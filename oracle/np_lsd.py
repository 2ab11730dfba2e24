"""ORACLE (test infrastructure only): plain numpy / Python-set restatement of localised statistics decoding of order 0
(LSD-0), written from the definition in ``csrc/fbgnn_lsd.cuh`` / DESIGN.md §4 and independent of ``lsd_oracle.c``:
clusters are explicit (set of checks, set of columns) pairs, merged pairwise until disjoint; validity is a GF(2) rank
comparison; the solution picks the independent columns greedily in rank order and solves on them.  It pins the C
oracle, which in turn pins ``k_lsd``."""
import numpy as np


def key(x, v):
    """osd_key: order-preserving map of float32 x to uint32, then the column index (-0.0 ranks before +0.0)."""
    u = int(np.array([x], np.float32).view(np.uint32)[0])
    u ^= 0xFFFFFFFF if u >> 31 else 0x80000000
    return (u << 32) | int(v)


def _rank(A):
    A = np.array(A, np.uint8) & 1
    r = 0
    rows, cols = A.shape
    for c in range(cols):
        hit = [i for i in range(r, rows) if A[i, c]]
        if not hit:
            continue
        A[[r, hit[0]]] = A[[hit[0], r]]
        for i in range(rows):
            if i != r and A[i, c]:
                A[i] ^= A[r]
        r += 1
        if r == rows:
            break
    return r


def _valid(H, s, C, V):
    rows, cols = sorted(C), sorted(V)
    sub = H[np.ix_(rows, cols)] if cols else np.zeros((len(rows), 0), np.uint8)
    return _rank(sub) == _rank(np.concatenate([sub, s[rows][:, None]], 1))


def _solve(H, s, C, V, keys):
    """The unique solution supported on the greedy independent columns (in rank order) of H[C, V]."""
    rows = sorted(C)
    order = sorted(V, key=lambda v: keys[v])
    P = []
    for v in order:
        if _rank(H[np.ix_(rows, P + [v])]) == len(P) + 1:
            P.append(v)
    A = np.concatenate([H[np.ix_(rows, P)], s[rows][:, None]], 1).astype(np.uint8)
    # Gaussian elimination on the independent columns; the last column is the right-hand side
    r = 0
    pivot_row = {}
    for j in range(len(P)):
        hit = [i for i in range(r, len(rows)) if A[i, j]]
        A[[r, hit[0]]] = A[[hit[0], r]]
        for i in range(len(rows)):
            if i != r and A[i, j]:
                A[i] ^= A[r]
        pivot_row[j] = r
        r += 1
    return {P[j]: int(A[pivot_row[j], -1]) for j in range(len(P))}


def lsd_frame(H, llr, s, max_cols, max_checks, sign=1.0, clusters_out=None):
    """LSD-0 of one frame: H [m,n], llr [n], s [m].  Returns (e [n] uint8, status); a solved frame's final clusters are
    appended to ``clusters_out`` when it is a list."""
    H = np.asarray(H, np.uint8) & 1
    s = np.asarray(s, np.uint8) & 1
    m, n = H.shape
    keys = [key(np.float32(sign) * np.float32(llr[v]), v) for v in range(n)]
    checks_of = [set(np.flatnonzero(H[:, v]).tolist()) for v in range(n)]
    cols_of = [set(np.flatnonzero(H[c]).tolist()) for c in range(m)]
    clusters = [({c}, set()) for c in range(m) if s[c]]
    while True:
        if sum(len(V) for _, V in clusters) > max_cols or sum(len(C) for C, _ in clusters) > max_checks:
            return np.zeros(n, np.uint8), 1
        valid = [_valid(H, s, C, V) for C, V in clusters]
        if all(valid):
            break
        clustered = set().union(*(V for _, V in clusters))
        picks = []
        for (C, V), ok in zip(clusters, valid):
            if ok:
                continue
            near = set().union(*(cols_of[c] for c in C)) - clustered
            if not near:
                return np.zeros(n, np.uint8), 2
            picks.append(min(near, key=lambda v: keys[v]))
        grown = []
        it = iter(picks)
        for (C, V), ok in zip(clusters, valid):
            if ok:
                grown.append((set(C), set(V)))
            else:
                v = next(it)
                grown.append((C | checks_of[v], V | {v}))
        merged = True
        while merged:                                   # unite clusters that share a check, until none do
            merged = False
            for i in range(len(grown)):
                for j in range(i + 1, len(grown)):
                    if grown[i][0] & grown[j][0]:
                        grown[i] = (grown[i][0] | grown[j][0], grown[i][1] | grown[j][1])
                        del grown[j]
                        merged = True
                        break
                if merged:
                    break
        clusters = grown
    if clusters_out is not None:
        clusters_out.extend(clusters)
    e = np.zeros(n, np.uint8)
    for C, V in clusters:
        for v, x in _solve(H, s, C, V, keys).items():
            e[v] = x
    return e, 0


def lsd(H, llr, s, max_cols, max_checks, sign=1.0):
    """lsd_frame over a batch: llr [B,n], s [m,B] -> (e_hat [B,n] uint8, status [B] uint8)."""
    llr, s = np.asarray(llr), np.asarray(s)
    out = [lsd_frame(H, llr[b], s[:, b], max_cols, max_checks, sign) for b in range(llr.shape[0])]
    return np.stack([e for e, _ in out]), np.array([st for _, st in out], np.uint8)
