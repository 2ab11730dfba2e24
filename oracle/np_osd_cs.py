"""ORACLE (test infrastructure only): numpy restatement of ordered-statistics decoding with the combination sweep
(OSD-CS; Roffe et al. 2020, the ``ldpc`` package's ``osd_method="osd_cs"``).  Independent of ``osd_cs_oracle.c``:
dense boolean elimination with the same row-wise pivot rule, then the candidate list written out explicitly.  It pins
the C oracle, which in turn pins ``k_osd``."""
import numpy as np

F = np.float32


def osd_cs_frame(basis, llr, s, order):
    """Ordered-statistics decoding of one frame with the combination sweep of order ``order`` (OSD-CS; 0 = OSD-0),
    restated on dense boolean arrays.  basis [R,n] full-rank rows, llr [n], s [R].  Returns (e_hat [n] uint8, weights):
    ``weights[t]`` is the Hamming weight of candidate t's solution, candidates in their index order -- the empty set,
    every single non-pivot column (order > 0), then the pairs of the first min(order, n - R) non-pivot columns in
    lexicographic order."""
    basis = np.asarray(basis, bool)
    R, n = basis.shape
    perm = np.argsort(np.asarray(llr, F), kind="stable")          # ascending reliability, ties by index
    aug = np.concatenate([basis[:, perm], np.asarray(s, bool)[:, None]], 1)
    piv = np.zeros(R, np.int64)
    for r in range(R):                                             # row-wise: the first remaining one of row r
        nz = np.flatnonzero(aug[r, :n])
        p = nz[0] if len(nz) else 0
        hit = aug[:, p].copy()
        hit[r] = False
        aug[hit] ^= aug[r]
        piv[r] = p
    sp = aug[:, n]
    nonpiv = np.setdiff1d(np.arange(n), piv)                       # increasing permuted position
    cands = [()]
    if order > 0:
        lp = min(order, max(n - R, 0))
        I, J = np.triu_indices(lp, k=1)                            # i < j, lexicographic
        cands += [(int(c),) for c in nonpiv] + [(int(nonpiv[i]), int(nonpiv[j])) for i, j in zip(I, J)]
    weights = np.empty(len(cands), np.int64)
    sols = []
    for t, T in enumerate(cands):
        sol = sp.copy()
        for c in T:
            sol ^= aug[:, c]
        weights[t] = int(sol.sum()) + len(T)
        sols.append(sol)
    best = int(np.argmin(weights))                                 # least weight, then least index
    e = np.zeros(n, np.uint8)
    e[perm[piv]] = sols[best]
    for c in cands[best]:
        e[perm[c]] = 1
    return e, weights


def osd_cs(basis, llr, s, order):
    """osd_cs_frame over a batch: llr [B,n], s [R,B] -> e_hat [B,n] uint8."""
    llr, s = np.asarray(llr), np.asarray(s)
    return np.stack([osd_cs_frame(basis, llr[b], s[:, b], order)[0] for b in range(llr.shape[0])])

