"""LSD-0 (localised statistics decoding of order 0) in the CPU oracle: the C oracle against its numpy restatement,
hand-worked answers on a repetition-code chain, H e = s on every solved frame, OSD-0 when one cluster holds every
column, and the Python layer's argument checks."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def lsd(oracle):
    from oracle import lsd_oracle
    lsd_oracle.build()
    return lsd_oracle


@pytest.fixture(scope="module")
def hp1922():
    import fbgnn as F
    h = F.create_circulant_matrix(31, [0, 2, 5])
    return F.hypergraph_product(h, h)


def _frames(H, B, seed, p):
    """Reliabilities with forced ties (low on the error's columns) and the syndromes of random errors on H."""
    rng = np.random.default_rng(seed)
    n = H.shape[1]
    noise = (rng.random((B, n)) < p).astype(np.int64)
    llr = rng.normal(3, 1, (B, n)).astype(np.float32)
    llr[noise == 1] -= 2.5
    llr[:, ::7] = 1.25                                   # ties: broken by index
    s = ((np.asarray(H, np.int64) @ noise.T) & 1).astype(np.uint8)
    return llr, s


_P = {"steane": 0.15, "rsurf3": 0.15, "toric4": 0.1, "gb48": 0.06, "c882": 0.02, "hp1922": 0.02}


@pytest.mark.parametrize("name", ["steane", "rsurf3", "toric4", "gb48", "c882", "hp1922"])
@pytest.mark.parametrize("matrix", ["full", "basis"])
def test_numpy_restatement_equals_c_oracle(codes, hp1922, lsd, name, matrix):
    from oracle import np_lsd
    code = hp1922 if name == "hp1922" else codes[name]
    H = np.asarray(code.hx if matrix == "full" else code.hx_basis)
    B = 4 if name in ("c882", "hp1922") else 16
    llr, s = _frames(H, B, seed=5, p=_P[name])
    for mc, mk in ((0, 0), (6, 10), (40, 512)):
        e, st = lsd.lsd(H, llr, s, mc, mk)
        ref_e, ref_st = np_lsd.lsd(H, llr, s, mc or 256, mk or 256)
        assert np.array_equal(st, ref_st) and np.array_equal(e, ref_e), (name, matrix, mc, mk)
        for b in np.flatnonzero(st == 0):                    # a solved frame meets its syndrome
            assert np.array_equal((H.astype(np.int64) @ e[b]) & 1, s[:, b])
        assert not e[st != 0].any()                           # an abandoned frame gets e = 0


def _chain(n=8, ring=False):
    """Repetition-code chain: row i checks columns i and i + 1 (a ring closes it with row n - 1 on n - 1 and 0)."""
    H = np.zeros((n if ring else n - 1, n), np.uint8)
    for i in range(H.shape[0]):
        H[i, i] = H[i, (i + 1) % n] = 1
    return H


def _one(lsd, H, llr, rows, **kw):
    s = np.zeros((H.shape[0], 1), np.uint8)
    s[list(rows), 0] = 1
    e, st = lsd.lsd(H, np.asarray([llr], np.float32), s, **kw)
    return list(np.flatnonzero(e[0])), int(st[0])


def test_chain_two_defects_grow_and_meet(lsd):
    # error on columns 3, 4: defects on rows 2 and 4; each takes its least reliable neighbour (3 and 4), and the two
    # clusters meet on row 3
    assert _one(lsd, _chain(), [5, 5, 5, 0, 0.5, 5, 5, 5], (2, 4)) == ([3, 4], 0)


def test_chain_two_clusters_pick_the_same_column(lsd):
    # defects on rows 2 and 3 both pick column 3 in the first round: one cluster, valid
    assert _one(lsd, _chain(), [5, 5, 4, 0, 4, 5, 5, 5], (2, 3)) == ([3], 0)


def test_chain_valid_cluster_absorbed_by_a_growing_neighbour(lsd):
    # round 1: rows 1, 2 take column 2 (valid); row 4 takes column 4 (checks 3, 4: invalid).  Round 2: it takes column
    # 3, whose check 2 unites it with the valid cluster: checks 1..4, columns 2, 3, 4, still invalid.  Rounds 3, 4, 5
    # add columns 5, 1 (tie with 6 by index) and 0; checks 0..5 over columns 0..5 are then full rank, and the unique
    # solution is {0, 1, 3, 4}.
    llr = [5, 5, 0, 1, 0.5, 2, 5, 5]
    assert _one(lsd, _chain(), llr, (1, 2, 4)) == ([0, 1, 3, 4], 0)
    # the same frame abandoned once its clusters hold more than two columns (after round 2)
    assert _one(lsd, _chain(), llr, (1, 2, 4), max_cols=2) == ([], 1)
    assert _one(lsd, _chain(), llr, (1, 2, 4), max_cols=3) == ([], 1)
    assert _one(lsd, _chain(), llr, (1, 2, 4), max_checks=3) == ([], 1)        # four checks after round 1
    assert _one(lsd, _chain(), llr, (1, 2, 4), max_checks=2) == ([], 1)        # three defects: over at the start


def test_inconsistent_syndrome_has_status_2(lsd):
    # a ring has even-weight syndromes only: one defect grows over every column, then has no candidate
    assert _one(lsd, _chain(ring=True), [1, 2, 3, 4, 5, 6, 7, 8], (3,)) == ([], 2)
    assert _one(lsd, _chain(ring=True), [1, 2, 3, 4, 5, 6, 7, 8], (3,), max_cols=4) == ([], 1)


def test_one_cluster_over_every_column_is_osd0(codes, lsd):
    """Where the final partition is one cluster holding every column, LSD-0 is OSD-0 on that (full-rank) matrix.  Growth
    reaches every column on a bidiagonal square chain when the defect's far end is the most reliable column; the small
    codes' bases add the frames where it happens by chance.  Inputs without signed zeros: the CPU OSD-0 compares floats."""
    from oracle import np_lsd, osd_cs_oracle
    rng = np.random.default_rng(9)
    sq = _chain(9)[:8, :8].copy()
    sq[7, 7] = 1                                          # row 7 checks column 7 only: 8 x 8, full rank
    cases = [(sq, np.array([9, 1, 2, 3, 4, 5, 6, 7], np.float32), np.eye(8, dtype=np.uint8)[0])]
    for _ in range(48):
        cases.append((sq, rng.normal(0, 1, 8).astype(np.float32), rng.integers(0, 2, 8).astype(np.uint8)))
    for name in ("steane", "rsurf3", "toric4"):
        H = np.asarray(codes[name].hx_basis)
        for _ in range(48):
            cases.append((H, rng.normal(0, 1, H.shape[1]).astype(np.float32), rng.integers(0, 2, H.shape[0]).astype(np.uint8)))
    hits = 0
    for H, llr, s in cases:
        cl = []
        ref_e, st = np_lsd.lsd_frame(H, llr, s, 256, 256, clusters_out=cl)
        if st or len(cl) != 1 or len(cl[0][1]) != H.shape[1]:
            continue
        e, st = lsd.lsd(H, llr[None], s[:, None])
        osd0 = osd_cs_oracle.osd(H, llr[None], np.ascontiguousarray(s[:, None]), 0)
        assert st[0] == 0 and np.array_equal(e, osd0) and np.array_equal(e[0], ref_e)
        hits += 1
    assert hits >= 2


def test_lsd_decoder_validation():
    import fbgnn as F
    for bad in (dict(max_cols=-1), dict(max_cols=513), dict(max_checks=-1), dict(max_checks=513)):
        with pytest.raises(ValueError):
            F.LSD_Decoder(10, **bad)
    d = F.LSD_Decoder(10, max_cols=7, max_checks=512)
    assert (d.max_cols, d.max_checks, d.last_status) == (7, 512, None)


def test_models_route_an_lsd_decoder(codes):
    import fbgnn as F
    code = codes["steane"]
    dec = F.QLDPCBPDecoder(code, num_iter=4, cn_type="minsum", stage_one=True)
    lsd = F.LSD_Decoder(code.N, max_cols=20, max_checks=30)
    inner = F.BP4_OSD_Model(code, dec, lsd)._inner
    assert inner.lsd is lsd and not inner.osd0
    assert F.BP4_OSD_Model(code, dec, F.OSD0_Decoder(code.N))._inner.lsd is None
    with pytest.raises(ValueError):
        F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, osd0=True, lsd=lsd)
    with pytest.raises(TypeError):
        F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, lsd=F.OSD0_Decoder(code.N))


def test_pipeline_oracles_flag_exactly_the_unsolved_frames(codes, oracle, lsd):
    """After LSD-0 a frame stays flagged exactly when LSD-0 abandoned a side whose BP decision missed its syndrome; with
    a budget no frame can meet, the BP decisions (and so the flags) are those of the pipeline without post-processing."""
    code = codes["c882"]
    g = oracle.CodeGraph(code)
    kw = dict(p0=None, factors=[0.8], cn_types=["minsum"], seed=4, B=200, want_diff=True)
    bp = oracle.pipeline(g, [20], [], 0.09, **kw)
    for mc, mk in ((0, 0), (12, 16), (1, 1)):
        r = lsd.pipeline(g, [20], [], 0.09, max_cols=mc, max_checks=mk, **kw)
        assert np.array_equal(r["flags"] & 1, r["unsolved"]), (mc, mk)
        assert r["counters"][1] == r["unsolved"].sum()
        assert r["unsolved"].sum() <= bp["counters"][1]
    assert np.array_equal(r["x_diff"], bp["x_diff"]) and np.array_equal(r["z_diff"], bp["z_diff"])
    assert bp["counters"][1] > 0
    bkw = dict(factor=0.8, cn_type="minsum", seed=6, B=1000)
    bbp = oracle.bsc_pipeline(code.hx, code.lx, 20, 0.03, **bkw)
    for mc, mk in ((0, 0), (12, 16)):
        b = lsd.bsc_pipeline(code.hx, code.lx, 20, 0.03, max_cols=mc, max_checks=mk, **bkw)
        assert np.array_equal(b["flags"] & 1, b["unsolved"]) and b["counters"][1] == b["unsolved"].sum()
        assert b["unsolved"].sum() <= bbp["counters"][1]
    assert b["unsolved"].sum() > 0                                  # the small budget abandons frames ...
    assert lsd.bsc_pipeline(code.hx, code.lx, 20, 0.03, **bkw)["unsolved"].sum() < bbp["counters"][1]   # ... LSD-0 solves some
