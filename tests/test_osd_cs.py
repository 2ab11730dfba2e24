"""OSD-CS (the combination sweep of ordered-statistics decoding) in the CPU oracle: the C oracle against its numpy
restatement, properties of the candidate sweep, OSD-0 unchanged at order 0, and the Python layer's argument checks."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def cs(oracle):
    from oracle import osd_cs_oracle
    osd_cs_oracle.build()
    return osd_cs_oracle


def _frames(code, B, seed, full=False):
    """Random reliabilities with forced ties, and the syndromes on hx of random errors reduced to the basis rows."""
    rng = np.random.default_rng(seed)
    n = code.N
    llr = rng.normal(2, 1.5, (B, n)).astype(np.float32)
    llr[:, ::7] = 1.25                                   # ties: broken by index
    noise = (rng.random((B, n)) < 0.3).astype(np.int64)
    s = ((code.hx.astype(np.int64) @ noise.T) & 1).astype(np.uint8)
    red = np.ascontiguousarray(s[code.pivot_hx])
    return (code.hx_basis, llr, red, s) if full else (code.hx_basis, llr, red)


def _orders(code):
    R, n = code.hx_basis.shape
    return (0, 1, 2, 5, n - R, n - R + 7)


def _weight(e):
    return e.astype(np.int64).sum(1)


@pytest.mark.parametrize("name", ["steane", "rsurf3", "toric4", "gb48", "c882"])
def test_numpy_restatement_equals_c_oracle(codes, cs, name):
    from oracle import np_osd_cs
    code = codes[name]
    basis, llr, red = _frames(code, 3 if name == "c882" else 12, seed=5)
    R, n = basis.shape
    for lam in _orders(code):
        B = 2 if name == "c882" and lam >= n - R else llr.shape[0]      # the full pair sweep of [[882,24]] is slow in numpy
        ref = np_osd_cs.osd_cs(basis, llr[:B], red[:, :B], lam)
        got = cs.osd(basis, llr[:B], np.ascontiguousarray(red[:, :B]), lam)
        assert np.array_equal(got, ref), (name, lam)


@pytest.mark.parametrize("name", ["steane", "rsurf3", "toric4", "gb48", "c882"])
def test_order_zero_is_osd0(codes, oracle, cs, name):
    code = codes[name]
    basis, llr, red = _frames(code, 16, seed=6)
    assert np.array_equal(cs.osd(basis, llr, red, 0), oracle.osd0(basis, llr, red))


@pytest.mark.parametrize("name", ["steane", "rsurf3", "toric4", "gb48", "c882"])
def test_osd_cs_properties(codes, cs, name):
    """Every solution meets the full syndrome; OSD-CS is never heavier than OSD-0 and its weight does not grow with the
    order; on the small codes no listed candidate is lighter than the one returned."""
    from oracle import np_osd_cs
    code = codes[name]
    basis, llr, red, s = _frames(code, 24, seed=7, full=True)
    R, n = basis.shape
    prev = None
    for lam in (0, 1, 2, 5, 10, n - R):
        e = cs.osd(basis, llr, red, lam)
        assert np.array_equal((code.hx.astype(np.int64) @ e.T.astype(np.int64)) & 1, s)
        w = _weight(e)
        if prev is not None:
            assert np.all(w <= prev), (name, lam)
        prev = w
        if name != "c882":
            for b in range(llr.shape[0]):
                _, weights = np_osd_cs.osd_cs_frame(basis, llr[b], red[:, b], lam)
                assert w[b] == weights.min(), (name, lam, b)


def test_osd_cs_finds_lighter_solutions(codes, cs):
    """On [[882,24]] with syndromes of light errors, the sweep does find strictly lighter solutions than OSD-0."""
    code = codes["c882"]
    rng = np.random.default_rng(8)
    B, n = 32, code.N
    noise = (rng.random((B, n)) < 0.05).astype(np.uint8)
    red = np.ascontiguousarray(((code.hx_basis.astype(np.int64) @ noise.T) & 1).astype(np.uint8))
    llr = rng.normal(3, 1, (B, n)).astype(np.float32)
    w0 = _weight(cs.osd(code.hx_basis, llr, red, 0))
    w10 = _weight(cs.osd(code.hx_basis, llr, red, 10))
    assert np.all(w10 <= w0) and np.any(w10 < w0)


def test_pipelines_at_order_zero_match_osd0(codes, oracle, cs):
    """BP4 + OSD and BP2 + OSD at order 0 reproduce the oracle's OSD-0 pipelines; order 10 changes the residual errors
    of some frames and still meets every syndrome."""
    code = codes["c882"]
    g = oracle.CodeGraph(code)
    kw = dict(p0=None, factors=[0.8], cn_types=["minsum"], seed=4, B=200, want_diff=True)
    ref = oracle.pipeline(g, [30], [], 0.11, osd0=True, **kw)
    r = cs.pipeline(g, [30], [], 0.11, osd_order=0, **kw)
    for k in ("flags", "counters", "x_diff", "z_diff"):
        assert np.array_equal(r[k], ref[k]), k
    bkw = dict(factor=0.8, cn_type="minsum", seed=6, B=1000)
    bref = oracle.bsc_pipeline(code.hx, code.lx, 30, 0.06, osd_basis=code.hx_basis, osd_pivot=code.pivot_hx, **bkw)
    b = cs.bsc_pipeline(code.hx, code.lx, 30, 0.06, code.hx_basis, code.pivot_hx, osd_order=0, **bkw)
    assert np.array_equal(b["flags"], bref["flags"]) and np.array_equal(b["counters"], bref["counters"])
    r10 = cs.pipeline(g, [30], [], 0.11, osd_order=10, **kw)
    assert r10["counters"][1] == 0                                   # OSD-CS meets the syndrome as OSD-0 does
    assert not np.array_equal(r10["x_diff"], ref["x_diff"])


def test_sandwich_pipeline_at_order_zero_matches_osd0(codes, oracle, cs, weights):
    """The same after BP -> GNN -> BP with round skipping, and in the SFU arithmetic."""
    code = codes["c882"]
    g = oracle.CodeGraph(code)
    G = oracle.Gnn(weights["c882"])
    for math in ("exact", "sfu"):
        with oracle.math(math):
            kw = dict(seed=8, B=60, want_diff=True, skip_inactive=True)
            ref = oracle.pipeline(g, [12, 12], [G], 0.12, osd0=True, **kw)
            r = cs.pipeline(g, [12, 12], [G], 0.12, osd_order=0, **kw)
        for k in ("flags", "counters", "x_diff", "z_diff"):
            assert np.array_equal(r[k], ref[k]), (math, k)


def test_osd_decoder_validation():
    import fbgnn as F
    with pytest.raises(ValueError):
        F.OSD_Decoder(10, osd_order=-1)
    with pytest.raises(ValueError):
        F.OSD_Decoder(10, osd_order=65536)
    with pytest.raises(ValueError):
        F.OSD_Decoder(10, osd_order=4, osd_method="osd_e")
    assert F.OSD_Decoder(10, osd_order=7).osd_order == 7
    assert F.OSD_Decoder(10, osd_order=7, osd_method="osd0").osd_order == 0
    assert F.OSD0_Decoder(10).osd_order == 0 and isinstance(F.OSD0_Decoder(10), F.OSD_Decoder)


def test_models_take_the_order_of_their_osd_decoder(codes):
    import fbgnn as F
    code = codes["steane"]
    dec = F.QLDPCBPDecoder(code, num_iter=4, cn_type="minsum", stage_one=True)
    assert F.BP4_OSD_Model(code, dec, F.OSD_Decoder(code.N, osd_order=3))._inner.osd_order == 3
    assert F.BP4_OSD_Model(code, dec, F.OSD0_Decoder(code.N))._inner.osd_order == 0
    with pytest.raises(ValueError):
        F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, osd0=True, osd_order=-2)
