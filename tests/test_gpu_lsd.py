"""LSD-0 on the GPU: k_lsd against the CPU oracle, bit for bit on e_hat and status -- small codes, [[882,24]],
[[1270,28]], [[1922,50]] and [[7688,50]] (whose OSD basis no CTA cluster holds), at the default and at small budgets --
and the layer's argument checks."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lsd(oracle):
    from oracle import lsd_oracle
    lsd_oracle.build()
    return lsd_oracle


def _hp(L):
    import fbgnn as F
    h = F.create_circulant_matrix(L, [0, 2, 5])
    return F.hypergraph_product(h, h)


def _frames(H, B, seed, p, tie_stride=7):
    """Reliabilities low on the error's columns, with ties every tie_stride-th column (broken by index) and a few
    signed zeros (-0.0 ranks before +0.0 on both sides), and the syndromes of the errors."""
    rng = np.random.default_rng(seed)
    n = H.shape[1]
    noise = (rng.random((B, n)) < p).astype(np.int64)
    llr = rng.normal(3, 1, (B, n)).astype(np.float32)
    llr[noise == 1] -= 2.5 if tie_stride <= 7 else 4.0
    llr[:, ::tie_stride] = 1.25
    llr[:, 5::max(11, 8 * tie_stride)] = -0.0
    llr[:, 6::max(11, 8 * tie_stride)] = 0.0
    s = ((np.asarray(H, np.int64) @ noise.T) & 1).astype(np.uint8)
    return llr, s


def _check(H, lsd, llr, s, budgets):
    import fbgnn as F
    H = np.asarray(H)
    n = H.shape[1]
    seen = set()
    for mc, mk in budgets:
        dec = F.LSD_Decoder(n, max_cols=mc, max_checks=mk)
        e = dec(llr, H, s, llr.shape[0])
        ref_e, ref_st = lsd.lsd(H, llr, s, mc, mk)
        assert e.dtype == bool and np.array_equal(dec.last_status, ref_st), (mc, mk)
        assert np.array_equal(e.astype(np.uint8), ref_e), (mc, mk)
        ok = ref_st == 0
        assert np.array_equal((H.astype(np.int64) @ e[ok].T.astype(np.int64)) & 1, s[:, ok])
        seen |= set(ref_st.tolist())
    return seen


_SMALL = [(0, 0), (8, 12), (512, 512)]


@pytest.mark.parametrize("name,p", [("steane", 0.15), ("rsurf3", 0.15), ("toric4", 0.1), ("gb48", 0.06),
                                    ("c882", 0.03)])
@pytest.mark.parametrize("matrix", ["full", "basis"])
def test_layer_bitexact(codes, lsd, name, p, matrix):
    code = codes[name]
    H = code.hx if matrix == "full" else code.hx_basis
    llr, s = _frames(H, 64, seed=3, p=p)
    _check(H, lsd, llr, s, _SMALL)


def test_layer_bitexact_c1270(c1270, lsd):
    llr, s = _frames(c1270.hx, 48, seed=4, p=0.02, tie_stride=97)
    _check(c1270.hx, lsd, llr, s, _SMALL)


@pytest.mark.parametrize("side", ["hx", "hz"])
def test_layer_bitexact_1922(lsd, side):
    code = _hp(31)
    H = code.hx if side == "hx" else code.hz
    llr, s = _frames(H, 48, seed=5, p=0.01, tie_stride=97)
    seen = _check(H, lsd, llr, s, _SMALL)
    assert 0 in seen and 1 in seen                      # both solved and abandoned frames were compared


def test_layer_bitexact_7688(lsd):
    """[[7688,50]]: OSD refuses its basis (test_gpu_osd_cluster.py); LSD-0 decodes the full hx."""
    code = _hp(62)
    assert (code.N, code.K) == (7688, 50)
    llr, s = _frames(code.hx, 24, seed=6, p=0.003, tie_stride=97)
    seen = _check(code.hx, lsd, llr, s, [(0, 0), (512, 512), (16, 24)])
    assert 0 in seen


def test_inconsistent_syndrome_status_2(lsd):
    import fbgnn as F
    n = 12
    H = np.zeros((n, n), np.uint8)                      # a ring: only even-weight syndromes are reachable
    for i in range(n):
        H[i, i] = H[i, (i + 1) % n] = 1
    llr = np.random.default_rng(7).normal(0, 1, (3, n)).astype(np.float32)
    s = np.zeros((n, 3), np.uint8)
    s[4, 0] = 1                                         # odd: status 2
    s[[1, 7], 1] = 1                                    # even: solved
    dec = F.LSD_Decoder(n)
    e = dec(llr, H, s, 3)
    ref_e, ref_st = lsd.lsd(H, llr, s)
    assert list(dec.last_status) == list(ref_st) == [2, 0, 0]
    assert np.array_equal(e.astype(np.uint8), ref_e)


def test_budget_validation(codes):
    import fbgnn as F
    from fbgnn import _ffi
    code = codes["gb48"]
    g = _ffi.Graph(code.hx)
    ctx = g.ctx
    llr, s = _frames(code.hx, 4, seed=8, p=0.05)
    llr_d, s_d = ctx.asarray(llr, np.float32), ctx.asarray(s, np.uint8)
    e = ctx.empty((4, code.N), np.uint8)
    for mc, mk in ((-1, 0), (513, 0), (0, -1), (0, 513)):
        with pytest.raises(F.FbgnnError, match=f"fbgnn error {-1}"):           # FBGNN_E_INVALID
            _ffi.call("fbgnn_lsd_decode", g.handle, mc, mk, 4, llr_d.t2(), s_d.t2(), e.t2(), None)
    _ffi.call("fbgnn_lsd_decode", g.handle, 512, 1, 4, llr_d.t2(), s_d.t2(), e.t2(), None)   # status is optional
    with pytest.raises(ValueError):
        F.LSD_Decoder(code.N)(llr[:, :-1], code.hx, s, 4)


# ---------------------------------------------------------------------------------------------- pipelines ----------
# (code, p, BP4 iterations, frames, LSD budgets): BP4 (min-sum, factor 0.8) leaves failed frames at these points, and
# LSD-0 solves some of them and abandons others
_BP4_CASES = {"c882": (0.09, 20, 300, (0, 0)), "hp1922": (0.05, 12, 96, (0, 0)), "hp7688": (0.03, 3, 24, (512, 512))}


def _code(codes, name):
    return codes[name] if name in codes else _hp(31 if name == "hp1922" else 62)


@pytest.mark.parametrize("name", list(_BP4_CASES))
@pytest.mark.parametrize("skip", [False, True])
def test_bp4_lsd_pipeline_bitexact(codes, oracle, lsd, name, skip):
    import fbgnn as F
    code = _code(codes, name)
    p, it, B, (mc, mk) = _BP4_CASES[name]
    dec = F.QLDPCBPDecoder(code, num_iter=it, normalization_factor=0.8, cn_type="minsum", stage_one=True)
    model = F.BP4_OSD_Model(code, dec, F.LSD_Decoder(code.N, max_cols=mc, max_checks=mk), seed=4)
    model._inner.skip_inactive = skip
    res = model.run(B, p, want_counters=True)
    ref = lsd.pipeline(oracle.CodeGraph(code), [it], [], p, p0=None, factors=[0.8], cn_types=["minsum"], seed=4, B=B,
                       want_diff=True, max_cols=mc, max_checks=mk)
    assert np.array_equal(res["flags"].numpy(), ref["flags"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])
    assert np.array_equal(res["counters"], ref["counters"])
    bp4 = F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, p0=None, seed=4).run(B, p, want_counters=True)
    assert res["counters"][1] == ref["unsolved"].sum()            # flagged == frames LSD-0 left unsolved
    assert res["counters"][1] < bp4["counters"][1]                 # LSD-0 ran and solved frames BP4 failed


@pytest.mark.parametrize("name,p", [("c882", 0.03), ("hp1922", 0.02)])
def test_bp2_lsd_pipeline_bitexact(codes, lsd, name, p):
    import fbgnn as F
    code = _code(codes, name)
    dec = F.LDPCBPDecoder(code.hx, is_syndrome=True, hard_out=False, cn_type="minsum", num_iter=20, normalization_factor=0.8)
    model = F.BP2_OSD_Model(code.hx, code.hx_basis, code.pivot_hx, code.lx, dec, F.LSD_Decoder(code.N), seed=6)
    B = 1000
    res = model.run(B, p, want_counters=True)
    ref = lsd.bsc_pipeline(code.hx, code.lx, 20, p, factor=0.8, cn_type="minsum", seed=6, B=B)
    assert np.array_equal(res["flags"].numpy(), ref["flags"]) and np.array_equal(res["counters"], ref["counters"])
    assert res["counters"][1] == ref["unsolved"].sum()
    bp2 = F.BP_BSC_Model(code.hx, dec, logical_pcm=code.lx, seed=6).run(B, p, want_counters=True)
    assert res["counters"][1] < bp2["counters"][1]


@pytest.mark.parametrize("name,p", [("c882", 0.12), ("hp1922", 0.06)])
def test_sandwich_then_lsd_bitexact(codes, oracle, lsd, weights, name, p):
    import fbgnn as F
    from fbgnn.feedback_gnn import unpack_bits
    code = _code(codes, name)
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
    G.set_weights(weights["c882"])
    d1 = F.QLDPCBPDecoder(code, num_iter=8, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code, num_iter=4, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    B = 96
    ref = lsd.pipeline(oracle.CodeGraph(code), [8, 4], [oracle.Gnn(weights["c882"])], p, seed=3, B=B, want_diff=True)
    model = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1, d2], [G], num_layers=2, seed=3, lsd=F.LSD_Decoder(code.N))
    res = model.run(B, p, want_counters=True)
    assert np.array_equal(res["flags"].numpy(), ref["flags"]) and np.array_equal(res["counters"], ref["counters"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])
    model = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1, d2], [G], num_layers=2, seed=3, lsd=F.LSD_Decoder(code.N))
    rb = model.run_bits(B, p, want_diff=True, want_counters=True)
    planes = rb["frame_bits"].numpy()
    flagged = (planes[0][np.arange(B) >> 5] >> (np.arange(B) & 31)) & 1
    assert np.array_equal(flagged.astype(np.uint8), ref["flags"] & 1)
    assert np.array_equal(rb["counters"], ref["counters"])
    assert np.array_equal(unpack_bits(rb["x_diff_bits"].numpy(), code.N), ref["x_diff"])
    assert ref["counters"][1] == ref["unsolved"].sum()


def test_pipeline_budget_validation(codes):
    import fbgnn as F
    code = codes["gb48"]
    dec = F.QLDPCBPDecoder(code, num_iter=4, cn_type="minsum", stage_one=True)
    model = F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, lsd=F.LSD_Decoder(code.N))
    model.lsd.max_cols = 513                                       # past the layer's own check
    with pytest.raises(F.FbgnnError, match=f"fbgnn error {-1}"):
        model.run(8, 0.05)
    bsc = F.BP_BSC_Model(code.hx, F.LDPCBPDecoder(code.hx, is_syndrome=True, hard_out=False, num_iter=4),
                         logical_pcm=code.lx)
    bsc._lsd = F.LSD_Decoder(code.N)
    bsc._lsd.max_checks = -1
    with pytest.raises(F.FbgnnError, match=f"fbgnn error {-1}"):
        bsc.run(8, 0.05)
