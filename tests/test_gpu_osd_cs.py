"""BP + OSD-CS: the order-λ combination sweep of k_osd against the CPU oracle, bit for bit -- the layer, the BP4 and BP2
OSD models and the Sandwich pipeline followed by OSD-CS."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cs(oracle):
    from oracle import osd_cs_oracle
    osd_cs_oracle.build()
    return osd_cs_oracle


def _frames(code, B, seed):
    rng = np.random.default_rng(seed)
    n = code.N
    noise = (rng.random((B, n)) < 0.06).astype(np.uint8)
    synd = ((code.hx @ noise.T.astype(np.int64)) & 1).astype(np.uint8)
    llr = rng.normal(3, 1, (B, n)).astype(np.float32)
    llr[noise == 1] -= 2.5
    llr[:, ::7] = 1.25                                  # ties: broken by index on both sides
    return llr, synd, np.ascontiguousarray(synd[code.pivot_hx])


def _check_layer(code, cs, orders, B, seed):
    import fbgnn as F
    llr, synd, red = _frames(code, B, seed)
    basis = code.hx_basis
    for lam in orders:
        e = F.OSD_Decoder(code.N, osd_order=lam)(llr, basis, red, B)
        ref = cs.osd(basis, llr, red, lam)
        assert e.dtype == bool and np.array_equal(e.astype(np.uint8), ref), (code.name, lam)
        assert np.array_equal((code.hx @ e.T.astype(np.int64)) & 1, synd)   # satisfies the full syndrome


@pytest.mark.parametrize("name", ["c882", "gb48", "rsurf3"])
def test_osd_cs_layer_bitexact(codes, cs, name):
    code = codes[name]
    R, n = code.hx_basis.shape
    _check_layer(code, cs, (1, 8, 60, n - R), B=40, seed=2)


def test_osd_cs_layer_bitexact_c1270(c1270, cs):
    """[[1270,28]] at λ = 60: the largest shared-memory footprint of the kernel."""
    _check_layer(c1270, cs, (60,), B=24, seed=3)


def test_order_zero_equals_osd0_decode(codes):
    import fbgnn as F
    for name in ("c882", "gb48"):
        code = codes[name]
        llr, _, red = _frames(code, 40, 4)
        basis = code.hx_basis
        e0 = F.OSD0_Decoder(code.N)(llr, basis, red, 40)                       # fbgnn_osd0_decode
        e = F.OSD_Decoder(code.N, osd_order=0)(llr, basis, red, 40)             # fbgnn_osd_decode, order 0
        assert np.array_equal(e, e0)


def test_negative_order_is_invalid(codes):
    import fbgnn as F
    from fbgnn import _ffi
    code = codes["gb48"]
    llr, _, red = _frames(code, 4, 5)
    g = _ffi.Graph(code.hx_basis)
    ctx = g.ctx
    llr_d, s_d = ctx.asarray(llr, np.float32), ctx.asarray(red, np.uint8)
    e = ctx.empty((4, code.N), np.uint8)
    for bad in (-1, 65536):
        with pytest.raises(F.FbgnnError, match=f"fbgnn error {-1}"):           # FBGNN_E_INVALID
            _ffi.call("fbgnn_osd_decode", g.handle, bad, 4, llr_d.t2(), s_d.t2(), e.t2())


@pytest.mark.parametrize("skip", [False, True])
def test_bp4_osd_cs_pipeline_bitexact(codes, oracle, cs, skip):
    import fbgnn as F
    code = codes["c882"]
    dec = F.QLDPCBPDecoder(code, num_iter=30, normalization_factor=0.8, cn_type="minsum", stage_one=True)
    model = F.BP4_OSD_Model(code, dec, F.OSD_Decoder(code.N, osd_order=10), seed=4)
    model._inner.skip_inactive = skip
    B, p = 600, 0.11
    res = model.run(B, p, want_counters=True)
    ref = cs.pipeline(oracle.CodeGraph(code), [30], [], p, p0=None, factors=[0.8], cn_types=["minsum"], seed=4,
                      B=B, want_diff=True, osd_order=10)
    assert np.array_equal(res["flags"].numpy(), ref["flags"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])
    assert np.array_equal(res["counters"], ref["counters"])
    assert res["counters"][1] == 0                               # OSD-CS always meets the syndrome


def test_sandwich_then_osd_cs_bitexact(codes, oracle, cs, weights):
    import fbgnn as F
    code = codes["c882"]
    G = F.Feedback_GNN(code=code, num_msg_dims=20, num_hidden_units=40, num_mlp_layers=2, use_bias=True)
    G.set_weights(weights["c882"])
    d = F.QLDPCBPDecoder(code, num_iter=12, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    model = F.Sandwich_BP_GNN_Evaluation_Model(code, [d, d], [G], num_layers=2, seed=8, osd0=True, osd_order=10)
    res = model.run(300, 0.12, want_counters=True)
    ref = cs.pipeline(oracle.CodeGraph(code), [12, 12], [oracle.Gnn(weights["c882"])], 0.12, seed=8, B=300,
                      want_diff=True, osd_order=10)
    assert np.array_equal(res["flags"].numpy(), ref["flags"]) and np.array_equal(res["counters"], ref["counters"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])


def test_bp2_osd_cs_pipeline_bitexact(codes, cs):
    import fbgnn as F
    code = codes["c882"]
    dec = F.LDPCBPDecoder(code.hx, is_syndrome=True, hard_out=False, cn_type="minsum", num_iter=30, normalization_factor=0.8)
    model = F.BP2_OSD_Model(code.hx, code.hx_basis, code.pivot_hx, code.lx, dec, F.OSD_Decoder(code.N, osd_order=10),
                            seed=6)
    B, p = 3000, 0.06
    res = model.run(B, p, want_counters=True)
    ref = cs.bsc_pipeline(code.hx, code.lx, 30, p, code.hx_basis, code.pivot_hx, factor=0.8, cn_type="minsum", seed=6,
                          B=B, osd_order=10)
    assert np.array_equal(res["flags"].numpy(), ref["flags"]) and np.array_equal(res["counters"], ref["counters"])
    assert res["counters"][1] == 0
