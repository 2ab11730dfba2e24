"""OSD on bases whose reduced matrix exceeds one SM's shared memory: the thread-block-cluster form of k_osd
(csrc/fbgnn_osd_cluster.cuh) against the CPU oracle and against k_osd itself, bit for bit -- the layer and the BP4 / BP2 /
Sandwich pipelines on the [[1922,50]] hypergraph-product code, every small code forced onto clusters of 2, 4 and 8 CTAs
with FBGNN_OSD_CLUSTER, and the clean refusal of [[7688,50]]."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cs(oracle):
    from oracle import osd_cs_oracle
    osd_cs_oracle.build()
    return osd_cs_oracle


@pytest.fixture(scope="module")
def hp1922():
    import fbgnn as F
    h = F.create_circulant_matrix(31, [0, 2, 5])
    code = F.hypergraph_product(h, h)
    assert (code.N, code.K) == (1922, 50)
    return code


def _frames(code, side, B, seed):
    """As test_gpu_osd_cs._frames, on either basis: (llr, full syndrome, reduced syndrome [rank, B], basis, pcm)."""
    H, piv = (code.hx, code.pivot_hx) if side == "hx" else (code.hz, code.pivot_hz)
    rng = np.random.default_rng(seed)
    n = code.N
    noise = (rng.random((B, n)) < 0.06).astype(np.uint8)
    synd = ((H @ noise.T.astype(np.int64)) & 1).astype(np.uint8)
    llr = rng.normal(3, 1, (B, n)).astype(np.float32)
    llr[noise == 1] -= 2.5
    llr[:, ::7] = 1.25                                  # ties: broken by index on both sides
    return llr, synd, np.ascontiguousarray(synd[piv]), H[piv], H


@pytest.mark.parametrize("side", ["hx", "hz"])
def test_layer_1922_bitexact(hp1922, cs, side):
    """The [[1922,50]] bases do not fit one CTA (about 238 KB at order 0): the cluster kernel runs by default."""
    import fbgnn as F
    code = hp1922
    llr, synd, red, basis, H = _frames(code, side, 24, seed=11 if side == "hx" else 12)
    R, n = basis.shape
    for lam in (0, 1, 10, 60, n - R):
        e = F.OSD_Decoder(n, osd_order=lam)(llr, basis, red, 24)
        ref = cs.osd(basis, llr, red, lam)
        assert e.dtype == bool and np.array_equal(e.astype(np.uint8), ref), (side, lam)
        assert np.array_equal((H @ e.T.astype(np.int64)) & 1, synd), (side, lam)


@pytest.mark.parametrize("name", ["steane", "rsurf3", "toric4", "gb48", "c882", "c1270"])
def test_forced_cluster_equals_k_osd(codes, c1270, cs, monkeypatch, name):
    """FBGNN_OSD_CLUSTER=C runs the cluster kernel on codes one CTA holds; Steane (3 basis rows) at C = 8 leaves seven
    CTAs without rows."""
    import fbgnn as F
    code = c1270 if name == "c1270" else codes[name]
    llr, _, red, basis, _ = _frames(code, "hx", 24, seed=13)
    R, n = basis.shape
    for lam in sorted({0, 10, n - R}):
        monkeypatch.delenv("FBGNN_OSD_CLUSTER", raising=False)
        one = F.OSD_Decoder(n, osd_order=lam)(llr, basis, red, 24)              # k_osd
        ref = cs.osd(basis, llr, red, lam)
        assert np.array_equal(one.astype(np.uint8), ref), (name, lam)
        for C in (2, 4, 8):
            monkeypatch.setenv("FBGNN_OSD_CLUSTER", str(C))
            e = F.OSD_Decoder(n, osd_order=lam)(llr, basis, red, 24)
            assert np.array_equal(e, one), (name, lam, C)


def test_forced_cluster_bad_value_is_invalid(codes, monkeypatch):
    import fbgnn as F
    code = codes["gb48"]
    llr, _, red, basis, _ = _frames(code, "hx", 4, seed=14)
    monkeypatch.setenv("FBGNN_OSD_CLUSTER", "3")
    with pytest.raises(F.FbgnnError, match=f"fbgnn error {-1}"):                 # FBGNN_E_INVALID
        F.OSD_Decoder(code.N)(llr, basis, red, 4)


@pytest.mark.parametrize("skip", [False, True])
def test_bp4_osd_cs_pipeline_1922_bitexact(hp1922, oracle, cs, skip):
    import fbgnn as F
    code = hp1922
    dec = F.QLDPCBPDecoder(code, num_iter=30, normalization_factor=0.8, cn_type="minsum", stage_one=True)
    model = F.BP4_OSD_Model(code, dec, F.OSD_Decoder(code.N, osd_order=10), seed=4)
    model._inner.skip_inactive = skip
    B, p = 200, 0.10
    res = model.run(B, p, want_counters=True)
    ref = cs.pipeline(oracle.CodeGraph(code), [30], [], p, p0=None, factors=[0.8], cn_types=["minsum"], seed=4,
                      B=B, want_diff=True, osd_order=10)
    assert np.array_equal(res["flags"].numpy(), ref["flags"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])
    assert np.array_equal(res["counters"], ref["counters"])
    bp4 = F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, p0=None, seed=4).run(B, p, want_counters=True)
    assert bp4["counters"][1] >= 20                              # frames BP4 left flagged: the ones OSD decoded
    assert res["counters"][1] == 0                               # OSD-CS always meets the syndrome


@pytest.mark.parametrize("lam", [0, 10])
def test_sandwich_osd_1922_bitexact(hp1922, oracle, cs, weights, lam):
    import fbgnn as F
    code = hp1922
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
    G.set_weights(weights["c882"])
    d1 = F.QLDPCBPDecoder(code, num_iter=8, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code, num_iter=4, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    model = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1, d2], [G], num_layers=2, seed=3, osd0=True, osd_order=lam)
    B, p = 64, 0.08
    res = model.run(B, p, want_counters=True)
    ref = cs.pipeline(oracle.CodeGraph(code), [8, 4], [oracle.Gnn(weights["c882"])], p, seed=3, B=B, want_diff=True,
                      osd_order=lam)
    assert np.array_equal(res["flags"].numpy(), ref["flags"]) and np.array_equal(res["counters"], ref["counters"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])


def test_bp2_osd_cs_pipeline_1922_bitexact(hp1922, cs):
    import fbgnn as F
    code = hp1922
    dec = F.LDPCBPDecoder(code.hx, is_syndrome=True, hard_out=False, cn_type="minsum", num_iter=30, normalization_factor=0.8)
    model = F.BP2_OSD_Model(code.hx, code.hx_basis, code.pivot_hx, code.lx, dec, F.OSD_Decoder(code.N, osd_order=10),
                            seed=6)
    B, p = 400, 0.08
    res = model.run(B, p, want_counters=True)
    ref = cs.bsc_pipeline(code.hx, code.lx, 30, p, code.hx_basis, code.pivot_hx, factor=0.8, cn_type="minsum", seed=6,
                          B=B, osd_order=10)
    assert np.array_equal(res["flags"].numpy(), ref["flags"]) and np.array_equal(res["counters"], ref["counters"])
    assert res["counters"][1] == 0


def test_7688_is_out_of_reach():
    """[[7688,50]]: even 8 CTAs cannot hold the reduced matrix; FBGNN_E_UNSUPPORTED names the bytes, nothing runs."""
    import fbgnn as F
    h = F.create_circulant_matrix(62, [0, 2, 5])
    code = F.hypergraph_product(h, h)
    assert (code.N, code.K) == (7688, 50)
    llr, _, red, basis, _ = _frames(code, "hx", 2, seed=15)
    with pytest.raises(F.FbgnnError, match=f"fbgnn error {-3}") as ei:        # FBGNN_E_UNSUPPORTED
        F.OSD_Decoder(code.N)(llr, basis, red, 2)
    m = re.search(r"needs (\d+) bytes of shared memory per frame in one CTA and (\d+) per CTA in a cluster of 8", str(ei.value))
    assert m and int(m.group(1)) > 8 * 232448 and int(m.group(2)) > 232448, str(ei.value)
