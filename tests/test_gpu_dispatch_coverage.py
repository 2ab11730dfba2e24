"""Every kernel instantiation the dispatchers of csrc/fbgnn_bp.cu, csrc/fbgnn_gnn.cu and csrc/fbgnn_gbp.cu can select,
compared with the CPU oracle on a code that routes to it.  The suite's other parity files use codes whose check degrees
are at most 8 and whose variable degrees are at most 4, and the shipped 40 / 20 GNN; the cells below are reached by
the (5,10) generalized-bicycle codes, the overcomplete codes of the reference's QLDPC notebook, a (5,10) hypergraph
product too large for one SM, and the other GNN widths, activations and depths.

Each case first asserts, from the matrices and the layer configuration alone, the property that makes the dispatcher
pick its cell (`bp4_cell` and its siblings below restate the dispatchers), so that a change of code or dispatcher
fails loudly instead of quietly testing another kernel.  CLAIMS maps every cell to the cases that exercise it;
tests/test_dispatch_coverage.py extracts the cells from the dispatcher sources and fails on any cell without a claim.

Float32 outputs are BIT-EXACT against the oracle in the same arithmetic, except the GNN_BP4 tensor-core form, which is
held to its stated tolerance (tests/test_gnn_bp4.py)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# cell (as written in the dispatcher, whitespace removed) -> the cases of this file that run it
CLAIMS = {
    # fbgnn_bp.cu: launch_bp4
    "launch_bp4_m<3,6>": ["test_bp4_layer_bitexact"],
    "launch_bp4_m<4,8>": ["test_bp4_layer_bitexact"],
    "launch_bp4_m<5,10>": ["test_bp4_layer_bitexact", "test_bp4_fixed_point_exit_dv5", "test_bp4_stage_two_dv5",
                           "test_pipeline_dv5"],
    "launch_bp4_m<0,0>": ["test_bp4_layer_bitexact", "test_bp4_early_stop"],
    "launch_bp4_cluster_t<64>": ["test_large_code_layer"],
    "launch_bp4_cluster_t<8>": ["test_large_code_layer_dc8"],
    "launch_bp4_gstate<MathExact>": ["test_large_code_layer", "test_bp4_early_stop"],
    "launch_bp4_gstate<MathSfu>": ["test_large_code_layer", "test_large_code_default_route", "test_bp4_early_stop",
                                   "test_large_code_pipeline"],
    # fbgnn_bp.cu: launch_bp2
    "launch_bp2_m<3,6>": ["test_bp2_layer_bitexact"],
    "launch_bp2_m<4,8>": ["test_bp2_layer_bitexact"],
    "launch_bp2_m<5,10>": ["test_bp2_layer_bitexact"],
    "launch_bp2_m<0,0>": ["test_bp2_layer_bitexact"],
    # fbgnn_gnn.cu: launch_gnn
    "k_gnn_deep<MathSfu>": ["test_gnn_deep"],
    "k_gnn_deep<MathExact>": ["test_gnn_deep"],
    "tc::k_gnn_tc<3,MathSfu>": ["test_gnn_tc"],
    "tc::k_gnn_tc<3,MathExact>": ["test_gnn_tc"],
    "launch_gnn_m<40,20,0,false,false>": ["test_gnn_layer_overcomplete"],
    "launch_gnn_m<40,20,3,true>": ["test_gnn_reg3_variants"],
    "launch_gnn_m<40,20,3,false>": ["test_gnn_reg3_variants"],
    "launch_gnn_m<40,20,0,true>": ["test_gnn_layer_overcomplete", "test_large_code_pipeline"],
    "launch_gnn_m<40,20,0,false>": ["test_gnn_reg3_variants"],
    "launch_gnn_m<20,20,0,false>": ["test_gnn_other_dims", "test_pipeline_gnn_20_20"],
    "launch_gnn_m<20,20,0,false,false>": ["test_gnn_other_dims"],
    "launch_gnn_m<64,32,0,false>": ["test_gnn_other_dims"],
    "launch_gnn_m<64,32,0,false,false>": ["test_gnn_other_dims"],
    # fbgnn_gbp.cu: gbp_run
    "k_gbp_pre_vn<20,40,20>": ["test_gnn_bp4_high_degree", "test_gnn_bp4_overcomplete"],
    "k_gbp_logit<20,MATH>": ["test_gnn_bp4_high_degree", "test_gnn_bp4_overcomplete"],
    "tc::k_gbp_cn_tc<MATH>": ["test_gnn_bp4_tensor_core_sfu", "test_gnn_bp4_overcomplete"],
    "tc::k_gbp_vn_tc<MATH>": ["test_gnn_bp4_tensor_core_sfu", "test_gnn_bp4_overcomplete"],
    "k_gbp_cn_f<20,40,20,true,MATH>": ["test_gnn_bp4_high_degree", "test_gnn_bp4_overcomplete"],
    "k_gbp_cn_f<20,40,20,false,MATH>": ["test_gnn_bp4_high_degree"],
    "k_gbp_cn<20,40,20,MATH>": ["test_gnn_bp4_high_degree", "test_gnn_bp4_overcomplete"],
    "k_gbp_vn_f<20,40,20,true,MATH>": ["test_gnn_bp4_high_degree", "test_gnn_bp4_overcomplete"],
    "k_gbp_vn_f<20,40,20,false,MATH>": ["test_gnn_bp4_high_degree"],
    "k_gbp_vn<20,40,20,MATH>": ["test_gnn_bp4_high_degree", "test_gnn_bp4_overcomplete"],
}

# ------------------------------------------------------------------ routing, restated from the dispatchers --------
SMEM_OPTIN = 227 * 1024          # shared memory a B200 block may opt in to (cudaDevAttrMaxSharedMemoryPerBlockOptin)
GBP_CODE_CAP = 8                 # fbgnn_kernels.cuh: edge codes staged per receiver in the GNN_BP4 kernels


def _regular(pcm):
    """(dv, dc) as fbgnn_core.cu records them: a degree is 0 unless it is the same for every node of the side."""
    pcm = np.asarray(pcm)
    col, row = pcm.sum(0), pcm.sum(1)
    dv = int(col[0]) if col.min() == col.max() else 0
    dc = int(row[0]) if pcm.shape[0] > 0 and row.min() == row.max() else 0
    return dv, dc


def _pad(x, k):
    return (x + k - 1) // k * k


def bp4_state_bytes(code, const_prior=False, iter_logits=False):
    """fbgnn_bp.cu bp4_smem: one frame's decoder state in the one-CTA kernel."""
    n, mt = code.N, code.hx.shape[0] + code.hz.shape[0]
    E = int(np.sum(code.hx)) + int(np.sum(code.hz))
    return 4 * (E + ((2 if const_prior else 3) + (2 if iter_logits else 0)) * _pad(n, 4)) + _pad(mt, 16) + \
        2 * ((n + 1) & ~1) + n + 16


def bp4_cell(code, large=None, math="exact", early_stop=False):
    """The launcher launch_bp4 picks for this code."""
    if bp4_state_bytes(code) > SMEM_OPTIN:
        want_cluster = (large == "cluster") if large else math != "sfu"
        if want_cluster and not early_stop:
            (_, dcx), (_, dcz) = _regular(code.hx), _regular(code.hz)
            max_dc = max(dcx, dcz) if dcx and dcz else 64
            return f"launch_bp4_cluster_t<{8 if max_dc <= 8 else 64}>"
        return "launch_bp4_gstate<MathSfu>" if math == "sfu" else "launch_bp4_gstate<MathExact>"
    (dvx, dcx), (dvz, dcz) = _regular(code.hx), _regular(code.hz)
    if dvx and dvx == dvz and dcx and dcx == dcz and (dvx, dcx) in ((3, 6), (4, 8), (5, 10)):
        return f"launch_bp4_m<{dvx},{dcx}>"
    return "launch_bp4_m<0,0>"


def bp2_cell(pcm):
    dv, dc = _regular(pcm)
    return f"launch_bp2_m<{dv},{dc}>" if (dv, dc) in ((3, 6), (4, 8), (5, 10)) else "launch_bp2_m<0,0>"


def gnn_cell(code, H, M, activation, reduce_op, use_bias):
    reg3 = _regular(code.hx)[0] == 3 and _regular(code.hz)[0] == 3
    tb = activation == "tanh" and use_bias
    fact = reduce_op in ("mean", "sum")
    if (H, M) == (40, 20):
        if not fact:
            return "launch_gnn_m<40,20,0,false,false>"
        if reg3:
            return f"launch_gnn_m<40,20,3,{'true' if tb else 'false'}>"
        return f"launch_gnn_m<40,20,0,{'true' if tb else 'false'}>"
    assert (H, M) in ((20, 20), (64, 32))
    return f"launch_gnn_m<{H},{M},0,false>" if fact else f"launch_gnn_m<{H},{M},0,false,false>"


def max_node_degree(code):
    return max(int(np.asarray(h).sum(a).max()) for h in (code.hx, code.hz) for a in (0, 1))


# ------------------------------------------------------------------ codes and helpers -----------------------------
@pytest.fixture(scope="module")
def dcodes(codes):
    """The suite's codes plus the (5,10) generalized-bicycle codes and the overcomplete codes (QLDPC.ipynb cell 12)."""
    import fbgnn as F
    import test_gpu_published as PUB
    c = dict(codes)
    for name in ("GB_n254_k28", "GB_n126_k28", "GB_n46_k2_oc", "GB_n48_k6_oc"):
        c[name] = PUB._code(F, name, codes, None)
    return c


@pytest.fixture(scope="module")
def hp(dcodes):
    """(5,10) hypergraph product of a weight-5 circulant of size 62 with itself: 7688 qubits, 38 440 edges per side
    (76 880 in all), check degree 10.  x^62 - 1 and 1 + x + x^2 + x^3 + x^5 share a factor of degree 5, so K = 50."""
    import fbgnn as F
    h = F.create_circulant_matrix(62, [0, 1, 2, 3, 5])
    code = F.hypergraph_product(h, h)
    assert (code.N, code.K) == (7688, 50)
    assert _regular(code.hx) == _regular(code.hz) == (5, 10)
    assert int(code.hx.sum()) == int(code.hz.sum()) == 38440
    return code


@pytest.fixture(params=["exact", "sfu"])
def arith(request, oracle):
    import fbgnn as F
    ctx = F.default_context()
    ctx.set_math(request.param)
    oracle.set_math(request.param)
    yield request.param
    ctx.set_math("exact")
    oracle.set_math("exact")


def _syndromes(oracle, code, B, p, seed):
    nx, nz = oracle.pauli(seed, 0, B, code.N, p)
    return (((code.hx @ nz.T.astype(np.int64)) & 1).astype(np.uint8),
            ((code.hz @ nx.T.astype(np.int64)) & 1).astype(np.uint8))


def _layer(F, oracle, code, llr_or_prior, sx, sz, it, factor, cn_type, tag, g=None):
    """fbgnn_bp4_decode (per-variable or constant prior) vs oracle.bp4: all outputs and the final messages."""
    import test_gpu_parity as P
    g = g or oracle.CodeGraph(code)
    dec = F.QLDPCBPDecoder(code, num_iter=it, normalization_factor=factor, cn_type=cn_type, stage_one=True)
    ctx = dec._device().ctx
    const = np.isscalar(llr_or_prior)
    out = dec.decode_device(None if const else ctx.asarray(llr_or_prior), ctx.asarray(sx), ctx.asarray(sz),
                            want_msgs=True, prior=float(llr_or_prior) if const else None)
    ref = oracle.bp4(g, float(llr_or_prior) if const else llr_or_prior, sx, sz, it, factor, cn_type, want_msgs=True)
    for k, o in zip(("Lx", "Ly", "Lz", "x_hat", "z_hat", "x_logit", "z_logit", "msg_x", "msg_z"), out):
        P.assert_bitexact(o.numpy(), ref[k], f"{tag} {cn_type} it={it} {k}")
    return ref


# ------------------------------------------------------------------ quaternary BP ---------------------------------
BP4_CODES = [("c882", "launch_bp4_m<3,6>", 0.09), ("gb48", "launch_bp4_m<4,8>", 0.05),
             ("GB_n254_k28", "launch_bp4_m<5,10>", 0.07), ("GB_n126_k28", "launch_bp4_m<5,10>", 0.05),
             ("GB_n46_k2_oc", "launch_bp4_m<0,0>", 0.06), ("GB_n48_k6_oc", "launch_bp4_m<0,0>", 0.06)]


@pytest.mark.parametrize("name,cell,p", BP4_CODES, ids=[c[0] for c in BP4_CODES])
def test_bp4_layer_bitexact(dcodes, oracle, arith, name, cell, p):
    """The BP4 layer on every regular instantiation and the generic one (the overcomplete codes: m > n, irregular
    checks of degree 8 / 10 / 12), three check-node rules, per-variable and constant priors, 0 to 64 iterations."""
    import fbgnn as F
    code = dcodes[name]
    assert bp4_cell(code) == cell
    if name.endswith("_oc"):
        assert code.hx.shape[0] > code.N and max(int(code.hx.sum(1).max()), int(code.hz.sum(1).max())) > 8
    B = 40
    sx, sz = _syndromes(oracle, code, B, p, 11)
    g = oracle.CodeGraph(code)
    prior = oracle.prior_llr(0.05)
    llr = (prior + np.random.default_rng(3).normal(0, 0.3, (B, 3, code.N))).astype(np.float32)
    for cn_type, factor in (("boxplus-phi", 0.625), ("minsum", 0.8), ("boxplus", 1.0)):
        for it in (0, 1, 7, 32, 64):
            _layer(F, oracle, code, llr, sx, sz, it, factor, cn_type, f"{name} per-variable", g)
            _layer(F, oracle, code, prior, sx, sz, it, factor, cn_type, f"{name} const", g)


@pytest.mark.parametrize("name", ["GB_n254_k28", "GB_n126_k28"])
@pytest.mark.parametrize("factor", [1.0, 0.625])
def test_bp4_fixed_point_exit_dv5(dcodes, oracle, arith, name, factor):
    """64 iterations of boxplus-phi at low p on the (5,10) codes: k_bp4<., 5, 10, ., FPX> leaves its loop once every
    frame is at a saturated fixed point (its record holds 2 x 5 sign bits per variable).  The outputs must equal the
    oracle's full 64 iterations bit for bit, and the kernel must indeed have left early."""
    import fbgnn as F
    code = dcodes[name]
    assert bp4_cell(code) == "launch_bp4_m<5,10>"
    B = 96
    sx, sz = _syndromes(oracle, code, B, 0.02, 77)
    prior = oracle.prior_llr(0.05)
    ctx = F.default_context()
    g = oracle.CodeGraph(code)
    for llr in (prior, (prior + np.random.default_rng(5).normal(0, 0.2, (B, 3, code.N))).astype(np.float32)):
        ctx.stats(reset=True)
        ref = _layer(F, oracle, code, llr, sx, sz, 64, factor, "boxplus-phi", f"{name} fpx", g)
        frames, iters = ctx.stats(reset=True)
        ok = np.all(((code.hx @ ref["z_hat"].T.astype(np.int64)) & 1) == sx, axis=0) & \
            np.all(((code.hz @ ref["x_hat"].T.astype(np.int64)) & 1) == sz, axis=0)
        assert ok.mean() > 0.9
        assert frames == B and iters < 0.75 * 64 * B, (frames, iters)       # the exit was taken


@pytest.mark.parametrize("name", ["GB_n254_k28", "GB_n126_k28"])
def test_bp4_stage_two_dv5(dcodes, oracle, arith, name):
    """stage_two per-iteration soft syndromes through the (5,10) kernel."""
    import test_gpu_parity as P
    assert bp4_cell(dcodes[name]) == "launch_bp4_m<5,10>"
    P.test_bp4_stage_two_per_iteration_soft_syndromes(dcodes, oracle, name)


@pytest.mark.parametrize("skip", [False, True])
def test_pipeline_dv5(dcodes, oracle, weights, arith, skip):
    """Sandwich (64, G, 16) on GB_n254_k28: the first stage runs the (5,10) fixed-point-exit kernel in the pipeline."""
    import fbgnn as F
    import test_gpu_parity as P
    code = dcodes["GB_n254_k28"]
    assert bp4_cell(code) == "launch_bp4_m<5,10>"
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
    G.set_weights(weights["c882"])
    d1 = F.QLDPCBPDecoder(code, num_iter=64, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code, num_iter=16, normalization_factor=0.9, cn_type="boxplus-phi", stage_one=True)
    B, p = 192, 0.07
    res = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1, d2], [G], num_layers=2, seed=7, first_frame=300,
                                             skip_inactive=skip).run(B, p, want_counters=True)
    ref = oracle.pipeline(oracle.CodeGraph(code), [64, 16], [oracle.Gnn(weights["c882"])], p, factors=[1.0, 0.9],
                          seed=7, first_frame=300, B=B, want_diff=True)
    P.assert_bitexact(res["flags"].numpy(), ref["flags"], "GB_n254 pipeline flags")
    P.assert_bitexact(res["x_diff"].numpy(), ref["x_diff"], "x_diff")
    P.assert_bitexact(res["z_diff"].numpy(), ref["z_diff"], "z_diff")
    assert res["counters"].tolist() == ref["counters"].tolist() and ref["counters"][3] > 0


@pytest.mark.parametrize("name", ["GB_n254_k28", "GB_n46_k2_oc", "large"])
def test_bp4_early_stop(dcodes, hp, oracle, arith, name):
    """Opt-in early stop on a (5,10) code, an overcomplete code and the large code (iters_out makes the cluster launcher
    decline, so the large code runs the HBM-state kernel): iteration counts and outputs equal the oracle's."""
    import fbgnn as F
    import test_gpu_parity as P
    code = hp if name == "large" else dcodes[name]
    expect = {"GB_n254_k28": "launch_bp4_m<5,10>", "GB_n46_k2_oc": "launch_bp4_m<0,0>",
              "large": "launch_bp4_gstate<MathSfu>" if arith == "sfu" else "launch_bp4_gstate<MathExact>"}[name]
    assert bp4_cell(code, math=arith, early_stop=True) == expect
    B = 6 if name == "large" else 96
    sx, sz = _syndromes(oracle, code, B, 0.02 if name == "large" else 0.04, 3)
    llr = np.full((B, 3, code.N), oracle.prior_llr(0.05), np.float32)
    dec = F.QLDPCBPDecoder(code, num_iter=40, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True,
                           early_stop=True)
    out = dec((llr, sx, sz))
    ref = oracle.bp4(oracle.CodeGraph(code), llr, sx, sz, 40, 1.0, "boxplus-phi", early_stop=True)
    P.assert_bitexact(dec.last_iterations, ref["iters"], f"{name} iterations")
    assert ref["iters"].min() < 40                                       # frames do stop early
    for k, o in zip(("Lx", "Ly", "Lz", "x_hat", "z_hat", "x_logit", "z_logit"), out):
        P.assert_bitexact(np.asarray(o, dtype=ref[k].dtype), ref[k], f"{name} early stop {k}")


# ------------------------------------------------------------------ binary BP -------------------------------------
BP2_CODES = [("c882", "launch_bp2_m<3,6>"), ("gb48", "launch_bp2_m<4,8>"), ("GB_n254_k28", "launch_bp2_m<5,10>"),
             ("GB_n126_k28", "launch_bp2_m<5,10>"), ("GB_n46_k2_oc", "launch_bp2_m<0,0>")]


@pytest.mark.parametrize("name,cell", BP2_CODES, ids=[c[0] for c in BP2_CODES])
@pytest.mark.parametrize("cn_type", ["boxplus-phi", "minsum", "boxplus"])
def test_bp2_layer_bitexact(dcodes, oracle, arith, name, cell, cn_type):
    import test_gpu_parity as P
    assert bp2_cell(dcodes[name].hx) == cell
    P.test_bp2_layer_bitexact(dcodes, oracle, name, cn_type)


# ------------------------------------------------------------------ the large (5,10) code -------------------------
def _large_layer_cases(F, oracle, code):
    B = 4
    sx, sz = _syndromes(oracle, code, B, 0.03, 5)
    g = oracle.CodeGraph(code)
    prior = oracle.prior_llr(0.03)
    llr = (prior + np.random.default_rng(1).normal(0, 0.3, (B, 3, code.N))).astype(np.float32)
    for cn_type, it in (("boxplus-phi", 6), ("minsum", 3)):
        _layer(F, oracle, code, llr, sx, sz, it, 0.9, cn_type, "large per-variable", g)
    _layer(F, oracle, code, prior, sx, sz, 5, 1.0, "boxplus-phi", "large const", g)


@pytest.mark.parametrize("large", ["cluster", "gstate"])
def test_large_code_layer(hp, oracle, arith, large, monkeypatch):
    """76 880 edges, 7688 qubits: no single SM holds a frame.  FBGNN_BP4_LARGE=cluster runs k_bp4_cluster with
    DCMAX = 64 (check degree 10 > 8), =gstate the kernel whose state lives in HBM; both arithmetics."""
    import fbgnn as F
    assert bp4_state_bytes(hp) > SMEM_OPTIN and bp4_state_bytes(hp, const_prior=True) > SMEM_OPTIN
    want = "launch_bp4_cluster_t<64>" if large == "cluster" else f"launch_bp4_gstate<{'MathSfu' if arith == 'sfu' else 'MathExact'}>"
    assert bp4_cell(hp, large=large, math=arith) == want
    monkeypatch.setenv("FBGNN_BP4_LARGE", large)
    _large_layer_cases(F, oracle, hp)


def test_large_code_layer_dc8(oracle, arith, monkeypatch):
    """The cluster kernel's DCMAX = 8 form, on a (4,8) hypergraph product of 7688 qubits (the [[7688,50]] code of
    test_gpu_parity.py is (3,6) and also takes it): both arithmetics through the cluster."""
    import fbgnn as F
    h = F.create_circulant_matrix(62, [0, 3, 11, 25])
    code = F.hypergraph_product(h, h)
    assert _regular(code.hx) == _regular(code.hz) == (4, 8)
    assert bp4_cell(code, large="cluster", math=arith) == "launch_bp4_cluster_t<8>"
    monkeypatch.setenv("FBGNN_BP4_LARGE", "cluster")
    _large_layer_cases(F, oracle, code)


def test_large_code_default_route(hp, oracle, monkeypatch):
    """Without an override SFU arithmetic takes the HBM-state kernel in its own arithmetic (the exact one would
    differ in the last bits of almost every message)."""
    import fbgnn as F
    monkeypatch.delenv("FBGNN_BP4_LARGE", raising=False)
    assert bp4_cell(hp, math="sfu") == "launch_bp4_gstate<MathSfu>"
    ctx = F.default_context()
    ctx.set_math("sfu")
    try:
        with oracle.math("sfu"):
            _large_layer_cases(F, oracle, hp)
    finally:
        ctx.set_math("exact")


def test_large_code_pipeline(hp, oracle, weights, arith, monkeypatch):
    """Two-stage Sandwich pipeline (8, G, 4) on the large code, default route: flags and counters."""
    import fbgnn as F
    import test_gpu_parity as P
    monkeypatch.delenv("FBGNN_BP4_LARGE", raising=False)
    assert bp4_cell(hp, math=arith).startswith("launch_bp4_" + ("gstate" if arith == "sfu" else "cluster_t<64>"))
    assert gnn_cell(hp, 40, 20, "tanh", "mean", True) == "launch_gnn_m<40,20,0,true>"
    G = F.Feedback_GNN(hp, 20, 40, 2, "mean", "tanh", True)
    G.set_weights(weights["c882"])
    d1 = F.QLDPCBPDecoder(hp, num_iter=8, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(hp, num_iter=4, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    B, p = 6, 0.05
    res = F.Sandwich_BP_GNN_Evaluation_Model(hp, [d1, d2], [G], num_layers=2, seed=3).run(B, p, want_counters=True)
    ref = oracle.pipeline(oracle.CodeGraph(hp), [8, 4], [oracle.Gnn(weights["c882"])], p, seed=3, B=B, want_diff=True)
    P.assert_bitexact(res["flags"].numpy(), ref["flags"], "large code pipeline flags")
    P.assert_bitexact(res["x_diff"].numpy(), ref["x_diff"], "large code pipeline x_diff")
    assert res["counters"].tolist() == ref["counters"].tolist()


# ------------------------------------------------------------------ the overcomplete codes beyond BP --------------
OC = ["GB_n46_k2_oc", "GB_n48_k6_oc"]


@pytest.mark.parametrize("name", OC)
@pytest.mark.parametrize("reduce_op", ["mean", "sum", "max", "min"])
def test_gnn_layer_overcomplete(dcodes, oracle, weights, arith, name, reduce_op):
    """Feedback GNN (generic kernels) where every qubit sits in 76 to 261 checks per side."""
    import test_gpu_parity as P
    code = dcodes[name]
    assert gnn_cell(code, 40, 20, "tanh", reduce_op, True) == (
        "launch_gnn_m<40,20,0,true>" if reduce_op in ("mean", "sum") else "launch_gnn_m<40,20,0,false,false>")
    assert min(int(code.hx.sum(0).min()), int(code.hz.sum(0).min())) > 70
    P.test_gnn_layer_bitexact(dcodes, oracle, weights, name, "c882", reduce_op)


@pytest.mark.parametrize("name", OC)
def test_gnn_bp4_overcomplete(dcodes, oracle, arith, name):
    """GNN_BP4 with every variable node past the GBP_CODE_CAP staged edge codes: factored (mean / sum) and max / min
    FMA forms bit-exact, the tensor-core form within its stated tolerance."""
    import test_gnn_bp4 as GB
    code = dcodes[name]
    assert min(int(code.hx.sum(0).min()), int(code.hz.sum(0).min())) > GBP_CODE_CAP
    for reduce_op, bias in (("mean", True), ("sum", False), ("max", True), ("min", False)):
        GB.test_cuda_gnn_bp4_bitexact(oracle, dcodes, name, reduce_op, bias)
    GB.test_cuda_gnn_bp4_tensor_core_path(oracle, dcodes, name, "mean", True)


@pytest.fixture(scope="module")
def cs(oracle):
    from oracle import osd_cs_oracle
    osd_cs_oracle.build()
    return osd_cs_oracle


@pytest.mark.parametrize("name", OC)
def test_osd_overcomplete(dcodes, oracle, cs, name):
    """OSD-0 and OSD-CS (λ = 10) on the pivot basis of a code whose rank is far below its number of checks."""
    import fbgnn as F
    import test_gpu_osd_cs as OCS
    code = dcodes[name]
    assert code.hx_basis.shape[0] < code.hx.shape[0] // 8
    OCS._check_layer(code, cs, (0, 10), B=48, seed=2)
    llr, synd, red = OCS._frames(code, 48, 3)
    e = F.OSD0_Decoder(code.N)(llr, code.hx_basis, red, 48)
    assert np.array_equal(e.astype(np.uint8), oracle.osd0(code.hx_basis, llr, red))
    assert np.array_equal((code.hx @ e.T.astype(np.int64)) & 1, synd)


@pytest.mark.parametrize("name", OC)
@pytest.mark.parametrize("order", [0, 10])
def test_bp4_osd_model_overcomplete(dcodes, oracle, cs, name, order):
    """BP4_OSD_Model: BP on the full overcomplete matrices, then the syndrome reduced to the pivot rows for OSD."""
    import fbgnn as F
    code = dcodes[name]
    assert bp4_cell(code) == "launch_bp4_m<0,0>"
    dec = F.QLDPCBPDecoder(code, num_iter=6, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    osd = F.OSD0_Decoder(code.N) if order == 0 else F.OSD_Decoder(code.N, osd_order=order)
    model = F.BP4_OSD_Model(code, dec, osd, seed=4)
    B, p = 600, 0.08
    res = model.run(B, p, want_counters=True)
    kw = dict(p0=None, factors=[1.0], seed=4, B=B, want_diff=True)
    ref = oracle.pipeline(oracle.CodeGraph(code), [6], [], p, osd0=True, **kw) if order == 0 else \
        cs.pipeline(oracle.CodeGraph(code), [6], [], p, osd_order=order, **kw)
    assert np.array_equal(res["flags"].numpy(), ref["flags"])
    assert np.array_equal(res["x_diff"].numpy(), ref["x_diff"]) and np.array_equal(res["z_diff"].numpy(), ref["z_diff"])
    assert np.array_equal(res["counters"], ref["counters"])
    assert res["counters"][1] == 0


# ------------------------------------------------------------------ feedback GNN widths and variants --------------
def _random_gnn(F, code, H, M, reduce_op, act, bias, seed, L=2):
    G = F.Feedback_GNN(code=code, num_msg_dims=M, num_hidden_units=H, num_mlp_layers=L, reduce_op=reduce_op,
                       activation=act, use_bias=bias)
    rng = np.random.default_rng(seed)
    w = [(a + rng.normal(0, 0.3, a.shape)).astype(np.float32) for a in G.get_weights()]
    G.set_weights(w)
    return G, w


def _gnn_inputs(oracle, code, B, seed):
    sx, sz = _syndromes(oracle, code, B, 0.1, seed)
    r = oracle.bp4(oracle.CodeGraph(code), float(oracle.prior_llr(0.05)), sx, sz, 8)
    return np.stack([r["Lx"], r["Ly"], r["Lz"]], -1), r["z_logit"], r["x_logit"], sx, sz


@pytest.mark.parametrize("name", ["c882", "rsurf3"])
@pytest.mark.parametrize("H,M", [(20, 20), (64, 32)])
@pytest.mark.parametrize("reduce_op", ["mean", "sum", "max", "min"])
def test_gnn_other_dims(codes, oracle, arith, name, H, M, reduce_op):
    import fbgnn as F
    import test_gpu_parity as P
    code = codes[name]
    cell = gnn_cell(code, H, M, "tanh", reduce_op, True)
    assert cell == (f"launch_gnn_m<{H},{M},0,false>" if reduce_op in ("mean", "sum") else f"launch_gnn_m<{H},{M},0,false,false>")
    G, w = _random_gnn(F, code, H, M, reduce_op, "tanh", True, seed=H + M)
    h_vn, lhx, lhz, sx, sz = _gnn_inputs(oracle, code, 36, 4)
    out = G((h_vn, lhx, lhz, sx, sz))
    ref = oracle.gnn(oracle.CodeGraph(code), oracle.Gnn(w, "tanh", reduce_op), h_vn, lhx, lhz, sx, sz)
    P.assert_bitexact(out, ref, f"gnn {H}/{M} {name} {reduce_op}")


@pytest.mark.parametrize("act,bias,name", [("relu", True, "c882"), ("tanh", False, "c882"), ("relu", True, "rsurf3"),
                                           ("linear", False, "rsurf3")])
@pytest.mark.parametrize("reduce_op", ["mean", "sum"])
def test_gnn_reg3_variants(codes, oracle, arith, act, bias, name, reduce_op):
    """40 / 20 GNN off the shipped tanh + bias: the (3,.)-regular kernel <40,20,3,false> on c882 and the generic
    <40,20,0,false> on rsurf3."""
    import fbgnn as F
    import test_gpu_parity as P
    code = codes[name]
    assert gnn_cell(code, 40, 20, act, reduce_op, bias) == (
        "launch_gnn_m<40,20,3,false>" if name == "c882" else "launch_gnn_m<40,20,0,false>")
    G, w = _random_gnn(F, code, 40, 20, reduce_op, act, bias, seed=7)
    h_vn, lhx, lhz, sx, sz = _gnn_inputs(oracle, code, 36, 9)
    out = G((h_vn, lhx, lhz, sx, sz))
    ref = oracle.gnn(oracle.CodeGraph(code), oracle.Gnn(w, act, reduce_op, use_bias=bias), h_vn, lhx, lhz, sx, sz)
    P.assert_bitexact(out, ref, f"gnn 40/20 {name} {act} bias={bias} {reduce_op}")


def test_pipeline_gnn_20_20(codes, oracle, arith):
    """A 20 / 20 GNN between two BP stages of the fused pipeline."""
    import fbgnn as F
    import test_gpu_parity as P
    code = codes["c882"]
    assert gnn_cell(code, 20, 20, "tanh", "mean", True) == "launch_gnn_m<20,20,0,false>"
    G, w = _random_gnn(F, code, 20, 20, "mean", "tanh", True, seed=21)
    d1 = F.QLDPCBPDecoder(code, num_iter=24, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code, num_iter=8, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    B, p = 160, 0.12
    res = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1, d2, d2], [G, G], num_layers=3, seed=9).run(B, p, want_counters=True)
    ref = oracle.pipeline(oracle.CodeGraph(code), [24, 8, 8], [oracle.Gnn(w)] * 2, p, seed=9, B=B, want_diff=True)
    P.assert_bitexact(res["flags"].numpy(), ref["flags"], "20/20 pipeline flags")
    P.assert_bitexact(res["x_diff"].numpy(), ref["x_diff"], "x_diff")
    assert res["counters"].tolist() == ref["counters"].tolist() and ref["counters"][3] > 0


@pytest.mark.parametrize("L,reduce_op,bias", [(1, "mean", True), (3, "max", False), (3, "sum", True)])
def test_gnn_deep(codes, oracle, arith, L, reduce_op, bias):
    """k_gnn_deep (num_mlp_layers != 2) in both arithmetics."""
    import test_gpu_parity as P
    P.test_gnn_any_mlp_depth_bitexact(codes, oracle, L, reduce_op, bias)


def test_gnn_tc(codes, oracle, weights, arith):
    """The tensor-core feedback GNN in both arithmetics against the oracle's emulation of it."""
    import fbgnn as F
    import test_gpu_parity as P
    code = codes["c882"]
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True, gemm="tf32x3")
    G.set_weights(weights["c882"])
    h_vn, lhx, lhz, sx, sz = _gnn_inputs(oracle, code, 40, 6)
    out = G((h_vn, lhx, lhz, sx, sz))
    ref = oracle.gnn(oracle.CodeGraph(code), oracle.Gnn(weights["c882"], gemm="tf32x3"), h_vn, lhx, lhz, sx, sz)
    P.assert_bitexact(out, ref, f"gnn tc {arith}")


# ------------------------------------------------------------------ GNN_BP4 ---------------------------------------
@pytest.mark.parametrize("reduce_op", ["mean", "sum", "max", "min"])
@pytest.mark.parametrize("act", ["tanh", "relu", "linear"])
@pytest.mark.parametrize("bias", [True, False])
def test_gnn_bp4_high_degree(dcodes, oracle, arith, reduce_op, act, bias):
    """GNN_BP4 on GB_n254_k28, whose checks have 10 edges: the codes of edges 9 and 10 are re-read past the staged
    slots.  Every reduction, activation and bias setting of the FMA kernels, bit-exact."""
    import fbgnn as F
    import test_gnn_bp4 as GB
    import test_gpu_parity as P
    code = dcodes["GB_n254_k28"]
    assert max_node_degree(code) == 10 > GBP_CODE_CAP
    W = oracle.gnn_bp4_random_weights(seed=6, use_bias=bias)
    B, it = 29, 3
    sx, sz = GB._syndromes(oracle, code, B, 0.06, 9)
    G = F.GNN_BP4(code, 20, 20, 40, 2, it, reduce_op=reduce_op, activation=act, use_bias=bias)
    G.set_weights(GB._weights_list(W, bias))
    llr_hat, x_hat, z_hat = G((sx, sz))
    ref = oracle.gnn_bp4(oracle.CodeGraph(code), W, sx, sz, it, activation=act, reduce_op=reduce_op)
    for i in range(it):
        P.assert_bitexact(llr_hat[i][0], ref["x_logit"][i], f"gnn_bp4 {act} {reduce_op} it={i} x")
        P.assert_bitexact(llr_hat[i][1], ref["z_logit"][i], f"gnn_bp4 {act} {reduce_op} it={i} z")
    P.assert_bitexact(x_hat.astype(np.uint8), ref["x_hat"], "x_hat")
    P.assert_bitexact(z_hat.astype(np.uint8), ref["z_hat"], "z_hat")


@pytest.mark.parametrize("name", ["c882", "GB_n254_k28"])
def test_gnn_bp4_tensor_core_sfu(dcodes, oracle, name):
    """The tensor-core GNN_BP4 in SFU arithmetic, chunked batches with a ragged tail (53 frames, 16 per pass), against
    the SFU oracle at the stated tolerance."""
    import fbgnn as F
    import test_gnn_bp4 as GB
    code = dcodes[name]
    ctx = F.default_context()
    ctx.set_math("sfu")
    try:
        with oracle.math("sfu"):
            W = oracle.gnn_bp4_random_weights(seed=4, use_bias=True)
            B, it = 53, 4
            sx, sz = GB._syndromes(oracle, code, B, 0.06, 19)
            ref = oracle.gnn_bp4(oracle.CodeGraph(code), W, sx, sz, it, reduce_op="mean")
            G = F.GNN_BP4(code, 20, 20, 40, 2, it, reduce_op="mean", activation="tanh", use_bias=True, gemm="tf32x3",
                          chunk_frames=16)
            G.set_weights(GB._weights_list(W, True))
            llr_hat, x_hat, z_hat = G((sx, sz))
    finally:
        ctx.set_math("exact")
    for i in range(it):
        for got, want in ((llr_hat[i][0], ref["x_logit"][i]), (llr_hat[i][1], ref["z_logit"][i])):
            assert np.all(np.abs(got - want) <= 2e-5 + 1e-5 * np.abs(want)), (name, i, float(np.abs(got - want).max()))
    agree = np.mean((x_hat.astype(np.uint8) == ref["x_hat"]) & (z_hat.astype(np.uint8) == ref["z_hat"]))
    assert agree >= 0.9999, agree
