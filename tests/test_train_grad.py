"""The gradient of the second training stage (fbgnn_second_stage_grad: k_bp4_grad, k_gnn_bwd_rows, k_atb_partial /
k_atb_reduce in csrc/fbgnn_train.cuh) pinned element by element against a float64 autograd reference.

* CPU: the torch reference oracle/torch_grad_oracle.py equals the numpy restatement oracle/np_grad_oracle.py (loss to
  1e-12) and float64 central differences of itself (gradient to 1e-6); seven deliberate bugs move some gradient array
  by more than 20 x the GPU tolerance, so the GPU tests would see each of them.
* B200: the CUDA gradient against the float64 reference on [[882,24]] at B = 4 / 37 / 300 (k_atb_partial at its
  2·SM cap with an uneven last block), reduce "sum" with factor 0.8, irregular codes, codes with degree-0 columns and
  m_x != m_z, [[1270,28]] (k_bp4_grad at 167 640 B of shared memory), the converged training regime against the
  reference with the kernel's own phi; exact properties (zero loss, want_grad, determinism, math mode) bit for bit;
  refusals.

Tolerances (TOL_*) are the errors measured on a B200 (profiles/grad_error_b200.txt, tools/grad_error_report.py) with
a margin of 2-3x; torch float32 against float64 sits at 1e-6 to 7e-5 in the same cases.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

# per-array relative error of the CUDA gradient against the float64 smooth-phi reference, unconverged cases:
# ||g - g_ref|| / ||g_ref|| and max|g - g_ref| / max|g_ref|.  Measured on one B200 (profiles/grad_error_b200.txt):
# at most 5.1e-5 ([[1270,28]]), 3.1e-5 on [[882,24]] at any B
TOL_GRAD = 1e-4
# the loss against the reference evaluated with the library's phi (measured <= 2.9e-6), and against the smooth one:
# at loss_from = num_iter - 1 the loss is ~5e-3 and phi's float32 staircase moves it by up to 1.6e-4 (torch float32
# likewise)
TOL_LOSS = 1e-5
TOL_LOSS_SMOOTH = 5e-4
# converged regime (profiles/r01_gradient_check.txt's configuration) against the specified-phi reference: measured
# 4.2e-5 (loss) and 3.1e-5 (gradient); against the smooth reference the gradient is off by 8.6e-4, as is torch float32
TOL_LOSS_CONVERGED = 1e-4
TOL_GRAD_CONVERGED = 1e-4
SMEM_OPTIN_B200 = 232448


# ------------------------------------------------------------------------------------------------ codes and inputs
def asym_code():
    """[[7,2]] with m_x = 3, m_z = 2: qubit 0 is in no Z check."""
    import fbgnn as F
    return F.css_code(F.hamming_code(3), F.hamming_code(3)[:2], name="asym_n7_k2")


def steane_plus_code():
    """Steane with an eighth qubit that is in every Z check and in no X check: hx = [H | 0], hz = [H | 1]."""
    import fbgnn as F
    H = F.hamming_code(3)
    return F.css_code(np.hstack([H, np.zeros((3, 1), H.dtype)]), np.hstack([H, np.ones((3, 1), H.dtype)]),
                      name="steane_plus_n8_k2")


def _code(codes, c1270, key):
    if key == "asym":
        return asym_code()
    if key == "steane_plus":
        return steane_plus_code()
    if key == "c1270":
        return c1270
    return codes[key]


def _syndromes(code, nx, nz):
    sx = ((code.hx @ nz.T.astype(np.int64)) & 1).astype(np.uint8)
    sz = ((code.hz @ nx.T.astype(np.int64)) & 1).astype(np.uint8)
    return sx, sz


def cpu_inputs(oracle, code, B, p, seed, stage1=8):
    """Stage-one BP on the CPU oracle: (h_vn, logit over hx rows, logit over hz rows, sx, sz)."""
    nx, nz = oracle.pauli(seed, 0, B, code.N, p)
    sx, sz = _syndromes(code, nx, nz)
    r = oracle.bp4(oracle.CodeGraph(code), float(oracle.prior_llr(0.05)), sx, sz, stage1)
    return np.stack([r["Lx"], r["Ly"], r["Lz"]], -1), r["z_logit"], r["x_logit"], sx, sz


def perturbed_weights(seed, sigma=0.3):
    """Freshly initialised Feedback_GNN weights (Keras initialisers) plus N(0, sigma) noise."""
    import fbgnn as F
    G = F.Feedback_GNN(asym_code(), 20, 40, 2, "sum", "tanh", True)
    rng = np.random.default_rng(seed)
    return [(a + sigma * rng.standard_normal(a.shape)).astype(np.float32) for a in G.get_weights()]


def rel_errors(g, ref):
    """Per array: (||g - ref|| / ||ref||, max|g - ref| / max|ref|)."""
    out = []
    for a, b in zip(g, ref):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        d = a - b
        out.append((np.linalg.norm(d) / max(np.linalg.norm(b), 1e-300), np.max(np.abs(d)) / max(np.max(np.abs(b)), 1e-300)))
    return out


def worst(errs):
    return max(max(e) for e in errs)


# ------------------------------------------------------------------------------------------------ CPU: the reference
def _np_loss_sum(code, w, h_vn, lhx, lhz, sx, sz, num_iter, factor, loss_from):
    """np_grad_oracle.second_stage_loss with the GNN's reduce = "sum" (messages summed, bias counted per edge)."""
    from oracle import np_grad_oracle as NG
    W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3 = [np.asarray(a, np.float64) for a in w]
    B, n, _ = h_vn.shape
    ms = []
    for pcm, lg, sy, W1, b1, W2, b2 in ((code.hx, lhx, sx, W1x, b1x, W2x, b2x), (code.hz, lhz, sz, W1z, b1z, W2z, b2z)):
        c, v = np.nonzero(np.asarray(pcm))
        h_cn = (np.asarray(lg, np.float64) * (1.0 - 2.0 * np.asarray(sy, np.float64))).T
        f = np.concatenate([h_cn[:, c, None], np.asarray(h_vn, np.float64)[:, v, :]], axis=-1)
        msg = np.tanh(f @ W1 + b1) @ W2 + b2
        acc = np.zeros((B, n, msg.shape[-1]))
        np.add.at(acc, (slice(None), v), msg)
        ms.append(acc)
    x = np.concatenate([ms[0], ms[1], h_vn], axis=-1)
    new_llr = np.tanh(x @ W3 + b3) @ W0 + b0
    lg = NG.bp4_logits(code, np.transpose(new_llr, (0, 2, 1)), sx, sz, num_iter, factor)
    gt_x, gt_z = 1.0 - np.asarray(sz, np.float64).T, 1.0 - np.asarray(sx, np.float64).T
    return sum(NG._bce(gt_x, lg[i + 1][0]) + NG._bce(gt_z, lg[i + 1][1]) for i in range(loss_from, num_iter))


@pytest.mark.parametrize("key", ["c882", "rsurf3", "asym"])
@pytest.mark.parametrize("reduce", ["mean", "sum"])
@pytest.mark.parametrize("factor", [1.0, 0.8])
def test_reference_loss_matches_the_numpy_restatement(oracle, codes, weights, key, reduce, factor):
    from oracle import np_grad_oracle as NG, torch_grad_oracle as TG
    code = _code(codes, None, key)
    h_vn, lhx, lhz, sx, sz = cpu_inputs(oracle, code, 3, 0.1, 7)
    w = weights["c882"] if reduce == "mean" else perturbed_weights(1)
    T = 6
    for lf in (0, T // 2, T):
        want = (NG.second_stage_loss(code, w, h_vn, lhx, lhz, sx, sz, T, factor, lf) if reduce == "mean"
                else _np_loss_sum(code, w, h_vn, lhx, lhz, sx, sz, T, factor, lf))
        got, _ = TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, T, factor, lf, reduce, want_grad=False)
        assert abs(got - want) <= 1e-12 * abs(want), (lf, got, want)
        assert (got == 0.0) == (lf == T)


def _fd(f, w, u, eps=1e-6):
    return (f([a + eps * d for a, d in zip(w, u)]) - f([a - eps * d for a, d in zip(w, u)])) / (2 * eps)


@pytest.mark.parametrize("key,reduce,factor,loss_from", [("c882", "mean", 1.0, 2), ("rsurf3", "sum", 0.8, 0),
                                                          ("asym", "mean", 0.8, 1), ("steane_plus", "sum", 1.0, 3)])
def test_reference_gradient_matches_central_differences(oracle, codes, weights, key, reduce, factor, loss_from):
    """Autograd (with phi' = -1/sinh and the detached signs) against float64 central differences of the same loss: three
    random directions per array, and every element of the bias arrays.  1e-6 relative, plus the rounding of the two
    float64 losses over 2 eps (about 1e-10 |loss| at eps = 1e-6; allowed: 1e-9 |loss|)."""
    from oracle import torch_grad_oracle as TG
    code = _code(codes, None, key)
    h_vn, lhx, lhz, sx, sz = cpu_inputs(oracle, code, 3, 0.1, 9)
    w = [np.asarray(a, np.float64) for a in (weights["c882"] if reduce == "mean" else perturbed_weights(2))]
    T = 5
    loss, g = TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, T, factor, loss_from, reduce)
    f = lambda ww: TG.second_stage_loss_and_grad(code, ww, h_vn, lhx, lhz, sx, sz, T, factor, loss_from, reduce,
                                                 want_grad=False)[0]
    rng = np.random.default_rng(4)
    for i, name in enumerate(TG.NAMES):
        for _ in range(3):
            u = [np.zeros_like(a) for a in w]
            u[i] = rng.standard_normal(w[i].shape)
            fd, an = _fd(f, w, u), float(np.sum(g[i] * u[i]))
            assert abs(an - fd) <= 1e-6 * abs(fd) + 1e-9 * loss, (name, an, fd)
        if name.startswith("b"):
            for j in range(w[i].size):
                u = [np.zeros_like(a) for a in w]
                u[i].flat[j] = 1.0
                fd = _fd(f, w, u)
                assert abs(g[i].flat[j] - fd) <= 1e-6 * abs(fd) + 1e-9 * loss, (name, j, g[i].flat[j], fd)


# ------------------------------------------------------------------------------------------------ CPU: tolerance power
MUTATION_CASES = [
    # name, code, correct arguments, mutated arguments
    ("factor applied as 1.0", "c882", dict(factor=0.8), dict(factor=1.0)),
    ("loss_from off by one", "c882", dict(loss_from=2), dict(loss_from=3)),
    ("mean and sum swapped", "c882", dict(reduce="mean"), dict(reduce="sum")),
    ("wx and wz swapped", "asym", dict(), dict(mutate={"swap_bce_weights"})),
    ("soft-syndrome pairing swapped", "c882", dict(), dict(mutate={"swap_pairing"})),
    ("bias factor 1 for sum", "c882", dict(reduce="sum"), dict(reduce="sum", mutate={"bias_factor_one"})),
    ("one edge of each check dropped", "c882", dict(), dict(mutate={"drop_cn_edge"})),
]


@pytest.mark.parametrize("name,key,good,bad", MUTATION_CASES, ids=[c[0] for c in MUTATION_CASES])
def test_gpu_tolerance_sees_each_mutation(oracle, codes, weights, name, key, good, bad):
    """Each bug moves some gradient array by more than 20 x TOL_GRAD on one of the two measures the GPU tests assert."""
    from oracle import torch_grad_oracle as TG
    code = _code(codes, None, key)
    h_vn, lhx, lhz, sx, sz = cpu_inputs(oracle, code, 4, 0.11, 12, stage1=16)
    base = dict(num_iter=6, factor=1.0, loss_from=2, reduce="mean")
    w = weights["c882"]
    _, g = TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, **{**base, **good})
    _, gm = TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, **{**base, **bad})
    margin = worst(rel_errors(gm, g)) / TOL_GRAD
    assert margin > 20, (name, margin)


def test_reference_accepts_degree_zero_columns_and_extreme_loss_from(oracle):
    from oracle import torch_grad_oracle as TG
    for code in (asym_code(), steane_plus_code()):
        assert (code.N, code.K) in ((7, 2), (8, 2))
        assert np.any(np.asarray(code.hx).sum(0) == 0) or np.any(np.asarray(code.hz).sum(0) == 0)
        h_vn, lhx, lhz, sx, sz = cpu_inputs(oracle, code, 2, 0.15, 3)
        w = perturbed_weights(5)
        loss, g = TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, 4, 1.0, 4, "sum")
        assert loss == 0.0 and all(np.all(a == 0) for a in g)
        loss, g = TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, 4, 1.0, 0, "sum")
        assert loss > 0 and all(np.all(np.isfinite(a)) for a in g) and all(np.any(a != 0) for a in g)
    with pytest.raises(ValueError):
        TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, 4, 1.0, 5)
    with pytest.raises(ValueError):
        TG.second_stage_loss_and_grad(code, w, h_vn, lhx, lhz, sx, sz, 4, mutate={"no_such_bug"})


# ------------------------------------------------------------------------------------------------ GPU
def gpu_case(oracle, code, w, B, p, seed, stage1, num_iter, loss_from, reduce="mean", factor=1.0, gemm="fma"):
    """Stage one on the device (First_Stage_BP_Model), then Second_Stage_GNN_BP_Model: (loss, grads, inputs), inputs in
    the reference's argument order (h_vn, logit over hx rows, logit over hz rows, sx, sz)."""
    import fbgnn as F
    nx, nz = oracle.pauli(seed, 0, B, code.N, p)
    nx, nz = nx.astype(bool), nz.astype(bool)
    d1 = F.QLDPCBPDecoder(code, num_iter=stage1, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code, num_iter=num_iter, normalization_factor=factor, cn_type="boxplus-phi", stage_two=True)
    G = F.Feedback_GNN(code, 20, 40, 2, reduce, "tanh", True, gemm=gemm)
    G.set_weights(w)
    m1 = F.First_Stage_BP_Model(code, d1)
    m2 = F.Second_Stage_GNN_BP_Model(code, G, d2, num_iter=num_iter, loss_from=loss_from)
    h_vn, lhxp, lhzp = m1(nx, nz)
    if code.hx.shape[0] == code.hz.shape[0]:
        _, _, loss = m2(nx, nz, h_vn, lhxp, lhzp)
        grads = m2.gradients()
    else:       # the model's decision pass stacks the x and z soft syndromes as the reference does: m_x = m_z only
        loss, grads = grad_call(m2, nx, nz, h_vn, lhxp, lhzp)
    sx, sz = _syndromes(code, nx, nz)
    return loss, grads, (h_vn, lhzp, lhxp, sx, sz)


def grad_call(m2, nx, nz, h_vn, lhxp, lhzp):
    """The gradient part of Second_Stage_GNN_BP_Model.__call__ alone (fbgnn_second_stage_grad): (loss, grads)."""
    import ctypes as C
    from fbgnn import _ffi, training
    dev, sx, sz = training._syndromes(m2.code, None, nx, nz)
    ctx = dev.ctx
    h, lhx, lhz = ctx.asarray(h_vn, np.float32), ctx.asarray(lhzp, np.float32), ctx.asarray(lhxp, np.float32)
    loss = C.c_double()
    flat = np.zeros(sum(r * c for r, c in training._GRAD_BLOCKS), np.float32)
    _ffi.call("fbgnn_second_stage_grad", dev.handle, m2.feedback.device_handle(ctx), m2.num_iter,
              m2.decoder.normalization_factor, m2.loss_from, nx.shape[0], h.t3(), lhx.t2(), lhz.t2(), sx.t2(), sz.t2(),
              1, C.byref(loss), flat.ctypes.data_as(C.POINTER(C.c_float)))
    return float(loss.value), m2._unpack(flat)


def reference(code, w, inputs, num_iter, loss_from, reduce="mean", factor=1.0, **kw):
    from oracle import torch_grad_oracle as TG
    return TG.second_stage_loss_and_grad(code, w, *inputs, num_iter, factor, loss_from, reduce, **kw)


# name: (code, weights, B, p, seed, stage-one iterations, num_iter, loss_from, reduce, factor)
UNCONVERGED = {f"c882_B{B}_T{T}_lf{lf}": ("c882", "c882", B, 0.11, 20 + B, 16, T, lf, "mean", 1.0)
               for B in (4, 37, 300) for T in (6, 16) for lf in (0, T - 1)}
UNCONVERGED.update({
    "c882_sum_f0.8_perturbed": ("c882", "perturbed", 8, 0.10, 31, 16, 6, 2, "sum", 0.8),
    "rsurf3": ("rsurf3", "c882", 64, 0.10, 32, 16, 6, 0, "mean", 1.0),
    "gb48": ("gb48", "c882", 32, 0.10, 33, 16, 6, 0, "mean", 1.0),
    "toric4": ("toric4", "perturbed", 32, 0.10, 34, 16, 6, 1, "sum", 0.8),
    "asym_B1": ("asym", "c882", 1, 0.15, 35, 8, 6, 0, "mean", 1.0),
    "asym_B33_sum": ("asym", "perturbed", 33, 0.15, 36, 8, 6, 0, "sum", 1.0),
    "steane_plus_B1_sum": ("steane_plus", "perturbed", 1, 0.15, 37, 8, 6, 0, "sum", 0.8),
    "steane_plus_B33": ("steane_plus", "c882", 33, 0.15, 38, 8, 6, 0, "mean", 1.0),
    "c1270_B8": ("c1270", "c1270", 8, 0.08, 39, 16, 6, 0, "mean", 1.0),
})
# profiles/r01_gradient_check.txt: stage one 64, num_iter 16, loss_from 8, p = 0.09, B = 4, seed 12
CONVERGED = ("c882", "c882", 4, 0.09, 12, 64, 16, 8, "mean", 1.0)


def run_named_case(oracle, codes, c1270, weights, case, gemm="fma"):
    key, wkey, B, p, seed, s1, T, lf, reduce, factor = case
    code = _code(codes, c1270, key)
    w = perturbed_weights(seed) if wkey == "perturbed" else weights[wkey]
    loss, g, inputs = gpu_case(oracle, code, w, B, p, seed, s1, T, lf, reduce, factor, gemm)
    return code, w, loss, g, inputs


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(UNCONVERGED))
def test_gradient_matches_the_float64_reference(oracle, codes, c1270, weights, name):
    case = UNCONVERGED[name]
    code, w, loss, g, inputs = run_named_case(oracle, codes, c1270, weights, case)
    T, lf, reduce, factor = case[6:]
    want, ref = reference(code, w, inputs, T, lf, reduce, factor)
    want_spec, _ = reference(code, w, inputs, T, lf, reduce, factor, want_grad=False, phi="specified")
    assert abs(loss - want_spec) <= TOL_LOSS * abs(want_spec), (loss, want_spec)
    assert abs(loss - want) <= TOL_LOSS_SMOOTH * abs(want), (loss, want)
    from oracle import torch_grad_oracle as TG
    for nm, (e_norm, e_max) in zip(TG.NAMES, rel_errors(g, ref)):
        assert e_norm <= TOL_GRAD and e_max <= TOL_GRAD, (nm, e_norm, e_max)


@pytest.mark.gpu
def test_converged_regime_matches_the_specified_phi_reference(oracle, codes, c1270, weights):
    """Near convergence the loss is ~3e-4 and phi's float32 staircase near its clip dominates it: the reference uses
    the kernel's phi in its forward pass (phi="specified")."""
    code, w, loss, g, inputs = run_named_case(oracle, codes, c1270, weights, CONVERGED)
    want, ref = reference(code, w, inputs, 16, 8, phi="specified")
    assert abs(loss - want) <= TOL_LOSS_CONVERGED * abs(want), (loss, want)
    assert worst(rel_errors(g, ref)) <= TOL_GRAD_CONVERGED


@pytest.mark.gpu
def test_tensor_core_forward_gradient_matches_the_reference(oracle, codes, c1270, weights):
    """gemm="tf32x3": the forward GNN runs in k_gnn_tc, the reverse sweep recomputes it in FMA form."""
    case = UNCONVERGED["c882_B37_T6_lf0"]
    code, w, loss, g, inputs = run_named_case(oracle, codes, c1270, weights, case, gemm="tf32x3")
    want, ref = reference(code, w, inputs, 6, 0)
    assert abs(loss - want) <= TOL_LOSS_SMOOTH * abs(want), (loss, want)
    assert worst(rel_errors(g, ref)) <= TOL_GRAD


def _model(code, w, num_iter, loss_from, trainable=True, reduce="mean", activation="tanh", use_bias=True, layers=2):
    import fbgnn as F
    G = F.Feedback_GNN(code, 20, 40, layers, reduce, activation, use_bias)
    if w is not None:
        G.set_weights(w)
    d2 = F.QLDPCBPDecoder(code, num_iter=num_iter, normalization_factor=1.0, cn_type="boxplus-phi", stage_two=True)
    return F.Second_Stage_GNN_BP_Model(code, G, d2, num_iter=num_iter, loss_from=loss_from, trainable=trainable)


def _stage_one(oracle, code, B, p, seed):
    import fbgnn as F
    nx, nz = oracle.pauli(seed, 0, B, code.N, p)
    nx, nz = nx.astype(bool), nz.astype(bool)
    d1 = F.QLDPCBPDecoder(code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    return (nx, nz) + tuple(F.First_Stage_BP_Model(code, d1)(nx, nz))


@pytest.mark.gpu
def test_exact_properties_bit_for_bit(oracle, codes, weights):
    import fbgnn as F
    code, w = codes["c882"], weights["c882"]
    args = _stage_one(oracle, code, 37, 0.11, 41)
    # loss_from == num_iter: nothing to learn from
    m = _model(code, w, 6, 6)
    _, _, loss = m(*args)
    assert loss == 0.0 and all(np.all(a == 0) for a in m.gradients())
    # want_grad = 0 computes the same loss
    m_t, m_f = _model(code, w, 6, 1), _model(code, w, 6, 1, trainable=False)
    _, _, l_t = m_t(*args)
    _, _, l_f = m_f(*args)
    assert l_t == l_f and l_t > 0
    g1 = m_t.gradients()
    # the two-stage reduction is deterministic
    _, _, l_2 = m_t(*args)
    assert l_2 == l_t and all(np.array_equal(a, b) for a, b in zip(g1, m_t.gradients()))
    # the call forces exact arithmetic and restores the context's mode afterwards
    ctx = F.default_context()
    before = ctx.get_math()
    try:
        for mode in ("sfu", "exact"):
            ctx.set_math(mode)
            _, _, l_m = m_t(*args)
            assert ctx.get_math() == mode
            assert l_m == l_t and all(np.array_equal(a, b) for a, b in zip(g1, m_t.gradients())), mode
    finally:
        ctx.set_math(before)


@pytest.mark.gpu
def test_code_beyond_one_cta_is_refused_and_the_context_stays_usable(oracle, codes, weights):
    """[[1922,50]]: k_bp4_grad would need 4 (3E + 14n + m_x + m_z) bytes of shared memory in one CTA."""
    import ctypes as C
    import fbgnn as F
    from fbgnn import _ffi, training
    h = F.create_circulant_matrix(31, [0, 2, 5])
    code = F.hypergraph_product(h, h)
    E, n, mt = int(np.sum(code.hx) + np.sum(code.hz)), code.N, code.hx.shape[0] + code.hz.shape[0]
    need = 4 * (3 * E + 14 * n + mt)
    assert need > SMEM_OPTIN_B200, need
    B = 2
    rng = np.random.default_rng(0)
    m = _model(code, weights["c882"], 4, 0)
    nx, nz = rng.random((B, n)) < 0.02, rng.random((B, n)) < 0.02
    dev, sx, sz = training._syndromes(code, None, nx, nz)
    ctx = dev.ctx
    hv = ctx.asarray(rng.normal(3.0, 1.0, (B, n, 3)), np.float32)
    lhx, lhz = ctx.asarray(np.ones((dev.mx, B)), np.float32), ctx.asarray(np.ones((dev.mz, B)), np.float32)
    gnn = m.feedback.device_handle(ctx)
    ctx.sync()
    launches = ctx.launch_count()
    loss = C.c_double(-1.0)
    grads = np.full(3923, 7.0, np.float32)
    with pytest.raises(F.FbgnnError, match=r"BP4 gradient needs (\d+) bytes of shared memory") as ei:
        _ffi.call("fbgnn_second_stage_grad", dev.handle, gnn, 4, 1.0, 0, B, hv.t3(), lhx.t2(), lhz.t2(), sx.t2(), sz.t2(),
                  1, C.byref(loss), grads.ctypes.data_as(C.POINTER(C.c_float)))
    assert str(need) in str(ei.value)
    assert ctx.launch_count() == launches and loss.value == -1.0 and np.all(grads == 7.0)
    ctx.sync()
    # the same context still trains a code that fits
    small = codes["rsurf3"]
    args = _stage_one(oracle, small, 8, 0.1, 43)
    m2 = _model(small, weights["c882"], 6, 0)
    _, _, l = m2(*args)
    assert l > 0 and all(np.all(np.isfinite(a)) for a in m2.gradients())


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [dict(reduce="max"), dict(activation="relu"), dict(use_bias=False), dict(layers=3)],
                         ids=["reduce_max", "relu", "no_bias", "depth3"])
def test_configurations_without_a_gradient_are_refused(oracle, codes, cfg):
    import fbgnn as F
    code = codes["rsurf3"]
    args = _stage_one(oracle, code, 4, 0.1, 44)
    m = _model(code, None, 6, 0, **cfg)
    with pytest.raises(F.FbgnnError, match="gradients are provided for"):
        m(*args)
    with pytest.raises(RuntimeError):
        m.gradients()
