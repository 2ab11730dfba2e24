"""Training path (SURVEY.md section 8(f) N3): First_Stage_BP_Model / Second_Stage_GNN_BP_Model
(feedback_gnn.py:364-460), the gradient tf.GradientTape would return, Adam, and the dataset generators of
examples/Generate_dataset.ipynb.

Parity of the gradient with TensorFlow is unpinned (no TensorFlow in the image, no recorded gradients in the
repository).  Here: the loss against the float64 numpy restatement oracle/np_grad_oracle.py, and the gradient
against central finite differences of that restatement.  The element-by-element pin of the gradient against a float64
autograd reference (oracle/torch_grad_oracle.py) over many codes, batch sizes and configurations is
tests/test_train_grad.py."""
import numpy as np
import pytest


def _setup(codes, weights, B, p, seed):
    import fbgnn as F
    from oracle import c_oracle as O
    code = codes["c882"]
    nx, nz = O.pauli(seed, 0, B, code.N, p)
    dec1 = F.QLDPCBPDecoder(code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    dec2 = F.QLDPCBPDecoder(code, num_iter=6, normalization_factor=1.0, cn_type="boxplus-phi", stage_two=True)
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
    G.set_weights(weights["c882"])
    m1 = F.First_Stage_BP_Model(code, dec1)
    m2 = F.Second_Stage_GNN_BP_Model(code, G, dec2, num_iter=6, loss_from=2)
    return code, nx.astype(bool), nz.astype(bool), G, m1, m2


def test_adam_matches_the_keras_update_rule():
    import fbgnn as F

    class Layer:
        def __init__(self): self.w = [np.array([1.0, -2.0], np.float32)]
        def get_weights(self): return [a.copy() for a in self.w]
        def set_weights(self, w): self.w = w
    lay, opt = Layer(), F.Adam(learning_rate=0.1)
    g = np.array([0.5, -0.25])
    m = v = np.zeros(2)
    w = lay.w[0].astype(np.float64)
    for t in range(1, 4):
        opt.apply_gradients([g], lay)
        m = 0.9 * m + 0.1 * g
        v = 0.999 * v + 0.001 * g * g
        w = w - 0.1 * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t) * m / (np.sqrt(v) + 1e-7)
        assert np.allclose(lay.w[0], w, rtol=1e-6)
    assert [a.tolist() for a in F.clip_by_value([np.array([-20.0, 3.0, 11.0])], -10, 10)] == [[-10.0, 3.0, 10.0]]


def test_float64_restatement_is_consistent_with_the_float32_oracle(oracle, codes, weights):
    """The float64 loss restatement agrees with the pinned C oracle on the quantities they share: the GNN output and
    the per-iteration soft syndromes (away from the float32 cancellation noise of phi)."""
    from oracle import np_grad_oracle as NG
    code = codes["c882"]
    g = oracle.CodeGraph(code)
    B = 3
    nx, nz = oracle.pauli(5, 0, B, code.N, 0.08)
    sx = ((code.hx @ nz.T.astype(np.int64)) & 1).astype(np.uint8)
    sz = ((code.hz @ nx.T.astype(np.int64)) & 1).astype(np.uint8)
    r = oracle.bp4(g, float(oracle.prior_llr(0.05)), sx, sz, 8)
    h_vn = np.stack([r["Lx"], r["Ly"], r["Lz"]], -1)
    out_c = oracle.gnn(g, oracle.Gnn(weights["c882"]), h_vn, r["z_logit"], r["x_logit"], sx, sz)
    out_n = NG.gnn_forward(code, weights["c882"], h_vn, r["z_logit"], r["x_logit"], sx, sz)
    assert np.allclose(out_c, out_n, rtol=1e-4, atol=1e-5)
    r2 = oracle.bp4(g, np.ascontiguousarray(np.transpose(out_c, (0, 2, 1))), sx, sz, 3, want_iter_logits=True)
    lg = NG.bp4_logits(code, np.transpose(out_c, (0, 2, 1)), sx, sz, 3, 1.0)
    for k in range(4):
        for got, want in ((r2["llr_hat"][2 * k], lg[k][0].T), (r2["llr_hat"][2 * k + 1], lg[k][1].T)):
            ok = np.abs(want) < 8.0                      # larger soft syndromes sit in phi's float32 noise
            assert np.allclose(got[ok], want[ok], rtol=2e-3, atol=2e-3)
    loss = NG.second_stage_loss(code, weights["c882"], h_vn, r["z_logit"], r["x_logit"], sx, sz, 3, loss_from=1)
    assert np.isfinite(loss) and loss > 0


@pytest.mark.gpu
def test_second_stage_loss_and_outputs(codes, weights):
    from oracle import np_grad_oracle as NG
    code, nx, nz, G, m1, m2 = _setup(codes, weights, 6, 0.09, 11)
    h_vn, lhxp, lhzp = m1(nx, nz)
    assert h_vn.shape == (6, code.N, 3) and lhxp.shape == (code.hz.shape[0], 6) and lhzp.shape == (code.hx.shape[0], 6)
    s_hat, ls_hat, loss = m2(nx, nz, h_vn, lhxp, lhzp)
    assert s_hat.shape == (6, code.hx.shape[0] + code.hz.shape[0])
    assert ls_hat.shape == (6, code.hx_perp.shape[0] + code.hz_perp.shape[0])
    sx = ((code.hx @ nz.T.astype(np.int64)) & 1).astype(np.uint8)
    sz = ((code.hz @ nx.T.astype(np.int64)) & 1).astype(np.uint8)
    want = NG.second_stage_loss(code, G.get_weights(), h_vn, lhzp, lhxp, sx, sz, 6, 1.0, 2)
    assert abs(loss - want) <= 2e-3 * abs(want) + 1e-6, (loss, want)
    # a logical error implies nothing about flags, but an all-zero residual has neither
    assert not np.any(ls_hat[~np.any(s_hat, axis=1) & ~np.any(ls_hat, axis=1)])


@pytest.mark.gpu
def test_gradient_against_finite_differences(codes, weights):
    """<grad, u> against (L(w + eps u) - L(w - eps u)) / (2 eps) of the float64 restatement, for one random direction per
    weight array and one over all weights.  Tolerance: 3 % of the larger magnitude plus 2 % of the gradient norm in that
    block (float32 forward values in the analytic derivative)."""
    from oracle import np_grad_oracle as NG
    code, nx, nz, G, m1, m2 = _setup(codes, weights, 4, 0.09, 12)
    h_vn, lhxp, lhzp = m1(nx, nz)
    _, _, loss = m2(nx, nz, h_vn, lhxp, lhzp)
    grads = m2.gradients()
    w = G.get_weights()
    assert [g.shape for g in grads] == [a.shape for a in w]
    assert all(np.all(np.isfinite(g)) for g in grads) and any(np.any(g != 0) for g in grads)
    sx = ((code.hx @ nz.T.astype(np.int64)) & 1).astype(np.uint8)
    sz = ((code.hz @ nx.T.astype(np.int64)) & 1).astype(np.uint8)
    f = lambda ww: NG.second_stage_loss(code, ww, h_vn, lhzp, lhxp, sx, sz, 6, 1.0, 2)
    rng = np.random.default_rng(0)
    dirs = []
    for i in range(len(w)):
        u = [np.zeros_like(a, dtype=np.float64) for a in w]
        u[i] = rng.standard_normal(w[i].shape)
        dirs.append((f"array {i}", u))
    dirs.append(("all", [rng.standard_normal(a.shape) for a in w]))
    for name, u in dirs:
        eps = 1e-4
        fd = (f([a + eps * d for a, d in zip(w, u)]) - f([a - eps * d for a, d in zip(w, u)])) / (2 * eps)
        an = sum(float(np.sum(g.astype(np.float64) * d)) for g, d in zip(grads, u))
        scale = np.sqrt(sum(float(np.sum(g.astype(np.float64) ** 2)) for g, d in zip(grads, u) if np.any(d)))
        assert abs(an - fd) <= 0.03 * max(abs(an), abs(fd)) + 0.02 * scale + 1e-7, (name, an, fd)


@pytest.mark.gpu
def test_training_steps_reduce_the_loss_on_a_fixed_batch(codes, weights):
    import fbgnn as F
    code, nx, nz, G, m1, m2 = _setup(codes, weights, 16, 0.1, 13)
    rng = np.random.default_rng(3)
    G.set_weights([a + 0.05 * rng.standard_normal(a.shape).astype(np.float32) for a in weights["c882"]])   # de-tune
    opt = F.Adam(learning_rate=2e-3)
    losses = [F.train_step(m1, m2, opt, nx, nz)[0] for _ in range(8)]
    assert losses[-1] < losses[0], losses
    assert opt.iterations == 8


@pytest.mark.gpu
def test_dataset_generators_return_undecoded_error_strings(codes, weights):
    import fbgnn as F
    code = codes["c882"]
    dec = F.QLDPCBPDecoder(code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi")
    model = F.BP4_Error_Model(code, dec, wt=True, seed=21)
    ex, ez = model(400, 60)
    assert ex.shape == ez.shape and ex.shape[1] == code.N and 0 < ex.shape[0] <= 400
    assert np.all(np.sum(ex | ez, axis=1) == 60)                       # every string has the requested weight
    # they are failures: decoding them again leaves a syndrome mismatch
    sx = (code.hx @ ez.T.astype(np.int64)) & 1
    sz = (code.hz @ ex.T.astype(np.int64)) & 1
    llr = np.full((ex.shape[0], 3, code.N), np.log(3 * 0.95 / 0.05), np.float32)
    xh, zh = dec((llr, sx, sz))
    bad = np.any((code.hz @ xh.T.astype(np.int64)) & 1 != sz, axis=0) | np.any((code.hx @ zh.T.astype(np.int64)) & 1 != sx, axis=0)
    assert np.all(bad)
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
    G.set_weights(weights["c882"])
    d1 = F.QLDPCBPDecoder(code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    hard = F.Feedback_GNN_Error_Model(code, d1, G, dec, wt=True, seed=21)
    hx_, hz_ = hard(400, 60)
    assert hx_.shape[0] <= ex.shape[0]                                  # the GNN round rescues some of them


def test_second_stage_model_host_contract(codes):
    """Constructor checks and the mapping of the packed gradient onto the Keras weight order (no GPU needed)."""
    import fbgnn as F
    from fbgnn import training as T
    code = codes["steane"]
    G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
    d_one = F.QLDPCBPDecoder(code, num_iter=4, cn_type="boxplus-phi", stage_one=True)
    d_two = F.QLDPCBPDecoder(code, num_iter=4, cn_type="boxplus-phi", stage_two=True)
    with pytest.raises(TypeError):
        F.Second_Stage_GNN_BP_Model(code, G, d_one, num_iter=4)              # needs a stage_two decoder
    with pytest.raises(TypeError):
        F.First_Stage_BP_Model(code, d_two)                                  # needs a stage_one decoder
    with pytest.raises(ValueError):
        F.Second_Stage_GNN_BP_Model(code, G, d_two, num_iter=5)              # num_iter must match the decoder
    with pytest.raises(NotImplementedError):
        F.Second_Stage_GNN_BP_Model(code, G, F.QLDPCBPDecoder(code, num_iter=4, cn_type="minsum", stage_two=True), num_iter=4)
    m = F.Second_Stage_GNN_BP_Model(code, G, d_two, num_iter=4)
    with pytest.raises(RuntimeError):
        m.gradients()
    n_flat = sum(r * c for r, c in T._GRAD_BLOCKS)
    assert n_flat == G.count_params() == 3923
    g = m._unpack(np.arange(n_flat, dtype=np.float32))
    assert [a.shape for a in g] == [a.shape for a in G.get_weights()]
    assert g[0][0, 0] == 0 and g[1][0] == 40 * 3                             # [W0; b0] block: bias row last
    assert g[2][0, 0] == 41 * 3 and g[3][0] == 41 * 3 + 4 * 40               # [W1x; b1x]
    assert len(m.trainable_variables) == 12


def test_weights_trained_by_this_framework_load(codes):
    """weights/feedback_GNN_n882_k24_trained_by_fbgnn.npy: written by save_weights after examples/train_recipe.py
    (profiles/r01_train_recipe.txt) -- the pickle format the reference's load_weights reads."""
    import os, pickle
    import fbgnn as F
    path = os.path.join(F.WEIGHTS_DIR, "feedback_GNN_n882_k24_trained_by_fbgnn.npy")
    with open(path, "rb") as f:
        raw = pickle.load(f)                                   # plain pickle of ndarrays: no custom classes needed
    assert len(raw) == 12 and all(isinstance(a, np.ndarray) and a.dtype == np.float32 for a in raw)
    G = F.Feedback_GNN(codes["c882"], 20, 40, 2, "mean", "tanh", True)
    F.load_weights(G, path)
    assert [a.shape for a in G.get_weights()] == [a.shape for a in raw] and G.count_params() == 3923


@pytest.mark.gpu
def test_weights_trained_by_this_framework_match_the_shipped_ones(codes, weights):
    """BP -> (GNN -> BP) x 3 at p = 0.12 on [[882,24]]: the weights trained here and the reference's decode the same
    40 000 frames with error rates within 15 % of each other (recorded run: 7 772 vs 7 778 per 10^5)."""
    import os
    import fbgnn as F
    code = codes["c882"]
    d1 = F.QLDPCBPDecoder(code, num_iter=64, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    res = {}
    for name in ("trained", "shipped"):
        G = F.Feedback_GNN(code, 20, 40, 2, "mean", "tanh", True)
        if name == "trained":
            F.load_weights(G, os.path.join(F.WEIGHTS_DIR, "feedback_GNN_n882_k24_trained_by_fbgnn.npy"))
        else:
            G.set_weights(weights["c882"])
        m = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1, d2, d2, d2], [G] * 3, num_layers=4, seed=11, skip_inactive=True)
        res[name] = int(m.run(40000, 0.12, want_flags=False, want_diff=False, want_counters=True)["counters"][2])
    assert 2400 < res["shipped"] < 3800, res
    assert abs(res["trained"] - res["shipped"]) <= 0.15 * res["shipped"], res
