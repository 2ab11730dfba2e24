"""Parity against THE REFERENCE'S OWN CODE.  tests/golden/ref_*.npz were written by executing the unmodified
reference sources (sionna/fec/ldpc/{codes_q,decoding_q,feedback_gnn,gnn}.py, sionna/channel/pauli.py, sionna/fec/utils.py)
on seeded inputs, with TensorFlow's primitives restated in numpy (oracle/tfshim; generator:
tests/golden/make_reference_golden.py).  They pin, for the CPU oracle (both arithmetics) and -- in the ``gpu`` tests --
for the CUDA path through the C ABI:

  * code construction and GF(2) algebra: every matrix, pivot list and parameter, exactly;
  * the noise source: same uniforms -> the reference's Pauli.call gives exactly our noise bits;
  * QLDPCBPDecoder.call: hard decisions identical on every qubit of every case; float32 marginals within 2e-5 after one
    iteration and 2e-3 after two (phi = softplus(x) - log(exp(x) - 1) cancels catastrophically, SURVEY.md H2, so the
    float32 noise of any two libms grows by ~10x per iteration; from iteration 3 on only robust statistics are asserted);
    soft syndromes within the float32 noise model of phi(sum phi(|.|)) (error ~ 4e-6 exp|logit|, saturating in steps of ln 2);
  * LDPCBPDecoder.call (binary, is_syndrome): hard decisions identical, soft outputs within 5e-6 after one iteration,
    5e-3 after five; min-sum bit-identical;
  * Feedback_GNN.call with the shipped weights loaded by the reference's load_weights: 1e-6 absolute, all four reduce ops;
  * Sandwich_BP_GNN_Evaluation_Model.call on the same uniforms: per-frame flagged / block-error indicators and the dense
    s_hat rows, identical on >= 97 % of the frames at p = 0.06 (>= 85 % in the chaotic regime p >= 0.08, F6 noise floor).
"""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
W = {"c882": "feedback_GNN_n882_k24_wt_4_60_iter_64_16_mixed.npy",
     "c1270": "feedback_GNN_n1270_k28_wt_10_80_iter_64_16_mixed.npy"}
LN2 = 0.6931472


@pytest.fixture(scope="module")
def ref():
    r = {k: np.load(os.path.join(GOLDEN, f"ref_{k}.npz")) for k in ("codes", "bp4", "bp2", "gnn", "sandwich")}
    # the QLDPCBPDecoder cases are stored in two files (c882 / the other codes) so that each stays under 1 MB
    r["bp4"] = {**r["bp4"], **np.load(os.path.join(GOLDEN, "ref_bp4_c1270_rsurf3.npz"))}
    return r


@pytest.fixture(scope="module")
def allcodes(codes, c1270):
    import fbgnn as F
    d = dict(codes)
    d["c1270"] = c1270
    d["rsurf5"] = F.create_rotated_surface_codes(5)
    d["surf3"] = F.create_surface_codes(3)
    d["hp162"] = F.hypergraph_product(F.create_circulant_matrix(9, [0, 2, 5]), F.create_circulant_matrix(9, [0, 2, 5]))
    d["ibm72"] = F.create_bivariate_QC_codes(6, 6, [3], [1, 2], [1, 2], [3])
    return d


def _unpack(Z, key):
    shape = tuple(Z[f"{key}.shape"])
    return np.unpackbits(Z[f"{key}.bits"])[:int(np.prod(shape))].reshape(shape)


def test_code_construction_matches_the_reference_code(ref, allcodes):
    """css_code and every constructor against sionna/fec/ldpc/codes_q.py + sionna/fec/utils.py executed as they are."""
    Z = ref["codes"]
    names = sorted({k.split(".")[0] for k in Z.files})
    assert len(names) == 10
    for name in names:
        c = allcodes[name]
        for attr in ("hx", "hz", "lx", "lz", "hx_perp", "hz_perp"):
            assert np.array_equal(np.asarray(getattr(c, attr)), _unpack(Z, f"{name}.{attr}")), (name, attr)
        assert list(c.pivot_hx) == Z[f"{name}.pivot_hx"].tolist() and list(c.pivot_hz) == Z[f"{name}.pivot_hz"].tolist()
        assert [c.N, c.K, c.rank_hx, c.rank_hz, int(c.L), int(c.Q), int(c.D)] == Z[f"{name}.params"].tolist(), name
        assert c.name == str(Z[f"{name}.name"]), name


def _bp_cases(Z):
    return sorted({k.rsplit(".", 1)[0] for k in Z if k.endswith(".Lx")})


def _check_bp4(Z, key, got, what):
    it = int(key.rsplit(".", 1)[1])
    minsum = ".minsum." in key
    assert np.array_equal(got["x_hat"], Z[f"{key}.x_hat"]) and np.array_equal(got["z_hat"], Z[f"{key}.z_hat"]), (what, key)
    for k in ("Lx", "Ly", "Lz"):
        r, g = Z[f"{key}.{k}"], got[k]
        err = np.abs(g - r)
        if minsum or it == 1:
            assert err.max() <= 2e-5, (what, key, k, float(err.max()))
        elif it == 2:
            assert err.max() <= 2e-3, (what, key, k, float(err.max()))
        rel = err / (np.abs(r) + 1.0)
        assert np.median(rel) < (2e-6 if it <= 2 else 2e-5) and np.quantile(rel, 0.99) < 5e-3, (what, key, k)
        assert np.mean(np.sign(g) == np.sign(r)) > 0.9999
    for k in ("x_logit", "z_logit"):
        r, g = Z[f"{key}.{k}"], got[k]
        err = np.abs(g - r)
        # float32 noise model of phi(sum phi(|.|)) (tests/test_oracle.py::_tol): the absolute error of a soft syndrome of
        # magnitude a grows like exp(a) until it saturates in steps of ln 2 at the clip (phi_max = 16.64)
        a = np.maximum(np.abs(r), np.abs(g))
        tol = 2e-5 * a + 1e-5 + np.minimum(4e-6 * np.exp(np.minimum(a, 20.0)), 4 * LN2)
        # (the SFU arithmetic rounds the two terms of phi where the reference does but through other operations: one
        # float32 quantum more per term, see tests/test_sfu_oracle.py)
        if minsum or it <= 2:
            assert np.all(err <= (9 if "sfu" in what else 6) * tol), (what, key, k, float((err / tol).max()))
        assert np.median(err / (a + 1.0)) < 2e-4, (what, key, k)
        assert np.mean(np.sign(g) == np.sign(r)) > 0.999


@pytest.mark.parametrize("arith", ["exact", "sfu"])
def test_oracle_bp4_matches_the_reference_code(ref, allcodes, oracle, arith):
    Z = ref["bp4"]
    with oracle.math(arith):
        for key in _bp_cases(Z):
            cname, cn_type, rest = key.split(".", 2)
            factor, it = rest.rsplit(".", 1)
            code = allcodes[cname]
            B = Z[f"{cname}.noise_x"].shape[0]
            nx, nz = oracle.pauli(11, 0, B, code.N, float(Z[f"{cname}.p"]))
            assert np.array_equal(nx, Z[f"{cname}.noise_x"]) and np.array_equal(nz, Z[f"{cname}.noise_z"]), "noise source"
            got = oracle.bp4(oracle.CodeGraph(code), Z[f"{cname}.llr"], Z[f"{cname}.sx"], Z[f"{cname}.sz"], int(it),
                             float(factor), cn_type)
            _check_bp4(Z, key, got, f"oracle[{arith}]")
            assert Z[f"{key}.dtypes"].tolist() == ["float32"] * 3 + ["int64", "float64", "float32", "float32"]
        # stage_two: (2 it + 2) soft-syndrome slices, slot 2i = x_logit before iteration i (decoding_q.py:743-746)
        code = allcodes["c882"]
        got = oracle.bp4(oracle.CodeGraph(code), Z["c882.llr"], Z["c882.sx"], Z["c882.sz"], 2, 1.0, "boxplus-phi",
                         want_iter_logits=True)["llr_hat"]
        r = Z["c882.stage_two.llr_hat"]
        assert got.shape == r.shape == (6, code.hx.shape[0], Z["c882.llr"].shape[0])
        a = np.maximum(np.abs(r), np.abs(got))
        assert np.all(np.abs(got - r) <= 6 * (2e-5 * a + 1e-5 + np.minimum(4e-6 * np.exp(np.minimum(a, 20.0)), 4 * LN2)))


def _check_bp2(Z, key, soft, hard, what):
    """LDPCBPDecoder (decoding.py, run with the column-major scipy.sparse.find it was written for, SURVEY.md F8)."""
    it = int(key.rsplit(".", 1)[1])
    r = Z[f"{key}.soft"]
    err = np.abs(soft - r)
    assert np.array_equal(hard, Z[f"{key}.hard"]), (what, key)
    if ".minsum." in key:
        assert err.max() == 0.0, (what, key)                  # no transcendental: bit-identical to the reference's code
    elif ".boxplus." in key:
        # tanh variant: |llr| = 20 (the clip) drives tanh(10) into saturation, where implementations differ in the last
        # float32 step (numpy: exactly 1; Eigen's rational form as restated in fb_math.h: 1 - 2.4e-7) and atanh amplifies
        # it -- a handful of saturated entries may differ by < 0.7, everything else agrees to rounding
        bad = int(np.count_nonzero(err > (5e-6 if it == 1 else 2e-3)))
        assert bad <= max(3, err.size // 1000) and err.max() <= 0.7, (what, key, bad, float(err.max()))
    else:
        assert err.max() <= (5e-6 if it == 1 else 1e-4 if it == 2 else 5e-3), (what, key, float(err.max()))


def _bp2_cases(Z):
    return sorted({k.rsplit(".", 1)[0] for k in Z.files if k.endswith(".soft") and k.split(".")[-2].isdigit()})


@pytest.mark.parametrize("arith", ["exact", "sfu"])
def test_oracle_bp2_matches_the_reference_code(ref, allcodes, oracle, arith):
    Z = ref["bp2"]
    with oracle.math(arith):
        for key in _bp2_cases(Z):
            cname, cn_type, it = key.split(".")
            soft, hard = oracle.bp2(allcodes[cname].hx, Z[f"{cname}.llr"], Z[f"{cname}.synd"], int(it), 0.9, cn_type)
            _check_bp2(Z, key, soft, hard, f"oracle[{arith}]")


def _logit_tol(r, g):
    a = np.maximum(np.abs(r), np.abs(g))
    return 6 * (2e-5 * a + 1e-5 + np.minimum(4e-6 * np.exp(np.minimum(a, 20.0)), 4 * LN2))


def test_oracle_trainable_mode_matches_the_reference_code(ref, allcodes, oracle):
    """trainable=True without stage_one / stage_two: llr_hat over the dense hx_perp / hz_perp rows (decoding_q.py:32-37)."""
    Z = ref["bp4"]
    code = allcodes["c882"]
    r = Z["c882.trainable.llr_hat"]
    got = oracle.bp4(oracle.CodeGraph(code), Z["c882.llr"][:4], Z["c882.sx"][:, :4], Z["c882.sz"][:, :4], 2, 1.0,
                     "boxplus-phi", rows_x=code.hx_perp, rows_z=code.hz_perp, want_iter_logits=True)["llr_hat"]
    assert got.shape == r.shape == (6, code.hx_perp.shape[0], 4)
    assert np.all(np.abs(got - r) <= _logit_tol(r, got))


@pytest.mark.gpu
def test_cuda_trainable_mode_matches_oracle_and_reference(ref, allcodes, oracle):
    import fbgnn as F
    Z = ref["bp4"]
    code = allcodes["c882"]
    llr, sx, sz = Z["c882.llr"][:4], Z["c882.sx"][:, :4], Z["c882.sz"][:, :4]
    dec = F.QLDPCBPDecoder(code, num_iter=2, normalization_factor=1.0, cn_type="boxplus-phi", trainable=True)
    llr_hat, xh, zh = dec((llr, sx, sz))
    want = oracle.bp4(oracle.CodeGraph(code), llr, sx, sz, 2, 1.0, "boxplus-phi", rows_x=code.hx_perp, rows_z=code.hz_perp,
                      want_iter_logits=True)
    assert np.array_equal(llr_hat.view(np.uint32), want["llr_hat"].view(np.uint32))          # bit-exact vs the oracle
    assert np.array_equal(xh.astype(np.uint8), want["x_hat"]) and np.array_equal(zh.astype(np.uint8), want["z_hat"])
    r = Z["c882.trainable.llr_hat"]
    assert np.all(np.abs(llr_hat - r) <= _logit_tol(r, llr_hat))                             # float32 noise vs the reference's code


def test_oracle_bp2_trainable_and_stateful_match_the_reference_code(ref, allcodes, oracle):
    Z = ref["bp2"]
    hx = allcodes["c882"].hx
    soft, _ = oracle.bp2(hx, Z["c882.llr"], Z["c882.synd"], 3, 0.9, "boxplus-phi", edge_weights=Z["c882.trainable.edge_weights"])
    assert np.abs(soft - Z["c882.trainable.soft"]).max() <= 2e-4
    x1, _, m1 = oracle.bp2(hx, Z["c882.llr"], None, 2, 0.9, "minsum", want_msgs=True)
    x2, _, m2 = oracle.bp2(hx, Z["c882.llr"], None, 2, 0.9, "minsum", msg_in=m1, want_msgs=True)
    for got, key in ((x1, "x1"), (x2, "x2"), (m1.T, "m1"), (m2.T, "m2")):
        assert np.array_equal(got, Z[f"c882.stateful.{key}"]), key           # min-sum: bit-identical to the reference's code
    x4, _ = oracle.bp2(hx, Z["c882.llr"], None, 4, 0.9, "minsum")
    assert np.array_equal(x4, x2)


@pytest.mark.gpu
def test_cuda_bp2_trainable_and_stateful(ref, allcodes, oracle):
    import fbgnn as F
    Z = ref["bp2"]
    hx = allcodes["c882"].hx
    llr, synd, ew = Z["c882.llr"], Z["c882.synd"], Z["c882.trainable.edge_weights"]
    dec = F.LDPCBPDecoder(hx, trainable=True, is_syndrome=True, num_iter=3, normalization_factor=0.9, cn_type="boxplus-phi",
                          hard_out=False)
    assert dec.has_weights and np.all(dec.edge_weights == 1.0) and len(dec.get_weights()) == 1
    plain = F.LDPCBPDecoder(hx, is_syndrome=True, num_iter=3, normalization_factor=0.9, cn_type="boxplus-phi", hard_out=False)
    assert np.array_equal(dec((llr, synd)), plain((llr, synd)))                 # unit weights change nothing
    dec.set_weights([ew])
    got = dec((llr, synd))
    want, _ = oracle.bp2(hx, llr, synd, 3, 0.9, "boxplus-phi", edge_weights=ew)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.abs(got - Z["c882.trainable.soft"]).max() <= 2e-4
    st = F.LDPCBPDecoder(hx, stateful=True, num_iter=2, normalization_factor=0.9, cn_type="minsum", hard_out=False)
    x1, m1 = st((llr, None))
    x2, m2 = st((llr, m1))
    for got, key in ((x1, "x1"), (x2, "x2"), (m1, "m1"), (m2, "m2")):
        assert np.array_equal(got, Z[f"c882.stateful.{key}"]), key


def test_llr2mi_known_answers():
    """fec/utils.py:151-218: I = 1 - mean(log2(1 + exp(llr))), LLRs clipped to +-20."""
    from fbgnn.decoding import _llr2mi
    assert _llr2mi(np.zeros(7, np.float32)) == 0.0                              # no knowledge
    assert abs(float(_llr2mi(np.full(5, -30.0, np.float32))) - 1.0) < 1e-6      # certain and right (clipped at -20)
    assert abs(float(_llr2mi(np.full(5, 30.0, np.float32))) - (1.0 - 20.0 / np.log(2.0))) < 1e-4


@pytest.mark.gpu
def test_cuda_bp2_track_exit_matches_the_reference_code(allcodes):
    """track_exit=True (decoding.py:955-1000): the EXIT trajectory ie_v / ie_c of the reference's own decoder, executed
    under oracle/tfshim (tests/golden/make_reference_golden_exit.py)."""
    import fbgnn as F
    Z = np.load(os.path.join(GOLDEN, "ref_exit.npz"))
    hx = allcodes["c882"].hx
    for cn_type in ("boxplus-phi", "minsum"):
        dec = F.LDPCBPDecoder(hx, track_exit=True, num_iter=6, normalization_factor=0.9, cn_type=cn_type, hard_out=False)
        assert dec.ie_c == 0 and dec.ie_v == 0                                  # before the first call, as in the reference
        soft = dec(Z["llr"])
        plain = F.LDPCBPDecoder(hx, num_iter=6, normalization_factor=0.9, cn_type=cn_type, hard_out=False)(Z["llr"])
        assert np.array_equal(soft, plain)                                      # tracking does not change the decoding
        assert dec.ie_v.shape == dec.ie_c.shape == (7,) and dec.ie_v[0] == 0 and dec.ie_c[0] == 0
        assert np.abs(dec.ie_v - Z[f"{cn_type}.ie_v"]).max() < 2e-5, cn_type
        assert np.abs(dec.ie_c - Z[f"{cn_type}.ie_c"]).max() < 2e-5, cn_type
        assert np.abs(soft - Z[f"{cn_type}.soft"]).max() < (1e-5 if cn_type == "minsum" else 5e-3)
    # with a syndrome as well, and zero iterations
    Zb = np.load(os.path.join(GOLDEN, "ref_bp2.npz"))
    dec = F.LDPCBPDecoder(hx, track_exit=True, is_syndrome=True, num_iter=3, normalization_factor=0.9, hard_out=False)
    ref3 = F.LDPCBPDecoder(hx, is_syndrome=True, num_iter=3, normalization_factor=0.9, hard_out=False)
    assert np.array_equal(dec((Zb["c882.llr"], Zb["c882.synd"])), ref3((Zb["c882.llr"], Zb["c882.synd"])))
    assert np.all(np.diff(dec.ie_c[1:]) != 0)
    z = F.LDPCBPDecoder(hx, track_exit=True, num_iter=0, hard_out=False)
    z(Z["llr"])
    assert z.ie_c.tolist() == [0.0] and z.ie_v.tolist() == [0.0]


@pytest.mark.parametrize("arith", ["exact", "sfu"])
def test_oracle_gnn_matches_the_reference_code(ref, allcodes, oracle, weights, arith):
    Z = ref["gnn"]
    with oracle.math(arith):
        for cname in ("c882", "c1270"):
            assert int(Z[f"{cname}.count_params"]) == 3923
            assert [tuple(s[:2 if s[1] else 1]) for s in Z[f"{cname}.weight_shapes"]] == [w.shape for w in weights[cname]]
            g = oracle.CodeGraph(allcodes[cname])
            for red in ("mean", "sum", "max", "min"):
                r = Z[f"{cname}.out"] if red == "mean" else Z[f"{cname}.out.{red}"]
                got = oracle.gnn(g, oracle.Gnn(weights[cname], "tanh", red), Z[f"{cname}.h_vn"], Z[f"{cname}.logit_hx"],
                                 Z[f"{cname}.logit_hz"], Z[f"{cname}.sx"], Z[f"{cname}.sz"])
                assert np.abs(got - r).max() <= 1e-6, (cname, red, float(np.abs(got - r).max()))


def _sandwich_cases(Z):
    return sorted({k.rsplit(".", 1)[0] for k in Z.files})


def _check_sandwich(Z, key, code, flags, xd, zd, what):
    n_s = int(Z[f"{key}.shapes"][0][1])
    s_ref = np.unpackbits(Z[f"{key}.s_hat_bits"], axis=1)[:, :n_s]
    s_got = np.concatenate([(xd.astype(np.int64) @ code.hz.T) & 1, (zd.astype(np.int64) @ code.hx.T) & 1], axis=1)
    fl, bl = (flags & 1).astype(bool), ((flags >> 1) & 1).astype(bool)
    p = float(key.rsplit(".", 2)[-2] + "." + key.rsplit(".", 1)[-1])
    need = 0.97 if p <= 0.06 else 0.78        # p = 0.08 / 0.10: the F6 noise floor of a chaotic decoder (25 of 32 frames)
    agree = [np.mean(fl == Z[f"{key}.s_hat_any"]), np.mean(bl == Z[f"{key}.ls_hat_any"]), np.mean(np.all(s_ref == s_got, axis=1))]
    assert min(agree) >= need, (what, key, agree)
    assert abs(int(bl.sum()) - int(Z[f"{key}.ls_hat_any"].sum())) <= 3


@pytest.mark.parametrize("arith", ["exact", "sfu"])
def test_oracle_pipeline_matches_the_reference_model(ref, allcodes, oracle, weights, arith):
    Z = ref["sandwich"]
    with oracle.math(arith):
        for key in _sandwich_cases(Z):
            cname, its, _ = key.split(".", 2)
            its = [int(i) for i in its.split("_")]
            p = float(key.split(".", 2)[2])
            seed, first, B = (int(v) for v in Z[f"{key}.meta"])
            code = allcodes[cname]
            r = oracle.pipeline(oracle.CodeGraph(code), its, [oracle.Gnn(weights[cname])] * (len(its) - 1), p, p0=0.05,
                                seed=seed, first_frame=first, B=B, want_diff=True)
            _check_sandwich(Z, key, code, r["flags"], r["x_diff"], r["z_diff"], f"oracle[{arith}]")


# ------------------------------------------------------------------ the CUDA path against the reference's code ----
@pytest.fixture()
def arith_gpu(request, oracle):
    import fbgnn as F
    ctx = F.default_context()
    ctx.set_math(request.param)
    yield request.param
    ctx.set_math("exact")


@pytest.mark.gpu
@pytest.mark.parametrize("arith_gpu", ["exact", "sfu"], indirect=True)
def test_cuda_bp4_and_gnn_match_the_reference_code(ref, allcodes, weights, arith_gpu):
    import fbgnn as F
    Z = ref["bp4"]
    for key in _bp_cases(Z):
        cname, cn_type, rest = key.split(".", 2)
        factor, it = rest.rsplit(".", 1)
        dec = F.QLDPCBPDecoder(allcodes[cname], num_iter=int(it), normalization_factor=float(factor), cn_type=cn_type,
                               stage_one=True)
        out = dec((Z[f"{cname}.llr"], Z[f"{cname}.sx"], Z[f"{cname}.sz"]))
        got = dict(zip(("Lx", "Ly", "Lz", "x_hat", "z_hat", "x_logit", "z_logit"), out))
        got["x_hat"], got["z_hat"] = got["x_hat"].astype(np.uint8), got["z_hat"].astype(np.uint8)
        assert [o.dtype for o in out] == [np.dtype(d) for d in Z[f"{key}.dtypes"]]           # the reference's output dtypes
        _check_bp4(Z, key, got, f"cuda[{arith_gpu}]")
    Zb = ref["bp2"]
    for key in _bp2_cases(Zb):
        cname, cn_type, it = key.split(".")
        kw = dict(is_syndrome=True, num_iter=int(it), normalization_factor=0.9, cn_type=cn_type)
        soft = F.LDPCBPDecoder(allcodes[cname].hx, hard_out=False, **kw)((Zb[f"{cname}.llr"], Zb[f"{cname}.synd"]))
        hard = F.LDPCBPDecoder(allcodes[cname].hx, **kw)((Zb[f"{cname}.llr"], Zb[f"{cname}.synd"]))
        _check_bp2(Zb, key, soft, hard.astype(np.uint8), f"cuda[{arith_gpu}]")
    Zg = ref["gnn"]
    for cname in ("c882", "c1270"):
        for red in ("mean", "sum", "max", "min"):
            G = F.Feedback_GNN(code=allcodes[cname], num_msg_dims=20, num_hidden_units=40, num_mlp_layers=2, reduce_op=red,
                               activation="tanh", use_bias=True)
            G.set_weights(weights[cname])
            got = G((Zg[f"{cname}.h_vn"], Zg[f"{cname}.logit_hx"], Zg[f"{cname}.logit_hz"], Zg[f"{cname}.sx"], Zg[f"{cname}.sz"]))
            r = Zg[f"{cname}.out"] if red == "mean" else Zg[f"{cname}.out.{red}"]
            assert np.abs(got - r).max() <= 1e-6, (cname, red)


@pytest.mark.gpu
@pytest.mark.parametrize("arith_gpu", ["exact", "sfu"], indirect=True)
def test_cuda_pipeline_matches_the_reference_model(ref, allcodes, weights, arith_gpu):
    import fbgnn as F
    Z = ref["sandwich"]
    for key in _sandwich_cases(Z):
        cname, its, _ = key.split(".", 2)
        its = [int(i) for i in its.split("_")]
        p = float(key.split(".", 2)[2])
        seed, first, B = (int(v) for v in Z[f"{key}.meta"])
        code = allcodes[cname]
        G = F.Feedback_GNN(code=code, num_msg_dims=20, num_hidden_units=40, num_mlp_layers=2, reduce_op="mean",
                           activation="tanh", use_bias=True)
        G.set_weights(weights[cname])
        decs = [F.QLDPCBPDecoder(code, num_iter=i, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True) for i in its]
        model = F.Sandwich_BP_GNN_Evaluation_Model(code, decs, [G] * (len(its) - 1), num_layers=len(its), p0=0.05, seed=seed,
                                                   first_frame=first)
        res = model.run(B, p)
        _check_sandwich(Z, key, code, res["flags"].numpy(), res["x_diff"].numpy(), res["z_diff"].numpy(), f"cuda[{arith_gpu}]")
