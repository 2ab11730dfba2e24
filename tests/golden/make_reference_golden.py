"""Generates tests/golden/ref_*.npz by EXECUTING THE REFERENCE'S OWN SOURCE FILES (from /root/reference, unmodified)
on seeded inputs -- possible without TensorFlow because oracle/tfshim restates the few TensorFlow / Keras primitives
those files call in numpy (see its docstring for the semantics it keeps).  What these fixtures pin is therefore the
reference's code path itself: code construction and GF(2) algebra (numpy only, exact), edge orders / permutations /
x-z swaps / clip constants of QLDPCBPDecoder.call, the weight order and feature layout of Feedback_GNN.call with the
shipped weights loaded by the reference's own load_weights, and the flag logic of
Sandwich_BP_GNN_Evaluation_Model.call.  Elementary functions come from numpy's libm, so float outputs carry float32
rounding noise relative to TensorFlow's (and to the oracle's); tests/test_reference_goldens.py states the tolerances.

    python tests/golden/make_reference_golden.py          (only where /root/reference exists; ~1 min)
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "feedback-gnn_b200"))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

from oracle import run_reference as R                      # noqa: E402

W882 = "feedback_GNN_n882_k24_wt_4_60_iter_64_16_mixed.npy"
W1270 = "feedback_GNN_n1270_k28_wt_10_80_iter_64_16_mixed.npy"
REF_WEIGHTS = os.path.join(R.REF, "sionna", "fec", "ldpc", "weights")


# ---- the noise source of this repository (Philox4x32-10 keyed by (seed, global frame id)), in numpy, so that the
# ---- reference can be driven with exactly the uniforms the oracle / the GPU use
def philox4x32_10(c0, c1, c2, c3, k0, k1):
    c0, c1, c2, c3 = (np.asarray(c, np.uint64) for c in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0), np.uint64(k1)
    M0, M1, MASK = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & MASK, p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = (hi1 ^ c1 ^ k0) & MASK, lo1, (hi0 ^ c3 ^ k1) & MASK, lo0
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK, (k1 + np.uint64(0xBB67AE85)) & MASK
    return c0, c1, c2, c3


def frame_uniforms(seed, first_frame, B, n, stream=0):
    frames = (np.arange(B, dtype=np.uint64) + np.uint64(first_frame))[:, None]
    q4 = np.arange((n + 3) // 4, dtype=np.uint64)[None, :]
    r = philox4x32_10(frames & np.uint64(0xFFFFFFFF), frames >> np.uint64(32), q4 + 0 * frames, np.uint64(stream) + 0 * frames + 0 * q4,
                      seed & 0xFFFFFFFF, seed >> 32)
    words = np.stack(r, axis=-1).reshape(B, -1)[:, :n]
    return ((words >> np.uint64(8)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)


def syndromes(code, nx, nz):
    return ((code.hx @ nz.T.astype(np.int64)) & 1), ((code.hz @ nx.T.astype(np.int64)) & 1)


def main():
    ns = R.load()
    tf, Q = ns.tf, ns.codes_q
    out = {}

    # ---------------------------------------------------------------- 1. code construction (exact integers)
    codes = {
        "steane": lambda: Q.css_code(Q.hamming_code(3), Q.hamming_code(3), name="Steane_n7_k1_d3"),
        "rsurf3": lambda: Q.create_rotated_surface_codes(3),
        "rsurf5": lambda: Q.create_rotated_surface_codes(5),
        "toric4": lambda: Q.create_checkerboard_toric_codes(4),
        "surf3": lambda: Q.create_surface_codes(3),
        "gb48": lambda: Q.create_generalized_bicycle_codes(24, [0, 2, 8, 15], [0, 2, 12, 17], name="GB_n48_k6_d8"),
        "hp162": lambda: Q.hypergraph_product(Q.create_circulant_matrix(9, [0, 2, 5]), Q.create_circulant_matrix(9, [0, 2, 5])),
        "ibm72": lambda: Q.create_bivariate_QC_codes(6, 6, [3], [1, 2], [1, 2], [3]),
        "c882": lambda: Q.create_QC_GHP_codes(63, Q.create_cyclic_permuting_matrix(7, [27, 54, 0]), [0, 1, 6]),
        "c1270": lambda: Q.create_QC_GHP_codes(127, np.array([[0, -1, 51, 52, -1], [-1, 0, -1, 111, 20], [0, -1, 98, -1, 122],
                                                             [0, 80, -1, 119, -1], [-1, 0, 5, -1, 106]]), [0, 1, 7],
                                               name="GHP_n1270_k28"),
    }
    built = {}
    cz = {}
    for name, make in codes.items():
        c = built[name] = make()
        for attr in ("hx", "hz", "lx", "lz", "hx_perp", "hz_perp"):
            m = np.asarray(getattr(c, attr)).astype(np.uint8)
            cz[f"{name}.{attr}.shape"] = np.array(m.shape)
            cz[f"{name}.{attr}.bits"] = np.packbits(m, axis=None)
        cz[f"{name}.pivot_hx"], cz[f"{name}.pivot_hz"] = np.array(c.pivot_hx), np.array(c.pivot_hz)
        cz[f"{name}.params"] = np.array([c.N, c.K, c.rank_hx, c.rank_hz, int(c.L), int(c.Q), int(c.D)])
        cz[f"{name}.name"] = np.array(c.name)
        print("code", name, c.N, c.K, c.name)
    np.savez_compressed(os.path.join(HERE, "ref_codes.npz"), **cz)

    # ---------------------------------------------------------------- 2. QLDPCBPDecoder.call (decoding_q.py:661-797)
    bp = {}
    for cname, B, p, cases in (("c882", 8, 0.06, [("boxplus-phi", 1.0, (1, 2, 3)), ("boxplus-phi", 0.625, (2,)),
                                                  ("minsum", 0.8, (1, 3)), ("boxplus", 1.0, (1, 2))]),
                               ("rsurf3", 16, 0.08, [("boxplus-phi", 1.0, (1, 2, 4)), ("minsum", 0.8, (2,))]),
                               ("c1270", 4, 0.06, [("boxplus-phi", 1.0, (1, 2))])):
        code = built[cname]
        u = frame_uniforms(11, 0, B, code.N)
        tf.random.provider = lambda shape, u=u: u
        nx, nz = ns.Pauli()([tf.zeros([B, code.N]), None, 2 * p / 3, p / 3, 2 * p / 3])
        tf.random.provider = None
        nx, nz = np.asarray(nx), np.asarray(nz)
        sx, sz = syndromes(code, nx, nz)
        rng = np.random.default_rng(3)
        prior = np.float32(np.log(np.float64(np.float32(3. * (1. - 0.05) / 0.05))))
        llr = (prior + rng.normal(0, 0.3, (B, 3, code.N))).astype(np.float32)
        bp[f"{cname}.noise_x"], bp[f"{cname}.noise_z"] = nx, nz
        bp[f"{cname}.llr"], bp[f"{cname}.sx"], bp[f"{cname}.sz"] = llr, sx.astype(np.uint8), sz.astype(np.uint8)
        bp[f"{cname}.p"] = np.float64(p)
        for cn_type, factor, iters in cases:
            for it in iters:
                dec = ns.QLDPCBPDecoder(code=code, num_iter=tf.constant(it), normalization_factor=tf.constant(factor),
                                        cn_type=cn_type, trainable=False, stage_one=True)
                res = dec((tf.constant(llr), tf.constant(sx), tf.constant(sz)))
                key = f"{cname}.{cn_type}.{factor}.{it}"
                for k, o in zip(("Lx", "Ly", "Lz", "x_hat", "z_hat", "x_logit", "z_logit"), res):
                    o = np.asarray(o)
                    bp[f"{key}.{k}"] = o.astype(np.uint8) if k.endswith("hat") else o
                bp[f"{key}.dtypes"] = np.array([str(np.asarray(o).dtype) for o in res])
                print("bp4", key)
        if cname == "c882":          # stage_two output: per-iteration soft syndromes (decoding_q.py:743-746, 794-795)
            dec = ns.QLDPCBPDecoder(code=code, num_iter=tf.constant(2), normalization_factor=tf.constant(1.0),
                                    cn_type="boxplus-phi", trainable=False, stage_two=True)
            llr_hat, xh, zh = dec((tf.constant(llr), tf.constant(sx), tf.constant(sz)))
            bp["c882.stage_two.llr_hat"] = np.asarray(llr_hat)
            # trainable=True without stage flags: the same output over the DENSE hx_perp / hz_perp rows (decoding_q.py:32-33)
            dec = ns.QLDPCBPDecoder(code=code, num_iter=tf.constant(2), normalization_factor=tf.constant(1.0),
                                    cn_type="boxplus-phi", trainable=True)
            llr_hat, xh, zh = dec((tf.constant(llr[:4]), tf.constant(sx[:, :4]), tf.constant(sz[:, :4])))
            bp["c882.trainable.llr_hat"] = np.asarray(llr_hat)
    # two files, so that each stays under 1 MB
    np.savez_compressed(os.path.join(HERE, "ref_bp4.npz"), **{k: v for k, v in bp.items() if k.startswith("c882.")})
    np.savez_compressed(os.path.join(HERE, "ref_bp4_c1270_rsurf3.npz"),
                        **{k: v for k, v in bp.items() if not k.startswith("c882.")})

    # ---------------------------------------------------------------- 2b. LDPCBPDecoder.call, is_syndrome (decoding.py:875-1048)
    from oracle import c_oracle as O
    b2 = {}
    for cname, B in (("c882", 12), ("rsurf3", 24), ("c1270", 6)):
        code = built[cname]
        noise = O.bsc(5, 0, B, code.N, 0.04)
        synd = (code.hx @ noise.T.astype(np.int64)) & 1
        rng = np.random.default_rng(0)
        llr = (-np.log((1 - 0.1) / 0.1) + rng.normal(0, 0.2, (B, code.N))).astype(np.float32)
        llr[0, :3] = [30.0, -30.0, 0.0]                                      # exercises the +-20 clip
        b2[f"{cname}.llr"], b2[f"{cname}.synd"] = llr, synd.astype(np.uint8)
        for cn_type in ("boxplus-phi", "minsum", "boxplus"):
            for it in (1, 2, 5):
                dec = ns.LDPCBPDecoder(code.hx, is_syndrome=True, num_iter=it, normalization_factor=0.9, cn_type=cn_type,
                                       hard_out=False)
                b2[f"{cname}.{cn_type}.{it}.soft"] = np.asarray(dec((tf.constant(llr), tf.constant(synd))))
                hard = ns.LDPCBPDecoder(code.hx, is_syndrome=True, num_iter=it, normalization_factor=0.9, cn_type=cn_type)
                b2[f"{cname}.{cn_type}.{it}.hard"] = np.asarray(hard((tf.constant(llr), tf.constant(synd)))).astype(np.uint8)
        if cname == "c882":
            # trainable=True: per-edge weights on the v2c messages (decoding.py:361-366, 981-983), here set to random values
            dec = ns.LDPCBPDecoder(code.hx, trainable=True, is_syndrome=True, num_iter=3, normalization_factor=0.9,
                                   cn_type="boxplus-phi", hard_out=False)
            ew = (1.0 + 0.2 * np.random.default_rng(9).standard_normal(int(code.hx.sum()))).astype(np.float32)
            dec._edge_weights.assign(ew)
            b2["c882.trainable.edge_weights"] = ew
            b2["c882.trainable.soft"] = np.asarray(dec((tf.constant(llr), tf.constant(synd))))
            # stateful=True: (llr, msg_vn) -> (x, msg_vn); two calls of 2 iterations == one call of 4 (decoding.py:947-953)
            dec = ns.LDPCBPDecoder(code.hx, stateful=True, num_iter=2, normalization_factor=0.9, cn_type="minsum", hard_out=False)
            x1, m1 = dec((tf.constant(llr), None))
            x2, m2 = dec((tf.constant(llr), m1))
            b2["c882.stateful.x1"], b2["c882.stateful.x2"] = np.asarray(x1), np.asarray(x2)
            b2["c882.stateful.m1"], b2["c882.stateful.m2"] = np.asarray(m1.flat_values), np.asarray(m2.flat_values)
        print("bp2", cname)
    np.savez_compressed(os.path.join(HERE, "ref_bp2.npz"), **b2)

    # ---------------------------------------------------------------- 3. Feedback_GNN.call with the shipped weights
    gn = {}
    for cname, wfile, B in (("c882", W882, 8), ("c1270", W1270, 4)):
        code = built[cname]
        bs, n = tf.constant(B), tf.constant(code.N)
        mx, mz = tf.constant(code.hx.shape[0]), tf.constant(code.hz.shape[0])
        G = ns.Feedback_GNN(code=code, num_msg_dims=tf.constant(20), num_hidden_units=tf.constant(40), num_mlp_layers=2,
                            reduce_op="mean", activation="tanh", use_bias=True)
        G((tf.zeros((bs, n, 3)), tf.zeros((mx, bs)), tf.zeros((mz, bs)), tf.zeros((mx, bs)), tf.zeros((mz, bs))))
        ns.load_weights(G, os.path.join(REF_WEIGHTS, wfile))              # the reference's own pickle.load + set_weights
        gn[f"{cname}.weight_shapes"] = np.array([w.shape + (0,) * (2 - w.ndim) for w in G.get_weights()])
        gn[f"{cname}.count_params"] = np.array(G.count_params())
        # inputs: a real first-stage state, produced by the reference decoder itself (16 iterations)
        u = frame_uniforms(12, 0, B, code.N)
        tf.random.provider = lambda shape, u=u: u
        nx, nz = ns.Pauli()([tf.zeros([B, code.N]), None, 2 * 0.1 / 3, 0.1 / 3, 2 * 0.1 / 3])
        tf.random.provider = None
        sx, sz = syndromes(code, np.asarray(nx), np.asarray(nz))
        prior = np.float32(np.log(np.float64(np.float32(57.0))))
        llr = np.full((B, 3, code.N), prior, np.float32)
        dec = ns.QLDPCBPDecoder(code=code, num_iter=tf.constant(16), normalization_factor=tf.constant(1.0),
                                cn_type="boxplus-phi", trainable=False, stage_one=True)
        llrx, llry, llrz, xh, zh, xl, zl = dec((tf.constant(llr), tf.constant(sx), tf.constant(sz)))
        h_vn = tf.stack([llrx, llry, llrz], axis=-1)
        new_llr = G((h_vn, zl, xl, tf.constant(sx), tf.constant(sz)))         # argument order of feedback_gnn.py:335
        for k, v in (("h_vn", h_vn), ("logit_hx", zl), ("logit_hz", xl), ("sx", sx.astype(np.uint8)),
                     ("sz", sz.astype(np.uint8)), ("out", new_llr)):
            gn[f"{cname}.{k}"] = np.asarray(v)
        for red in ("sum", "max", "min"):
            G2 = ns.Feedback_GNN(code=code, num_msg_dims=tf.constant(20), num_hidden_units=tf.constant(40),
                                 num_mlp_layers=2, reduce_op=red, activation="tanh", use_bias=True)
            G2((tf.zeros((bs, n, 3)), tf.zeros((mx, bs)), tf.zeros((mz, bs)), tf.zeros((mx, bs)), tf.zeros((mz, bs))))
            G2.set_weights(G.get_weights())
            gn[f"{cname}.out.{red}"] = np.asarray(G2((h_vn, zl, xl, tf.constant(sx), tf.constant(sz))))
        print("gnn", cname, G.count_params())
    np.savez_compressed(os.path.join(HERE, "ref_gnn.npz"), **gn)

    # ---------------------------------------------------------------- 4. Sandwich_BP_GNN_Evaluation_Model.call
    sw = {}
    for cname, wfile, iters, B, p, seed in (("c882", W882, [16, 8, 8], 96, 0.06, 21), ("c882", W882, [32, 16], 64, 0.10, 22),
                                            ("c1270", W1270, [24, 8], 32, 0.08, 23)):
        code = built[cname]
        bs, n = tf.constant(B), tf.constant(code.N)
        mx, mz = tf.constant(code.hx.shape[0]), tf.constant(code.hz.shape[0])
        G = ns.Feedback_GNN(code=code, num_msg_dims=tf.constant(20), num_hidden_units=tf.constant(40), num_mlp_layers=2,
                            reduce_op="mean", activation="tanh", use_bias=True)
        G((tf.zeros((bs, n, 3)), tf.zeros((mx, bs)), tf.zeros((mz, bs)), tf.zeros((mx, bs)), tf.zeros((mz, bs))))
        ns.load_weights(G, os.path.join(REF_WEIGHTS, wfile))
        decs = [ns.QLDPCBPDecoder(code=code, num_iter=tf.constant(it), normalization_factor=tf.constant(1.0),
                                  cn_type="boxplus-phi", trainable=False, stage_one=True) for it in iters]
        model = ns.Sandwich_BP_GNN_Evaluation_Model(code, decs, [G] * (len(iters) - 1), num_layers=len(iters))
        u = frame_uniforms(seed, 1000, B, code.N)
        tf.random.provider = lambda shape, u=u: u
        s_hat, ls_hat = model(tf.constant(B), p)
        tf.random.provider = None
        key = f"{cname}.{'_'.join(map(str, iters))}.{p}"
        sw[f"{key}.s_hat_any"] = np.any(np.asarray(s_hat), axis=1)
        sw[f"{key}.ls_hat_any"] = np.any(np.asarray(ls_hat), axis=1)
        sw[f"{key}.s_hat_bits"] = np.packbits(np.asarray(s_hat).astype(np.uint8), axis=1)
        sw[f"{key}.ls_hat_bits"] = np.packbits(np.asarray(ls_hat).astype(np.uint8), axis=1)
        sw[f"{key}.shapes"] = np.array([s_hat.shape, ls_hat.shape])
        sw[f"{key}.meta"] = np.array([seed, 1000, B])
        print("sandwich", key, int(sw[f"{key}.s_hat_any"].sum()), int(sw[f"{key}.ls_hat_any"].sum()))
    np.savez_compressed(os.path.join(HERE, "ref_sandwich.npz"), **sw)


if __name__ == "__main__":
    main()
