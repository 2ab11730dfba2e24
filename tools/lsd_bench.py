"""LSD-0 on a B200: block errors of BP + LSD-0 beside BP + OSD on identical frames, frames LSD-0 abandons, and the device
time of the post-processing launches.  One run writes one JSON (default profiles/lsd_bench.json):

  c882       [[882,24]], p = 0.10, the frames and seed of profiles/osd_bench.json (300 000, seed 70): BP4 (minsum, 100 it.,
             f = 0.8) + OSD-0 / OSD-CS-10 / LSD-0, and the n882.py Sandwich (nG = 5) + OSD-CS-10 / LSD-0.
  hp1922     [[1922,50]], p = 0.06, 10^5 frames: BP4 alone, + OSD-0, + OSD-CS-10, + LSD-0.
  hp7688     [[7688,50]]: BP4 alone against BP4 + LSD-0 at the smallest p of P_GRID where BP4 alone fails on at least 5 % of
             a 4 000-frame probe, on 20 000 frames (about a thousand failed frames).  Every frame BP4 + LSD-0 leaves
             flagged is one LSD-0 abandoned (a solved side meets its syndrome), so its flagged count is the abandoned count.
  kernel     fbgnn_osd_decode (order 0, on the basis) and fbgnn_lsd_decode (default budgets, on the full matrix) on the same
             B frames per side -- the reliabilities and syndromes of a minsum BP4 decode at p = 0.10 -- CUDA events, one
             warm-up and 7 timed launches, µs per frame (every frame of the launch is processed).

Usage: python tools/lsd_bench.py [--out FILE] [--frames 300000]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "feedback-gnn_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402

import fbgnn as F  # noqa: E402
from fbgnn import _ffi  # noqa: E402
from osd_bench import c882, count, gpu_info, hp1922, summary, time_launch  # noqa: E402

P_GRID_7688 = (0.02, 0.025, 0.03, 0.035, 0.04, 0.05)


def hp7688():
    h = F.create_circulant_matrix(62, [0, 2, 5])
    return F.hypergraph_product(h, h)


def bp4(code):
    return F.QLDPCBPDecoder(code, num_iter=100, normalization_factor=0.8, cn_type="minsum", stage_one=True)


def post_models(code, seed, osd_orders=(0, 10), lsd=True, alone=False):
    dec = bp4(code)
    models = {}
    if alone:
        models["bp4"] = F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, p0=None, seed=seed)
    for lam in osd_orders:
        models[f"bp4_osd_{'0' if lam == 0 else f'cs{lam}'}"] = F.BP4_OSD_Model(code, dec, F.OSD_Decoder(code.N, lam),
                                                                              seed=seed)
    if lsd:
        models["bp4_lsd0"] = F.BP4_OSD_Model(code, dec, F.LSD_Decoder(code.N), seed=seed)
    for m in models.values():
        (m._inner if hasattr(m, "_inner") else m).skip_inactive = True
    return models


def count_flagged(model, frames, batch, p):
    k = b = 0
    for _ in range(frames // batch):
        c = model.run(batch, p, want_flags=False, want_diff=False, want_counters=True)["counters"]
        k += int(c[2]); b += int(c[1])
    return {"frames": frames, "block_errors": k, "flagged": b}


def c882_rows(frames, p=0.10, batch=50000, seed=70):
    code = c882()
    res = {name: count(m, frames, batch, p) for name, m in post_models(code, seed).items()}
    G = F.Feedback_GNN(code=code, num_msg_dims=20, num_hidden_units=40, num_mlp_layers=2, reduce_op="mean",
                       activation="tanh", use_bias=True)
    F.load_weights(G, os.path.join(F.WEIGHTS_DIR, "feedback_GNN_n882_k24_wt_4_60_iter_64_16_mixed.npy"))
    d1 = F.QLDPCBPDecoder(code=code, num_iter=64, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code=code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    for name, kw in (("sandwich_nG5_osd_cs10", dict(osd0=True, osd_order=10)),
                     ("sandwich_nG5_lsd0", dict(lsd=F.LSD_Decoder(code.N)))):
        model = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1] + [d2] * 5, [G] * 5, num_layers=6, skip_inactive=True,
                                                   seed=seed, **kw)
        res[name] = count(model, frames, batch, p)
    return dict(p=p, **res)


def hp1922_rows(frames=100000, p=0.06, batch=20000, seed=71):
    models = post_models(hp1922(), seed, alone=True)
    return dict(p=p, **{name: count_flagged(m, frames, batch, p) for name, m in models.items()})


def hp7688_rows(frames=20000, batch=4000, seed=72):
    models = post_models(hp7688(), seed, osd_orders=(), alone=True)
    probe = {}
    for p in P_GRID_7688:
        probe[str(p)] = count_flagged(models["bp4"], batch, batch, p)["flagged"]
        if probe[str(p)] >= 0.05 * batch:
            break
    res = {"p": p, "probe_bp4_flagged_of_4000": probe}
    for name, m in models.items():
        res[name] = count_flagged(m, frames, batch, p)
    res["bp4_lsd0"]["abandoned"] = res["bp4_lsd0"]["flagged"]
    return res


def kernel_rows(code, ctx, seed, B):
    """Per side: OSD-0 on the basis and LSD-0 on the full matrix, the same frames (llr_z' with hx, llr_x' with hz)."""
    n = code.N
    nx, nz = F.Pauli(seed=seed).sample_device(B, n, F.pauli_thresholds(0.10))
    gx, gz = _ffi.Graph(code.hx, ctx), _ffi.Graph(code.hz, ctx)
    sx, sz = ctx.empty((B, gx.m), np.uint8), ctx.empty((B, gz.m), np.uint8)
    _ffi.call("fbgnn_syndrome", gx.handle, B, nz.t2(), sx.T.t2())
    _ffi.call("fbgnn_syndrome", gz.handle, B, nx.t2(), sz.T.t2())
    Lx, Ly, Lz = (a.numpy().astype(np.float64) for a in bp4(code)((ctx.asarray(np.full((B, 3, n), np.log(27.0),
                                                                                         np.float32)), sx.T, sz.T))[:3])
    sp = lambda x: np.logaddexp(0.0, x)                                              # noqa: E731
    llr_z = (sp(-Lx) - np.logaddexp(-Lz, -Ly)).astype(np.float32)
    llr_x = (sp(-Lz) - np.logaddexp(-Lx, -Ly)).astype(np.float32)
    out = {}
    for side, g, H, piv, llr, s in (("x", gx, code.hx, code.pivot_hx, llr_z, sx.numpy()),
                                    ("z", gz, code.hz, code.pivot_hz, llr_x, sz.numpy())):
        llr_d = ctx.asarray(llr, np.float32)
        full = ctx.asarray(np.ascontiguousarray(s.T), np.uint8)                      # [m, B]
        red = ctx.asarray(np.ascontiguousarray(s[:, piv].T), np.uint8)               # [rank, B]
        gb = _ffi.Graph(H[piv], ctx)
        e = ctx.empty((B, n), np.uint8)
        st = ctx.empty((B,), np.uint8)
        osd = lambda: _ffi.call("fbgnn_osd_decode", gb.handle, 0, B, llr_d.t2(), red.t2(), e.t2())       # noqa: E731
        lsd = lambda: _ffi.call("fbgnn_lsd_decode", g.handle, 0, 0, B, llr_d.t2(), full.t2(), e.t2(), st.ptr)  # noqa: E731
        row = {"osd0": summary(time_launch(ctx, osd, B), B), "lsd0": summary(time_launch(ctx, lsd, B), B)}
        row["lsd0"]["status_counts"] = np.bincount(st.numpy(), minlength=3).tolist()
        out[side] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lsd_bench.json"))
    ap.add_argument("--frames", type=int, default=300000)
    args = ap.parse_args()
    ctx = F.default_context()
    res = {"device": ctx.name, "nvidia_smi": gpu_info(), "math": ctx.get_math(),
           "kernel_B4096": {"c882": kernel_rows(c882(), ctx, 1, 4096), "hp1922": kernel_rows(hp1922(), ctx, 2, 4096)},
           "c882": c882_rows(args.frames), "hp1922": hp1922_rows(), "hp7688": hp7688_rows()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res)[:6000])


if __name__ == "__main__":
    main()
