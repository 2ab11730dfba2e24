"""OSD-CS on a B200: kernel time per frame of fbgnn_osd_decode by order, and block errors of BP + OSD-{0, CS} on identical
frames.  One run writes one JSON (default profiles/osd_bench.json):

  kernel     fbgnn_osd_decode at B = 8192 for λ in {0, 1, 10, 30, 60}, on both sides of [[882,24]] and [[1270,28]]; the
             reliabilities are the llr_x' / llr_z' (bp_osd.py:135-144) of a minsum BP4 decode (100 it., f = 0.8) at p = 0.10.
             CUDA events around each launch, one warm-up launch, 7 timed launches: median, min and max.
  ler        BP4(minsum, 100 it., f = 0.8) + OSD-{0, CS-10, CS-60} on [[882,24]], 300 000 frames at p = 0.10, the same seed
             for all (examples/OSD.ipynb cell 2; published OSD-0: 111 / 300 000), and the n882.py Sandwich (nG = 5) without
             OSD, with OSD-0 and with OSD-CS-10 at p = 0.10.

With --cluster it measures the thread-block-cluster form of the kernel (csrc/fbgnn_osd_cluster.cuh) instead and writes
profiles/osd_cluster_bench.json:

  kernel     fbgnn_osd_decode at B = 4096 for λ in {0, 10, 60}, on both sides of the [[1922,50]] hypergraph-product code
             (one CTA cannot hold its reduced matrix), reliabilities as above.
  overhead   [[1270,28]] (hx side), which one CTA holds: k_osd against the cluster kernel forced with FBGNN_OSD_CLUSTER=2,
             same frames, the two launches alternated 7 times per order.
  ler        BP4(minsum, 100 it., f = 0.8) alone, + OSD-0 and + OSD-CS-10 on the same --frames frames of [[1922,50]], at
             the smallest p of P_GRID where BP4 alone fails on at least 1 % of a 20 000-frame probe.

Usage: python tools/osd_bench.py [--out FILE] [--frames 300000] [--kernel-only] [--cluster]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "feedback-gnn_b200"))
import numpy as np  # noqa: E402

import fbgnn as F  # noqa: E402
from fbgnn import _ffi  # noqa: E402

ORDERS = (0, 1, 10, 30, 60)
B_KERNEL = 8192
REPS = 7


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def smem_optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def c882():
    return F.create_QC_GHP_codes(63, F.create_cyclic_permuting_matrix(7, [27, 54, 0]), [0, 1, 6])


def c1270():
    return F.create_QC_GHP_codes(127, np.array([[0, -1, 51, 52, -1], [-1, 0, -1, 111, 20], [0, -1, 98, -1, 122],
                                                [0, 80, -1, 119, -1], [-1, 0, 5, -1, 106]]), [0, 1, 7],
                                 name="GHP_n1270_k28")


def smem_bytes(n, R, lam, C=1):
    """Dynamic shared memory of one k_osd CTA, or with C > 1 of each CTA of k_osd_cluster (osd_smem in
    csrc/fbgnn_pipeline.cu)."""
    rows = R if C == 1 else ((R + 31) // 32 + C - 1) // C * 32
    W, Rp = (n + 32) // 32, rows | 1
    npad = 1 << (n - 1).bit_length()
    main = (max(npad * 8, W * Rp * 4) + 7) & ~7
    u16 = 2 * (2 * n + R)
    smem, base = main + u16 + 16, main + ((u16 + 15) & ~15)
    if C > 1:
        smem = base + 4 * (3 * (W + 1) + rows // 32)
        base = (smem + 15) & ~15
    if lam == 0:
        return smem
    lp, RW = min(lam, max(n - R, 0)), (R + 31) // 32
    return base + (lp + 1) * RW * 4 + (4 * n if C > 1 else 0)


def cluster_size(n, R, lam, optin):
    """CTAs per frame launch_osd picks: 1 if one CTA fits, else the smallest of 2 / 4 / 8 (None: unsupported)."""
    return next((C for C in (1, 2, 4, 8) if smem_bytes(n, R, lam, C) <= optin), None)


def osd_inputs(code, ctx, seed, B):
    """Per side (x: hx with llr_z', z: hz with llr_x'): (basis graph, rank, llr [B, n], reduced syndrome [rank, B]) on
    the device, from a minsum BP4 decode at p = 0.10."""
    n = code.N
    nx, nz = F.Pauli(seed=seed).sample_device(B, n, F.pauli_thresholds(0.10))
    gx, gz = _ffi.Graph(code.hx, ctx), _ffi.Graph(code.hz, ctx)
    sx, sz = ctx.empty((B, gx.m), np.uint8), ctx.empty((B, gz.m), np.uint8)
    _ffi.call("fbgnn_syndrome", gx.handle, B, nz.t2(), sx.T.t2())
    _ffi.call("fbgnn_syndrome", gz.handle, B, nx.t2(), sz.T.t2())
    dec = F.QLDPCBPDecoder(code, num_iter=100, normalization_factor=0.8, cn_type="minsum", stage_one=True)
    Lx, Ly, Lz = (a.numpy().astype(np.float64) for a in dec((ctx.asarray(np.full((B, 3, n), np.log(27.0), np.float32)),
                                                             sx.T, sz.T))[:3])
    sp = lambda x: np.logaddexp(0.0, x)                                              # noqa: E731
    llr_z = (sp(-Lx) - np.logaddexp(-Lz, -Ly)).astype(np.float32)                   # pairs with hx
    llr_x = (sp(-Lz) - np.logaddexp(-Lx, -Ly)).astype(np.float32)                   # pairs with hz
    sxh, szh = sx.numpy(), sz.numpy()
    out = {}
    for side, H, piv, llr, s in (("x", code.hx, code.pivot_hx, llr_z, sxh), ("z", code.hz, code.pivot_hz, llr_x, szh)):
        basis = H[piv]
        out[side] = (_ffi.Graph(basis, ctx), basis.shape[0], ctx.asarray(llr, np.float32),
                     ctx.asarray(np.ascontiguousarray(s[:, piv].T), np.uint8))              # [rank, B]
    return out


def time_launch(ctx, run, B):
    """Per-frame time of run(): one warm-up launch, then REPS launches timed with CUDA events."""
    run()
    ctx.sync()
    ms = []
    for _ in range(REPS):
        ctx.timer_start()
        run()
        ms.append(ctx.timer_stop())
    return np.array(ms)


def summary(ms, B):
    return {"us_per_frame_median": float(np.median(ms)) * 1e3 / B, "us_per_frame_min": float(ms.min()) * 1e3 / B,
            "us_per_frame_max": float(ms.max()) * 1e3 / B, "ms_per_launch": ms.tolist()}


def kernel_times(code, ctx, seed, orders=ORDERS, B=B_KERNEL):
    """Per side: {order: {median_us_per_frame, min, max, ms_per_launch}}."""
    n = code.N
    out = {}
    for side, (g, R, llr_d, red_d) in osd_inputs(code, ctx, seed, B).items():
        e = ctx.empty((B, n), np.uint8)
        res = {"rank": R, "n_minus_rank": n - R}
        for lam in orders:
            run = lambda: _ffi.call("fbgnn_osd_decode", g.handle, lam, B, llr_d.t2(), red_d.t2(), e.t2())  # noqa: E731
            C = cluster_size(n, R, lam, smem_optin())
            res[str(lam)] = dict(summary(time_launch(ctx, run, B), B), ctas_per_frame=C,
                                 smem_bytes_per_cta=smem_bytes(n, R, lam, C or 8),
                                 candidates=1 + (0 if lam == 0 else (n - R) + min(lam, n - R) * (min(lam, n - R) - 1) // 2))
        out[side] = res
    return out


def hp1922():
    h = F.create_circulant_matrix(31, [0, 2, 5])
    return F.hypergraph_product(h, h)


def cluster_overhead(ctx, B=4096, seed=3):
    """[[1270,28]], hx side: k_osd and the cluster kernel forced onto 2 CTAs, alternated on the same frames."""
    code = c1270()
    g, R, llr_d, red_d = osd_inputs(code, ctx, seed, B)["x"]
    e = ctx.empty((B, code.N), np.uint8)
    out = {"rank": R}
    for lam in (0, 10, 60):
        run = lambda: _ffi.call("fbgnn_osd_decode", g.handle, lam, B, llr_d.t2(), red_d.t2(), e.t2())  # noqa: E731
        ms = {"k_osd": [], "cluster2": []}
        for _ in range(REPS):
            for key in ms:
                if key == "cluster2":
                    os.environ["FBGNN_OSD_CLUSTER"] = "2"
                ms[key].append(float(np.median(time_launch(ctx, run, B))))
                os.environ.pop("FBGNN_OSD_CLUSTER", None)
        out[str(lam)] = {k: summary(np.array(v), B) for k, v in ms.items()}
        out[str(lam)]["ratio_median"] = (out[str(lam)]["cluster2"]["us_per_frame_median"] /
                                         out[str(lam)]["k_osd"]["us_per_frame_median"])
    return out


P_GRID = (0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.10)


def cluster_block_errors(frames, batch=20000, seed=71):
    code = hp1922()
    dec = F.QLDPCBPDecoder(code, num_iter=100, normalization_factor=0.8, cn_type="minsum", stage_one=True)
    models = {"bp4": F.Sandwich_BP_GNN_Evaluation_Model(code, [dec], [], num_layers=1, p0=None, seed=seed)}
    for lam in (0, 10):
        models[f"bp4_osd_{'0' if lam == 0 else f'cs{lam}'}"] = F.BP4_OSD_Model(
            code, dec, F.OSD_Decoder(code.N, osd_order=lam), seed=seed)
    for m in models.values():
        (m._inner if hasattr(m, "_inner") else m).skip_inactive = True
    probe = {}
    for p in P_GRID:
        probe[str(p)] = count(models["bp4"], batch, batch, p)["block_errors"]
        if probe[str(p)] >= 0.01 * batch:
            break
    res = {"p": p, "probe_bp4_block_errors_of_20000": probe}
    for name, m in models.items():
        res[name] = count(m, frames, batch, p)
    return res


def count(model, frames, batch, p):
    k, t0 = 0, time.perf_counter()
    for _ in range(frames // batch):
        k += int(model.run(batch, p, want_flags=False, want_diff=False, want_counters=True)["counters"][2])
    return {"frames": frames, "block_errors": k, "seconds": time.perf_counter() - t0}


def block_errors(frames, p=0.10, batch=50000, seed=70):
    code = c882()
    res = {}
    dec = F.QLDPCBPDecoder(code, num_iter=100, normalization_factor=0.8, cn_type="minsum", stage_one=True)
    for lam in (0, 10, 60):
        model = F.BP4_OSD_Model(code, dec, F.OSD_Decoder(code.N, osd_order=lam), seed=seed)
        model._inner.skip_inactive = True
        res[f"bp4_osd_{'0' if lam == 0 else f'cs{lam}'}"] = count(model, frames, batch, p)
    G = F.Feedback_GNN(code=code, num_msg_dims=20, num_hidden_units=40, num_mlp_layers=2, reduce_op="mean",
                       activation="tanh", use_bias=True)
    F.load_weights(G, os.path.join(F.WEIGHTS_DIR, "feedback_GNN_n882_k24_wt_4_60_iter_64_16_mixed.npy"))
    d1 = F.QLDPCBPDecoder(code=code, num_iter=64, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code=code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    for name, kw in (("sandwich_nG5", {}), ("sandwich_nG5_osd0", dict(osd0=True)),
                     ("sandwich_nG5_osd_cs10", dict(osd0=True, osd_order=10))):
        model = F.Sandwich_BP_GNN_Evaluation_Model(code, [d1] + [d2] * 5, [G] * 5, num_layers=6, skip_inactive=True,
                                                   seed=seed, **kw)
        res[name] = count(model, frames, batch, p)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "osd_bench.json"))
    ap.add_argument("--frames", type=int, default=300000)
    ap.add_argument("--kernel-only", action="store_true")
    ap.add_argument("--cluster", action="store_true")
    args = ap.parse_args()
    ctx = F.default_context()
    if args.cluster:
        out = args.out if args.out != ap.get_default("out") else os.path.join(ROOT, "profiles", "osd_cluster_bench.json")
        res = {"device": ctx.name, "nvidia_smi": gpu_info(), "math": ctx.get_math(), "B": 4096, "reps": REPS,
               "smem_optin": smem_optin(),
               "kernel": {"hp1922": kernel_times(hp1922(), ctx, 1, orders=(0, 10, 60), B=4096)},
               "overhead_c1270": cluster_overhead(ctx)}
        if not args.kernel_only:
            res["block_errors"] = cluster_block_errors(args.frames)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res)[:4000])
        return
    res = {"device": ctx.name, "nvidia_smi": gpu_info(), "math": ctx.get_math(), "B": B_KERNEL, "reps": REPS,
           "kernel": {"c882": kernel_times(c882(), ctx, 1), "c1270": kernel_times(c1270(), ctx, 2)}}
    if not args.kernel_only:
        res["block_errors_p010"] = block_errors(args.frames)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res)[:4000])


if __name__ == "__main__":
    main()
