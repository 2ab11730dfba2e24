#!/usr/bin/env python
"""bench.py -- headline benchmark of the BP -> feedback-GNN -> BP hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Every timed section runs K steps.

Workload (BASELINE.json configs[2], named in config.workload): the [[1270,28]] GHP code, decoders
(64, G, 16, G, 16, G, 16) with the shipped weights (the configuration of n1270.py / the reference's
published table, examples/n1270.ipynb cell 2), depolarising noise p = 0.10, BP prior p0 = 0.05,
every frame runs every round (reference-equivalent work; no round skipping), B frames per step per
GPU.  A "step" = one pass of the whole pipeline over one batch of B synthetic frames.

  value         frames/s, device-timed (CUDA events on the launching stream), noise sampled in-kernel; --math sfu
                (default: exp / log on the special-function unit) or exact (FP32 polynomials) -- both bit-exact
                against the CPU oracle in the same arithmetic; the other arithmetic is timed beside it
  e2e           frames/s through the public Python API with HOST buffers: per step the noise bit-planes
                (packed, 32 qubits per word) are copied from pinned host memory, the pipeline runs on them
                (fbgnn_pipeline_run_bits) and the indicator planes + counters are read back to the host
  roofline      the dominant kernel (k_bp4, stage 0) against the MEASURED MUFU peak (SURVEY.md 8(d): the path
                is transcendental-bound, not HBM- or tensor-bound): frac on the algorithmic work, executed_frac
                on the iterations the kernel reports as executed, issue_frac / traffic / pipe utilisation from the
                committed ncu capture of the same launch (profiles/r02_ncu_k_bp4_stage0_<math>.json)
  cpu_baseline  the CPU oracle (oracle/fbgnn_oracle.c, the restatement of the reference; TensorFlow is not
                installable in this image) on the box's host cores, bounded sample; the numpy oracle beside it
  --impl reference   times that same CPU restatement alone (all host threads) and prints its line
  N > 1         one process per GPU (RANK / WORLD_SIZE from the launcher), frames sharded by global frame id, one
                NCCL all-reduce of the four counters per step inside the timed region (libfbgnn.so; no PyTorch)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "feedback-gnn_b200"))
sys.path.insert(0, ROOT)

import numpy as np

P_NOISE = 0.10
P0 = 0.05
N_G = 3
NUM_ITERS = [64] + [16] * N_G
WEIGHTS = "feedback_GNN_n1270_k28_wt_10_80_iter_64_16_mixed.npy"
WORKLOAD = ("[[1270,28]] GHP code, BP4(64)->(GNN->BP4(16))x3 with trained weights (n1270.py -nG 3), "
            "depolarising p=0.10, p0=0.05, f=1.0, boxplus-phi, full work (no round skipping)")
# algorithmic transcendental evaluations (SURVEY.md 8(d)): BP4 iteration 52n, epilogue 29n, GNN 560n
N_Q = 1270
TE_ITER = 52 * N_Q
TE_EPI = 29 * N_Q
TE_GNN = 560 * N_Q
TE_PER_FRAME = sum(NUM_ITERS) * TE_ITER + len(NUM_ITERS) * TE_EPI + N_G * TE_GNN


def build_code():
    import fbgnn as F
    return F.create_QC_GHP_codes(127, np.array([[0, -1, 51, 52, -1], [-1, 0, -1, 111, 20], [0, -1, 98, -1, 122],
                                                [0, 80, -1, 119, -1], [-1, 0, 5, -1, 106]]), [0, 1, 7],
                                 name="GHP_n1270_k28")


def build_model(code, seed=2, first_frame=0, gemm="fma"):
    import fbgnn as F
    G = F.Feedback_GNN(code=code, num_msg_dims=20, num_hidden_units=40, num_mlp_layers=2, reduce_op="mean",
                       activation="tanh", use_bias=True, gemm=gemm)
    F.load_weights(G, os.path.join(F.WEIGHTS_DIR, WEIGHTS))
    d1 = F.QLDPCBPDecoder(code=code, num_iter=64, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    d2 = F.QLDPCBPDecoder(code=code, num_iter=16, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
    return F.Sandwich_BP_GNN_Evaluation_Model(code, [d1] + [d2] * N_G, [G] * N_G, num_layers=N_G + 1, p0=P0,
                                              seed=seed, first_frame=first_frame)


# ------------------------------------------------------------------ clocks --------------
class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, pw, reasons = [], [], [], set()
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "sm_min_mhz": min(sm) if sm else None, "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ CPU arm -------------
def cpu_reference_run(code, frames, steps=1, warmup=0, seed=2):
    """The CPU restatement of the reference on all host threads; returns (frames/s, threads, ms/step)."""
    from oracle import c_oracle as O
    import fbgnn as F
    g = O.CodeGraph(code)
    G = O.Gnn(F.read_weights(os.path.join(F.WEIGHTS_DIR, WEIGHTS)))
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core
    O.lib().orc_set_num_threads(os.cpu_count() or 1)
    threads = O.num_threads()
    kw = dict(num_iters=NUM_ITERS, gnns=[G] * N_G, p=P_NOISE, p0=P0, seed=seed, skip_inactive=False)
    for i in range(warmup):
        O.pipeline(g, B=max(threads, 8), first_frame=10 ** 9 + i * 1000, **kw)
    t0 = time.perf_counter()
    for i in range(steps):
        O.pipeline(g, B=frames, first_frame=i * frames, **kw)
    dt = time.perf_counter() - t0
    return frames * steps / dt, threads, dt / steps * 1e3


def run_reference_arm(args, rank):
    if rank != 0:
        return
    code = build_code()
    cores = os.cpu_count() or 1
    frames = max(16 * cores, 64)                     # ~2 s of CPU work per step on the GPU box
    fps, threads, ms = cpu_reference_run(code, frames, steps=args.steps, warmup=min(args.warmup, 1))
    line = {"impl": "reference", "metric": "decoded frames/sec (BP->GNN->BP, [[1270,28]])", "value": fps,
            "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": shared_config(args.frames_per_step),
            "note": "CPU restatement of the reference (oracle/fbgnn_oracle.c, exact arithmetic, OpenMP over frames); the "
                    "reference's own TensorFlow path cannot be installed in this image.  Each step is a bounded sample of "
                    f"{frames} frames of the workload in `config`",
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                             "sample": f"{args.steps} x {frames} frames of the same workload"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm -------------
def shared_config(B):
    """The `config` object both arms print (same keys, same values: the workload is the same)."""
    return {"workload": WORKLOAD, "frames_per_step_per_gpu": B, "num_iter": NUM_ITERS, "rounds_of_gnn": N_G,
            "p": P_NOISE, "p0": P0,
            "l2": "per-step working set (~23 KB/frame of HBM state, %d MB) exceeds the 126 MB L2" % (B * 23 // 1000)}


def time_pipeline(ctx, comm, model, B, steps, warmup, allreduce=True, keep_last=False):
    """`steps` passes of the whole pipeline, CUDA events on the context's stream, max over ranks.  One counter
    all-reduce per step sits inside the timed region (the poll of sim_ber's stopping rule, misc.py:710-716).
    With `keep_last` the last step also writes its per-frame outputs (flags, x_diff, z_diff), which only adds
    stores to the final kernel, and returns them as the third value."""
    for _ in range(warmup):
        model.run(B, P_NOISE, want_flags=False, want_diff=False)
    comm.barrier()
    counters = np.zeros(4, np.int64)
    last = None
    ctx.timer_start()
    for i in range(steps):
        want = keep_last and i == steps - 1
        r = model.run(B, P_NOISE, want_flags=want, want_diff=want, want_counters=True)
        counters = counters + (comm.allreduce_sum(r["counters"]) if allreduce else r["counters"])
        if want:
            last = r
    ms = ctx.timer_stop()
    comm.barrier()
    return float(comm.allreduce_f64([ms], "max")[0]), counters, last


DUMP_FRAMES = 4096        # frames of the last step whose residuals are written (x_diff + z_diff: 41.6 MB in float32)


def dump_outputs(path, res, first_frame, B):
    """What the last timed step returned to its caller, as float32 / float64 .npy files: `counters` (frames, flagged,
    block errors, stage-0 failures over the whole step) and, for a fixed seeded sample of its frames, `flags`
    (bit 0 flagged, bit 1 block error, bits 2+ the stages before the last that left the frame active), `x_diff` /
    `z_diff` (residual error: noise XOR correction, one row per frame) and `frames` (their global frame ids, which
    key the in-kernel noise)."""
    os.makedirs(path, exist_ok=True)
    rows = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_FRAMES), replace=False))
    out = {"counters": res["counters"].astype(np.float64),
           "frames": (first_frame + rows).astype(np.float64),
           "flags": res["flags"].numpy()[rows].astype(np.float32),
           "x_diff": res["x_diff"].numpy()[rows].astype(np.float32),
           "z_diff": res["z_diff"].numpy()[rows].astype(np.float32)}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fbgnn", choices=["fbgnn", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=32768, help="frames per step per GPU")
    ap.add_argument("--gnn-gemm", default="tf32x3", choices=["tf32x3", "fma"],
                    help="dense products of the feedback GNN: on the tcgen05 tensor cores (default; three-product TF32 "
                         "split, bit-exact against the oracle's emulation of the tensor-core arithmetic, csrc/fb_umma.h) "
                         "or as FP32 FMAs")
    ap.add_argument("--math", default="sfu", choices=["sfu", "exact"],
                    help="arithmetic of the headline: exp/log on the SFU (default) or as FP32 polynomials; both are "
                         "bit-exact against the CPU oracle in the same arithmetic (csrc/fb_math.h)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline returned (rank 0) to DIR/<name>.npy, so that two "
                         "builds can be compared output for output; the same arguments give the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3
    os.environ.setdefault("FBGNN_DEVICE", str(local_rank))
    import fbgnn as F
    from fbgnn import _ffi
    from fbgnn.distributed import init_from_env
    ctx = F.default_context()
    # one process per GPU; the only collective is the counter all-reduce (NCCL inside libfbgnn.so, on ctx's stream)
    comm = init_from_env(ctx)
    code = build_code()
    B = args.frames_per_step
    per_rank_frames = (args.steps + args.warmup) * B
    model = build_model(code, seed=2, first_frame=rank * per_rank_frames, gemm=args.gnn_gemm)
    other_gemm = "fma" if args.gnn_gemm == "tf32x3" else "tf32x3"
    other = "exact" if args.math == "sfu" else "sfu"

    # ---- headline: device-timed throughput, noise sampled in-kernel, nothing leaves the GPU but the counters
    ctx.set_math(args.math)
    ctx.stats(reset=True)
    sampler = ClockSampler(local_rank)
    for _ in range(args.warmup):
        model.run(B, P_NOISE, want_flags=False, want_diff=False)
    comm.barrier()
    ctx.stats(reset=True)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    dump = args.dump_outputs is not None and rank == 0
    ms, counters, last = time_pipeline(ctx, comm, model, B, args.steps, 0, keep_last=dump)
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    bp_frames, bp_iters = ctx.stats(reset=True)
    value = args.steps * B * world / (ms * 1e-3)
    if dump:
        dump_outputs(args.dump_outputs, last, model.next_frame - B, B)

    # ---- the other arithmetic on the same workload, reported beside the headline
    ctx.set_math(other)
    o_steps = args.steps
    o_ms, o_counters, _ = time_pipeline(ctx, comm, model, B, o_steps, 2)
    o_value = o_steps * B * world / (o_ms * 1e-3)
    ctx.set_math(args.math)

    # ---- the same workload with round skipping (result-identical; what low-p sweeps use)
    model.skip_inactive = True
    s_steps = args.steps
    s_ms, s_counters, _ = time_pipeline(ctx, comm, model, B, s_steps, 2)
    model.skip_inactive = False
    s_value = s_steps * B * world / (s_ms * 1e-3)

    # ---- the same workload with the other evaluation of the feedback GNN's dense products (tensor cores <-> FP32 FMAs)
    tc_model = build_model(code, seed=2, first_frame=rank * per_rank_frames, gemm=other_gemm)
    t_steps = args.steps
    t_ms, t_counters, _ = time_pipeline(ctx, comm, tc_model, B, t_steps, 2)
    t_value = t_steps * B * world / (t_ms * 1e-3)

    # ---- end to end through the public API with HOST buffers: packed noise bit-planes in, packed indicator planes out
    # (32 qubits / 32 frames per word: 10.5 MB in, 12 KB out per step instead of 83 MB / 33 KB as byte arrays)
    host_src = F.Pauli(seed=2, first_frame=10 ** 10 + rank * B).sample_device(B, N_Q, F.pauli_thresholds(P_NOISE))
    nx_host, nz_host = host_src[0].numpy(), host_src[1].numpy()                # synthetic samples, host resident
    wq, fw = F.packed_words(N_Q), (B + 31) // 32
    nx_h = _ffi.PinnedArray((B, wq), np.uint32)
    nz_h = _ffi.PinnedArray((B, wq), np.uint32)
    nx_h.array[:], nz_h.array[:] = F.pack_bits(nx_host), F.pack_bits(nz_host)
    planes_h = _ffi.PinnedArray((3, fw), np.uint32)
    nxb_d, nzb_d = ctx.empty((B, wq), np.uint32), ctx.empty((B, wq), np.uint32)
    nx_d, nz_d = ctx.asarray(nx_host), ctx.asarray(nz_host)                    # byte form, for the roofline probe below
    import ctypes as C

    def e2e_step():
        _ffi.copy_h2d_async(ctx, nxb_d, nx_h.array)
        _ffi.copy_h2d_async(ctx, nzb_d, nz_h.array)
        res = model.run_bits(B, P_NOISE, noise_bits=(nxb_d, nzb_d), want_counters=True)
        _ffi.call("fbgnn_memcpy_d2h", ctx.handle, planes_h.array.ctypes.data_as(C.c_void_p), res["frame_bits"].ptr,
                  planes_h.array.nbytes)
        return int(F.unpack_bits(planes_h.array[1], B).sum()), res["counters"]

    e2e_step()
    comm.barrier()
    t0 = time.perf_counter()
    ctx.timer_start()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        blk, c = e2e_step()
        assert blk == c[2]
    e2e_ms_dev = ctx.timer_stop()
    e2e_wall = time.perf_counter() - t0
    e2e_ms = max(e2e_ms_dev, e2e_wall * 1e3)          # wall clock includes the Python host side
    e2e_ms = float(comm.allreduce_f64([e2e_ms], "max")[0])
    e2e_value = e2e_steps * B * world / (e2e_ms * 1e-3)
    h2d_bytes, d2h_bytes = 2 * B * wq * 4, 3 * fw * 4 + 32

    if rank != 0:
        comm.close()
        return

    # ---- roofline of the dominant kernel (k_bp4, 64 iterations from the constant prior), timed alone
    sfu_peak = ctx.sfu_peak()
    fma_peak = ctx.fma_peak()
    dev = _ffi.device_code(code)
    dec = model.decoders[0]
    sx = ctx.empty((B, dev.mx), np.uint8).T
    sz = ctx.empty((B, dev.mz), np.uint8).T
    gx, gz = _ffi.Graph(code.hx), _ffi.Graph(code.hz)
    _ffi.call("fbgnn_syndrome", gx.handle, B, nz_d.t2(), sx.t2())
    _ffi.call("fbgnn_syndrome", gz.handle, B, nx_d.t2(), sz.t2())
    prior = float(model.prior(P_NOISE))
    for _ in range(2):
        dec.decode_device(None, sx, sz, want_logits=True, prior=prior)
    ctx.sync()
    ctx.stats(reset=True)
    reps = 3
    kt = 0.0
    for _ in range(reps):
        ctx.flush_l2()
        ctx.sync()
        ctx.timer_start()
        dec.decode_device(None, sx, sz, want_logits=True, prior=prior)
        kt += ctx.timer_stop()
    k_ms = kt / reps
    k_frames, k_iters = ctx.stats(reset=True)
    te_launch = B * (64 * TE_ITER + TE_EPI)                       # algorithmic: every frame, every iteration
    te_executed = k_iters / reps * TE_ITER + B * TE_EPI           # the iterations the kernel actually ran
    achieved = te_launch / (k_ms * 1e-3)
    prof = _profile_summary(args.math, B)
    roofline = {"bound": "sfu", "kernel": "k_bp4<const prior, fixed-point exit>, 64 iterations, arithmetic " + args.math,
                "achieved": achieved / 1e9, "peak": sfu_peak / 1e9, "unit": "G transcendental evals/s",
                "frac": achieved / sfu_peak,
                "frac_note": "ALGORITHMIC transcendental evaluations of the reference formulas (SURVEY.md 8(d): 52n per "
                             "iteration, all 64 iterations of every frame) / launch time / MUFU peak.  It can exceed 1: the "
                             "fixed-point exit proves part of the iterations redundant and the SFU arithmetic shares one "
                             "exp between the two terms of phi, so the kernel needs fewer MUFU instructions than the "
                             "reference formulas have transcendentals.  What bounds the executed work is instruction "
                             "issue: see executed_frac, issue_frac and profile.*_pipe_pct",
                "peak_source": "measured live: ex2.approx micro-benchmark (fbgnn_sfu_peak); SURVEY.md 8(d) names the SFU "
                               "as the bound of this path, MEASURED_PEAKS.json holds only HBM / bf16 figures",
                "units_per_launch": B, "te_per_unit": 64 * TE_ITER + TE_EPI, "launch_ms": k_ms,
                "executed_iterations_per_frame": k_iters / max(k_frames, 1),
                "executed_frac": te_executed / (k_ms * 1e-3) / sfu_peak,
                "executed_note": "TE of the iterations actually run (the fixed-point exit leaves the loop once an iteration "
                                 "reproduces every message bit for bit) / MUFU peak; inside an iteration warps whose lanes "
                                 "are all saturated skip evaluations as well -- the MUFU pipe utilisation ncu measured for "
                                 "this launch is `profile.xu_pipe_pct`",
                "fp32_issue_peak_ginstr_s": fma_peak / 1e9,
                "whole_step_frac": value * TE_PER_FRAME / (sfu_peak * world),
                "whole_step_executed_iterations_per_frame": bp_iters / max(bp_frames, 1) * (1 + N_G),
                "hbm_peak_gbs": _measured_peaks().get("hbm_gbs"),
                "traffic": prof.get("dram_bytes") if prof else None,
                "profile": prof}
    if prof and prof.get("dram_bytes") and _measured_peaks().get("hbm_gbs"):
        roofline["hbm_achieved_gbs"] = prof["dram_bytes"] / (k_ms * 1e-3) / 1e9
        roofline["hbm_frac"] = roofline["hbm_achieved_gbs"] / _measured_peaks()["hbm_gbs"]
    if prof and prof.get("thread_inst"):
        roofline["issue_frac"] = prof["thread_inst"] / (k_ms * 1e-3) / fma_peak
        roofline["issue_note"] = ("thread-instructions of this launch (ncu, profiles/) / live launch time / measured FP32 "
                                  "issue peak")

    cpu_baseline = None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        frames = max(96 * cores, 256)                # ~10-20 s of CPU work
        fps, threads, _ = cpu_reference_run(code, frames, steps=1, warmup=1)
        cpu_baseline = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                        "sample": f"{frames} frames of the same workload (oracle/fbgnn_oracle.c, exact arithmetic, "
                                  f"OpenMP over frames)",
                        "numpy_oracle": numpy_reference_run(code)}

    line = {"metric": "decoded frames/sec (BP->GNN->BP, [[1270,28]])", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": shared_config(B),
            "arithmetic": {"mode": args.math,
                           "note": "float32 throughout; 'sfu' evaluates exp/log on MUFU.EX2/LG2 (2-3 ulp), 'exact' as FP32 "
                                   "polynomials (1 ulp).  Both are bit-exact against the CPU oracle in the same arithmetic "
                                   "and reproduce the published error rates (tests/test_gpu_sfu.py, test_gpu_fullsize.py)",
                           other: {"value": o_value, "unit": "frames/s", "steps": o_steps,
                                   "block_errors": int(o_counters[2]), "frames": int(o_counters[0])}},
            "counters": {"frames": int(counters[0]), "flagged": int(counters[1]),
                         "block_errors": int(counters[2]), "stage0_failures": int(counters[3])},
            "collectives_in_timed_region": args.steps if world > 1 else 0,
            "context": {"published_rtx4090_tf_xla_frames_per_s": 6389},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": d2h_bytes, "steps": e2e_steps,
                    "path": "Sandwich_BP_GNN_Evaluation_Model.run_bits(noise_bits=host bit-planes) -> indicator planes + "
                            "counters on host (fbgnn_pipeline_run_bits)"},
            "gpu_launches": int(launches),
            "skip_inactive": {"value": s_value, "unit": "frames/s", "steps": s_steps,
                              "block_errors": int(s_counters[2]), "frames": int(s_counters[0]),
                              "note": "frames whose correction already matches the syndrome skip the remaining "
                                      "GNN/BP rounds: bit-identical results (the reference masks those updates, "
                                      "feedback_gnn.py:339-340) but less work than the reference executes, so it "
                                      "is reported beside the headline, not as the headline"},
            "gnn_gemm": {"mode": args.gnn_gemm,
                         "note": "tf32x3: the three dense products of the feedback GNN's node update on the tcgen05 tensor "
                                 "cores (csrc/fbgnn_gnn_tc.cuh, operands in TMEM, three-product TF32 split).  The arithmetic "
                                 "of a tcgen05.mma step is an integer model characterised on B200 (csrc/fb_umma.h), so this "
                                 "form is bit-exact against the CPU oracle as well (tests/test_gpu_gnn_tc.py); its outputs "
                                 "are within 5e-7 of the FMA form.  fma: FP32 FMAs in the oracle's order",
                         other_gemm: {"value": t_value, "unit": "frames/s", "steps": t_steps,
                                      "block_errors": int(t_counters[2]), "frames": int(t_counters[0])}},
            "roofline": roofline,
            "cpu_baseline": cpu_baseline}
    print(json.dumps(line), flush=True)
    comm.close()


def numpy_reference_run(code, frames=24):
    """The independent numpy restatement (oracle/np_oracle.py) on the same workload: a second CPU figure
    (BASELINE.md 2.2), single-threaded elementwise numpy."""
    from oracle import c_oracle as O
    from oracle import np_oracle as N
    import fbgnn as F
    w = F.read_weights(os.path.join(F.WEIGHTS_DIR, WEIGHTS))
    nx, nz = O.pauli(2, 0, frames, code.N, P_NOISE)
    X, Z = N.Side(code.hx), N.Side(code.hz)
    t0 = time.perf_counter()
    N.pipeline(code, X, Z, NUM_ITERS, [w] * N_G, nx, nz, O.prior_llr(P0))
    dt = time.perf_counter() - t0
    return {"value": frames / dt, "unit": "frames/s", "sample": f"{frames} frames, one process"}


def _profile_summary(math_mode, B):
    """Per-launch ncu figures of the dominant kernel from the committed capture of this round (same B, same arithmetic),
    written by tools/ncu_to_json.py; None when there is no matching capture."""
    path = os.path.join(ROOT, "profiles", f"r02_ncu_k_bp4_stage0_{math_mode}.json")
    try:
        with open(path) as f:
            p = json.load(f)
    except Exception:
        return None
    if p.get("frames") != B:
        return None
    p["source"] = os.path.relpath(path, ROOT)
    return p


def _measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


if __name__ == "__main__":
    main()
