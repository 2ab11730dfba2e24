"""Per-array error of the CUDA training gradient (fbgnn_second_stage_grad) over the case matrix of
tests/test_train_grad.py, against the float64 autograd reference with the smooth phi and with the library's phi
("specified"), beside the noise floor of a float32 evaluation of the same reference (torch float32 vs float64).

    python tools/grad_error_report.py [--out profiles/grad_error_b200.txt]

Columns per array: ||g - ref|| / ||ref||  and  max|g - ref| / max|ref|.  Needs a CUDA device (the library) and torch
(the reference).  The tolerances of tests/test_train_grad.py cite this report's B200 output."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "feedback-gnn_b200"), ROOT):
    sys.path.insert(0, p)

import numpy as np
import torch

import fbgnn as F
from oracle import c_oracle as O, torch_grad_oracle as TG
import test_train_grad as T


def codes():
    c = {"rsurf3": F.create_rotated_surface_codes(3), "toric4": F.create_checkerboard_toric_codes(4),
         "gb48": F.create_generalized_bicycle_codes(24, [0, 2, 8, 15], [0, 2, 12, 17], name="GB_n48_k6_d8"),
         "c882": F.create_QC_GHP_codes(63, F.create_cyclic_permuting_matrix(7, [27, 54, 0]), [0, 1, 6])}
    c1270 = F.create_QC_GHP_codes(127, np.array([[0, -1, 51, 52, -1], [-1, 0, -1, 111, 20], [0, -1, 98, -1, 122],
                                                 [0, 80, -1, 119, -1], [-1, 0, 5, -1, 106]]), [0, 1, 7], name="GHP_n1270_k28")
    return c, c1270


def fmt(errs):
    return "  ".join("%8.1e %8.1e" % e for e in errs)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    O.build()
    cs, c1270 = codes()
    d = F.WEIGHTS_DIR
    weights = {"c882": F.read_weights(os.path.join(d, "feedback_GNN_n882_k24_wt_4_60_iter_64_16_mixed.npy")),
               "c1270": F.read_weights(os.path.join(d, "feedback_GNN_n1270_k28_wt_10_80_iter_64_16_mixed.npy"))}
    ctx = F.default_context()
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                 # the report still stands without it; say so
        smi = f"nvidia-smi unavailable ({e})"
    lines = [f"# tools/grad_error_report.py -- {ctx.name}; name, power limit, max SM clock: {smi}",
             "# per array: ||g - ref|| / ||ref||  max|g - ref| / max|ref|",
             "#   cuda-smooth: CUDA vs float64 reference (smooth phi); cuda-spec: vs float64 reference (library phi);",
             "#   f32-floor: torch float32 vs float64, smooth phi (the float32 noise floor of the same computation)"]
    print("\n".join(lines), flush=True)
    cases = [(name, case, "fma") for name, case in T.UNCONVERGED.items()]
    cases += [("c882_B37_T6_lf0_tf32x3", T.UNCONVERGED["c882_B37_T6_lf0"], "tf32x3"), ("converged", T.CONVERGED, "fma")]
    summary = []
    for name, case, gemm in cases:
        t0 = time.time()
        code, w, loss, g, inputs = T.run_named_case(O, cs, c1270, weights, case, gemm=gemm)
        Tn, lf, reduce, factor = case[6:]
        l64, r64 = T.reference(code, w, inputs, Tn, lf, reduce, factor)
        lsp, rsp = T.reference(code, w, inputs, Tn, lf, reduce, factor, phi="specified")
        l32, r32 = T.reference(code, w, inputs, Tn, lf, reduce, factor, dtype=torch.float32)
        e64, esp, e32 = T.rel_errors(g, r64), T.rel_errors(g, rsp), T.rel_errors(r32, r64)
        out = [f"{name}  gemm={gemm} (code {case[0]}, B {case[2]}, p {case[3]}, stage one {case[5]}, num_iter {Tn}, "
               f"loss_from {lf}, {reduce}, factor {factor}; {time.time() - t0:.1f} s)",
               "  loss cuda %.9e  smooth %.9e (rel %.1e)  spec %.9e (rel %.1e)  f32 %.9e (rel %.1e)" % (
                   loss, l64, abs(loss - l64) / l64, lsp, abs(loss - lsp) / lsp, l32, abs(l32 - l64) / l64),
               "  %-4s %17s  %17s  %17s" % ("", "cuda-smooth", "cuda-spec", "f32-floor")]
        for nm, a, b, c in zip(TG.NAMES, e64, esp, e32):
            out.append("  %-4s %s    %s    %s" % (nm, fmt([a]), fmt([b]), fmt([c])))
        summary.append("%-26s worst cuda-smooth %.1e  cuda-spec %.1e  f32-floor %.1e  loss rel %.1e / %.1e" % (
            name, T.worst(e64), T.worst(esp), T.worst(e32), abs(loss - l64) / l64, abs(loss - lsp) / lsp))
        print("\n".join(out), flush=True)
        lines += out
    lines += ["# summary"] + summary
    print("# summary\n" + "\n".join(summary))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
