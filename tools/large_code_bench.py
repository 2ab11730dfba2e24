"""Timing of the two paths for codes beyond one SM's shared memory ([[7688,50]] HP code): thread-block cluster with
distributed shared memory vs the HBM-state fallback (development aid; profiles/r02_cluster_vs_gstate.txt)."""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "feedback-gnn_b200"))
import numpy as np
import fbgnn as F
from fbgnn import _ffi

h = F.create_circulant_matrix(62, [0, 2, 5])
code = F.hypergraph_product(h, h)
ctx = F.default_context()
B, it = 2048, 32
dec = F.QLDPCBPDecoder(code, num_iter=it, normalization_factor=1.0, cn_type="boxplus-phi", stage_one=True)
dev = dec._device()
nx, nz = F.Pauli(seed=1).sample_device(B, code.N, F.pauli_thresholds(0.04))
gx, gz = _ffi.Graph(code.hx), _ffi.Graph(code.hz)
sx = ctx.empty((B, dev.mx), np.uint8).T
sz = ctx.empty((B, dev.mz), np.uint8).T
_ffi.call("fbgnn_syndrome", gx.handle, B, nz.t2(), sx.t2())
_ffi.call("fbgnn_syndrome", gz.handle, B, nx.t2(), sz.t2())
prior = float(np.log(3 * 0.95 / 0.05))
res = {"code": code.name, "n": code.N, "frames": B, "iterations": it, "device": ctx.name}
for arith in ("exact", "sfu"):
    ctx.set_math(arith)
    for mode in ("cluster", "gstate"):
        os.environ["FBGNN_BP4_LARGE"] = mode
        out = dec.decode_device(None, sx, sz, prior=prior)
        ctx.sync()
        ctx.timer_start()
        for _ in range(3):
            out = dec.decode_device(None, sx, sz, prior=prior)
        ms = ctx.timer_stop() / 3
        res[f"{arith}.{mode}"] = {"ms": round(ms, 3), "frames_per_s": round(B / (ms * 1e-3)), "checksum": int(out[3].numpy().sum())}
print(json.dumps(res))
