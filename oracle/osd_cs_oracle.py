"""ORACLE (test infrastructure only): ctypes front end of ``oracle/osd_cs_oracle.c`` -- ordered-statistics decoding
with the combination sweep of order λ (OSD-CS; λ = 0 is OSD-0) on top of the CPU oracle of ``c_oracle``:

* ``osd(basis, llr, s, order)``            ~ ``fbgnn_osd_decode`` / ``OSD_Decoder(n, osd_order)``
* ``pipeline(..., osd_order=λ)``           ~ ``Sandwich_BP_GNN_Evaluation_Model(..., osd0=True, osd_order=λ)``
* ``bsc_pipeline(..., osd_order=λ)``       ~ ``BP2_OSD_Model`` with ``OSD_Decoder(n, osd_order=λ)``

The library compiles ``fbgnn_oracle.c`` into itself (same flags as ``oracle/Makefile``), so it has its own copy of
the arithmetic selection; every call first mirrors ``c_oracle``'s current one.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import c_oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "osd_cs_oracle.c")
_SO = os.path.join(_HERE, "_build", "libosd_cs_oracle.so")
_DEPS = (_SRC, os.path.join(_HERE, "fbgnn_oracle.c"), os.path.join(_HERE, "..", "feedback-gnn_b200", "csrc", "fb_math.h"))
_CFLAGS = ["-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-Wall", "-Wextra"]
_lib = None


def build(force=False):
    """Compile the library (the oracle's recipe, plus -Bsymbolic so that it never binds to libfbgnn_oracle.so)."""
    stale = not os.path.exists(_SO) or any(os.path.getmtime(f) > os.path.getmtime(_SO) for f in _DEPS)
    if force or stale:
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        tmp = f"{_SO}.{os.getpid()}.tmp"
        subprocess.run(["gcc"] + _CFLAGS + ["-I" + os.path.join(_HERE, "..", "feedback-gnn_b200", "csrc"), "-shared",
                        _SRC, "-o", tmp, "-lm", "-Wl,-Bsymbolic"], check=True)
        os.replace(tmp, _SO)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
    mode = O.get_math()
    if mode == "sfu":
        t = O._sfu_keep
        _lib.orc_set_sfu_tables(O._p(t[0]), O._p(t[1]), O._p(t[2]), O._p(t[3]))
    assert _lib.orc_set_math(1 if mode == "sfu" else 0) == 0
    return _lib


def osd(basis, llr, s, order):
    """OSD of order ``order``: basis [rank,n] full-rank rows, llr [B,n], s [rank,B] -> e_hat [B,n]."""
    R = O.Rows(basis)
    llr = O._f32(llr)
    B, n = llr.shape
    s = O._u8(s)
    assert s.shape == (R.m, B) and order >= 0
    out = np.empty((B, n), np.uint8)
    lib().orc_osd(C.byref(R.c), C.c_int(n), C.c_int(int(order)), C.c_int64(B), O._p(llr), O._p(s), O._p(out))
    return out


def pipeline(g, num_iters, gnns, p, p0=0.05, factors=None, cn_types=None, seed=0, first_frame=0, B=1, noise=None,
             skip_inactive=False, want_diff=False, wt=0, early_stop=False, osd_order=0):
    """``c_oracle.pipeline(..., osd0=True)`` with OSD of order ``osd_order`` after the last stage."""
    S = len(num_iters)
    assert len(gnns) == S - 1
    ni = O._i32(num_iters)
    fa = O._f32([1.0] * S if factors is None else factors)
    ct = O._i32([O.CN_TYPES[c] for c in (cn_types or ["boxplus-phi"] * S)])
    garr = (C.c_void_p * max(S - 1, 1))(*[C.addressof(G.c) for G in gnns])
    code = g.code
    bx, bz = O.Rows(np.asarray(code.hx)[code.pivot_hx]), O.Rows(np.asarray(code.hz)[code.pivot_hz])
    pvx, pvz = O._i32(code.pivot_hx), O._i32(code.pivot_hz)
    cfg = O._PipeCfg(S, O._p(ni), O._p(fa), O._p(ct), C.cast(garr, C.c_void_p),
                     C.c_float(O.prior_llr(p if p0 is None else p0)), int(wt), 1,
                     C.cast(C.pointer(bx.c), C.c_void_p), O._p(pvx), C.cast(C.pointer(bz.c), C.c_void_p), O._p(pvz),
                     int(early_stop), int(skip_inactive))
    thr = O.pauli_thresholds(p)
    flags = np.empty(B, np.uint8)
    counters = np.zeros(4, np.int64)
    nx = nz = None
    if noise is not None:
        nx, nz = O._u8(noise[0]), O._u8(noise[1])
        assert nx.shape == (B, g.n)
    xd = np.empty((B, g.n), np.uint8) if want_diff else None
    zd = np.empty((B, g.n), np.uint8) if want_diff else None
    lib().orc_pipeline_osd(C.byref(g.X.c), C.byref(g.Z.c), C.byref(g.lx.c), C.byref(g.lz.c), C.byref(cfg),
                           C.c_int(int(osd_order)), O._p(thr), C.c_uint64(seed), C.c_uint64(first_frame), C.c_int64(B),
                           O._p(nx), O._p(nz), O._p(flags), O._p(counters), O._p(xd), O._p(zd))
    return dict(flags=flags, counters=counters, x_diff=xd, z_diff=zd)


def bsc_pipeline(pcm, logical_pcm, num_iter, p, osd_basis, osd_pivot, p0=None, factor=1.0, cn_type="boxplus-phi",
                 seed=0, first_frame=0, B=1, noise=None, osd_order=0):
    """``c_oracle.bsc_pipeline(..., osd_basis, osd_pivot)`` with OSD of order ``osd_order``."""
    S = O.Side(pcm)
    L = None if logical_pcm is None else O.Rows(logical_pcm)
    p0 = np.float32(p if p0 is None else p0)
    llr_const = np.float32(-np.log((np.float32(1.0) - p0) / p0))
    flags = np.empty(B, np.uint8)
    counters = np.zeros(4, np.int64)
    nz = None if noise is None else O._u8(noise)
    basis, pivot = O.Rows(osd_basis), O._i32(osd_pivot)
    lib().orc_bsc_pipeline_osd(C.byref(S.c), None if L is None else C.byref(L.c), C.c_int(O.CN_TYPES[cn_type]),
                               C.c_int(num_iter), C.c_float(factor), C.c_float(llr_const), C.c_float(np.float32(p)),
                               C.c_uint64(seed), C.c_uint64(first_frame), C.c_int64(B), O._p(nz), O._p(flags),
                               O._p(counters), C.byref(basis.c), O._p(pivot), C.c_int(int(osd_order)))
    return dict(flags=flags, counters=counters)
