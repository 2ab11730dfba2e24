"""ctypes binding of libfbgnn.so (include/fbgnn.h) and the device-array type the layers exchange.

There is no CPU fallback: if the shared library is missing, or there is no CUDA device, the
first call that needs it raises ``FbgnnError`` -- the package never computes on the host.

``DeviceArray`` is a minimal strided view of device memory.  It speaks DLPack in both
directions (``__dlpack__`` / ``__dlpack_device__`` for export, ``from_dlpack`` for import), so
tensors are exchanged zero-copy with any DLPack-aware library (CuPy, PyTorch, JAX, TF's
``tf.experimental.dlpack``); ``numpy()`` copies to the host.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("FBGNN_LIB", os.path.join(_HERE, "libfbgnn.so"))
_lib = None


class FbgnnError(RuntimeError):
    pass


class Tensor2(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("s0", C.c_int64), ("s1", C.c_int64)]


class Tensor3(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("s0", C.c_int64), ("s1", C.c_int64), ("s2", C.c_int64)]


class PipelineCfg(C.Structure):
    _fields_ = [("num_stages", C.c_int32), ("num_iter", C.POINTER(C.c_int32)),
                ("factor", C.POINTER(C.c_float)), ("cn_type", C.POINTER(C.c_int32)),
                ("gnn", C.POINTER(C.c_void_p)), ("prior", C.c_float), ("thr", C.c_float * 3),
                ("fixed_weight", C.c_int32), ("osd0", C.c_int32), ("skip_inactive", C.c_int32),
                ("early_stop", C.c_int32), ("osd_order", C.c_int32), ("lsd", C.c_int32),
                ("lsd_max_cols", C.c_int32), ("lsd_max_checks", C.c_int32)]


class Bp4Opts(C.Structure):
    _fields_ = [("iters_out", C.c_void_p), ("rows_x", C.c_void_p), ("rows_z", C.c_void_p)]


NULL2 = Tensor2(None, 0, 0)
NULL3 = Tensor3(None, 0, 0, 0)

_i32p = C.POINTER(C.c_int32)
_f32p = C.POINTER(C.c_float)
_vpp = C.POINTER(C.c_void_p)

# name -> (argtypes); every function returns int
_SIGNATURES = {
    "fbgnn_device_count": [C.POINTER(C.c_int)],
    "fbgnn_ctx_create": [C.c_int, _vpp],
    "fbgnn_ctx_destroy": [C.c_void_p],
    "fbgnn_ctx_sync": [C.c_void_p],
    "fbgnn_ctx_device": [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_int],
    "fbgnn_timer_start": [C.c_void_p],
    "fbgnn_timer_stop": [C.c_void_p, C.POINTER(C.c_float)],
    "fbgnn_launch_count": [C.c_void_p, C.POINTER(C.c_int64)],
    "fbgnn_ctx_stats": [C.c_void_p, C.POINTER(C.c_int64), C.c_int32],
    "fbgnn_ctx_set_math": [C.c_void_p, C.c_int32],
    "fbgnn_ctx_get_math": [C.c_void_p, C.POINTER(C.c_int32)],
    "fbgnn_malloc": [C.c_void_p, C.c_size_t, _vpp],
    "fbgnn_free": [C.c_void_p, C.c_void_p],
    "fbgnn_memset": [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t],
    "fbgnn_memcpy_h2d": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t],
    "fbgnn_memcpy_d2h": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t],
    "fbgnn_memcpy_d2d": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t],
    "fbgnn_host_alloc": [C.c_size_t, _vpp],
    "fbgnn_host_free": [C.c_void_p],
    "fbgnn_flush_l2": [C.c_void_p],
    "fbgnn_graph_create": [C.c_void_p, C.c_int32, C.c_int32, _i32p, _i32p, _vpp],
    "fbgnn_graph_destroy": [C.c_void_p],
    "fbgnn_code_create": [C.c_void_p, C.c_int32, C.c_int32, _i32p, _i32p, C.c_int32, _i32p, _i32p,
                          C.c_int32, _i32p, _i32p, C.c_int32, _i32p, _i32p, _vpp],
    "fbgnn_code_destroy": [C.c_void_p],
    "fbgnn_code_edges": [C.c_void_p, _i32p, _i32p],
    "fbgnn_code_set_basis": [C.c_void_p, C.c_int32, _i32p, C.c_int32, _i32p],
    "fbgnn_pauli_sample": [C.c_void_p, C.c_int32, C.c_int64, _f32p, C.c_uint64, C.c_uint64, Tensor2, Tensor2],
    "fbgnn_pauli_sample_wt": [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64, Tensor2, Tensor2],
    "fbgnn_bsc_sample": [C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint64, C.c_uint64, Tensor2],
    "fbgnn_syndrome": [C.c_void_p, C.c_int64, Tensor2, Tensor2],
    "fbgnn_bp4_decode": [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int64, Tensor3, C.c_float,
                         Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2,
                         Tensor2, Tensor2, Tensor3],
    "fbgnn_bp4_decode_ex": [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int64, Tensor3, C.c_float,
                            Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2, Tensor2,
                            Tensor2, Tensor2, Tensor3, C.POINTER(Bp4Opts)],
    "fbgnn_rows_create": [C.c_void_p, C.c_int32, C.c_int32, _i32p, _i32p, _vpp],
    "fbgnn_rows_destroy": [C.c_void_p],
    "fbgnn_bp2_decode": [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int64, Tensor2, Tensor2, Tensor2,
                         Tensor2],
    "fbgnn_bp2_decode_ex": [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int64, Tensor2, Tensor2, Tensor2,
                            Tensor2, C.c_void_p, Tensor2, Tensor2],
    "fbgnn_osd0_decode": [C.c_void_p, C.c_int64, Tensor2, Tensor2, Tensor2],
    "fbgnn_osd_decode": [C.c_void_p, C.c_int32, C.c_int64, Tensor2, Tensor2, Tensor2],
    "fbgnn_lsd_decode": [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, Tensor2, Tensor2, Tensor2, C.c_void_p],
    "fbgnn_gnn_create": [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32] + [_f32p] * 12 + [_vpp],
    "fbgnn_gnn_create_deep": [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _f32p,
                              C.c_int64, _vpp],
    "fbgnn_gnn_destroy": [C.c_void_p],
    "fbgnn_gnn_forward": [C.c_void_p, C.c_void_p, C.c_int64, Tensor3, Tensor2, Tensor2, Tensor2, Tensor2,
                          Tensor3],
    "fbgnn_gbp_create": [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_f32p), _vpp],
    "fbgnn_gbp_destroy": [C.c_void_p],
    "fbgnn_gbp_set_gemm": [C.c_void_p, C.c_int32],
    "fbgnn_gnn_set_gemm": [C.c_void_p, C.c_int32],
    "fbgnn_umma_probe": [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32],
    "fbgnn_gbp_set_chunk": [C.c_void_p, C.c_int64],
    "fbgnn_second_stage_grad": [C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_int32, C.c_int64, Tensor3, Tensor2,
                                Tensor2, Tensor2, Tensor2, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_float)],
    "fbgnn_gbp_decode": [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, Tensor2, Tensor2, Tensor3, Tensor3, Tensor2,
                         Tensor2],
    "fbgnn_pipeline_run": [C.c_void_p, C.POINTER(PipelineCfg), C.c_uint64, C.c_uint64, C.c_int64, Tensor2,
                           Tensor2, C.c_void_p, Tensor2, Tensor2, C.POINTER(C.c_int64)],
    "fbgnn_pipeline_run_bits": [C.c_void_p, C.POINTER(PipelineCfg), C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)],
    "fbgnn_bsc_pipeline_run": [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float,
                               C.c_uint64, C.c_uint64, C.c_int64, Tensor2, C.c_void_p, C.POINTER(C.c_int64),
                               C.c_void_p, _i32p],
    "fbgnn_bsc_pipeline_run_ex": [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float,
                                  C.c_uint64, C.c_uint64, C.c_int64, Tensor2, C.c_void_p, C.POINTER(C.c_int64),
                                  C.c_void_p, _i32p, C.c_int32],
    "fbgnn_bsc_pipeline_run_lsd": [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float,
                                   C.c_uint64, C.c_uint64, C.c_int64, Tensor2, C.c_void_p, C.POINTER(C.c_int64),
                                   C.c_int32, C.c_int32],
    "fbgnn_comm_unique_id": [C.POINTER(C.c_uint8)],
    "fbgnn_comm_init_rank": [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_uint8)],
    "fbgnn_comm_info": [C.c_void_p, _i32p, _i32p, _i32p],
    "fbgnn_allreduce_counters": [C.c_void_p, C.POINTER(C.c_int64), C.c_int32],
    "fbgnn_allreduce_f64": [C.c_void_p, C.POINTER(C.c_double), C.c_int32, C.c_int32],
    "fbgnn_comm_barrier": [C.c_void_p],
    "fbgnn_comm_destroy": [C.c_void_p],
    "fbgnn_sfu_peak": [C.c_void_p, C.POINTER(C.c_double)],
    "fbgnn_fma_peak": [C.c_void_p, C.POINTER(C.c_double)],
    "fbgnn_math_probe": [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int64],
}

EXPORTED_SYMBOLS = ["fbgnn_version", "fbgnn_last_error"] + list(_SIGNATURES)


def lib():
    """Load libfbgnn.so (once).  Raises FbgnnError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise FbgnnError(f"{_LIB_PATH} not found: build it with `make -C feedback-gnn_b200/csrc` "
                             f"(or __graft_entry__.build()); fbgnn has no CPU fallback")
        L = C.CDLL(_LIB_PATH)
        L.fbgnn_version.restype = C.c_int
        L.fbgnn_last_error.restype = C.c_char_p
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = C.c_int
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise FbgnnError(f"fbgnn error {rc}: {lib().fbgnn_last_error().decode()}")


def call(name, *args):
    check(getattr(lib(), name)(*args))


# ----------------------------------------------------------------------------- context --
class Context:
    """One GPU (stream + scratch).  ``default_context()`` returns a per-process singleton for
    the device given by FBGNN_DEVICE / LOCAL_RANK (default 0)."""

    def __init__(self, device=0):
        self.handle = C.c_void_p()
        call("fbgnn_ctx_create", int(device), C.byref(self.handle))
        dev, sms = C.c_int(), C.c_int()
        name = C.create_string_buffer(256)
        call("fbgnn_ctx_device", self.handle, C.byref(dev), C.byref(sms), name, 256)
        self.device, self.num_sms, self.name = dev.value, sms.value, name.value.decode()

    def sync(self):
        call("fbgnn_ctx_sync", self.handle)

    def set_math(self, mode):
        """Arithmetic of the decoders launched from now on: "exact" (exp / log as polynomials on the FP32 pipe) or
        "sfu" (exp / log on the special-function unit; "fast" is the former name).  Both are bit-identical to the CPU
        oracle in the same arithmetic (csrc/fb_math.h)."""
        call("fbgnn_ctx_set_math", self.handle, {"exact": 0, "sfu": 1, "fast": 1}[mode])

    def get_math(self):
        m = C.c_int32()
        call("fbgnn_ctx_get_math", self.handle, C.byref(m))
        return ["exact", "sfu"][m.value]

    def timer_start(self):
        call("fbgnn_timer_start", self.handle)

    def timer_stop(self):
        ms = C.c_float()
        call("fbgnn_timer_stop", self.handle, C.byref(ms))
        return ms.value

    def launch_count(self):
        v = C.c_int64()
        call("fbgnn_launch_count", self.handle, C.byref(v))
        return v.value

    def stats(self, reset=False):
        """(frames decoded, BP iterations executed) by the quaternary BP kernels since the last reset; the first call
        switches the counting on."""
        v = (C.c_int64 * 2)()
        call("fbgnn_ctx_stats", self.handle, v, 1 if reset else 0)
        return int(v[0]), int(v[1])

    def flush_l2(self):
        call("fbgnn_flush_l2", self.handle)

    def sfu_peak(self):
        v = C.c_double()
        call("fbgnn_sfu_peak", self.handle, C.byref(v))
        return v.value

    def fma_peak(self):
        v = C.c_double()
        call("fbgnn_fma_peak", self.handle, C.byref(v))
        return v.value

    # allocation helpers
    def empty(self, shape, dtype):
        return DeviceArray.empty(self, shape, dtype)

    def zeros(self, shape, dtype):
        a = DeviceArray.empty(self, shape, dtype)
        call("fbgnn_memset", self.handle, a.ptr, 0, a.nbytes)
        return a

    def asarray(self, x, dtype=None):
        """Host array / DLPack object / DeviceArray -> DeviceArray on this context."""
        if isinstance(x, DeviceArray):
            if dtype is not None and x.dtype != np.dtype(dtype):
                raise FbgnnError(f"device tensor has dtype {x.dtype}, expected {np.dtype(dtype)}")
            return x
        if not isinstance(x, np.ndarray) and hasattr(x, "__dlpack__") and hasattr(x, "__dlpack_device__"):
            if x.__dlpack_device__()[0] in (2, 3, 13):      # kDLCUDA, kDLCUDAHost, kDLCUDAManaged
                a = DeviceArray.from_dlpack(self, x)
                if dtype is not None and a.dtype != np.dtype(dtype):
                    raise FbgnnError(f"device tensor has dtype {a.dtype}, expected {np.dtype(dtype)}")
                return a
        h = np.ascontiguousarray(np.asarray(x), dtype=dtype)
        a = DeviceArray.empty(self, h.shape, h.dtype)
        if h.nbytes:
            call("fbgnn_memcpy_h2d", self.handle, a.ptr, h.ctypes.data_as(C.c_void_p), h.nbytes)
            self.sync()                                    # h may be a temporary
        return a

    def edge_vn(self):
        """Variable node of every edge, edges sorted by (variable, check) -- the order of the message vectors."""
        return self._vn_of_edge

    def __del__(self):
        try:
            if self.handle:
                lib().fbgnn_ctx_destroy(self.handle)
        except Exception:
            pass


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        dev = int(os.environ.get("FBGNN_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        _default_ctx = Context(dev)
        if os.environ.get("FBGNN_MATH", "exact") != "exact":
            _default_ctx.set_math(os.environ["FBGNN_MATH"])
    return _default_ctx


def device_count():
    n = C.c_int()
    call("fbgnn_device_count", C.byref(n))
    return n.value


# ----------------------------------------------------------------------------- DLPack ---
class _DLDevice(C.Structure):
    _fields_ = [("device_type", C.c_int32), ("device_id", C.c_int32)]


class _DLDataType(C.Structure):
    _fields_ = [("code", C.c_uint8), ("bits", C.c_uint8), ("lanes", C.c_uint16)]


class _DLTensor(C.Structure):
    _fields_ = [("data", C.c_void_p), ("device", _DLDevice), ("ndim", C.c_int32), ("dtype", _DLDataType),
                ("shape", C.POINTER(C.c_int64)), ("strides", C.POINTER(C.c_int64)), ("byte_offset", C.c_uint64)]


class _DLManagedTensor(C.Structure):
    pass


_DLDeleter = C.CFUNCTYPE(None, C.POINTER(_DLManagedTensor))
_DLManagedTensor._fields_ = [("dl_tensor", _DLTensor), ("manager_ctx", C.c_void_p), ("deleter", _DLDeleter)]

_DL_CODES = {"i": 0, "u": 1, "f": 2, "b": 6}
_DL_CODES_INV = {0: "i", 1: "u", 2: "f", 6: "b"}
_live_exports = {}          # id -> (managed tensor, owner, shape/stride arrays) kept alive until the deleter runs

C.pythonapi.PyCapsule_New.restype = C.py_object
C.pythonapi.PyCapsule_New.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]
C.pythonapi.PyCapsule_GetPointer.restype = C.c_void_p
C.pythonapi.PyCapsule_GetPointer.argtypes = [C.py_object, C.c_char_p]
C.pythonapi.PyCapsule_SetName.argtypes = [C.py_object, C.c_char_p]
C.pythonapi.PyCapsule_IsValid.argtypes = [C.py_object, C.c_char_p]


@_DLDeleter
def _dl_deleter(mt_ptr):
    _live_exports.pop(C.addressof(mt_ptr.contents), None)


class _Owner:
    """Owns one device allocation."""

    def __init__(self, ctx, ptr):
        self.ctx, self.ptr = ctx, ptr

    def __del__(self):
        try:
            if self.ptr:
                lib().fbgnn_free(self.ctx.handle, self.ptr)
        except Exception:
            pass


class DeviceArray:
    """Strided view of device memory (element strides)."""

    def __init__(self, ctx, owner, ptr, shape, strides, dtype):
        self.ctx, self._owner, self.ptr = ctx, owner, ptr
        self.shape, self.strides, self.dtype = tuple(int(s) for s in shape), tuple(int(s) for s in strides), np.dtype(dtype)

    @staticmethod
    def empty(ctx, shape, dtype):
        shape = tuple(int(s) for s in (shape if hasattr(shape, "__len__") else (shape,)))
        dtype = np.dtype(dtype)
        count = int(np.prod(shape)) if len(shape) else 1
        p = C.c_void_p()
        call("fbgnn_malloc", ctx.handle, max(count * dtype.itemsize, 1), C.byref(p))
        strides, acc = [], 1
        for s in reversed(shape):
            strides.append(acc)
            acc *= max(s, 1)
        return DeviceArray(ctx, _Owner(ctx, p.value), p.value, shape, tuple(reversed(strides)), dtype)

    # -- structure -----------------------------------------------------------------------
    @property
    def ndim(self):
        return len(self.shape)

    @property
    def size(self):
        return int(np.prod(self.shape)) if self.shape else 1

    @property
    def nbytes(self):
        return self.size * self.dtype.itemsize

    @property
    def T(self):
        return self.transpose(tuple(reversed(range(self.ndim))))

    def transpose(self, axes):
        return DeviceArray(self.ctx, self._owner, self.ptr, [self.shape[a] for a in axes],
                           [self.strides[a] for a in axes], self.dtype)

    def is_contiguous(self):
        acc = 1
        for s, st in zip(reversed(self.shape), reversed(self.strides)):
            if s != 1 and st != acc:
                return False
            acc *= s
        return True

    def __getitem__(self, idx):
        """Basic slicing along the leading axis only (enough for batching)."""
        if isinstance(idx, slice):
            start, stop, step = idx.indices(self.shape[0])
            if step != 1:
                raise FbgnnError("only unit-step slices are supported")
            n = max(stop - start, 0)
            return DeviceArray(self.ctx, self._owner, self.ptr + start * self.strides[0] * self.dtype.itemsize,
                               (n,) + self.shape[1:], self.strides, self.dtype)
        raise FbgnnError("unsupported index")

    def t2(self):
        assert self.ndim == 2
        t = Tensor2(self.ptr, self.strides[0], self.strides[1])
        t._keep = self          # the view keeps its allocation alive (frees are stream-ordered)
        return t

    def t3(self):
        assert self.ndim == 3
        t = Tensor3(self.ptr, self.strides[0], self.strides[1], self.strides[2])
        t._keep = self
        return t

    # -- host transfer -------------------------------------------------------------------
    def numpy(self):
        """Copy to a host ndarray of the same logical shape."""
        if self.size == 0:
            return np.empty(self.shape, self.dtype)
        order = sorted(range(self.ndim), key=lambda a: -self.strides[a])
        base = self.transpose(order)
        if not base.is_contiguous():
            raise FbgnnError("numpy() needs a view that is a permutation of a contiguous array")
        h = np.empty(base.shape, self.dtype)
        call("fbgnn_memcpy_d2h", self.ctx.handle, h.ctypes.data_as(C.c_void_p), self.ptr, h.nbytes)
        inv = np.argsort(order)
        return h.transpose(inv)

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a if dtype is None else a.astype(dtype)

    # -- DLPack ---------------------------------------------------------------------------
    def __dlpack_device__(self):
        return (2, self.ctx.device)                        # kDLCUDA

    def __dlpack__(self, stream=None, **kwargs):
        self.ctx.sync()
        nd = self.ndim
        shape = (C.c_int64 * max(nd, 1))(*self.shape)
        strides = (C.c_int64 * max(nd, 1))(*self.strides)
        mt = _DLManagedTensor()
        mt.dl_tensor.data = self.ptr
        mt.dl_tensor.device = _DLDevice(2, self.ctx.device)
        mt.dl_tensor.ndim = nd
        mt.dl_tensor.dtype = _DLDataType(_DL_CODES[self.dtype.kind], self.dtype.itemsize * 8, 1)
        mt.dl_tensor.shape = C.cast(shape, C.POINTER(C.c_int64))
        mt.dl_tensor.strides = C.cast(strides, C.POINTER(C.c_int64))
        mt.dl_tensor.byte_offset = 0
        mt.manager_ctx = None
        mt.deleter = _dl_deleter
        _live_exports[C.addressof(mt)] = (mt, self._owner, shape, strides)
        return C.pythonapi.PyCapsule_New(C.addressof(mt), b"dltensor", None)

    @staticmethod
    def from_dlpack(ctx, obj):
        """Zero-copy import of a CUDA tensor from any object with ``__dlpack__``."""
        cap = obj.__dlpack__()
        if not C.pythonapi.PyCapsule_IsValid(cap, b"dltensor"):
            raise FbgnnError("object did not produce a valid DLPack capsule")
        mt = C.cast(C.pythonapi.PyCapsule_GetPointer(cap, b"dltensor"), C.POINTER(_DLManagedTensor)).contents
        t = mt.dl_tensor
        if t.device.device_type not in (2, 3, 13):
            raise FbgnnError("DLPack tensor is not in CUDA memory")
        if t.device.device_type == 2 and t.device.device_id != ctx.device:
            raise FbgnnError(f"DLPack tensor lives on GPU {t.device.device_id}, context is GPU {ctx.device}")
        if t.dtype.lanes != 1 or t.dtype.code not in _DL_CODES_INV:
            raise FbgnnError("unsupported DLPack dtype")
        kind = _DL_CODES_INV[t.dtype.code]
        dtype = np.dtype(np.bool_) if kind == "b" else np.dtype(f"{kind}{t.dtype.bits // 8}")
        shape = [t.shape[i] for i in range(t.ndim)]
        if t.strides:
            strides = [t.strides[i] for i in range(t.ndim)]
        else:
            strides, acc = [], 1
            for s in reversed(shape):
                strides.insert(0, acc)
                acc *= max(s, 1)
        C.pythonapi.PyCapsule_SetName(cap, b"used_dltensor")

        class _Imported:
            def __init__(self, mt_ptr, keep):
                self.mt_ptr, self.keep = mt_ptr, keep

            def __del__(self):
                try:
                    m = self.mt_ptr.contents
                    if m.deleter:
                        m.deleter(self.mt_ptr)
                except Exception:
                    pass

        owner = _Imported(C.cast(C.addressof(mt), C.POINTER(_DLManagedTensor)), (cap, obj))
        return DeviceArray(ctx, owner, (t.data or 0) + t.byte_offset, shape, strides, dtype)


def from_dlpack(obj, ctx=None):
    return DeviceArray.from_dlpack(ctx or default_context(), obj)


# ----------------------------------------------------------------------------- graphs ---
def _csr(mat):
    """(m, n, indptr, indices) int32 CSR of a dense / scipy-sparse binary matrix."""
    if hasattr(mat, "toarray"):
        mat = mat.toarray()
    mat = np.asarray(mat)
    if mat.ndim != 2:
        raise ValueError("parity-check matrix must be 2-D")
    if mat.size and not np.array_equal(mat, mat.astype(bool)):
        raise AssertionError("PC matrix must be binary.")
    m, n = mat.shape
    r, c = np.nonzero(mat)
    indptr = np.concatenate([[0], np.cumsum(np.bincount(r, minlength=m))]).astype(np.int32)
    return m, n, np.ascontiguousarray(indptr), np.ascontiguousarray(c.astype(np.int32))


def _ip(a):
    return a.ctypes.data_as(_i32p)


class Graph:
    """Device-side Tanner graph of one parity-check matrix (fbgnn_graph)."""

    def __init__(self, pcm, ctx=None):
        self.ctx = ctx or default_context()
        self.m, self.n, indptr, indices = _csr(pcm)
        self.E = int(indptr[-1])
        self._vn_of_edge = np.sort(np.asarray(indices[:self.E], np.int64))
        self.handle = C.c_void_p()
        call("fbgnn_graph_create", self.ctx.handle, self.n, self.m, _ip(indptr), _ip(indices), C.byref(self.handle))

    def edge_vn(self):
        """Variable node of every edge, edges sorted by (variable, check) -- the order of the message vectors."""
        return self._vn_of_edge

    def __del__(self):
        try:
            if self.handle:
                lib().fbgnn_graph_destroy(self.handle)
        except Exception:
            pass


class Rows:
    """Device-side CSR rows of a binary matrix (fbgnn_rows): a row set for soft syndromes."""

    def __init__(self, mat, ctx=None):
        self.ctx = ctx or default_context()
        self.m, self.n, indptr, indices = _csr(mat)
        self.handle = C.c_void_p()
        call("fbgnn_rows_create", self.ctx.handle, self.n, self.m, _ip(indptr), _ip(indices), C.byref(self.handle))

    def __del__(self):
        try:
            if self.handle:
                lib().fbgnn_rows_destroy(self.handle)
        except Exception:
            pass


class Code:
    """Device-side CSS code (fbgnn_code): graphs of hx and hz plus bit-packed logicals."""

    def __init__(self, code, ctx=None):
        self.ctx = ctx or default_context()
        # css_code objects of fbgnn.codes_q carry their CSR; anything else with hx / hz matrices works too
        (mx, n, hxp, hxi), (mz, n2, hzp, hzi) = _csr(code.hx), _csr(code.hz)
        assert n == n2
        lx = np.asarray(code.lx) if np.asarray(code.lx).size else np.zeros((0, n), int)
        lz = np.asarray(code.lz) if np.asarray(code.lz).size else np.zeros((0, n), int)
        kx, _, lxp, lxi = _csr(lx.reshape(-1, n))
        kz, _, lzp, lzi = _csr(lz.reshape(-1, n))
        self.n, self.mx, self.mz, self.Ex, self.Ez = n, mx, mz, int(hxp[-1]), int(hzp[-1])
        self.handle = C.c_void_p()
        call("fbgnn_code_create", self.ctx.handle, n, mx, _ip(hxp), _ip(hxi), mz, _ip(hzp), _ip(hzi),
             kx, _ip(lxp), _ip(lxi), kz, _ip(lzp), _ip(lzi), C.byref(self.handle))
        self.has_basis = False
        if hasattr(code, "pivot_hx") and hasattr(code, "pivot_hz"):
            px = np.ascontiguousarray(code.pivot_hx, np.int32)
            pz = np.ascontiguousarray(code.pivot_hz, np.int32)
            if len(px) and len(pz):
                call("fbgnn_code_set_basis", self.handle, len(px), _ip(px), len(pz), _ip(pz))
                self.has_basis = True

    def __del__(self):
        try:
            if self.handle:
                lib().fbgnn_code_destroy(self.handle)
        except Exception:
            pass


_code_cache = {}


def device_code(code, ctx=None):
    """One device copy per (css_code object, context)."""
    ctx = ctx or default_context()
    key = (id(code), id(ctx))
    ent = _code_cache.get(key)
    if ent is None or ent[0] is not code:
        ent = (code, Code(code, ctx))
        _code_cache[key] = ent
    return ent[1]


# ----------------------------------------------------------------------------- pinned host memory ---
class PinnedArray:
    """numpy view of page-locked host memory (so H2D / D2H copies run at full PCIe rate)."""

    def __init__(self, shape, dtype):
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        self._ptr = C.c_void_p()
        call("fbgnn_host_alloc", max(count * dtype.itemsize, 1), C.byref(self._ptr))
        buf = (C.c_uint8 * max(count * dtype.itemsize, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)

    def __del__(self):
        try:
            if self._ptr:
                self.array = None
                lib().fbgnn_host_free(self._ptr)
        except Exception:
            pass


def copy_h2d_async(ctx, dst, host_array):
    """Enqueue a host->device copy of a C-contiguous host array into a contiguous DeviceArray."""
    assert dst.is_contiguous() and host_array.flags.c_contiguous and dst.nbytes == host_array.nbytes
    call("fbgnn_memcpy_h2d", ctx.handle, dst.ptr, host_array.ctypes.data_as(C.c_void_p), host_array.nbytes)
