"""Feedback GNN layer and the Monte-Carlo evaluation models built around it.

Mirrors ``sionna/fec/ldpc/feedback_gnn.py`` of the reference:

* ``Feedback_GNN`` (``:20-188``) -- one-shot GNN that turns the marginals and soft syndromes of
  a BP run into new per-qubit priors; ``get_weights`` / ``set_weights`` use the Keras order
  ``[W0, b0, W1_x, b1_x, W2_x, b2_x, W1_z, b1_z, W2_z, b2_z, W3, b3]`` so the shipped
  ``weights/*.npy`` load unchanged (``fbgnn.gnn.load_weights``).
* ``Sandwich_BP_GNN_Evaluation_Model`` (``:232-361``) -- ``model(batch_size, p)`` runs
  sample -> syndrome -> BP -> (GNN -> BP) x nG -> residual-syndrome / logical check and returns
  ``(s_hat, ls_hat)``.  It runs as the fused device pipeline ``fbgnn_pipeline_run``.
* ``BP_BSC_Model`` (``:190-229``) -- the binary counterpart on a BSC.

``s_hat`` / ``ls_hat`` are returned as ``ErrorIndicator`` objects: they carry the per-frame
"any bit set" flags computed on the GPU (all that ``sim_ber`` / ``count_block_errors`` need)
and materialise the reference's dense ``[B, m]`` 0/1 matrices on demand (``numpy()`` /
``np.asarray``) from the residual error kept on the device.
"""
import numpy as np

from . import _ffi
from .decoding_q import QLDPCBPDecoder, CN_TYPES, _is_device, _to_u8
from .decoding import LDPCBPDecoder
from .pauli import Pauli, pauli_thresholds

ACTS = {"tanh": 0, "relu": 1, None: 2, "linear": 2}
REDUCE = {"mean": 0, "sum": 1, "max": 2, "min": 3}


def _glorot_uniform(rng, fan_in, fan_out):
    limit = np.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-limit, limit, size=(fan_in, fan_out)).astype(np.float32)


class Feedback_GNN:
    def __init__(self,
                 code,
                 num_msg_dims,
                 num_hidden_units,
                 num_mlp_layers,
                 reduce_op="mean",
                 activation="tanh",
                 use_bias=False,
                 ctx=None,
                 gemm="fma"):
        """``gemm`` (extension): "fma" (default; bit-exact against the oracle) or "tf32x3" -- the dense products of the
        node update on the tcgen05 tensor cores (csrc/fbgnn_gnn_tc.cuh): within 5e-7 of the FMA form, bit-exact against
        the oracle's emulation of the tensor-core arithmetic (csrc/fb_umma.h); built for the shipped configuration (20 / 40, two layers, tanh, mean or sum, (3,.)-regular codes)."""
        if gemm not in ("fma", "tf32x3"):
            raise ValueError("gemm must be 'fma' or 'tf32x3'")
        self._gemm = gemm
        self._code = code
        self._num_cn_x, self._num_vn = code.hx.shape
        self._num_cn_z = code.hz.shape[0]
        self._num_edges_x = int(np.sum(code.hx))
        self._num_edges_z = int(np.sum(code.hz))
        self._num_msg_dims = int(num_msg_dims)
        self._num_hidden_units = int(num_hidden_units)
        self._num_mlp_layers = int(num_mlp_layers)
        if not 1 <= self._num_mlp_layers <= 8:
            raise ValueError("num_mlp_layers must be in [1, 8]")
        if self._num_mlp_layers != 2 and max(self._num_hidden_units, self._num_msg_dims) > 128:
            raise ValueError("hidden / message dims above 128 are supported for 2-layer MLPs only")
        if reduce_op not in REDUCE:
            raise ValueError("unknown reduce operation")
        if activation not in ACTS:
            raise ValueError(f"unsupported activation {activation!r}")
        self._reduce_op = reduce_op
        self._activation = activation
        self._use_bias = bool(use_bias)
        self._ctx = ctx
        self._weights = None
        self._handles = {}
        self._is_built = False

    # -- Keras-like weight handling --------------------------------------------------------
    def build(self, input_shape=None):
        """Create the variables with the reference's initialisers (feedback_gnn.py:110-128,
        gnn.py:52-58): Dense kernels Glorot-uniform, biases ones, ``_llr_inv_embed`` kernel zeros."""
        if self._is_built:
            return
        self._is_built = True
        H, M, L = self._num_hidden_units, self._num_msg_dims, self._num_mlp_layers
        rng = np.random.default_rng(0)
        ones = lambda k: np.ones(k, np.float32)

        def mlp(k_in, units):                 # gnn.py:46-58: Dense layers, Glorot-uniform kernels, biases of ones
            out = []
            for k_out in units:
                out += [_glorot_uniform(rng, k_in, k_out), ones(k_out)]
                k_in = k_out
            return out
        # _llr_inv_embed acts on the embedding MLP's output -- for L = 1 that MLP is empty and it sees the concatenated
        # input itself; edge MLPs: L-1 hidden layers + a linear output of M; embedding MLP: L-1 hidden layers
        w = [np.zeros((H if L > 1 else 2 * M + 3, 3), np.float32), ones(3)]
        for _ in range(2):
            w += mlp(4, [H] * (L - 1) + [M])
        w += mlp(2 * M + 3, [H] * (L - 1))
        if not self._use_bias:
            w = w[0::2]
        self._weights = w

    def get_weights(self):
        self.build()
        return [a.copy() for a in self._weights]

    def set_weights(self, weights):
        self.build()
        weights = [np.ascontiguousarray(np.asarray(w), dtype=np.float32) for w in weights]
        if len(weights) != len(self._weights):
            raise ValueError(f"You called `set_weights(weights)` with a weight list of length {len(weights)}, "
                             f"but the layer was expecting {len(self._weights)} weights.")
        for new, old in zip(weights, self._weights):
            if new.shape != old.shape:
                raise ValueError(f"Layer weight shape {old.shape} not compatible with provided weight "
                                 f"shape {new.shape}")
        self._weights = weights
        self._drop_handle()

    def count_params(self):
        self.build()
        return int(sum(w.size for w in self._weights))

    def _drop_handle(self):
        for h in getattr(self, "_handles", {}).values():
            try:
                _ffi.lib().fbgnn_gnn_destroy(h[1])
            except Exception:
                pass
        self._handles = {}

    def __del__(self):
        self._drop_handle()

    def device_handle(self, ctx=None):
        """fbgnn_gnn handle holding the current weights."""
        self.build()
        ctx = ctx or self._ctx or _ffi.default_context()
        ent = self._handles.get(id(ctx))          # one device copy of the weights per context (GPU)
        if (ent is None or ent[0] is not ctx) and self._num_mlp_layers != 2:
            import ctypes as C
            if self._gemm != "fma":
                raise _ffi.FbgnnError("the tensor-core form of the feedback GNN is built for 2-layer MLPs")
            packed = []
            step = 2 if self._use_bias else 1
            for i in range(0, len(self._weights), step):
                W = self._weights[i]
                packed += [W.reshape(-1), self._weights[i + 1] if self._use_bias else np.zeros(W.shape[1], np.float32)]
            packed = np.ascontiguousarray(np.concatenate(packed), np.float32)
            h = C.c_void_p()
            _ffi.call("fbgnn_gnn_create_deep", ctx.handle, self._num_hidden_units, self._num_msg_dims,
                      self._num_mlp_layers, ACTS[self._activation], REDUCE[self._reduce_op], int(self._use_bias),
                      packed.ctypes.data_as(C.POINTER(C.c_float)), packed.size, C.byref(h))
            self._handles[id(ctx)] = (ctx, h)
            ent = self._handles[id(ctx)]
        if ent is None or ent[0] is not ctx:
            import ctypes as C
            if self._use_bias:
                W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3 = self._weights
            else:
                W0, W1x, W2x, W1z, W2z, W3 = self._weights
                b0 = b1x = b2x = b1z = b2z = b3 = None
            fp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))
            h = C.c_void_p()
            _ffi.call("fbgnn_gnn_create", ctx.handle, self._num_hidden_units, self._num_msg_dims,
                      ACTS[self._activation], REDUCE[self._reduce_op],
                      *[fp(a) for a in (W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3)], C.byref(h))
            if self._gemm == "tf32x3":
                _ffi.call("fbgnn_gnn_set_gemm", h, 1)
            self._handles[id(ctx)] = (ctx, h)
        return self._handles[id(ctx)][1]

    # -- forward ---------------------------------------------------------------------------
    def __call__(self, inputs):
        """``(h_vn [B,n,3], logit_hx [m_x,B], logit_hz [m_z,B], syndrome_x [m_x,B],
        syndrome_z [m_z,B]) -> new priors [B,n,3]`` (feedback_gnn.py:161-188)."""
        h_vn, logit_hx, logit_hz, syndrome_x, syndrome_z = inputs
        dev = _ffi.device_code(self._code, self._ctx)
        ctx = dev.ctx
        on_device = any(_is_device(t) for t in inputs)
        h = ctx.asarray(h_vn, np.float32)
        B = h.shape[0]
        if h.shape != (B, dev.n, 3):
            raise ValueError(f"h_vn must have shape [B,{dev.n},3]")
        lhx = ctx.asarray(logit_hx, np.float32)
        lhz = ctx.asarray(logit_hz, np.float32)
        sx = ctx.asarray(_to_u8(syndrome_x), np.uint8)
        sz = ctx.asarray(_to_u8(syndrome_z), np.uint8)
        for t, m in ((lhx, dev.mx), (sx, dev.mx), (lhz, dev.mz), (sz, dev.mz)):
            if t.shape != (m, B):
                raise ValueError(f"check-node inputs must have shape [{m},{B}], got {t.shape}")
        out = ctx.empty((B, dev.n, 3), np.float32)
        _ffi.call("fbgnn_gnn_forward", dev.handle, self.device_handle(ctx), B, h.t3(), lhx.t2(), lhz.t2(),
                  sx.t2(), sz.t2(), out.t3())
        return out if on_device else out.numpy()

    call = __call__


def packed_words(n):
    """Words per packed bit-plane row of n bits: ceil(n / 32) rounded up to a multiple of 4 (16-byte rows)."""
    return (((int(n) + 31) // 32) + 3) & ~3


def pack_bits(a):
    """[B, n] 0/1 array -> uint32 [B, packed_words(n)]: entry v = bit (v & 31) of word v >> 5."""
    a = np.asarray(a).astype(bool)
    B, n = a.shape
    wq = packed_words(n)
    padded = np.zeros((B, wq * 32), np.uint8)
    padded[:, :n] = a
    return np.ascontiguousarray(np.packbits(padded, axis=1, bitorder="little").view("<u4"))


def unpack_bits(words, n):
    """Inverse of ``pack_bits`` (also for the frame planes: unpack_bits(frame_bits, B))."""
    w = np.ascontiguousarray(np.asarray(words), dtype="<u4")
    return np.unpackbits(w.view(np.uint8), axis=-1, bitorder="little")[..., :n]


class ErrorIndicator:
    """Lazy ``[B, rows]`` 0/1 matrix whose row-wise "any" is already known (see module doc)."""

    def __init__(self, flags_fn, rows, materialise=None):
        self._flags_fn, self._rows, self._materialise = flags_fn, rows, materialise
        self._flags = None

    def has_dense(self):
        """False when only the per-frame flags exist (the dense matrix was not kept on the device)."""
        return self._materialise is not None

    def frame_flags(self):
        """uint8 [B]: 1 where the row of the matrix has any non-zero entry."""
        if self._flags is None:
            self._flags = self._flags_fn()
        return self._flags

    @property
    def shape(self):
        return (len(self.frame_flags()), self._rows)

    def count_nonzero_rows(self):
        return int(self.frame_flags().sum())

    def numpy(self):
        if self._materialise is None:
            raise _ffi.FbgnnError("the dense matrix is not kept by this model; use frame_flags() / count_nonzero_rows()")
        return self._materialise()

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        return a if dtype is None else a.astype(dtype)


class Sandwich_BP_GNN_Evaluation_Model:
    """``model(batch_size, p) -> (s_hat, ls_hat)`` for BP -> (GNN -> BP) x nG under depolarising noise.

    Extra keyword arguments (not in the reference):
      seed            Philox key of the noise source (default 0)
      first_frame     global id of the first frame; every call advances it by ``batch_size``,
                      so shards of one Monte-Carlo run can be given disjoint id ranges
      skip_inactive   stop frames once their correction matches the syndrome (result-identical
                      to the reference, which masks the later updates: feedback_gnn.py:339-340)
      early_stop      opt-in: every BP stage leaves a frame's iteration loop at the first iteration whose decision
                      reproduces the syndrome (SURVEY.md H8).  NOT what the reference computes -- it always runs
                      num_iter iterations -- so it is off by default and excluded from parity claims
      osd_order       with osd0: 0 runs OSD-0, λ > 0 the combination sweep OSD-CS of order λ (bp_osd.OSD_Decoder)
      lsd             a bp_osd.LSD_Decoder: the frames still mismatching after the last stage are re-solved by LSD-0 on
                      each side's full matrix, with its budgets; a side LSD-0 abandons keeps its BP decision.  Not
                      together with osd0=True
    """

    def __init__(self, code, decoders, feedbacks, num_layers=4, wt=False, p0=0.05, seed=0, first_frame=0,
                 skip_inactive=False, osd0=False, ctx=None, early_stop=False, osd_order=0, lsd=None):
        self.k, self.n = code.K, code.N
        self.code = code
        self.hx, self.hz, self.lx, self.lz = code.hx, code.hz, code.lx, code.lz
        self.hx_perp, self.hz_perp = code.hx_perp, code.hz_perp
        self.code_name = code.name
        self.num_checks = code.hx.shape[0] + code.hz.shape[0]
        self.channel = Pauli(wt=wt)
        self.decoders = list(decoders)
        self.feedbacks = list(feedbacks)
        self.num_layers = int(num_layers)
        if len(self.decoders) < self.num_layers or len(self.feedbacks) < self.num_layers - 1:
            raise ValueError("need num_layers decoders and num_layers-1 feedbacks")
        for d in self.decoders[:self.num_layers]:
            if not isinstance(d, QLDPCBPDecoder):
                raise TypeError("decoders must be fbgnn QLDPCBPDecoder layers")
        for g in self.feedbacks[:self.num_layers - 1]:
            if not isinstance(g, Feedback_GNN):
                raise TypeError("feedbacks must be fbgnn Feedback_GNN layers")
        self.wt = wt
        self.p0 = p0
        if wt and p0 is None:
            raise ValueError("wt=True needs an explicit p0 (the model input is then an error weight, not a rate)")
        self.seed = int(seed)
        self.next_frame = int(first_frame)
        self.skip_inactive = bool(skip_inactive)
        self.osd0 = bool(osd0)          # OSD-0 on the frames the last BP stage leaves mismatching (bp_osd.py)
        self.early_stop = bool(early_stop)   # opt-in: BP stages stop per frame at the first syndrome match (not the reference)
        self.osd_order = int(osd_order)
        if not 0 <= self.osd_order <= 65535:
            raise ValueError(f"osd_order must be in [0, 65535], got {osd_order}")
        if lsd is not None:
            from .bp_osd import LSD_Decoder
            if not isinstance(lsd, LSD_Decoder):
                raise TypeError("lsd must be an fbgnn LSD_Decoder")
            if self.osd0:
                raise ValueError("give osd0=True or lsd, not both")
        self.lsd = lsd
        self._ctx = ctx
        self.last_counters = None

    def prior(self, p):
        """log(3(1-p0)/p0) as float32 (feedback_gnn.py:311-312)."""
        p0 = float(p) if self.p0 is None else float(self.p0)
        return np.float32(np.log(np.float64(np.float32(3. * (1. - p0) / p0))))

    def _cfg(self, ctx, p):
        """fbgnn_pipeline_cfg of this model at noise level ``p`` (+ the ctypes arrays it points into)."""
        import ctypes as C
        S = self.num_layers
        ni = (C.c_int32 * S)(*[d.num_iter for d in self.decoders[:S]])
        fa = (C.c_float * S)(*[d.normalization_factor for d in self.decoders[:S]])
        ct = (C.c_int32 * S)(*[CN_TYPES[d.cn_type] for d in self.decoders[:S]])
        gh = (C.c_void_p * max(S - 1, 1))(*[g.device_handle(ctx).value for g in self.feedbacks[:S - 1]])
        # wt=True: `p` is the error weight (feedback_gnn.py:300-301) and p0 must be given
        thr = pauli_thresholds(0.0 if self.wt else float(p))
        lsd = self.lsd
        cfg = _ffi.PipelineCfg(S, ni, fa, ct, gh, float(self.prior(p)), (C.c_float * 3)(*thr),
                               int(round(float(p))) if self.wt else 0, 1 if (self.osd0 or lsd is not None) else 0,
                               1 if self.skip_inactive else 0, 1 if self.early_stop else 0, self.osd_order,
                               1 if lsd is not None else 0, lsd.max_cols if lsd is not None else 0,
                               lsd.max_checks if lsd is not None else 0)
        return cfg, (ni, fa, ct, gh)

    def run(self, batch_size, p, noise=None, want_flags=True, want_diff=True, want_counters=False):
        """Device-level entry.  Returns dict(flags, x_diff, z_diff DeviceArrays, counters ndarray)."""
        import ctypes as C
        dev = _ffi.device_code(self.code, self._ctx)
        ctx = dev.ctx
        B = int(batch_size)
        cfg, keepalive = self._cfg(ctx, p)
        nx = nz = _ffi.NULL2
        keep = None
        if noise is not None:
            keep = (ctx.asarray(_to_u8(noise[0]), np.uint8), ctx.asarray(_to_u8(noise[1]), np.uint8))
            if keep[0].shape != (B, dev.n) or keep[1].shape != (B, dev.n):
                raise ValueError(f"noise_x / noise_z must have shape [{B},{dev.n}], got {keep[0].shape} / {keep[1].shape}")
            nx, nz = keep[0].t2(), keep[1].t2()
        flags = ctx.empty((B,), np.uint8) if want_flags else None
        xd = ctx.empty((B, dev.n), np.uint8) if want_diff else None
        zd = ctx.empty((B, dev.n), np.uint8) if want_diff else None
        counters = (C.c_int64 * 4)() if want_counters else None
        _ffi.call("fbgnn_pipeline_run", dev.handle, C.byref(cfg), self.seed, self.next_frame, B, nx, nz,
                  flags.ptr if flags is not None else None,
                  xd.t2() if xd is not None else _ffi.NULL2, zd.t2() if zd is not None else _ffi.NULL2,
                  counters)
        if noise is None:
            self.next_frame += B
        res = dict(flags=flags, x_diff=xd, z_diff=zd,
                   counters=np.array(list(counters), np.int64) if want_counters else None)
        self.last_counters = res["counters"]
        return res

    def run_bits(self, batch_size, p, noise_bits=None, want_frame_bits=True, want_diff=False, want_counters=False):
        """Packed-bitmask entry (fbgnn_pipeline_run_bits): what a Monte-Carlo host loop exchanges with the GPU is 32 qubits /
        32 frames per word.  ``noise_bits``: optional pair of uint32 [B, wq] arrays (host or device; ``pack_bits``), qubit v of
        frame b = bit (v & 31) of word [b, v >> 5].  Returns dict(frame_bits uint32 [3, ceil(B/32)] device: planes flagged /
        block error / failed stage 0; x_diff_bits, z_diff_bits uint32 [B, wq]; counters)."""
        import ctypes as C
        dev = _ffi.device_code(self.code, self._ctx)
        ctx = dev.ctx
        B = int(batch_size)
        cfg, keepalive = self._cfg(ctx, p)
        wq = packed_words(dev.n)
        nx = nz = None
        if noise_bits is not None:
            nx, nz = (ctx.asarray(a, np.uint32) for a in noise_bits)
            if nx.shape != (B, wq) or nz.shape != (B, wq):
                raise ValueError(f"packed noise planes must have shape [{B},{wq}], got {nx.shape} / {nz.shape}")
        fb = ctx.empty((3, (B + 31) // 32), np.uint32) if want_frame_bits else None
        xd = ctx.empty((B, wq), np.uint32) if want_diff else None
        zd = ctx.empty((B, wq), np.uint32) if want_diff else None
        counters = (C.c_int64 * 4)() if want_counters else None
        ptr = lambda a: a.ptr if a is not None else None
        _ffi.call("fbgnn_pipeline_run_bits", dev.handle, C.byref(cfg), self.seed, self.next_frame, B, ptr(nx), ptr(nz),
                  ptr(fb), ptr(xd), ptr(zd), counters)
        if noise_bits is None:
            self.next_frame += B
        res = dict(frame_bits=fb, x_diff_bits=xd, z_diff_bits=zd,
                   counters=np.array(list(counters), np.int64) if want_counters else None)
        self.last_counters = res["counters"]
        return res

    def __call__(self, batch_size, ebno_db):
        res = self.run(batch_size, float(np.asarray(ebno_db)))
        flags, xd, zd = res["flags"], res["x_diff"], res["z_diff"]
        cache = {}

        def host_flags():
            if "f" not in cache:
                cache["f"] = flags.numpy()
            return cache["f"]

        def diffs():
            if "d" not in cache:
                cache["d"] = (xd.numpy().astype(np.int64), zd.numpy().astype(np.int64))
            return cache["d"]

        def s_hat():       # feedback_gnn.py:349-350,355
            x, z = diffs()
            return np.concatenate([(x @ self.hz.T) & 1, (z @ self.hx.T) & 1], axis=1)

        def ls_hat():      # feedback_gnn.py:352-353,356
            x, z = diffs()
            return np.concatenate([(x @ self.hx_perp.T) & 1, (z @ self.hz_perp.T) & 1], axis=1)

        return (ErrorIndicator(lambda: host_flags() & 1, self.num_checks, s_hat),
                ErrorIndicator(lambda: (host_flags() >> 1) & 1,
                               self.hx_perp.shape[0] + self.hz_perp.shape[0], ls_hat))

    call = __call__


class BP_BSC_Model:
    """``model(batch_size, p)`` for binary syndrome BP on a BSC (feedback_gnn.py:190-229)."""

    def __init__(self, pcm, decoder, logical_pcm=None, p0=None, seed=0, first_frame=0, ctx=None):
        if not isinstance(decoder, LDPCBPDecoder):
            raise TypeError("decoder must be an fbgnn LDPCBPDecoder layer")
        self.pcm = np.asarray(pcm.toarray() if hasattr(pcm, "toarray") else pcm)
        self.logical_pcm = None if logical_pcm is None else np.asarray(logical_pcm)
        _, self.n = self.pcm.shape
        self.decoder = decoder
        self.p0 = p0
        self.seed = int(seed)
        self.next_frame = int(first_frame)
        self._ctx = ctx
        self._graph = None
        self._logical = None
        self._osd_basis = None          # set by BP2_OSD_Model
        self._osd_pivot = None
        self._osd_order = 0
        self._lsd = None                # set by BP2_OSD_Model with an LSD_Decoder
        self.last_counters = None

    def llr_const(self, p):
        """-log((1-p0)/p0) as float32 (feedback_gnn.py:210-211)."""
        p0 = float(p) if self.p0 is None else float(self.p0)
        return np.float32(-np.log(np.float64(np.float32((1. - p0) / p0))))

    def _graphs(self):
        if self._graph is None:
            self._graph = _ffi.Graph(self.pcm, self._ctx)
            if self.logical_pcm is not None:
                self._logical = _ffi.Graph(self.logical_pcm, self._graph.ctx)
        return self._graph, self._logical

    def run(self, batch_size, p, noise=None, want_counters=False):
        import ctypes as C
        g, lg = self._graphs()
        ctx = g.ctx
        B = int(batch_size)
        flags = ctx.empty((B,), np.uint8)
        counters = (C.c_int64 * 4)() if want_counters else None
        nz = _ffi.NULL2
        keep = None
        if noise is not None:
            keep = ctx.asarray(_to_u8(noise), np.uint8)
            if keep.shape != (B, self.n):
                raise ValueError(f"noise must have shape [{B},{self.n}], got {keep.shape}")
            nz = keep.t2()
        d = self.decoder
        if self._lsd is not None:
            _ffi.call("fbgnn_bsc_pipeline_run_lsd", g.handle, lg.handle if lg is not None else None,
                      CN_TYPES[d.cn_type], d.num_iter, d.normalization_factor, float(self.llr_const(p)),
                      float(np.float32(p)), self.seed, self.next_frame, B, nz, flags.ptr, counters,
                      self._lsd.max_cols, self._lsd.max_checks)
        else:
            _ffi.call("fbgnn_bsc_pipeline_run_ex", g.handle, lg.handle if lg is not None else None,
                      CN_TYPES[d.cn_type], d.num_iter, d.normalization_factor, float(self.llr_const(p)),
                      float(np.float32(p)), self.seed, self.next_frame, B, nz, flags.ptr, counters,
                      self._osd_basis.handle if self._osd_basis is not None else None,
                      self._osd_pivot.ctypes.data_as(C.POINTER(C.c_int32)) if self._osd_pivot is not None else None,
                      self._osd_order)
        if noise is None:
            self.next_frame += B
        self.last_counters = np.array(list(counters), np.int64) if want_counters else None
        return dict(flags=flags, counters=self.last_counters)

    def __call__(self, batch_size, ebno_db):
        p = float(np.asarray(ebno_db))
        if self.logical_pcm is None:
            # reference returns (noise, noise_hat): run the layers one by one
            g, _ = self._graphs()
            ctx = g.ctx
            B = int(batch_size)
            noise = ctx.empty((B, self.n), np.uint8)
            _ffi.call("fbgnn_bsc_sample", ctx.handle, self.n, B, float(np.float32(p)), self.seed,
                      self.next_frame, noise.t2())
            self.next_frame += B
            synd = ctx.empty((B, g.m), np.uint8).T
            _ffi.call("fbgnn_syndrome", g.handle, B, noise.t2(), synd.t2())
            llr = ctx.asarray(np.full((B, self.n), self.llr_const(p), np.float32))
            noise_hat = self.decoder((llr, synd))
            return noise.numpy().astype(np.float32), np.asarray(noise_hat.numpy(), np.float32)
        res = self.run(batch_size, p)
        flags = res["flags"]
        cache = {}

        def host_flags():
            if "f" not in cache:
                cache["f"] = flags.numpy()
            return cache["f"]

        return (ErrorIndicator(lambda: host_flags() & 1, self.pcm.shape[0]),
                ErrorIndicator(lambda: (host_flags() >> 1) & 1, self.logical_pcm.shape[0]))

    call = __call__
