"""BP + OSD post-processing -- ``OSD_Decoder``, ``OSD0_Decoder``, ``BP4_OSD_Model``, ``BP2_OSD_Model``.

Mirrors ``sionna/fec/ldpc/bp_osd.py`` of the reference: the frames whose BP decision misses the
syndrome are re-solved by ordered-statistics decoding of order 0 (``:8-77``): columns ordered by the
reliabilities BP produced, row-wise Gaussian elimination of the full-rank basis ``[H_basis | s]``,
solution on the pivot columns.  The models keep the reference's contract: ``model(batch_size, p)``
returns ``(zeros_like(ls_hat), ls_hat)`` with ``ls_hat`` the logical-operator parities of the
residual error (``:183-197``, ``:262-274``), so ``PlotBER.simulate(..., qldpc=False)`` counts block
errors from it.  Everything runs on the GPU (``k_osd`` and the fused pipelines).

``OSD_Decoder(n, osd_order=λ)`` adds the combination sweep of Roffe et al., "Decoding across the quantum LDPC code
landscape" (2020) -- the ``ldpc`` package's ``osd_method="osd_cs"`` -- on the matrix OSD-0 has reduced: every single
non-pivot column, then every pair of the first λ non-pivot columns (least reliable first), each flipped on top of the
OSD-0 solution; the lightest solution (Hamming weight, ties to the earlier candidate) is returned.  Order 0 is OSD-0.

Ties between equal reliabilities are broken by qubit index (the reference's ``tf.argsort`` leaves
them to the backend).

A frame's reduced matrix sits in the shared memory of one CTA (``k_osd``).  Where it does not fit, as for the
[[1922,50]] hypergraph-product code, a thread-block cluster of 2, 4 or 8 CTAs splits it by rows (``k_osd_cluster``,
the same result bit for bit).  A basis beyond a cluster of 8 (about 1.8 MB, e.g. [[7688,50]]) raises ``FbgnnError``
with ``FBGNN_E_UNSUPPORTED`` (-3).
"""
import numpy as np

from . import _ffi
from .decoding import LDPCBPDecoder
from .decoding_q import QLDPCBPDecoder, _is_device, _to_u8
from .feedback_gnn import BP_BSC_Model, ErrorIndicator, Sandwich_BP_GNN_Evaluation_Model


OSD_METHODS = ("osd0", "osd_cs")


class OSD_Decoder:
    """``OSD_Decoder(n, osd_order=0, osd_method="osd_cs")(llr [bs,n], pcm [bs,rank,n] or [rank,n], s [rank,bs], bs)
    -> e_hat [bs,n]`` bool.  ``osd_method="osd0"`` or ``osd_order=0``: OSD-0; otherwise OSD-CS of order
    ``osd_order`` (at most 65535)."""

    def __init__(self, n, osd_order=0, osd_method="osd_cs", ctx=None):
        if osd_method not in OSD_METHODS:
            raise ValueError(f"osd_method must be one of {OSD_METHODS}, got {osd_method!r}")
        osd_order = int(osd_order)
        if not 0 <= osd_order <= 65535:
            raise ValueError(f"osd_order must be in [0, 65535], got {osd_order}")
        self.n = int(n)
        self.osd_method = osd_method
        self.osd_order = 0 if osd_method == "osd0" else osd_order
        self._ctx = ctx
        self._graphs = {}

    def _basis_graph(self, pcm):
        pcm = np.asarray(pcm)
        if pcm.ndim == 3:               # the reference broadcasts one basis over the batch (bp_osd.py:159-162)
            pcm = pcm[0]
        key = (pcm.shape, hash(pcm.tobytes()))
        if key not in self._graphs:
            self._graphs[key] = _ffi.Graph(pcm, self._ctx)
        return self._graphs[key]

    def __call__(self, llr, pcm, s, bs=None):
        g = self._basis_graph(pcm)
        ctx = g.ctx
        on_device = _is_device(llr) or _is_device(s)
        llr_d = ctx.asarray(llr, np.float32)
        B = llr_d.shape[0]
        s_d = ctx.asarray(_to_u8(s), np.uint8)
        if llr_d.shape != (B, self.n) or g.n != self.n or s_d.shape != (g.m, B):
            raise ValueError(f"expected llr [bs,{self.n}], pcm [rank,{self.n}], s [rank,bs]")
        e_hat = ctx.empty((B, self.n), np.uint8)
        _ffi.call("fbgnn_osd_decode", g.handle, self.osd_order, B, llr_d.t2(), s_d.t2(), e_hat.t2())
        return e_hat if on_device else e_hat.numpy().astype(bool)

    call = __call__


class OSD0_Decoder(OSD_Decoder):
    """``OSD0_Decoder(n)``: ``OSD_Decoder`` of order 0 (bp_osd.py:8-77)."""

    def __init__(self, n, ctx=None):
        super().__init__(n, osd_order=0, osd_method="osd0", ctx=ctx)


def _osd_order(osd_decoder):
    return int(getattr(osd_decoder, "osd_order", 0))


def _indicators(flags, rows, dense=None):
    """(zeros_like(ls_hat), ls_hat) of the reference (bp_osd.py:196-197, 273-274) as lazy indicators; ``dense``
    materialises ls_hat when the model kept the residual errors."""
    cache = {}

    def host_flags():
        if "f" not in cache:
            cache["f"] = flags.numpy()
        return cache["f"]

    ls_hat = ErrorIndicator(lambda: (host_flags() >> 1) & 1, rows, dense)
    zeros = ErrorIndicator(lambda: np.zeros_like(host_flags()), rows,
                           None if dense is None else (lambda: np.zeros((len(host_flags()), rows), np.int64)))
    return zeros, ls_hat


class BP4_OSD_Model:
    """Quaternary BP followed by OSD on the failed frames (bp_osd.py:80-197), of the order of ``osd_decoder``
    (``OSD0_Decoder``: OSD-0).  The prior is log(3(1-p)/p) with the simulated p (``:121``)."""

    def __init__(self, code, bp4_decoder, osd_decoder, seed=0, first_frame=0, ctx=None):
        if not isinstance(bp4_decoder, QLDPCBPDecoder):
            raise TypeError("bp4_decoder must be an fbgnn QLDPCBPDecoder layer")
        self.code, self.k, self.n = code, code.K, code.N
        self.bp4_decoder, self.osd_decoder = bp4_decoder, osd_decoder
        self._inner = Sandwich_BP_GNN_Evaluation_Model(code, [bp4_decoder], [], num_layers=1, p0=None, seed=seed,
                                                       first_frame=first_frame, osd0=True,
                                                       osd_order=_osd_order(osd_decoder), ctx=ctx)

    @property
    def last_counters(self):
        return self._inner.last_counters

    def run(self, batch_size, p, **kw):
        return self._inner.run(batch_size, p, **kw)

    def __call__(self, batch_size, ebno_db):
        res = self._inner.run(batch_size, float(np.asarray(ebno_db)), want_diff=True)
        xd, zd = res["x_diff"], res["z_diff"]

        def dense():      # ls_hat = [lz . x_diff ; lx . z_diff] (bp_osd.py:188-194)
            x, z = xd.numpy().astype(np.int64), zd.numpy().astype(np.int64)
            return np.concatenate([(x @ np.asarray(self.code.lz).T) & 1, (z @ np.asarray(self.code.lx).T) & 1], axis=1)

        return _indicators(res["flags"], self.code.lx.shape[0] + self.code.lz.shape[0], dense)

    call = __call__


class BP2_OSD_Model:
    """Binary syndrome BP on a BSC followed by OSD on the failed frames (bp_osd.py:199-274), of the order of
    ``osd_decoder``; the BP logit is -log((1-p)/p) with the simulated p (``:221``)."""

    def __init__(self, pcm, pcm_basis, pivot_pcm, logical_pcm, bp2_decoder, osd_decoder, seed=0, first_frame=0,
                 ctx=None):
        if not isinstance(bp2_decoder, LDPCBPDecoder):
            raise TypeError("bp2_decoder must be an fbgnn LDPCBPDecoder layer")
        self.pcm, self.pcm_basis = np.asarray(pcm), np.asarray(pcm_basis)
        self.pivot_pcm = np.ascontiguousarray(pivot_pcm, np.int32)
        self.logical_pcm = np.asarray(logical_pcm)
        self.rank, self.n = self.pcm_basis.shape
        if not np.array_equal(self.pcm[self.pivot_pcm], self.pcm_basis):
            raise ValueError("pcm_basis must be pcm[pivot_pcm]")
        self.bp2_decoder, self.osd_decoder = bp2_decoder, osd_decoder
        self._inner = BP_BSC_Model(self.pcm, bp2_decoder, logical_pcm=self.logical_pcm, p0=None, seed=seed,
                                   first_frame=first_frame, ctx=ctx)

    @property
    def last_counters(self):
        return self._inner.last_counters

    def run(self, batch_size, p, **kw):
        inner = self._inner
        if inner._osd_basis is None:
            g, _ = inner._graphs()
            inner._osd_basis = _ffi.Graph(self.pcm_basis, g.ctx)
            inner._osd_pivot = self.pivot_pcm
            inner._osd_order = _osd_order(self.osd_decoder)
        return inner.run(batch_size, p, **kw)

    def __call__(self, batch_size, ebno_db):
        res = self.run(batch_size, float(np.asarray(ebno_db)))
        return _indicators(res["flags"], self.logical_pcm.shape[0])

    call = __call__
