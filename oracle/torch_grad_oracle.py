"""TEST INFRASTRUCTURE -- the second-stage loss of oracle/np_grad_oracle.py restated in torch, so that autograd gives
the gradient csrc/fbgnn_train.cuh computes, element by element (Feedback_GNN -> BP4 stage_two with boxplus-phi ->
multi-loss BCE over the message states loss_from + 1 .. num_iter, in the same literal per-edge form).

Only tests/ and tools/ may import this module; it is the only place torch is imported (the product has no torch).

* ``dtype``: torch.float64 is the reference; torch.float32 measures the noise floor of a float32 evaluation.
* ``reduce``: the GNN's "mean" or "sum".  Any ``factor``, any ``loss_from`` in 0 .. num_iter, any CSS code (columns of
  degree 0 on either side included).
* Derivative rules as the header of fbgnn_train.cuh states them (TensorFlow's): signs and comparisons are detached,
  a clip passes the gradient inside its range only, phi'(x) = -1 / sinh(x).
* ``phi``: "smooth" is np_grad_oracle._phi (float64 formula after the clip); "specified" evaluates the library's
  exact-arithmetic phi (fb_phi4f through oracle.c_oracle) on the float32-rounded argument -- the staircase the kernel's
  forward pass sees near the clip -- with the same backward, the kernel's dphi.
* ``mutate``: a set of deliberate bugs (``MUTATIONS``) for the tests that show the tolerances would see them.
"""
import numpy as np
import torch

CLIP_LO, CLIP_HI = 8.5e-8, 16.635532
NAMES = ("W0", "b0", "W1x", "b1x", "W2x", "b2x", "W1z", "b1z", "W2z", "b2z", "W3", "b3")
MUTATIONS = ("swap_bce_weights", "swap_pairing", "bias_factor_one", "drop_cn_edge")


def _dphi(x, g):
    inside = (x >= CLIP_LO) & (x <= CLIP_HI)
    return torch.where(inside, -g / torch.sinh(torch.where(inside, x, torch.ones_like(x))), torch.zeros_like(g))


class _PhiSmooth(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        xc = x.clamp(CLIP_LO, CLIP_HI)
        return torch.logaddexp(torch.zeros_like(xc), xc) - torch.log(torch.expm1(xc))

    @staticmethod
    def backward(ctx, g):
        return _dphi(ctx.saved_tensors[0], g)


class _PhiSpecified(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        from oracle import c_oracle
        ctx.save_for_backward(x)
        x32 = x.detach().cpu().to(torch.float32).numpy()
        return torch.from_numpy(np.asarray(c_oracle.math_fn("phi4f", x32), np.float32)).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return _dphi(ctx.saved_tensors[0], g)


def _edges(pcm):
    c, v = np.nonzero(np.asarray(pcm))          # row-major (cn, vn): feedback_gnn.py:88
    return torch.as_tensor(c), torch.as_tensor(v)


def _scatter(n_out, idx, src):
    """sum of src[:, e] into out[:, idx[e]] (src [B, E, ...])."""
    return src.new_zeros((src.shape[0], n_out) + tuple(src.shape[2:])).index_add(1, idx, src)


def _parity(m, c, neg):
    """(-1)^(number of True in neg[:, e] over the edges e of each row), detached: [B, m]."""
    cnt = _scatter(m, c, neg.to(torch.int64))
    return (1 - 2 * (cnt % 2))


def gnn_forward(code, w, h_vn, logit_hx, logit_hz, sx, sz, reduce="mean", mutate=()):
    """Feedback_GNN.call, literal per-edge form (np_grad_oracle.gnn_forward) with reduce "mean" or "sum".  Torch
    tensors in, [B, n, 3] out."""
    W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3 = w
    B, n, _ = h_vn.shape
    ms = []
    for pcm, lg, sy, W1, b1, W2, b2 in ((code.hx, logit_hx, sx, W1x, b1x, W2x, b2x), (code.hz, logit_hz, sz, W1z, b1z, W2z, b2z)):
        c, v = _edges(pcm)
        h_cn = (lg * (1.0 - 2.0 * sy)).T                                                            # [B, m]
        f = torch.cat([h_cn[:, c, None], h_vn[:, v, :]], dim=-1)                                     # [B, E, 4]
        t = torch.tanh(f @ W1 + b1)                                                                 # [B, E, H]
        deg = torch.bincount(v, minlength=n).to(h_vn.dtype)
        if reduce == "mean":
            acc = _scatter(n, v, t @ W2 + b2)
            ms.append(acc / deg.clamp(min=1.0)[None, :, None])
        elif reduce == "sum":
            if "bias_factor_one" in mutate:   # value deg * b2, gradient of b2 counted once per node of nonzero degree
                b2v = deg[:, None] * b2.detach() + (deg > 0).to(deg.dtype)[:, None] * (b2 - b2.detach())
                ms.append(_scatter(n, v, t @ W2) + b2v[None])
            else:
                ms.append(_scatter(n, v, t @ W2 + b2))
        else:
            raise ValueError("reduce must be 'mean' or 'sum'")
    x = torch.cat([ms[0], ms[1], h_vn], dim=-1)
    return torch.tanh(x @ W3 + b3) @ W0 + b0                                                         # [B, n, 3]


def bp4_logits(code, llr, sx, sz, num_iter, factor, phi, mutate=()):
    """QLDPCBPDecoder.call with stage_two, boxplus-phi (np_grad_oracle.bp4_logits): (x_logit, z_logit) [B, m] of the
    message states 0 .. num_iter.  llr [B, 3, n] = priors (x, y, z)."""
    B, _, n = llr.shape
    ex, ez = _edges(code.hx), _edges(code.hz)
    mxn, mzn = code.hx.shape[0], code.hz.shape[0]
    synx, synz = (1 - 2 * sx.to(torch.int64)).T, (1 - 2 * sz.to(torch.int64)).T                    # [B, m]
    mx, mz = llr.new_zeros((B, len(ex[0]))), llr.new_zeros((B, len(ez[0])))
    zero = llr.new_zeros(())
    first = {}
    for key, (c, _) in (("x", ex), ("z", ez)):     # the first edge of every row (edges are row-major)
        f = torch.ones(len(c), dtype=torch.bool)
        f[1:] = c[1:] != c[:-1]
        first[key] = f

    def marg():
        Sx, Sz = _scatter(n, ex[1], mx), _scatter(n, ez[1], mz)
        return Sz + llr[:, 0], Sz + Sx + llr[:, 1], Sx + llr[:, 2]

    def soft_syndrome(edges, m, l):
        c, v = edges
        val = l[:, v]
        par = _parity(m, c, (val < 0).detach())
        return par * phi(_scatter(m, c, phi(val.abs())))

    def logits(Lx, Ly, Lz):
        llr_z = torch.logaddexp(zero, -Lx) - torch.logaddexp(-Lz, -Ly)
        llr_x = torch.logaddexp(zero, -Lz) - torch.logaddexp(-Lx, -Ly)
        if "swap_pairing" in mutate:
            llr_x, llr_z = llr_z, llr_x
        return soft_syndrome(ez, mzn, llr_x), soft_syndrome(ex, mxn, llr_z)

    def cn(edges, m, v2c, syn, key):
        c, _ = edges
        if "drop_cn_edge" in mutate:
            v2c = torch.where(first[key], v2c.detach(), v2c)
        neg = (v2c < 0).detach()
        sgn = 1 - 2 * neg.to(torch.int64)
        par = syn * _parity(m, c, neg)
        a = phi(v2c.abs())
        T = _scatter(m, c, a)
        return (sgn * par[:, c]) * phi(T[:, c] - a) * factor

    out = []
    for _ in range(num_iter):
        Lx, Ly, Lz = marg()
        out.append(logits(Lx, Ly, Lz))
        vx = torch.logaddexp(zero, -Lx[:, ex[1]]) - torch.logaddexp(-(Lz[:, ex[1]] - mx), -(Ly[:, ex[1]] - mx))
        vz = torch.logaddexp(zero, -Lz[:, ez[1]]) - torch.logaddexp(-(Lx[:, ez[1]] - mz), -(Ly[:, ez[1]] - mz))
        mx, mz = cn(ex, mxn, vx, synx, "x"), cn(ez, mzn, vz, synz, "z")
    out.append(logits(*marg()))
    return out


def _bce_sum(label, logit):
    """sum of tf.keras BinaryCrossentropy(from_logits=True) terms; the caller divides by the count."""
    return torch.sum(logit.clamp(min=0.0) - logit * label + torch.log1p(torch.exp(-logit.abs())))


def second_stage_loss_and_grad(code, w, h_vn, logit_hx, logit_hz, sx, sz, num_iter, factor=1.0, loss_from=8,
                               reduce="mean", dtype=torch.float64, phi="smooth", mutate=(), want_grad=True):
    """(loss, [12 gradients in Keras order]) of np_grad_oracle.second_stage_loss (argument order and pairing as
    there: logit_hx pairs with the rows of hx).  Inputs are numpy arrays; gradients come back as float64 arrays."""
    unknown = set(mutate) - set(MUTATIONS)
    if unknown:
        raise ValueError(f"unknown mutations {sorted(unknown)}")
    if not 0 <= loss_from <= num_iter:
        raise ValueError("loss_from must be in 0 .. num_iter")
    phi_fn = {"smooth": _PhiSmooth.apply, "specified": _PhiSpecified.apply}[phi]
    t = lambda a: torch.as_tensor(np.asarray(a, np.float64)).to(dtype)
    wt = [t(a).requires_grad_(want_grad) for a in w]
    sx_t, sz_t = torch.as_tensor(np.asarray(sx, np.uint8)), torch.as_tensor(np.asarray(sz, np.uint8))
    new_llr = gnn_forward(code, wt, t(h_vn), t(logit_hx), t(logit_hz), sx_t.to(dtype), sz_t.to(dtype), reduce, mutate)
    lg = bp4_logits(code, new_llr.permute(0, 2, 1), sx_t, sz_t, num_iter, factor, phi_fn, mutate)
    B = h_vn.shape[0]
    gt_x, gt_z = (1 - sz_t.to(dtype)).T, (1 - sx_t.to(dtype)).T
    cx, cz = B * code.hz.shape[0], B * code.hx.shape[0]          # entries of x_logit (rows of hz) / z_logit (rows of hx)
    if "swap_bce_weights" in mutate:
        cx, cz = cz, cx
    loss = new_llr.new_zeros(())
    for i in range(loss_from, num_iter):
        x_logit, z_logit = lg[i + 1]
        loss = loss + _bce_sum(gt_x, x_logit) / cx + _bce_sum(gt_z, z_logit) / cz
    if not want_grad:
        return float(loss.detach()), None
    if loss.requires_grad:
        grads = torch.autograd.grad(loss, wt, allow_unused=True)
    else:
        grads = [None] * len(wt)
    return float(loss.detach()), [np.zeros(a.shape) if g is None else g.detach().to(torch.float64).numpy() for a, g in zip(w, grads)]
