"""TEST INFRASTRUCTURE -- float64 numpy restatement of the loss of Second_Stage_GNN_BP_Model.call
(sionna/fec/ldpc/feedback_gnn.py:412-431: Feedback_GNN -> QLDPCBPDecoder(stage_two) -> multi-loss BCE), used
to check the hand-written gradient of csrc/fbgnn_train.cuh.

Only tests/ may import this module.  Everything is evaluated with the exact mathematical functions in
float64 (no float32 thresholds), so it is the smooth function whose derivative the CUDA reverse sweep
approximates at float32 accuracy.  Parity of the gradient with TensorFlow is unpinned (TensorFlow is not
available).  oracle/torch_grad_oracle.py restates this loss in torch (equal to 1e-12, reduce "sum" added) and
differentiates it by autograd; tests/test_train_grad.py compares the CUDA gradient with that, array by array and
element by element (profiles/grad_error_b200.txt).
"""
import numpy as np

CLIP_LO, CLIP_HI = 8.5e-8, 16.635532


def _phi(x):
    x = np.clip(x, CLIP_LO, CLIP_HI)
    return np.logaddexp(0.0, x) - np.log(np.expm1(x))


def _edges(pcm):
    c, v = np.nonzero(np.asarray(pcm))          # row-major (cn, vn): feedback_gnn.py:88
    return c, v


def gnn_forward(code, w, h_vn, logit_hx, logit_hz, sx, sz):
    """Feedback_GNN.call (feedback_gnn.py:161-188), literal per-edge form.  h_vn [B,n,3]; logits / syndromes [m,B]."""
    W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3 = [np.asarray(a, np.float64) for a in w]
    h_vn = np.asarray(h_vn, np.float64)
    B, n, _ = h_vn.shape
    ms = []
    for pcm, lg, sy, W1, b1, W2, b2 in ((code.hx, logit_hx, sx, W1x, b1x, W2x, b2x), (code.hz, logit_hz, sz, W1z, b1z, W2z, b2z)):
        c, v = _edges(pcm)
        h_cn = (np.asarray(lg, np.float64) * (1.0 - 2.0 * np.asarray(sy, np.float64))).T          # [B, m]
        f = np.concatenate([h_cn[:, c, None], h_vn[:, v, :]], axis=-1)                              # [B, E, 4]
        msg = np.tanh(f @ W1 + b1) @ W2 + b2                                                        # [B, E, M]
        acc = np.zeros((B, n, msg.shape[-1]))
        np.add.at(acc, (slice(None), v), msg)
        deg = np.bincount(v, minlength=n).astype(np.float64)
        ms.append(acc / np.maximum(deg, 1.0)[None, :, None])
    x = np.concatenate([ms[0], ms[1], h_vn], axis=-1)
    return np.tanh(x @ W3 + b3) @ W0 + b0                                                           # [B, n, 3]


def _soft_syndrome(pcm_edges, m, llr):
    c, v = pcm_edges
    val = llr[:, v]                                                                                 # [B, E]
    sgn = np.where(val < 0, -1.0, 1.0)
    B = llr.shape[0]
    T = np.zeros((B, m)); par = np.ones((B, m))
    np.add.at(T, (slice(None), c), _phi(np.abs(val)))
    np.multiply.at(par, (slice(None), c), sgn)
    return par * _phi(T)                                                                            # [B, m]


def bp4_logits(code, llr, sx, sz, num_iter, factor):
    """QLDPCBPDecoder.call with stage_two (decoding_q.py:732-780), boxplus-phi: list of (x_logit, z_logit) [B,m] for
    the message states 0..num_iter.  llr [B,3,n] = priors (x, y, z)."""
    llr = np.asarray(llr, np.float64)
    B, _, n = llr.shape
    ex, ez = _edges(code.hx), _edges(code.hz)
    mxn, mzn = code.hx.shape[0], code.hz.shape[0]
    synx = (1.0 - 2.0 * np.asarray(sx, np.float64)).T                                               # [B, m_x]
    synz = (1.0 - 2.0 * np.asarray(sz, np.float64)).T
    mx = np.zeros((B, len(ex[0]))); mz = np.zeros((B, len(ez[0])))
    out = []

    def marg():
        Sx = np.zeros((B, n)); Sz = np.zeros((B, n))
        np.add.at(Sx, (slice(None), ex[1]), mx)
        np.add.at(Sz, (slice(None), ez[1]), mz)
        return Sz + llr[:, 0], Sz + Sx + llr[:, 1], Sx + llr[:, 2]

    def logits(Lx, Ly, Lz):
        llr_z = np.logaddexp(0.0, -Lx) - np.logaddexp(-Lz, -Ly)
        llr_x = np.logaddexp(0.0, -Lz) - np.logaddexp(-Lx, -Ly)
        return _soft_syndrome(ez, mzn, llr_x), _soft_syndrome(ex, mxn, llr_z)

    def cn(edges, m, v2c, syn):
        c, _ = edges
        sgn = np.where(v2c < 0, -1.0, 1.0)
        par = syn.copy()
        np.multiply.at(par, (slice(None), c), sgn)
        a = _phi(np.abs(v2c))
        T = np.zeros((B, m))
        np.add.at(T, (slice(None), c), a)
        return sgn * par[:, c] * _phi(T[:, c] - a) * factor

    for _ in range(num_iter):
        Lx, Ly, Lz = marg()
        out.append(logits(Lx, Ly, Lz))
        vx = np.logaddexp(0.0, -Lx[:, ex[1]]) - np.logaddexp(-(Lz[:, ex[1]] - mx), -(Ly[:, ex[1]] - mx))
        vz = np.logaddexp(0.0, -Lz[:, ez[1]]) - np.logaddexp(-(Lx[:, ez[1]] - mz), -(Ly[:, ez[1]] - mz))
        mx, mz = cn(ex, mxn, vx, synx), cn(ez, mzn, vz, synz)
    out.append(logits(*marg()))
    return out


def _bce(label, logit):
    """tf.keras.losses.BinaryCrossentropy(from_logits=True): mean over all entries."""
    return np.mean(np.maximum(logit, 0.0) - logit * label + np.log1p(np.exp(-np.abs(logit))))


def second_stage_loss(code, w, h_vn, logit_hx, logit_hz, sx, sz, num_iter, factor=1.0, loss_from=8):
    """loss of feedback_gnn.py:425-431.  logit_hx pairs with hx rows (the caller's logit_hz_perp), logit_hz with hz."""
    new_llr = gnn_forward(code, w, h_vn, logit_hx, logit_hz, sx, sz)
    lg = bp4_logits(code, np.transpose(new_llr, (0, 2, 1)), sx, sz, num_iter, factor)
    gt_x = 1.0 - np.asarray(sz, np.float64).T
    gt_z = 1.0 - np.asarray(sx, np.float64).T
    loss = 0.0
    for i in range(loss_from, num_iter):
        x_logit, z_logit = lg[i + 1]
        loss += _bce(gt_x, x_logit) + _bce(gt_z, z_logit)
    return loss
