"""Shared helpers of the parity tests (test infrastructure; may import oracle/)."""
import json
import os

import numpy as np

from oracle.make_golden import MODEL_CASES, VQ_CASES, make_vq_inputs, window  # noqa: F401
from oracle.weights import make_images, make_state_dict

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HP_KEYS = ("h_dim", "res_h_dim", "n_res_layers", "n_embeddings", "embedding_dim")


def load_golden(name):
    """A golden case.  Model cases also carry the reference's VQ step on the stored z_e (vq_idx, vq_loss,
    vq_perplexity) and its decoder on the resulting z_q (dec_x_hat): for a full-size fixture these are the forward's
    own idx, loss, perplexity and x_hat; a windowed fixture (cfg3_s256) stores them for its window."""
    with np.load(os.path.join(GOLDEN, name + ".npz")) as d:
        out = {k: d[k] for k in d.files}
    out["case"] = json.loads(str(out["case"]))
    if "z_e" in out:
        for k, full in (("vq_idx", "idx"), ("vq_loss", "loss"), ("vq_perplexity", "perplexity"), ("dec_x_hat", "x_hat")):
            out.setdefault(k, out[full])
    return out


def model_case_inputs(case):
    hp = {k: case[k] for k in HP_KEYS}
    sd = make_state_dict(seed=case["wseed"], codebook=case["codebook"],
                         codebook_scale=case["codebook_scale"], **hp)
    x = make_images(case["batch"], case["size"], case["xseed"])
    return hp, sd, x


def build_model(hp, sd, device="cuda"):
    """The product model (drop-in import path) loaded with a numpy state dict."""
    import torch
    from models.vqvae import VQVAE
    m = VQVAE(hp["h_dim"], hp["res_h_dim"], hp["n_res_layers"], hp["n_embeddings"],
              hp["embedding_dim"], 0.25)
    m.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    return m.to(device).eval()


def expected_zq(g, E=None):
    """The reference's z_q (NCHW) of a golden case, or None when only its hash is stored.  Cases that do not store z_q
    to stay small (cfg3_s256) hold z_e and vq_idx, from which z_q = fl(z_e + fl(E[idx] - z_e)) follows
    (quantizer.py:60,67)."""
    if "z_q" in g:
        return g["z_q"]
    if "z_e" in g and E is not None:
        z = g["z_e"]
        B, D, H, W = z.shape
        rows = np.ascontiguousarray(z.transpose(0, 2, 3, 1)).reshape(-1, D)
        e = np.asarray(E, dtype=np.float32)[g["vq_idx"].ravel()]
        zq = (rows + (e - rows).astype(np.float32)).astype(np.float32)
        return np.ascontiguousarray(zq.reshape(B, H, W, D).transpose(0, 3, 1, 2))
    return None


# --------------------------------------------------------------------------- TF32 layer reference and bound
# A tcgen05 kind::tf32 MMA reads fp32 operands and drops the low 13 mantissa bits (round toward zero to a 10-bit
# mantissa; tests/test_tf32_bound.py pins this on the GPU).  Products of two TF32 values are exact in float64, so the
# centre c = sum t(x) t(w) + b (+ skip) is computed exactly up to float64 rounding.  The kernel adds the products in
# K = 8 blocks into fp32 accumulators (2 or 4 partials), then adds the partials, the bias and the skip in fp32; for
# any faithful fp32 accumulation of the blocks
#     |y - c| <= rho(K) * S,   S = sum |t(x)| |t(w)| + |b| (+ |skip|),   rho(K) = (ceil(K / 8) + 8) * 2^-22,
# with K the number of products summed into one output (a stride-2 transposed conv: the taps of that output's
# parity only).  ReLU is 1-Lipschitz, so the bound holds after it.  No bound is propagated through layers: every
# layer is checked on the input it really received.
TF32_MASK = np.uint32(0xFFFFE000)


def tf32(a):
    """fp32 -> TF32 operand of a tcgen05 kind::tf32 MMA (float32 array): mantissa truncated to 10 bits."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
    return (a.view(np.uint32) & TF32_MASK).view(np.float32)


def rho(K):
    return (-(-K // 8) + 8) * 2.0 ** -22


def conv_products(x, w, stride, pad, transposed):
    """Float64 conv / conv-transpose (NCHW, torch CPU) and the number of products summed into one output."""
    import torch
    import torch.nn.functional as F
    tx, tw = torch.from_numpy(np.asarray(x, np.float64)), torch.from_numpy(np.asarray(w, np.float64))
    kh, kw = w.shape[2], w.shape[3]
    if transposed:
        y = F.conv_transpose2d(tx, tw, None, stride, pad)
        K = -(-kh // stride) * -(-kw // stride) * w.shape[0]
    else:
        y = F.conv2d(tx, tw, None, stride, pad)
        K = kh * kw * w.shape[1]
    return y.numpy(), K


def tf32_layer_ref(x, w, b=None, *, stride=1, pad=0, transposed=False, skip=None, relu=False, operand=tf32):
    """(c, bound) of one TF32 conv / conv-transpose layer (NCHW float64) on the observable fp32 input x.
    `operand` maps an fp32 operand to what the MMA multiplies (tf32 for the kernels; the identity gives the plain
    reference the sensitivity checks use)."""
    xt, wt = operand(x).astype(np.float64), operand(w).astype(np.float64)
    c, K = conv_products(xt, wt, stride, pad, transposed)
    S, _ = conv_products(np.abs(xt), np.abs(wt), stride, pad, transposed)
    if b is not None:
        b = np.asarray(b, np.float64).reshape(1, -1, 1, 1)
        c, S = c + b, S + np.abs(b)
    if skip is not None:
        c, S = c + skip, S + np.abs(np.asarray(skip, np.float64))
    if relu:
        c = np.maximum(c, 0)
    return c, rho(K) * S


def tf32_residual_ref(r, w1, w2, *, relu_out=True, operand=tf32):
    """(c, bound, straddle share) of one residual layer out = act(r + W2 . relu(W1 (*) r)) (residual.py:18-29) as
    res_tc runs it: GEMM1 3x3 C -> Cmid, mid = relu(GEMM1) stored fp32 and truncated again as GEMM2's A operand,
    GEMM2 1x1 Cmid -> C + the skip r.  mid is not observable: with r1 = rho(K1) S1 the kernel's GEMM2 operand lies in
    [t(fl(relu(c1 - r1))), t(fl(relu(c1 + r1)))] (rounding, ReLU and t are monotone); GEMM2 is centred on
    t(fl(relu(c1))) and the bound gains sum |t(w2)| dev, dev = the larger distance to either end.  dev is non-zero only
    where mid straddles a TF32 boundary; the share of such mid values is returned."""
    r = np.asarray(r, np.float32)
    c1, b1 = tf32_layer_ref(r, w1, stride=1, pad=1, operand=operand)
    mid = operand(np.maximum(c1, 0).astype(np.float32)).astype(np.float64)
    lo = operand(np.maximum(c1 - b1, 0).astype(np.float32)).astype(np.float64)
    hi = operand(np.maximum(c1 + b1, 0).astype(np.float32)).astype(np.float64)
    dev = np.maximum(hi - mid, mid - lo)
    wt2 = operand(w2).astype(np.float64)
    c, K2 = conv_products(mid, wt2, 1, 0, False)
    S, _ = conv_products(np.abs(mid) + dev, np.abs(wt2), 1, 0, False)
    spread, _ = conv_products(dev, np.abs(wt2), 1, 0, False)
    c, S = c + r, S + np.abs(r.astype(np.float64))
    if relu_out:
        c = np.maximum(c, 0)
    return c, rho(K2) * S + spread, float((dev > 0).mean())


def bound_ratio(y, c, bound):
    """|y - c| / bound elementwise (inf where the bound is 0 and y != c)."""
    err = np.abs(np.asarray(y, np.float64) - c)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(err == 0, 0.0, err / bound)


def assert_within_bound(y, c, bound, what=""):
    """Every |y - c| <= bound; prints (and returns) the largest |y - c| / bound.  On failure reports the worst
    element, its ratio and the share of elements above the bound."""
    y = np.asarray(y, np.float64)
    assert y.shape == c.shape == bound.shape, (y.shape, c.shape, bound.shape)
    q = bound_ratio(y, c, bound)
    worst = np.unravel_index(int(np.argmax(q)), q.shape)
    qmax = float(q[worst])
    print("%s: max |y-c|/bound = %.4f over %d outputs" % (what, qmax, q.size))
    assert qmax <= 1.0, ("%s: |y-c| > bound at %s: y=%.9g c=%.9g bound=%.3g ratio %.3g; %.2f %% of outputs above"
                         % (what, tuple(int(i) for i in worst), y[worst], c[worst], bound[worst], qmax,
                            100 * float((q > 1).mean())))
    return qmax


def share_above_bound(y, c, bound):
    return float((bound_ratio(y, c, bound) > 1).mean())


def assert_zq_matches(g, zq_nchw, E=None):
    """Bitwise comparison of a z_q (NCHW fp32 array) with the golden case, through the stored array, the
    reconstruction above, or the stored SHA-256 of the reference's bytes."""
    import hashlib
    zq_nchw = np.ascontiguousarray(zq_nchw, dtype=np.float32)
    want = expected_zq(g, E)
    if want is not None:
        assert np.array_equal(zq_nchw, want, equal_nan=True)
    else:
        assert hashlib.sha256(zq_nchw.tobytes()).hexdigest() == str(g["z_q_sha256"])
