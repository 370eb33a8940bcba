"""The TF32 layer bar of tests/helpers.py (tf32_layer_ref / tf32_residual_ref / assert_within_bound).

CPU: the checker passes an emulated correct TF32 kernel and rejects each way a kernel can be subtly wrong (untruncated
or bf16 operands, round-to-nearest conversion, a dropped tap / k-step / bias, a border pixel read one pixel off), at
the shapes of E3 (K = 1152), the pre-quant 1x1 (K = 128) and D2 (K = 4 x 128 per output parity).
GPU: the operand conversion of tcgen05 kind::tf32 is pinned (truncation), and on the real kernels the plain float64
reference breaks the bound on a clear share of outputs, so the bar resolves TF32 operand precision.
"""
import numpy as np
import pytest
import torch

from tests.helpers import (assert_within_bound, conv_products, share_above_bound, tf32, tf32_layer_ref,
                           tf32_residual_ref)


def _identity(a):
    return np.asarray(a, np.float32)


def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(torch.bfloat16).float().numpy()


def _tf32_rna(a):
    """Round-to-nearest (ties away) TF32 conversion, what cvt.rna.tf32.f32 gives."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
    return ((a.view(np.uint32) + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def emulate_tf32_kernel(x, w, b, *, stride, pad, transposed, skip=None, relu=False, operand=tf32, drop_tap=None,
                        drop_kstep=None):
    """A TF32 tensor-core conv in numpy: converted operands, one K = 8 block (one tap x 8 input channels) at a time
    added into fp32 accumulators, two partials by block parity, then partials + bias (+ skip) (+ ReLU) in fp32."""
    xt, wt = operand(x).astype(np.float64), operand(w).astype(np.float64)
    cax = 0 if transposed else 1
    kh, kw = w.shape[2], w.shape[3]
    zero = np.zeros_like(conv_products(xt[:, :1], wt[:1] if transposed else wt[:, :1], stride, pad, transposed)[0],
                         dtype=np.float32)
    acc = [zero, zero]
    i = 0
    for r in range(kh):
        for s in range(kw):
            if (r, s) == drop_tap:
                continue
            for c0 in range(0, w.shape[cax], 8):
                if (r, s, c0) == drop_kstep:
                    continue
                sl = [slice(None)] * 4
                sl[cax] = slice(c0, c0 + 8)
                wk = np.zeros_like(wt[tuple(sl)])
                wk[:, :, r, s] = wt[tuple(sl)][:, :, r, s]
                blk, _ = conv_products(xt[:, c0:c0 + 8], wk, stride, pad, transposed)
                p = i & 1
                acc[p] = (acc[p] + blk).astype(np.float32)
                i += 1
    y = acc[0] + acc[1]
    if b is not None:
        y = y + np.asarray(b, np.float32).reshape(1, -1, 1, 1)
    if skip is not None:
        y = y + skip
    return np.maximum(y, np.float32(0)) if relu else y


SHAPES = {
    # Cin, k, stride, pad, transposed     (B = 1, 8 x 8 input, Cout = 16: the bound depends on K, not on Cout)
    "E3": (128, 3, 1, 1, False),          # encoder.py:35-36, K = 1152
    "1x1": (128, 1, 1, 0, False),         # vqvae.py:16-17, K = 128
    "D2": (128, 4, 2, 1, True),           # decoder.py:31-33, K = 512 per output parity
}


def _layer(name, seed=0):
    Cin, k, stride, pad, transposed = SHAPES[name]
    rng = np.random.RandomState(seed)
    x = np.maximum(rng.standard_normal((1, Cin, 8, 8)), 0).astype(np.float32)      # post-ReLU activations
    w = (rng.standard_normal((Cin, 16, k, k) if transposed else (16, Cin, k, k)) / np.sqrt(Cin * k * k)).astype(np.float32)
    b = (rng.standard_normal(16) * 0.1).astype(np.float32)
    return x, w, b, dict(stride=stride, pad=pad, transposed=transposed)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_emulated_tf32_kernel_is_within_bound(name):
    x, w, b, geo = _layer(name)
    c, bound = tf32_layer_ref(x, w, b, relu=True, **geo)
    assert_within_bound(emulate_tf32_kernel(x, w, b, relu=True, **geo), c, bound, "emulated %s" % name)
    c, bound = tf32_layer_ref(x, w, b, **geo)
    q = assert_within_bound(emulate_tf32_kernel(x, w, b, **geo), c, bound, "emulated %s, no ReLU" % name)
    assert q > 0          # the bound is not met by an accident of exact arithmetic


def _mutant(kind, x, w, b, geo):
    emu = emulate_tf32_kernel
    if kind == "plain_float64":
        return conv_products(x, w, geo["stride"], geo["pad"], geo["transposed"])[0] + b.reshape(1, -1, 1, 1)
    if kind == "bf16_operands":
        return emu(x, w, b, operand=_bf16, **geo)
    if kind == "round_to_nearest_tf32":
        return emu(x, w, b, operand=_tf32_rna, **geo)
    if kind == "tap_dropped":
        return emu(x, w, b, drop_tap=(w.shape[2] // 2, w.shape[3] // 2), **geo)
    if kind == "kstep_dropped":
        return emu(x, w, b, drop_kstep=(w.shape[2] - 1, w.shape[3] - 1, 120), **geo)
    if kind == "bias_dropped":
        return emu(x, w, None, **geo)
    if kind == "border_pixel_shifted":
        y = emu(x, w, b, **geo)
        y[..., 0] = emu(np.ascontiguousarray(np.roll(x, -1, axis=3)), w, b, **geo)[..., 0]   # column 0 reads column 1
        return y
    raise ValueError(kind)


MUTANTS = ["plain_float64", "bf16_operands", "round_to_nearest_tf32", "tap_dropped", "kstep_dropped", "bias_dropped",
           "border_pixel_shifted"]


@pytest.mark.parametrize("kind", MUTANTS)
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_checker_rejects_wrong_arithmetic(name, kind):
    x, w, b, geo = _layer(name)
    c, bound = tf32_layer_ref(x, w, b, **geo)
    y = _mutant(kind, x, w, b, geo)
    with pytest.raises(AssertionError, match="above"):
        assert_within_bound(y, c, bound, "%s %s" % (name, kind))
    print("%s %s: %.1f %% of outputs above the bound" % (name, kind, 100 * share_above_bound(y, c, bound)))


def _emulate_residual(r, w1, w2, mid_operand=tf32):
    """res_tc in numpy: GEMM1 as above (no bias), mid = relu(.) in fp32, GEMM2 on mid_operand(mid), + r, ReLU."""
    mid = emulate_tf32_kernel(r, w1, None, stride=1, pad=1, transposed=False, relu=True)
    out = emulate_tf32_kernel(mid, w2, None, stride=1, pad=0, transposed=False, skip=r,
                              operand=lambda a: mid_operand(a) if a is mid else tf32(a))
    return np.maximum(out, np.float32(0))


def _residual_inputs(seed=0, C=128, Cmid=32):
    rng = np.random.RandomState(seed)
    r = np.maximum(rng.standard_normal((1, C, 8, 8)), 0).astype(np.float32)
    w1 = (rng.standard_normal((Cmid, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
    w2 = (rng.standard_normal((C, Cmid, 1, 1)) / np.sqrt(Cmid)).astype(np.float32)
    return r, w1, w2


def test_emulated_residual_layer_is_within_bound_and_wrong_operands_are_not():
    """At K1 = 1152 the rigorous GEMM1 bound (about 4e-4 here) exceeds half a TF32 ulp of a typical mid value, so the
    interval of the kernel's GEMM2 operand spans a TF32 boundary for nearly every positive mid: the mid term absorbs
    about one TF32 ulp per mid value.  The bar still rejects bf16 operands and the plain float64 layer."""
    r, w1, w2 = _residual_inputs()
    c, bound, straddle = tf32_residual_ref(r, w1, w2)
    print("residual mid straddle share %.2f %%" % (100 * straddle))
    assert_within_bound(_emulate_residual(r, w1, w2), c, bound, "emulated residual layer")
    c_bf16, _, _ = tf32_residual_ref(r, w1, w2, operand=_bf16)
    c_plain, _, _ = tf32_residual_ref(r, w1, w2, operand=_identity)
    for what, y in (("bf16 operands", c_bf16), ("bf16 mid", _emulate_residual(r, w1, w2, mid_operand=_bf16)),
                    ("plain float64", c_plain)):
        with pytest.raises(AssertionError, match="above"):
            assert_within_bound(y, c, bound, "residual layer, " + what)
        print("residual layer, %s: %.1f %% of outputs above the bound" % (what, 100 * share_above_bound(y, c, bound)))


def test_tf32_truncates_and_ratio_handles_a_zero_bound():
    v = np.array([1 + 7 * 2.0 ** -13, -(1 + 7 * 2.0 ** -13), 3.0, 0.0], np.float32)
    assert tf32(v).tolist() == [1.0, -1.0, 3.0, 0.0]
    assert _tf32_rna(v).tolist() == [1 + 2.0 ** -10, -(1 + 2.0 ** -10), 3.0, 0.0]
    z = np.zeros(3)
    assert_within_bound(np.zeros(3), z, z, "exact zeros")
    with pytest.raises(AssertionError):
        assert_within_bound(np.array([0.0, 1e-30, 0.0]), z, z, "a zero bound admits only y == c")


# --------------------------------------------------------------------------- GPU
def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
def test_tcgen05_tf32_operand_conversion_truncates():
    """conv_tc 1x1 (Cin 32 -> Cout 16): one input channel holds +-(1 + 7 * 2^-13) and its weights are 1 (then the roles
    swapped).  Truncation to a 10-bit mantissa gives exactly +-1; round-to-nearest would give +-(1 + 2^-10)."""
    from vqvae_b200 import ops
    from vqvae_b200._lib import TF32
    v = np.float32(1 + 7 * 2.0 ** -13)
    sign = np.where(np.arange(64).reshape(1, 8, 8, 1) % 2 == 0, 1, -1).astype(np.float32)
    for role in ("x", "w"):
        x = np.zeros((1, 8, 8, 32), np.float32)
        w = np.zeros((16, 32, 1, 1), np.float32)
        if role == "x":
            x[..., 5:6] = v * sign
            w[:, 5] = 1
        else:
            x[..., 5:6] = sign
            w[:, 5] = v
        y = ops.conv2d(_cuda(x), ops.pack_conv_weight(_cuda(w), False), None, B=1, Cin=32, H=8, W=8, Cout=16, kh=1, kw=1,
                       stride=1, pad=0, precision=TF32).cpu().numpy()
        got = sorted(set(np.abs(y).ravel().tolist()))
        print("tf32 conversion probe (%s operand): |y| in %s" % (role, got))
        assert got == [1.0], got
        assert np.array_equal(y, np.broadcast_to(sign, y.shape))


def _run_conv(x, w, b, *, stride, pad, transposed, in_layout, out_layout, relu=False):
    from vqvae_b200 import ops
    from vqvae_b200._lib import NCHW, TF32
    B, Cin, H, W = x.shape
    Cout, k = (w.shape[1] if transposed else w.shape[0]), w.shape[2]
    xin = x if in_layout == NCHW else np.ascontiguousarray(x.transpose(0, 2, 3, 1))
    wp = ops.pack_conv_weight(_cuda(w), transposed)
    n0 = ops.launch_count()
    y = ops.conv2d(_cuda(xin), wp, _cuda(b), B=B, Cin=Cin, H=H, W=W, Cout=Cout,
                   kh=k, kw=k, stride=stride, pad=pad, transposed=transposed, in_layout=in_layout,
                   out_layout=out_layout, relu=relu, precision=TF32)
    assert ops.launch_count() - n0 == 1             # one tcgen05 launch (the FFMA path runs k4s2 phases one by one)
    y = y.cpu().numpy()
    return y if out_layout == NCHW else y.transpose(0, 3, 1, 2)


# The largest-K layer of each kernel family, without ReLU (a clamped output would hide the operand precision).
FAMILIES = [
    # family,        B, Cin, H,  W,  Cout, k, s, p, transposed, in, out
    ("conv_halo",    2, 128, 8, 8, 128, 3, 1, 1, False, 1, 1),      # E3, K = 1152
    ("conv_tc",      2, 64, 16, 16, 128, 4, 2, 1, False, 1, 1),     # E2, K = 1024
    ("conv_tc_k4s2T", 2, 128, 8, 8, 64, 4, 2, 1, True, 1, 1),       # D2, K = 512 per parity
    ("convt_shuffle", 2, 64, 16, 16, 3, 4, 2, 1, True, 1, 0),       # D3, K = 256 per parity
    ("conv_in_tc",   2, 3, 32, 32, 64, 4, 2, 1, False, 0, 1),       # E1, K = 48
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FAMILIES, ids=[f[0] for f in FAMILIES])
def test_plain_reference_breaks_the_bound_on_the_real_kernels(case):
    """The kernel is within the bound of the truncated-operand reference, and the plain float64 reference (untruncated
    operands) is not, on >= 20 % of outputs: the bar sees TF32 operand precision on this kernel."""
    family, B, Cin, H, W, Cout, k, stride, pad, transposed, lin, lout = case
    rng = np.random.RandomState(11)
    x = rng.standard_normal((B, Cin, H, W)).astype(np.float32)
    w = (rng.standard_normal((Cin, Cout, k, k) if transposed else (Cout, Cin, k, k)) / np.sqrt(Cin * k * k)).astype(np.float32)
    b = (rng.standard_normal(Cout) * 0.1).astype(np.float32)
    geo = dict(stride=stride, pad=pad, transposed=transposed)
    y = _run_conv(x, w, b, in_layout=lin, out_layout=lout, **geo)
    c, bound = tf32_layer_ref(x, w, b, **geo)
    assert_within_bound(y, c, bound, family)
    c_plain, _ = tf32_layer_ref(x, w, b, operand=_identity, **geo)
    share = share_above_bound(y, c_plain, bound)
    print("%s: plain float64 reference above the bound on %.1f %% of outputs" % (family, 100 * share))
    assert share >= 0.2, share


@pytest.mark.gpu
def test_plain_reference_breaks_the_residual_bound():
    from vqvae_b200 import ops
    from vqvae_b200._lib import TF32
    r, w1, w2 = _residual_inputs(seed=3)
    r = np.concatenate([r, np.maximum(np.random.RandomState(4).standard_normal(r.shape), 0).astype(np.float32)])
    p1, p2 = ops.pack_conv_weight(_cuda(w1), False), ops.pack_conv_weight(_cuda(w2), False)
    y = ops.residual_layer(_cuda(r.transpose(0, 2, 3, 1)), p1, p2, B=2, H=8, W=8, C=128, Cmid=32, relu_out=False,
                           precision=TF32).cpu().numpy().transpose(0, 3, 1, 2)
    c, bound, straddle = tf32_residual_ref(r, w1, w2, relu_out=False)
    print("res_tc: mid straddle share %.4f %%" % (100 * straddle))
    assert_within_bound(y, c, bound, "res_tc")
    # the mid term absorbs about one TF32 ulp of every positive mid value (test above): the plain float64 reference
    # breaks this bound on a smaller share (13-15 % in the CPU emulation) than a bf16-operand one (about 50 %)
    shares = {}
    for what, op in (("plain float64", _identity), ("bf16 operands", _bf16)):
        shares[what] = share_above_bound(y, tf32_residual_ref(r, w1, w2, relu_out=False, operand=op)[0], bound)
        print("res_tc: %s reference above the bound on %.1f %% of outputs" % (what, 100 * shares[what]))
    assert shares["plain float64"] >= 0.05 and shares["bf16 operands"] >= 0.2, shares
