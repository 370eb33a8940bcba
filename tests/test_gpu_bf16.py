"""VQB_BF16 path: the persistent tcgen05 kind::f16 kernels (hconv.cu, res_bf16.cu) against the C oracle.

Operands are rounded to bf16 (8-bit mantissa) and accumulated in fp32, so each kernel is compared with the oracle
evaluated on the SAME bf16-rounded inputs and weights: what is left is the fp32 accumulation order (~1e-5) plus, for
bf16 outputs, one rounding of the result (relative 2^-9).  Tolerances: bf16 outputs rtol 2^-8 + atol 2e-3, fp32
outputs atol 2e-4.  Needs a B200 (``-m gpu``).
"""
import numpy as np
import pytest
import torch

from oracle import cref

pytestmark = pytest.mark.gpu


def _bf(a):
    """Round an fp32 array to bf16 and back (the operand precision of the kernels)."""
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).float().numpy()


def _nhwc_bf16(x_nchw):
    return torch.from_numpy(np.ascontiguousarray(x_nchw.transpose(0, 2, 3, 1))).to(torch.bfloat16).cuda().contiguous()


def _run_layer(rng, B, Cin, H, W, Cout, k, stride, transposed, relu, out_f32):
    from vqvae_b200 import ops
    from vqvae_b200 import _lib
    x = _bf(rng.standard_normal((B, Cin, H, W)).astype(np.float32))
    wshape = (Cin, Cout, k, k) if transposed else (Cout, Cin, k, k)
    w = (rng.standard_normal(wshape) / np.sqrt(Cin * k * k)).astype(np.float32)
    b = (rng.standard_normal(Cout) * 0.1).astype(np.float32)
    pad = 0 if k == 1 else 1
    wq = _bf(w)
    ref = cref.conv_transpose2d(x, wq, b, stride, pad) if transposed else cref.conv2d(x, wq, b, stride, pad)
    if relu:
        ref = np.maximum(ref, 0)
    kind = ops.conv_kind(k, stride, transposed, Cout)
    assert kind is not None
    packed = ops.pack_conv_weight_bf16(torch.from_numpy(w).cuda(), kind)
    assert packed is not None
    y = ops.conv2d_bf16(_nhwc_bf16(x), packed, torch.from_numpy(b).cuda(), B=B, Cin=Cin, H=H, W=W, Cout=Cout, kind=kind,
                        relu=relu, out_f32=out_f32)
    torch.cuda.synchronize()
    y = y.float().cpu().numpy()
    if kind != _lib.CONVT_K4S2_OUT:
        y = y.transpose(0, 3, 1, 2)
    assert y.shape == ref.shape
    if out_f32 or kind == _lib.CONVT_K4S2_OUT:
        np.testing.assert_allclose(y, ref, atol=2e-4, rtol=1e-4)
    else:
        np.testing.assert_allclose(y, ref, atol=2e-3, rtol=2.0 ** -8)


BF16_LAYER_CASES = [
    # B, Cin, H, W, Cout, k, stride, transposed, relu, out_f32          (reference layer)
    (2, 128, 16, 32, 128, 3, 1, False, True, False),    # encoder.py:35-36, two M-tiles per weight stage
    (1, 128, 64, 64, 128, 3, 1, False, False, False),   # same at the cfg3 latent size (32 tiles)
    (3, 128, 8, 8, 128, 3, 1, False, True, False),      # cfg2 latent size: TW = 8, two images per tile
    (2, 64, 20, 36, 128, 3, 1, True, True, False),      # decoder.py:28-29, ragged tiles in x and y
    (2, 64, 32, 32, 128, 4, 2, False, True, False),     # encoder.py:32-34 (space-to-depth planes)
    (1, 64, 128, 128, 128, 4, 2, False, True, False),   # same, cfg3 size
    (3, 64, 16, 16, 128, 4, 2, False, False, False),    # cfg2 size
    (2, 128, 16, 16, 64, 4, 2, True, True, False),      # decoder.py:31-33: two passes, paired column parities
    (1, 128, 64, 64, 64, 4, 2, True, True, False),      # cfg3 size
    (3, 128, 8, 8, 64, 4, 2, True, False, False),       # cfg2 size
    (2, 128, 16, 32, 64, 1, 1, False, False, True),     # vqvae.py:16-17 -> fp32 z_e, resident weights
    (5, 128, 8, 8, 64, 1, 1, False, False, True),       # cfg2 size, ragged batch (5 images, 2 per tile)
    (2, 64, 32, 32, 3, 4, 2, True, False, True),        # decoder.py:34-35 -> fp32 NCHW, pixel shuffle
    (1, 64, 128, 128, 3, 4, 2, True, False, True),      # cfg3 size
    (3, 64, 16, 16, 3, 4, 2, True, True, True),         # cfg2 size (ReLU asked: the gather-form kernel)
    (2, 64, 20, 37, 3, 4, 2, True, False, True),        # scatter form (convt_out_bf16.cu), ragged 14x14 interiors, odd width
    (5, 64, 14, 14, 3, 4, 2, True, False, True),        # one exact tile per image
    (3, 64, 15, 29, 3, 4, 2, True, False, True),        # one-pixel remainders
    (1, 64, 12, 20, 48, 3, 1, False, True, False),      # Cout = 48 (16-column tail group), ragged
    (1, 256, 16, 16, 64, 3, 1, False, False, False),    # four 64-channel chunks
]


@pytest.mark.parametrize("case", BF16_LAYER_CASES)
def test_bf16_conv_layers_vs_oracle(case):
    rng = np.random.RandomState(abs(hash(case)) % (2 ** 31))
    _run_layer(rng, *case)


def test_bf16_conv_many_tiles_persistent_loop():
    """More tiles than SMs: every CTA walks several tiles (ring wrap-around, TMEM double buffering)."""
    rng = np.random.RandomState(7)
    _run_layer(rng, 8, 128, 64, 64, 128, 3, 1, False, True, False)        # 512 tiles of 256 pixels
    _run_layer(rng, 4, 128, 64, 64, 64, 4, 2, True, True, False)          # 2 passes x 256 tiles


def test_bf16_kernels_back_to_back_launches():
    """40 launches of each persistent kernel enqueued without a host sync (programmatic dependent launch lets a launch start
    while its predecessor drains): every launch must give the first launch's bits.  Written after a two-issuer variant of
    the residual kernel passed all single-launch tests and faulted about once in thirty launches (r02_hconv_notes.txt)."""
    from vqvae_b200 import ops, _lib
    g = torch.Generator(device="cuda").manual_seed(5)
    B, L = 48, 64
    jobs = []

    def conv(Cin, H, W, Cout, k, stride, transposed, out_f32=False, relu=True):
        x = torch.randn((B, H, W, Cin), device="cuda", generator=g).to(torch.bfloat16)
        wshape = (Cin, Cout, k, k) if transposed else (Cout, Cin, k, k)
        w = torch.randn(wshape, device="cuda", generator=g) / np.sqrt(Cin * k * k)
        b = torch.randn((Cout,), device="cuda", generator=g) * 0.1
        kind = ops.conv_kind(k, stride, transposed, Cout)
        pk = ops.pack_conv_weight_bf16(w, kind)
        jobs.append(lambda: ops.conv2d_bf16(x, pk, b, B=B, Cin=Cin, H=H, W=W, Cout=Cout, kind=kind, relu=relu, out_f32=out_f32))

    conv(64, 2 * L, 2 * L, 128, 4, 2, False)          # E2
    conv(128, L, L, 128, 3, 1, False)                 # E3 (two MMA issuer warps, streamed weights)
    conv(64, L, L, 128, 3, 1, True)                   # D1
    conv(128, L, L, 64, 4, 2, True)                   # D2 (two passes)
    conv(128, L, L, 64, 1, 1, False, True, False)     # pre-quant 1x1 (resident weights)
    conv(64, 2 * L, 2 * L, 3, 4, 2, True, True, False)  # D3, scatter form
    r = torch.randn((B, L, L, 128), device="cuda", generator=g).clamp_min(0).to(torch.bfloat16)
    w1 = torch.randn((32, 128, 3, 3), device="cuda", generator=g) / np.sqrt(1152)
    w2 = torch.randn((128, 32, 1, 1), device="cuda", generator=g) / np.sqrt(32)
    p1, p2 = ops.pack_conv_weight_bf16(w1, _lib.CONV_K3), ops.pack_conv_weight_bf16(w2, _lib.RES_W2)
    jobs.append(lambda: ops.residual_layer_bf16(r, p1, p2, B=B, H=L, W=L, C=128, Cmid=32, relu_out=True))
    xi = torch.rand((B, 3, 4 * L, 4 * L), device="cuda", generator=g) * 2 - 1
    wi = ops.pack_conv_weight(torch.randn((64, 3, 4, 4), device="cuda", generator=g) / 7, False)
    bi = torch.zeros((64,), device="cuda")
    jobs.append(lambda: ops.conv_in_bf16(xi, wi, bi, B=B, H=4 * L, W=4 * L, Cout=64))
    for job in jobs:
        outs = [job() for _ in range(40)]
        torch.cuda.synchronize()
        for o in outs[1:]:
            assert torch.equal(o, outs[0])
        del outs


@pytest.mark.parametrize("B,H,W,C,Cmid,relu_out", [(2, 16, 32, 128, 32, True), (1, 64, 64, 128, 32, True), (3, 8, 8, 128, 32, True),
                                                   (2, 20, 36, 128, 32, False), (5, 8, 8, 64, 16, True), (6, 64, 64, 128, 32, True)])
def test_bf16_residual_layer_vs_oracle(B, H, W, C, Cmid, relu_out):
    """res_bf16.cu: out = act(r + W2.relu(W1 (*) r)) with bf16 operands; the intermediate relu(W1 (*) r) is rounded
    to bf16 before the second GEMM (it is that GEMM's A operand), which the oracle side mirrors."""
    from vqvae_b200 import ops, _lib
    rng = np.random.RandomState(B * 1000 + H * 100 + C)
    r = _bf(np.maximum(rng.standard_normal((B, C, H, W)).astype(np.float32), 0))
    w1 = (rng.standard_normal((Cmid, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
    w2 = (rng.standard_normal((C, Cmid, 1, 1)) / np.sqrt(Cmid)).astype(np.float32)
    mid = _bf(np.maximum(cref.conv2d(r, _bf(w1), None, 1, 1), 0))
    ref = r + cref.conv2d(mid, _bf(w2), None, 1, 0)
    if relu_out:
        ref = np.maximum(ref, 0)
    p1 = ops.pack_conv_weight_bf16(torch.from_numpy(w1).cuda(), _lib.CONV_K3)
    p2 = ops.pack_conv_weight_bf16(torch.from_numpy(w2).cuda(), _lib.RES_W2)
    y = ops.residual_layer_bf16(_nhwc_bf16(r), p1, p2, B=B, H=H, W=W, C=C, Cmid=Cmid, relu_out=relu_out)
    torch.cuda.synchronize()
    y = y.float().cpu().numpy().transpose(0, 3, 1, 2)
    # a mid value that sits on a bf16 rounding boundary may round the other way (fp32 accumulation order): one such
    # flip moves an output by 2^-9 |mid| |w2| ~ 1e-3, hence the absolute term
    np.testing.assert_allclose(y, ref, atol=6e-3, rtol=2.0 ** -7)


# --------------------------------------------------------------------------- whole model, VQB_BF16 pipeline
# The reference reaches bf16 only through torch.autocast(dtype=torch.bfloat16) (SURVEY Q6).  Run that way on the CPU
# it differs from its own fp32 forward by (measured in the authoring container, unmodified reference):
#   z_e max-abs 0.8-0.9e-3;  index flips 0 % (cifar_spread), 0.9 % (cfg3_s256), 1.0 % (k1024_s64), 3.1 % (cifar_default,
#   the near-tie stress init);  x_hat max-abs 0.7e-3 without flips, up to 1e-2 around flipped latents.
# Bars for this pipeline (bf16 operands + bf16 activations between layers, fp32 accumulation, fp32 z_e, exact VQ):
#   z_e within 2.5e-3 abs of the reference's fp32 z_e; VQ bit-exact ON THE PIPELINE'S OWN z_e (every flip is explained
#   by the z_e perturbation); flips vs the fp32 reference <= 4 %; x_hat within 3e-3 abs of the fp32 oracle decoder run
#   on the pipeline's own codes.
@pytest.mark.parametrize("name", ["cifar_spread", "cifar_default", "k1024_s64", "cfg3_s256"])
def test_bf16_model_forward_tolerance(name):
    import vqvae_b200
    from tests.helpers import build_model, load_golden, model_case_inputs, window
    g = load_golden(name)
    hp, sd, x = model_case_inputs(g["case"])
    m = build_model(hp, sd)
    xc = torch.from_numpy(x).cuda()
    E = sd["vector_quantization.embedding.weight"]
    with vqvae_b200.precision("bf16"):
        assert m._bf16_pipeline()
        z_e, B, H, W = m._encode_rows(xc, True)
        loss, x_hat, perp = m(xc)
    torch.cuda.synchronize()
    z_rows = z_e.reshape(-1, hp["embedding_dim"]).cpu().numpy()
    z_nchw = z_rows.reshape(B, H, W, -1).transpose(0, 3, 1, 2)
    np.testing.assert_allclose(window(z_nchw, g["case"]), g["z_e"], atol=2.5e-3, rtol=0)
    idx = m.last_min_encoding_indices.cpu().numpy().ravel()
    o = cref.vq_rows(z_rows, E)
    assert np.array_equal(idx, o["idx"])                         # bit-exact at the VQ boundary, on our own z_e
    flips = float((idx != g["idx"].ravel()).mean())
    assert flips <= 0.04, flips
    # decoder: fp32 oracle on the codes this forward chose (z_q = z + (e - z) ~ e to 1 ulp)
    zq = np.ascontiguousarray(o["zq"].reshape(B, H, W, -1).transpose(0, 3, 1, 2))
    xh_ref = cref.decoder(zq, sd, hp["n_res_layers"])
    np.testing.assert_allclose(x_hat.cpu().numpy(), xh_ref, atol=3e-3, rtol=0)
    assert x_hat.dtype == torch.float32 and x_hat.shape == x.shape
    np.testing.assert_allclose(loss.item(), 1.25 * o["sse"] / z_rows.size, rtol=1e-5)
    if flips == 0.0:
        np.testing.assert_allclose(window(x_hat.cpu().numpy(), g["case"]), g["x_hat"], atol=3e-3, rtol=0)


@pytest.mark.parametrize("B,H,W,relu", [(2, 256, 256, True), (5, 32, 32, True), (3, 64, 64, False), (2, 16, 16, True), (1, 12, 20, True), (300, 32, 32, True)])
def test_bf16_input_conv_vs_oracle(B, H, W, relu):
    """encoder.py:29-31 in the bf16 pipeline: fp32 NCHW image -> bf16 NHWC.  The 48-tap contraction runs as kind::tf32 on the
    fp32 pixels (operands truncated to 10-bit mantissas), the result is rounded once to bf16: within the TF32 layer bound
    rho(48) S of tests/helpers.py plus the bf16 rounding.  bf16 keeps 8 significant bits, so rounding to nearest moves
    a value in [2^e, 2^(e+1)) by at most half an ulp, 2^(e-8) <= 2^-8 |y| (the rounded y never drops below 2^e)."""
    from vqvae_b200 import ops
    from tests.helpers import assert_within_bound, tf32_layer_ref
    rng = np.random.RandomState(B + H)
    x = (2 * rng.random_sample((B, 3, H, W)) - 1).astype(np.float32)
    w = (rng.standard_normal((64, 3, 4, 4)) / 7).astype(np.float32)
    b = (rng.standard_normal(64) * 0.1).astype(np.float32)
    y = ops.conv_in_bf16(torch.from_numpy(x).cuda(), ops.pack_conv_weight(torch.from_numpy(w).cuda(), False), torch.from_numpy(b).cuda(),
                         B=B, H=H, W=W, Cout=64, relu=relu)
    torch.cuda.synchronize()
    y = y.float().cpu().numpy().transpose(0, 3, 1, 2)
    c, bound = tf32_layer_ref(x, w, b, stride=2, pad=1, relu=relu)
    assert_within_bound(y, c, bound + 2.0 ** -8 * np.abs(y), "conv_in_bf16 %s" % ((B, H, W),))
