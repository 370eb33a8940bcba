"""Parity of the CUDA path (through the C ABI) against the oracle and the committed
golden vectors of the unmodified reference.  Needs a B200: run with ``-m gpu``.

Bars: integer / index outputs bit-exact; fp32 z_q bitwise at the VQ boundary; fp32
conv outputs within 2e-6 absolute of the double-accumulated oracle at |y| = O(1e-1)
(fp32 FFMA path); scalars within 2e-5 relative.
"""
import numpy as np
import pytest
import torch

from oracle import cref
from tests.helpers import (MODEL_CASES, VQ_CASES, assert_zq_matches, build_model, expected_zq, load_golden,
                           make_vq_inputs, model_case_inputs, window)

pytestmark = pytest.mark.gpu

# The tcgen05 VQ kernel sums (e - z)^2 of one row in four fp32 partials (64 terms) and adds rows in double; the FFMA kernel and
# the oracle add every term in double.  Per-row relative error <= 16 * 2^-24 ~ 1e-6, random in sign across rows.
SSE_RTOL = 2e-6

CONV_ATOL = 2e-6     # fp32 FFMA vs double-accumulated oracle, activations O(0.1..1)


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# --------------------------------------------------------------------------- VQ kernel
@pytest.mark.parametrize("name", sorted(VQ_CASES))
def test_vq_kernel_bit_exact_vs_oracle_and_reference(name):
    from vqvae_b200 import ops
    g = load_golden(name)
    z, E = make_vq_inputs(**g["case"])
    B, D, H, W = z.shape
    rows = np.ascontiguousarray(z.transpose(0, 2, 3, 1)).reshape(-1, D)
    o = cref.vq_rows(rows, E)
    idx, zq, sse, hist = ops.vq_forward(_cuda(rows), _cuda(E))
    loss, perp = ops.vq_finish(sse, hist, rows.shape[0], E.shape[0], D, 0.25)
    torch.cuda.synchronize()
    assert idx.dtype == torch.int64
    assert np.array_equal(idx.cpu().numpy(), o["idx"])                       # vs oracle
    assert np.array_equal(idx.cpu().numpy(), g["idx"].ravel())               # vs reference
    assert np.array_equal(zq.cpu().numpy(), o["zq"], equal_nan=True)         # bitwise vs oracle
    assert_zq_matches(g, zq.cpu().numpy().reshape(B, H, W, D).transpose(0, 3, 1, 2))   # bitwise vs reference
    assert np.array_equal(hist.cpu().numpy(), g["hist"])
    np.testing.assert_allclose(sse.item(), o["sse"], rtol=SSE_RTOL, equal_nan=True)
    np.testing.assert_allclose(loss.item(), g["loss"], rtol=1e-6, equal_nan=True)
    np.testing.assert_allclose(perp.item(), g["perplexity"], rtol=2e-5)


def test_vq_module_five_tuple_matches_reference():
    from models.quantizer import VectorQuantizer
    g = load_golden("vq_k512_d64")
    z, E = make_vq_inputs(**g["case"])
    vq = VectorQuantizer(512, 64, 0.25)
    vq.embedding.weight.data.copy_(torch.from_numpy(E))
    vq = vq.cuda()
    with torch.enable_grad():                  # grad mode + a trainable codebook: the differentiable path, like the reference
        loss, z_q, perp, onehot, idx = vq(_cuda(z))
    assert idx.shape == (z.shape[0] * z.shape[2] * z.shape[3], 1) and idx.dtype == torch.int64
    assert np.array_equal(idx.cpu().numpy(), g["idx"])
    assert z_q.shape == z.shape and z_q.is_contiguous()
    assert z_q.requires_grad
    assert np.array_equal(z_q.detach().cpu().numpy(), g["z_q"])
    assert onehot.shape == (idx.shape[0], 512) and onehot.dtype == torch.float32
    oh = onehot.cpu().numpy()
    assert np.array_equal(oh.argmax(1), g["idx"].ravel()) and np.all(oh.sum(1) == 1.0)
    assert np.array_equal(oh.sum(0).astype(np.int32), g["hist"])
    np.testing.assert_allclose(loss.item(), g["loss"], rtol=1e-6)
    np.testing.assert_allclose(perp.item(), g["perplexity"], rtol=2e-5)


def test_vq_rejects_wrong_channel_count_and_cpu_tensor():
    from models.quantizer import VectorQuantizer
    vq = VectorQuantizer(16, 8, 0.25).cuda()
    with pytest.raises(RuntimeError):
        vq(torch.zeros(1, 4, 2, 2, device="cuda"))
    with pytest.raises(RuntimeError):
        vq(torch.zeros(1, 8, 2, 2))          # CPU tensor: no CPU fallback


@pytest.mark.parametrize("N,K,D", [(1, 1, 4), (63, 65, 12), (64, 64, 64), (65, 129, 32), (1000, 513, 256)])
def test_vq_ragged_sizes(N, K, D):
    from vqvae_b200 import ops
    rng = np.random.RandomState(N + K + D)
    rows = rng.standard_normal((N, D)).astype(np.float32)
    E = rng.standard_normal((K, D)).astype(np.float32)
    o = cref.vq_rows(rows, E)
    idx, zq, sse, hist = ops.vq_forward(_cuda(rows), _cuda(E))
    assert np.array_equal(idx.cpu().numpy(), o["idx"])
    assert np.array_equal(zq.cpu().numpy(), o["zq"])
    assert np.array_equal(hist.cpu().numpy(), o["hist"])


# --------------------------------------------------------------------------- conv layers
def _conv_case(rng, B, Cin, H, W, Cout, k, stride, pad, transposed, in_layout, out_layout, relu, skip,
               precision=0, atol=5e-6, rtol=1e-5):
    from vqvae_b200 import ops
    from vqvae_b200._lib import NCHW
    x = rng.standard_normal((B, Cin, H, W)).astype(np.float32)
    wshape = (Cin, Cout, k, k) if transposed else (Cout, Cin, k, k)
    w = (rng.standard_normal(wshape) / np.sqrt(Cin * k * k)).astype(np.float32)
    b = rng.standard_normal(Cout).astype(np.float32) * 0.1
    ref = cref.conv_transpose2d(x, w, b, stride, pad) if transposed else cref.conv2d(x, w, b, stride, pad)
    sk = None
    if skip:
        sk = rng.standard_normal(ref.shape).astype(np.float32)
        ref = ref + sk
    if relu:
        ref = np.maximum(ref, 0)
    xin = x if in_layout == NCHW else np.ascontiguousarray(x.transpose(0, 2, 3, 1))
    wp = ops.pack_conv_weight(_cuda(w), transposed)
    y = ops.conv2d(_cuda(xin), wp, _cuda(b), B=B, Cin=Cin, H=H, W=W, Cout=Cout, kh=k, kw=k,
                   stride=stride, pad=pad, transposed=transposed, in_layout=in_layout,
                   out_layout=out_layout, relu=relu, precision=precision,
                   skip=_cuda(np.ascontiguousarray(sk.transpose(0, 2, 3, 1))) if skip else None)
    y = y.cpu().numpy()
    if out_layout != NCHW:
        y = y.transpose(0, 3, 1, 2)
    assert y.shape == ref.shape
    np.testing.assert_allclose(y, ref, atol=atol, rtol=rtol)


CONV_CASES = [
    # B, Cin, H,  W,  Cout, k, s, p, transposed, in, out, relu, skip     (reference layer)
    (2, 3, 32, 32, 64, 4, 2, 1, False, 0, 1, True, False),     # encoder.py:29-31, NCHW in
    (2, 64, 16, 16, 128, 4, 2, 1, False, 1, 1, True, False),   # encoder.py:32-34
    (2, 128, 8, 8, 128, 3, 1, 1, False, 1, 1, False, False),   # encoder.py:35-36
    (2, 128, 8, 8, 32, 3, 1, 1, False, 1, 1, True, False),     # residual.py:20-22
    (2, 32, 8, 8, 128, 1, 1, 0, False, 1, 1, True, True),      # residual.py:23-24,28 (+skip)
    (2, 128, 8, 8, 64, 1, 1, 0, False, 1, 1, False, False),    # vqvae.py:16-17
    (2, 128, 8, 8, 64, 1, 1, 0, False, 0, 0, False, False),    # same, NCHW in/out (piecewise API)
    (2, 64, 8, 8, 128, 3, 1, 1, True, 1, 1, False, False),     # decoder.py:28-29
    (2, 128, 8, 8, 64, 4, 2, 1, True, 1, 1, True, False),      # decoder.py:31-33
    (2, 64, 16, 16, 3, 4, 2, 1, True, 1, 0, False, False),     # decoder.py:34-35, NCHW out
    (3, 5, 7, 9, 6, 3, 1, 1, False, 0, 0, False, False),       # odd everything
    (1, 8, 5, 6, 10, 4, 2, 1, True, 1, 1, True, False),        # odd transposed
    (1, 12, 6, 5, 2, 3, 1, 1, True, 1, 0, False, False),       # small-Cout kernel, k3
    (2, 6, 9, 7, 3, 4, 2, 1, True, 0, 0, False, False),        # Cout=3 from NCHW input
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_layers_vs_oracle(case):
    rng = np.random.RandomState(abs(hash(case)) % (2 ** 31))
    _conv_case(rng, *case)


# tcgen05 implicit-GEMM path (VQB_TF32): operands truncated to TF32 (rel. 2^-10 each),
# fp32 accumulation -> |err| <= 2^-9 * sum|x||w| ~ 2e-3 * O(1) per output at these scales.
TC_CONV_CASES = [
    (2, 64, 16, 16, 128, 4, 2, 1, False, 1, 1, True, False),   # encoder.py:32-34 (element-strided TMA)
    (2, 128, 8, 8, 128, 3, 1, 1, False, 1, 1, False, False),   # encoder.py:35-36
    (2, 128, 8, 8, 32, 3, 1, 1, False, 1, 1, True, False),     # residual.py:20-22
    (2, 32, 8, 8, 128, 1, 1, 0, False, 1, 1, True, True),      # residual.py:23-24,28 (+skip)
    (2, 128, 8, 8, 64, 1, 1, 0, False, 1, 1, False, False),    # vqvae.py:16-17
    (2, 64, 8, 8, 128, 3, 1, 1, True, 1, 1, False, False),     # decoder.py:28-29
    (2, 128, 8, 8, 64, 4, 2, 1, True, 1, 1, True, False),      # decoder.py:31-33 (4 phases)
    (3, 64, 5, 7, 48, 3, 1, 1, False, 1, 1, True, False),      # ragged tile: masked rows, Cout=48
    (1, 32, 20, 36, 16, 3, 1, 1, False, 1, 1, False, False),   # multi-tile in x and y, Cout=16
    (5, 96, 4, 4, 64, 4, 2, 1, True, 1, 1, False, False),      # small image, 3 k-chunks, BN=8 tile
    (1, 32, 33, 17, 32, 4, 2, 1, False, 1, 1, False, False),   # odd sizes, stride 2
    (2, 64, 16, 16, 3, 4, 2, 1, True, 1, 0, False, False),     # decoder.py:34-35: 3x3-neighbourhood GEMM + pixel shuffle
    (1, 32, 5, 9, 2, 4, 2, 1, True, 1, 0, True, False),        # same, ragged tile, Cout=2
    (2, 3, 32, 32, 64, 4, 2, 1, False, 0, 1, True, False),     # encoder.py:29-31: hand-built im2col tile
    (3, 3, 12, 20, 128, 4, 2, 1, False, 0, 1, False, False),   # same, partial last tile, Cout=128 (generic gather)
    (3, 3, 64, 64, 64, 4, 2, 1, False, 0, 1, True, False),     # staged-rows fast path, 4 output rows per tile
    (1, 3, 8, 256, 64, 4, 2, 1, False, 0, 1, False, False),    # fast path, one output row per tile (OW = 128)
    (5, 3, 16, 16, 64, 4, 2, 1, False, 0, 1, True, False),     # tile straddles images: generic gather + TMA store
    (2, 3, 32, 32, 128, 4, 2, 1, False, 0, 1, True, False),    # fast path, Cout=128 (direct stores)
    (3, 3, 6, 8, 64, 4, 2, 1, False, 0, 1, True, False),       # partial tile (36 pixels), TMA store clips
]


def test_tf32_full_size_properties_cfg2():
    """BASELINE cfg2 at its full size (B=256, 32x32, K=512) in the default VQB_TF32 mode, through size-independent
    properties: (1) the VQ step is bit-exact on the z_e the TF32 encoder produced (C oracle on all 16384 rows);
    (2) z_e is within 1e-3 of the all-fp32 product forward (itself oracle-checked at small sizes); (3) the share of
    min_encoding_indices that differ from the all-fp32 forward stays below 0.5 %; (4) the decoder output is within
    1.5e-3 of the fp32 decoder run on the SAME codes."""
    import vqvae_b200
    from vqvae_b200.synth import make_images, make_state_dict
    hp = dict(h_dim=128, res_h_dim=32, n_res_layers=2, n_embeddings=512, embedding_dim=64)
    sd = make_state_dict(seed=0, codebook="normal", codebook_scale=0.05, **hp)
    m = build_model(hp, sd)
    x = _cuda(make_images(256, 32, seed=1))
    with vqvae_b200.precision("fp32"):
        ze32, B, H, W = m._encode_rows(x.clone())
        m(x.clone())
        idx32 = m.last_min_encoding_indices.clone()
    with vqvae_b200.precision("tf32"):
        ze, B, H, W = m._encode_rows(x.clone())
        loss, x_hat, perp = m(x.clone())
        idx = m.last_min_encoding_indices.clone()
    assert (ze - ze32).abs().max().item() <= 1e-3
    rows = ze.reshape(-1, 64).cpu().numpy()
    o = cref.vq_rows(rows, sd["vector_quantization.embedding.weight"])
    assert np.array_equal(idx.cpu().numpy().ravel(), o["idx"])
    np.testing.assert_allclose(loss.item(), 1.25 * o["sse"] / rows.size, rtol=1e-5)
    flips = float((idx != idx32).float().mean().item())
    assert flips <= 0.005, flips
    with vqvae_b200.precision("fp32"):
        xh32 = m.decoder(_cuda(np.ascontiguousarray(o["zq"].reshape(B, H, W, 64).transpose(0, 3, 1, 2))))
    assert (x_hat - xh32).abs().max().item() <= 1.5e-3
    print("cfg2 full size tf32: flips vs fp32 %.4f %%" % (100 * flips))


@pytest.mark.parametrize("case", TC_CONV_CASES)
def test_tc_conv_layers_vs_oracle(case):
    from vqvae_b200._lib import TF32
    rng = np.random.RandomState(abs(hash(case)) % (2 ** 31))
    _conv_case(rng, *case, precision=TF32, atol=4e-3, rtol=2e-3)


def test_tc_model_forward_tf32_tolerance():
    """Whole forward in VQB_TF32 mode vs the reference golden: x_hat within 5e-4 abs
    (SURVEY 8c: TF32 convs give 1-2e-4), index flips below 0.5 % (0.02-0.13 % observed)."""
    import vqvae_b200
    for name in ("cifar_default", "cifar_spread", "k1024_s64"):
        g = load_golden(name)
        hp, sd, x = model_case_inputs(g["case"])
        m = build_model(hp, sd)
        with vqvae_b200.precision("tf32"):
            loss, x_hat, perp = m(_cuda(x))
        idx = m.last_min_encoding_indices.cpu().numpy()
        nflip = int((idx != g["idx"]).sum())
        flips = nflip / idx.size
        assert nflip <= max(3, int(0.005 * idx.size)), (name, nflip, idx.size)   # 256..512 rows: 1 flip = 0.2-0.4 %
        if flips == 0.0:
            np.testing.assert_allclose(x_hat.cpu().numpy(), g["x_hat"], atol=5e-4, rtol=0)
        np.testing.assert_allclose(loss.item(), g["loss"], rtol=2e-2)


# --------------------------------------------------------------------------- whole path
@pytest.mark.parametrize("name", sorted(MODEL_CASES))
def test_vqvae_forward_vs_reference_golden(name):
    g = load_golden(name)
    hp, sd, x = model_case_inputs(g["case"])
    m = build_model(hp, sd)
    xc = _cuda(x)
    # piecewise API the notebook uses (visualization.ipynb cell 1 `reconstruct`)
    z_e = m.pre_quantization_conv(m.encoder(xc.clone()))
    np.testing.assert_allclose(window(z_e.cpu().numpy(), g["case"]), g["z_e"], atol=CONV_ATOL, rtol=0)
    # VQ boundary: the reference's own z_e in -> bit-exact indices, bitwise z_q
    loss_b, zq_b, perp_b, _, idx_b = m.vector_quantization(_cuda(g["z_e"]))
    assert np.array_equal(idx_b.cpu().numpy(), g["vq_idx"])
    E_np = sd["vector_quantization.embedding.weight"]
    assert_zq_matches(g, zq_b.cpu().numpy(), E_np)
    np.testing.assert_allclose(loss_b.item(), g["vq_loss"], rtol=1e-5)
    np.testing.assert_allclose(perp_b.item(), g["vq_perplexity"], rtol=2e-5)
    # decoder on the reference's z_q
    xh_b = m.decoder(_cuda(expected_zq(g, E_np)))
    np.testing.assert_allclose(xh_b.cpu().numpy(), g["dec_x_hat"], atol=CONV_ATOL, rtol=0)
    # fused forward
    loss, x_hat, perp = m(xc)
    idx = m.last_min_encoding_indices.cpu().numpy()
    mism = int((idx != g["idx"]).sum())
    if mism:
        # an end-to-end flip is only acceptable on a provable near-tie of the oracle's
        # fp64 distances computed from OUR z_e (SURVEY 7.3.2)
        rows = z_e.permute(0, 2, 3, 1).reshape(-1, hp["embedding_dim"]).double().cpu().numpy()
        E = sd["vector_quantization.embedding.weight"].astype(np.float64)
        d = (rows ** 2).sum(1, keepdims=True) + (E ** 2).sum(1) - 2 * rows @ E.T
        bad = np.nonzero((idx != g["idx"]).ravel())[0]
        gap = np.abs(d[bad, idx.ravel()[bad]] - d[bad, g["idx"].ravel()[bad]])
        assert np.all(gap <= 4 * np.spacing(np.float32(np.abs(d[bad]).max()))), (mism, gap)
    assert mism <= max(1, idx.size // 1000)
    if mism == 0:
        np.testing.assert_allclose(window(x_hat.cpu().numpy(), g["case"]), g["x_hat"], atol=CONV_ATOL, rtol=0)
        np.testing.assert_allclose(loss.item(), g["loss"], rtol=1e-5)
        np.testing.assert_allclose(perp.item(), g["perplexity"], rtol=2e-5)
    assert x_hat.shape == x.shape and x_hat.is_contiguous() and x_hat.dtype == torch.float32


def test_encode_decode_entry_points_match_forward():
    g = load_golden("cifar_spread")
    hp, sd, x = model_case_inputs(g["case"])
    m = build_model(hp, sd)
    xc = _cuda(x)
    _, x_hat, _ = m(xc)
    idx = m.encode(xc)
    assert torch.equal(idx, m.last_min_encoding_indices)
    x_dec = m.decode(idx, (x.shape[2] // 4, x.shape[3] // 4))
    # decode() feeds E[idx]; forward feeds z + (E[idx] - z): differ by <= 1 ulp of z_q (Q4)
    np.testing.assert_allclose(x_dec.cpu().numpy(), x_hat.cpu().numpy(), atol=1e-6, rtol=0)


def test_residual_layer_in_place_relu_and_shared_weights():
    """SURVEY Q1/Q2: the caller's tensor is ReLU'd in place; the stack shares one layer."""
    from models.residual import ResidualLayer, ResidualStack
    rng = np.random.RandomState(3)
    x = rng.standard_normal((2, 16, 5, 6)).astype(np.float32)
    layer = ResidualLayer(16, 16, 8).cuda()
    w1 = layer.res_block[1].weight.detach().cpu().numpy()
    w2 = layer.res_block[3].weight.detach().cpu().numpy()
    xc = _cuda(x)
    y = layer(xc)
    r = np.maximum(x, 0)
    ref = r + cref.conv2d(np.maximum(cref.conv2d(r, w1, None, 1, 1), 0), w2, None, 1, 0)
    np.testing.assert_allclose(y.cpu().numpy(), ref, atol=5e-6)
    assert np.array_equal(xc.cpu().numpy(), r)            # mutated like nn.ReLU(True)
    st = ResidualStack(16, 16, 8, 3).cuda()
    assert st.stack[0] is st.stack[1] is st.stack[2]
    w1 = st.stack[0].res_block[1].weight.detach().cpu().numpy()
    w2 = st.stack[0].res_block[3].weight.detach().cpu().numpy()
    y = st(_cuda(x))
    np.testing.assert_allclose(y.cpu().numpy(), cref.residual_stack(x, w1, w2, 3), atol=1e-5)


def test_verbose_path_prints_and_asserts(capsys):
    g = load_golden("no_res")
    hp, sd, x = model_case_inputs(g["case"])
    m = build_model(hp, sd)
    with pytest.raises(AssertionError):
        m(_cuda(x), verbose=True)
    out = capsys.readouterr().out
    assert "original data shape" in out and "encoded data shape" in out and "recon data shape" in out


# ------------------------------------------------------- full-size properties (cfg2)
def test_full_size_properties_cfg2():
    """BASELINE cfg2 (B=256, 32x32, K=512, D=64): size-independent properties."""
    from oracle.weights import make_images, make_state_dict
    hp = dict(h_dim=128, res_h_dim=32, n_res_layers=2, n_embeddings=512, embedding_dim=64)
    sd = make_state_dict(seed=0, codebook="normal", codebook_scale=0.05, **hp)
    m = build_model(hp, sd)
    x = _cuda(make_images(256, 32, seed=1))
    loss, x_hat, perp = m(x)
    idx = m.last_min_encoding_indices
    N = 256 * 8 * 8
    assert idx.shape == (N, 1) and int(idx.min()) >= 0 and int(idx.max()) < 512
    # batch independence: a slice of the batch gives the slice of the outputs, bitwise
    loss_h, x_hat_h, _ = m(x[64:128].contiguous())
    assert torch.equal(x_hat_h, x_hat[64:128])
    assert torch.equal(m.last_min_encoding_indices, idx.view(256, 64)[64:128].reshape(-1, 1))
    # idempotence: quantising z_q again returns the same codes
    z_e = m.pre_quantization_conv(m.encoder(x.clone()))
    l1, zq1, p1, _, i1 = m.vector_quantization(z_e)
    assert torch.equal(i1, idx)
    l2, zq2, p2, _, i2 = m.vector_quantization(zq1)
    assert torch.equal(i2, i1)
    # straight-through value is within 1 ulp of the gathered code (Q4)
    E = m.vector_quantization.embedding.weight
    e = E[i1.view(-1)].view(256, 8, 8, 64).permute(0, 3, 1, 2)
    assert float((zq1 - e).abs().max()) <= 1.5e-8 * 4
    # loss = (1+beta) * mse(e, z_e) and perplexity from the histogram of idx
    mse = ((e - z_e).double() ** 2).mean().item()
    np.testing.assert_allclose(loss.item(), 1.25 * mse, rtol=1e-5)
    p = torch.bincount(idx.view(-1), minlength=512).double() / N
    np.testing.assert_allclose(perp.item(), float(torch.exp(-(p * torch.log(p + 1e-10)).sum())), rtol=1e-5)
    # oracle spot check of the first 4 images at full depth
    o = cref.vqvae_forward(x[:4].cpu().numpy(), sd, 2)
    np.testing.assert_allclose(x_hat[:4].cpu().numpy(), o["x_hat"], atol=CONV_ATOL, rtol=0)
    assert np.array_equal(idx.view(256, 64)[:4].reshape(-1, 1).cpu().numpy(), o["idx"])


@pytest.mark.parametrize("B,H,W,C,Cmid,relu_out", [(2, 8, 8, 128, 32, True), (3, 5, 7, 64, 32, False),
                                                   (1, 20, 36, 128, 64, True), (5, 4, 4, 32, 32, True)])
def test_fused_residual_layer_tc_vs_oracle(B, H, W, C, Cmid, relu_out):
    """res_tc.cu (one tcgen05 kernel, two chained GEMMs) vs residual.py:18-29 semantics."""
    from vqvae_b200 import ops
    from vqvae_b200._lib import FP32, TF32
    rng = np.random.RandomState(B * 1000 + H * 100 + C)
    r = np.maximum(rng.standard_normal((B, C, H, W)).astype(np.float32), 0)       # r = relu(x)
    w1 = (rng.standard_normal((Cmid, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
    w2 = (rng.standard_normal((C, Cmid, 1, 1)) / np.sqrt(Cmid)).astype(np.float32)
    ref = r + cref.conv2d(np.maximum(cref.conv2d(r, w1, None, 1, 1), 0), w2, None, 1, 0)
    if relu_out:
        ref = np.maximum(ref, 0)
    rn = _cuda(np.ascontiguousarray(r.transpose(0, 2, 3, 1)))
    p1, p2 = ops.pack_conv_weight(_cuda(w1), False), ops.pack_conv_weight(_cuda(w2), False)
    for prec, atol in ((FP32, 1e-5), (TF32, 6e-3)):
        y = ops.residual_layer(rn, p1, p2, B=B, H=H, W=W, C=C, Cmid=Cmid, relu_out=relu_out, precision=prec)
        np.testing.assert_allclose(y.cpu().numpy().transpose(0, 3, 1, 2), ref, atol=atol, rtol=2e-3)


@pytest.mark.parametrize("B,H,W,C,Cmid,n", [(256, 8, 8, 128, 32, 2), (5, 8, 8, 128, 32, 3), (3, 6, 7, 128, 32, 2),
                                            (9, 4, 4, 64, 32, 4), (2, 16, 16, 128, 32, 2), (1, 8, 8, 128, 32, 1)])
def test_fused_residual_stack_tc(B, H, W, C, Cmid, n):
    """vqb_residual_stack_f32 (residual.py:45-51): all n shared-weight applications in ONE tcgen05 launch when a
    128-pixel tile holds whole images.  Same arithmetic as n separate vqb_residual_layer_f32 launches, so the two
    are bit-identical; both are held to the oracle at the TF32 tolerance, the fp32 mode at 1e-5 per layer."""
    from vqvae_b200 import ops
    from vqvae_b200._lib import FP32, TF32
    rng = np.random.RandomState(B * 1000 + H * 100 + C + n)
    r = np.maximum(rng.standard_normal((B, C, H, W)).astype(np.float32), 0)
    w1 = (rng.standard_normal((Cmid, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
    w2 = (rng.standard_normal((C, Cmid, 1, 1)) / np.sqrt(Cmid)).astype(np.float32)
    ref = r
    for _ in range(n):
        ref = np.maximum(ref + cref.conv2d(np.maximum(cref.conv2d(ref, w1, None, 1, 1), 0), w2, None, 1, 0), 0)
    rn = _cuda(np.ascontiguousarray(r.transpose(0, 2, 3, 1)))
    p1, p2 = ops.pack_conv_weight(_cuda(w1), False), ops.pack_conv_weight(_cuda(w2), False)
    for prec, atol in ((FP32, 1e-5 * n), (TF32, 6e-3 * n)):
        l0 = ops.launch_count()
        y = ops.residual_stack(rn, p1, p2, B=B, H=H, W=W, C=C, Cmid=Cmid, n_layers=n, precision=prec)
        launches = ops.launch_count() - l0
        np.testing.assert_allclose(y.cpu().numpy().transpose(0, 3, 1, 2), ref, atol=atol, rtol=2e-3 * n)
        seq = rn
        for _ in range(n):
            seq = ops.residual_layer(seq, p1, p2, B=B, H=H, W=W, C=C, Cmid=Cmid, relu_out=True, precision=prec)
        assert torch.equal(y, seq)
        if prec == TF32 and W <= 8 and H <= 16:
            assert launches == 1, launches          # the fused path really ran
    assert torch.equal(rn.cpu(), torch.from_numpy(np.ascontiguousarray(r.transpose(0, 2, 3, 1))))   # input untouched


def test_checkpoint_load_packs_weights_and_reproduces_the_golden_forward():
    """SURVEY 8f rank 2: a checkpoint in the reference's own format -> load_checkpoint -> forward equals the golden outputs of
    the unmodified reference for the same weights; the weight packings exist before the first forward."""
    import os
    import vqvae_b200
    g = load_golden("small_odd")
    hp, sd, x = model_case_inputs(g["case"])
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ckpt_small_odd.pth")
    m, data = vqvae_b200.load_checkpoint(path, device="cuda")
    w = m.encoder.conv_stack[2].weight
    assert getattr(w, "_vqb_packed", None), "conv weights must be packed at load time"
    loss, x_hat, perp = m(_cuda(x))
    assert np.array_equal(m.last_min_encoding_indices.cpu().numpy(), g["idx"])
    np.testing.assert_allclose(x_hat.cpu().numpy(), g["x_hat"], atol=CONV_ATOL, rtol=0)
    np.testing.assert_allclose(loss.item(), g["loss"], rtol=1e-5)


def test_vq_backward_matches_autograd_of_the_reference_formula():
    """SURVEY 8f rank 3: VectorQuantizer in training mode (grad enabled): loss.backward() + a downstream gradient on z_q give the
    straight-through gradient on z and the scatter-added codebook gradient of quantizer.py:63-67 (torch autograd on CPU as oracle)."""
    from models.quantizer import VectorQuantizer
    rng = np.random.RandomState(3)
    K, D = 37, 16
    z0 = rng.standard_normal((3, D, 5, 7)).astype(np.float32)
    E0 = rng.standard_normal((K, D)).astype(np.float32)
    gq = rng.standard_normal((3, D, 5, 7)).astype(np.float32)
    torch.set_grad_enabled(True)               # (the conftest default is no_grad; restored by its context on exit)
    # reference formula with torch autograd (CPU)
    z = torch.tensor(z0, requires_grad=True)
    E = torch.tensor(E0, requires_grad=True)
    zf = z.permute(0, 2, 3, 1).contiguous().view(-1, D)
    d = (zf ** 2).sum(1, keepdim=True) + (E ** 2).sum(1) - 2 * zf @ E.t()
    idx = d.argmin(1)
    zq = E[idx].view(3, 5, 7, D)
    zp = z.permute(0, 2, 3, 1)
    loss = ((zq.detach() - zp) ** 2).mean() + 0.25 * ((zq - zp.detach()) ** 2).mean()
    out = (zp + (zq - zp).detach()).permute(0, 3, 1, 2)
    (loss * 1.7 + (out * torch.tensor(gq)).sum()).backward()
    # product
    vq = VectorQuantizer(K, D, 0.25).cuda()
    vq.embedding.weight.data.copy_(torch.from_numpy(E0))
    zc = torch.tensor(z0, device="cuda", requires_grad=True)
    l2, zq2, perp2, oh2, idx2 = vq(zc)
    assert np.array_equal(idx2.view(-1).cpu().numpy(), idx.numpy())
    (l2 * 1.7 + (zq2 * torch.tensor(gq, device="cuda")).sum()).backward()
    np.testing.assert_allclose(l2.item(), loss.item(), rtol=1e-6)
    np.testing.assert_allclose(zc.grad.cpu().numpy(), z.grad.numpy(), atol=1e-6, rtol=1e-5)
    np.testing.assert_allclose(vq.embedding.weight.grad.cpu().numpy(), E.grad.numpy(), atol=1e-6, rtol=1e-5)
    assert perp2.requires_grad is False and oh2.shape == (105, K)
