"""The fused TF32 latent stage (vqb_latent_encoder_f32 / vqb_latent_decoder_f32) against the per-layer chain it
replaces, in one process on the same seeded data: outputs must be bitwise equal (same TF32 operands, same k-step order
and accumulator split, same epilogue order)."""
import ctypes

import numpy as np
import pytest
import torch


def test_latent_entry_points_validate_arguments_without_a_gpu():
    from vqvae_b200 import _lib
    lib = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    enc, dec = lib.vqb_latent_encoder_f32, lib.vqb_latent_decoder_f32
    assert enc(None, p, None, p, p, p, None, p, 2, 8, 8, 128, 32, 64, 2, None) == -1          # null input
    assert enc(p, p, None, p, p, p, None, p, 0, 8, 8, 128, 32, 64, 2, None) == -1              # B <= 0
    assert enc(p, p, None, p, p, p, None, p, 2, 8, 8, 128, 32, 64, 0, None) == -1              # no residual layer
    assert enc(p, p, None, p, p, p, None, p, 2, 8, 8, 256, 32, 64, 2, None) == -2              # C != 128
    assert enc(p, p, None, p, p, p, None, p, 2, 8, 8, 128, 32, 64, 5, None) == -2              # n_res > 4
    assert enc(p, p, None, p, p, p, None, p, 2, 8, 16, 128, 32, 64, 2, None) in (-2, -5)       # W > 8: not one tile
    assert dec(p, p, None, p, p, None, None, p, 2, 8, 8, 64, 128, 32, 64, 2, None) == -1       # null D2 weight
    assert dec(p, p, None, p, p, p, None, p, 2, 8, 8, 64, 128, 32, 3, 2, None) == -2           # Cout != 64
    assert dec(p, p, None, p, p, p, None, p, 2, 32, 8, 64, 128, 32, 64, 2, None) in (-2, -5)   # H > 16


def _weights(g, cout, cin, k, transposed=False):
    shape = (cin, cout, k, k) if transposed else (cout, cin, k, k)
    return torch.randn(shape, device="cuda", generator=g) / np.sqrt(cin * k * k)


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", [(2, 8, 8), (3, 8, 8), (256, 8, 8), (5, 4, 4)])
def test_fused_latent_stage_equals_per_layer_chain(B, H, W):
    from vqvae_b200 import ops
    from vqvae_b200._lib import TF32
    g = torch.Generator(device="cuda").manual_seed(1234 + B)
    C, Cmid, D, n = 128, 32, 64, 2
    pk = ops.pack_conv_weight
    w3, w1, w2, wq = _weights(g, C, C, 3), _weights(g, Cmid, C, 3), _weights(g, C, Cmid, 1), _weights(g, D, C, 1)
    wt1, wt2 = _weights(g, C, D, 3, True), _weights(g, C // 2, C, 4, True)
    b3, bq, bt1, bt2 = (torch.randn((c,), device="cuda", generator=g) * 0.1 for c in (C, D, C, C // 2))
    p3, p1, p2, pq = pk(w3, False), pk(w1, False), pk(w2, False), pk(wq, False)
    pt1, pt2 = pk(wt1, True), pk(wt2, True)
    h = torch.randn((B, H, W, C), device="cuda", generator=g).clamp_min(0)      # E2's output, after its ReLU
    zq = torch.randn((B, H, W, D), device="cuda", generator=g) * 0.5

    conv = dict(precision=TF32)
    e = ops.conv2d(h, p3, b3, B=B, Cin=C, H=H, W=W, Cout=C, kh=3, kw=3, stride=1, pad=1, relu=True, **conv)
    e = ops.residual_stack(e, p1, p2, B=B, H=H, W=W, C=C, Cmid=Cmid, n_layers=n, precision=TF32)
    z_chain = ops.conv2d(e, pq, bq, B=B, Cin=C, H=H, W=W, Cout=D, kh=1, kw=1, stride=1, pad=0, **conv)
    z_fused = ops.latent_encoder(h, p3, b3, p1, p2, pq, bq, B=B, H=H, W=W, C=C, Cmid=Cmid, D=D, n_res=n)
    assert z_fused is not None
    assert torch.equal(z_fused, z_chain), float((z_fused - z_chain).abs().max())

    d = ops.conv2d(zq, pt1, bt1, B=B, Cin=D, H=H, W=W, Cout=C, kh=3, kw=3, stride=1, pad=1, transposed=True, relu=True,
                   **conv)
    d = ops.residual_stack(d, p1, p2, B=B, H=H, W=W, C=C, Cmid=Cmid, n_layers=n, precision=TF32)
    d_chain = ops.conv2d(d, pt2, bt2, B=B, Cin=C, H=H, W=W, Cout=C // 2, kh=4, kw=4, stride=2, pad=1, transposed=True,
                         relu=True, **conv)
    d_fused = ops.latent_decoder(zq, pt1, bt1, p1, p2, pt2, bt2, B=B, H=H, W=W, D=D, C=C, Cmid=Cmid, Cout=C // 2,
                                 n_res=n)
    assert d_fused is not None
    assert torch.equal(d_fused, d_chain), float((d_fused - d_chain).abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cifar_default", "cifar_spread"])
def test_tf32_forward_fused_equals_unfused(name, monkeypatch):
    import vqvae_b200
    from vqvae_b200 import modules, ops
    from tests.helpers import build_model, load_golden, model_case_inputs
    g = load_golden(name)
    hp, sd, x = model_case_inputs(g["case"])
    m = build_model(hp, sd)
    xc = torch.from_numpy(x).cuda()
    with vqvae_b200.precision("tf32"):
        m(xc)                                           # packs the weights (counted as launches)
        n0 = ops.launch_count()
        _, x_fused, _ = m(xc)
        launches_fused = ops.launch_count() - n0
        idx_fused = m.last_min_encoding_indices.clone()
        monkeypatch.setattr(modules.Encoder, "_fused_tail", lambda self, *a: None)
        monkeypatch.setattr(modules.Decoder, "_fused_head", lambda self, *a: None)
        n0 = ops.launch_count()
        _, x_chain, _ = m(xc)
        launches_chain = ops.launch_count() - n0
        idx_chain = m.last_min_encoding_indices.clone()
    assert torch.equal(idx_fused, idx_chain)
    assert torch.equal(x_fused, x_chain)
    assert launches_chain - launches_fused == 4        # E3 + stack + 1x1 and D1 + stack + D2 became two kernels
