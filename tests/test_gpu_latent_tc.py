"""The fused TF32 latent stage (vqb_latent_encoder_f32 / vqb_latent_decoder_f32) against the per-layer chain it
replaces, in one process on the same seeded data: outputs must be bitwise equal (same TF32 operands, same k-step order
and accumulator split, same epilogue order), across the dispatch domain (H <= 16, W <= 8, 1 <= n_res <= 4).  The
chain's links are in turn held to the TF32 bar of tests/helpers.py on the inputs they received."""
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


def _tile_bn(H):
    """Images per 128-pixel tile of the fused kernels (and conv_halo / res_tc): 16 / BH, BH = pow2_ceil(H) <= 16."""
    bh = 1
    while bh < H:
        bh *= 2
    return 16 // min(bh, 16)


class _Latent:
    """Seeded weights and inputs of both latent halves at C = 128, Cmid = 32, D = 64; the per-layer chains and the
    fused kernels on them."""
    C, Cmid, D = 128, 32, 64

    def __init__(self, seed, B, H, W, n, biases=True):
        from vqvae_b200 import ops
        g = torch.Generator(device="cuda").manual_seed(seed)
        C, Cmid, D = self.C, self.Cmid, self.D
        self.B, self.H, self.W, self.n = B, H, W, n
        self.w3, self.w1, self.w2 = _weights(g, C, C, 3), _weights(g, Cmid, C, 3), _weights(g, C, Cmid, 1)
        self.wq, self.wt1, self.wt2 = _weights(g, D, C, 1), _weights(g, C, D, 3, True), _weights(g, C // 2, C, 4, True)
        self.b3, self.bq, self.bt1, self.bt2 = (torch.randn((c,), device="cuda", generator=g) * 0.1 if biases else None
                                                for c in (C, D, C, C // 2))
        pk = ops.pack_conv_weight
        self.p3, self.p1, self.p2, self.pq = pk(self.w3, False), pk(self.w1, False), pk(self.w2, False), pk(self.wq, False)
        self.pt1, self.pt2 = pk(self.wt1, True), pk(self.wt2, True)
        self.h = torch.randn((B, H, W, C), device="cuda", generator=g).clamp_min(0)      # E2's output, after its ReLU
        self.zq = torch.randn((B, H, W, D), device="cuda", generator=g) * 0.5

    def _stack(self, x, links):
        """n separate residual_layer launches (each one a link), checked bitwise against the one-launch stack."""
        from vqvae_b200 import ops
        from vqvae_b200._lib import TF32
        geo = dict(B=self.B, H=self.H, W=self.W, C=self.C, Cmid=self.Cmid)
        stack = ops.residual_stack(x, self.p1, self.p2, n_layers=self.n, precision=TF32, **geo)
        for i in range(self.n):
            y = ops.residual_layer(x, self.p1, self.p2, relu_out=True, precision=TF32, **geo)
            links.append(("residual %d/%d" % (i + 1, self.n), x, y))
            x = y
        assert torch.equal(stack, x), "residual stack in one launch != %d separate launches" % self.n
        return x

    def encoder_chain(self):
        """E3 (conv_halo) -> residual layers -> pre-quant 1x1 (conv_tc): (z_e, [(link, input, output)])."""
        from vqvae_b200 import ops
        from vqvae_b200._lib import TF32
        C, D, B, H, W, links = self.C, self.D, self.B, self.H, self.W, []
        conv = dict(B=B, H=H, W=W, stride=1, precision=TF32)
        e = ops.conv2d(self.h, self.p3, self.b3, Cin=C, Cout=C, kh=3, kw=3, pad=1, relu=True, **conv)
        links.append(("E3", self.h, e))
        e = self._stack(e, links)
        z = ops.conv2d(e, self.pq, self.bq, Cin=C, Cout=D, kh=1, kw=1, pad=0, **conv)
        links.append(("1x1", e, z))
        return z, links

    def decoder_chain(self):
        """D1 convT 3x3 (conv_halo) -> residual layers -> D2 convT k4s2 (conv_tc, 4 phases)."""
        from vqvae_b200 import ops
        from vqvae_b200._lib import TF32
        C, D, B, H, W, links = self.C, self.D, self.B, self.H, self.W, []
        conv = dict(B=B, H=H, W=W, transposed=True, relu=True, precision=TF32)
        d = ops.conv2d(self.zq, self.pt1, self.bt1, Cin=D, Cout=C, kh=3, kw=3, stride=1, pad=1, **conv)
        links.append(("D1", self.zq, d))
        d = self._stack(d, links)
        y = ops.conv2d(d, self.pt2, self.bt2, Cin=C, Cout=C // 2, kh=4, kw=4, stride=2, pad=1, **conv)
        links.append(("D2", d, y))
        return y, links

    def encoder_fused(self):
        from vqvae_b200 import ops
        return ops.latent_encoder(self.h, self.p3, self.b3, self.p1, self.p2, self.pq, self.bq, B=self.B, H=self.H,
                                  W=self.W, C=self.C, Cmid=self.Cmid, D=self.D, n_res=self.n)

    def decoder_fused(self):
        from vqvae_b200 import ops
        return ops.latent_decoder(self.zq, self.pt1, self.bt1, self.p1, self.p2, self.pt2, self.bt2, B=self.B, H=self.H,
                                  W=self.W, D=self.D, C=self.C, Cmid=self.Cmid, Cout=self.C // 2, n_res=self.n)

    def assert_fused_equals_chain(self):
        z_chain, enc_links = self.encoder_chain()
        z_fused = self.encoder_fused()
        assert z_fused is not None
        assert torch.equal(z_fused, z_chain), float((z_fused - z_chain).abs().max())
        d_chain, dec_links = self.decoder_chain()
        d_fused = self.decoder_fused()
        assert d_fused is not None
        assert torch.equal(d_fused, d_chain), float((d_fused - d_chain).abs().max())
        return enc_links + dec_links


# The dispatch domain of Encoder._fused_tail / Decoder._fused_head: H <= 16, W <= 8, 1 <= n_res <= 4.  The (H, W) points
# cover every tile class (BH = 2: BN = 8 images per tile and a ring of only 2 stages; BH = 4, 8, 16: BN = 4, 2, 1) with
# full and masked (W < 8) tile columns.  B = BN + 1 leaves a ragged last tile; 2 * 148 * BN + 1 images give more CTAs
# than a B200 has SMs (one CTA per SM).
LATENT_HW = [(2, 8), (2, 3), (3, 5), (4, 4), (5, 7), (7, 8), (8, 8), (8, 1), (9, 8), (12, 6), (16, 8), (16, 3)]
LATENT_CASES = [(H, W, n, B) for H, W in LATENT_HW for n in (1, 2, 3, 4)
                for B in (_tile_bn(H) + 1, 2 * 148 * _tile_bn(H) + 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n,B", LATENT_CASES)
def test_fused_latent_stage_equals_per_layer_chain(H, W, n, B):
    _Latent(1234 + B + 17 * H + W, B, H, W, n).assert_fused_equals_chain()


@pytest.mark.gpu
def test_fused_latent_stage_without_biases():
    """The ABI takes null biases (a layer built with bias=False): the fused kernels then add zeros, like the chain."""
    _Latent(77, 3, 8, 8, 2, biases=False).assert_fused_equals_chain()


@pytest.mark.gpu
def test_fused_latent_stage_declines_a_one_row_latent():
    """At H = 1 a tile holds 16 images and the halo buffers leave no room for a ring of two stages: both entry points
    answer UNSUPPORTED (None) without launching, and the caller runs the chain."""
    from vqvae_b200 import ops
    lat = _Latent(5, 17, 1, 8, 2)
    n0 = ops.launch_count()
    assert lat.encoder_fused() is None
    assert lat.decoder_fused() is None
    assert ops.launch_count() == n0


# One (H, W) with W = 8 and one with W < 8 per tile class BH = 2, 4, 8, 16; small B (the reference runs on the host).
BOUND_CASES = [(2, 8, 1), (2, 3, 4), (4, 8, 2), (3, 5, 3), (8, 8, 2), (5, 7, 1), (16, 8, 3), (12, 6, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n", BOUND_CASES)
def test_latent_chain_links_within_tf32_bound(H, W, n):
    """fused == chain bitwise, and every link of the chain is held to the truncated-operand bound of tests/helpers.py
    on the input that link really received (no bound is carried through layers)."""
    from tests.helpers import assert_within_bound, tf32_layer_ref, tf32_residual_ref
    B = _tile_bn(H) + 1
    lat = _Latent(4321 + 17 * H + W, B, H, W, n)
    links = lat.assert_fused_equals_chain()

    def a(t):
        return None if t is None else t.cpu().numpy()

    w = {k: a(getattr(lat, k)) for k in ("w3", "w1", "w2", "wq", "wt1", "wt2", "b3", "bq", "bt1", "bt2")}
    for name, x, y in links:
        x, y = a(x).transpose(0, 3, 1, 2), a(y).transpose(0, 3, 1, 2)
        if name == "E3":
            c, bound = tf32_layer_ref(x, w["w3"], w["b3"], stride=1, pad=1, relu=True)
        elif name == "1x1":
            c, bound = tf32_layer_ref(x, w["wq"], w["bq"])
        elif name == "D1":
            c, bound = tf32_layer_ref(x, w["wt1"], w["bt1"], stride=1, pad=1, transposed=True, relu=True)
        elif name == "D2":
            c, bound = tf32_layer_ref(x, w["wt2"], w["bt2"], stride=2, pad=1, transposed=True, relu=True)
        else:
            c, bound, straddle = tf32_residual_ref(x, w["w1"], w["w2"])
            print("%s: mid straddle share %.2f %%" % (name, 100 * straddle))
        assert_within_bound(y, c, bound, "latent %dx%d n=%d B=%d %s" % (H, W, n, B, name))


def _synth_model(img_h, img_w, n_res, batch=4):
    from tests.helpers import build_model
    from vqvae_b200.synth import make_state_dict
    hp = dict(h_dim=128, res_h_dim=32, n_res_layers=n_res, n_embeddings=512, embedding_dim=64)
    sd = make_state_dict(seed=n_res, codebook="normal", codebook_scale=0.05, **hp)
    x = (2 * np.random.RandomState(img_h + img_w).random_sample((batch, 3, img_h, img_w)) - 1).astype(np.float32)
    return build_model(hp, sd), x


# name: (image H, image W, n_res) of a synthetic model, or a golden case; launches the fused stage saves per forward
FORWARD_CASES = {
    "cifar_default": None, "cifar_spread": None,
    "synth_64x32_n3": (64, 32, 3),      # 16 x 8 latent: BN = 1
    "synth_20x28_n1": (20, 28, 1),      # 5 x 7 latent: masked tile columns
    "synth_8x32_n4": (8, 32, 4),        # 2 x 8 latent: BN = 8, two ring stages
    "synth_4x32_n2": (4, 32, 2),        # 1 x 8 latent: not covered, both halves run the chain
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FORWARD_CASES))
def test_tf32_forward_fused_equals_unfused(name, monkeypatch):
    import vqvae_b200
    from vqvae_b200 import modules, ops
    from tests.helpers import build_model, load_golden, model_case_inputs
    if FORWARD_CASES[name] is None:
        g = load_golden(name)
        hp, sd, x = model_case_inputs(g["case"])
        m = build_model(hp, sd)
    else:
        m, x = _synth_model(*FORWARD_CASES[name])
    saved = 0 if x.shape[2] // 4 < 2 else 4          # E3 + stack + 1x1 and D1 + stack + D2 became two kernels
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
    assert launches_chain - launches_fused == saved, (launches_chain, launches_fused)
