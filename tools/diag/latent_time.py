"""The TF32 latent stage at cfg2's shape (B=256, 8x8 latent, C=128, Cmid=32, D=64, two residual applications):
per-layer chain (E3 + stack + 1x1; D1 + stack + D2) vs the two fused kernels (vqb_latent_encoder_f32 /
vqb_latent_decoder_f32).  Each variant is captured in a CUDA graph and replayed with a 256 MiB L2 flush before every
replay; CUDA events around the replay only.  Prints us per stage (median, min), launches and the TF32 share."""
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from vqvae_b200 import ops  # noqa: E402
from vqvae_b200._lib import TF32  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
H = W = 8
C, CM, D, NRES = 128, 32, 64, 2
REPS = 200
TF32_PEAK = 1125.0      # TFLOP/s, dense TF32 of one B200 per NVIDIA's HGX B200 data sheet (1000 W card)
dev = torch.device("cuda")
g = torch.Generator(device="cuda").manual_seed(0)


def wt(cout, cin, k, transposed=False):
    shape = (cin, cout, k, k) if transposed else (cout, cin, k, k)
    return ops.pack_conv_weight(torch.randn(shape, device=dev, generator=g) / np.sqrt(cin * k * k), transposed)


p3, p1, p2, pq, pt1, pt2 = wt(C, C, 3), wt(CM, C, 3), wt(C, CM, 1), wt(D, C, 1), wt(C, D, 3, True), wt(C // 2, C, 4, True)
b3, bq, bt1, bt2 = (torch.randn((c,), device=dev, generator=g) * 0.1 for c in (C, D, C, C // 2))
h = torch.randn((B, H, W, C), device=dev, generator=g).clamp_min(0)
zq = torch.randn((B, H, W, D), device=dev, generator=g) * 0.5


def enc_chain():
    e = ops.conv2d(h, p3, b3, B=B, Cin=C, H=H, W=W, Cout=C, kh=3, kw=3, stride=1, pad=1, relu=True, precision=TF32)
    e = ops.residual_stack(e, p1, p2, B=B, H=H, W=W, C=C, Cmid=CM, n_layers=NRES, precision=TF32)
    return ops.conv2d(e, pq, bq, B=B, Cin=C, H=H, W=W, Cout=D, kh=1, kw=1, stride=1, pad=0, precision=TF32)


def dec_chain():
    d = ops.conv2d(zq, pt1, bt1, B=B, Cin=D, H=H, W=W, Cout=C, kh=3, kw=3, stride=1, pad=1, transposed=True, relu=True,
                   precision=TF32)
    d = ops.residual_stack(d, p1, p2, B=B, H=H, W=W, C=C, Cmid=CM, n_layers=NRES, precision=TF32)
    return ops.conv2d(d, pt2, bt2, B=B, Cin=C, H=H, W=W, Cout=C // 2, kh=4, kw=4, stride=2, pad=1, transposed=True,
                      relu=True, precision=TF32)


def enc_fused():
    return ops.latent_encoder(h, p3, b3, p1, p2, pq, bq, B=B, H=H, W=W, C=C, Cmid=CM, D=D, n_res=NRES)


def dec_fused():
    return ops.latent_decoder(zq, pt1, bt1, p1, p2, pt2, bt2, B=B, H=H, W=W, D=D, C=C, Cmid=CM, Cout=C // 2, n_res=NRES)


flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def measure(fn):
    n0 = ops.launch_count()
    ref = fn()
    launches = ops.launch_count() - n0
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    for _ in range(5):
        graph.replay()
    ts = []
    for _ in range(REPS):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    assert torch.equal(out, ref)
    return float(np.median(ts)), float(np.min(ts)), launches, out


flop_enc = 2.0 * B * H * W * (9 * C * C + NRES * (9 * C * CM + CM * C) + C * D)
flop_dec = 2.0 * B * H * W * (9 * D * C + NRES * (9 * C * CM + CM * C) + 16 * C * (C // 2))
print(f"device {torch.cuda.get_device_name()}, B={B}, latent {H}x{W}, {REPS} graph replays each, L2 flushed before each")
res = {}
for name, fn, flop in (("encoder tail, chain", enc_chain, flop_enc), ("encoder tail, fused", enc_fused, flop_enc),
                       ("decoder head, chain", dec_chain, flop_dec), ("decoder head, fused", dec_fused, flop_dec)):
    med, mn, nl, out = measure(fn)
    res[name] = out
    tf = flop / (med * 1e-6) / 1e12
    print(f"{name:22s} {med:8.2f} us median  {mn:8.2f} us min  {nl} launches  {tf:6.1f} TFLOP/s = "
          f"{100 * tf / TF32_PEAK:4.1f} % of dense TF32", flush=True)
print("fused == chain (bitwise):", torch.equal(res["encoder tail, fused"], res["encoder tail, chain"].view(B, H, W, D)),
      torch.equal(res["decoder head, fused"], res["decoder head, chain"]))
