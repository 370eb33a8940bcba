"""Torch-tensor front end of the C ABI: allocation and stream plumbing only.

PyTorch owns every buffer and the current stream; all arithmetic happens inside
libvqvae_b200.so.  There is NO CPU path: a non-CUDA tensor raises.
"""
import torch

from . import _lib
from ._lib import BF16, FP32, NCHW, NHWC, TF32, check, lib  # noqa: F401


def _require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(
            f"vqvae_b200: {what} must be a CUDA tensor -- this implementation is sm_100a-only "
            "and has no CPU fallback")
    if t.device.index != torch.cuda.current_device():
        # the C ABI launches on the CURRENT device's stream (header: "the caller selects the device"); a tensor that lives
        # elsewhere would be read through a peer mapping at best and fault at worst (ADVICE r1)
        raise RuntimeError(
            f"vqvae_b200: {what} is on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
            "wrap the call in `with torch.cuda.device(tensor.device):`")


def _stream():
    return torch.cuda.current_stream().cuda_stream


# Optional per-call CUDA-event timing (bench.py's kernel breakdown): when PROFILE is a
# list, every C-ABI compute call appends (label, start_event, end_event).
PROFILE = None


class _Span:
    __slots__ = ("label", "start", "end")

    def __init__(self, label):
        self.label = label
        self.start = self.end = None
        if PROFILE is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.end = torch.cuda.Event(enable_timing=True)
            self.start.record()

    def done(self):
        if self.start is not None:
            self.end.record()
            PROFILE.append((self.label, self.start, self.end))


def launch_count() -> int:
    """Kernels launched so far through the C ABI by this process."""
    return int(lib().vqb_launch_count())


def _f32c(t):
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def pack_conv_weight(w, transposed, out=None):
    """(Cout,Cin,kh,kw) conv / (Cin,Cout,kh,kw) conv-transpose weight -> the two tap-major
    fp32 GEMM operand layouts of vqb_pack_conv_weight_f32, back to back:
    [(r*kw+s)*Cin+ci][co] for the FFMA kernel and [(r*kw+s)][co][ci] for tcgen05."""
    _require_cuda(w, "weight")
    w = _f32c(w.detach())
    if transposed:
        cin, cout, kh, kw = w.shape
    else:
        cout, cin, kh, kw = w.shape
    # 2 GEMM layouts + (for the k4s2 output layer) the 9x16xCin pixel-shuffle packing
    n = 2 * kh * kw * cin * cout + 9 * 16 * cin
    if out is None or out.numel() != n or out.dtype != torch.float32 or out.device != w.device:
        out = torch.empty((n,), dtype=torch.float32, device=w.device)      # else: repacked in place
    check(lib().vqb_pack_conv_weight_f32(w.data_ptr(), out.data_ptr(), cout, cin, kh, kw,
                                         int(bool(transposed)), _stream()), "pack_conv_weight")
    return out


def conv_out_hw(h, w, kh, kw, stride, pad, transposed):
    if transposed:
        return (h - 1) * stride - 2 * pad + kh, (w - 1) * stride - 2 * pad + kw
    return (h + 2 * pad - kh) // stride + 1, (w + 2 * pad - kw) // stride + 1


def conv2d(x, w_packed, bias, *, B, Cin, H, W, Cout, kh, kw, stride, pad, transposed=False,
           in_layout=NHWC, out_layout=NHWC, relu=False, skip=None, precision=FP32):
    """One nn.Conv2d / nn.ConvTranspose2d forward (+bias, +skip, +ReLU) on raw buffers.
    `x` is any contiguous CUDA fp32 tensor holding the (B,Cin,H,W) activation in
    `in_layout`; returns a new tensor in `out_layout` ((B,Cout,OH,OW) or (B,OH,OW,Cout))."""
    _require_cuda(x, "input")
    oh, ow = conv_out_hw(H, W, kh, kw, stride, pad, transposed)
    if oh <= 0 or ow <= 0:
        raise RuntimeError(f"conv output size is non-positive ({oh}x{ow})")
    shape = (B, Cout, oh, ow) if out_layout == NCHW else (B, oh, ow, Cout)
    out = torch.empty(shape, dtype=torch.float32, device=x.device)
    span = _Span(f"conv{'T' if transposed else ''} {Cin}->{Cout} k{kh}s{stride} {H}x{W}"
                 f"{' +skip' if skip is not None else ''}")
    check(lib().vqb_conv2d_f32(
        x.data_ptr(), w_packed.data_ptr(), bias.data_ptr() if bias is not None else None,
        skip.data_ptr() if skip is not None else None, out.data_ptr(),
        B, Cin, H, W, Cout, kh, kw, stride, pad, int(bool(transposed)), in_layout, out_layout,
        int(bool(relu)), precision, _stream()), "conv2d")
    span.done()
    return out


def conv_kind(kh, stride, transposed, cout):
    """enum vqb_conv_kind of a layer of the hot path, or None when the bf16 kernels do not cover it."""
    if not transposed:
        return {(1, 1): _lib.CONV_K1, (3, 1): _lib.CONV_K3, (4, 2): _lib.CONV_K4S2}.get((kh, stride))
    if (kh, stride) == (3, 1):
        return _lib.CONVT_K3
    if (kh, stride) == (4, 2):
        return _lib.CONVT_K4S2_OUT if cout <= 4 else _lib.CONVT_K4S2
    return None


def pack_conv_weight_bf16(w, kind, out=None):
    """fp32 conv / conv-transpose weight -> the bf16 k-step-ordered packing of vqb_pack_conv_weight_bf16
    (None when the shape is not covered).  `out`: repack into an existing buffer (same shape) in place."""
    _require_cuda(w, "weight")
    w = _f32c(w.detach())
    transposed = kind in (_lib.CONVT_K3, _lib.CONVT_K4S2, _lib.CONVT_K4S2_OUT)
    cin, cout = (w.shape[0], w.shape[1]) if transposed else (w.shape[1], w.shape[0])
    nbytes = lib().vqb_conv_bf16_packed_bytes(kind, cout, cin)
    if nbytes == 0:
        return None
    if out is None or out.numel() != nbytes or out.dtype != torch.uint8 or out.device != w.device:
        # (torch's caching allocator hands out 512-byte aligned blocks: the 128-byte alignment the TMA maps need)
        out = torch.empty((nbytes,), dtype=torch.uint8, device=w.device)
    check(lib().vqb_pack_conv_weight_bf16(w.data_ptr(), out.data_ptr(), kind, cout, cin, _stream()), "pack_conv_weight_bf16")
    return out


def conv2d_bf16(x, packed, bias, *, B, Cin, H, W, Cout, kind, relu=False, out_f32=False):
    """One layer on bf16 NHWC input through vqb_conv2d_bf16; returns bf16 NHWC, fp32 NHWC (out_f32) or, for
    CONVT_K4S2_OUT, the fp32 NCHW module output."""
    _require_cuda(x, "input")
    if x.dtype != torch.bfloat16 or not x.is_contiguous():
        raise RuntimeError("conv2d_bf16: input must be a contiguous bf16 NHWC tensor")
    if kind == _lib.CONV_K4S2:
        shape, dt = (B, H // 2, W // 2, Cout), (torch.float32 if out_f32 else torch.bfloat16)
    elif kind == _lib.CONVT_K4S2:
        shape, dt = (B, 2 * H, 2 * W, Cout), (torch.float32 if out_f32 else torch.bfloat16)
    elif kind == _lib.CONVT_K4S2_OUT:
        shape, dt = (B, Cout, 2 * H, 2 * W), torch.float32
    else:
        shape, dt = (B, H, W, Cout), (torch.float32 if out_f32 else torch.bfloat16)
    out = torch.empty(shape, dtype=dt, device=x.device)
    k, st, tr = {_lib.CONV_K1: (1, 1, ""), _lib.CONV_K3: (3, 1, ""), _lib.CONVT_K3: (3, 1, "T"), _lib.CONV_K4S2: (4, 2, ""),
                 _lib.CONVT_K4S2: (4, 2, "T"), _lib.CONVT_K4S2_OUT: (4, 2, "T")}[kind]
    span = _Span(f"bf16 conv{tr} {Cin}->{Cout} k{k}s{st} {H}x{W}")
    check(lib().vqb_conv2d_bf16(x.data_ptr(), packed.data_ptr(), bias.data_ptr() if bias is not None else None,
                                out.data_ptr(), B, Cin, H, W, Cout, kind, int(bool(relu)), int(bool(out_f32)),
                                _stream()), "conv2d_bf16")
    span.done()
    return out


def conv_in_bf16(x, w_packed_f32, bias, *, B, H, W, Cout, relu=True):
    """encoder.py:29-31 for the bf16 pipeline: fp32 NCHW image -> bf16 NHWC (B, H/2, W/2, Cout) (vqb_conv_in_bf16)."""
    _require_cuda(x, "input")
    out = torch.empty((B, H // 2, W // 2, Cout), dtype=torch.bfloat16, device=x.device)
    span = _Span(f"bf16 conv 3->{Cout} k4s2 {H}x{W}")
    check(lib().vqb_conv_in_bf16(x.data_ptr(), w_packed_f32.data_ptr(), bias.data_ptr() if bias is not None else None,
                                 out.data_ptr(), B, H, W, Cout, int(bool(relu)), _stream()), "conv_in_bf16")
    span.done()
    return out


def vq_forward_bf16zq(z_rows, codebook):
    """Fused VectorQuantizer core, fp32 rows in, bit-exact int64 idx, z_q as bf16 rows (vqb_vq_forward_bf16zq_f32).
    Deferred SSE: returns (idx, zq_bf16, sse, hist, ws); run vq_reduce_sse(ws, ...) before reading sse."""
    _require_cuda(z_rows, "z")
    N, D = z_rows.shape
    K = codebook.shape[0]
    dev = z_rows.device
    idx = torch.empty((N,), dtype=torch.int64, device=dev)
    zq = torch.empty((N, D), dtype=torch.bfloat16, device=dev)
    sse = torch.empty((1,), dtype=torch.float64, device=dev)
    hist = torch.empty((K,), dtype=torch.int32, device=dev)
    ws_bytes = lib().vqb_vq_workspace_bytes(N, K, D)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    span = _Span(f"vq N={N} K={K} D={D} (bf16 zq)")
    check(lib().vqb_vq_forward_bf16zq_f32(z_rows.data_ptr(), codebook.data_ptr(), N, K, D, idx.data_ptr(), zq.data_ptr(),
                                          sse.data_ptr(), hist.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "vq_forward_bf16zq")
    span.done()
    return idx, zq, sse, hist, ws


def residual_layer_bf16(r, w1_packed, w2_packed, *, B, H, W, C, Cmid, relu_out):
    """out = act(r + W2.relu(W1 (*) r)) on bf16 NHWC buffers, one persistent tcgen05 kernel (vqb_residual_layer_bf16)."""
    _require_cuda(r, "input")
    if r.dtype != torch.bfloat16 or not r.is_contiguous():
        raise RuntimeError("residual_layer_bf16: input must be a contiguous bf16 NHWC tensor")
    out = torch.empty((B, H, W, C), dtype=torch.bfloat16, device=r.device)
    span = _Span(f"bf16 res {C}->{Cmid}->{C} {H}x{W}")
    check(lib().vqb_residual_layer_bf16(r.data_ptr(), w1_packed.data_ptr(), w2_packed.data_ptr(), out.data_ptr(),
                                        B, H, W, C, Cmid, int(bool(relu_out)), _stream()), "residual_layer_bf16")
    span.done()
    return out


def residual_layer(r, w1_packed, w2_packed, *, B, H, W, C, Cmid, relu_out, precision=FP32):
    """out = act(r + W2.relu(W1 (*) r)) on NHWC buffers (vqb_residual_layer_f32)."""
    _require_cuda(r, "input")
    out = torch.empty((B, H, W, C), dtype=torch.float32, device=r.device)
    tmp = torch.empty((B, H, W, Cmid), dtype=torch.float32, device=r.device)
    span = _Span(f"res {C}->{Cmid}->{C} {H}x{W}")
    check(lib().vqb_residual_layer_f32(r.data_ptr(), w1_packed.data_ptr(), w2_packed.data_ptr(), out.data_ptr(),
                                       tmp.data_ptr(), B, H, W, C, Cmid, int(bool(relu_out)), precision,
                                       _stream()), "residual_layer")
    span.done()
    return out


def residual_stack(r, w1_packed, w2_packed, *, B, H, W, C, Cmid, n_layers, precision=FP32):
    """n_layers applications of one shared-weight layer, each followed by ReLU, on NHWC buffers
    (vqb_residual_stack_f32; one kernel in tensor-core mode when a tile holds whole images)."""
    _require_cuda(r, "input")
    if n_layers < 1:
        return r
    out = torch.empty((B, H, W, C), dtype=torch.float32, device=r.device)
    scratch = torch.empty((B, H, W, C), dtype=torch.float32, device=r.device) if n_layers > 1 else out
    tmp = torch.empty((B, H, W, Cmid), dtype=torch.float32, device=r.device)
    span = _Span(f"res x{n_layers} {C}->{Cmid}->{C} {H}x{W}")
    check(lib().vqb_residual_stack_f32(r.data_ptr(), w1_packed.data_ptr(), w2_packed.data_ptr(), out.data_ptr(),
                                       scratch.data_ptr(), tmp.data_ptr(), B, H, W, C, Cmid, n_layers, precision,
                                       _stream()), "residual_stack")
    span.done()
    return out


def _ptr(t):
    return t.data_ptr() if t is not None else None


def latent_encoder(h, w3, b3, w1, w2, wq, bq, *, B, H, W, C, Cmid, D, n_res):
    """E3 conv 3x3 + ReLU -> residual stack -> pre-quant 1x1 as ONE kernel (vqb_latent_encoder_f32): NHWC
    relu(conv 2) in, z_e NHWC (B, H, W, D) = the VQ's rows out.  None when the shape is not covered (the caller runs
    the layers)."""
    _require_cuda(h, "input")
    z_e = torch.empty((B, H, W, D), dtype=torch.float32, device=h.device)
    span = _Span(f"latent enc {C}->{Cmid}->{D} x{n_res} {H}x{W}")
    rc = lib().vqb_latent_encoder_f32(h.data_ptr(), w3.data_ptr(), _ptr(b3), w1.data_ptr(), w2.data_ptr(), wq.data_ptr(),
                                      _ptr(bq), z_e.data_ptr(), B, H, W, C, Cmid, D, n_res, _stream())
    if rc == -2:            # VQB_ERR_UNSUPPORTED: nothing was launched
        return None
    check(rc, "latent_encoder")
    span.done()
    return z_e


def latent_decoder(zq, wt1, bt1, w1, w2, wt2, bt2, *, B, H, W, D, C, Cmid, Cout, n_res):
    """ConvT 3x3 + ReLU -> residual stack -> ConvT k4s2 + ReLU as ONE kernel (vqb_latent_decoder_f32): z_q rows in,
    NHWC (B, 2H, 2W, Cout) out.  None when the shape is not covered (the caller runs the layers)."""
    _require_cuda(zq, "input")
    out = torch.empty((B, 2 * H, 2 * W, Cout), dtype=torch.float32, device=zq.device)
    span = _Span(f"latent dec {D}->{C}->{Cout} x{n_res} {H}x{W}")
    rc = lib().vqb_latent_decoder_f32(zq.data_ptr(), wt1.data_ptr(), _ptr(bt1), w1.data_ptr(), w2.data_ptr(),
                                      wt2.data_ptr(), _ptr(bt2), out.data_ptr(), B, H, W, D, C, Cmid, Cout, n_res,
                                      _stream())
    if rc == -2:
        return None
    check(rc, "latent_decoder")
    span.done()
    return out


def vq_forward(z_rows, codebook, defer=False):
    """Fused VectorQuantizer core on (N,D) rows -> (idx int64 (N,), zq (N,D), sse f64 (1,),
    hist int32 (K,)).  defer=True (vqb_vq_forward_deferred_f32) additionally returns the workspace:
    `sse` is final only after vq_reduce_sse(ws, ...) has run (e.g. on a side stream)."""
    _require_cuda(z_rows, "z")
    N, D = z_rows.shape
    K = codebook.shape[0]
    dev = z_rows.device
    idx = torch.empty((N,), dtype=torch.int64, device=dev)
    zq = torch.empty((N, D), dtype=torch.float32, device=dev)
    sse = torch.empty((1,), dtype=torch.float64, device=dev)
    hist = torch.empty((K,), dtype=torch.int32, device=dev)
    ws_bytes = lib().vqb_vq_workspace_bytes(N, K, D)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    span = _Span(f"vq N={N} K={K} D={D}")
    fn = lib().vqb_vq_forward_deferred_f32 if defer else lib().vqb_vq_forward_f32
    check(fn(z_rows.data_ptr(), codebook.data_ptr(), N, K, D, idx.data_ptr(), zq.data_ptr(), sse.data_ptr(),
             hist.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "vq_forward")
    span.done()
    if defer:
        return idx, zq, sse, hist, ws
    return idx, zq, sse, hist


def vq_reduce_sse(ws, N, K, D, sse):
    """Completes `sse` after vq_forward(..., defer=True) (vqb_vq_reduce_sse_f32), on the current stream."""
    check(lib().vqb_vq_reduce_sse_f32(ws.data_ptr(), N, K, D, sse.data_ptr(), _stream()), "vq_reduce_sse")


def vq_finish(sse, hist, N, K, D, beta):
    """(loss, perplexity) fp32 0-dim CUDA tensors from the (all-reduced) sse / hist."""
    out = torch.empty((2,), dtype=torch.float32, device=hist.device)
    check(lib().vqb_vq_finish_f32(sse.data_ptr(), hist.data_ptr(), N, K, D, float(beta),
                                  out.data_ptr(), out.data_ptr() + 4, _stream()), "vq_finish")
    return out[0], out[1]


def vq_backward(g_zq, g_loss, z_rows, codebook, idx, beta):
    """(dz (N,D), dE (K,D)) of the VectorQuantizer forward (vqb_vq_backward_f32); g_zq / g_loss may be None."""
    _require_cuda(z_rows, "z")
    N, D = z_rows.shape
    K = codebook.shape[0]
    dz = torch.empty_like(z_rows)
    dE = torch.empty((K, D), dtype=torch.float32, device=z_rows.device)
    gz = _f32c(g_zq) if g_zq is not None else None
    gl = _f32c(g_loss).reshape(1) if g_loss is not None else None
    check(lib().vqb_vq_backward_f32(gz.data_ptr() if gz is not None else None, gl.data_ptr() if gl is not None else None,
                                    z_rows.data_ptr(), codebook.data_ptr(), idx.data_ptr(), N, K, D, float(beta),
                                    dz.data_ptr(), dE.data_ptr(), _stream()), "vq_backward")
    return dz, dE


def onehot(idx, K):
    N = idx.numel()
    out = torch.empty((N, K), dtype=torch.float32, device=idx.device)
    check(lib().vqb_onehot_f32(idx.data_ptr(), N, K, out.data_ptr(), _stream()), "onehot")
    return out


def gather_rows(idx, codebook):
    _require_cuda(idx, "indices")
    idx = idx.reshape(-1).to(torch.int64).contiguous()
    K, D = codebook.shape
    out = torch.empty((idx.numel(), D), dtype=torch.float32, device=idx.device)
    check(lib().vqb_gather_rows_f32(idx.data_ptr(), codebook.data_ptr(), idx.numel(), K, D,
                                    out.data_ptr(), _stream()), "gather_rows")
    return out


def nchw_to_nhwc(x):
    _require_cuda(x, "input")
    x = _f32c(x)
    B, C, H, W = x.shape
    out = torch.empty((B, H, W, C), dtype=torch.float32, device=x.device)
    check(lib().vqb_nchw_to_nhwc_f32(x.data_ptr(), out.data_ptr(), B, C, H, W, _stream()), "nchw_to_nhwc")
    return out


def nhwc_to_nchw(x):
    B, H, W, C = x.shape
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=x.device)
    check(lib().vqb_nhwc_to_nchw_f32(x.data_ptr(), out.data_ptr(), B, C, H, W, _stream()), "nhwc_to_nchw")
    return out


def relu_(x):
    """In-place ReLU on a contiguous fp32 CUDA tensor (residual.py:19 side effect)."""
    check(lib().vqb_relu_f32(x.data_ptr(), x.numel(), _stream()), "relu_")
    return x


VQ_KERNELS = {"auto": 0, "exact": 1, "tc": 2, "tc_r1": 3}


def set_vq_kernel(name: str):
    """Kernel used by vq_forward: "auto" (tcgen05 when D == 64), "exact" (FFMA) or "tc"."""
    check(lib().vqb_set_vq_kernel(VQ_KERNELS[name]), "set_vq_kernel")


def vq_debug_scores(z_rows, codebook):
    """Diagnostic: tcgen05 VQ kernel + dump of its approximate TF32 scores (N, Kpad)."""
    N, D = z_rows.shape
    K = codebook.shape[0]
    dev = z_rows.device
    kpad = (K + 255) // 256 * 256
    idx = torch.empty((N,), dtype=torch.int64, device=dev)
    zq = torch.empty((N, D), dtype=torch.float32, device=dev)
    sse = torch.empty((1,), dtype=torch.float64, device=dev)
    hist = torch.empty((K,), dtype=torch.int32, device=dev)
    scores = torch.full((N, kpad), float("nan"), dtype=torch.float32, device=dev)
    ws_bytes = lib().vqb_vq_workspace_bytes(N, K, D)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    check(lib().vqb_debug_vq_scores_f32(z_rows.data_ptr(), codebook.data_ptr(), N, K, D, idx.data_ptr(),
                                        zq.data_ptr(), sse.data_ptr(), hist.data_ptr(), ws.data_ptr(),
                                        ws_bytes, scores.data_ptr(), _stream()), "vq_debug_scores")
    return idx, zq, sse, hist, scores
