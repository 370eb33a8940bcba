"""Host-side mirror of the reference's nn.Module API for the VQVAE.forward hot path.

Same class names, constructor signatures, attribute names and state-dict keys as
MishaLaskin/vqvae ``models/{vqvae,quantizer,encoder,decoder,residual}.py`` (SURVEY 8b),
so ``from models.vqvae import VQVAE`` keeps working (the top-level ``models`` package
re-exports these classes).  The nn.Conv2d / nn.ConvTranspose2d / nn.Embedding children
are kept ONLY as parameter containers (identical init order => identical weights under
the same torch seed, identical ``state_dict()``); their own ``forward`` is never used.
Every ``forward`` here launches the hand-written sm_100a kernels through the C ABI
(``include/vqvae_b200.h``).  Inference only: outputs carry no autograd graph.

Reference semantics reproduced on purpose (SURVEY 3.3):
  Q1  ResidualStack applies ONE shared ResidualLayer n times (residual.py:44-45)
  Q2  the in-place ReLU makes a layer relu(x) + f(relu(x)) and mutates the caller's x
  Q3  final F.relu after the stack; no activation after encoder conv 4 / decoder convT 0
  Q4  z_q is bitwise z + (e - z)
  Q7  the dense one-hot is built only for direct VectorQuantizer.forward callers
  Q8  verbose=True prints three shapes and then ``assert False``
"""
import contextlib

import torch
import torch.nn as nn

from . import ops
from .dist import reduce_vq_stats
from ._lib import (CONV_K1, CONV_K3, CONV_K4S2, CONVT_K3, CONVT_K4S2, CONVT_K4S2_OUT, NCHW, NHWC, PRECISIONS,
                   RES_W2, TF32)

# Default = what the reference itself computes on a GPU: fp32 tensors, convolutions on tensor cores in TF32 with fp32
# accumulation (PyTorch's torch.backends.cudnn.allow_tf32 default, SURVEY 2.2), bit-exact fp32 VQ.
DEFAULT_PRECISION = "tf32"
_PRECISION = {"value": DEFAULT_PRECISION}


def set_precision(name: str):
    """Arithmetic of the convolution layers:
    "tf32" (default) tcgen05 kind::tf32 on fp32 activations, fp32 accumulation -- the reference's GPU arithmetic;
    "fp32"  FFMA on CUDA cores -- the reference's CPU numerics (end-to-end indices equal the CPU reference);
    "bf16"  bf16 activations and operands between layers (tcgen05 kind::f16), fp32 accumulation -- the arithmetic the
            reference reaches through torch.autocast(dtype=torch.bfloat16); fastest.
    The VQ distances / argmin are bit-exact fp32 in every mode."""
    if name not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}")
    _PRECISION["value"] = name


def get_precision() -> str:
    return _PRECISION["value"]


@contextlib.contextmanager
def precision(name: str):
    old = get_precision()
    set_precision(name)
    try:
        yield
    finally:
        set_precision(old)


def _param_tag(param):
    """Identity of a parameter's current value as far as torch tracks it.  ``.data`` edits (``w.data.mul_()``) do
    not bump ``_version`` and inference-mode tensors have no version counter at all: call
    ``vqvae_b200.invalidate_packed(model)`` after such edits (documented in INTEGRATION.md)."""
    try:
        ver = param._version
    except RuntimeError:            # "Inference tensors do not track version counter"
        ver = None
    return (ver, param.data_ptr(), str(param.device))


class _PackedWeights:
    """Packed conv weights cached ON the parameter object (so the cache dies with it) per packing kind:
    ("f32", transposed) = the tap-major fp32 layouts of vqb_pack_conv_weight_f32, ("bf16", kind) = the k-step-ordered
    bf16 layout of vqb_pack_conv_weight_bf16.  When the parameter changes (load_state_dict, optimizer step, .to())
    the SAME device buffer is repacked in place whenever its size still fits, so CUDA graphs captured around a
    forward keep reading current weights after ``repack`` (HostPipeline checks the tags before every replay)."""

    def get(self, param, key):
        tag = _param_tag(param)
        cache = getattr(param, "_vqb_packed", None)
        if cache is None:
            cache = {}
            param._vqb_packed = cache
        hit = cache.get(key)
        if hit is not None and hit[0] == tag and tag[0] is not None:
            return hit[1]
        old = hit[1] if hit is not None and hit[1] is not None and hit[1].device == param.device else None
        if key[0] == "f32":
            buf = ops.pack_conv_weight(param, key[1], out=old)
        else:
            buf = ops.pack_conv_weight_bf16(param, key[1], out=old)
        cache[key] = (tag, buf)
        return buf

    def f32(self, param, transposed):
        return self.get(param, ("f32", bool(transposed)))

    def bf16(self, param, kind):
        return self.get(param, ("bf16", int(kind)))


_PACKED = _PackedWeights()


_INVALIDATIONS = {"n": 0}


def invalidate_packed(model):
    """Drop every cached weight packing of ``model`` (after ``param.data`` edits, which torch does not version).
    Buffers are kept and refilled in place at the next forward / ``HostPipeline.push``."""
    _INVALIDATIONS["n"] += 1
    for p in model.parameters():
        cache = getattr(p, "_vqb_packed", None)
        if cache:
            for k, (tag, buf) in list(cache.items()):
                cache[k] = ((None, None, None), buf)


def packed_state(model):
    """Tuple of the parameters' tags: changes whenever a weight packing may be stale."""
    return tuple(_param_tag(p) for p in model.parameters())


def _conv_precision():
    """Arithmetic of the fp32-activation entry points (vqb_conv2d_f32 & co): "bf16" has no meaning for them -- bf16
    operands exist only inside the fused VQVAE.forward / encode / decode pipeline -- so piecewise sub-module calls
    run the TF32 kernels in that mode (more accurate than asked, never less)."""
    name = get_precision()
    return PRECISIONS["tf32" if name == "bf16" else name]


def _bias(conv):
    if conv.bias is None:
        return None
    b = conv.bias.detach()
    return b if b.dtype == torch.float32 else b.float()


def _run_conv(conv, x, B, H, W, *, in_layout=NHWC, out_layout=NHWC, relu=False, skip=None):
    """Forward of one nn.Conv2d / nn.ConvTranspose2d container through vqb_conv2d_f32."""
    transposed = isinstance(conv, nn.ConvTranspose2d)
    kh, kw = conv.kernel_size
    stride, pad = conv.stride[0], conv.padding[0]
    w = _PACKED.f32(conv.weight, transposed)
    return ops.conv2d(x, w, _bias(conv), B=B, Cin=conv.in_channels, H=H, W=W, Cout=conv.out_channels,
                      kh=kh, kw=kw, stride=stride, pad=pad, transposed=transposed, in_layout=in_layout,
                      out_layout=out_layout, relu=relu, skip=skip,
                      precision=_conv_precision())


def _prep_input(x, channels, what):
    if x.dim() != 4:
        raise RuntimeError(f"{what}: expected a 4-D (B,C,H,W) tensor, got {tuple(x.shape)}")
    if x.shape[1] != channels:
        raise RuntimeError(f"{what}: expected {channels} input channels, got {x.shape[1]}")
    ops._require_cuda(x, what + " input")
    x = x.detach()
    if x.dtype != torch.float32:
        x = x.float()
    return x if x.is_contiguous() else x.contiguous()


class ResidualLayer(nn.Module):
    """One residual layer (reference models/residual.py:8-29)."""

    def __init__(self, in_dim, h_dim, res_h_dim):
        super().__init__()
        self.res_block = nn.Sequential(
            nn.ReLU(True),
            nn.Conv2d(in_dim, res_h_dim, kernel_size=3, stride=1, padding=1, bias=False),
            nn.ReLU(True),
            nn.Conv2d(res_h_dim, h_dim, kernel_size=1, stride=1, bias=False),
        )

    def _apply_nhwc(self, r, B, H, W, relu_out):
        """r = relu(x) in NHWC.  Returns r + W2.relu(W1 (*) r), optionally ReLU'd
        (the next consumer always applies ReLU first, residual.py:19,50)."""
        c1, c2 = self.res_block[1], self.res_block[3]
        return ops.residual_layer(r, _PACKED.f32(c1.weight, False), _PACKED.f32(c2.weight, False), B=B, H=H, W=W,
                                  C=c1.in_channels, Cmid=c1.out_channels, relu_out=relu_out,
                                  precision=_conv_precision())

    def forward(self, x):
        xin = x
        x = _prep_input(x, self.res_block[1].in_channels, "ResidualLayer")
        B, _, H, W = x.shape
        # Q2: nn.ReLU(True) rewrites the caller's tensor before the sum is formed.
        if xin.is_contiguous() and xin.dtype == torch.float32 and not xin.requires_grad:
            ops.relu_(xin)
            x = xin
        else:
            x = ops.relu_(x.clone())
        r = ops.nchw_to_nhwc(x)
        return ops.nhwc_to_nchw(self._apply_nhwc(r, B, H, W, relu_out=False))


class ResidualStack(nn.Module):
    """n applications of ONE shared ResidualLayer, then ReLU (models/residual.py:32-51)."""

    def __init__(self, in_dim, h_dim, res_h_dim, n_res_layers):
        super().__init__()
        self.n_res_layers = n_res_layers
        self.stack = nn.ModuleList([ResidualLayer(in_dim, h_dim, res_h_dim)] * n_res_layers)

    def _apply_nhwc(self, r, B, H, W):
        """r = relu(stack input), NHWC.  Output = the stack's result (post F.relu)."""
        if len(self.stack) == 0:
            return r
        layer = self.stack[0]
        if any(l is not layer for l in self.stack):      # not the reference's [layer] * n construction
            for l in self.stack:
                r = l._apply_nhwc(r, B, H, W, relu_out=True)
            return r
        c1, c2 = layer.res_block[1], layer.res_block[3]
        return ops.residual_stack(r, _PACKED.f32(c1.weight, False), _PACKED.f32(c2.weight, False), B=B, H=H, W=W,
                                  C=c1.in_channels, Cmid=c1.out_channels, n_layers=len(self.stack),
                                  precision=_conv_precision())

    def _shared_layer(self):
        """(conv 3x3, conv 1x1, n) of the reference's ``[layer] * n`` construction, else None."""
        if len(self.stack) == 0 or any(l is not self.stack[0] for l in self.stack):
            return None
        layer = self.stack[0]
        return layer.res_block[1], layer.res_block[3], len(self.stack)

    def _bf16_ok(self):
        if len(self.stack) == 0:
            return True
        layer = self.stack[0]
        c1 = layer.res_block[1]
        return all(l is layer for l in self.stack) and c1.in_channels in (64, 128) and \
            c1.out_channels % 16 == 0 and c1.out_channels <= 64

    def _apply_nhwc_bf16(self, r, B, H, W):
        """bf16 NHWC twin of _apply_nhwc: one persistent tcgen05 kernel per application of the shared layer."""
        if len(self.stack) == 0:
            return r
        c1, c2 = self.stack[0].res_block[1], self.stack[0].res_block[3]
        w1, w2 = _PACKED.bf16(c1.weight, CONV_K3), _PACKED.bf16(c2.weight, RES_W2)
        for _ in range(len(self.stack)):
            r = ops.residual_layer_bf16(r, w1, w2, B=B, H=H, W=W, C=c1.in_channels, Cmid=c1.out_channels, relu_out=True)
        return r

    def forward(self, x):
        ch = self.stack[0].res_block[1].in_channels if len(self.stack) else x.shape[1]
        xin = x
        x = _prep_input(x, ch, "ResidualStack")
        B, _, H, W = x.shape
        if len(self.stack) and xin.is_contiguous() and xin.dtype == torch.float32 \
                and not xin.requires_grad:
            ops.relu_(xin)      # side effect of the first layer's in-place ReLU (Q2)
            x = xin
        else:
            x = ops.relu_(x.clone())
        return ops.nhwc_to_nchw(self._apply_nhwc(ops.nchw_to_nhwc(x), B, H, W))


class Encoder(nn.Module):
    """q_theta(z|x): models/encoder.py:9-43."""

    def __init__(self, in_dim, h_dim, n_res_layers, res_h_dim):
        super().__init__()
        kernel, stride = 4, 2
        self.conv_stack = nn.Sequential(
            nn.Conv2d(in_dim, h_dim // 2, kernel_size=kernel, stride=stride, padding=1),
            nn.ReLU(),
            nn.Conv2d(h_dim // 2, h_dim, kernel_size=kernel, stride=stride, padding=1),
            nn.ReLU(),
            nn.Conv2d(h_dim, h_dim, kernel_size=kernel - 1, stride=stride - 1, padding=1),
            ResidualStack(h_dim, h_dim, res_h_dim, n_res_layers),
        )

    def _head_nhwc(self, x):
        """x: prepared NCHW fp32 CUDA tensor -> (NHWC output of conv 2 after its ReLU, B, H, W)."""
        B, _, H, W = x.shape
        cs = self.conv_stack
        h = _run_conv(cs[0], x, B, H, W, in_layout=NCHW, relu=True)
        H, W = h.shape[1], h.shape[2]
        h = _run_conv(cs[2], h, B, H, W, relu=True)
        return h, B, h.shape[1], h.shape[2]

    def _tail_nhwc(self, h, B, H, W):
        """conv 4 and the stack, one launch per layer: NHWC in -> NHWC stack output."""
        cs = self.conv_stack
        # the only consumer of conv 4 is the stack, whose first op is ReLU (or, with an
        # empty stack, its final F.relu): fold that ReLU into this epilogue (Q2/Q3).
        h = _run_conv(cs[4], h, B, H, W, relu=True)
        return cs[5]._apply_nhwc(h, B, H, W)

    def _forward_nhwc(self, x):
        """x: prepared NCHW fp32 CUDA tensor -> (NHWC activation, B, H, W)."""
        h, B, H, W = self._head_nhwc(x)
        return self._tail_nhwc(h, B, H, W), B, H, W

    def _fused_tail(self, h, B, H, W, pq):
        """conv 4 -> stack -> ``pq`` (the pre-quant 1x1) as one kernel, z_e NHWC out: tf32 arithmetic, a shared-weight
        stack and a latent whose tiles hold whole images.  None when not covered (the caller runs the layers)."""
        st = self.conv_stack[5]._shared_layer()
        if _conv_precision() != TF32 or st is None:
            return None
        c1, c2, n = st
        e3 = self.conv_stack[4]
        return ops.latent_encoder(h, _PACKED.f32(e3.weight, False), _bias(e3), _PACKED.f32(c1.weight, False),
                                  _PACKED.f32(c2.weight, False), _PACKED.f32(pq.weight, False), _bias(pq), B=B, H=H,
                                  W=W, C=e3.in_channels, Cmid=c1.out_channels, D=pq.out_channels, n_res=n)

    def _bf16_ok(self):
        cs = self.conv_stack
        return (cs[0].in_channels == 3 and cs[0].out_channels == 64 and cs[2].out_channels % 16 == 0
                and cs[2].out_channels <= 256 and cs[4].in_channels % 64 == 0 and cs[4].in_channels <= 512
                and cs[5]._bf16_ok())

    def _forward_nhwc_bf16(self, x):
        """VQB_BF16 pipeline: fp32 NCHW image -> bf16 NHWC latent activation (ReLU of the stack applied)."""
        B, _, H, W = x.shape
        cs = self.conv_stack
        h = ops.conv_in_bf16(x, _PACKED.f32(cs[0].weight, False), _bias(cs[0]), B=B, H=H, W=W, Cout=cs[0].out_channels, relu=True)
        H, W = H // 2, W // 2
        h = ops.conv2d_bf16(h, _PACKED.bf16(cs[2].weight, CONV_K4S2), _bias(cs[2]), B=B, Cin=cs[2].in_channels, H=H, W=W,
                            Cout=cs[2].out_channels, kind=CONV_K4S2, relu=True)
        H, W = H // 2, W // 2
        h = ops.conv2d_bf16(h, _PACKED.bf16(cs[4].weight, CONV_K3), _bias(cs[4]), B=B, Cin=cs[4].in_channels, H=H, W=W,
                            Cout=cs[4].out_channels, kind=CONV_K3, relu=True)      # the stack's first ReLU folded in (Q2/Q3)
        h = cs[5]._apply_nhwc_bf16(h, B, H, W)
        return h, B, H, W

    def forward(self, x):
        x = _prep_input(x, self.conv_stack[0].in_channels, "Encoder")
        h, _, _, _ = self._forward_nhwc(x)
        return ops.nhwc_to_nchw(h)


class Decoder(nn.Module):
    """p_phi(x|z): models/decoder.py:9-39."""

    def __init__(self, in_dim, h_dim, n_res_layers, res_h_dim):
        super().__init__()
        kernel, stride = 4, 2
        self.inverse_conv_stack = nn.Sequential(
            nn.ConvTranspose2d(in_dim, h_dim, kernel_size=kernel - 1, stride=stride - 1, padding=1),
            ResidualStack(h_dim, h_dim, res_h_dim, n_res_layers),
            nn.ConvTranspose2d(h_dim, h_dim // 2, kernel_size=kernel, stride=stride, padding=1),
            nn.ReLU(),
            nn.ConvTranspose2d(h_dim // 2, 3, kernel_size=kernel, stride=stride, padding=1),
        )

    def _forward_from_nhwc(self, z, B, H, W):
        """z: NHWC (B,H,W,in_dim) -> x_hat NCHW."""
        ics = self.inverse_conv_stack
        h = self._fused_head(z, B, H, W)
        if h is None:
            h = _run_conv(ics[0], z, B, H, W, relu=True)     # ReLU of the stack folded in (Q2/Q3)
            H, W = h.shape[1], h.shape[2]
            h = ics[1]._apply_nhwc(h, B, H, W)
            h = _run_conv(ics[2], h, B, H, W, relu=True)
        H, W = h.shape[1], h.shape[2]
        return _run_conv(ics[4], h, B, H, W, out_layout=NCHW)

    def _fused_head(self, z, B, H, W):
        """convT 0 -> stack -> convT 2 (+ReLU) as one kernel: tf32 arithmetic, a shared-weight stack and a latent whose
        tiles hold whole images.  None when not covered (the caller runs the layers)."""
        ics = self.inverse_conv_stack
        st = ics[1]._shared_layer()
        if _conv_precision() != TF32 or st is None:
            return None
        c1, c2, n = st
        return ops.latent_decoder(z, _PACKED.f32(ics[0].weight, True), _bias(ics[0]), _PACKED.f32(c1.weight, False),
                                  _PACKED.f32(c2.weight, False), _PACKED.f32(ics[2].weight, True), _bias(ics[2]), B=B,
                                  H=H, W=W, D=ics[0].in_channels, C=ics[0].out_channels, Cmid=c1.out_channels,
                                  Cout=ics[2].out_channels, n_res=n)

    def _bf16_ok(self):
        ics = self.inverse_conv_stack
        return (ics[0].in_channels % 64 == 0 and ics[0].out_channels % 16 == 0 and ics[0].out_channels <= 256
                and ics[1]._bf16_ok() and ics[2].in_channels % 64 == 0 and ics[2].out_channels % 32 == 0
                and ics[2].out_channels <= 128 and ics[4].in_channels % 64 == 0 and ics[4].out_channels <= 4)

    def _forward_from_nhwc_bf16(self, z, B, H, W):
        """z: bf16 NHWC (B,H,W,in_dim) -> x_hat fp32 NCHW, every layer on the bf16 tcgen05 kernels."""
        ics = self.inverse_conv_stack
        h = ops.conv2d_bf16(z, _PACKED.bf16(ics[0].weight, CONVT_K3), _bias(ics[0]), B=B, Cin=ics[0].in_channels, H=H, W=W,
                            Cout=ics[0].out_channels, kind=CONVT_K3, relu=True)
        h = ics[1]._apply_nhwc_bf16(h, B, H, W)
        h = ops.conv2d_bf16(h, _PACKED.bf16(ics[2].weight, CONVT_K4S2), _bias(ics[2]), B=B, Cin=ics[2].in_channels, H=H, W=W,
                            Cout=ics[2].out_channels, kind=CONVT_K4S2, relu=True)
        H, W = 2 * H, 2 * W
        return ops.conv2d_bf16(h, _PACKED.bf16(ics[4].weight, CONVT_K4S2_OUT), _bias(ics[4]), B=B, Cin=ics[4].in_channels,
                               H=H, W=W, Cout=ics[4].out_channels, kind=CONVT_K4S2_OUT, relu=False)

    def forward(self, x):
        x = _prep_input(x, self.inverse_conv_stack[0].in_channels, "Decoder")
        B, _, H, W = x.shape
        return self._forward_from_nhwc(ops.nchw_to_nhwc(x), B, H, W)


class _VQFunction(torch.autograd.Function):
    """Training-mode VectorQuantizer core (SURVEY 8f rank 3): the fused forward kernel plus vqb_vq_backward_f32 --
    straight-through gradient to z, commitment / codebook gradients scatter-added by index (quantizer.py:63-67)."""

    @staticmethod
    def forward(ctx, z_rows, codebook, beta):
        z_rows, codebook = z_rows.detach().contiguous(), codebook.detach().contiguous()
        idx, zq, sse, hist = ops.vq_forward(z_rows, codebook)
        N, D = z_rows.shape
        loss, perp = ops.vq_finish(sse, hist, N, codebook.shape[0], D, beta)
        ctx.save_for_backward(z_rows, codebook, idx)
        ctx.beta = beta
        ctx.mark_non_differentiable(perp, idx)
        return loss, zq, perp, idx

    @staticmethod
    def backward(ctx, g_loss, g_zq, _g_perp, _g_idx):
        z_rows, codebook, idx = ctx.saved_tensors
        dz, dE = ops.vq_backward(g_zq, g_loss, z_rows, codebook, idx, ctx.beta)
        return dz, dE, None


class VectorQuantizer(nn.Module):
    """Discretisation bottleneck: models/quantizer.py:10-76."""

    def __init__(self, n_e, e_dim, beta):
        super().__init__()
        self.n_e = n_e
        self.e_dim = e_dim
        self.beta = beta
        self.embedding = nn.Embedding(self.n_e, self.e_dim)
        self.embedding.weight.data.uniform_(-1.0 / self.n_e, 1.0 / self.n_e)

    def _codebook(self):
        w = self.embedding.weight.detach()
        if w.dtype != torch.float32:
            w = w.float()
        return w if w.is_contiguous() else w.contiguous()

    def _scalars(self, sse, hist, n_local, group=None):
        """(loss, perplexity) from the VQ kernel's sufficient statistics (quantizer.py:63-64, :70-71)."""
        n_total = n_local
        if group is not None and torch.distributed.get_world_size(group) > 1:
            # batch-sharded forward (SURVEY 8e): loss and perplexity are the only
            # cross-sample quantities; reduce their sufficient statistics.
            # one tiny all-reduce of [hist (K) | sse]; shards are equal-sized (contiguous batch
            # split), so the global row count is n_local * world_size: no host sync needed
            hist, sse = reduce_vq_stats(hist, sse, group)
            n_total = n_total * torch.distributed.get_world_size(group)
        return ops.vq_finish(sse, hist, n_total, self.n_e, self.e_dim, self.beta)

    def _quantize_rows(self, rows, group=None):
        """rows (N, e_dim) fp32 CUDA -> (loss, zq_rows, perplexity, idx (N,))."""
        idx, zq, sse, hist = ops.vq_forward(rows, self._codebook())
        loss, perp = self._scalars(sse, hist, rows.shape[0], group)
        return loss, zq, perp, idx

    def _forward_train(self, z):
        """Differentiable path (z or the codebook requires grad): same kernels, gradients through _VQFunction; the
        NCHW <-> row layout changes are plain torch views/copies so autograd carries them."""
        if z.dim() != 4 or z.shape[1] != self.e_dim:
            raise RuntimeError(f"VectorQuantizer: expected (B,{self.e_dim},H,W), got {tuple(z.shape)}")
        ops._require_cuda(z, "VectorQuantizer input")
        B, D, H, W = z.shape
        rows = z.float().permute(0, 2, 3, 1).contiguous().view(-1, D)                   # quantizer.py:45-46
        loss, zq, perp, idx = _VQFunction.apply(rows, self.embedding.weight.float(), float(self.beta))
        z_q = zq.view(B, H, W, D).permute(0, 3, 1, 2).contiguous()                      # :74
        return loss, z_q, perp, ops.onehot(idx, self.n_e), idx.view(-1, 1)

    def forward(self, z):
        if torch.is_grad_enabled() and (z.requires_grad or self.embedding.weight.requires_grad) and z.is_cuda:
            return self._forward_train(z)
        z = _prep_input(z, self.e_dim, "VectorQuantizer")   # Q11: channels must equal e_dim
        B, D, H, W = z.shape
        rows = ops.nchw_to_nhwc(z).view(-1, D)                              # quantizer.py:45-46
        loss, zq, perp, idx = self._quantize_rows(rows)
        z_q = ops.nhwc_to_nchw(zq.view(B, H, W, D))                         # :74
        min_encoding_indices = idx.view(-1, 1)                              # :54
        min_encodings = ops.onehot(idx, self.n_e)                           # :55-57 (Q7)
        return loss, z_q, perp, min_encodings, min_encoding_indices


class _PointwiseConv2d(nn.Conv2d):
    """nn.Conv2d container whose forward runs vqb_conv2d_f32 (vqvae.py:16-17,33)."""

    def forward(self, x):
        x = _prep_input(x, self.in_channels, "pre_quantization_conv")
        B, _, H, W = x.shape
        return _run_conv(self, x, B, H, W, in_layout=NCHW, out_layout=NCHW)


class VQVAE(nn.Module):
    """models/vqvae.py:10-44."""

    def __init__(self, h_dim, res_h_dim, n_res_layers, n_embeddings, embedding_dim, beta,
                 save_img_embedding_map=False):
        super().__init__()
        self.encoder = Encoder(3, h_dim, n_res_layers, res_h_dim)
        self.pre_quantization_conv = _PointwiseConv2d(h_dim, embedding_dim, kernel_size=1, stride=1)
        self.vector_quantization = VectorQuantizer(n_embeddings, embedding_dim, beta)
        self.decoder = Decoder(embedding_dim, h_dim, n_res_layers, res_h_dim)
        if save_img_embedding_map:
            self.img_to_embedding_map = {i: [] for i in range(n_embeddings)}
        else:
            self.img_to_embedding_map = None
        # batch-sharded inference: set to a torch.distributed process group so that
        # embedding_loss / perplexity equal the single-process values (SURVEY 8e)
        self.process_group = None
        # True: every sharded forward all-reduces the VQ statistics (one 4 KB collective per step: every step is a
        # rank rendezvous).  False: forward returns THIS SHARD's loss / perplexity and keeps the statistics;
        # reduce_scalars() all-reduces them on demand (e.g. every M steps, or when a caller reads the scalars).
        self.sync_scalars = True
        self.last_vq_stats = None            # (hist int32 (K,), sse f64 (1,), rows of this shard) of the last forward
        self._side_stream = None
        self.last_min_encoding_indices = None

    def _bf16_pipeline(self):
        """True when set_precision("bf16") is active AND every layer of this model has a bf16 tcgen05 kernel
        (h_dim = 128 family: 64-channel first layer, channel counts in multiples of 64, embedding_dim = 64,
        n_embeddings <= 8192 for the VQ kernel that writes bf16 z_q).
        Other shapes run the TF32 kernels on fp32 activations, with a one-time warning."""
        if get_precision() != "bf16":
            return False
        pq = self.pre_quantization_conv
        vq = self.vector_quantization
        ok = (self.encoder._bf16_ok() and self.decoder._bf16_ok() and pq.in_channels % 64 == 0
              and pq.out_channels == 64 and vq.e_dim == 64 and vq.n_e <= 8192)
        if not ok and not getattr(self, "_warned_bf16", False):
            import warnings
            warnings.warn("vqvae_b200: this model shape has no bf16 kernels; precision 'bf16' runs the TF32 kernels")
            self._warned_bf16 = True
        return ok

    def _encode_rows(self, x, bf16=False):
        x = _prep_input(x, 3, "VQVAE")
        if x.shape[2] % 4 or x.shape[3] % 4:
            raise RuntimeError("VQVAE: image height and width must be divisible by 4 (Q11)")
        if bf16:
            h, B, H, W = self.encoder._forward_nhwc_bf16(x)
            pq = self.pre_quantization_conv
            z_e = ops.conv2d_bf16(h, _PACKED.bf16(pq.weight, CONV_K1), _bias(pq), B=B, Cin=pq.in_channels, H=H, W=W,
                                  Cout=pq.out_channels, kind=CONV_K1, relu=False, out_f32=True)   # fp32: feeds the exact VQ
            return z_e, B, H, W
        h, B, H, W = self.encoder._head_nhwc(x)
        z_e = self.encoder._fused_tail(h, B, H, W, self.pre_quantization_conv)
        if z_e is None:
            h = self.encoder._tail_nhwc(h, B, H, W)
            z_e = _run_conv(self.pre_quantization_conv, h, B, H, W)          # NHWC (B,H,W,D)
        return z_e, B, H, W

    def forward(self, x, verbose=False):
        bf16 = self._bf16_pipeline()
        z_e, B, H, W = self._encode_rows(x, bf16)                            # vqvae.py:31-33
        vq = self.vector_quantization
        D = vq.e_dim
        group = self.process_group
        # The decoder does not depend on the loss / perplexity scalars (vqvae.py:36 vs quantizer.py:63-71), so
        # the SSE reduction, the batch-sharded all-reduce (SURVEY 8e) and the scalar finisher run on a side
        # stream and overlap the decoder; fork/join with events, so the whole forward stays capturable in one
        # CUDA graph.
        n_rows = z_e.shape[0] * H * W
        if bf16:
            idx, zq, sse, hist, ws = ops.vq_forward_bf16zq(z_e.view(-1, D), vq._codebook())
        else:
            idx, zq, sse, hist, ws = ops.vq_forward(z_e.view(-1, D), vq._codebook(), defer=True)
        main = torch.cuda.current_stream()
        if self._side_stream is None or self._side_stream.device != z_e.device:
            self._side_stream = torch.cuda.Stream(device=z_e.device)
        side = self._side_stream
        side.wait_stream(main)
        with torch.cuda.stream(side):
            ops.vq_reduce_sse(ws, n_rows, vq.n_e, D, sse)
            embedding_loss, perplexity = vq._scalars(sse, hist, n_rows, group if self.sync_scalars else None)
            self.last_vq_stats = (hist, sse, n_rows)
            if not torch.cuda.is_current_stream_capturing():
                for t in (ws, sse, hist, embedding_loss, perplexity):
                    t.record_stream(side)
        if bf16:
            x_hat = self.decoder._forward_from_nhwc_bf16(zq.view(B, H, W, D), B, H, W)
        else:
            x_hat = self.decoder._forward_from_nhwc(zq.view(B, H, W, D), B, H, W)  # :36
        main.wait_stream(side)
        if not torch.cuda.is_current_stream_capturing():
            # the two scalars were allocated in the side stream's pool and are consumed on the caller's stream: without this
            # their block could be handed out again on the side stream while the caller still reads them (ADVICE r1)
            embedding_loss.record_stream(main)
            perplexity.record_stream(main)
        self.last_min_encoding_indices = idx.view(-1, 1)
        if verbose:                                                          # :38-42 (Q8)
            print('original data shape:', x.shape)
            print('encoded data shape:', torch.Size((B, D, H, W)))
            print('recon data shape:', x_hat.shape)
            assert False
        return embedding_loss, x_hat, perplexity

    def reduce_scalars(self):
        """(embedding_loss, perplexity) over the WHOLE sharded batch from the statistics of the last forward: the one
        collective of the path (SURVEY 8e), issued on demand when ``sync_scalars`` is False.  Equals the
        single-process values on the concatenated batch (tests/test_dist_cpu.py, tests/test_gpu_dist.py)."""
        if self.last_vq_stats is None:
            raise RuntimeError("reduce_scalars: no forward has run yet")
        hist, sse, n_rows = self.last_vq_stats
        return self.vector_quantization._scalars(sse, hist, n_rows, self.process_group)

    def repack(self):
        """Refresh every cached weight packing whose parameter changed (load_state_dict, optimizer step), IN PLACE
        in the buffers earlier forwards -- and CUDA graphs captured around them -- already read.  A plain forward
        does this by itself; HostPipeline calls it before replaying a captured graph."""
        enc, dec, pq = self.encoder.conv_stack, self.decoder.inverse_conv_stack, self.pre_quantization_conv
        bf16 = self._bf16_pipeline()
        _PACKED.f32(enc[0].weight, False)
        stacks = [s for s in (enc[5], dec[1]) if len(s.stack)]
        if bf16:
            _PACKED.bf16(enc[2].weight, CONV_K4S2); _PACKED.bf16(enc[4].weight, CONV_K3); _PACKED.bf16(pq.weight, CONV_K1)
            _PACKED.bf16(dec[0].weight, CONVT_K3); _PACKED.bf16(dec[2].weight, CONVT_K4S2)
            _PACKED.bf16(dec[4].weight, CONVT_K4S2_OUT)
            for st in stacks:
                _PACKED.bf16(st.stack[0].res_block[1].weight, CONV_K3); _PACKED.bf16(st.stack[0].res_block[3].weight, RES_W2)
        else:
            for conv in (enc[2], enc[4], pq):
                _PACKED.f32(conv.weight, False)
            for conv in (dec[0], dec[2], dec[4]):
                _PACKED.f32(conv.weight, True)
            for st in stacks:
                for layer in set(st.stack):
                    _PACKED.f32(layer.res_block[1].weight, False); _PACKED.f32(layer.res_block[3].weight, False)

    # ---- SURVEY 8(f) rank 1: the two halves callers use around the path ----------
    def encode(self, x):
        """images -> min_encoding_indices (N,1) int64 (README step 2 / notebook cell 1)."""
        z_e, B, H, W = self._encode_rows(x, self._bf16_pipeline())
        _, _, _, idx = self.vector_quantization._quantize_rows(z_e.view(-1, self.vector_quantization.e_dim))
        return idx.view(-1, 1)

    def decode(self, indices, latent_hw):
        """min_encoding_indices -> images (notebook cell 13 ``generate_samples``): the
        one-hot matmul replaced by a codebook row gather."""
        H, W = latent_hw
        vq = self.vector_quantization
        rows = ops.gather_rows(indices, vq._codebook())
        B = rows.shape[0] // (H * W)
        if self._bf16_pipeline():
            return self.decoder._forward_from_nhwc_bf16(rows.to(torch.bfloat16).view(B, H, W, vq.e_dim), B, H, W)
        return self.decoder._forward_from_nhwc(rows.view(B, H, W, vq.e_dim), B, H, W)
