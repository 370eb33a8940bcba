/*
 * vqvae_b200.h -- C ABI of the B200 (sm_100a) VQ-VAE inference hot path.
 *
 * The reference (MishaLaskin/vqvae) is pure Python on top of PyTorch and exposes no
 * FFI of its own (SURVEY.md 8b); its "plugin API" for this path is the nn.Module
 * tree models.{vqvae,quantizer,encoder,decoder,residual}.  This header is the
 * boundary UNDER those modules: each entry point replaces one PyTorch operator call
 * site of the reference (file:line cited per function, paths under the reference
 * root).  models/*.py in this repo binds them with ctypes; INTEGRATION.md shows the
 * stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch in practice)
 *     unless stated otherwise;
 *     the library never allocates, frees or retains device memory;
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous, make no
 *     host synchronisation and are CUDA-graph capturable;
 *   - one CUDA device per process (the deployment model is one process per GPU,
 *     SURVEY.md 8e): the opt-in shared-memory size of each kernel is configured once
 *     per process, on the device that is current at its first launch; calls may come
 *     from any host thread but are not re-entrant on the same workspace;
 *   - host pointers appear only in vqb_device_info and vqb_memcpy_async;
 *   - return value: 0 = success, >0 = cudaError_t, <0 = vqb_status below; no C++
 *     exception crosses the boundary;
 *   - activations between layers are NHWC ("pixel rows": (B*H*W, C) row-major); the
 *     module boundary of the reference is NCHW, so every conv entry point takes an
 *     explicit layout for its input and output.
 */
#ifndef VQVAE_B200_H
#define VQVAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQB_ABI_VERSION 3

enum vqb_status {
    VQB_OK = 0,
    VQB_ERR_BAD_ARG = -1,       /* NULL pointer, non-positive size, bad enum          */
    VQB_ERR_UNSUPPORTED = -2,   /* shape outside what the kernels implement          */
    VQB_ERR_WORKSPACE = -3,     /* workspace too small (see *_workspace_bytes)       */
    VQB_ERR_NO_DEVICE = -4,     /* no sm_100 device / driver                         */
    VQB_ERR_ALIGNMENT = -5      /* pointer not aligned as documented                 */
};

enum vqb_layout { VQB_NCHW = 0, VQB_NHWC = 1 };

/* arithmetic of a convolution entry point that takes fp32 activations (vqb_conv2d_f32,
 * vqb_residual_*_f32).  VQB_BF16 names the bf16-operand pipeline, whose activations are bf16:
 * the *_f32 entry points answer VQB_ERR_UNSUPPORTED to it -- use vqb_conv2d_bf16 & co.   */
enum vqb_precision {
    VQB_FP32 = 0,  /* fp32 FFMA accumulate (CUDA cores): the reference's CPU numerics   */
    VQB_TF32 = 1,  /* tcgen05 kind::tf32, fp32 accumulate in TMEM (cuDNN's default)     */
    VQB_BF16 = 2   /* tcgen05 kind::f16 on bf16 operands and activations (bf16 entry points only) */
};

int vqb_abi_version(void);
/* 0: release library.  1: built with -DVQB_DIAG=1, which adds the in-kernel timelines of
 * tools/diag and computes the same results.  Neither reads the environment.               */
int vqb_diag_build(void);
const char *vqb_error_string(int code);
/* SM count and compute capability of the current device. */
int vqb_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* Number of kernels this process has launched through the library so far (bench.py
 * reports it as gpu_launches).                                                     */
unsigned long long vqb_launch_count(void);

/* ---- weight packing (once per load_state_dict) --------------------------------
 * nn.Conv2d weight (Cout,Cin,kh,kw)          encoder.py:29-36, residual.py:20-24,
 *                                            vqvae.py:16-17
 * nn.ConvTranspose2d weight (Cin,Cout,kh,kw) decoder.py:28-35   (transposed = 1)
 * -> `packed` holds 2*Cout*Cin*kh*kw + 144*Cin floats: the tap-major GEMM operand in both
 *    layouts the kernels read, [(r*kw+s)*Cin + ci][co] (FFMA path) followed by
 *    [(r*kw+s)][co][ci] (K-major rows for the tcgen05 path); for a k4 s2 transposed
 *    conv with Cout <= 4 a third region [9][16][Cin] (3x3-neighbourhood + pixel-shuffle
 *    form of decoder.py:34-35) follows.                                           */
int vqb_pack_conv_weight_f32(const float *w, float *packed, int Cout, int Cin, int kh,
                             int kw, int transposed, void *stream);

/* ---- convolution layers ---------------------------------------------------------
 * One call = one nn.Conv2d (transposed=0) or nn.ConvTranspose2d (transposed=1)
 * forward, optionally fused with what follows it in the reference:
 *   out = act( conv(in) + bias [+ skip] ),  act = ReLU if relu else identity
 * `skip` (NHWC, shape of out, may be NULL) implements `x + res_block(x)` of
 * residual.py:27-29; out_layout must be NHWC when skip is given.
 * w_packed comes from vqb_pack_conv_weight_f32.  Stride-2 transposed convs are run
 * as 4 sub-pixel phase launches.  Replaces: encoder.py:29-36 (stride 2/2/1, pad 1),
 * residual.py:20-24, vqvae.py:16-17 (1x1), decoder.py:28-35.                      */
int vqb_conv2d_f32(const float *in, const float *w_packed, const float *bias,
                   const float *skip, float *out, int B, int Cin, int H, int W, int Cout,
                   int kh, int kw, int stride, int pad, int transposed, int in_layout,
                   int out_layout, int relu, int precision, void *stream);

/* ---- bf16 activation path (VQB_BF16): persistent tcgen05 kind::f16 kernels ------------
 * Between layers the activations are bf16 NHWC; weights are packed to bf16 once per
 * load_state_dict; accumulation is fp32 in TMEM.  This is the arithmetic the reference
 * reaches through torch.autocast(dtype=torch.bfloat16) around vqvae.py:29-44 (SURVEY Q6).
 * The layer shapes are named, not parameterised:                                         */
enum vqb_conv_kind {
    VQB_CONV_K1 = 0,        /* nn.Conv2d k1 s1 p0           vqvae.py:16-17                 */
    VQB_CONV_K3 = 1,        /* nn.Conv2d k3 s1 p1           encoder.py:35-36               */
    VQB_CONVT_K3 = 2,       /* nn.ConvTranspose2d k3 s1 p1  decoder.py:28-29               */
    VQB_CONV_K4S2 = 3,      /* nn.Conv2d k4 s2 p1           encoder.py:32-33 (H, W even)   */
    VQB_CONVT_K4S2 = 4,     /* nn.ConvTranspose2d k4 s2 p1  decoder.py:31-32 (Cout % 32 == 0, Cout <= 128) */
    VQB_CONVT_K4S2_OUT = 5  /* same to Cout <= 4 channels, fp32 NCHW output: decoder.py:34-35 */
};
/* Bytes of the packed bf16 weight of one layer (0 = shape not covered: Cin % 64 != 0, ...). */
size_t vqb_conv_bf16_packed_bytes(int kind, int Cout, int Cin);
/* w: the layer's fp32 weight as PyTorch stores it ((Cout,Cin,kh,kw), or (Cin,Cout,kh,kw) for
 * the transposed kinds) -> `packed` (128-byte aligned): one 128-byte row of 64 input channels
 * per (k-step, output column), in the order the kernel's k-steps consume them.            */
int vqb_pack_conv_weight_bf16(const float *w, void *packed, int kind, int Cout, int Cin,
                              void *stream);
/* One layer forward on bf16 NHWC input (B,H,W,Cin):  out = act(conv(in) + bias).
 * out: bf16 NHWC, or fp32 NHWC when out_f32 != 0 (z_e for the bit-exact VQ), or fp32 NCHW
 * (B,Cout,2H,2W) for VQB_CONVT_K4S2_OUT.  All pointers 16-byte aligned.                   */
int vqb_conv2d_bf16(const void *in, const void *packed, const float *bias, void *out, int B,
                    int Cin, int H, int W, int Cout, int kind, int relu, int out_f32,
                    void *stream);

/* encoder.py:29-31 for the bf16 pipeline: fp32 NCHW image (B,3,H,W) -> bf16 NHWC (B,H/2,W/2,Cout),
 * Cout == 64; w_packed from vqb_pack_conv_weight_f32.                                       */
int vqb_conv_in_bf16(const float *x, const float *w_packed, const float *bias, void *out, int B,
                     int H, int W, int Cout, int relu, void *stream);
/* VectorQuantizer core for the bf16 pipeline: as vqb_vq_forward_deferred_f32 (fp32 z, bit-exact
 * idx, deferred SSE) but zq is written as bf16 rows (N, D); D == 64 and K <= 8192 only.      */
int vqb_vq_forward_bf16zq_f32(const float *z, const float *codebook, int64_t N, int K, int D,
                              int64_t *idx, void *zq_bf16, double *sse, int32_t *hist,
                              void *workspace, size_t workspace_bytes, void *stream);

/* One ResidualLayer application on bf16 NHWC activations (residual.py:18-29 as evaluated,
 * SURVEY Q2):  out = act( r + W2 . relu( W1 (*) r ) ),  act = ReLU iff relu_out.
 * w1_packed: vqb_pack_conv_weight_bf16(kind VQB_CONV_K3, Cout = Cmid, Cin = C) of res_block.1.weight;
 * w2_packed: vqb_pack_conv_weight_bf16(kind VQB_RES_W2 = 6, Cout = C, Cin = Cmid) of res_block.3.weight.
 * One persistent tcgen05 kernel: both GEMMs chained per tile, W1 and W2 resident in shared memory.
 * C in {64, 128}, Cmid % 16 == 0, Cmid <= 64; other shapes return VQB_ERR_UNSUPPORTED.      */
#define VQB_RES_W2 6
int vqb_residual_layer_bf16(const void *r, const void *w1_packed, const void *w2_packed, void *out,
                            int B, int H, int W, int C, int Cmid, int relu_out, void *stream);

/* ---- one ResidualLayer application, residual.py:18-29 -----------------------------
 * As the reference evaluates it (the in-place ReLU of :19 has already replaced x by
 * r = relu(x), SURVEY Q2):   out = act( r + W2 . relu( W1 (*) r ) )
 * r, out NHWC (B,H,W,C); W1 = res_block.1.weight (Cmid,C,3,3), W2 = res_block.3.weight
 * (C,Cmid,1,1), both packed by vqb_pack_conv_weight_f32; act = ReLU iff relu_out (inside
 * a ResidualStack the next consumer always applies ReLU first, residual.py:19,50).
 * tmp: B*H*W*Cmid floats of scratch (used only by the two-launch FFMA fallback).
 * With precision != VQB_FP32 and C % 32 == Cmid % 32 == 0 this is ONE tcgen05 kernel
 * (two chained GEMMs, the Cmid-channel intermediate never leaves the SM).            */
int vqb_residual_layer_f32(const float *r, const float *w1_packed, const float *w2_packed,
                           float *out, float *tmp, int B, int H, int W, int C, int Cmid,
                           int relu_out, int precision, void *stream);

/* ---- a whole ResidualStack, residual.py:45-51 --------------------------------------
 * n_layers applications of ONE shared-weight layer (residual.py:43 builds the list as
 * [layer] * n), each followed by the ReLU its consumer applies (the next layer's in-place
 * ReLU, or the stack's F.relu at :50):  r_{i+1} = relu( r_i + W2 . relu( W1 (*) r_i ) ),
 * r_0 = r = relu(stack input), out = r_{n_layers}.   r, out NHWC (B,H,W,C).
 * scratch: B*H*W*C floats (needed when n_layers > 1; used when the applications run as
 * separate launches), tmp: B*H*W*Cmid floats (FFMA fallback only).
 * With precision != VQB_FP32, whole images per 128-pixel tile (W <= 8, H <= 16) and the
 * layer shape vqb_residual_layer_f32 accepts, ALL applications run inside ONE tcgen05
 * kernel: the activation tile stays in shared memory and is rewritten in place.        */
int vqb_residual_stack_f32(const float *r, const float *w1_packed, const float *w2_packed,
                           float *out, float *scratch, float *tmp, int B, int H, int W, int C,
                           int Cmid, int n_layers, int precision, void *stream);

/* ---- the latent stage as two fused kernels (TF32), encoder.py:35-36 + residual.py + vqvae.py:16-17
 * and decoder.py:28-33 -----------------------------------------------------------------------------
 * For latents whose 128-pixel tile holds whole images (W <= 8, H <= 16): one tcgen05 kernel runs the
 * whole chain with the activation resident in shared memory, bitwise equal to the per-layer calls.
 * Weights are the vqb_pack_conv_weight_f32 buffers of the layers, biases may be NULL (= 0).
 * Encoder tail: in = relu(conv 2) NHWC (B,H,W,C) ->
 *   E3 conv 3x3 C->C +bias, ReLU -> n_res applications of the shared ResidualLayer (w1: C->Cmid 3x3,
 *   w2: Cmid->C 1x1), each followed by ReLU -> pre-quant 1x1 C->D +bias -> z_e (B*H*W, D) rows.
 * Decoder head: zq (B*H*W, D) rows ->
 *   ConvTranspose 3x3 s1 D->C +bias, ReLU -> the residual stack as above -> ConvTranspose k4 s2 p1
 *   C->Cout +bias, ReLU -> out NHWC (B,2H,2W,Cout).
 * C == 128, Cmid == 32, D == 64, Cout == 64, 1 <= n_res <= 4; pointers 16-byte aligned.  Other
 * shapes return VQB_ERR_UNSUPPORTED (the caller then runs the layers one by one).              */
int vqb_latent_encoder_f32(const float *in, const float *w3_packed, const float *b3,
                           const float *w1_packed, const float *w2_packed, const float *wq_packed,
                           const float *bq, float *z_e, int B, int H, int W, int C, int Cmid,
                           int D, int n_res, void *stream);
int vqb_latent_decoder_f32(const float *zq, const float *wt1_packed, const float *bt1,
                           const float *w1_packed, const float *w2_packed, const float *wt2_packed,
                           const float *bt2, float *out, int B, int H, int W, int D, int C,
                           int Cmid, int Cout, int n_res, void *stream);

/* ---- VectorQuantizer.forward, quantizer.py:45-76 --------------------------------
 * z        (N, D) fp32 pixel rows (= z.permute(0,2,3,1).view(-1, e_dim), :45-46)
 * codebook (K, D) fp32 embedding.weight (:26)
 * idx      (N)    int64 min_encoding_indices, first minimum wins, NaN wins (:54)
 * zq       (N, D) fp32 straight-through value fl(z + fl(e_idx - z)) (:60,:67)
 * hist     (K)    int32 code counts, ZEROED by the call (column sums of the one-hot
 *                 of :55-57; feeds the perplexity of :70-71)
 * sse      (1)    double, sum of fl(e_idx - z)^2, OVERWRITTEN by the call (numerator
 *                 of the two mean() terms of :63-64)
 * workspace       vqb_vq_workspace_bytes(N,K,D) bytes, 16-byte aligned
 * Distances follow the canonical fp32 order documented in DESIGN.md / oracle.c, so
 * idx and zq are bit-exact against the oracle.                                    */
size_t vqb_vq_workspace_bytes(int64_t N, int K, int D);
int vqb_vq_forward_f32(const float *z, const float *codebook, int64_t N, int K, int D,
                       int64_t *idx, float *zq, double *sse, int32_t *hist,
                       void *workspace, size_t workspace_bytes, void *stream);

/* Deferred variant: identical outputs, except that `sse` is only final after
 * vqb_vq_reduce_sse_f32 has run on the same workspace (stream-ordered after this call).
 * The per-CTA SSE partials stay in the workspace, so the tiny reduction -- and the scalar
 * finisher that needs it -- can run on a side stream while the decoder consumes zq
 * (vqvae.py:36 does not depend on the loss terms of quantizer.py:63-64).              */
int vqb_vq_forward_deferred_f32(const float *z, const float *codebook, int64_t N, int K, int D,
                                int64_t *idx, float *zq, double *sse, int32_t *hist,
                                void *workspace, size_t workspace_bytes, void *stream);
int vqb_vq_reduce_sse_f32(const void *workspace, int64_t N, int K, int D, double *sse,
                          void *stream);

/* Kernel choice of vqb_vq_forward_f32: 0 = auto (tcgen05 kernel when D == 64 and K <= 8192,
 * else the exact FFMA kernel), 1 = always the FFMA kernel, 2 = require the tcgen05 kernel
 * (vq2.cu; VQB_ERR_UNSUPPORTED outside its domain).  Both produce bit-identical idx / zq;
 * the switch exists for tests and benchmarks.                                         */
int vqb_set_vq_kernel(int which);

/* ---- backward of VectorQuantizer.forward, quantizer.py:63-67 (training-mode callers, main.py:74-79) ----
 * g_zq (N,D) = gradient arriving at the returned z_q (straight-through: passes to z unchanged), g_loss = device
 * scalar gradient of the returned loss (either may be NULL = zero).  Writes
 *   dz (N,D) = g_zq + g_loss * 2/(N D) * (z - E[idx])
 *   dE (K,D) = g_loss * 2 beta/(N D) * sum_{i: idx[i]=k} (E[k] - z[i])      (zeroed, then scatter-added by index)
 * argmin / one-hot / perplexity carry no gradient.  D % 4 == 0, 16-byte aligned pointers.                */
int vqb_vq_backward_f32(const float *g_zq, const float *g_loss, const float *z, const float *codebook,
                        const int64_t *idx, int64_t N, int K, int D, float beta, float *dz, float *dE,
                        void *stream);

/* loss = (1+beta)*sse/(N*D) and perplexity = exp(-sum p log(p+1e-10)), p = hist/N,
 * written as two fp32 device scalars (quantizer.py:63-64, :70-71).  Separate from
 * the VQ kernel so a batch-sharded caller can all-reduce (hist, sse) in between.  */
int vqb_vq_finish_f32(const double *sse, const int32_t *hist, int64_t N, int K, int D,
                      float beta, float *loss, float *perplexity, void *stream);

/* Dense one-hot min_encodings (N,K) fp32 for direct VectorQuantizer.forward callers
 * (quantizer.py:55-57,76); VQVAE.forward discards it (vqvae.py:34) so it is never
 * built on that path.                                                             */
int vqb_onehot_f32(const int64_t *idx, int64_t N, int K, float *onehot, void *stream);

/* z_q rows from indices: matmul(one_hot, embedding.weight) of quantizer.py:60 and of
 * the notebook's generate_samples (visualization.ipynb cell 13) as a row gather.
 * Indices outside [0, K) are clamped to the nearest valid row.                    */
int vqb_gather_rows_f32(const int64_t *idx, const float *codebook, int64_t N, int K, int D,
                        float *rows, void *stream);

/* In-place ReLU over n floats: the nn.ReLU(True) of residual.py:19, which mutates
 * the caller's tensor when a ResidualLayer is called directly (SURVEY Q2).         */
int vqb_relu_f32(float *x, int64_t n, void *stream);

/* ---- layout changes at the module boundary (quantizer.py:45, :74) ---------------- */
int vqb_nchw_to_nhwc_f32(const float *in, float *out, int B, int C, int H, int W, void *stream);
int vqb_nhwc_to_nchw_f32(const float *in, float *out, int B, int C, int H, int W, void *stream);

/* Stream-ordered copy used by the host-buffer streaming front end (vqvae_b200.HostPipeline):
 * kind 1 = host -> device, 2 = device -> host, 3 = device -> device.  Host buffers should be
 * pinned (the copy is only asynchronous then).                                          */
int vqb_memcpy_async(void *dst, const void *src, size_t bytes, int kind, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* VQVAE_B200_H */
