// api.cu -- the extern "C" boundary declared in include/vqvae_b200.h.
#include "common.cuh"

size_t vq_exact_workspace_bytes(int K);
int launch_vq_exact(const float *z, const float *E, long long N, int K, int D, long long *idx, float *zq,
                    double *sse, int *hist, void *ws, cudaStream_t s);

size_t vq2_workspace_bytes(int K);
size_t vq_ws_marker_offset(int K);
int launch_vq_reduce_sse(const void *ws, int K, double *sse, cudaStream_t s);
int launch_conv_in_tc_ex(const float *x, const float *wp, const float *bias, void *y, int B, int H, int W, int Cout,
                         int relu, int out_bf16, cudaStream_t s);

bool conv_in_bf16_persistent_ok(int H, int W, const void *x);
int launch_conv_in_bf16_persistent(const float *x, const float *wp, const float *bias, void *y, int B, int H, int W, int relu,
                                   cudaStream_t s);
bool vq2_supported(long long N, int K, int D);
int launch_vq2(const float *z, const float *E, long long N, int K, int D, long long *idx, void *zq, double *sse, int *hist,
               void *ws, int defer, int zq_bf16, cudaStream_t s);
int launch_conv_in_k4s2(const float *x, const float *wp, const float *bias, float *y, int B, int Cin, int H, int W,
                        int Cout, int relu, cudaStream_t s);
int launch_convt_out_k4s2(const float *x, const float *wp, const float *bias, float *y, int B, int Cin, int H, int W,
                          int Cout, int relu, cudaStream_t s);
bool res_tc_supported(int C, int Cmid, const void *r, const void *out);
int launch_res_tc(const float *r, const float *w1_tc, const float *w2_tc, float *out, int B, int H, int W, int C,
                  int Cmid, int relu_out, int napp, cudaStream_t s);
bool conv_in_tc_supported(int Cin, int Cout, int H, int W, const void *y);
int launch_conv_in_tc(const float *x, const float *wp, const float *bias, float *y, int B, int H, int W, int Cout,
                      int relu, cudaStream_t s);
bool convt_shuffle_supported(int Cin, int Cout, const void *in, const void *out);
int launch_convt_shuffle(const float *in, const float *w_shuffle, const float *bias, float *out, int B, int Cin, int H,
                         int W, int Cout, int relu, cudaStream_t s);
bool conv_halo_supported(const ConvLaunch &p);
int launch_conv_halo(const ConvLaunch &p, const float *w_tc, cudaStream_t s);
bool conv_tc_supported(const ConvLaunch &p);
int launch_conv_tc(const ConvLaunch *ph, int nph, const float *w_tc, int total_taps, cudaStream_t s);

unsigned long long g_vqb_launches = 0;
static int g_vq_kernel = 0;   // 0 auto, 1 exact FFMA kernel, 2 tcgen05 kernel (vq2.cu)
extern "C" int vqb_set_vq_kernel(int which) {
    if (which < 0 || which > 2) return VQB_ERR_BAD_ARG;
    g_vq_kernel = which;
    return 0;
}
extern "C" unsigned long long vqb_launch_count(void) { return g_vqb_launches; }

extern "C" int vqb_abi_version(void) { return VQB_ABI_VERSION; }

// 0 = release library; 1 = diagnostic build (adds in-kernel timelines, same results)
extern "C" int vqb_diag_build(void) { return VQB_DIAG; }

extern "C" const char *vqb_error_string(int code) {
    switch (code) {
        case VQB_OK: return "success";
        case VQB_ERR_BAD_ARG: return "bad argument (null pointer, non-positive size or bad enum)";
        case VQB_ERR_UNSUPPORTED: return "shape not supported by the sm_100a kernels";
        case VQB_ERR_WORKSPACE: return "workspace too small";
        case VQB_ERR_NO_DEVICE: return "no CUDA device";
        case VQB_ERR_ALIGNMENT: return "pointer not 16-byte aligned";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown vqb error";
    }
}

extern "C" int vqb_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return VQB_ERR_NO_DEVICE;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) return VQB_ERR_NO_DEVICE;
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return 0;
}

static void set_strides(int layout, int C, int H, int W, long long &sn, long long &sh, long long &sw,
                        long long &sc) {
    if (layout == VQB_NCHW) {
        sn = (long long)C * H * W; sc = (long long)H * W; sh = W; sw = 1;
    } else {
        sn = (long long)H * W * C; sh = (long long)W * C; sw = C; sc = 1;
    }
}

extern "C" int vqb_conv2d_f32(const float *in, const float *w_packed, const float *bias, const float *skip,
                              float *out, int B, int Cin, int H, int W, int Cout, int kh, int kw, int stride,
                              int pad, int transposed, int in_layout, int out_layout, int relu, int precision,
                              void *stream) {
    if (!in || !w_packed || !out) return VQB_ERR_BAD_ARG;
    if (B <= 0 || Cin <= 0 || H <= 0 || W <= 0 || Cout <= 0 || kh <= 0 || kw <= 0 || stride <= 0 || pad < 0)
        return VQB_ERR_BAD_ARG;
    if ((in_layout != VQB_NCHW && in_layout != VQB_NHWC) || (out_layout != VQB_NCHW && out_layout != VQB_NHWC))
        return VQB_ERR_BAD_ARG;
    if (precision < VQB_FP32 || precision > VQB_BF16) return VQB_ERR_BAD_ARG;
    if (precision == VQB_BF16) return VQB_ERR_UNSUPPORTED;      // bf16 operands need bf16 activations: vqb_conv2d_bf16
    if (skip && out_layout != VQB_NHWC) return VQB_ERR_BAD_ARG;
    if (kh * kw > VQB_MAX_TAPS) return VQB_ERR_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;

    const int OH = transposed ? (H - 1) * stride - 2 * pad + kh : (H + 2 * pad - kh) / stride + 1;
    const int OW = transposed ? (W - 1) * stride - 2 * pad + kw : (W + 2 * pad - kw) / stride + 1;
    if (OH <= 0 || OW <= 0) return VQB_ERR_BAD_ARG;

    // the two HBM-bound end layers have dedicated kernels (conv_edge.cu)
    if (kh == 4 && kw == 4 && stride == 2 && pad == 1 && !skip) {
        if (!transposed && precision != VQB_FP32 && in_layout == VQB_NCHW && out_layout == VQB_NHWC &&
            conv_in_tc_supported(Cin, Cout, H, W, out)) {     // tcgen05 with a hand-built im2col tile
            const int rc = launch_conv_in_tc(in, w_packed, bias, out, B, H, W, Cout, relu, s);
            if (rc != VQB_ERR_UNSUPPORTED) return rc;
        }
        if (!transposed && Cin == 3 && Cout % 32 == 0 && in_layout == VQB_NCHW && out_layout == VQB_NHWC &&
            H % 2 == 0 && W % 2 == 0 && (size_t)16 * Cin * Cout * 4 <= 48 * 1024)
            return launch_conv_in_k4s2(in, w_packed, bias, out, B, Cin, H, W, Cout, relu, s);
        if (transposed && precision != VQB_FP32 && in_layout == VQB_NHWC && out_layout == VQB_NCHW &&
            convt_shuffle_supported(Cin, Cout, in, out)) {    // tcgen05: one 3x3-neighbourhood GEMM + pixel shuffle
            const int rc = launch_convt_shuffle(in, w_packed + (size_t)2 * 16 * Cin * Cout, bias, out, B, Cin, H, W, Cout, relu, s);
            if (rc != VQB_ERR_UNSUPPORTED) return rc;
        }
        if (transposed && Cout == 3 && Cin % 4 == 0 && Cin <= 128 && ((Cin / 4) & (Cin / 4 - 1)) == 0 &&
            in_layout == VQB_NHWC && out_layout == VQB_NCHW)
            return launch_convt_out_k4s2(in, w_packed, bias, out, B, Cin, H, W, Cout, relu, s);
    }

    ConvLaunch p;
    p.in = in; p.w = w_packed; p.bias = bias; p.skip = skip; p.out = out;
    p.B = B; p.Cin = Cin; p.H = H; p.W = W; p.Cout = Cout; p.relu = relu;
    set_strides(in_layout, Cin, H, W, p.in_sn, p.in_sh, p.in_sw, p.in_sc);
    set_strides(out_layout, Cout, OH, OW, p.out_sn, p.out_sh, p.out_sw, p.out_sc);
    const bool small = (Cout <= 4);
    const float *w_tc = w_packed + (size_t)kh * kw * Cin * Cout;   // K-major copy for the tcgen05 path
    const bool want_tc = precision != VQB_FP32;

    if (!transposed || stride == 1) {
        p.OHg = OH; p.OWg = OW;
        p.in_step = transposed ? 1 : stride;
        p.out_step = 1; p.out_py = 0; p.out_px = 0;
        p.ntaps = kh * kw;
        for (int r = 0; r < kh; ++r)
            for (int c = 0; c < kw; ++c) {
                const int t = r * kw + c;
                p.tap_w[t] = t;
                p.tap_dy[t] = transposed ? pad - r : r - pad;
                p.tap_dx[t] = transposed ? pad - c : c - pad;
            }
        // a tensor-core launcher that cannot fit the shape (shared memory, ring depth) answers VQB_ERR_UNSUPPORTED
        // before launching anything: fall through to the next kernel that can run it
        if (want_tc && conv_halo_supported(p)) {
            const int rc = launch_conv_halo(p, w_tc, s);
            if (rc != VQB_ERR_UNSUPPORTED) return rc;
        }
        if (want_tc && conv_tc_supported(p)) {
            const int rc = launch_conv_tc(&p, 1, w_tc, kh * kw, s);
            if (rc != VQB_ERR_UNSUPPORTED) return rc;
        }
        return small ? launch_conv_small_cout(p, s) : launch_conv_ffma(p, s);
    }
    // stride-s transposed conv: s*s sub-pixel phases, each a stride-1 gather conv
    // over the taps whose parity matches (decoder.py:31-35).
    p.in_step = 1; p.out_step = stride;
    ConvLaunch phases[4];
    int nph = 0;
    const bool tc_multi = want_tc && stride == 2 && conv_tc_supported(p);
    for (int py = 0; py < stride; ++py)
        for (int px = 0; px < stride; ++px) {
            p.out_py = py; p.out_px = px;
            p.OHg = (OH - py + stride - 1) / stride;
            p.OWg = (OW - px + stride - 1) / stride;
            if (p.OHg <= 0 || p.OWg <= 0) continue;
            int nt = 0;
            for (int r = 0; r < kh; ++r) {
                if ((py + pad - r) % stride != 0) continue;
                for (int c = 0; c < kw; ++c) {
                    if ((px + pad - c) % stride != 0) continue;
                    p.tap_w[nt] = r * kw + c;
                    p.tap_dy[nt] = (py + pad - r) / stride;
                    p.tap_dx[nt] = (px + pad - c) / stride;
                    ++nt;
                }
            }
            p.ntaps = nt;
            int rc;
            if (nt == 0) {
                // a phase no tap reaches still gets bias/skip/activation
                p.ntaps = 0;
            }
            if (tc_multi) { phases[nph++] = p; continue; }
            rc = small ? launch_conv_small_cout(p, s) : launch_conv_ffma(p, s);
            if (rc != 0) return rc;
        }
    if (tc_multi && nph > 0) {
        const int rc = launch_conv_tc(phases, nph, w_tc, kh * kw, s);   // one launch, blockIdx.y = phase
        if (rc != VQB_ERR_UNSUPPORTED) return rc;
        for (int i = 0; i < nph; ++i) {                                 // did not fit: the phases one by one on CUDA cores
            const int rc2 = small ? launch_conv_small_cout(phases[i], s) : launch_conv_ffma(phases[i], s);
            if (rc2 != 0) return rc2;
        }
    }
    return 0;
}

extern "C" size_t vqb_vq_workspace_bytes(int64_t N, int K, int D) {
    (void)N; (void)D;
    if (K <= 0) return 0;
    return vq_ws_marker_offset(K) + 256;
}

// [exact / vq2 kernel workspace (whichever is larger)][256 B: deferred-reduction marker]
size_t vq_ws_marker_offset(int K) {
    const size_t a = vq_exact_workspace_bytes(K), b = vq2_workspace_bytes(K);
    return ((a > b ? a : b) + 255) / 256 * 256;
}

static int vq_forward_impl(const float *z, const float *codebook, int64_t N, int K, int D, int64_t *idx, float *zq,
                           double *sse, int32_t *hist, void *workspace, size_t workspace_bytes, int defer,
                           void *stream);

extern "C" int vqb_vq_forward_deferred_f32(const float *z, const float *codebook, int64_t N, int K, int D, int64_t *idx,
                                           float *zq, double *sse, int32_t *hist, void *workspace,
                                           size_t workspace_bytes, void *stream) {
    return vq_forward_impl(z, codebook, N, K, D, idx, zq, sse, hist, workspace, workspace_bytes, 1, stream);
}

extern "C" int vqb_vq_reduce_sse_f32(const void *workspace, int64_t N, int K, int D, double *sse, void *stream) {
    if (!workspace || !sse || N <= 0 || K <= 0 || D <= 0) return VQB_ERR_BAD_ARG;
    return launch_vq_reduce_sse(workspace, K, sse, (cudaStream_t)stream);
}

extern "C" int vqb_vq_forward_f32(const float *z, const float *codebook, int64_t N, int K, int D, int64_t *idx,
                                  float *zq, double *sse, int32_t *hist, void *workspace,
                                  size_t workspace_bytes, void *stream) {
    return vq_forward_impl(z, codebook, N, K, D, idx, zq, sse, hist, workspace, workspace_bytes, 0, stream);
}

static int vq_forward_impl(const float *z, const float *codebook, int64_t N, int K, int D, int64_t *idx, float *zq,
                           double *sse, int32_t *hist, void *workspace, size_t workspace_bytes, int defer,
                           void *stream) {
    if (!z || !codebook || !idx || !zq || !sse || !hist || !workspace) return VQB_ERR_BAD_ARG;
    if (N <= 0 || K <= 0 || D <= 0) return VQB_ERR_BAD_ARG;
    if (D % 4 != 0) return VQB_ERR_UNSUPPORTED;
    if (workspace_bytes < vqb_vq_workspace_bytes(N, K, D)) return VQB_ERR_WORKSPACE;
    const uintptr_t al = reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(codebook) |
                         reinterpret_cast<uintptr_t>(zq) | reinterpret_cast<uintptr_t>(workspace);
    if (al & 15) return VQB_ERR_ALIGNMENT;
    const bool v2_ok = vq2_supported(N, K, D);
    if (g_vq_kernel == 2 && !v2_ok) return VQB_ERR_UNSUPPORTED;
    if (v2_ok && g_vq_kernel != 1)
        return launch_vq2(z, codebook, N, K, D, reinterpret_cast<long long *>(idx), zq, sse, hist, workspace, defer, 0,
                          (cudaStream_t)stream);
    const int rc = launch_vq_exact(z, codebook, N, K, D, reinterpret_cast<long long *>(idx), zq, sse, hist, workspace,
                                   (cudaStream_t)stream);
    if (rc || !defer) return rc;
    // sse is final: nothing pending for vqb_vq_reduce_sse_f32
    return vqb_cuda_status(cudaMemsetAsync(reinterpret_cast<unsigned char *>(workspace) + vq_ws_marker_offset(K), 0, 4,
                                           (cudaStream_t)stream));
}

// VQB_BF16 pipeline: same contract as vqb_vq_forward_deferred_f32 (fp32 z in, bit-exact idx) but z_q leaves as bf16
// rows for the decoder's first conv; vq2 kernel only (D == 64, K <= 8192).
extern "C" int vqb_vq_forward_bf16zq_f32(const float *z, const float *codebook, int64_t N, int K, int D, int64_t *idx,
                                         void *zq_bf16, double *sse, int32_t *hist, void *workspace,
                                         size_t workspace_bytes, void *stream) {
    if (!z || !codebook || !idx || !zq_bf16 || !sse || !hist || !workspace) return VQB_ERR_BAD_ARG;
    if (N <= 0 || K <= 0 || D <= 0) return VQB_ERR_BAD_ARG;
    if (workspace_bytes < vqb_vq_workspace_bytes(N, K, D)) return VQB_ERR_WORKSPACE;
    const uintptr_t al = reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(codebook) |
                         reinterpret_cast<uintptr_t>(zq_bf16) | reinterpret_cast<uintptr_t>(workspace);
    if (al & 15) return VQB_ERR_ALIGNMENT;
    if (!vq2_supported(N, K, D)) return VQB_ERR_UNSUPPORTED;
    return launch_vq2(z, codebook, N, K, D, reinterpret_cast<long long *>(idx), zq_bf16, sse, hist, workspace, 1, 1,
                      (cudaStream_t)stream);
}

// encoder.py:29-31 in the VQB_BF16 pipeline: fp32 NCHW image in, bf16 NHWC activation out (Cout == 64); the 48-tap
// contraction itself runs as kind::tf32 on the fp32 pixels.  w_packed: vqb_pack_conv_weight_f32 of the layer.
extern "C" int vqb_conv_in_bf16(const float *x, const float *w_packed, const float *bias, void *out, int B, int H, int W,
                                int Cout, int relu, void *stream) {
    if (!x || !w_packed || !out) return VQB_ERR_BAD_ARG;
    if (B <= 0 || H <= 0 || W <= 0 || Cout <= 0) return VQB_ERR_BAD_ARG;
    if (!conv_in_tc_supported(3, Cout, H, W, out) || Cout != 64) return VQB_ERR_UNSUPPORTED;
    if (conv_in_bf16_persistent_ok(H, W, x)) {          // one CTA per SM, pipelined over tiles (conv_in_bf16.cu)
        const int rc = launch_conv_in_bf16_persistent(x, w_packed, bias, out, B, H, W, relu, (cudaStream_t)stream);
        if (rc != VQB_ERR_UNSUPPORTED) return rc;
    }
    return launch_conv_in_tc_ex(x, w_packed, bias, out, B, H, W, Cout, relu, 1, (cudaStream_t)stream);
}

extern "C" int vqb_residual_layer_f32(const float *r, const float *w1_packed, const float *w2_packed, float *out,
                                      float *tmp, int B, int H, int W, int C, int Cmid, int relu_out, int precision,
                                      void *stream) {
    if (!r || !w1_packed || !w2_packed || !out || !tmp) return VQB_ERR_BAD_ARG;
    if (B <= 0 || H <= 0 || W <= 0 || C <= 0 || Cmid <= 0) return VQB_ERR_BAD_ARG;
    if (precision < VQB_FP32 || precision > VQB_BF16) return VQB_ERR_BAD_ARG;
    if (precision == VQB_BF16) return VQB_ERR_UNSUPPORTED;      // see vqb_residual_layer_bf16
    if (precision != VQB_FP32 && res_tc_supported(C, Cmid, r, out)) {
        const int rc = launch_res_tc(r, w1_packed + (size_t)9 * C * Cmid, w2_packed + (size_t)C * Cmid, out, B, H, W, C, Cmid,
                                     relu_out, 1, (cudaStream_t)stream);
        if (rc != VQB_ERR_UNSUPPORTED) return rc;               // (e.g. C = 256, Cmid = 128: shared memory) -> generic path
    }
    // two launches through the generic path (residual.py:20-24 then :23-24,:28)
    int rc = vqb_conv2d_f32(r, w1_packed, nullptr, nullptr, tmp, B, C, H, W, Cmid, 3, 3, 1, 1, 0, VQB_NHWC, VQB_NHWC, 1,
                            precision, stream);
    if (rc) return rc;
    return vqb_conv2d_f32(tmp, w2_packed, nullptr, r, out, B, Cmid, H, W, C, 1, 1, 1, 0, 0, VQB_NHWC, VQB_NHWC,
                          relu_out, precision, stream);
}

extern "C" int vqb_residual_stack_f32(const float *r, const float *w1_packed, const float *w2_packed, float *out,
                                      float *scratch, float *tmp, int B, int H, int W, int C, int Cmid, int n_layers,
                                      int precision, void *stream) {
    if (!r || !w1_packed || !w2_packed || !out || !tmp) return VQB_ERR_BAD_ARG;
    if (B <= 0 || H <= 0 || W <= 0 || C <= 0 || Cmid <= 0 || n_layers < 1) return VQB_ERR_BAD_ARG;
    if (n_layers > 1 && !scratch) return VQB_ERR_BAD_ARG;
    if (precision < VQB_FP32 || precision > VQB_BF16) return VQB_ERR_BAD_ARG;
    if (precision == VQB_BF16) return VQB_ERR_UNSUPPORTED;
    if (n_layers > 1 && precision != VQB_FP32 && res_tc_supported(C, Cmid, r, out)) {
        // all applications in ONE launch: the activation never leaves shared memory between them
        const int rc = launch_res_tc(r, w1_packed + (size_t)9 * C * Cmid, w2_packed + (size_t)C * Cmid, out, B, H, W, C,
                                     Cmid, 1, n_layers, (cudaStream_t)stream);
        if (rc != VQB_ERR_UNSUPPORTED) return rc;
    }
    // one launch per application, ping-ponging so that the last one lands in `out`
    const float *src = r;
    for (int i = 0; i < n_layers; ++i) {
        float *dst = ((n_layers - 1 - i) % 2 == 0) ? out : scratch;
        const int rc = vqb_residual_layer_f32(src, w1_packed, w2_packed, dst, tmp, B, H, W, C, Cmid, 1, precision, stream);
        if (rc) return rc;
        src = dst;
    }
    return 0;
}

// Thin stream-ordered copy for the host-buffer front end (vqvae_b200/pipeline.py): one ctypes call instead of
// a torch stream context + Tensor.copy_ per transfer (the Python overhead per step was larger than the kernels).
extern "C" int vqb_memcpy_async(void *dst, const void *src, size_t bytes, int kind, void *stream) {
    if (!dst || !src) return VQB_ERR_BAD_ARG;
    if (bytes == 0) return 0;
    if (kind < 1 || kind > 3) return VQB_ERR_BAD_ARG;
    // Driver entry point (unified addressing: the driver knows which side is pinned host memory).  The copy must
    // not go through THIS library's statically linked runtime: host buffers pinned by another runtime instance
    // (torch's) were copied at pageable speed, synchronously, through cudaMemcpyAsync (measured: 8 GB/s).
    typedef int (*PFN_cuMemcpyAsync)(unsigned long long, unsigned long long, size_t, void *);
    static PFN_cuMemcpyAsync fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemcpyAsync", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<PFN_cuMemcpyAsync>(p);
    }();
    if (fn) {
        const int rc = fn((unsigned long long)(uintptr_t)dst, (unsigned long long)(uintptr_t)src, bytes, stream);
        return rc == 0 ? 0 : VQB_ERR_BAD_ARG;
    }
    const cudaMemcpyKind k = kind == 1 ? cudaMemcpyHostToDevice : kind == 2 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    return vqb_cuda_status(cudaMemcpyAsync(dst, src, bytes, k, (cudaStream_t)stream));
}
