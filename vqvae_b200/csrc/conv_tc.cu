// conv_tc.cu -- tcgen05 implicit-GEMM convolution for sm_100a (VQB_TF32 arithmetic).
//
// Replaces the nn.Conv2d / nn.ConvTranspose2d call sites of the hot path whose channel
// counts fill a tensor-core tile: encoder.py:32-36 (64->128 k4s2, 128->128 k3),
// residual.py:20-24 (128->32 k3, 32->128 k1 + skip), vqvae.py:16-17 (128->64 k1),
// decoder.py:28-33 (ConvT 64->128 k3s1, ConvT 128->64 k4s2 as four sub-pixel phases).
//
// GEMM view (one CTA = one 128-pixel output tile, all Cout columns):
//   D[128 px][Cout] = sum over (tap t, 32-channel chunk c) A_t,c[128 px][32] * W_t,c[Cout][32]^T
//   * A_t,c is fetched by ONE 4-D TMA box {32 ch, BW, BH, BN} of the NHWC input, shifted
//     by the tap offset (dy,dx): the box lands in shared memory as 128 rows of 128 bytes
//     in the 128-byte-swizzled K-major layout UMMA reads; out-of-image pixels are
//     zero-filled by TMA (= the convolution's zero padding) and stride-2 convolutions use
//     the tensor map's element strides.  Nothing like an im2col matrix ever exists.
//   * W_t,c is a 2-D TMA box {32 ch, Cout} of the tap-major packed weight [t][Cout][Cin].
//   * warp 0 = TMA producer, warp 1 = tcgen05.mma kind::tf32 issuer (fp32 accumulators
//     in TMEM), warp 2 = TMEM allocator, warps 4-7 = epilogue: tcgen05.ld -> +bias
//     -> +skip -> ReLU -> coalesced 16-byte NHWC stores.  Up to 8-stage mbarrier ring
//     (the k-loop of one tile is TMA-latency bound, so the ring is as deep as smem allows).
//   * the sub-pixel phases of a stride-2 transposed conv run in ONE launch (blockIdx.y).
#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int CT_THREADS = 256;
constexpr int CT_MAX_STAGES = 8;
constexpr int CT_GROUP = 2;            // ring stages released per tcgen05.commit (a commit costs ~230 cycles)
constexpr int A_BYTES = 128 * 128;                 // 128 pixels x 32 fp32

struct ConvTcParams {
    const float *bias, *skip;
    float *out;
    int B, Cin, Cout;
    int BW, BH, BN;                                // tile = BN images x BH rows x BW cols = 128 pixels
    int tiles_x, tiles_y;                          // of the largest phase grid
    int in_step, out_step;
    int stages;
    int nmma;                                      // MMA issuer warps (1 or 2), see res_tc.cu
    // blockIdx.y = phase (1 for a plain conv, stride^2 sub-pixel phases of a transposed conv)
    int OHg[4], OWg[4], out_py[4], out_px[4], ntaps[4];
    int tap_w[4][VQB_MAX_TAPS], tap_dy[4][VQB_MAX_TAPS], tap_dx[4][VQB_MAX_TAPS];
    long long out_sn, out_sh, out_sw;              // NHWC element strides of out / skip
    int relu;
};

__global__ void __launch_bounds__(CT_THREADS, 2)
conv_tc_kernel(const __grid_constant__ CUtensorMap tma_in, const __grid_constant__ CUtensorMap tma_w,
               const ConvTcParams p) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = ptx::smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (sbase - raw);
    const int b_bytes = p.Cout * 128;
    const int stage_bytes = A_BYTES + b_bytes;
    const int CT_STAGES = p.stages;
    const int ph = blockIdx.y;
    const uint32_t bars = sbase + CT_STAGES * stage_bytes;      // full[S], empty[S], tfull
    float *bias_s = reinterpret_cast<float *>(sm + CT_STAGES * stage_bytes + 192);
    volatile uint32_t *tmem_holder = reinterpret_cast<volatile uint32_t *>(sm + CT_STAGES * stage_bytes + 176);
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (CT_MAX_STAGES + s); };
    const uint32_t tfull = bars + 8u * (2 * CT_MAX_STAGES);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int tcols = 32;
    while (tcols < p.nmma * p.Cout + ((p.Cout & 31) ? 16 : 0)) tcols <<= 1;

    // tile origin
    int tile = blockIdx.x;
    const int tx = tile % p.tiles_x; tile /= p.tiles_x;
    const int ty = tile % p.tiles_y; tile /= p.tiles_y;
    const int gx0 = tx * p.BW, gy0 = ty * p.BH, n0 = tile * p.BN;

    if (tid < CT_STAGES) { ptx::mbar_init(full(tid), 1); ptx::mbar_init(empty(tid), (uint32_t)p.nmma); }      // init spread over threads
    if (tid == 32) ptx::mbar_init(tfull, (uint32_t)p.nmma);
    if (tid == 64) { ptx::prefetch_tmap(&tma_in); ptx::prefetch_tmap(&tma_w); }
    ptx::fence_mbar_init();
    for (int c = tid; c < p.Cout; c += CT_THREADS) bias_s[c] = p.bias ? __ldg(p.bias + c) : 0.f;
    if (warp == 2) ptx::tmem_alloc(sbase + CT_STAGES * stage_bytes + 176, (uint32_t)tcols);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    pdl_launch_dependents();       // the next layer may start its prologue
    pdl_wait();                    // ... and this one waits here for the previous layer's output

    const int kchunks = p.Cin / 32;
    const int ksteps = p.ntaps[ph] * kchunks;

    // Issuer warps run fully converged; only the elected leader lane issues TMA / MMA / commits and every
    // per-k-step quantity is a running pointer (profiles/r01_res_tc_timeline.txt).
    if (warp == 0) {
        const bool leader = ptx::elect_one();
        uint32_t st = 0, par = 0, full_bar = bars, empty_bar = bars + 8u * CT_MAX_STAGES, dst = sbase;
        const int ix0 = gx0 * p.in_step, iy0 = gy0 * p.in_step;
        for (int t = 0; t < p.ntaps[ph]; ++t) {
            const int cx = ix0 + p.tap_dx[ph][t], cy = iy0 + p.tap_dy[ph][t], wrow = p.tap_w[ph][t] * p.Cout;
            for (int cc = 0; cc < kchunks; ++cc) {
                if ((st & (CT_GROUP - 1)) == 0) ptx::mbar_wait(empty_bar, par ^ 1);
                if (leader) {
                    ptx::mbar_expect_tx(full_bar, (uint32_t)stage_bytes);
                    ptx::tma_load_4d(dst, &tma_in, full_bar, cc * 32, cx, cy, n0);
                    ptx::tma_load_2d(dst + A_BYTES, &tma_w, full_bar, cc * 32, wrow);
                }
                ++st; full_bar += 8; dst += (uint32_t)stage_bytes;
                if ((st & (CT_GROUP - 1)) == 0) empty_bar += 8;
                if (st == (uint32_t)CT_STAGES) { st = 0; par ^= 1; full_bar = bars; empty_bar = bars + 8u * CT_MAX_STAGES; dst = sbase; }
            }
        }
    } else if (warp == 1 || (warp == 3 && p.nmma == 2)) {
        // issuer mi takes k-steps mi, mi + nmma, ... into its own accumulator (columns mi * Cout ..)
        const int mi = warp >> 1, nm = p.nmma;
        const bool leader = ptx::elect_one();
        const uint32_t idesc = ptx::instr_desc(ptx::FMT_TF32, 128, (uint32_t)p.Cout);
        const uint32_t d_hi = ptx::desc_hi_sw128(1024);
        const uint32_t a_lo0 = sbase >> 4, step16 = (uint32_t)stage_bytes >> 4;
        const uint32_t dacc = tmem_base + (uint32_t)(mi * p.Cout);
        uint32_t st = (uint32_t)mi, par = 0, acc = 0;
        for (int i = mi; i < ksteps; i += nm) {
            ptx::mbar_wait(full((int)st), par);
            ptx::tc_fence_after();
            const uint32_t a_lo = a_lo0 + st * step16;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                if (leader) ptx::mma_tf32_w(dacc, a_lo + 2u * kk, d_hi, a_lo + (A_BYTES >> 4) + 2u * kk, d_hi, idesc, acc);
                acc = 1;
            }
            if ((st & (CT_GROUP - 1)) + (uint32_t)nm >= (uint32_t)CT_GROUP) {
                if (leader) ptx::tc_commit(empty((int)(st / CT_GROUP)));
            }
            st += (uint32_t)nm;
            if (st >= (uint32_t)CT_STAGES) { st -= (uint32_t)CT_STAGES; par ^= 1; }
        }
        if (leader) ptx::tc_commit(tfull);
        __syncwarp();
    } else if (warp >= 4) {
        // ---- epilogue: this thread owns output pixel `row` of the tile ----
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const int bw = row % p.BW, bh = (row / p.BW) % p.BH, bn = row / (p.BW * p.BH);
        const int gx = gx0 + bw, gy = gy0 + bh, n = n0 + bn;
        const bool valid = gx < p.OWg[ph] && gy < p.OHg[ph] && n < p.B;
        const long long ob = (long long)n * p.out_sn + (long long)(gy * p.out_step + p.out_py[ph]) * p.out_sh +
                             (long long)(gx * p.out_step + p.out_px[ph]) * p.out_sw;
        if (ksteps > 0) {
            ptx::mbar_wait(tfull, 0);
            ptx::tc_fence_after();
        }
        {
            const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
            const bool two = (p.nmma == 2 && ksteps >= 2), have = (ksteps > 0);
            auto emit = [&](float (&v)[32], int c0) {
                if (!have) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = 0.f;
                }
                if (valid) {
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        if (c0 + i < p.Cout) {             // Cout % 16 == 0: whole float4s
                            const float4 bb = *reinterpret_cast<const float4 *>(bias_s + c0 + i);
                            float4 o = make_float4(v[i] + bb.x, v[i + 1] + bb.y, v[i + 2] + bb.z, v[i + 3] + bb.w);
                            if (p.skip) {
                                const float4 sk = __ldg(reinterpret_cast<const float4 *>(p.skip + ob + c0 + i));
                                o.x += sk.x; o.y += sk.y; o.z += sk.z; o.w += sk.w;
                            }
                            if (p.relu) {
                                o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
                            }
                            *reinterpret_cast<float4 *>(p.out + ob + c0 + i) = o;
                        }
                    }
                }
            };
            // the TMEM loads of the next 32 columns travel while the current ones are stored (a tcgen05.ld round
            // trip is ~0.2 us); three register arrays: the partial `u` is folded into its `v` before the next load
            float va[32], vb[32], u[32];
            auto load = [&](float (&v)[32], int c0) {
                if (have) {
                    ptx::tmem_ld32(trow + (uint32_t)c0, v);
                    if (two) ptx::tmem_ld32(trow + (uint32_t)(p.Cout + c0), u);
                }
            };
            auto wait = [&](float (&v)[32]) {
                if (have) {
                    ptx::tmem_ld_wait32(v);
                    if (two) {
                        ptx::tmem_ld_wait32(u);
#pragma unroll
                        for (int i = 0; i < 32; ++i) v[i] = __fadd_rn(v[i], u[i]);      // + the second issuer's partial
                    }
                }
            };
            load(va, 0);
            for (int c0 = 0; c0 < p.Cout; c0 += 64) {
                wait(va);
                if (c0 + 32 < p.Cout) load(vb, c0 + 32);
                emit(va, c0);
                if (c0 + 32 < p.Cout) {
                    wait(vb);
                    if (c0 + 64 < p.Cout) load(va, c0 + 64);
                    emit(vb, c0 + 32);
                }
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, (uint32_t)tcols);
}

int pow2_ceil(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

}  // namespace

bool conv_tc_supported(const ConvLaunch &p) {
    const bool in_nhwc = p.in_sc == 1 && p.in_sw == p.Cin;
    const bool out_nhwc = p.out_sc == 1 && p.out_sw == p.Cout;
    return in_nhwc && out_nhwc && p.Cin % 32 == 0 && p.Cout % 16 == 0 && p.Cout >= 16 && p.Cout <= 256 &&
           p.in_step >= 1 && p.in_step <= 2 &&
           (reinterpret_cast<uintptr_t>(p.in) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 &&
           (p.skip == nullptr || (reinterpret_cast<uintptr_t>(p.skip) & 15) == 0);
}

// ph[0..nph): the phases of ONE layer (same tensors, strides and steps; they differ in the
// output grid, the sub-pixel offset and the tap list).  w_tc: tap-major K-major weight
// [tap][Cout][Cin] (vqb_pack_conv_weight_f32, second half).
int launch_conv_tc(const ConvLaunch *ph, int nph, const float *w_tc, int total_taps, cudaStream_t s) {
    if (nph < 1 || nph > 4) return VQB_ERR_UNSUPPORTED;
    const ConvLaunch &p = ph[0];
    ConvTcParams q;
    q.bias = p.bias; q.skip = p.skip; q.out = p.out;
    q.B = p.B; q.Cin = p.Cin; q.Cout = p.Cout;
    int maxw = 0, maxh = 0;
    for (int i = 0; i < 4; ++i) {
        const ConvLaunch &r = ph[i < nph ? i : 0];
        q.OHg[i] = i < nph ? r.OHg : 0; q.OWg[i] = i < nph ? r.OWg : 0;
        q.out_py[i] = r.out_py; q.out_px[i] = r.out_px; q.ntaps[i] = i < nph ? r.ntaps : 0;
        for (int t = 0; t < VQB_MAX_TAPS; ++t) {
            q.tap_w[i][t] = t < r.ntaps ? r.tap_w[t] : 0;
            q.tap_dy[i][t] = t < r.ntaps ? r.tap_dy[t] : 0;
            q.tap_dx[i][t] = t < r.ntaps ? r.tap_dx[t] : 0;
        }
        if (q.OWg[i] > maxw) maxw = q.OWg[i];
        if (q.OHg[i] > maxh) maxh = q.OHg[i];
    }
    if (maxw <= 0 || maxh <= 0) return 0;
    q.BW = pow2_ceil(maxw) < 16 ? pow2_ceil(maxw) : 16;
    q.BH = pow2_ceil(maxh) < 128 / q.BW ? pow2_ceil(maxh) : 128 / q.BW;
    q.BN = 128 / (q.BW * q.BH);
    q.tiles_x = (maxw + q.BW - 1) / q.BW;
    q.tiles_y = (maxh + q.BH - 1) / q.BH;
    const int tiles_n = (p.B + q.BN - 1) / q.BN;
    q.in_step = p.in_step; q.out_step = p.out_step;
    q.out_sn = p.out_sn; q.out_sh = p.out_sh; q.out_sw = p.out_sw; q.relu = p.relu;

    CUtensorMap tin, tw;
    const uint64_t dims[4] = {(uint64_t)p.Cin, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.B};
    const uint64_t strides[3] = {(uint64_t)p.Cin * 4, (uint64_t)p.W * p.Cin * 4, (uint64_t)p.H * p.W * p.Cin * 4};
    const uint32_t box[4] = {32u, (uint32_t)(q.BW * p.in_step), (uint32_t)(q.BH * p.in_step), (uint32_t)q.BN};
    const uint32_t es[4] = {1u, (uint32_t)p.in_step, (uint32_t)p.in_step, 1u};
    int rc = vqb_encode_tmap_4d(&tin, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, p.in, dims, strides, box, es,
                                CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = vqb_encode_tmap_2d(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w_tc, (uint64_t)p.Cin,
                            (uint64_t)total_taps * p.Cout, (uint64_t)p.Cin * 4, 32, (uint32_t)p.Cout,
                            CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    const int stage_bytes = A_BYTES + p.Cout * 128;
    int maxk = 1;
    for (int i = 0; i < nph; ++i) if (q.ntaps[i] * (p.Cin / 32) > maxk) maxk = q.ntaps[i] * (p.Cin / 32);
    int stages = (200 * 1024) / stage_bytes;
    {
        // more CTAs than one wave of 1-CTA/SM residency (e.g. the 4 phases of a stride-2 transposed conv):
        // keep the ring small enough for 2 CTAs per SM instead of running 2x the waves
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const long long ctas = (long long)q.tiles_x * q.tiles_y * tiles_n * nph;
        if (ctas > sms && stages > (108 * 1024) / stage_bytes) stages = (108 * 1024) / stage_bytes;
    }
    if (stages > CT_MAX_STAGES) stages = CT_MAX_STAGES;
    if (stages > maxk) stages = maxk;
    else stages -= stages % CT_GROUP;             // a reused ring must hold whole commit groups
    if (stages < 1) stages = 1;
    q.stages = stages;
    q.nmma = (2 * p.Cout <= 256 && stages >= 2 && (stages % 2 == 0 || stages >= maxk)) ? 2 : 1;
    const int smem = stages * stage_bytes + 192 + p.Cout * 4 + 1024;
    static int attr_max = 0;
    if (smem > attr_max) {
        cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr_max = smem;
    }
    const long long grid = (long long)q.tiles_x * q.tiles_y * tiles_n;
    if (grid <= 0 || grid > 0x7fffffffLL) return VQB_ERR_UNSUPPORTED;
    if (cudaError_t le = vqb_launch(conv_tc_kernel, dim3((unsigned)grid, (unsigned)nph), dim3(CT_THREADS), (size_t)smem, s, tin, tw, q)) return (int)le;
    VQB_COUNT_LAUNCH(1);
    return vqb_cuda_status(cudaGetLastError());
}
