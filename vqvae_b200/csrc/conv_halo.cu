// conv_halo.cu -- tcgen05 implicit GEMM for 3x3 / stride-1 / pad-1 layers with A-operand reuse.
//
// conv_tc.cu fetches the 128-pixel A tile once per tap (9x for a 3x3), which makes the k-loop
// L2->SM feed bound (profiles/r01: tensor pipe 7-30 % active).  Here the input tile is loaded
// ONCE per 32-channel chunk, with its 1-pixel halo, as a TMA box {32 ch, WP px, BN img, BH+2 rows}
// (tensor-map dims ordered c,w,n,h so the rows of the BN images interleave), and the nine taps are
// nine UMMA shared-memory descriptors into that one tile: tap (dy,dx) starts (dy+1)*BN*WP+(dx+1)
// 128-byte rows further in and 8-pixel row groups stay WP rows apart (the descriptor's base_offset
// stays 0: the hardware uses absolute address bits).  Only the weight tiles stream through the ring.
// Used for encoder.py:35-36, decoder.py:28-29 (ConvTranspose k3s1 = same neighbourhood, tap
// offsets pad - r) and the 3x3 of residual.py:20.
#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int CH_THREADS = 256;
constexpr int CH_MAX_STAGES = 32;     // weight-tile ring: as deep as shared memory allows (the k-loop is
                                      // bound by bytes in flight, not by bandwidth)
constexpr int CH_GROUP = 4;           // ring stages released per tcgen05.commit (a commit costs ~230 cycles)
constexpr int CH_HALO_BUFS = 2;       // halo tiles are double buffered: chunk c+2 loads while c+1 computes
constexpr int CH_MAX_CHUNKS = 8;       // Cin <= 256
// Halo tile width (p.WP = VQB_HALO_WP): 8 pixels + 1 each side = 10.  Not a multiple of 8 on purpose: the swizzle phase
// of a row comes from its absolute address, for TMA and UMMA alike, so an 8-row operand group may start at any row
// (SBO = WP rows); padding to 16 wasted 37 % of the tile.

struct ConvHaloParams {
    const float *bias, *skip;
    float *out;
    int B, H, W, Cin, Cout;
    int BH, BN, tiles_x, tiles_y;
    int stages, relu;
    int nmma;               // MMA issuer warps (1 or 2): k-step i goes to issuer i % nmma, private accumulators summed
                            // by the epilogue in a fixed order (see res_tc.cu)
    int WP;                 // halo tile width in pixels (VQB_HALO_WP)
    int shuffle_cout;       // > 0: the GEMM's 16 columns are (py, px, co) of a k4s2p1 transposed conv with this
                            // many real output channels; the epilogue pixel-shuffles them into the NCHW output
    int tap_w[9], tap_dy[9], tap_dx[9];
};

__global__ void __launch_bounds__(CH_THREADS, 2)
conv_halo_kernel(const __grid_constant__ CUtensorMap tma_in, const __grid_constant__ CUtensorMap tma_w,
                 const ConvHaloParams p) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = ptx::smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (sbase - raw);

    const int chunks = p.Cin / 32;
    const int WP = p.WP;
    const int halo_bytes = (p.BH + 2) * p.BN * WP * 128;        // per 32-channel chunk
    const int halo_stride = (halo_bytes + 1023) & ~1023;        // buffers start on swizzle-pattern boundaries
    const int b_bytes = p.Cout * 128;
    const int S = p.stages;
    const int hbufs = chunks < CH_HALO_BUFS ? chunks : CH_HALO_BUFS;
    const uint32_t ring_off = (uint32_t)(hbufs * halo_stride);
    const uint32_t bar_off = ring_off + (uint32_t)(S * b_bytes);
    const uint32_t bars = sbase + bar_off;
    auto bfull = [&](int s) { return bars + 8u * s; };
    auto bempty = [&](int s) { return bars + 8u * (CH_MAX_STAGES + s); };
    auto hfull = [&](int b) { return bars + 8u * (2 * CH_MAX_STAGES + b); };
    auto hempty = [&](int b) { return bars + 8u * (2 * CH_MAX_STAGES + CH_HALO_BUFS + b); };
    const uint32_t tfull = bars + 8u * (2 * CH_MAX_STAGES + 2 * CH_HALO_BUFS);
    const int misc = 8 * (2 * CH_MAX_STAGES + 2 * CH_HALO_BUFS + 1);
    volatile uint32_t *tmem_holder = reinterpret_cast<volatile uint32_t *>(sm + bar_off + misc);
    float *bias_s = reinterpret_cast<float *>(sm + bar_off + misc + 8);    // 16-byte aligned (misc % 16 == 8)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int tcols = 32;
    // (the epilogue reads 32-column groups: a Cout that is not a multiple of 32 needs 16 columns of slack)
    while (tcols < p.nmma * p.Cout + ((p.Cout & 31) ? 16 : 0)) tcols <<= 1;

    int tile = blockIdx.x;
    const int tx = tile % p.tiles_x; tile /= p.tiles_x;
    const int ty = tile % p.tiles_y; tile /= p.tiles_y;
    const int gx0 = tx * 8, gy0 = ty * p.BH, n0 = tile * p.BN;

    if (tid < S) { ptx::mbar_init(bfull(tid), 1); ptx::mbar_init(bempty(tid), (uint32_t)p.nmma); }     // init spread over threads
    if (tid >= 64 && tid < 64 + CH_HALO_BUFS) { ptx::mbar_init(hfull(tid - 64), 1); ptx::mbar_init(hempty(tid - 64), (uint32_t)p.nmma); }
    if (tid == 96) ptx::mbar_init(tfull, (uint32_t)p.nmma);
    if (tid == 128) { ptx::prefetch_tmap(&tma_in); ptx::prefetch_tmap(&tma_w); }
    ptx::fence_mbar_init();
    for (int c = tid; c < p.Cout; c += CH_THREADS) {
        if (p.shuffle_cout > 0) bias_s[c] = (p.bias && c < 4 * p.shuffle_cout) ? __ldg(p.bias + c % p.shuffle_cout) : 0.f;
        else bias_s[c] = p.bias ? __ldg(p.bias + c) : 0.f;
    }
    if (warp == 2) ptx::tmem_alloc(sbase + bar_off + misc, (uint32_t)tcols);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    pdl_launch_dependents();       // the next layer may start its prologue (it blocks in its own pdl_wait)

    // Issuer warps run fully converged; only the elected leader lane issues TMA / MMA / commits, and
    // every per-k-step quantity is a running pointer (profiles/r01_res_tc_timeline.txt: the issue loops
    // are bound by their own scalar instructions, not by TMA or the tensor pipe).
    if (warp == 0) {
        const bool leader = ptx::elect_one();
        auto load_halo = [&](int c) {
            const int b = c % CH_HALO_BUFS;
            if (c >= CH_HALO_BUFS) ptx::mbar_wait(hempty(b), (uint32_t)(((c / CH_HALO_BUFS) - 1) & 1));
            if (leader) {
                ptx::mbar_expect_tx(hfull(b), (uint32_t)halo_bytes);
                ptx::tma_load_4d(sbase + b * halo_stride, &tma_in, hfull(b), c * 32, gx0 - 1, n0, gy0 - 1);
            }
        };
        // weights do not depend on the previous layer: the first ring-full of weight tiles is requested
        // BEFORE pdl_wait(), i.e. while the previous kernel is still draining
        const int prefill = S < 9 * chunks ? S : 9 * chunks;
        if (leader)
            for (int i = 0; i < prefill; ++i) {
                ptx::mbar_expect_tx(bars + 8u * i, (uint32_t)b_bytes);
                ptx::tma_load_2d(sbase + ring_off + i * b_bytes, &tma_w, bars + 8u * i, (i / 9) * 32, p.tap_w[i % 9] * p.Cout);
            }
        pdl_wait();                                     // the input activation is the previous layer's output
        for (int c = 0; c < hbufs; ++c) load_halo(c);
        uint32_t st = 0, par = 0, full_bar = bars, empty_bar = bars + 8u * CH_MAX_STAGES, dst = sbase + ring_off;
        int kidx = 0;
        for (int c = 0; c < chunks; ++c) {
            // refill the halo buffer chunk c-1 just vacated with chunk c+1 (the ring keeps the MMAs fed)
            if (c >= 1 && c + 1 < chunks && c + 1 >= CH_HALO_BUFS) load_halo(c + 1);
#pragma unroll
            for (int t = 0; t < 9; ++t, ++kidx) {
                if (kidx >= prefill) {
                    if ((st & (CH_GROUP - 1)) == 0) ptx::mbar_wait(empty_bar, par ^ 1);
                    if (leader) {
                        ptx::mbar_expect_tx(full_bar, (uint32_t)b_bytes);
                        ptx::tma_load_2d(dst, &tma_w, full_bar, c * 32, p.tap_w[t] * p.Cout);
                    }
                }
                ++st; full_bar += 8; dst += (uint32_t)b_bytes;
                if ((st & (CH_GROUP - 1)) == 0) empty_bar += 8;
                if (st == (uint32_t)S) { st = 0; par ^= 1; full_bar = bars; empty_bar = bars + 8u * CH_MAX_STAGES; dst = sbase + ring_off; }
            }
        }
    } else if (warp == 1 || (warp == 3 && p.nmma == 2)) {
        // issuer mi takes k-steps mi, mi + nmma, ... (ring position advances by nmma) into its own accumulator
        const int mi = warp >> 1, nm = p.nmma;
        const bool leader = ptx::elect_one();
        const uint32_t idesc = ptx::instr_desc(ptx::FMT_TF32, 128, (uint32_t)p.Cout);
        const uint32_t a_hi = ptx::desc_hi_sw128(WP * 128), b_hi = ptx::desc_hi_sw128(1024);
        const uint32_t rs16 = (uint32_t)(p.BN * WP * 128) >> 4;        // one padded halo row in 16-byte units
        const uint32_t b_lo0 = (sbase + ring_off) >> 4, b_step = (uint32_t)b_bytes >> 4;
        const uint32_t dacc = tmem_base + (uint32_t)(mi * p.Cout);
        uint32_t st = (uint32_t)mi, par = 0, acc = 0;
        int kbase = 0;
        for (int c = 0; c < chunks; ++c, kbase += 9) {
            const int hb = c % CH_HALO_BUFS;
            ptx::mbar_wait(hfull(hb), (uint32_t)((c / CH_HALO_BUFS) & 1));
            const uint32_t h_lo = (sbase + (uint32_t)(hb * halo_stride)) >> 4;
            for (int t = (mi - kbase) & (nm - 1); t < 9; t += nm) {
                ptx::mbar_wait(bfull((int)st), par);
                ptx::tc_fence_after();
                // tap (dy,dx): the halo tile read (dy+1) padded rows and (dx+1) pixels further in; the
                // descriptor's base_offset stays 0 (swizzle phase = absolute address bits, measured)
                const uint32_t a_lo = h_lo + (uint32_t)(p.tap_dy[t] + 1) * rs16 + (uint32_t)(p.tap_dx[t] + 1) * 8u;
                const uint32_t b_lo = b_lo0 + st * b_step;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    if (leader) ptx::mma_tf32_w(dacc, a_lo + 2u * kk, a_hi, b_lo + 2u * kk, b_hi, idesc, acc);
                    acc = 1;
                }
                // a ring group (CH_GROUP stages) is released by one commit per issuer, after its last stage of the group
                if ((st & (CH_GROUP - 1)) + (uint32_t)nm >= (uint32_t)CH_GROUP) {
                    if (leader) ptx::tc_commit(bempty((int)(st / CH_GROUP)));
                }
                st += (uint32_t)nm;
                if (st >= (uint32_t)S) { st -= (uint32_t)S; par ^= 1; }
            }
            if (leader) ptx::tc_commit(hempty(hb));            // chunk done: its halo buffer may be refilled
            __syncwarp();
        }
        if (leader) ptx::tc_commit(tfull);
    } else if (warp >= 4) {
        const int q = warp & 3;
        const int row = q * 32 + lane;                 // = (y * BN + bn) * 8 + x
        const int x = row & 7, g = row >> 3;
        const int bn = g % p.BN, yy = g / p.BN;
        const int gx = gx0 + x, gy = gy0 + yy, n = n0 + bn;
        const bool valid = gx < p.W && gy < p.H && n < p.B;
        const long long ob = (((long long)n * p.H + gy) * p.W + gx) * p.Cout;
        pdl_wait();                                     // (skip, if any, is the previous layers' output)
        ptx::mbar_wait(tfull, 0);
        ptx::tc_fence_after();
        if (p.shuffle_cout > 0) {
            // decoder.py:34-35 as a 3x3-neighbourhood GEMM: column (py*2+px)*Cout+co of input pixel (gy,gx)
            // is output pixel (2gy+py, 2gx+px), channel co, of the NCHW module output.
            float v[32];
            ptx::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16), v);
            ptx::tmem_ld_wait32(v);
            if (p.nmma == 2) {                          // + the second issuer's partial (columns Cout..)
                float u[32];
                ptx::tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)p.Cout, u);
                ptx::tmem_ld_wait32(u);
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = __fadd_rn(v[i], u[i]);
            }
            if (valid) {
                const int co_n = p.shuffle_cout, OH = 2 * p.H, OW = 2 * p.W;
                for (int co = 0; co < co_n; ++co)
#pragma unroll
                    for (int py = 0; py < 2; ++py) {
                        float2 o = make_float2(v[(py * 2 + 0) * co_n + co] + bias_s[co],
                                               v[(py * 2 + 1) * co_n + co] + bias_s[co]);
                        if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); }
                        *reinterpret_cast<float2 *>(p.out + (((long long)n * co_n + co) * OH + 2 * gy + py) * OW + 2 * gx) = o;
                    }
            }
        } else {
            const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
            const bool two = p.nmma == 2, have = true;
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

int ch_pow2_ceil(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

}  // namespace

bool conv_halo_supported(const ConvLaunch &p) {
    const bool nhwc = p.in_sc == 1 && p.in_sw == p.Cin && p.out_sc == 1 && p.out_sw == p.Cout;
    if (!nhwc || p.ntaps != 9 || p.in_step != 1 || p.out_step != 1 || p.OHg != p.H || p.OWg != p.W) return false;
    for (int t = 0; t < 9; ++t)
        if (p.tap_dy[t] < -1 || p.tap_dy[t] > 1 || p.tap_dx[t] < -1 || p.tap_dx[t] > 1) return false;
    return p.Cin % 32 == 0 && p.Cin <= 32 * CH_MAX_CHUNKS && p.Cout % 16 == 0 && p.Cout >= 16 && p.Cout <= 256 &&
           (reinterpret_cast<uintptr_t>(p.in) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 &&
           (p.skip == nullptr || (reinterpret_cast<uintptr_t>(p.skip) & 15) == 0);
}

int launch_conv_halo_ex(const ConvLaunch &p, const float *w_tc, int shuffle_cout, cudaStream_t s);
int launch_conv_halo(const ConvLaunch &p, const float *w_tc, cudaStream_t s) { return launch_conv_halo_ex(p, w_tc, 0, s); }

int launch_conv_halo_ex(const ConvLaunch &p, const float *w_tc, int shuffle_cout, cudaStream_t s) {
    ConvHaloParams q;
    q.bias = p.bias; q.skip = p.skip; q.out = p.out;
    q.B = p.B; q.H = p.H; q.W = p.W; q.Cin = p.Cin; q.Cout = p.Cout; q.relu = p.relu;
    q.BH = ch_pow2_ceil(p.H) < 16 ? ch_pow2_ceil(p.H) : 16;
    q.BN = 16 / q.BH;
    q.tiles_x = (p.W + 7) / 8;
    q.tiles_y = (p.H + q.BH - 1) / q.BH;
    const int tiles_n = (p.B + q.BN - 1) / q.BN;
    q.nmma = 2 * p.Cout <= 256 ? 2 : 1;       // <= 256 TMEM columns: two CTAs per SM can still allocate
    q.shuffle_cout = shuffle_cout;
    for (int t = 0; t < 9; ++t) { q.tap_w[t] = p.tap_w[t]; q.tap_dy[t] = p.tap_dy[t]; q.tap_dx[t] = p.tap_dx[t]; }

    CUtensorMap tin, tw;
    // dims ordered (c, w, n, h): the BN images of a tile interleave row by row in shared memory
    const uint64_t dims[4] = {(uint64_t)p.Cin, (uint64_t)p.W, (uint64_t)p.B, (uint64_t)p.H};
    const uint64_t strides[3] = {(uint64_t)p.Cin * 4, (uint64_t)p.H * p.W * p.Cin * 4, (uint64_t)p.W * p.Cin * 4};
    const int WP = VQB_HALO_WP;
    q.WP = WP;
    const uint32_t box[4] = {32u, (uint32_t)WP, (uint32_t)q.BN, (uint32_t)(q.BH + 2)};
    const uint32_t es[4] = {1u, 1u, 1u, 1u};
    int rc = vqb_encode_tmap_4d(&tin, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, p.in, dims, strides, box, es,
                                CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = vqb_encode_tmap_2d(&tw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w_tc, (uint64_t)p.Cin, (uint64_t)9 * p.Cout,
                            (uint64_t)p.Cin * 4, 32, (uint32_t)p.Cout, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    const int chunks = p.Cin / 32;
    const int halo_bytes = (((q.BH + 2) * q.BN * WP * 128) + 1023) & ~1023;
    const int b_bytes = p.Cout * 128;
    const int hbufs = chunks < CH_HALO_BUFS ? chunks : CH_HALO_BUFS;
    const int fixed = hbufs * halo_bytes + 8 * (2 * CH_MAX_STAGES + 2 * CH_HALO_BUFS + 1) + 8 + 256 * 4 + 1024;
    int stages = (226 * 1024 - fixed) / b_bytes;
    if (stages > CH_MAX_STAGES) stages = CH_MAX_STAGES;
    if (stages >= 9 * chunks) stages = 9 * chunks;
    else stages -= stages % CH_GROUP;             // a reused ring must hold whole commit groups
    if (stages < CH_GROUP) return VQB_ERR_UNSUPPORTED;
    q.stages = stages;
    const int smem = fixed + stages * b_bytes;
    static int attr_max = 0;
    if (smem > attr_max) {
        cudaError_t e = cudaFuncSetAttribute(conv_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr_max = smem;
    }
    const long long grid = (long long)q.tiles_x * q.tiles_y * tiles_n;
    if (grid <= 0 || grid > 0x7fffffffLL) return VQB_ERR_UNSUPPORTED;
    if (cudaError_t le = vqb_launch(conv_halo_kernel, dim3((unsigned)grid), dim3(CH_THREADS), (size_t)smem, s, tin, tw, q)) return (int)le;
    VQB_COUNT_LAUNCH(1);
    return vqb_cuda_status(cudaGetLastError());
}

// ConvTranspose2d(Cin -> Cout <= 4, k4 s2 p1), NHWC in -> NCHW out, as ONE 3x3-neighbourhood GEMM with 16 columns
// (py, px, co): w_shuffle = [9 taps][16][Cin] packed by vqb_pack_conv_weight_f32 (third region).
bool convt_shuffle_supported(int Cin, int Cout, const void *in, const void *out) {
    return Cin % 32 == 0 && Cin <= 32 * CH_MAX_CHUNKS && Cout >= 1 && Cout <= 4 &&
           (reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0;
}

int launch_convt_shuffle(const float *in, const float *w_shuffle, const float *bias, float *out, int B, int Cin, int H,
                         int W, int Cout, int relu, cudaStream_t s) {
    ConvLaunch p;
    p.in = in; p.w = nullptr; p.bias = bias; p.skip = nullptr; p.out = out;
    p.B = B; p.Cin = Cin; p.H = H; p.W = W; p.Cout = 16; p.relu = relu;
    p.OHg = H; p.OWg = W; p.in_step = 1; p.out_step = 1; p.out_py = 0; p.out_px = 0;
    p.ntaps = 9;
    for (int t = 0; t < 9; ++t) { p.tap_w[t] = t; p.tap_dy[t] = t / 3 - 1; p.tap_dx[t] = t % 3 - 1; }
    p.in_sc = 1; p.in_sw = Cin; p.in_sh = (long long)W * Cin; p.in_sn = (long long)H * W * Cin;
    p.out_sc = 1; p.out_sw = 16; p.out_sh = 0; p.out_sn = 0;      // unused by the shuffle epilogue
    return launch_conv_halo_ex(p, w_shuffle, Cout, s);
}
