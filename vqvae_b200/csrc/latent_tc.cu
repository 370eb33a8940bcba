// latent_tc.cu -- the TF32 latent stage of VQVAE.forward as two whole-image tcgen05 kernels (sm_100a).
//
// At latents of <= 8 x 16 pixels one 128-pixel tile holds BN whole images, and no receptive field crosses an image
// border, so a chain of layers can run back to back inside one CTA with the activation resident in shared memory:
//   encoder tail  E3 conv 3x3 C->C +bias +ReLU -> ResidualLayer x n (shared weights, last with the stack's ReLU)
//                 -> pre-quant 1x1 C->D +bias                       -> z_e, fp32 (N, D) rows (what the VQ reads)
//   decoder head  D1 convT 3x3 s1 D->C +bias +ReLU -> ResidualLayer x n -> D2 convT k4s2 C->C/2 +bias +ReLU
//                                                                       -> fp32 NHWC (B, 2H, 2W, C/2)
// The C-channel activation lives in C/32 halo buffers of the conv_halo / res_tc layout ({32 ch, WP px, BN img,
// BH+2 rows}, 128B-swizzled K-major rows); their zero borders are every layer's padding.  A layer's epilogue
// rewrites the buffers in place once the layer's MMAs have completed, and the next layer's MMAs wait for that.
// Every tap of every layer is a shifted UMMA descriptor into the resident tile (D2: four output parities x 2x2
// taps); only weights stream.
//
// One host-built plan of k-steps (one k-step = one 32-channel weight tile x four K = 8 MMAs) covers the whole chain;
// the weight producer streams it through one ring of 16 KB stages without ever looking at layer boundaries, so the
// first stages of layer n+1 are resident when layer n's epilogue finishes.
//
// Numerics: each layer keeps the k-step order and the split of k-steps over TMEM accumulators of the per-layer
// kernel it replaces (conv_halo: 2 partials by k-step parity; res_tc: 4 partials by k-step mod 4; conv_tc 1x1 and
// k4s2 phases: 2 partials by chunk parity), and the epilogues sum the partials and apply bias / skip / ReLU in the
// same order, so the outputs are bitwise those of the per-layer chain.  Which warp issues an MMA does not change
// the arithmetic: two issuer warps split the partials between them.
#include "bf16_common.cuh"
#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int LT_THREADS = 384;       // warp 0 weight producer, 1-2 MMA issuers (2 also TMEM), 3 input loader,
                                      // 4-11 epilogue (two warps per TMEM lane quadrant, half the columns each)
constexpr int LT_NISS = 2;            // MMA issuer warps
constexpr int LT_MAX_STAGES = 8;
constexpr int LT_STAGE = 16384;       // ring stage: one 128-row weight tile, or several smaller ones
constexpr int LT_MAXK = 320;          // k-steps in the plan
constexpr int LT_MAXG = 16;           // GEMM groups (layers; D2 counts one per output parity)
constexpr int LT_A2 = 128 * 128;      // relu(GEMM1) of a residual layer: the A operand of its 1x1 GEMM
constexpr int LT_TMEM_COLS = 512;

// epilogue kinds
enum { EPI_ACT = 0,        // sum 2 partials (cols 0, C) + bias -> ReLU -> halo buffers in place (E3, D1)
       EPI_RES1 = 1,       // sum 4 partials (cols 0, 32, 64, 96) -> ReLU -> A2
       EPI_RES2 = 2,       // D (col 128) + skip (the resident activation) -> ReLU -> halo buffers in place
       EPI_ROWS = 3,       // sum 2 partials (cols 0, 64) + bias -> z_e rows (pre-quant 1x1)
       EPI_D2 = 4 };       // sum 2 partials (cols 128 ph, +64) + bias -> ReLU -> NHWC output pixel (2y+py, 2x+px)

// plan word 0 (issuer): a_off16 [0,14) | TMEM column [14,23) | accumulate [23] | first of stage [24] |
//                       last of stage [25] | issuer [26] | offset in the stage, KB [27,31)
// plan word 1 (producer): weight row [0,12) | 32-channel chunk [12,15) | tensor map [15,17) | stage KB [17,22)
constexpr uint32_t PL_FIRST = 1u << 24, PL_LAST = 1u << 25;

struct LatGroup {
    short k0, k1;           // plan k-steps [k0, k1)
    short n, sbo;           // MMA N; A-operand stride between 8-row groups (halo: WP*128, A2: 1024)
    short wait;             // the group whose epilogue must have finished (-1: the input tile)
    short epi, ph, boff;    // epilogue kind, D2 output parity, bias offset in shared memory
};

struct LatParams {
    float *out;
    const float *bias0, *bias1;     // C floats (E3 / D1) at smem bias[0..C), D or C/2 floats (1x1 / D2) at [C..)
    int B, H, W, BN, WP;
    int nin;                        // 32-channel chunks of the input (E2 output: C/32, z_q: D/32)
    int in_bytes;                   // bytes of one input chunk's halo box
    int nbias1;
    int S, halo_stride, ngroups, nk;
    LatGroup grp[LT_MAXG];
    uint2 plan[LT_MAXK];
};

__global__ void __launch_bounds__(LT_THREADS, 1)
latent_tc_kernel(const __grid_constant__ CUtensorMap tma_in, const __grid_constant__ CUtensorMap tw0,
                 const __grid_constant__ CUtensorMap tw1, const __grid_constant__ CUtensorMap tw2,
                 const __grid_constant__ CUtensorMap tw3, const __grid_constant__ LatParams p) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = ptx::smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (sbase - raw);

    constexpr int NBUF = 4;                                     // C = 128: four 32-channel halo buffers
    const int S = p.S, hs = p.halo_stride;
    const uint32_t a2_off = (uint32_t)(NBUF * hs);
    const uint32_t ring_off = a2_off + LT_A2;
    const uint32_t plan_off = ring_off + (uint32_t)(S * LT_STAGE);
    const uint32_t bias_off = plan_off + LT_MAXK * 8;
    const uint32_t bar_off = bias_off + 256 * 4;
    const uint32_t bars = sbase + bar_off;
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (LT_MAX_STAGES + s); };
    auto accfull = [&](int g) { return bars + 8u * (2 * LT_MAX_STAGES + g); };
    auto actready = [&](int g) { return bars + 8u * (2 * LT_MAX_STAGES + LT_MAXG + g); };
    const uint32_t inready = bars + 8u * (2 * LT_MAX_STAGES + 2 * LT_MAXG);
    volatile uint32_t *tmem_holder = reinterpret_cast<volatile uint32_t *>(sm + bar_off + 8 * (2 * LT_MAX_STAGES + 2 * LT_MAXG + 1));
    uint2 *plan_s = reinterpret_cast<uint2 *>(sm + plan_off);
    float *bias_s = reinterpret_cast<float *>(sm + bias_off);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0 = blockIdx.x * p.BN;

    if (tid < S) { ptx::mbar_init(full(tid), 1); ptx::mbar_init(empty(tid), LT_NISS); }
    if (tid >= 32 && tid < 32 + p.ngroups) {
        ptx::mbar_init(accfull(tid - 32), LT_NISS);             // one commit per issuer
        ptx::mbar_init(actready(tid - 32), 8);                  // one arrival per epilogue warp
    }
    if (tid == 64) ptx::mbar_init(inready, 1);
    if (tid == 96) { ptx::prefetch_tmap(&tma_in); ptx::prefetch_tmap(&tw0); ptx::prefetch_tmap(&tw1); }
    if (tid == 97) { ptx::prefetch_tmap(&tw2); ptx::prefetch_tmap(&tw3); }
    ptx::fence_mbar_init();
    for (int k = tid; k < p.nk; k += LT_THREADS) plan_s[k] = p.plan[k];
    for (int c = tid; c < 128 + p.nbias1; c += LT_THREADS)
        bias_s[c] = c < 128 ? (p.bias0 ? __ldg(p.bias0 + c) : 0.f) : (p.bias1 ? __ldg(p.bias1 + c - 128) : 0.f);
    if (warp == 2) ptx::tmem_alloc(sbase + bar_off + 8 * (2 * LT_MAX_STAGES + 2 * LT_MAXG + 1), LT_TMEM_COLS);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    pdl_launch_dependents();       // the next kernel may start its prologue (it blocks in its own pdl_wait)

    if (warp == 0) {
        // ---- weight producer: the whole plan through the ring, paced by ring space only ----
        const bool leader = ptx::elect_one();
        uint32_t st = 0, par = 0;
        bool wrapped = false;
        for (int k = 0; k < p.nk; ++k) {
            const uint2 e = plan_s[k];
            if (e.x & PL_FIRST) {
                if (wrapped) ptx::mbar_wait(empty((int)st), par ^ 1u);
                if (leader) ptx::mbar_expect_tx(full((int)st), ((e.y >> 17) & 31u) * 1024u);
            }
            if (leader) {
                const uint32_t m = (e.y >> 15) & 3u;
                const CUtensorMap *map = m == 0 ? &tw0 : m == 1 ? &tw1 : m == 2 ? &tw2 : &tw3;
                ptx::tma_load_2d(sbase + ring_off + st * LT_STAGE + ((e.x >> 27) & 15u) * 1024u, map, full((int)st),
                                 (int)((e.y >> 12) & 7u) * 32, (int)(e.y & 4095u));
            }
            if (e.x & PL_LAST) {
                if (++st == (uint32_t)S) { st = 0; par ^= 1u; wrapped = true; }
            }
            __syncwarp();
        }
    } else if (warp == 1 || warp == 2) {
        // ---- MMA issuers: issuer mi issues the k-steps of its partials; both wait for and release EVERY ring
        // stage (a parity wait cannot tell use k from use k+2, DESIGN 4.0) ----
        const uint32_t mi = (uint32_t)(warp - 1);
        const bool leader = ptx::elect_one();
        const uint32_t b_hi = ptx::desc_hi_sw128(1024);
        const uint32_t s16 = sbase >> 4, ring16 = (sbase + ring_off) >> 4;
        uint32_t st = 0, par = 0;
        for (int g = 0; g < p.ngroups; ++g) {
            const LatGroup G = p.grp[g];
            ptx::mbar_wait(G.wait < 0 ? inready : actready(G.wait), 0);
            ptx::tc_fence_after();
            const uint32_t idesc = ptx::instr_desc(ptx::FMT_TF32, 128, (uint32_t)G.n);
            const uint32_t a_hi = ptx::desc_hi_sw128((uint32_t)G.sbo);
            for (int k = G.k0; k < G.k1; ++k) {
                const uint32_t e = plan_s[k].x;
                if (e & PL_FIRST) {
                    ptx::mbar_wait(full((int)st), par);
                    ptx::tc_fence_after();
                }
                if (((e >> 26) & 1u) == mi) {
                    const uint32_t a_lo = s16 + (e & 0x3FFFu);
                    const uint32_t b_lo = ring16 + st * (LT_STAGE >> 4) + ((e >> 27) & 15u) * 64u;
                    const uint32_t d = tmem_base + ((e >> 14) & 511u);
                    uint32_t acc = (e >> 23) & 1u;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        if (leader) ptx::mma_tf32_w(d, a_lo + 2u * kk, a_hi, b_lo + 2u * kk, b_hi, idesc, acc);
                        acc = 1;
                    }
                }
                if (e & PL_LAST) {
                    if (leader) ptx::tc_commit(empty((int)st));
                    if (++st == (uint32_t)S) { st = 0; par ^= 1u; }
                }
                __syncwarp();
            }
            if (leader) ptx::tc_commit(accfull(g));
            __syncwarp();
        }
    } else if (warp == 3) {
        // ---- input tile: the previous kernel's output, with a zero-filled 1-pixel halo ----
        const bool leader = ptx::elect_one();
        pdl_wait();
        if (leader) {
            ptx::mbar_expect_tx(inready, (uint32_t)(p.nin * p.in_bytes));
            for (int c = 0; c < p.nin; ++c)         // box {32 ch, WP px, BN img, BH+2 rows} from (x, y) = (-1, -1)
                ptx::tma_load_4d(sbase + (uint32_t)(c * hs), &tma_in, inready, c * 32, -1, n0, -1);
        }
        __syncwarp();
    } else {
        // ---- epilogue: thread = one row of the 128-row accumulator (= one pixel of the tile) ----
        const int q = warp & 3, h = (warp - 4) >> 2;
        const int row = q * 32 + lane;                      // row = (y * BN + bn) * 8 + x
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        const int x = row & 7, grp = row >> 3;
        const int bn = grp % p.BN, y = grp / p.BN;
        const int n = n0 + bn;
        const bool valid = x < p.W && y < p.H && n < p.B;
        const int hrow = ((y + 1) * p.BN + bn) * p.WP + x + 1;        // this pixel's row of a halo buffer
        const int sw = hrow & 7;
        pdl_wait();                                         // outputs may still be read by earlier kernels
        // buffers the input does not fill (decoder: D channels in, C out) start as zeros: their borders are padding
        for (int b = p.nin; b < NBUF; ++b) {
            float4 *z = reinterpret_cast<float4 *>(sm + b * hs);
            for (int i = tid - 128; i < hs / 16; i += 256) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        // every thread's zeros land before any thread writes its own rows of those buffers (first EPI_ACT below)
        if (p.nin < NBUF) ptx::named_bar_sync(1, 256);
        for (int g = 0; g < p.ngroups; ++g) {
            const LatGroup G = p.grp[g];
            ptx::mbar_wait_sleep(accfull(g), 0);
            ptx::tc_fence_after();
            if (G.epi == EPI_ACT) {
                for (int cc = 2 * h; cc < 2 * h + 2; ++cc) {
                    float v[32], u[32];
                    ptx::tmem_ld32(taddr + (uint32_t)(cc * 32), v);
                    ptx::tmem_ld32(taddr + (uint32_t)(128 + cc * 32), u);
                    ptx::tmem_ld_wait32(v); ptx::tmem_ld_wait32(u);
                    unsigned char *dst = sm + cc * hs + hrow * 128;
#pragma unroll
                    for (int c16 = 0; c16 < 8; ++c16) {
                        const float *bb = bias_s + G.boff + cc * 32 + c16 * 4;
                        float4 o;
                        o.x = fmaxf(__fadd_rn(v[c16 * 4 + 0], u[c16 * 4 + 0]) + bb[0], 0.f);
                        o.y = fmaxf(__fadd_rn(v[c16 * 4 + 1], u[c16 * 4 + 1]) + bb[1], 0.f);
                        o.z = fmaxf(__fadd_rn(v[c16 * 4 + 2], u[c16 * 4 + 2]) + bb[2], 0.f);
                        o.w = fmaxf(__fadd_rn(v[c16 * 4 + 3], u[c16 * 4 + 3]) + bb[3], 0.f);
                        if (!valid) o = make_float4(0.f, 0.f, 0.f, 0.f);
                        *reinterpret_cast<float4 *>(dst + ((c16 ^ sw) << 4)) = o;
                    }
                }
            } else if (G.epi == EPI_RES1) {
                if (h == 0) {
                    float v[32], u1[32], u2[32], u3[32];
                    ptx::tmem_ld32(taddr, v);
                    ptx::tmem_ld32(taddr + 32u, u1);
                    ptx::tmem_ld32(taddr + 64u, u2);
                    ptx::tmem_ld32(taddr + 96u, u3);
                    ptx::tmem_ld_wait32(v); ptx::tmem_ld_wait32(u1); ptx::tmem_ld_wait32(u2); ptx::tmem_ld_wait32(u3);
                    unsigned char *arow = sm + a2_off + row * 128;
#pragma unroll
                    for (int c16 = 0; c16 < 8; ++c16) {
                        float4 o;
                        o.x = fmaxf(__fadd_rn(__fadd_rn(__fadd_rn(v[c16 * 4 + 0], u1[c16 * 4 + 0]), u2[c16 * 4 + 0]), u3[c16 * 4 + 0]), 0.f);
                        o.y = fmaxf(__fadd_rn(__fadd_rn(__fadd_rn(v[c16 * 4 + 1], u1[c16 * 4 + 1]), u2[c16 * 4 + 1]), u3[c16 * 4 + 1]), 0.f);
                        o.z = fmaxf(__fadd_rn(__fadd_rn(__fadd_rn(v[c16 * 4 + 2], u1[c16 * 4 + 2]), u2[c16 * 4 + 2]), u3[c16 * 4 + 2]), 0.f);
                        o.w = fmaxf(__fadd_rn(__fadd_rn(__fadd_rn(v[c16 * 4 + 3], u1[c16 * 4 + 3]), u2[c16 * 4 + 3]), u3[c16 * 4 + 3]), 0.f);
                        *reinterpret_cast<float4 *>(arow + ((c16 ^ (row & 7)) << 4)) = o;
                    }
                }
            } else if (G.epi == EPI_RES2) {
                for (int cc = 2 * h; cc < 2 * h + 2; ++cc) {
                    float v[32];
                    ptx::tmem_ld32(taddr + (uint32_t)(128 + cc * 32), v);
                    ptx::tmem_ld_wait32(v);
                    unsigned char *srow = sm + cc * hs + hrow * 128;
#pragma unroll
                    for (int c16 = 0; c16 < 8; ++c16) {
                        float4 *ptr = reinterpret_cast<float4 *>(srow + ((c16 ^ sw) << 4));
                        const float4 sk = *ptr;
                        float4 o = make_float4(fmaxf(v[c16 * 4] + sk.x, 0.f), fmaxf(v[c16 * 4 + 1] + sk.y, 0.f),
                                               fmaxf(v[c16 * 4 + 2] + sk.z, 0.f), fmaxf(v[c16 * 4 + 3] + sk.w, 0.f));
                        if (!valid) o = make_float4(0.f, 0.f, 0.f, 0.f);
                        *ptr = o;
                    }
                }
            } else {
                // EPI_ROWS / EPI_D2: 32 of the 64 output channels per thread, straight to global memory in 32-byte stores
                const bool d2 = G.epi == EPI_D2;
                const uint32_t col = d2 ? (uint32_t)(G.ph * 128) : 0u;
                float v[32], u[32];
                ptx::tmem_ld32(taddr + col + (uint32_t)(h * 32), v);
                ptx::tmem_ld32(taddr + col + 64u + (uint32_t)(h * 32), u);
                ptx::tmem_ld_wait32(v); ptx::tmem_ld_wait32(u);
                if (valid) {
                    long long pix;
                    if (d2) {
                        const int py = G.ph >> 1, px = G.ph & 1;
                        pix = ((long long)n * 2 * p.H + 2 * y + py) * (2 * p.W) + 2 * x + px;
                    } else {
                        pix = ((long long)n * p.H + y) * p.W + x;
                    }
                    float *dst = p.out + pix * 64 + h * 32;
                    const float *bb = bias_s + G.boff + h * 32;
                    uint32_t o[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        float t = __fadd_rn(v[i], u[i]) + bb[i];
                        if (d2) t = fmaxf(t, 0.f);
                        o[i] = __float_as_uint(t);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        st_global_256(dst + 8 * j, o[8 * j], o[8 * j + 1], o[8 * j + 2], o[8 * j + 3], o[8 * j + 4],
                                      o[8 * j + 5], o[8 * j + 6], o[8 * j + 7]);
                }
            }
            ptx::fence_proxy_async();       // generic smem writes -> visible to the tensor core's async proxy
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(actready(g));
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, LT_TMEM_COLS);
}

}  // namespace

namespace {

constexpr int LT_MAX_RES = 4;         // residual applications a plan holds (k-steps and groups above)

// Host-side plan: k-steps appended layer by layer, grouped into ring stages of <= 16 KB that never span two layers.
struct LatPlan {
    LatParams &p;
    int first = -1, used = 0;
    bool ok = true;
    explicit LatPlan(LatParams &q) : p(q) { p.ngroups = 0; p.nk = 0; }
    void close_stage() {
        if (first < 0) return;
        p.plan[p.nk - 1].x |= PL_LAST;
        p.plan[first].y |= (uint32_t)(used / 1024) << 17;
        first = -1; used = 0;
    }
    // a_off: byte offset of the A window from the smem base; col: TMEM column of the partial; acc: not the partial's
    // first k-step; map / chunk / wrow: the weight tile; bytes: its size (N rows x 128 B)
    void step(uint32_t a_off, int col, int acc, int issuer, int map, int chunk, int wrow, int bytes) {
        if (first >= 0 && used + bytes > LT_STAGE) close_stage();
        if (p.nk >= LT_MAXK || (a_off >> 4) >= (1u << 14)) { ok = false; return; }
        uint2 e;
        e.x = (a_off >> 4) | (uint32_t)col << 14 | (uint32_t)acc << 23 | (uint32_t)issuer << 26 | (uint32_t)(used / 1024) << 27;
        e.y = (uint32_t)wrow | (uint32_t)chunk << 12 | (uint32_t)map << 15;
        if (first < 0) { first = p.nk; e.x |= PL_FIRST; }
        used += bytes;
        p.plan[p.nk++] = e;
    }
    void begin(int n, int sbo, int epi, int ph, int boff) {
        if (p.ngroups >= LT_MAXG) { ok = false; return; }
        LatGroup &g = p.grp[p.ngroups];
        g.k0 = (short)p.nk; g.n = (short)n; g.sbo = (short)sbo; g.wait = (short)(p.ngroups - 1);
        g.epi = (short)epi; g.ph = (short)ph; g.boff = (short)boff;
    }
    void end() {
        if (!ok) return;
        close_stage();
        p.grp[p.ngroups++].k1 = (short)p.nk;
    }
};

int lt_pow2_ceil(int x) {
    int v = 1;
    while (v < x) v <<= 1;
    return v;
}

// Tile geometry and shared-memory plan of conv_halo / res_tc at a one-tile latent; VQB_ERR_UNSUPPORTED when the
// resident activation and a ring of at least two stages do not fit.
int lat_geometry(LatParams &q, int B, int H, int W, int *smem) {
    if (W > 8 || H > 16) return VQB_ERR_UNSUPPORTED;
    const int BH = lt_pow2_ceil(H) < 16 ? lt_pow2_ceil(H) : 16;
    q.B = B; q.H = H; q.W = W; q.BN = 16 / BH; q.WP = vqb_halo_wp();
    q.in_bytes = (BH + 2) * q.BN * q.WP * 128;
    q.halo_stride = (q.in_bytes + 1023) & ~1023;
    const int fixed = 4 * q.halo_stride + LT_A2 + LT_MAXK * 8 + 256 * 4 + 8 * (2 * LT_MAX_STAGES + 2 * LT_MAXG + 2);
    int S = (227 * 1024 - 1024 - fixed) / LT_STAGE;
    if (S > LT_MAX_STAGES) S = LT_MAX_STAGES;
    if (S < 2) return VQB_ERR_UNSUPPORTED;
    q.S = S;
    *smem = 1024 + fixed + S * LT_STAGE;
    return 0;
}

// the residual applications: GEMM1 (3x3 C -> 32, four partials by k-step mod 4, as res_tc) and GEMM2 (1x1 32 -> C)
void plan_residual(LatPlan &pl, const LatParams &q, int n_res) {
    const int rs = q.BN * q.WP * 128, hs = q.halo_stride;
    for (int app = 0; app < n_res; ++app) {
        pl.begin(32, q.WP * 128, EPI_RES1, 0, 0);
        for (int c = 0; c < 4; ++c)
            for (int t = 0; t < 9; ++t) {
                const int k = c * 9 + t, part = k & 3;
                pl.step((uint32_t)(c * hs + (t / 3) * rs + (t % 3) * 128), part * 32, k >= 4, part & 1, 1, c, t * 32, 32 * 128);
            }
        pl.end();
        pl.begin(128, 1024, EPI_RES2, 0, 0);
        pl.step((uint32_t)(4 * hs), 128, 0, 0, 2, 0, 0, 128 * 128);
        pl.end();
    }
}

int launch_latent(const CUtensorMap &tin, const CUtensorMap (&tw)[4], const LatParams &q, int smem, cudaStream_t s) {
    static int attr_max = 0;
    if (smem > attr_max) {
        cudaError_t e = cudaFuncSetAttribute(latent_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr_max = smem;
    }
    const long long grid = ((long long)q.B + q.BN - 1) / q.BN;
    if (grid <= 0 || grid > 0x7fffffffLL) return VQB_ERR_UNSUPPORTED;
    if (cudaError_t le = vqb_launch(latent_tc_kernel, dim3((unsigned)grid), dim3(LT_THREADS), (size_t)smem, s, tin, tw[0],
                                    tw[1], tw[2], tw[3], q))
        return (int)le;
    VQB_COUNT_LAUNCH(1);
    return vqb_cuda_status(cudaGetLastError());
}

int tmap_input(CUtensorMap *m, const float *in, const LatParams &q, int Cin) {
    // dims ordered (c, w, n, h): the BN images of a tile interleave row by row in shared memory
    const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)q.W, (uint64_t)q.B, (uint64_t)q.H};
    const uint64_t strides[3] = {(uint64_t)Cin * 4, (uint64_t)q.H * q.W * Cin * 4, (uint64_t)q.W * Cin * 4};
    const uint32_t box[4] = {32u, (uint32_t)q.WP, (uint32_t)q.BN, (uint32_t)(q.in_bytes / (q.BN * q.WP * 128))};
    const uint32_t es[4] = {1u, 1u, 1u, 1u};
    return vqb_encode_tmap_4d(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, in, dims, strides, box, es, CU_TENSOR_MAP_SWIZZLE_128B);
}

// K-major weight tiles [taps * Cout][Cin] (the second region of vqb_pack_conv_weight_f32), boxes {32 ch, Cout rows}
int tmap_weight(CUtensorMap *m, const float *w_tc, int taps, int Cout, int Cin) {
    return vqb_encode_tmap_2d(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w_tc, (uint64_t)Cin, (uint64_t)taps * Cout,
                              (uint64_t)Cin * 4, 32, (uint32_t)Cout, CU_TENSOR_MAP_SWIZZLE_128B);
}

bool lt_aligned(const void *a, const void *b, const void *c, const void *d, const void *e, const void *f) {
    return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
             reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(e) | reinterpret_cast<uintptr_t>(f)) & 15) == 0;
}

}  // namespace

extern "C" int vqb_latent_encoder_f32(const float *in, const float *w3_packed, const float *b3, const float *w1_packed,
                                      const float *w2_packed, const float *wq_packed, const float *bq, float *z_e, int B,
                                      int H, int W, int C, int Cmid, int D, int n_res, void *stream) {
    if (!in || !w3_packed || !w1_packed || !w2_packed || !wq_packed || !z_e) return VQB_ERR_BAD_ARG;
    if (B <= 0 || H <= 0 || W <= 0 || C <= 0 || Cmid <= 0 || D <= 0 || n_res < 1) return VQB_ERR_BAD_ARG;
    if (C != 128 || Cmid != 32 || D != 64 || n_res > LT_MAX_RES) return VQB_ERR_UNSUPPORTED;
    if (!lt_aligned(in, w3_packed, w1_packed, w2_packed, wq_packed, z_e)) return VQB_ERR_ALIGNMENT;
    LatParams q;
    int smem = 0;
    if (int rc = lat_geometry(q, B, H, W, &smem)) return rc;
    q.out = z_e; q.bias0 = b3; q.bias1 = bq; q.nbias1 = D; q.nin = C / 32;
    LatPlan pl(q);
    const int rs = q.BN * q.WP * 128, hs = q.halo_stride;
    // E3: conv 3x3 C -> C, two partials by k-step parity (conv_halo), + bias, ReLU (the stack's first ReLU)
    pl.begin(128, q.WP * 128, EPI_ACT, 0, 0);
    for (int c = 0; c < 4; ++c)
        for (int t = 0; t < 9; ++t) {
            const int k = c * 9 + t, part = k & 1;
            pl.step((uint32_t)(c * hs + (t / 3) * rs + (t % 3) * 128), part * 128, k >= 2, part, 0, c, t * 128, 128 * 128);
        }
    pl.end();
    plan_residual(pl, q, n_res);
    // pre-quant 1x1 C -> D: two partials by chunk parity (conv_tc), + bias
    pl.begin(64, q.WP * 128, EPI_ROWS, 0, 128);
    for (int c = 0; c < 4; ++c) pl.step((uint32_t)(c * hs + rs + 128), (c & 1) * 64, c >= 2, c & 1, 3, c, 0, 64 * 128);
    pl.end();
    if (!pl.ok) return VQB_ERR_UNSUPPORTED;

    CUtensorMap tin, tw[4];
    int rc = tmap_input(&tin, in, q, C);
    if (!rc) rc = tmap_weight(&tw[0], w3_packed + (size_t)9 * C * C, 9, C, C);
    if (!rc) rc = tmap_weight(&tw[1], w1_packed + (size_t)9 * C * Cmid, 9, Cmid, C);
    if (!rc) rc = tmap_weight(&tw[2], w2_packed + (size_t)C * Cmid, 1, C, Cmid);
    if (!rc) rc = tmap_weight(&tw[3], wq_packed + (size_t)C * D, 1, D, C);
    if (rc) return rc;
    return launch_latent(tin, tw, q, smem, (cudaStream_t)stream);
}

extern "C" int vqb_latent_decoder_f32(const float *zq, const float *wt1_packed, const float *bt1, const float *w1_packed,
                                      const float *w2_packed, const float *wt2_packed, const float *bt2, float *out, int B,
                                      int H, int W, int D, int C, int Cmid, int Cout, int n_res, void *stream) {
    if (!zq || !wt1_packed || !w1_packed || !w2_packed || !wt2_packed || !out) return VQB_ERR_BAD_ARG;
    if (B <= 0 || H <= 0 || W <= 0 || D <= 0 || C <= 0 || Cmid <= 0 || Cout <= 0 || n_res < 1) return VQB_ERR_BAD_ARG;
    if (D != 64 || C != 128 || Cmid != 32 || Cout != 64 || n_res > LT_MAX_RES) return VQB_ERR_UNSUPPORTED;
    if (!lt_aligned(zq, wt1_packed, w1_packed, w2_packed, wt2_packed, out)) return VQB_ERR_ALIGNMENT;
    LatParams q;
    int smem = 0;
    if (int rc = lat_geometry(q, B, H, W, &smem)) return rc;
    q.out = out; q.bias0 = bt1; q.bias1 = bt2; q.nbias1 = Cout; q.nin = D / 32;
    LatPlan pl(q);
    const int rs = q.BN * q.WP * 128, hs = q.halo_stride;
    // D1: ConvTranspose 3x3 s1 D -> C = 3x3 conv with taps (dy, dx) = (1 - r, 1 - s), two partials by k-step parity
    // (conv_halo), + bias, ReLU (the stack's first ReLU)
    pl.begin(128, q.WP * 128, EPI_ACT, 0, 0);
    for (int c = 0; c < D / 32; ++c)
        for (int t = 0; t < 9; ++t) {
            const int k = c * 9 + t, part = k & 1;
            pl.step((uint32_t)(c * hs + (2 - t / 3) * rs + (2 - t % 3) * 128), part * 128, k >= 2, part, 0, c, t * 128,
                    128 * 128);
        }
    pl.end();
    plan_residual(pl, q, n_res);
    // D2: ConvTranspose k4 s2 p1 C -> Cout, output parity (py, px) = the 2x2 taps r = py+1-2dy, s = px+1-2dx, k-steps
    // tap-major with two partials by chunk parity (conv_tc), + bias, ReLU
    const int gres = q.ngroups - 1;
    for (int py = 0; py < 2; ++py)
        for (int px = 0; px < 2; ++px) {
            const int ph = py * 2 + px;
            pl.begin(64, q.WP * 128, EPI_D2, ph, 128);
            q.grp[q.ngroups].wait = (short)gres;
            int k = 0;
            for (int r = 0; r < 4; ++r) {
                if ((py + 1 - r) % 2 != 0) continue;
                const int dy = (py + 1 - r) / 2;
                for (int s = 0; s < 4; ++s) {
                    if ((px + 1 - s) % 2 != 0) continue;
                    const int dx = (px + 1 - s) / 2;
                    for (int c = 0; c < 4; ++c, ++k)
                        pl.step((uint32_t)(c * hs + (dy + 1) * rs + (dx + 1) * 128), ph * 128 + (k & 1) * 64, k >= 2, k & 1, 3,
                                c, (r * 4 + s) * Cout, Cout * 128);
                }
            }
            pl.end();
        }
    if (!pl.ok) return VQB_ERR_UNSUPPORTED;

    CUtensorMap tin, tw[4];
    int rc = tmap_input(&tin, zq, q, D);
    if (!rc) rc = tmap_weight(&tw[0], wt1_packed + (size_t)9 * D * C, 9, C, D);
    if (!rc) rc = tmap_weight(&tw[1], w1_packed + (size_t)9 * C * Cmid, 9, Cmid, C);
    if (!rc) rc = tmap_weight(&tw[2], w2_packed + (size_t)C * Cmid, 1, C, Cmid);
    if (!rc) rc = tmap_weight(&tw[3], wt2_packed + (size_t)16 * C * Cout, 16, Cout, C);
    if (rc) return rc;
    return launch_latent(tin, tw, q, smem, (cudaStream_t)stream);
}
