// res_tc.cu -- one ResidualLayer application as ONE tcgen05 kernel (sm_100a, TF32 operands).
//
// Replaces residual.py:18-29 as it is actually evaluated (SURVEY Q2: the in-place ReLU makes the
// layer relu(x) + W2 . relu(W1 (*) relu(x)); the caller passes r = relu(x) >= 0):
//     out = act( r + W2 . relu( W1 (*) r ) )          W1: 3x3 C->Cmid (no bias), W2: 1x1 Cmid->C
// with act = ReLU when the next consumer applies one first (always inside a ResidualStack).
// Five PyTorch launches (relu, conv, relu, conv, add) and the (B,Cmid,H,W) intermediate's HBM
// round trip become two chained GEMMs inside one CTA per 128-pixel tile:
//   GEMM1  D1[128][Cmid] = sum_{9 taps, C/32 chunks} A[128][32] * W1[Cmid][32]^T   (A = one halo tile per
//          chunk, the nine taps are shifted UMMA descriptors into it, as conv_halo.cu; W1 streams)
//   epi1   tcgen05.ld D1 -> ReLU -> written back to shared memory as the K-major, 128B-swizzled
//          A operand of GEMM2 (one 128-byte row per pixel per 32 channels)
//   GEMM2  D2[128][C] = A2[128][Cmid] * W2[C][Cmid]^T
//   epi2   tcgen05.ld D2 -> + r (skip, from global/L2) -> ReLU -> NHWC store
#include "common.cuh"
#include "ptx.cuh"

namespace {

constexpr int RT_THREADS = 320;       // warps 0-3 epilogue, 4 TMA producer, 5 TMEM allocator, 6-9 MMA issuers
constexpr int RT_MAX_STAGES = 32;     // W1 tile ring, as deep as shared memory allows
constexpr int RT_GROUP = 4;           // ring stages released per tcgen05.commit (a commit costs ~230 cycles)
constexpr int RT_HALO_BUFS = 2;       // double-buffered halo tiles
constexpr int RT_A_BYTES = 128 * 128;
constexpr int RT_MAX_CHUNKS = 8;

struct ResTcParams {
    const float *skip;      // r, NHWC (B,H,W,C)
    float *out;             // NHWC (B,H,W,C)
    int B, H, W, C, Cmid;
    int BH, BN, tiles_x, tiles_y;          // tile = 8 px wide x (BH rows x BN images = 16)
    int stages;
    int WP;                 // halo tile width in pixels: 8 + 1 each side = VQB_HALO_WP (see conv_halo.cu)
    int relu_out;
    int nprod;              // W1 producer warps (2 in staged mode: warp 5 takes the odd k-steps; one warp issuing a 4 KB
                            // box per k-step behind an mbarrier wait could not keep four MMA issuers fed)
    int nmma;               // GEMM1 issuer warps (1, 2 or 4): k-step i goes to issuer i % nmma, each accumulates its own
                            // D1 partial in TMEM; epilogue 1 sums them in a fixed order (deterministic)
    int napp;               // applications of the (shared-weight) layer chained inside the kernel (residual.py:45-50);
                            // > 1 only in staged mode with tiles that hold whole images: the activation then stays
                            // in the halo buffers (borders = the conv's zero padding) and is rewritten in place
    int staged;             // 1: all halo chunks resident (skip read from smem) and the output tile is
                            //    staged in smem (ring + A2 + W2 region) and TMA-stored
};

__global__ void __launch_bounds__(RT_THREADS)
res_tc_kernel(const __grid_constant__ CUtensorMap tma_in, const __grid_constant__ CUtensorMap tma_w1,
              const __grid_constant__ CUtensorMap tma_w2, const __grid_constant__ CUtensorMap tma_out,
              const ResTcParams p) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = ptx::smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (sbase - raw);

    const int S = p.stages;
    const int chunks = p.C / 32;
    const int RT_WP = p.WP;
    const int halo_bytes = (p.BH + 2) * p.BN * RT_WP * 128; // per 32-channel chunk
    const int halo_stride = (halo_bytes + 1023) & ~1023;    // buffers start on swizzle-pattern boundaries
    const int stage_bytes = p.Cmid * 128;                   // W1 tile of one (tap, chunk)
    const int matoms = p.Cmid / 32;                         // 128-byte atoms of the GEMM2 K dimension
    const int hbufs = (p.staged || chunks < RT_HALO_BUFS) ? chunks : RT_HALO_BUFS;
    const uint32_t ring_off = (uint32_t)(hbufs * halo_stride);
    const uint32_t a2_off = ring_off + (uint32_t)(S * stage_bytes);    // A2: matoms x [128 rows][128 B]
    const uint32_t w2_off = a2_off + (uint32_t)(matoms * RT_A_BYTES);   // W2: matoms x [C rows][128 B]
    const uint32_t bar_off = w2_off + (uint32_t)(matoms * p.C * 128);
    const uint32_t bars = sbase + bar_off;
    auto full = [&](int s) { return bars + 8u * s; };
    auto empty = [&](int s) { return bars + 8u * (RT_MAX_STAGES + s); };
    const uint32_t w2full = bars + 8u * (2 * RT_MAX_STAGES + 0);
    const uint32_t d1full = bars + 8u * (2 * RT_MAX_STAGES + 1);
    const uint32_t a2ready = bars + 8u * (2 * RT_MAX_STAGES + 2);
    const uint32_t d2full = bars + 8u * (2 * RT_MAX_STAGES + 3);
    auto hfull = [&](int b) { return bars + 8u * (2 * RT_MAX_STAGES + 4 + b); };
    auto hempty = [&](int b) { return bars + 8u * (2 * RT_MAX_STAGES + 4 + RT_MAX_CHUNKS + b); };
    const uint32_t actready = bars + 8u * (2 * RT_MAX_STAGES + 4 + 2 * RT_MAX_CHUNKS);   // in-place activation rewritten
    constexpr int RT_MISC = 8 * (2 * RT_MAX_STAGES + 4 + 2 * RT_MAX_CHUNKS + 2);
    volatile uint32_t *tmem_holder = reinterpret_cast<volatile uint32_t *>(sm + bar_off + RT_MISC);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int tcols = 32;
    while (tcols < p.nmma * p.Cmid + p.C) tcols <<= 1;
    const uint32_t d2col = (uint32_t)(p.nmma * p.Cmid);     // D1 partials at columns 0.., D2 right after them

    int tile = blockIdx.x;
    const int tx = tile % p.tiles_x; tile /= p.tiles_x;
    const int ty = tile % p.tiles_y; tile /= p.tiles_y;
    const int gx0 = tx * 8, gy0 = ty * p.BH, n0 = tile * p.BN;

    // barrier init spread over the threads (one thread initialising ~80 barriers cost 0.7 us of every launch)
    if (tid < S) { ptx::mbar_init(full(tid), 1); ptx::mbar_init(empty(tid), (uint32_t)p.nmma); }
    if (tid >= 64 && tid < 64 + hbufs) { ptx::mbar_init(hfull(tid - 64), 1); ptx::mbar_init(hempty(tid - 64), (uint32_t)p.nmma); }
    if (tid == 96) {
        ptx::mbar_init(w2full, 1);
        ptx::mbar_init(d1full, (uint32_t)p.nmma);           // one commit per issuer
        ptx::mbar_init(a2ready, 4);                         // one arrival per epilogue warp
        ptx::mbar_init(d2full, 1);
        ptx::mbar_init(actready, p.staged ? 8u : 4u);       // one arrival per epilogue warp (+ the four helper warps)
    }
    if (tid == 128) { ptx::prefetch_tmap(&tma_in); ptx::prefetch_tmap(&tma_w1); }
    if (tid == 160) { ptx::prefetch_tmap(&tma_w2); ptx::prefetch_tmap(&tma_out); }
    ptx::fence_mbar_init();
    if (warp == 5) ptx::tmem_alloc(sbase + bar_off + RT_MISC, (uint32_t)tcols);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    pdl_launch_dependents();       // the next layer may start its prologue (it blocks in its own pdl_wait)


    // ---- epilogue 2 of the staged layout, columns [c_beg, c_end) of this thread's row: D2 + skip (centre tap of
    // the resident halo tile) -> ReLU -> either back into the halo buffers in place (chained application: same
    // thread, same address; pixels outside the image stay zero = the conv's padding) or into the output tile
    // staged over the dead W1 ring + A2 + W2 (MMA row order, TMA-stored).  Run by the epilogue warps for the
    // first half of the columns and by warps 6-9 (idle issuers) for the second: one warp per scheduler cannot
    // hide its own tcgen05.ld / LDS latencies.
    auto epilogue2_staged = [&](int c_beg, int c_end, bool last) {
        const int q = warp & 3;
        const int row = q * 32 + lane;                      // row = (y * BN + bn) * 8 + x
        const uint32_t lane_taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        const int bw = row & 7, grp = row >> 3;
        const int bn = grp % p.BN, bh = grp / p.BN;
        const bool valid = gx0 + bw < p.W && gy0 + bh < p.H && n0 + bn < p.B;
        const int hrow = ((bh + 1) * p.BN + bn) * RT_WP + bw + 1;      // this pixel's row of a halo buffer
        auto emit = [&](const float (&v)[32], int c0) {
            unsigned char *srow = sm + (c0 >> 5) * halo_stride + hrow * 128;
            unsigned char *orow = sm + ring_off + (c0 >> 5) * RT_A_BYTES + row * 128;
#pragma unroll
            for (int c16 = 0; c16 < 8; ++c16) {
                float4 *ptr = reinterpret_cast<float4 *>(srow + ((c16 ^ (hrow & 7)) << 4));
                const float4 sk = *ptr;
                float4 o = make_float4(v[c16 * 4] + sk.x, v[c16 * 4 + 1] + sk.y, v[c16 * 4 + 2] + sk.z, v[c16 * 4 + 3] + sk.w);
                if (p.relu_out) {
                    o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
                }
                if (last) {
                    *reinterpret_cast<float4 *>(orow + ((c16 ^ (row & 7)) << 4)) = o;
                } else {
                    if (!valid) o = make_float4(0.f, 0.f, 0.f, 0.f);
                    *ptr = o;
                }
            }
        };
        if (c_beg >= c_end) return;
        float va[32], vb[32];                               // two TMEM loads in flight
        ptx::tmem_ld32(lane_taddr + d2col + (uint32_t)c_beg, va);
        for (int c0 = c_beg; c0 < c_end; c0 += 64) {
            ptx::tmem_ld_wait32(va);
            if (c0 + 32 < c_end) ptx::tmem_ld32(lane_taddr + d2col + (uint32_t)(c0 + 32), vb);
            emit(va, c0);
            if (c0 + 32 < c_end) {
                ptx::tmem_ld_wait32(vb);
                if (c0 + 64 < c_end) ptx::tmem_ld32(lane_taddr + d2col + (uint32_t)(c0 + 64), va);
                emit(vb, c0 + 32);
            }
        }
    };
    const int c_split = ((p.C / 32 + 1) / 2) * 32;          // epilogue warps: [0, c_split), helper warps: [c_split, C)

    // Warp roles: 0-3 epilogue (TMEM lane quadrant = warp id), 4 TMA producer, 5 TMEM allocator, 6.. MMA
    // issuers.  GEMM1 has N = Cmid = 32: the tensor pipe needs ~22 cycles per MMA, one issuing warp manages
    // one per ~135 (barrier wait + descriptor arithmetic per k-step are dependent scalar code), so the k-steps
    // are dealt round-robin to up to four issuer warps with private accumulators.
    if (warp == 4 || (warp == 5 && p.nprod == 2)) {
        {
            const int pi = warp - 4, np = p.nprod;
            const bool leader = ptx::elect_one();       // converged warp, one issuing lane
            auto load_halo = [&](int c) {               // input tile + halo of one 32-channel chunk
                const int b = c % hbufs;
                if (c >= hbufs) ptx::mbar_wait(hempty(b), (uint32_t)(((c / hbufs) - 1) & 1));
                if (leader) {
                    ptx::mbar_expect_tx(hfull(b), (uint32_t)halo_bytes);
                    ptx::tma_load_4d(sbase + b * halo_stride, &tma_in, hfull(b), c * 32, gx0 - 1, n0, gy0 - 1);
                }
            };
            // weights do not depend on the previous layer: W2 and the first ring-full of W1 tiles are
            // requested BEFORE pdl_wait(), i.e. while the previous kernel is still draining
            if (leader && pi == 0) {
                ptx::mbar_expect_tx(w2full, (uint32_t)(matoms * p.C * 128));      // W2 (all of it) once
                for (int a = 0; a < matoms; ++a)
                    ptx::tma_load_2d(sbase + w2_off + a * p.C * 128, &tma_w2, w2full, a * 32, 0);
            }
            const int ksteps = 9 * chunks * p.napp;     // the same W1 tiles stream once per application
            const int prefill = S < ksteps ? S : ksteps;
            if (leader)
                for (int i = pi; i < prefill; i += np) {
                    ptx::mbar_expect_tx(bars + 8u * i, (uint32_t)stage_bytes);
                    ptx::tma_load_2d(sbase + ring_off + i * stage_bytes, &tma_w1, bars + 8u * i, ((i / 9) % chunks) * 32, (i % 9) * p.Cmid);
                }
            if (pi == 0) {
                pdl_wait();                             // the input activation is the previous layer's output
                for (int c = 0; c < hbufs; ++c) load_halo(c);
            }
            if (np == 2) {
                // staged mode (no halo reloads): this producer streams the k-steps >= prefill of its parity
                int kidx = prefill + ((pi - prefill) & 1);
                uint32_t st = (uint32_t)(kidx % S), pass = (uint32_t)(kidx / S);
                int t = kidx % 9, c = (kidx / 9) % chunks;
                for (; kidx < ksteps; kidx += 2) {
                    ptx::mbar_wait(empty((int)(st / RT_GROUP)), (pass - 1u) & 1u);      // the group's previous use is released
                    if (leader) {
                        ptx::mbar_expect_tx(full((int)st), (uint32_t)stage_bytes);
                        ptx::tma_load_2d(sbase + ring_off + st * (uint32_t)stage_bytes, &tma_w1, full((int)st), c * 32, t * p.Cmid);
                    }
                    st += 2; if (st >= (uint32_t)S) { st -= (uint32_t)S; ++pass; }
                    t += 2; if (t >= 9) { t -= 9; if (++c == chunks) c = 0; }
                }
            } else {
            // W1 tiles stream through the ring; running pointers, no div/mod in the loop
            uint32_t st = 0, par = 0, full_bar = bars, empty_bar = bars + 8u * RT_MAX_STAGES;
            uint32_t dst = sbase + ring_off;
            int kidx = 0;
            for (int app = 0; app < p.napp; ++app)
            for (int c = 0; c < chunks; ++c) {
                if (c >= 1 && c + 1 < chunks && c + 1 >= hbufs) load_halo(c + 1);
#pragma unroll
                for (int t = 0; t < 9; ++t, ++kidx) {
                    if (kidx >= prefill) {
                        if ((st & (RT_GROUP - 1)) == 0) ptx::mbar_wait(empty_bar, par ^ 1);
                        if (leader) {
                            ptx::mbar_expect_tx(full_bar, (uint32_t)stage_bytes);
                            ptx::tma_load_2d(dst, &tma_w1, full_bar, c * 32, t * p.Cmid);
                        }
                    }
                    ++st; full_bar += 8; dst += (uint32_t)stage_bytes;
                    if ((st & (RT_GROUP - 1)) == 0) empty_bar += 8;
                    if (st == (uint32_t)S) {
                        st = 0; par ^= 1; full_bar = bars; empty_bar = bars + 8u * RT_MAX_STAGES; dst = sbase + ring_off;
                    }
                }
            }
            }
        }
    } else if (warp >= 6) {
        {
            const int mi = warp - 6, nm = p.nmma;
            const bool issuer = mi < nm;
            const bool leader = ptx::elect_one();       // all 32 lanes run the loop; only `leader` issues
            const uint32_t idesc1 = ptx::instr_desc(ptx::FMT_TF32, 128, (uint32_t)p.Cmid);
            const uint32_t idesc2 = ptx::instr_desc(ptx::FMT_TF32, 128, (uint32_t)p.C);
            const uint32_t a_hi = ptx::desc_hi_sw128(RT_WP * 128), b_hi = ptx::desc_hi_sw128(1024);
            const uint32_t rs16 = (uint32_t)(p.BN * RT_WP * 128) >> 4;      // one padded halo row, in 16-byte units
            const uint32_t b_lo0 = (sbase + ring_off) >> 4, b_step = (uint32_t)stage_bytes >> 4;
            const uint32_t dacc = tmem_base + (uint32_t)(mi * p.Cmid);      // this issuer's D1 partial
            // this issuer's k-steps are mi, mi + nm, ...: its ring position advances by nm (S is a multiple of 4)
            uint32_t st = (uint32_t)mi, par = 0;
            int kbase = 0;                              // global index of the current chunk's first k-step
            for (int app = 0; app < p.napp; ++app) {
                const uint32_t ap = (uint32_t)(app & 1);
                uint32_t acc = 0;
                if (app > 0) {
                    // the epilogue has rewritten the activation in place (and drained D1/D2 of the previous application)
                    ptx::mbar_wait(actready, ap ^ 1u);
                    ptx::tc_fence_after();
                }
                for (int c = 0; issuer && c < chunks; ++c, kbase += 9) {
                    const int hb = c % hbufs;
                    ptx::mbar_wait(hfull(hb), (uint32_t)((c / hbufs) & 1));
                    const uint32_t h_lo = (sbase + (uint32_t)(hb * halo_stride)) >> 4;
                    for (int t = (mi - kbase) & (nm - 1); t < 9; t += nm) {
                        ptx::mbar_wait(full((int)st), par);
                        ptx::tc_fence_after();
                        // tap (dy,dx) = (t/3-1, t%3-1): the halo tile read (dy+1) padded rows and (dx+1) pixels
                        // further in; base_offset stays 0 (the swizzle phase comes from the absolute address)
                        const uint32_t t3 = ((uint32_t)t * 11u) >> 5;           // t / 3 for t < 9
                        const uint32_t a_lo = h_lo + t3 * rs16 + ((uint32_t)t - 3u * t3) * 8u;
                        const uint32_t b_lo = b_lo0 + st * b_step;
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            if (leader) ptx::mma_tf32_w(dacc, a_lo + 2u * kk, a_hi, b_lo + 2u * kk, b_hi, idesc1, acc);
                            acc = 1;
                        }
                        // a ring group (RT_GROUP stages) is released by one commit per issuer, after its last stage of the group
                        if ((st & (RT_GROUP - 1)) + (uint32_t)nm >= (uint32_t)RT_GROUP) {
                            if (leader) ptx::tc_commit(empty((int)(st / RT_GROUP)));
                        }
                        st += (uint32_t)nm;
                        if (st >= (uint32_t)S) { st -= (uint32_t)S; par ^= 1; }
                    }
                    if (leader && !p.staged) ptx::tc_commit(hempty(hb));     // chunk done: its halo buffer may be refilled
                    __syncwarp();
                }
                if (leader && issuer) ptx::tc_commit(d1full);    // this issuer's GEMM1 MMAs issued
                if (mi == 0) {
                    // GEMM2 once the epilogue has written relu(D1) as the A2 operand
                    if (app == 0) ptx::mbar_wait(w2full, 0);
                    ptx::mbar_wait(a2ready, ap);
                    ptx::tc_fence_after();
                    for (int a = 0; a < matoms; ++a)
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            if (leader)
                                ptx::mma_tf32(tmem_base + d2col, ptx::smem_desc_sw128(sbase + a2_off + a * RT_A_BYTES + kk * 32),
                                              ptx::smem_desc_sw128(sbase + w2_off + a * p.C * 128 + kk * 32), idesc2,
                                              (a > 0 || kk > 0) ? 1u : 0u);
                    if (leader) ptx::tc_commit(d2full);   // GEMM2 issued
                }
                __syncwarp();
                if (p.staged) {
                    // second half of epilogue 2 (this warp's TMEM lane quadrant is warp % 4)
                    const bool last = app + 1 == p.napp;
                    ptx::mbar_wait_sleep(d2full, ap, 64);
                    ptx::tc_fence_after();
                    epilogue2_staged(c_split, p.C, last);
                    ptx::fence_proxy_async();
                    if (last) {
                        ptx::named_bar_sync(1, 256);             // with the four epilogue warps; tid 0 then stores the tile
                    } else {
                        ptx::tc_fence_before();
                        __syncwarp();
                        if (lane == 0) ptx::mbar_arrive(actready);
                    }
                }
            }
        }
    } else if (warp < 4) {
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t lane_taddr = tmem_base + ((uint32_t)(q * 32) << 16);
        pdl_wait();     // (non-staged path reads the skip tensor from global memory)
        const int bw = row & 7, grp = row >> 3;             // row = (y * BN + bn) * 8 + x
        const int bn = grp % p.BN, bh = grp / p.BN;
        const int gx = gx0 + bw, gy = gy0 + bh, n = n0 + bn;
        const bool valid = gx < p.W && gy < p.H && n < p.B;
        const long long ob = (((long long)n * p.H + gy) * p.W + gx) * p.C;
        const int hrow = ((bh + 1) * p.BN + bn) * RT_WP + bw + 1;      // this pixel's row of a halo buffer
        for (int app = 0; app < p.napp; ++app) {
        const uint32_t ap = (uint32_t)(app & 1);
        const bool last = app + 1 == p.napp;
        // ---- epilogue 1: relu(D1) -> A2 operand in shared memory ----
        ptx::mbar_wait_sleep(d1full, ap);
        ptx::tc_fence_after();
        for (int a = 0; a < matoms; ++a) {
            float v[32];
            if (p.nmma == 4) {                              // all four partials in flight, then one fixed-order sum
                float u1[32], u2[32], u3[32];
                ptx::tmem_ld32(lane_taddr + (uint32_t)(a * 32), v);
                ptx::tmem_ld32(lane_taddr + (uint32_t)(p.Cmid + a * 32), u1);
                ptx::tmem_ld32(lane_taddr + (uint32_t)(2 * p.Cmid + a * 32), u2);
                ptx::tmem_ld32(lane_taddr + (uint32_t)(3 * p.Cmid + a * 32), u3);
                ptx::tmem_ld_wait32(v); ptx::tmem_ld_wait32(u1); ptx::tmem_ld_wait32(u2); ptx::tmem_ld_wait32(u3);
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = __fadd_rn(__fadd_rn(__fadd_rn(v[i], u1[i]), u2[i]), u3[i]);
            } else {
                ptx::tmem_ld32(lane_taddr + (uint32_t)(a * 32), v);
                ptx::tmem_ld_wait32(v);
                for (int m = 1; m < p.nmma; ++m) {              // + the other issuers' partials, fixed order
                    float u[32];
                    ptx::tmem_ld32(lane_taddr + (uint32_t)(m * p.Cmid + a * 32), u);
                    ptx::tmem_ld_wait32(u);
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = __fadd_rn(v[i], u[i]);
                }
            }
            unsigned char *arow = sm + a2_off + a * RT_A_BYTES + row * 128;
#pragma unroll
            for (int c16 = 0; c16 < 8; ++c16) {
                const float4 o = make_float4(fmaxf(v[c16 * 4 + 0], 0.f), fmaxf(v[c16 * 4 + 1], 0.f),
                                             fmaxf(v[c16 * 4 + 2], 0.f), fmaxf(v[c16 * 4 + 3], 0.f));
                *reinterpret_cast<float4 *>(arow + ((c16 ^ (row & 7)) << 4)) = o;
            }
        }
        ptx::fence_proxy_async();       // generic-proxy smem writes -> visible to the tensor core's async proxy
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(a2ready);

        // ---- epilogue 2: D2 + skip -> ReLU -> next application's input / NHWC store ----
        ptx::mbar_wait_sleep(d2full, ap, 64);
        ptx::tc_fence_after();
        if (!last) {
            // chained application (staged mode, whole images per tile): r_{a+1} = act(r_a + D2) replaces r_a
            epilogue2_staged(0, c_split, false);
            ptx::fence_proxy_async();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(actready);
            continue;
        }
        if (p.staged) {
            epilogue2_staged(0, c_split, true);
            ptx::fence_proxy_async();
            ptx::named_bar_sync(1, 256);                       // the four epilogue warps + the four helper warps
            if (tid == 0) {
                for (int a = 0; a < p.C / 32; ++a)               // box {32 ch, 8 px, BN img, BH rows}; OOB rows are clipped
                    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::
                                     "l"(reinterpret_cast<uint64_t>(&tma_out)), "r"(sbase + ring_off + a * RT_A_BYTES),
                                     "r"(a * 32), "r"(gx0), "r"(n0), "r"(gy0) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
        } else
        for (int c0 = 0; c0 < p.C; c0 += 32) {
            float v[32];
            ptx::tmem_ld32(lane_taddr + d2col + (uint32_t)c0, v);
            ptx::tmem_ld_wait32(v);
            if (valid) {
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    const float4 sk = __ldg(reinterpret_cast<const float4 *>(p.skip + ob + c0 + i));
                    float4 o = make_float4(v[i] + sk.x, v[i + 1] + sk.y, v[i + 2] + sk.z, v[i + 3] + sk.w);
                    if (p.relu_out) {
                        o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
                    }
                    *reinterpret_cast<float4 *>(p.out + ob + c0 + i) = o;
                }
            }
        }
        }   // applications
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 5) ptx::tmem_dealloc(tmem_base, (uint32_t)tcols);
}

int rt_pow2_ceil(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

}  // namespace

bool res_tc_supported(int C, int Cmid, const void *r, const void *out) {
    return C % 32 == 0 && C >= 32 && C <= 256 && Cmid % 32 == 0 && Cmid >= 32 && Cmid <= 128 &&
           (reinterpret_cast<uintptr_t>(r) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
}

// w1_tc: [9][Cmid][C], w2_tc: [1][C][Cmid]  (the K-major halves of vqb_pack_conv_weight_f32)
// napp > 1 chains that many applications of the layer in one launch; it needs tiles that hold whole images
// (W <= 8, H <= 16) and the staged shared-memory layout, else VQB_ERR_UNSUPPORTED (the caller then launches
// the applications one by one).
int launch_res_tc(const float *r, const float *w1_tc, const float *w2_tc, float *out, int B, int H, int W, int C,
                  int Cmid, int relu_out, int napp, cudaStream_t s) {
    if (!res_tc_supported(C, Cmid, r, out) || napp < 1) return VQB_ERR_UNSUPPORTED;
    if (napp > 1 && !relu_out) return VQB_ERR_UNSUPPORTED;      // a chained layer input must be relu(x)
    ResTcParams q;
    q.napp = napp;
    q.nmma = 4;
    while (q.nmma > 1 && q.nmma * Cmid + C > 512) q.nmma >>= 1;      // TMEM columns: nmma D1 partials + D2
    // the k-steps of every application must deal out the same way (fused == separate launches, bit for bit)
    while (q.nmma > 1 && (9 * (C / 32)) % q.nmma != 0) q.nmma >>= 1;
    q.skip = r; q.out = out; q.B = B; q.H = H; q.W = W; q.C = C; q.Cmid = Cmid; q.relu_out = relu_out;
    q.BH = rt_pow2_ceil(H) < 16 ? rt_pow2_ceil(H) : 16;
    q.BN = 16 / q.BH;
    q.tiles_x = (W + 7) / 8;
    q.tiles_y = (H + q.BH - 1) / q.BH;
    const int tiles_n = (B + q.BN - 1) / q.BN;

    const int RT_WP = VQB_HALO_WP;
    q.WP = RT_WP;
    CUtensorMap tin, tw1, tw2, tout;
    // dims ordered (c, w, n, h): the BN images of a tile interleave row by row in shared memory
    const uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)B, (uint64_t)H};
    const uint64_t strides[3] = {(uint64_t)C * 4, (uint64_t)H * W * C * 4, (uint64_t)W * C * 4};
    const uint32_t box[4] = {32u, (uint32_t)RT_WP, (uint32_t)q.BN, (uint32_t)(q.BH + 2)};
    const uint32_t es[4] = {1u, 1u, 1u, 1u};
    int rc = vqb_encode_tmap_4d(&tin, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, r, dims, strides, box, es,
                                CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    {
        const uint32_t obox[4] = {32u, 8u, (uint32_t)q.BN, (uint32_t)q.BH};
        rc = vqb_encode_tmap_4d(&tout, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, out, dims, strides, obox, es,
                                CU_TENSOR_MAP_SWIZZLE_128B);
        if (rc) return rc;
    }
    rc = vqb_encode_tmap_2d(&tw1, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w1_tc, (uint64_t)C, (uint64_t)9 * Cmid,
                            (uint64_t)C * 4, 32, (uint32_t)Cmid, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = vqb_encode_tmap_2d(&tw2, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, w2_tc, (uint64_t)Cmid, (uint64_t)C,
                            (uint64_t)Cmid * 4, 32, (uint32_t)C, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;

    const int stage_bytes = Cmid * 128;
    const int chunks = C / 32;
    const int halo_b = (((q.BH + 2) * q.BN * RT_WP * 128) + 1023) & ~1023;
    const int tail = (Cmid / 32) * RT_A_BYTES + (Cmid / 32) * C * 128;            // A2 + W2
    const int misc = 8 * (2 * RT_MAX_STAGES + 4 + 2 * RT_MAX_CHUNKS + 2) + 16 + 1024;
    // staged mode: every halo chunk resident + a ring that, together with A2 + W2, holds the 128 x C output tile
    int stages = 0;
    q.staged = 0;
    {
        int need = 128 * C * 4 - tail;                       // ring bytes needed for the output staging
        int st = (need + stage_bytes - 1) / stage_bytes;
        if (st < RT_GROUP) st = RT_GROUP;
        st = (st + RT_GROUP - 1) / RT_GROUP * RT_GROUP;
        // ... and as deep as shared memory allows beyond that: the W1 tiles in flight (stages x Cmid x 128 B)
        // over the L2 latency are what feeds GEMM1 (8 stages = 32 KB kept the tensor pipe 14 % busy)
        int fit = (227 * 1024 - (chunks * halo_b + tail + misc)) / stage_bytes;
        if (fit > RT_MAX_STAGES) fit = RT_MAX_STAGES;
        fit -= fit % RT_GROUP;
        if (st <= fit && chunks <= RT_MAX_CHUNKS) {
            q.staged = 1;
            const int all = (9 * chunks * napp + RT_GROUP - 1) / RT_GROUP * RT_GROUP;
            stages = fit < all ? fit : (all > st ? all : st);
        }
    }
    if (napp > 1 && !(q.staged && q.tiles_x == 1 && q.tiles_y == 1)) return VQB_ERR_UNSUPPORTED;
    const int hbufs = q.staged ? chunks : (chunks < RT_HALO_BUFS ? chunks : RT_HALO_BUFS);
    const int fixed = hbufs * halo_b + tail + misc;
    if (!q.staged) {
        stages = (226 * 1024 - fixed) / stage_bytes;
        if (stages > RT_MAX_STAGES) stages = RT_MAX_STAGES;
        if (stages >= 9 * chunks) stages = 9 * chunks;
        else stages -= stages % RT_GROUP;             // a reused ring must hold whole commit groups
        if (stages < RT_GROUP) return VQB_ERR_UNSUPPORTED;
    }
    q.stages = stages;
    q.nprod = (q.staged && stages % 2 == 0) ? 2 : 1;
    const int smem = stages * stage_bytes + fixed;
    static int attr_max = 0;
    if (smem > attr_max) {
        cudaError_t e = cudaFuncSetAttribute(res_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr_max = smem;
    }
    const long long grid = (long long)q.tiles_x * q.tiles_y * tiles_n;
    if (grid <= 0 || grid > 0x7fffffffLL) return VQB_ERR_UNSUPPORTED;
    if (cudaError_t le = vqb_launch(res_tc_kernel, dim3((unsigned)grid), dim3(RT_THREADS), (size_t)smem, s, tin, tw1, tw2, tout, q)) return (int)le;
    VQB_COUNT_LAUNCH(1);
    return vqb_cuda_status(cudaGetLastError());
}
