// vq2.cu -- fused VectorQuantizer.forward on tcgen05 (sm_100a), D = 64, K <= 8192.
//
// Replaces quantizer.py:45-71.  Contract: idx / z_q are bit-identical to vq_exact.cu and to the oracle.  The TF32
// scores s_k = ||e_k||^2 - 2 z.e_k only SELECT; tau bounds twice the worst-case error of a score (tf32 truncation of
// both operands, fp32 accumulation and the rounding of the canonical formula), so every code whose canonical fp32
// distance could be the minimum -- the winner and all its ties -- has s_k <= min_k s_k + tau; codes inside that
// window are re-scored with the canonical chain of oracle/csrc/oracle.c (sequential fmaf over d,
// fl(fl(A+B) - fl(2M)), first minimum wins, NaN wins).
//
// Design (against the round-1 kernel, profiles/r01_vq_tc_epilogue_timeline.txt: 8.7 us per 128-row tile against a
// 1.5 us HBM budget, all phases serial, every row re-scoring 8-16 codes although 82-86 % of the rows have ONE code
// inside the window):
//   * the sweep over the scores only takes MINIMA, over several partitions of a thread's codes at once: P1 = the
//     column's residue mod 16 (16 running minima), P2 = its 16-column block inside the chunk pair (16 minima, reduced
//     by a min3 tree as the block passes), and for streamed codebooks P3 / P4 = the chunk pair mod 8 / div 8.  That is
//     one 3-input FMNMX per score (plus the FFMA that forms the score) -- no index packing, no second minima, no
//     lists, no branches (profiles/r02_vq2_profile_notes.txt: the first version's 4.5 ALU-pipe instructions per score
//     were the kernel's bound);
//   * after the sweep the window {s_k <= min + tau} is covered exactly by a GRID: a code inside the window pulls the
//     minimum of every class it belongs to under the threshold, so window is a subset of R x B x C x Q with R, B, C, Q
//     the classes whose minimum is inside the window.  One grid point -> it is the canonical argmin, NO exact
//     arithmetic at all (82-86 % of the rows); a few -> those codes are re-scored with the canonical chain (grid points
//     outside the window are harmless: the exact distance decides); a big grid, non-finite data or overflow -> the row
//     is queued and all finish threads scan the whole codebook for it together;
//   * sweep (8 warps, TMEM readers) and finish (4 warps: decision, exact chains, gather, z_q = z + (e - z), SSE,
//     histogram, idx) are different warps and work on different tiles at the same time; the TMA producer / MMA issuer
//     run ahead of both.  16 warps per CTA, one CTA per SM, persistent.
//   * z_q can leave as fp32 rows (module contract) or as bf16 rows (the bf16 decoder reads them; VQVAE.forward never
//     returns z_q).
#include <cuda_bf16.h>

#include <cstdlib>

#include "common.cuh"
#include "ptx.cuh"

#if VQB_DIAG
// in-kernel timeline of CTA 0 (SM cycle counter), tools/diag/vq2_timeline.py; diagnostic builds only
__device__ unsigned long long g_vq2_tl[32 * 32];
extern "C" int vqb_debug_read_vq2_timeline(unsigned long long *dst, int n) {
    if (!dst || n < 1 || n > 32 * 32) return VQB_ERR_BAD_ARG;
    return vqb_cuda_status(cudaMemcpyFromSymbol(dst, g_vq2_tl, sizeof(unsigned long long) * n));
}
#define VQ2_TL(it_, ev_)                                                                      \
    do {                                                                                      \
        if (blockIdx.x == 0 && (it_) >= 0 && (it_) < 32) {                                    \
            unsigned long long t_;                                                            \
            asm volatile("mov.u64 %0, %%clock64;" : "=l"(t_));                                \
            g_vq2_tl[(it_) * 32 + (ev_)] = t_;                                                \
        }                                                                                     \
    } while (0)
#else
#define VQ2_TL(it_, ev_) do { } while (0)
#endif

namespace {

constexpr int TM = 128;          // latent rows per tile (UMMA M)
constexpr int CN = 256;          // codes per chunk (UMMA N)
constexpr int DD = 64;
constexpr int NT2 = 512;         // 16 warps
constexpr int NTRK = 16;         // minima per partition and thread
constexpr int GCAP = 24;         // grid points a half row can hand over; more -> whole-codebook scan
constexpr int ZSTAGE = TM * DD * 4, ZATOM = TM * 128;
constexpr int ESTAGE = CN * DD * 4, EATOM = CN * 128;
constexpr int HIST_MAX = 1024;

constexpr int OFF_Z = 0;
constexpr int OFF_E = OFF_Z + 2 * ZSTAGE;
constexpr int OFF_B = OFF_E + 2 * ESTAGE;                    // float[2 * CN]
constexpr int OFF_CAND = OFF_B + 2 * CN * 4;                 // 2 tiles x 256 half rows x int4 (grid size or -1, R | B << 16, C | Q << 8, 0)
constexpr int OFF_XCH = OFF_CAND + 2 * 256 * 16;             // float2[256]: (half-row min, partial ||z||^2)
constexpr int PCAP = 512;                                    // (row, code) pairs re-scored per tile (typically 100-250); one list per tile parity:
                                                             // a warp may push tile t+1's pairs while another still reads tile t's distances
constexpr int OFF_Q = OFF_XCH + 256 * 8;                     // per tile parity: int[136] = full-scan queue (count + rows) + pair count
constexpr int OFF_QR = OFF_Q + 2 * 136 * 4;                  // per finish warp (d, k) partials: 4 x (float,int) x 8 slots
constexpr int OFF_PAIR = OFF_QR + 4 * 8 * 8;                 // pairs: int2 (row, k)[PCAP] then float dist[PCAP]
constexpr int OFF_HIST = OFF_PAIR + 2 * PCAP * 12;
constexpr int OFF_BAR = OFF_HIST + HIST_MAX * 4;
constexpr int OFF_TMEM = OFF_BAR + 24 * 8;
constexpr int OFF_RED = OFF_TMEM + 64;
constexpr int SMEM_TOTAL = OFF_RED + 64;
constexpr int SMEM_ALLOC = SMEM_TOTAL + 1024;
static_assert(SMEM_ALLOC <= 227 * 1024, "shared memory budget");

enum { Z_FULL = 0, Q_DONE = 2, E_FULL = 4, E_EMPTY = 6, T_FULL = 8, T_EMPTY = 10, C_FULL = 12, C_EMPTY = 14 };

struct Vq2Params {
    const float *E;        // (K, 64) codebook
    const float *bn;       // (nchunks*256) canonical ||e_k||^2, +inf past K (streamed codebooks)
    const float *scal;     // [0] = upper bound of max ||e_k||, [1] = non-finite flag (streamed codebooks)
    long long N;
    int K, nchunks, nbits;
    long long *idx;
    double *partials;
    unsigned *pending;
    int *hist;
    int zq_bf16;
    void *zq;              // (N, 64) fp32 or bf16 rows
};

__device__ __forceinline__ bool vq2_better(float dn, int kn, float db, int kb) {
    const bool nn = dn != dn, nb = db != db;            // torch.argmin: NaN is the minimum
    if (nn || nb) return nn && (!nb || kn < kb);
    return dn < db || (dn == db && kn < kb);
}
template <bool RESIDENT, bool ZQBF>
__global__ void __launch_bounds__(NT2, 1)
vq2_kernel(const __grid_constant__ CUtensorMap tmz, const __grid_constant__ CUtensorMap tme,
           const Vq2Params p) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = ptx::smem_u32(smem_raw);
    const uint32_t sbase = (raw + 1023u) & ~1023u;
    unsigned char *sm = smem_raw + (sbase - raw);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t bars = sbase + OFF_BAR;
    auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };
    float *bsm = reinterpret_cast<float *>(sm + OFF_B);
    int *hist_s = reinterpret_cast<int *>(sm + OFF_HIST);
    int *cand = reinterpret_cast<int *>(sm + OFF_CAND);
    float2 *xch = reinterpret_cast<float2 *>(sm + OFF_XCH);
    volatile int *fq_all = reinterpret_cast<volatile int *>(sm + OFF_Q);
    volatile uint32_t *tmem_holder = reinterpret_cast<volatile uint32_t *>(sm + OFF_TMEM);

    const long long ntiles = (p.N + TM - 1) / TM;
    const int nchunks = p.nchunks;
    constexpr bool resident = RESIDENT;           // the whole codebook (<= 2 chunks) stays in shared memory
    const bool smem_hist = p.K <= HIST_MAX;
    const float INF = __int_as_float(0x7f800000);

    if (tid == 0) {
        ptx::prefetch_tmap(&tmz); ptx::prefetch_tmap(&tme);
        for (int s = 0; s < 2; ++s) {
            ptx::mbar_init(bar(Z_FULL + s), 1);
            ptx::mbar_init(bar(Q_DONE + s), 4);       // 4 finish warps
            ptx::mbar_init(bar(E_FULL + s), 1);
            ptx::mbar_init(bar(E_EMPTY + s), 9);      // MMA commit + 8 sweep warps
            ptx::mbar_init(bar(T_FULL + s), 1);
            ptx::mbar_init(bar(T_EMPTY + s), 8);
            ptx::mbar_init(bar(C_FULL + s), 8);
            ptx::mbar_init(bar(C_EMPTY + s), 4);
        }
        ptx::fence_mbar_init();
    }
    if (smem_hist)
        for (int k = tid; k < p.K; k += NT2) hist_s[k] = 0;
    if (tid == 0) { fq_all[0] = 0; fq_all[135] = 0; fq_all[136] = 0; fq_all[136 + 135] = 0; }
    if (warp == 2) ptx::tmem_alloc(sbase + OFF_TMEM, 512);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    pdl_launch_dependents();
    pdl_wait();                    // z_e is written by the previous layer

    auto code_ptr_smem = [&](int k) -> const unsigned char * { return sm + OFF_E + (k >> 8) * ESTAGE + (k & 255) * 128; };

    if (warp == 0) {
        // ===================== TMA producer (+ z_q tile stores) =====================
        if (lane == 0) {
            long long gc = 0;
            int it = 0;
            long long tile = blockIdx.x;
            for (; tile < ntiles; tile += gridDim.x, ++it) {
                const int zs = it & 1;
                if (it >= 2) {                   // the finish warps have emitted tile it-2 from this stage
                    ptx::mbar_wait_sleep(bar(Q_DONE + zs), (uint32_t)(((it - 2) >> 1) & 1), 32);
                    VQ2_TL(it - 2, 1);
                }
                VQ2_TL(it, 0);
                ptx::mbar_expect_tx(bar(Z_FULL + zs), ZSTAGE);
                const uint32_t zdst = sbase + OFF_Z + zs * ZSTAGE;
                ptx::tma_load_2d(zdst, &tmz, bar(Z_FULL + zs), 0, (int)(tile * TM));
                ptx::tma_load_2d(zdst + ZATOM, &tmz, bar(Z_FULL + zs), 32, (int)(tile * TM));
                if (resident && it > 0) continue;
                for (int c = 0; c < nchunks; ++c, ++gc) {
                    const int es = resident ? c : (int)(gc & 1);
                    const uint32_t par = resident ? 0u : (uint32_t)((gc >> 1) & 1);
                    ptx::mbar_wait(bar(E_EMPTY + es), par ^ 1);
                    ptx::mbar_expect_tx(bar(E_FULL + es), resident ? ESTAGE : ESTAGE + CN * 4);
                    const uint32_t edst = sbase + OFF_E + es * ESTAGE;
                    ptx::tma_load_2d(edst, &tme, bar(E_FULL + es), 0, c * CN);
                    ptx::tma_load_2d(edst + EATOM, &tme, bar(E_FULL + es), 32, c * CN);
                    if (!resident)
                        ptx::bulk_load_1d(sbase + OFF_B + es * CN * 4, p.bn + (size_t)c * CN, CN * 4, bar(E_FULL + es));
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (converged warp, elected leader lane issues) =====================
        const bool leader = ptx::elect_one();
        constexpr uint32_t idesc = ptx::instr_desc(ptx::FMT_TF32, TM, CN);
        const uint32_t d_hi = ptx::desc_hi_sw128(1024);
        int it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int zs = it & 1;
            ptx::mbar_wait(bar(Z_FULL + zs), (it >> 1) & 1);
            if (leader) VQ2_TL(it, 3);
            const uint32_t za_lo = (sbase + OFF_Z + zs * ZSTAGE) >> 4;
            for (int c = 0; c < nchunks; ++c) {
                const long long gc = (long long)it * nchunks + c;
                int es;
                if (resident) {
                    es = c;
                    if (it == 0) ptx::mbar_wait(bar(E_FULL + es), 0);
                } else {
                    es = (int)(gc & 1);
                    ptx::mbar_wait(bar(E_FULL + es), (uint32_t)((gc >> 1) & 1));
                }
                const int ab = (int)(gc & 1);
                ptx::mbar_wait(bar(T_EMPTY + ab), (uint32_t)(((gc >> 1) & 1) ^ 1));
                ptx::tc_fence_after();
                if (leader && c < 2) VQ2_TL(it, 4 + 2 * c);
                const uint32_t ea_lo = (sbase + OFF_E + es * ESTAGE) >> 4;
#pragma unroll
                for (int ks = 0; ks < DD / 8; ++ks)
                    if (leader)
                        ptx::mma_tf32_w(tmem_base + ab * CN, za_lo + (ks >> 2) * (ZATOM >> 4) + (ks & 3) * 2, d_hi,
                                        ea_lo + (ks >> 2) * (EATOM >> 4) + (ks & 3) * 2, d_hi, idesc, ks > 0 ? 1u : 0u);
                if (leader) {
                    if (c < 2) VQ2_TL(it, 5 + 2 * c);
                    ptx::tc_commit(bar(T_FULL + ab));
                    if (!resident) ptx::tc_commit(bar(E_EMPTY + es));
                }
                __syncwarp();
            }
        }
    } else if (warp >= 4 && warp < 12) {
        // ===================== sweep warps: thread = (row, column half) =====================
        const int et = tid - 128;               // 0..255
        const int q = warp & 3;                 // TMEM lane quadrant
        const int h = (warp - 4) >> 2;          // column half of every chunk
        const int row = q * 32 + lane;
        const int rsw = row & 7;
        float Emax;
        bool bad_codebook;
        if (resident) {
            // canonical ||e_k||^2 (quantizer.py:50), their maximum and a non-finite flag from the resident copy
            float mymax = 0.f;
            unsigned mybad = 0u;
            for (int c = 0; c < nchunks; ++c) ptx::mbar_wait(bar(E_FULL + c), 0);
            for (int k = et; k < nchunks * CN; k += 256) {
                float sn = INF;
                if (k < p.K) {
                    const unsigned char *er = sm + OFF_E + (k >> 8) * ESTAGE + (k & 255) * 128;
                    sn = 0.f;
#pragma unroll
                    for (int a = 0; a < 2; ++a)
#pragma unroll
                        for (int c16 = 0; c16 < 8; ++c16) {
                            const float4 v = *reinterpret_cast<const float4 *>(er + a * EATOM + ((c16 ^ (k & 7)) << 4));
                            sn = __fadd_rn(sn, __fmul_rn(v.x, v.x)); sn = __fadd_rn(sn, __fmul_rn(v.y, v.y));
                            sn = __fadd_rn(sn, __fmul_rn(v.z, v.z)); sn = __fadd_rn(sn, __fmul_rn(v.w, v.w));
                        }
                    if (!(sn < INF)) mybad = 1u;
                    else mymax = fmaxf(mymax, sqrtf(sn) * 1.00001f);
                }
                bsm[k] = sn;
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                mymax = fmaxf(mymax, __shfl_xor_sync(0xffffffffu, mymax, off));
                mybad |= __shfl_xor_sync(0xffffffffu, mybad, off);
            }
            if (lane == 0) xch[warp - 4] = make_float2(mymax, __uint_as_float(mybad));
            ptx::named_bar_sync(5, 256);
            float mx = 0.f;
            unsigned bad = 0u;
            for (int w = 0; w < 8; ++w) { mx = fmaxf(mx, xch[w].x); bad |= __float_as_uint(xch[w].y); }
            ptx::named_bar_sync(5, 256);
            Emax = mx;
            bad_codebook = bad != 0u;
        } else {
            Emax = __uint_as_float(reinterpret_cast<const unsigned *>(p.scal)[0]);
            bad_codebook = reinterpret_cast<const unsigned *>(p.scal)[1] != 0u;
        }
        const uint32_t lane_taddr = tmem_base + ((uint32_t)(q * 32) << 16);

        int it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int zs = it & 1;
            const unsigned char *zrow = sm + OFF_Z + zs * ZSTAGE + row * 128;
            ptx::mbar_wait_sleep(bar(Z_FULL + zs), (it >> 1) & 1, 100);
            if (tid == 128) VQ2_TL(it, 8);
            // this thread's half of ||z||^2 (any order: it only feeds the error bound tau)
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
            for (int c16 = 0; c16 < 8; ++c16) {
                const float4 v = *reinterpret_cast<const float4 *>(zrow + h * ZATOM + ((c16 ^ rsw) << 4));
                a0 = fmaf(v.x, v.x, a0); a1 = fmaf(v.y, v.y, a1); a2 = fmaf(v.z, v.z, a2); a3 = fmaf(v.w, v.w, a3);
            }
            const float Apart = (a0 + a1) + (a2 + a3);

            // running minima of the partitions (header): m1 residue mod 16, mb block of the chunk pair, mc / m4 chunk pair
            float m1[NTRK], mb[NTRK], mc[8], m4[2];
#pragma unroll
            for (int i = 0; i < NTRK; ++i) { m1[i] = INF; mb[i] = INF; }
#pragma unroll
            for (int i = 0; i < 8; ++i) mc[i] = INF;
            m4[0] = INF; m4[1] = INF;
            float cur = INF;                                          // minimum of the current chunk pair (streamed codebooks)

            for (int c0 = 0; c0 < nchunks; c0 += 2) {
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) {
                    const int c = c0 + cc;
                    if (c < nchunks) {
                        const long long gc = (long long)it * nchunks + c;
                        const int ab = (int)(gc & 1);
                        const int es = resident ? c : (int)(gc & 1);
                        ptx::mbar_wait_sleep(bar(T_FULL + ab), (uint32_t)((gc >> 1) & 1), 64);
                        ptx::tc_fence_after();
                        if (tid == 128 && c < 2) VQ2_TL(it, 9 + 2 * c);
                        const float *bch = bsm + es * CN + h * 128;
                        const uint32_t tcol = lane_taddr + (uint32_t)(ab * CN + h * 128);
                        float va[32], vb[32];
                        auto process = [&](const float (&v)[32], const int j) {
                            float sc[32];
#pragma unroll
                            for (int i = 0; i < 8; ++i) {                 // ||e_k||^2 of the 32 columns (broadcast 16-byte loads)
                                const float4 b4 = *reinterpret_cast<const float4 *>(bch + j * 32 + 4 * i);
                                sc[4 * i] = fmaf(v[4 * i], -2.f, b4.x); sc[4 * i + 1] = fmaf(v[4 * i + 1], -2.f, b4.y);
                                sc[4 * i + 2] = fmaf(v[4 * i + 2], -2.f, b4.z); sc[4 * i + 3] = fmaf(v[4 * i + 3], -2.f, b4.w);
                            }
#pragma unroll
                            for (int i = 0; i < NTRK; ++i) m1[i] = ptx::fmin3(m1[i], sc[i], sc[i + 16]);
#pragma unroll
                            for (int u = 0; u < 2; ++u) {                 // the two 16-column blocks of this load
                                const float *b = sc + 16 * u;
                                float &acc = mb[cc * 8 + j * 2 + u];
                                const float t1 = ptx::fmin3(b[2], b[3], b[4]), t2 = ptx::fmin3(b[5], b[6], b[7]);
                                const float t3 = ptx::fmin3(b[8], b[9], b[10]), t4 = ptx::fmin3(b[11], b[12], b[13]);
                                const float t6 = ptx::fmin3(t1, t2, t3);
                                if (resident) {
                                    const float t0 = ptx::fmin3(acc, b[0], b[1]);
                                    const float t5 = ptx::fmin3(b[14], b[15], t0);
                                    acc = ptx::fmin3(t4, t5, t6);
                                } else {
                                    const float t0 = ptx::fmin3(b[0], b[1], b[14]);
                                    const float t5 = ptx::fmin3(b[15], t0, t4);
                                    const float blk = fminf(t5, t6);
                                    acc = fminf(acc, blk);
                                    cur = fminf(cur, blk);
                                }
                            }
                        };
                        ptx::tmem_ld32(tcol, va);
                        ptx::tmem_ld_wait32(va);
                        ptx::tmem_ld32(tcol + 32, vb);
                        process(va, 0);
                        ptx::tmem_ld_wait32(vb);
                        ptx::tmem_ld32(tcol + 64, va);
                        process(vb, 1);
                        ptx::tmem_ld_wait32(va);
                        ptx::tmem_ld32(tcol + 96, vb);
                        process(va, 2);
                        ptx::tmem_ld_wait32(vb);
                        process(vb, 3);
                        ptx::tc_fence_before();
                        __syncwarp();
                        if (tid == 128 && c < 2) VQ2_TL(it, 10 + 2 * c);
                        if (tid == 352 && c < 2) VQ2_TL(it, 16 + c);
                        if (lane == 0) {
                            ptx::mbar_arrive(bar(T_EMPTY + ab));
                            if (!resident) ptx::mbar_arrive(bar(E_EMPTY + es));
                        }
                    }
                }
                if (!resident) {                                       // close the chunk pair
                    const int cp = c0 >> 1;
#pragma unroll
                    for (int i = 0; i < 8; ++i) if (i == (cp & 7)) mc[i] = fminf(mc[i], cur);
#pragma unroll
                    for (int i = 0; i < 2; ++i) if (i == (cp >> 3)) m4[i] = fminf(m4[i], cur);
                    cur = INF;
                }
            }

            // ---- half-row minimum, exchange with the partner thread (same row, other column half) ----
            float hmin;
            {
                const float t0 = ptx::fmin3(m1[0], m1[1], m1[2]), t1 = ptx::fmin3(m1[3], m1[4], m1[5]), t2 = ptx::fmin3(m1[6], m1[7], m1[8]);
                const float t3 = ptx::fmin3(m1[9], m1[10], m1[11]), t4 = ptx::fmin3(m1[12], m1[13], m1[14]);
                hmin = fminf(ptx::fmin3(t0, t1, t2), ptx::fmin3(t3, t4, m1[15]));
            }
            xch[et] = make_float2(hmin, Apart);
            ptx::named_bar_sync(1 + q, 64);
            const float2 px = xch[et ^ 128];
            const float rowmin = fminf(hmin, px.x);
            const float A = Apart + px.y;
            // S >= sum_d |z_d e_kd| for every k (Cauchy-Schwarz, rounded up); tau = 2 x (tf32 truncation of both
            // operands on 2M: 2*2^-9*S, fp32 accumulation + the canonical formula's own rounding), with margin.
            const float S = sqrtf(A) * 1.00002f * Emax;
            const float tau = S * (0.0078125f + 0.0009765625f) + (A + Emax * Emax + S) * 1.9073486e-6f + 1e-30f;
            const bool slow_row = bad_codebook || !(A < INF) || !(tau < INF) || !(rowmin == rowmin);
            const float thr = rowmin + tau;
            ptx::named_bar_sync(1 + q, 64);               // xch is reused by the next tile
            if (tid == 128) VQ2_TL(it, 13);

            // ---- this half's grid: the classes of every partition whose minimum is inside the window ----
            unsigned R = 0u, Bm = 0u, Cm = 1u, Qm = 1u;
#pragma unroll
            for (int i = 0; i < NTRK; ++i) {
                R |= m1[i] <= thr ? (1u << i) : 0u;
                Bm |= mb[i] <= thr ? (1u << i) : 0u;
            }
            if (!resident) {
                Cm = 0u; Qm = 0u;
#pragma unroll
                for (int i = 0; i < 8; ++i) Cm |= mc[i] <= thr ? (1u << i) : 0u;
                Qm = (m4[0] <= thr ? 1u : 0u) | (m4[1] <= thr ? 2u : 0u);
            }
            const int n = __popc(R) * __popc(Bm) * __popc(Cm) * __popc(Qm);
            const bool needfull = slow_row || n > GCAP;
            const int par = it & 1;
            ptx::mbar_wait_sleep(bar(C_EMPTY + par), (uint32_t)(((it >> 1) & 1) ^ 1), 100);       // finish warps are done with tile it-2's records
            if (tid == 128) VQ2_TL(it, 14);
            *reinterpret_cast<int4 *>(cand + (par * 256 + et) * 4) = make_int4(needfull ? -1 : n, (int)(R | (Bm << 16)), (int)(Cm | (Qm << 8)), 0);
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(bar(C_FULL + par));
            if (tid == 128) VQ2_TL(it, 15);
        }
    } else if (warp >= 12) {
        // ===================== finish warps: thread = row =====================
        const int ft = tid - 384;               // 0..127 = row of the tile
        const int row = ft;
        double sse = 0.0;
        float *qr = reinterpret_cast<float *>(sm + OFF_QR);
        int2 *prk_all = reinterpret_cast<int2 *>(sm + OFF_PAIR);
        float *pdist_all = reinterpret_cast<float *>(sm + OFF_PAIR + 2 * PCAP * 8);
        for (int i = ft; i < 2 * PCAP; i += 128) prk_all[i] = make_int2(0, -1);      // slots a list overflow leaves unwritten must stay harmless
        ptx::named_bar_sync(6, 128);
        // canonical distance of code k to the z row at `zr_s` (shared memory, swizzled): A = sum fl(z^2) left to right,
        // M = one sequential fmaf chain, d = fl(fl(A + B_k) - fl(2 M))   (quantizer.py:49-51, oracle.c)
        auto exact_dist = [&](const unsigned char *zr_s, int zsw, int k) -> float {
            float A = 0.f, M = 0.f;
            const unsigned char *es = code_ptr_smem(k);
            const float4 *eg = reinterpret_cast<const float4 *>(p.E + (size_t)k * DD);
#pragma unroll
            for (int c16 = 0; c16 < 16; ++c16) {
                const float4 v = *reinterpret_cast<const float4 *>(zr_s + (c16 >> 3) * ZATOM + (((c16 & 7) ^ zsw) << 4));
                const float4 e = resident ? *reinterpret_cast<const float4 *>(es + (c16 >> 3) * EATOM + (((c16 & 7) ^ (k & 7)) << 4)) : __ldg(eg + c16);
                A = __fadd_rn(A, __fmul_rn(v.x, v.x)); A = __fadd_rn(A, __fmul_rn(v.y, v.y));
                A = __fadd_rn(A, __fmul_rn(v.z, v.z)); A = __fadd_rn(A, __fmul_rn(v.w, v.w));
                M = __fmaf_rn(v.x, e.x, M); M = __fmaf_rn(v.y, e.y, M); M = __fmaf_rn(v.z, e.z, M); M = __fmaf_rn(v.w, e.w, M);
            }
            const float bnk = resident ? bsm[k] : __ldg(p.bn + k);
            return __fsub_rn(__fadd_rn(A, bnk), __fmul_rn(2.0f, M));
        };
        auto exact_dist2 = [&](const unsigned char *za, int zswa, int ka, const unsigned char *zb, int zswb, int kb, float &da, float &db) {
            float Aa = 0.f, Ma = 0.f, Ab = 0.f, Mb = 0.f;
            const unsigned char *esa = code_ptr_smem(ka), *esb = code_ptr_smem(kb);
            const float4 *ega = reinterpret_cast<const float4 *>(p.E + (size_t)ka * DD), *egb = reinterpret_cast<const float4 *>(p.E + (size_t)kb * DD);
#pragma unroll
            for (int c16 = 0; c16 < 16; ++c16) {
                const float4 va = *reinterpret_cast<const float4 *>(za + (c16 >> 3) * ZATOM + (((c16 & 7) ^ zswa) << 4));
                const float4 vb = *reinterpret_cast<const float4 *>(zb + (c16 >> 3) * ZATOM + (((c16 & 7) ^ zswb) << 4));
                const float4 ea = resident ? *reinterpret_cast<const float4 *>(esa + (c16 >> 3) * EATOM + (((c16 & 7) ^ (ka & 7)) << 4)) : __ldg(ega + c16);
                const float4 eb = resident ? *reinterpret_cast<const float4 *>(esb + (c16 >> 3) * EATOM + (((c16 & 7) ^ (kb & 7)) << 4)) : __ldg(egb + c16);
                Aa = __fadd_rn(Aa, __fmul_rn(va.x, va.x)); Ab = __fadd_rn(Ab, __fmul_rn(vb.x, vb.x));
                Aa = __fadd_rn(Aa, __fmul_rn(va.y, va.y)); Ab = __fadd_rn(Ab, __fmul_rn(vb.y, vb.y));
                Aa = __fadd_rn(Aa, __fmul_rn(va.z, va.z)); Ab = __fadd_rn(Ab, __fmul_rn(vb.z, vb.z));
                Aa = __fadd_rn(Aa, __fmul_rn(va.w, va.w)); Ab = __fadd_rn(Ab, __fmul_rn(vb.w, vb.w));
                Ma = __fmaf_rn(va.x, ea.x, Ma); Mb = __fmaf_rn(vb.x, eb.x, Mb);
                Ma = __fmaf_rn(va.y, ea.y, Ma); Mb = __fmaf_rn(vb.y, eb.y, Mb);
                Ma = __fmaf_rn(va.z, ea.z, Ma); Mb = __fmaf_rn(vb.z, eb.z, Mb);
                Ma = __fmaf_rn(va.w, ea.w, Ma); Mb = __fmaf_rn(vb.w, eb.w, Mb);
            }
            const float bna = resident ? bsm[ka] : __ldg(p.bn + ka), bnb = resident ? bsm[kb] : __ldg(p.bn + kb);
            da = __fsub_rn(__fadd_rn(Aa, bna), __fmul_rn(2.0f, Ma));
            db = __fsub_rn(__fadd_rn(Ab, bnb), __fmul_rn(2.0f, Mb));
        };
        int it = 0;
        for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
            const int zs = it & 1, par = it & 1;
            volatile int *fq = fq_all + par * 136;                 // [0] queue count, [1..128] queued rows, [135] pair count
            int2 *prk = prk_all + par * PCAP;
            float *pdist = pdist_all + par * PCAP;
            unsigned char *ztile = sm + OFF_Z + zs * ZSTAGE;
            ptx::mbar_wait_sleep(bar(Z_FULL + zs), (it >> 1) & 1, 200);
            ptx::mbar_wait_sleep(bar(C_FULL + par), (uint32_t)((it >> 1) & 1), 32);
            if (ft == 0) VQ2_TL(it, 20);
            const int4 g0 = *reinterpret_cast<const int4 *>(cand + (par * 256 + row) * 4);
            const int4 g1 = *reinterpret_cast<const int4 *>(cand + (par * 256 + 128 + row) * 4);
            const int n0 = g0.x, n1 = g1.x;
            // grid point (i, b, c, q) of column half hh -> code: chunk pair 8 q + c, chunk (b >> 3), 16-column block b & 7, residue i
            auto for_grid = [&](const int4 g, const int hh, auto &&f) {
                for (unsigned qm = ((unsigned)g.z >> 8) & 3u; qm; qm &= qm - 1u)
                    for (unsigned cm = (unsigned)g.z & 0xffu; cm; cm &= cm - 1u)
                        for (unsigned bm = (unsigned)g.y >> 16; bm; bm &= bm - 1u)
                            for (unsigned rm = (unsigned)g.y & 0xffffu; rm; rm &= rm - 1u) {
                                const int qi = __ffs((int)qm) - 1, ci = __ffs((int)cm) - 1, bi = __ffs((int)bm) - 1, ri = __ffs((int)rm) - 1;
                                f(((qi * 8 + ci) * 2 + (bi >> 3)) * CN + hh * 128 + (bi & 7) * 16 + ri);
                            }
            };
            int bk = -1, pbase = -1;
            float bd = 0.f;
            const int ncand = n0 + n1;
            bool queued = n0 < 0 || n1 < 0;
            if (!queued && ncand == 1) {
                // the only grid point: it holds the window's only code, provably the canonical argmin
                const int4 g = n0 == 1 ? g0 : g1;
                const int qi = __ffs(((int)g.z >> 8) & 3) - 1, ci = __ffs((int)g.z & 0xff) - 1;
                const int bi = __ffs((int)((unsigned)g.y >> 16)) - 1, ri = __ffs((int)g.y & 0xffff) - 1;
                bk = ((qi * 8 + ci) * 2 + (bi >> 3)) * CN + (n0 == 1 ? 0 : 128) + (bi & 7) * 16 + ri;
                if (bk >= p.K) { bk = -1; queued = true; }
            } else if (!queued) {
                // a few grid points: their (row, code) pairs join the tile's work list, re-scored densely below
                pbase = atomicAdd(const_cast<int *>(&fq[135]), ncand);
                if (pbase + ncand > PCAP) {
                    for (int w = pbase; w < PCAP; ++w) prk[w] = make_int2(0, -1);       // (stale pairs of an earlier tile)
                    queued = true; pbase = -1;
                }
                else {
                    int w = pbase;
                    auto push = [&](int k) { prk[w++] = make_int2(row, k < p.K ? k : -1); };
                    if (n0 > 0) for_grid(g0, 0, push);
                    if (n1 > 0) for_grid(g1, 1, push);
                }
            }
            if (queued) {
                const int slot = atomicAdd(const_cast<int *>(&fq[0]), 1);
                fq[1 + slot] = row;
            }
            ptx::named_bar_sync(6, 128);                   // work list and queue are complete
            if (ft == 0) VQ2_TL(it, 21);
            {
                const int np = min((int)fq[135], PCAP);
                for (int pi = ft; pi < np; pi += 256) {        // two independent chains per thread: the chain latency, not the issue rate, bounds this phase
                    const int2 ra = prk[pi];
                    const int pj = pi + 128 < np ? pi + 128 : pi;
                    const int2 rb2 = prk[pj];
                    float da, db;
                    exact_dist2(ztile + ra.x * 128, ra.x & 7, ra.y < 0 ? 0 : ra.y, ztile + rb2.x * 128, rb2.x & 7, rb2.y < 0 ? 0 : rb2.y, da, db);
                    pdist[pi] = da;
                    pdist[pj] = db;
                }
            }
            if (ft == 0) VQ2_TL(it, 22);
            const int nq = fq[0];
            // whole-codebook exact scans, all 128 finish threads per queued row: thread t takes codes t, t+128, ...
            for (int qi = 0; qi < nq; ++qi) {
                const int qrow = fq[1 + qi];
                float sd = 0.f;
                int sk = -1;
                for (int k = ft; k < p.K; k += 128) {
                    const float dist = exact_dist(ztile + qrow * 128, qrow & 7, k);
                    if (sk < 0 || vq2_better(dist, k, sd, sk)) { sd = dist; sk = k; }
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    const float od = __shfl_xor_sync(0xffffffffu, sd, off);
                    const int ok = __shfl_xor_sync(0xffffffffu, sk, off);
                    if (ok >= 0 && (sk < 0 || vq2_better(od, ok, sd, sk))) { sd = od; sk = ok; }
                }
                if (lane == 0) { qr[((warp - 12) * 8 + (qi & 7)) * 2] = sd; reinterpret_cast<int *>(qr)[((warp - 12) * 8 + (qi & 7)) * 2 + 1] = sk; }
                ptx::named_bar_sync(6, 128);
                if (row == qrow) {
                    for (int w = 0; w < 4; ++w) {
                        const float od = qr[(w * 8 + (qi & 7)) * 2];
                        const int ok = reinterpret_cast<int *>(qr)[(w * 8 + (qi & 7)) * 2 + 1];
                        if (ok >= 0 && (bk < 0 || vq2_better(od, ok, bd, bk))) { bd = od; bk = ok; }
                    }
                }
                if ((qi & 7) == 7) ptx::named_bar_sync(6, 128);      // the 8 partial slots are recycled
            }
            ptx::named_bar_sync(6, 128);                   // pair distances (and queue results) are complete
            if (ft == 0) VQ2_TL(it, 23);
            if (pbase >= 0) {
                for (int s2 = 0; s2 < ncand; ++s2) {
                    const int k = prk[pbase + s2].y;
                    const float dist = pdist[pbase + s2];
                    if (k >= 0 && (bk < 0 || vq2_better(dist, k, bd, bk))) { bd = dist; bk = k; }
                }
            }
            if (ft == 0) { fq[0] = 0; fq[135] = 0; }      // this parity's counters are next used two tiles (>= two barriers) later
            if (bk < 0) bk = 0;

            // ---- idx, histogram ----
            const long long grow = tile * TM + row;
            if (grow < p.N) {
                p.idx[grow] = bk;
                if (smem_hist) atomicAdd(&hist_s[bk], 1);
                else atomicAdd(&p.hist[bk], 1);
            }
            // ---- gather e_idx, straight-through z_q, SSE: one row per warp step, the lanes across its 64 columns (two
            // each): two-wavefront shared-memory reads of the z row and of the code row, one coalesced 256- / 128-byte
            // store of z_q.  (Thread-per-row with an in-place z_q tile + TMA store took 3700 + 1400 cycles of the tile's
            // dependent chain, profiles/r02_vq2_timeline_k512_before.txt.) ----
            {
                const int wr0 = (warp - 12) * 32;
                const int c16 = lane >> 1;
                const uint32_t zc = (uint32_t)(c16 & 7);
                const unsigned char *zb0 = ztile + wr0 * 128 + (c16 >> 3) * ZATOM + (lane & 1) * 8;
                const uint32_t eoff = (uint32_t)((c16 >> 3) * EATOM + (lane & 1) * 8);
                const long long g0r = tile * TM + wr0;
                const bool full = g0r + 32 <= p.N;                  // every row of this warp is live (all tiles but the last)
                float2 *zqf = reinterpret_cast<float2 *>(p.zq) + g0r * 32 + lane;
                __nv_bfloat162 *zqh = reinterpret_cast<__nv_bfloat162 *>(p.zq) + g0r * 32 + lane;
                float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
                for (int rb = 0; rb < 32; rb += 8) {
                    float2 zv[8], ev[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int k = __shfl_sync(0xffffffffu, bk, rb + j);
                        zv[j] = *reinterpret_cast<const float2 *>(zb0 + (rb + j) * 128 + ((zc ^ (uint32_t)j) << 4));      // (wr0 + rb + j) & 7 == j
                        if (resident) ev[j] = *reinterpret_cast<const float2 *>(code_ptr_smem(k) + eoff + ((zc ^ (uint32_t)(k & 7)) << 4));
                        else ev[j] = __ldg(reinterpret_cast<const float2 *>(p.E + (size_t)k * DD) + lane);
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float dx = __fsub_rn(ev[j].x, zv[j].x), dy = __fsub_rn(ev[j].y, zv[j].y);
                        const float ox = __fadd_rn(zv[j].x, dx), oy = __fadd_rn(zv[j].y, dy);                    // quantizer.py:67
                        if (full || g0r + rb + j < p.N) {
                            acc0 = fmaf(dx, dx, acc0); acc1 = fmaf(dy, dy, acc1);
                            if (ZQBF) zqh[(rb + j) * 32] = __floats2bfloat162_rn(ox, oy);
                            else zqf[(rb + j) * 32] = make_float2(ox, oy);
                        }
                    }
                }
                sse += (double)(acc0 + acc1);       // this lane's 2 columns x 32 rows: fp32 partial, one double add per tile
            }
            __syncwarp();
            if (ft == 0) VQ2_TL(it, 24);
            if (ft == 96) VQ2_TL(it, 25);
            if (lane == 0) { ptx::mbar_arrive(bar(Q_DONE + zs)); ptx::mbar_arrive(bar(C_EMPTY + par)); }
        }
        // ---- CTA reduction of the SSE partial, histogram flush ----
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, off);
        double *red = reinterpret_cast<double *>(sm + OFF_RED);
        if (lane == 0) red[warp - 12] = sse;
        ptx::named_bar_sync(6, 128);
        if (ft == 0) {
            p.partials[blockIdx.x] = (red[0] + red[1]) + (red[2] + red[3]);
            if (blockIdx.x == 0) *p.pending = gridDim.x;
        }
        if (smem_hist)
            for (int k = ft; k < p.K; k += 128) {
                const int cval = hist_s[k];
                if (cval) atomicAdd(&p.hist[k], cval);
            }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}

// workspace prep of a streamed codebook: canonical code norms (quantizer.py:50), their maximum, a non-finite flag
__global__ void vq2_prep_kernel(const float *__restrict__ E, int K, int Kpad, float *__restrict__ bn,
                                unsigned *__restrict__ scal) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Kpad) return;
    if (k >= K) { bn[k] = __int_as_float(0x7f800000); return; }
    const float *e = E + (size_t)k * DD;
    float s = 0.f;
    for (int d = 0; d < DD; ++d) s = __fadd_rn(s, __fmul_rn(e[d], e[d]));
    bn[k] = s;
    if (!(s < __int_as_float(0x7f800000))) atomicOr(&scal[1], 1u);       // inf or NaN
    else atomicMax(&scal[0], __float_as_uint(sqrtf(s) * 1.00001f));       // positive floats order as uints
}

// SSE of the per-CTA partials; n < 0: the count is read from *pending (deferred reduction; 0 = sse is already final)
__global__ void vq2_sum_partials(const double *__restrict__ partials, int n, const unsigned *__restrict__ pending,
                                 double *__restrict__ out) {
    __shared__ double sh[256];
    if (n < 0) n = (int)*pending;
    if (n <= 0) return;
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s += partials[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int off = 128; off >= 1; off >>= 1) {
        if (threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}

size_t align256(size_t x) { return (x + 255) / 256 * 256; }

}  // namespace

bool vq2_supported(long long N, int K, int D) {
    return D == DD && N >= 1 && N < (1LL << 31) && K >= 1 && K <= 8192;
}

// workspace: [bn: Kpad floats][scal: 256 B][partials: 256 doubles]; the deferred-reduction marker lives behind
// both VQ kernels' workspace layouts (vq_ws_marker_offset)
size_t vq2_workspace_bytes(int K) {
    const size_t Kpad = (size_t)((K + CN - 1) / CN) * CN;
    return align256(Kpad * 4) + 256 + 256 * sizeof(double);
}

size_t vq_ws_marker_offset(int K);

int launch_vq_reduce_sse(const void *ws, int K, double *sse, cudaStream_t s) {
    const int Kpad = (K + CN - 1) / CN * CN;
    const unsigned char *w = reinterpret_cast<const unsigned char *>(ws);
    const double *partials = reinterpret_cast<const double *>(w + align256((size_t)Kpad * 4) + 256);
    vq2_sum_partials<<<1, 256, 0, s>>>(partials, -1, reinterpret_cast<const unsigned *>(w + vq_ws_marker_offset(K)), sse);
    VQB_COUNT_LAUNCH(1);
    return vqb_cuda_status(cudaGetLastError());
}

// defer != 0: the SSE partials stay in the workspace (vqb_vq_reduce_sse_f32 sums them later, e.g. on a side stream)
int launch_vq2(const float *z, const float *E, long long N, int K, int D, long long *idx, void *zq, double *sse, int *hist,
               void *ws, int defer, int zq_bf16, cudaStream_t s) {
    if (!vq2_supported(N, K, D)) return VQB_ERR_UNSUPPORTED;
    const int nchunks = (K + CN - 1) / CN;
    const int Kpad = nchunks * CN;
    unsigned char *w = reinterpret_cast<unsigned char *>(ws);
    float *bn = reinterpret_cast<float *>(w);
    unsigned *scal = reinterpret_cast<unsigned *>(w + align256((size_t)Kpad * 4));
    double *partials = reinterpret_cast<double *>(w + align256((size_t)Kpad * 4) + 256);

    CUtensorMap tmz, tme;
    int rc = vqb_encode_tmap_2d(&tmz, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, z, DD, (uint64_t)N, DD * 4, 32, TM, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = vqb_encode_tmap_2d(&tme, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, E, DD, (uint64_t)K, DD * 4, 32, CN, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;

    cudaError_t e = cudaMemsetAsync(hist, 0, sizeof(int) * (size_t)K, s);
    if (e != cudaSuccess) return (int)e;
    int nlaunch = 2;
    if (nchunks > 2) {          // streamed codebook: norms / max / flag from a prep launch
        e = cudaMemsetAsync(scal, 0, 256, s);
        if (e != cudaSuccess) return (int)e;
        vq2_prep_kernel<<<(Kpad + 127) / 128, 128, 0, s>>>(E, K, Kpad, bn, scal);
        nlaunch = 3;
    }
    static bool attr_set = false;
    if (!attr_set) {
        const void *kernels[4] = {(const void *)vq2_kernel<true, false>, (const void *)vq2_kernel<true, true>,
                                  (const void *)vq2_kernel<false, false>, (const void *)vq2_kernel<false, true>};
        for (const void *kf : kernels) {
            e = cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_ALLOC);
            if (e != cudaSuccess) return (int)e;
        }
        attr_set = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long ntiles = (N + TM - 1) / TM;
    int grid = (int)(ntiles < sms ? ntiles : sms);
    if (grid > 256) grid = 256;
    Vq2Params p;
    p.E = E; p.bn = bn; p.scal = reinterpret_cast<const float *>(scal);
    p.N = N; p.K = K; p.nchunks = nchunks;
    p.nbits = 0;
    p.idx = idx; p.partials = partials; p.hist = hist; p.zq_bf16 = zq_bf16; p.zq = zq;
    p.pending = reinterpret_cast<unsigned *>(w + vq_ws_marker_offset(K));
    const dim3 gd((unsigned)grid), bd(NT2);
    cudaError_t le;
    if (nchunks <= 2) le = zq_bf16 ? vqb_launch(vq2_kernel<true, true>, gd, bd, (size_t)SMEM_ALLOC, s, tmz, tme, p)
                                   : vqb_launch(vq2_kernel<true, false>, gd, bd, (size_t)SMEM_ALLOC, s, tmz, tme, p);
    else le = zq_bf16 ? vqb_launch(vq2_kernel<false, true>, gd, bd, (size_t)SMEM_ALLOC, s, tmz, tme, p)
                      : vqb_launch(vq2_kernel<false, false>, gd, bd, (size_t)SMEM_ALLOC, s, tmz, tme, p);
    if (le != cudaSuccess)
        return (int)le;
    if (!defer) vq2_sum_partials<<<1, 256, 0, s>>>(partials, grid, nullptr, sse);
    VQB_COUNT_LAUNCH(defer ? nlaunch - 1 : nlaunch);
    return vqb_cuda_status(cudaGetLastError());
}
