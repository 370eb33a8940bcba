// vq_exact.cu -- fused VectorQuantizer.forward in canonical fp32 arithmetic (sm_100a).
//
// Replaces quantizer.py:45-71 (distance matrix, argmin, one-hot, one-hot @ codebook,
// loss numerator, straight-through, code histogram) with ONE persistent kernel that
// never materialises the (N,K) distance / one-hot matrices:
//   * a CTA owns 64 latent rows at a time and streams the codebook through shared
//     memory in 64-code chunks (so K*D of any size works);
//   * each thread owns a 4x4 (row, code) block and runs the dot products as
//     sequential fmaf chains over d = 0..D-1 -- exactly the canonical order of
//     oracle/csrc/oracle.c, which matched the reference bit for bit on every golden
//     case -- then d = fl(fl(A+B) - fl(2*M)) with non-contracted intrinsics;
//   * (min, idx) is kept per thread (ascending k => first minimum wins, NaN wins like
//     torch.argmin), merged across the 16 threads of a row with shuffles;
//   * the same launch gathers e_idx, writes z_q = z + (e - z), accumulates the SSE and a
//     shared-memory code histogram that is flushed once per CTA.
// This is the bit-exact kernel, the checker for the tcgen05 kernel in vq2.cu and the kernel for every shape vq2 does
// not cover (D != 64 or K > 8192).
#include "common.cuh"

namespace {

constexpr int VR = 64;    // rows per tile
constexpr int VC = 64;    // codes per chunk
constexpr int VNT = 256;  // threads
constexpr int VPAD = 4;

__device__ __forceinline__ bool vq_better(float dn, int kn, float db, int kb) {
    // torch.argmin order (quantizer.py:54): NaN is the minimum; ties -> lowest index.
    const bool nn = dn != dn, nb = db != db;
    if (nn || nb) return nn && (!nb || kn < kb);
    return dn < db || (dn == db && kn < kb);
}

__global__ void code_norms_kernel(const float *__restrict__ E, int K, int D, float *__restrict__ bn) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const float *e = E + (size_t)k * D;
    float s = 0.f;
    for (int d = 0; d < D; ++d) s = __fadd_rn(s, __fmul_rn(e[d], e[d]));  // quantizer.py:50
    bn[k] = s;
}

__global__ void __launch_bounds__(VNT)
vq_exact_kernel(const float *__restrict__ z, const float *__restrict__ E, const float *__restrict__ bn,
                long long N, int K, int D, long long *__restrict__ idx, float *__restrict__ zq,
                double *__restrict__ partials, int *__restrict__ hist, int use_smem_hist) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *zs = reinterpret_cast<float *>(smem_raw);          // [D][VR+VPAD]
    float *es = zs + (size_t)D * (VR + VPAD);                 // [D][VC+VPAD]
    float *an = es + (size_t)D * (VC + VPAD);                 // [VR]
    float *bs = an + VR;                                      // [VC]
    int *best_k = reinterpret_cast<int *>(bs + VC);           // [VR]
    int *shist = best_k + VR;                                 // [K] when use_smem_hist
    __shared__ double red[VNT / 32];

    const int tid = threadIdx.x;
    const int ty = tid >> 4, tx = tid & 15;
    const long long ntiles = (N + VR - 1) / VR;
    double my_sse = 0.0;
    if (use_smem_hist)
        for (int k = tid; k < K; k += VNT) shist[k] = 0;

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long r0 = tile * VR;
        __syncthreads();
        // z tile -> smem, transposed to [d][row]; rows past N read as zero
        for (int e4 = tid; e4 < VR * (D / 4); e4 += VNT) {
            const int row = e4 / (D / 4), d = (e4 % (D / 4)) * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + row < N) v = __ldg(reinterpret_cast<const float4 *>(z + (size_t)(r0 + row) * D + d));
            zs[(size_t)(d + 0) * (VR + VPAD) + row] = v.x;
            zs[(size_t)(d + 1) * (VR + VPAD) + row] = v.y;
            zs[(size_t)(d + 2) * (VR + VPAD) + row] = v.z;
            zs[(size_t)(d + 3) * (VR + VPAD) + row] = v.w;
        }
        __syncthreads();
        if (tid < VR) {  // A_i = sum_d fl(z^2), left to right (quantizer.py:49)
            float s = 0.f;
            for (int d = 0; d < D; ++d) {
                const float v = zs[(size_t)d * (VR + VPAD) + tid];
                s = __fadd_rn(s, __fmul_rn(v, v));
            }
            an[tid] = s;
        }
        float bd[4];
        int bk[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { bd[i] = 0.f; bk[i] = -1; }

        for (int c0 = 0; c0 < K; c0 += VC) {
            __syncthreads();
            for (int e4 = tid; e4 < VC * (D / 4); e4 += VNT) {
                const int c = e4 / (D / 4), d = (e4 % (D / 4)) * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c0 + c < K) v = __ldg(reinterpret_cast<const float4 *>(E + (size_t)(c0 + c) * D + d));
                es[(size_t)(d + 0) * (VC + VPAD) + c] = v.x;
                es[(size_t)(d + 1) * (VC + VPAD) + c] = v.y;
                es[(size_t)(d + 2) * (VC + VPAD) + c] = v.z;
                es[(size_t)(d + 3) * (VC + VPAD) + c] = v.w;
            }
            if (tid < VC) bs[tid] = (c0 + tid < K) ? __ldg(bn + c0 + tid) : 0.f;
            __syncthreads();
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 4
            for (int d = 0; d < D; ++d) {
                const float4 a = *reinterpret_cast<const float4 *>(zs + (size_t)d * (VR + VPAD) + ty * 4);
                const float4 b = *reinterpret_cast<const float4 *>(es + (size_t)d * (VC + VPAD) + tx * 4);
                const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = __fmaf_rn(av[i], bv[j], acc[i][j]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float A = an[ty * 4 + i];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int k = c0 + tx * 4 + j;
                    if (k < K) {
                        // d = fl(fl(A + B) - fl(2*M))   quantizer.py:49-51
                        const float dist = __fsub_rn(__fadd_rn(A, bs[tx * 4 + j]), __fmul_rn(2.0f, acc[i][j]));
                        if (bk[i] < 0 || vq_better(dist, k, bd[i], bk[i])) { bd[i] = dist; bk[i] = k; }
                    }
                }
            }
        }
        // merge the 16 threads (tx) that share a row: lanes differ in the low 4 bits
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int off = 8; off >= 1; off >>= 1) {
                const float od = __shfl_xor_sync(0xffffffffu, bd[i], off);
                const int ok = __shfl_xor_sync(0xffffffffu, bk[i], off);
                if (ok >= 0 && (bk[i] < 0 || vq_better(od, ok, bd[i], bk[i]))) { bd[i] = od; bk[i] = ok; }
            }
            if (tx == 0) best_k[ty * 4 + i] = bk[i];
        }
        __syncthreads();
        // gather + straight-through + SSE + histogram; 16 threads per row, float4 each
        for (int rr = 0; rr < VR; rr += VNT / 16) {
            const int row = rr + (tid >> 4);
            const long long grow = r0 + row;
            if (grow < N) {
                const int k = best_k[row];
                const float *zr = z + (size_t)grow * D;
                const float *er = E + (size_t)k * D;
                float *qr = zq + (size_t)grow * D;
                for (int d = tx * 4; d < D; d += 64) {
                    const float4 zv = __ldg(reinterpret_cast<const float4 *>(zr + d));
                    const float4 ev = __ldg(reinterpret_cast<const float4 *>(er + d));
                    float4 df, q;
                    df.x = __fsub_rn(ev.x, zv.x); df.y = __fsub_rn(ev.y, zv.y);
                    df.z = __fsub_rn(ev.z, zv.z); df.w = __fsub_rn(ev.w, zv.w);
                    q.x = __fadd_rn(zv.x, df.x); q.y = __fadd_rn(zv.y, df.y);   // quantizer.py:67
                    q.z = __fadd_rn(zv.z, df.z); q.w = __fadd_rn(zv.w, df.w);
                    *reinterpret_cast<float4 *>(qr + d) = q;
                    my_sse += (double)df.x * df.x + (double)df.y * df.y + (double)df.z * df.z + (double)df.w * df.w;
                }
                if (tx == 0) {
                    idx[grow] = k;
                    if (use_smem_hist) atomicAdd(&shist[k], 1);
                    else atomicAdd(&hist[k], 1);
                }
            }
        }
    }
    // CTA reduction of the SSE partial (fixed order => deterministic)
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) my_sse += __shfl_xor_sync(0xffffffffu, my_sse, off);
    if ((tid & 31) == 0) red[tid >> 5] = my_sse;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int w = 0; w < VNT / 32; ++w) s += red[w];
        partials[blockIdx.x] = s;
    }
    if (use_smem_hist)
        for (int k = tid; k < K; k += VNT) {
            const int c = shist[k];
            if (c) atomicAdd(&hist[k], c);
        }
}

__global__ void sum_partials_kernel(const double *__restrict__ partials, int n, double *__restrict__ out) {
    __shared__ double sh[256];
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

}  // namespace

// workspace: [K floats code norms | pad to 256 B | VQ_MAX_CTAS doubles]
constexpr int VQ_MAX_CTAS = 2048;

size_t vq_exact_workspace_bytes(int K) {
    return (((size_t)K * sizeof(float) + 255) / 256) * 256 + (size_t)VQ_MAX_CTAS * sizeof(double);
}

int launch_vq_exact(const float *z, const float *E, long long N, int K, int D, long long *idx, float *zq,
                    double *sse, int *hist, void *ws, cudaStream_t s) {
    float *bn = reinterpret_cast<float *>(ws);
    double *partials = reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(ws) +
                                                  (((size_t)K * sizeof(float) + 255) / 256) * 256);
    cudaError_t e = cudaMemsetAsync(hist, 0, sizeof(int) * (size_t)K, s);
    if (e != cudaSuccess) return (int)e;
    code_norms_kernel<<<(K + 127) / 128, 128, 0, s>>>(E, K, D, bn);
    const size_t base = ((size_t)D * (VR + VPAD) + (size_t)D * (VC + VPAD) + VR + VC) * sizeof(float) +
                        VR * sizeof(int);
    const int use_smem_hist = (base + (size_t)K * sizeof(int) <= 200 * 1024) ? 1 : 0;
    const size_t smem = base + (use_smem_hist ? (size_t)K * sizeof(int) : 0);
    constexpr size_t kMaxDyn = 227 * 1024 - 1024;   // 227 KB per CTA minus static smem
    if (smem > kMaxDyn) return VQB_ERR_UNSUPPORTED;
    static bool attr_set = false;
    if (!attr_set) {
        e = cudaFuncSetAttribute(vq_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDyn);
        if (e != cudaSuccess) return (int)e;
        attr_set = true;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int per_sm = (int)((227 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    const long long ntiles = (N + VR - 1) / VR;
    long long grid = (long long)sms * per_sm;
    if (grid > ntiles) grid = ntiles;
    if (grid > VQ_MAX_CTAS) grid = VQ_MAX_CTAS;
    if (grid < 1) grid = 1;
    vq_exact_kernel<<<(unsigned)grid, VNT, smem, s>>>(z, E, bn, N, K, D, idx, zq, partials, hist, use_smem_hist);
    sum_partials_kernel<<<1, 256, 0, s>>>(partials, (int)grid, sse);
    VQB_COUNT_LAUNCH(3);
    return vqb_cuda_status(cudaGetLastError());
}
