// common.cuh -- shared declarations of the sm_100a VQ-VAE kernels (internal).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vqvae_b200.h"

#define VQB_MAX_TAPS 16

// The library never reads the environment.  A library built with -DVQB_DIAG=1 (VQB_DIAG=1 python -m
// vqvae_b200.build, used by tools/diag) differs from the release build only by the in-kernel timelines of vq2,
// hconv and res_bf16 (#if VQB_DIAG); it computes the same results with the same launches.
#ifndef VQB_DIAG
#define VQB_DIAG 0
#endif

// halo tile width in pixels of conv_halo.cu / res_tc.cu / latent_tc.cu: an 8-pixel tile + 1 each side
constexpr int VQB_HALO_WP = 10;

// One launch of the generalised gather-form convolution
//   out[n, gy*out_step+out_py, gx*out_step+out_px, co] =
//       act( bias[co] + skip + sum_{t<ntaps, ci} in[n, gy*in_step+dy[t], gx*in_step+dx[t], ci]
//                                                * w[tap_w[t]*Cin + ci][co] )
// which covers nn.Conv2d (in_step = stride, out_step = 1, dy = r - pad), stride-1
// nn.ConvTranspose2d (dy = pad - r) and one sub-pixel phase of a stride-2
// nn.ConvTranspose2d (in_step = 1, out_step = 2, taps of matching parity).
struct ConvLaunch {
    const float *in, *w, *bias, *skip;
    float *out;
    int B, Cin, H, W, Cout;
    int OHg, OWg;                 // output grid of this launch
    int in_step, out_step, out_py, out_px;
    int ntaps;
    int tap_w[VQB_MAX_TAPS], tap_dy[VQB_MAX_TAPS], tap_dx[VQB_MAX_TAPS];
    long long in_sn, in_sh, in_sw, in_sc;      // element strides of `in`
    long long out_sn, out_sh, out_sw, out_sc;  // element strides of `out` (and `skip`)
    int relu;
};

int launch_conv_ffma(const ConvLaunch &p, cudaStream_t s);
int launch_conv_small_cout(const ConvLaunch &p, cudaStream_t s);

// process-wide count of kernels launched through the C ABI (vqb_launch_count)
extern unsigned long long g_vqb_launches;
#define VQB_COUNT_LAUNCH(n) (g_vqb_launches += (n))

// Programmatic dependent launch: the next kernel of the layer chain may start its prologue (barrier init,
// TMEM allocation, tensor-map prefetch) while this one drains; it blocks in pdl_wait() until the previous
// grid has completed and its writes are visible.
#ifdef __CUDACC__
#include <utility>
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
static inline cudaError_t vqb_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                     Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
// same, as thread-block clusters of `cluster` CTAs along x (the grid must be a multiple of it)
template <typename... KArgs, typename... Args>
static inline cudaError_t vqb_launch_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                                             unsigned cluster, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
#endif

static inline int vqb_cuda_status(cudaError_t e) { return e == cudaSuccess ? 0 : (int)e; }
