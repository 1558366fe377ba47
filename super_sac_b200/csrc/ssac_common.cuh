// Shared helpers for libssac_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <string>

#include "../../include/ssac_b200.h"

namespace ssac {

void set_error(const std::string& msg);
int fail(int code, const char* what);

#define SSAC_REQUIRE(cond, msg)                               \
  do {                                                        \
    if (!(cond)) return ::ssac::fail(SSAC_E_BADARG, msg);     \
  } while (0)

#define SSAC_CHECK_LAUNCH(name)                                        \
  do {                                                                 \
    cudaError_t e__ = cudaGetLastError();                              \
    if (e__ != cudaSuccess) {                                          \
      ::ssac::set_error(std::string(name) + ": " + cudaGetErrorString(e__)); \
      return (int)e__;                                                 \
    }                                                                  \
  } while (0)

constexpr int kNumSMs = 148;  // B200

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------------
// A kernel launched with launch_pdl() may start while its predecessor in the stream is still running; it must execute
// pdl_wait() before touching anything an earlier kernel produced (or still reads), and only then pdl_trigger(), so that
// at most ONE predecessor is ever in flight behind it.  Whatever precedes pdl_wait() (TMEM allocation, barrier set-up,
// loads of parameters that only Adam / Polyak write -- kernels that never trigger early) overlaps the predecessor's
// tail.  Without the launch attribute both instructions are no-ops, so the same kernels serve every launch site.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();   // ssac_set_pdl (ssac_elementwise.cu)

// cluster_x > 1: thread-block clusters of that many CTAs along x (the attribute comes first so that it survives PDL off)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_cluster_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                      int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  return launch_cluster_pdl(kernel, grid, block, smem, stream, 1, static_cast<Args&&>(args)...);
}

// ---- Adam (torch/optim/adam.py _single_tensor_adam as configured at main.py:188-239) --------------------------------
struct AdamScalars {
  float step_size, bc2_sqrt, clip_coef;
};
// Every operation is spelled out (no compiler-chosen FMA contraction).  The contractions are the ones torch's CUDA
// kernels compile to: lerp = fma(w, end - start, start), addcmul = fma(value * t1, t2, self),
// addcdiv = fma(value, t1 / t2, self).
__device__ __forceinline__ void adam1(float& p, float& g, float& m, float& v, const AdamScalars& sc, float one_m_b1,
                                      float b2, float one_m_b2, float eps, float wd, bool clip) {
  if (clip) g = __fmul_rn(g, sc.clip_coef);
  float ge = g;
  if (wd != 0.f) ge = __fmaf_rn(wd, p, ge);                                   // grad.add(param, alpha=wd)
  m = __fmaf_rn(one_m_b1, __fsub_rn(ge, m), m);                               // exp_avg.lerp_(grad, 1-beta1)
  v = __fmaf_rn(__fmul_rn(one_m_b2, ge), ge, __fmul_rn(v, b2));               // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1-beta2)
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), sc.bc2_sqrt), eps);  // exp_avg_sq.sqrt() / bc2_sqrt + eps
  p = __fmaf_rn(-sc.step_size, __fdiv_rn(m, denom), p);                       // param.addcdiv_(exp_avg, denom, value=-step_size)
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide reductions for blockDim.x <= 1024 (multiple of 32).  `scratch` is 32 floats of shared memory.
// Every thread gets the result.
template <typename Op>
__device__ __forceinline__ float block_reduce(float v, float* scratch, Op op, float identity) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();  // protect scratch reuse
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  float r = (lane < nw) ? scratch[lane] : identity;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) r = op(r, __shfl_xor_sync(0xffffffffu, r, o));
  return r;
}
struct OpSum { __device__ float operator()(float a, float b) const { return a + b; } };
struct OpMax { __device__ float operator()(float a, float b) const { return fmaxf(a, b); } };
struct OpMin { __device__ float operator()(float a, float b) const { return fminf(a, b); } };

}  // namespace ssac
