// Shared helpers for the lcao_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "lcao_b200.h"

void lcao_set_error(const char* fmt, ...);

#define LCAO_REQUIRE(cond, ...)            \
  do {                                     \
    if (!(cond)) {                         \
      lcao_set_error(__VA_ARGS__);         \
      return LCAO_E_ARG;                   \
    }                                      \
  } while (0)

#define LCAO_CUDA(call)                                                              \
  do {                                                                               \
    cudaError_t err__ = (call);                                                      \
    if (err__ != cudaSuccess) {                                                      \
      lcao_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(err__)); \
      return LCAO_E_CUDA;                                                            \
    }                                                                                \
  } while (0)

extern unsigned long long g_lcao_launches;  // kernels launched by this library (reported by lcao_launch_count)
#define LCAO_LAUNCH_CHECK()        \
  do {                             \
    ++g_lcao_launches;             \
    LCAO_CUDA(cudaGetLastError()); \
  } while (0)

// ---- programmatic dependent launch (PDL): a kernel launched through launch_pdl may begin — block scheduling, barrier /
// TMEM set-up, the split of its resident weights — while the kernel before it in the stream is still draining, once every
// CTA of that kernel has executed pdl_trigger() (or exited).  It must call pdl_wait() before it touches anything the
// stream's earlier work produces or still reads; pdl_wait() returns when ALL earlier grids have completed and flushed.
// Kernels without the launch attribute, and predecessors that never trigger (torch's kernels, memsets), behave as usual.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool lcao_pdl_enabled();  // abi.cu: LCAO_PDL=0 switches the launch attribute off
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = lcao_pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// sum over the 8 lanes of an aligned lane-octet
__device__ __forceinline__ float octet_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float siluf(float x) { return x * sigmoidf_acc(x); }
__device__ __forceinline__ float silu_gradf(float x) {
  float s = sigmoidf_acc(x);
  return s * (1.0f + x * (1.0f - s));
}
// generic activation and its derivative as functions of the PRE-activation (torch semantics: F.softplus threshold 20,
// exact-erf GELU, ELU alpha 1, LeakyReLU slope 0.01; ReLU maps NaN to NaN and passes the gradient at a NaN input, as
// torch.relu / threshold_backward do); SiLU is the hot case and comes first
__device__ __forceinline__ float softplusf_acc(float x) { return x > 20.0f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float act_fwdf(int act, float x) {
  switch (act) {
    case LCAO_ACT_SILU: return siluf(x);
    case LCAO_ACT_SSP: return softplusf_acc(x) - 0.69314718055994530942f;
    case LCAO_ACT_SOFTPLUS: return softplusf_acc(x);
    case LCAO_ACT_RELU: return x < 0.0f ? 0.0f : x;
    case LCAO_ACT_TANH: return tanhf(x);
    case LCAO_ACT_SIGMOID: return sigmoidf_acc(x);
    case LCAO_ACT_GELU: return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
    case LCAO_ACT_ELU: return x > 0.0f ? x : expm1f(x);
    case LCAO_ACT_LEAKY_RELU: return x > 0.0f ? x : 0.01f * x;
    default: return x;
  }
}
__device__ __forceinline__ float act_gradf(int act, float x) {
  switch (act) {
    case LCAO_ACT_SILU: return silu_gradf(x);
    case LCAO_ACT_SSP:
    case LCAO_ACT_SOFTPLUS: return x > 20.0f ? 1.0f : sigmoidf_acc(x);
    case LCAO_ACT_RELU: return x <= 0.0f ? 0.0f : 1.0f;
    case LCAO_ACT_TANH: { const float t = tanhf(x); return 1.0f - t * t; }
    case LCAO_ACT_SIGMOID: { const float s = sigmoidf_acc(x); return s * (1.0f - s); }
    case LCAO_ACT_GELU:
      return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * 0.39894228040143267794f * expf(-0.5f * x * x);
    case LCAO_ACT_ELU: return x > 0.0f ? 1.0f : expf(x);
    case LCAO_ACT_LEAKY_RELU: return x > 0.0f ? 1.0f : 0.01f;
    default: return 1.0f;
  }
}
// GEN = false: SiLU only.  The bandwidth-bound edge kernels are instantiated twice so that the default activation does
// not carry the code (and registers) of the other eight.
template <bool GEN>
__device__ __forceinline__ float act_fwd_t(int act, float x) { return GEN ? act_fwdf(act, x) : siluf(x); }
template <bool GEN>
__device__ __forceinline__ float act_grad_t(int act, float x) { return GEN ? act_gradf(act, x) : silu_gradf(x); }
template <bool GEN>
__device__ __forceinline__ float4 act_fwd4(int act, float4 v) {
  return make_float4(act_fwd_t<GEN>(act, v.x), act_fwd_t<GEN>(act, v.y), act_fwd_t<GEN>(act, v.z), act_fwd_t<GEN>(act, v.w));
}
template <bool GEN>
__device__ __forceinline__ float4 act_grad4(int act, float4 v) {
  return make_float4(act_grad_t<GEN>(act, v.x), act_grad_t<GEN>(act, v.y), act_grad_t<GEN>(act, v.z), act_grad_t<GEN>(act, v.w));
}
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// Sum 8 per-lane partials over the 32 lanes with 9 shuffles; every lane ends up with the total of
// element  4*bit4(lane) + 2*bit3(lane) + bit2(lane).
__device__ __forceinline__ float bfly8(const float (&p)[8], int lane) {
  float q4[4], q2[2];
  bool up = (lane & 16) != 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float recv = __shfl_xor_sync(0xffffffffu, up ? p[k] : p[k + 4], 16);
    q4[k] = (up ? p[k + 4] : p[k]) + recv;
  }
  up = (lane & 8) != 0;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float recv = __shfl_xor_sync(0xffffffffu, up ? q4[k] : q4[k + 2], 8);
    q2[k] = (up ? q4[k + 2] : q4[k]) + recv;
  }
  up = (lane & 4) != 0;
  const float recv = __shfl_xor_sync(0xffffffffu, up ? q2[0] : q2[1], 4);
  float r = (up ? q2[1] : q2[0]) + recv;
  r += __shfl_xor_sync(0xffffffffu, r, 2);
  r += __shfl_xor_sync(0xffffffffu, r, 1);
  return r;
}
__device__ __forceinline__ int bfly8_index(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }

// real spherical harmonics Y_l^0(c) and derivatives (shbf.py:41-63)
#define LCAO_Y0 0.28209479177387814f
#define LCAO_Y1 0.4886025119029199f
#define LCAO_Y2A 0.9461746957575601f
#define LCAO_Y2B 0.31539156525252005f
#define LCAO_Y3 0.3731763325901154f
