// Shared device/host helpers for libtcavp (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include "../../include/tcavp.h"

namespace tcavp {

// ---------------------------------------------------------------------------------------------
// Host-side error plumbing: every entry point returns 0 or a negative code and records a
// thread-local message readable through tcavp_last_error(). Nothing throws, nothing syncs.
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int  fail_arg(const char* fmt, ...);
int  check_launch(const char* what);
int  sm_count();

#define TCAVP_REQUIRE(cond, ...)                         \
  do {                                                   \
    if (!(cond)) return ::tcavp::fail_arg(__VA_ARGS__);  \
  } while (0)

#define TCAVP_CUDA(expr)                                                          \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      ::tcavp::set_error("%s failed: %s", #expr, cudaGetErrorString(_e));         \
      return TCAVP_ERR_CUDA;                                                      \
    }                                                                             \
  } while (0)

// ---------------------------------------------------------------------------------------------
// Device helpers
// ---------------------------------------------------------------------------------------------
template <typename T> struct Cvt;
template <> struct Cvt<float> {
  __device__ __forceinline__ static float to_f(float v) { return v; }
  __device__ __forceinline__ static float from_f(float v) { return v; }
};
template <> struct Cvt<__nv_bfloat16> {
  __device__ __forceinline__ static float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ __forceinline__ static __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};

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

// Load element i of a tensor whose dtype is only known at run time (TCAVP_F32 / TCAVP_BF16).
__device__ __forceinline__ float load_as_f(const void* p, size_t i, int dtype) {
  return dtype == TCAVP_F32 ? reinterpret_cast<const float*>(p)[i]
                            : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
}
__device__ __forceinline__ void store_from_f(void* p, size_t i, int dtype, float v) {
  if (dtype == TCAVP_F32) reinterpret_cast<float*>(p)[i] = v;
  else reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------------------------------------
// GEMM epilogue shared by the SIMT fp32 kernel and the tcgen05 bf16 kernel.
//   v = acc (+bias[n]);  v = relu(v) if act == RELU   (SwiGLU is applied by the caller on column pairs)
//   v += residual[m_out, n];  out[m_out, n] = v   with m_out = (m / remap_gi) * remap_go + m % remap_gi + remap_off
// ---------------------------------------------------------------------------------------------
struct EpilogueParams {
  int M, N;                 // logical output extent (N is the post-SwiGLU width when act == SWIGLU)
  void* out; int ldo; int out_dtype;
  const float* bias;
  const void* residual; int ldr; int res_dtype;
  int act;
  int remap_gi, remap_go, remap_off;
  const float* rope; int rope_L, rope_dh, rope_cols;   // fused rotary embedding on adjacent column pairs
  const float* row_scale;                              // per-row factor applied to the raw accumulators (fused RMSNorm)
  unsigned long long* sumsq_out;                       // += sum of squares of the final output row, Q44.20 fixed point (order-independent)
  const unsigned long long* row_sumsq; float ss_inv, ss_eps;   // row factor rsqrt(row_sumsq[m] * 2^-20 * ss_inv + ss_eps) (alternative to row_scale)
  __nv_bfloat16* aux; int ld_aux;                      // SwiGLU only: raw (row-scaled) gate/up accumulators for the backward pass
  const float* col_scale;                              // e4m3 operands: per-accumulator-column factor applied to the raw accumulators
};

__device__ __forceinline__ int remap_row(int gi, int go, int off, int m) {
  return gi > 0 ? (m / gi) * go + (m % gi) + off : m;
}

__device__ __forceinline__ float silu_f(float g) { return g / (1.f + __expf(-g)); }
// HF ACT2FN["gelu_new"] (GPT-2): tanh form of GELU
__device__ __forceinline__ float gelu_tanh_f(float x) { return 0.5f * x * (1.f + tanhf(0.7978845608028654f * (x + 0.044715f * x * x * x))); }

// Scalar epilogue (SIMT kernel and the ragged edges of the tensor-core kernel).
__device__ __forceinline__ void epilogue_store(const EpilogueParams& p, int m, int mo, int n, float v) {
  if (m >= p.M || n >= p.N) return;
  if (p.bias) v += __ldg(p.bias + n);
  if (p.act == TCAVP_ACT_RELU) v = fmaxf(v, 0.f);
  else if (p.act == TCAVP_ACT_GELU_TANH) v = gelu_tanh_f(v);
  if (p.residual) v += load_as_f(p.residual, (size_t)mo * p.ldr + n, p.res_dtype);
  store_from_f(p.out, (size_t)mo * p.ldo + n, p.out_dtype, v);
}

constexpr float SUMSQ_FIX = 1048576.f;   // 2^20
__device__ __forceinline__ void sumsq_add(unsigned long long* dst, float partial) {
  atomicAdd(dst, __float2ull_rn(fminf(partial, 1e12f) * SUMSQ_FIX));
}
__device__ __forceinline__ float sumsq_rstd(const unsigned long long* src, float inv_cols, float eps) {
  return rsqrtf((float)__ldg(src) * (1.f / SUMSQ_FIX) * inv_cols + eps);
}

// ---------------------------------------------------------------------------------------------
// Counter-based dropout mask (include/tcavp.h: tcavp_dropout): a pure function of (seed, site, element index).
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ uint32_t drop_key(const uint32_t* seed, uint32_t site) {
  return mix32(__ldg(seed) ^ mix32(site + 0x9E3779B9U * (__ldg(seed + 1) + 1U)));
}
__device__ __forceinline__ bool drop_keep(uint32_t key, unsigned long long idx, uint32_t thresh) {
  uint32_t u = mix32((uint32_t)idx ^ key);
  const uint32_t hi = (uint32_t)(idx >> 32);
  if (hi) u = mix32(u ^ (hi * 0x85EBCA6BU));
  return u >= thresh;
}

void count_launch();

}  // namespace tcavp
