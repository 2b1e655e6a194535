// LayerNorm (+residual, +row remap, +row vector) and RMSNorm.  Bandwidth-bound: one warp per row,
// 16-byte vector accesses, warp-shuffle reductions, fp32 statistics for both storage dtypes.
#include "common.cuh"

namespace tcavp {

// Load / store 8 consecutive elements (16 bytes for bf16, 32 bytes for fp32).
__device__ __forceinline__ void load8(const void* base, size_t idx, int dtype, float (&v)[8]) {
  if (dtype == TCAVP_BF16) {
    uint4 u = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(base) + idx);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 f = __bfloat1622float2(h[e]);
      v[2 * e] = f.x;
      v[2 * e + 1] = f.y;
    }
  } else {
    const float4* p = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + idx);
    float4 a = p[0], b = p[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
}
__device__ __forceinline__ void store8(void* base, size_t idx, int dtype, const float (&v)[8]) {
  if (dtype == TCAVP_BF16) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int e = 0; e < 4; ++e) h[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
    *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(base) + idx) = u;
  } else {
    float4* p = reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + idx);
    p[0] = make_float4(v[0], v[1], v[2], v[3]);
    p[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
}

// VEC = true: cols % 8 == 0 and all row starts are 16B (bf16) / 32B (fp32) aligned.
template <bool VEC>
__global__ void __launch_bounds__(256) layernorm_kernel(const void* x, const void* res,
                                                        const float* __restrict__ w, const float* __restrict__ b,
                                                        void* out, int rows, int cols, float eps, int in_dtype,
                                                        int out_dtype, int gi, int go, int off, const float* __restrict__ rowvec) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const size_t base = (size_t)row * cols;
  float s = 0.f;
  if (VEC) {
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      load8(x, base + c, in_dtype, v);
      if (res) {
        float r[8];
        load8(res, base + c, in_dtype, r);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] += r[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) s += v[e];
    }
  } else {
    for (int c = lane; c < cols; c += 32) s += load_as_f(x, base + c, in_dtype) + (res ? load_as_f(res, base + c, in_dtype) : 0.f);
  }
  const float mean = warp_sum(s) / cols;
  float q = 0.f;
  if (VEC) {
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      load8(x, base + c, in_dtype, v);
      if (res) {
        float r[8];
        load8(res, base + c, in_dtype, r);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] += r[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) q += (v[e] - mean) * (v[e] - mean);
    }
  } else {
    for (int c = lane; c < cols; c += 32) {
      float v = load_as_f(x, base + c, in_dtype) + (res ? load_as_f(res, base + c, in_dtype) : 0.f);
      q += (v - mean) * (v - mean);
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / cols + eps);
  const size_t obase = (size_t)remap_row(gi, go, off, row) * cols;
  if (VEC) {
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      load8(x, base + c, in_dtype, v);
      if (res) {
        float r[8];
        load8(res, base + c, in_dtype, r);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] += r[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[e] = (v[e] - mean) * rstd * __ldg(w + c + e) + __ldg(b + c + e);
        if (rowvec) v[e] += __ldg(rowvec + c + e);
      }
      store8(out, obase + c, out_dtype, v);
    }
  } else {
    for (int c = lane; c < cols; c += 32) {
      float v = load_as_f(x, base + c, in_dtype) + (res ? load_as_f(res, base + c, in_dtype) : 0.f);
      v = (v - mean) * rstd * __ldg(w + c) + __ldg(b + c);
      if (rowvec) v += __ldg(rowvec + c);
      store_from_f(out, obase + c, out_dtype, v);
    }
  }
}

// Register-resident LayerNorm for rows of <= G * NV * 8 elements: G lanes share a row (32 / G rows per warp), every lane
// keeps NV 8-element vectors, so the row is read ONCE and narrow rows (d_model = 64: G = 8) still use all 32 lanes.
template <int G, int NV>
__global__ void __launch_bounds__(256) layernorm_reg_kernel(const void* __restrict__ x, const void* __restrict__ res,
                                                            const float* __restrict__ w, const float* __restrict__ b,
                                                            void* __restrict__ out, int rows, int cols, float eps, int in_dtype,
                                                            int out_dtype, int gi, int go, int off, const float* __restrict__ rowvec) {
  constexpr int RPW = 32 / G;
  const int lane = threadIdx.x & 31, sub = lane % G;
  const int row = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * RPW + lane / G;
  const bool live = row < rows;
  const size_t base = (size_t)(live ? row : 0) * cols;
  float v[NV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * G + sub) * 8;
    if (live && c < cols) {
      load8(x, base + c, in_dtype, v[i]);
      if (res) {
        float r[8];
        load8(res, base + c, in_dtype, r);
#pragma unroll
        for (int e = 0; e < 8; ++e) v[i][e] += r[e];
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) s += v[i][e];
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[i][e] = 0.f;
    }
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / cols;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    if ((i * G + sub) * 8 < cols) {
#pragma unroll
      for (int e = 0; e < 8; ++e) q += (v[i][e] - mean) * (v[i][e] - mean);
    }
  }
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / cols + eps);
  if (!live) return;
  const size_t obase = (size_t)remap_row(gi, go, off, row) * cols;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * G + sub) * 8;
    if (c < cols) {
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + c)), w1 = __ldg(reinterpret_cast<const float4*>(w + c + 4));
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(b + c)), b1 = __ldg(reinterpret_cast<const float4*>(b + c + 4));
      const float ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      float o8[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        o8[e] = (v[i][e] - mean) * rstd * ww[e] + bb[e];
        if (rowvec) o8[e] += __ldg(rowvec + c + e);
      }
      store8(out, obase + c, out_dtype, o8);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over many bf16 rows (the 25 LayerNorm passes of a GPT-2-arch backbone at M = scenes x 144 rows): rows staged through shared
// memory by the bulk-copy engine.  The register-resident kernel above keeps one row per warp in flight (1.5 KB at 768 columns, 32 warps
// per SM at 56 registers = 48 KB per SM), which is latency-bound at ~2.9 TB/s; here every warp owns a ring of PIPE_STAGES row buffers
// filled by cp.async.bulk (one elected lane, mbarrier complete_tx), so the bytes in flight per SM are the ring (8 warps x 8 rows x 1.5 KB
// per block, two blocks per SM) and no longer cost registers.  Warps stride over the rows (persistent grid); statistics and the affine map are the same
// fp32 arithmetic, in the same order, as layernorm_reg_kernel<32, NV>.
// ------------------------------------------------------------------------------------------------
namespace lnp {
constexpr int MAX_STAGES = 8, WARPS = 8;
__host__ __device__ inline int stages_for(int cols) { return cols <= 768 ? 8 : 6; }      // ~98 KB of ring per block: two blocks per SM
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
}  // namespace lnp

template <int NV>
__global__ void __launch_bounds__(lnp::WARPS * 32, 2) layernorm_pipe_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                                                                        const float* __restrict__ b, void* __restrict__ out, int rows, int cols,
                                                                        float eps, int out_dtype, int gi, int go, int off,
                                                                        const float* __restrict__ rowvec, int ldo) {
  using namespace lnp;
  extern __shared__ __align__(128) uint8_t ln_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t row_bytes = (uint32_t)cols * 2u;
  const int PIPE_STAGES = stages_for(cols);
  const uint32_t ring = smem_u32(ln_smem) + (uint32_t)warp * PIPE_STAGES * row_bytes;
  const uint32_t bars = smem_u32(ln_smem) + (uint32_t)WARPS * PIPE_STAGES * row_bytes + (uint32_t)warp * PIPE_STAGES * 8u;
  const int wstride = gridDim.x * WARPS;
  const int row0 = blockIdx.x * WARPS + warp;
  if (lane == 0) {
    for (int s = 0; s < PIPE_STAGES; ++s) mbar_init(bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (lane == 0) {      // prologue: the first PIPE_STAGES rows of this warp
    for (int s = 0; s < PIPE_STAGES; ++s) {
      const long long r = (long long)row0 + (long long)s * wstride;
      if (r < rows) {
        mbar_expect_tx(bars + 8 * s, row_bytes);
        bulk_load(ring + s * row_bytes, x + (size_t)r * cols, row_bytes, bars + 8 * s);
      }
    }
  }
  // a lane handles the same columns of every row: its slice of the affine parameters lives in registers for the whole kernel (loaded
  // per row they were 4x the row's own bytes through L1TEX: ncu showed l1tex 86 % busy against 45 % DRAM)
  float wr[NV][8], br[NV][8];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 8;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      wr[i][e] = c < cols ? __ldg(w + c + e) : 0.f;
      br[i][e] = c < cols ? __ldg(b + c + e) : 0.f;
    }
  }
  int stage = 0;
  uint32_t phase = 0;
  for (long long row = row0; row < rows; row += wstride) {
    mbar_wait(bars + 8 * stage, phase);
    float v[NV][8];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
        uint4 u;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(ring + stage * row_bytes + c * 2));
        const uint32_t q[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          v[i][2 * e] = __uint_as_float(q[e] << 16);
          v[i][2 * e + 1] = __uint_as_float(q[e] & 0xffff0000u);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) sum += v[i][e];
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[i][e] = 0.f;
      }
    }
    // the row is in registers: hand the buffer back to the copy engine (every lane has read its part once the shuffle below has run;
    // the refill is issued after the first reduction, which all lanes take part in)
    sum = warp_sum(sum);
    if (lane == 0) {
      const long long nxt = row + (long long)PIPE_STAGES * wstride;
      if (nxt < rows) {
        mbar_expect_tx(bars + 8 * stage, row_bytes);
        bulk_load(ring + stage * row_bytes, x + (size_t)nxt * cols, row_bytes, bars + 8 * stage);
      }
    }
    const float mean = sum / cols;
    float q2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      if ((i * 32 + lane) * 8 < cols) {
#pragma unroll
        for (int e = 0; e < 8; ++e) q2 += (v[i][e] - mean) * (v[i][e] - mean);
      }
    }
    const float rstd = rsqrtf(warp_sum(q2) / cols + eps);
    const size_t obase = (size_t)remap_row(gi, go, off, (int)row) * ldo;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
        float o8[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          o8[e] = (v[i][e] - mean) * rstd * wr[i][e] + br[i][e];
          if (rowvec) o8[e] += __ldg(rowvec + c + e);
        }
        store8(out, obase + c, out_dtype, o8);
      }
    }
    if (++stage == PIPE_STAGES) { stage = 0; phase ^= 1; }
  }
}

// Per-row e4m3 quantisation (tcavp_quant_e4m3_rows) on the same bulk-copy row ring: each warp owns `stages` row buffers filled by
// cp.async.bulk.  The whole row stays in shared memory while the warp finds its amax (and sum of squares), then is read a second time to
// quantise it, so rows of any width up to the ring size take the same path (768-class rows: eight per warp in flight, 7B-class MLP
// rows of 11 008 columns: one).
namespace q8 {
__device__ __forceinline__ uint32_t e4m3x4(float a, float b, float c, float d) {     // a lands in the lowest byte
  uint16_t lo, hi;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(b), "f"(a));
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(d), "f"(c));
  return (uint32_t)lo | ((uint32_t)hi << 16);
}
__device__ __forceinline__ void lds8(uint32_t addr, float (&v)[8]) {
  uint4 u;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr));
  const uint32_t q[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    v[2 * e] = __uint_as_float(q[e] << 16);
    v[2 * e + 1] = __uint_as_float(q[e] & 0xffff0000u);
  }
}
constexpr int RING_BYTES = 96 << 10;     // per block (lnp::WARPS warps); two blocks per SM at 768-class rows
__host__ __device__ inline int stages_for(int cols) {
  const int s = RING_BYTES / (lnp::WARPS * (cols * 2 + 8));
  return s < 1 ? 1 : (s > lnp::MAX_STAGES ? lnp::MAX_STAGES : s);
}
}  // namespace q8

__global__ void __launch_bounds__(lnp::WARPS * 32) quant_e4m3_kernel(const __nv_bfloat16* __restrict__ x, int ldi, uint8_t* __restrict__ q, int ldo,
                                                                    float* __restrict__ f, int rows, int cols, int rms, float eps) {
  using namespace lnp;
  extern __shared__ __align__(128) uint8_t ln_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t row_bytes = (uint32_t)cols * 2u;
  const int stages = q8::stages_for(cols);
  const uint32_t ring = smem_u32(ln_smem) + (uint32_t)warp * stages * row_bytes;
  const uint32_t bars = smem_u32(ln_smem) + (uint32_t)WARPS * stages * row_bytes + (uint32_t)warp * stages * 8u;
  const int wstride = gridDim.x * WARPS;
  const int row0 = blockIdx.x * WARPS + warp;
  if (lane == 0) {
    for (int s = 0; s < stages; ++s) mbar_init(bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (lane == 0) {
    for (int s = 0; s < stages; ++s) {
      const long long r = (long long)row0 + (long long)s * wstride;
      if (r < rows) {
        mbar_expect_tx(bars + 8 * s, row_bytes);
        bulk_load(ring + s * row_bytes, x + (size_t)r * ldi, row_bytes, bars + 8 * s);
      }
    }
  }
  int stage = 0;
  uint32_t phase = 0;
  for (long long row = row0; row < rows; row += wstride) {
    mbar_wait(bars + 8 * stage, phase);
    const uint32_t buf = ring + stage * row_bytes;
    float amax = 0.f, ss = 0.f;
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      q8::lds8(buf + c * 2, v);
      float p = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        amax = fmaxf(amax, fabsf(v[e]));
        p = fmaf(v[e], v[e], p);
      }
      ss += p;      // per-8-element partials keep the rounding error of long rows (11 008 columns) near 1e-7
    }
    amax = warp_max(amax);
    const float s = amax > 0.f ? __fdiv_rn(448.f, amax) : 0.f;
    uint8_t* qrow = q + (size_t)row * ldo;
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      q8::lds8(buf + c * 2, v);
      const uint32_t lo = q8::e4m3x4(v[0] * s, v[1] * s, v[2] * s, v[3] * s), hi = q8::e4m3x4(v[4] * s, v[5] * s, v[6] * s, v[7] * s);
      asm volatile("st.global.v2.b32 [%0], {%1, %2};" ::"l"(qrow + c), "r"(lo), "r"(hi) : "memory");
    }
    float fr = __fdiv_rn(amax, 448.f);
    if (rms) fr *= rsqrtf(warp_sum(ss) / cols + eps);
    __syncwarp();     // every lane has read the row: the buffer goes back to the copy engine
    if (lane == 0) {
      f[row] = fr;
      const long long nxt = row + (long long)stages * wstride;
      if (nxt < rows) {
        mbar_expect_tx(bars + 8 * stage, row_bytes);
        bulk_load(buf, x + (size_t)nxt * ldi, row_bytes, bars + 8 * stage);
      }
    }
    if (++stage == stages) { stage = 0; phase ^= 1; }
  }
}

// Row-strided LayerNorm for shapes outside the bulk-copy kernel (narrow / unaligned rows, fp32): warp per row, element-wise.
__global__ void __launch_bounds__(256) layernorm_strided_kernel(const void* __restrict__ x, int ldx, const float* __restrict__ w,
                                                                const float* __restrict__ b, void* __restrict__ out, int ldo, int rows, int cols,
                                                                float eps, int in_dtype, int out_dtype) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const size_t base = (size_t)row * ldx, obase = (size_t)row * ldo;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += load_as_f(x, base + c, in_dtype);
  const float mean = warp_sum(s) / cols;
  float q = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float d = load_as_f(x, base + c, in_dtype) - mean;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / cols + eps);
  for (int c = lane; c < cols; c += 32)
    store_from_f(out, obase + c, out_dtype, (load_as_f(x, base + c, in_dtype) - mean) * rstd * __ldg(w + c) + __ldg(b + c));
}

template <bool VEC>
__global__ void __launch_bounds__(256) rmsnorm_kernel(const void* __restrict__ x, const float* __restrict__ w,
                                                      void* __restrict__ out, int rows, int cols, int ldi, int ldo, float eps,
                                                      int in_dtype, int out_dtype) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const size_t base = (size_t)row * ldi, obase = (size_t)row * ldo;
  float q = 0.f;
  if (VEC) {
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      load8(x, base + c, in_dtype, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) q += v[e] * v[e];
    }
  } else {
    for (int c = lane; c < cols; c += 32) {
      float v = load_as_f(x, base + c, in_dtype);
      q += v * v;
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / cols + eps);
  if (VEC) {
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      load8(x, base + c, in_dtype, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[e] = __ldg(w + c + e) * (v[e] * rstd);
      }
      store8(out, obase + c, out_dtype, v);
    }
  } else {
    for (int c = lane; c < cols; c += 32) {
      store_from_f(out, obase + c, out_dtype, __ldg(w + c) * (load_as_f(x, base + c, in_dtype) * rstd));
    }
  }
}

// rstd[r] = rsqrt(mean(x[r,:]^2) + eps): one warp per row, 16-byte loads
template <bool VEC>
__global__ void __launch_bounds__(256) row_rstd_kernel(const void* __restrict__ x, int ldx, int rows, int cols, float eps, int dtype,
                                                       float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const size_t base = (size_t)row * ldx;
  float q = 0.f;
  if (VEC) {
    for (int c = lane * 8; c < cols; c += 256) {
      float v[8];
      load8(x, base + c, dtype, v);
#pragma unroll
      for (int e = 0; e < 8; ++e) q += v[e] * v[e];
    }
  } else {
    for (int c = lane; c < cols; c += 32) {
      const float v = load_as_f(x, base + c, dtype);
      q += v * v;
    }
  }
  q = warp_sum(q);
  if (lane == 0) out[row] = rsqrtf(q / cols + eps);
}

static bool aligned_rows(const void* p, int ld, int dtype) {
  const size_t es = dtype == TCAVP_BF16 ? 2 : 4;
  return p == nullptr || (reinterpret_cast<uintptr_t>(p) % (8 * es) == 0 && ((size_t)ld * es) % (8 * es) == 0);
}

}  // namespace tcavp

namespace tcavp {
// Register-resident RMSNorm for rows of <= 1024 elements: the row is read once (NV 8-element vectors per lane).
template <int NV>
__global__ void __launch_bounds__(256) rmsnorm_reg_kernel(const void* __restrict__ x, const float* __restrict__ w, void* __restrict__ out, int rows,
                                                          int cols, int ldi, int ldo, float eps, int in_dtype, int out_dtype) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const size_t base = (size_t)row * ldi, obase = (size_t)row * ldo;
  float v[NV][8];
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 8;
    if (c < cols) {
      load8(x, base + c, in_dtype, v[i]);
#pragma unroll
      for (int e = 0; e < 8; ++e) q += v[i][e] * v[i][e];
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / cols + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = (i * 32 + lane) * 8;
    if (c < cols) {
      const float4 w0 = __ldg(reinterpret_cast<const float4*>(w + c)), w1 = __ldg(reinterpret_cast<const float4*>(w + c + 4));
      const float ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
      float o8[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) o8[e] = v[i][e] * rstd * ww[e];
      store8(out, obase + c, out_dtype, o8);
    }
  }
}
}  // namespace tcavp

extern "C" int tcavp_layernorm(const void* x, const void* residual, const float* w, const float* b, void* out, int rows,
                               int cols, float eps, int in_dtype, int out_dtype, int remap_gi, int remap_go, int remap_off,
                               const float* rowvec, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(rows >= 0 && cols > 0, "tcavp_layernorm: bad shape rows=%d cols=%d", rows, cols);
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && w && b && out, "tcavp_layernorm: null pointer");
  TCAVP_REQUIRE((in_dtype | 1) == 1 && (out_dtype | 1) == 1, "tcavp_layernorm: bad dtype");
  const bool vec = cols % 8 == 0 && aligned_rows(x, cols, in_dtype) && aligned_rows(residual, cols, in_dtype) &&
                   aligned_rows(out, cols, out_dtype);
  const int wpb = 8;
  const int grid = (rows + wpb - 1) / wpb;
  const bool wb_al = reinterpret_cast<uintptr_t>(w) % 16 == 0 && reinterpret_cast<uintptr_t>(b) % 16 == 0;
  // many bf16 rows, no residual: rows staged through shared memory by the bulk-copy engine (see layernorm_pipe_kernel)
  static int pipe_on = -1, pipe_min_rows = 24576;      // 36 864 x 768: 31 us through the ring vs 39 us register-resident; 16 384 rows: equal
  if (pipe_on < 0) {
    const char* e = getenv("TCAVP_LN_PIPE");
    pipe_on = e ? atoi(e) : 1;
    e = getenv("TCAVP_LN_PIPE_MIN_ROWS");
    if (e) pipe_min_rows = atoi(e);
  }
  if (pipe_on && vec && wb_al && !residual && in_dtype == TCAVP_BF16 && cols >= 256 && cols <= 1024 && rows >= pipe_min_rows &&
      (!rowvec || reinterpret_cast<uintptr_t>(rowvec) % 4 == 0)) {
    const size_t smem = (size_t)lnp::WARPS * lnp::stages_for(cols) * ((size_t)cols * 2 + 8);
    const int blocks_per_sm = (int)((200u << 10) / smem) > 2 ? 2 : (int)((200u << 10) / smem);
    int grid_p = sm_count() * (blocks_per_sm < 1 ? 1 : blocks_per_sm);
    if (grid_p > (rows + lnp::WARPS - 1) / lnp::WARPS) grid_p = (rows + lnp::WARPS - 1) / lnp::WARPS;
#define TCAVP_LN_PIPE(NV)                                                                                                              \
  do {                                                                                                                                 \
    TCAVP_CUDA(cudaFuncSetAttribute(layernorm_pipe_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
    layernorm_pipe_kernel<NV><<<grid_p, lnp::WARPS * 32, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), w, b, out, rows, cols, eps, \
                                                                         out_dtype, remap_gi, remap_go, remap_off, rowvec, cols);      \
  } while (0)
    if (cols <= 512) TCAVP_LN_PIPE(2);
    else if (cols <= 768) TCAVP_LN_PIPE(3);
    else TCAVP_LN_PIPE(4);
#undef TCAVP_LN_PIPE
    return check_launch("layernorm_kernel");
  }
  if (vec && wb_al && cols <= 1024) {
#define TCAVP_LN_REG(G, NV)                                                                                                         \
  do {                                                                                                                              \
    const int rpb = wpb * (32 / G);                                                                                                 \
    layernorm_reg_kernel<G, NV><<<(rows + rpb - 1) / rpb, wpb * 32, 0, stream>>>(x, residual, w, b, out, rows, cols, eps, in_dtype, \
                                                                               out_dtype, remap_gi, remap_go, remap_off, rowvec); \
  } while (0)
    if (cols <= 64) TCAVP_LN_REG(8, 1);
    else if (cols <= 128) TCAVP_LN_REG(16, 1);
    else if (cols <= 256) TCAVP_LN_REG(32, 1);
    else if (cols <= 512) TCAVP_LN_REG(32, 2);
    else if (cols <= 768) TCAVP_LN_REG(32, 3);
    else TCAVP_LN_REG(32, 4);
#undef TCAVP_LN_REG
  } else if (vec)
    layernorm_kernel<true><<<grid, wpb * 32, 0, stream>>>(x, residual, w, b, out, rows, cols, eps, in_dtype, out_dtype, remap_gi, remap_go, remap_off, rowvec);
  else
    layernorm_kernel<false><<<grid, wpb * 32, 0, stream>>>(x, residual, w, b, out, rows, cols, eps, in_dtype, out_dtype, remap_gi, remap_go, remap_off, rowvec);
  return check_launch("layernorm_kernel");
}

extern "C" int tcavp_layernorm_strided(const void* x, int ldx, const float* w, const float* b, void* out, int ldo, int rows, int cols, float eps,
                                       int in_dtype, int out_dtype, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && ldx >= cols && ldo >= cols, "tcavp_layernorm_strided: bad shape rows=%d cols=%d ldx=%d ldo=%d", rows, cols, ldx, ldo);
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && w && b && out, "tcavp_layernorm_strided: null pointer");
  TCAVP_REQUIRE((in_dtype | 1) == 1 && (out_dtype | 1) == 1, "tcavp_layernorm_strided: bad dtype");
  const size_t osz = out_dtype == TCAVP_BF16 ? 2 : 4;
  auto al = [](const void* p, size_t a) { return reinterpret_cast<uintptr_t>(p) % a == 0; };
  if (in_dtype == TCAVP_BF16 && ldx == cols && cols % 8 == 0 && cols >= 256 && cols <= 1024 && al(x, 16) && al(w, 16) && al(b, 16) &&
      al(out, 8 * osz) && ((size_t)ldo * osz) % (8 * osz) == 0) {
    const size_t smem = (size_t)lnp::WARPS * lnp::stages_for(cols) * ((size_t)cols * 2 + 8);
    const int bps = (int)((200u << 10) / smem) > 2 ? 2 : (int)((200u << 10) / smem);
    int grid_p = sm_count() * (bps < 1 ? 1 : bps);
    if (grid_p > (rows + lnp::WARPS - 1) / lnp::WARPS) grid_p = (rows + lnp::WARPS - 1) / lnp::WARPS;
#define TCAVP_LN_PIPE(NV)                                                                                                              \
  do {                                                                                                                                 \
    TCAVP_CUDA(cudaFuncSetAttribute(layernorm_pipe_kernel<NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
    layernorm_pipe_kernel<NV><<<grid_p, lnp::WARPS * 32, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), w, b, out, rows, cols, eps, \
                                                                         out_dtype, 0, 0, 0, nullptr, ldo);                            \
  } while (0)
    if (cols <= 512) TCAVP_LN_PIPE(2);
    else if (cols <= 768) TCAVP_LN_PIPE(3);
    else TCAVP_LN_PIPE(4);
#undef TCAVP_LN_PIPE
    return check_launch("layernorm_kernel");
  }
  layernorm_strided_kernel<<<(rows + 7) / 8, 256, 0, stream>>>(x, ldx, w, b, out, ldo, rows, cols, eps, in_dtype, out_dtype);
  return check_launch("layernorm_kernel");
}

extern "C" int tcavp_row_rstd(const void* x, int ldx, int rows, int cols, float eps, int dtype, float* out, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && ldx >= cols, "tcavp_row_rstd: bad shape rows=%d cols=%d ldx=%d", rows, cols, ldx);
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && out && (dtype | 1) == 1, "tcavp_row_rstd: bad pointer/dtype");
  const int grid = (rows + 7) / 8;
  if (cols % 8 == 0 && aligned_rows(x, ldx, dtype))
    row_rstd_kernel<true><<<grid, 256, 0, stream>>>(x, ldx, rows, cols, eps, dtype, out);
  else
    row_rstd_kernel<false><<<grid, 256, 0, stream>>>(x, ldx, rows, cols, eps, dtype, out);
  return check_launch("row_rstd_kernel");
}

extern "C" int tcavp_rmsnorm(const void* x, int ldi, const float* w, void* out, int rows, int cols, int ldo, float eps, int in_dtype,
                             int out_dtype, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && ldo >= cols && ldi >= cols, "tcavp_rmsnorm: bad shape rows=%d cols=%d ldi=%d ldo=%d", rows, cols, ldi, ldo);
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && w && out, "tcavp_rmsnorm: null pointer");
  TCAVP_REQUIRE((in_dtype | 1) == 1 && (out_dtype | 1) == 1, "tcavp_rmsnorm: bad dtype");
  const bool vec = cols % 8 == 0 && aligned_rows(x, ldi, in_dtype) && aligned_rows(out, ldo, out_dtype);
  const int wpb = 8;
  const int grid = (rows + wpb - 1) / wpb;
  if (vec && cols <= 1024 && reinterpret_cast<uintptr_t>(w) % 16 == 0) {
    if (cols <= 256) rmsnorm_reg_kernel<1><<<grid, wpb * 32, 0, stream>>>(x, w, out, rows, cols, ldi, ldo, eps, in_dtype, out_dtype);
    else if (cols <= 512) rmsnorm_reg_kernel<2><<<grid, wpb * 32, 0, stream>>>(x, w, out, rows, cols, ldi, ldo, eps, in_dtype, out_dtype);
    else if (cols <= 768) rmsnorm_reg_kernel<3><<<grid, wpb * 32, 0, stream>>>(x, w, out, rows, cols, ldi, ldo, eps, in_dtype, out_dtype);
    else rmsnorm_reg_kernel<4><<<grid, wpb * 32, 0, stream>>>(x, w, out, rows, cols, ldi, ldo, eps, in_dtype, out_dtype);
  } else if (vec)
    rmsnorm_kernel<true><<<grid, wpb * 32, 0, stream>>>(x, w, out, rows, cols, ldi, ldo, eps, in_dtype, out_dtype);
  else
    rmsnorm_kernel<false><<<grid, wpb * 32, 0, stream>>>(x, w, out, rows, cols, ldi, ldo, eps, in_dtype, out_dtype);
  return check_launch("rmsnorm_kernel");
}

extern "C" int tcavp_quant_e4m3_rows(const void* x, int ldi, void* q, int ldo, float* f, int rows, int cols, int rms, float eps, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(rows >= 0 && cols >= 16 && cols <= 14336 && cols % 16 == 0 && ldi >= cols && ldo >= cols,
                "tcavp_quant_e4m3_rows: bad shape rows=%d cols=%d ldi=%d ldo=%d (cols %% 16 == 0, 16 <= cols <= 14336)", rows, cols, ldi, ldo);
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && q && f, "tcavp_quant_e4m3_rows: null pointer");
  TCAVP_REQUIRE(ldi % 8 == 0 && ldo % 16 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(q) % 16 == 0,
                "tcavp_quant_e4m3_rows: needs ldi %% 8 == 0, ldo %% 16 == 0 and 16-byte aligned x / q (ldi=%d ldo=%d)", ldi, ldo);
  const size_t smem = (size_t)lnp::WARPS * q8::stages_for(cols) * ((size_t)cols * 2 + 8);
  int bps = (int)((200u << 10) / smem);
  bps = bps < 1 ? 1 : (bps > 4 ? 4 : bps);
  int grid = sm_count() * bps;
  if (grid > (rows + lnp::WARPS - 1) / lnp::WARPS) grid = (rows + lnp::WARPS - 1) / lnp::WARPS;
  TCAVP_CUDA(cudaFuncSetAttribute(quant_e4m3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  quant_e4m3_kernel<<<grid, lnp::WARPS * 32, smem, stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), ldi, reinterpret_cast<uint8_t*>(q), ldo, f,
                                                             rows, cols, rms, eps);
  return check_launch("quant_e4m3_kernel");
}
