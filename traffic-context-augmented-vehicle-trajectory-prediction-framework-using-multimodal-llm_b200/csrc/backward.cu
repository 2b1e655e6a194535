// Backward-pass kernels of the fine-tune step (reference scripts/im_kim_train_GRN.py:1039-1040: loss.backward() +
// AdamW).  The reference leaves all of this to torch autograd; here every gradient is a hand-written kernel behind
// the C ABI.  Dense gradient contractions reuse tcavp_gemm on explicitly transposed operands (tcavp_transpose);
// this file holds the rest: transposes, reductions over rows, the norm / activation / attention / NLinear / head
// backward kernels, the skinny (rank-r) weight-gradient kernel used for LoRA, and the fused AdamW update.
// All arithmetic is fp32; bf16 is a storage type only.
#include "common.cuh"

namespace tcavp {

static int grid_cap(long long blocks, int per_sm) {
  const long long cap = (long long)sm_count() * per_sm;
  return (int)(blocks < 1 ? 1 : (blocks > cap ? cap : blocks));
}

// ------------------------------------------------------------------------------------------------
// transpose: out[b][c][r] = in[b][r][c]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) transpose_kernel(const void* __restrict__ in, long long in_bs, int ldi, int in_dtype,
                                                        void* __restrict__ out, long long out_bs, int ldo, int out_dtype, int rows,
                                                        int cols) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < rows && c < cols) ? load_as_f(in, (size_t)b * in_bs + (size_t)r * ldi + c, in_dtype) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;
    if (c < cols && r < rows) store_from_f(out, (size_t)b * out_bs + (size_t)c * ldo + r, out_dtype, tile[tx][i]);
  }
}

// bf16 -> bf16 form: 64 x 64 tiles, 4-byte (two-element) global accesses on both sides (128 contiguous bytes per warp and tile row;
// the generic kernel moves 2 bytes per thread: 0.8 TB/s on the [B L, 2H] activations the fine-tune step transposes)
__global__ void __launch_bounds__(256) transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in, long long in_bs, int ldi,
                                                             __nv_bfloat16* __restrict__ out, long long out_bs, int ldo, int rows, int cols) {
  __shared__ __nv_bfloat16 tile[64][66];
  const int b = blockIdx.z;
  const int r0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const __nv_bfloat16* ip = in + (size_t)b * in_bs;
  __nv_bfloat16* op = out + (size_t)b * out_bs;
  for (int i = ty; i < 64; i += 8) {
    const int r = r0 + i, c = c0 + 2 * tx;
    __nv_bfloat162 v = __floats2bfloat162_rn(0.f, 0.f);
    if (r < rows && c + 1 < cols) v = *reinterpret_cast<const __nv_bfloat162*>(ip + (size_t)r * ldi + c);
    else if (r < rows && c < cols) v.x = ip[(size_t)r * ldi + c];
    tile[i][2 * tx] = v.x;
    tile[i][2 * tx + 1] = v.y;
  }
  __syncthreads();
  for (int i = ty; i < 64; i += 8) {
    const int c = c0 + i, r = r0 + 2 * tx;
    if (c >= cols) continue;
    if (r + 1 < rows) {
      __nv_bfloat162 v;
      v.x = tile[2 * tx][i];
      v.y = tile[2 * tx + 1][i];
      *reinterpret_cast<__nv_bfloat162*>(op + (size_t)c * ldo + r) = v;
    } else if (r < rows) {
      op[(size_t)c * ldo + r] = tile[2 * tx][i];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// period_sum: out[r % period][c] += x[r][c]   (period 1 = bias gradient; period P = positional-table gradient)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) period_sum_kernel(const void* __restrict__ x, int ldx, int dtype, long long rows, int cols,
                                                         int period, float* __restrict__ out, long long k_per_split) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  const int p = blockIdx.y;
  if (c >= cols) return;
  const long long K = (rows - p + period - 1) / period;   // rows r = p + period * k, k < K
  const long long k0 = (long long)blockIdx.z * k_per_split;
  long long k1 = k0 + k_per_split;
  if (k1 > K) k1 = K;
  float acc = 0.f;
  for (long long k = k0; k < k1; ++k) acc += load_as_f(x, (size_t)(p + period * k) * ldx + c, dtype);
  if (k1 > k0) atomicAdd(out + (size_t)p * cols + c, acc);
}

// ------------------------------------------------------------------------------------------------
// elementwise: relu backward, axpby, SwiGLU forward / backward
// ------------------------------------------------------------------------------------------------
__global__ void relu_bwd_kernel(const void* __restrict__ dy, int lddy, const void* __restrict__ y, int ldy, void* __restrict__ dx, int lddx,
                                int dtype, long long rows, int cols) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i % cols);
    const float g = load_as_f(dy, (size_t)r * lddy + c, dtype);
    store_from_f(dx, (size_t)r * lddx + c, dtype, load_as_f(y, (size_t)r * ldy + c, dtype) > 0.f ? g : 0.f);
  }
}

// HF ACT2FN["gelu_new"] (GPT-2 mlp.act) as a pass of its own, and its backward on the stored pre-activation (the fine-tune step of a
// GPT-2-arch backbone keeps c_fc's output x; the inference path applies the activation in the GEMM epilogue instead).
//   y = 0.5 x (1 + t),  t = tanh(c (x + a x^3));   dy/dx = 0.5 (1 + t) + 0.5 x (1 - t^2) c (1 + 3 a x^2)
// bf16 tensors take the 16-byte path (8 elements per thread, hardware tanh: its 2^-11 relative error is below the output rounding);
// fp32 tensors (the parity mode) use tanhf.
template <bool BWD>
__device__ __forceinline__ float gelu_new_eval(float x, float g, bool approx) {
  const float u = 0.7978845608028654f * fmaf(0.044715f * x * x, x, x);
  float t;
  if (approx) asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  else t = tanhf(u);
  if (!BWD) return 0.5f * x * (1.f + t);
  return g * (0.5f * (1.f + t) + 0.5f * x * (1.f - t * t) * 0.7978845608028654f * fmaf(3.f * 0.044715f * x, x, 1.f));
}
template <bool BWD>
__global__ void __launch_bounds__(256) gelu_new_kernel(const void* __restrict__ dy, int lddy, const void* __restrict__ x, int ldx,
                                                       void* __restrict__ out, int ldo, int dtype, long long rows, int cols, int vec) {
  if (vec) {      // bf16, cols / strides multiples of 8, 16-byte aligned bases
    const int c8 = cols >> 3;
    const long long total = rows * c8;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
      const long long r = i / c8;
      const int c = (int)(i % c8) << 3;
      const uint4 xv = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(x) + (size_t)r * ldx + c);
      uint4 gv = make_uint4(0, 0, 0, 0);
      if (BWD) gv = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(dy) + (size_t)r * lddy + c);
      const uint32_t xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
      uint32_t o[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float lo = gelu_new_eval<BWD>(__uint_as_float(xs[e] << 16), __uint_as_float(gs[e] << 16), true);
        const float hi = gelu_new_eval<BWD>(__uint_as_float(xs[e] & 0xffff0000u), __uint_as_float(gs[e] & 0xffff0000u), true);
        const __nv_bfloat162 pk = __floats2bfloat162_rn(lo, hi);
        o[e] = *reinterpret_cast<const uint32_t*>(&pk);
      }
      *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(out) + (size_t)r * ldo + c) = make_uint4(o[0], o[1], o[2], o[3]);
    }
    return;
  }
  const long long total = rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i % cols);
    const float g = BWD ? load_as_f(dy, (size_t)r * lddy + c, dtype) : 0.f;
    store_from_f(out, (size_t)r * ldo + c, dtype, gelu_new_eval<BWD>(load_as_f(x, (size_t)r * ldx + c, dtype), g, dtype == TCAVP_BF16));
  }
}

__global__ void axpby_kernel(const void* __restrict__ a, int lda, int a_dtype, float alpha, const void* __restrict__ b, int ldb, int b_dtype,
                             float beta, void* __restrict__ out, int ldo, int out_dtype, long long rows, int cols) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i % cols);
    float v = alpha * load_as_f(a, (size_t)r * lda + c, a_dtype);
    if (b) v += beta * load_as_f(b, (size_t)r * ldb + c, b_dtype);
    store_from_f(out, (size_t)r * ldo + c, out_dtype, v);
  }
}

// gu rows are interleaved (g0,u0,g1,u1,...): out[r][j] = silu(g_j) * u_j   (HF:190)
__global__ void swiglu_kernel(const void* __restrict__ gu, void* __restrict__ out, int dtype, long long rows, int I) {
  const long long total = rows * I;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const float g = load_as_f(gu, 2 * (size_t)i, dtype), u = load_as_f(gu, 2 * (size_t)i + 1, dtype);
    store_from_f(out, (size_t)i, dtype, g / (1.f + __expf(-g)) * u);
  }
}
__global__ void swiglu_bwd_kernel(const void* __restrict__ dout, const void* __restrict__ gu, void* __restrict__ dgu, int dtype, long long rows,
                                  int I) {
  const long long total = rows * I;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const float g = load_as_f(gu, 2 * (size_t)i, dtype), u = load_as_f(gu, 2 * (size_t)i + 1, dtype);
    const float d = load_as_f(dout, (size_t)i, dtype);
    const float sg = 1.f / (1.f + __expf(-g));
    store_from_f(dgu, 2 * (size_t)i, dtype, d * u * sg * (1.f + g * (1.f - sg)));
    store_from_f(dgu, 2 * (size_t)i + 1, dtype, d * g * sg);
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward (input was x + res): dx, dw += sum_r dy * xhat, db += sum_r dy.  Warp per row.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const void* __restrict__ dy, int dy_dtype, const void* __restrict__ x,
                                                            const void* __restrict__ res, int x_dtype, const float* __restrict__ w, int rows,
                                                            int cols, float eps, void* __restrict__ dx, int dx_dtype, float* __restrict__ dw,
                                                            float* __restrict__ db) {
  extern __shared__ float sacc[];   // [2][cols]
  float* s_dw = sacc;
  float* s_db = sacc + cols;
  for (int c = threadIdx.x; c < 2 * cols; c += blockDim.x) sacc[c] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    const size_t base = (size_t)row * cols;
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) s += load_as_f(x, base + c, x_dtype) + (res ? load_as_f(res, base + c, x_dtype) : 0.f);
    const float mean = warp_sum(s) / cols;
    float q = 0.f;
    for (int c = lane; c < cols; c += 32) {
      const float v = load_as_f(x, base + c, x_dtype) + (res ? load_as_f(res, base + c, x_dtype) : 0.f) - mean;
      q += v * v;
    }
    const float rstd = rsqrtf(warp_sum(q) / cols + eps);
    float s1 = 0.f, s2 = 0.f;
    for (int c = lane; c < cols; c += 32) {
      const float xh = (load_as_f(x, base + c, x_dtype) + (res ? load_as_f(res, base + c, x_dtype) : 0.f) - mean) * rstd;
      const float d = load_as_f(dy, base + c, dy_dtype);
      const float g = d * __ldg(w + c);
      s1 += g;
      s2 += g * xh;
      if (dw) {
        atomicAdd(s_dw + c, d * xh);
        atomicAdd(s_db + c, d);
      }
    }
    s1 = warp_sum(s1) / cols;
    s2 = warp_sum(s2) / cols;
    if (dx) {
      for (int c = lane; c < cols; c += 32) {
        const float xh = (load_as_f(x, base + c, x_dtype) + (res ? load_as_f(res, base + c, x_dtype) : 0.f) - mean) * rstd;
        const float g = load_as_f(dy, base + c, dy_dtype) * __ldg(w + c);
        store_from_f(dx, base + c, dx_dtype, rstd * (g - s1 - xh * s2));
      }
    }
  }
  __syncthreads();
  if (dw) {
    for (int c = threadIdx.x; c < cols; c += blockDim.x) {
      atomicAdd(dw + c, s_dw[c]);
      atomicAdd(db + c, s_db[c]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// RMSNorm backward.  y = w * (x * rstd)  (w == nullptr: unit weight, the folded-weight form used by the LLM stack):
//   g = dy * w;  dx = rstd * (g - xhat * mean(g * xhat)) + add,   xhat = x * rstd
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rmsnorm_bwd_kernel(const void* __restrict__ dy, int lddy, const void* __restrict__ x, int ldx,
                                                          const float* __restrict__ w, const void* __restrict__ add, int ldadd,
                                                          void* __restrict__ dx, int lddx, int dtype, int rows, int cols, float eps) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    float ss = 0.f;
    for (int c = lane; c < cols; c += 32) {
      const float v = load_as_f(x, (size_t)row * ldx + c, dtype);
      ss += v * v;
    }
    const float rstd = rsqrtf(warp_sum(ss) / cols + eps);
    float dot = 0.f;
    for (int c = lane; c < cols; c += 32) {
      const float g = load_as_f(dy, (size_t)row * lddy + c, dtype) * (w ? __ldg(w + c) : 1.f);
      dot += g * load_as_f(x, (size_t)row * ldx + c, dtype) * rstd;
    }
    dot = warp_sum(dot) / cols;
    for (int c = lane; c < cols; c += 32) {
      const float g = load_as_f(dy, (size_t)row * lddy + c, dtype) * (w ? __ldg(w + c) : 1.f);
      const float xh = load_as_f(x, (size_t)row * ldx + c, dtype) * rstd;
      float v = rstd * (g - xh * dot);
      if (add) v += load_as_f(add, (size_t)row * ldadd + c, dtype);
      store_from_f(dx, (size_t)row * lddx + c, dtype, v);
    }
  }
}

// Vectorised bf16 variant: 16-byte accesses, one warp per row; NV > 0 keeps the row (x and dy, NV 8-element vectors per lane)
// in registers so both are read exactly once, NV == 0 streams wider rows three times (the re-reads hit L1).
__device__ __forceinline__ void ld8_bf16(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    v[2 * e] = __uint_as_float(w[e] << 16);
    v[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u);
  }
}
__device__ __forceinline__ void st8_bf16(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 u;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
  for (int e = 0; e < 4; ++e) h[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
  *reinterpret_cast<uint4*>(p) = u;
}

template <int NV>
__global__ void __launch_bounds__(256) rmsnorm_bwd_vec_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, const __nv_bfloat16* __restrict__ x,
                                                              int ldx, const float* __restrict__ w, const __nv_bfloat16* __restrict__ add,
                                                              int ldadd, __nv_bfloat16* __restrict__ dx, int lddx, int rows, int cols, float eps) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    const __nv_bfloat16* xr = x + (size_t)row * ldx;
    const __nv_bfloat16* gr = dy + (size_t)row * lddy;
    float xv[NV > 0 ? NV : 1][8], gv[NV > 0 ? NV : 1][8];
    float ss = 0.f, dot = 0.f;
    if (NV > 0) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (i * 32 + lane) * 8;
        if (c < cols) {
          ld8_bf16(xr + c, xv[i]);
          ld8_bf16(gr + c, gv[i]);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            if (w) gv[i][e] *= __ldg(w + c + e);
            ss += xv[i][e] * xv[i][e];
            dot += gv[i][e] * xv[i][e];
          }
        }
      }
    } else {
      for (int c = lane * 8; c < cols; c += 256) {
        float a[8], g[8];
        ld8_bf16(xr + c, a);
        ld8_bf16(gr + c, g);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          ss += a[e] * a[e];
          dot += g[e] * (w ? __ldg(w + c + e) : 1.f) * a[e];
        }
      }
    }
    const float rstd = rsqrtf(warp_sum(ss) / cols + eps);
    dot = warp_sum(dot) * rstd / cols;          // mean(g * xhat)
    if (NV > 0) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = (i * 32 + lane) * 8;
        if (c < cols) {
          float o[8], ad[8];
          if (add) ld8_bf16(add + (size_t)row * ldadd + c, ad);
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = rstd * (gv[i][e] - xv[i][e] * rstd * dot) + (add ? ad[e] : 0.f);
          st8_bf16(dx + (size_t)row * lddx + c, o);
        }
      }
    } else {
      for (int c = lane * 8; c < cols; c += 256) {
        float a[8], g[8], o[8], ad[8];
        ld8_bf16(xr + c, a);
        ld8_bf16(gr + c, g);
        if (add) ld8_bf16(add + (size_t)row * ldadd + c, ad);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = rstd * (g[e] * (w ? __ldg(w + c + e) : 1.f) - a[e] * rstd * dot) + (add ? ad[e] : 0.f);
        st8_bf16(dx + (size_t)row * lddx + c, o);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Rotary embedding on ADJACENT column pairs (the layout tcavp_gemm's fused RoPE produces), forward or inverse.
// Table layout 1: [dh/4][L] x float4 = (cos, sin) of pairs (2k, 2k+1).
// ------------------------------------------------------------------------------------------------
__global__ void rope_adjacent_kernel(void* __restrict__ buf, int dtype, long long rows, int L, int ld, int cols, int dh,
                                     const float* __restrict__ table, int inverse) {
  const int quads = cols >> 2;
  const long long total = rows * quads;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / quads;
    const int c = (int)(i % quads) * 4;
    const int pos = (int)(r % L);
    const float4 t = __ldg(reinterpret_cast<const float4*>(table) + (size_t)((c % dh) >> 2) * L + pos);
    const float sg = inverse ? -1.f : 1.f;
    const size_t o = (size_t)r * ld + c;
    const float a0 = load_as_f(buf, o, dtype), a1 = load_as_f(buf, o + 1, dtype), a2 = load_as_f(buf, o + 2, dtype),
                a3 = load_as_f(buf, o + 3, dtype);
    store_from_f(buf, o, dtype, a0 * t.x - sg * a1 * t.y);
    store_from_f(buf, o + 1, dtype, a1 * t.x + sg * a0 * t.y);
    store_from_f(buf, o + 2, dtype, a2 * t.z - sg * a3 * t.w);
    store_from_f(buf, o + 3, dtype, a3 * t.z + sg * a2 * t.w);
  }
}

// ------------------------------------------------------------------------------------------------
// copy_rows: out[remap_out(r), :] = in[remap_in(r), :]  with dtype conversion (scatter into / gather from the fused
// (B, L, H) sequence buffer; reference scripts/train.py:528 torch.cat and its backward split)
// ------------------------------------------------------------------------------------------------
__global__ void copy_rows_kernel(const void* __restrict__ in, int ldi, int in_dtype, int igi, int igo, int ioff, void* __restrict__ out, int ldo,
                                 int out_dtype, int ogi, int ogo, int ooff, long long rows, int cols) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const size_t ri = (size_t)remap_row(igi, igo, ioff, r), ro = (size_t)remap_row(ogi, ogo, ooff, r);
    store_from_f(out, ro * ldo + c, out_dtype, load_as_f(in, ri * ldi + c, in_dtype));
  }
}

// ------------------------------------------------------------------------------------------------
// masked mean backward (reference scripts/train.py:373-382): dx[b,p,:] = p < len[b] ? dout[b,:] / len[b] : 0
// ------------------------------------------------------------------------------------------------
__global__ void masked_mean_bwd_kernel(const void* __restrict__ dout, int dout_dtype, const int32_t* __restrict__ len, void* __restrict__ dx,
                                       int dx_dtype, int B, int P, int D) {
  const long long total = (long long)B * P * D;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const long long bp = i / D;
    const int p = (int)(bp % P), b = (int)(bp / P);
    int n = __ldg(len + b);
    n = n < 0 ? 0 : (n > P ? P : n);
    store_from_f(dx, (size_t)i, dx_dtype, p < n ? load_as_f(dout, (size_t)b * D + d, dout_dtype) / (float)n : 0.f);
  }
}

// ------------------------------------------------------------------------------------------------
// NLinear backward (reference scripts/train.py:701-716 / 769-785):
//   out[b,t,c] = sum_s W[t][s][c] * (in[b,s,c] - in[b,T_in-1,c]) + bias[t][c] + in[b,T_in-1,c]
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) nlinear_bwd_in_kernel(const void* __restrict__ g, int g_dtype, const float* __restrict__ w,
                                                             void* __restrict__ din, int din_dtype, int B, int C, int T_in, int T_out) {
  const long long total = (long long)B * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long b = i / C;
    float sum_g = 0.f, sum_du = 0.f, du_last = 0.f;
    for (int t = 0; t < T_out; ++t) sum_g += load_as_f(g, ((size_t)b * T_out + t) * C + c, g_dtype);
    for (int s = 0; s < T_in; ++s) {
      float du = 0.f;
      for (int t = 0; t < T_out; ++t)
        du = fmaf(load_as_f(g, ((size_t)b * T_out + t) * C + c, g_dtype), __ldg(w + ((size_t)t * T_in + s) * C + c), du);
      sum_du += du;
      if (s < T_in - 1) store_from_f(din, ((size_t)b * T_in + s) * C + c, din_dtype, du);
      else du_last = du;
    }
    store_from_f(din, ((size_t)b * T_in + T_in - 1) * C + c, din_dtype, du_last + sum_g - sum_du);
  }
}

// dW[t][s][c] += sum_b g[b,t,c] * (in[b,s,c] - in[b,T_in-1,c]);  grid (T_out*T_in, splits), block = (256/C) b-lanes x C
__global__ void __launch_bounds__(256) nlinear_bwd_w_kernel(const void* __restrict__ g, int g_dtype, const void* __restrict__ in, int in_dtype,
                                                            float* __restrict__ dw, int B, int C, int T_in, int T_out, int b_per_split) {
  const int t = blockIdx.x / T_in, s = blockIdx.x % T_in;
  const int c = threadIdx.x % C, bl = threadIdx.x / C, nb = blockDim.x / C;
  if (bl >= nb) return;
  const int b0 = blockIdx.y * b_per_split;
  int b1 = b0 + b_per_split;
  if (b1 > B) b1 = B;
  float acc = 0.f;
  for (int b = b0 + bl; b < b1; b += nb) {
    const float u = load_as_f(in, ((size_t)b * T_in + s) * C + c, in_dtype) - load_as_f(in, ((size_t)b * T_in + T_in - 1) * C + c, in_dtype);
    acc = fmaf(load_as_f(g, ((size_t)b * T_out + t) * C + c, g_dtype), u, acc);
  }
  atomicAdd(dw + ((size_t)t * T_in + s) * C + c, acc);
}

// ------------------------------------------------------------------------------------------------
// head: decoded[b,f,t] = o[b,t,f] + x[b,f,T_in-1]  (reference scripts/train.py:941-943) and the loss gradient
//   d_o[b,t,f] = gscale * 2 * (decoded - y) * range_f^2 / (B * T_out)       (reference scripts/train.py:945-962)
// ------------------------------------------------------------------------------------------------
__global__ void head_assemble_kernel(const float* __restrict__ o, const float* __restrict__ x, float* __restrict__ decoded, int B, int T_in,
                                     int T_out) {
  const long long total = (long long)B * 2 * T_out;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i % T_out);
    const long long bf = i / T_out;
    const int f = (int)(bf % 2);
    const long long b = bf / 2;
    decoded[i] = o[((size_t)b * T_out + t) * 2 + f] + x[(size_t)bf * T_in + T_in - 1];
  }
}
__global__ void traj_loss_bwd_kernel(const float* __restrict__ decoded, const float* __restrict__ y, const float* __restrict__ norm_stat,
                                     const float* __restrict__ gscale, float* __restrict__ d_o, int B, int T_out) {
  const long long total = (long long)B * 2 * T_out;
  const float gs = gscale ? __ldg(gscale) : 1.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i % T_out);
    const long long bf = i / T_out;
    const int f = (int)(bf % 2);
    const long long b = bf / 2;
    const float range = norm_stat[b * 4 + 2 * f + 1] - norm_stat[b * 4 + 2 * f];
    d_o[((size_t)b * T_out + t) * 2 + f] = gs * 2.f * (decoded[i] - y[i]) * range * range / ((float)B * (float)T_out);
  }
}

// ------------------------------------------------------------------------------------------------
// Skinny weight gradient (LoRA A / B): out[n][j] += sum_m scale[m] * Y[m][n] * Z[m][j],  J <= 32.
// One thread per output column n (coalesced reads of Y), Z rows staged in shared memory, atomics at the end.
// ------------------------------------------------------------------------------------------------
template <int J>
__global__ void __launch_bounds__(128) skinny_dw_kernel(const void* __restrict__ Y, int ldy, int y_dtype, const void* __restrict__ Z, int ldz,
                                                        int z_dtype, const float* __restrict__ scale, float* __restrict__ out, int ldo,
                                                        long long M, int N, int jn, int m_per_block) {
  constexpr int MB = 32;
  __shared__ float sz[MB][J];
  const int n = blockIdx.x * 128 + threadIdx.x;
  const long long m0 = (long long)blockIdx.y * m_per_block;
  long long m1 = m0 + m_per_block;
  if (m1 > M) m1 = M;
  float acc[J];
#pragma unroll
  for (int j = 0; j < J; ++j) acc[j] = 0.f;
  for (long long mb = m0; mb < m1; mb += MB) {
    __syncthreads();
    for (int e = threadIdx.x; e < MB * J; e += 128) {
      const int r = e / J, j = e % J;
      const long long m = mb + r;
      float v = 0.f;
      if (m < m1 && j < jn) v = load_as_f(Z, (size_t)m * ldz + j, z_dtype) * (scale ? __ldg(scale + m) : 1.f);
      sz[r][j] = v;
    }
    __syncthreads();
    if (n < N) {
      const int lim = (int)((m1 - mb) < MB ? (m1 - mb) : MB);
      for (int r = 0; r < lim; ++r) {
        const float y = load_as_f(Y, (size_t)(mb + r) * ldy + n, y_dtype);
#pragma unroll
        for (int j = 0; j < J; ++j) acc[j] = fmaf(y, sz[r][j], acc[j]);
      }
    }
  }
  if (n < N) {
#pragma unroll
    for (int j = 0; j < J; ++j)
      if (j < jn) atomicAdd(out + (size_t)n * ldo + j, acc[j]);
  }
}

// ------------------------------------------------------------------------------------------------
// Weight gradient of a linear map without operand transposes: out[n][k] += sum_m dY[m][n] * X[m][k]   (fp32 FFMA).
// Both operands are read in their natural row-major [M, *] layout (rows of dY / X are coalesced over n / k), a CTA owns a
// 64 x 64 output tile and one slice of the M rows (grid.z splits M so small outputs still fill the GPU), partial tiles are
// combined with fp32 atomics into the zero-initialised output.  Used for the fp32 temporal / fusion / polygon layers, whose
// outputs are at most a few hundred rows wide while M = scenes x positions is large.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dw_simt_kernel(const void* __restrict__ dY, int lddy, int dy_dtype, const void* __restrict__ X, int ldx,
                                                      int x_dtype, float* __restrict__ out, int ldo, long long M, int N, int K, int m_per_block) {
  constexpr int T = 64, MB = 16;
  __shared__ float sy[MB][T + 4];
  __shared__ float sx[MB][T + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int n0 = blockIdx.y * T, k0 = blockIdx.x * T;
  const long long m0 = (long long)blockIdx.z * m_per_block;
  long long m1 = m0 + m_per_block;
  if (m1 > M) m1 = M;
  float acc[4][4] = {};
  for (long long mb = m0; mb < m1; mb += MB) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = threadIdx.x + i * 256;     // 0..1023
      const int r = e >> 6, c = e & 63;        // row of the M slice, column of the tile (consecutive lanes -> consecutive columns)
      const long long m = mb + r;
      sy[r][c] = (m < m1 && n0 + c < N) ? load_as_f(dY, (size_t)m * lddy + n0 + c, dy_dtype) : 0.f;
      sx[r][c] = (m < m1 && k0 + c < K) ? load_as_f(X, (size_t)m * ldx + k0 + c, x_dtype) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < MB; ++r) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sy[r][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = sx[r][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k < K) {
        if (gridDim.z == 1) out[(size_t)n * ldo + k] += acc[i][j];
        else atomicAdd(out + (size_t)n * ldo + k, acc[i][j]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Attention backward.  One CTA per (batch, head, 16-query block); probabilities are recomputed (no saved
// statistics), head_dim is streamed in chunks so any width works (LTSF cross-attention: dh = H/2).
//   P = softmax(scale * Q K^T + mask);  dP = dO V^T;  D_i = sum_j P_ij dP_ij;  dS = scale * P o (dP - D)
//   dQ = dS K (owned rows, plain stores);  dK += dS^T Q;  dV += P^T dO  (fp32 atomics: q-blocks and GQA groups share keys)
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// LayerNorm backward for a FROZEN LayerNorm (GPT-2-arch backbone under peft: ln_1 / ln_2 / ln_f get no gradient): dx only, with the
// gradient of the residual branch added in the same pass.   g = dy * w;  dx = rstd * (g - mean(g) - xhat * mean(g * xhat)) + add
// bf16 rows up to 1024 columns live in registers (one 16-byte load per 8 elements, x and dy read once); anything else takes the
// generic warp-per-row loop.
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) layernorm_bwd_dx_vec_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, const __nv_bfloat16* __restrict__ x,
                                                                   int ldx, const float* __restrict__ w, const __nv_bfloat16* __restrict__ add,
                                                                   int ldadd, __nv_bfloat16* __restrict__ dx, int lddx, int rows, int cols, float eps) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    const __nv_bfloat16* xr = x + (size_t)row * ldx;
    const __nv_bfloat16* gr = dy + (size_t)row * lddy;
    float xv[NV][8], gv[NV][8];
    float s = 0.f, sg = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
        ld8_bf16(xr + c, xv[i]);
        ld8_bf16(gr + c, gv[i]);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          gv[i][e] *= __ldg(w + c + e);
          s += xv[i][e];
          sg += gv[i][e];
        }
      }
    }
    const float mean = warp_sum(s) / cols;
    float q = 0.f, dot = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          xv[i][e] -= mean;
          q += xv[i][e] * xv[i][e];
          dot += gv[i][e] * xv[i][e];
        }
      }
    }
    const float rstd = rsqrtf(warp_sum(q) / cols + eps);
    const float s1 = warp_sum(sg) / cols;                    // mean(g)
    const float s2 = warp_sum(dot) * rstd / cols;            // mean(g * xhat)
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
        float o[8], ad[8];
        if (add) ld8_bf16(add + (size_t)row * ldadd + c, ad);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = rstd * (gv[i][e] - s1 - xv[i][e] * rstd * s2) + (add ? ad[e] : 0.f);
        st8_bf16(dx + (size_t)row * lddx + c, o);
      }
    }
  }
}

__global__ void __launch_bounds__(256) layernorm_bwd_dx_kernel(const void* __restrict__ dy, int lddy, const void* __restrict__ x, int ldx,
                                                               const float* __restrict__ w, const void* __restrict__ add, int ldadd,
                                                               void* __restrict__ dx, int lddx, int dtype, int rows, int cols, float eps) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += gridDim.x * wpb) {
    float s = 0.f;
    for (int c = lane; c < cols; c += 32) s += load_as_f(x, (size_t)row * ldx + c, dtype);
    const float mean = warp_sum(s) / cols;
    float q = 0.f, sg = 0.f, dot = 0.f;
    for (int c = lane; c < cols; c += 32) {
      const float v = load_as_f(x, (size_t)row * ldx + c, dtype) - mean;
      const float g = load_as_f(dy, (size_t)row * lddy + c, dtype) * __ldg(w + c);
      q += v * v;
      sg += g;
      dot += g * v;
    }
    const float rstd = rsqrtf(warp_sum(q) / cols + eps);
    const float s1 = warp_sum(sg) / cols, s2 = warp_sum(dot) * rstd / cols;
    for (int c = lane; c < cols; c += 32) {
      const float xh = (load_as_f(x, (size_t)row * ldx + c, dtype) - mean) * rstd;
      const float g = load_as_f(dy, (size_t)row * lddy + c, dtype) * __ldg(w + c);
      store_from_f(dx, (size_t)row * lddx + c, dtype, rstd * (g - s1 - xh * s2) + (add ? load_as_f(add, (size_t)row * ldadd + c, dtype) : 0.f));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// RMSNorm / frozen-LayerNorm backward over a long bf16 token stream, rows staged through shared memory by the bulk-copy engine (the
// scheme of layernorm_pipe_kernel in norm.cu): every warp owns a three-deep ring of (x, dy[, add]) row triples filled by cp.async.bulk
// + mbarrier complete_tx, so the bytes in flight per SM are the rings of 16 resident warps (~220 KB) instead of what the registers of
// the *_vec kernels hold (~70 KB: they were latency-bound at 2.8 TB/s).  Same formulas as rmsnorm_bwd_vec_kernel /
// layernorm_bwd_dx_vec_kernel.
// ------------------------------------------------------------------------------------------------
namespace nbp {
constexpr int STAGES = 3, WARPS = 8;      // ~100 registers per thread: two blocks per SM, 2 x 8 x 3 row triples in flight
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
__device__ __forceinline__ void lds8_bf16(uint32_t addr, float (&v)[8]) {
  uint32_t q[4];
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(q[0]), "=r"(q[1]), "=r"(q[2]), "=r"(q[3]) : "r"(addr));
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    v[2 * e] = __uint_as_float(q[e] << 16);
    v[2 * e + 1] = __uint_as_float(q[e] & 0xffff0000u);
  }
}
}  // namespace nbp

template <int NV, bool LN>
__global__ void __launch_bounds__(nbp::WARPS * 32) norm_bwd_pipe_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, const __nv_bfloat16* __restrict__ x,
                                                                       int ldx, const float* __restrict__ w, const __nv_bfloat16* __restrict__ add,
                                                                       int ldadd, __nv_bfloat16* __restrict__ dx, int lddx, int rows, int cols, float eps) {
  using namespace nbp;
  extern __shared__ __align__(128) uint8_t nb_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t row_bytes = (uint32_t)cols * 2u;
  const uint32_t n_in = add ? 3u : 2u;
  const uint32_t stage_bytes = 3u * row_bytes;
  const uint32_t ring = smem_u32(nb_smem) + (uint32_t)warp * STAGES * stage_bytes;
  const uint32_t bars = smem_u32(nb_smem) + (uint32_t)WARPS * STAGES * stage_bytes + (uint32_t)warp * STAGES * 8u;
  const int wstride = gridDim.x * WARPS;
  const int row0 = blockIdx.x * WARPS + warp;
  auto issue = [&](long long r, int s) {      // lane 0 only
    const uint32_t dst = ring + s * stage_bytes, bar = bars + 8 * s;
    mbar_expect_tx(bar, n_in * row_bytes);
    bulk_load(dst, x + (size_t)r * ldx, row_bytes, bar);
    bulk_load(dst + row_bytes, dy + (size_t)r * lddy, row_bytes, bar);
    if (add) bulk_load(dst + 2 * row_bytes, add + (size_t)r * ldadd, row_bytes, bar);
  };
  if (lane == 0) {
    for (int s = 0; s < STAGES; ++s) mbar_init(bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int s = 0; s < STAGES; ++s) {
      const long long r = (long long)row0 + (long long)s * wstride;
      if (r < rows) issue(r, s);
    }
  }
  __syncwarp();
  // LayerNorm: this lane's slice of the weight lives in registers for the whole kernel (per-row loads made the kernel L1TEX-bound)
  float wr[LN ? NV : 1][8];
  if (LN) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
#pragma unroll
      for (int e = 0; e < 8; ++e) wr[LN ? i : 0][e] = c < cols ? __ldg(w + c + e) : 0.f;
    }
  }
  int stage = 0;
  uint32_t phase = 0;
  for (long long row = row0; row < rows; row += wstride) {
    mbar_wait(bars + 8 * stage, phase);
    const uint32_t sx = ring + stage * stage_bytes, sg = sx + row_bytes, sa = sg + row_bytes;
    float xv[NV][8], gv[NV][8];
    float a0 = 0.f, a1 = 0.f;      // RMSNorm: sum x^2, sum g x;   LayerNorm: sum x, sum g
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
        lds8_bf16(sx + c * 2, xv[i]);
        lds8_bf16(sg + c * 2, gv[i]);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          if (LN) gv[i][e] *= wr[LN ? i : 0][e];
          else if (w) gv[i][e] *= __ldg(w + c + e);
          if (LN) {
            a0 += xv[i][e];
            a1 += gv[i][e];
          } else {
            a0 += xv[i][e] * xv[i][e];
            a1 += gv[i][e] * xv[i][e];
          }
        }
      }
    }
    a0 = warp_sum(a0);
    a1 = warp_sum(a1);
    float rstd, s1 = 0.f, s2;
    if (LN) {
      const float mean = a0 / cols;
      float q = 0.f, dot = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        if ((i * 32 + lane) * 8 < cols) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            xv[i][e] -= mean;
            q += xv[i][e] * xv[i][e];
            dot += gv[i][e] * xv[i][e];
          }
        }
      }
      rstd = rsqrtf(warp_sum(q) / cols + eps);
      s1 = a1 / cols;
      s2 = warp_sum(dot) * rstd / cols;
    } else {
      rstd = rsqrtf(a0 / cols + eps);
      s2 = a1 * rstd / cols;
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = (i * 32 + lane) * 8;
      if (c < cols) {
        float o[8], ad[8];
        if (add) lds8_bf16(sa + c * 2, ad);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = rstd * (gv[i][e] - s1 - xv[i][e] * rstd * s2) + (add ? ad[e] : 0.f);
        st8_bf16(dx + (size_t)row * lddx + c, o);
      }
    }
    __syncwarp();                 // every lane has read its part of the stage: hand it back to the copy engine
    if (lane == 0) {
      const long long nxt = row + (long long)STAGES * wstride;
      if (nxt < rows) issue(nxt, stage);
    }
    if (++stage == STAGES) { stage = 0; phase ^= 1; }
  }
}

// host side: 1 = launched, 0 = not eligible
template <bool LN>
static int norm_bwd_pipe_launch(const void* dy, int lddy, const void* x, int ldx, const float* w, const void* add, int ldadd, void* dx, int lddx,
                                int dtype, int rows, int cols, float eps, cudaStream_t stream) {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("TCAVP_NORM_BWD_PIPE");
    on = e ? atoi(e) : 1;
  }
  auto al = [](const void* p, int ld) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % 16 == 0 && ld % 8 == 0); };
  if (!on || dtype != TCAVP_BF16 || cols % 8 || cols < 256 || cols > 1024 || rows < 32768 || !al(dy, lddy) || !al(x, ldx) || !al(add, ldadd) ||
      !al(dx, lddx) || (LN && !w))
    return 0;
  const size_t smem = (size_t)nbp::WARPS * nbp::STAGES * ((size_t)cols * 6 + 8);
  int bps = (int)((220u << 10) / (smem + 1024));
  bps = bps > 2 ? 2 : (bps < 1 ? 1 : bps);
  int grid = sm_count() * bps;
  if (grid > (rows + nbp::WARPS - 1) / nbp::WARPS) grid = (rows + nbp::WARPS - 1) / nbp::WARPS;
  const __nv_bfloat16* dyb = reinterpret_cast<const __nv_bfloat16*>(dy);
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* ab = reinterpret_cast<const __nv_bfloat16*>(add);
  __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(dx);
#define TCAVP_NBP(NV)                                                                                                            \
  do {                                                                                                                           \
    if (cudaFuncSetAttribute(norm_bwd_pipe_kernel<NV, LN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0; \
    norm_bwd_pipe_kernel<NV, LN><<<grid, nbp::WARPS * 32, smem, stream>>>(dyb, lddy, xb, ldx, w, ab, ldadd, ob, lddx, rows, cols, eps);       \
  } while (0)
  if (cols <= 512) TCAVP_NBP(2);
  else if (cols <= 768) TCAVP_NBP(3);
  else TCAVP_NBP(4);
#undef TCAVP_NBP
  return 1;
}

namespace ab {
constexpr int QB = 16;
constexpr int THREADS = 256;
constexpr int JJ = 3;          // keys per thread in the score phase: Tk <= JJ * THREADS

template <typename T>
__global__ void __launch_bounds__(THREADS) attn_bwd_kernel(tcavp_attn_args a, const T* __restrict__ dout, long long do_sb, long long do_st,
                                                           T* __restrict__ dq, long long dq_sb, long long dq_st, float* __restrict__ dk,
                                                           long long dk_sb, long long dk_st, float* __restrict__ dv, long long dv_sb,
                                                           long long dv_st, int DC) {
  extern __shared__ float sm[];
  const int Tk = a.Tk, LD = DC + 1;
  float* sP = sm;                       // [QB][Tk]   probabilities, later unchanged
  float* sdS = sP + QB * Tk;            // [QB][Tk]   dP, then dS
  float* sQ = sdS + QB * Tk;            // [QB][LD]
  float* sdO = sQ + QB * LD;            // [QB][LD]
  float* sK = sdO + QB * LD;            // [Tk][LD]
  float* sV = sK + (size_t)Tk * LD;     // [Tk][LD]
  const int nqb = (a.Tq + QB - 1) / QB;
  const int qb = blockIdx.x % nqb;
  const int bh = blockIdx.x / nqb;
  const int b = bh / a.H, h = bh % a.H, hk = h / (a.H / a.Hkv);
  const int q0 = qb * QB;
  const int tid = threadIdx.x;
  const T* gq = reinterpret_cast<const T*>(a.q) + (size_t)b * a.q_sb + (size_t)h * a.dh;
  const T* gk = reinterpret_cast<const T*>(a.k) + (size_t)b * a.k_sb + (size_t)hk * a.dh;
  const T* gv = reinterpret_cast<const T*>(a.v) + (size_t)b * a.v_sb + (size_t)hk * a.dh;
  const T* gdo = dout + (size_t)b * do_sb + (size_t)h * a.dh;

  // ---- phase A: S = Q K^T and dP = dO V^T, accumulated over head-dim chunks ----
  float accS[JJ][QB], accP[JJ][QB];
#pragma unroll
  for (int jj = 0; jj < JJ; ++jj)
#pragma unroll
    for (int i = 0; i < QB; ++i) accS[jj][i] = accP[jj][i] = 0.f;
  for (int d0 = 0; d0 < a.dh; d0 += DC) {
    const int dc = min(DC, a.dh - d0);
    __syncthreads();
    for (int e = tid; e < QB * DC; e += THREADS) {
      const int i = e / DC, d = e % DC;
      const bool ok = (q0 + i < a.Tq) && d < dc;
      sQ[i * LD + d] = ok ? Cvt<T>::to_f(gq[(size_t)(q0 + i) * a.q_st + d0 + d]) : 0.f;
      sdO[i * LD + d] = ok ? Cvt<T>::to_f(gdo[(size_t)(q0 + i) * do_st + d0 + d]) : 0.f;
    }
    for (int e = tid; e < Tk * DC; e += THREADS) {
      const int j = e / DC, d = e % DC;
      const bool ok = d < dc;
      sK[j * LD + d] = ok ? Cvt<T>::to_f(gk[(size_t)j * a.k_st + d0 + d]) : 0.f;
      sV[j * LD + d] = ok ? Cvt<T>::to_f(gv[(size_t)j * a.v_st + d0 + d]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int jj = 0; jj < JJ; ++jj) {
      const int j = tid + jj * THREADS;
      if (j < Tk) {
        for (int d = 0; d < dc; ++d) {
          const float kv = sK[j * LD + d], vv = sV[j * LD + d];
#pragma unroll
          for (int i = 0; i < QB; ++i) {
            accS[jj][i] = fmaf(sQ[i * LD + d], kv, accS[jj][i]);
            accP[jj][i] = fmaf(sdO[i * LD + d], vv, accP[jj][i]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int jj = 0; jj < JJ; ++jj) {
    const int j = tid + jj * THREADS;
    if (j < Tk) {
      const bool okj = !a.key_mask || a.key_mask[(size_t)b * Tk + j] != 0;
#pragma unroll
      for (int i = 0; i < QB; ++i) {
        const bool ok = okj && (q0 + i < a.Tq) && (!a.causal || j <= q0 + i);
        sP[i * Tk + j] = ok ? accS[jj][i] * a.scale : -INFINITY;
        sdS[i * Tk + j] = accP[jj][i];
      }
    }
  }
  __syncthreads();
  // ---- phase B: softmax rows and dS (warp per row) ----
  {
    const int warp = tid >> 5, lane = tid & 31;
    for (int i = warp; i < QB; i += THREADS / 32) {
      float mx = -INFINITY;
      for (int j = lane; j < Tk; j += 32) mx = fmaxf(mx, sP[i * Tk + j]);
      mx = warp_max(mx);
      float l = 0.f;
      for (int j = lane; j < Tk; j += 32) {
        const float p = mx == -INFINITY ? 0.f : __expf(sP[i * Tk + j] - mx);
        sP[i * Tk + j] = p;
        l += p;
      }
      l = warp_sum(l);
      const float inv = l > 0.f ? 1.f / l : 0.f;
      float dsum = 0.f;
      if (a.drop_thresh == 0) {
        for (int j = lane; j < Tk; j += 32) {
          const float p = sP[i * Tk + j] * inv;
          sP[i * Tk + j] = p;
          dsum += p * sdS[i * Tk + j];
        }
        dsum = warp_sum(dsum);
        for (int j = lane; j < Tk; j += 32) sdS[i * Tk + j] = a.scale * sP[i * Tk + j] * (sdS[i * Tk + j] - dsum);
      } else {
        // O = P_d V with P_d = keep ? P / (1 - p_drop) : 0:  dP = mask-scaled (dO V^T),  D = sum_j P dP,  dS = scale P (dP - D),
        // and dV uses P_d (kept in sP for phase C)
        const uint32_t dkey = drop_key(a.drop_seed, a.drop_site);
        const unsigned long long drow = ((unsigned long long)bh * a.Tq + (unsigned)(q0 + i)) * (unsigned long long)Tk;
        for (int j = lane; j < Tk; j += 32) {
          const float p = sP[i * Tk + j] * inv;
          const float f = (q0 + i < a.Tq && drop_keep(dkey, drow + (unsigned)j, a.drop_thresh)) ? a.drop_scale : 0.f;
          const float dp = f * sdS[i * Tk + j];
          dsum += p * dp;
          sdS[i * Tk + j] = dp;
          sP[i * Tk + j] = p;
        }
        dsum = warp_sum(dsum);
        for (int j = lane; j < Tk; j += 32) {
          const float p = sP[i * Tk + j];
          const float f = (q0 + i < a.Tq && drop_keep(dkey, drow + (unsigned)j, a.drop_thresh)) ? a.drop_scale : 0.f;
          sdS[i * Tk + j] = a.scale * p * (sdS[i * Tk + j] - dsum);
          sP[i * Tk + j] = p * f;
        }
      }
    }
  }
  // ---- phase C: dQ, dK, dV per head-dim chunk ----
  T* gdq = dq + (size_t)b * dq_sb + (size_t)h * a.dh;
  float* gdk = dk + (size_t)b * dk_sb + (size_t)hk * a.dh;
  float* gdv = dv + (size_t)b * dv_sb + (size_t)hk * a.dh;
  for (int d0 = 0; d0 < a.dh; d0 += DC) {
    const int dc = min(DC, a.dh - d0);
    __syncthreads();
    for (int e = tid; e < QB * DC; e += THREADS) {
      const int i = e / DC, d = e % DC;
      const bool ok = (q0 + i < a.Tq) && d < dc;
      sQ[i * LD + d] = ok ? Cvt<T>::to_f(gq[(size_t)(q0 + i) * a.q_st + d0 + d]) : 0.f;
      sdO[i * LD + d] = ok ? Cvt<T>::to_f(gdo[(size_t)(q0 + i) * do_st + d0 + d]) : 0.f;
    }
    for (int e = tid; e < Tk * DC; e += THREADS) {
      const int j = e / DC, d = e % DC;
      sK[j * LD + d] = d < dc ? Cvt<T>::to_f(gk[(size_t)j * a.k_st + d0 + d]) : 0.f;
    }
    __syncthreads();
    for (int e = tid; e < QB * DC; e += THREADS) {     // dQ[i][d] = sum_j dS[i][j] K[j][d]
      const int i = e / DC, d = e % DC;
      if (q0 + i < a.Tq && d < dc) {
        float acc = 0.f;
        for (int j = 0; j < Tk; ++j) acc = fmaf(sdS[i * Tk + j], sK[j * LD + d], acc);
        gdq[(size_t)(q0 + i) * dq_st + d0 + d] = Cvt<T>::from_f(acc);
      }
    }
    for (int e = tid; e < Tk * DC; e += THREADS) {     // dK[j][d] += sum_i dS[i][j] Q[i][d];  dV[j][d] += sum_i P[i][j] dO[i][d]
      const int j = e / DC, d = e % DC;
      if (d < dc) {
        float ak = 0.f, av = 0.f;
#pragma unroll
        for (int i = 0; i < QB; ++i) {
          ak = fmaf(sdS[i * Tk + j], sQ[i * LD + d], ak);
          av = fmaf(sP[i * Tk + j], sdO[i * LD + d], av);
        }
        atomicAdd(gdk + (size_t)j * dk_st + d0 + d, ak);
        atomicAdd(gdv + (size_t)j * dv_st + d0 + d, av);
      }
    }
  }
}
}  // namespace ab

int attention_x_bwd_launch(const tcavp_attn_args& a, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb, long long dq_st,
                           void* dk, long long dk_sb, long long dk_st, void* dv, long long dv_sb, long long dv_st, int dkv_dtype, cudaStream_t stream);
int dw_tc_launch(const void* Y, int ldy, const void* X, int ldx, const float* scale, float* out, int ldo, long long M, int N, int K,
                 cudaStream_t stream);
int attention_bwd_tc_launch(const tcavp_attn_args& a, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                            long long dq_st, void* dk, long long dk_sb, long long dk_st, void* dv, long long dv_sb, long long dv_st,
                            int dkv_dtype, cudaStream_t stream);   // attention_bwd_tc.cu

// ------------------------------------------------------------------------------------------------
// AdamW (torch.optim.AdamW semantics, reference scripts/im_kim_train_GRN.py:1008): decoupled weight decay,
// bias-corrected moments.  One flat fp32 buffer per state.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void adamw_update(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                             long long n, float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt,
                                             float gscale) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * gscale;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    pi -= (lr / bc1) * (mi / denom);
    p[i] = pi;
  }
}

__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                             float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt, float gscale) {
  adamw_update(p, g, m, v, n, lr, b1, b2, eps, wd, bc1, bc2_sqrt, gscale);
}

// ------------------------------------------------------------------------------------------------
// Gradient-norm clipping and non-finite step skipping (reference modify_scripts/modify_train.py:1190-1196: skip a step whose loss
// is NaN, clip_grad_norm_; scripts/modify_im_kim_train.py: clip_grad_norm_(…, 1.0) before optimizer.step()).
// The norm is a two-launch deterministic reduction: a fixed partition of the buffer over at most CLIP_BLOCKS blocks, one fp64
// partial per block, then one block combines the partials in a fixed order.  No atomics and no counters to reset, so repeated
// calls and graph replays give the same bits.
// ------------------------------------------------------------------------------------------------
constexpr int CLIP_BLOCKS = TCAVP_CLIP_WORKSPACE_BYTES / 8;   // 1184 = 8 resident blocks on each of the 148 SMs of a B200
constexpr int CLIP_THREADS = 256;
constexpr int CLIP_UNROLL = 4;                                // float4 loads in flight per thread

__device__ __forceinline__ double block_sum_f64(double v, double* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < CLIP_THREADS / 32; ++w) s += red[w];
  return s;   // valid in thread 0
}

// Squares of four elements summed in fp32 (at most 4 roundings, < 2.4e-7 relative), accumulated across the buffer in fp64.
__device__ __forceinline__ double sumsq4(float4 x) {
  return (double)fmaf(x.w, x.w, fmaf(x.z, x.z, fmaf(x.y, x.y, x.x * x.x)));
}

// Block b reduces g[b * chunk, min(n, (b + 1) * chunk)); chunk is a multiple of 4, so with VEC every block's float4 run is aligned.
template <bool VEC>
__global__ void __launch_bounds__(CLIP_THREADS, CLIP_BLOCKS / 148) clip_norm_partial_kernel(const float* __restrict__ g, long long n, long long chunk,
                                                                         double* __restrict__ partial) {
  __shared__ double red[CLIP_THREADS / 32];
  const long long lo = blockIdx.x * chunk;
  const long long hi = min(n, lo + chunk);
  double acc = 0.0;
  long long tail = lo;
  if (VEC) {
    const float4* v = reinterpret_cast<const float4*>(g + lo);
    const long long nv = (hi - lo) >> 2;
    long long i = threadIdx.x;
#pragma unroll 1
    for (; i + (CLIP_UNROLL - 1) * CLIP_THREADS < nv; i += CLIP_UNROLL * CLIP_THREADS) {
      float4 x[CLIP_UNROLL];
#pragma unroll
      for (int u = 0; u < CLIP_UNROLL; ++u) x[u] = __ldcs(v + i + u * CLIP_THREADS);
#pragma unroll
      for (int u = 0; u < CLIP_UNROLL; ++u) acc += sumsq4(x[u]);
    }
#pragma unroll 1
    for (; i < nv; i += CLIP_THREADS) acc += sumsq4(__ldcs(v + i));
    tail = lo + (nv << 2);
  }
#pragma unroll 1
  for (long long i = tail + threadIdx.x; i < hi; i += CLIP_THREADS) {
    const float x = g[i];
    acc += (double)(x * x);
  }
  const double s = block_sum_f64(acc, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(CLIP_THREADS) clip_finish_kernel(const double* __restrict__ partial, int nparts, float grad_scale,
                                                                   float max_norm, const float* __restrict__ loss, int skip_nonfinite,
                                                                   tcavp_clip_record* __restrict__ rec) {
  __shared__ double red[CLIP_THREADS / 32];
  double s = 0.0;
  for (int i = threadIdx.x; i < nparts; i += CLIP_THREADS) s += partial[i];
  s = block_sum_f64(s, red);
  if (threadIdx.x != 0) return;
  const float norm = (float)(sqrt(s) * fabs((double)grad_scale));
  float coef = 1.f;
  if (max_norm > 0.f) {
    // torch.nn.utils.clip_grad_norm_: max_norm / (total_norm + 1e-6) on an fp32 tensor is reciprocal() * max_norm, then
    // clamp(max=1), which keeps a NaN (fminf would return 1 and let a NaN gradient through unclipped)
    coef = __frcp_rn(norm + 1e-6f) * max_norm;
    coef = coef > 1.f ? 1.f : coef;
  }
  rec->total_norm = norm;
  rec->clip_coef = coef;
  rec->skip = skip_nonfinite && (!isfinite(norm) || (loss != nullptr && !isfinite(*loss)));
  rec->reserved = 0;
}

// tcavp_adamw with the gradient factor, the skip and the step number read from the device: the bias corrections are the host
// expressions of tcavp_adamw evaluated for step = *step + 1.  The counter itself moves in adamw_count_kernel, after every block
// has read it.
__global__ void adamw_clipped_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                     long long n, float lr, float b1, float b2, float eps, float wd, float gscale,
                                     const tcavp_clip_record* __restrict__ clip, const int* __restrict__ step) {
  if (clip->skip) return;
  const float t = (float)(*step + 1);
  adamw_update(p, g, m, v, n, lr, b1, b2, eps, wd, 1.f - powf(b1, t), sqrtf(1.f - powf(b2, t)), gscale * clip->clip_coef);
}

__global__ void adamw_count_kernel(const tcavp_clip_record* __restrict__ clip, int* __restrict__ step, int* __restrict__ skipped) {
  if (!clip->skip)
    ++*step;
  else if (skipped != nullptr)
    ++*skipped;
}

__global__ void mark_nonfinite_kernel(const float* __restrict__ loss, float* __restrict__ dst) {
  if (!isfinite(*loss)) *dst = __int_as_float(0x7fc00000);
}

}  // namespace tcavp

using namespace tcavp;
#define STREAM(s) reinterpret_cast<cudaStream_t>(s)
#define DT_OK(d) ((d) == TCAVP_F32 || (d) == TCAVP_BF16)

extern "C" int tcavp_transpose(const void* in, long long in_bstride, int ldi, int in_dtype, void* out, long long out_bstride, int ldo,
                               int out_dtype, int batch, int rows, int cols, tcavp_stream_t stream) {
  TCAVP_REQUIRE(batch >= 0 && rows >= 0 && cols >= 0 && batch <= 65535, "tcavp_transpose: bad shape");
  if (batch == 0 || rows == 0 || cols == 0) return TCAVP_OK;
  TCAVP_REQUIRE(in && out && DT_OK(in_dtype) && DT_OK(out_dtype) && ldi >= cols && ldo >= rows, "tcavp_transpose: bad pointer/dtype/ld");
  TCAVP_REQUIRE((cols + 31) / 32 <= 65535, "tcavp_transpose: too many columns");
  if (in_dtype == TCAVP_BF16 && out_dtype == TCAVP_BF16 && ldi % 2 == 0 && ldo % 2 == 0 && in_bstride % 2 == 0 && out_bstride % 2 == 0 &&
      reinterpret_cast<uintptr_t>(in) % 4 == 0 && reinterpret_cast<uintptr_t>(out) % 4 == 0 && (cols + 63) / 64 <= 65535) {
    dim3 grid64((rows + 63) / 64, (cols + 63) / 64, batch);
    transpose_bf16_kernel<<<grid64, 256, 0, STREAM(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(in), in_bstride, ldi,
                                                               reinterpret_cast<__nv_bfloat16*>(out), out_bstride, ldo, rows, cols);
    return check_launch("transpose_kernel");
  }
  dim3 grid((rows + 31) / 32, (cols + 31) / 32, batch);
  transpose_kernel<<<grid, 256, 0, STREAM(stream)>>>(in, in_bstride, ldi, in_dtype, out, out_bstride, ldo, out_dtype, rows, cols);
  return check_launch("transpose_kernel");
}

extern "C" int tcavp_period_sum(const void* x, int ldx, int dtype, long long rows, int cols, int period, float* out, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && period > 0 && period <= 65535, "tcavp_period_sum: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && out && DT_OK(dtype) && ldx >= cols, "tcavp_period_sum: bad pointer/dtype");
  const long long K = (rows + period - 1) / period;
  const int cblocks = (cols + 127) / 128;
  long long want = ((long long)sm_count() * 8) / ((long long)cblocks * period);
  if (want < 1) want = 1;
  if (want > K) want = K;
  if (want > 4096) want = 4096;
  const long long kper = (K + want - 1) / want;
  dim3 grid(cblocks, period, (unsigned)((K + kper - 1) / kper));
  period_sum_kernel<<<grid, 128, 0, STREAM(stream)>>>(x, ldx, dtype, rows, cols, period, out, kper);
  return check_launch("period_sum_kernel");
}

extern "C" int tcavp_relu_bwd(const void* dy, int lddy, const void* y, int ldy, void* dx, int lddx, int dtype, long long rows, int cols,
                              tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0, "tcavp_relu_bwd: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dy && y && dx && DT_OK(dtype), "tcavp_relu_bwd: bad pointer/dtype");
  relu_bwd_kernel<<<grid_cap((rows * cols + 255) / 256, 16), 256, 0, STREAM(stream)>>>(dy, lddy, y, ldy, dx, lddx, dtype, rows, cols);
  return check_launch("relu_bwd_kernel");
}

static int gelu_vec_ok(const void* a, int lda, const void* b, int ldb, const void* c, int ldc, int dtype, int cols) {
  auto al = [](const void* p, int ld) { return !p || (reinterpret_cast<uintptr_t>(p) % 16 == 0 && ld % 8 == 0); };
  return dtype == TCAVP_BF16 && cols % 8 == 0 && al(a, lda) && al(b, ldb) && al(c, ldc);
}
extern "C" int tcavp_gelu_tanh(const void* x, int ldx, void* out, int ldo, int dtype, long long rows, int cols, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && ldx >= cols && ldo >= cols, "tcavp_gelu_tanh: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(x && out && DT_OK(dtype), "tcavp_gelu_tanh: bad pointer/dtype");
  const int vec = gelu_vec_ok(nullptr, 0, x, ldx, out, ldo, dtype, cols);
  const long long work = vec ? rows * (cols / 8) : rows * cols;
  gelu_new_kernel<false><<<grid_cap((work + 255) / 256, 16), 256, 0, STREAM(stream)>>>(nullptr, 0, x, ldx, out, ldo, dtype, rows, cols, vec);
  return check_launch("gelu_new_kernel");
}
extern "C" int tcavp_gelu_tanh_bwd(const void* dy, int lddy, const void* x, int ldx, void* dx, int lddx, int dtype, long long rows, int cols,
                                   tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && lddy >= cols && ldx >= cols && lddx >= cols, "tcavp_gelu_tanh_bwd: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dy && x && dx && DT_OK(dtype), "tcavp_gelu_tanh_bwd: bad pointer/dtype");
  const int vec = gelu_vec_ok(dy, lddy, x, ldx, dx, lddx, dtype, cols);
  const long long work = vec ? rows * (cols / 8) : rows * cols;
  gelu_new_kernel<true><<<grid_cap((work + 255) / 256, 16), 256, 0, STREAM(stream)>>>(dy, lddy, x, ldx, dx, lddx, dtype, rows, cols, vec);
  return check_launch("gelu_new_bwd_kernel");
}

extern "C" int tcavp_axpby(const void* a, int lda, int a_dtype, float alpha, const void* b, int ldb, int b_dtype, float beta, void* out,
                           int ldo, int out_dtype, long long rows, int cols, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0, "tcavp_axpby: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(a && out && DT_OK(a_dtype) && DT_OK(out_dtype) && (!b || DT_OK(b_dtype)), "tcavp_axpby: bad pointer/dtype");
  axpby_kernel<<<grid_cap((rows * cols + 255) / 256, 16), 256, 0, STREAM(stream)>>>(a, lda, a_dtype, alpha, b, ldb, b_dtype, beta, out, ldo,
                                                                                  out_dtype, rows, cols);
  return check_launch("axpby_kernel");
}

extern "C" int tcavp_swiglu(const void* gu, void* out, int dtype, long long rows, int I, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && I > 0, "tcavp_swiglu: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(gu && out && DT_OK(dtype), "tcavp_swiglu: bad pointer/dtype");
  swiglu_kernel<<<grid_cap((rows * I + 255) / 256, 16), 256, 0, STREAM(stream)>>>(gu, out, dtype, rows, I);
  return check_launch("swiglu_kernel");
}

extern "C" int tcavp_swiglu_bwd(const void* dout, const void* gu, void* dgu, int dtype, long long rows, int I, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && I > 0, "tcavp_swiglu_bwd: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dout && gu && dgu && DT_OK(dtype), "tcavp_swiglu_bwd: bad pointer/dtype");
  swiglu_bwd_kernel<<<grid_cap((rows * I + 255) / 256, 16), 256, 0, STREAM(stream)>>>(dout, gu, dgu, dtype, rows, I);
  return check_launch("swiglu_bwd_kernel");
}

extern "C" int tcavp_layernorm_bwd(const void* dy, int dy_dtype, const void* x, const void* residual, int x_dtype, const float* w, int rows,
                                   int cols, float eps, void* dx, int dx_dtype, float* dw, float* db, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && cols <= 8192, "tcavp_layernorm_bwd: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dy && x && w && DT_OK(dy_dtype) && DT_OK(x_dtype) && (!dx || DT_OK(dx_dtype)) && ((dw == nullptr) == (db == nullptr)),
                "tcavp_layernorm_bwd: bad pointer/dtype");
  const size_t smem = (size_t)2 * cols * sizeof(float);
  TCAVP_CUDA(cudaFuncSetAttribute(layernorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  layernorm_bwd_kernel<<<grid_cap((rows + 7) / 8, 4), 256, smem, STREAM(stream)>>>(dy, dy_dtype, x, residual, x_dtype, w, rows, cols, eps, dx,
                                                                                 dx_dtype, dw, db);
  return check_launch("layernorm_bwd_kernel");
}

extern "C" int tcavp_layernorm_bwd_dx(const void* dy, int lddy, const void* x, int ldx, const float* w, const void* add, int ldadd, void* dx,
                                      int lddx, int dtype, int rows, int cols, float eps, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0 && lddy >= cols && ldx >= cols && lddx >= cols && (!add || ldadd >= cols), "tcavp_layernorm_bwd_dx: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dy && x && w && dx && DT_OK(dtype), "tcavp_layernorm_bwd_dx: bad pointer/dtype");
  if (norm_bwd_pipe_launch<true>(dy, lddy, x, ldx, w, add, ldadd, dx, lddx, dtype, rows, cols, eps, STREAM(stream)))
    return check_launch("layernorm_bwd_dx_kernel");
  auto al = [](const void* p, int ld) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % 16 == 0 && ld % 8 == 0); };
  if (dtype == TCAVP_BF16 && cols % 8 == 0 && cols <= 1024 && al(dy, lddy) && al(x, ldx) && al(add, ldadd) && al(dx, lddx)) {
    const __nv_bfloat16* dyb = reinterpret_cast<const __nv_bfloat16*>(dy);
    const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x);
    const __nv_bfloat16* ab = reinterpret_cast<const __nv_bfloat16*>(add);
    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(dx);
    const int grid = grid_cap((rows + 7) / 8, 16);
#define TCAVP_LB(NV) layernorm_bwd_dx_vec_kernel<NV><<<grid, 256, 0, STREAM(stream)>>>(dyb, lddy, xb, ldx, w, ab, ldadd, ob, lddx, rows, cols, eps)
    if (cols <= 256) TCAVP_LB(1);
    else if (cols <= 512) TCAVP_LB(2);
    else if (cols <= 768) TCAVP_LB(3);
    else TCAVP_LB(4);
#undef TCAVP_LB
    return check_launch("layernorm_bwd_dx_kernel");
  }
  layernorm_bwd_dx_kernel<<<grid_cap((rows + 7) / 8, 8), 256, 0, STREAM(stream)>>>(dy, lddy, x, ldx, w, add, ldadd, dx, lddx, dtype, rows, cols, eps);
  return check_launch("layernorm_bwd_dx_kernel");
}

extern "C" int tcavp_rmsnorm_bwd(const void* dy, int lddy, const void* x, int ldx, const float* w, const void* add, int ldadd, void* dx,
                                 int lddx, int dtype, int rows, int cols, float eps, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0, "tcavp_rmsnorm_bwd: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dy && x && dx && DT_OK(dtype), "tcavp_rmsnorm_bwd: bad pointer/dtype");
  if (norm_bwd_pipe_launch<false>(dy, lddy, x, ldx, w, add, ldadd, dx, lddx, dtype, rows, cols, eps, STREAM(stream)))
    return check_launch("rmsnorm_bwd_kernel");
  auto al = [](const void* p, int ld) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % 16 == 0 && ld % 8 == 0); };
  if (dtype == TCAVP_BF16 && cols % 8 == 0 && al(dy, lddy) && al(x, ldx) && al(add, ldadd) && al(dx, lddx)) {
    const __nv_bfloat16* dyb = reinterpret_cast<const __nv_bfloat16*>(dy);
    const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x);
    const __nv_bfloat16* ab = reinterpret_cast<const __nv_bfloat16*>(add);
    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(dx);
    const int grid = grid_cap((rows + 7) / 8, 16);
#define TCAVP_RB(NV) rmsnorm_bwd_vec_kernel<NV><<<grid, 256, 0, STREAM(stream)>>>(dyb, lddy, xb, ldx, w, ab, ldadd, ob, lddx, rows, cols, eps)
    if (cols <= 256) TCAVP_RB(1);
    else if (cols <= 512) TCAVP_RB(2);
    else if (cols <= 768) TCAVP_RB(3);
    else if (cols <= 1024) TCAVP_RB(4);
    else TCAVP_RB(0);
#undef TCAVP_RB
    return check_launch("rmsnorm_bwd_kernel");
  }
  rmsnorm_bwd_kernel<<<grid_cap((rows + 7) / 8, 8), 256, 0, STREAM(stream)>>>(dy, lddy, x, ldx, w, add, ldadd, dx, lddx, dtype, rows, cols, eps);
  return check_launch("rmsnorm_bwd_kernel");
}

// bf16 rows with 16-byte aligned starts: 8 elements (two rotation quads) per thread, one 16-byte load + store.
__global__ void __launch_bounds__(256) rope_adjacent_vec_kernel(__nv_bfloat16* __restrict__ buf, long long rows, int L, int ld, int cols, int dh,
                                                                const float* __restrict__ table, int inverse) {
  const int octs = cols >> 3;
  const long long total = rows * octs;
  const float sg = inverse ? -1.f : 1.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / octs;
    const int c = (int)(i % octs) * 8;
    const int pos = (int)(r % L);
    float v[8];
    ld8_bf16(buf + (size_t)r * ld + c, v);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(table) + (size_t)(((c + 4 * h) % dh) >> 2) * L + pos);
      const float a0 = v[4 * h], a1 = v[4 * h + 1], a2 = v[4 * h + 2], a3 = v[4 * h + 3];
      v[4 * h] = a0 * t.x - sg * a1 * t.y;
      v[4 * h + 1] = a1 * t.x + sg * a0 * t.y;
      v[4 * h + 2] = a2 * t.z - sg * a3 * t.w;
      v[4 * h + 3] = a3 * t.z + sg * a2 * t.w;
    }
    st8_bf16(buf + (size_t)r * ld + c, v);
  }
}

extern "C" int tcavp_rope_adjacent(void* buf, int dtype, long long rows, int L, int ld, int cols, int dh, const float* table, int inverse,
                                   tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && L > 0 && cols >= 0 && dh >= 4 && dh % 4 == 0 && cols % dh == 0 && ld >= cols, "tcavp_rope_adjacent: bad shape");
  if (rows == 0 || cols == 0) return TCAVP_OK;
  TCAVP_REQUIRE(buf && table && DT_OK(dtype), "tcavp_rope_adjacent: bad pointer/dtype");
  if (dtype == TCAVP_BF16 && cols % 8 == 0 && dh % 8 == 0 && ld % 8 == 0 && reinterpret_cast<uintptr_t>(buf) % 16 == 0) {
    rope_adjacent_vec_kernel<<<grid_cap((rows * (cols / 8) + 255) / 256, 16), 256, 0, STREAM(stream)>>>(reinterpret_cast<__nv_bfloat16*>(buf), rows, L,
                                                                                                        ld, cols, dh, table, inverse);
    return check_launch("rope_adjacent_kernel");
  }
  rope_adjacent_kernel<<<grid_cap((rows * (cols / 4) + 255) / 256, 16), 256, 0, STREAM(stream)>>>(buf, dtype, rows, L, ld, cols, dh, table, inverse);
  return check_launch("rope_adjacent_kernel");
}

extern "C" int tcavp_copy_rows(const void* in, int ldi, int in_dtype, int in_gi, int in_go, int in_off, void* out, int ldo, int out_dtype,
                               int out_gi, int out_go, int out_off, long long rows, int cols, tcavp_stream_t stream) {
  TCAVP_REQUIRE(rows >= 0 && cols > 0, "tcavp_copy_rows: bad shape");
  if (rows == 0) return TCAVP_OK;
  TCAVP_REQUIRE(in && out && DT_OK(in_dtype) && DT_OK(out_dtype), "tcavp_copy_rows: bad pointer/dtype");
  copy_rows_kernel<<<grid_cap((rows * cols + 255) / 256, 16), 256, 0, STREAM(stream)>>>(in, ldi, in_dtype, in_gi, in_go, in_off, out, ldo,
                                                                                      out_dtype, out_gi, out_go, out_off, rows, cols);
  return check_launch("copy_rows_kernel");
}

extern "C" int tcavp_masked_mean_bwd(const void* dout, int dout_dtype, const int32_t* len, void* dx, int dx_dtype, int B, int P, int D,
                                     tcavp_stream_t stream) {
  TCAVP_REQUIRE(B >= 0 && P > 0 && D > 0, "tcavp_masked_mean_bwd: bad shape");
  if (B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dout && len && dx && DT_OK(dout_dtype) && DT_OK(dx_dtype), "tcavp_masked_mean_bwd: bad pointer/dtype");
  masked_mean_bwd_kernel<<<grid_cap(((long long)B * P * D + 255) / 256, 16), 256, 0, STREAM(stream)>>>(dout, dout_dtype, len, dx, dx_dtype, B, P, D);
  return check_launch("masked_mean_bwd_kernel");
}

extern "C" int tcavp_nlinear_bwd(const void* g, int g_dtype, const void* in, int in_dtype, const float* w, void* din, int din_dtype,
                                 float* dw, int B, int C, int T_in, int T_out, tcavp_stream_t stream) {
  TCAVP_REQUIRE(B >= 0 && C > 0 && C <= 256 && T_in > 0 && T_out > 0, "tcavp_nlinear_bwd: bad shape");
  if (B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(g && DT_OK(g_dtype) && (!din || (w && DT_OK(din_dtype))) && (!dw || (in && DT_OK(in_dtype))), "tcavp_nlinear_bwd: bad pointer/dtype");
  if (din) {
    nlinear_bwd_in_kernel<<<grid_cap(((long long)B * C + 127) / 128, 16), 128, 0, STREAM(stream)>>>(g, g_dtype, w, din, din_dtype, B, C, T_in, T_out);
    int rc = check_launch("nlinear_bwd_in_kernel");
    if (rc) return rc;
  }
  if (dw) {
    int splits = (sm_count() * 4) / (T_in * T_out);
    if (splits < 1) splits = 1;
    if (splits > B) splits = B;
    const int bper = (B + splits - 1) / splits;
    dim3 grid(T_out * T_in, (B + bper - 1) / bper);
    nlinear_bwd_w_kernel<<<grid, (256 / C) * C, 0, STREAM(stream)>>>(g, g_dtype, in, in_dtype, dw, B, C, T_in, T_out, bper);
    return check_launch("nlinear_bwd_w_kernel");
  }
  return TCAVP_OK;
}

extern "C" int tcavp_head_assemble(const float* o, const float* x, float* decoded, int B, int T_in, int T_out, tcavp_stream_t stream) {
  TCAVP_REQUIRE(B >= 0 && T_in > 0 && T_out > 0, "tcavp_head_assemble: bad shape");
  if (B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(o && x && decoded, "tcavp_head_assemble: null pointer");
  head_assemble_kernel<<<grid_cap(((long long)B * 2 * T_out + 255) / 256, 16), 256, 0, STREAM(stream)>>>(o, x, decoded, B, T_in, T_out);
  return check_launch("head_assemble_kernel");
}

extern "C" int tcavp_traj_loss_bwd(const float* decoded, const float* y, const float* norm_stat, const float* gscale, float* d_o, int B,
                                   int T_out, tcavp_stream_t stream) {
  TCAVP_REQUIRE(B >= 0 && T_out > 0, "tcavp_traj_loss_bwd: bad shape");
  if (B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(decoded && y && norm_stat && d_o, "tcavp_traj_loss_bwd: null pointer");
  traj_loss_bwd_kernel<<<grid_cap(((long long)B * 2 * T_out + 255) / 256, 16), 256, 0, STREAM(stream)>>>(decoded, y, norm_stat, gscale, d_o, B, T_out);
  return check_launch("traj_loss_bwd_kernel");
}

extern "C" int tcavp_skinny_dw(const void* Y, int ldy, int y_dtype, const void* Z, int ldz, int z_dtype, const float* row_scale, float* out,
                               int ldo, long long M, int N, int J, tcavp_stream_t stream) {
  TCAVP_REQUIRE(M >= 0 && N > 0 && J > 0 && J <= 32 && ldo >= J, "tcavp_skinny_dw: bad shape (J=%d, max 32)", J);
  if (M == 0) return TCAVP_OK;
  TCAVP_REQUIRE(Y && Z && out && DT_OK(y_dtype) && DT_OK(z_dtype), "tcavp_skinny_dw: bad pointer/dtype");
  if (y_dtype == TCAVP_BF16 && z_dtype == TCAVP_BF16 && M < (1ll << 31)) {   // bound by the one pass over Y instead of FFMA issue
    const int rc = dw_tc_launch(Y, ldy, Z, ldz, row_scale, out, ldo, M, N, J, STREAM(stream));
    if (rc <= 0) return rc;
  }
  const int nblocks = (N + 127) / 128;
  long long splits = ((long long)sm_count() * 8) / nblocks;
  if (splits < 1) splits = 1;
  long long mper = (M + splits - 1) / splits;
  mper = (mper + 31) / 32 * 32;
  dim3 grid(nblocks, (unsigned)((M + mper - 1) / mper));
  if (J <= 8) skinny_dw_kernel<8><<<grid, 128, 0, STREAM(stream)>>>(Y, ldy, y_dtype, Z, ldz, z_dtype, row_scale, out, ldo, M, N, J, (int)mper);
  else if (J <= 16) skinny_dw_kernel<16><<<grid, 128, 0, STREAM(stream)>>>(Y, ldy, y_dtype, Z, ldz, z_dtype, row_scale, out, ldo, M, N, J, (int)mper);
  else skinny_dw_kernel<32><<<grid, 128, 0, STREAM(stream)>>>(Y, ldy, y_dtype, Z, ldz, z_dtype, row_scale, out, ldo, M, N, J, (int)mper);
  return check_launch("skinny_dw_kernel");
}

extern "C" int tcavp_dw(const void* dY, int lddy, int dy_dtype, const void* X, int ldx, int x_dtype, float* out, int ldo, long long M, int N,
                        int K, tcavp_stream_t stream) {
  TCAVP_REQUIRE(M >= 0 && N > 0 && K > 0 && lddy >= N && ldx >= K && ldo >= K, "tcavp_dw: bad shape M=%lld N=%d K=%d", M, N, K);
  if (M == 0) return TCAVP_OK;
  TCAVP_REQUIRE(dY && X && out && DT_OK(dy_dtype) && DT_OK(x_dtype), "tcavp_dw: bad pointer/dtype");
  if (dy_dtype == TCAVP_BF16 && x_dtype == TCAVP_BF16) {     // tensor cores on the row-major operands (ldmatrix.trans)
    const int rc = dw_tc_launch(dY, lddy, X, ldx, nullptr, out, ldo, M, N, K, STREAM(stream));
    if (rc <= 0) return rc;
  }
  const int tn = (N + 63) / 64, tk = (K + 63) / 64;
  long long splits = ((long long)sm_count() * 4) / ((long long)tn * tk);
  if (splits < 1) splits = 1;
  long long mper = (M + splits - 1) / splits;
  mper = (mper + 15) / 16 * 16;
  if (mper < 64) mper = 64;
  const long long nz = (M + mper - 1) / mper;
  TCAVP_REQUIRE(nz <= 65535 && tn <= 65535, "tcavp_dw: grid too large");
  dim3 grid(tk, tn, (unsigned)nz);
  dw_simt_kernel<<<grid, 256, 0, STREAM(stream)>>>(dY, lddy, dy_dtype, X, ldx, x_dtype, out, ldo, M, N, K, (int)mper);
  return check_launch("dw_simt_kernel");
}

extern "C" int tcavp_attention_bwd(const tcavp_attn_args* a, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                                   long long dq_st, float* dk, long long dk_sb, long long dk_st, float* dv, long long dv_sb, long long dv_st,
                                   tcavp_stream_t stream) {
  TCAVP_REQUIRE(a != nullptr, "tcavp_attention_bwd: null args");
  TCAVP_REQUIRE(a->B >= 0 && a->H > 0 && a->Hkv > 0 && a->H % a->Hkv == 0 && a->Tq > 0 && a->Tk > 0 && a->dh > 0, "tcavp_attention_bwd: bad shape");
  TCAVP_REQUIRE(a->Tk <= ab::JJ * ab::THREADS, "tcavp_attention_bwd: Tk %d > %d", a->Tk, ab::JJ * ab::THREADS);
  TCAVP_REQUIRE(!a->causal || a->Tq == a->Tk, "tcavp_attention_bwd: causal needs Tq == Tk");
  if (a->B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(a->q && a->k && a->v && dout && dq && dk && dv && DT_OK(a->dtype), "tcavp_attention_bwd: bad pointer/dtype");
  TCAVP_REQUIRE(a->drop_thresh == 0 || (a->drop_seed != nullptr && a->drop_scale > 0.f), "tcavp_attention_bwd: dropout needs a device seed and a scale");
  {   // tensor-core path: bf16, MHA, small head, forward output available (args->out)
    const int rc = attention_bwd_tc_launch(*a, dout, do_sb, do_st, dq, dq_sb, dq_st, dk, dk_sb, dk_st, dv, dv_sb, dv_st, TCAVP_F32, STREAM(stream));
    if (rc <= 0) return rc;
  }
  int DC = a->dh < 32 ? a->dh : 32;
  auto smem_for = [&](int dc) { return (size_t)(2 * ab::QB * a->Tk + 2 * ab::QB * (dc + 1) + 2 * (size_t)a->Tk * (dc + 1)) * sizeof(float); };
  if (smem_for(DC) > 200 * 1024) DC = 16 < a->dh ? 16 : a->dh;
  const size_t smem = smem_for(DC);
  TCAVP_REQUIRE(smem <= 220 * 1024, "tcavp_attention_bwd: Tk %d needs %zu bytes of shared memory", a->Tk, smem);
  const int nqb = (a->Tq + ab::QB - 1) / ab::QB;
  const long long blocks = (long long)a->B * a->H * nqb;
  TCAVP_REQUIRE(blocks <= 0x7fffffffLL, "tcavp_attention_bwd: grid too large");
  if (a->dtype == TCAVP_BF16) {
    TCAVP_CUDA(cudaFuncSetAttribute(ab::attn_bwd_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ab::attn_bwd_kernel<__nv_bfloat16><<<(unsigned)blocks, ab::THREADS, smem, STREAM(stream)>>>(
        *a, reinterpret_cast<const __nv_bfloat16*>(dout), do_sb, do_st, reinterpret_cast<__nv_bfloat16*>(dq), dq_sb, dq_st, dk, dk_sb, dk_st, dv,
        dv_sb, dv_st, DC);
  } else {
    TCAVP_CUDA(cudaFuncSetAttribute(ab::attn_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ab::attn_bwd_kernel<float><<<(unsigned)blocks, ab::THREADS, smem, STREAM(stream)>>>(
        *a, reinterpret_cast<const float*>(dout), do_sb, do_st, reinterpret_cast<float*>(dq), dq_sb, dq_st, dk, dk_sb, dk_st, dv, dv_sb, dv_st, DC);
  }
  return check_launch("attn_bwd_kernel");
}

extern "C" int tcavp_attention_bwd_owned(const tcavp_attn_args* a, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                                         long long dq_st, void* dk, long long dk_sb, long long dk_st, void* dv, long long dv_sb, long long dv_st,
                                         int dkv_dtype, tcavp_stream_t stream) {
  TCAVP_REQUIRE(a != nullptr, "tcavp_attention_bwd_owned: null args");
  TCAVP_REQUIRE(a->B >= 0 && a->H > 0 && a->H == a->Hkv && a->Tq > 0 && a->Tk > 0, "tcavp_attention_bwd_owned: bad shape (needs H == Hkv)");
  TCAVP_REQUIRE(!a->causal || a->Tq == a->Tk, "tcavp_attention_bwd_owned: causal needs Tq == Tk");
  if (a->B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(a->q && a->k && a->v && dout && dq && dk && dv && DT_OK(dkv_dtype), "tcavp_attention_bwd_owned: bad pointer/dtype");
  TCAVP_REQUIRE(a->drop_thresh == 0 || (a->drop_seed != nullptr && a->drop_scale > 0.f), "tcavp_attention_bwd_owned: dropout needs a device seed and a scale");
  int rc = 1;
  if (a->out) rc = attention_bwd_tc_launch(*a, dout, do_sb, do_st, dq, dq_sb, dq_st, dk, dk_sb, dk_st, dv, dv_sb, dv_st, dkv_dtype, STREAM(stream));
  if (rc > 0)   // few queries against wide heads (LTSF cross-attention): head_dim % 64 == 0, Tq <= 64, no causal mask
    rc = attention_x_bwd_launch(*a, dout, do_sb, do_st, dq, dq_sb, dq_st, dk, dk_sb, dk_st, dv, dv_sb, dv_st, dkv_dtype, STREAM(stream));
  if (rc > 0)
    return fail_arg("tcavp_attention_bwd_owned: shape not covered (bf16 and either head_dim 16/32/64/96/128 with Tq, Tk <= 256 and the forward "
                    "output in args->out, or head_dim %% 64 == 0 with Tq <= 64, Tk <= 256, not causal)");
  return rc;
}

extern "C" int tcavp_adamw(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1, float beta2,
                           float eps, float weight_decay, int step, float grad_scale, tcavp_stream_t stream) {
  TCAVP_REQUIRE(n >= 0 && step >= 1, "tcavp_adamw: bad n/step");
  if (n == 0) return TCAVP_OK;
  TCAVP_REQUIRE(param && grad && exp_avg && exp_avg_sq, "tcavp_adamw: null pointer");
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2 = sqrtf(1.f - powf(beta2, (float)step));
  adamw_kernel<<<grid_cap((n + 255) / 256, 16), 256, 0, STREAM(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                                                                        bc1, bc2, grad_scale);
  return check_launch("adamw_kernel");
}

extern "C" int tcavp_clip_prologue(const float* grad, long long n, float grad_scale, float max_norm, const float* loss, int skip_nonfinite,
                                   void* workspace, long long workspace_bytes, tcavp_clip_record* record, tcavp_stream_t stream) {
  TCAVP_REQUIRE(n >= 0, "tcavp_clip_prologue: bad n");
  TCAVP_REQUIRE(record && (n == 0 || (grad && workspace)), "tcavp_clip_prologue: null pointer");
  TCAVP_REQUIRE(n == 0 || workspace_bytes >= TCAVP_CLIP_WORKSPACE_BYTES, "tcavp_clip_prologue: workspace below TCAVP_CLIP_WORKSPACE_BYTES");
  TCAVP_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 8 == 0, "tcavp_clip_prologue: workspace not 8-byte aligned");
  int parts = 0;
  if (n > 0) {
    // equal 4-aligned chunks, at most CLIP_BLOCKS of them and at least one unrolled block sweep (4096 elements) each
    const long long sweep = (long long)CLIP_THREADS * CLIP_UNROLL * 4;
    const long long want = (n + sweep - 1) / sweep;
    const long long blocks = want < CLIP_BLOCKS ? want : CLIP_BLOCKS;
    const long long chunk = ((n + blocks - 1) / blocks + 3) / 4 * 4;
    parts = (int)((n + chunk - 1) / chunk);
    double* partial = static_cast<double*>(workspace);
    if (reinterpret_cast<uintptr_t>(grad) % 16 == 0)
      clip_norm_partial_kernel<true><<<parts, CLIP_THREADS, 0, STREAM(stream)>>>(grad, n, chunk, partial);
    else
      clip_norm_partial_kernel<false><<<parts, CLIP_THREADS, 0, STREAM(stream)>>>(grad, n, chunk, partial);
    int rc = check_launch("clip_norm_partial_kernel");
    if (rc) return rc;
  }
  clip_finish_kernel<<<1, CLIP_THREADS, 0, STREAM(stream)>>>(static_cast<const double*>(workspace), parts, grad_scale, max_norm, loss,
                                                             skip_nonfinite != 0, record);
  return check_launch("clip_finish_kernel");
}

extern "C" int tcavp_adamw_clipped(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1,
                                   float beta2, float eps, float weight_decay, float grad_scale, const tcavp_clip_record* clip, int* step,
                                   int* skipped, tcavp_stream_t stream) {
  TCAVP_REQUIRE(n >= 0, "tcavp_adamw_clipped: bad n");
  TCAVP_REQUIRE(clip && step && (n == 0 || (param && grad && exp_avg && exp_avg_sq)), "tcavp_adamw_clipped: null pointer");
  if (n > 0) {
    adamw_clipped_kernel<<<grid_cap((n + 255) / 256, 16), 256, 0, STREAM(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                                                  weight_decay, grad_scale, clip, step);
    int rc = check_launch("adamw_clipped_kernel");
    if (rc) return rc;
  }
  adamw_count_kernel<<<1, 1, 0, STREAM(stream)>>>(clip, step, skipped);
  return check_launch("adamw_count_kernel");
}

extern "C" int tcavp_mark_nonfinite(const float* loss, float* dst, tcavp_stream_t stream) {
  TCAVP_REQUIRE(loss && dst, "tcavp_mark_nonfinite: null pointer");
  mark_nonfinite_kernel<<<1, 1, 0, STREAM(stream)>>>(loss, dst);
  return check_launch("mark_nonfinite_kernel");
}
