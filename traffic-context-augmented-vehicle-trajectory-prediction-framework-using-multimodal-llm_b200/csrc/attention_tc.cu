// Tensor-core flash attention: the LLM self-attention (HF:251-289 with the causal + key-padding mask of HF:399)
// and the small nn.MultiheadAttention cores of the Q-Former / lane-polygon encoder (train.py:371, 411-413).
// bf16 operands, head_dim 16/32/64/96/128, Tq, Tk <= 256, optional causal mask, optional key mask, GQA.
//
// One CTA per (batch, head): K and V of that head are staged ONCE in shared memory (padded rows, conflict-free
// ldmatrix), every warp owns two 16-row query slabs (one from each end of the range: balanced causal work) and runs the FlashAttention-2 register pipeline
// (mma.sync m16n8k16: S = Q.K^T -> online softmax in fp32 -> O += P.V) over 64-key blocks, skipping blocks
// beyond its causal bound.  Scores and probabilities never touch shared or global memory.
#include "common.cuh"

namespace tcavp {
namespace fa {

constexpr int PAD = 8;      // bf16 elements of row padding (16 bytes): ldmatrix rows land in distinct banks

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// MAXT / MINB: launch bounds.  (288, 2) keeps two 9-warp CTAs (L = 144) resident per SM so the K/V staging of one
// overlaps the MMAs of the other.
// KB = keys per iteration (16 / 48 / 64): chosen by the host so that Tk pads to the fewest dead keys (L = 144 = 3 x 48).
template <int DH, int MAXT, int MINB, int KB>
__global__ void __launch_bounds__(MAXT, MINB) attn_flash_kernel(tcavp_attn_args a, int tk_pad_all, int tq_pad) {
  constexpr int LDS = DH + PAD;            // smem row stride in elements
  constexpr int KS = DH / 16;              // k-steps of the Q.K^T contraction
  constexpr int NT = DH / 8;               // n8 tiles of the output
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sV = sK + (size_t)tk_pad_all * LDS;
  __nv_bfloat16* sQ = sV + (size_t)tk_pad_all * LDS;                    // [tq_pad] rows, zero-filled beyond Tq
  int* sMask = reinterpret_cast<int*>(sQ + (size_t)tq_pad * LDS);       // [tk_pad_all] 1 = attend
  int* sBlkValid = sMask + tk_pad_all;                                  // [tk_pad_all / KB] all keys of the block attendable

  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int hk = h / (a.H / a.Hkv);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tk_pad = tk_pad_all;
  const __nv_bfloat16* gq = reinterpret_cast<const __nv_bfloat16*>(a.q) + (size_t)b * a.q_sb + (size_t)h * DH;
  const __nv_bfloat16* gk = reinterpret_cast<const __nv_bfloat16*>(a.k) + (size_t)b * a.k_sb + (size_t)hk * DH;
  const __nv_bfloat16* gv = reinterpret_cast<const __nv_bfloat16*>(a.v) + (size_t)b * a.v_sb + (size_t)hk * DH;

  // ---- stage K, V (zero-filled beyond Tk) and the key mask ----
  constexpr int VPR = DH / 8;              // 16-byte vectors per row
  // cp.async: every 16-byte copy is in flight at once (no register staging, no per-iteration round trip); rows
  // beyond Tk are zero-filled (src-size 0) so masked probabilities never meet NaN payloads.
  {
    const uint32_t sK_a = (uint32_t)__cvta_generic_to_shared(sK), sV_a = (uint32_t)__cvta_generic_to_shared(sV);
    for (int i = threadIdx.x; i < tk_pad * VPR; i += blockDim.x) {
      const int r = i / VPR, c = (i % VPR) * 8;
      const int sz = r < a.Tk ? 16 : 0;
      const size_t rr = r < a.Tk ? r : 0;
      const uint32_t off = (uint32_t)((r * LDS + c) * 2);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sK_a + off), "l"(gk + rr * a.k_st + c), "r"(sz) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sV_a + off), "l"(gv + rr * a.v_st + c), "r"(sz) : "memory");
    }
    const uint32_t sQ_a = (uint32_t)__cvta_generic_to_shared(sQ);
    for (int i = threadIdx.x; i < tq_pad * VPR; i += blockDim.x) {
      const int r = i / VPR, c = (i % VPR) * 8;
      const int sz = r < a.Tq ? 16 : 0;
      const size_t rr = r < a.Tq ? r : 0;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sQ_a + (uint32_t)((r * LDS + c) * 2)), "l"(gq + rr * a.q_st + c), "r"(sz) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int j = threadIdx.x; j < tk_pad; j += blockDim.x)
    sMask[j] = (j < a.Tk) && (!a.key_mask || a.key_mask[(size_t)b * a.Tk + j] != 0);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < tk_pad / KB) {
    int all = 1;
    for (int j = 0; j < KB; ++j) all &= sMask[threadIdx.x * KB + j];
    sBlkValid[threadIdx.x] = all;
  }
  __syncthreads();

  // Causal work grows with the row index, so every warp takes one slab from each end of the query range:
  // slabs (w, nslabs-1-w) cost about the same for every w and no warp idles while the last rows finish.
  const int nslabs = (a.Tq + 15) / 16;
  const int g = lane >> 2, t4 = lane & 3;
  const uint32_t sK_u = (uint32_t)__cvta_generic_to_shared(sK), sV_u = (uint32_t)__cvta_generic_to_shared(sV);
  const uint32_t sQ_u = (uint32_t)__cvta_generic_to_shared(sQ);
  // ldmatrix lane -> row/col offsets.  K (non-transposed, x4 = keys [0,8)/[8,16) x dims [0,8)/[8,16)):
  const int k_row = (lane & 7) + ((lane >> 4) << 3), k_col = ((lane >> 3) & 1) * 8;
  // V (transposed, x4 = keys [0,8)/[8,16) x dims [0,8)/[8,16)):
  const int v_row = (lane & 7) + (((lane >> 3) & 1) << 3), v_col = (lane >> 4) * 8;
  const float sl2 = a.scale * 1.4426950408889634f;   // softmax in base 2
  const bool drop = a.drop_thresh != 0;
  const uint32_t dkey = drop ? drop_key(a.drop_seed, a.drop_site) : 0u;
  __nv_bfloat16* go = reinterpret_cast<__nv_bfloat16*>(a.out) + (size_t)b * a.o_sb + (size_t)h * DH;
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
  const int slab = pass == 0 ? nslabs - 1 - warp : warp;
  if (slab < 0 || slab >= nslabs || (pass == 1 && slab >= nslabs - 1 - warp)) continue;
  const int row0 = slab * 16;
  const int r_lo = row0 + g, r_hi = row0 + g + 8;

  // ---- Q fragments from the staged tile (A operand, row-major m16k16 per k-step; x4 = rows [0,8)/[8,16) x dims [0,8)/[8,16)) ----
  uint32_t qf[KS][4];
  if (tq_pad > 0) {
#pragma unroll
    for (int ks = 0; ks < KS; ++ks)
      ldsm_x4(sQ_u + (uint32_t)(((row0 + v_row) * LDS + ks * 16 + v_col) * 2), qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
  } else {   // tq_pad == 0: Q was not staged (shared memory is better spent on a second resident CTA): fragments from global
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const int c = ks * 16 + t4 * 2;
      const __nv_bfloat16* p_lo = gq + (size_t)r_lo * a.q_st + c;
      const __nv_bfloat16* p_hi = gq + (size_t)r_hi * a.q_st + c;
      qf[ks][0] = r_lo < a.Tq ? *reinterpret_cast<const uint32_t*>(p_lo) : 0u;
      qf[ks][1] = r_hi < a.Tq ? *reinterpret_cast<const uint32_t*>(p_hi) : 0u;
      qf[ks][2] = r_lo < a.Tq ? *reinterpret_cast<const uint32_t*>(p_lo + 8) : 0u;
      qf[ks][3] = r_hi < a.Tq ? *reinterpret_cast<const uint32_t*>(p_hi + 8) : 0u;
    }
  }

  float o[NT][4];
#pragma unroll
  for (int n = 0; n < NT; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
  float m_lo = -INFINITY, m_hi = -INFINITY, l_lo = 0.f, l_hi = 0.f;
  // train-mode dropout on the probabilities: P.V uses keep ? p / (1 - p_drop) : 0, the row sums the undropped p (warp-uniform switch)
  const unsigned long long drow_lo = ((unsigned long long)blockIdx.x * a.Tq + (unsigned)r_lo) * (unsigned long long)a.Tk;
  const unsigned long long drow_hi = drow_lo + 8ull * (unsigned long long)a.Tk;

  const int k_end = a.causal ? min(a.Tk, row0 + 16) : a.Tk;   // keys this warp can ever see
  for (int kb = 0; kb < k_end; kb += KB) {
    float s[KB / 8][4];
#pragma unroll
    for (int n = 0; n < KB / 8; ++n) s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
    // ---- S = Q . K^T for 64 keys ----
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
      for (int np = 0; np < KB / 16; ++np) {      // pairs of n8 tiles (16 keys)
        uint32_t b0, b1, b2, b3;
        ldsm_x4(sK_u + (uint32_t)(((kb + np * 16 + k_row) * LDS + ks * 16 + k_col) * 2), b0, b1, b2, b3);
        mma16816(s[2 * np], qf[ks], b0, b1);       // keys [0,8) of the pair: dims [0,8), [8,16)
        mma16816(s[2 * np + 1], qf[ks], b2, b3);   // keys [8,16)
      }
    }
    // ---- mask + online softmax ----
    float mx_lo = m_lo, mx_hi = m_hi;
    const bool need_mask = !sBlkValid[kb / KB] || (a.causal && kb + KB - 1 > row0);   // warp-uniform
    if (need_mask) {
#pragma unroll
      for (int n = 0; n < KB / 8; ++n) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int j = kb + n * 8 + t4 * 2 + e;
          const bool okj = sMask[j] != 0;
          const bool ok_lo = okj && (!a.causal || j <= r_lo), ok_hi = okj && (!a.causal || j <= r_hi);
          s[n][e] = ok_lo ? s[n][e] * sl2 : -INFINITY;
          s[n][2 + e] = ok_hi ? s[n][2 + e] * sl2 : -INFINITY;
        }
      }
    } else {
#pragma unroll
      for (int n = 0; n < KB / 8; ++n) {
        s[n][0] *= sl2; s[n][1] *= sl2; s[n][2] *= sl2; s[n][3] *= sl2;
      }
    }
#pragma unroll
    for (int n = 0; n < KB / 8; ++n) {
      mx_lo = fmaxf(mx_lo, fmaxf(s[n][0], s[n][1]));
      mx_hi = fmaxf(mx_hi, fmaxf(s[n][2], s[n][3]));
    }
    mx_lo = fmaxf(mx_lo, __shfl_xor_sync(0xffffffffu, mx_lo, 1));
    mx_lo = fmaxf(mx_lo, __shfl_xor_sync(0xffffffffu, mx_lo, 2));
    mx_hi = fmaxf(mx_hi, __shfl_xor_sync(0xffffffffu, mx_hi, 1));
    mx_hi = fmaxf(mx_hi, __shfl_xor_sync(0xffffffffu, mx_hi, 2));
    // rows with nothing attendable yet keep m = -inf: use 0 as the reference point so exp2(-inf - 0) = 0
    const float ref_lo = mx_lo == -INFINITY ? 0.f : mx_lo, ref_hi = mx_hi == -INFINITY ? 0.f : mx_hi;
    const float c_lo = ex2(m_lo - ref_lo), c_hi = ex2(m_hi - ref_hi);
    m_lo = mx_lo;
    m_hi = mx_hi;
    float ps_lo = 0.f, ps_hi = 0.f;
    uint32_t pf[KB / 16][4];
#pragma unroll
    for (int n = 0; n < KB / 8; ++n) {
      float p0 = ex2(s[n][0] - ref_lo), p1 = ex2(s[n][1] - ref_lo);
      float p2 = ex2(s[n][2] - ref_hi), p3 = ex2(s[n][3] - ref_hi);
      ps_lo += p0 + p1;
      ps_hi += p2 + p3;
      if (drop) {
        const unsigned j = (unsigned)(kb + n * 8 + t4 * 2);
        p0 = drop_keep(dkey, drow_lo + j, a.drop_thresh) ? p0 * a.drop_scale : 0.f;
        p1 = drop_keep(dkey, drow_lo + j + 1, a.drop_thresh) ? p1 * a.drop_scale : 0.f;
        p2 = drop_keep(dkey, drow_hi + j, a.drop_thresh) ? p2 * a.drop_scale : 0.f;
        p3 = drop_keep(dkey, drow_hi + j + 1, a.drop_thresh) ? p3 * a.drop_scale : 0.f;
      }
      // accumulator layout of two adjacent n8 tiles == A-operand layout of one k16 step
      pf[n >> 1][(n & 1) * 2] = pack2(p0, p1);
      pf[n >> 1][(n & 1) * 2 + 1] = pack2(p2, p3);
    }
    l_lo = l_lo * c_lo + ps_lo;
    l_hi = l_hi * c_hi + ps_hi;
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      o[n][0] *= c_lo; o[n][1] *= c_lo; o[n][2] *= c_hi; o[n][3] *= c_hi;
    }
    // ---- O += P . V ----
#pragma unroll
    for (int kk = 0; kk < KB / 16; ++kk) {        // 16 keys per k-step
#pragma unroll
      for (int np = 0; np < NT / 2; ++np) {       // pairs of output n8 tiles (16 dims)
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(sV_u + (uint32_t)(((kb + kk * 16 + v_row) * LDS + np * 16 + v_col) * 2), b0, b1, b2, b3);
        mma16816(o[2 * np], pf[kk], b0, b1);       // dims [0,8): keys [0,8), [8,16)
        mma16816(o[2 * np + 1], pf[kk], b2, b3);   // dims [8,16)
      }
    }
  }
  // ---- finalize: row sums across the quad, normalise, store ----
  l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1);
  l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
  l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1);
  l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
  const float i_lo = l_lo > 0.f ? 1.f / l_lo : 0.f, i_hi = l_hi > 0.f ? 1.f / l_hi : 0.f;
  if (a.lse && t4 == 0) {        // natural log of the row sum at the base-2 reference max; -inf for a row with no visible key
    float* lse = a.lse + (size_t)b * a.lse_sb + (size_t)h * a.Tq;
    if (r_lo < a.Tq) lse[r_lo] = (m_lo + log2f(l_lo)) * 0.6931471805599453f;
    if (r_hi < a.Tq) lse[r_hi] = (m_hi + log2f(l_hi)) * 0.6931471805599453f;
  }
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    const int c = n * 8 + t4 * 2;
    if (r_lo < a.Tq) *reinterpret_cast<uint32_t*>(go + (size_t)r_lo * a.o_st + c) = pack2(o[n][0] * i_lo, o[n][1] * i_lo);
    if (r_hi < a.Tq) *reinterpret_cast<uint32_t*>(go + (size_t)r_hi * a.o_st + c) = pack2(o[n][2] * i_hi, o[n][3] * i_hi);
  }
  }   // slab passes
}

}  // namespace fa

// Returns 1 when the shape is not covered (caller falls back to the generic kernel), <= 0 otherwise.
int attention_tc_launch(const tcavp_attn_args& a, cudaStream_t stream) {
  if (!(a.dh == 16 || a.dh == 32 || a.dh == 64 || a.dh == 96 || a.dh == 128) || a.Tk > 256 || a.Tq > 256 || a.Tk < 1) return 1;
  auto al16 = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  if (!al16(a.q) || !al16(a.k) || !al16(a.v) || !al16(a.out)) return 1;
  if (a.q_sb % 8 || a.q_st % 8 || a.k_sb % 8 || a.k_st % 8 || a.v_sb % 8 || a.v_st % 8 || a.o_sb % 2 || a.o_st % 2) return 1;
  auto pad_to = [](int n, int m) { return (n + m - 1) / m * m; };
  const int kb = a.Tk <= 16 ? 16 : (pad_to(a.Tk, 48) < pad_to(a.Tk, 64) ? 48 : 64);   // keys per iteration: fewest dead keys
  const int tk_pad = pad_to(a.Tk, kb);
  const int tq_pad = a.dh >= 128 ? 0 : pad_to(a.Tq, 16);   // dh 128: K + V + Q would leave room for one CTA per SM only
  const int warps = ((a.Tq + 15) / 16 + 1) / 2;                                // every warp owns a pair of 16-row slabs (<= 8 warps)
  const size_t smem = (size_t)(2 * tk_pad + tq_pad) * (a.dh + fa::PAD) * 2 + (size_t)tk_pad * 4 + (size_t)(tk_pad / kb) * 4;
  const dim3 grid(a.B * a.H);
#define TCAVP_FLASH_KB(DH, MAXT, MINB, KB_)                                                                                       \
  do {                                                                                                                            \
    TCAVP_CUDA(cudaFuncSetAttribute(fa::attn_flash_kernel<DH, MAXT, MINB, KB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    fa::attn_flash_kernel<DH, MAXT, MINB, KB_><<<grid, warps * 32, smem, stream>>>(a, tk_pad, tq_pad);                              \
  } while (0)
#define TCAVP_FLASH(DH, MAXT, MINB)                          \
  do {                                                       \
    if (kb == 16) TCAVP_FLASH_KB(DH, MAXT, MINB, 16);        \
    else if (kb == 48) TCAVP_FLASH_KB(DH, MAXT, MINB, 48);   \
    else TCAVP_FLASH_KB(DH, MAXT, MINB, 64);                 \
  } while (0)
  if (a.dh == 64) {
    if (warps <= 5) TCAVP_FLASH(64, 160, 3);   // L <= 160: three CTAs per SM
    else TCAVP_FLASH(64, 256, 2);
  } else if (a.dh == 128) {
    if (warps <= 5) TCAVP_FLASH(128, 160, 2);
    else TCAVP_FLASH(128, 256, 1);
  } else if (a.dh == 96) {       // Q-Former heads (768 / 8)
    TCAVP_FLASH(96, 256, 1);
  } else if (a.dh == 32) {
    TCAVP_FLASH(32, 256, 2);
  } else {                       // lane-polygon encoder heads (64 / 4)
    TCAVP_FLASH(16, 256, 2);
  }
#undef TCAVP_FLASH
#undef TCAVP_FLASH_KB
  return check_launch("attn_flash_kernel");
}

}  // namespace tcavp
