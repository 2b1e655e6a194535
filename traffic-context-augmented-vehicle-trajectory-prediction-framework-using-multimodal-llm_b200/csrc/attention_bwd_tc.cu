// Tensor-core attention backward (bf16, head_dim 16/32/64/96/128, Tq, Tk <= 256, H == Hkv): the gradient of the LLM
// self-attention (HF:251-289) and of the small nn.MultiheadAttention cores, used by the fine-tune step.  Longer sequences and GQA
// run on the key-blocked kernels at the end of this file, which take the softmax statistics from the forward's logsumexp.
//
// One CTA per (batch, head).  Q, K, V and dO of the head are staged ONCE in shared memory (cp.async, padded rows); no score,
// probability or gradient tile ever touches shared or global memory, and there are no atomics:
//   pass B (query-outer, a warp owns 16-row query slabs, paired from both ends for causal balance)
//       sweep 1: S = Q K^T -> row max m_i and 1 / row sum (online softmax statistics), D_i = dO_i . O_i
//       sweep 2: S again -> P = exp2(S - m_i) / l_i;  dP = dO V^T;  dS = scale * P o (dP - D_i);  dQ += dS K   (registers)
//   pass A (key-outer, a warp owns 16-key slabs): for every query slab
//       S^T = K_J Q_I^T, dP^T = V_J dO_I^T  (computed transposed so that P^T / dS^T come out in the A-operand layout)
//       dV_J += P^T dO_I;  dK_J += dS^T Q_I                                                                 (registers)
// mma.sync m16n8k16 bf16 -> fp32.  The scores are recomputed three times instead of being stored: the contraction work is
// tiny next to the GEMMs of the step, while stored probabilities would cost B*H*L*L*2 bytes of HBM per layer.
#include "common.cuh"

namespace tcavp {
namespace fb {

constexpr int PAD = 8;

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

// KB = keys per block of the query-outer pass (48 when that pads Tk to fewer dead keys, e.g. L = 144 = 3 x 48; 64 otherwise).
template <int DH, int MAXT, int MINB, int KB>
__global__ void __launch_bounds__(MAXT, MINB) attn_bwd_tc_kernel(tcavp_attn_args a, const __nv_bfloat16* __restrict__ dout, long long do_sb,
                                                                 long long do_st, __nv_bfloat16* __restrict__ dq, long long dq_sb,
                                                                 long long dq_st, void* __restrict__ dk, long long dk_sb, long long dk_st,
                                                                 void* __restrict__ dv, long long dv_sb, long long dv_st, int dkv_bf16,
                                                                 int tq_pad, int tk_pad) {
  constexpr int LDS = DH + PAD;
  constexpr int KS = DH / 16;
  constexpr int NT = DH / 8;
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem);
  __nv_bfloat16* sdO = sQ + (size_t)tq_pad * LDS;
  __nv_bfloat16* sK = sdO + (size_t)tq_pad * LDS;
  __nv_bfloat16* sV = sK + (size_t)tk_pad * LDS;
  float* sM = reinterpret_cast<float*>(sV + (size_t)tk_pad * LDS);   // [tq_pad] row max of the scaled base-2 logits (0 if none)
  float* sIL = sM + tq_pad;                                           // [tq_pad] 1 / row sum (0 for empty / padded rows)
  float* sD = sIL + tq_pad;                                           // [tq_pad] dO_i . O_i
  int* sMask = reinterpret_cast<int*>(sD + tq_pad);                   // [tk_pad]

  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const __nv_bfloat16* gq = reinterpret_cast<const __nv_bfloat16*>(a.q) + (size_t)b * a.q_sb + (size_t)h * DH;
  const __nv_bfloat16* gk = reinterpret_cast<const __nv_bfloat16*>(a.k) + (size_t)b * a.k_sb + (size_t)h * DH;
  const __nv_bfloat16* gv = reinterpret_cast<const __nv_bfloat16*>(a.v) + (size_t)b * a.v_sb + (size_t)h * DH;
  const __nv_bfloat16* go = reinterpret_cast<const __nv_bfloat16*>(a.out) + (size_t)b * a.o_sb + (size_t)h * DH;
  const __nv_bfloat16* gdo = dout + (size_t)b * do_sb + (size_t)h * DH;

  // ---- stage Q, dO (tq_pad rows) and K, V (tk_pad rows), zero-filled beyond the real extents ----
  {
    constexpr int VPR = DH / 8;
    const uint32_t sQ_a = (uint32_t)__cvta_generic_to_shared(sQ), sdO_a = (uint32_t)__cvta_generic_to_shared(sdO);
    const uint32_t sK_a = (uint32_t)__cvta_generic_to_shared(sK), sV_a = (uint32_t)__cvta_generic_to_shared(sV);
    for (int i = threadIdx.x; i < tq_pad * VPR; i += blockDim.x) {
      const int r = i / VPR, c = (i % VPR) * 8;
      const int sz = r < a.Tq ? 16 : 0;
      const size_t rr = r < a.Tq ? r : 0;
      const uint32_t off = (uint32_t)((r * LDS + c) * 2);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sQ_a + off), "l"(gq + rr * a.q_st + c), "r"(sz) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sdO_a + off), "l"(gdo + rr * do_st + c), "r"(sz) : "memory");
    }
    for (int i = threadIdx.x; i < tk_pad * VPR; i += blockDim.x) {
      const int r = i / VPR, c = (i % VPR) * 8;
      const int sz = r < a.Tk ? 16 : 0;
      const size_t rr = r < a.Tk ? r : 0;
      const uint32_t off = (uint32_t)((r * LDS + c) * 2);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sK_a + off), "l"(gk + rr * a.k_st + c), "r"(sz) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sV_a + off), "l"(gv + rr * a.v_st + c), "r"(sz) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int j = threadIdx.x; j < tk_pad; j += blockDim.x) sMask[j] = (j < a.Tk) && (!a.key_mask || a.key_mask[(size_t)b * a.Tk + j] != 0);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const int g = lane >> 2, t4 = lane & 3;
  const uint32_t sQ_u = (uint32_t)__cvta_generic_to_shared(sQ), sdO_u = (uint32_t)__cvta_generic_to_shared(sdO);
  const uint32_t sK_u = (uint32_t)__cvta_generic_to_shared(sK), sV_u = (uint32_t)__cvta_generic_to_shared(sV);
  // ldmatrix lane offsets: A operand (16 rows x 16 k, row-major), B operand from [n][k] storage, B operand from [k][n] storage
  const int a_row = lane & 15, a_col = (lane >> 4) * 8;
  const int bn_row = (lane & 7) + ((lane >> 4) << 3), bn_col = ((lane >> 3) & 1) * 8;
  const int bk_row = (lane & 7) + (((lane >> 3) & 1) << 3), bk_col = (lane >> 4) * 8;
  const float sl2 = a.scale * 1.4426950408889634f;
  // train-mode dropout (O = P_d V, P_d = keep ? P / (1 - p_drop) : 0): dP = f o (dO V^T) with f = keep ? 1 / (1 - p_drop) : 0,
  // D_i = dO_i . O_i is unchanged, dV uses P_d.  The mask is regenerated from (seed, site, ((b*H + h)*Tq + i)*Tk + j).
  const bool drop = a.drop_thresh != 0;
  const uint32_t dkey = drop ? drop_key(a.drop_seed, a.drop_site) : 0u;
  const unsigned long long dbase = (unsigned long long)blockIdx.x * a.Tq * (unsigned long long)a.Tk;

  // =========================== pass B: statistics, D and dQ (query-outer) ===========================
  const int nqs = (a.Tq + 15) / 16;
  for (int idx = warp; idx < (nqs + 1) / 2; idx += nwarps) {
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      const int slab = pass == 0 ? nqs - 1 - idx : idx;
      if (pass == 1 && slab == nqs - 1 - idx) continue;
      const int row0 = slab * 16;
      const int r_lo = row0 + g, r_hi = row0 + g + 8;
      uint32_t qf[KS][4];
#pragma unroll
      for (int ks = 0; ks < KS; ++ks)
        ldsm_x4(sQ_u + (uint32_t)(((row0 + a_row) * LDS + ks * 16 + a_col) * 2), qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
      const int k_end = a.causal ? min(a.Tk, row0 + 16) : a.Tk;
      // ---- sweep 1: softmax statistics ----
      float m_lo = -INFINITY, m_hi = -INFINITY, l_lo = 0.f, l_hi = 0.f;
      for (int kb = 0; kb < k_end; kb += KB) {
        float s[KB / 8][4];
#pragma unroll
        for (int n = 0; n < KB / 8; ++n) s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
          for (int np = 0; np < KB / 16; ++np) {
            uint32_t b0, b1, b2, b3;
            ldsm_x4(sK_u + (uint32_t)(((kb + np * 16 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
            mma16816(s[2 * np], qf[ks], b0, b1);
            mma16816(s[2 * np + 1], qf[ks], b2, b3);
          }
        }
        float mx_lo = m_lo, mx_hi = m_hi;
#pragma unroll
        for (int n = 0; n < KB / 8; ++n) {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = kb + n * 8 + t4 * 2 + e;
            const bool okj = sMask[j] != 0;
            s[n][e] = (okj && (!a.causal || j <= r_lo)) ? s[n][e] * sl2 : -INFINITY;
            s[n][2 + e] = (okj && (!a.causal || j <= r_hi)) ? s[n][2 + e] * sl2 : -INFINITY;
          }
          mx_lo = fmaxf(mx_lo, fmaxf(s[n][0], s[n][1]));
          mx_hi = fmaxf(mx_hi, fmaxf(s[n][2], s[n][3]));
        }
        mx_lo = fmaxf(mx_lo, __shfl_xor_sync(0xffffffffu, mx_lo, 1));
        mx_lo = fmaxf(mx_lo, __shfl_xor_sync(0xffffffffu, mx_lo, 2));
        mx_hi = fmaxf(mx_hi, __shfl_xor_sync(0xffffffffu, mx_hi, 1));
        mx_hi = fmaxf(mx_hi, __shfl_xor_sync(0xffffffffu, mx_hi, 2));
        const float ref_lo = mx_lo == -INFINITY ? 0.f : mx_lo, ref_hi = mx_hi == -INFINITY ? 0.f : mx_hi;
        l_lo *= ex2(m_lo - ref_lo);
        l_hi *= ex2(m_hi - ref_hi);
        m_lo = mx_lo;
        m_hi = mx_hi;
#pragma unroll
        for (int n = 0; n < KB / 8; ++n) {
          l_lo += ex2(s[n][0] - ref_lo) + ex2(s[n][1] - ref_lo);
          l_hi += ex2(s[n][2] - ref_hi) + ex2(s[n][3] - ref_hi);
        }
      }
      l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1);
      l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
      l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1);
      l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
      const float rm_lo = m_lo == -INFINITY ? 0.f : m_lo, rm_hi = m_hi == -INFINITY ? 0.f : m_hi;
      const float il_lo = (l_lo > 0.f && r_lo < a.Tq) ? 1.f / l_lo : 0.f, il_hi = (l_hi > 0.f && r_hi < a.Tq) ? 1.f / l_hi : 0.f;
      // ---- D_i = dO_i . O_i ----
      float d_lo = 0.f, d_hi = 0.f;
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        const int c = n * 8 + t4 * 2;
        if (r_lo < a.Tq) {
          const float2 o2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(go + (size_t)r_lo * a.o_st + c));
          const float2 d2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sdO + r_lo * LDS + c));
          d_lo += o2.x * d2.x + o2.y * d2.y;
        }
        if (r_hi < a.Tq) {
          const float2 o2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(go + (size_t)r_hi * a.o_st + c));
          const float2 d2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(sdO + r_hi * LDS + c));
          d_hi += o2.x * d2.x + o2.y * d2.y;
        }
      }
      d_lo += __shfl_xor_sync(0xffffffffu, d_lo, 1);
      d_lo += __shfl_xor_sync(0xffffffffu, d_lo, 2);
      d_hi += __shfl_xor_sync(0xffffffffu, d_hi, 1);
      d_hi += __shfl_xor_sync(0xffffffffu, d_hi, 2);
      if (t4 == 0) {
        sM[r_lo] = rm_lo; sIL[r_lo] = il_lo; sD[r_lo] = d_lo;
        sM[r_hi] = rm_hi; sIL[r_hi] = il_hi; sD[r_hi] = d_hi;
      }
      // ---- sweep 2: dQ ----
      float acc[NT][4];
#pragma unroll
      for (int n = 0; n < NT; ++n) acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
      for (int kb = 0; kb < k_end; kb += KB) {
        float s[KB / 8][4], dp[KB / 8][4];
#pragma unroll
        for (int n = 0; n < KB / 8; ++n) {
          s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
          dp[n][0] = dp[n][1] = dp[n][2] = dp[n][3] = 0.f;
        }
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
          uint32_t df[4];
          ldsm_x4(sdO_u + (uint32_t)(((row0 + a_row) * LDS + ks * 16 + a_col) * 2), df[0], df[1], df[2], df[3]);
#pragma unroll
          for (int np = 0; np < KB / 16; ++np) {
            uint32_t b0, b1, b2, b3;
            ldsm_x4(sK_u + (uint32_t)(((kb + np * 16 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
            mma16816(s[2 * np], qf[ks], b0, b1);
            mma16816(s[2 * np + 1], qf[ks], b2, b3);
            ldsm_x4(sV_u + (uint32_t)(((kb + np * 16 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
            mma16816(dp[2 * np], df, b0, b1);
            mma16816(dp[2 * np + 1], df, b2, b3);
          }
        }
        uint32_t pf[KB / 16][4];
#pragma unroll
        for (int n = 0; n < KB / 8; ++n) {
          float ds[4];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = kb + n * 8 + t4 * 2 + e;
            const bool okj = sMask[j] != 0;
            const float p_lo = (okj && (!a.causal || j <= r_lo)) ? ex2(s[n][e] * sl2 - rm_lo) * il_lo : 0.f;
            const float p_hi = (okj && (!a.causal || j <= r_hi)) ? ex2(s[n][2 + e] * sl2 - rm_hi) * il_hi : 0.f;
            float g_lo = dp[n][e], g_hi = dp[n][2 + e];
            if (drop) {
              g_lo = drop_keep(dkey, dbase + (unsigned long long)r_lo * a.Tk + (unsigned)j, a.drop_thresh) ? g_lo * a.drop_scale : 0.f;
              g_hi = drop_keep(dkey, dbase + (unsigned long long)r_hi * a.Tk + (unsigned)j, a.drop_thresh) ? g_hi * a.drop_scale : 0.f;
            }
            ds[e] = a.scale * p_lo * (g_lo - d_lo);
            ds[2 + e] = a.scale * p_hi * (g_hi - d_hi);
          }
          pf[n >> 1][(n & 1) * 2] = pack2(ds[0], ds[1]);
          pf[n >> 1][(n & 1) * 2 + 1] = pack2(ds[2], ds[3]);
        }
#pragma unroll
        for (int kk = 0; kk < KB / 16; ++kk) {
#pragma unroll
          for (int np = 0; np < NT / 2; ++np) {
            uint32_t b0, b1, b2, b3;
            ldsm_x4_t(sK_u + (uint32_t)(((kb + kk * 16 + bk_row) * LDS + np * 16 + bk_col) * 2), b0, b1, b2, b3);
            mma16816(acc[2 * np], pf[kk], b0, b1);
            mma16816(acc[2 * np + 1], pf[kk], b2, b3);
          }
        }
      }
      __nv_bfloat16* gdq = dq + (size_t)b * dq_sb + (size_t)h * DH;
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        const int c = n * 8 + t4 * 2;
        if (r_lo < a.Tq) *reinterpret_cast<uint32_t*>(gdq + (size_t)r_lo * dq_st + c) = pack2(acc[n][0], acc[n][1]);
        if (r_hi < a.Tq) *reinterpret_cast<uint32_t*>(gdq + (size_t)r_hi * dq_st + c) = pack2(acc[n][2], acc[n][3]);
      }
    }
  }
  __syncthreads();

  // =========================== pass A: dK, dV (key-outer) ===========================
  const int nks = (a.Tk + 15) / 16;
  for (int idx = warp; idx < (nks + 1) / 2; idx += nwarps) {
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      const int slab = pass == 0 ? idx : nks - 1 - idx;      // causal: key slab 0 sees every query slab, the last one only one
      if (pass == 1 && slab == idx) continue;
      const int j0 = slab * 16;
      const int j_lo = j0 + g, j_hi = j0 + g + 8;
      const bool ok_lo = sMask[j_lo] != 0, ok_hi = sMask[j_hi] != 0;
      float ak[NT][4], av[NT][4];
#pragma unroll
      for (int n = 0; n < NT; ++n) {
        ak[n][0] = ak[n][1] = ak[n][2] = ak[n][3] = 0.f;
        av[n][0] = av[n][1] = av[n][2] = av[n][3] = 0.f;
      }
      const int i_begin = a.causal ? j0 : 0;                 // queries i < j0 see none of this slab's keys
      for (int i0 = i_begin; i0 < tq_pad; i0 += 16) {
        float st[2][4], dpt[2][4];                           // S^T and dP^T: rows = keys (lo / hi), cols = queries i0 + n*8 + 2*t4 + e
#pragma unroll
        for (int n = 0; n < 2; ++n) {
          st[n][0] = st[n][1] = st[n][2] = st[n][3] = 0.f;
          dpt[n][0] = dpt[n][1] = dpt[n][2] = dpt[n][3] = 0.f;
        }
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
          uint32_t kf[4], vf[4], b0, b1, b2, b3;
          ldsm_x4(sK_u + (uint32_t)(((j0 + a_row) * LDS + ks * 16 + a_col) * 2), kf[0], kf[1], kf[2], kf[3]);
          ldsm_x4(sV_u + (uint32_t)(((j0 + a_row) * LDS + ks * 16 + a_col) * 2), vf[0], vf[1], vf[2], vf[3]);
          ldsm_x4(sQ_u + (uint32_t)(((i0 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
          mma16816(st[0], kf, b0, b1);
          mma16816(st[1], kf, b2, b3);
          ldsm_x4(sdO_u + (uint32_t)(((i0 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
          mma16816(dpt[0], vf, b0, b1);
          mma16816(dpt[1], vf, b2, b3);
        }
        uint32_t pT[4], dsT[4];
#pragma unroll
        for (int n = 0; n < 2; ++n) {
          float p[4], ds[4];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int i = i0 + n * 8 + t4 * 2 + e;
            const float m = sM[i], il = sIL[i], D = sD[i];
            p[e] = (ok_lo && (!a.causal || j_lo <= i)) ? ex2(st[n][e] * sl2 - m) * il : 0.f;
            p[2 + e] = (ok_hi && (!a.causal || j_hi <= i)) ? ex2(st[n][2 + e] * sl2 - m) * il : 0.f;
            float g_lo = dpt[n][e], g_hi = dpt[n][2 + e];
            float f_lo = 1.f, f_hi = 1.f;
            if (drop) {
              const unsigned long long irow = dbase + (unsigned long long)i * a.Tk;
              f_lo = drop_keep(dkey, irow + (unsigned)j_lo, a.drop_thresh) ? a.drop_scale : 0.f;
              f_hi = drop_keep(dkey, irow + (unsigned)j_hi, a.drop_thresh) ? a.drop_scale : 0.f;
              g_lo *= f_lo;
              g_hi *= f_hi;
            }
            ds[e] = a.scale * p[e] * (g_lo - D);
            ds[2 + e] = a.scale * p[2 + e] * (g_hi - D);
            p[e] *= f_lo;            // dV_J += P_d^T dO
            p[2 + e] *= f_hi;
          }
          pT[n * 2] = pack2(p[0], p[1]);
          pT[n * 2 + 1] = pack2(p[2], p[3]);
          dsT[n * 2] = pack2(ds[0], ds[1]);
          dsT[n * 2 + 1] = pack2(ds[2], ds[3]);
        }
#pragma unroll
        for (int np = 0; np < NT / 2; ++np) {
          uint32_t b0, b1, b2, b3;
          ldsm_x4_t(sdO_u + (uint32_t)(((i0 + bk_row) * LDS + np * 16 + bk_col) * 2), b0, b1, b2, b3);
          mma16816(av[2 * np], pT, b0, b1);
          mma16816(av[2 * np + 1], pT, b2, b3);
          ldsm_x4_t(sQ_u + (uint32_t)(((i0 + bk_row) * LDS + np * 16 + bk_col) * 2), b0, b1, b2, b3);
          mma16816(ak[2 * np], dsT, b0, b1);
          mma16816(ak[2 * np + 1], dsT, b2, b3);
        }
      }
      if (dkv_bf16) {     // this CTA owns every key row of its head: the activation dtype is written directly (no fp32 round trip)
        __nv_bfloat16* gdk = reinterpret_cast<__nv_bfloat16*>(dk) + (size_t)b * dk_sb + (size_t)h * DH;
        __nv_bfloat16* gdv = reinterpret_cast<__nv_bfloat16*>(dv) + (size_t)b * dv_sb + (size_t)h * DH;
#pragma unroll
        for (int n = 0; n < NT; ++n) {
          const int c = n * 8 + t4 * 2;
          if (j_lo < a.Tk) {
            *reinterpret_cast<uint32_t*>(gdk + (size_t)j_lo * dk_st + c) = pack2(ak[n][0], ak[n][1]);
            *reinterpret_cast<uint32_t*>(gdv + (size_t)j_lo * dv_st + c) = pack2(av[n][0], av[n][1]);
          }
          if (j_hi < a.Tk) {
            *reinterpret_cast<uint32_t*>(gdk + (size_t)j_hi * dk_st + c) = pack2(ak[n][2], ak[n][3]);
            *reinterpret_cast<uint32_t*>(gdv + (size_t)j_hi * dv_st + c) = pack2(av[n][2], av[n][3]);
          }
        }
      } else {
        float* gdk = reinterpret_cast<float*>(dk) + (size_t)b * dk_sb + (size_t)h * DH;
        float* gdv = reinterpret_cast<float*>(dv) + (size_t)b * dv_sb + (size_t)h * DH;
#pragma unroll
        for (int n = 0; n < NT; ++n) {
          const int c = n * 8 + t4 * 2;
          if (j_lo < a.Tk) {
            *reinterpret_cast<float2*>(gdk + (size_t)j_lo * dk_st + c) = make_float2(ak[n][0], ak[n][1]);
            *reinterpret_cast<float2*>(gdv + (size_t)j_lo * dv_st + c) = make_float2(av[n][0], av[n][1]);
          }
          if (j_hi < a.Tk) {
            *reinterpret_cast<float2*>(gdk + (size_t)j_hi * dk_st + c) = make_float2(ak[n][2], ak[n][3]);
            *reinterpret_cast<float2*>(gdv + (size_t)j_hi * dv_st + c) = make_float2(av[n][2], av[n][3]);
          }
        }
      }
    }
  }
}

// ================================================================================================
// Key-blocked backward from the forward's logsumexp (bf16, head_dim 64 / 128, any length, GQA): attn_bwd_kv_kernel + attn_bwd_q_kernel.
// P_ij = exp2(s_ij * scale * log2(e) - lse2_i) is recomputed from Q, K and the forward's row logsumexp (lse2 = lse * log2(e)), so no
// CTA has to see a whole key range to rebuild the softmax statistics; D_i = dO_i . O_i is recomputed where it is needed.
//   attn_bwd_kv_kernel  a CTA owns (scene, KV head, 64-key block), a warp 16 of its keys; it sweeps, in a fixed order, the query
//                       heads of its GQA group and the 64-row query chunks the causal mask lets see the block (double-buffered
//                       cp.async staging): dV += P^T dO, dK += dS^T Q in registers, then one plain store per key row.  The GQA sum
//                       over the group's query heads happens inside the CTA: no atomics, no fp32 staging, deterministic.
//   attn_bwd_q_kernel   a CTA owns (scene, query head, 64-row query block), a warp 16 rows; it sweeps the key blocks up to the
//                       causal bound (double-buffered K / V): dQ += dS K.
// ================================================================================================
constexpr int BQ = 64;        // query rows per chunk / block
constexpr int BK = 64;        // keys per block

// D_i = dO_i . O_i for rows [r0, r0 + 16) of one head, one warp: two lanes per row, each with all of its 16-byte loads of O and dO in
// flight at once (one global round trip per call); rows >= Tq get 0
template <int DH>
__device__ __forceinline__ void rows_d(const __nv_bfloat16* go, long long o_st, const __nv_bfloat16* gdo, long long do_st, int r0, int Tq,
                                       float* sD, int lane) {
  constexpr int NV = DH / 16;                                          // 16-byte vectors per half row
  const int r = r0 + (lane >> 1), c0 = (lane & 1) * (DH / 2);
  float d = 0.f;
  if (r < Tq) {
    uint4 o[NV], g[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      o[i] = *reinterpret_cast<const uint4*>(go + (size_t)r * o_st + c0 + 8 * i);
      g[i] = *reinterpret_cast<const uint4*>(gdo + (size_t)r * do_st + c0 + 8 * i);
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const __nv_bfloat162* op = reinterpret_cast<const __nv_bfloat162*>(&o[i]);
      const __nv_bfloat162* gp = reinterpret_cast<const __nv_bfloat162*>(&g[i]);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 a = __bfloat1622float2(op[e]), b = __bfloat1622float2(gp[e]);
        d += a.x * b.x + a.y * b.y;
      }
    }
  }
  d += __shfl_xor_sync(0xffffffffu, d, 1);
  if ((lane & 1) == 0) sD[lane >> 1] = d;
}
// base-2 logsumexp of a row; +inf for rows past Tq and rows with no visible key, so that exp2(x - lse2) = 0 there
__device__ __forceinline__ float row_lse2(const float* lse, int i, int Tq) {
  if (i >= Tq) return INFINITY;
  const float v = __ldg(lse + i);
  return v == -INFINITY ? INFINITY : v * 1.4426950408889634f;
}
// 16-byte cp.async of `rows` rows x DH columns into padded shared rows, zero-filled beyond `valid`
template <int DH>
__device__ __forceinline__ void stage_rows(uint32_t dst, const __nv_bfloat16* src, long long st, int rows, int valid) {
  constexpr int VPR = DH / 8;
  for (int i = threadIdx.x; i < rows * VPR; i += blockDim.x) {
    const int r = i / VPR, c = (i % VPR) * 8;
    const int sz = r < valid ? 16 : 0;
    const size_t rr = r < valid ? r : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + (uint32_t)((r * (DH + PAD) + c) * 2)), "l"(src + rr * st + c), "r"(sz)
                 : "memory");
  }
}

template <int DH>
__global__ void __launch_bounds__(128) attn_bwd_kv_kernel(tcavp_attn_args a, const __nv_bfloat16* __restrict__ dout, long long do_sb,
                                                          long long do_st, void* __restrict__ dk, long long dk_sb, long long dk_st,
                                                          void* __restrict__ dv, long long dv_sb, long long dv_st, int dkv_bf16) {
  constexpr int LDS = DH + PAD;
  constexpr int KS = DH / 16;
  constexpr int NT = DH / 8;
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sK = reinterpret_cast<__nv_bfloat16*>(smem);          // [BK][LDS]
  __nv_bfloat16* sV = sK + BK * LDS;
  __nv_bfloat16* sQ = sV + BK * LDS;                                   // [2][BQ][LDS]
  __nv_bfloat16* sdO = sQ + 2 * BQ * LDS;                              // [2][BQ][LDS]
  float* sL = reinterpret_cast<float*>(sdO + 2 * BQ * LDS);            // [2][BQ] base-2 logsumexp
  float* sD = sL + 2 * BQ;                                             // [2][BQ]
  int* sMask = reinterpret_cast<int*>(sD + 2 * BQ);                    // [BK]

  const int bhk = a.B * a.Hkv;
  const int kb = blockIdx.x / bhk;                                     // low key blocks (the most causal work) first
  const int b = (blockIdx.x % bhk) / a.Hkv, hk = (blockIdx.x % bhk) % a.Hkv;
  const int hrep = a.H / a.Hkv;
  const int j0 = kb * BK;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const float sl2 = a.scale * 1.4426950408889634f;

  const __nv_bfloat16* gk = reinterpret_cast<const __nv_bfloat16*>(a.k) + (size_t)b * a.k_sb + (size_t)j0 * a.k_st + (size_t)hk * DH;
  const __nv_bfloat16* gv = reinterpret_cast<const __nv_bfloat16*>(a.v) + (size_t)b * a.v_sb + (size_t)j0 * a.v_st + (size_t)hk * DH;
  const uint32_t sK_u = (uint32_t)__cvta_generic_to_shared(sK), sV_u = (uint32_t)__cvta_generic_to_shared(sV);
  const uint32_t sQ_u = (uint32_t)__cvta_generic_to_shared(sQ), sdO_u = (uint32_t)__cvta_generic_to_shared(sdO);
  stage_rows<DH>(sK_u, gk, a.k_st, BK, a.Tk - j0);
  stage_rows<DH>(sV_u, gv, a.v_st, BK, a.Tk - j0);
  for (int j = threadIdx.x; j < BK; j += blockDim.x)
    sMask[j] = (j0 + j < a.Tk) && (!a.key_mask || a.key_mask[(size_t)b * a.Tk + j0 + j] != 0);

  // the (query head, query chunk) sweep, in a fixed order
  const int c_begin = a.causal ? j0 / BQ : 0;                          // chunks wholly before the block see none of its keys
  const int nchunk = (a.Tq + BQ - 1) / BQ - c_begin;
  const int total = hrep * nchunk;
  auto load = [&](int it, int buf) {
    const int h = hk * hrep + it / nchunk, i0 = (c_begin + it % nchunk) * BQ;
    const __nv_bfloat16* gq = reinterpret_cast<const __nv_bfloat16*>(a.q) + (size_t)b * a.q_sb + (size_t)i0 * a.q_st + (size_t)h * DH;
    const __nv_bfloat16* gdo = dout + (size_t)b * do_sb + (size_t)i0 * do_st + (size_t)h * DH;
    stage_rows<DH>(sQ_u + (uint32_t)(buf * BQ * LDS * 2), gq, a.q_st, BQ, a.Tq - i0);
    stage_rows<DH>(sdO_u + (uint32_t)(buf * BQ * LDS * 2), gdo, do_st, BQ, a.Tq - i0);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const float* lse = a.lse + (size_t)b * a.lse_sb + (size_t)h * a.Tq;
    for (int r = threadIdx.x; r < BQ; r += blockDim.x) sL[buf * BQ + r] = row_lse2(lse, i0 + r, a.Tq);
    const __nv_bfloat16* go = reinterpret_cast<const __nv_bfloat16*>(a.out) + (size_t)b * a.o_sb + (size_t)h * DH;
    rows_d<DH>(go, a.o_st, dout + (size_t)b * do_sb + (size_t)h * DH, do_st, i0 + warp * 16, a.Tq, sD + buf * BQ + warp * 16, lane);
  };

  const int a_row = lane & 15, a_col = (lane >> 4) * 8;
  const int bn_row = (lane & 7) + ((lane >> 4) << 3), bn_col = ((lane >> 3) & 1) * 8;
  const int bk_row = (lane & 7) + (((lane >> 3) & 1) << 3), bk_col = (lane >> 4) * 8;
  const int jw = warp * 16;                                            // this warp's keys within the block
  float ak[NT][4], av[NT][4];
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    ak[n][0] = ak[n][1] = ak[n][2] = ak[n][3] = 0.f;
    av[n][0] = av[n][1] = av[n][2] = av[n][3] = 0.f;
  }
  if (total > 0) load(0, 0);
  else asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
  for (int it = 0; it < total; ++it) {
    const int buf = it & 1;
    if (it + 1 < total) {
      load(it + 1, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const int i0 = (c_begin + it % nchunk) * BQ;
    const bool ok_lo = sMask[jw + g] != 0, ok_hi = sMask[jw + g + 8] != 0;
    const int j_lo = j0 + jw + g, j_hi = j_lo + 8;
    const uint32_t q_u = sQ_u + (uint32_t)(buf * BQ * LDS * 2), do_u = sdO_u + (uint32_t)(buf * BQ * LDS * 2);
    const float* cL = sL + buf * BQ;
    const float* cD = sD + buf * BQ;
    for (int ii = 0; ii < BQ; ii += 16) {
      if (i0 + ii >= a.Tq || (a.causal && i0 + ii + 15 < j0 + jw)) continue;   // warp-uniform
      float st[2][4], dpt[2][4];
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        st[n][0] = st[n][1] = st[n][2] = st[n][3] = 0.f;
        dpt[n][0] = dpt[n][1] = dpt[n][2] = dpt[n][3] = 0.f;
      }
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t kf[4], vf[4], b0, b1, b2, b3;
        ldsm_x4(sK_u + (uint32_t)(((jw + a_row) * LDS + ks * 16 + a_col) * 2), kf[0], kf[1], kf[2], kf[3]);
        ldsm_x4(sV_u + (uint32_t)(((jw + a_row) * LDS + ks * 16 + a_col) * 2), vf[0], vf[1], vf[2], vf[3]);
        ldsm_x4(q_u + (uint32_t)(((ii + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
        mma16816(st[0], kf, b0, b1);
        mma16816(st[1], kf, b2, b3);
        ldsm_x4(do_u + (uint32_t)(((ii + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
        mma16816(dpt[0], vf, b0, b1);
        mma16816(dpt[1], vf, b2, b3);
      }
      uint32_t pT[4], dsT[4];
#pragma unroll
      for (int n = 0; n < 2; ++n) {
        float p[4], ds[4];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int il = ii + n * 8 + t4 * 2 + e, i = i0 + il;
          const float l2 = cL[il], D = cD[il];
          p[e] = (ok_lo && (!a.causal || j_lo <= i)) ? ex2(st[n][e] * sl2 - l2) : 0.f;
          p[2 + e] = (ok_hi && (!a.causal || j_hi <= i)) ? ex2(st[n][2 + e] * sl2 - l2) : 0.f;
          ds[e] = a.scale * p[e] * (dpt[n][e] - D);
          ds[2 + e] = a.scale * p[2 + e] * (dpt[n][2 + e] - D);
        }
        pT[n * 2] = pack2(p[0], p[1]);
        pT[n * 2 + 1] = pack2(p[2], p[3]);
        dsT[n * 2] = pack2(ds[0], ds[1]);
        dsT[n * 2 + 1] = pack2(ds[2], ds[3]);
      }
#pragma unroll
      for (int np = 0; np < NT / 2; ++np) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(do_u + (uint32_t)(((ii + bk_row) * LDS + np * 16 + bk_col) * 2), b0, b1, b2, b3);
        mma16816(av[2 * np], pT, b0, b1);
        mma16816(av[2 * np + 1], pT, b2, b3);
        ldsm_x4_t(q_u + (uint32_t)(((ii + bk_row) * LDS + np * 16 + bk_col) * 2), b0, b1, b2, b3);
        mma16816(ak[2 * np], dsT, b0, b1);
        mma16816(ak[2 * np + 1], dsT, b2, b3);
      }
    }
    __syncthreads();       // buffer `buf` is refilled by the next iteration's prefetch
  }
  const int j_lo = j0 + jw + g, j_hi = j_lo + 8;
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    const int c = n * 8 + t4 * 2;
    if (dkv_bf16) {
      __nv_bfloat16* gdk = reinterpret_cast<__nv_bfloat16*>(dk) + (size_t)b * dk_sb + (size_t)hk * DH + c;
      __nv_bfloat16* gdv = reinterpret_cast<__nv_bfloat16*>(dv) + (size_t)b * dv_sb + (size_t)hk * DH + c;
      if (j_lo < a.Tk) {
        *reinterpret_cast<uint32_t*>(gdk + (size_t)j_lo * dk_st) = pack2(ak[n][0], ak[n][1]);
        *reinterpret_cast<uint32_t*>(gdv + (size_t)j_lo * dv_st) = pack2(av[n][0], av[n][1]);
      }
      if (j_hi < a.Tk) {
        *reinterpret_cast<uint32_t*>(gdk + (size_t)j_hi * dk_st) = pack2(ak[n][2], ak[n][3]);
        *reinterpret_cast<uint32_t*>(gdv + (size_t)j_hi * dv_st) = pack2(av[n][2], av[n][3]);
      }
    } else {
      float* gdk = reinterpret_cast<float*>(dk) + (size_t)b * dk_sb + (size_t)hk * DH + c;
      float* gdv = reinterpret_cast<float*>(dv) + (size_t)b * dv_sb + (size_t)hk * DH + c;
      if (j_lo < a.Tk) {
        *reinterpret_cast<float2*>(gdk + (size_t)j_lo * dk_st) = make_float2(ak[n][0], ak[n][1]);
        *reinterpret_cast<float2*>(gdv + (size_t)j_lo * dv_st) = make_float2(av[n][0], av[n][1]);
      }
      if (j_hi < a.Tk) {
        *reinterpret_cast<float2*>(gdk + (size_t)j_hi * dk_st) = make_float2(ak[n][2], ak[n][3]);
        *reinterpret_cast<float2*>(gdv + (size_t)j_hi * dv_st) = make_float2(av[n][2], av[n][3]);
      }
    }
  }
}

template <int DH>
__global__ void __launch_bounds__(128) attn_bwd_q_kernel(tcavp_attn_args a, const __nv_bfloat16* __restrict__ dout, long long do_sb,
                                                         long long do_st, __nv_bfloat16* __restrict__ dq, long long dq_sb, long long dq_st) {
  constexpr int LDS = DH + PAD;
  constexpr int KS = DH / 16;
  constexpr int NT = DH / 8;
  extern __shared__ __align__(16) uint8_t smem[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(smem);          // [BQ][LDS]
  __nv_bfloat16* sdO = sQ + BQ * LDS;
  __nv_bfloat16* sK = sdO + BQ * LDS;                                  // [2][BK][LDS]
  __nv_bfloat16* sV = sK + 2 * BK * LDS;                               // [2][BK][LDS]
  float* sD = reinterpret_cast<float*>(sV + 2 * BK * LDS);             // [BQ]
  int* sMask = reinterpret_cast<int*>(sD + BQ);                        // [2][BK]

  const int bh = a.B * a.H;
  const int nqb = (a.Tq + BQ - 1) / BQ;
  const int qb = nqb - 1 - (int)blockIdx.x / bh;                       // high query blocks (the most causal work) first
  const int b = (blockIdx.x % bh) / a.H, h = (blockIdx.x % bh) % a.H;
  const int hk = h / (a.H / a.Hkv);
  const int i0 = qb * BQ;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const float sl2 = a.scale * 1.4426950408889634f;

  const __nv_bfloat16* gq = reinterpret_cast<const __nv_bfloat16*>(a.q) + (size_t)b * a.q_sb + (size_t)i0 * a.q_st + (size_t)h * DH;
  const __nv_bfloat16* gdo = dout + (size_t)b * do_sb + (size_t)h * DH;
  const __nv_bfloat16* gk = reinterpret_cast<const __nv_bfloat16*>(a.k) + (size_t)b * a.k_sb + (size_t)hk * DH;
  const __nv_bfloat16* gv = reinterpret_cast<const __nv_bfloat16*>(a.v) + (size_t)b * a.v_sb + (size_t)hk * DH;
  const uint32_t sQ_u = (uint32_t)__cvta_generic_to_shared(sQ), sdO_u = (uint32_t)__cvta_generic_to_shared(sdO);
  const uint32_t sK_u = (uint32_t)__cvta_generic_to_shared(sK), sV_u = (uint32_t)__cvta_generic_to_shared(sV);
  stage_rows<DH>(sQ_u, gq, a.q_st, BQ, a.Tq - i0);
  stage_rows<DH>(sdO_u, gdo + (size_t)i0 * do_st, do_st, BQ, a.Tq - i0);
  const int k_end = a.causal ? min(a.Tk, i0 + BQ) : a.Tk;
  const int nkb = (k_end + BK - 1) / BK;
  auto load = [&](int kb, int buf) {
    const int j0 = kb * BK;
    stage_rows<DH>(sK_u + (uint32_t)(buf * BK * LDS * 2), gk + (size_t)j0 * a.k_st, a.k_st, BK, a.Tk - j0);
    stage_rows<DH>(sV_u + (uint32_t)(buf * BK * LDS * 2), gv + (size_t)j0 * a.v_st, a.v_st, BK, a.Tk - j0);
    asm volatile("cp.async.commit_group;" ::: "memory");
    for (int j = threadIdx.x; j < BK; j += blockDim.x)
      sMask[buf * BK + j] = (j0 + j < a.Tk) && (!a.key_mask || a.key_mask[(size_t)b * a.Tk + j0 + j] != 0);
  };
  if (nkb > 0) load(0, 0);     // (commits the Q / dO copies in the same group)
  else asm volatile("cp.async.commit_group;" ::: "memory");
  const __nv_bfloat16* go = reinterpret_cast<const __nv_bfloat16*>(a.out) + (size_t)b * a.o_sb + (size_t)h * DH;
  rows_d<DH>(go, a.o_st, gdo, do_st, i0 + warp * 16, a.Tq, sD + warp * 16, lane);
  __syncwarp();
  const int row0 = warp * 16;                                          // this warp's rows within the block
  const int r_lo = i0 + row0 + g, r_hi = r_lo + 8;
  const float* lse = a.lse + (size_t)b * a.lse_sb + (size_t)h * a.Tq;
  const float l2_lo = row_lse2(lse, r_lo, a.Tq), l2_hi = row_lse2(lse, r_hi, a.Tq);
  const float d_lo = sD[row0 + g], d_hi = sD[row0 + g + 8];

  const int a_row = lane & 15, a_col = (lane >> 4) * 8;
  const int bn_row = (lane & 7) + ((lane >> 4) << 3), bn_col = ((lane >> 3) & 1) * 8;
  const int bk_row = (lane & 7) + (((lane >> 3) & 1) << 3), bk_col = (lane >> 4) * 8;
  float acc[NT][4];
#pragma unroll
  for (int n = 0; n < NT; ++n) acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
  for (int kb = 0; kb < nkb; ++kb) {
    const int buf = kb & 1;
    if (kb + 1 < nkb) {
      load(kb + 1, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const int j0 = kb * BK;
    if (i0 + row0 < a.Tq && !(a.causal && j0 > i0 + row0 + 15)) {     // warp-uniform
      uint32_t qf[KS][4];
#pragma unroll
      for (int ks = 0; ks < KS; ++ks)
        ldsm_x4(sQ_u + (uint32_t)(((row0 + a_row) * LDS + ks * 16 + a_col) * 2), qf[ks][0], qf[ks][1], qf[ks][2], qf[ks][3]);
      const uint32_t k_u = sK_u + (uint32_t)(buf * BK * LDS * 2), v_u = sV_u + (uint32_t)(buf * BK * LDS * 2);
      const int* m = sMask + buf * BK;
      float s[BK / 8][4], dp[BK / 8][4];
#pragma unroll
      for (int n = 0; n < BK / 8; ++n) {
        s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
        dp[n][0] = dp[n][1] = dp[n][2] = dp[n][3] = 0.f;
      }
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        uint32_t df[4];
        ldsm_x4(sdO_u + (uint32_t)(((row0 + a_row) * LDS + ks * 16 + a_col) * 2), df[0], df[1], df[2], df[3]);
#pragma unroll
        for (int np = 0; np < BK / 16; ++np) {
          uint32_t b0, b1, b2, b3;
          ldsm_x4(k_u + (uint32_t)(((np * 16 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
          mma16816(s[2 * np], qf[ks], b0, b1);
          mma16816(s[2 * np + 1], qf[ks], b2, b3);
          ldsm_x4(v_u + (uint32_t)(((np * 16 + bn_row) * LDS + ks * 16 + bn_col) * 2), b0, b1, b2, b3);
          mma16816(dp[2 * np], df, b0, b1);
          mma16816(dp[2 * np + 1], df, b2, b3);
        }
      }
      uint32_t pf[BK / 16][4];
#pragma unroll
      for (int n = 0; n < BK / 8; ++n) {
        float ds[4];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int jl = n * 8 + t4 * 2 + e, j = j0 + jl;
          const bool okj = m[jl] != 0;
          const float p_lo = (okj && (!a.causal || j <= r_lo)) ? ex2(s[n][e] * sl2 - l2_lo) : 0.f;
          const float p_hi = (okj && (!a.causal || j <= r_hi)) ? ex2(s[n][2 + e] * sl2 - l2_hi) : 0.f;
          ds[e] = a.scale * p_lo * (dp[n][e] - d_lo);
          ds[2 + e] = a.scale * p_hi * (dp[n][2 + e] - d_hi);
        }
        pf[n >> 1][(n & 1) * 2] = pack2(ds[0], ds[1]);
        pf[n >> 1][(n & 1) * 2 + 1] = pack2(ds[2], ds[3]);
      }
#pragma unroll
      for (int kk = 0; kk < BK / 16; ++kk) {
#pragma unroll
        for (int np = 0; np < NT / 2; ++np) {
          uint32_t b0, b1, b2, b3;
          ldsm_x4_t(k_u + (uint32_t)(((kk * 16 + bk_row) * LDS + np * 16 + bk_col) * 2), b0, b1, b2, b3);
          mma16816(acc[2 * np], pf[kk], b0, b1);
          mma16816(acc[2 * np + 1], pf[kk], b2, b3);
        }
      }
    }
    __syncthreads();
  }
  __nv_bfloat16* gdq = dq + (size_t)b * dq_sb + (size_t)h * DH;
#pragma unroll
  for (int n = 0; n < NT; ++n) {
    const int c = n * 8 + t4 * 2;
    if (r_lo < a.Tq) *reinterpret_cast<uint32_t*>(gdq + (size_t)r_lo * dq_st + c) = pack2(acc[n][0], acc[n][1]);
    if (r_hi < a.Tq) *reinterpret_cast<uint32_t*>(gdq + (size_t)r_hi * dq_st + c) = pack2(acc[n][2], acc[n][3]);
  }
}

}  // namespace fb

// Returns 1 when the shape is not covered, <= 0 otherwise.  Needs the forward output (args->out) and its logsumexp (args->lse).
int attention_bwd_blk_launch(const tcavp_attn_args& a, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                             long long dq_st, void* dk, long long dk_sb, long long dk_st, void* dv, long long dv_sb, long long dv_st,
                             int dkv_dtype, cudaStream_t stream) {
  if (a.dtype != TCAVP_BF16 || a.out == nullptr || a.lse == nullptr || a.drop_thresh != 0 || !(a.dh == 64 || a.dh == 128)) return 1;
  if (!(a.Tk > 256 || a.Tq > 256 || a.H != a.Hkv)) return 1;         // MHA at <= 256 positions: attn_bwd_tc_kernel
  auto al16 = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  if (!al16(a.q) || !al16(a.k) || !al16(a.v) || !al16(dout) || !al16(a.out) || reinterpret_cast<uintptr_t>(dq) % 4 ||
      reinterpret_cast<uintptr_t>(dk) % 8 || reinterpret_cast<uintptr_t>(dv) % 8)
    return 1;
  if (a.q_sb % 8 || a.q_st % 8 || a.k_sb % 8 || a.k_st % 8 || a.v_sb % 8 || a.v_st % 8 || do_sb % 8 || do_st % 8 || a.o_sb % 8 || a.o_st % 8 ||
      dq_sb % 2 || dq_st % 2 || dk_sb % 2 || dk_st % 2 || dv_sb % 2 || dv_st % 2)
    return 1;
  const int nkb = (a.Tk + fb::BK - 1) / fb::BK, nqb = (a.Tq + fb::BQ - 1) / fb::BQ;
  if ((long long)nkb * a.B * a.Hkv > 0x7fffffffLL || (long long)nqb * a.B * a.H > 0x7fffffffLL) return 1;
  const size_t lds = (size_t)(a.dh + fb::PAD) * 2;
  const size_t smem_kv = (size_t)(fb::BK + fb::BK + 4 * fb::BQ) * lds + (size_t)4 * fb::BQ * 4 + (size_t)fb::BK * 4;
  const size_t smem_q = (size_t)(2 * fb::BQ + 4 * fb::BK) * lds + (size_t)fb::BQ * 4 + (size_t)2 * fb::BK * 4;
  const int bf = dkv_dtype == TCAVP_BF16 ? 1 : 0;
  const __nv_bfloat16* dob = reinterpret_cast<const __nv_bfloat16*>(dout);
  __nv_bfloat16* dqb = reinterpret_cast<__nv_bfloat16*>(dq);
  if (a.dh == 64) {
    TCAVP_CUDA(cudaFuncSetAttribute(fb::attn_bwd_kv_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_kv));
    fb::attn_bwd_kv_kernel<64><<<nkb * a.B * a.Hkv, 128, smem_kv, stream>>>(a, dob, do_sb, do_st, dk, dk_sb, dk_st, dv, dv_sb, dv_st, bf);
    int rc = check_launch("attn_bwd_kv_kernel");
    if (rc) return rc;
    TCAVP_CUDA(cudaFuncSetAttribute(fb::attn_bwd_q_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_q));
    fb::attn_bwd_q_kernel<64><<<nqb * a.B * a.H, 128, smem_q, stream>>>(a, dob, do_sb, do_st, dqb, dq_sb, dq_st);
  } else {
    TCAVP_CUDA(cudaFuncSetAttribute(fb::attn_bwd_kv_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_kv));
    fb::attn_bwd_kv_kernel<128><<<nkb * a.B * a.Hkv, 128, smem_kv, stream>>>(a, dob, do_sb, do_st, dk, dk_sb, dk_st, dv, dv_sb, dv_st, bf);
    int rc = check_launch("attn_bwd_kv_kernel");
    if (rc) return rc;
    TCAVP_CUDA(cudaFuncSetAttribute(fb::attn_bwd_q_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_q));
    fb::attn_bwd_q_kernel<128><<<nqb * a.B * a.H, 128, smem_q, stream>>>(a, dob, do_sb, do_st, dqb, dq_sb, dq_st);
  }
  return check_launch("attn_bwd_q_kernel");
}

// Returns 1 when the shape is not covered (caller uses the generic SIMT kernel), <= 0 otherwise.
int attention_bwd_tc_launch(const tcavp_attn_args& a, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                            long long dq_st, void* dk, long long dk_sb, long long dk_st, void* dv, long long dv_sb, long long dv_st,
                            int dkv_dtype, cudaStream_t stream) {
  if (a.dtype != TCAVP_BF16 || a.out == nullptr || a.H != a.Hkv) return 1;
  if (!(a.dh == 16 || a.dh == 32 || a.dh == 64 || a.dh == 96 || a.dh == 128) || a.Tk > 256 || a.Tq > 256) return 1;
  auto al16 = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  if (!al16(a.q) || !al16(a.k) || !al16(a.v) || !al16(dout) || reinterpret_cast<uintptr_t>(a.out) % 4 || reinterpret_cast<uintptr_t>(dq) % 4 ||
      reinterpret_cast<uintptr_t>(dk) % 8 || reinterpret_cast<uintptr_t>(dv) % 8)
    return 1;
  if (a.q_sb % 8 || a.q_st % 8 || a.k_sb % 8 || a.k_st % 8 || a.v_sb % 8 || a.v_st % 8 || do_sb % 8 || do_st % 8 || a.o_sb % 2 || a.o_st % 2 ||
      dq_sb % 2 || dq_st % 2 || dk_sb % 2 || dk_st % 2 || dv_sb % 2 || dv_st % 2)
    return 1;
  const int tq_pad = (a.Tq + 15) / 16 * 16;
  auto pad_to = [](int n, int m) { return (n + m - 1) / m * m; };
  const int kb = pad_to(a.Tk, 48) < pad_to(a.Tk, 64) ? 48 : 64;
  const int tk_pad = pad_to(a.Tk, kb);
  const int nqs = (a.Tq + 15) / 16, nks = (a.Tk + 15) / 16;
  const int slabs = nqs > nks ? nqs : nks;
  int warps = (slabs + 1) / 2;
  if (warps > 8) warps = 8;
  const size_t smem = (size_t)2 * (tq_pad + tk_pad) * (a.dh + fb::PAD) * 2 + (size_t)3 * tq_pad * 4 + (size_t)tk_pad * 4;
  if (smem > 220 * 1024) return 1;
  const dim3 grid(a.B * a.H);
#define TCAVP_BWD_KB(DH, MAXT, MINB, KB_)                                                                                                   \
  do {                                                                                                                                      \
    TCAVP_CUDA(cudaFuncSetAttribute(fb::attn_bwd_tc_kernel<DH, MAXT, MINB, KB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
    fb::attn_bwd_tc_kernel<DH, MAXT, MINB, KB_><<<grid, warps * 32, smem, stream>>>(                                                        \
        a, reinterpret_cast<const __nv_bfloat16*>(dout), do_sb, do_st, reinterpret_cast<__nv_bfloat16*>(dq), dq_sb, dq_st, dk, dk_sb, dk_st, \
        dv, dv_sb, dv_st, dkv_dtype == TCAVP_BF16 ? 1 : 0, tq_pad, tk_pad);                                                                  \
  } while (0)
#define TCAVP_BWD(DH, MAXT, MINB)                      \
  do {                                                 \
    if (kb == 48) TCAVP_BWD_KB(DH, MAXT, MINB, 48);    \
    else TCAVP_BWD_KB(DH, MAXT, MINB, 64);             \
  } while (0)
  if (a.dh == 64) {
    if (warps <= 5) TCAVP_BWD(64, 160, 2);
    else TCAVP_BWD(64, 256, 1);
  } else if (a.dh == 128) {
    TCAVP_BWD(128, 256, 1);
  } else if (a.dh == 96) {
    TCAVP_BWD(96, 256, 1);
  } else if (a.dh == 32) {
    TCAVP_BWD(32, 256, 2);
  } else {
    TCAVP_BWD(16, 256, 2);
  }
#undef TCAVP_BWD
#undef TCAVP_BWD_KB
  return check_launch("attn_bwd_tc_kernel");
}

}  // namespace tcavp
