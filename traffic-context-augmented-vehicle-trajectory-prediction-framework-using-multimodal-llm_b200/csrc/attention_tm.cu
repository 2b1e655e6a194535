// tcgen05 flash attention for the LLM self-attention (HF:251-289 with the causal + key-padding mask of HF:399; GQA):
// bf16, causal, head_dim 64 / 128, L >= 128.  attn_tm_kernel below covers 128 <= L <= 256 (the fused sequence is 16 image + 128 text
// tokens = 144) with whole-row tiles; attn_tml_kernel (further down) covers L > 256 with 128-key blocks and an online softmax.
// Both optionally write the row logsumexp (tcavp_attn_args::lse) that the key-blocked backward rebuilds the probabilities from.
//
// Persistent, warp-specialised, one CTA per SM looping over (scene, head) items:
//   warp 0      TMA producer: Q, K, V tiles of the item ([L16 rows] x 64-column boxes, 128-byte swizzle) straight out of the packed
//               [rows, (nh + 2 nkv) dh] QKV activation into a 2-stage shared-memory ring (the next item lands under this item's math)
//   warp 1      one thread issues tcgen05.mma:  S = Q K^T (both operands K-major from shared memory, fp32 accumulators in TMEM) and
//               O = P V  (A = P read from TENSOR MEMORY, B = V as an MN-major shared-memory operand: no transposed copy of V)
//   warps 4-7   softmax of tile A, one thread per query row: tcgen05.ld the row's scores, mask, exp2, row sum, and write the bf16
//               probabilities back over the scores with tcgen05.st (P aliases S in TMEM); later drain O, scale by 1 / row sum, store
//   warps 8-11  the same for tile B
// L = 144 does not fit a 128-row UMMA tile, and padding to 256 would waste a whole second tile.  The causal structure gives a cheap
// split instead: tile A = the LAST 128 query rows [L16-128, L16) against all L16 keys, tile B = the first L16-128 rows (16 for L = 144),
// which can only see the first L16-128 keys — an M = 128, N = 16 MMA with 16 live rows.  TMEM: S_A (L16 cols) + S_B + O_A + O_B (dh each).
// Scores / probabilities never leave the SM; Q, K, V are read once and O written once (the HBM floor of the op).
#include <cuda.h>
#include <mutex>
#include "common.cuh"

namespace tcavp {
namespace tm {

constexpr int THREADS = 384;      // 12 warps: 0 TMA, 1 MMA (+ TMEM owner), 2-3 idle, 4-7 softmax of slot 0, 8-11 softmax of slot 1
constexpr int BOXC = 64;          // bf16 columns per TMA box = 128 bytes = one swizzle row

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
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
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// Shared-memory operand descriptors (cute::UMMA::SmemDescriptor, SWIZZLE_128B, version 1).
//   K-major  (Q, K):  rows of 128 bytes, 8-row groups 1024 bytes apart (SBO); the k-step advances the start address by 32 bytes.
//   MN-major (V as the B operand of P.V, N = head dim contiguous, K = keys): canonical ((8,8,m),(8,k)) : ((1,8,LBO),(64,SBO)) in
//            elements — 64 contiguous head-dim elements (128 bytes) per key row, 8-key groups 1024 bytes apart (SBO), the next 64
//            head-dim elements LBO bytes away (the second 64-column TMA box of a 128-wide head).
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// kind::f16 instruction descriptor: D fp32, A / B bf16, A K-major, B K-major or MN-major (bit 16).
__device__ __forceinline__ uint32_t idesc_f16(int M, int N, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {   // A from TMEM
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// tcgen05.ld is asynchronous: several loads are issued back to back and ONE tcgen05.wait::ld covers them (a wait per load would expose
// the TMEM round trip 18 times per score row).  `tmem_ld_fence` ties the destination registers to the wait so no use can move above it.
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_fence(uint32_t (&r)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) asm volatile("" : "+r"(r[i]));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void stg256(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]),
               "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

struct Geo {
  int B, H, Hkv, L, L16, NB;          // NB = L16 - 128: rows / keys of tile B (0: no tile B)
  int stages, slots;                  // shared-memory ring depth; items in flight per CTA (each slot owns a TMEM region + 4 softmax warps)
  uint32_t box_bytes, stage_bytes;    // one [L16 x 64] box; Q + K + V of one item
  uint32_t sb_col, o_col, slot_cols;  // per slot: S_A at +0, S_B at +sb_col, O (O_B, then O_A) at +o_col
  float sl2;                          // softmax scale * log2(e)
  const int32_t* key_mask;
  __nv_bfloat16* out; long long o_sb, o_st;
  float* lse; long long lse_sb;       // optional [B, H, L] logsumexp output
};

// Valid-key bits of the 16 score columns [16u, 16u + 16) for query row q: key-padding bits AND the causal bound j <= q.
__device__ __forceinline__ uint32_t unit_bits(const uint32_t* s_mask, int u, int q) {
  const uint32_t key16 = (s_mask[u >> 1] >> ((u & 1) * 16)) & 0xFFFFu;
  const int n_ok = q - u * 16 + 1;                       // leading columns the causal mask allows
  const uint32_t c16 = n_ok >= 16 ? 0xFFFFu : (n_ok <= 0 ? 0u : ((1u << n_ok) - 1u));
  return key16 & c16;
}

// Softmax of one score row per thread (TMEM lane = row): two sweeps over the row's scores (row max, then exp2 / row sum / P), each one
// 16-column unit (one x16 load, one wait) at a time: batches of two units in flight cost more in instruction-cache misses than they hid
// (211 us against 202 us on the 768-class shape).  The bf16 probabilities overwrite the score columns (P aliases S).  A
// 16-column unit whose keys are all attendable for every row of the warp (the common case left of the causal diagonal) takes a
// select-free path.  `q`: query index of the row, `ncols`: key columns of the tile, `warp_kmax`: largest key any row of the warp sees.
// Returns (row sum, base-2 reference max the probabilities were taken against).
// (__noinline__: tile A and tile B share one copy — ten warps in different places of a 60 KB kernel thrash the instruction caches)
__device__ __noinline__ float2 softmax_rows(const Geo& g, uint32_t srow, int q, int ncols, int warp_kmax, const uint32_t* s_mask) {
  const int nu = min(ncols, (warp_kmax + 16) & ~15) >> 4;
  const int nu_all = ncols >> 4;
  float m = -INFINITY;
  for (int u = 0; u < nu; ++u) {
    uint32_t r[16];
    tmem_ld16_issue(srow + u * 16, r);
    tmem_ld_wait();
    tmem_ld_fence(r);
    const uint32_t vb = unit_bits(s_mask, u, q);
    if (__all_sync(0xffffffffu, vb == 0xFFFFu)) {
#pragma unroll
      for (int c = 0; c < 16; ++c) m = fmaxf(m, __uint_as_float(r[c]));
    } else {
#pragma unroll
      for (int c = 0; c < 16; ++c) m = fmaxf(m, ((vb >> c) & 1u) ? __uint_as_float(r[c]) : -INFINITY);
    }
  }
  const float mref = m == -INFINITY ? 0.f : m * g.sl2;
  float l = 0.f;
  for (int u = 0; u < nu; ++u) {
    uint32_t r[16];
    tmem_ld16_issue(srow + u * 16, r);
    tmem_ld_wait();
    // the unit's score columns are in registers: its bf16 probabilities may now overwrite score columns (8u + 8 <= 16u + 16)
    tmem_ld_fence(r);
    uint32_t pk[8];
    const uint32_t vb = unit_bits(s_mask, u, q);
    if (__all_sync(0xffffffffu, vb == 0xFFFFu)) {
#pragma unroll
      for (int c = 0; c < 16; c += 2) {
        const float p0 = ex2(fmaf(__uint_as_float(r[c]), g.sl2, -mref)), p1 = ex2(fmaf(__uint_as_float(r[c + 1]), g.sl2, -mref));
        l += p0 + p1;
        pk[c >> 1] = pack2(p0, p1);
      }
    } else {
#pragma unroll
      for (int c = 0; c < 16; c += 2) {
        const float p0 = ((vb >> c) & 1u) ? ex2(fmaf(__uint_as_float(r[c]), g.sl2, -mref)) : 0.f;
        const float p1 = ((vb >> (c + 1)) & 1u) ? ex2(fmaf(__uint_as_float(r[c + 1]), g.sl2, -mref)) : 0.f;
        l += p0 + p1;
        pk[c >> 1] = pack2(p0, p1);
      }
    }
    tmem_st8(srow + u * 8, pk);
  }
  {
    const uint32_t z[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    for (int u = nu; u < nu_all; ++u) tmem_st8(srow + u * 8, z);    // keys beyond the causal bound of this warp's rows
  }
  tmem_st_wait();
  tc_fence_before();
  return make_float2(l, mref);
}

// lse[b, h, q] = ln(sum_j exp(scale * s_qj)) from the row sum l taken against the base-2 reference mref (-inf when l == 0)
__device__ __forceinline__ void store_lse(float* lse, long long lse_sb, int H, int L, int b, int h, int q, float l, float mref) {
  if (lse && q < L) lse[(size_t)b * lse_sb + (size_t)h * L + q] = (mref + log2f(l)) * 0.6931471805599453f;
}

// Drains one output row per thread: O / row sum -> bf16 -> global (128 or 256 contiguous bytes per row).
template <int DH>
__device__ __noinline__ void drain_rows(const Geo& g, uint32_t orow, float l, int q, int b, int h) {
  const float inv = l > 0.f ? 1.f / l : 0.f;
  __nv_bfloat16* op = g.out + (size_t)b * g.o_sb + (size_t)q * g.o_st + (size_t)h * DH;
  const bool live = q < g.L;
#pragma unroll
  for (int c0 = 0; c0 < DH; c0 += 64) {
    uint32_t r[4][16];
#pragma unroll
    for (int i = 0; i < 4; ++i) tmem_ld16_issue(orow + c0 + i * 16, r[i]);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      tmem_ld_fence(r[i]);
      uint32_t w[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) w[e] = pack2(__uint_as_float(r[i][2 * e]) * inv, __uint_as_float(r[i][2 * e + 1]) * inv);
      if (live) stg256(op + c0 + i * 16, w);
    }
  }
  tc_fence_before();
}

// Barrier block (8 bytes each) behind the stage ring:  per stage: qkv_full, qkv_empty, mask_ready;  per slot: s_full, pb_ready, pa_ready,
// ob_full, ob_drained, oa_full, o_free.
constexpr int MAX_STAGES = 4, MAX_SLOTS = 2;
constexpr uint32_t BAR_FULL = 0, BAR_EMPTY = 8 * MAX_STAGES, BAR_MASK = 16 * MAX_STAGES, BAR_SLOT = 24 * MAX_STAGES;
constexpr uint32_t SL_SFULL = 0, SL_PB = 8, SL_PA = 16, SL_OBFULL = 24, SL_OBDRAINED = 32, SL_OAFULL = 40, SL_OFREE = 48, SL_BYTES = 56;
constexpr uint32_t BAR_BYTES = BAR_SLOT + MAX_SLOTS * SL_BYTES + 8;     // + the TMEM base address slot

template <int DH>
__global__ void __launch_bounds__(THREADS, 1)
attn_tm_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k, const __grid_constant__ CUtensorMap tma_v, Geo g) {
  constexpr int NBOX = DH / BOXC;      // 64-column boxes per operand
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint32_t s_mask[MAX_STAGES][8];    // per stage: key-valid bits of the item's scene (written by the producer warp)
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = smem_base + g.stages * g.stage_bytes;
  const uint32_t tmem_slot = bars + BAR_SLOT + MAX_SLOTS * SL_BYTES;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nbw = (g.NB + 31) >> 5;                                   // warps of a slot with live tile-B rows
  const int n_items = g.B * g.H;
  const int my_items = blockIdx.x < n_items ? (n_items - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  // (scene, head) of this CTA's n-th item without a division per item: it = blockIdx.x + n * gridDim.x
  const int step_b = (int)gridDim.x / g.H, step_h = (int)gridDim.x % g.H;
  const int b0 = (int)blockIdx.x / g.H, h0 = (int)blockIdx.x % g.H;
  const int hrep = g.H / g.Hkv;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_q)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_k)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_v)) : "memory");
    for (int s = 0; s < MAX_STAGES; ++s) {
      mbar_init(bars + BAR_FULL + 8 * s, 1);
      mbar_init(bars + BAR_EMPTY + 8 * s, 1);
      mbar_init(bars + BAR_MASK + 8 * s, 1);
    }
    for (int k = 0; k < MAX_SLOTS; ++k) {
      const uint32_t sb = bars + BAR_SLOT + k * SL_BYTES;
      mbar_init(sb + SL_SFULL, 1);
      mbar_init(sb + SL_PB, nbw > 0 ? nbw : 1);
      mbar_init(sb + SL_PA, 4);
      mbar_init(sb + SL_OBFULL, 1);
      mbar_init(sb + SL_OBDRAINED, nbw > 0 ? nbw : 1);
      mbar_init(sb + SL_OAFULL, 1);
      mbar_init(sb + SL_OFREE, 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer (+ the scene's key-valid bits, off the softmax warps' critical path) =====================
    int b = b0, h = h0, s = 0;
    uint32_t use = 0;
    for (int n = 0; n < my_items; ++n) {
      // key-valid words of the scene: every load is issued before the first ballot (a ballot per load would serialise eight global
      // round trips per item and make this warp the bottleneck of the whole pipeline), and before the wait on the stage
      int kv[8];
#pragma unroll
      for (int w = 0; w < 8; ++w) {                                          // HF:399: padding keys are masked for every query
        const int j = w * 32 + lane;
        kv[w] = j < g.L ? (g.key_mask ? __ldg(g.key_mask + (size_t)b * g.L + j) : 1) : 0;
      }
      if (lane == 0) {
        mbar_wait(bars + BAR_EMPTY + 8 * s, (use & 1u) ^ 1u);                // also frees the stage's mask words (read before P is ready)
        const uint32_t full = bars + BAR_FULL + 8 * s;
        mbar_expect_tx(full, g.stage_bytes);
        const uint32_t st = smem_base + s * g.stage_bytes;
        const int hk = h / hrep;
#pragma unroll
        for (int c = 0; c < NBOX; ++c) {
          tma_load_2d(st + c * g.box_bytes, &tma_q, full, h * DH + c * BOXC, b * g.L);
          tma_load_2d(st + (NBOX + c) * g.box_bytes, &tma_k, full, hk * DH + c * BOXC, b * g.L);
          tma_load_2d(st + (2 * NBOX + c) * g.box_bytes, &tma_v, full, hk * DH + c * BOXC, b * g.L);
        }
      }
      __syncwarp();
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const uint32_t bits = __ballot_sync(0xffffffffu, kv[w] != 0);
        if (lane == 0) s_mask[s][w] = bits;
      }
      if (lane == 0) mbar_arrive(bars + BAR_MASK + 8 * s);
      __syncwarp();
      b += step_b; h += step_h;
      if (h >= g.H) { h -= g.H; ++b; }
      if (++s == g.stages) { s = 0; ++use; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // Software pipeline over this CTA's items with a skew of (slots - 1):  iteration n issues S(n) = Q K^T of item n, then the P.V
    // products of item n - (slots - 1), whose softmax ran while S(n) was being issued / computed.  tcgen05.mma executes in issue order,
    // so an accumulator region is never overwritten before the products that read it (issued earlier by this thread) have retired.
    if (lane == 0) {
      const uint32_t id_sa = idesc_f16(128, g.L16, 0), id_sb = idesc_f16(128, g.NB > 0 ? g.NB : 16, 0), id_pv = idesc_f16(128, DH, 1);
      const int qa0 = g.L16 - 128;      // first query row of tile A
      const int skew = g.slots - 1;
      for (int n = 0; n < my_items + skew; ++n) {
        if (n < my_items) {
          const int s = n % g.stages, k = n % g.slots;
          const uint32_t use = (uint32_t)(n / g.stages);
          const uint32_t sq = smem_base + s * g.stage_bytes, sk = sq + NBOX * g.box_bytes;
          const uint32_t tS = tmem_base + k * g.slot_cols, sbar = bars + BAR_SLOT + k * SL_BYTES;
          mbar_wait(bars + BAR_FULL + 8 * s, use & 1u);
          tc_fence_after();
#pragma unroll
          for (int kk = 0; kk < DH / 16; ++kk) {        // S_A = Q[qa0 .. qa0 + 128) . K^T over all L16 keys
            const uint32_t boff = (uint32_t)(kk >> 2) * g.box_bytes + (uint32_t)(kk & 3) * 32u;
            umma_ss(tS, desc_kmajor(sq + boff + (uint32_t)qa0 * 128u), desc_kmajor(sk + boff), id_sa, kk != 0);
          }
          if (g.NB > 0) {
#pragma unroll
            for (int kk = 0; kk < DH / 16; ++kk) {      // S_B = Q[0 .. 128) . K[0 .. NB)^T
              const uint32_t boff = (uint32_t)(kk >> 2) * g.box_bytes + (uint32_t)(kk & 3) * 32u;
              umma_ss(tS + g.sb_col, desc_kmajor(sq + boff), desc_kmajor(sk + boff), id_sb, kk != 0);
            }
          }
          umma_commit(sbar + SL_SFULL);
        }
        const int m = n - skew;
        if (m >= 0) {
          const int s = m % g.stages, k = m % g.slots;
          const uint32_t ph = (uint32_t)(m / g.slots) & 1u;
          const uint32_t sv = smem_base + s * g.stage_bytes + 2 * NBOX * g.box_bytes;
          const uint32_t tS = tmem_base + k * g.slot_cols, tO = tS + g.o_col, sbar = bars + BAR_SLOT + k * SL_BYTES;
          mbar_wait(sbar + SL_OFREE, ph ^ 1u);          // the slot's previous output has been drained
          if (g.NB > 0) {                               // O_B = P_B . V[0 .. NB)
            mbar_wait(sbar + SL_PB, ph);
            tc_fence_after();
            for (int kk = 0; kk < g.NB / 16; ++kk)
              umma_ts(tO, tS + g.sb_col + kk * 8, desc_mnmajor(sv + (uint32_t)kk * 2048u, g.box_bytes), id_pv, kk != 0);
            umma_commit(sbar + SL_OBFULL);
          }
          mbar_wait(sbar + SL_PA, ph);                  // O_A = P_A . V   (into the columns O_B was drained from)
          if (g.NB > 0) mbar_wait(sbar + SL_OBDRAINED, ph);
          tc_fence_after();
          for (int kk = 0; kk < g.L16 / 16; ++kk)
            umma_ts(tO, tS + kk * 8, desc_mnmajor(sv + (uint32_t)kk * 2048u, g.box_bytes), id_pv, kk != 0);
          umma_commit(sbar + SL_OAFULL);
          umma_commit(bars + BAR_EMPTY + 8 * s);        // every MMA that reads this stage has retired when this arrives
        }
      }
    }
  } else if (warp >= 4 && ((warp - 4) >> 2) < g.slots) {
    // ===================== softmax / output warps: slot k = (warp - 4) / 4, TMEM lane quarter wq = warp % 4 =====================
    const int k = (warp - 4) >> 2, wq = warp & 3;
    const uint32_t lane_base = tmem_base + ((uint32_t)(wq * 32) << 16) + k * g.slot_cols;
    const uint32_t sbar = bars + BAR_SLOT + k * SL_BYTES;
    const int qa0 = g.L16 - 128;
    const bool has_b = wq < nbw;
    // this slot's items: n = k, k + slots, ...
    int b = b0, h = h0;
    for (int i = 0; i < k; ++i) {
      b += step_b; h += step_h;
      if (h >= g.H) { h -= g.H; ++b; }
    }
    int j = 0;
    for (int n = k; n < my_items; n += g.slots, ++j) {
      const int st = n % g.stages;
      const uint32_t ph = (uint32_t)j & 1u;
      mbar_wait(bars + BAR_MASK + 8 * st, (uint32_t)(n / g.stages) & 1u);
      mbar_wait(sbar + SL_SFULL, ph);
      tc_fence_after();
      float l_b = 0.f;
      const int qb = wq * 32 + lane;                    // tile B row = query index
      if (has_b) {
        // rows >= NB of tile B are not part of the problem: their query index is pushed past L so nothing is stored for them
        const float2 r = softmax_rows(g, lane_base + g.sb_col, qb < g.NB ? qb : g.L + qb, g.NB, min(wq * 32 + 31, g.NB - 1), s_mask[st]);
        l_b = r.x;
        __syncwarp();
        if (lane == 0) mbar_arrive(sbar + SL_PB);
        store_lse(g.lse, g.lse_sb, g.H, g.L, b, h, qb < g.NB ? qb : g.L + qb, r.x, r.y);
      }
      const int qa = qa0 + wq * 32 + lane;
      const float2 ra = softmax_rows(g, lane_base, qa, g.L16, qa0 + wq * 32 + 31, s_mask[st]);
      const float l_a = ra.x;
      __syncwarp();
      if (lane == 0) mbar_arrive(sbar + SL_PA);
      store_lse(g.lse, g.lse_sb, g.H, g.L, b, h, qa, ra.x, ra.y);
      if (has_b) {
        mbar_wait(sbar + SL_OBFULL, ph);
        tc_fence_after();
        drain_rows<DH>(g, lane_base + g.o_col, l_b, qb < g.NB ? qb : g.L + qb, b, h);
        __syncwarp();
        if (lane == 0) mbar_arrive(sbar + SL_OBDRAINED);
      }
      mbar_wait(sbar + SL_OAFULL, ph);
      tc_fence_after();
      drain_rows<DH>(g, lane_base + g.o_col, l_a, qa, b, h);
      __syncwarp();
      if (lane == 0) mbar_arrive(sbar + SL_OFREE);
      for (int i = 0; i < g.slots; ++i) {
        b += step_b; h += step_h;
        if (h >= g.H) { h -= g.H; ++b; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}


// ------------------------------------------------------------------------------------------------
// Key-blocked form for L > 256 (attn_tml_kernel): one work item = (scene, head, 128-row query tile t), which iterates over the
// 128-key blocks 0 .. t (causal: block t is the diagonal one, the only block that needs the causal mask).  Same roles as above:
//   warp 0      TMA producer: the item's Q tile into a 2-deep Q ring, then K and V of every key block into a stage ring, plus the
//               block's four key-valid words (ballots over key_mask, so the mask costs no shared memory that grows with L)
//   warp 1      one thread issues S(g) = Q K_g^T into one of two S buffers, ONE BLOCK AHEAD of O += P(g-1) V(g-1) (A = P from TMEM,
//               B = V MN-major), so the softmax of block g overlaps the score product of block g + 1
//   warps 4-7   online softmax, one thread per query row: running reference max and row sum in registers, P written over S
// TMEM: S0 [0, 128), S1 [128, 256), O [256, 256 + dh).  O accumulates across the key blocks of an item.
//
// Rescaling O: a row's probabilities are taken against a reference max that is only raised when the block max exceeds it by more
// than RESCALE_LOG2 (2^8 in probability): every probability stays <= 256, exact enough in bf16 and far from fp32 overflow, and
// the final normalisation divides by the row sum taken against the same stale reference, so the result does not depend on when the
// reference moved.  When it does move, the row's thread tcgen05.ld's its O row, scales it and tcgen05.st's it back after the
// previous P.V has retired and before it releases P of this block.  Random and trained scores raise it in the first block or two
// only, so almost every block skips the O round trip.
// Items are ordered longest first (query tile NT-1 of every (scene, head) before tile NT-2, ...) and dealt round-robin to the
// persistent CTAs, so the uneven causal work of the tiles evens out across the grid.
constexpr int L_THREADS = 256;           // 8 warps: 0 TMA, 1 MMA (+ TMEM owner), 2-3 idle, 4-7 softmax
constexpr int L_MAX_STAGES = 4;
constexpr float RESCALE_LOG2 = 8.f;

struct GeoL {
  int B, H, Hkv, L, NT;                  // NT = 128-row query tiles per (scene, head)
  int stages;
  uint32_t q_bytes, stage_bytes;         // one Q tile; K + V of one key block
  float sl2;
  const int32_t* key_mask;
  __nv_bfloat16* out; long long o_sb, o_st;
  float* lse; long long lse_sb;
};

// barriers (8 bytes each): q_full[2], q_empty[2], kv_full[S], kv_empty[S], mask[S], s_full[2], p_ready, pv_done, o_free, TMEM slot
constexpr uint32_t LB_QFULL = 0, LB_QEMPTY = 16, LB_KVFULL = 32, LB_KVEMPTY = LB_KVFULL + 8 * L_MAX_STAGES,
                   LB_MASK = LB_KVEMPTY + 8 * L_MAX_STAGES, LB_SFULL = LB_MASK + 8 * L_MAX_STAGES, LB_PREADY = LB_SFULL + 16,
                   LB_PVDONE = LB_PREADY + 8, LB_OFREE = LB_PVDONE + 8, LB_TMEM = LB_OFREE + 8, LB_BYTES = LB_TMEM + 8;

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
      "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// item -> (scene, head, query tile), longest tiles first
__device__ __forceinline__ void item_coords(const GeoL& g, int it, int& b, int& h, int& t) {
  const int bh = g.B * g.H;
  t = g.NT - 1 - it / bh;
  const int r = it % bh;
  b = r / g.H;
  h = r % g.H;
}

template <int DH>
__global__ void __launch_bounds__(L_THREADS, 1)
attn_tml_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k, const __grid_constant__ CUtensorMap tma_v, GeoL g) {
  constexpr int NBOX = DH / BOXC;
  constexpr uint32_t BOX = 128u * 128u;                        // one [128 rows x 64 columns] bf16 box
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint32_t s_mask[L_MAX_STAGES][4];                 // per stage: key-valid bits of the block's 128 keys
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sq0 = smem_base, skv0 = smem_base + 2u * g.q_bytes;
  const uint32_t bars = skv0 + (uint32_t)g.stages * g.stage_bytes;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (bars + LB_TMEM - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_items = g.B * g.H * g.NT;
  const int my_items = blockIdx.x < n_items ? (n_items - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int hrep = g.H / g.Hkv;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_q)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_k)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_v)) : "memory");
    for (int i = 0; i < 2; ++i) {
      mbar_init(bars + LB_QFULL + 8 * i, 1);
      mbar_init(bars + LB_QEMPTY + 8 * i, 1);
      mbar_init(bars + LB_SFULL + 8 * i, 1);
    }
    for (int s = 0; s < L_MAX_STAGES; ++s) {
      mbar_init(bars + LB_KVFULL + 8 * s, 1);
      mbar_init(bars + LB_KVEMPTY + 8 * s, 1);
      mbar_init(bars + LB_MASK + 8 * s, 1);
    }
    mbar_init(bars + LB_PREADY, 4);
    mbar_init(bars + LB_PVDONE, 1);
    mbar_init(bars + LB_OFREE, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bars + LB_TMEM), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    uint32_t gblk = 0;                                            // running key-block counter of this CTA
    for (int n = 0; n < my_items; ++n) {
      int b, h, t;
      item_coords(g, (int)blockIdx.x + n * (int)gridDim.x, b, h, t);
      const int hk = h / hrep;
      if (lane == 0) {
        const uint32_t qf = bars + LB_QFULL + 8 * (n & 1);
        mbar_wait(bars + LB_QEMPTY + 8 * (n & 1), (((uint32_t)n >> 1) & 1u) ^ 1u);
        mbar_expect_tx(qf, g.q_bytes);
#pragma unroll
        for (int c = 0; c < NBOX; ++c) tma_load_2d(sq0 + (n & 1) * g.q_bytes + c * BOX, &tma_q, qf, h * DH + c * BOXC, b * g.L + t * 128);
      }
      for (int j = 0; j <= t; ++j, ++gblk) {
        const int s = (int)(gblk % (uint32_t)g.stages);
        const uint32_t use = gblk / (uint32_t)g.stages;
        int kv[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) {                             // HF:399: padding keys are masked for every query
          const int key = j * 128 + w * 32 + lane;
          kv[w] = key < g.L ? (g.key_mask ? __ldg(g.key_mask + (size_t)b * g.L + key) : 1) : 0;
        }
        if (lane == 0) {
          mbar_wait(bars + LB_KVEMPTY + 8 * s, (use & 1u) ^ 1u);   // also frees the stage's mask words (read before P is ready)
          const uint32_t full = bars + LB_KVFULL + 8 * s;
          mbar_expect_tx(full, g.stage_bytes);
          const uint32_t st = skv0 + (uint32_t)s * g.stage_bytes;
#pragma unroll
          for (int c = 0; c < NBOX; ++c) {
            tma_load_2d(st + c * BOX, &tma_k, full, hk * DH + c * BOXC, b * g.L + j * 128);
            tma_load_2d(st + (NBOX + c) * BOX, &tma_v, full, hk * DH + c * BOXC, b * g.L + j * 128);
          }
        }
        __syncwarp();
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const uint32_t bits = __ballot_sync(0xffffffffu, kv[w] != 0);
          if (lane == 0) s_mask[s][w] = bits;
        }
        if (lane == 0) mbar_arrive(bars + LB_MASK + 8 * s);
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: S one key block ahead of P.V =====================
    if (lane == 0) {
      const uint32_t id_s = idesc_f16(128, 128, 0), id_pv = idesc_f16(128, DH, 1);
      const uint32_t tO = tmem_base + 256;
      // S cursor: (item sn, block sj, global block sg); the P.V cursor trails it by one block
      int sn = 0, sj = 0, st_ = 0;
      uint32_t sg = 0;
      auto issue_s = [&]() {
        if (sn >= my_items) return;
        int b, h, t;
        item_coords(g, (int)blockIdx.x + sn * (int)gridDim.x, b, h, t);
        (void)b; (void)h;
        st_ = t;
        if (sj == 0) mbar_wait(bars + LB_QFULL + 8 * (sn & 1), ((uint32_t)sn >> 1) & 1u);
        const int s = (int)(sg % (uint32_t)g.stages);
        mbar_wait(bars + LB_KVFULL + 8 * s, (sg / (uint32_t)g.stages) & 1u);
        tc_fence_after();
        const uint32_t sq = sq0 + (sn & 1) * g.q_bytes, sk = skv0 + (uint32_t)s * g.stage_bytes;
        const uint32_t tS = tmem_base + (sg & 1u) * 128u;
#pragma unroll
        for (int kk = 0; kk < DH / 16; ++kk) {
          const uint32_t boff = (uint32_t)(kk >> 2) * BOX + (uint32_t)(kk & 3) * 32u;
          umma_ss(tS, desc_kmajor(sq + boff), desc_kmajor(sk + boff), id_s, kk != 0);
        }
        umma_commit(bars + LB_SFULL + 8 * (sg & 1u));
        if (sj == st_) {                                          // last score product of the item: its Q buffer may be refilled
          umma_commit(bars + LB_QEMPTY + 8 * (sn & 1));
          ++sn; sj = 0;
        } else {
          ++sj;
        }
        ++sg;
      };
      issue_s();
      uint32_t pg = 0;
      for (int n = 0; n < my_items; ++n) {
        int b, h, t;
        item_coords(g, (int)blockIdx.x + n * (int)gridDim.x, b, h, t);
        for (int j = 0; j <= t; ++j, ++pg) {
          issue_s();                                              // S(pg + 1) overwrites P(pg - 1): its P.V was issued earlier
          if (j == 0) mbar_wait(bars + LB_OFREE, ((uint32_t)n & 1u) ^ 1u);   // the previous item's O has been drained
          mbar_wait(bars + LB_PREADY, pg & 1u);
          tc_fence_after();
          const int s = (int)(pg % (uint32_t)g.stages);
          const uint32_t sv = skv0 + (uint32_t)s * g.stage_bytes + NBOX * BOX;
          const uint32_t tP = tmem_base + (pg & 1u) * 128u;
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
            umma_ts(tO, tP + kk * 8, desc_mnmajor(sv + (uint32_t)kk * 2048u, BOX), id_pv, (j > 0 || kk != 0) ? 1u : 0u);
          umma_commit(bars + LB_PVDONE);
          umma_commit(bars + LB_KVEMPTY + 8 * s);                 // every MMA that reads this stage has retired when this arrives
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== softmax / output warps: TMEM lane quarter wq, one query row per thread =====================
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    const uint32_t lane_off = (uint32_t)(wq * 32) << 16;
    const uint32_t orow = tmem_base + lane_off + 256;
    uint32_t gblk = 0;
    for (int n = 0; n < my_items; ++n) {
      int b, h, t;
      item_coords(g, (int)blockIdx.x + n * (int)gridDim.x, b, h, t);
      const int q = t * 128 + row;
      float ref = -INFINITY, l = 0.f;                             // base-2 reference max, row sum against it
      for (int j = 0; j <= t; ++j, ++gblk) {
        const int st = (int)(gblk % (uint32_t)g.stages);
        mbar_wait(bars + LB_MASK + 8 * st, (gblk / (uint32_t)g.stages) & 1u);
        mbar_wait(bars + LB_SFULL + 8 * (gblk & 1u), (gblk >> 1) & 1u);
        tc_fence_after();
        const uint32_t srow = tmem_base + lane_off + (gblk & 1u) * 128u;
        const bool diag = j == t;
        // units past the causal bound of every row of this warp are not read (their P is stored as zeros)
        const int nu = diag ? min(8, (wq * 32 + 31) / 16 + 1) : 8;
        auto bits = [&](int u) {
          const uint32_t key16 = (s_mask[st][u >> 1] >> ((u & 1) * 16)) & 0xFFFFu;
          if (!diag) return key16;
          const int n_ok = row - u * 16 + 1;
          return key16 & (n_ok >= 16 ? 0xFFFFu : (n_ok <= 0 ? 0u : ((1u << n_ok) - 1u)));
        };
        float m = -INFINITY;
        for (int u = 0; u < nu; ++u) {
          uint32_t r[16];
          tmem_ld16_issue(srow + u * 16, r);
          tmem_ld_wait();
          tmem_ld_fence(r);
          const uint32_t vb = bits(u);
#pragma unroll
          for (int c = 0; c < 16; ++c) m = fmaxf(m, ((vb >> c) & 1u) ? __uint_as_float(r[c]) : -INFINITY);
        }
        const float mb = m == -INFINITY ? -INFINITY : m * g.sl2;
        // raise the reference only when the block max clears it by RESCALE_LOG2; a row with no visible key so far has O = 0, l = 0
        const bool raise = ref == -INFINITY ? mb != -INFINITY : mb > ref + RESCALE_LOG2;
        const float corr = (raise && ref != -INFINITY) ? ex2(ref - mb) : 1.f;
        if (raise) ref = mb;
        l *= corr;
        const float mref = ref == -INFINITY ? 0.f : ref;
        for (int u = 0; u < nu; ++u) {
          uint32_t r[16];
          tmem_ld16_issue(srow + u * 16, r);
          tmem_ld_wait();
          tmem_ld_fence(r);                                       // the unit's scores are in registers: P may overwrite them
          const uint32_t vb = bits(u);
          uint32_t pk[8];
#pragma unroll
          for (int c = 0; c < 16; c += 2) {
            const float p0 = ((vb >> c) & 1u) ? ex2(fmaf(__uint_as_float(r[c]), g.sl2, -mref)) : 0.f;
            const float p1 = ((vb >> (c + 1)) & 1u) ? ex2(fmaf(__uint_as_float(r[c + 1]), g.sl2, -mref)) : 0.f;
            l += p0 + p1;
            pk[c >> 1] = pack2(p0, p1);
          }
          tmem_st8(srow + u * 8, pk);
        }
        {
          const uint32_t z[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          for (int u = nu; u < 8; ++u) tmem_st8(srow + u * 8, z);
        }
        if (j > 0) {
          mbar_wait(bars + LB_PVDONE, (gblk - 1) & 1u);           // O holds every earlier block of the item
          tc_fence_after();
          if (__any_sync(0xffffffffu, corr != 1.f)) {
#pragma unroll
            for (int c0 = 0; c0 < DH; c0 += 64) {
              uint32_t r[4][16];
#pragma unroll
              for (int i = 0; i < 4; ++i) tmem_ld16_issue(orow + c0 + i * 16, r[i]);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                tmem_ld_fence(r[i]);
#pragma unroll
                for (int e = 0; e < 16; ++e) r[i][e] = __float_as_uint(__uint_as_float(r[i][e]) * corr);
                tmem_st16(orow + c0 + i * 16, r[i]);
              }
            }
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars + LB_PREADY);
      }
      // ---- drain: O / l -> bf16 -> global, lse ----
      mbar_wait(bars + LB_PVDONE, (gblk - 1) & 1u);
      tc_fence_after();
      const float inv = l > 0.f ? 1.f / l : 0.f;
      __nv_bfloat16* op = g.out + (size_t)b * g.o_sb + (size_t)q * g.o_st + (size_t)h * DH;
      const bool live = q < g.L;
#pragma unroll
      for (int c0 = 0; c0 < DH; c0 += 64) {
        uint32_t r[4][16];
#pragma unroll
        for (int i = 0; i < 4; ++i) tmem_ld16_issue(orow + c0 + i * 16, r[i]);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          tmem_ld_fence(r[i]);
          uint32_t w[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) w[e] = pack2(__uint_as_float(r[i][2 * e]) * inv, __uint_as_float(r[i][2 * e + 1]) * inv);
          if (live) stg256(op + c0 + i * 16, w);
        }
      }
      store_lse(g.lse, g.lse_sb, g.H, g.L, b, h, q, l, ref == -INFINITY ? 0.f : ref);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + LB_OFREE);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}
// [rows, cols] bf16 view with row stride ld; box = box_rows x 64 columns, 128-byte swizzle, zero fill out of bounds.
static int make_map(CUtensorMap* map, const void* base, long long rows, int cols, long long ld, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return 1;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BOXC, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS
             ? 0
             : 1;
}

}  // namespace tm

// Key-blocked launch (L > 256).  Same operand conditions as the tile form; returns 1 when the shape is not covered.
static int attention_tml_launch(const tcavp_attn_args& a, cudaStream_t stream) {
  using namespace tm;
  const int L = a.Tq;
  GeoL g;
  g.B = a.B; g.H = a.H; g.Hkv = a.Hkv; g.L = L; g.NT = (L + 127) / 128;
  g.q_bytes = (uint32_t)(a.dh / BOXC) * 128u * 128u;
  g.stage_bytes = 2u * g.q_bytes;
  int stages = (int)((225u * 1024u - 2u * g.q_bytes - LB_BYTES - 1024u) / g.stage_bytes);
  if (stages < 2) return 1;
  g.stages = stages > L_MAX_STAGES ? L_MAX_STAGES : stages;
  g.sl2 = a.scale * 1.4426950408889634f;
  g.key_mask = a.key_mask;
  g.out = reinterpret_cast<__nv_bfloat16*>(a.out); g.o_sb = a.o_sb; g.o_st = a.o_st;
  g.lse = a.lse; g.lse_sb = a.lse_sb;
  if ((long long)a.B * a.H * g.NT > 0x7fffffffLL || (long long)a.B * L > 0x7fffffffLL) return 1;
  CUtensorMap mq, mk, mv;
  const long long rows = (long long)a.B * L;
  if (make_map(&mq, a.q, rows, a.H * a.dh, a.q_st, 128) || make_map(&mk, a.k, rows, a.Hkv * a.dh, a.k_st, 128) ||
      make_map(&mv, a.v, rows, a.Hkv * a.dh, a.v_st, 128))
    return 1;
  const size_t smem = (size_t)2 * g.q_bytes + (size_t)g.stages * g.stage_bytes + LB_BYTES + 1024;   // > 118 KB: one CTA per SM
  const int items = a.B * a.H * g.NT;
  const int grid = items < sm_count() ? items : sm_count();
  if (a.dh == 64) {
    TCAVP_CUDA(cudaFuncSetAttribute(attn_tml_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_tml_kernel<64><<<grid, L_THREADS, smem, stream>>>(mq, mk, mv, g);
  } else {
    TCAVP_CUDA(cudaFuncSetAttribute(attn_tml_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_tml_kernel<128><<<grid, L_THREADS, smem, stream>>>(mq, mk, mv, g);
  }
  return check_launch("attn_tml_kernel");
}

// Returns 1 when the shape is not covered (caller falls back to the mma.sync flash kernel), <= 0 otherwise.
int attention_tm_launch(const tcavp_attn_args& a, cudaStream_t stream) {
  using namespace tm;
  static int enabled = -1;
  if (enabled < 0) {
    const char* e = getenv("TCAVP_ATTN_TCGEN05");      // 0: keep the mma.sync kernel (A/B runs)
    enabled = e ? atoi(e) : 1;
  }
  if (!enabled) return 1;
  if (a.dtype != TCAVP_BF16 || !a.causal || a.Tq != a.Tk || a.drop_thresh != 0) return 1;
  if (!(a.dh == 64 || a.dh == 128) || a.Tq < 128 || a.B < 1) return 1;
  const int L = a.Tq, L16 = (L + 15) / 16 * 16, NB = L16 - 128;
  // rows of consecutive scenes must be contiguous (one 2-D tensor map per operand) and TMA-addressable
  if (a.q_sb != (long long)L * a.q_st || a.k_sb != (long long)L * a.k_st || a.v_sb != (long long)L * a.v_st) return 1;
  auto al16 = [](const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; };
  if (!al16(a.q) || !al16(a.k) || !al16(a.v) || reinterpret_cast<uintptr_t>(a.out) % 32 || a.q_st % 8 || a.k_st % 8 || a.v_st % 8 || a.o_st % 16 ||
      a.o_sb % 16)
    return 1;
  if (L > 256) return attention_tml_launch(a, stream);
  Geo g;
  g.B = a.B; g.H = a.H; g.Hkv = a.Hkv; g.L = L; g.L16 = L16; g.NB = NB;
  g.box_bytes = (uint32_t)L16 * 128u;
  g.stage_bytes = 3u * (uint32_t)(a.dh / BOXC) * g.box_bytes;
  // TMEM per item in flight: S_A (L16 columns), S_B (NB columns) right behind it, one output region (O_B, then O_A)
  g.sb_col = (uint32_t)L16;
  g.o_col = (uint32_t)((L16 + NB + 31) / 32 * 32);
  g.slot_cols = g.o_col + (uint32_t)a.dh;
  if (g.slot_cols > 512u) return 1;
  const int fit = (int)((225u * 1024u - 2048u) / g.stage_bytes);     // stages that fit in shared memory
  if (fit < 1) return 1;
  g.slots = (2u * g.slot_cols <= 512u && fit >= 2) ? MAX_SLOTS : 1;
  g.stages = fit >= 2 * g.slots ? 2 * g.slots : (fit >= g.slots ? (fit / g.slots) * g.slots : 1);
  if (g.stages > MAX_STAGES) g.stages = MAX_STAGES;
  if (g.stages < g.slots) g.slots = 1;
  g.sl2 = a.scale * 1.4426950408889634f;
  g.key_mask = a.key_mask;
  g.out = reinterpret_cast<__nv_bfloat16*>(a.out); g.o_sb = a.o_sb; g.o_st = a.o_st;
  g.lse = a.lse; g.lse_sb = a.lse_sb;
  CUtensorMap mq, mk, mv;
  const long long rows = (long long)a.B * L;
  if (make_map(&mq, a.q, rows, a.H * a.dh, a.q_st, L16) || make_map(&mk, a.k, rows, a.Hkv * a.dh, a.k_st, L16) ||
      make_map(&mv, a.v, rows, a.Hkv * a.dh, a.v_st, L16))
    return 1;
  // at least 118 KB so that a second CTA can never become co-resident on an SM (each CTA allocates all 512 TMEM columns)
  size_t smem = (size_t)g.stages * g.stage_bytes + BAR_BYTES + 1024;
  if (smem < 118 * 1024) smem = 118 * 1024;
  const int items = a.B * a.H;
  const int grid = items < sm_count() ? items : sm_count();
  if (a.dh == 64) {
    TCAVP_CUDA(cudaFuncSetAttribute(attn_tm_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_tm_kernel<64><<<grid, THREADS, smem, stream>>>(mq, mk, mv, g);
  } else {
    TCAVP_CUDA(cudaFuncSetAttribute(attn_tm_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attn_tm_kernel<128><<<grid, THREADS, smem, stream>>>(mq, mk, mv, g);
  }
  return check_launch("attn_tm_kernel");
}

}  // namespace tcavp
