// tcavp_gemm: out = act(A . W^T + bias) + residual, with row remap and the fused epilogues of include/tcavp.h
// (RMSNorm row factor / statistics, RoPE, SwiGLU forward + stash, SwiGLU backward).
//
//   bf16 : persistent, warp-specialised tcgen05 kernels.  Warp 0: one elected thread issues TMA loads (cp.async.bulk.tensor,
//          128-byte swizzle) into a multi-stage shared-memory ring; warp 1: one elected thread issues tcgen05.mma (bf16 -> fp32)
//          into TMEM; 16 epilogue warps drain TMEM with tcgen05.ld, apply the fused epilogue and store 32 bytes per lane.
//          Variants, picked by tcavp_gemm from the problem shape:
//            gemm_tc_kernel<BN>       one CTA per 128 x BN tile (BN 32..256), double-buffered accumulators
//            gemm_tc_pair_kernel<256> CTA pair (cta_group::2) on a 256 x 256 tile, double-buffered accumulators (the default for
//                                     large problems: the epilogue of tile i overlaps the MMAs of tile i+1)
//            gemm_tc_wide_kernel      CTA pair on a 512 x 256 tile, all 512 TMEM columns, for long contractions (K >= 2048)
//   e4m3 : the gemm_tc_kernel and gemm_tc_pair_kernel pipelines with tcgen05.mma.kind::f8f6f4 and per-column dequantisation.
//   fp32 : SIMT FFMA kernel with exact fp32 accumulation (the rtol 1e-4 parity mode; no TF32).
//
// LoRA (peft lora.Linear, reference scripts/train.py:432-440) is expressed by the caller as extra K columns
// ([x | x.A^T] . [W | (alpha/r) B]^T), i.e. it accumulates in the same TMEM tile as the base product.
#include <cuda.h>
#include <stdlib.h>
#include <mutex>
#include "common.cuh"

namespace tcavp {
namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;   // 64 bf16 = 128 bytes = one SWIZZLE_128B atom row
constexpr int UMMA_K = 16;
constexpr int NUM_EPI_WARPS = 16;  // four warps per TMEM lane quarter, each draining every fourth 32-column chunk
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;  // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2..: epilogue
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;
// Operand geometry per element type.  e4m3 (kind::f8f6f4) keeps the byte geometry of bf16: a k-block is one 128-byte swizzle row
// (128 elements) and one MMA covers 32 bytes of K (32 elements), so stage sizes, descriptor advances and TMEM budgets are shared.
template <bool F8>
struct Op {
  static constexpr int KB = F8 ? 128 : BLOCK_K;   // elements per k-block
  static constexpr int UK = F8 ? 32 : UMMA_K;     // elements per MMA
  static constexpr int ESZ = F8 ? 1 : 2;          // bytes per element
};

template <int BLOCK_N>
struct Cfg {
  static constexpr int B_STAGE_BYTES = BLOCK_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int STAGES = (BLOCK_N >= 256) ? 4 : (BLOCK_N >= 128 ? 6 : 8);
  static constexpr int TMEM_COLS = (2 * BLOCK_N < 32) ? 32 : 2 * BLOCK_N;  // two accumulator buffers
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256 /*barriers*/ + 1024 /*alignment slack*/;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// K-major operand tile in shared memory, SWIZZLE_128B: rows are 128 bytes, 8-row groups are 1024 bytes apart.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);   // start address, 16-byte units
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset between 8-row groups
  d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f8f6f4 instruction descriptor: D fp32, A/B E4M3 (format code 0 in bits 7-9 / 10-12), both K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_e4m3(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_e4m3(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// silu(g) * u with one EX2 and one RCP: g * u / (1 + 2^(-g log2 e)); saturates correctly at +-inf.
__device__ __forceinline__ float swiglu_f(float g, float u) {
  return __fdividef(g * u, 1.f + ex2_approx(-1.4426950408889634f * g));
}

// 256-bit global accesses (sm_100): one full 32-byte sector per lane per instruction.
__device__ __forceinline__ void stg256(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]),
               "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
// ... streaming form for outputs far larger than L2 (panelled 7B-class GEMMs): the written lines are the first to leave L2, so they do not
// push out the W panel the next wave of tiles needs.
__device__ __forceinline__ void stg256_stream(void* p, const uint32_t (&v)[8]) {
  asm volatile("st.global.L1::no_allocate.L2::evict_first.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void ldg256(const void* p, uint32_t (&v)[8]) {
  asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(p));
}

// Tile order of the persistent kernels.  Units are swept n-fastest inside PANELS of `pw` n-tiles: the W rows of a panel stay resident in
// L2 while every row block of A streams past them once, so W is read from DRAM once and A once per panel.  With pw >= tiles_n (any
// problem whose whole W fits in L2, e.g. the 768-class shapes) this is the plain row-major order.  Without panels a 7B-class gate/up
// GEMM (W = 180 MB > L2) re-read W for every 512-row block: 12.7 GB of DRAM reads per launch against 0.5 GB algorithmic.
__host__ __device__ __forceinline__ void unit_to_tile(int u, int tiles_mg, int tiles_n, int pw, int& mg, int& nt) {
  if (pw >= tiles_n) {
    mg = u / tiles_n;
    nt = u % tiles_n;
    return;
  }
  const int per_panel = tiles_mg * pw;
  const int full = tiles_n / pw;
  int p = u / per_panel, r, w;
  if (p < full) {
    r = u - p * per_panel;
    w = pw;
  } else {
    p = full;
    r = u - full * per_panel;
    w = tiles_n - full * pw;
  }
  mg = r / w;
  nt = p * pw + r % w;
}
constexpr int PANEL_SHIFT = 16;   // flags >> PANEL_SHIFT = panel width in n-tiles (0: no panels)

enum { EPI_VEC_OUT = 1, EPI_VEC_RES = 2, EPI_VEC_BIAS = 4, EPI_TMA_OUT = 8,    // EPI_TMA_OUT: bf16 output staged in shared memory, stored by TMA
       L2_W_LAST = 256, L2_OUT_FIRST = 1024 };      // L2 eviction priorities of a panelled problem (see panel_flags)

// e4m3 operands: accumulator column n carries the dequantisation factor col_scale[n] of its weight row.  Applied to the raw accumulators
// (before the row factor, RoPE and SwiGLU, which mix or pair columns with different scales); columns past Nacc get 0.
__device__ __forceinline__ void scale_cols(uint32_t (&r)[32], const float* __restrict__ cs, int nacc0, int nacc) {
  if (nacc0 + 32 <= nacc) {
    const float4* p = reinterpret_cast<const float4*>(cs + nacc0);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 s = __ldg(p + q);
      r[4 * q] = __float_as_uint(__uint_as_float(r[4 * q]) * s.x);
      r[4 * q + 1] = __float_as_uint(__uint_as_float(r[4 * q + 1]) * s.y);
      r[4 * q + 2] = __float_as_uint(__uint_as_float(r[4 * q + 2]) * s.z);
      r[4 * q + 3] = __float_as_uint(__uint_as_float(r[4 * q + 3]) * s.w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * (nacc0 + j < nacc ? __ldg(cs + nacc0 + j) : 0.f));
  }
}

// Epilogue of 32 accumulator columns [nacc0, nacc0+32) of row m for one thread.  The interior-tile path (full chunk,
// 16-byte aligned rows) is branch-light and fully vectorised; ragged edges take the scalar path.
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// `stage_row` / `half` / `lane` (EPI_TMA_OUT only): shared-memory address of this lane's row in the warp's staging tile, which half of
// the warp's 64 accumulator columns this call covers, and the lane (= row of the 32-row tile, for the swizzle).
__device__ __forceinline__ void epilogue_chunk(const EpilogueParams& p, int m, int pos, int nacc0, const uint32_t (&r)[32], float rs, int flags,
                                               float& ssq, uint32_t stage_row = 0, int half = 0, int lane = 0) {
  if (m >= p.M) return;
  const int mo = remap_row(p.remap_gi, p.remap_go, p.remap_off, m);
  if (p.act == TCAVP_ACT_SWIGLU_BWD) {
    // accumulators = d(mid) for 32 hidden units; (gate, up) pairs come from the forward stash, (d gate, d up) pairs go out
    if (nacc0 >= p.N) return;
    const __nv_bfloat16* gp = p.aux + (size_t)mo * p.ld_aux + 2 * nacc0;
    __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)mo * p.ldo + 2 * nacc0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {          // 8 hidden units = 16 bf16 = 32 bytes per step
      uint32_t gu[8], du[8];
      ldg256(gp + q * 16, gu);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float g = __uint_as_float(gu[e] << 16), u = __uint_as_float(gu[e] & 0xffff0000u);
        const float d = __uint_as_float(r[q * 8 + e]) * rs;
        const float sg = __fdividef(1.f, 1.f + ex2_approx(-1.4426950408889634f * g));
        du[e] = pack_bf16(d * u * sg * (1.f + g * (1.f - sg)), d * g * sg);
      }
      stg256(op + q * 16, du);
    }
    return;
  }
  float o[32];
  int cnt, n0;
  if (p.act == TCAVP_ACT_SWIGLU) {
    cnt = 16;
    n0 = nacc0 >> 1;
    if (p.aux && nacc0 + 32 <= 2 * p.N) {     // stash (gate, up) pairs for the backward pass: 32 bf16 = two 32-byte stores
      __nv_bfloat16* ap = p.aux + (size_t)remap_row(p.remap_gi, p.remap_go, p.remap_off, m) * p.ld_aux + nacc0;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        uint32_t u[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) u[e] = pack_bf16(__uint_as_float(r[q * 16 + 2 * e]) * rs, __uint_as_float(r[q * 16 + 2 * e + 1]) * rs);
        stg256(ap + q * 16, u);
      }
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) o[j] = swiglu_f(__uint_as_float(r[2 * j]) * rs, __uint_as_float(r[2 * j + 1]) * rs);
  } else {
    cnt = 32;
    n0 = nacc0;
#pragma unroll
    for (int j = 0; j < 32; ++j) o[j] = __uint_as_float(r[j]) * rs;
  }
  if (n0 >= p.N) return;
  const bool full = (n0 + cnt <= p.N);
  if (p.rope_cols > 0 && n0 < p.rope_cols) {
    // chunk = 32 columns = 16 rotation pairs of one head (rope_dh is a multiple of 32).  The table is laid out
    // [dh/4][L] x float4 (cos, sin of two adjacent pairs): consecutive rows (= consecutive positions = consecutive lanes)
    // read consecutive 16-byte entries, so each load is 4 wavefronts instead of 32.
    const float4* cs = reinterpret_cast<const float4*>(p.rope) + (size_t)((n0 % p.rope_dh) >> 2) * p.rope_L + pos;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 t = __ldg(cs + (size_t)j * p.rope_L);   // (cos, sin) of two adjacent pairs
      const float a0 = o[4 * j], a1 = o[4 * j + 1], a2 = o[4 * j + 2], a3 = o[4 * j + 3];
      o[4 * j] = a0 * t.x - a1 * t.y;
      o[4 * j + 1] = a1 * t.x + a0 * t.y;
      o[4 * j + 2] = a2 * t.z - a3 * t.w;
      o[4 * j + 3] = a3 * t.z + a2 * t.w;
    }
  }
  if (p.bias) {
    if (full && (flags & EPI_VEC_BIAS)) {
      const float4* bp = reinterpret_cast<const float4*>(p.bias + n0);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (q * 4 < cnt) {
          const float4 b = __ldg(bp + q);
          o[q * 4] += b.x; o[q * 4 + 1] += b.y; o[q * 4 + 2] += b.z; o[q * 4 + 3] += b.w;
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < cnt && n0 + j < p.N) o[j] += __ldg(p.bias + n0 + j);
    }
  }
  if (p.act == TCAVP_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) o[j] = fmaxf(o[j], 0.f);
  } else if (p.act == TCAVP_ACT_GELU_TANH) {
    // bf16 outputs: the hardware tanh (MUFU.TANH, relative error ~2^-11) is below the output rounding; the fp32 SIMT path keeps tanhf
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float x = o[j];
      float t;
      asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.7978845608028654f * fmaf(0.044715f * x * x, x, x)));
      o[j] = 0.5f * x * (1.f + t);
    }
  }
  if (p.residual) {
    if ((flags & EPI_VEC_RES) && full) {
      if (p.res_dtype == TCAVP_BF16) {
        const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(p.residual) + (size_t)mo * p.ldr + n0;
        uint32_t u[2][8];
#pragma unroll
        for (int q = 0; q < 2; ++q)
          if (q * 16 < cnt) ldg256(rp + q * 16, u[q]);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if (q * 16 < cnt) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {     // bf16 -> fp32 is a 16-bit shift
              o[q * 16 + 2 * e] += __uint_as_float(u[q][e] << 16);
              o[q * 16 + 2 * e + 1] += __uint_as_float(u[q][e] & 0xffff0000u);
            }
          }
        }
      } else {
        const float4* rp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.residual) + (size_t)mo * p.ldr + n0);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (q * 4 < cnt) {
            float4 f = rp[q];
            o[q * 4] += f.x; o[q * 4 + 1] += f.y; o[q * 4 + 2] += f.z; o[q * 4 + 3] += f.w;
          }
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < cnt && n0 + j < p.N) o[j] += load_as_f(p.residual, (size_t)mo * p.ldr + n0 + j, p.res_dtype);
    }
  }
  if (p.sumsq_out) {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < cnt && (full || n0 + j < p.N)) ssq = fmaf(o[j], o[j], ssq);
  }
  if (flags & EPI_TMA_OUT) {
    // bf16 rows of the warp's 32 x 64 (SwiGLU: 32 x 32) output tile in the swizzled layout the TMA store expects: 16-byte chunk j of
    // row r sits at chunk j ^ (r & 7) of a 128-byte row (SWIZZLE_128B) / j ^ ((r >> 1) & 3) of a 64-byte row (SWIZZLE_64B).
    // Columns past N are written too (their accumulators come from zero-filled weight rows) and clipped by the store.
    if (cnt == 32) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = half * 4 + q;
        sts128(stage_row + (uint32_t)((j ^ (lane & 7)) << 4), pack_bf16(o[q * 8], o[q * 8 + 1]), pack_bf16(o[q * 8 + 2], o[q * 8 + 3]),
               pack_bf16(o[q * 8 + 4], o[q * 8 + 5]), pack_bf16(o[q * 8 + 6], o[q * 8 + 7]));
      }
    } else {
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int j = half * 2 + q;
        sts128(stage_row + (uint32_t)((j ^ ((lane >> 1) & 3)) << 4), pack_bf16(o[q * 8], o[q * 8 + 1]), pack_bf16(o[q * 8 + 2], o[q * 8 + 3]),
               pack_bf16(o[q * 8 + 4], o[q * 8 + 5]), pack_bf16(o[q * 8 + 6], o[q * 8 + 7]));
      }
    }
    return;
  }
  if ((flags & EPI_VEC_OUT) && full) {
    if (p.out_dtype == TCAVP_BF16) {
      __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)mo * p.ldo + n0;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (q * 16 < cnt) {
          uint32_t u[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) u[e] = pack_bf16(o[q * 16 + 2 * e], o[q * 16 + 2 * e + 1]);
          if (flags & L2_OUT_FIRST) stg256_stream(op + q * 16, u);
          else stg256(op + q * 16, u);
        }
      }
    } else {
      float* op = reinterpret_cast<float*>(p.out) + (size_t)mo * p.ldo + n0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (q * 8 < cnt) {
          uint32_t u[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) u[e] = __float_as_uint(o[q * 8 + e]);
          stg256(op + q * 8, u);
        }
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < cnt && n0 + j < p.N) store_from_f(p.out, (size_t)mo * p.ldo + n0 + j, p.out_dtype, o[j]);
  }
}

template <int BLOCK_N, bool F8 = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, EpilogueParams ep,
               int M, int Nacc, int K, int flags) {
  using C = Cfg<BLOCK_N>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_base + C::STAGES * A_STAGE_BYTES;
  const uint32_t bars = smem_base + C::STAGES * C::STAGE_BYTES;
  const uint32_t full_bar = bars;                         // STAGES x 8 bytes
  const uint32_t empty_bar = bars + 8 * C::STAGES;        // STAGES x 8 bytes
  const uint32_t tmem_full_bar = bars + 16 * C::STAGES;   // 2 x 8
  const uint32_t tmem_empty_bar = tmem_full_bar + 16;     // 2 x 8
  const uint32_t tmem_slot = tmem_empty_bar + 16;         // 4 bytes: TMEM base address
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_n = (Nacc + BLOCK_N - 1) / BLOCK_N;
  const int tiles_m = (M + BLOCK_M - 1) / BLOCK_M;
  const int num_units = tiles_m * tiles_n;
  const int unit0 = blockIdx.x, unit_stride = gridDim.x;
  using O = Op<F8>;
  const int num_kb = (K + O::KB - 1) / O::KB;
  const int pw = (flags >> PANEL_SHIFT) > 0 ? (flags >> PANEL_SHIFT) : tiles_n;   // n-tiles per L2-resident panel of W

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_b)) : "memory");
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar + 8 * s, 1);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tmem_full_bar + 8 * s, 1);
      mbar_init(tmem_empty_bar + 8 * s, NUM_EPI_WARPS);   // one arrive per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = unit0; unit < num_units; unit += unit_stride) {
        int mg, nt;
        unit_to_tile(unit, tiles_m, tiles_n, pw, mg, nt);
        const int m0 = mg * BLOCK_M;
        const int n0 = nt * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar + 8 * stage, phase ^ 1);
          mbar_expect_tx(full_bar + 8 * stage, C::STAGE_BYTES);
          tma_load_2d(smem_a + stage * A_STAGE_BYTES, &tma_a, full_bar + 8 * stage, kb * O::KB, m0);
          tma_load_2d(smem_b + stage * C::B_STAGE_BYTES, &tma_b, full_bar + 8 * stage, kb * O::KB, n0);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = F8 ? umma_idesc_e4m3(BLOCK_M, BLOCK_N) : umma_idesc(BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int unit = unit0; unit < num_units; unit += unit_stride, ++it) {
        const int acc = it & 1;
        mbar_wait(tmem_empty_bar + 8 * acc, ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar + 8 * stage, phase);
          tc_fence_after();
          const int k_left = K - kb * O::KB;
          const int ksteps = k_left >= O::KB ? O::KB / O::UK : (k_left + O::UK - 1) / O::UK;
          const uint32_t a_addr = smem_a + stage * A_STAGE_BYTES;
          const uint32_t b_addr = smem_b + stage * C::B_STAGE_BYTES;
          for (int k = 0; k < ksteps; ++k) {
            const uint64_t ad = umma_smem_desc(a_addr + k * O::UK * O::ESZ), bd = umma_smem_desc(b_addr + k * O::UK * O::ESZ);
            if constexpr (F8) umma_e4m3(tmem_d, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
            else umma_bf16(tmem_d, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar + 8 * stage);   // frees the smem slot once the MMAs above retire
          if (kb == num_kb - 1) umma_commit(tmem_full_bar + 8 * acc);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..) =====================
    const int quarter = warp & 3;           // TMEM lanes [32*quarter, +32) are the ones this warp may read
    const int chunk0 = (warp - 2) >> 2;     // the two warps of a quarter take alternate 32-column chunks
    int it = 0;
    for (int unit = unit0; unit < num_units; unit += unit_stride, ++it) {
      const int acc = it & 1;
      int mg, nt;
      unit_to_tile(unit, tiles_m, tiles_n, pw, mg, nt);
      const int m0 = mg * BLOCK_M;
      const int n0 = nt * BLOCK_N;
      mbar_wait(tmem_full_bar + 8 * acc, (it >> 1) & 1);
      tc_fence_after();
      const int m = m0 + quarter * 32 + lane;
      float rs = 1.f;
      if (m < M) {
        if (ep.row_scale) rs = __ldg(ep.row_scale + m);
        else if (ep.row_sumsq) rs = sumsq_rstd(ep.row_sumsq + m, ep.ss_inv, ep.ss_eps);
      }
      float ssq = 0.f;
      const int pos = ep.rope_cols > 0 ? m % ep.rope_L : 0;
#pragma unroll 1
      for (int c = chunk0; c < BLOCK_N / 32; c += NUM_EPI_WARPS / 4) {
        if (n0 + c * 32 >= Nacc) break;   // warp-uniform
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BLOCK_N + c * 32, r);
        if constexpr (F8) scale_cols(r, ep.col_scale, n0 + c * 32, Nacc);
        epilogue_chunk(ep, m, pos, n0 + c * 32, r, rs, flags, ssq);
      }
      if (ep.sumsq_out && m < M) sumsq_add(ep.sumsq_out + remap_row(ep.remap_gi, ep.remap_go, ep.remap_off, m), ssq);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty_bar + 8 * acc);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2): the two CTAs of a cluster (one TPC) compute ONE 256 x BLOCK_N tile.  Each CTA
// stages its own 128 rows of A and its own BLOCK_N/2 rows of W; the leader CTA's single thread issues
// tcgen05.mma.cta_group::2 (UMMA 256 x BLOCK_N x 16), which reads both shared memories and writes rows [0,128) of the
// tile into the leader's TMEM and rows [128,256) into the peer's.  Per k-block an SM ingests 16 KB (A) + BLOCK_N*64 B
// (half of W) instead of A + the whole W tile, which is what bounds the K <= 1024 GEMMs, and the ring gets 6 stages.
// Synchronisation: every TMA load (both CTAs) completes on the LEADER's full barrier; the MMA thread's commits are
// multicast to both CTAs' empty / tmem_full barriers; epilogue warps of both CTAs arrive on the leader's tmem_empty.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
// ... with an L2 eviction-priority policy: the W panel of a problem larger than L2 is loaded evict_last so that the A rows and the
// output lines streaming through L2 do not push it out between waves of tiles (without it a 58 MB panel was re-read every wave).
__device__ __forceinline__ void tma_load_2d_pair_hint(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy(bool evict_last) {   // evict_last, or evict_normal
  uint64_t p;
  if (evict_last) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_e4m3_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {   // arrives on the same barrier offset in both CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

template <int BLOCK_N, bool TMA_OUT = false>
struct PairCfg {
  static constexpr int HALF_N = BLOCK_N / 2;
  static constexpr int B_STAGE_BYTES = HALF_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int OUT_BYTES = TMA_OUT ? NUM_EPI_WARPS * 4096 : 0;     // one 32 x 64 bf16 staging tile per epilogue warp
  static constexpr int STAGES = BLOCK_N >= 256 ? (TMA_OUT ? 5 : 6) : 8;
  static constexpr int TMEM_COLS = 2 * BLOCK_N;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + OUT_BYTES + 256 + 1024;
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src),
               "r"(c0), "r"(c1)
               : "memory");
}

// TMA_OUT: the epilogue warps do not store to global memory themselves.  Each warp owns 32 rows x 64 adjacent accumulator columns of
// the tile, writes its bf16 results into a private 4 KB swizzled staging tile and lets one lane issue a cp.async.bulk.tensor store
// (the copy engine writes full 128-byte lines and clips the tensor edges); the staging tile is reused once the previous store has
// read it (cp.async.bulk.wait_group.read).  One operand stage is given up for the staging tiles.
template <int BLOCK_N, bool TMA_OUT = false, bool F8 = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ CUtensorMap tma_o,
                    EpilogueParams ep, int M, int Nacc, int K, int flags) {
  using C = PairCfg<BLOCK_N, TMA_OUT>;
  constexpr int PAIR_M = 2 * BLOCK_M;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_base + C::STAGES * A_STAGE_BYTES;
  const uint32_t smem_out = smem_base + C::STAGES * C::STAGE_BYTES;          // TMA_OUT: NUM_EPI_WARPS x 4 KB staging tiles (1024-byte aligned)
  const uint32_t bars = smem_out + C::OUT_BYTES;
  const uint32_t full_bar = bars;                         // leader's copy is the live one
  const uint32_t empty_bar = bars + 8 * C::STAGES;        // per CTA, signalled by the multicast commit
  const uint32_t tmem_full_bar = bars + 16 * C::STAGES;   // per CTA, signalled by the multicast commit
  const uint32_t tmem_empty_bar = tmem_full_bar + 16;     // leader's copy is the live one
  const uint32_t tmem_slot = tmem_empty_bar + 16;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_n = (Nacc + BLOCK_N - 1) / BLOCK_N;
  const int tiles_m = (M + PAIR_M - 1) / PAIR_M;
  const int num_units = tiles_m * tiles_n;
  const int unit0 = blockIdx.x >> 1, unit_stride = gridDim.x >> 1;
  using O = Op<F8>;
  const int num_kb = (K + O::KB - 1) / O::KB;
  const int pw = (flags >> PANEL_SHIFT) > 0 ? (flags >> PANEL_SHIFT) : tiles_n;   // n-tiles per L2-resident panel of W

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_b)) : "memory");
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar + 8 * s, 1);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tmem_full_bar + 8 * s, 1);
      mbar_init(tmem_empty_bar + 8 * s, 2 * NUM_EPI_WARPS);   // epilogue warps of both CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // the same warp of both CTAs allocates the pair's TMEM columns
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      const uint32_t leader_full = mapa_shared(full_bar, 0);
      const bool hinted = (flags & L2_W_LAST) != 0;
      const uint64_t pol_w = l2_policy(hinted), pol_a = l2_policy(false);
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = unit0; unit < num_units; unit += unit_stride) {
        int mg, nt;
        unit_to_tile(unit, tiles_m, tiles_n, pw, mg, nt);
        const int m0 = mg * PAIR_M + (int)cta_rank * BLOCK_M;
        const int n0 = nt * BLOCK_N + (int)cta_rank * C::HALF_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar + 8 * stage, phase ^ 1);
          if (leader) mbar_expect_tx(full_bar + 8 * stage, 2 * C::STAGE_BYTES);
          if (hinted) {
            tma_load_2d_pair_hint(smem_a + stage * A_STAGE_BYTES, &tma_a, leader_full + 8 * stage, kb * O::KB, m0, pol_a);
            tma_load_2d_pair_hint(smem_b + stage * C::B_STAGE_BYTES, &tma_b, leader_full + 8 * stage, kb * O::KB, n0, pol_w);
          } else {
            tma_load_2d_pair(smem_a + stage * A_STAGE_BYTES, &tma_a, leader_full + 8 * stage, kb * O::KB, m0);
            tma_load_2d_pair(smem_b + stage * C::B_STAGE_BYTES, &tma_b, leader_full + 8 * stage, kb * O::KB, n0);
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = F8 ? umma_idesc_e4m3(PAIR_M, BLOCK_N) : umma_idesc(PAIR_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int unit = unit0; unit < num_units; unit += unit_stride, ++it) {
        const int acc = it & 1;
        mbar_wait(tmem_empty_bar + 8 * acc, ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(full_bar + 8 * stage, phase);
          tc_fence_after();
          const int k_left = K - kb * O::KB;
          const int ksteps = k_left >= O::KB ? O::KB / O::UK : (k_left + O::UK - 1) / O::UK;
          const uint32_t a_addr = smem_a + stage * A_STAGE_BYTES;
          const uint32_t b_addr = smem_b + stage * C::B_STAGE_BYTES;
          for (int k = 0; k < ksteps; ++k) {
            const uint64_t ad = umma_smem_desc(a_addr + k * O::UK * O::ESZ), bd = umma_smem_desc(b_addr + k * O::UK * O::ESZ);
            if constexpr (F8) umma_e4m3_pair(tmem_d, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
            else umma_bf16_pair(tmem_d, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit_pair(empty_bar + 8 * stage);
          if (kb == num_kb - 1) umma_commit_pair(tmem_full_bar + 8 * acc);
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2.., both CTAs: each drains its own 128 rows) =====================
    const int quarter = warp & 3;
    const int chunk0 = (warp - 2) >> 2;
    const uint32_t leader_tmem_empty = mapa_shared(tmem_empty_bar, 0);
    const uint32_t my_stage = smem_out + (uint32_t)(warp - 2) * 4096u;
    const bool swiglu = ep.act == TCAVP_ACT_SWIGLU;
    const uint32_t stage_row = my_stage + (uint32_t)lane * (swiglu ? 64u : 128u);
    int it = 0;
    for (int unit = unit0; unit < num_units; unit += unit_stride, ++it) {
      const int acc = it & 1;
      int mg, nt;
      unit_to_tile(unit, tiles_m, tiles_n, pw, mg, nt);
      const int m0 = mg * PAIR_M + (int)cta_rank * BLOCK_M;
      const int n0 = nt * BLOCK_N;
      mbar_wait(tmem_full_bar + 8 * acc, (it >> 1) & 1);
      tc_fence_after();
      const int m = m0 + quarter * 32 + lane;
      float rs = 1.f;
      if (m < M) {
        if (ep.row_scale) rs = __ldg(ep.row_scale + m);
        else if (ep.row_sumsq) rs = sumsq_rstd(ep.row_sumsq + m, ep.ss_inv, ep.ss_eps);
      }
      float ssq = 0.f;
      const int pos = ep.rope_cols > 0 ? m % ep.rope_L : 0;
      if (TMA_OUT) {
        // this warp: accumulator columns [n0 + 64 chunk0, + 64) of rows [m0 + 32 quarter, + 32)
        const int c_first = 2 * chunk0;
        if (n0 + c_first * 32 < Nacc) {                       // warp-uniform
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous store has read the staging tile
          __syncwarp();
#pragma unroll 1
          for (int hh = 0; hh < 2; ++hh) {
            const int c = c_first + hh;
            if (n0 + c * 32 >= Nacc) break;
            uint32_t r[32];
            tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BLOCK_N + c * 32, r);
            if constexpr (F8) scale_cols(r, ep.col_scale, n0 + c * 32, Nacc);
            epilogue_chunk(ep, m, pos, n0 + c * 32, r, rs, flags, ssq, stage_row, hh, lane);
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            const int col_acc = n0 + c_first * 32;
            tma_store_2d(&tma_o, my_stage, swiglu ? col_acc >> 1 : col_acc, m0 + quarter * 32);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      } else {
#pragma unroll 1
        for (int c = chunk0; c < BLOCK_N / 32; c += NUM_EPI_WARPS / 4) {
          if (n0 + c * 32 >= Nacc) break;   // warp-uniform
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BLOCK_N + c * 32, r);
          if constexpr (F8) scale_cols(r, ep.col_scale, n0 + c * 32, Nacc);
          epilogue_chunk(ep, m, pos, n0 + c * 32, r, rs, flags, ssq);
        }
      }
      if (ep.sumsq_out && m < M) sumsq_add(ep.sumsq_out + remap_row(ep.remap_gi, ep.remap_go, ep.remap_off, m), ssq);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(leader_tmem_empty + 8 * acc);
    }
    if (TMA_OUT && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // stores complete before the CTA retires
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Wide variant for long contractions (K >= 2048: down_proj, every 7B-class projection): a CTA pair computes a 512 x 256 tile,
// each CTA accumulating 256 x 256 fp32 = ALL 512 TMEM columns (rows [0,128) in columns [0,256), rows [128,256) in [256,512)).
// Per k-block an SM stages 32 KB of A + 16 KB of W for 8.4 MFLOP (175 FLOP per staged byte against 128 for the pair kernel,
// and one W fetch from shared memory feeds two 128-row MMAs), which is what the power-capped mainloop pays for.  The price is
// a single accumulator buffer: the epilogue of a tile is not hidden behind the next tile's MMAs (only behind its TMA prefetch),
// ~4-8k cycles against >= 32 x 1024 cycles of MMAs per tile at K >= 2048.
// ------------------------------------------------------------------------------------------------
struct WideCfg {
  static constexpr int BLOCK_N = 256, HALF_N = 128;
  static constexpr int A_BYTES = 2 * A_STAGE_BYTES;                 // 256 rows x 64 x bf16
  static constexpr int B_BYTES = HALF_N * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;             // 48 KB
  static constexpr int STAGES = 4;
  static constexpr int TMEM_COLS = 512;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256 + 1024;
};

__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_wide_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, EpilogueParams ep,
                    int M, int Nacc, int K, int flags, int split_g) {
  using C = WideCfg;
  constexpr int CTA_M = 2 * BLOCK_M, PAIR_M = 4 * BLOCK_M;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_base + C::STAGES * C::A_BYTES;
  const uint32_t bars = smem_base + C::STAGES * C::STAGE_BYTES;
  const uint32_t full_bar = bars;
  const uint32_t empty_bar = bars + 8 * C::STAGES;
  const uint32_t tmem_full_bar = bars + 16 * C::STAGES;   // 2 x 8: one per 128-row half
  const uint32_t tmem_empty_bar = tmem_full_bar + 16;     // 2 x 8: one per 128-row half
  const uint32_t tmem_slot = tmem_empty_bar + 16;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_n = (Nacc + C::BLOCK_N - 1) / C::BLOCK_N;
  const int tiles_m = (M + PAIR_M - 1) / PAIR_M;
  const int num_units = tiles_m * tiles_n;
  const int unit0 = blockIdx.x >> 1, unit_stride = gridDim.x >> 1;
  const int num_kb = (K + BLOCK_K - 1) / BLOCK_K;
  const int pw = (flags >> PANEL_SHIFT) > 0 ? (flags >> PANEL_SHIFT) : tiles_n;   // n-tiles per L2-resident panel of W

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_a)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_b)) : "memory");
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar + 8 * s, 1);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int h = 0; h < 2; ++h) {
      mbar_init(tmem_full_bar + 8 * h, 1);
      mbar_init(tmem_empty_bar + 8 * h, 2 * NUM_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      const uint32_t leader_full = mapa_shared(full_bar, 0);
      const bool hinted = (flags & L2_W_LAST) != 0;
      const uint64_t pol_w = l2_policy(hinted), pol_a = l2_policy(false);
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = unit0; unit < num_units; unit += unit_stride) {
        int mg, nt;
        unit_to_tile(unit, tiles_m, tiles_n, pw, mg, nt);
        const int m0 = mg * PAIR_M + (int)cta_rank * CTA_M;
        const int n0 = nt * C::BLOCK_N + (int)cta_rank * C::HALF_N;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(empty_bar + 8 * stage, phase ^ 1);
          if (leader) mbar_expect_tx(full_bar + 8 * stage, 2 * C::STAGE_BYTES);
          if (hinted) {
            tma_load_2d_pair_hint(smem_a + stage * C::A_BYTES, &tma_a, leader_full + 8 * stage, kb * BLOCK_K, m0, pol_a);
            tma_load_2d_pair_hint(smem_b + stage * C::B_BYTES, &tma_b, leader_full + 8 * stage, kb * BLOCK_K, n0, pol_w);
          } else {
            tma_load_2d_pair(smem_a + stage * C::A_BYTES, &tma_a, leader_full + 8 * stage, kb * BLOCK_K, m0);              // 256 rows
            tma_load_2d_pair(smem_b + stage * C::B_BYTES, &tma_b, leader_full + 8 * stage, kb * BLOCK_K, n0);              // 128 rows
          }
          if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = umma_idesc(2 * BLOCK_M, C::BLOCK_N);
      // Order of the (k-block, row half) MMAs of a tile.  The first `g` and the last `g` k-blocks are issued HALF-MAJOR (half 0 of all g
      // k-blocks, then half 1): at the end of a tile half 0's accumulator is complete - and its drain starts - g k-blocks of half-1 MMAs
      // before the tile ends, and at the start of the next tile half 0 is re-armed first while half 1 is still draining.  Each half's
      // drain overlaps g x 512 cycles of tensor work on the other half instead of stalling the pipe (single accumulator buffer: all 512
      // TMEM columns hold this tile).  The k-blocks in between are issued k-major, which frees a stage after every k-block.
      int g = split_g < C::STAGES ? split_g : C::STAGES;
      if (2 * g > num_kb) g = num_kb / 2;
      if (g < 1) g = 1;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int unit = unit0; unit < num_units; unit += unit_stride, ++it) {
        int kb0 = 0;
        while (kb0 < num_kb) {
          const int gn = (kb0 == 0 || kb0 + g >= num_kb) ? (kb0 + g <= num_kb ? g : num_kb - kb0) : 1;
          const bool last = kb0 + gn == num_kb;
#pragma unroll 1
          for (int h = 0; h < 2; ++h) {
            int st = stage;
            uint32_t ph = phase;
            for (int j = 0; j < gn; ++j) {
              const int kb = kb0 + j;
              if (h == 0) {
                mbar_wait(full_bar + 8 * st, ph);
                tc_fence_after();
              }
              if (kb == 0) {     // this half's accumulator columns must have been drained by the previous tile's epilogue
                mbar_wait(tmem_empty_bar + 8 * h, (it & 1) ^ 1);
                tc_fence_after();
              }
              const int k_left = K - kb * BLOCK_K;
              const int ksteps = k_left >= BLOCK_K ? BLOCK_K / UMMA_K : (k_left + UMMA_K - 1) / UMMA_K;
              const uint32_t a_addr = smem_a + st * C::A_BYTES + h * A_STAGE_BYTES;
              const uint32_t b_addr = smem_b + st * C::B_BYTES;
              for (int k = 0; k < ksteps; ++k) {
                umma_bf16_pair(tmem_base + h * C::BLOCK_N, umma_smem_desc(a_addr + k * UMMA_K * 2), umma_smem_desc(b_addr + k * UMMA_K * 2), idesc,
                               (kb | k) != 0 ? 1u : 0u);
              }
              if (h == 1) umma_commit_pair(empty_bar + 8 * st);
              if (++st == C::STAGES) { st = 0; ph ^= 1; }
            }
            if (last) umma_commit_pair(tmem_full_bar + 8 * h);
            if (h == 1) { stage = st; phase = ph; }
          }
          kb0 += gn;
        }
      }
    }
  } else {
    // ===================== epilogue: every CTA drains its own 256 rows, half by half =====================
    const int quarter = warp & 3;
    const int chunk0 = (warp - 2) >> 2;
    const uint32_t leader_tmem_empty = mapa_shared(tmem_empty_bar, 0);
    int it = 0;
    for (int unit = unit0; unit < num_units; unit += unit_stride, ++it) {
      int mg, nt;
      unit_to_tile(unit, tiles_m, tiles_n, pw, mg, nt);
      const int m_cta = mg * PAIR_M + (int)cta_rank * CTA_M;
      const int n0 = nt * C::BLOCK_N;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        mbar_wait(tmem_full_bar + 8 * h, it & 1);
        tc_fence_after();
        const int m = m_cta + h * BLOCK_M + quarter * 32 + lane;
        float rs = 1.f;
        if (m < M) {
          if (ep.row_scale) rs = __ldg(ep.row_scale + m);
          else if (ep.row_sumsq) rs = sumsq_rstd(ep.row_sumsq + m, ep.ss_inv, ep.ss_eps);
        }
        float ssq = 0.f;
        const int pos = ep.rope_cols > 0 ? m % ep.rope_L : 0;
#pragma unroll 1
        for (int c = chunk0; c < C::BLOCK_N / 32; c += NUM_EPI_WARPS / 4) {
          if (n0 + c * 32 >= Nacc) break;   // warp-uniform
          uint32_t rr[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + h * C::BLOCK_N + c * 32, rr);
          epilogue_chunk(ep, m, pos, n0 + c * 32, rr, rs, flags, ssq);
        }
        if (ep.sumsq_out && m < M) sumsq_add(ep.sumsq_out + remap_row(ep.remap_gi, ep.remap_go, ep.remap_off, m), ssq);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(leader_tmem_empty + 8 * h);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host side: TMA descriptors through the driver entry point (no link-time dependency on libcuda)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// rows x cols bf16 (f8: e4m3) matrix with leading dimension ld; box = box_rows x one 128-byte row (64 bf16 / 128 e4m3), 128-byte swizzle.
static int make_map(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_rows, bool f8 = false) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
    return TCAVP_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * (f8 ? 1 : 2)};
  cuuint32_t box[2] = {(cuuint32_t)(f8 ? Op<true>::KB : BLOCK_K), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, f8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
    return TCAVP_ERR_CUDA;
  }
  return TCAVP_OK;
}

// Vector-path switches of the epilogue: 256-bit output / residual accesses need 32-byte aligned rows, the bias loads 16-byte alignment.
static int epilogue_flags(const EpilogueParams& ep) {
  const size_t osz = ep.out_dtype == TCAVP_BF16 ? 2 : 4, rsz = ep.res_dtype == TCAVP_BF16 ? 2 : 4;
  int flags = 0;
  if (((size_t)ep.ldo * osz) % 32 == 0 && (reinterpret_cast<uintptr_t>(ep.out) % 32) == 0) flags |= EPI_VEC_OUT;
  if (ep.residual && ((size_t)ep.ldr * rsz) % 32 == 0 && (reinterpret_cast<uintptr_t>(ep.residual) % 32) == 0) flags |= EPI_VEC_RES;
  if (ep.bias && (reinterpret_cast<uintptr_t>(ep.bias) % 16) == 0) flags |= EPI_VEC_BIAS;
  return flags;
}

// Panel width (n-tiles) of the persistent tile order + L2 hints, packed into the kernel's flags (see unit_to_tile).
// A panel of W is sized to stay in L2 (40 of the 126 MB; loaded evict_last) while A streams past it.
// Modelled DRAM reads: W + A x panels with panels, A + (W rows one wave of resident units touches) x waves without (ncu: without
// evict_last even a 33 MB W is re-streamed by most waves) - the smaller one decides.  The hints (pair and wide kernels): W evict_last,
// and streaming (evict_first) stores for outputs larger than 256 MB.
static int panel_flags(long long M, long long N, long long K, int unit_m, int tile_n, int resident_units, bool can_hint) {
  constexpr long long budget = 40ll << 20;
  static const int force = [] {      // test hook: this many n-tiles per panel whatever the problem size
    const char* e = getenv("TCAVP_GEMM_PANEL_FORCE");
    return e ? atoi(e) : 0;
  }();
  if (force > 0 && force <= 0x7fff) return (force << PANEL_SHIFT) | (can_hint ? L2_W_LAST : 0);
  const long long w_bytes = N * K * 2, a_bytes = M * K * 2;
  // streaming stores only for outputs the next kernel cannot find in L2 anyway (> 2 x L2 of bf16)
  const int out_first = M * N * 2 > (256ll << 20) ? L2_OUT_FIRST : 0;
  const int hint_flags = can_hint ? (L2_W_LAST | out_first) : 0;
  if (w_bytes <= budget) return w_bytes * 4 > budget ? hint_flags : 0;     // whole W is one resident panel (tiny W: nothing to protect)
  const long long tiles_n = (N + tile_n - 1) / tile_n, tiles_m = (M + unit_m - 1) / unit_m;
  long long pw = budget / ((long long)tile_n * K * 2);
  if (pw < 1) pw = 1;
  const long long panels = (tiles_n + pw - 1) / pw;
  pw = (tiles_n + panels - 1) / panels;          // equal-width panels
  const long long waves = (tiles_m * tiles_n + resident_units - 1) / resident_units;
  const long long rows_per_wave = resident_units >= tiles_n ? tiles_n : resident_units;   // n-tiles of W one wave touches
  const long long plain = a_bytes + waves * rows_per_wave * tile_n * K * 2;
  const long long panelled = w_bytes + a_bytes * panels;
  if (panelled >= plain || pw >= tiles_n || pw > 0x7fff) return 0;
  return ((int)pw << PANEL_SHIFT) | hint_flags;
}

// tcavp_last_kernel() name of a single-CTA form: the template shape, and the operand type for e4m3
template <int BLOCK_N, bool F8> constexpr const char* tc_name() {
  if (F8) return BLOCK_N == 32 ? "gemm_tc_kernel<32,e4m3>" : BLOCK_N == 64 ? "gemm_tc_kernel<64,e4m3>" : BLOCK_N == 128 ? "gemm_tc_kernel<128,e4m3>"
                                                                                                                     : "gemm_tc_kernel<256,e4m3>";
  return BLOCK_N == 32 ? "gemm_tc_kernel<32>" : BLOCK_N == 64 ? "gemm_tc_kernel<64>" : BLOCK_N == 128 ? "gemm_tc_kernel<128>" : "gemm_tc_kernel<256>";
}

template <int BLOCK_N, bool F8 = false>
static int launch_tc(const tcavp_gemm_args& a, const EpilogueParams& ep, cudaStream_t stream) {
  using C = Cfg<BLOCK_N>;
  CUtensorMap ma, mb;
  int rc = make_map(&ma, a.A, a.M, a.K, a.lda, BLOCK_M, F8);
  if (rc) return rc;
  rc = make_map(&mb, a.W, a.N, a.K, a.ldw, BLOCK_N, F8);
  if (rc) return rc;
  TCAVP_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BLOCK_N, F8>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  const int tiles_m = (a.M + BLOCK_M - 1) / BLOCK_M, tiles_n = (a.N + BLOCK_N - 1) / BLOCK_N;
  const int units = tiles_m * tiles_n;
  const int max_ctas = sm_count();
  const int grid = units < max_ctas ? units : max_ctas;
  int flags = epilogue_flags(ep);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  flags |= panel_flags(a.M, a.N, a.K, BLOCK_M, BLOCK_N, max_ctas, false);
  TCAVP_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BLOCK_N, F8>, ma, mb, ep, a.M, a.N, a.K, flags));
  return check_launch(tc_name<BLOCK_N, F8>());
}

// [rows, cols] bf16 output view for the TMA-store epilogue: box = 32 rows x box_cols (64: SWIZZLE_128B, 32: SWIZZLE_64B)
static int make_out_map(CUtensorMap* map, void* base, int rows, int cols, int ld, int box_cols) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is unavailable (no CUDA driver?)");
    return TCAVP_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, 32u};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (output) failed (%d) rows=%d cols=%d ld=%d", (int)r, rows, cols, ld);
    return TCAVP_ERR_CUDA;
  }
  return TCAVP_OK;
}

template <int BLOCK_N, bool F8 = false>
static int launch_tc_pair(const tcavp_gemm_args& a, const EpilogueParams& ep, cudaStream_t stream) {
  // TMA-store epilogue: bf16 output rows in place (no row remap), 16-byte aligned rows, not the SwiGLU-backward form.  Measured on
  // B200 (profiles/gemm_tmastore_ab_r02.txt) within +-1 % of the 256-bit global stores on the K = 768 shapes; it frees the epilogue
  // warps' LSU work and writes whole lines.
  const bool tma_out = ep.out_dtype == TCAVP_BF16 && ep.remap_gi == 0 && ep.act != TCAVP_ACT_SWIGLU_BWD &&
                       (ep.ldo % 8) == 0 && reinterpret_cast<uintptr_t>(ep.out) % 16 == 0;
  CUtensorMap ma, mb, mo;
  int rc = make_map(&ma, a.A, a.M, a.K, a.lda, BLOCK_M, F8);
  if (rc) return rc;
  rc = make_map(&mb, a.W, a.N, a.K, a.ldw, BLOCK_N / 2, F8);
  if (rc) return rc;
  if (tma_out) {
    rc = make_out_map(&mo, ep.out, ep.M, ep.N, ep.ldo, ep.act == TCAVP_ACT_SWIGLU ? 32 : 64);
    if (rc) return rc;
  } else {
    mo = ma;      // unused by the kernel
  }
  const int smem_bytes = tma_out ? PairCfg<BLOCK_N, true>::SMEM_BYTES : PairCfg<BLOCK_N, false>::SMEM_BYTES;
  if (tma_out) TCAVP_CUDA(cudaFuncSetAttribute(gemm_tc_pair_kernel<BLOCK_N, true, F8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  else TCAVP_CUDA(cudaFuncSetAttribute(gemm_tc_pair_kernel<BLOCK_N, false, F8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  const int tiles_m = (a.M + 2 * BLOCK_M - 1) / (2 * BLOCK_M), tiles_n = (a.N + BLOCK_N - 1) / BLOCK_N;
  const int units = tiles_m * tiles_n;
  const int max_pairs = sm_count() / 2;
  const int grid = (units < max_pairs ? units : max_pairs) * 2;
  int flags = epilogue_flags(ep);
  if (tma_out) flags |= EPI_TMA_OUT;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  flags |= panel_flags(a.M, a.N, a.K, 2 * BLOCK_M, BLOCK_N, max_pairs, true);
  if (tma_out) TCAVP_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_pair_kernel<BLOCK_N, true, F8>, ma, mb, mo, ep, a.M, a.N, a.K, flags));
  else TCAVP_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_pair_kernel<BLOCK_N, false, F8>, ma, mb, mo, ep, a.M, a.N, a.K, flags));
  return check_launch(F8 ? "gemm_tc_pair_kernel<256,e4m3>" : "gemm_tc_pair_kernel<256>");
}

// k-blocks at the head and tail of a tile that the wide kernel issues half-major (1 would be plain k-major order).
// Measured on B200 (profiles/wide_split_ab_r02v.txt, same box, A-B-A-B): K = 3072 down_proj 775 -> 766 us, 7B o_proj 1263 -> 1258 us with 4;
// on K = 768 the wide tile gains 13 % from it (gate/up 844 -> 954 TF/s) but the double-buffered pair kernel stays ahead (1041 TF/s).
constexpr int WIDE_SPLIT = 4;

static int launch_tc_wide(const tcavp_gemm_args& a, const EpilogueParams& ep, cudaStream_t stream) {
  using C = WideCfg;
  CUtensorMap ma, mb;
  int rc = make_map(&ma, a.A, a.M, a.K, a.lda, 2 * BLOCK_M);
  if (rc) return rc;
  rc = make_map(&mb, a.W, a.N, a.K, a.ldw, C::HALF_N);
  if (rc) return rc;
  TCAVP_CUDA(cudaFuncSetAttribute(gemm_tc_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  const int tiles_m = (a.M + 4 * BLOCK_M - 1) / (4 * BLOCK_M), tiles_n = (a.N + C::BLOCK_N - 1) / C::BLOCK_N;
  const int units = tiles_m * tiles_n;
  const int max_pairs = sm_count() / 2;
  const int grid = (units < max_pairs ? units : max_pairs) * 2;
  int flags = epilogue_flags(ep);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  flags |= panel_flags(a.M, a.N, a.K, 4 * BLOCK_M, C::BLOCK_N, max_pairs, true);
  TCAVP_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_wide_kernel, ma, mb, ep, a.M, a.N, a.K, flags, WIDE_SPLIT));
  return check_launch("gemm_tc_wide_kernel");
}

// TCAVP_GEMM_WIDE_K: contractions at least this long use the 512 x 256 pair tile (0 disables it).  Without the variable the value is
// tunable at run time (tcavp_gemm_wide_min_k): which of the two kernels wins on K >= 2048 differs from one B200 to the next (measured:
// wide +6-15 % on some boards, pair +6-12 % on others of the same pool — profiles/wide_vs_pair_r02y.txt), so ops.py times both once per process.
static int g_wide_k = -2;      // -2: not initialised
static int wide_min_k() {
  if (g_wide_k == -2) {
    const char* e = getenv("TCAVP_GEMM_WIDE_K");
    int v = e ? atoi(e) : 2048;
    if (v < 0) v = 0;
    g_wide_k = v;
  }
  return g_wide_k;
}

}  // namespace tc

// ------------------------------------------------------------------------------------------------
// fp32 SIMT kernel (exact FFMA accumulation: the rtol 1e-4 parity mode and the fp32 temporal / fusion layers).
// BM x BN output tile, 16-deep K slices, 256 threads as a 16 x 16 grid of (BM/16) x (BN/16) register tiles read from shared
// memory with 16-byte loads; the next K slice is fetched into registers while the current one is multiplied, so the global
// latency is hidden inside a CTA.  Tile shapes: 128x128 (8x8 per thread) for big problems, 64x64, and 32x64 / 16x64 when the
// 64x64 grid would not fill the GPU (e.g. post_mlp: 4096 x 64 outputs with K = 3200).
// ------------------------------------------------------------------------------------------------
namespace simt {
constexpr int BK = 16;

template <typename T, int BM, int BN>
__global__ void __launch_bounds__(256) gemm_simt_kernel(const T* __restrict__ A, int lda, const T* __restrict__ W, int ldw,
                                                        EpilogueParams ep, int M, int Nacc, int K, int vec4) {
  constexpr int TM = BM / 16, TN = BN / 16;
  constexpr int LA = (BM * BK + 255) / 256, LW = (BN * BK + 255) / 256;     // elements fetched per thread and slice
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Ws[BK][BN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int jn = 0; jn < TN; ++jn) acc[i][jn] = 0.f;
  float ra[LA], rw[LW];
  auto fetch = [&](int k0) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = threadIdx.x + i * 256, r = e >> 4, c = e & 15;
      const int gm = m0 + r, gk = k0 + c;
      ra[i] = (e < BM * BK && gm < M && gk < K) ? Cvt<T>::to_f(A[(size_t)gm * lda + gk]) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < LW; ++i) {
      const int e = threadIdx.x + i * 256, r = e >> 4, c = e & 15;
      const int gn = n0 + r, gk = k0 + c;
      rw[i] = (e < BN * BK && gn < Nacc && gk < K) ? Cvt<T>::to_f(W[(size_t)gn * ldw + gk]) : 0.f;
    }
  };
  auto publish = [&]() {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      const int e = threadIdx.x + i * 256;
      if (e < BM * BK) As[e & 15][e >> 4] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < LW; ++i) {
      const int e = threadIdx.x + i * 256;
      if (e < BN * BK) Ws[e & 15][e >> 4] = rw[i];
    }
  };
  fetch(0);
  publish();
  __syncthreads();
  for (int k0 = 0; k0 < K; k0 += BK) {
    const bool more = k0 + BK < K;
    if (more) fetch(k0 + BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], w[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = As[k][ty * TM + i];
#pragma unroll
      for (int jn = 0; jn < TN; ++jn) w[jn] = Ws[k][tx * TN + jn];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int jn = 0; jn < TN; ++jn) acc[i][jn] = fmaf(a[i], w[jn], acc[i][jn]);
    }
    __syncthreads();
    if (more) {
      publish();
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int m = m0 + ty * TM + i;
    if (m >= M) continue;
    const int mo = remap_row(ep.remap_gi, ep.remap_go, ep.remap_off, m);
    if (ep.row_scale) {
      const float rs = __ldg(ep.row_scale + m);
#pragma unroll
      for (int jn = 0; jn < TN; ++jn) acc[i][jn] *= rs;
    }
#pragma unroll
    for (int q = 0; q < TN / 4; ++q) {     // four adjacent accumulator columns at a time (SwiGLU pairs / RoPE quads stay together)
      const int n = n0 + tx * TN + 4 * q;
      const float c0 = acc[i][4 * q], c1 = acc[i][4 * q + 1], c2 = acc[i][4 * q + 2], c3 = acc[i][4 * q + 3];
      if (ep.act == TCAVP_ACT_SWIGLU) {
        epilogue_store(ep, m, mo, n / 2, silu_f(c0) * c1);
        epilogue_store(ep, m, mo, n / 2 + 1, silu_f(c2) * c3);
      } else if (ep.rope_cols > 0 && n < ep.rope_cols) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(ep.rope) + (size_t)((n % ep.rope_dh) >> 2) * ep.rope_L + (m % ep.rope_L));
        epilogue_store(ep, m, mo, n, c0 * t.x - c1 * t.y);
        epilogue_store(ep, m, mo, n + 1, c1 * t.x + c0 * t.y);
        epilogue_store(ep, m, mo, n + 2, c2 * t.z - c3 * t.w);
        epilogue_store(ep, m, mo, n + 3, c3 * t.z + c2 * t.w);
      } else if (vec4 && n + 3 < ep.N) {     // four adjacent outputs: one 16-byte (fp32) / 8-byte (bf16) store
        float v[4] = {c0, c1, c2, c3};
        if (ep.bias) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + n));
          v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
        }
        if (ep.act == TCAVP_ACT_RELU) {
#pragma unroll
          for (int e = 0; e < 4; ++e) v[e] = fmaxf(v[e], 0.f);
        } else if (ep.act == TCAVP_ACT_GELU_TANH) {
#pragma unroll
          for (int e = 0; e < 4; ++e) v[e] = gelu_tanh_f(v[e]);
        }
        if (ep.residual) {
          if (ep.res_dtype == TCAVP_F32) {
            const float4 rr = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ep.residual) + (size_t)mo * ep.ldr + n);
            v[0] += rr.x; v[1] += rr.y; v[2] += rr.z; v[3] += rr.w;
          } else {
            const uint2 rr = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(ep.residual) + (size_t)mo * ep.ldr + n);
            v[0] += __uint_as_float(rr.x << 16); v[1] += __uint_as_float(rr.x & 0xffff0000u);
            v[2] += __uint_as_float(rr.y << 16); v[3] += __uint_as_float(rr.y & 0xffff0000u);
          }
        }
        if (ep.out_dtype == TCAVP_F32) {
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out) + (size_t)mo * ep.ldo + n) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
          uint2 u;
          u.x = tc::pack_bf16(v[0], v[1]);
          u.y = tc::pack_bf16(v[2], v[3]);
          *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(ep.out) + (size_t)mo * ep.ldo + n) = u;
        }
      } else {
        epilogue_store(ep, m, mo, n, c0);
        epilogue_store(ep, m, mo, n + 1, c1);
        epilogue_store(ep, m, mo, n + 2, c2);
        epilogue_store(ep, m, mo, n + 3, c3);
      }
    }
  }
}

template <typename T, int BM, int BN>
static void launch_simt(const tcavp_gemm_args& a, const EpilogueParams& ep, cudaStream_t stream) {
  dim3 grid((a.N + BN - 1) / BN, (a.M + BM - 1) / BM);
  // vector epilogue: rows of out / residual / bias start on 16-byte (fp32) or 8-byte (bf16) boundaries
  auto al = [](const void* p, int ld, int dtype) {
    const size_t esz = dtype == TCAVP_BF16 ? 2 : 4;
    return p == nullptr || (reinterpret_cast<uintptr_t>(p) % (4 * esz) == 0 && ((size_t)ld * esz) % (4 * esz) == 0);
  };
  const int vec4 = (ep.act == TCAVP_ACT_NONE || ep.act == TCAVP_ACT_RELU || ep.act == TCAVP_ACT_GELU_TANH) && ep.rope_cols == 0 && al(ep.out, ep.ldo, ep.out_dtype) &&
                   al(ep.residual, ep.ldr, ep.res_dtype) && (ep.bias == nullptr || reinterpret_cast<uintptr_t>(ep.bias) % 16 == 0);
  gemm_simt_kernel<T, BM, BN><<<grid, 256, 0, stream>>>(reinterpret_cast<const T*>(a.A), a.lda, reinterpret_cast<const T*>(a.W), a.ldw, ep, a.M,
                                                        a.N, a.K, vec4);
}
}  // namespace simt
}  // namespace tcavp

extern "C" int tcavp_gemm_wide_min_k(int new_value) {
  const int old = tcavp::tc::wide_min_k();
  if (new_value >= 0) tcavp::tc::g_wide_k = new_value;
  return old;
}

extern "C" int tcavp_gemm_tile_order(int tiles_m, int tiles_n, int panel_w, int* mg, int* nt) {
  TCAVP_REQUIRE(tiles_m > 0 && tiles_n > 0 && panel_w > 0 && mg != nullptr && nt != nullptr, "tcavp_gemm_tile_order: bad arguments");
  for (int u = 0; u < tiles_m * tiles_n; ++u) tcavp::tc::unit_to_tile(u, tiles_m, tiles_n, panel_w, mg[u], nt[u]);
  return 0;
}

extern "C" int tcavp_gemm(const tcavp_gemm_args* a, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(a != nullptr, "tcavp_gemm: null args");
  TCAVP_REQUIRE(a->M >= 0 && a->N > 0 && a->K > 0, "tcavp_gemm: bad shape M=%d N=%d K=%d", a->M, a->N, a->K);
  if (a->M == 0) return TCAVP_OK;
  TCAVP_REQUIRE(a->A && a->W && a->out, "tcavp_gemm: null A/W/out");
  TCAVP_REQUIRE(a->lda >= a->K && a->ldw >= a->K, "tcavp_gemm: lda/ldw smaller than K");
  TCAVP_REQUIRE(a->act == TCAVP_ACT_NONE || a->act == TCAVP_ACT_RELU || a->act == TCAVP_ACT_SWIGLU || a->act == TCAVP_ACT_SWIGLU_BWD ||
                    a->act == TCAVP_ACT_GELU_TANH,
                "tcavp_gemm: bad act %d", a->act);
  if (a->act == TCAVP_ACT_SWIGLU_BWD) {
    TCAVP_REQUIRE(a->in_dtype == TCAVP_BF16 && a->out_dtype == TCAVP_BF16 && a->aux_out && !a->bias && !a->residual && !a->rope_cos_sin &&
                      !a->sumsq_out && a->remap_gi == 0,
                  "tcavp_gemm: SWIGLU_BWD needs bf16 operands / output, the (gate, up) stash in aux_out and no other epilogue term");
    TCAVP_REQUIRE(a->N % 32 == 0 && a->ldo >= 2 * a->N && a->ld_aux >= 2 * a->N && a->ldo % 16 == 0 && a->ld_aux % 16 == 0 &&
                      reinterpret_cast<uintptr_t>(a->out) % 32 == 0 && reinterpret_cast<uintptr_t>(a->aux_out) % 32 == 0,
                  "tcavp_gemm: SWIGLU_BWD needs N %% 32 == 0, ldo / ld_aux >= 2N and multiples of 16, 32-byte aligned out / aux_out");
  }
  TCAVP_REQUIRE(a->act != TCAVP_ACT_SWIGLU || (a->N % 2 == 0), "tcavp_gemm: SwiGLU needs an even number of interleaved rows");
  TCAVP_REQUIRE(a->out_dtype == TCAVP_F32 || a->out_dtype == TCAVP_BF16, "tcavp_gemm: bad out_dtype");
  TCAVP_REQUIRE(!a->residual || a->res_dtype == TCAVP_F32 || a->res_dtype == TCAVP_BF16, "tcavp_gemm: bad res_dtype");
  EpilogueParams ep;
  ep.M = a->M;
  ep.N = a->act == TCAVP_ACT_SWIGLU ? a->N / 2 : a->N;
  ep.out = a->out; ep.ldo = a->ldo; ep.out_dtype = a->out_dtype;
  ep.bias = a->bias;
  ep.residual = a->residual; ep.ldr = a->ldr; ep.res_dtype = a->res_dtype;
  ep.act = a->act;
  ep.remap_gi = a->remap_gi; ep.remap_go = a->remap_go; ep.remap_off = a->remap_off;
  ep.row_scale = a->row_scale;
  ep.rope = a->rope_cos_sin; ep.rope_L = a->rope_L; ep.rope_dh = a->rope_dh; ep.rope_cols = a->rope_cos_sin ? a->rope_cols : 0;
  ep.sumsq_out = a->sumsq_out;
  ep.row_sumsq = a->row_sumsq; ep.ss_inv = a->sumsq_inv_cols; ep.ss_eps = a->sumsq_eps;
  TCAVP_REQUIRE(!(a->row_scale && a->row_sumsq), "tcavp_gemm: row_scale and row_sumsq are exclusive");
  TCAVP_REQUIRE((!a->sumsq_out && !a->row_sumsq) || a->in_dtype == TCAVP_BF16, "tcavp_gemm: sumsq_out / row_sumsq need bf16 operands");
  TCAVP_REQUIRE(!a->sumsq_out || a->act != TCAVP_ACT_SWIGLU, "tcavp_gemm: sumsq_out is not defined for the SwiGLU epilogue");
  ep.aux = reinterpret_cast<__nv_bfloat16*>(a->aux_out); ep.ld_aux = a->ld_aux;
  ep.col_scale = a->col_scale;
  TCAVP_REQUIRE(!a->col_scale || a->in_dtype == TCAVP_E4M3, "tcavp_gemm: col_scale needs e4m3 operands");
  if (ep.aux && a->act != TCAVP_ACT_SWIGLU_BWD) {
    TCAVP_REQUIRE(a->act == TCAVP_ACT_SWIGLU && a->in_dtype == TCAVP_BF16, "tcavp_gemm: aux_out needs act SWIGLU and bf16 operands");
    TCAVP_REQUIRE(a->N % 32 == 0 && a->ld_aux >= a->N && a->ld_aux % 16 == 0 && reinterpret_cast<uintptr_t>(a->aux_out) % 32 == 0,
                  "tcavp_gemm: aux_out needs N %% 32 == 0, ld_aux >= N, ld_aux %% 16 == 0 and a 32-byte aligned pointer");
  }
  if (ep.rope_cols > 0) {
    TCAVP_REQUIRE(a->act == TCAVP_ACT_NONE && !a->bias, "tcavp_gemm: fused RoPE needs act NONE and no bias");
    TCAVP_REQUIRE(a->rope_L > 0 && a->rope_dh >= 32 && a->rope_dh % 32 == 0 && a->rope_cols % a->rope_dh == 0 && a->rope_cols <= a->N,
                  "tcavp_gemm: bad RoPE geometry (L=%d dh=%d cols=%d)", a->rope_L, a->rope_dh, a->rope_cols);
  }
  TCAVP_REQUIRE(ep.ldo >= ep.N, "tcavp_gemm: ldo %d < output width %d", ep.ldo, ep.N);
  TCAVP_REQUIRE(!ep.residual || ep.ldr >= ep.N, "tcavp_gemm: ldr too small");

  if (a->in_dtype == TCAVP_BF16) {
    TCAVP_REQUIRE(a->K % 8 == 0 && a->lda % 8 == 0 && a->ldw % 8 == 0, "tcavp_gemm(bf16): K, lda, ldw must be multiples of 8 (K=%d lda=%d ldw=%d)", a->K, a->lda, a->ldw);
    TCAVP_REQUIRE(reinterpret_cast<uintptr_t>(a->A) % 16 == 0 && reinterpret_cast<uintptr_t>(a->W) % 16 == 0, "tcavp_gemm(bf16): A and W must be 16-byte aligned");
    if (a->N <= 32) return tc::launch_tc<32>(*a, ep, stream);
    if (a->N <= 64) return tc::launch_tc<64>(*a, ep, stream);
    if (a->N <= 128) return tc::launch_tc<128>(*a, ep, stream);
    // large problems: CTA pairs (one 256 x 256 tile per TPC)
    // wide tile: long contraction AND at least ~4 waves of 512 x 256 tiles (coarser tiles quantise worse on mid-size problems).
    // ops.py's _long_k_gemm mirrors this condition to autotune the wide-vs-pair choice before the first such GEMM.
    if (tc::wide_min_k() > 0 && a->K >= tc::wide_min_k() && a->M >= 64 * tc::BLOCK_M &&
        (long long)((a->M + 511) / 512) * ((a->N + 255) / 256) >= 4LL * (sm_count() / 2))
      return tc::launch_tc_wide(*a, ep, stream);
    if (a->M >= 16 * tc::BLOCK_M) return tc::launch_tc_pair<256>(*a, ep, stream);
    return tc::launch_tc<256>(*a, ep, stream);
  }
  if (a->in_dtype == TCAVP_E4M3) {
    TCAVP_REQUIRE(a->col_scale && reinterpret_cast<uintptr_t>(a->col_scale) % 16 == 0, "tcavp_gemm(e4m3): needs a 16-byte aligned col_scale");
    TCAVP_REQUIRE(a->K % 16 == 0 && a->lda % 16 == 0 && a->ldw % 16 == 0, "tcavp_gemm(e4m3): K, lda, ldw must be multiples of 16 (K=%d lda=%d ldw=%d)",
                  a->K, a->lda, a->ldw);
    TCAVP_REQUIRE(reinterpret_cast<uintptr_t>(a->A) % 16 == 0 && reinterpret_cast<uintptr_t>(a->W) % 16 == 0, "tcavp_gemm(e4m3): A and W must be 16-byte aligned");
    TCAVP_REQUIRE(!a->row_sumsq && !a->sumsq_out && !a->aux_out && a->act != TCAVP_ACT_SWIGLU_BWD,
                  "tcavp_gemm(e4m3): row_sumsq, sumsq_out, aux_out and SWIGLU_BWD are bf16-only epilogues");
    if (a->N <= 32) return tc::launch_tc<32, true>(*a, ep, stream);
    if (a->N <= 64) return tc::launch_tc<64, true>(*a, ep, stream);
    if (a->N <= 128) return tc::launch_tc<128, true>(*a, ep, stream);
    if (a->M >= 16 * tc::BLOCK_M) return tc::launch_tc_pair<256, true>(*a, ep, stream);
    return tc::launch_tc<256, true>(*a, ep, stream);
  }
  if (a->in_dtype == TCAVP_F32) {
    const long long t64 = (long long)((a->N + 63) / 64) * ((a->M + 63) / 64);
    const long long t128 = (long long)((a->N + 127) / 128) * ((a->M + 127) / 128);
    const int sms = sm_count();
    if (a->N >= 128 && t128 >= 2LL * sms) simt::launch_simt<float, 128, 128>(*a, ep, stream);
    else if (t64 >= sms) simt::launch_simt<float, 64, 64>(*a, ep, stream);
    else if (t64 * 2 >= sms) simt::launch_simt<float, 32, 64>(*a, ep, stream);
    else simt::launch_simt<float, 16, 64>(*a, ep, stream);
    return check_launch("gemm_simt_kernel");
  }
  return fail_arg("tcavp_gemm: unsupported in_dtype %d", a->in_dtype);
}
