// Text generation on the device (include/tcavp.h: tcavp_sample_next, tcavp_decode_attention, tcavp_decode_embed).
//
// Every kernel here reads the decode position from device memory (position = offset + *counter) and the sampler advances that
// counter itself, so one decode iteration can be captured in a CUDA graph and replayed without host-side step numbers.
//
//   sample_next_kernel     one CTA per sequence: HF's logits processors (repetition penalty, no-repeat-n-gram, temperature, top-k,
//                          top-p) over the fp32 logits row, then a counter-hash inverse-CDF draw (or argmax), EOS -> pad, history append.
//                          Top-k and top-p find their thresholds by MSB-first radix descent over order-preserving keys (no sort).
//   decode_attn_kernel     one query row per (sequence, head) against the KV cache, keys split over CTAs in chunks of DEC_CHUNK
//   decode_combine_kernel  (flash-decoding); the combine merges the per-chunk (max, sum, accumulator) partials.  A bandwidth kernel:
//                          SIMT fp32 math, one pass over the live cache rows, no tensor cores.
//   decode_embed_kernel    the sampled tokens' embedding rows (+ GPT-2's wpe row) and the RoPE table row of the device position.
#include "common.cuh"

namespace tcavp {

constexpr int SAMPLE_THREADS = 1024;
constexpr int DEC_CHUNK = 128;        // keys per attention CTA
constexpr int DEC_THREADS = 128;      // 4 warps
constexpr float W_FIX = 1099511627776.f;   // 2^40: fixed-point scale of the sampling weights

__device__ __forceinline__ uint32_t order_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// Block-wide reductions for SAMPLE_THREADS threads (red: >= 32 slots of shared scratch).
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  if (w == 0) {
    v = lane < (int)(blockDim.x >> 5) ? red[lane] : -INFINITY;
    v = warp_max(v);
    if (lane == 0) red[0] = v;
  }
  __syncthreads();
  return red[0];
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v, unsigned long long* red) {
  v = warp_sum_u64(v);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  if (w == 0) {
    v = lane < (int)(blockDim.x >> 5) ? red[lane] : 0ull;
    v = warp_sum_u64(v);
    if (lane == 0) red[0] = v;
  }
  __syncthreads();
  return red[0];
}

__device__ __forceinline__ uint32_t sample_hash(uint32_t seed_lo, uint32_t seed_hi, uint32_t row, uint32_t step) {
  const uint32_t key = mix32(seed_lo ^ mix32(seed_hi + 0x9E3779B9U));
  return mix32(mix32(key ^ step) ^ (row * 0x85EBCA6BU + 0x632BE5ABU));
}

__global__ void __launch_bounds__(SAMPLE_THREADS) sample_next_kernel(
    const float* __restrict__ logits, long long ld, int V, float* __restrict__ work, long long* __restrict__ hist, int ld_hist,
    int hist_offset, int* __restrict__ state, const uint32_t* __restrict__ seed, int do_sample, float temperature, int top_k, float top_p,
    float rep_penalty, int ngram, long long eos, long long pad, int* __restrict__ done, long long* __restrict__ tokens_out, int B) {
  __shared__ unsigned int cnt[256];
  __shared__ unsigned long long mass[256];
  __shared__ unsigned long long red64[32];
  __shared__ float redf[32];
  __shared__ uint32_t s_prefix;
  __shared__ unsigned long long s_above;
  __shared__ int s_rem, s_tok;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int step = state[0];
  const int n = hist_offset + step;                 // history length (prompt + generated)
  const float* x = logits + (size_t)b * ld;
  float* w = work + (size_t)b * V;
  long long* h = hist + (size_t)b * ld_hist;

  for (int i = tid; i < V; i += SAMPLE_THREADS) w[i] = x[i];
  __syncthreads();
  // repetition penalty: the value of every distinct history token is recomputed from the raw logit, so duplicates write the same value
  if (rep_penalty != 1.f) {
    for (int j = tid; j < n; j += SAMPLE_THREADS) {
      const long long t = h[j];
      if (t >= 0 && t < V) {
        const float s = x[t];
        w[t] = s < 0.f ? s * rep_penalty : s / rep_penalty;
      }
    }
    __syncthreads();
  }
  // no-repeat-n-gram: every earlier n-gram whose first n - 1 tokens equal the last n - 1 tokens bans its last token
  if (ngram > 0 && n + 1 >= ngram) {
    for (int i = tid; i + ngram <= n; i += SAMPLE_THREADS) {
      bool same = true;
      for (int k = 0; k < ngram - 1 && same; ++k) same = h[i + k] == h[n - (ngram - 1) + k];
      if (same) {
        const long long t = h[i + ngram - 1];
        if (t >= 0 && t < V) w[t] = -INFINITY;
      }
    }
    __syncthreads();
  }
  const bool sample = do_sample != 0;
  if (sample && temperature != 1.f) {
    for (int i = tid; i < V; i += SAMPLE_THREADS) w[i] = w[i] / temperature;
    __syncthreads();
  }
  if (!sample) {      // argmax, lowest index on ties
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < V; i += SAMPLE_THREADS) {
      const float v = w[i];
      if (v > best || (v == best && i < bi)) { best = v; bi = i; }
    }
    const float m = block_max(best, redf);
    unsigned long long cand = (best == m) ? (unsigned long long)(unsigned)bi : 0xffffffffull;   // lowest index among the maxima
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
    if ((tid & 31) == 0) red64[tid >> 5] = cand;
    __syncthreads();
    if (tid < 32) {
      cand = red64[tid];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
      if (tid == 0) s_tok = cand == 0xffffffffull ? 0 : (int)cand;
    }
    __syncthreads();
  } else {
    // top-k: the k-th largest value by radix descent over counts; values below it are removed (ties at the k-th value are kept)
    if (top_k > 0 && top_k < V) {
      if (tid == 0) { s_prefix = 0u; s_rem = top_k; }
      uint32_t mask = 0u;
      for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += SAMPLE_THREADS) cnt[i] = 0u;
        __syncthreads();
        const uint32_t prefix = s_prefix;
        for (int i = tid; i < V; i += SAMPLE_THREADS) {
          const uint32_t k = order_key(w[i]);
          if ((k & mask) == prefix) atomicAdd(&cnt[(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid == 0) {
          int rem = s_rem;
          for (int bin = 255; bin >= 0; --bin) {
            if ((int)cnt[bin] >= rem) { s_prefix = prefix | ((uint32_t)bin << shift); break; }
            rem -= (int)cnt[bin];
          }
          s_rem = rem;
        }
        mask |= 255u << shift;
        __syncthreads();
      }
      const float kth = key_to_float(s_prefix);
      for (int i = tid; i < V; i += SAMPLE_THREADS)
        if (w[i] < kth) w[i] = -INFINITY;
      __syncthreads();
    }
    // weights of the survivors: w_i = floor(exp(x_i - max) * 2^40), exact integers, so every sum below is order-independent
    float mloc = -INFINITY;
    for (int i = tid; i < V; i += SAMPLE_THREADS) mloc = fmaxf(mloc, w[i]);
    const float m = block_max(mloc, redf);
    if (top_p > 0.f && top_p < 1.f && m > -INFINITY) {
      // top-p: keep the tokens whose mass strictly above them is < top_p (HF removes cum <= 1 - top_p in ascending order);
      // the smallest kept key is found by radix descent over per-bin weight sums
      unsigned long long tot = 0ull;
      for (int i = tid; i < V; i += SAMPLE_THREADS) tot += __float2ull_rz(expf(w[i] - m) * W_FIX);
      tot = block_sum_u64(tot, red64);
      const unsigned long long thresh = (unsigned long long)((double)top_p * (double)tot);
      if (tid == 0) { s_prefix = 0u; s_above = 0ull; }
      uint32_t mask = 0u;
      for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += SAMPLE_THREADS) { cnt[i] = 0u; mass[i] = 0ull; }
        __syncthreads();
        const uint32_t prefix = s_prefix;
        for (int i = tid; i < V; i += SAMPLE_THREADS) {
          const float v = w[i];
          const uint32_t k = order_key(v);
          if (v > -INFINITY && (k & mask) == prefix) {
            const uint32_t bin = (k >> shift) & 255u;
            atomicAdd(&cnt[bin], 1u);
            atomicAdd(&mass[bin], __float2ull_rz(expf(v - m) * W_FIX));
          }
        }
        __syncthreads();
        if (tid == 0) {
          unsigned long long above = s_above, best_above = 0ull;
          int best = -1;
          for (int bin = 255; bin >= 0; --bin) {
            if (cnt[bin] == 0u) continue;
            if (best >= 0 && above >= thresh) break;
            best = bin;
            best_above = above;
            above += mass[bin];
          }
          s_prefix = prefix | ((uint32_t)best << shift);
          s_above = best_above;
        }
        mask |= 255u << shift;
        __syncthreads();
      }
      const uint32_t kmin = s_prefix;
      for (int i = tid; i < V; i += SAMPLE_THREADS)
        if (order_key(w[i]) < kmin) w[i] = -INFINITY;
      __syncthreads();
    }
    // inverse CDF over the kept tokens in ascending token id: the first i with sum_{j <= i} w_j > r, r = floor(u * W / 2^32)
    const int per = (V + SAMPLE_THREADS - 1) / SAMPLE_THREADS;
    const int i0 = min(tid * per, V), i1 = min(i0 + per, V);
    unsigned long long mine = 0ull;
    if (m > -INFINITY)
      for (int i = i0; i < i1; ++i) mine += __float2ull_rz(expf(w[i] - m) * W_FIX);
    // exclusive scan of the per-thread sums (warp shuffles, then the warp totals)
    const int lane = tid & 31, wid = tid >> 5;
    unsigned long long inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) red64[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      unsigned long long t = red64[lane], s = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += u;
      }
      red64[lane] = s - t;          // exclusive prefix of the warp totals
      if (lane == 31) s_above = s;  // total W
    }
    if (tid == 0) s_tok = -1;
    __syncthreads();
    const unsigned long long W = s_above;
    const unsigned long long excl = red64[wid] + inc - mine;
    const uint32_t u = sample_hash(seed[0], seed[1], (uint32_t)b, (uint32_t)step);
    const unsigned long long r = __umul64hi(W, (unsigned long long)u << 32);
    if (W > 0ull && r >= excl && r < excl + mine) {
      unsigned long long c = excl;
      for (int i = i0; i < i1; ++i) {
        c += __float2ull_rz(expf(w[i] - m) * W_FIX);
        if (c > r) { s_tok = i; break; }
      }
    }
    __syncthreads();
    if (tid == 0 && s_tok < 0) {      // nothing drawable (every logit -inf or underflowed): the first maximum
      int t = 0;
      for (int i = 0; i < V; ++i) if (w[i] == m) { t = i; break; }
      s_tok = t;
    }
    __syncthreads();
  }
  if (tid == 0) {
    long long t = s_tok;
    if (eos >= 0) {
      if (done[b]) t = pad;
      if (t == eos) done[b] = 1;
    }
    if (n < ld_hist) h[n] = t;
    tokens_out[b] = t;
    // the last CTA to finish advances the step counter and records whether every row is done
    __threadfence();
    if (atomicAdd(&state[1], 1) == B - 1) {
      __threadfence();
      int all = eos >= 0;
      for (int i = 0; i < B && all; ++i) all = ((volatile int*)done)[i] != 0;
      state[1] = 0;
      state[0] = step + 1;
      if (all && state[2] == 0) state[2] = step + 1;
    }
  }
}

// ---- decode attention ---------------------------------------------------------------------------------------------------------------
template <typename T, int DH>
__global__ void __launch_bounds__(DEC_THREADS) decode_attn_kernel(tcavp_decode_attn_args a, int nsplit) {
  constexpr int NE = DH / 32;
  __shared__ float s_m[4], s_l[4], s_acc[4][DH];
  const int s = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int p = a.offset + *a.counter;            // position of the new row; keys 0 .. p
  const int j0 = s * DEC_CHUNK;
  if (p < 0 || p >= a.capacity || j0 > p) return;
  const int j1 = min(j0 + DEC_CHUNK, p + 1);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ratio = a.H / a.Hkv, hk = h / ratio;
  const T* q = reinterpret_cast<const T*>(a.q) + (size_t)b * a.q_sb + (size_t)h * DH;
  const T* kc = reinterpret_cast<const T*>(a.k_cache) + (size_t)b * a.cache_sb + (size_t)hk * DH;
  const T* vc = reinterpret_cast<const T*>(a.v_cache) + (size_t)b * a.cache_sb + (size_t)hk * DH;
  const T* kn = reinterpret_cast<const T*>(a.k_new) + (size_t)b * a.new_sb + (size_t)hk * DH;
  const T* vn = reinterpret_cast<const T*>(a.v_new) + (size_t)b * a.new_sb + (size_t)hk * DH;
  // the new row is read from its source in this launch and appended to the cache by the first query head of its group
  if (j1 == p + 1 && h % ratio == 0 && warp == 0) {
    T* kd = reinterpret_cast<T*>(a.k_cache) + (size_t)b * a.cache_sb + (size_t)p * a.cache_st + (size_t)hk * DH;
    T* vd = reinterpret_cast<T*>(a.v_cache) + (size_t)b * a.cache_sb + (size_t)p * a.cache_st + (size_t)hk * DH;
#pragma unroll
    for (int e = 0; e < NE; ++e) { kd[lane + 32 * e] = kn[lane + 32 * e]; vd[lane + 32 * e] = vn[lane + 32 * e]; }
  }
  float qr[NE], acc[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) { qr[e] = Cvt<T>::to_f(q[lane + 32 * e]) * a.scale; acc[e] = 0.f; }
  float m = -INFINITY, l = 0.f;
  for (int jb = j0 + warp * 4; jb < j1; jb += 16) {   // each warp takes 4 consecutive keys of every 16
    float sc[4];
    const T* kr[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = jb + u;
      kr[u] = j == p ? kn : kc + (size_t)j * a.cache_st;
      float d = 0.f;
      if (j < j1) {
#pragma unroll
        for (int e = 0; e < NE; ++e) d = fmaf(qr[e], Cvt<T>::to_f(kr[u][lane + 32 * e]), d);
      }
      sc[u] = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < 4; ++u) sc[u] += __shfl_xor_sync(0xffffffffu, sc[u], o);
    }
    float mn = m;
#pragma unroll
    for (int u = 0; u < 4; ++u) if (jb + u < j1) mn = fmaxf(mn, sc[u]);
    const float corr = __expf(m - mn);
    float pr[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) pr[u] = jb + u < j1 ? __expf(sc[u] - mn) : 0.f;
    l = l * corr + (pr[0] + pr[1]) + (pr[2] + pr[3]);
#pragma unroll
    for (int e = 0; e < NE; ++e) acc[e] *= corr;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = jb + u;
      if (j < j1) {
        const T* vr = j == p ? vn : vc + (size_t)j * a.cache_st;
#pragma unroll
        for (int e = 0; e < NE; ++e) acc[e] = fmaf(pr[u], Cvt<T>::to_f(vr[lane + 32 * e]), acc[e]);
      }
    }
    m = mn;
  }
  if (lane == 0) { s_m[warp] = m; s_l[warp] = l; }
#pragma unroll
  for (int e = 0; e < NE; ++e) s_acc[warp][lane + 32 * e] = acc[e];
  __syncthreads();
  // merge the 4 warps; partial record = (max, sum, acc[DH]) in fp32
  float* rec = a.workspace + ((size_t)(b * a.H + h) * nsplit + s) * (DH + 2);
  const float M = fmaxf(fmaxf(s_m[0], s_m[1]), fmaxf(s_m[2], s_m[3]));
  for (int d = threadIdx.x; d < DH; d += DEC_THREADS) {
    float v = 0.f;
#pragma unroll
    for (int w4 = 0; w4 < 4; ++w4) v += s_m[w4] == -INFINITY ? 0.f : s_acc[w4][d] * __expf(s_m[w4] - M);
    rec[2 + d] = v;
  }
  if (threadIdx.x == 0) {
    float L = 0.f;
#pragma unroll
    for (int w4 = 0; w4 < 4; ++w4) L += s_m[w4] == -INFINITY ? 0.f : s_l[w4] * __expf(s_m[w4] - M);
    rec[0] = M;
    rec[1] = L;
  }
}

template <typename T, int DH>
__global__ void __launch_bounds__(DH) decode_combine_kernel(tcavp_decode_attn_args a, int nsplit) {
  const int h = blockIdx.x, b = blockIdx.y, d = threadIdx.x;
  const int p = a.offset + *a.counter;
  if (p < 0 || p >= a.capacity) return;
  const int live = p / DEC_CHUNK + 1;
  const float* rec = a.workspace + (size_t)(b * a.H + h) * nsplit * (DH + 2);
  float M = -INFINITY;
  for (int s = 0; s < live; ++s) M = fmaxf(M, rec[(size_t)s * (DH + 2)]);
  float L = 0.f, v = 0.f;
  for (int s = 0; s < live; ++s) {
    const float* r = rec + (size_t)s * (DH + 2);
    const float f = r[0] == -INFINITY ? 0.f : __expf(r[0] - M);
    L = fmaf(r[1], f, L);
    v = fmaf(r[2 + d], f, v);
  }
  T* o = reinterpret_cast<T*>(a.out) + (size_t)b * a.o_sb + (size_t)h * DH;
  o[d] = Cvt<T>::from_f(L > 0.f ? v / L : 0.f);
}

template <typename T, int DH>
static int launch_decode(const tcavp_decode_attn_args& a, int nsplit, cudaStream_t stream) {
  decode_attn_kernel<T, DH><<<dim3(nsplit, a.H, a.B), DEC_THREADS, 0, stream>>>(a, nsplit);
  int rc = check_launch("decode_attn_kernel");
  if (rc) return rc;
  decode_combine_kernel<T, DH><<<dim3(a.H, a.B), DH, 0, stream>>>(a, nsplit);
  return check_launch("decode_combine_kernel");
}

// ---- embedding rows / RoPE row of the device position ----------------------------------------------------------------------------------
template <typename T>
__global__ void decode_embed_kernel(const long long* __restrict__ tokens, const T* __restrict__ embed, int vocab, const T* __restrict__ wpe,
                                    int n_pos, T* __restrict__ out, int ldo, int H, const float* __restrict__ rope_full, int rope_L, int dh,
                                    int rope_layout, float* __restrict__ rope_out, const int* __restrict__ counter, int offset, int B) {
  const int p = offset + *counter;
  if (blockIdx.x == B) {          // the RoPE table row of position p (layout 0: [L, dh/2, 2]; layout 1: [dh/4, L, 4])
    if (p < 0 || p >= rope_L) return;
    for (int i = threadIdx.x; i < dh; i += blockDim.x)
      rope_out[i] = rope_layout == 0 ? rope_full[(size_t)p * dh + i] : rope_full[((size_t)(i >> 2) * rope_L + p) * 4 + (i & 3)];
    return;
  }
  const long long t = tokens[blockIdx.x];
  const bool ok = t >= 0 && t < vocab;
  const bool pos_ok = wpe == nullptr || (p >= 0 && p < n_pos);
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    float v = ok ? Cvt<T>::to_f(embed[(size_t)t * H + i]) : 0.f;
    if (wpe != nullptr && pos_ok) v += Cvt<T>::to_f(wpe[(size_t)p * H + i]);
    out[(size_t)blockIdx.x * ldo + i] = Cvt<T>::from_f(v);
  }
}

}  // namespace tcavp

extern "C" {

int tcavp_sample_next(const float* logits, long long ld, int B, int V, float* work, long long* hist, int ld_hist, int hist_offset, int* state,
                      const uint32_t* seed, int do_sample, float temperature, int top_k, float top_p, float repetition_penalty,
                      int no_repeat_ngram_size, long long eos_token_id, long long pad_token_id, int* done, long long* tokens_out,
                      tcavp_stream_t stream) {
  using namespace tcavp;
  TCAVP_REQUIRE(B >= 0 && V > 0 && ld >= V && ld_hist > 0 && hist_offset >= 0, "tcavp_sample_next: bad shape B=%d V=%d ld=%lld ld_hist=%d",
                B, V, ld, ld_hist);
  if (B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(logits && work && hist && state && done && tokens_out, "tcavp_sample_next: null tensor");
  TCAVP_REQUIRE(!do_sample || (seed != nullptr && temperature > 0.f), "tcavp_sample_next: sampling needs a device seed and temperature > 0");
  TCAVP_REQUIRE(repetition_penalty > 0.f && no_repeat_ngram_size >= 0 && top_k >= 0, "tcavp_sample_next: bad processor arguments");
  sample_next_kernel<<<B, SAMPLE_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      logits, ld, V, work, hist, ld_hist, hist_offset, state, seed, do_sample, temperature, top_k, top_p, repetition_penalty,
      no_repeat_ngram_size, eos_token_id, pad_token_id, done, tokens_out, B);
  return check_launch("sample_next_kernel");
}

long long tcavp_decode_attention_workspace_bytes(int B, int H, int dh, int capacity) {
  const long long nsplit = (capacity + tcavp::DEC_CHUNK - 1) / tcavp::DEC_CHUNK;
  return (long long)B * H * nsplit * (dh + 2) * 4;
}

int tcavp_decode_attention(const tcavp_decode_attn_args* a, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(a != nullptr, "tcavp_decode_attention: null args");
  TCAVP_REQUIRE(a->B >= 0 && a->H > 0 && a->Hkv > 0 && a->H % a->Hkv == 0 && a->capacity > 0,
                "tcavp_decode_attention: bad shape B=%d H=%d Hkv=%d capacity=%d", a->B, a->H, a->Hkv, a->capacity);
  TCAVP_REQUIRE(a->dh == 32 || a->dh == 64 || a->dh == 128, "tcavp_decode_attention: head_dim %d (32, 64 or 128)", a->dh);
  TCAVP_REQUIRE(a->dtype == TCAVP_F32 || a->dtype == TCAVP_BF16, "tcavp_decode_attention: bad dtype");
  if (a->B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(a->q && a->k_new && a->v_new && a->k_cache && a->v_cache && a->out && a->counter && a->workspace,
                "tcavp_decode_attention: null tensor");
  TCAVP_REQUIRE(a->workspace_bytes >= tcavp_decode_attention_workspace_bytes(a->B, a->H, a->dh, a->capacity),
                "tcavp_decode_attention: workspace of %lld bytes < %lld", a->workspace_bytes,
                tcavp_decode_attention_workspace_bytes(a->B, a->H, a->dh, a->capacity));
  const int nsplit = (a->capacity + DEC_CHUNK - 1) / DEC_CHUNK;
  if (a->dtype == TCAVP_BF16) {
    if (a->dh == 32) return launch_decode<__nv_bfloat16, 32>(*a, nsplit, stream);
    return a->dh == 64 ? launch_decode<__nv_bfloat16, 64>(*a, nsplit, stream) : launch_decode<__nv_bfloat16, 128>(*a, nsplit, stream);
  }
  if (a->dh == 32) return launch_decode<float, 32>(*a, nsplit, stream);
  return a->dh == 64 ? launch_decode<float, 64>(*a, nsplit, stream) : launch_decode<float, 128>(*a, nsplit, stream);
}

int tcavp_decode_embed(const long long* tokens, const void* embed, int vocab, const void* wpe, int n_pos, void* out, int ldo, int H, int dtype,
                       const float* rope_full, int rope_L, int dh, int rope_layout, float* rope_out, const int* counter, int offset, int B,
                       tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(B >= 0 && H > 0 && ldo >= H && vocab > 0, "tcavp_decode_embed: bad shape B=%d H=%d ldo=%d", B, H, ldo);
  TCAVP_REQUIRE(dtype == TCAVP_F32 || dtype == TCAVP_BF16, "tcavp_decode_embed: bad dtype");
  TCAVP_REQUIRE(rope_full == nullptr || (rope_out != nullptr && rope_L > 0 && dh > 0 && dh % 4 == 0 && (rope_layout == 0 || rope_layout == 1)),
                "tcavp_decode_embed: bad RoPE table arguments");
  if (B == 0) return TCAVP_OK;
  TCAVP_REQUIRE(tokens && embed && out && counter, "tcavp_decode_embed: null tensor");
  const int grid = B + (rope_full != nullptr ? 1 : 0);
  if (dtype == TCAVP_BF16)
    decode_embed_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(tokens, reinterpret_cast<const __nv_bfloat16*>(embed), vocab,
        reinterpret_cast<const __nv_bfloat16*>(wpe), n_pos, reinterpret_cast<__nv_bfloat16*>(out), ldo, H, rope_full, rope_L, dh, rope_layout,
        rope_out, counter, offset, B);
  else
    decode_embed_kernel<float><<<grid, 256, 0, stream>>>(tokens, reinterpret_cast<const float*>(embed), vocab, reinterpret_cast<const float*>(wpe),
        n_pos, reinterpret_cast<float*>(out), ldo, H, rope_full, rope_L, dh, rope_layout, rope_out, counter, offset, B);
  return check_launch("decode_embed_kernel");
}

}  // extern "C"
