// tcavp_attention: softmax(scale * q.k^T + mask) . v for strided (b, t, h, d) views.
//
//   generic path : one warp per (batch, head, query row); lanes stride over the head dimension, keys are
//                  processed four at a time (four interleaved warp-shuffle reductions), online softmax in
//                  fp32.  Handles every head_dim on the path (16 ... 2048), causal and key-padding masks.
//   flash path   : bf16, head_dim 64/128 (the LLM self-attention, HF:251-289) — see attention_tc.cu.
//   wide path    : bf16, few queries against a wide head (LTSF cross-attention) — see attention_x.cu.
#include "common.cuh"

namespace tcavp {

int attention_tc_launch(const tcavp_attn_args& a, cudaStream_t stream);   // attention_tc.cu; returns 1 if not applicable
int attention_tm_launch(const tcavp_attn_args& a, cudaStream_t stream);   // attention_tm.cu (tcgen05 / TMEM / TMA); returns 1 if not applicable
int attention_x_launch(const tcavp_attn_args& a, cudaStream_t stream);    // attention_x.cu;  returns 1 if not applicable
int attention_xt_launch(const tcavp_attn_args& a, cudaStream_t stream);   // attention_xt.cu (tcgen05: two heads on one shared K = V head); returns 1 if not applicable

template <typename T, int NE>   // NE = ceil(dh / 32) head-dim elements per lane
__global__ void __launch_bounds__(128) attn_warp_kernel(tcavp_attn_args a) {
  const int lane = threadIdx.x & 31;
  const long long w = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long total = (long long)a.B * a.H * a.Tq;
  if (w >= total) return;
  const int i = (int)(w % a.Tq);
  const int h = (int)((w / a.Tq) % a.H);
  const int b = (int)(w / ((long long)a.Tq * a.H));
  const int hk = h / (a.H / a.Hkv);
  const T* q = reinterpret_cast<const T*>(a.q) + (size_t)b * a.q_sb + (size_t)i * a.q_st + (size_t)h * a.dh;
  const T* k = reinterpret_cast<const T*>(a.k) + (size_t)b * a.k_sb + (size_t)hk * a.dh;
  const T* v = reinterpret_cast<const T*>(a.v) + (size_t)b * a.v_sb + (size_t)hk * a.dh;
  const int32_t* km = a.key_mask ? a.key_mask + (size_t)b * a.Tk : nullptr;

  float qr[NE], acc[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    const int d = lane + 32 * e;
    qr[e] = d < a.dh ? Cvt<T>::to_f(q[d]) * a.scale : 0.f;
    acc[e] = 0.f;
  }
  float m = -INFINITY, l = 0.f;
  const int kend = a.causal ? i + 1 : a.Tk;
  // dropout on the probabilities (train mode): the PV product uses keep ? p / (1 - p_drop) : 0, the row sum the undropped p
  const bool drop = a.drop_thresh != 0;
  const uint32_t dkey = drop ? drop_key(a.drop_seed, a.drop_site) : 0u;
  const unsigned long long drow = (unsigned long long)w * (unsigned long long)a.Tk;     // w = (b*H + h)*Tq + i
  for (int j0 = 0; j0 < kend; j0 += 4) {
    float s[4];
    bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = j0 + u;
      ok[u] = j < kend && (!km || km[j] != 0);
      float p = 0.f;
      if (ok[u]) {
        const T* kj = k + (size_t)j * a.k_st;
#pragma unroll
        for (int e = 0; e < NE; ++e) {
          const int d = lane + 32 * e;
          if (d < a.dh) p = fmaf(qr[e], Cvt<T>::to_f(kj[d]), p);
        }
      }
      s[u] = p;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < 4; ++u) s[u] += __shfl_xor_sync(0xffffffffu, s[u], o);
    }
    float mn = m;
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (ok[u]) mn = fmaxf(mn, s[u]);
    if (mn == -INFINITY) continue;   // nothing attendable so far (warp-uniform)
    const float corr = __expf(m - mn);   // m == -inf -> 0
    float p[4];
    float ps = 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      p[u] = ok[u] ? __expf(s[u] - mn) : 0.f;
      ps += p[u];
    }
    l = l * corr + ps;
    if (drop) {
#pragma unroll
      for (int u = 0; u < 4; ++u) p[u] = drop_keep(dkey, drow + (unsigned)(j0 + u), a.drop_thresh) ? p[u] * a.drop_scale : 0.f;
    }
#pragma unroll
    for (int e = 0; e < NE; ++e) acc[e] *= corr;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (ok[u]) {
        const T* vj = v + (size_t)(j0 + u) * a.v_st;
#pragma unroll
        for (int e = 0; e < NE; ++e) {
          const int d = lane + 32 * e;
          if (d < a.dh) acc[e] = fmaf(p[u], Cvt<T>::to_f(vj[d]), acc[e]);
        }
      }
    }
    m = mn;
  }
  const float inv = l > 0.f ? 1.f / l : 0.f;
  if (a.lse && lane == 0) a.lse[(size_t)b * a.lse_sb + (size_t)h * a.Tq + i] = m + logf(l);   // -inf when no key is visible
  T* o = reinterpret_cast<T*>(a.out) + (size_t)b * a.o_sb + (size_t)i * a.o_st + (size_t)h * a.dh;
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    const int d = lane + 32 * e;
    if (d < a.dh) o[d] = Cvt<T>::from_f(acc[e] * inv);
  }
}

// Narrow heads (dh <= 32: lane-polygon encoder dh = 16, LTSF attention block dh = 32): one CTA per (batch, head), K and V
// staged once in shared memory as fp32, ONE THREAD per query row (q and the output accumulator live in registers, K/V
// reads are warp-wide broadcasts), online softmax.  No cross-lane reductions at all.
template <typename T, int DH>
__global__ void __launch_bounds__(128) attn_row_kernel(tcavp_attn_args a) {
  extern __shared__ float sm_kv[];
  float* sK = sm_kv;
  float* sV = sK + (size_t)a.Tk * DH;
  int* sM = reinterpret_cast<int*>(sV + (size_t)a.Tk * DH);
  const int b = blockIdx.x / a.H, h = blockIdx.x % a.H;
  const int hk = h / (a.H / a.Hkv);
  const T* k = reinterpret_cast<const T*>(a.k) + (size_t)b * a.k_sb + (size_t)hk * DH;
  const T* v = reinterpret_cast<const T*>(a.v) + (size_t)b * a.v_sb + (size_t)hk * DH;
  for (int i = threadIdx.x; i < a.Tk * DH; i += blockDim.x) {
    const int j = i / DH, d = i % DH;
    sK[i] = Cvt<T>::to_f(k[(size_t)j * a.k_st + d]);
    sV[i] = Cvt<T>::to_f(v[(size_t)j * a.v_st + d]);
  }
  for (int j = threadIdx.x; j < a.Tk; j += blockDim.x) sM[j] = !a.key_mask || a.key_mask[(size_t)b * a.Tk + j] != 0;
  __syncthreads();
  const bool drop = a.drop_thresh != 0;
  const uint32_t dkey = drop ? drop_key(a.drop_seed, a.drop_site) : 0u;
  for (int i = threadIdx.x; i < a.Tq; i += blockDim.x) {
    const unsigned long long drow = ((unsigned long long)blockIdx.x * a.Tq + i) * (unsigned long long)a.Tk;   // blockIdx.x = b*H + h
    const T* q = reinterpret_cast<const T*>(a.q) + (size_t)b * a.q_sb + (size_t)i * a.q_st + (size_t)h * DH;
    float qr[DH], acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      qr[d] = Cvt<T>::to_f(q[d]) * a.scale;
      acc[d] = 0.f;
    }
    float m = -INFINITY, l = 0.f;
    const int kend = a.causal ? i + 1 : a.Tk;
    for (int j = 0; j < kend; ++j) {
      if (!sM[j]) continue;
      const float4* kj = reinterpret_cast<const float4*>(sK + (size_t)j * DH);
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int d4 = 0; d4 < DH / 4; ++d4) {
        const float4 kk = kj[d4];
        s0 = fmaf(qr[4 * d4], kk.x, s0);
        s1 = fmaf(qr[4 * d4 + 1], kk.y, s1);
        s0 = fmaf(qr[4 * d4 + 2], kk.z, s0);
        s1 = fmaf(qr[4 * d4 + 3], kk.w, s1);
      }
      const float s = s0 + s1;
      const float mn = fmaxf(m, s);
      const float corr = __expf(m - mn);
      float p = __expf(s - mn);
      l = l * corr + p;
      if (drop) p = drop_keep(dkey, drow + (unsigned)j, a.drop_thresh) ? p * a.drop_scale : 0.f;
      const float4* vj = reinterpret_cast<const float4*>(sV + (size_t)j * DH);
#pragma unroll
      for (int d4 = 0; d4 < DH / 4; ++d4) {
        const float4 vv = vj[d4];
        acc[4 * d4] = fmaf(acc[4 * d4], corr, p * vv.x);
        acc[4 * d4 + 1] = fmaf(acc[4 * d4 + 1], corr, p * vv.y);
        acc[4 * d4 + 2] = fmaf(acc[4 * d4 + 2], corr, p * vv.z);
        acc[4 * d4 + 3] = fmaf(acc[4 * d4 + 3], corr, p * vv.w);
      }
      m = mn;
    }
    const float inv = l > 0.f ? 1.f / l : 0.f;
    if (a.lse) a.lse[(size_t)b * a.lse_sb + (size_t)h * a.Tq + i] = m + logf(l);
    T* o = reinterpret_cast<T*>(a.out) + (size_t)b * a.o_sb + (size_t)i * a.o_st + (size_t)h * DH;
#pragma unroll
    for (int d = 0; d < DH; ++d) o[d] = Cvt<T>::from_f(acc[d] * inv);
  }
}

template <typename T>
static int launch_row(const tcavp_attn_args& a, cudaStream_t stream) {
  const size_t smem = (size_t)a.Tk * a.dh * 8 + (size_t)a.Tk * 4;
  const int threads = a.Tq <= 32 ? 32 : (a.Tq <= 64 ? 64 : 128);
  if (a.dh == 16) attn_row_kernel<T, 16><<<a.B * a.H, threads, smem, stream>>>(a);
  else attn_row_kernel<T, 32><<<a.B * a.H, threads, smem, stream>>>(a);
  return check_launch("attn_row_kernel");
}

template <typename T>
static int launch_warp(const tcavp_attn_args& a, cudaStream_t stream) {
  if ((a.dh == 16 || a.dh == 32) && a.Tk <= 128) return launch_row<T>(a, stream);
  const long long total = (long long)a.B * a.H * a.Tq;
  const int grid = (int)((total + 3) / 4);
  const int ne = (a.dh + 31) / 32;
#define CASE(N)                                              \
  if (ne <= N) {                                             \
    attn_warp_kernel<T, N><<<grid, 128, 0, stream>>>(a);     \
    return check_launch("attn_warp_kernel");                 \
  }
  CASE(1) CASE(2) CASE(3) CASE(4) CASE(8) CASE(12) CASE(16) CASE(32) CASE(64)
#undef CASE
  return fail_arg("tcavp_attention: head_dim %d > 2048 unsupported", a.dh);
}

}  // namespace tcavp

extern "C" int tcavp_attention(const tcavp_attn_args* a, tcavp_stream_t stream_) {
  using namespace tcavp;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  TCAVP_REQUIRE(a != nullptr, "tcavp_attention: null args");
  TCAVP_REQUIRE(a->B >= 0 && a->H > 0 && a->Hkv > 0 && a->H % a->Hkv == 0 && a->Tq >= 0 && a->Tk >= 0 && a->dh > 0,
                "tcavp_attention: bad shape B=%d H=%d Hkv=%d Tq=%d Tk=%d dh=%d", a->B, a->H, a->Hkv, a->Tq, a->Tk, a->dh);
  if (a->B == 0 || a->Tq == 0) return TCAVP_OK;
  TCAVP_REQUIRE(a->q && a->k && a->v && a->out, "tcavp_attention: null tensor");
  TCAVP_REQUIRE(!a->causal || a->Tq == a->Tk, "tcavp_attention: causal needs Tq == Tk");
  TCAVP_REQUIRE(a->dtype == TCAVP_F32 || a->dtype == TCAVP_BF16, "tcavp_attention: bad dtype");
  TCAVP_REQUIRE(a->drop_thresh == 0 || (a->drop_seed != nullptr && a->drop_scale > 0.f), "tcavp_attention: dropout needs a device seed and a scale");
  TCAVP_REQUIRE(!a->lse || a->dtype == TCAVP_F32 || a->dh <= 128, "tcavp_attention: lse needs head_dim <= 128 in bf16");
  if (a->dtype == TCAVP_BF16) {
    // two heads on one shared K = V head (checks its own shape conditions first; writes no lse)
    int rc = a->lse ? 1 : attention_xt_launch(*a, stream);
    if (rc > 0) rc = a->dh > 128 ? attention_x_launch(*a, stream) : attention_tm_launch(*a, stream);
    if (rc > 0 && a->dh <= 128) rc = attention_tc_launch(*a, stream);
    if (rc <= 0) return rc;
    return launch_warp<__nv_bfloat16>(*a, stream);
  }
  return launch_warp<float>(*a, stream);
}
