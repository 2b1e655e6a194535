/*
 * libtcavp — C ABI of the B200-native (sm_100a) forward hot path of the Traffic-Context-Augmented
 * Vehicle Trajectory Prediction model.
 *
 * The reference (imjaegyun/Traffic-Context-Augmented-...-Multimodal-LLM) has no FFI/plugin layer: its
 * boundary is the Python class `MultiModalTrajectoryModel` (reference scripts/train.py:847-964).  This
 * header is the C boundary *beneath* our Python mirror of that class; each entry point names the
 * reference call site (file:line, relative to the reference root; "HF:" = transformers 5.5.0
 * models/llama/modeling_llama.py, "torch:" = torch.nn) whose arithmetic it replaces.
 *
 * Conventions
 *   - All pointers are DEVICE pointers.  The caller owns every buffer; the library allocates no device
 *     memory and keeps no state besides the cached driver entry point used to encode TMA descriptors.
 *   - Every call is asynchronous on `stream` (a cudaStream_t passed as void*), never synchronises,
 *     returns 0 on success or a negative TCAVP_ERR_* code; tcavp_last_error() gives the thread-local text.
 *   - dtype codes: TCAVP_F32 (fp32 storage, exact fp32 SIMT math, no TF32) / TCAVP_BF16 (bf16 storage,
 *     fp32 accumulate; dense contractions on tcgen05 tensor cores) / TCAVP_E4M3 (one-byte OCP e4m3fn GEMM operands
 *     with per-row / per-column fp32 scales: the opt-in fp8 serving mode of the decoder stack).
 *   - Matrices are row-major; "ld*" are leading dimensions in ELEMENTS.  Weights keep nn.Linear's
 *     [out_features, in_features] layout so state_dict tensors are consumed without transposition.
 *   - There is no CPU fallback anywhere: without an sm_100 device every compute entry point fails.
 */
#ifndef TCAVP_H_
#define TCAVP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* tcavp_stream_t; /* cudaStream_t */

enum { TCAVP_F32 = 0, TCAVP_BF16 = 1, TCAVP_E4M3 = 2 };
enum { TCAVP_OK = 0, TCAVP_ERR_ARG = -1, TCAVP_ERR_CUDA = -2, TCAVP_ERR_UNSUPPORTED = -3 };
enum { TCAVP_ACT_NONE = 0, TCAVP_ACT_RELU = 1, TCAVP_ACT_SWIGLU = 2, TCAVP_ACT_SWIGLU_BWD = 3,
       TCAVP_ACT_GELU_TANH = 4 /* HF "gelu_new" (GPT-2 mlp.c_fc): 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))) */ };

/* ---- library ------------------------------------------------------------------------------- */
const char* tcavp_last_error(void);
int tcavp_version(void);
/* Fills SM count and compute capability of the current device. */
int tcavp_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
long long tcavp_launch_count(void);
/* Name of the kernel the calling thread's most recent entry-point call launched last (static string; "" before the first launch).
 * Test aid: proves which variant a shape was routed to (e.g. the tcgen05 kernel rather than its mma.sync fallback). */
const char* tcavp_last_kernel(void);
/* Profiling aid: one warp spins for `ns` nanoseconds on `stream` and writes (elapsed SM cycles, elapsed ns) to out2[0..1]
 * (device memory) — the true average SM clock while other kernels run next to it. */
int tcavp_clock_probe(unsigned long long* out2, unsigned long long ns, tcavp_stream_t stream);

/* Routing threshold of the two CTA-pair tcgen05 GEMM kernels: contractions with K >= the value run the 512 x 256 "wide" tile, shorter
 * ones the double-buffered 256 x 256 tile; 0 disables the wide kernel.  Returns the previous value; a negative argument only queries.
 * (Which kernel wins at K >= 2048 differs from board to board; the Python front end times both once per process.) */
int tcavp_gemm_wide_min_k(int new_value);
/* Host-only test aid (no device work): the tile order of the persistent tcgen05 GEMM kernels.  For unit = 0 .. tiles_m*tiles_n-1 writes the
 * row-block index to mg[unit] and the n-tile index to nt[unit]; `panel_w` n-tiles per L2-resident W panel (>= tiles_n: row-major order).
 * Same function the kernels run (csrc/gemm.cu: unit_to_tile). */
int tcavp_gemm_tile_order(int tiles_m, int tiles_n, int panel_w, int* mg, int* nt);

/* ---- dense contraction with fused epilogue --------------------------------------------------
 * out[m', n] = act( sum_k A[m,k] * W[n,k] + bias[n] ) + residual[m', n]
 *
 * Replaces every nn.Linear / F.linear on the path: HF LlamaAttention q/k/v/o_proj (HF:251-289) and
 * LlamaMLP gate/up/down (HF:182-196), peft lora.Linear (y = Wx + (alpha/r) B(A x), train.py:432-440),
 * nn.MultiheadAttention / nn.Transformer* in/out projections and FFNs (train.py:358-359, 402-406,
 * 663-670, 754), q_proj (train.py:521), lane_fc / post_mlp / dec_proj / dec_unproj (train.py:784-799).
 *
 *   in_dtype   TCAVP_BF16: A and W are bf16 -> TMA-fed tcgen05.mma, fp32 accumulators in TMEM.
 *              Requires K % 8 == 0, lda % 8 == 0, ldw % 8 == 0 and 16-byte aligned A / W.
 *              TCAVP_F32 : A and W are fp32 -> SIMT FFMA kernel (exact fp32 accumulate).
 *              TCAVP_E4M3: A and W are e4m3fn bytes -> tcgen05.mma.kind::f8f6f4, fp32 accumulators in TMEM.  Requires
 *              col_scale, K % 16 == 0, lda % 16 == 0, ldw % 16 == 0 and 16-byte aligned A / W; output and residual stay
 *              bf16 / fp32.  row_sumsq, sumsq_out, aux_out and SWIGLU_BWD are bf16-only (TCAVP_ERR_ARG).
 *   LoRA       is NOT an epilogue term: the caller appends T = x.A^T (rank r, from a skinny call of
 *              this same function) as extra K columns of A and (alpha/r).B as extra K columns of W,
 *              so the rank-r update accumulates in the same TMEM tile as the base product.
 *   act        RELU, or SWIGLU: W rows are interleaved (gate_0, up_0, gate_1, up_1, ...), N counts the
 *              interleaved rows, the output has N/2 columns silu(gate_j) * up_j (HF:190); bias,
 *              residual and ldo refer to the N/2 output columns.
 *   row remap  remap_gi > 0: m' = (m / remap_gi) * remap_go + (m % remap_gi) + remap_off (writes the
 *              16 image-token rows of each scene straight into the fused (B, L, H) buffer,
 *              train.py:521-528).  Otherwise m' = m.
 *   residual   optional [M', N] tensor added after the activation; may alias `out`.
 *   row scale  row_scale != NULL: every accumulator of row m is multiplied by row_scale[m] before anything else.
 *              With the RMSNorm weight folded into W at pack time this fuses HF's LlamaRMSNorm (HF:53-70) into the
 *              projection that consumes it: w * (x * rstd) . W^T == rstd * (x . (W diag(w))^T); rstd comes from
 *              tcavp_row_rstd.
 *   RoPE       rope_cols > 0 fuses HF's apply_rotary_pos_emb (HF:146-170) into the epilogue of the packed QKV
 *              projection: output columns [0, rope_cols) are heads of width rope_dh whose W rows were
 *              permuted at pack time so that the rotation partners (i, i + dh/2) sit in adjacent columns
 *              (2i, 2i+1); row m has position m % rope_L; rope_cos_sin is the layout-1 table of
 *              tcavp_rope_table.  q.k is invariant under the shared permutation, v is not permuted.
 */
typedef struct tcavp_gemm_args {
  int M, N, K;
  const void* A; int lda;
  const void* W; int ldw;
  int in_dtype;
  void* out; int ldo; int out_dtype;
  const float* bias;
  const void* residual; int ldr; int res_dtype;
  int act;
  int remap_gi, remap_go, remap_off;
  const float* rope_cos_sin; int rope_L, rope_dh, rope_cols;
  const float* row_scale;
  /* Fused RMSNorm statistics across GEMMs (bf16 tensor-core path): a producer GEMM adds sum_n out[m', n]^2 of its final
   * (post-residual) output rows into sumsq_out[m'] — unsigned 64-bit FIXED POINT with 20 fractional bits (zeroed by the caller):
   * integer atomics make the sum independent of the order in which tiles finish, so results stay bit-reproducible and scenes
   * stay independent of their batch.  A consumer GEMM given row_sumsq applies rsqrt(row_sumsq[m] * 2^-20 * sumsq_inv_cols +
   * sumsq_eps) to the raw accumulators exactly like row_scale.  Removes the separate tcavp_row_rstd pass over the residual
   * stream between decoder sub-blocks (HF:53-70 LlamaRMSNorm). */
  unsigned long long* sumsq_out;
  const unsigned long long* row_sumsq; float sumsq_inv_cols, sumsq_eps;
  void* aux_out; int ld_aux;   /* bf16 operands only.  SWIGLU: also store the raw (row-scaled) gate/up accumulators, interleaved
                                  [M', N] bf16, for the backward pass (the fine-tune step stashes them; NULL otherwise).
                                  SWIGLU_BWD (fine-tune step): INPUT — the stashed (gate, up) pairs [M', 2N]; the N accumulator
                                  columns are d(mid) and the epilogue writes the 2N interleaved columns (d gate, d up) to `out`
                                  (bf16, ldo >= 2N): d gate = d u s (1 + g (1 - s)), d up = d g s, s = sigmoid(g) — the backward of
                                  HF LlamaMLP's act_fn(gate) * up (HF:190) fused into the down_proj^T GEMM. */
  const float* col_scale;      /* e4m3 operands only (required there, 16-byte aligned, N floats): accumulator column n is multiplied by
                                  col_scale[n] (the weight row's dequantisation factor) before the row factor, RoPE and SwiGLU — for
                                  SwiGLU n indexes the interleaved accumulator rows of W.  With row_scale = the activation rows'
                                  factors: out = act(acc * row_scale[m] * col_scale[n] + bias) + residual.  NULL for bf16 / fp32. */
} tcavp_gemm_args;

int tcavp_gemm(const tcavp_gemm_args* args, tcavp_stream_t stream);

/* fp32 rows -> bf16 [hi | hi | lo] (3 * cols columns; hi = bf16(x), lo = bf16(x - hi)).  Against weights packed [hi | lo | hi] one
 * bf16 tcavp_gemm over K = 3 * cols returns the fp32 product to ~2^-16 relative with fp32 accumulation — the tensor-core route for
 * the narrow fp32 layers of the temporal encoder / decoder (train.py:674-686, 784-790) in bf16 compute mode. */
int tcavp_split_bf16x3(const float* x, int ldx, void* out, int ldo, long long rows, int cols, tcavp_stream_t stream);

/* ---- attention ----------------------------------------------------------------------------------
 * out[b, i, h, :] = softmax_j( scale * q[b,i,h,:].k[b,j,hk,:] + mask ) . v[b,j,hk,:],  hk = h / (H/Hkv)
 *
 * Replaces torch: F.multi_head_attention_forward's core (train.py:371, 411-413, 678, 798) and HF
 * sdpa_attention_forward with the causal+padding mask of create_causal_mask (HF:399, 251-289).
 * q/k/v/out are strided views: element (b, t, h, d) lives at  ptr[b*s_b + t*s_t + h*dh + d].
 *   causal      != 0: key j allowed only if j <= i (requires Tq == Tk).
 *   key_mask    optional int32 [B, Tk], 1 = attend, 0 = masked (key padding).  Rows whose keys are all
 *               masked produce zeros (the reference discards such rows, train.py:378-380).
 * Softmax statistics and accumulation are fp32 for both dtypes.  `dtype` applies to q, k, v and out.
 * bf16 with dh in {16,32,64,96,128} and Tq,Tk <= 256 (flash kernel), causal self-attention with dh 64 / 128 and Tq == Tk >= 128 at
 * any length (tcgen05 kernels), or few queries against a wide head (Tq <= 32, dh % 64 == 0: LTSF cross-attention) runs on tensor cores;
 * everything else on the SIMT kernel.
 */
typedef struct tcavp_attn_args {
  int B, H, Hkv, Tq, Tk, dh;
  const void* q; long long q_sb, q_st;
  const void* k; long long k_sb, k_st;
  const void* v; long long v_sb, v_st;
  void* out; long long o_sb, o_st;
  int dtype;
  float scale;
  int causal;
  const int32_t* key_mask;
  /* dropout on the attention probabilities (nn.MultiheadAttention(dropout=p) in train mode: train.py:663, 754 and the nn.Transformer
   * layers of train.py:358, 402-405): P_drop = keep(b, h, i, j) ? P / (1 - p) : 0, applied after the softmax (row sums on the undropped
   * P).  drop_thresh == 0 disables it.  See tcavp_dropout for the mask function; element index = ((b*H + h)*Tq + i)*Tk + j. */
  const uint32_t* drop_seed; uint32_t drop_site; uint32_t drop_thresh; float drop_scale;
  /* optional fp32 [B, H, Tq] output (element (b, h, i) at lse[b*lse_sb + h*Tq + i]): the natural-log logsumexp of the scaled scores over
   * the keys row i may see, -inf for a row with no visible key.  Written by the self-attention routes (head_dim <= 128 bf16 and every
   * fp32 shape); the backward of tcavp_attention_bwd_owned recomputes the probabilities from it.  NULL writes nothing. */
  float* lse; long long lse_sb;
} tcavp_attn_args;

int tcavp_attention(const tcavp_attn_args* args, tcavp_stream_t stream);

/* ---- normalisation ---------------------------------------------------------------------------- */
/* out[r,:] = LayerNorm(x[r,:] + residual[r,:]) * w + b      (torch: nn.LayerNorm eps 1e-5; residual
 * optional — post-norm nn.Transformer*Layer, train.py:358, 402-405; attn_block 677-681; fusion 759-764).
 * remap/rowvec: optional scatter of row r to (r/gi)*go + r%gi + off with `rowvec[:]` added after the
 * affine (writes Q-Former tokens + vision_modality_embedding into the fused buffer, train.py:522-528). */
int tcavp_layernorm(const void* x, const void* residual, const float* w, const float* b, void* out, int rows, int cols,
                    float eps, int in_dtype, int out_dtype, int remap_gi, int remap_go, int remap_off,
                    const float* rowvec, tcavp_stream_t stream);
/* The same LayerNorm (no residual) with explicit row strides: out may be the leading columns of a wider operand — the GPT-2-arch path
 * writes ln_1(x) straight into the K-extended [ln_1(x) | LoRA side columns] operand of the fused c_attn GEMM (HF modeling_gpt2.py
 * GPT2Block.forward: ln_1 -> attn), which saves the copy into it.  bf16 rows of 256..1024 columns go through the bulk-copy ring. */
int tcavp_layernorm_strided(const void* x, int ldx, const float* w, const float* b, void* out, int ldo, int rows, int cols, float eps,
                            int in_dtype, int out_dtype, tcavp_stream_t stream);
/* out[r,:] = w * (x[r,:] * rsqrt(mean(x^2) + eps))          (HF:53-70 LlamaRMSNorm).  ldi / ldo are the row strides of
 * x / out in elements (the residual stream lives in K-extended rows that also carry the LoRA side columns). */
int tcavp_rmsnorm(const void* x, int ldi, const float* w, void* out, int rows, int cols, int ldo, float eps, int in_dtype,
                  int out_dtype, tcavp_stream_t stream);
/* out[r] = rsqrt(mean(x[r, 0:cols]^2) + eps)  — the per-row factor of LlamaRMSNorm, consumed by tcavp_gemm's row_scale. */
int tcavp_row_rstd(const void* x, int ldx, int rows, int cols, float eps, int dtype, float* out, tcavp_stream_t stream);
/* Per-row e4m3 quantisation of bf16 rows (the activation operand of the fp8 decoder projections, HF:182-196 / 251-289):
 *   s = 448 / amax(|x[r, :]|) (fp32, correctly rounded), q[r, c] = e4m3_rn_satfinite(x[r, c] * s), f[r] = amax / 448;
 *   an all-zero row gives q = 0, f = 0.  rms != 0 folds LlamaRMSNorm (HF:53-70; its weight is folded into the e4m3 weight) into the
 *   factor: f[r] = rsqrt(mean(x[r, :]^2) + eps) * amax / 448, so one read of x gives the QKV / gate-up operand and its row_scale.
 * x bf16 [rows, ldi], q e4m3 [rows, ldo] (bytes), f fp32 [rows].  cols % 16 == 0, 16 <= cols <= 14336, ldi % 8 == 0, ldo % 16 == 0, 16-byte
 * aligned x / q.  Rows stream through shared memory by the bulk-copy engine; every row is quantised independently of its batch. */
int tcavp_quant_e4m3_rows(const void* x, int ldi, void* q, int ldo, float* f, int rows, int cols, int rms, float eps, tcavp_stream_t stream);

/* ---- rotary embedding (HF:146-170 apply_rotary_pos_emb, default rope HF:73-136) ----------------
 * In place on the q and k head blocks of a packed [rows, ld] qkv buffer (q heads first, then k heads);
 * position of row r is r % L.  cos_sin is an fp32 [L, dh/2, 2] table. */
int tcavp_rope(void* qkv, int rows, int L, int ld, int n_q_heads, int n_k_heads, int dh, const float* cos_sin,
               int dtype, tcavp_stream_t stream);
/* Fills the cos/sin table as HF does: angle = pos * inv_freq[j] in fp32, cosf / sinf.  inv_freq is a device fp32
 * [dh/2] vector the host computes with HF's formula 1 / theta^(2j/dh) (HF:86-88).
 *   layout 0: [L, dh/2, 2]  (tcavp_rope)
 *   layout 1: [dh/4, L, 4]  (tcavp_gemm's fused RoPE: consecutive positions are contiguous, so the row-per-thread
 *                            epilogue reads it coalesced) */
int tcavp_rope_table(float* cos_sin, const float* inv_freq, int L, int dh, int layout, tcavp_stream_t stream);

/* ---- fused-sequence assembly (train.py:526-528) -------------------------------------------------
 * fused[b, n_img + j, :] = embed[ids[b, j], :] + text_mod[:]   for j < L_text; mask_out[b, :] = [1]*n_img ++ mask. */
int tcavp_embed_text(const int64_t* ids, const int64_t* attn_mask, const void* embed, int embed_dtype,
                     const float* text_mod, void* fused, int fused_dtype, int32_t* mask_out, int B, int L_text,
                     int n_img, int H, int vocab, tcavp_stream_t stream);
/* out[r', :] = x[r, :] + rowvec[:] with the row remap above (Identity q_proj case, train.py:492-495, 522). */
int tcavp_add_rowvec(const void* x, const float* rowvec, void* out, int rows, int cols, int in_dtype, int out_dtype,
                     int remap_gi, int remap_go, int remap_off, tcavp_stream_t stream);
/* dtype conversion / strided copy / row broadcast: out[r, 0:cols] = in[r % in_row_mod, 0:cols]
 * (in_row_mod <= 0: no modulo).  The broadcast form expands the Q-Former query tokens over the batch
 * (train.py:412). */
int tcavp_cast(const void* in, int ldi, int in_dtype, void* out, int ldo, int out_dtype, int rows, int cols,
               int in_row_mod, tcavp_stream_t stream);

/* ---- lane polygon encoder ends (train.py:364-365, 373-382) -------------------------------------- */
/* out[b,p,:] = W[:, 0:2] . polygon[b,p,:] + bias + pos[p,:];  key_mask[b,p] = p < len[b] */
int tcavp_poly_embed(const float* polygon, const int32_t* len, const float* w, const float* bias, const float* pos,
                     void* out, int out_dtype, int32_t* key_mask, int B, int P, int D, tcavp_stream_t stream);
/* out[b,:] = mean over p < len[b] of x[b,p,:]  (zeros when len[b] == 0) */
int tcavp_masked_mean(const void* x, int in_dtype, const int32_t* len, void* out, int out_dtype, int B, int P, int D,
                      tcavp_stream_t stream);

/* ---- temporal encoder / NLinear decoder (train.py:701-716, 837-839, 769-785) --------------------
 * enc[b, t, c] = sum_s We[c,t,s] * (xp[b,c,s] - xp[b,c,T-1]) + be[c,t] + xp[b,c,T-1] + pos[c,t],
 *   xp[b,c,s] = sum_f Wt[c,f] * x[b,f,s] + bt[c]                (token_proj, 1x1 conv)
 * Output layout is (B, T_in, C) — rows (b,t) with channels contiguous — so the attention block's
 * projections are plain row-major GEMMs.  Weight layouts (permuted once at pack time so that the channel
 * index is contiguous): we [T_in(t), T_in(s), C], be / pos [T_in, C], wt [C, F], bt [C]; T_in <= 64. */
int tcavp_ltsf_encode(const float* x, const float* wt, const float* bt, const float* we, const float* be,
                      const float* pos, void* enc, int out_dtype, int B, int F, int C, int T_in,
                      tcavp_stream_t stream);
/* dec[b, t, c] = sum_s Wd[c,t,s] * (enc[b,s,c] - enc[b,T-1,c]) + bd[c,t] + enc[b,T-1,c] + lane_adj[b,t,c]
 * (lane_adj optional; (B, T_out, C) layout — post_mlp / lane_fc weights are permuted accordingly at pack time).
 * wd [T_out, T_in(s), C], bd [T_out, C]. */
int tcavp_nlinear_decode(const void* enc, int enc_dtype, const float* wd, const float* bd, const void* lane_adj,
                         int adj_dtype, void* dec, int out_dtype, int B, int C, int T_in, int T_out,
                         tcavp_stream_t stream);

/* ---- fusion head + metrics (train.py:801-805, 941-943, 945-962, 1302-1322) ----------------------
 * Per (b, t): f = LN(fused[b,t,:]); f = W2.relu(W1.f + b1) + b2; o = Wo.f + bo (2 values);
 * decoded[b, :, t] = o + x[b, :, T_in-1].  With y and norm_stat (fp32 [B,4] = min_x,max_x,min_y,max_y):
 * metrics[0..4] += (sum of squared de-normalised x error, same for y, sum_b ADE_b, sum_b FDE_b,
 * MSE_x + MSE_y = the reference's training loss) and per_scene[b] = (ADE_b, FDE_b) — `metrics` is a
 * float[8] zeroed by the caller. */
int tcavp_fusion_head(const void* fused, int in_dtype, const float* ln_w, const float* ln_b, const float* w1,
                      const float* b1, const float* w2, const float* b2, const float* wo, const float* bo,
                      const float* x, float* decoded, const float* y, const float* norm_stat, float* metrics,
                      float* per_scene, int B, int C, int T_in, int T_out, tcavp_stream_t stream);
/* Same contract for d_model = 64 on the tensor cores (mma.sync tiles over (scene, step) rows, weights resident in shared memory,
 * split-bf16 operands: three products per linear, fp32 accumulation, relative error ~2^-16) — what the bf16 compute mode calls;
 * tcavp_fusion_head stays the exact-fp32 FFMA path of the rtol 1e-4 parity mode. */
int tcavp_fusion_head_tc(const void* fused, int in_dtype, const float* ln_w, const float* ln_b, const float* w1,
                      const float* b1, const float* w2, const float* b2, const float* wo, const float* bo,
                      const float* x, float* decoded, const float* y, const float* norm_stat, float* metrics,
                      float* per_scene, int B, int C, int T_in, int T_out, tcavp_stream_t stream);
/* Same metrics for an existing prediction (train.py:1302-1322; RMSE: ablation_study_without_lora.py:1237). */
int tcavp_traj_metrics(const float* decoded, const float* y, const float* norm_stat, float* metrics, float* per_scene,
                       int B, int T_out, tcavp_stream_t stream);

/* ==== fine-tune step: backward kernels (reference scripts/im_kim_train_GRN.py:1039-1040 loss.backward() + AdamW; the
 * reference leaves these to torch autograd).  Dense gradient contractions are tcavp_gemm calls on transposed operands:
 *   dX = dY . W      -> tcavp_gemm(A = dY, W = W^T)          dW = dY^T . X  -> tcavp_gemm(A = dY^T, W = X^T) ======== */

/* out[b][c][r] = in[b][r][c] for r < rows, c < cols (batch strides / leading dimensions in elements). */
int tcavp_transpose(const void* in, long long in_bstride, int ldi, int in_dtype, void* out, long long out_bstride, int ldo,
                    int out_dtype, int batch, int rows, int cols, tcavp_stream_t stream);
/* out[r % period][c] += x[r][c]  (fp32 [period, cols], accumulated): bias gradients (period 1) and the gradients of
 * broadcast tables — pos_embedding / pos_encoding / query_tokens / modality embeddings (train.py:365, 412, 522, 527, 839). */
int tcavp_period_sum(const void* x, int ldx, int dtype, long long rows, int cols, int period, float* out, tcavp_stream_t stream);
/* dx = y > 0 ? dy : 0  (nn.ReLU backward on the stored activation output). */
int tcavp_relu_bwd(const void* dy, int lddy, const void* y, int ldy, void* dx, int lddx, int dtype, long long rows, int cols,
                   tcavp_stream_t stream);
/* out = alpha * a + beta * b  (b optional): gradient accumulation where two consumers share a tensor, LoRA scaling. */
int tcavp_axpby(const void* a, int lda, int a_dtype, float alpha, const void* b, int ldb, int b_dtype, float beta, void* out, int ldo,
                int out_dtype, long long rows, int cols, tcavp_stream_t stream);
/* SwiGLU on interleaved (gate, up) columns (HF:190) and its backward; gu / dgu are [rows, 2I], out / dout [rows, I]. */
int tcavp_swiglu(const void* gu, void* out, int dtype, long long rows, int I, tcavp_stream_t stream);
int tcavp_swiglu_bwd(const void* dout, const void* gu, void* dgu, int dtype, long long rows, int I, tcavp_stream_t stream);
/* LayerNorm backward for a FROZEN LayerNorm (no residual input, no dw / db): dx = rstd (g - mean(g) - xhat mean(g xhat)) [+ add],
 * g = dy * w.  `add` (optional) is the gradient arriving on the residual branch, summed in the same pass.  Used by the fine-tune step
 * of a GPT-2-arch backbone, whose ln_1 / ln_2 / ln_f are frozen under peft (HF modeling_gpt2.py GPT2Block.forward). */
int tcavp_layernorm_bwd_dx(const void* dy, int lddy, const void* x, int ldx, const float* w, const void* add, int ldadd, void* dx, int lddx,
                           int dtype, int rows, int cols, float eps, tcavp_stream_t stream);
/* HF ACT2FN["gelu_new"] (GPT-2 mlp.act: 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))) on [rows, cols] as a pass of its own, and its
 * backward on the stored pre-activation x: dx = dy * d gelu_new(x) / dx.  The fine-tune step of a GPT-2-arch backbone (HF
 * modeling_gpt2.py GPT2MLP.forward, reached through reference scripts/train.py:445-453) keeps c_fc's output for the backward pass;
 * inference applies the activation in the tcavp_gemm epilogue (TCAVP_ACT_GELU_TANH). */
int tcavp_gelu_tanh(const void* x, int ldx, void* out, int ldo, int dtype, long long rows, int cols, tcavp_stream_t stream);
int tcavp_gelu_tanh_bwd(const void* dy, int lddy, const void* x, int ldx, void* dx, int lddx, int dtype, long long rows, int cols,
                        tcavp_stream_t stream);
/* Backward of tcavp_layernorm (input x + residual): dx (optional), dw += sum_r dy*xhat, db += sum_r dy (optional pair). */
int tcavp_layernorm_bwd(const void* dy, int dy_dtype, const void* x, const void* residual, int x_dtype, const float* w, int rows,
                        int cols, float eps, void* dx, int dx_dtype, float* dw, float* db, tcavp_stream_t stream);
/* Backward of LlamaRMSNorm (HF:53-70): dx = rstd * (g - xhat * mean(g * xhat)) + add, g = dy * w (w NULL = unit weight,
 * the folded-weight form of the LLM stack); `add` (optional) is the residual-branch gradient. */
int tcavp_rmsnorm_bwd(const void* dy, int lddy, const void* x, int ldx, const float* w, const void* add, int ldadd, void* dx, int lddx,
                      int dtype, int rows, int cols, float eps, tcavp_stream_t stream);
/* Rotary embedding on adjacent column pairs (the layout of tcavp_gemm's fused RoPE), in place on columns [0, cols) of a
 * [rows, ld] buffer; inverse != 0 applies the transpose rotation (= the backward of HF:146-170). Table layout 1. */
int tcavp_rope_adjacent(void* buf, int dtype, long long rows, int L, int ld, int cols, int dh, const float* table, int inverse,
                        tcavp_stream_t stream);
/* out[remap_out(r), :] = in[remap_in(r), :], remap(r) = (r / gi) * go + r % gi + off (gi = 0: identity): scatter into /
 * gather from the fused (B, L, H) sequence (train.py:528 torch.cat and its backward). */
int tcavp_copy_rows(const void* in, int ldi, int in_dtype, int in_gi, int in_go, int in_off, void* out, int ldo, int out_dtype,
                    int out_gi, int out_go, int out_off, long long rows, int cols, tcavp_stream_t stream);
/* Backward of tcavp_masked_mean (train.py:373-382). */
int tcavp_masked_mean_bwd(const void* dout, int dout_dtype, const int32_t* len, void* dx, int dx_dtype, int B, int P, int D,
                          tcavp_stream_t stream);
/* Backward of the per-channel NLinear map out[b,t,c] = sum_s W[t][s][c] (in[b,s,c] - in[b,T-1,c]) + bias[t][c] + in[b,T-1,c]
 * (train.py:701-716, 769-785): din (optional, needs w) and dw[t][s][c] += ... (optional, needs in).  The bias gradient is
 * tcavp_period_sum(g, period = T_out). */
int tcavp_nlinear_bwd(const void* g, int g_dtype, const void* in, int in_dtype, const float* w, void* din, int din_dtype, float* dw,
                      int B, int C, int T_in, int T_out, tcavp_stream_t stream);
/* decoded[b,f,t] = o[b,t,f] + x[b,f,T_in-1]  (train.py:941-943; o = out_proj rows). */
int tcavp_head_assemble(const float* o, const float* x, float* decoded, int B, int T_in, int T_out, tcavp_stream_t stream);
/* d_o[b,t,f] = gscale * d loss / d decoded[b,f,t] for loss = MSE_x + MSE_y on de-normalised coordinates (train.py:945-962);
 * gscale: optional device scalar (the incoming loss gradient). */
int tcavp_traj_loss_bwd(const float* decoded, const float* y, const float* norm_stat, const float* gscale, float* d_o, int B, int T_out,
                        tcavp_stream_t stream);
/* Rank-r weight gradients of peft lora.Linear (train.py:432-440): out[n][j] += sum_m row_scale[m] * Y[m][n] * Z[m][j], J <= 32
 * (row_scale optional: the RMSNorm rstd of the folded-norm form). */
int tcavp_skinny_dw(const void* Y, int ldy, int y_dtype, const void* Z, int ldz, int z_dtype, const float* row_scale, float* out, int ldo,
                    long long M, int N, int J, tcavp_stream_t stream);
/* Feed-forward sub-layer of a d_model = 64 post-norm encoder layer in ONE kernel (torch nn.TransformerEncoderLayer: the lane-polygon
 * encoder, train.py:358 — d_model 64, dim_feedforward F):  out = LayerNorm(x + linear2(relu(linear1(x)))) * ln_w + ln_b.
 * x, out: bf16 [M, 64] (contiguous rows); w1: bf16 [F, 64]; w2: bf16 [64, F]; biases / LayerNorm parameters fp32; F % 128 == 0.
 * tcgen05 / TMEM / TMA: the [M, F] hidden activation stays in tensor memory (bf16, A operand of the second product). */
int tcavp_ffn64_ln(const void* x, const void* w1, const float* b1, const void* w2, const float* b2, const float* ln_w, const float* ln_b,
                   float eps, void* out, long long M, int F, tcavp_stream_t stream);
/* peft lora.Linear in train() mode (train.py:432-440, lora_dropout): every target module t (q_proj, k_proj, v_proj) applies lora_A to
 * dropout(x) with its OWN mask keep_t(m H + h) = tcavp_dropout's mask function at site sites[t] / threshold thresh[t].  These three
 * entry points regenerate the masks on the operand fragments, so the masked copies of the [M, H] input never exist in memory.
 * sites / thresh are HOST arrays of n_targets entries; r (LoRA rank) is 8 or 16, n_targets <= 4; all tensors bf16 except out of da.
 *   lora_a_drop : T[m, j]   = sum_h keep_{j / r}(m H + h) x[m, h] A[j, h]           A: [n_targets r, H] (caller folds 1 / (1 - p) in); T = out[:, 0 : n_targets r)
 *   lora_dx_drop: dx[m, h] += sum_t keep_t(m H + h) sum_{j in target t} dT[m, j] A[j, h]
 *   lora_da_drop: out[h, j] += sum_m row_scale[m] keep_{j / r}(m H + h) x[m, h] dT[m, j]   (fp32 [H, ldo], zero-initialised by the caller) */
int tcavp_lora_a_drop(const void* x, int ldx, const void* A, int lda, void* out, int ldo, long long M, int H, int r, int n_targets,
                      const uint32_t* seed, const uint32_t* sites, const uint32_t* thresh, tcavp_stream_t stream);
int tcavp_lora_dx_drop(const void* dT, int lddt, const void* A, int lda, void* dx, int lddx, long long M, int H, int r, int n_targets,
                       const uint32_t* seed, const uint32_t* sites, const uint32_t* thresh, tcavp_stream_t stream);
int tcavp_lora_da_drop(const void* x, int ldx, const void* dT, int lddt, const float* row_scale, float* out, int ldo, long long M, int H, int r,
                       int n_targets, const uint32_t* seed, const uint32_t* sites, const uint32_t* thresh, tcavp_stream_t stream);
/* Best-of-K candidate reduction (reference scripts/test.py:1336-1368): candidates (B, K, 2, T_out) fp32, y (B, 2, T_out), norm_stat (B, 4).
 * per_scene[b] = (min_k ADE, min_k FDE, min_k RMSE) after de-normalisation; totals[0..2] += their sums over the batch (caller zeroes). */
int tcavp_best_of_k(const float* candidates, const float* y, const float* norm_stat, float* per_scene, float* totals, int B, int K, int T_out,
                    tcavp_stream_t stream);

/* Weight gradient of a linear map (autograd of F.linear, reference loop im_kim_train_GRN.py:1039):
 * out[n][k] += sum_m dY[m][n] * X[m][k], out fp32 [N, ldo] (caller zero-initialises; M-slices are combined with atomics), dY / X in
 * their row-major [M, *] layouts (fp32 or bf16, may differ) — no transposed copies.  fp32 FFMA: meant for the narrow fp32 layers
 * (temporal encoder / decoder, fusion head, polygon input projection); wide bf16 layers go through tcavp_transpose + tcavp_gemm. */
int tcavp_dw(const void* dY, int lddy, int dy_dtype, const void* X, int ldx, int x_dtype, float* out, int ldo, long long M, int N, int K,
             tcavp_stream_t stream);
/* Backward of tcavp_attention (probabilities recomputed; any head_dim; Tk <= 768).  dq has the dtype/layout convention of q;
 * dk / dv are fp32 (caller zeroes them: the generic kernel accumulates with atomics because query blocks and GQA groups add
 * into the same keys).  When args->out / o_sb / o_st hold the FORWARD OUTPUT and the shape is bf16, H == Hkv, head_dim in
 * {16,32,64,96,128}, Tq, Tk <= 256, a tensor-core kernel (mma.sync, one CTA per (batch, head), no atomics) is used. */
int tcavp_attention_bwd(const tcavp_attn_args* args, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                        long long dq_st, float* dk, long long dk_sb, long long dk_st, float* dv, long long dv_sb, long long dv_st,
                        tcavp_stream_t stream);
/* Tensor-core-only form of tcavp_attention_bwd: the CTAs that own a key range sum its gradient over every query (and every query head
 * of a GQA group), so dk / dv are plain stores in `dkv_dtype` (TCAVP_BF16: straight into the packed d(qkv) activation buffer — no
 * fp32 staging, no zero-fill, no cast) with the same stride convention as k / v; no atomics, repeated calls give the same bits.
 * args->out must hold the forward output.  With args->lse holding the forward's logsumexp (tcavp_attention with lse set), bf16,
 * head_dim 64 / 128 and no dropout, any length and any H % Hkv == 0 is covered (key-blocked kernels; MHA at <= 256 positions keeps the
 * one-CTA-per-head kernel); without it H == Hkv and Tq, Tk <= 256.  Fails (TCAVP_ERR_ARG) on shapes the tensor-core kernels do not
 * cover; callers then use tcavp_attention_bwd. */
int tcavp_attention_bwd_owned(const tcavp_attn_args* args, const void* dout, long long do_sb, long long do_st, void* dq, long long dq_sb,
                              long long dq_st, void* dk, long long dk_sb, long long dk_st, void* dv, long long dv_sb, long long dv_st,
                              int dkv_dtype, tcavp_stream_t stream);
/* Stage-1 (CausalLM) objective on the labelled rows of a logits chunk — HF ForCausalLMLoss behind LlamaForCausalLM.forward(labels=...)
 * (HF:487-491; reference scripts/check_generation.py:131-151): fp32 logits [rows, V] (row stride ld), targets int64 [rows] (already
 * shifted, no -100 rows).  loss_sum[0] += sum_rows (logsumexp(row) - row[target]); when grad != NULL, grad[row, :] = (softmax(row) -
 * onehot(target)) * scale in grad_dtype (TCAVP_F32 / TCAVP_BF16; scale = incoming gradient / number of labelled positions). */
int tcavp_ce_loss(const float* logits, long long ld, const long long* targets, float* loss_sum, void* grad, long long ldg, int grad_dtype,
                  long long rows, int V, float scale, tcavp_stream_t stream);
/* Fused AdamW over flat fp32 buffers, torch.optim.AdamW semantics (im_kim_train_GRN.py:1008); grad_scale multiplies the
 * gradient first (1/world_size after a sum all-reduce). */
int tcavp_adamw(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1, float beta2,
                float eps, float weight_decay, int step, float grad_scale, tcavp_stream_t stream);

/* ---- gradient-norm clipping and non-finite step skipping, decided on the device (reference modify_scripts/modify_train.py:1190-1196:
 * a step whose loss is NaN is skipped, the gradient norm is clipped; scripts/modify_im_kim_train.py: clip_grad_norm_(…, 1.0) before
 * optimizer.step()) ------------------------------------------------------------------------------------------------------------------ */
typedef struct {
  float total_norm; /* L2 norm of grad_scale * grad before clipping: the value torch.nn.utils.clip_grad_norm_ returns */
  float clip_coef;  /* min(1, max_norm / (total_norm + 1e-6)) evaluated as torch does (NaN norm -> NaN); 1 when max_norm <= 0 */
  int skip;         /* skip_nonfinite && (total_norm or *loss is not finite) */
  int reserved;
} tcavp_clip_record;
#define TCAVP_CLIP_WORKSPACE_BYTES 9472 /* 1184 fp64 block partials, 8-byte aligned */
/* Writes *record for the flat fp32 gradient buffer grad[n].  The norm is accumulated deterministically (fixed partition, fp64 block
 * partials in `workspace`, fixed-order combine), so repeated calls and graph replays give the same bits.  Reads grad once.
 * max_norm <= 0: no clipping (clip_coef = 1).  loss (one fp32 device value) may be NULL. */
int tcavp_clip_prologue(const float* grad, long long n, float grad_scale, float max_norm, const float* loss, int skip_nonfinite,
                        void* workspace, long long workspace_bytes, tcavp_clip_record* record, tcavp_stream_t stream);
/* tcavp_adamw driven by a record of tcavp_clip_prologue and a device step counter.  record->skip set: param, exp_avg, exp_avg_sq and
 * *step are left untouched and *skipped (may be NULL) is incremented.  Otherwise the gradient is multiplied by
 * grad_scale * record->clip_coef, the bias corrections are those of tcavp_adamw for step = *step + 1, and *step is incremented. */
int tcavp_adamw_clipped(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1, float beta2,
                        float eps, float weight_decay, float grad_scale, const tcavp_clip_record* record, int* step, int* skipped,
                        tcavp_stream_t stream);
/* *dst = NaN when *loss is not finite.  Run on a gradient element before its all-reduce, it makes the global norm of every rank
 * non-finite, so every rank skips the step a non-finite loss on one rank asks to skip. */
int tcavp_mark_nonfinite(const float* loss, float* dst, tcavp_stream_t stream);

/* ---- dropout (train mode: lora_dropout train.py:432-440 -> peft lora.Linear; nn.Dropout of train.py:664-671, 745-750; the
 * dropout / dropout1 / dropout2 / dropout3 of torch's nn.TransformerEncoderLayer / DecoderLayer, train.py:358, 402-405) --------------
 * Counter-based mask, a pure function of (seed, site, element index) — nothing is stored, the backward pass regenerates it:
 *     mix(x)  : x ^= x >> 16; x *= 0x7feb352d; x ^= x >> 15; x *= 0x846ca68b; x ^= x >> 16          (32-bit)
 *     key     = mix(seed[0] ^ mix(site + 0x9E3779B9 * (seed[1] + 1)))
 *     u       = mix(idx_lo ^ key);  if idx_hi != 0: u = mix(u ^ idx_hi * 0x85EBCA6B)
 *     keep    = u >= thresh                         thresh = round(p * 2^32)
 * `seed` is a DEVICE pointer to two uint32 (base seed, step counter) so a captured CUDA graph draws fresh masks on every replay.
 *     out[r, c] = (accumulate ? out[r, c] : 0) + (residual ? residual[r, c] : 0) + (keep(r * cols + c) ? in[r, c] * scale : 0)
 * (scale = 1 / (1 - p) for the forward pass; the same call on a gradient is the backward pass).  in == out is allowed. */
int tcavp_dropout(const void* in, int ldi, int in_dtype, const void* residual, int ldr, int res_dtype, void* out, int ldo, int out_dtype,
                  long long rows, int cols, const uint32_t* seed, uint32_t site, uint32_t thresh, float scale, int accumulate,
                  tcavp_stream_t stream);

/* ---- text generation on the device (reference scripts/train.py:577-654 -> HF generate(do_sample=True, ...) with past_key_values) -------
 * Every entry point below reads the decode position from device memory, position = offset + *counter, and tcavp_sample_next advances
 * the counter itself: one decode iteration captured in a CUDA graph stays correct over any number of replays. */

/* One step of HF's logits-processor chain and the draw, one CTA per sequence.  logits fp32 [B, V] (row stride ld); work fp32 [B, V]
 * receives the processed logits (removed tokens -inf: what generate.py process_logits returns); hist int64 [B, ld_hist] holds the
 * prompt ids followed by the generated ones, n = hist_offset + state[0] of them valid.  In order:
 *   repetition penalty over hist[0, n) (once per distinct token: s < 0 ? s * penalty : s / penalty of the raw logit; 1 = off);
 *   no-repeat-n-gram (0 = off); do_sample: temperature, top-k (0 or >= V = off; values below the k-th largest removed, ties kept),
 *   top-p (outside (0, 1) = off; a token is kept when the mass strictly above it is < top_p, so a tie group at the boundary is kept
 *   whole; the largest is always kept);
 *   do_sample: inverse-CDF draw over the kept tokens in ascending token id with integer weights w_i = floor(exp(x_i - max) * 2^40):
 *     key = mix(seed[0] ^ mix(seed[1] + 0x9E3779B9)),  u = mix(mix(key ^ step) ^ (row * 0x85EBCA6B + 0x632BE5AB))   (mix: tcavp_dropout)
 *     r = floor(u * W / 2^32), W = sum w_i;  token = the first i with sum_{j <= i} w_j > r     (step = state[0], row = sequence index)
 *   else argmax of the processed logits, lowest index on ties.
 * eos_token_id >= 0: a row whose done[b] is set emits pad_token_id, a row that emits eos sets done[b].  The token goes to hist[b, n]
 * (when n < ld_hist) and tokens_out[b].  int state[3] = {step, 0, first step count at which every row was done (0 = not yet)}: the last
 * CTA increments state[0] and fills state[2]; state[1] is its arrival counter and must be 0 between launches. */
int tcavp_sample_next(const float* logits, long long ld, int B, int V, float* work, long long* hist, int ld_hist, int hist_offset, int* state,
                      const uint32_t* seed, int do_sample, float temperature, int top_k, float top_p, float repetition_penalty,
                      int no_repeat_ngram_size, long long eos_token_id, long long pad_token_id, int* done, long long* tokens_out,
                      tcavp_stream_t stream);

/* One query row per (sequence, head) over a KV cache filled up to position p - 1, p = offset + *counter: the new key / value rows
 * (k_new / v_new, the projection output of position p) are appended to the cache at p and the query attends over positions 0 .. p.
 * GQA (Hkv divides H), head_dim 32 / 64 / 128, TCAVP_F32 or TCAVP_BF16.  Keys are split over CTAs in chunks of 128 and the partials merged
 * by a second kernel (flash-decoding); fp32 SIMT arithmetic: a bandwidth-bound kernel, no tensor cores.  Strides in elements:
 * q / k_new / v_new / out rows of sequence b at b * q_sb / b * new_sb / b * o_sb, cache rows at b * cache_sb + t * cache_st, head h at
 * h * dh.  workspace: tcavp_decode_attention_workspace_bytes(B, H, dh, capacity) bytes of fp32 partials.  p >= capacity: no work. */
typedef struct {
  int B, H, Hkv, dh, capacity;
  const void* q; long long q_sb;
  const void* k_new; const void* v_new; long long new_sb;
  void* k_cache; void* v_cache; long long cache_sb, cache_st;
  void* out; long long o_sb;
  int dtype; float scale;
  const int* counter; int offset;
  float* workspace; long long workspace_bytes;
} tcavp_decode_attn_args;
long long tcavp_decode_attention_workspace_bytes(int B, int H, int dh, int capacity);
int tcavp_decode_attention(const tcavp_decode_attn_args* args, tcavp_stream_t stream);

/* The position-dependent gathers of a decode step, p = offset + *counter: out[b, 0:H] = embed[tokens[b]] (+ wpe[p] when wpe != NULL:
 * GPT-2) in `dtype` (row stride ldo), and, when rope_full != NULL, rope_out[0:dh] = row p of a tcavp_rope_table table of rope_L
 * positions (layout 0 or 1), i.e. the one-position table of the GEMM's fused RoPE epilogue. */
int tcavp_decode_embed(const long long* tokens, const void* embed, int vocab, const void* wpe, int n_pos, void* out, int ldo, int H, int dtype,
                       const float* rope_full, int rope_L, int dh, int rope_layout, float* rope_out, const int* counter, int offset, int B,
                       tcavp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TCAVP_H_ */
