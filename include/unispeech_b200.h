/*
 * unispeech_b200 -- C ABI of the B200-native WavLM / UniSpeech-SAT encoder hot path.
 *
 * Every entry point enqueues hand-written sm_100a kernels on the given CUDA stream and returns without
 * synchronising.  All pointers are DEVICE pointers owned by the caller (PyTorch tensors); the library never
 * allocates or frees caller memory on the hot path.  Return value: 0 on success, negative on error (message via
 * b200s_last_error(), thread-local).  There is no CPU fallback: on a device that is not compute capability 10.x
 * b200s_check_device() fails and so does every kernel launch.
 *
 * The reference (microsoft/UniSpeech) has no FFI for this path: it is plain PyTorch module code.  Each function
 * below cites the reference lines whose library calls (cuDNN conv, cuBLAS GEMM, F.multi_head_attention_forward,
 * F.layer_norm, F.group_norm, F.gelu, autograd) it replaces.  Paths are relative to /root/reference.
 * Conventions: activations bf16, accumulation fp32, parameters / gradients fp32 masters in the reference
 * state_dict layout.  "bs" = batch stride, "rs"/"ld" = row stride, always in ELEMENTS.  Gradient outputs marked
 * (+=) are accumulated with fp32 atomics: the caller zeroes them once per optimisation step.
 */
#ifndef UNISPEECH_B200_H_
#define UNISPEECH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* b200s_stream; /* cudaStream_t */

int b200s_version(void);
const char* b200s_last_error(void);
/* 0 if the current device can run the kernels (sm_100), negative otherwise */
int b200s_check_device(void);
/* number of kernels launched by this library so far (bench.py reports the per-step count) */
long long b200s_launch_count(void);
/* zero `bytes` bytes of device memory on the stream (cudaMemsetAsync): the per-step reset of the flat gradient buffer that the
 * backward kernels accumulate into (the reference's `optimizer.zero_grad()`, src/fairseq/trainer.py:627) */
int b200s_memset_zero(void* p, unsigned long long bytes, b200s_stream stream);

/* ---- fused GEMM epilogue description (all tensors optional) ------------------------------------------------
 * value = acc (+ bias[col]);  if gelu: out_pre <- value (gelu = 1) or gelu'(value) (gelu = 2) (optional), value = gelu_erf(value)
 *         if dgelu: value *= gelu'(gelu_aux[row,col]) (dgelu = 1) or gelu_aux[row,col] (dgelu = 2, aux written by a gelu = 2
 *         forward: the backward epilogue is then a plain multiply);  value += res1 + res2;  out <- value
 * colsum (fp32[N], +=) accumulates column sums of the stored values (bias gradients). */
typedef struct {
  const float* bias;
  const void* res1; long long res1_bs, res1_ld;
  const void* res2; long long res2_bs, res2_ld;
  const void* gelu_aux; long long aux_bs, aux_ld;
  void* out_pre; long long pre_bs, pre_ld;
  float* colsum;
  int gelu;
  int dgelu;
} b200s_epilogue;

/* ============================ tcgen05 GEMM family (csrc/gemm.cuh, gemm.cu) ============================ */

/* out[b, r, 0:N] = epilogue( A[b, r, 0:K] . W[N,K]^T ),  bf16 in / bf16 out, fp32 accumulate in TMEM.
 * A rows live at a + b*a_bs + r*a_rs and may OVERLAP (a_rs < K): this is how the strided Conv1d layers 1-6 of
 * ConvFeatureExtractionModel (WavLM/WavLM.py:400-403,485-504) and their input gradients become GEMMs on
 * channels-last [B,T,C] activations (row = k*C window, row stride = stride*C).  Also every nn.Linear forward /
 * input-gradient: q,k,v,out_proj (WavLM/modules.py:540-563), fc1/fc2 (WavLM/WavLM.py:706-739),
 * post_extract_proj (WavLM/WavLM.py:347-348).  K % 64 == 0, N % 8 == 0. */
int b200s_gemm_rows(const void* a, long long a_bs, long long a_rs, int rows, int batches, int K,
                    const void* w, int N, void* out, long long out_bs, long long out_ld,
                    const b200s_epilogue* epi, b200s_stream stream);

/* dW[n, k] (+=) sum_{b,r} Y[b,r,n] * X[b,r,k]   (fp32, row stride dw_ld): the weight gradient of the GEMMs above
 * (autograd of nn.Linear / nn.Conv1d).  Both operands are read MN-major by tcgen05.mma; X rows may overlap
 * (conv im2col view).  Split-K over (batch, row) blocks.  N % 8 == 0, K % 8 == 0. */
int b200s_gemm_wgrad(const void* y, long long y_bs, long long y_rs, const void* x, long long x_bs,
                     long long x_rs, int rows, int batches, int N, int K, float* dw, long long dw_ld,
                     b200s_stream stream);
/* Ragged batches (utterances of different lengths, zero-padded to the longest: BASELINE.json configs[4]).  Same contracts as
 * b200s_gemm_rows / b200s_gemm_wgrad with batches = utterances and rows = padded frames per utterance, plus a DEVICE int32 array
 * `valid[batches]` = frames of each utterance that hold real audio (padding is a suffix).  gemm_rows_ragged: an M tile that
 * starts at or beyond valid[b] is not computed; its output rows (and the saved pre-activation) are written as ZEROS (padded rows
 * must stay finite).  gemm_wgrad_ragged: 64-row blocks that start at or beyond valid[b] are neither loaded nor multiplied --
 * exact whenever the loss does not read padded frames (their gradient rows are then zero; the reference computes them anyway,
 * WavLM/WavLM.py:574-575 zeroes the inputs but every row-wise op still runs on them).  Small shapes that take the single-CTA
 * kernel ignore `valid` (they compute every row). */
int b200s_gemm_rows_ragged(const void* a, long long a_bs, long long a_rs, int rows, int batches, int K, const void* w, int N,
                           void* out, long long out_bs, long long out_ld, const b200s_epilogue* epi, const int* valid,
                           b200s_stream stream);
int b200s_gemm_wgrad_ragged(const void* y, long long y_bs, long long y_rs, const void* x, long long x_bs, long long x_rs,
                            int rows, int batches, int N, int K, float* dw, long long dw_ld, const int* valid,
                            b200s_stream stream);

/* Grouped positional convolution as an implicit GEMM (TransformerEncoder.pos_conv, WavLM/WavLM.py:514-527,577-579;
 * SamePad WavLM/modules.py:72-83), also used for its input gradient with flipped/transposed taps:
 *   out[b,t,g*Cg+n] = epilogue( sum_{j<taps} sum_{c<Cg} xpad[b, t+j, g*Cg+c] * wp[g*64+n, j*64+c] )
 * xpad: [B, Tpad, D] bf16 (row stride D) with zero rows around the T valid frames, pointer offset so that tap j of
 * output frame t reads row t+j;  wp: [G*64, taps*64] bf16 zero padded (b200s_posconv_prep). Cg = D/G <= 64. */
int b200s_posconv_gemm(const void* xpad, long long xpad_bs, int T, int B, int D, int G, int taps,
                       const void* wp, void* out, long long out_bs, long long out_ld,
                       const b200s_epilogue* epi, b200s_stream stream);

/* dwp[g, n, j, c] (+=) sum_{b,t} dy[b,t,g*Cg+n] * xpad[b,t+j,g*Cg+c];  dwp fp32 [G, Cg, taps, 64], only c < Cg is
 * meaningful. */
int b200s_posconv_wgrad(const void* dy, long long dy_bs, long long dy_rs, const void* xpad, long long xpad_bs,
                        int T, int B, int D, int G, int taps, float* dwp, b200s_stream stream);

/* ============================ attention (csrc/attn_fwd.cu, attn_bwd.cu) ============================ */

/* out[b,t,h*64+d] = sum_j softmax_j(scale q_i.k_j + gate[b,h,i]*tab[h,j-i+T-1], -inf at padded keys) v_j
 * Replaces compute_bias + gate multiply + F.multi_head_attention_forward (WavLM/modules.py:417-455,504-563); the
 * [B*H,T,T] bias is never materialised (it is Toeplitz).  qkv: bf16 [B,T,3D] fused projection output; gate: fp32
 * [B,H,T] or NULL (=1); tab: fp32 [H,2T-1] or NULL (no bias); key_pad: uint8 [B,T] or NULL; out: bf16 [B,T,D];
 * lse: fp32 [B,H,T] log2-domain log-sum-exp (saved for backward).  head_dim = 64; T <= b200s_attn_fwd_max_frames(tab != NULL)
 * (3072 with the bias, 16384 without): the kernel keeps the CTA's table slice and key mask in shared memory. */
int b200s_attn_fwd(const void* qkv, const float* gate, const float* tab, const uint8_t* key_pad, void* out,
                   float* lse, int B, int T, int H, float scale, b200s_stream stream);

/* Backward of b200s_attn_fwd (autograd of the same lines).  delta: fp32 [B,H,T] workspace; dqkv: bf16 [B,T,3D];
 * dgate: fp32 [B,H,T] (written); dtab: fp32 [H,2T-1] (+=, shared by all layers: WavLM/WavLM.py:549,594-599). */
int b200s_attn_bwd(const void* qkv, const void* out, const void* dout, const float* gate, const float* tab,
                   const uint8_t* key_pad, const float* lse, float* delta, void* dqkv, float* dgate, float* dtab,
                   int B, int T, int H, float scale, b200s_stream stream);

/* Same contract as b200s_attn_bwd, computed by ONE fused tensor-core kernel (csrc/attn_bwd2.cu: probabilities recomputed
 * once, dK/dV accumulated in TMEM, dQ reduced across key tiles in fp32).  dq_acc: fp32 [B,T,D] workspace that must be ZERO
 * on entry and is zero again on return.  T <= 2048. */
int b200s_attn_bwd_fused(const void* qkv, const void* out, const void* dout, const float* gate, const float* tab,
                         const uint8_t* key_pad, const float* lse, float* delta, float* dq_acc, void* dqkv,
                         float* dgate, float* dtab, int B, int T, int H, float scale, b200s_stream stream);

/* Attention with dropout on the probabilities (attention_dropout; the dropout_p argument of
 * F.multi_head_attention_forward, WavLM/modules.py:551): O = (softmax(..) o M) V / (1 - p).  M comes from the counter-based
 * hash of csrc/dropout.cuh keyed by (key0, key1, (b*H+h)*T + i, j); the forward kernel also records it as a bit mask
 * (drop_mask: b200s_attn_dropout_mask_words(B,T,H) uint32 words) which the fused backward re-reads, so the backward needs
 * no key.  drop_p = 0 is exactly b200s_attn_fwd / b200s_attn_bwd_fused (drop_mask may be NULL). */
int b200s_attn_fwd_dropout(const void* qkv, const float* gate, const float* tab, const uint8_t* key_pad, void* out,
                           float* lse, int B, int T, int H, float scale, float drop_p, uint32_t key0, uint32_t key1,
                           uint32_t* drop_mask, b200s_stream stream);
int b200s_attn_bwd_fused_dropout(const void* qkv, const void* out, const void* dout, const float* gate,
                                 const float* tab, const uint8_t* key_pad, const float* lse, float* delta,
                                 float* dq_acc, void* dqkv, float* dgate, float* dtab, int B, int T, int H, float scale,
                                 float drop_p, const uint32_t* drop_mask, b200s_stream stream);
long long b200s_attn_dropout_mask_words(int B, int T, int H);

/* Longest T that b200s_attn_fwd accepts, with (has_bias != 0) or without the relative-position table. */
int b200s_attn_fwd_max_frames(int has_bias);

/* ============================ long-utterance attention (csrc/attn_long.cu) ============================ */

/* Same inputs, outputs and numerics as b200s_attn_fwd (no dropout) for 1 <= T <= 16384, with shared memory that does not
 * depend on T.  tab is required.  tab_radius R (0 <= R <= T-1) promises tab[h, delta] = tab[h, +-R] for |delta| >= R (the
 * WavLM bucketing saturates beyond some distance); R = T-1 is exact for any table.  Key tiles whose every (query, key)
 * distance lies beyond R on one side use the per-row constant gate * tab[h, +-R] and skip the table.  head_dim = 64. */
int b200s_attn_fwd_long(const void* qkv, const float* gate, const float* tab, int tab_radius, const uint8_t* key_pad,
                        void* out, float* lse, int B, int T, int H, float scale, b200s_stream stream);

/* Backward of b200s_attn_fwd_long, same contract as b200s_attn_bwd for 1 <= T <= 16384 (tab = NULL: no bias, tab_radius
 * ignored).  dgate is written; dtab is += and shared by all layers.  With R < T-1 the gradient of every saturated diagonal
 * |delta| >= R is summed into dtab at delta = +-R and the entries beyond are left untouched: the bucket scatter
 * (b200s_relpos_table_bwd) then yields the same embedding gradient, since all those deltas share one bucket per side. */
int b200s_attn_bwd_long(const void* qkv, const void* out, const void* dout, const float* gate, const float* tab,
                        int tab_radius, const uint8_t* key_pad, const float* lse, float* delta, void* dqkv, float* dgate,
                        float* dtab, int B, int T, int H, float scale, b200s_stream stream);

/* SMs the persistent CTA-pair GEMM kernels leave free (0 = none, the default).  Data-parallel runs overlap the NCCL gradient exchange
 * with the backward pass; its CTAs (bounded by NCCL_MAX_CTAS) then find free SMs instead of displacing clusters of a grid that was
 * sized for the whole chip (legacy_distributed_data_parallel.py:76-165 runs the exchange strictly after backward, so the reference
 * has no counterpart). */
int b200s_reserve_sms(int sms);

/* ============================ row kernels (csrc/rowops.cu) ============================ */

/* y = LayerNorm(x) * gamma + beta [then exact GELU]; saves mean / rstd (fp32 [rows]).  nn.LayerNorm / Fp32LayerNorm
 * (WavLM/WavLM.py:342,559,666,675; WavLM/modules.py:30-42) and the LN+GELU of the layer_norm extractor
 * (WavLM/WavLM.py:409-419).  D in {64,128,256,512,768,1024}. */
int b200s_layer_norm_fwd(const void* x, long long x_bs, long long x_rs, const float* gamma, const float* beta,
                         void* y, long long y_bs, long long y_rs, float* mean, float* rstd, int rows_per_batch,
                         int batches, int D, int gelu, b200s_stream stream);

/* LayerNorm forward fused with the gru_rel_pos gate of the attention that consumes y (b200s_gate_fwd semantics on the stored
 * bf16 y): saves one pass over y per layer.  D = H * 64; gate: fp32 [B, H, T]; rows = B * T with the usual views. */
int b200s_layer_norm_gate_fwd(const void* x, long long x_bs, long long x_rs, const float* gamma, const float* beta,
                              void* y, long long y_bs, long long y_rs, float* mean, float* rstd, int T, int B, int D,
                              const float* grep_w, const float* grep_b, const float* grep_a, int H, float* gate,
                              b200s_stream stream);

/* dx = LN-backward(dy) [+ dres];  dgamma, dbeta (+=);  colsum (+=) = column sums of dx (bias gradient of x's producer). */
int b200s_layer_norm_bwd(const void* dy, long long dy_bs, long long dy_rs, const void* x, long long x_bs,
                         long long x_rs, const float* mean, const float* rstd, const float* gamma,
                         const float* beta, const void* dres, long long dres_bs, long long dres_rs, void* dx,
                         long long dx_bs, long long dx_rs, float* dgamma, float* dbeta, float* colsum,
                         int rows_per_batch, int batches, int D, int gelu, b200s_stream stream);

/* Ragged-batch forms of the row kernels (BASELINE configs[4]; the reference pads and computes every frame, WavLM.py:574-575).
 * valid[b] (int32, device): rows of batch b that hold real frames.  Rows at or beyond it are PADDING: the forward kernels write
 * zeros (mean = rstd = 0, gate = 1) without reading x, the backward kernels write a zero gradient row (nothing downstream of a
 * padded frame reaches the loss), the column sum skips them.  valid == NULL: identical to the plain entry point. */
int b200s_layer_norm_fwd_ragged(const void* x, long long x_bs, long long x_rs, const float* gamma, const float* beta,
                                void* y, long long y_bs, long long y_rs, float* mean, float* rstd, int rows_per_batch,
                                int batches, int D, int gelu, const int* valid, b200s_stream stream);
int b200s_layer_norm_gate_fwd_ragged(const void* x, long long x_bs, long long x_rs, const float* gamma, const float* beta,
                                     void* y, long long y_bs, long long y_rs, float* mean, float* rstd, int T, int B, int D,
                                     const float* grep_w, const float* grep_b, const float* grep_a, int H, float* gate,
                                     const int* valid, b200s_stream stream);
int b200s_layer_norm_bwd_ragged(const void* dy, long long dy_bs, long long dy_rs, const void* x, long long x_bs,
                                long long x_rs, const float* mean, const float* rstd, const float* gamma,
                                const float* beta, const void* dres, long long dres_bs, long long dres_rs, void* dx,
                                long long dx_bs, long long dx_rs, float* dgamma, float* dbeta, float* colsum,
                                int rows_per_batch, int batches, int D, int gelu, const int* valid, b200s_stream stream);
int b200s_colsum_ragged(const void* x, long long x_bs, long long x_rs, int rows_per_batch, int batches, int N, float* out,
                        const int* valid, b200s_stream stream);
int b200s_gate_bwd_ragged(const void* x, long long x_bs, long long x_rs, int T, int B, int H, const float* grep_w,
                          const float* grep_b, const float* grep_a, const float* dgate, void* dxg, long long dx_bs,
                          long long dx_rs, float* dgrep_w, float* dgrep_b, float* dgrep_a, const int* valid,
                          b200s_stream stream);

/* out[c] (+=) sum_rows x[r,c]  -- nn.Linear bias gradients */
int b200s_colsum(const void* x, long long x_bs, long long x_rs, int rows_per_batch, int batches, int N, float* out,
                 b200s_stream stream);

/* out = dy * gelu'(pre); colsum (+=) optional.  Backward of x + gelu(pos_conv(x)) (WavLM/WavLM.py:577-579) and of the
 * last conv layer's GELU. */
int b200s_dgelu_mul(const void* dy, long long dy_bs, long long dy_rs, const void* pre, long long pre_bs,
                    long long pre_rs, void* out, long long out_bs, long long out_rs, int rows_per_batch, int batches,
                    int N, float* colsum, b200s_stream stream);
/* Same; pre_is_grad != 0: `pre` already holds gelu'(pre-activation) (written by a gelu = 2 epilogue), out = dy * pre. */
int b200s_dgelu_mul_ex(const void* dy, long long dy_bs, long long dy_rs, const void* pre, long long pre_bs,
                       long long pre_rs, void* out, long long out_bs, long long out_rs, int rows_per_batch, int batches,
                       int N, float* colsum, int pre_is_grad, b200s_stream stream);

/* *out += sum of x^2 over a bf16 rows view (fp64 accumulator, caller zeroes it): numerator of the feature penalty
 * `features.float().pow(2).mean()` (src/fairseq/models/wavlm/wavlm.py:484).  N % 8 == 0. */
int b200s_sumsq_rows(const void* x, long long x_bs, long long x_rs, int rows_per_batch, int batches, int N, double* out,
                     b200s_stream stream);
/* Backward of GradMultiply.apply(features, scale) (WavLM/modules.py:60-69, WavLM/WavLM.py:333-336) fused with the gradient of
 * the feature penalty taken on its output (fairseq wavlm.py:477-484), in place on the bf16 gradient rows g:
 *   g <- scale * (g + (*pen_grad * pen_mul) * x);   pen_grad = DEVICE float (upstream gradient of the penalty scalar) or NULL. */
int b200s_grad_multiply(void* g, long long g_bs, long long g_rs, const void* x, long long x_bs, long long x_rs,
                        int rows_per_batch, int batches, int N, float scale, const float* pen_grad, float pen_mul,
                        b200s_stream stream);
/* y = [res +] dropout(x), y may alias x.  nn.Dropout / F.dropout of the transformer stack (WavLM/WavLM.py:350,584,659-661,
 * 702-738): keep(row, col) is a pure function of (key0, key1, logical row = b*rows_per_batch + r, col) (csrc/dropout.cuh),
 * kept values are scaled by 1/(1-p).  The backward pass is the same call on the incoming gradient with the same key and
 * res = NULL.  N % 8 == 0, 0 <= p < 1. */
int b200s_dropout_rows(const void* x, long long x_bs, long long x_rs, const void* res, long long res_bs,
                       long long res_rs, void* y, long long y_bs, long long y_rs, int rows_per_batch, int batches,
                       int N, float p, uint32_t key0, uint32_t key1, b200s_stream stream);

/* Host-side evaluation of the mask formulas (csrc/dropout.cuh), no device involved: bits word of counter `ctr`; per-row key
 * of the attention mask (which = 0 / 1 for key0 / key1); 16-bit keep threshold of probability p. */
uint32_t b200s_dropout_bits(uint32_t key0, uint32_t key1, uint32_t ctr);
uint32_t b200s_dropout_row_key(uint32_t key, uint32_t row, int which);
uint32_t b200s_dropout_threshold16(float p);

/* x[b,t,:] = mask_emb where mask[b,t]; = 0 where pad[b,t]   (apply_mask WavLM/WavLM.py:285-286; x[padding_mask]=0 :574-575) */
int b200s_frame_mask_fwd(void* x, long long x_bs, long long x_rs, int T, int B, int D, const uint8_t* mask,
                         const uint8_t* pad, const float* mask_emb, b200s_stream stream);
int b200s_frame_mask_bwd(void* dx, long long x_bs, long long x_rs, int T, int B, int D, const uint8_t* mask,
                         const uint8_t* pad, float* dmask_emb, b200s_stream stream);

/* gate[b,h,t] of gru_rel_pos from the RAW layer input (WavLM/modules.py:523-533) and its backward */
int b200s_gate_fwd(const void* x, long long x_bs, long long x_rs, int T, int B, int H, const float* grep_w,
                   const float* grep_b, const float* grep_a, float* gate, b200s_stream stream);
int b200s_gate_bwd(const void* x, long long x_bs, long long x_rs, int T, int B, int H, const float* grep_w,
                   const float* grep_b, const float* grep_a, const float* dgate, void* dxg, long long dx_bs,
                   long long dx_rs, float* dgrep_w, float* dgrep_b, float* dgrep_a, b200s_stream stream);

/* tab[h, i] = emb[lut[i], h]  (Toeplitz form of compute_bias, WavLM/modules.py:445-455) and the scatter-add backward */
int b200s_relpos_table_fwd(const float* emb, const int* lut, int n, int H, float* tab, b200s_stream stream);
int b200s_relpos_table_bwd(const float* dtab, const int* lut, int n, int H, float* demb, b200s_stream stream);

/* ============================ conv layer 0 (csrc/conv0.cu) ============================ */

/* Conv1d(1,C,k,stride s, no bias) + GroupNorm(C,C) (mode 0) or LayerNorm over channels (mode 1) + GELU on the raw
 * waveform (WavLM/WavLM.py:400-426).  wav fp32 [B,L]; w fp32 [C,1,k]; out bf16 channels-last.  stats: fp64 [B,C,2]
 * (mode 0);  fmean/frstd: fp32 [B,T] (mode 1).  C in {64, 512}. */
int b200s_conv0_fwd(const float* wav, long long L, int B, int T, int C, int k, int s, const float* w,
                    const float* gamma, const float* beta, int mode, double* stats, float* fmean, float* frstd,
                    void* out, long long out_bs, b200s_stream stream);
int b200s_conv0_bwd(const float* wav, long long L, int B, int T, int C, int k, int s, const float* w,
                    const float* gamma, const float* beta, int mode, const double* stats, float* bstats,
                    const float* fmean, const float* frstd, const void* da, long long da_bs, float* dw,
                    float* dgamma, float* dbeta, b200s_stream stream);
/* Same, with a bf16 workspace [B, ws_bs/C rows >= T, C] for the gradient w.r.t. the raw convolution output (mode 1 only; may
 * alias `da`, which is then consumed): the LayerNorm-mode backward becomes one pass over the frames plus one streaming
 * weight-gradient reduction instead of two full recomputing passes. */
int b200s_conv0_bwd_ws(const float* wav, long long L, int B, int T, int C, int k, int s, const float* w,
                       const float* gamma, const float* beta, int mode, const double* stats, float* bstats,
                       const float* fmean, const float* frstd, const void* da, long long da_bs, void* dconv_ws,
                       long long ws_bs, float* dw, float* dgamma, float* dbeta, b200s_stream stream);

/* ============================ parameter preparation (csrc/prep.cu) ============================ */

int b200s_scale_copy_f32(const float* src, float* dst, long long n, float scale, b200s_stream stream);
/* fp32 [N,K] -> bf16 dst[n*ld+k] and/or its transpose dstT[k*ldT+n] */
int b200s_prep_linear(const float* src, int N, int K, float scale, void* dst, long long ld, void* dstT,
                      long long ldT, b200s_stream stream);
/* all nn.Linear operands of the model in ONE launch: descs = device array of n_descs 56-byte records
 * {const float* src; bf16* dst; bf16* dstT; int64 ld, ldT; int32 N, K, tile_begin, tiles_k} (64x64 tiles: tiles_k = ceil(K/64),
 * tile_begin = prefix sum of ceil(N/64)*ceil(K/64)) */
int b200s_prep_linear_batched(const void* descs, int n_descs, int total_tiles, b200s_stream stream);
/* nn.Conv1d weight [Co,Ci,k] -> forward operand [Co, k*Ci] / per-phase input-gradient operand / gradient un-layout */
int b200s_prep_conv_fwd(const float* src, int Co, int Ci, int k, void* dst, b200s_stream stream);
int b200s_prep_conv_dgrad(const float* src, int Co, int Ci, int k, int s, int rho, void* dst, b200s_stream stream);
int b200s_unprep_conv_wgrad(const float* dwk, int Co, int Ci, int k, float* dw, b200s_stream stream);
/* weight_norm(dim=2) of pos_conv (WavLM/WavLM.py:526) -> padded per-group operands; and its backward.  Workspaces (8-byte aligned,
 * zeroed inside): norm2 = 2 * taps floats, work = 4 * taps floats -- the per-tap sums are accumulated in fp64 so that the norm, and
 * with it every bf16 pos_conv weight, is the same value on every run (the forward pass is bit-reproducible). */
int b200s_posconv_prep(const float* weight_v, const float* weight_g, int D, int G, int taps, float* norm2,
                       void* wp_fwd, void* wp_dgrad, b200s_stream stream);
int b200s_posconv_unprep(const float* weight_v, const float* weight_g, const float* dwp, int D, int G, int taps,
                         float* work, float* dweight_v, float* dweight_g, b200s_stream stream);

/* ============================ optimizer step on the flat gradient buffer (csrc/optim.cu) ============================ */

/* *out += sum_i g[i]^2 (fp64 accumulator on the device; the caller zeroes it).  With the flat gradient buffer this is the global
 * gradient norm of utils.clip_grad_norm_ (src/fairseq/utils.py:338-377) in one launch and without a host round trip. */
int b200s_sumsq_f32(const float* g, long long n, double* out, b200s_stream stream);

/* Same sum restricted to the tensors of an optimizer descriptor table (the layout b200s_adam_step takes): gradients of
 * parameters the optimizer does not own (excluded / frozen) are not counted -- fairseq's clip_grad_norm_ only sees
 * parameters whose .grad exists (src/fairseq/utils.py:338-345). */
int b200s_sumsq_table(const void* table, int n_tensors, long long total_chunks, const float* g, double* out,
                      b200s_stream stream);

/* Fused fairseq Adam update (src/fairseq/optim/adam.py:150-228) of n_tensors fp32 master tensors whose gradients (g) and
 * moments (m = exp_avg, v = exp_avg_sq) live in flat buffers:
 *   g' = g * grad_scale * clip,   clip = max_norm > 0 ? min(1, max_norm / (|grad_scale| * sqrt(*sumsq) + 1e-6)) : 1
 *        (multiply_grads + clip_grad_norm, src/fairseq/optim/fp16_optimizer.py:176-214, utils.py:378-381)
 *   m = beta1 m + (1-beta1) g';  v = beta2 v + (1-beta2) g'^2;  p -= weight_decay*lr*p;
 *   p -= lr*sqrt(1-beta2^step)/(1-beta1^step) * m / (sqrt(v) + eps);   g = 0 if zero_grad.
 * table: DEVICE array of n_tensors records {float* param; int64 goff; int64 numel; int64 chunk0} (32 bytes; goff = element
 * offset in g/m/v, multiple of 4; chunk0 = prefix sum of ceil(numel/2048)); total_chunks = sum of all chunks; step >= 1. */
int b200s_adam_step(const void* table, int n_tensors, long long total_chunks, float* g, float* m, float* v,
                    const double* sumsq, float grad_scale, float max_norm, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, int zero_grad, b200s_stream stream);

/* ============================ masked-prediction loss head (csrc/nce.cu) ============================ */
/* final_proj + cosine-similarity NCE logits + sum-reduced cross entropy of the pre-training models
 * (src/fairseq/models/wavlm/wavlm.py:426-438,525-576; src/fairseq/criterions/wavlm_criterion.py:63-87), built around the
 * tcgen05 GEMMs above: z[s,c] = cos(proj_s, E_c)/temp = (proj En^T)[s,c] / (|proj_s| temp), loss = w * sum_s CE(z[s,:], target_s)
 * (the reference's {positive} U {negatives != positive} softmax IS the softmax over the C classes). */

/* out[s,:] = x[idx[s],:]  (x[masked_indices], wavlm.py:541,558) and its autograd dx[idx[s],:] += src[s,:] (distinct rows) */
int b200s_gather_rows(const void* x, long long x_rs, const int* idx, int S, int D, void* out, long long out_rs,
                      b200s_stream stream);
int b200s_scatter_add_rows(const void* src, long long src_rs, const int* idx, int S, int D, void* dx, long long dx_rs,
                           b200s_stream stream);
/* en[c,:] = bf16(E_c / max(|E_c|,1e-8)) for c < C, zero rows up to Cpad; en_t = its transpose [Dp, Cpad]; invn[c] = 1/max(|E_c|,1e-8) */
int b200s_nce_prep(const float* label_embs, int C, int Cpad, int Dp, void* en, void* en_t, float* invn,
                   b200s_stream stream);
/* zraw = proj En^T (bf16 [S,Cpad], from b200s_gemm_rows).  Writes g[s,c] = weight (softmax(z)_c - [c==target_s]) / (|proj_s| temp)
 * (bf16 [S,Cpad], zero in the padded columns), pn[s] = 1/|proj_s|, rvec[s] = sum_c g[s,c] cos[s,c]; adds weight * sum_s CE to
 * *loss_sum (fp64) and the number of frames whose target has the largest logit to *correct (compute_correct,
 * wavlm_criterion.py:116-126; may be NULL). */
int b200s_nce_ce(const void* proj, long long proj_rs, int Dp, const void* zraw, long long z_rs, const int* target, int S,
                 int C, int Cpad, float logit_temp, float weight, void* g, long long g_rs, float* pn, float* rvec,
                 double* loss_sum, int* correct, b200s_stream stream);
/* dproj[s,:] -= rvec[s] * pn[s] * proj[s,:]   (dproj holds g En on entry: the gradient through 1/|proj_s|) */
int b200s_nce_dproj(void* dproj, long long d_rs, const void* proj, long long p_rs, int S, int Dp, const float* pn,
                    const float* rvec, b200s_stream stream);
/* d_label_embs[c,:] += (d_en_c - (d_en_c . En_c) En_c) / |E_c|,  d_en = g^T proj (fp32 [>=C, Dp], from b200s_gemm_wgrad) */
int b200s_nce_dlabel(const float* d_en, const float* label_embs, const float* invn, int C, int Dp, float* d_label_embs,
                     b200s_stream stream);

/* ============================ UniSpeech-SAT utterance-contrastive head (csrc/sat.cu) ============================ */
/* Utterance-contrastive loss of src/fairseq/models/unispeech_sat/unispeech_sat.py:699-758 (compute_pred_spk, compute_nce with
 * replace_inf=False :545-557, F.binary_cross_entropy_with_logits(...).mean() :736) without the [N+1, S, Dp] gathered instances:
 *   logit[s,0] = cos(proj_s, y_s)/temp, logit[s,1+n] = cos(proj_s, y[idx[n*S+s]])/temp; target[s,0] = 1, target[s,1+n] = same[n*S+s].
 * proj, y: bf16 [S, Dp] rows; idx: int32 [N, S] (host-drawn like sample_instances :487-543); same: uint8 [N, S].
 * Outputs: g fp32 [S, N+1] = d loss / d logit; *loss_sum (fp64, +=) the mean loss; stats[0] += #{(logit >= 0) == target},
 * stats[1] += #{target == 1} (contrastive_acc and mean_targets are these / (S (N+1))).  Dp % 4 == 0, Dp <= 1024. */
int b200s_sat_nce_fwd(const void* proj, long long proj_rs, const void* y, long long y_rs, const int* idx, const uint8_t* same,
                      int S, int N, int Dp, float logit_temp, float* g, double* loss_sum, int* stats, b200s_stream stream);
/* Backward: dproj_acc[s,:] += d loss/d proj_s, dy_acc[r,:] += d loss/d y_r (fp32 [S, Dp], vector reductions; pass the SAME buffer
 * for both when y IS proj, i.e. no quantizer); upstream = DEVICE float, the gradient of the loss scalar. */
/* wav2vec 2.0 InfoNCE (src/fairseq/models/wav2vec/wav2vec2.py:533-553 compute_preds; criterions/wav2vec_criterion.py:57-62,103-118) on
 * the same operands: logit[s,0] = cos(x_s, y_s)/temp, logit[s,1+n] = cos(x_s, y[idx[n*S+s]])/temp, a negative equal to the positive
 * is masked with -inf; *loss_sum += sum_s cross_entropy(logit[s,:], 0); g fp32 [S, N+1] = softmax - onehot(0) (consumed by
 * b200s_sat_nce_bwd); stats[0] += correct (argmax == 0, not also argmin == 0), stats[1] += S.  Dp % 4 == 0, Dp <= 1024. */
int b200s_w2v_nce_fwd(const void* proj, long long proj_rs, const void* y, long long y_rs, const int* idx, int S, int N, int Dp,
                      float logit_temp, float* g, double* loss_sum, int* stats, b200s_stream stream);
int b200s_sat_nce_bwd(const void* proj, long long proj_rs, const void* y, long long y_rs, const int* idx, int S, int N, int Dp,
                      float logit_temp, const float* g, const float* upstream, float* dproj_acc, float* dy_acc,
                      b200s_stream stream);
/* dst (bf16 rows) = src (fp32 rows); N and the row strides multiples of 4 elements */
int b200s_f32_to_bf16_rows(const float* src, long long src_rs, void* dst, long long dst_rs, long long rows, int N,
                           b200s_stream stream);
/* GumbelVectorQuantizer.forward with hard codes (src/fairseq/modules/gumbel_vector_quantizer.py:141-201; time_first,
 * combine_groups = False): logits bf16 [S, G*V] = weight_proj(x); codes[s*G+g] = argmax_v logits (eval) or argmax_v (logits +
 * Gumbel noise from the counter hash with (key0, key1)) (training: the hard sample of F.gumbel_softmax);
 * q[s, g*dv ..] = vars[g*V + code, :] (bf16; vars fp32 [G*V, dv]); counts[g*V+v] += [v == argmax of the NOISE-FREE logits], probs[g*V+v] += softmax(logits)_v
 * (fp32, the caller zeroes them: hard_probs / avg_probs of :152-170 are these / S). */
int b200s_vq_hard(const void* logits, long long logits_rs, const float* vars, int S, int G, int V, int dv, int* codes, void* q,
                  long long q_rs, float* counts, float* probs, int gumbel, uint32_t key0, uint32_t key1, b200s_stream stream);
/* d loss / d logits (bf16 [S, G*V], fully written) = p (c - <c, p>) / S  [c: fp32 [G*V] = d loss / d avg_probs, or NULL]
 *   + ys (h - <h, ys>) / tau  [h: bf16 [S, G*V] = dq . vars^T, or NULL: straight-through gradient of F.gumbel_softmax(hard=True),
 *     ys = softmax((logits + the same noise) / tau)]. */
int b200s_vq_logits_bwd(const void* logits, long long logits_rs, int S, int G, int V, const float* c, const void* h, long long h_rs,
                        float tau, uint32_t key0, uint32_t key1, void* dlogits, long long dlogits_rs, b200s_stream stream);
/* dvars[g*V + codes[s*G+g], :] += dq[s, g*dv ..]   (backward of the codebook lookup) */
int b200s_vq_dvars(const void* dq, long long dq_rs, const int* codes, int S, int G, int V, int dv, float* dvars,
                   b200s_stream stream);

/* ============================ on-device data path (csrc/datapath.cu) ============================ */
/* Span masking of compute_mask_indices (WavLM/WavLM.py:35-159; static span length, overlapping spans) on the device, with the
 * library's counter-based RNG instead of numpy's (statistical parity): per row count = max(min_masks, floor(mask_prob sz / L + u)),
 * `count` distinct uniform starts in [0, sz - L), union of the spans, every row trimmed to the batch-minimum number of masked
 * frames.  valid_len: int32 [B] unpadded frames per row, or NULL (all T).  mask: uint8 [B, T] out; counts: int32 [B] workspace.
 * T <= 4096. */
int b200s_span_mask(const int* valid_len, int B, int T, float mask_prob, int mask_length, int min_masks, uint32_t key0,
                    uint32_t key1, uint8_t* mask, int* counts, b200s_stream stream);
/* power[b] += sum_t x[b,t]^2 (fp32 waveforms [B, L], batch stride x_bs; fp64 accumulators zeroed by the caller) */
int b200s_row_power(const float* x, long long x_bs, int B, int L, double* power, b200s_stream stream);
/* Utterance mixing (src/fairseq/data/audio/utterance_mixing_dataset.py:415-432): plan = DEVICE array of B records
 * {int32 c (-1: not mixed), int32 len, int32 c_start, int32 s_start, float snr_db} drawn by the caller;
 * dst[b, s_start + t] += src[c, c_start + t] * sqrt(P_b / (P_c 10^(snr/10))), P = power / L (from b200s_row_power of src). */
int b200s_mix_apply(const float* src, long long bs, int B, int L, const void* plan, const double* power, float* dst,
                    b200s_stream stream);
/* x[b, :n_b] = (x - mean) / sqrt(var + 1e-5) over the row's n_b = valid_len[b] (or L) samples (F.layer_norm(wav, wav.shape),
 * utterance_mixing_dataset.py:433-435,571-573); stats: fp64 [B, 2] zeroed by the caller; plan != NULL: only rows with c >= 0. */
int b200s_row_normalize(float* x, long long bs, int B, int L, const int* valid_len, double* stats, const void* plan,
                        b200s_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* UNISPEECH_B200_H_ */
