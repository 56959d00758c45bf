/*
 * tinyrec.h -- C ABI of libtinyrec.so: the B200 (sm_100a) kernels behind the
 * Tiny-NewsRec training / scoring hot path.
 *
 * The reference (yflyl613/Tiny-NewsRec) is pure Python/PyTorch and has no FFI or
 * operator registry: its boundary for this path is the nn.Module API consumed by
 * Tiny-NewsRec/run.py (SURVEY.md section 8b).  Each entry point below therefore cites the
 * reference *torch call site* it replaces (paths relative to /root/reference).
 * The Python modules in tiny-newsrec_b200/ keep the reference signatures and bind
 * these functions with ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named h_*; the caller owns all
 *     memory (kernels never allocate or free device memory);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no
 *     device synchronisation inside;
 *   - return 0 on success, non-zero on error; `tnr_last_error()` returns a
 *     thread-local message.  There is no CPU fallback and no other backend: a
 *     device that is not sm_100 is an error;
 *   - "bf16" buffers are raw uint16 bfloat16, row-major; `ld*` are leading
 *     dimensions in ELEMENTS.
 */
#ifndef TINYREC_H_
#define TINYREC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TNR_ABI_VERSION 6

const char* tnr_last_error(void);
int tnr_abi_version(void);
/* Fails unless the current device is compute capability 10.x. Returns SM count in *num_sms. */
int tnr_device_check(int* num_sms);
/* Leave `n_sms` SMs of the current device out of the persistent GEMM grids launched from now on (0 = use all).
 * Data-parallel training sets it while gradient all-reduces are in flight (the replacement of Horovod's background
 * exchange, Tiny-NewsRec/run.py:144-149): a persistent one-CTA-per-SM GEMM whose grid covers every SM makes the
 * collective's CTAs wait for a whole GEMM, and the GEMM CTAs displaced by them then run as a second wave. */
int tnr_set_sm_reserve(int n_sms);
/* Host staging copy of the loaders: dst (pinned) <- src (pageable), split over up to n_threads host threads (1..16).
 * No CUDA call inside.  The job of the reference loader's producer thread (Tiny-NewsRec/dataloader.py:303-314). */
int tnr_host_copy_mt(void* dst, const void* src, long long bytes, int n_threads);

/* ------------------------------------------------------------------ dropout */
/* Training-mode dropout (the reference trains with dropout 0.1 active: run.py never calls
 * model.eval() in train(), SURVEY.md section 3.1).  Masks are counter-based (Philox4x32-7 keyed by
 * *seed, per-tensor `site`, element index) so the backward regenerates them instead of storing
 * them; oracle/dropout.py restates the generator bit-for-bit.  `seed` is a DEVICE pointer so a
 * captured CUDA graph replays with a fresh seed.  NULL struct, NULL seed or p <= 0 disables. */
typedef struct {
  const unsigned long long* seed;
  unsigned int site;
  float p;
} tnr_dropout;

/* keep[i] = 1/0 for the first n elements of dropout tensor `site` (linear element index; tests). */
int tnr_dropout_mask(const tnr_dropout* drop, long long n, unsigned char* keep, void* stream);

/* ------------------------------------------------------------------ GEMM */
enum { TNR_ACT_NONE = 0, TNR_ACT_GELU = 1, TNR_ACT_TANH = 2, TNR_ACT_DGELU = 3,
       TNR_ACT_GELU_DAUX = 4,   /* C = gelu(z), aux <- gelu'(z) (instead of z): what the FFN1 forward of a trained layer uses */
       TNR_ACT_MULAUX = 5 };    /* C = acc * aux: the matching dgrad epilogue (dz = (dy W2) * gelu'(z)) */
enum { TNR_BF16 = 0, TNR_F32 = 1 };

/* C[M,N] = epilogue( A[M,K] . B[N,K]^T )       bf16 operands, fp32 accumulate in TMEM
 * (tcgen05.mma kind::f16, TMA-fed, warp-specialised persistent kernel).
 *   a_mn_major = 0: A memory is [M,K] row-major (lda >= K).
 *   a_mn_major = 1: A memory is [K,M] row-major (lda >= M)  -- A used transposed (wgrad).
 *   b_mn_major = 0: B memory is [N,K] row-major (nn.Linear weight [out,in]).
 *   b_mn_major = 1: B memory is [K,N] row-major (dgrad through weight; wgrad activations).
 * epilogue:  v = acc (+ bias[n]);  GELU: (aux <- bf16(v) if aux) v = gelu_erf(v);
 *            TANH: v = tanh(v);  DGELU: v *= gelu_erf'(aux[m,n]);  v = dropout(v);  v += residual[m,n];
 *            c_dtype bf16 | f32;  split_k > 1 or accumulate: fp32 atomic add into C.
 * Replaces torch nn.Linear call sites: tnlrv3/modeling.py:236-248 (QKV), transformers
 * BertSelfOutput/BertIntermediate/BertOutput dense (used at modeling.py:287,305-306),
 * model_bert.py:24 (att_fc1), :136 (dense) and their autograd backward. */
typedef struct {
  int M, N, K;
  const void* A; int lda; int a_mn_major;
  const void* B; int ldb; int b_mn_major;
  void* C; int ldc; int c_dtype;
  const float* bias;
  const void* residual; int ldr;
  int act;
  void* aux; int ldaux;
  int split_k;
  int accumulate;
  const tnr_dropout* drop;   /* v = dropout(acc + bias) before the residual add; NULL = off (plain epilogue only) */
  float* colsum;             /* if != NULL (bf16 output only): colsum[n] += sum_m C[m,n] of the rounded bf16 output --
                                the bias gradient of the layer in front (fp32 atomics), fused into the dgrad epilogue */
} tnr_gemm_args;
int tnr_gemm_bf16(const tnr_gemm_args* args, void* stream);

/* ------------------------------------------------- encoder row kernels (HBM-bound) */
/* out[t,:] = LayerNorm_eps( word[ids[t]] + pos[t % L] + type0 )  ->  bf16 [n_rows*L, E].
 * ids: int64, row r at ids + r*ids_ld (the reference packs ids|mask as x[n, 2L]).
 * word_dtype: TNR_BF16 or TNR_F32 table [vocab, E]; pos fp32 [>=L, E]; type0 fp32 [E].
 * Replaces BertEmbeddings.forward, tnlrv3/modeling.py:153-178 (dropout :177 applied when `drop` is given). */
int tnr_embed_ln_fwd(const int64_t* ids, int ids_ld, int n_rows, int L, int vocab, const void* word,
                     int word_dtype, const float* pos, const float* type0, const float* gamma,
                     const float* beta, float eps, int E, void* out_bf16, const tnr_dropout* drop,
                     void* stream);

/* y = LayerNorm(x) over rows of a bf16 [rows, E] buffer (the "dense + bias + residual" sum the
 * GEMM epilogue wrote).  Replaces the LayerNorm of transformers BertSelfOutput / BertOutput
 * (imported at tnlrv3/modeling.py:12-14, used at :287 and :306). */
int tnr_layernorm_fwd(const void* x_bf16, int rows, int E, const float* gamma, const float* beta,
                      float eps, void* y_bf16, void* stream);
/* dx = dLN(dy; x) ; dgamma += , dbeta += (fp32, caller zero-initialises).  autograd of the above.
 * If dx_drop_bf16 != NULL it receives dx * keep / (1-p) for dropout tensor `drop` -- the gradient
 * w.r.t. the dense output that was dropped out before the residual add (dx itself is the residual
 * branch); with drop disabled it is a plain copy of dx.  If dsum != NULL, dsum[c] += sum_r
 * (dropout-masked) dx[r,c]: the bias gradient of that dense layer, fused here. */
int tnr_layernorm_bwd(const void* dy_bf16, const void* x_bf16, int rows, int E, const float* gamma,
                      float eps, void* dx_bf16, float* dgamma, float* dbeta, void* dx_drop_bf16,
                      float* dsum, const tnr_dropout* drop, void* stream);
/* out[c] += sum_r x[r,c]  (bias gradients of nn.Linear). */
int tnr_colsum_bf16(const void* x_bf16, int rows, int cols, int ld, float* out, void* stream);

/* ------------------------------------------------------------ fused attention */
/* ctx = dropout(softmax(Q K^T / 8 + (1-mask)*-10000 + relbias[h][j-i])) V, head dim 64, 1 <= L <= 512.
 * qkv bf16 [n*L, 3E] (Q | K | V), mask int64 (row r at mask + r*mask_ld, 1 = attend), ctx bf16 [n*L, E].
 * relbias fp32 [A, 2L-1]: bias of key j for query i at index (j - i) + L - 1.  The reference builds a
 * [n, A, L, L] bias per forward from one-hot buckets (tnlrv3/modeling.py:458-463); position_ids are always
 * arange(L) (:162-163), so it is batch-invariant and a function of j - i only.
 * L <= 32: one warp per (news, head); L > 32: streamed-KV online-softmax kernel (attention_long.cu).
 * `drop` applies dropout to the probabilities (:223).
 * Replaces BertSelfAttention.multi_head_attention, tnlrv3/modeling.py:205-231. */
int tnr_attn_relpos_fwd(const void* qkv_bf16, const int64_t* mask, int mask_ld, const float* relbias,
                        void* ctx_bf16, int n_news, int L, int A, int E, const tnr_dropout* drop,
                        void* stream);
/* dqkv bf16 [n*L, 3E] from dctx (probabilities recomputed, dropout mask regenerated).
 * L <= 32: one warp per (news, head), workspace unused (may be NULL).  32 < L <= 512: two streamed kernels
 * (dQ with its own online softmax statistics, then dK / dV per key block) that need `workspace`:
 * 2 * n_news * A * L floats (row log-sum-exp and delta_i = sum_j P_ij dP_ij).
 * If dbias_qkv != NULL: dbias_qkv[3E] += column sums of dqkv (the fused [bq|bk|bv] gradient, fp32 atomics). */
int tnr_attn_relpos_bwd(const void* qkv_bf16, const int64_t* mask, int mask_ld, const float* relbias,
                        const void* dctx_bf16, void* dqkv_bf16, float* dbias_qkv, float* workspace, int n_news,
                        int L, int A, int E, const tnr_dropout* drop, void* stream);

/* ------------------------------------------------- fp32 inference path of the news encoder */
/* The 1e-4 parity mode of NewsEncoder (args.precision = 'fp32'): fp32 activations end to end, no dropout (inference
 * only).  Each GEMM is tnr_gemm_bf16 with K' = 3K over operands split by tnr_split_bf16x3: A' = [A_hi | A_lo | A_hi],
 * B' = [W_hi | W_hi | W_lo], so A' B'^T = A_hi W_hi + A_lo W_hi + A_hi W_lo (about 5e-6 relative instead of bf16's
 * 2.6e-3), written as fp32 C with the bias epilogue.  All buffers below are fp32 unless named otherwise. */
enum { TNR_SPLIT_ACT = 0,        /* [hi | lo | hi] */
       TNR_SPLIT_WEIGHT = 1 };   /* [hi | hi | lo] */
/* out bf16 [rows, 3K] (row stride 3K) from x [rows, K] (row stride ldx): hi = bf16_rn(v), lo = bf16_rn(v - hi) with
 * v = x, or v = gelu_erf(x) = 0.5 x erfc(-x / sqrt 2) (fp32 erfcf, a few ulps) when gelu != 0 (the FFN2 input). */
int tnr_split_bf16x3(const float* x, int rows, int K, int ldx, int layout, int gelu, void* out_bf16, void* stream);
/* out[n*L, E] = LayerNorm_eps(word[ids[t]] + pos[t % L] + type0) from the fp32 word table (gathered bit-exactly; ids
 * outside [0, vocab) are clamped as in tnr_embed_ln_fwd); two-pass statistics. */
int tnr_embed_ln_fwd_f32(const int64_t* ids, int ids_ld, int n_rows, int L, int vocab, const float* word,
                         const float* pos, const float* type0, const float* gamma, const float* beta, float eps, int E,
                         float* out, void* stream);
/* y = LayerNorm(x + residual), [rows, E] (the residual add of BertSelfOutput / BertOutput, modeling.py:287,306). */
int tnr_add_layernorm_f32(const float* x, const float* residual, int rows, int E, const float* gamma,
                          const float* beta, float eps, float* y, void* stream);
/* ctx [n*L, E] = softmax(Q K^T / 8 + (1-mask)*-10000 + relbias[h][j-i]) V from qkv [n*L, 3E]; mask and relbias as in
 * tnr_attn_relpos_fwd.  Head dim 64, 1 <= L <= 512, n_news <= 65535.  Fully padded rows get the reference's softmax
 * over the shifted scores. */
int tnr_attn_relpos_fwd_f32(const float* qkv, const int64_t* mask, int mask_ld, const float* relbias, float* ctx,
                            int n_news, int L, int A, int E, void* stream);
/* Word pooling from the fc1 pre-activation u [n*S, ldq] (bias included): a = exp(tanh(u) . w2 + b2) / (sum + 1e-8)
 * (no max subtraction, as the reference), out [n, C] = sum_s a_s x[n, s, :]; x [n*S, C]. */
int tnr_attnpool_fwd_f32(const float* x, const float* u, int ldq, int Q, const float* w2, const float* b2, float* out,
                         int n, int S, int C, void* stream);

/* ------------------------------------------------------- additive attention pooling (words) */
/* a = normalise(exp(e.w2 + b2) [* mask]);  out[n,:] = sum_s a[n,s] x[n,s,:]
 * x bf16 [n,S,C]; e = tanh(fc1 x) bf16 [n*S, ldq] (from tnr_gemm_bf16 with TNR_ACT_TANH);
 * mask fp32 [n,S] or NULL; out bf16 [n,C]; a_out fp32 [n,S] (saved for backward).
 * Replaces AttentionPooling.forward, Tiny-NewsRec/model_bert.py:15-34 (word level, :133). */
int tnr_attnpool_fwd(const void* x_bf16, const void* e_bf16, int ldq, int Q, const float* w2,
                     const float* b2, const float* mask, void* out_bf16, float* a_out, int n, int S,
                     int C, void* stream);
/* dout fp32 [n,C] -> dx_direct bf16 [n,S,C] (= a*dout), du bf16 [n*S, ldq] (grad at fc1
 * pre-activation), dw2 += [Q], db2 += [1]. */
int tnr_attnpool_bwd(const void* x_bf16, const void* e_bf16, int ldq, int Q, const float* w2,
                     const float* a_in, const float* dout, void* dx_bf16, void* du_bf16, float* dw2,
                     float* db2, int n, int S, int C, void* stream);

/* ------------------------------------------------- user encoder / scoring / KD loss (fp32) */
/* Additive-attention user encoder, NAML branch.  vecs fp32 [B,H,D], mask fp32 [B,H].
 *   use_mask = 0 (args.user_log_mask False): v = vec*m + pad_doc*(1-m), unmasked pooling
 *   use_mask = 1: masked pooling (alpha *= m).  All-masked history -> exactly 0.
 * user fp32 [B,D]; a_out [B,H] normalised weights; e_out [B,H,Q] tanh activations (or NULL).
 * 1 <= H <= 512 (user_log_length): H <= 64 is one 64-row tile per impression; longer histories walk the rows in
 * 64-row chunks and normalise once over all H.  The same holds for _multi, _gather, _score and _bwd.
 * Replaces UserEncoder.forward, Tiny-NewsRec/model_bert.py:155-176 (+ AttentionPooling :15-34). */
int tnr_user_encoder_fwd(const float* vecs, const float* mask, const float* pad_doc, const float* W1,
                         const float* b1, const float* w2, const float* b2, int use_mask, float* user,
                         float* a_out, float* e_out, int B, int H, int D, int Q, void* stream);
/* The same for n_enc (<= 9) encoders sharing `mask` in ONE launch (grid B x n_enc): the student
 * user encoder and the M teacher user encoders of Model.forward (model_bert.py:269,281). */
typedef struct {
  const float *vecs, *pad_doc, *W1, *b1, *w2, *b2;
  float *user, *a_out, *e_out;
} tnr_user_encoder_io;
int tnr_user_encoder_fwd_multi(const tnr_user_encoder_io* enc, int n_enc, const float* mask, int use_mask,
                               int B, int H, int D, int Q, void* stream);
/* One encoder with the history rows gathered inside the kernel: vecs[b,h] = table[idx[b,h]] (idx int32 [B,H];
 * ids outside [0, n_rows) read row 0 like the loader, dataloader.py:74).  Fuses news_scoring[log_ids] with
 * the user encoder of the scoring loop (Tiny-NewsRec/run.py:340-343, dataloader.py:292-301): the
 * [B,H,D] gathered copy is never written.  a_out may be NULL. */
int tnr_user_encoder_fwd_gather(const float* table, long long n_rows, const int32_t* idx, const float* mask,
                                const float* pad_doc, const float* W1, const float* b1, const float* w2,
                                const float* b2, int use_mask, float* user, float* a_out, int B, int H, int D,
                                int Q, void* stream);
/* fp32 inference mode (args.precision = 'fp32') of tnr_user_encoder_fwd / _gather: same arguments and checks, the
 * fc1 contraction as 3xTF32 (hi = tf32_rn(x), lo = x - hi for both operands; lo_a hi_b + hi_a lo_b + hi_a hi_b, three
 * mma.sync per product) over the unrounded fp32 rows, tanhf / expf in the epilogue: fp32 accuracy (~1e-6 relative)
 * where the TF32 forms give ~1e-4 and more with sharp attention logits.  Forward only. */
int tnr_user_encoder_fwd_f32(const float* vecs, const float* mask, const float* pad_doc, const float* W1,
                             const float* b1, const float* w2, const float* b2, int use_mask, float* user,
                             float* a_out, float* e_out, int B, int H, int D, int Q, void* stream);
int tnr_user_encoder_fwd_gather_f32(const float* table, long long n_rows, const int32_t* idx, const float* mask,
                                    const float* pad_doc, const float* W1, const float* b1, const float* w2,
                                    const float* b2, int use_mask, float* user, float* a_out, int B, int H, int D,
                                    int Q, void* stream);
/* Scoring path of the same encoder for thousands of impressions per launch (the eval loop, run.py:335-361):
 * the fc1 contraction runs as ONE flat TF32 GEMM over the history rows with mask != 0 on the tcgen05 tensor cores
 * (kind::tf32, CTA pairs, 256-row tiles, W1 resident in the pair's shared memory, rows gathered by index from the
 * table) that emits the logits, then a warp per impression normalises and pools.  `w1_packed`:
 * tnr_user_encoder_packed_w1_floats(D) floats filled by tnr_user_encoder_pack_w1 from att_fc1.weight / .bias,
 * att_fc2.weight and pad_doc (re-pack when any of them changes): the swizzled TF32 image of W1, W1 pad_doc and the
 * logit of a pad_doc row.  idx NULL: vecs is [B*H, D]; else vecs is the [n_rows, D] table and idx int32 [B,H]
 * (unknown ids read row 0).  a_out [B,H] is required (it holds the logits between the two kernels).
 * D % 32 == 0, D <= 256, Q <= 208, H <= 512. */
long long tnr_user_encoder_packed_w1_floats(int D);
int tnr_user_encoder_pack_w1(const float* W1, const float* pad_doc, const float* b1, const float* w2, float* packed,
                             int D, int Q, void* stream);
long long tnr_user_encoder_score_ws_bytes(int B, int H);
int tnr_user_encoder_score(const float* vecs, long long n_rows, const int32_t* idx, const float* mask,
                           const float* pad_doc, const float* w1_packed, const float* b1, const float* w2,
                           const float* b2, int use_mask, float* user, float* a_out, void* workspace, int B,
                           int H, int D, int Q, void* stream);
/* d_user [B,D] -> d_vecs += [B*H, D]; dpad/dW1/db1/dw2/db2 += (fp32 atomics).
 * scratch: fp32 [B*H*(Q+D)] workspace (grad at the fc1 pre-activation + blended inputs; dW1 is then
 * one TN GEMM over all impressions). */
int tnr_user_encoder_bwd(const float* vecs, const float* mask, const float* pad_doc, const float* W1,
                         const float* w2, int use_mask, const float* a_in, const float* e_in,
                         const float* d_user, float* d_vecs, float* dpad, float* dW1, float* db1,
                         float* dw2, float* db2, float* scratch, int B, int H, int D, int Q, void* stream);

/* Click score + CE + multi-teacher KD loss and its gradients in one pass.
 * Row layout of the [R, D] news matrices: history block (b,h) -> b*H+h, then candidate block
 * (b,k) -> B*H + b*K + k; teacher matrices T_ext / TP_ext / G_ext are [M, B*(H+K)+B, D] with the
 * B per-impression user rows appended (raw / projected by transform_matrix / gradient).
 * losses: fp32 [4 + 4B + 1], zero-initialised ONCE by the caller: [0..3] = {distill, emb, target, total}
 * batch means (assigned; summed in impression order, so bit-reproducible), [4 + 4b ..] per-impression
 * terms, last word a ticket counter the kernel resets.  score_out [B,K];
 * if want_grad: d_news [R,D] (assigned), d_user [B,D], G_ext (grad w.r.t. TP_ext).
 * M == 0 gives the PLM-NR loss (CE only, coef scales it).
 * Replaces Model.forward, Tiny-NewsRec/model_bert.py:262-306 (+ kd_ce_loss :208-219,
 * hid_mse_loss :222-244, score :204) and its autograd backward. */
int tnr_kd_loss_fwdbwd(const float* s_news, const float* s_user, const int64_t* label,
                       const float* T_ext, const float* TP_ext, int M, int B, int H, int K, int D,
                       float temperature, float coef, int want_grad, float* score_out, float* losses,
                       float* d_news, float* d_user, float* G_ext, void* stream);

/* Small batched fp32 GEMMs (TF32 mma.sync, fp32 accumulate) for transform_matrix (model_bert.py:277-278,283):
 *   nt:     C[b][M,N]  = A[b][M,K] . B[b][N,K]^T + bias[b][N]
 *   tn_acc: C[b][N1,N2] += A[b][R,N1]^T . B[b][R,N2];  cbias[b][N1] += colsum(A[b])   */
int tnr_sgemm_nt(const float* A, const float* B, const float* bias, float* C, int M, int N, int K,
                 int batch, long long sA, long long sB, long long sbias, long long sC, void* stream);
/* tnr_sgemm_nt to fp32 accuracy (3xTF32, as tnr_user_encoder_fwd_f32): the NRMS Q/K/V projections of the fp32
 * inference mode. */
int tnr_sgemm_nt_f32(const float* A, const float* B, const float* bias, float* C, int M, int N, int K,
                     int batch, long long sA, long long sB, long long sbias, long long sC, void* stream);
int tnr_sgemm_tn_acc(const float* A, const float* B, float* C, float* cbias, int R, int N1, int N2,
                     int batch, long long sA, long long sB, long long sC, long long sbias, void* stream);

/* ------------------------------------------------- NRMS user encoder (multi-head self-attention) */
/* The self-attention in front of the additive pooling when args.model == 'NRMS'
 * (Tiny-NewsRec/model_bert.py:37-100; wired in at :145-148,:162-164,:171-173).  d_k = d_v = 16 (:146).
 *   blend_fwd:  out = vecs * m + pad_doc * (1 - m)            (user_log_mask False, model_bert.py:169-170)
 *   blend_bwd:  d_vecs += d_blend * m, dpad += sum_r d_blend (1 - m)   (mask NULL: d_vecs += d_blend)
 *   attn_fwd:   q, k, v, ctx fp32 [B*H, n_heads*16]; s_ij = exp(q_i.k_j / 4) [* mask_j] (NO max subtraction),
 *               ctx_i = sum_j s_ij v_j / (sum_j s_ij + 1e-8); mask fp32 [B,H] or NULL (unmasked branch)
 *   attn_bwd:   d_ctx -> dq, dk, dv (assigned; scores recomputed)
 *   1 <= H <= 512: H <= 64 runs a block per impression (warp per head), longer histories a block per (impression, head)
 * The Q/K/V projections are tnr_sgemm_nt (batch 3), their weight gradients tnr_sgemm_tn_acc, and the input
 * gradient dX = dQ W_Q + dK W_K + dV W_V is tnr_sgemm_nn:  C[M,N] = sum_p A[p][M,K] . B[p][K,N]. */
int tnr_nrms_blend_fwd(const float* vecs, const float* mask, const float* pad_doc, float* out, int rows, int D,
                       void* stream);
int tnr_nrms_blend_bwd(const float* d_blend, const float* mask, float* d_vecs, float* dpad, int rows, int D,
                       void* stream);
int tnr_nrms_attn_fwd(const float* q, const float* k, const float* v, const float* mask, float* ctx, int B, int H,
                      int n_heads, void* stream);
int tnr_nrms_attn_bwd(const float* q, const float* k, const float* v, const float* mask, const float* d_ctx,
                      float* dq, float* dk, float* dv, int B, int H, int n_heads, void* stream);
int tnr_sgemm_nn(const float* A, const float* B, float* C, int M, int N, int K, int parts, long long sA,
                 long long sB, void* stream);

/* ------------------------------------------------------------------ optimiser */
/* Adam(amsgrad=True) on a flat fp32 buffer (torch.optim.Adam semantics, run.py:134) fused with
 * the bf16 shadow-weight refresh; grad_scale pre-multiplies g.  vmax == NULL: plain Adam (amsgrad=False, the
 * optimiser of Post-train_KD.ipynb cell 18): the denominator uses v. */
int tnr_adam_amsgrad(float* p, const float* g, float* m, float* v, float* vmax, void* shadow_bf16,
                     long long n, float lr, float beta1, float beta2, float eps, int step,
                     float grad_scale, void* stream);
/* The same with the step counter ON THE DEVICE (int32; bc_ws: 2 floats of workspace for the bias corrections): a
 * captured CUDA graph of the train step replays with the right step number.  advance != 0: ++step and refresh
 * bc_ws first; advance == 0: update this range with the corrections of the current step (the optimiser steps the flat
 * buffer in two ranges so that the last gradient all-reduce of the step overlaps the update of everything else). */
int tnr_adam_amsgrad_devstep(float* p, const float* g, float* m, float* v, float* vmax, void* shadow_bf16,
                             long long n, float lr, float beta1, float beta2, float eps, int* step_dev,
                             float* bc_ws, float grad_scale, int advance, void* stream);
int tnr_cast_f32_bf16(const float* x, void* y_bf16, long long n, void* stream);

/* ------------------------------------------------------------------ gradient exchange over peer memory */
/* In-place SUM all-reduce of floats [off, off + n) of a symmetric fp32 buffer across the `world` GPUs of one NVSwitch
 * node, over peer-mapped memory in ONE kernel of n_ctas CTAs (two-shot: rank r reduces slice r from every peer in rank
 * order and stores the sum into every peer's buffer; flag barriers before and after; bit-identical results on all
 * ranks).  ptrs_dev / flags_dev: DEVICE arrays of `world` pointers -- rank r's copy of the buffer and of a zero-
 * initialised flag page of tnr_allreduce_p2p_flag_words() uint32 (both symmetric allocations, e.g.
 * torch.distributed._symmetric_memory).  multicast_ptr != NULL: the NVLS multicast mapping of the same buffer -- the
 * reduce becomes multimem.ld_reduce (sum inside the NVSwitch) + multimem.st (one store reaches every rank); NULL: peer
 * loads / stores.  Every rank must launch it with the same (off, n, n_ctas) in the same order;
 * it is graph-capturable (no host-side sequence state).  Replaces the Horovod gradient all-reduce of
 * Tiny-NewsRec/run.py:144-149 (hvd.DistributedOptimizer, op=Average: the 1/world is folded into the Adam kernel). */
long long tnr_allreduce_p2p_flag_words(void);
int tnr_allreduce_p2p(void* const* ptrs_dev, void* multicast_ptr, void* const* flags_dev, int rank, int world,
                      long long off, long long n, int n_ctas, void* stream);

/* ------------------------------------------------------------------ batch assembly */
/* out[r,:] = (int64) table[idx[r], :]   (news_combined[idx] -> LongTensor, dataloader.py:131,138,152-156);
 * idx outside [0, n_rows_table) maps to row 0 (dataloader.py:74).  Bit-exact. */
int tnr_gather_rows_i32_i64(const int32_t* table, long long n_rows_table, const int32_t* idx,
                            long long n, int W, int64_t* out, void* stream);
/* A whole training batch from its index arrays in one launch (dataloader.py:129-144): rows [history | candidates] of
 * tokens_out int64 [n_hist + n_cand, W] = news[idx] widened, and for each of the M <= 8 teacher tables (host arrays of
 * device pointers) teacher_out[i][r, :D] (row stride out_ld floats) = teacher_tables[i][idx[r], :].  Unknown ids read
 * row 0.  Bit-exact copies. */
int tnr_train_batch_gather(const int32_t* news, long long n_rows, int W, const float* const* teacher_tables,
                           float* const* teacher_out, int M, int D, long long out_ld, const int32_t* hist_idx,
                           long long n_hist, const int32_t* cand_idx, long long n_cand, long long* tokens_out,
                           void* stream);
/* out[r, :D] = table[idx[r], :]  fp32 (teacher_embs[i][idx], dataloader.py:142,144; news_scoring[idx] :295,301). */
int tnr_gather_rows_f32(const float* table, long long n_rows_table, const int32_t* idx, long long n,
                        int D, float* out, long long out_ld, void* stream);

/* ------------------------------------------------------------------ impression scoring */
/* Per impression b: score_c = table[cand[ptr[b]+c]] . user[b]; AUC / MRR / nDCG@5 / nDCG@10 with
 * binary labels; impressions with constant labels are skipped (valid = 0).
 * ptr int64 [n_imp + 1] (CSR offsets, ptr[n_imp] == nnz), cand int32 [nnz] (ids outside 0..n_rows-1 read row 0),
 * label int8 [nnz]; per_imp double [n_imp, 5] = {auc, mrr, ndcg5, ndcg10, valid}; sums double [5] += column sums
 * (NULL to skip); scores fp32 [nnz]: REQUIRED, the dot scores (output, and the workspace between the flat scoring
 * kernel and the per-impression ranking kernel); max_c >= the largest candidate count of the batch.
 * Replaces the Python loop at Tiny-NewsRec/run.py:346-361 + metrics.py:5-23 + sklearn roc_auc_score. */
int tnr_eval_metrics(const float* table, long long n_rows, const float* user, const long long* ptr,
                     const int32_t* cand, const int8_t* label, long long n_imp, long long nnz, int D, int max_c,
                     double* per_imp, double* sums, float* scores, void* stream);

/* doc-sim diagnostic: *sum_out += sum over pairs (i, j) int32 [n_pairs, 2] with i != j of the fp32 cosine of
 * table rows i and j (pairs with i == j or out of range add 0, as the reference skips them).
 * Replaces the 1 000 000-iteration numpy loop at Tiny-NewsRec/run.py:292-299. */
int tnr_doc_sim(const float* table, long long n_rows, const int32_t* pairs, long long n_pairs, int D,
                double* sum_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TINYREC_H_ */
