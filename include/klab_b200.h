/*
 * klab_b200.h -- C ABI of libklab_b200.so: hand-written sm_100a kernels for the image-caption
 * training step of Da-Tsuchi/KLab_MultiModalModel (Swin-V2 encoder + T5 encoder/decoder + LM-head CE).
 *
 * The reference has no FFI of its own: its seam is the Python class `MyModel`
 * (/root/reference/models/model.py:8-42) and all arithmetic is delegated to `transformers`
 * (HF/ below = site-packages/transformers 5.5.0).  Each entry point therefore cites the HF function
 * whose eager op chain it replaces (SURVEY.md section 2.3 K1..K14, section 8a).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero otherwise (never throws); klab_last_error() gives
 *     the message of the calling thread's last failure;
 *   - all pointers are DEVICE pointers unless stated; tensors are row-major; `ld*` are row strides in
 *     ELEMENTS; `stream` is a cudaStream_t passed as void*;
 *   - dtypes: KLAB_F32 (strict path, fp32 SIMT arithmetic) or KLAB_BF16 (bf16 storage, tcgen05 tensor
 *     cores, fp32 accumulation and statistics);
 *   - the library borrows pointers for the duration of a call and keeps none;
 *   - there is no CPU fallback: on a device that is not sm_100 every compute entry fails with
 *     KLAB_ERR_UNSUPPORTED.
 */
#ifndef KLAB_B200_H
#define KLAB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLAB_ABI_VERSION 1

enum { KLAB_F32 = 0, KLAB_BF16 = 1 };
enum { KLAB_OK = 0, KLAB_ERR_INVALID = 1, KLAB_ERR_CUDA = 2, KLAB_ERR_UNSUPPORTED = 3 };

/* ---- library / device probes -------------------------------------------------------------- */
int klab_abi_version(void);
const char* klab_last_error(void);
/* 0 iff the current CUDA device is compute capability 10.x (sm_100a code is present in the library). */
int klab_check_device(void);
/* number of kernels this library has launched since load (bench.py's `gpu_launches`). */
long long klab_launch_count(void);
/* Data parallelism (replaces nothing in HF; serves /root/reference/train.py:26): the persistent kernels of this library size
 * their grids to the SM count minus `n_sms`, leaving those SMs to the CTAs of a concurrently running NCCL collective (a
 * 230 KB-shared-memory CTA cannot share an SM with them; without the reserve every persistent kernel that overlaps a
 * collective runs a second, nearly empty wave).  0 = use every SM (default).  klab_sm_budget returns the SMs in use. */
int klab_set_sm_reserve(int n_sms);
int klab_sm_budget(void);
/* 1: the persistent GEMM / T5-attention kernels launched from now on take their work items from a per-launch counter (first
 * item static), so CTAs that find their SM held by a collective do not stretch the kernel by a whole wave; 0 (default, also
 * KLAB_DYNAMIC_SCHED=0/1): static stride, ~1 us per launch cheaper when nothing else shares the GPU.  Set before the first
 * forward: CUDA graphs bake the choice. */
int klab_set_dynamic_sched(int on);

/* ---- K5: GEMM with fused epilogue -----------------------------------------------------------
 * Replaces every nn.Linear on the path: HF/models/swinv2/modeling_swinv2.py:535,578-579,591,385 and
 * HF/models/t5/modeling_t5.py:93-102,178-181,277,298-299,338,1110 (forward, dgrad and wgrad).
 *
 *   D[M,N] = epilogue( alpha * sum_k A(m,k) * B(n,k) )
 *
 * A(m,k) is read from A[m*lda + k]  (a_mn_major = 0)  or  A[k*lda + m]  (a_mn_major = 1);
 * B(n,k) is read from B[n*ldb + k]  (b_mn_major = 0)  or  B[k*ldb + n]  (b_mn_major = 1).
 *   forward  y = x W^T      : A = x  [M,K] (0), B = W [N,K] (0)
 *   dgrad    dx = dy W      : A = dy [M,N'](0), B = W [N',K'] read as B(n=k', k=n') (1)
 *   wgrad    dW = dy^T x    : A = dy read as A(m=n', k=row) (1), B = x read as B(n=k', k=row) (1)
 * epilogue, in order:  v += bias[n];  aux_out[m,n] = v (GELU_SAVE_GRAD: gelu'(v));  v = act(v) or v *= act'(aux_in[m,n]);
 *                      v *= dropout_keep(seed, m*N+n)/(1-p);  v += residual[m,n];  v += D_old (accumulate);
 * in_dtype KLAB_BF16 runs the tcgen05/TMEM/TMA kernel (requires lda, ldb multiples of 8 and 16-byte
 * aligned bases); in_dtype KLAB_F32 runs the fp32 SIMT kernel (strict parity path). */
enum { KLAB_ACT_NONE = 0, KLAB_ACT_RELU = 1, KLAB_ACT_GELU = 2, KLAB_ACT_RELU_BWD = 3, KLAB_ACT_GELU_BWD = 4,
       /* GELU whose DERIVATIVE is saved: forward writes aux_out = gelu'(pre-activation) (instead of the pre-activation) next to
        * D = gelu(pre-activation) -- both come out of the same erfc / exp evaluation -- and the backward GEMM only multiplies:
        * KLAB_ACT_MUL_AUX: v *= aux_in.  Saves the ~19-instruction gelu' evaluation per element in an issue-bound epilogue. */
       KLAB_ACT_GELU_SAVE_GRAD = 5, KLAB_ACT_MUL_AUX = 6 };

typedef struct klab_gemm_epilogue {
    const float* bias;      /* [N] fp32, or NULL */
    const void* residual;   /* [M,N] ld = ldr, dtype res_dtype, or NULL */
    const void* aux_in;     /* RELU_BWD: saved post-activation; GELU_BWD: saved pre-activation */
    void* aux_out;          /* optional copy of the pre-activation value, dtype out_dtype */
    long long ldr, ld_aux_in, ld_aux_out;
    float alpha;
    int act;
    int accumulate;         /* D += result (D must be initialised) */
    int out_dtype, res_dtype, aux_in_dtype;
    float dropout_p;        /* 0 = off */
    unsigned long long dropout_seed;
    const unsigned long long* dropout_seed_ptr; /* optional DEVICE counter added to dropout_seed (CUDA-graph friendly) */
} klab_gemm_epilogue;

int klab_gemm(void* stream, int in_dtype, int M, int N, int K,
              const void* A, long long lda, int a_mn_major,
              const void* B, long long ldb, int b_mn_major,
              void* D, long long ldd, const klab_gemm_epilogue* epi);
/* Test / tuning aid for the bf16 tensor-core path: pin the kernel kind (cta2: 0 = one-CTA kernel, 1 = CTA-pair kernel with
 * tcgen05.mma.cta_group::2), the N tile and the split-K count of the klab_gemm calls that follow; -1 leaves a choice to the
 * library (default; KLAB_GEMM_FORCE_CTA2 / _BN / _SPLITS preset it at load).  A pin the shape cannot honour is ignored.
 * klab_gemm_last_config reports what the calling thread's last bf16 klab_gemm actually launched. */
int klab_gemm_set_force(int cta2, int bn, int splits);
int klab_gemm_last_config(int* bn, int* splits, int* cta2);
/* Same contract, forced onto the fp32-accumulating SIMT kernel (on-device cross-check of the tensor-core path). */
int klab_gemm_simt(void* stream, int in_dtype, int M, int N, int K,
                   const void* A, long long lda, int a_mn_major,
                   const void* B, long long ldb, int b_mn_major,
                   void* D, long long ldd, const klab_gemm_epilogue* epi);

/* ---- K8: T5 RMSNorm (HF/models/t5/modeling_t5.py:55-68) -------------------------------------
 * y = x * rsqrt(mean(x^2) + eps) * gamma; fp32 statistics; gamma is fp32.  Output rows may be "grouped":
 * row r is written at y + (r / y_rows_per_group) * y_group_stride + (r % y_rows_per_group) * ldy
 * (y_rows_per_group = 0: plain r * ldy) so the frozen text encoder writes straight into the concatenated
 * [image tokens; text tokens] buffer (/root/reference/models/model.py:23).  rstd_out (fp32 [rows]) may be NULL.
 * bwd: dx = rstd * (dy*gamma - xhat * mean(dy*gamma*xhat)) + dres;  dgamma (+)= sum_rows dy * xhat. */
int klab_rmsnorm_fwd(void* stream, int dtype, long long rows, int d, const void* x, long long ldx, const float* gamma, float eps,
                     void* y, long long ldy, int y_rows_per_group, long long y_group_stride, float* rstd_out);
int klab_rmsnorm_bwd(void* stream, int dtype, long long rows, int d, const void* dy, long long lddy, const void* x, long long ldx,
                     const float* gamma, const float* rstd, const void* dres, long long lddres, void* dx, long long lddx,
                     float* dgamma, int accumulate_dgamma, void* workspace);
/* Same, and in the same pass dx_drop[rows, d] = dropout(dx) with the mask klab_dropout_apply(p, seed, seed_ptr) draws for a
 * contiguous [rows, d] tensor: the consumer of dx (T5LayerSelfAttention / T5LayerCrossAttention backward,
 * HF/models/t5/modeling_t5.py:375,406) starts by applying its forward dropout mask to its output gradient. */
int klab_rmsnorm_bwd_dropout(void* stream, int dtype, long long rows, int d, const void* dy, long long lddy, const void* x, long long ldx,
                             const float* gamma, const float* rstd, const void* dres, long long lddres, void* dx, long long lddx,
                             float* dgamma, int accumulate_dgamma, void* workspace, void* dx_drop, float p, unsigned long long seed,
                             const unsigned long long* seed_ptr);
long long klab_norm_bwd_workspace_bytes(long long rows, int d);

/* ---- K6: LayerNorm, Swin-V2 res-post-norm form (HF/models/swinv2/modeling_swinv2.py:273,386,707-712,969) ----
 * y = LN(x) * gamma + beta (+ residual).  bwd: dx = LN'(dy) (+ dres); dgamma/dbeta (+)= column sums.
 * The backward can read dy through the same grouped row map (gradient of the concat buffer). */
int klab_layernorm_fwd(void* stream, int dtype, long long rows, int d, const void* x, long long ldx, const float* gamma,
                       const float* beta, float eps, const void* residual, long long ldres, void* y, long long ldy,
                       int y_rows_per_group, long long y_group_stride, float* mean_out, float* rstd_out);
int klab_layernorm_bwd(void* stream, int dtype, long long rows, int d, const void* dy, long long lddy, int dy_rows_per_group,
                       long long dy_group_stride, const void* x, long long ldx, const float* gamma, const float* mean,
                       const float* rstd, const void* dres, long long lddres, void* dx, long long lddx, float* dgamma,
                       float* dbeta, int accumulate_dparams, void* workspace);

/* out[c] (+)= sum_r x[r,c]: bias gradients of the Swin linears. */
int klab_colsum(void* stream, int dtype, long long rows, int d, const void* x, long long ldx, float* out, int accumulate,
                void* workspace);
long long klab_colsum_workspace_bytes(long long rows, int d);

/* ---- K9: T5 attention (HF/models/t5/modeling_t5.py:253-344; bias :189-251; causal mask :704) ----
 * q/k/v/out live in the [B*L, H*d_kv] layout of the projection GEMMs (row strides ld*); head h uses columns
 * [h*d_kv, (h+1)*d_kv).  scores = q k^T (unscaled) + bias_table[rel_bucket[(j - i - q_offset) + rel_zero], h];
 * causal: key j visible iff j <= i + q_offset.  bias_table NULL = cross-attention (zero bias).  rel_bucket is
 * the int32 LUT of T5Attention._relative_position_bucket built by the host with the reference's own torch ops
 * (bit-exact bucket edges).  lse fp32 [B,H,Lq] is saved for backward.  dropout_p > 0 drops probabilities with a
 * counter-based RNG keyed by (seed + *seed_ptr, b, h, i, j) that backward regenerates.  d_kv = 64 with Lq, Lk <= 256 in bf16
 * runs the tcgen05 kernel (t5_attention_tc.cu); other shapes / fp32 run the exact-fp32 CUDA-core kernel.
 * bwd: dq/dk/dv in the same layouts; dbias_table [num_buckets,H] is ACCUMULATED (the table of block 0 receives
 * the gradient of every block, :758). */
int klab_t5_attention_fwd(void* stream, int dtype, int B, int H, int Lq, int Lk, int d_kv, const void* q, long long ldq,
                          const void* k, long long ldk, const void* v, long long ldv, void* out, long long ldo,
                          const float* bias_table, const int* rel_bucket, int rel_zero, int num_buckets, int causal,
                          int q_offset, float* lse, float dropout_p, unsigned long long seed,
                          const unsigned long long* seed_ptr);
int klab_t5_attention_bwd(void* stream, int dtype, int B, int H, int Lq, int Lk, int d_kv, const void* q, long long ldq,
                          const void* k, long long ldk, const void* v, long long ldv, const void* out, const void* dout,
                          long long ldo, void* dq, void* dk, void* dv, const float* bias_table, const int* rel_bucket,
                          int rel_zero, int num_buckets, int causal, int q_offset, const float* lse, float* dbias_table,
                          float dropout_p, unsigned long long seed, const unsigned long long* seed_ptr, void* workspace);
long long klab_t5_attention_bwd_workspace_bytes(int B, int H, int Lq, int num_buckets);
/* Beam-search decode attention (one query row per hypothesis; the rows of one sample are consecutive).  Same arithmetic as the
 * Lq = 1 forward above, except where keys come from:
 *   src != NULL (self-attention): key / value position j of query row r is cache row src[r * ld_src + j] * Lk + j of k / v
 *     (Lk = cache positions per hypothesis); causal bound j <= q_offset; T5 bias as above.  src is the beam ancestry table of
 *     klab_beam_update: it replaces HF's per-step cache reorder (HF/generation/utils.py:3330-3336).
 *   src == NULL (cross-attention): the kv_group consecutive query rows r of one sample share its K/V rows
 *     [(r / kv_group) * Lk, ... + Lk) -- the encoder output is projected once per sample, not per beam
 *     (HF's _expand_inputs_for_generation repeats it).  No bias, no mask.
 * kv_group query rows (1..32) run in one CTA and consume each K/V chunk from shared memory.  bf16 (16-byte loads) or fp32 (the
 * exact path); fp32 arithmetic either way. */
int klab_t5_attention_decode_beam(void* stream, int dtype, int rows, int H, int Lk, int d_kv, const void* q, long long ldq,
                                  const void* k, long long ldk, const void* v, long long ldv, void* out, long long ldo,
                                  int kv_group, const int* src, long long ld_src, const float* bias_table, const int* rel_bucket,
                                  int rel_zero, int q_offset);

/* ---- K2+K3+K4: Swin-V2 shifted-window cosine attention (HF/models/swinv2/modeling_swinv2.py:421-487,
 * window_partition/roll/reverse :146-166,:678,:698, shift mask :627-653) -------------------------------
 * q/k/v (row stride ld; dq/dk/dv use the same) and ctx/dctx (row stride ldc) are [B*res*res, heads*head_dim] in natural token order; the window partition, the
 * cyclic shift and the {0,-200} shift mask are computed from coordinates inside the kernel.
 * bias = 16*sigmoid(CPB) [heads,N,N] from klab_swin_cpb_fwd; logit_scale is the raw parameter [heads].
 * bwd OVERWRITES dbias [heads,N,N] and dlogit_scale [heads]. */
int klab_swin_attention_fwd(void* stream, int dtype, int B, int res, int heads, int head_dim, int window, int shift,
                            const void* q, const void* k, const void* v, long long ld, void* ctx, long long ldc,
                            const float* logit_scale, const float* bias, float* lse);
int klab_swin_attention_bwd(void* stream, int dtype, int B, int res, int heads, int head_dim, int window, int shift,
                            const void* q, const void* k, const void* v, long long ld, const void* ctx, const void* dctx,
                            long long ldc, void* dq, void* dk, void* dv, const float* logit_scale, const float* bias,
                            const float* lse, float* dbias, float* dlogit_scale);
/* Continuous position bias MLP (:408-410,:450-460; tables :489-524 are built by the host). */
int klab_swin_cpb_fwd(void* stream, int table_rows, int hidden_units, int heads, int n_tokens, const float* coords,
                      const int* index, const float* w1, const float* b1, const float* w2, float* hidden, float* tab, float* bias);
int klab_swin_cpb_bwd(void* stream, int table_rows, int hidden_units, int heads, int n_tokens, const float* coords,
                      const int* index, const float* w2, const float* hidden, const float* tab, const float* dbias, float* dtab,
                      float* dw1, float* db1, float* dw2, int accumulate);

/* ---- K11 + T8: embedding gather with _shift_right fused (HF/models/t5/modeling_t5.py:595-614,:682) and its
 * scatter-add backward into the tied fp32 embedding gradient. ids are int64 [B,L]. */
int klab_embedding_fwd(void* stream, int dtype, int B, int L, const long long* ids, int shift_right, int start_id, int pad_id,
                       const void* table, long long vocab, int d, void* out, long long ldo, int* err_flag);
int klab_embedding_bwd(void* stream, int dtype, int B, int L, const long long* ids, int shift_right, int start_id, int pad_id,
                       const void* dout, long long ldo, int d, float* dtable, long long vocab);

/* ---- K1 / K7 data movement: patch-embedding im2col (Conv2d k=s=P, :329) and patch-merging 2x2 gather (:374-383;
 * scatter = 1 is the inverse permutation used by backward). */
int klab_patchify(void* stream, int out_dtype, int B, int C, int H, int W, int P, const float* pixels, void* out, long long ldo);
int klab_patch_merge(void* stream, int dtype, int B, int res, int C, const void* in, void* out, int scatter);

/* ---- N2 (SURVEY.md 8f): the arithmetic of the reference's host-side image processor (/root/reference/train.py:39,55:
 * AutoImageProcessor -> transformers ViTImageProcessor: rescale by 1/255, then (x - mean[c]) / std[c]) on the device.
 * in: [B, C, H*W] uint8 (in_is_u8 = 1) or fp32; out fp32, same layout.  mean / std are HOST pointers to C floats (has_norm = 0:
 * rescale only).  Rounding follows the numpy code it replaces: r = float32(double(x) * rescale); y = (r - mean) / std in fp32. */
int klab_image_normalize(void* stream, int in_is_u8, int B, int C, long long hw, const void* in, double rescale, const float* mean,
                         const float* std, int has_norm, float* out);

/* ---- K10 (generic path): cross entropy with ignore_index = -100 over materialised logits
 * (HF/models/t5/modeling_t5.py:1114-1117). stats = {mean loss, #non-ignored rows}.  bwd overwrites the logits
 * with d loss / d logits scaled by *gscale (device scalar, may be NULL = 1). */
int klab_ce_fwd(void* stream, int dtype, long long rows, int V, const void* logits, long long ld, const long long* labels,
                float* lse, float* row_loss, float* stats, int* err_flag);
int klab_ce_bwd(void* stream, int dtype, long long rows, int V, void* logits, long long ld, int ld_pad, const long long* labels,
                const float* lse, const float* stats, const float* gscale);

/* ---- K10 (hot path): LM head fused with the cross entropy, vocab-tiled, logits never written
 * (HF/models/t5/modeling_t5.py:1105-1117: logits = (h * d^-0.5) E^T with the tied embedding, CrossEntropyLoss(ignore_index=-100)).
 * bf16 tcgen05 path only.  fwd: the LM-head GEMM's epilogue keeps, per (row, vocab tile), an online-softmax partial
 * (max, sum exp) and the label's logit in fp32 straight out of TMEM; a second kernel combines them into lse[rows] and
 * stats = {mean loss over non-ignored rows, #non-ignored rows}.  workspace: klab_lmhead_ce_workspace_bytes(rows, V).
 * bwd is vocab-chunked by the caller: klab_lmhead_ce_bwd_chunk recomputes the logits of vocabulary columns [v0, v0 + vc)
 * (E_chunk = E + v0 * lde) and writes d loss / d logits * (*gscale) as bf16 into dlogits [rows, vc] (a chunk-sized scratch that
 * stays in L2); the caller then runs dH += dlogits E_chunk and dE[v0:v0+vc] = dlogits^T H with klab_gemm. */
long long klab_lmhead_ce_workspace_bytes(long long rows, int V);
int klab_lmhead_ce_fwd(void* stream, long long rows, int V, int d, const void* h, long long ldh, const void* E, long long lde, float alpha,
                       const long long* labels, float* lse, float* stats, void* workspace, int* err_flag);
int klab_lmhead_ce_bwd_chunk(void* stream, long long rows, int d, const void* h, long long ldh, const void* E_chunk, long long lde, float alpha,
                             const long long* labels, const float* lse, const float* stats, const float* gscale, int v0, int vc,
                             void* dlogits, long long ldd);

/* ---- K14 (part): greedy decode step (HF/generation/utils.py:2762-2800): ids[b,t] = unfinished[b] ? argmax(logits[b,:]) : pad;
 * unfinished[b] &= ids[b,t] != eos.  logits are fp32 [B,V]; ties resolve to the lowest index. */
int klab_greedy_step(void* stream, int B, int V, const float* logits, long long ld, long long* ids, long long ld_ids, int t,
                     int* unfinished, int pad_id, int eos_id);

/* ---- K14 (part): multinomial sampling step (HF/generation/utils.py:2658-2800 with do_sample=True): per row of the fp32
 * logits [rows, V], unfinished rows draw ids[row, t] from softmax(warped logits), finished rows get pad_id;
 * unfinished[row] &= ids[row, t] != eos.  Warpers in HF's order: logits / temperature; top_k > 0 keeps scores >= the k-th
 * largest (ties kept; top_k >= V keeps all); top_p < 1 keeps token i iff the mass of the tokens with a strictly greater score
 * is < top_p, or i holds the maximum (ties at the boundary are all kept; top_p = 0 keeps the maximum and its ties).
 * The draw: u = u(*seed, row, t - 1) -- t - 1 is the number of tokens generated before this one -- with
 *   z = seed + 0x9E3779B97F4A7C15 * (1 + row * 2^16 + (t - 1)) mod 2^64, the splitmix64 finaliser on z, u = (z >> 40) * 2^-24;
 * the token is the smallest index i with sum_{j <= i, kept} exp(s_j - max) > u * Z, Z the sum over the kept tokens (the last
 * kept token if rounding leaves none).  seed is a DEVICE pointer (read at run time, so a captured graph draws anew when the
 * value there changes).  The row is held in shared memory: V too large for it returns an error.  t in 1..65536. */
int klab_sample_step(void* stream, int rows, int V, const float* logits, long long ld, long long* ids, long long ld_ids, int t,
                     int* unfinished, int pad_id, int eos_id, float temperature, int top_k, float top_p,
                     const unsigned long long* seed);

/* ---- K14 (part): beam search step on device state (HF/generation/utils.py:3076-3386, GenerationMixin._beam_search of 5.5.0,
 * one EOS id so k = 2 * num_beams candidates are kept).  Ties resolve to the lower flat index beam * V + token.
 * klab_beam_topk: per row of the fp32 logits [rows, V]: log_softmax (fp32) + run_scores[row], its k largest values, descending,
 *   as cand_val [rows, k] and token ids cand_tok [rows, k].  k even, 4..16.
 * klab_beam_update: one step for the token at position t + 1 of B samples of nb (2..8) running beams (rows b * nb + i):
 *   merges the nb * 2nb candidates, applies EOS / max-length (T new tokens), chooses the next running beams (run_scores,
 *   next_tok [B * nb] int64), merges the finished set (fin_scores: score / generated_len ** length_penalty, fin_seq, fin_flag,
 *   fin_len), updates the early-stop heuristic (unsat [B]) and done [B] (early_stopping 0 False, 1 True, 2 "never").
 *   src (int32), run_seq and fin_seq (int64) are double-buffered [2][B * nb][ld], ld >= T + 1: buffer t & 1 is read and
 *   (t + 1) & 1 written; src[r, j] is the cache row that holds position j of hypothesis r.  A sample with done[b] set no longer
 *   changes (its tables are carried forward unchanged); unsat and done must start at 1 and 0. */
int klab_beam_topk(void* stream, int rows, int V, int k, const float* logits, long long ld, const float* run_scores, float* cand_val,
                   int* cand_tok);
int klab_beam_update(void* stream, int B, int nb, int V, int T, int t, int eos_id, float length_penalty, int early_stopping,
                     const float* cand_val, const int* cand_tok, float* run_scores, int* src, long long* run_seq, long long ld,
                     float* fin_scores, long long* fin_seq, int* fin_flag, int* fin_len, int* unsat, int* done, long long* next_tok);

/* y = x * keep(seed, linear index)/(1-p): the mask klab_gemm's epilogue dropout applied to a contiguous [M,N] output
 * (T5 dropout sites, HF/models/t5/modeling_t5.py:95,149,375,406,734,768), regenerated for the backward pass. */
int klab_dropout_apply(void* stream, int dtype, long long n, const void* x, void* y, float p, unsigned long long seed,
                       const unsigned long long* seed_ptr);
/* Every dropout site takes `seed` (host scalar) plus an optional DEVICE counter `seed_ptr` whose value is added to it inside
 * the kernel; klab_seed_advance steps that counter on the device once per training step, so a captured CUDA graph replays
 * with fresh masks and without a host round trip. */
int klab_seed_advance(void* stream, unsigned long long* seed_counter);

/* Gated-GELU feed-forward of T5 v1.1 / Flan-T5 (T5DenseGatedActDense, HF/models/t5/modeling_t5.py:106-132), elementwise part.
 * u [rows, 2*d_ff] contiguous = [a | b], the output of ONE GEMM against the [wi_0; wi_1] operand.
 * fwd: h [rows, d_ff] = dropout(gelu_new(a) * b), gelu_new(x) = 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))).
 * bwd: du [rows, 2*d_ff] = [dh' * b * gelu_new'(a) | dh' * gelu_new(a)] with dh' = dropout(dh).
 * The mask is the one klab_dropout_apply(p, seed, seed_ptr) draws for a contiguous [rows, d_ff] tensor.  bf16 or fp32 in and
 * out, fp32 arithmetic; d_ff must be a multiple of 8 and every pointer 16-byte aligned (KLAB_ERR_INVALID otherwise). */
int klab_geglu_fwd(void* stream, int dtype, long long rows, int d_ff, const void* u, void* h, float p, unsigned long long seed,
                   const unsigned long long* seed_ptr);
int klab_geglu_bwd(void* stream, int dtype, long long rows, int d_ff, const void* dh, const void* u, void* du, float p,
                   unsigned long long seed, const unsigned long long* seed_ptr);

/* ---- N1: fused multi-tensor Adam (the optimizer step that follows the path: /root/reference/train.py:28,66,
 * torch.optim.Adam over model.transformer.parameters(); semantics of torch/optim/adam.py with amsgrad = False).
 * table (DEVICE, int64 [n_tensors][6]) = {param fp32*, grad fp32*, exp_avg fp32*, exp_avg_sq fp32*, bf16 operand copy* or 0,
 * numel}; blockmap (DEVICE, int32 [n_blocks][2]) = {tensor index, chunk index}, one CTA per chunk of klab_adam_chunk_elems()
 * elements.  `step` is the 1-based step count (bias corrections); grad_scale multiplies the gradient first.
 * When the bf16 pointer is non-zero the refreshed parameter is also written there (the operand the tensor cores read). */
int klab_adam_chunk_elems(void);
int klab_adam_step(void* stream, const long long* table_dev, const int* blockmap_dev, int n_blocks, double lr, double beta1,
                   double beta2, double eps, double weight_decay, long long step, double grad_scale);

/* dtype conversion (fp32 master weights -> bf16 operand copies). */
int klab_cast(void* stream, int src_dtype, int dst_dtype, long long n, const void* src, void* dst);

#ifdef __cplusplus
}
#endif
#endif /* KLAB_B200_H */
