/* egom2p_b200 -- C ABI of the B200 (sm_100a) kernels behind the EgoM2P masked multimodal training step.
 *
 * Every entry point takes plain device pointers + sizes + a cudaStream_t (passed as void*), launches on
 * that stream only, never synchronises the device, never allocates device memory, and returns 0 or a
 * negative EGOM2P_ERR_* code (message via egom2p_last_error(), thread-local). No torch types cross this
 * boundary. The reference is pure Python/PyTorch (no FFI of its own), so each group below names the
 * reference code (path:line under the upstream repo) whose eager-op sequence it replaces; the Python
 * binding a maintainer adds is a ctypes stub (INTEGRATION.md).
 *
 * Conventions: row-major; "rows" = tokens (batch*sequence flattened); bf16 = __nv_bfloat16 bits (uint16_t);
 * masks are uint8 (torch.bool) with 1 = masked-out, as in the reference's input_mask / target_mask.
 */
#ifndef EGOM2P_B200_H_
#define EGOM2P_B200_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EGOM2P_OK 0
#define EGOM2P_ERR_INVALID (-1) /* bad argument / unsupported shape */
#define EGOM2P_ERR_CUDA (-2)    /* CUDA runtime / driver error at launch */

#define EGOM2P_MAX_MODS 8

const char* egom2p_last_error(void);
int egom2p_abi_version(void);
/* Number of kernels this library has launched on behalf of the calling process (bench.py: gpu_launches). */
int64_t egom2p_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * (1) Index plan + fused embedding gather.
 * Replaces cat_encoder_tensors / forward_mask_encoder (egom2p/models/egom2p_model.py:251-283,344-396),
 * cat_decoder_tensors / forward_mask_decoder / adapt_decoder_attention_mask (:285-342,398-481) and the
 * adapter forwards (egom2p/models/encoder_embeddings.py:181-210,272-301; decoder_embeddings.py:337-370,455-487).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t n_mods;                          /* modalities in CONCAT order (encoder: mod_dict order; decoder: shuffled order) */
  int32_t batch;                           /* B */
  int32_t budget;                          /* num_encoder_tokens / num_decoder_tokens */
  int32_t is_decoder;                      /* 0: encoder plan, 1: decoder plan (needs attn_cnt, ids) */
  int32_t causal;                          /* decoder_causal_mask */
  int32_t sep;                             /* decoder_sep_mask */
  int32_t len[EGOM2P_MAX_MODS];            /* tokens per sample of each modality */
  int32_t mod_id[EGOM2P_MAX_MODS];         /* modality_info[mod]['id'] (int16 range) */
  const uint8_t* mask[EGOM2P_MAX_MODS];    /* (B, len) input_mask / target_mask */
  const int32_t* attn_cnt[EGOM2P_MAX_MODS];/* (B, len) decoder_attention_mask, decoder only */
  const int64_t* ids[EGOM2P_MAX_MODS];     /* (B, len) token ids, decoder only (target ids) */
} egom2p_plan_desc;

/* Stable partition of the concatenated mask (== argsort(mask + arange*1e-6)[:, :budget]).
 * Outputs (device): keep_idx (B,budget) int32 concat index; keep_mod / keep_pos (B,budget) int32 modality slot and
 * position inside it; pad (B,budget) uint8 (1 = pad slot); mod_mask (B,budget) int16 (-1 on pads);
 * n_valid (B) int32. Decoder only: target_ids (B,budget) int64 (0 on pads); key_lo/key_hi (B,budget) int32 = the
 * contiguous key range each decoder row may attend (empty range == every key masked). */
int egom2p_index_plan(const egom2p_plan_desc* desc, int32_t* keep_idx, int32_t* keep_mod, int32_t* keep_pos,
                      uint8_t* pad, int16_t* mod_mask, int32_t* n_valid, int64_t* target_ids, int32_t* key_lo,
                      int32_t* key_hi, void* stream);

/* Row lists of the vocabulary heads: for each of n_mods modality ids (host array), the flat indices i (ascending) with
 * mod_mask[i] == id, written to rows + m * cap (int64, cap >= total), and their number to counts[m] (device int32).
 * Replaces the per-modality boolean row-select y[decoder_mod_mask == id] (egom2p/models/egom2p_model.py:633). */
int egom2p_plan_rows(const int16_t* mod_mask, int64_t total, const int32_t* mod_ids, int32_t n_mods, int64_t cap,
                     int64_t* rows, int32_t* counts, void* stream);

typedef struct {
  int32_t n_mods;
  int32_t dim;
  int32_t len[EGOM2P_MAX_MODS];
  int32_t vocab[EGOM2P_MAX_MODS];
  const int64_t* ids[EGOM2P_MAX_MODS];     /* (B, len) token ids (encoder) or NULL (decoder: mask token) */
  const float* token_emb[EGOM2P_MAX_MODS]; /* (vocab, dim) fp32 or NULL */
  const float* pos_emb[EGOM2P_MAX_MODS];   /* (len, dim) fp32 */
  const float* mod_emb[EGOM2P_MAX_MODS];   /* (dim) fp32 */
} egom2p_embed_desc;

/* x0[r] = tok[r] + (pos_emb[p] + mod_emb)  and  emb[r] = pos_emb[p] + mod_emb  for kept slot r; pads -> 0.
 * tok[r] = token_emb[ids] (encoder) or mask_token (decoder, mask_token != NULL). emb may be NULL.
 * A token id outside [0, vocab) is clamped to 0 or vocab - 1 here and in the backward (the reference raises on it).
 * row_batch: sample index of every row (int32, rows), or NULL when the rows are the (B, budget) slots in order (sample =
 * r / budget). A non-NULL row_batch is what lets the rows of a ragged batch be PACKED (valid slots only, sample after
 * sample), so that every per-row kernel downstream works on the valid tokens only. */
int egom2p_embed_gather_fwd(const egom2p_embed_desc* desc, const float* mask_token, const int32_t* keep_mod,
                            const int32_t* keep_pos, const uint8_t* pad, const int32_t* row_batch, int64_t rows,
                            int32_t budget, float* x0, float* emb, void* stream);
/* Gradients of the above: d_token_emb[m][id] += dx0[r] (atomic scatter-add), d_mod_emb[m] += sum_r (dx0[r] + demb[r]),
 * d_mask_token += sum_r dx0[r]; all accumulate into the given fp32 buffers (any may be NULL). demb may be NULL. */
int egom2p_embed_gather_bwd(const egom2p_embed_desc* desc, const float* dx0, const float* demb, const int32_t* keep_mod,
                            const int32_t* keep_pos, const uint8_t* pad, const int32_t* row_batch, int64_t rows, int32_t budget,
                            float* const* d_token_emb, float* const* d_mod_emb, float* d_mask_token, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (3a) LayerNorm (no bias, eps) -- egom2p/models/egom2p_utils.py:118-133. fp32 in; bf16 and/or fp32 out.
 * ------------------------------------------------------------------------------------------------ */
int egom2p_layernorm_fwd(const float* x, const float* weight, int64_t rows, int32_t dim, float eps, uint16_t* y_bf16,
                         float* y_f32, float* mean, float* rstd, void* stream);
/* dx_out = dx_in (may be NULL) + LN'(dy); dy given as bf16 or fp32 (exactly one non-NULL); d_weight += sum_r dy*xhat
 * (NULL: not reduced, for a frozen weight). dx_bf16 (optional) receives a bf16 copy of dx_out. */
int egom2p_layernorm_bwd(const uint16_t* dy_bf16, const float* dy_f32, const float* x, const float* weight,
                         const float* mean, const float* rstd, const float* dx_in, int64_t rows, int32_t dim,
                         float* dx_out, uint16_t* dx_bf16, float* d_weight, void* stream);
/* nn.LayerNorm(dim, eps) with a learnable bias (the GELU / bias family, egom2p_model.py:882-978): the forward adds bias[c]
 * after the weight; the backward is the one above plus d_bias += sum_r dy in the same pass. d_weight and d_bias may each be
 * NULL (a frozen parameter's gradient is not reduced). */
int egom2p_layernorm_bias_fwd(const float* x, const float* weight, const float* bias, int64_t rows, int32_t dim, float eps,
                              uint16_t* y_bf16, float* y_f32, float* mean, float* rstd, void* stream);
int egom2p_layernorm_bias_bwd(const uint16_t* dy_bf16, const float* dy_f32, const float* x, const float* weight,
                              const float* mean, const float* rstd, const float* dx_in, int64_t rows, int32_t dim,
                              float* dx_out, uint16_t* dx_bf16, float* d_weight, float* d_bias, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (3b) bf16 GEMM on tcgen05/TMEM fed by TMA -- every nn.Linear on the path (egom2p_utils.py:167-169,187,203,226-228,
 * egom2p_model.py:722) and their dgrad / wgrad.  C[M,N] = op(A) * op(B)^T with fp32 accumulation:
 *   a_mn = 0: A is (M,K) row-major (K contiguous);  a_mn = 1: A is stored (K,M) row-major (M contiguous)
 *   b_mn = 0: B is (N,K) row-major (K contiguous);  b_mn = 1: B is stored (K,N) row-major (N contiguous)
 * lda/ldb = row pitch in elements of the stored matrices. Epilogue: out = acc (+ bias[n]) (+ addend[m,n]);
 * written as bf16 (c_bf16) or fp32 (c_f32) -- exactly one; addend may alias c_f32 (accumulate). A bias with bf16 output
 * (the biased qkv / q / kv projections) needs a_mn = b_mn = 0, no addend and a 16-byte aligned bias. fp32 outputs with few
 * tiles and long K (wgrad) are split along K and accumulated with TMA reduce-add.
 * ------------------------------------------------------------------------------------------------ */
int egom2p_gemm_bf16(const uint16_t* A, const uint16_t* B, int32_t M, int32_t N, int32_t K, int64_t lda, int64_t ldb,
                     int32_t a_mn, int32_t b_mn, const float* bias, const float* addend, int64_t ld_add,
                     uint16_t* c_bf16, float* c_f32, int64_t ldc, void* stream);

/* SwiGLU MLP with the gate fused into the GEMM epilogues (egom2p/models/egom2p_utils.py:154-169). W13 holds the rows of
 * fc1 and fc3 interleaved in groups of 32 (rows [64g, 64g+32) = fc1[32g..], rows [64g+32, 64g+64) = fc3[32g..]), so a
 * 64-column accumulator group is [a | b] of the same 32 hidden units.
 *   fwd: ab (M, N2) bf16 = X W13^T (saved for backward) and g (M, N2/2) bf16 = silu(a) * b, in one pass.
 *   bwd: dg = dY W2 (W2 stored (K, hidden), consumed MN-major) never leaves TMEM: dab (M, 2*hidden) bf16 =
 *        [dg * b * silu'(a) | dg * silu(a)] in the same interleaved layout. */
int egom2p_gemm_swiglu_fwd(const uint16_t* X, const uint16_t* W13, int32_t M, int32_t N2, int32_t K, int64_t ldx, int64_t ldw,
                           uint16_t* ab, int64_t ld_ab, uint16_t* g, int64_t ldg, void* stream);
int egom2p_gemm_swiglu_bwd(const uint16_t* dY, const uint16_t* W2, const uint16_t* ab, int32_t M, int32_t hidden, int32_t K,
                           int64_t ldy, int64_t ldw, int64_t ld_ab, uint16_t* dab, int64_t ld_dab, void* stream);

/* GELU MLP (fc2(GELU(fc1 x)) with biases, nn.GELU() exact erf form) with the activation fused into the GEMM epilogues.
 *   fwd: u (M, N) bf16 = X W1^T + b1 (saved for backward; b1 fp32, may be NULL) and h (M, N) bf16 = GELU(u), in one pass.
 *   bwd: dh = dY W2 (W2 stored (K, hidden), consumed MN-major) never leaves TMEM: du (M, hidden) bf16 = dh * GELU'(u).
 * N / hidden must be multiples of 64. */
int egom2p_gemm_gelu_fwd(const uint16_t* X, const uint16_t* W1, const float* b1, int32_t M, int32_t N, int32_t K, int64_t ldx,
                         int64_t ldw, uint16_t* u, int64_t ld_u, uint16_t* h, int64_t ldh, void* stream);
int egom2p_gemm_gelu_bwd(const uint16_t* dY, const uint16_t* W2, const uint16_t* u, int32_t M, int32_t hidden, int32_t K,
                         int64_t ldy, int64_t ldw, int64_t ld_u, uint16_t* du, int64_t ld_du, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (4) Vocabulary head fused with softmax cross-entropy (egom2p/models/decoder_embeddings.py:489-500,
 * egom2p_model.py:614-644): logits = Y W^T are produced tile-by-tile in TMEM and never written to HBM.
 * ------------------------------------------------------------------------------------------------ */
/* Pass 1: per (row, vocab tile) partial max / sum-exp and the target logit. part_* are (n_tiles, R) fp32 with
 * n_tiles = 2 * ceil(V / 256) (two column halves per 256-wide vocabulary tile); tgt_logit (R) fp32. */
int egom2p_ce_partials(const uint16_t* Y, const uint16_t* W, const int64_t* target, int32_t R, int32_t V, int32_t K,
                       int64_t ldy, int64_t ldw, float* part_max, float* part_sum, float* tgt_logit, void* stream);
/* Pass 1 of a head that needs a backward: the same partials, and the softmax numerators
 * probs[r, v] = 2^(logit * log2 e - ref[r]) as bf16 (R, V), row pitch ldp. ref (R) fp32 from egom2p_ce_row_ref. */
int egom2p_ce_probs(const uint16_t* Y, const uint16_t* W, const int64_t* target, const float* ref, int32_t R, int32_t V,
                    int32_t K, int64_t ldy, int64_t ldw, uint16_t* probs, int64_t ldp, float* part_max, float* part_sum,
                    float* tgt_logit, void* stream);
/* ref[r] = ||Y_r|| * max_v ||W_v|| * log2 e (an upper bound of every logit of row r, in log2 units); wmax2: one fp32 of
 * scratch. K, ldy, ldw multiples of 8. */
int egom2p_ce_row_ref(const uint16_t* Y, const uint16_t* W, int32_t R, int32_t V, int32_t K, int64_t ldy, int64_t ldw,
                      float* wmax2, float* ref, void* stream);
/* Pass 2: lse[r] = logsumexp over tiles; loss_sum += sum_r (lse[r] - tgt_logit[r]) (one fp32, atomically).
 * After egom2p_ce_probs (ref non-null, else the last six arguments are ignored): per 128-row tile, tile_flag = 1 when a
 * row has ref[r] - max logit * log2 e > 60 (its numerators are not exact in bf16); otherwise rscale[r] = 1 / sum_v probs[r, v]
 * and probs[r, target[r]] -= that sum, so that rscale[r] * probs[r, :] = softmax - onehot. Flagged tiles get rscale = 1. */
int egom2p_ce_finalize(const float* part_max, const float* part_sum, const float* tgt_logit, int32_t R,
                       int32_t n_tiles, float* lse, float* loss_sum, const float* ref, const int64_t* target, int32_t V,
                       uint16_t* probs, int64_t ldp, float* rscale, uint8_t* tile_flag, void* stream);
/* Backward recompute: dlogits[r, v0:v0+Vc] = (exp(logit - lse[r]) - [v == target[r]]) * gscale[0] as bf16 (R, Vc),
 * for the vocab chunk [v0, v0+Vc). gscale is a device scalar (upstream grad / R), or null for 1. With tile_flag
 * (the loss pass's flags) only the flagged 128-row tiles are computed and written; the launch is one round of CTA pairs. */
int egom2p_ce_dlogits(const uint16_t* Y, const uint16_t* W, const int64_t* target, const float* lse,
                      const float* gscale, const uint8_t* tile_flag, int32_t R, int32_t v0, int32_t Vc, int32_t K,
                      int64_t ldy, int64_t ldw, uint16_t* dlogits, int64_t ldd, void* stream);
/* Row scales of the head backward: s[r] = gscale[0] * rscale[r]; ys (R, K) bf16 = s[r] * Y[r, :] when ys is non-null. */
int egom2p_ce_row_scale(const uint16_t* Y, int32_t R, int32_t K, int64_t ldy, const float* rscale, const float* gscale,
                        float* s, uint16_t* ys, void* stream);

/* ------------------------------------------------------------------------------------------------
 * (2) Attention, head_dim 64, tcgen05/TMEM tiles fed by TMA, online softmax in fp32
 * (egom2p/models/egom2p_utils.py:185-205 self, :222-244 cross). Q rows live at Q + (b*Mq + i)*ldq + h*64 (same for
 * K/V with Nk, ldk/ldv; O with ldo), so packed qkv / kv projections are consumed in place. Each query row attends
 * one contiguous key range [key_lo, key_hi) of its sample (NULL: [0, Nk)); that is every mask this path produces
 * (encoder key padding, decoder cross, decoder per-modality self-attention, causal). An empty range reproduces the
 * reference's masked_fill(-finfo.max) behaviour: uniform attention over all Nk keys.
 * ------------------------------------------------------------------------------------------------ */
int egom2p_attn_lse_stride(int32_t Mq);                 /* S = Mq rounded up to 128 */
int64_t egom2p_attn_ranges_bytes(int32_t B, int32_t Mq); /* bytes of the range metadata buffer */
/* Builds the per-row / per-block range metadata once per forward; it is shared by every layer and head and by the
 * forward and backward kernels. key_lo / key_hi are (B, Mq) int32 or both NULL. meta: 256-byte aligned.
 * empty_zero = 0: a row with an empty range attends all Nk keys uniformly (the reference's masked_fill(-finfo.max));
 * empty_zero = 1: such a row has NO keys and its output is exactly 0 -- a sample whose context is empty inside a batch
 * that also holds non-empty contexts (the unconditional branch of guided decoding, egom2p/models/generate.py:793-802,
 * batched with the conditional one). Forward only. */
int egom2p_attn_ranges(const int32_t* key_lo, const int32_t* key_hi, int32_t B, int32_t Mq, int32_t Nk, float scale,
                       int32_t empty_zero, void* meta, void* stream);
/* lse is (B, H, S) fp32 in log2 units (reference + log2(sum) of scale*log2e*scores), saved for the backward pass.
 * kmax_scratch: B*H floats of device scratch for the pre-pass of the bound-path softmax (max_k |k|^2 per batch and head,
 * see csrc/attn.cu), or NULL to force the online-maximum softmax. */
int egom2p_attn_fwd(const uint16_t* Q, const uint16_t* K, const uint16_t* V, int32_t B, int32_t H, int32_t Mq, int32_t Nk,
                    int64_t ldq, int64_t ldk, int64_t ldv, const void* meta, uint16_t* O, int64_t ldo, float* lse,
                    float* kmax_scratch, void* stream);
/* Bytes of device scratch egom2p_attn_bwd needs (per-row delta terms + the fp32 dQ accumulator). */
int64_t egom2p_attn_bwd_scratch_bytes(int32_t B, int32_t H, int32_t Mq);
/* dQ/dK/dV use the same addressing as Q/K/V with their own row pitches; dO shares O's pitch. */
int egom2p_attn_bwd(const uint16_t* Q, const uint16_t* K, const uint16_t* V, const uint16_t* O, const uint16_t* dO,
                    const float* lse, int32_t B, int32_t H, int32_t Mq, int32_t Nk, int64_t ldq, int64_t ldk, int64_t ldv,
                    int64_t ldo, const void* meta, float scale, void* scratch, uint16_t* dQ, uint16_t* dK, uint16_t* dV,
                    int64_t lddq, int64_t lddk, int64_t lddv, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Elementwise helpers on the path.
 * ------------------------------------------------------------------------------------------------ */
int egom2p_cast_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, void* stream);
/* One launch for a list of casts: the per-step refresh of the bf16 GEMM operands from the fp32 master weights
 * (the reference gets this from torch.autocast's weight cache, run_training_egom2p.py:716). Item i casts a contiguous
 * (rows, cols) fp32 matrix into a bf16 matrix of row pitch dst_ld; group > 0 writes row r to row
 * (r / group) * 2 * group + slot * group + r % group (the interleaved fc1 | fc3 operand of egom2p_gemm_swiglu_fwd).
 * first_chunk = running sum of ceil(rows / rows_per_chunk) over the items before i; n_chunks = the total. The array
 * lives in device memory. */
typedef struct {
  const float* src;
  uint16_t* dst;
  int64_t rows;
  int64_t first_chunk;
  int32_t cols, dst_ld, group, slot, rows_per_chunk, pad_;
} egom2p_cast_item;
int egom2p_cast_f32_to_bf16_multi(const void* items_dev, int32_t n_items, int64_t n_chunks, void* stream);
/* out = a + b (fp32), optional bf16 copy. */
int egom2p_add_f32(const float* a, const float* b, int64_t n, float* out, uint16_t* out_bf16, void* stream);
/* Optimizer tail over ALL trainable tensors in two launches (the reference: clip_grad_norm_ + AdamW.step driven by
 * NativeScalerWithGradNormCount.__call__, egom2p/utils/native_scaler.py:27-47; AdamW groups from
 * egom2p/utils/optim_factory.py:206-226). The item table lives in device memory; first_chunk = running sum of
 * ceil(n / 8192) over the items before i, n_chunks = the total.
 *   egom2p_sumsq_multi: *sumsq = sum over all items of sum(g^2); deterministic (per-chunk partial sums in `partials`,
 *     n_chunks floats of scratch, added in a fixed order) so that data-parallel replicas compute identical clip factors.
 *   egom2p_adamw_multi_steps: torch.optim.AdamW update of every item with its own lr / weight decay; the gradient is read as
 *     g * min(1, max_norm / (sqrt(*sumsq) + 1e-6)) when sumsq != NULL (clip folded in: gradients are not rewritten; a NaN
 *     norm gives a NaN coefficient, as torch's clamp does). `steps` is a device array of n_items int32 step counts, one per
 *     item: item i's bias corrections use steps[i] + 1, and steps[0 .. n_items) are incremented afterwards (CUDA-graph
 *     capturable). It replaces egom2p_adamw_multi, which read one count shared by all items from the same argument
 *     position: the old symbol is gone, so a caller built against it fails to resolve it instead of passing a single
 *     counter where an array is read, and the ABI version is unchanged. */
typedef struct {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t n;
  int64_t first_chunk;
  float lr, weight_decay;
} egom2p_opt_item;
int egom2p_sumsq_multi(const void* items_dev, int32_t n_items, int64_t n_chunks, float* partials, float* sumsq, void* stream);
int egom2p_adamw_multi_steps(const void* items_dev, int32_t n_items, int64_t n_chunks, float beta1, float beta2, float eps,
                             int32_t* steps, const float* sumsq, float max_norm, void* stream);
/* out[c] += sum_r x[r, c] -- bias gradient of decoder_proj_context (egom2p_model.py:157,722). */
int egom2p_colsum_f32(const float* x, int64_t rows, int32_t cols, float* out, void* stream);
/* out[c] += sum_r x[r, c] for a bf16 (rows, cols) matrix of row pitch ld (cols, ld multiples of 8): the bias gradients of
 * the GELU / bias family's Linears from the bf16 output gradients, one atomic per column and row slab. */
int egom2p_colsum_bf16(const uint16_t* x, int64_t rows, int32_t cols, int64_t ld, float* out, void* stream);
/* dst[i, :] = src[idx[i], :] (bf16) and dst[idx[i], :] = src[i, :] (fp32; times row_scale[i] when row_scale is given):
 * compaction of the rows of one modality for its vocabulary head, replacing the boolean row-select
 * y[decoder_mod_mask == id] (egom2p_model.py:633). */
int egom2p_gather_rows_bf16(const uint16_t* src, const int64_t* idx, int64_t n, int32_t cols, uint16_t* dst, void* stream);
int egom2p_scatter_rows_f32(const float* src, const int64_t* idx, int64_t n, int32_t cols, const float* row_scale, float* dst,
                            void* stream);

/* ------------------------------------------------------------------------------------------------
 * Device-side masking of the token modalities: UnifiedMasking.image_mask (egom2p/data/masking.py:236-266) for a whole batch
 * of one modality. Positions are ranked by a random key per position (32-bit Philox draws from (seed, offset), subsequences
 * separated by stream_id; or the caller's noise (B, L) fp32 >= 0, ordered like a stable argsort): with ids_shuffle =
 * argsort(keys), position r is an input (input_mask 0) iff ids_shuffle[r] < input_budget[b] and a target (target_mask 0) iff
 * input_budget[b] <= ids_shuffle[r] < input_budget[b] + target_budget[b] (NULL: all the rest) -- the reference's gather --
 * and attn_cnt holds the target count at the lowest target position (0 elsewhere). L <= 8192.
 * ------------------------------------------------------------------------------------------------ */
int egom2p_image_masks(const float* noise, uint64_t seed, uint64_t offset, int32_t stream_id, int32_t B, int32_t L,
                       const int32_t* input_budget, const int32_t* target_budget, uint8_t* input_mask, uint8_t* target_mask,
                       int32_t* attn_cnt, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Generation (guided ROAR / MaskGIT decoding, egom2p/models/generate.py): fused sampling.
 * ------------------------------------------------------------------------------------------------ */
/* One token per row from fp32 logits (rows, V), row pitch ld, with the semantics of GenerationSampler.sample_tokens /
 * top_k_top_p_filtering (egom2p/models/generate.py:332-371): top-k (logits below the k-th largest are removed; 0 = off),
 * then top-p on softmax(remaining) at temperature 1 (a token is removed when the mass ranked strictly above it exceeds
 * top_p; 0 = off), then one draw from softmax(kept / temperature) -- here by inverse CDF in ascending token order with the
 * uniform u[row] in [0, 1); temperature == 0: argmax, prob 1. No sort and no second copy of the logits: threshold search by
 * nested 2048-bin mass histograms. The filtered set is always the n_kept largest logits, and tokens of equal logit are kept
 * or removed together: at top-k this is the reference's rule (nothing equal to the k-th value is removed); at top-p, where
 * the reference's stable sort keeps only the lower-index part of a tie group that straddles top_p, the whole group is kept.
 * Outputs: token (rows) int64, prob (rows) fp32 of the drawn token (may be NULL), n_kept (rows) int32 size of the filtered
 * set (may be NULL). V <= 65536. */
int egom2p_sample_rows(const float* logits, int64_t ld, int32_t rows, int32_t V, float temperature, float top_p,
                       int32_t top_k, const float* u, int64_t* token, float* prob, int32_t* n_kept, void* stream);
/* out = bf16(y_uncond + (y_cond - y_uncond) * scale): classifier-free guidance (generate.py:804) applied to the decoder
 * outputs before the (linear, bias-free) vocabulary head, so that one head GEMM yields the guided logits. */
int egom2p_cfg_combine_bf16(const float* y_uncond, const float* y_cond, int64_t n, float scale, uint16_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EGOM2P_B200_H_ */
