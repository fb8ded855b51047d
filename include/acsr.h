/* acsr.h -- flat C ABI of the B200-native AC-SASRec hot path (libacsr.so).
 *
 * The reference (AIM-SE/AC-TSR, a RecBole 1.0.1 fork) has no native code and no FFI:
 * every "kernel" is an ATen call made from Python.  Each entry point below therefore
 * cites the reference *Python call site* it replaces (paths relative to
 * /root/reference/recbole).  The reference-side binding is ctypes; INTEGRATION.md
 * shows the stub a maintainer adds to recbole/model/sequential_recommender/acsasrec.py.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch tensors), contiguous
 *    row-major; activations/parameters float32, ids int64 (RecBole's dtype).
 *  - `stream` is a cudaStream_t passed as void*; calls only enqueue work, never
 *    synchronise, never allocate.  Workspaces are passed in by the caller.
 *  - return 0 on success, <0 on error (ACSR_ERR_*); acsr_last_error() returns the
 *    message of the last failing call on this thread.  No exceptions cross the ABI.
 *  - dropout: `p` keep-complement probability.  If `mask` != NULL it holds the
 *    multiplicative mask (0 or 1/(1-p)) to apply (test / parity mode).  Otherwise, if
 *    p > 0, the mask is generated in-kernel with Philox4x32-10 keyed by
 *    (rng->seed, rng->step, rng_stream, element index); `rng` points to DEVICE memory
 *    {uint64 seed; uint64 step} so CUDA-graph replays see a new step.  Backward
 *    kernels regenerate the identical mask from the same triple.
 */
#ifndef ACSR_H_
#define ACSR_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACSR_ABI_VERSION 1
#define ACSR_OK 0
#define ACSR_ERR_ARG (-1)
#define ACSR_ERR_UNSUPPORTED (-2)
#define ACSR_ERR_CUDA (-3)

int acsr_version(void);
const char* acsr_last_error(void);
/* number of SMs the persistent kernels size their grids for (148 on B200) */
int acsr_num_sms(void);
/* launch the library's kernels with programmatic dependent launch (next kernel's prologue overlaps the tail of the
 * previous one).  Returns the previous setting.  Default: off (environment ACSR_PDL=1 turns it on). */
int acsr_set_pdl(int on);

/* Registers [ptr, ptr + bytes) as parameter memory: within a chain of kernels launched with programmatic dependent launch nothing
 * but the optimizer step (the chain's last node) writes it, so the GEMM kernels may stage weights that live there before they wait
 * for the previous kernel (their weight staging then overlaps its tail).  ptr == NULL clears the registry. */
int acsr_register_static(const void* ptr, int64_t bytes);

/* caller-owned scratch memory of the CURRENT device (the library allocates nothing).  Only the attention backward for
 * sequences longer than 64 needs it: acsr_attn_workspace_bytes(L, H, n_streams) bytes per sequence (0 for L <= 64;
 * n_streams = 1 for acsr_attn_calib_bwd, 2 for acsr_attn_calib_bwd2); with less than B sequences' worth the batch is
 * processed in chunks, with less than one the call fails.  The pointer must stay valid until the work enqueued with it
 * has completed. */
int acsr_set_workspace(void* ptr, int64_t bytes);
int64_t acsr_attn_workspace_bytes(int L, int H, int n_streams);

/* rng state helper: rng->step += 1 (one tiny kernel; keeps graph replays distinct) */
int acsr_rng_advance(void* rng, void* stream);

/* ---- K1: item-embedding gather (+position add) + LayerNorm + dropout ------------------
 * replaces model/sequential_recommender/acsasrec.py:87-95.
 * item_seq [T] int64 (T = B*L tokens), table [V,d], pos_emb [L,d] or NULL, out [T,d],
 * stats [T,2] (mean, rstd) saved for backward.  d in {32,64,128,256}.  Ids outside [0,V) are treated as the padding id 0 (no
 * out-of-bounds access; nn.Embedding would raise -- the host pipeline, dataset.py, guarantees the range). */
int acsr_embed_ln_dropout_fwd(const int64_t* item_seq, const float* table, const float* pos_emb,
                              const float* ln_w, const float* ln_b, float eps,
                              int T, int L, int d, int64_t V,
                              float p, const float* mask, const void* rng, uint32_t rng_stream,
                              float* out, float* stats, void* stream);
/* backward: d_table [V,d] += scatter (row 0 = padding_idx gets nothing, nn.Embedding(padding_idx=0)),
 * d_pos [L,d] +=, d_ln_w [d] +=, d_ln_b [d] += (all accumulate with atomics). */
int acsr_embed_ln_dropout_bwd(const float* d_out, const int64_t* item_seq, const float* table, const float* pos_emb,
                              const float* ln_w, const float* stats,
                              int T, int L, int d, int64_t V,
                              float p, const float* mask, const void* rng, uint32_t rng_stream,
                              float* d_table, float* d_pos, float* d_ln_w, float* d_ln_b, void* stream);

/* ---- K4-K7 core, K11: fused calibrated causal attention -------------------------------
 * replaces model/layers.py:657-674 (cal_attack_mask), 686-742 (cal_origin_qkv after the
 * projections), 883-896 (combine_attention), 917-936 and the probs.V of 676-678; the
 * additive mask of model/abstract_recommender.py:136-143 is derived from item_seq in-kernel.
 * mq,mk,mv,aq,ak [B,L,d] projected tensors; gate_logit [B,L,L] (combine_option gate) or NULL.
 * order_w [2*dh], order_b [1] or NULL (use_order False); dist_w, dist_b, scalar likewise.
 * flags: see ACSR_ATTN_*.  comb_scalar: annealing rate (combine_option annealing).
 * rich_ratio: device float* (rich_calibrated_combine trainable) or NULL (fixed -> 0.5).
 * D1,D2,D3 explicit dropout masks [B,H,L,L] or NULL; noise [B,H,L,L] or NULL (Philox normal).
 * ctx_att (may be NULL: attacked branch skipped), ctx_cal [B,L,d]; pen_sq [1] double,
 * accumulated: sum over b,h,i,j of (1-M)^2 (acsasrec.py:135).  probs_out NULL or
 * [6,B,H,L,L] = P0,P,M,A,C,R for introspection (layers.py:899-950).  L <= 64, dh <= 64. */
/* order: NULL, or int32 [B] from acsr_seq_order: CTA group g works on sequence order[g] (longest first), which trims
 * the tail of the launch when lengths vary.  Results do not depend on it.
 * ctx_rows: NULL, or int64 [B] (the item_length tensor) for the LAST layer, where only context row ctx_rows[b]-1 of each
 * sequence is consumed (gather_indexes, abstract_recommender.py:130-134): the other rows only compute their attack mask
 * for the penalty, their context rows are not written, and in the backward their d_ctx rows are taken as zero. */
int acsr_seq_order(const int64_t* item_seq, int B, int L, int32_t* order, void* stream);
#define ACSR_ATTN_TWO_LEVEL 1
/* second bit of the `two_level` argument: bidirectional attention mask, i.e. get_attention_mask(item_seq, bidirectional=True)
 * of model/abstract_recommender.py:136-143 as AcBERT4Rec uses it (acbert4rec.py:168): only padded KEYS are masked, query
 * row i sees keys j > i too (both branches of the order calibrator, layers.py:715-719, are then in play).  L <= 64. */
#define ACSR_ATTN_BIDIRECTIONAL 2
/* third bit: the layer of model/transformer_layers.py:873-953 (ACSSEPT, acssept.py:61-75) instead of model/layers.py:859-951.
 * Same projections, calibrators, attack mask and combine options, but attacked = origin*M + noise*(1-M), calibrated =
 * origin*exp(1-M) and the combination are used AS THEY ARE (transformer_layers.py:919-927), without the masked softmax
 * layers.py:917-925 puts around each of them.  Masked keys (future or padding) therefore keep an attacked weight -- the bare
 * noise -- and, with combine_option fixed, a share of softmax(origin + 0.5*calibrated): all L keys of every row are in play.
 * L <= 64. */
#define ACSR_ATTN_PLAIN 4
#define ACSR_ATTN_COMBINE_GATE 0
#define ACSR_ATTN_COMBINE_FIXED 1
#define ACSR_ATTN_COMBINE_ANNEAL 2
#define ACSR_ATTN_RICH_NONE 0
#define ACSR_ATTN_RICH_FIXED 1
#define ACSR_ATTN_RICH_TRAINABLE 2
int acsr_attn_calib_fwd(const float* mq, const float* mk, const float* mv, const float* aq, const float* ak,
                        const float* gate_logit, const int64_t* item_seq,
                        const float* order_w, const float* order_b,
                        const float* dist_w, const float* dist_b, const float* scalar,
                        int B, int L, int H, int dh,
                        int two_level, int combine_option, float comb_scalar, int rich_mode, const float* rich_ratio,
                        float p_attn, const float* D1, const float* D2, const float* D3, const float* noise,
                        const void* rng, uint32_t rng_stream,
                        float* ctx_att, float* ctx_cal, double* pen_sq, float* probs_out,
                        const int32_t* order, const int64_t* ctx_rows, void* stream);
/* backward of the same block.  d_ctx_att / d_ctx_cal [B,L,d] (either may be NULL == zero),
 * d_pen_sq device float[1] or NULL.  Outputs (written, not accumulated): d_mq,d_mk,d_mv,d_aq,d_ak [B,L,d].
 * Accumulated with atomics (caller zeroes): d_gate_logit [B,L,L], d_order_w [2dh], d_order_b [1],
 * d_dist_w [2dh], d_dist_b [1], d_scalar [1], d_rich_ratio [1] (NULL when the parameter is absent or when this
 * cotangent stream does not own it: the attacked-loss stream only trains the attack transforms, trainer.py:672-686). */
int acsr_attn_calib_bwd(const float* d_ctx_att, const float* d_ctx_cal, const float* d_pen_sq,
                        const float* mq, const float* mk, const float* mv, const float* aq, const float* ak,
                        const float* gate_logit, const int64_t* item_seq,
                        const float* order_w, const float* order_b,
                        const float* dist_w, const float* dist_b, const float* scalar,
                        int B, int L, int H, int dh,
                        int two_level, int combine_option, float comb_scalar, int rich_mode, const float* rich_ratio,
                        float p_attn, const float* D1, const float* D2, const float* D3, const float* noise,
                        const void* rng, uint32_t rng_stream,
                        float* d_mq, float* d_mk, float* d_mv, float* d_aq, float* d_ak,
                        float* d_gate_logit, float* d_order_w, float* d_order_b,
                        float* d_dist_w, float* d_dist_b, float* d_scalar, float* d_rich_ratio,
                        const int32_t* order, const int64_t* ctx_rows, void* stream);
/* the same backward for BOTH cotangent streams of the adversarial step in one launch (the reference's two
 * backward() traversals, trainer/trainer.py:672-684): stream 0 = d(calibrated loss) carries d_ctx_cal0 (+ d_pen_sq0),
 * stream 1 = d(attacked loss) carries d_ctx_att1 (last layer) OR d_ctx_cal1 (lower layers) and d_pen_sq1; any may be
 * NULL.  The row probabilities are recomputed once and shared.  Outputs are [2*B*L, .]: stream 1 writes B*L rows below
 * stream 0 in d_mq..d_ak and in d_gate_logit ([2*B*L, L]).  Parameter gradients (d_order_* .. d_rich_ratio) are taken
 * from stream 0 only: stream 1 trains nothing but the attack transforms. */
int acsr_attn_calib_bwd2(const float* d_ctx_cal0, const float* d_pen_sq0,
                         const float* d_ctx_att1, const float* d_ctx_cal1, const float* d_pen_sq1,
                         const float* mq, const float* mk, const float* mv, const float* aq, const float* ak,
                         const float* gate_logit, const int64_t* item_seq,
                         const float* order_w, const float* order_b,
                         const float* dist_w, const float* dist_b, const float* scalar,
                         int B, int L, int H, int dh,
                         int two_level, int combine_option, float comb_scalar, int rich_mode, const float* rich_ratio,
                         float p_attn, const float* D1, const float* D2, const float* D3, const float* noise,
                         const void* rng, uint32_t rng_stream,
                         float* d_mq, float* d_mk, float* d_mv, float* d_aq, float* d_ak,
                         float* d_gate_logit, float* d_order_w, float* d_order_b,
                         float* d_dist_w, float* d_dist_b, float* d_scalar, float* d_rich_ratio,
                        const int32_t* order, const int64_t* ctx_rows, void* stream);

/* ---- epilogue of the output projection and of the FFN: LN(dropout(h + bias) + res) ----
 * replaces model/layers.py:681-683 and 794-796 (bias add of the preceding nn.Linear folded in).
 * h,out [T,d]; bias [d] or NULL; res [res_rows,d] is read with period res_rows (res_rows == T for a plain call;
 * res_rows == T/2 when the attacked and calibrated branches are stacked and share the layer input). */
int acsr_bias_dropout_res_ln_fwd(const float* h, const float* bias, const float* res,
                                 const float* ln_w, const float* ln_b, float eps, int T, int d, int res_rows,
                                 float p, const float* mask, const void* rng, uint32_t rng_stream,
                                 float* out, float* stats, void* stream);
/* backward over T cotangent rows.  The saved forward tensors h/stats/mask repeat with period act_rows and res with
 * period res_rows (two stacked cotangent streams of one shared activation: act_rows = T/2); only rows
 * [0,param_rows) feed d_bias,d_ln_w,d_ln_b [d] (accumulated).  d_h (= grad of the GEMM output), d_res [T,d] written. */
int acsr_bias_dropout_res_ln_bwd(const float* d_out, const float* h, const float* bias, const float* res,
                                 const float* ln_w, const float* stats, int T, int d,
                                 int act_rows, int res_rows, int param_rows,
                                 float p, const float* mask, const void* rng, uint32_t rng_stream,
                                 float* d_h, float* d_res, float* d_bias, float* d_ln_w, float* d_ln_b, void* stream);

/* ---- FFN activation: out = act(h + bias)   (model/layers.py:776-792) -------------------
 * act: 0 gelu(erf) 1 relu 2 swish 3 tanh 4 sigmoid.  h,out [T,n].  Backward: h repeats with period act_rows,
 * rows [0,param_rows) feed d_bias. */
int acsr_bias_act_fwd(const float* h, const float* bias, int T, int n, int act, float* out, void* stream);
int acsr_bias_act_bwd(const float* d_out, const float* h, const float* bias, int T, int n, int act,
                      int act_rows, int param_rows, float* d_h, float* d_bias, void* stream);

/* ---- K9: gather the hidden state at position len-1 (abstract_recommender.py:130-134) ---
 * x_att (may be NULL), x_cal [B,L,d]; out [2B,d] rows [0,B) attacked, [B,2B) calibrated
 * (or [B,d] when x_att is NULL). */
int acsr_gather_last_fwd(const float* x_att, const float* x_cal, const int64_t* item_len,
                         int B, int L, int d, float* out, void* stream);
/* d_x_att/d_x_cal [B,L,d] must be zero-filled by the caller; rows len-1 are written. */
int acsr_gather_last_bwd(const float* d_out, const int64_t* item_len, int B, int L, int d,
                         float* d_x_att, float* d_x_cal, void* stream);

/* ---- K10/K12: full-catalogue logits out.E^T on tcgen05 tensor cores --------------------
 * replaces acsasrec.py:118-120 (logits + CrossEntropyLoss), 162-163 (full-sort scores),
 * trainer/trainer.py:941-942 + evaluator/collector.py:147-153 (scores[:,0]=-inf, topk, hit flags).
 * out [M,64] float32 (d must be 64 in ABI v1), table [V,64].  passes: 1 = TF32, 3 = 3xTF32
 * (hi/lo split, fp32-level accuracy).  All kernels are persistent over [m_tile(128), n_chunk];
 * n_chunks = acsr_logits_num_chunks(M, V).
 */
int acsr_logits_num_chunks(int M, int64_t V);
/* number of (max, sum exp) parts per row acsr_logits_ce_partial writes at hidden size d: the chunk plan above at d = 64; at every
 * other width the scores / CE / CE-gradient run on the K-streamed tcgen05 GEMM (acsr_gemm_batch, ACSR_EPI_CE*), one part per
 * 256-column block (d = 128 of config/yelp.yaml:39-42, d = 256 of BASELINE config #5).  Only the streaming top-k of a
 * catalogue too large for acsr_topk_select still takes the fp32 FMA kernel (logits_simt.cu) at d != 64. */
int acsr_logits_num_chunks_d(int M, int64_t V, int d);
/* scores [M, ldc] = out.E^T  (full_sort_predict, predict-all) */
int acsr_logits_store(const float* out, const float* table, int M, int64_t V, int d, int passes,
                      float* scores, int64_t ldc, void* stream);
/* CE forward: partial [M, n_chunks, 2] = (running max, sum exp) over this call's vocabulary
 * range; combine with acsr_ce_finalize (after an all-gather when vocab-sharded). */
int acsr_logits_ce_partial(const float* out, const float* table, int M, int64_t V, int d, int passes,
                           float* partial, void* stream);
/* combine partial (max, sumexp) pairs -> lse [M]; tgt_logit[m] = out[m].E[target[m]-idx_offset] as an
 * fp32 dot when the target row lives in this table shard (else 0; sum across shards);
 * row_loss[m] = lse - tgt_logit; loss[g] = mean of row_loss over each of n_groups groups of
 * M/n_groups consecutive rows (attacked rows first, calibrated second).  Warp per row, then one CTA for the means. */
int acsr_ce_finalize(const float* partial, int n_parts, const float* out, const float* table,
                     const int64_t* target, int M, int d, int64_t V, int64_t idx_offset, int n_groups,
                     float* lse, float* tgt_logit, float* row_loss, float* loss, void* stream);
/* scalar glue of the adversarial losses (acsasrec.py:129-142) in one launch: pen_l = sqrt(pen_sq[l]);
 * loss_attacked[0] = -ce_attacked[0] + w * mean_l pen_l ; d_pen_sq[l] = w / (2 n_layers pen_l) (NULL: skip).
 * w = mask_loss_weight[0] when the pointer is given (trainable_mask_loss_weight), else mask_loss_weight_value. */
int acsr_loss_combine(const double* pen_sq, int n_layers, const float* ce_attacked, const float* mask_loss_weight,
                      float mask_loss_weight_value, float* loss_attacked, float* d_pen_sq, void* stream);
/* acsr_ce_finalize + acsr_loss_combine in ONE launch (they sit on the training step's critical path): same outputs;
 * loss_attacked[0] = -loss[n_groups-1] + w * mean_l sqrt(pen_sq[l]) (the attacked rows are the last group); loss_attacked may
 * be NULL (then pen_sq / d_pen_sq are ignored).  counter: one uint32 in device memory, zero before the first call; the last
 * CTA to finish does the reductions and resets it. */
int acsr_ce_finalize_losses(const float* partial, int n_parts, const float* out, const float* table, const int64_t* target, int M, int d,
                            int64_t V, int64_t idx_offset, int n_groups, float* lse, float* tgt_logit, float* row_loss, float* loss,
                            const double* pen_sq, int n_layers, const float* mask_loss_weight, float mask_loss_weight_value,
                            float* loss_attacked, float* d_pen_sq, uint32_t* counter, void* stream);
/* CE backward part 1: Gt [V, ldg] (ldg >= M) = transpose of (exp(out.E^T - lse) - onehot(target)) * row_scale[m];
 * then d_E = Gt.out is a plain GEMM and d_out = Gt^T.E goes through acsr_linear_wgrad (reduction over V). */
int acsr_logits_ce_grad(const float* out, const float* table, const float* lse, const int64_t* target,
                        const float* row_scale, int M, int64_t V, int d, int passes,
                        float* Gt, int64_t ldg, void* stream);
/* CE backward WITHOUT the [M,V] gradient matrix (hidden size 64; the backward of acsasrec.py:117-121 as autograd runs it through
 * CrossEntropyLoss and the matmul with item_embedding.weight^T).  G = (exp(out.E^T - lse) - onehot(target)) * row_scale is
 * recomputed tile by tile on the tensor cores and consumed in registers by the thread that owns the logits row:
 *   acsr_ce_bwd_dout   : d_out [M,64]   += G . E        (critical path of the step)
 *   acsr_ce_bwd_dtable : d_table [V,64] += G^T . out    (nothing but the embedding scatter / optimizer consumes it)
 * Both ACCUMULATE into their output with vector reductions (clear it first); target[m] outside [0,V) = no one-hot in this
 * table (shard-local targets of the vocab-sharded path).  Other hidden sizes: ACSR_ERR_UNSUPPORTED (acsr_logits_ce_grad). */
int acsr_ce_bwd_dout(const float* out, const float* table, const float* lse, const int64_t* target, const float* row_scale, int M,
                     int64_t V, int d, int passes, float* d_out, void* stream);
int acsr_ce_bwd_dtable(const float* out, const float* table, const float* lse, const int64_t* target, const float* row_scale, int M,
                       int64_t V, int d, int passes, float* d_table, void* stream);
/* fused logits + streaming top-k: partial_val/partial_idx [M, n_chunks, k] (each chunk's k best, UNSORTED,
 * padded with -inf/-1); column 0 is excluded (trainer.py:942); idx_offset is added to indices (vocab shards). */
int acsr_logits_topk_partial(const float* out, const float* table, int M, int64_t V, int d, int passes,
                             int k, int64_t idx_offset, int skip_col0,
                             float* partial_val, int64_t* partial_idx, void* stream);
/* the same with a caller-owned scratch row_bound [2 * M * acsr_logits_num_chunks(M, V)] (int32, contents irrelevant): every warp set
 * of every CTA of a row tile publishes the best score of its own stream; once at least k streams have, the minimum of those (k or more different
 * items) is a lower bound of the row's overall k-th best, and scores at or below it never touch a candidate list.  Results are
 * identical (up to exact score ties).  row_bound == NULL, or fewer than k CTAs per row tile: acsr_logits_topk_partial. */
int acsr_logits_topk_partial_ws(const float* out, const float* table, int M, int64_t V, int d, int passes,
                                int k, int64_t idx_offset, int skip_col0,
                                float* partial_val, int64_t* partial_idx, int32_t* row_bound, void* stream);
/* merge n_parts partial lists per row (any order) -> topk_val [M,k], topk_idx [M,k] int64 and, when
 * positive != NULL, rec_topk [M,k+1] int32 = hit flags + pos_len(=1) (collector.py:148-153). */
int acsr_topk_merge(const float* partial_val, const int64_t* partial_idx, int M, int n_parts, int k,
                    const int64_t* positive, float* topk_val, int64_t* topk_idx, int32_t* rec_topk, void* stream);

/* ---- rank counts of the positive for GAUC (evaluator/metrics.py GAUC, collector.py rec.meanrank) ----
 * The reference sorts the whole [B, V] score matrix to find the positive's average rank.  Here the top-k kernels count, per row,
 * G = #items scoring strictly above s_pos and E = #items scoring equal to it, column 0 (when skipped) and the positive's own column
 * excluded, so the counts do not depend on how a path rounds the positive's own score.  s_pos = pos_score[m] comes from
 * acsr_row_dot (one fp32 dot in a fixed order, as the CE target logit); the 1-based average rank is G + (E + 2) / 2.
 * acsr_row_dot: dot[m] = out[m] . table[ids[m] - idx_offset] when 0 <= ids[m] - idx_offset < V, else 0 (the shards' answers sum). */
int acsr_row_dot(const float* out, const float* table, const int64_t* ids, int M, int d, int64_t V, int64_t idx_offset, float* dot,
                 void* stream);
/* acsr_logits_topk_partial_ws that also writes partial_counts [M, acsr_logits_num_chunks(M, V), 2] int32 = (G, E) of each chunk
 * (zero for the lists no CTA produces); positive [M] = item ids (idx_offset is subtracted, as for the output ids).  Plain stores:
 * deterministic.  Every score is counted, including tiles the shared bound lets skip the candidate bookkeeping. */
int acsr_logits_topk_rank_partial(const float* out, const float* table, int M, int64_t V, int d, int passes, int k, int64_t idx_offset,
                                  int skip_col0, const int64_t* positive, const float* pos_score, float* partial_val,
                                  int64_t* partial_idx, int32_t* partial_counts, int32_t* row_bound, void* stream);
/* acsr_topk_merge that also sums partial_counts [M, n_count_parts, 2] into counts [M, 2]; positive may be NULL (no rec_topk). */
int acsr_topk_merge_rank(const float* partial_val, const int64_t* partial_idx, int M, int n_parts, int k,
                         const int64_t* positive, const int32_t* partial_counts, int n_count_parts, float* topk_val,
                         int64_t* topk_idx, int32_t* rec_topk, int32_t* counts, void* stream);

/* dense variant for catalogues of at most acsr_topk_select_max_items() items (one row's scores as 32-bit keys in shared
 * memory): top-k of every row of scores [M, ld] (first V columns) by a 4-pass radix select + a sort of the k winners.
 * skip_col0 excludes column 0 (trainer.py:942); item id = column + idx_offset.  Together with acsr_logits_store this is the
 * full-sort evaluation of small catalogues (the scores stay L2-resident); the fused acsr_logits_topk_partial path is for
 * large / sharded ones. */
int acsr_topk_select_max_items(void);
int acsr_topk_select(const float* scores, int M, int64_t V, int64_t ld, int k, int skip_col0, int64_t idx_offset,
                     const int64_t* positive, float* topk_val, int64_t* topk_idx, int32_t* rec_topk, void* stream);
/* acsr_topk_select that also counts counts [M, 2] = (G, E) against pos_score over the row in shared memory (see acsr_row_dot);
 * positive is required (its column, id - idx_offset, is not counted). */
int acsr_topk_select_rank(const float* scores, int M, int64_t V, int64_t ld, int k, int skip_col0, int64_t idx_offset,
                          const int64_t* positive, const float* pos_score, float* topk_val, int64_t* topk_idx, int32_t* rec_topk,
                          int32_t* counts, void* stream);

/* Fold the attack transforms into the first projections (layers.py:658-659, 687-689) so that the five projections of a layer
 * read the same input and run as ONE batched GEMM: out_W [5,d,d] / out_b [5,d] = {Wq, Wk, Wv, Waq.Wq, Wak.Wk} and
 * {bq, bk, bv, Waq.bq + baq, Wak.bk + bak}.  Wqkv [3,d,d], bqkv [3,d], Waqk [2,d,d], baqk [2,d] (row-major [out,in]). */
int acsr_fold_attack_weights(const float* Wqkv, const float* bqkv, const float* Waqk, const float* baqk, int d, float* out_W,
                             float* out_b, void* stream);

/* ---- encoder GEMMs on tcgen05 with the token rows on the UMMA M axis (3xTF32, fp32-level accuracy) ----
 * replaces the nn.Linear forward / input-gradient GEMMs of model/layers.py:658-659, 680, 687-689, 791-794, 887.
 * Y[r, n] (+)= sum_k X(r,k) * W(n,k) + bias[n], r < rows, n < N, k < K <= 256, with strided operands so that
 * transposed weights (input gradients) and K-concatenated inputs need no copies:
 *   X(r,k) = X[(k/64)*x_kblock_stride + r*ldx + k%64]
 *   W(n,k) = W[(k/64)*w_kblock_stride + n*w_stride_n + (k%64)*w_stride_k]
 * batch > 1 launches independent problems (pointer + b*stride_*).  bias NULL or [N]; accumulate != 0 adds to Y. */
int acsr_linear_tok(const float* X, int64_t ldx, int64_t x_kblock_stride, int64_t rows, int K,
                    const float* W, int64_t w_stride_n, int64_t w_stride_k, int64_t w_kblock_stride, int N,
                    const float* bias, int accumulate, float* Y, int64_t ldy,
                    int batch, int64_t stride_x, int64_t stride_w, int64_t stride_bias, int64_t stride_y,
                    int passes, void* stream);
/* projection + bias + dropout + residual + LayerNorm fused (model/layers.py:680-683, 793-796), output width 64:
 * HZ = X.W^T (saved for the backward), out = LN(dropout(HZ + bias) + res[r % res_rows]), stats[r] = (mean, rstd).
 * Dropout masks use the same Philox counters as acsr_bias_dropout_res_ln_{fwd,bwd}, which stays the backward. */
int acsr_linear_tok_bdrl(const float* X, int64_t ldx, int64_t rows, int K, const float* W, const float* bias,
                         const float* res, int64_t res_rows, const float* ln_w, const float* ln_b, float eps,
                         float p_drop, const float* mask, const void* rng, uint32_t rng_stream,
                         float* HZ, float* out, float* stats, int passes, void* stream);
/* input gradient of a layer's projections in ONE launch (backward of model/layers.py:658-659, 687-689, 887), hidden size d = 64:
 *   d_mq_tot = d_mq + d_aq.Waq (+ d_gl.Wg) ; d_mk_tot = d_mk + d_ak.Wak ; d_x[r] += d_mq_tot.Wq + d_mk_tot.Wk + d_mv.Wv,  r < rows
 * (the three acsr_linear_tok launches d_qkv[0:2] += d_aqk.Waqk, d_mq += d_gl.Wg, d_x += d_qkv.Wqkv).  d_qkv [3, plane_rows, 64] =
 * (d_mq, d_mk, d_mv), d_aqk [2, plane_rows, 64] = (d_aq, d_ak); rows r < rows_keep of d_mq_tot / d_mk_tot are written back into
 * d_qkv[0] / d_qkv[1], the others are left as they were.  d_gl [plane_rows, L] and Wg [L, 64] (L <= 64) are both NULL without
 * the gate.  Wqkv [3,64,64], Waqk [2,64,64] row-major [out, in]; d_x [rows, 64] already holds the residual-path gradient. */
int acsr_proj_input_grad(float* d_qkv, const float* d_aqk, int64_t plane_rows, const float* d_gl, int L, const float* Wqkv,
                         const float* Waqk, const float* Wg, int d, int64_t rows, int64_t rows_keep, float* d_x, int passes,
                         void* stream);

/* ---- token-parallel linear layer on tcgen05 (3xTF32):  Y[rows, N] (+)= X[rows, K] . Wt^T + bias,  K == 64 (ABI v1).
 * replaces the forward nn.Linear calls at layers.py:658-659, 680, 687-689, 791 and their input-gradient GEMMs.
 * The stationary operand is addressed as Wt[n][k] = W[n*w_stride_n + k*w_stride_k]: (K,1) for y = x.W^T with W [N,K]
 * row-major, (1,ldw) for dx = dy.W.  accumulate != 0 adds into Y.  `batch` independent problems per launch with
 * float strides stride_x/w/bias/y (stacked Q/K/V).  X rows must be contiguous (row pitch K). */
int acsr_linear_tc(const float* X, int64_t rows, int K, const float* W, int N, int64_t w_stride_n, int64_t w_stride_k,
                   const float* bias, int accumulate, float* Y, int64_t ldy, int batch, int64_t stride_x, int64_t stride_w,
                   int64_t stride_bias, int64_t stride_y, int passes, void* stream);

/* ---- weight / bias gradient of a token-parallel linear layer (backward of the nn.Linear calls in
 * layers.py:658-659, 687-689, 680, 791-794, 887):  dW[N,K] += dY[T,N]^T . X[T,K],  db[N] += sum_t dY[t,:]
 * (db may be NULL).  Accumulates with atomics: the caller zeroes or passes its gradient buffer. */
int acsr_linear_wgrad(const float* dY, const float* X, int T, int N, int K, float* dW, float* db, void* stream);
/* `batch` independent problems in one launch; problem z uses dY + z*stride_dy, X + z*stride_x (0 = shared input),
 * dW + z*stride_dw, db + z*stride_db (strides in floats).  Used for the stacked Q/K/V and attack-Q/K projections. */
int acsr_linear_wgrad_batched(const float* dY, const float* X, int T, int N, int K, float* dW, float* db, int batch,
                              int64_t stride_dy, int64_t stride_x, int64_t stride_dw, int64_t stride_db, void* stream);

/* ---- general encoder GEMM on tcgen05 (3xTF32), any hidden size: K streamed in 32-wide slabs, up to 16 problems per launch ----
 * replaces EVERY nn.Linear forward, input-gradient and weight-gradient GEMM of model/layers.py:658-659, 680, 687-689,
 * 791-794, 887 (and their autograd backward) for hidden sizes the width-64 kernels above do not cover (d = 128 of
 * config/yelp.yaml:39-42, amazon-sports-outdoors.yaml:31-34, amazon-toys-games.yaml:29-32; d = 256 of BASELINE config #5).
 *   C[m, n] (+)= sum_k A(m,k) * B(n,k)        m < M, n < N, k < K
 *   A(m,k) = A[(k / a_kblk) * a_kb_stride + m * a_row_stride + (k % a_kblk) * a_k_stride]      (B alike; strides in floats)
 * so transposed operands (input gradients: B = W^T; weight gradients: A = dY^T, B = X^T with the token axis on K) and
 * K-concatenated inputs need no copies.  a_kblk / b_kblk: multiples of 4 (or >= K when the operand is one block).
 * Epilogues (thread-per-row out of TMEM):
 *   ACSR_EPI_STORE  C = acc + bias (accumulate != 0: C += ...)
 *   ACSR_EPI_ATOMIC C += acc with vector atomics; the K range is cut into k_splits work items (0 = chosen by the library);
 *                   colsum[m] += sum_k A(m,k) when colsum != NULL (the bias gradient of a weight-gradient problem; needs
 *                   a_k_stride != 1, i.e. the transposed-operand form)
 *   ACSR_EPI_ACT    C = acc (saved for the backward), C2 = act(acc + bias)                       layers.py:776-792
 *   ACSR_EPI_BDRL   C = acc (may be NULL), out = LayerNorm(dropout(acc + bias) + res[m % res_rows]), stats[m] = (mean, rstd);
 *                   N <= 256 and a multiple of 4                                                 layers.py:681-683, 794-796 */
#define ACSR_EPI_STORE 0
#define ACSR_EPI_ATOMIC 1
#define ACSR_EPI_ACT 2
#define ACSR_EPI_BDRL 3
/* full-catalogue logits at any hidden size (model/sequential_recommender/acsasrec.py:118-120; rows of `out` on M, table rows on N):
 *   ACSR_EPI_CE      C2 = partial [M, acsr_gemm_ce_parts(N), 2]: (max, sum exp) of every 256-column block, for acsr_ce_finalize
 *   ACSR_EPI_CE_GRAD C = Gt [N, ldc >= M] = ((softmax - onehot(target)) * row_scale)^T with lse = res [M], row_scale = ln_w [M],
 *                    target = rng (int64 [M]) */
#define ACSR_EPI_CE 4
#define ACSR_EPI_CE_GRAD 5
#define ACSR_GEMM_MAX_PROBLEMS 16
typedef struct acsr_gemm_problem {
  const float* A; int64_t a_row_stride; int64_t a_k_stride; int64_t a_kb_stride;
  const float* B; int64_t b_row_stride; int64_t b_k_stride; int64_t b_kb_stride;
  float* C; int64_t ldc;
  int64_t M;
  const float* bias;
  float* colsum;
  float* C2;
  const float* res; int64_t res_rows;
  const float* ln_w; const float* ln_b;
  const float* mask; const void* rng;
  float* out; float* stats;
  int32_t a_kblk; int32_t b_kblk;
  int32_t N; int32_t K;
  int32_t epilogue; int32_t accumulate; int32_t k_splits; int32_t act;
  uint32_t rng_stream; float eps; float p_drop; int32_t reserved;
} acsr_gemm_problem;
int acsr_gemm_batch(const acsr_gemm_problem* problems, int n_problems, int passes, void* stream);
int acsr_gemm_ce_parts(int64_t V);

/* ---- the last encoder layer after its attention, on the rows that feed the losses (one launch per direction) ----
 * Replaces, for hidden size 64 and inner size <= 256 (multiple of 16), the chain the reference runs on all T rows although only
 * position len-1 of every sequence reaches the loss (abstract_recommender.py:130-134 gather_indexes after layers.py:676-684 and
 * layers.py:790-798): gather -> dense + dropout + residual + LayerNorm -> FeedForward (dense_1, activation, dense_2, dropout,
 * residual, LayerNorm).  Rows [0,B) come from ctx_first (calibrated), rows [B,2B) from ctx_second (attacked; NULL: B rows only);
 * x [T,64] is the layer input (residual).  Saved for the backward, same meaning as in the unfused path: c_ctx [C,64], c_x [B,64],
 * hz / z2 = GEMM outputs before bias, st_a / st_f = (mean, rstd) [C,2], h, z1 / a1 [C,I], out [C,64].  Dropout: explicit masks
 * [C,64] or Philox streams stream_a / stream_f with the counters of acsr_bias_dropout_res_ln_fwd. */
int acsr_tail_fwd(const float* ctx_first, const float* ctx_second, const float* x, const int64_t* item_len, int B, int L, int d, int I,
                  int act, const float* Wo, const float* bo, const float* lnA_w, const float* lnA_b, float epsA, const float* W1,
                  const float* b1, const float* W2, const float* b2, const float* lnF_w, const float* lnF_b, float epsF, float p_drop,
                  const float* mask_a, const float* mask_f, const void* rng, uint32_t stream_a, uint32_t stream_f, float* c_ctx,
                  float* c_x, float* hz, float* st_a, float* h, float* z1, float* a1, float* z2, float* st_f, float* out, void* stream);
/* backward of acsr_tail_fwd over C = n_groups * B cotangent rows d_out [C,64]: writes d_z2, d_hz [C,64] and d_z1 [C,I] (the
 * left operands of the three weight-gradient reductions), scatters the gradients of the attention context and of the layer input
 * to position len-1 of the token-major buffers d_ctx_* / d_x_* [T,64] (cleared by the caller), and ACCUMULATES the bias /
 * LayerNorm gradients from rows [0,B) (the calibrated stream owns the parameters, trainer.py:672-686). */
int acsr_tail_bwd(const float* d_out, const int64_t* item_len, int B, int L, int d, int I, int act, int n_groups, const float* c_x,
                  const float* hz, const float* st_a, const float* h, const float* z1, const float* z2, const float* st_f,
                  const float* Wo, const float* bo, const float* lnA_w, const float* W1, const float* b1, const float* W2,
                  const float* b2, const float* lnF_w, float p_drop, const float* mask_a, const float* mask_f, const void* rng,
                  uint32_t stream_a, uint32_t stream_f, float* d_z2, float* d_z1, float* d_hz, float* d_x_first, float* d_x_second,
                  float* d_ctx_first, float* d_ctx_second, float* g_bo, float* g_lnA_w, float* g_lnA_b, float* g_b1, float* g_b2,
                  float* g_lnF_w, float* g_lnF_b, void* stream);

/* ---- backward of an encoder layer's dense part after its attention (layers.py:676-684, 790-798) as ONE tcgen05 kernel (hidden
 * size 64, inner size a multiple of 64 up to 256), the chain of two acsr_bias_dropout_res_ln_bwd calls, acsr_bias_act_bwd and
 * three input-gradient GEMMs:
 *   d_pre_f = LN_f backward of d_out ; d_z2 = d_pre_f * mask_f ; d_z1 = (d_z2.W2) * act'(z1 + b1) ; d_h = d_pre_f + d_z1.W1 ;
 *   d_xres = LN_a backward of d_h ; d_hz = d_xres * mask_a ; d_ctx = d_hz.Wo
 * with the argument meaning of those calls: `rows` cotangent rows; the saved tensors z2, h, st_f, z1 [., I], hz, st_a (and the
 * explicit masks [., 64]) repeat with period act_rows, x_res with period res_rows; rows < param_rows feed the parameter gradients.
 * `ops` = the weights pre-split by acsr_dense_bwd_prep (acsr_dense_bwd_prep_floats(I) floats).  Writes d_xres and d_ctx
 * [rows, 64] (overwritten) and rows < param_rows of d_z2, d_hz [., 64] and d_z1 [., I]; ADDS the LayerNorm weight / bias gradients
 * of both norms into g_ln*.  The bias gradients of dense_2, dense_1 and the out-projection are left to the weight-gradient launch
 * (column sums of d_z2, d_z1, d_hz).  Dropout: masks or Philox streams as acsr_bias_dropout_res_ln_bwd. */
int64_t acsr_dense_bwd_prep_floats(int I);
int acsr_dense_bwd_prep(const float* Wo, const float* W1, const float* W2, int d, int I, float* ops, void* stream);
int acsr_dense_bwd(const float* d_out, int64_t rows, int64_t act_rows, int64_t res_rows, int64_t param_rows, int d, int I, int act,
                   const float* ops, const float* z2, const float* b2, const float* h, const float* lnF_w, const float* st_f,
                   const float* z1, const float* b1, const float* hz, const float* bo, const float* x_res, const float* lnA_w,
                   const float* st_a, float p_drop, const float* mask_a, const float* mask_f, const void* rng, uint32_t stream_a,
                   uint32_t stream_f, float* d_z2, float* d_z1, float* d_hz, float* d_xres, float* d_ctx, float* g_lnF_w,
                   float* g_lnF_b, float* g_lnA_w, float* g_lnA_b, int passes, void* stream);

/* ---- loss_type BPR (model/sequential_recommender/acsasrec.py:109-116, model/loss.py:21-47) ----
 * x_m = out_m . (E[pos_m] - E[neg_m]); row_loss[m] = -log(gamma + sigmoid(x_m)); loss[g] = mean over row group g
 * (M rows in n_groups equal groups: [calibrated ; attacked] in the fused step).  row_x [M] is saved for the backward. */
int acsr_bpr_loss_fwd(const float* out, const float* table, const int64_t* pos_items, const int64_t* neg_items, int M, int d,
                      int n_groups, float gamma, float* row_x, float* row_loss, float* loss, void* stream);
/* d_out[m] = row_scale[m] * dloss/dx_m * (E[pos_m] - E[neg_m]) (may be NULL); rows m in [table_row_begin, table_row_end)
 * scatter +-row_scale[m] * dloss/dx_m * out_m into d_table rows pos_m / neg_m with atomics (d_table may be NULL). */
int acsr_bpr_loss_bwd(const float* out, const float* table, const int64_t* pos_items, const int64_t* neg_items, const float* row_x,
                      const float* row_scale, int M, int d, float gamma, int table_row_begin, int table_row_end, float* d_out,
                      float* d_table, void* stream);
/* the same over a vocab-sharded table (dist.VocabParallel): this rank holds rows [lo, hi) of the V-row table as shard[0, hi-lo).
 * acsr_bpr_dots_shard: dots [M, 2] = (out_m . E[pos_m], out_m . E[neg_m]) for owned ids, 0 for the others, in acsr_bpr_loss_fwd's
 * arithmetic: summed over ranks, the dots are acsr_bpr_loss_fwd's two scores bit for bit.  acsr_bpr_loss_from_dots: row_x,
 * row_loss and loss of acsr_bpr_loss_fwd from the summed dots.  acsr_bpr_loss_bwd_shard: acsr_bpr_loss_bwd with the rows of
 * unowned ids read as 0 in d_out (the ranks' d_out sum to g * (E[pos] - E[neg])) and only owned ids scattered into d_shard_grad
 * (rows [0, hi-lo)). */
int acsr_bpr_dots_shard(const float* out, const float* shard, int64_t lo, int64_t hi, int64_t V, const int64_t* pos_items,
                        const int64_t* neg_items, int M, int d, float* dots, void* stream);
int acsr_bpr_loss_from_dots(const float* dots, int M, int n_groups, float gamma, float* row_x, float* row_loss, float* loss,
                            void* stream);
int acsr_bpr_loss_bwd_shard(const float* out, const float* shard, int64_t lo, int64_t hi, int64_t V, const int64_t* pos_items,
                            const int64_t* neg_items, const float* row_x, const float* row_scale, int M, int d, float gamma,
                            int table_row_begin, int table_row_end, float* d_out, float* d_shard_grad, void* stream);

/* ---- vocab-sharded item table (north_star; the reference has only the dense nn.Embedding of acsasrec.py:37) ----
 * this rank stores table rows [row_lo, row_hi).  gather: out[i] = shard[ids[i] - row_lo] when the row is owned, else 0 (the owners'
 * answers are summed by a reduce-scatter, so every token gets its row from exactly one rank).  scatter_add: shard_grad[ids[i] -
 * row_lo] += rows[i] for owned ids != 0 (row 0 is nn.Embedding's padding_idx: no gradient through the gather). */
int acsr_shard_gather_rows(const int64_t* ids, int64_t n, const float* shard, int64_t row_lo, int64_t row_hi, int d, float* out,
                           void* stream);
int acsr_shard_scatter_add_rows(const int64_t* ids, int64_t n, const float* rows, int64_t row_lo, int64_t row_hi, int d,
                                float* shard_grad, void* stream);

/* ---- device-resident training data (SURVEY section 8 f-2) ----
 * replaces the per-epoch CPU shuffle + host slicing + per-step host->device copy of data/interaction.py:293-297,
 * data/dataloader/general_dataloader.py:62-65 and trainer/trainer.py:661.  seqs [n_rows, L], lens / targets / negs [n_rows]
 * (negs may be NULL) and the epoch permutation perm [n_rows] live in device memory; the batch cursor[0] (rows perm[cursor*B ..
 * cursor*B + B)) is written in the packed layout [item_id_list | item_length | item_id | neg_item_id] of the captured step's
 * static input buffer.  acsr_cursor_advance: cursor[0] += 1 (a second node of the captured step). */
int acsr_batch_gather(const int64_t* seqs, const int64_t* lens, const int64_t* targets, const int64_t* negs, const int64_t* perm,
                      const int64_t* cursor, int64_t n_rows, int B, int L, int64_t* out_packed, void* stream);
int acsr_cursor_advance(int64_t* cursor, void* stream);

/* ---- negative sampling and sampled-candidate ranking (negsample.cu) ----
 * acsr_neg_sample replaces recbole/sampler/sampler.py sample_by_user_ids (RecBole 1.0.1's non-repeatable Sampler, as called by
 * data/dataloader/general_dataloader.py for `neg_sampling` and for `eval_args.mode: uniN / popN`).  negs[m * ld_negs + j],
 * j < N, is a negative for row m: an item of [1, n_items) outside the user's used set used_items[used_offsets[u] ..
 * used_offsets[u+1]) (sorted ascending, unique, per user id u = users[row]) and != positives[row] (positives may be NULL).
 * Uniform (alias_prob == NULL): exactly uniform over that complement, one draw and a binary search per negative.  Popularity
 * (alias_prob [n_items] float32 / alias_idx [n_items] int64, a Walker alias table of the item counts): alias draws rejected
 * while they hit the excluded set, at most 16 per negative, after which the uniform-complement draw is taken.  Draws are with
 * replacement and keyed by Philox4x32-10 (rng->seed, rng->step, rng_stream, row * N + j): advance rng with acsr_rng_advance
 * for fresh draws.  With perm / cursor (both or neither), row m reads users / positives at perm[cursor[0] * M + m] of n_rows
 * rows -- the batch acsr_batch_gather writes, when launched between it and acsr_cursor_advance.  A user id outside [0, n_users)
 * or a user whose complement is empty gets item 0 (never a valid draw).  Graph-capturable. */
int acsr_neg_sample(const int64_t* users, const int64_t* positives, const int64_t* perm, const int64_t* cursor, int64_t n_rows, int M,
                    int N, const int64_t* used_offsets, const int64_t* used_items, int64_t n_users, int64_t n_items,
                    const float* alias_prob, const int64_t* alias_idx, const void* rng, uint32_t rng_stream, int64_t* negs,
                    int64_t ld_negs, void* stream);
/* acsr_candidate_rank replaces trainer/trainer.py _neg_sample_batch_eval (predict on the repeated interaction, scatter into a
 * -inf [B, n_items] matrix) and evaluator/collector.py eval_batch_collect (topk + hit flags) for sampled evaluation.
 * cand [M, n_cand] int64, column 0 the positive; scores[m, c] = out[m] . table[cand[m, c]] in fp32 (out [M, d], table [V, d],
 * d a multiple of 4 up to 1024; scores may be NULL).  rank = number of DISTINCT candidates c >= 1 whose score is strictly
 * greater than the positive's (duplicates collapse as in the scattered matrix; ties count for the positive).
 * rec [M, kmax+1] int32: rec[m, rank] = 1 when rank < kmax, rec[m, kmax] = 1 (pos_len), else 0.
 * n_cand <= acsr_candidate_rank_max_candidates() (8192) and kmax <= 1024, else ACSR_ERR_UNSUPPORTED. */
int acsr_candidate_rank_max_candidates(void);
int acsr_candidate_rank(const float* out, const float* table, int64_t V, int d, const int64_t* cand, int M, int n_cand, int kmax,
                        int32_t* rec, float* scores, void* stream);
/* the same plus counts [M, 3] int32 = (distinct negatives scoring above the positive, distinct negatives tied with it, distinct
 * candidates including the positive): GAUC's rank inputs and user_len, the number of finite entries of the scattered row. */
int acsr_candidate_rank_counts(const float* out, const float* table, int64_t V, int d, const int64_t* cand, int M, int n_cand, int kmax,
                               int32_t* rec, float* scores, int32_t* counts, void* stream);
/* acsr_candidate_rank split in two for a vocab-sharded table (dist.VocabParallel).  acsr_candidate_scores_shard: scores[m, c] =
 * out[m] . shard[id - lo] where id = cand[m, c] clamped to [0, V) lies in this rank's rows [lo, hi), else 0; each owned score is
 * bit for bit the one acsr_candidate_rank computes on the full table, so the sum over ranks is exact.  acsr_candidate_rank_scores:
 * the ranking of acsr_candidate_rank (counts == NULL) or acsr_candidate_rank_counts on precomputed scores [M, n_cand]. */
int acsr_candidate_scores_shard(const float* out, const float* shard, int64_t lo, int64_t hi, int64_t V, int d, const int64_t* cand,
                                int M, int n_cand, float* scores, void* stream);
int acsr_candidate_rank_scores(const float* scores, const int64_t* cand, int64_t V, int M, int n_cand, int kmax, int32_t* rec,
                               int32_t* counts, void* stream);

/* ---- K13: fused Adam over one flat fp32 buffer (trainer/trainer.py:614-615,687) ---------
 * torch.optim.Adam semantics (no amsgrad); step_count device int64[1], incremented by the call. */
int acsr_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                   float lr, float beta1, float beta2, float eps, float weight_decay,
                   int64_t* step_count, void* stream);

/* ---- gradient clipping by global norm (trainer.py `clip_grad_norm`: torch.nn.utils.clip_grad_norm_) -----------------------
 * acsr_grad_norm_partial: out[0] = the fp64 sum of |g|^q over grad[ranges[2r] .. ranges[2r+1]) for r < n_ranges (q = norm_type,
 * a positive number; q = 1 and 2 need no pow), or max |g| for q = inf.  NaN and Inf propagate.  grad holds n floats; ranges is
 * a HOST array of 2 * n_ranges int64 (1 <= n_ranges <= 8, 0 <= begin <= end <= n; no alignment needed).  block_partials: scratch of
 * acsr_grad_norm_max_blocks() doubles; counter: one uint32 in device memory, zero before the first call and reset by the last
 * CTA, which combines the per-CTA partials in a fixed order: bit-identical from run to run and under graph replay.
 * acsr_adam_step_clipped: acsr_adam_step on grad * coef with coef = min(1, max_norm / (total + 1e-6)) (NaN propagates), where
 * total = (sum of partials[0 .. n_partials) in index order)^(1/q), or their max for q = inf -- partials of disjoint ranges
 * of acsr_grad_norm_partial, e.g. the replicated part of the buffer and every rank's item-table shard.  The clipped gradient
 * is written back to grad and total_out[0] receives the norm (fp32, the value clip_grad_norm_ returns).  max_norm > 0,
 * 1 <= n_partials <= 1024. */
int acsr_grad_norm_max_blocks(void);
int acsr_grad_norm_partial(const float* grad, int64_t n, const int64_t* ranges, int n_ranges, double norm_type,
                           double* block_partials, uint32_t* counter, double* out, void* stream);
int acsr_adam_step_clipped(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                           float beta2, float eps, float weight_decay, int64_t* step_count, const double* partials, int n_partials,
                           double norm_type, float max_norm, float* total_out, void* stream);

/* ---- ACTiSASRec (SURVEY section 8 f-4): time-interval aware keys / values ----------------------------------------------
 * replaces model/sequential_recommender/actisasrec.py:104-124, 146-155 and the time-aware terms of
 * model/transformer_layers.py:1085-1091 (context) and 1116-1134 (scores).  The reference gathers two [B,L,L,d] tensors
 * (time_matrix_emb_K/V[t_ij]) and drops them out element-wise; here they never exist.  With the pair embedding
 *     E[b,i,j,c] = P[j,c]*Dp[b,j,c] + T[tmat[b,i,j],c]*Dt[b,i,j,c]
 * (P [L,d] absolute-position table, T [span1,d] interval table, span1 = time_span + 1, Dp / Dt inverted-dropout multipliers:
 * explicit tensors [B,L,d] / [B,L,L,d], or Philox streams stream_p / stream_t of `rng`, or none when p == 0):
 *   acsr_time_matrix   tmat[b,i,j] = (int) min(|ts[b,i] - ts[b,j]|, time_span)        (actisasrec.py:146-155, fp32 like the field)
 *   acsr_pair_score    s[b,h,i,j]  = sum_{c in head h} x[b,i,c] * E[b,i,j,c]          (x = mixed query: the score bias;
 *                                                                                      x = d context: d of the attention matrix)
 *   acsr_pair_context  y[b,i,c] (+)= sum_j prob[b,h(c),i,j] * E[b,i,j,c]              (prob = attention: the context term;
 *                                                                                      prob = d bias: d of the mixed query)
 *   acsr_pair_wgrad    dP[j,c] += sum_{b,i} a[b,h,i,j]*v[b,i,c]*Dp[b,j,c];  dT[t,c] += sum_{tmat=t} a*v*Dt     (row 0 of both
 *                      tables is nn.Embedding's padding_idx, actisasrec.py:55-58: no gradient)
 * causal != 0: pairs j > i are written as 0 without being computed.  L <= 64, head size a multiple of 4. */
int acsr_time_matrix(const float* time_seq, int B, int L, int time_span, int32_t* tmat, void* stream);
int acsr_pair_score(const float* x, const float* P, const float* T, const int32_t* tmat, int B, int L, int H, int dh, int span1,
                    float p, const float* Dp, const float* Dt, const void* rng, uint32_t stream_p, uint32_t stream_t, int causal,
                    float* s_out, void* stream);
int acsr_pair_context(const float* prob, const float* P, const float* T, const int32_t* tmat, int B, int L, int H, int dh, int span1,
                      float p, const float* Dp, const float* Dt, const void* rng, uint32_t stream_p, uint32_t stream_t,
                      int accumulate, float* y, void* stream);
int acsr_pair_wgrad(const float* a, const float* v, const int32_t* tmat, int B, int L, int H, int dh, int span1,
                    float p, const float* Dp, const float* Dt, const void* rng, uint32_t stream_p, uint32_t stream_t,
                    float* dP, float* dT, void* stream);
/* the fused attention of acsr_attn_calib_fwd / _bwd (ACSR_ATTN_PLAIN, L <= 64) around those terms: s_bias [B,H,L,L] is added to
 * the raw scores q_i.k_j before the calibrators (transformer_layers.py:1134); prob_att / prob_cal [B,H,L,L] receive the attacked
 * and the final calibrated attention (every entry written).  Backward: d_prob_att / d_prob_cal are the cotangents of those two
 * matrices (NULL == zero), d_s_bias [B,H,L,L] receives the gradient of the bias where a row's chain runs (caller zero-fills). */
int acsr_attn_calib_ti_fwd(const float* s_bias, const float* mq, const float* mk, const float* mv, const float* aq,
                           const float* ak, const float* gate_logit, const int64_t* item_seq, const float* order_w,
                           const float* order_b, const float* dist_w, const float* dist_b, const float* scalar, int B,
                           int L, int H, int dh, int two_level, int combine_option, float comb_scalar, int rich_mode,
                           const float* rich_ratio, float p_attn, const float* D1, const float* D2, const float* D3,
                           const float* noise, const void* rng, uint32_t rng_stream, float* ctx_att, float* ctx_cal,
                           double* pen_sq, float* prob_att, float* prob_cal, void* stream);
int acsr_attn_calib_ti_bwd(const float* d_ctx_att, const float* d_ctx_cal, const float* d_pen_sq, const float* d_prob_att,
                           const float* d_prob_cal, const float* s_bias, const float* mq, const float* mk,
                           const float* mv, const float* aq, const float* ak, const float* gate_logit, const int64_t* item_seq,
                           const float* order_w, const float* order_b, const float* dist_w, const float* dist_b, const float* scalar,
                           int B, int L, int H, int dh, int two_level, int combine_option, float comb_scalar, int rich_mode,
                           const float* rich_ratio, float p_attn, const float* D1, const float* D2, const float* D3,
                           const float* noise, const void* rng, uint32_t rng_stream, float* d_mq, float* d_mk, float* d_mv,
                           float* d_aq, float* d_ak, float* d_gate_logit, float* d_order_w, float* d_order_b, float* d_dist_w,
                           float* d_dist_b, float* d_scalar, float* d_rich_ratio, float* d_s_bias, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ACSR_H_ */
