/*
 * fedfr_b200 -- C ABI of the B200 (sm_100a) PartialFC CosFace / FedAvg hot path.
 *
 * This is the drop-in boundary.  The reference (jackie840129/FedFR) is pure Python; the functions
 * below are what its hot path binds to through ctypes (see INTEGRATION.md for the stub a reference
 * maintainer would add).  Each entry cites the reference lines it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only, no torch types; every pointer is a DEVICE pointer unless the
 *     name ends in _host;
 *   - every function enqueues on `stream` (a cudaStream_t passed as void*) and returns without
 *     synchronising unless stated;
 *   - return value: 0 = ok, < 0 = bad argument / unsupported shape / wrong GPU (see PFC_E_*),
 *     > 0 = a cudaError_t.  pfc_last_error() returns a thread-local message for the last failure;
 *   - row-major, dense tensors.  `emb` is the embedding size E (reference default 512).
 *   - there is NO CPU fallback anywhere: without an sm_100 device every compute entry fails.
 */
#ifndef FEDFR_B200_H_
#define FEDFR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFC_E_ARG         (-1)   /* null pointer / negative size / misaligned */
#define PFC_E_SHAPE       (-2)   /* shape not supported by the requested kernel path */
#define PFC_E_ARCH        (-3)   /* device is not compute capability 10.x */
#define PFC_E_WORKSPACE   (-4)   /* workspace too small */

/* margin applied to the target cosine in the logits epilogues */
#define PFC_MARGIN_COSFACE 0     /* s * (cos - m)                 losses.py:17-29 */
#define PFC_MARGIN_ARCFACE 1     /* s * cos(acos(cos) + m)        losses.py:32-45 */

/* kernel path selectors for the GEMM-shaped entries */
#define PFC_PATH_TENSOR   0      /* bf16 operands, tcgen05/TMEM fp32 accumulate (the product path) */
#define PFC_PATH_CHECK    1      /* fp32 operands, fp32 SIMT accumulate ("check mode", slow) */

int         pfc_version(void);
const char* pfc_last_error(void);
/* cc_major/cc_minor/sm_count may be NULL.  Returns PFC_E_ARCH when the device is not sm_100. */
int pfc_query_device(int device, int* cc_major, int* cc_minor, int* sm_count);

/* ------------------------------------------------------------------------------------------------
 * Row kernels (HBM bound)
 * ---------------------------------------------------------------------------------------------- */

/* norm_weight = normalize(sub_weight)                                   partial_fc.py:127
 * w [n_rows_src, emb] fp32.  If index != NULL row r of the output is w[index[r]] (fuses the gather of
 * partial_fc.py:105).  Writes w_hat (bf16 [n_rows, emb], may be NULL), w_hat_f32 (fp32, may be NULL;
 * check mode) and inv_norm[r] = 1 / max(||w_r||, 1e-12). */
int pfc_normalize_rows(const float* w, const int64_t* index, int64_t n_rows, int emb,
                       void* w_hat_bf16, float* w_hat_f32, float* inv_norm, void* stream);

/* total_features -> bf16 operand of the logits GEMM (features are used as passed, partial_fc.py:110). */
int pfc_cast_rows_bf16(const float* x, int64_t n_rows, int emb, void* x_bf16, void* stream);

/* sub_weight = weight[index]; sub_weight_mom = weight_mom[index]        partial_fc.py:105-106 */
int pfc_gather_rows2(const float* weight, const float* weight_mom, const int64_t* index, int64_t n_index,
                     int emb, float* sub_weight, float* sub_weight_mom, void* stream);

/* weight_mom[index] = sub_weight_mom; weight[index] = sub_weight        partial_fc.py:113-116 (update) */
int pfc_scatter_rows2(float* weight, float* weight_mom, const int64_t* index, int64_t n_index, int emb,
                      const float* sub_weight, const float* sub_weight_mom, void* stream);

/* optimizer.step() + update() for the head in one pass (the step either side of the path, SURVEY 8f):
 * torch.optim.SGD (momentum buffer always present, as injected at partial_fc.py:126) applied in place to the rows
 * weight[index[r]] / weight_mom[index[r]] with gradient row r (index == NULL: row r itself), operation by operation as
 * torch's foreach kernels do it (config.py:8-9: momentum 0.9, weight_decay 5e-4).  When index == NULL, w_hat_bf16 /
 * inv_norm (either may be NULL) receive normalize() of the UPDATED rows -- the operands of the next step's forward. */
int pfc_sgd_step(float* weight, float* weight_mom, const float* grad, const int64_t* index, int64_t n_rows,
                 int emb, float lr, float momentum, float dampening, float weight_decay, int nesterov,
                 void* w_hat_bf16, float* inv_norm, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sampling (integer exact)                                              partial_fc.py:89-106
 * ---------------------------------------------------------------------------------------------- */

/* label_out[i] = label_in[i] - class_start if owned by this shard else -1      partial_fc.py:91-93 */
int pfc_remap_labels(const int64_t* label_in, int64_t n, int64_t class_start, int64_t num_local,
                     int64_t* label_out, void* stream);

size_t pfc_sample_workspace_bytes(int64_t num_local);

/* index = sort(topk(perm with perm[positive] = 2.0, num_sample).indices), or the positives when they
 * outnumber num_sample; label[i] <- searchsorted(index, label[i]) for owned labels.
 *   label      in/out [n_label]   shard-local ids or -1 (output of pfc_remap_labels)
 *   perm       in/out [num_local] fp32 uniform draw (torch.rand, partial_fc.py:95); positives are set to 2.0
 *   index_out  [max(num_sample, min(n_label, num_local))]
 *   n_index_out device int64[1]: number of ids written
 * Ties at the k-th value are resolved like torch's CUDA topk: strictly greater first, then equal in
 * ascending index order. */
int pfc_sample_index(int64_t* label, int64_t n_label, float* perm, int64_t num_local, int64_t num_sample,
                     int64_t* index_out, int64_t* n_index_out, void* workspace, size_t workspace_bytes,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused margin-softmax forward                                          partial_fc.py:137-147, losses.py:23-29
 * ---------------------------------------------------------------------------------------------- */

/* Number of per-row partial (max, sum-exp) slots pfc_fwd_stats writes for this shape. */
int pfc_fwd_num_partials(int64_t n_rows, int64_t n_classes, int emb, int path);

/* z_ij = s * (x_i . w_hat_j - m [label_i == j]); for every row the running max and sum exp(z - max) over
 * the classes this call covers, plus the target logit z_{i,label_i} for owned rows.  Logits never
 * leave the chip.
 *   x, w_hat     bf16 (PFC_PATH_TENSOR) or fp32 (PFC_PATH_CHECK), [n_rows, emb] / [n_classes, emb]
 *   label        int64 [n_rows], -1 = class not in this shard
 *   part_max/part_sum  fp32 [pfc_fwd_num_partials(...), n_rows]
 *   target_logit fp32 [n_rows]; the library zero-fills target_logit and part_sum itself before the launch (only owning
 *                rows are then written), so the caller may pass a persistent, un-cleared buffer */
int pfc_fwd_stats(const void* x, const void* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes,
                  int emb, float s, float m, int margin_kind, float* part_max, float* part_sum, float* target_logit,
                  int path, void* stream);

/* prepare + forward in one call: norm_weight = normalize(sub_weight[index]) (partial_fc.py:105,127) fused with
 * pfc_fwd_stats (partial_fc.py:137-147).  The class axis is processed in chunks: the HBM-bound normalisation of
 * chunk k+1 is done by extra warps INSIDE the tensor-core logits kernel of chunk k (one replayed CUDA graph).
 *   w      fp32 [*, emb] (sub_weight, or the whole shard when index != NULL), index int64 [n_classes] or NULL
 *   w_hat  out: bf16 (PFC_PATH_TENSOR) / fp32 (PFC_PATH_CHECK) [n_classes, emb];  inv_norm out: fp32 [n_classes]
 *   the remaining arguments are those of pfc_fwd_stats; target_logit / part_sum are zero-filled here. */
int pfc_normalize_fwd_stats(const float* w, const int64_t* index, const void* x, const int64_t* label,
                            int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, void* w_hat,
                            float* inv_norm, float* part_max, float* part_sum, float* target_logit,
                            int path, void* stream);

/* Merge the partial slots of one shard into stats[n_rows, 3] = (max, sum-exp at that max, target logit). */
int pfc_merge_stats(const float* part_max, const float* part_sum, const float* target_logit, int n_partials,
                    int64_t n_rows, float* stats, void* stream);

/* Combine the shard stats of `world` ranks (all-gathered, [world, n_rows, 3]) -- replaces the three
 * all_reduces of partial_fc.py:142,147,161 -- into row_max, row_sum and
 * loss = -mean(log(max(p_target, 1e-30)))                               partial_fc.py:162 */
int pfc_finalize_stats(const float* gathered_stats, int world, int64_t n_rows, float* row_max, float* row_sum,
                       float* loss_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused backward                                                        partial_fc.py:165-168 (+ autograd)
 * ---------------------------------------------------------------------------------------------- */

size_t pfc_bwd_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb, int path);

/* G_ij = s * (softmax_ij - [label_i == j]) / total_batch  (recomputed from x, w_hat and the global stats)
 * dx    = G . w_hat                         [n_rows, emb]   fp32, overwritten (this shard's partial sum)
 * dw_j  = (dwh_j - w_hat_j (w_hat_j . dwh_j)) * inv_norm_j  with dwh = G^T . x    (normalize backward)
 *         [n_classes, emb] fp32; accumulate_dw != 0 adds into dw (torch .grad semantics).
 * w_hat_f32 is only read in PFC_PATH_CHECK (then x / w_hat are fp32 too). */
int pfc_bwd(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label,
            const float* row_max, const float* row_sum, int64_t n_rows, int64_t n_classes, int emb,
            float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
            void* workspace, size_t workspace_bytes, int path, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stored-probability variant (tensor path only; the default of fedfr_b200.PartialFC)
 *                                                  partial_fc.py:137-168 without the recomputation GEMM
 * ------------------------------------------------------------------------------------------------
 * pfc_normalize_fwd_prob = pfc_normalize_fwd_stats, and additionally keeps
 *     P_ij = exp2(s log2e (x_i . w_hat_j) - a_i)      bf16, blocked [ceil(C/256)*4][ceil(Bt/128)][128][64]
 * in prob_ws, where a_i = s log2e |x_i| (1 + 2^-7) - 58 is an upper bound of every logit of row i (in log2 units)
 * minus a fixed headroom, so no row maximum is needed before the GEMM.  The partial statistics it emits are
 * (a_i ln 2, sum_j P_ij): valid (max, sum-exp) pairs for pfc_merge_stats / pfc_finalize_stats, and equal on every rank.
 * The target column is stored as zero; pfc_bwd_prob writes it from fp32 statistics.
 * Domain: rows whose largest logit lies more than ~184 log2 units (127 nats) below s |x_i| underflow to P = 0
 * (cannot happen for unit-norm features with s <= 64; use pfc_normalize_fwd_stats + pfc_bwd otherwise).
 *   w == NULL: w_hat / inv_norm are already valid and only the logits kernels run.
 *   prob_ws: device scratch of pfc_prob_workspace_bytes(...) bytes, 1024-byte aligned, handed unchanged to pfc_bwd_prob. */
size_t pfc_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb);
int pfc_normalize_fwd_prob(const float* w, const int64_t* index, const void* x, const int64_t* label,
                           int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, void* w_hat,
                           float* inv_norm, float* part_max, float* part_sum, float* target_logit,
                           void* prob_ws, size_t prob_ws_bytes, void* stream);

/* Range guard of the stored-probability path.  `flag` = two ints in pinned host memory (or device memory), NULL disables:
 *   flag[0] := 1 by pfc_normalize_fwd_prob when s |x_i| of some row exceeds `limit_nats` (<= 0: keep the default 80) or is
 *              not finite -- the row would be referenced to a bound far above its real logits and underflow;
 *   flag[1] := 1 by pfc_bwd_prob when a row's sum of probabilities is 0 or not finite (its gradients are then zero).
 * Sticky plain stores, checked EVERY step on the device at no cost; the host polls them without synchronising and switches
 * to pfc_normalize_fwd_stats + pfc_bwd (no such domain limit).  Applies to the calling thread's current device. */
int pfc_set_range_flag(int* flag, float limit_nats);

/* Backward of pfc_normalize_fwd_prob: same outputs as pfc_bwd.  row_sum = the GLOBAL sum_j P_ij of
 * pfc_finalize_stats.  G_ij = (s / (row_sum_i total_batch)) P_ij is never formed: dx = row-scaled P . w_hat,
 * dwh = P^T . (row-scaled x); the radial term w_hat_j . dwh_j of the normalize backward is taken from the dw accumulator. */
size_t pfc_bwd_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb);
int pfc_bwd_prob(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_sum,
                 int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch,
                 float* dx, float* dw, int accumulate_dw, void* prob_ws, size_t prob_ws_bytes,
                 void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SpreadOut regulariser                                                 server.py:48-63 (SpreadOut_Module.forward)
 * ------------------------------------------------------------------------------------------------
 * similarity = w_hat . w_hat^T (w_hat = normalize(FC), bf16 [n, emb]); H_ij = relu(similarity_ij - margin) for i != j.
 *   part_sum [pfc_spreadout_num_partials(n, emb), n]: partial sums of H_ij^2 per row (their total is the 'sum' loss;
 *            part_max is scratch of the same shape).  The count depends on the shape and the device alone, not on the
 *            tuning knobs of the head's forward;
 *   hw_out   fp32 [n, emb] = H . w_hat.  d loss / d w_hat = 4 * hw_out (H is symmetric, each pair counted twice);
 *            the normalize backward to FC is row-wise and left to the caller.
 * The [n, n] similarity never exists; H lives as bf16 in `workspace` (pfc_spreadout_workspace_bytes, 1024-aligned). */
int pfc_spreadout_num_partials(int64_t n, int emb);
size_t pfc_spreadout_workspace_bytes(int64_t n, int emb);
int pfc_spreadout(const void* w_hat, int64_t n, int emb, float margin, float* part_max, float* part_sum, float* hw_out,
                  void* workspace, size_t workspace_bytes, void* stream);

/* losses.CosFace.forward on materialised logits (dense twin, client.py:430): in place
 * cosine[i, label[i]] -= m for label[i] != -1, then out = cosine * s.      losses.py:23-29 */
int pfc_cosface_dense(float* cosine, const int64_t* label, int64_t n_rows, int64_t n_classes, float s, float m,
                      float* out, void* stream);

/* losses.ArcFace.forward on materialised logits (client.py:430 with --loss ArcFace): IN PLACE, like the reference,
 * cosine = s * cos(acos(cosine) + m [label_i == j]) (rows with label -1 get no margin).              losses.py:38-45 */
int pfc_arcface_dense(float* cosine, const int64_t* label, int64_t n_rows, int64_t n_classes, float s, float m,
                      void* stream);

/* ------------------------------------------------------------------------------------------------
 * FedAvg                                                                server.py:25-46
 * ---------------------------------------------------------------------------------------------- */

#define FEDAVG_F32  0
#define FEDAVG_I64  1
#define FEDAVG_KEEP_FIRST_TERM 0x100   /* OR into a dtype code: the sum starts AT the first term (FedAvg_on_FC, server.py:38)
                                          instead of 0 + first term (FedPavg, server.py:30-32: -0.0 becomes +0.0) */

/* One segment = one state_dict entry: K source tensors of n elements and one fp32 output.
 * out[e] = sum_i fl32(w_i) * fl32(src_i[e]) evaluated as separate round-to-nearest multiply and add in
 * client order (bit-identical to the reference's `tmp += weights[i] * models[i][name]`).
 *   seg_src_host   [n_seg * K] device pointers, client-minor (segment s, client i -> s*K + i)
 *   seg_out_host   [n_seg]     device pointers (fp32)
 *   seg_len_host   [n_seg]     element counts
 *   seg_dtype_host [n_seg]     FEDAVG_F32 / FEDAVG_I64 [| FEDAVG_KEEP_FIRST_TERM]; fp32 segments with a source or output that is
 *                              not 16-byte aligned take a scalar path; K > 64 clients run as ceil(K / 64) launches, same sum order
 *   weights_host   [K]         already normalised (w_i / sum w), rounded to fp32 by the caller
 * table_dev: device scratch of at least fedavg_table_bytes(n_seg, K) bytes; the host arrays are copied
 * into it with cudaMemcpyAsync on `stream` (so they must stay valid until the stream reaches the copy;
 * pass pinned memory to keep the call asynchronous). */
size_t fedavg_table_bytes(int n_seg, int K);
int fedavg_weighted_sum(const void* const* seg_src_host, void* const* seg_out_host, const int64_t* seg_len_host,
                        const int32_t* seg_dtype_host, int n_seg, const float* weights_host, int K,
                        void* table_dev, size_t table_bytes, void* stream);

/* FedAvg_on_FC epilogue (server.py:42-45): out = fl32(1-p) * old + fl32(p) * aggr, elementwise fp32
 * (both scalars are rounded from the Python doubles by the caller; separate multiply and add). */
int fedavg_blend(const float* old_fc, const float* aggr, float one_minus_p, float p, int64_t n, float* out,
                 void* stream);

/* ------------------------------------------------------------------------------------------------
 * Cosine head of the personalised branch                        client.py:25-60 (BCE_module.forward :45-58)
 * ------------------------------------------------------------------------------------------------
 * feat fp32 [n_rows, emb] (output of the module's converter, NOT normalised), weight fp32 [n_classes, emb], bias fp32
 * [n_classes] or NULL, label int64 [n_rows] (labels >= n_classes and -1 have no positive column, client.py:49-52).
 *   cosine = normalize(feat) . normalize(weight)^T                                  client.py:47
 *   logits = r * (g(cosine) -/+ m) + bias,  g(x) = 2 ((x+1)/2)^t - 1,  "-" on gt     client.py:40,53-57
 *   gt     uint8 [n_rows, n_classes]  (the bool matrix the module returns)           client.py:48-52
 * cosine [n_rows, n_classes], inv_norm_feat [n_rows], inv_norm_w [n_classes] are kept for the backward.  One launch. */
int pfc_bce_head_fwd(const float* feat, const float* weight, const float* bias, const int64_t* label, int64_t n_rows,
                     int64_t n_classes, int emb, float m, float r, float t, float* logits, unsigned char* gt,
                     float* cosine, float* inv_norm_feat, float* inv_norm_w, void* stream);
/* autograd of the above from dlogits fp32 [n_rows, n_classes]: dfeat [n_rows, emb] (NULL = not needed),
 * dweight [n_classes, emb], dbias [n_classes] (NULL when there is no bias).  Overwrites its outputs.  One launch;
 * emb <= 1024. */
int pfc_bce_head_bwd(const float* feat, const float* weight, const float* cosine, const float* inv_norm_feat,
                     const float* inv_norm_w, const float* dlogits, int64_t n_rows, int64_t n_classes, int emb, float r,
                     float t, float* dfeat, float* dweight, float* dbias, void* stream);

/* The head with losses.BCE_loss on top (losses.py:4-15, client.py:382,393), without the [n_rows, n_classes] logits.
 * For row b and class c, cos, gt and the logit z are the fp32 values pfc_bce_head_fwd computes (same operations, same
 * target-column rule, same clamp of (cos + 1) / 2 at 0).  With pos_coef = fl32(lam / r_loss) and
 * neg_coef = fl32((1 - lam) / r_loss) (the Python doubles rounded once, as torch rounds a scalar factor; the reference
 * uses lam = 0.7, r_loss = 30, which is not the head's r):
 *   term(b, c) = gt ? pos_coef * log((1 + exp(-z)) + 1e-8) : neg_coef * log((1 + exp(z)) + 1e-8)
 *   loss       = (sum over b in row order of row_loss[b]) / n_rows,   row_loss[b] = sum over c in class order of term(b, c)
 * in fp32, each sum sequential from 0, so the loss is the same bits from run to run.  torch's literal formula, not log1p:
 * an exp that overflows fp32 (|z| > ~88.7) gives an infinite loss, as in the reference.  n_rows == 0 gives a NaN loss
 * (torch's mean of nothing); n_classes == 0 gives 0.
 * Writes loss [1], row_loss [n_rows], and cosine, inv_norm_feat, inv_norm_w as pfc_bce_head_fwd does (inv_norm_feat even
 * when n_classes == 0).  ticket: one device uint32 that is 0 before the call; the call returns it to 0.  Calls that may
 * run at the same time need tickets of their own.  bias may be NULL.  emb <= 1024.  One launch. */
int pfc_bce_loss_fwd(const float* feat, const float* weight, const float* bias, const int64_t* label, int64_t n_rows,
                     int64_t n_classes, int emb, float m, float r, float t, float pos_coef, float neg_coef, float* loss,
                     float* row_loss, unsigned int* ticket, float* cosine, float* inv_norm_feat, float* inv_norm_w,
                     void* stream);
/* Its autograd: pfc_bce_head_bwd with d loss / d z computed in the kernel from cosine, label and bias,
 *   d z = ((grad_out[0] / n_rows) * coef) / ((1 + e) + 1e-8) * e,   e = exp(-z), coef = pos_coef, negated, on gt;
 *                                                                   e = exp(z),  coef = neg_coef otherwise
 * (autograd's order of operations; an overflowing exp gives NaN, as in the reference).  grad_out is a DEVICE scalar (the
 * gradient arriving at the loss, e.g. 10 for 10 * loss), so no host synchronisation is needed.  Same outputs, NULL rules
 * and size limits as pfc_bce_head_bwd; bias may be NULL.  One launch. */
int pfc_bce_loss_bwd(const float* feat, const float* weight, const float* bias, const int64_t* label, const float* cosine,
                     const float* inv_norm_feat, const float* inv_norm_w, const float* grad_out, int64_t n_rows,
                     int64_t n_classes, int emb, float m, float r, float t, float pos_coef, float neg_coef, float* dfeat,
                     float* dweight, float* dbias, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Hard-negative mining by similarity threshold              client.py:208-215 and client.py:232-235
 * ------------------------------------------------------------------------------------------------
 * hit[j] = 1 when some row i has <a_i, b_j> > threshold, else 0  (a fp32 [n_a, emb], b fp32 [n_b, emb], hit uint8 [n_b],
 * fully overwritten).  nonzero(hit) is the reference's `unique(torch.where(a @ b.T > threshold)[1])`; the [n_a, n_b]
 * similarity matrix is never materialised.  fp32 FMA chains in k order (see csrc/hardneg.cu for why not bf16). */
int pfc_similar_columns(const float* a, int64_t n_a, const float* b, int64_t n_b, int emb, float threshold,
                        unsigned char* hit, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Pairwise-cosine ROC histogram                                 roc_cuda.py:14-28 (launch :40-51)
 * ------------------------------------------------------------------------------------------------
 * Replaces the numba kernel `calc_ROC(feature, label, subfeature, sublabel, out)`: for every pair (i, j) with
 * i < n_sub, j < n and sub_offset + i < j,
 *     tmp = sum_k fl32(subfeature[i,k] * feature[j,k])   (fp32 products, fp64 sum, k ascending -- the reference's arithmetic)
 *     hist[2 * int((tmp + 1) * 1000) + (sublabel[i] != label[j])] += 1
 * feature fp32 [n, emb], label int32 [n], subfeature fp32 [n_sub, emb], sublabel int32 [n_sub]; hist int64 [2001 * 2]
 * is ADDED to (the reference's `out`, float64 there and cast to int64 by its caller, roc_cuda.py:52).  The reference
 * always compares local indices (sub_offset = 0: roc_cuda.py:44-48 slices feature[start:] and its first rows); a
 * non-zero sub_offset lets one call, or one rank, take rows [sub_offset, sub_offset + n_sub) of `feature` as the sub
 * block, so the reference's whole batch loop (roc_cuda.py:30-53, :136-139) is ONE launch with n_sub = target_size.
 * Bins are clamped to [0, 2000] (the reference would write out of bounds for |cosine| > 1 by more than rounding). */
int pfc_roc_histogram(const float* feature, const int32_t* label, int64_t n, const float* subfeature,
                      const int32_t* sublabel, int64_t n_sub, int64_t sub_offset, int emb, int64_t* hist, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 1:1 template verification (IJB-B / IJB-C protocol)         ijbc_all.py / ijbc_conti.py
 * ------------------------------------------------------------------------------------------------
 * Template pooling.  feats fp32 [n, emb] (emb <= 4096), weights fp32 [n] or NULL (a per-image scale).  The images are
 * given in ascending (template, media, row) order as a CSR: order int64 [n] lists image rows, media j holds
 * order[media_start[j] .. media_start[j+1]), template t holds medias tmpl_start[t] .. tmpl_start[t+1]
 * (media_start [n_media + 1], tmpl_start [n_templates + 1], both ascending, every media non-empty; fedfr_b200.verify
 * builds them).  Writes template_feats fp32 [n_templates, emb]:
 *     x = feats_i (* weights_i, fp32);  media = fp32 sum of its images in order, / (float)count when count > 1;
 *     t = fp32 sum of the medias in order;  out_k = (float)((double)t_k / max(sqrt(sum_k (double)t_k^2), 1e-12)).
 * Deterministic (no atomics). */
int pfc_template_pool(const float* feats, const float* weights, const int64_t* order, const int64_t* media_start,
                      const int64_t* tmpl_start, int64_t n_templates, int emb, float* template_feats, void* stream);

/* scores[p] = (float)(sum_k (double)fl32(a_k * b_k)), k ascending, a = template_feats[row1[p]], b = template_feats[row2[p]]
 * (the pfc_roc_histogram chain).  A pair with a row outside [0, n_templates) scores NaN.  Pairs grouped by row1 read
 * that row once per 128 pairs. */
int pfc_pair_scores(const float* template_feats, int64_t n_templates, int emb, const int64_t* row1, const int64_t* row2,
                    int64_t n_pairs, float* scores, void* stream);

/* Exact TAR@FAR without sorting.  scores fp32 [n] (n < 2^31), issame uint8 [n] (nonzero = genuine); fars_host: n_far
 * (1..8) host doubles in (0, 1].  With n_imp impostors and k = floor(f * n_imp) (fp64), the threshold is the (k+1)-th
 * largest impostor score (-inf when k >= n_imp) and a pair is accepted iff score > threshold (-0.0 == +0.0).  Writes
 * counts int64 [3 + 2 n_far] = {n_gen, n_imp, n_nan, then accepted genuine, accepted impostor per FAR} and thresholds
 * fp32 [n_far]; NaN scores are counted in n_nan and in no class.  workspace: pfc_tar_at_far_workspace_bytes(n) bytes,
 * 8-byte aligned. */
size_t pfc_tar_at_far_workspace_bytes(int64_t n);
int pfc_tar_at_far(const float* scores, const unsigned char* issame, int64_t n, const double* fars_host, int n_far,
                   int64_t* counts, float* thresholds, void* workspace, size_t workspace_bytes, void* stream);

/* Exact ROC curve, element for element sklearn.metrics.roc_curve(issame, scores) (drop_intermediate=True).  scores fp32
 * [n] (n < 2^31), issame uint8 [n] (nonzero = genuine).  Defined on counts, with no float sort order:
 *   1. each score maps to the order-preserving uint32 key of pfc_tar_at_far, -0.0 folded onto +0.0;
 *   2. walking the distinct keys in descending order, key j has g_j genuine and i_j impostor scores (exact counts);
 *      tps = cumsum(g), fps = cumsum(i);
 *   3. thinning keeps the first and the last key, and an inner key j iff g_{j+1} != g_j or i_{j+1} != i_j (sklearn's
 *      nonzero second difference of fps / tps);
 *   4. the point (0, 0) at threshold +inf comes first; then fpr = (double)fps / n_imp, tpr = (double)tps / n_gen (one
 *      IEEE division each) and threshold = (double) of the key's fp32 value.
 * Writes n_points[0] = the curve's length (<= n + 1) and fpr, tpr, thresholds [n_points] (room for n + 1 each; nothing
 * past n_points is written), and counts int64 [3] = {n_gen, n_imp, n_nonfinite}: finite genuine, finite impostor, and
 * NaN or +-inf scores.  The curve means nothing unless n_nonfinite == 0, n_gen > 0 and n_imp > 0 (fedfr_b200.verify
 * raises otherwise).  Deterministic: integer counts and scans, no float atomics.  workspace:
 * pfc_roc_curve_workspace_bytes(n) bytes (about 19 n), 8-byte aligned. */
size_t pfc_roc_curve_workspace_bytes(int64_t n);
int pfc_roc_curve(const float* scores, const unsigned char* issame, int64_t n, double* fpr, double* tpr, double* thresholds,
                  int64_t* n_points, int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K-fold verification accuracy (LFW / CFP-FP / AgeDB)      eval/verification.py test() / evaluate() / calculate_roc
 * ------------------------------------------------------------------------------------------------
 * The per-round small-set test, exact on integer counts.  emb fp32 [2P, emb] (rows 2p and 2p+1 are pair p: evaluate's
 * embeddings[0::2] / [1::2]), flip fp32 [2P, emb] or NULL, issame uint8 [P] (nonzero = genuine), thr fp64 [T] strictly
 * ascending (the caller's grid, e.g. np.arange(0, 4, 0.01); never recomputed here), F = nfolds.
 *   1. fused row: x_k = fl32(emb_k + flip_k), or emb_k when flip is NULL;
 *   2. sklearn.preprocessing.normalize's formula with a pinned fp64 sum of squares:
 *        nrm = (float)sqrt(sum_k (double)x_k^2), nrm = 1 when it is 0, xh_k = x_k / nrm (one fp32 IEEE division).
 *      The sum: lane l of 32 adds k = l, l + 32, l + 64, ... in ascending order (fp64, round to nearest), then the 32
 *      partials are added by an xor butterfly s_l = s_l + s_{l^o} for o = 16, 8, 4, 2, 1 (all lanes end equal);
 *   3. dist[p] = (float)(sum_k (double)fl32(xh1_k - xh2_k)^2), summed in the same order (the fp64 square of an fp32
 *      difference is exact);
 *   4. b_p = #{j : !((double)dist[p] < thr_j)}: pair p is predicted "same" at threshold j iff dist < thr_j iff j >= b_p
 *      (numpy 2's np.less(dist, thr_j) with an np.float64 threshold; a NaN distance gets b_p = T, never "same");
 *   5. folds are sklearn's KFold(F, shuffle=False): contiguous test blocks of P / F pairs, the first P % F one longer;
 *      train is the complement.  F = 1 is insightface's LFold: train = test = all pairs;
 *   6. per fold f and threshold j, integer tp / fp / tn / fn on train and on test.  best_f = the first j maximising the
 *      train tp + tn (np.argmax of the train accuracy); accuracy[f] = (double)(tp + tn)_test[best_f] / n_test;
 *      best_thr[f] = thr[best_f]; the test rates tpr_fj = (double)tp / (tp + fn) and fpr_fj = (double)fp / (fp + tn),
 *      0 when the denominator is 0;
 *   7. tpr[j] = (tpr_0j + tpr_1j + ... + tpr_(F-1)j) / F, added in fold order, then one division (np.mean(tprs, 0));
 *      fpr the same.
 * Writes dist fp32 [P], accuracy and best_thr fp64 [F], tpr and fpr fp64 [T].  Limits: 1 <= emb <= 4096, 1 <= P < 2^31,
 * 1 <= T <= 16384, 1 <= F <= P.  Deterministic: integer histograms (shared-memory atomics), fixed-order scans and sums,
 * no sort, no float atomics; the host is never synchronised.  workspace: pfc_kfold_workspace_bytes(P, T, F) bytes
 * (about 4 P + 24 F T: the bins, the per-fold histograms and the per-fold rates), 8-byte aligned.  VAL@FAR
 * (calculate_val) and the pca > 0 branch are not part of this call. */
size_t pfc_kfold_workspace_bytes(int64_t n_pairs, int n_thresholds, int64_t nfolds);
int pfc_kfold_accuracy(const float* emb, const float* flip, const unsigned char* issame, int64_t n_pairs, int emb_dim,
                       const double* thr, int n_thresholds, int64_t nfolds, float* dist, double* accuracy, double* best_thr,
                       double* tpr, double* fpr, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * 1:N identification (IJB-B / IJB-C search protocol)         ijbc_all.py rank-k, local_1n.py
 * ------------------------------------------------------------------------------------------------
 * probe fp32 [P, emb], gallery fp32 [G, emb] (used as given; normally pfc_template_pool output, one gallery row per
 * subject), mate_row int64 [P]: the gallery row of the probe's subject, or -1 for a non-mated probe.  Gallery rows keep
 * the caller's order, and that order breaks ties.
 *   1. s(p, g) = (float)(sum_k (double)fl32(x_pk * y_gk)), k ascending: the pfc_pair_scores chain, so a pair's score
 *      is bit-identical to pfc_pair_scores on the same two rows;
 *   2. key(s) = the order-preserving uint32 key of pfc_tar_at_far: -0.0 folded onto +0.0; NaN maps to 0, below every
 *      number, and is counted in n_nan;
 *   3. mated probe with mate m: rank[p] = 1 + #{g : key_g > key_m} + #{g < m : key_g == key_m}, the mate's 1-based
 *      position in np.argsort(-s_p, kind="stable"); rank[p] = 0 for a non-mated probe;
 *      mate_score[p] = s(p, m), NaN without a mate;
 *   4. top1_row[p] = the first row with the largest key (np.argsort(-s_p, kind="stable")[0]); top1_score[p] = its
 *      score, read back from the key (so +0.0 for a zero score; NaN only when every score of the row is NaN).
 * CMC and TPIR@FPIR follow from rank, mate_score and top1_score alone (fedfr_b200.verify cmc / tpir_at_fpir):
 *   cmc[r-1] = #{mated p : rank_p <= r} / n_mated;  TPIR@FPIR at rank R is pfc_tar_at_far over s'_p = mate_score_p if
 *   1 <= rank_p <= R else -inf (mated, "genuine") and s'_p = top1_score_p (non-mated, "impostor").
 * A mate_row outside [-1, G) gets rank 0 and a NaN mate_score, like a bad row in pfc_pair_scores, and is counted.
 * Writes rank, top1_row int64 [P], mate_score, top1_score fp32 [P] and counts int64 [2] = {n_nan (NaN scores over
 * all P x G pairs), n_bad (mate rows outside [-1, G))}.  Limits: 1 <= emb <= 4096, 1 <= P, G < 2^31.  Deterministic:
 * integer atomics and a 64-bit maximum, no float atomics, no [P, G] matrix; the host is never synchronised.
 * workspace: pfc_identify_workspace_bytes(P) bytes (about 12 P), 8-byte aligned. */
size_t pfc_identify_workspace_bytes(int64_t n_probe);
int pfc_identify(const float* probe, int64_t n_probe, const float* gallery, int64_t n_gallery, int emb,
                 const int64_t* mate_row, int64_t* rank, float* mate_score, int64_t* top1_row, float* top1_score,
                 int64_t* counts, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* FEDFR_B200_H_ */
