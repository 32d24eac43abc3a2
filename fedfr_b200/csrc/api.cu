// extern "C" entries of the GEMM-shaped part of the hot path: dispatch between the tensor path
// (tc_kernels.cu) and check mode (simt_check.cu).  There is no CPU path.
#include "common.cuh"

namespace pfc {
int tc_fwd_num_partials(int64_t n_rows, int64_t n_classes);
int tc_fwd_stats(const void* x, const void* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind,
                 float* part_max, float* part_sum, float* target_logit, cudaStream_t st);
size_t tc_bwd_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb);
int tc_bwd(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_max, const float* row_sum,
           int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
           void* workspace, size_t workspace_bytes, cudaStream_t st);
int tc_normalize_fwd(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                     float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum, float* target_logit, cudaStream_t st);
size_t tc_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb);
int tc_normalize_fwd_prob(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                          float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum, float* target_logit,
                          void* prob_ws, size_t prob_ws_bytes, cudaStream_t st);
size_t tc_bwd_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb);
int tc_bwd_prob(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_sum, int64_t n_rows, int64_t n_classes,
                int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw, void* prob_ws,
                size_t prob_ws_bytes, void* workspace, size_t workspace_bytes, cudaStream_t st);
void tc_set_prob_split(int dx_sms, float dw_rate, int sweep_lead);
size_t tc_spreadout_workspace_bytes(int64_t n, int emb);
int tc_spreadout(const void* w_hat, int64_t n, int emb, float margin, float* part_max, float* part_sum, float* hw_out, void* workspace,
                 size_t workspace_bytes, cudaStream_t st);
void tc_set_fwd_overlap(int chunks, int norm_blocks_per_sm);
int launch_normalize_rows(const float* w, const int64_t* index, int64_t n_rows, int emb, __nv_bfloat16* ob, float* of, float* inv_norm,
                          int blocks_per_sm, cudaStream_t st);
void tc_set_fwd_bn(int bn);
void tc_set_clusters(int dx_cs, int dw_cs);
void tc_set_debug(long long* p);
void tc_set_logits_pair(int on);
void tc_set_graph(int on);
void tc_set_dw4(int on);
int tc_set_range_flag(int* flag, float limit_nats);
void tc_set_dx_pair(int on);
void tc_set_prefetch(int logits, int dx, int dw);
void tc_set_chunk_mb(int mb);
void tc_set_pipeline(int on, int sm_g, int sm_dx, int sm_dw, int ring);
int simt_fwd_num_partials(int64_t n_rows, int64_t n_classes);
int simt_fwd_stats(const float* x, const float* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind,
                   float* part_max, float* part_sum, float* target_logit, cudaStream_t st);
size_t simt_bwd_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb);
int simt_bwd(const float* x, const float* w_hat, const float* inv_norm, const int64_t* label, const float* row_max, const float* row_sum,
             int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
             void* workspace, size_t workspace_bytes, cudaStream_t st);
}  // namespace pfc

using namespace pfc;

extern "C" {

int pfc_fwd_num_partials(int64_t n_rows, int64_t n_classes, int emb, int path) {
  (void)emb;
  if (n_rows <= 0 || n_classes <= 0) return 0;
  return path == PFC_PATH_CHECK ? simt_fwd_num_partials(n_rows, n_classes) : tc_fwd_num_partials(n_rows, n_classes);
}

int pfc_fwd_stats(const void* x, const void* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind,
                  float* part_max, float* part_sum, float* target_logit, int path, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_fwd_stats");
  PFC_REQUIRE(x && w_hat && label && part_max && part_sum && target_logit, PFC_E_ARG, "pfc_fwd_stats: null argument");
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && emb > 0, PFC_E_ARG, "pfc_fwd_stats: empty shape (rows=%lld classes=%lld)", (long long)n_rows,
              (long long)n_classes);
  if (path == PFC_PATH_CHECK)
    return simt_fwd_stats(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(w_hat), label, n_rows, n_classes, emb, s, m, margin_kind,
                          part_max, part_sum, target_logit, as_stream(stream));
  PFC_REQUIRE(path == PFC_PATH_TENSOR, PFC_E_ARG, "pfc_fwd_stats: unknown path %d", path);
  return tc_fwd_stats(x, w_hat, label, n_rows, n_classes, emb, s, m, margin_kind, part_max, part_sum, target_logit, as_stream(stream));
}

int pfc_normalize_fwd_stats(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                            float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum, float* target_logit, int path,
                            void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_normalize_fwd_stats");
  PFC_REQUIRE(w && x && w_hat && inv_norm && label && part_max && part_sum && target_logit, PFC_E_ARG, "pfc_normalize_fwd_stats: null argument");
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && emb > 0, PFC_E_ARG, "pfc_normalize_fwd_stats: empty shape (rows=%lld classes=%lld)",
              (long long)n_rows, (long long)n_classes);
  if (path == PFC_PATH_CHECK) {
    if (int rc = launch_normalize_rows(w, index, n_classes, emb, nullptr, reinterpret_cast<float*>(w_hat), inv_norm, 0, as_stream(stream))) return rc;
    return simt_fwd_stats(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(w_hat), label, n_rows, n_classes, emb, s, m, margin_kind,
                          part_max, part_sum, target_logit, as_stream(stream));
  }
  PFC_REQUIRE(path == PFC_PATH_TENSOR, PFC_E_ARG, "pfc_normalize_fwd_stats: unknown path %d", path);
  return tc_normalize_fwd(w, index, x, label, n_rows, n_classes, emb, s, m, margin_kind, w_hat, inv_norm, part_max, part_sum, target_logit, as_stream(stream));
}

/* ---- stored-probability variant of the two calls above (tensor path only) ----------------------------------------
 * The forward keeps P_ij = exp2(s log2e cos_ij - a_i) in a bf16 workspace (a_i: a per-row upper bound of the logits),
 * so the backward needs no third logits GEMM.  w == NULL: w_hat / inv_norm are already valid.                       */
size_t pfc_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb) {
  if (n_rows <= 0 || n_classes <= 0 || emb <= 0) return 0;
  return tc_prob_workspace_bytes(n_rows, n_classes, emb);
}

int pfc_normalize_fwd_prob(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                           float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum, float* target_logit,
                           void* prob_ws, size_t prob_ws_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_normalize_fwd_prob");
  PFC_REQUIRE(x && w_hat && inv_norm && label && part_max && part_sum && target_logit && prob_ws, PFC_E_ARG, "pfc_normalize_fwd_prob: null argument");
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && emb > 0, PFC_E_ARG, "pfc_normalize_fwd_prob: empty shape (rows=%lld classes=%lld)", (long long)n_rows,
              (long long)n_classes);
  return tc_normalize_fwd_prob(w, index, x, label, n_rows, n_classes, emb, s, m, margin_kind, w_hat, inv_norm, part_max, part_sum, target_logit, prob_ws,
                               prob_ws_bytes, as_stream(stream));
}

size_t pfc_bwd_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb) {
  if (n_rows <= 0 || n_classes <= 0 || emb <= 0) return 0;
  return tc_bwd_prob_workspace_bytes(n_rows, n_classes, emb);
}

int pfc_bwd_prob(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_sum, int64_t n_rows, int64_t n_classes,
                 int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw, void* prob_ws,
                 size_t prob_ws_bytes, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_bwd_prob");
  PFC_REQUIRE(x && w_hat && inv_norm && label && row_sum && dx && dw && prob_ws && workspace, PFC_E_ARG, "pfc_bwd_prob: null argument");
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && emb > 0, PFC_E_ARG, "pfc_bwd_prob: empty shape");
  return tc_bwd_prob(x, w_hat, inv_norm, label, row_sum, n_rows, n_classes, emb, s, m, margin_kind, inv_total_batch, dx, dw, accumulate_dw, prob_ws,
                     prob_ws_bytes, workspace, workspace_bytes, as_stream(stream));
}

/* tuning: SM budget of the dx kernel (0 = from the shape), dw/dx per-SM rate (<= 0 = keep), classes dx / dw may drift apart (< 0 = keep, 0 = unpaced) */
int pfc_set_prob_split(int dx_sms, float dw_rate, int sweep_lead) {
  tc_set_prob_split(dx_sms, dw_rate, sweep_lead);
  return 0;
}

/* ---- SpreadOut (server.py:48-63) -------------------------------------------------------------------------------- */
size_t pfc_spreadout_workspace_bytes(int64_t n, int emb) {
  if (n <= 0 || emb <= 0) return 0;
  return tc_spreadout_workspace_bytes(n, emb);
}

int pfc_spreadout(const void* w_hat, int64_t n, int emb, float margin, float* part_max, float* part_sum, float* hw_out, void* workspace,
                  size_t workspace_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_spreadout");
  PFC_REQUIRE(w_hat && part_max && part_sum && hw_out && workspace, PFC_E_ARG, "pfc_spreadout: null argument");
  PFC_REQUIRE(n > 0 && emb > 0, PFC_E_ARG, "pfc_spreadout: empty shape");
  return tc_spreadout(w_hat, n, emb, margin, part_max, part_sum, hw_out, workspace, workspace_bytes, as_stream(stream));
}

int pfc_set_fwd_overlap(int chunks, int norm_blocks_per_sm) {   /* class chunks of the fused forward, normalise blocks per SM */
  tc_set_fwd_overlap(chunks, norm_blocks_per_sm);
  return 0;
}

size_t pfc_bwd_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb, int path) {
  if (n_rows <= 0 || n_classes <= 0 || emb <= 0) return 0;
  return path == PFC_PATH_CHECK ? simt_bwd_workspace_bytes(n_rows, n_classes, emb) : tc_bwd_workspace_bytes(n_rows, n_classes, emb);
}

int pfc_bwd(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_max, const float* row_sum,
            int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
            void* workspace, size_t workspace_bytes, int path, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_bwd");
  PFC_REQUIRE(x && w_hat && inv_norm && label && row_max && row_sum && dx && dw && workspace, PFC_E_ARG, "pfc_bwd: null argument");
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && emb > 0, PFC_E_ARG, "pfc_bwd: empty shape");
  if (path == PFC_PATH_CHECK)
    return simt_bwd(reinterpret_cast<const float*>(x), reinterpret_cast<const float*>(w_hat), inv_norm, label, row_max, row_sum, n_rows,
                    n_classes, emb, s, m, margin_kind, inv_total_batch, dx, dw, accumulate_dw, workspace, workspace_bytes, as_stream(stream));
  PFC_REQUIRE(path == PFC_PATH_TENSOR, PFC_E_ARG, "pfc_bwd: unknown path %d", path);
  return tc_bwd(x, w_hat, inv_norm, label, row_max, row_sum, n_rows, n_classes, emb, s, m, margin_kind, inv_total_batch, dx, dw, accumulate_dw, workspace,
                workspace_bytes, as_stream(stream));
}

/* tuning knob (not part of the reference-facing surface): class-tile width of the logits kernels */
int pfc_set_logits_tile(int bn) {
  PFC_REQUIRE(bn == 128 || bn == 256, PFC_E_ARG, "pfc_set_logits_tile: bn must be 128 or 256");
  tc_set_fwd_bn(bn);
  return 0;
}

int pfc_set_logits_pair(int on) {   /* 1 = CTA-pair (cta_group::2) logits kernels (default), 0 = single-CTA */
  tc_set_logits_pair(on);
  return 0;
}

int pfc_set_debug_buffer(void* dev_ptr) {
  tc_set_debug(reinterpret_cast<long long*>(dev_ptr));
  return 0;
}

/* Range guard of the stored-probability path: `flag` = two ints in pinned host (or device) memory, or NULL to disable.
 * flag[0] is set when s |x_i| of a row exceeds `limit_nats` (or is not finite) in pfc_normalize_fwd_prob, flag[1] when a
 * row sum is 0 / non-finite in pfc_bwd_prob.  Sticky; applies to the calling thread's current device. */
int pfc_set_range_flag(int* flag, float limit_nats) { return tc_set_range_flag(flag, limit_nats); }

int pfc_set_dw4(int on) {   /* E = 512 dw kernel: -1 auto (default), 0 e-split pair kernel, > 0 the 4-CTA-cluster kernel */
  tc_set_dw4(on);
  return 0;
}

int pfc_set_graph(int on) {   /* 1 = replay the backward as a cached CUDA graph (default), 0 = launch kernel by kernel */
  tc_set_graph(on);
  return 0;
}

int pfc_set_pipeline(int on, int sm_g, int sm_dx, int sm_dw, int ring) {   /* concurrent G / dx / dw chains; SMs per chain (0 = keep) */
  tc_set_pipeline(on, sm_g, sm_dx, sm_dw, ring);
  return 0;
}

int pfc_set_prefetch(int logits, int dx_distance, int dw) {   /* TMA L2 prefetch ahead of the smem rings */
  tc_set_prefetch(logits, dx_distance, dw);
  return 0;
}

int pfc_set_dx_pair(int on) {   /* 1 = CTA-pair dx kernel when the row blocks come in fours (ceil(Bt / 128) % 4 == 0), E >= 256 and the pair logits kernels are on (default), 0 = single-CTA kernel */
  tc_set_dx_pair(on);
  return 0;
}

int pfc_set_chunk_mb(int mb) {   /* bf16 G scratch per backward chunk in MiB (0 = default) */
  tc_set_chunk_mb(mb);
  return 0;
}

int pfc_set_clusters(int dx_cluster, int dw_cluster) {
  tc_set_clusters(dx_cluster, dw_cluster);
  return 0;
}

}  // extern "C"
