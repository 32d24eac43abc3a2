// Cosine head of FedFR's personalised branch (client.py:25-60 `BCE_module.forward`, lines 45-58) and its backward.
//
// forward, per (row b, class c):
//     cos   = <f_b, w_c> / (max(|f_b|, 1e-12) * max(|w_c|, 1e-12))        F.normalize x2 + matmul     client.py:47
//     g     = 2 * ((cos + 1) / 2)^t - 1                                    g_func                      client.py:40
//     logit = r * (g - m) + bias_c   when c is the row's class, else   r * (g + m) + bias_c            client.py:53-57
//     gt    = (c == label_b), labels >= n_class (and -1) select no column                              client.py:48-52
// backward from d logit (the caller's loss, losses.BCE_loss or anything else, runs in torch on the [B, C] logits):
//     d cos = d logit * r * t * ((cos + 1) / 2)^(t - 1),    d bias_c = sum_b d logit     ((cos + 1) / 2 clamped at 0)
//     d f_b = ( sum_c d cos * w^_c  -  f^_b * sum_c d cos * cos ) / |f_b|       (matmul + normalize backward)
//     d w_c = ( sum_b d cos * f^_b  -  w^_c * sum_b d cos * cos ) / |w_c|
// The reference runs ~20 ATen kernels over [B, C] temporaries for this (two normalisations, a matmul, a [B, C+1] bool
// scatter, two masked gathers / pows / scatters, a broadcast add, and their autograd twins).  Shapes are small (B = 64-256
// rows, C = a client's identities, E = 512): launch-latency territory, so the whole forward is ONE launch (a warp per
// logit: three dot products in one pass over the two rows, epilogue in lane 0) and the whole backward is ONE launch
// (a CTA per feature row and a CTA per class row, each streaming the other operand once through L2).  fp32 throughout.
#include "common.cuh"

namespace pfc {

constexpr float kNormEps = 1e-12f;        // F.normalize default eps
constexpr int kBceThreads = 128;
constexpr int kBceMaxKpt = 8;             // emb <= 1024
constexpr int kBceChunk = 256;

__device__ __forceinline__ float pow_small(float u, float t) {
  if (t == 1.f) return u;
  if (t == 2.f) return u * u;
  if (t == 3.f) return (u * u) * u;       // torch's pow special-cases these exponents the same way
  if (t == 0.f) return 1.f;
  return powf(u, t);
}

// column selected by gt[arange, tmp_labels] on a [B, C+1] matrix whose last column is dropped (client.py:48-52);
// negative labels index from the end like Python does.
__device__ __forceinline__ int64_t bce_target_col(int64_t label, int64_t n_classes) {
  if (label >= n_classes) return -1;
  if (label < 0) {
    label += n_classes + 1;
    if (label < 0 || label >= n_classes) return -1;
  }
  return label;
}

__global__ void __launch_bounds__(256)
bce_head_fwd_kernel(const float* __restrict__ feat, const float* __restrict__ weight, const float* __restrict__ bias,
                    const int64_t* __restrict__ label, int64_t n_rows, int64_t n_classes, int emb, float m, float r, float t,
                    float* __restrict__ logits, unsigned char* __restrict__ gt, float* __restrict__ cosine,
                    float* __restrict__ inv_nf, float* __restrict__ inv_nw) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t total = n_rows * n_classes;
  for (int64_t p = warp; p < total; p += n_warps) {
    const int64_t b = p / n_classes, c = p % n_classes;
    const float* f = feat + b * emb;
    const float* w = weight + c * emb;
    float fw = 0.f, ff = 0.f, ww = 0.f;
    for (int k = lane; k < emb; k += 32) {
      const float x = f[k], y = w[k];
      fw = fmaf(x, y, fw);
      ff = fmaf(x, x, ff);
      ww = fmaf(y, y, ww);
    }
    fw = warp_sum(fw);
    ff = warp_sum(ff);
    ww = warp_sum(ww);
    if (lane == 0) {
      const float inf = 1.f / fmaxf(sqrtf(ff), kNormEps);
      const float inw = 1.f / fmaxf(sqrtf(ww), kNormEps);
      const float cs = fw * inf * inw;
      const float u = fmaxf((cs + 1.f) * 0.5f, 0.f);     // an antipodal pair can round below -1: powf would give NaN
      const float g = 2.f * pow_small(u, t) - 1.f;
      const bool pos = (bce_target_col(label[b], n_classes) == c);
      const float z = __fadd_rn(__fmul_rn(r, pos ? (g - m) : (g + m)), bias ? bias[c] : 0.f);
      logits[p] = z;
      gt[p] = pos ? 1 : 0;
      cosine[p] = cs;
      if (c == 0) inv_nf[b] = inf;
      if (b == 0) inv_nw[c] = inw;
    }
  }
}

__device__ __forceinline__ float block_sum_128(float v, float* scratch) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  return (scratch[0] + scratch[1]) + (scratch[2] + scratch[3]);
}

// One CTA per output row.  mine = the operand whose gradient this CTA produces (feature row b, or class row c),
// other = the rows it sums over.  elem(o) gives the flat [B, C] index of (this row, other row o).
__global__ void __launch_bounds__(kBceThreads)
bce_head_bwd_kernel(const float* __restrict__ feat, const float* __restrict__ weight, const float* __restrict__ cosine,
                    const float* __restrict__ inv_nf, const float* __restrict__ inv_nw, const float* __restrict__ dlogits,
                    int64_t n_rows, int64_t n_classes, int emb, float r, float t,
                    float* __restrict__ dfeat, float* __restrict__ dweight, float* __restrict__ dbias) {
  __shared__ float s_d[kBceChunk];
  __shared__ float scratch[4];
  const bool row_role = (int64_t)blockIdx.x < n_rows;             // else: class role
  if (row_role && dfeat == nullptr) return;
  const int64_t me = row_role ? blockIdx.x : blockIdx.x - n_rows;
  const int64_t n_other = row_role ? n_classes : n_rows;
  const float* mine = (row_role ? feat : weight) + me * emb;
  const float* other = row_role ? weight : feat;
  const float* inv_other = row_role ? inv_nw : inv_nf;
  const float inv_me = row_role ? inv_nf[me] : inv_nw[me];
  const float slope_scale = r * t;

  float acc[kBceMaxKpt];
#pragma unroll
  for (int j = 0; j < kBceMaxKpt; ++j) acc[j] = 0.f;
  float radial = 0.f, bias_sum = 0.f;                              // sum d cos * cos ; sum d logit

  for (int64_t o0 = 0; o0 < n_other; o0 += kBceChunk) {
    const int n_chunk = (int)((n_other - o0 < kBceChunk) ? n_other - o0 : kBceChunk);
    __syncthreads();
    for (int o = threadIdx.x; o < n_chunk; o += kBceThreads) {
      const int64_t e = row_role ? me * n_classes + (o0 + o) : (o0 + o) * n_classes + me;
      const float dz = dlogits[e], cs = cosine[e];
      const float u = fmaxf((cs + 1.f) * 0.5f, 0.f);
      const float dcos = dz * slope_scale * pow_small(u, t - 1.f);
      s_d[o] = dcos * inv_other[o0 + o];
      radial = fmaf(dcos, cs, radial);
      bias_sum += dz;
    }
    __syncthreads();
    for (int o = 0; o < n_chunk; ++o) {
      const float d = s_d[o];
      const float* orow = other + (o0 + o) * emb;
#pragma unroll
      for (int j = 0; j < kBceMaxKpt; ++j) {
        const int k = threadIdx.x + j * kBceThreads;
        if (k < emb) acc[j] = fmaf(d, orow[k], acc[j]);
      }
    }
  }
  radial = block_sum_128(radial, scratch);
  if (!row_role && dbias) {
    bias_sum = block_sum_128(bias_sum, scratch);
    if (threadIdx.x == 0) dbias[me] = bias_sum;
  }
  // a row whose norm was clamped to eps (0 < |v| < 1e-12) has a constant denominator: autograd of F.normalize gives
  // it no radial term (inv_me == 1 / eps marks it: the forward computed 1 / max(|v|, eps) with the same division)
  if (inv_me >= 1.f / kNormEps) radial = 0.f;
  float* out = (row_role ? dfeat : dweight) + me * emb;
#pragma unroll
  for (int j = 0; j < kBceMaxKpt; ++j) {
    const int k = threadIdx.x + j * kBceThreads;
    if (k < emb) out[k] = inv_me * (acc[j] - mine[k] * inv_me * radial);
  }
}

}  // namespace pfc

using namespace pfc;

extern "C" {

int pfc_bce_head_fwd(const float* feat, const float* weight, const float* bias, const int64_t* label, int64_t n_rows,
                     int64_t n_classes, int emb, float m, float r, float t, float* logits, unsigned char* gt,
                     float* cosine, float* inv_norm_feat, float* inv_norm_w, void* stream) {
  if (int rc = require_sm100()) return rc;
  PFC_REQUIRE(n_rows >= 0 && n_classes >= 0 && emb >= 1, PFC_E_ARG, "pfc_bce_head_fwd: bad size");
  if (n_rows == 0 || n_classes == 0) return 0;
  PFC_REQUIRE(feat && weight && label && logits && gt && cosine && inv_norm_feat && inv_norm_w, PFC_E_ARG,
              "pfc_bce_head_fwd: null pointer");
  const int64_t warps = n_rows * n_classes;
  int64_t blocks = (warps + 7) / 8;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  bce_head_fwd_kernel<<<(int)blocks, 256, 0, as_stream(stream)>>>(feat, weight, bias, label, n_rows, n_classes, emb, m, r, t,
                                                                  logits, gt, cosine, inv_norm_feat, inv_norm_w);
  PFC_LAUNCH_CHECK();
  return 0;
}

int pfc_bce_head_bwd(const float* feat, const float* weight, const float* cosine, const float* inv_norm_feat,
                     const float* inv_norm_w, const float* dlogits, int64_t n_rows, int64_t n_classes, int emb, float r,
                     float t, float* dfeat, float* dweight, float* dbias, void* stream) {
  if (int rc = require_sm100()) return rc;
  PFC_REQUIRE(n_rows >= 0 && n_classes >= 0 && emb >= 1, PFC_E_ARG, "pfc_bce_head_bwd: bad size");
  PFC_REQUIRE(emb <= kBceMaxKpt * kBceThreads, PFC_E_SHAPE, "pfc_bce_head_bwd: emb %d > %d", emb, kBceMaxKpt * kBceThreads);
  PFC_REQUIRE(n_rows + n_classes < (int64_t)1 << 31, PFC_E_SHAPE, "pfc_bce_head_bwd: too many rows");
  if (n_rows == 0 || n_classes == 0) {
    // no pairs: every gradient is zero
    if (dfeat && n_rows) PFC_CUDA(cudaMemsetAsync(dfeat, 0, (size_t)n_rows * emb * 4, as_stream(stream)));
    if (dweight && n_classes) PFC_CUDA(cudaMemsetAsync(dweight, 0, (size_t)n_classes * emb * 4, as_stream(stream)));
    if (dbias && n_classes) PFC_CUDA(cudaMemsetAsync(dbias, 0, (size_t)n_classes * 4, as_stream(stream)));
    return 0;
  }
  PFC_REQUIRE(feat && weight && cosine && inv_norm_feat && inv_norm_w && dlogits && dweight, PFC_E_ARG,
              "pfc_bce_head_bwd: null pointer");
  bce_head_bwd_kernel<<<(int)(n_rows + n_classes), kBceThreads, 0, as_stream(stream)>>>(
      feat, weight, cosine, inv_norm_feat, inv_norm_w, dlogits, n_rows, n_classes, emb, r, t, dfeat, dweight, dbias);
  PFC_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
