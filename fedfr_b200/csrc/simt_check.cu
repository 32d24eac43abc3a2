// "Check mode" (PFC_PATH_CHECK): the same maths as the tensor path with fp32 operands and fp32 SIMT
// accumulation.  Slow on purpose -- it exists to separate bf16 rounding from logic errors (parity to
// 1e-4 against the oracle) and to cross-check the tcgen05 kernels on the device.
#include "common.cuh"

namespace pfc {
namespace simt {

constexpr int TM = 64, TN = 64, TK = 16;

// acc[4][4] of a 64x64 tile of C = A * B with generic element strides:
//   A(m,k) = A[m*a_sm + k*a_sk], B(k,n) = B[k*b_sk + n*b_sn];  out-of-range elements read as 0.
struct Tile {
  float acc[4][4];
};

__device__ __forceinline__ void tile_gemm(const float* __restrict__ A, int64_t a_sm, int64_t a_sk, const float* __restrict__ B, int64_t b_sk,
                                          int64_t b_sn, int m0, int n0, int M, int N, int K, float (*sA)[TM + 1], float (*sB)[TN + 1],
                                          Tile& t) {
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) t.acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += TK) {
    for (int e = threadIdx.x; e < TM * TK; e += 256) {
      const int mm = e / TK, kk = e % TK;
      const int m = m0 + mm, k = k0 + kk;
      sA[kk][mm] = (m < M && k < K) ? A[(int64_t)m * a_sm + (int64_t)k * a_sk] : 0.f;
    }
    for (int e = threadIdx.x; e < TN * TK; e += 256) {
      const int nn = e / TK, kk = e % TK;
      const int n = n0 + nn, k = k0 + kk;
      sB[kk][nn] = (n < N && k < K) ? B[(int64_t)k * b_sk + (int64_t)n * b_sn] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sA[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = sB[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) t.acc[i][j] = fmaf(a[i], b[j], t.acc[i][j]);
    }
    __syncthreads();
  }
}

// grid (n_row_tiles, n_split): each block scans its slice of class tiles for 64 rows.
__global__ void __launch_bounds__(256) fwd_stats_kernel(const float* __restrict__ x, const float* __restrict__ w_hat, const int64_t* __restrict__ label,
                                                        int n_rows, int n_classes, int emb, float s, float m, int margin_kind, float* __restrict__ part_max,
                                                        float* __restrict__ part_sum, float* __restrict__ target_logit) {
  __shared__ float sA[TK][TM + 1], sB[TK][TN + 1], sZ[TM][TN + 1];
  const int m0 = blockIdx.x * TM;
  const int n_ct = (n_classes + TN - 1) / TN;
  const int ct0 = (int)((int64_t)n_ct * blockIdx.y / gridDim.y), ct1 = (int)((int64_t)n_ct * (blockIdx.y + 1) / gridDim.y);
  float run_m = -INFINITY, run_l = 0.f;
  const int my_row = m0 + threadIdx.x;                 // threads 0..63 own a row each for the scan
  const int64_t my_label = (threadIdx.x < TM && my_row < n_rows) ? label[my_row] : -1;
  for (int ct = ct0; ct < ct1; ++ct) {
    Tile t;
    tile_gemm(x, emb, 1, w_hat, 1, emb, m0, ct * TN, n_rows, n_classes, emb, sA, sB, t);
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sZ[ty * 4 + i][tx * 4 + j] = t.acc[i][j];
    __syncthreads();
    if (threadIdx.x < TM && my_row < n_rows) {
      for (int j = 0; j < TN; ++j) {
        const int col = ct * TN + j;
        if (col >= n_classes) break;
        float cosv = sZ[threadIdx.x][j];
        if (col == my_label) cosv = margin_cos(cosv, m, margin_kind);   // losses.py:27 / :41-44
        const float z = cosv * s;                             // losses.py:28
        if (col == my_label) target_logit[my_row] = z;
        if (z > run_m) { run_l = run_l * expf(run_m - z) + 1.f; run_m = z; }
        else run_l += expf(z - run_m);
      }
    }
    __syncthreads();
  }
  if (threadIdx.x < TM && my_row < n_rows) {
    part_max[(int64_t)blockIdx.y * n_rows + my_row] = run_m;
    part_sum[(int64_t)blockIdx.y * n_rows + my_row] = run_l;
  }
}

// G[r, c] = s * (exp(z - M_r) / S_r - [c == y_r]) / Bt      (fp32 scratch [n_rows, ldg])
__global__ void __launch_bounds__(256) grad_logits_kernel(const float* __restrict__ x, const float* __restrict__ w_hat, const int64_t* __restrict__ label,
                                                          const float* __restrict__ row_max, const float* __restrict__ row_sum, int n_rows,
                                                          int n_classes, int class_base, int emb, float s, float m, int margin_kind, float g_scale,
                                                          float* __restrict__ g, int64_t ldg) {
  __shared__ float sA[TK][TM + 1], sB[TK][TN + 1];
  const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
  Tile t;
  tile_gemm(x, emb, 1, w_hat, 1, emb, m0, n0, n_rows, n_classes, emb, sA, sB, t);
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + ty * 4 + i;
    if (r >= n_rows) continue;
    const int64_t y = label[r];
    const float M = row_max[r], S = row_sum[r];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = n0 + tx * 4 + j;
      if (c >= n_classes) continue;
      const bool hit = (y >= 0) && (y == (int64_t)class_base + c);
      const float z = (hit ? margin_cos(t.acc[i][j], m, margin_kind) : t.acc[i][j]) * s;
      const float pr = expf(z - M) / S;
      g[(int64_t)r * ldg + c] = (pr - (hit ? 1.f : 0.f)) * g_scale * (hit ? margin_slope(t.acc[i][j], m, margin_kind) : 1.f);
    }
  }
}

// C[M,N] (+)= A*B with generic strides (used for dx = G.w_hat and dwh = G^T.x)
__global__ void __launch_bounds__(256) gemm_kernel(const float* __restrict__ A, int64_t a_sm, int64_t a_sk, const float* __restrict__ B, int64_t b_sk,
                                                   int64_t b_sn, int M, int N, int K, float* __restrict__ C, int64_t ldc, int accumulate) {
  __shared__ float sA[TK][TM + 1], sB[TK][TN + 1];
  const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
  Tile t;
  tile_gemm(A, a_sm, a_sk, B, b_sk, b_sn, m0, n0, M, N, K, sA, sB, t);
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + ty * 4 + i;
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = n0 + tx * 4 + j;
      if (c >= N) continue;
      float v = t.acc[i][j];
      if (accumulate) v += C[(int64_t)r * ldc + c];
      C[(int64_t)r * ldc + c] = v;
    }
  }
}

// dw_j = (dwh_j - w_hat_j (w_hat_j . dwh_j)) * inv_norm_j       one warp per row
// A row whose norm was clamped to eps (0 < |w_j| < 1e-12) has w_hat_j = w_j / eps and a constant denominator: autograd of
// F.normalize gives it dwh_j / eps with no radial term.  inv_norm_j == 1 / eps marks it (normalize_rows_warp computes
// 1 / max(|w|, eps) with the same correctly rounded division); a norm within an ulp above eps may read as clamped too,
// which is inside the rounding of the norm itself.
__global__ void __launch_bounds__(256) normalize_bwd_kernel(const float* __restrict__ dwh, const float* __restrict__ w_hat,
                                                            const float* __restrict__ inv_norm, int64_t n_rows, int emb, float* __restrict__ dw,
                                                            int accumulate) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const float inv = inv_norm[r];
  float dot = 0.f;
  if (inv < 1.f / 1e-12f) {
    for (int c = lane; c < emb; c += 32) dot += dwh[r * emb + c] * w_hat[r * emb + c];
    dot = warp_sum(dot);
  }
  for (int c = lane; c < emb; c += 32) {
    float v = (dwh[r * emb + c] - w_hat[r * emb + c] * dot) * inv;
    if (accumulate) v += dw[r * emb + c];
    dw[r * emb + c] = v;
  }
}

}  // namespace simt

static int check_splits(int64_t n_classes) {
  int64_t n_ct = (n_classes + simt::TN - 1) / simt::TN;
  return (int)(n_ct < 32 ? n_ct : 32);
}

int simt_fwd_num_partials(int64_t n_rows, int64_t n_classes) { (void)n_rows; return check_splits(n_classes); }

int simt_fwd_stats(const float* x, const float* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind,
                   float* part_max, float* part_sum, float* target_logit, cudaStream_t st) {
  const int splits = check_splits(n_classes);
  PFC_CUDA(cudaMemsetAsync(part_sum, 0, sizeof(float) * (size_t)splits * n_rows, st));
  PFC_CUDA(cudaMemsetAsync(target_logit, 0, sizeof(float) * (size_t)n_rows, st));
  dim3 grid((unsigned)((n_rows + simt::TM - 1) / simt::TM), (unsigned)splits);
  simt::fwd_stats_kernel<<<grid, 256, 0, st>>>(x, w_hat, label, (int)n_rows, (int)n_classes, emb, s, m, margin_kind, part_max, part_sum, target_logit);
  PFC_LAUNCH_CHECK();
  return 0;
}

// Class columns per backward chunk: a 64 MiB fp32 G scratch, at least one 64-column tile, and at most 65,535 tiles
// (grad_logits_kernel puts the class tiles on gridDim.y).
static int64_t check_chunk(int64_t n_rows, int64_t n_classes) {
  int64_t chunk = (64ll << 20) / (n_rows * 4);
  chunk = chunk / 64 * 64;
  if (chunk < 64) chunk = 64;
  if (chunk > 65535ll * 64) chunk = 65535ll * 64;
  const int64_t cpad = (n_classes + 63) / 64 * 64;
  return chunk < cpad ? chunk : cpad;
}

size_t simt_bwd_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb) {
  const int64_t chunk = check_chunk(n_rows, n_classes);
  return (size_t)n_rows * chunk * 4 + (size_t)chunk * emb * 4 + 2048;
}

int simt_bwd(const float* x, const float* w_hat, const float* inv_norm, const int64_t* label, const float* row_max, const float* row_sum,
             int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
             void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int64_t chunk = check_chunk(n_rows, n_classes);
  PFC_REQUIRE(workspace_bytes >= simt_bwd_workspace_bytes(n_rows, n_classes, emb) - 2048, PFC_E_WORKSPACE, "pfc_bwd(check): workspace too small");
  float* g = reinterpret_cast<float*>(workspace);
  float* dwh = g + (size_t)n_rows * chunk;
  int idx = 0;
  for (int64_t c0 = 0; c0 < n_classes; c0 += chunk, ++idx) {
    const int64_t cc = n_classes - c0 < chunk ? n_classes - c0 : chunk;
    dim3 g1((unsigned)((n_rows + 63) / 64), (unsigned)((cc + 63) / 64));
    simt::grad_logits_kernel<<<g1, 256, 0, st>>>(x, w_hat + c0 * emb, label, row_max, row_sum, (int)n_rows, (int)cc, (int)c0, emb, s, m, margin_kind,
                                                 s * inv_total_batch, g, chunk);
    PFC_LAUNCH_CHECK();
    // dx[r,e] (+)= sum_c G[r,c] w_hat[c,e]
    dim3 g2((unsigned)((n_rows + 63) / 64), (unsigned)((emb + 63) / 64));
    simt::gemm_kernel<<<g2, 256, 0, st>>>(g, chunk, 1, w_hat + c0 * emb, emb, 1, (int)n_rows, emb, (int)cc, dx, emb, idx > 0);
    PFC_LAUNCH_CHECK();
    // dwh[c,e] = sum_r G[r,c] x[r,e]
    dim3 g3((unsigned)((cc + 63) / 64), (unsigned)((emb + 63) / 64));
    simt::gemm_kernel<<<g3, 256, 0, st>>>(g, 1, chunk, x, emb, 1, (int)cc, emb, (int)n_rows, dwh, emb, 0);
    PFC_LAUNCH_CHECK();
    simt::normalize_bwd_kernel<<<(unsigned)((cc + 7) / 8), 256, 0, st>>>(dwh, w_hat + c0 * emb, inv_norm + c0, cc, emb, dw + c0 * emb, accumulate_dw);
    PFC_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace pfc
