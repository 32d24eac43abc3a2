// The exact pair-score chain shared by the ROC histogram (roc.cu), 1:1 template verification and 1:N identification
// (verify.cu):
//     tmp = tmp + (double)fl32(a[k] * b[k])      k ascending: fp32 products, fp64 adds, no FMA
// Kernel sources include it as "../../fedfr_b200/csrc/dot_chain.cuh": that path resolves from csrc/ for nvcc and from
// tests/emu/ for the CPU emulation of the kernels, which compiles the .cu files outside this directory.
#pragma once

namespace pfc {

__device__ __forceinline__ double dot_chain(double tmp, const float* __restrict__ a, const float* __restrict__ b, int n) {
  for (int k = 0; k < n; ++k) tmp = __dadd_rn(tmp, (double)__fmul_rn(a[k], b[k]));
  return tmp;
}

// The tiled form of the chain for a 64 x 64 tile of pairs, run by all 256 threads of a CTA (barriers inside):
//     acc[u][v] = dot_chain(0, a[i0 + ty + 16 u], b[j0 + tx + 16 v], emb),   tx = tid & 15, ty = tid >> 4
// Rows at or past n_a / n_b read as zeros.  32-wide k slices of both operands are staged in As / Bs (shared memory),
// and each pair adds exactly the k < emb terms in ascending order, so every sum equals dot_chain's bit for bit.
constexpr int kChainTile = 64;
constexpr int kChainK = 32;
constexpr int kChainThreads = 256;

__device__ __forceinline__ void tile_chain(const float* __restrict__ a, int64_t n_a, int64_t i0,
                                           const float* __restrict__ b, int64_t n_b, int64_t j0, int emb,
                                           float (*As)[kChainK + 1], float (*Bs)[kChainK + 1], double (&acc)[4][4]) {
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) acc[u][v] = 0.0;

  for (int k0 = 0; k0 < emb; k0 += kChainK) {
    __syncthreads();                                  // the previous slice (or tile) has been consumed
    {
      const int kk = tid & 31;
      const bool k_ok = (k0 + kk) < emb;
#pragma unroll
      for (int r = 0; r < kChainTile / 8; ++r) {
        const int row = (tid >> 5) + 8 * r;
        const int64_t gi = i0 + row, gj = j0 + row;
        As[row][kk] = (k_ok && gi < n_a) ? a[gi * emb + k0 + kk] : 0.f;
        Bs[row][kk] = (k_ok && gj < n_b) ? b[gj * emb + k0 + kk] : 0.f;
      }
    }
    __syncthreads();
    const int kc = (emb - k0 < kChainK) ? emb - k0 : kChainK;
#pragma unroll 4
    for (int kk = 0; kk < kc; ++kk) {
      float x[4], y[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) x[u] = As[ty + 16 * u][kk];
#pragma unroll
      for (int v = 0; v < 4; ++v) y[v] = Bs[tx + 16 * v][kk];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = __dadd_rn(acc[u][v], (double)__fmul_rn(x[u], y[v]));
    }
  }
}

}  // namespace pfc
