// Pairwise-cosine ROC histogram (roc_cuda.py:14-28 `calc_ROC`, launched at roc_cuda.py:40-51).
//
// For every pair (i, j) with i < n_sub, j < n and (sub_offset + i) < j:
//     tmp  = sum_k fl32(subfeature[i,k] * feature[j,k])      products rounded to fp32, summed in fp64, k ascending
//     bin  = int((tmp + 1) * 1000)                            fp64, truncation
//     hist[2*bin + (sublabel[i] != label[j])] += 1
// which is the reference kernel's arithmetic exactly (its `tmp = 0.` is a double, the product of two float32 is a
// float32), so the histogram is integer-identical.  The reference runs one thread per pair with both 512-float rows
// read from global memory; here a CTA owns a 64 x 64 tile of pairs, stages 32-wide k slices of both operands in shared
// memory, keeps 4 x 4 fp64 sums per thread, counts into a shared-memory histogram and adds the non-empty bins to the
// global int64 histogram once per CTA.  CTAs are persistent (grid = resident CTAs, stride over tiles); tiles entirely on
// or below the diagonal are skipped.  The bound is the fp32-multiply / convert / fp64-add chain per (pair, k), not HBM:
// a 64 x 64 tile reads 2 * 64 * emb * 4 bytes for 4096 * emb such chains.
#include "common.cuh"
#include "../../fedfr_b200/csrc/dot_chain.cuh"

namespace pfc {

constexpr int kRocBins = 2001;
constexpr int kRocTile = kChainTile;      // the exact kernel's tile loop is tile_chain (dot_chain.cuh)
constexpr int kRocK = kChainK;
constexpr int kRocThreads = kChainThreads;
constexpr int kRocFlushTiles = 1 << 19;   // 2^19 tiles * 4096 pairs < 2^32: the shared counters cannot wrap

__device__ __forceinline__ void roc_flush(unsigned int* h, unsigned long long* hist) {
  __syncthreads();
  for (int b = threadIdx.x; b < 2 * kRocBins; b += kRocThreads) {
    const unsigned int v = h[b];
    if (v) atomicAdd(hist + b, (unsigned long long)v);
    h[b] = 0u;
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kRocThreads, 2)
roc_hist_kernel(const float* __restrict__ feature, const int32_t* __restrict__ label, int64_t n,
                const float* __restrict__ sub, const int32_t* __restrict__ sublabel, int64_t n_sub, int64_t sub_offset,
                int emb, unsigned long long* __restrict__ hist) {
  __shared__ float As[kRocTile][kRocK + 1];
  __shared__ float Bs[kRocTile][kRocK + 1];
  __shared__ unsigned int h[2 * kRocBins];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  for (int b = tid; b < 2 * kRocBins; b += kRocThreads) h[b] = 0u;
  __syncthreads();

  const int64_t n_ti = (n_sub + kRocTile - 1) / kRocTile;
  const int64_t n_tj = (n + kRocTile - 1) / kRocTile;
  const int64_t total = n_ti * n_tj;
  int tiles_done = 0;
  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int64_t i0 = (t / n_tj) * kRocTile;
    const int64_t j0 = (t % n_tj) * kRocTile;
    const int64_t j_last = (j0 + kRocTile - 1 < n - 1) ? j0 + kRocTile - 1 : n - 1;
    if (j_last <= sub_offset + i0) continue;          // no pair with i < j in this tile (uniform over the CTA)

    double acc[4][4];
    tile_chain(sub, n_sub, i0, feature, n, j0, emb, As, Bs, acc);

#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = i0 + ty + 16 * u;
      if (i >= n_sub) continue;
      const int32_t li = sublabel[i];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int64_t j = j0 + tx + 16 * v;
        if (j >= n || sub_offset + i >= j) continue;
        int bin = (int)__dmul_rn(__dadd_rn(acc[u][v], 1.0), 1000.0);
        bin = bin < 0 ? 0 : (bin > kRocBins - 1 ? kRocBins - 1 : bin);   // the reference would write out of bounds
        atomicAdd(&h[2 * bin + (li != label[j] ? 1 : 0)], 1u);
      }
    }
    if (++tiles_done == kRocFlushTiles) {
      roc_flush(h, hist);
      tiles_done = 0;
    }
  }
  roc_flush(h, hist);
}

// ---------------------------------------------------------------------------------------------------------------------
// Two-tier variant (opt-in, pfc_set_roc_mode(1); not yet measured on a B200).  Same tiles; the common case runs on the
// fp32 FMA pipe and only pairs that could sit on a bin edge take the exact chain above.
//   A_ij  = blocked fp32 sum: 32-step FMA chain per k slice, slices added in fp32
//   T_ij  = the reference value (fp32 products summed in fp64)
//   |A - T| <= (32 + n_slices + 2) * 2^-24 * |a_i| |b_j|          (gamma_n bound of the two summation levels + the product
//                                                                   roundings of T; Cauchy-Schwarz for sum |a_k b_k|)
// so with x = (A + 1) * 1000 in fp64 and e = 1000 * bound (inflated for the fp32 norms, plus an absolute slack), the bin is
// int(x) whenever x is farther than e from an integer; otherwise the pair is queued in shared memory and the CTA later
// recomputes T for 256 queued pairs at a time (every lane busy, no divergence inside the tile epilogue).  The result
// is integer-identical to roc_hist_kernel for every input (tests/test_kernel_emulation.py drives both with rows that
// land exactly on bin edges).
constexpr int kRocQueue = 1024;

__device__ __forceinline__ double roc_exact_x(const float* __restrict__ a, const float* __restrict__ b, int emb) {
  return __dmul_rn(__dadd_rn(dot_chain(0.0, a, b, emb), 1.0), 1000.0);
}

// Exact chain for every queued pair, one pair per thread.  Called by the whole CTA (barriers inside); q_n may exceed the
// capacity when the queue overflowed -- those pairs were handled by their owners.
__device__ __forceinline__ void roc_drain(const unsigned int* q_i, const unsigned int* q_j, unsigned int* q_n,
                                          const float* __restrict__ sub, const int32_t* __restrict__ sublabel,
                                          const float* __restrict__ feature, const int32_t* __restrict__ label, int emb,
                                          unsigned int* h) {
  const unsigned int n_q = *q_n < (unsigned)kRocQueue ? *q_n : (unsigned)kRocQueue;
  for (unsigned int e = threadIdx.x; e < n_q; e += kRocThreads) {
    const int64_t i = q_i[e], j = q_j[e];
    int bin = (int)roc_exact_x(sub + i * emb, feature + j * emb, emb);
    bin = bin < 0 ? 0 : (bin > kRocBins - 1 ? kRocBins - 1 : bin);
    atomicAdd(&h[2 * bin + (sublabel[i] != label[j] ? 1 : 0)], 1u);
  }
  __syncthreads();
  if (threadIdx.x == 0) *q_n = 0u;
  __syncthreads();
}

__global__ void __launch_bounds__(kRocThreads, 2)
roc_hist2_kernel(const float* __restrict__ feature, const int32_t* __restrict__ label, int64_t n,
                 const float* __restrict__ sub, const int32_t* __restrict__ sublabel, int64_t n_sub, int64_t sub_offset,
                 int emb, float coef, unsigned long long* __restrict__ hist) {
  __shared__ float As[kRocTile][kRocK + 1];
  __shared__ float Bs[kRocTile][kRocK + 1];
  __shared__ float nA[kRocTile], nB[kRocTile];
  __shared__ unsigned int h[2 * kRocBins];
  __shared__ unsigned int q_i[kRocQueue], q_j[kRocQueue];   // pairs that need the exact chain, gathered over several tiles
  __shared__ unsigned int q_n;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int lane = tid & 31, wrow = tid >> 5;
  if (tid == 0) q_n = 0u;
  for (int b = tid; b < 2 * kRocBins; b += kRocThreads) h[b] = 0u;
  __syncthreads();

  const int64_t n_ti = (n_sub + kRocTile - 1) / kRocTile;
  const int64_t n_tj = (n + kRocTile - 1) / kRocTile;
  const int64_t total = n_ti * n_tj;
  int tiles_done = 0;
  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int64_t i0 = (t / n_tj) * kRocTile;
    const int64_t j0 = (t % n_tj) * kRocTile;
    const int64_t j_last = (j0 + kRocTile - 1 < n - 1) ? j0 + kRocTile - 1 : n - 1;
    if (j_last <= sub_offset + i0) continue;

    float acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) acc[u][v] = 0.f;
    float ssa[kRocTile / 8], ssb[kRocTile / 8];          // this lane's share of |row|^2 for the rows its warp loads
#pragma unroll
    for (int r = 0; r < kRocTile / 8; ++r) { ssa[r] = 0.f; ssb[r] = 0.f; }

    for (int k0 = 0; k0 < emb; k0 += kRocK) {
      __syncthreads();
      {
        const bool k_ok = (k0 + lane) < emb;
#pragma unroll
        for (int r = 0; r < kRocTile / 8; ++r) {
          const int row = wrow + 8 * r;
          const int64_t gi = i0 + row, gj = j0 + row;
          const float a = (k_ok && gi < n_sub) ? sub[gi * emb + k0 + lane] : 0.f;
          const float b = (k_ok && gj < n) ? feature[gj * emb + k0 + lane] : 0.f;
          As[row][lane] = a;
          Bs[row][lane] = b;
          ssa[r] = fmaf(a, a, ssa[r]);
          ssb[r] = fmaf(b, b, ssb[r]);
        }
      }
      __syncthreads();
      const int kc = (emb - k0 < kRocK) ? emb - k0 : kRocK;
      float part[4][4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) part[u][v] = 0.f;
#pragma unroll 4
      for (int kk = 0; kk < kc; ++kk) {
        float a[4], b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) a[u] = As[ty + 16 * u][kk];
#pragma unroll
        for (int v = 0; v < 4; ++v) b[v] = Bs[tx + 16 * v][kk];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) part[u][v] = fmaf(a[u], b[v], part[u][v]);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] += part[u][v];
    }
    // row norms (upper bounds): lanes of a warp hold the 32 k-residues of the rows that warp loaded
#pragma unroll
    for (int r = 0; r < kRocTile / 8; ++r) {
      const float sa = warp_sum(ssa[r]), sb = warp_sum(ssb[r]);
      if (lane == 0) {
        nA[wrow + 8 * r] = sqrtf(sa) * 1.001f;
        nB[wrow + 8 * r] = sqrtf(sb) * 1.001f;
      }
    }
    __syncthreads();

#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = i0 + ty + 16 * u;
      if (i >= n_sub) continue;
      const int32_t li = sublabel[i];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int64_t j = j0 + tx + 16 * v;
        if (j >= n || sub_offset + i >= j) continue;
        double x = __dmul_rn(__dadd_rn((double)acc[u][v], 1.0), 1000.0);
        const double e = 1000.0 * (double)coef * (double)nA[ty + 16 * u] * (double)nB[tx + 16 * v] + 1e-6;
        const double fl = floor(x);
        if (!(x - fl > e && fl + 1.0 - x > e && x > e)) {              // could be on a bin edge (or below zero, or NaN): exact chain
          const unsigned int slot = atomicAdd(&q_n, 1u);
          if (slot < (unsigned)kRocQueue) {                             // later, 256 pairs at a time with every lane busy
            q_i[slot] = (unsigned int)i;
            q_j[slot] = (unsigned int)j;
            continue;
          }
          x = roc_exact_x(sub + i * emb, feature + j * emb, emb);       // queue full (adversarial input): do it here
        }
        int bin = (int)x;
        bin = bin < 0 ? 0 : (bin > kRocBins - 1 ? kRocBins - 1 : bin);
        atomicAdd(&h[2 * bin + (li != label[j] ? 1 : 0)], 1u);
      }
    }
    __syncthreads();
    if (q_n >= (unsigned)(kRocQueue - kRocQueue / 4)) roc_drain(q_i, q_j, &q_n, sub, sublabel, feature, label, emb, h);   // uniform
    if (++tiles_done == kRocFlushTiles) {
      roc_flush(h, hist);
      tiles_done = 0;
    }
  }
  __syncthreads();
  roc_drain(q_i, q_j, &q_n, sub, sublabel, feature, label, emb, h);
  roc_flush(h, hist);
}

static int g_roc_mode = 1;      // 1 (default): two-tier, integer-identical and 2x faster on B200 (profiles/README.md r02a); 0: exact chain for every pair

static int roc_grid(int64_t total) {
  int64_t g = (int64_t)sm_count() * 2;
  if (g > total) g = total;
  return (int)(g < 1 ? 1 : g);
}

}  // namespace pfc

using namespace pfc;

extern "C" {

int pfc_roc_histogram(const float* feature, const int32_t* label, int64_t n, const float* subfeature,
                      const int32_t* sublabel, int64_t n_sub, int64_t sub_offset, int emb, int64_t* hist, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_roc_histogram");
  PFC_REQUIRE(n >= 0 && n_sub >= 0 && sub_offset >= 0 && emb >= 0 && hist, PFC_E_ARG, "pfc_roc_histogram: bad argument");
  if (n == 0 || n_sub == 0) return 0;
  PFC_REQUIRE(feature && label && subfeature && sublabel, PFC_E_ARG, "pfc_roc_histogram: null pointer");
  const int64_t total = ((n_sub + kRocTile - 1) / kRocTile) * ((n + kRocTile - 1) / kRocTile);
  if (g_roc_mode == 1 && n < (1ll << 32) && n_sub < (1ll << 32)) {        // the pair queue stores 32-bit row ids
    const float coef = (float)(kRocK + (emb + kRocK - 1) / kRocK + 2) * 5.9604645e-8f;      // (32 + n_slices + 2) * 2^-24
    roc_hist2_kernel<<<roc_grid(total), kRocThreads, 0, as_stream(stream)>>>(
        feature, label, n, subfeature, sublabel, n_sub, sub_offset, emb, coef, reinterpret_cast<unsigned long long*>(hist));
  } else {
    roc_hist_kernel<<<roc_grid(total), kRocThreads, 0, as_stream(stream)>>>(
        feature, label, n, subfeature, sublabel, n_sub, sub_offset, emb, reinterpret_cast<unsigned long long*>(hist));
  }
  PFC_LAUNCH_CHECK();
  return 0;
}

// developer hook (not in the reference-facing header): 0 = exact chain for every pair, 1 = two-tier kernel
int pfc_set_roc_mode(int mode) {
  if (mode != 0 && mode != 1) return PFC_E_ARG;
  g_roc_mode = mode;
  return 0;
}

}  // extern "C"
