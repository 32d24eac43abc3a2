// 1:1 template verification (the IJB-B / IJB-C protocol of FedFR's ijbc_all.py / ijbc_conti.py): template pooling,
// pair scores and exact TAR@FAR.  Every step is pinned so that a plain C restatement reproduces it bit for bit.
//
// Pooling (one CTA per template, threads over E, sequential over medias and images -- no atomics, deterministic).  The
// caller hands in the images in ascending (template, media, row) order as a CSR: order[] lists image rows,
// media_start[] cuts it into medias, tmpl_start[] cuts the medias into templates.
//     x_i   = feats_i  or  fl32(feats_i * weights_i)
//     media = x_first + x_2 + ...  (fp32, image order), then / (float)count when count > 1
//     t     = media_first + media_2 + ...  (fp32, ascending media id)
//     out_k = (float)((double)t_k / max(sqrt(sum_k (double)t_k^2), 1e-12))     fp64 adds over ascending k
//
// Pair scores: score = (float)dot_chain(0, a, b, E) -- the ROC histogram's chain.  A CTA owns 128 consecutive pairs (one
// per thread) and stages 32-wide k slices of their rows in shared memory; the distinct runs of row1 in the tile are
// staged once each, so a pair list grouped by its first template (as IJB-C's is) reads that row once per tile.
//
// TAR@FAR: scores map to order-preserving uint32 keys (-0.0 folded onto +0.0, NaN counted and left out).  A 4 x 8-bit
// radix select over the impostor keys finds the (k+1)-th largest for up to 8 FARs at once: per pass, the unresolved
// selections with the same key prefix share one histogram (prefixes of one length are equal or disjoint, so each key
// lands in at most one), counted with warp-aggregated shared atomics; the last block to finish a pass picks the bins.
// One counting pass then accepts score > threshold for every FAR.  No sort of the scores.
#include "common.cuh"
#include "../../fedfr_b200/csrc/dot_chain.cuh"

namespace pfc {

constexpr int kPoolThreads = 128;
constexpr int kPoolMaxEmb = 4096;

__device__ __forceinline__ float pool_x(const float* __restrict__ feats, const float* __restrict__ weights, int64_t row,
                                        int emb, int k) {
  const float f = feats[row * emb + k];
  return weights ? __fmul_rn(f, weights[row]) : f;
}

__global__ void __launch_bounds__(kPoolThreads)
template_pool_kernel(const float* __restrict__ feats, const float* __restrict__ weights, int emb,
                     const int64_t* __restrict__ order, const int64_t* __restrict__ media_start,
                     const int64_t* __restrict__ tmpl_start, float* __restrict__ out) {
  __shared__ float t_sh[kPoolMaxEmb];
  __shared__ double nrm_sh;
  const int64_t tpl = blockIdx.x;
  const int64_t m0 = tmpl_start[tpl], m1 = tmpl_start[tpl + 1];
  for (int k = threadIdx.x; k < emb; k += kPoolThreads) {
    float t = 0.f;
    for (int64_t m = m0; m < m1; ++m) {
      const int64_t i0 = media_start[m], i1 = media_start[m + 1];
      float s = pool_x(feats, weights, order[i0], emb, k);
      for (int64_t i = i0 + 1; i < i1; ++i) s = __fadd_rn(s, pool_x(feats, weights, order[i], emb, k));
      if (i1 - i0 > 1) s = s / (float)(i1 - i0);
      t = m == m0 ? s : __fadd_rn(t, s);
    }
    t_sh[k] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {                      // the pinned order: one fp64 chain over ascending k
    double ss = 0.0;
    for (int k = 0; k < emb; ++k) ss = __dadd_rn(ss, __dmul_rn((double)t_sh[k], (double)t_sh[k]));
    const double nrm = sqrt(ss);
    nrm_sh = nrm > 1e-12 ? nrm : 1e-12;
  }
  __syncthreads();
  const double nrm = nrm_sh;
  for (int k = threadIdx.x; k < emb; k += kPoolThreads) out[tpl * emb + k] = (float)((double)t_sh[k] / nrm);
}

constexpr int kPairTile = 128;
constexpr int kPairK = 32;

__global__ void __launch_bounds__(kPairTile)
pair_score_kernel(const float* __restrict__ tf, int64_t n_rows, int emb, const int64_t* __restrict__ row1,
                  const int64_t* __restrict__ row2, int64_t n_pairs, float* __restrict__ out) {
  __shared__ float As[kPairTile][kPairK + 1];
  __shared__ float Bs[kPairTile][kPairK + 1];
  __shared__ int64_t ra[kPairTile], rb[kPairTile];
  __shared__ unsigned int warp_runs[kPairTile / 32];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t p = (int64_t)blockIdx.x * kPairTile + tid;
  int64_t a = -1, b = -1;                      // -1: a zero row (past the end, or a row out of range -> NaN score)
  if (p < n_pairs) {
    a = row1[p];
    b = row2[p];
    if (a < 0 || a >= n_rows || b < 0 || b >= n_rows) a = b = -1;
  }
  ra[tid] = a;
  rb[tid] = b;
  __syncthreads();
  const bool first = tid == 0 || ra[tid - 1] != a;             // a new run of row1 starts here
  const unsigned int m = __ballot_sync(0xffffffffu, first);
  if (lane == 0) warp_runs[w] = (unsigned int)__popc(m);
  __syncthreads();
  unsigned int base = 0, n_a = 0;
  for (int v = 0; v < kPairTile / 32; ++v) {
    if (v < w) base += warp_runs[v];
    n_a += warp_runs[v];
  }
  const int slot = (int)(base + (unsigned int)__popc(m & (0xffffffffu >> (31 - lane)))) - 1;   // this pair's run
  if (first) ra[slot] = a;                     // every read of ra[] above happened before the barrier
  __syncthreads();

  double acc = 0.0;
  for (int k0 = 0; k0 < emb; k0 += kPairK) {
    __syncthreads();                           // the previous slice has been consumed
    const bool k_ok = k0 + lane < emb;
    for (int r = w; r < (int)n_a; r += kPairTile / 32) {
      const int64_t g = ra[r];
      As[r][lane] = (k_ok && g >= 0) ? tf[g * emb + k0 + lane] : 0.f;
    }
#pragma unroll 8
    for (int r = w; r < kPairTile; r += kPairTile / 32) {
      const int64_t g = rb[r];
      Bs[r][lane] = (k_ok && g >= 0) ? tf[g * emb + k0 + lane] : 0.f;
    }
    __syncthreads();
    acc = dot_chain(acc, As[slot], Bs[tid], emb - k0 < kPairK ? emb - k0 : kPairK);
  }
  if (p < n_pairs) out[p] = a >= 0 ? (float)acc : nanf("");
}

constexpr int kTarMaxFar = 8;
constexpr int kTarThreads = 256;

struct TarFars {
  double f[kTarMaxFar];
  int n;
};

struct TarState {
  unsigned int hist[kTarMaxFar][256];          // per prefix slot
  unsigned int slot_prefix[kTarMaxFar];        // distinct key prefixes of the unresolved selections
  unsigned int n_slot;
  int q_slot[kTarMaxFar];                      // slot of selection q, -1 once resolved
  unsigned int prefix[kTarMaxFar];
  unsigned int rank[kTarMaxFar];               // 1-based rank of the wanted key inside its prefix bucket, from the top
  unsigned int thr_key[kTarMaxFar];            // accept iff key > thr_key
  unsigned int blocks_done;
  unsigned long long n_gen, n_imp, n_nan;
  unsigned long long acc_gen[kTarMaxFar], acc_imp[kTarMaxFar];
};

// Order-preserving key of an fp32 score given as its bits: larger score -> larger key; -0.0 and +0.0 -> one key.
// NaN -> 0, which no number maps to (0 is the key of the bit pattern 0xffffffff, itself a NaN).
__device__ __forceinline__ unsigned int tar_key(unsigned int u) {
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0u;
  if ((u & 0x7fffffffu) == 0u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void tar_init_kernel(TarState* st) {
  unsigned int* h = &st->hist[0][0];
  for (int i = threadIdx.x; i < kTarMaxFar * 256; i += blockDim.x) h[i] = 0u;
  if (threadIdx.x < kTarMaxFar) {
    const int q = threadIdx.x;
    st->slot_prefix[q] = 0u; st->q_slot[q] = 0; st->prefix[q] = 0u; st->rank[q] = 0u; st->thr_key[q] = 0u;
    st->acc_gen[q] = 0ull; st->acc_imp[q] = 0ull;
  }
  if (threadIdx.x == 0) {
    st->n_slot = 1u;                           // the first pass: one histogram of the top byte for every selection
    st->blocks_done = 0u;
    st->n_gen = st->n_imp = st->n_nan = 0ull;
  }
}

// Run by one thread of the last block of a pass: pick each unresolved selection's bin, then regroup by prefix.
__device__ void tar_select(TarState* st, int pass, const TarFars& fars) {
  volatile TarState* v = st;
  const unsigned int shift = pass * 8;
  if (pass == 3) {
    const unsigned long long n_imp = v->n_imp;
    for (int q = 0; q < fars.n; ++q) {
      const unsigned long long k = (unsigned long long)floor(fars.f[q] * (double)n_imp);
      if (k >= n_imp) { v->q_slot[q] = -1; v->thr_key[q] = tar_key(0xff800000u); }      // tau = -inf
      else { v->q_slot[q] = 0; v->rank[q] = (unsigned int)(k + 1); v->prefix[q] = 0u; }
    }
  }
  for (int q = 0; q < fars.n; ++q) {
    const int s = v->q_slot[q];
    if (s < 0) continue;
    const unsigned int r = v->rank[q];
    unsigned int cum = 0;
    int b = 255;
    for (; b > 0; --b) {
      if (cum + v->hist[s][b] >= r) break;
      cum += v->hist[s][b];
    }
    v->prefix[q] = v->prefix[q] | ((unsigned int)b << shift);
    v->rank[q] = r - cum;
    if (pass == 0) { v->thr_key[q] = v->prefix[q]; v->q_slot[q] = -1; }
  }
  unsigned int n_slot = 0;
  for (int q = 0; q < fars.n; ++q) {
    if (v->q_slot[q] < 0) continue;
    unsigned int s = 0;
    while (s < n_slot && v->slot_prefix[s] != v->prefix[q]) ++s;
    if (s == n_slot) v->slot_prefix[n_slot++] = v->prefix[q];
    v->q_slot[q] = (int)s;
  }
  v->n_slot = n_slot;
  v->blocks_done = 0u;
}

// One radix pass over byte `pass` (3 = most significant) of the impostor keys; pass 3 also counts the classes.
__global__ void __launch_bounds__(kTarThreads)
tar_radix_kernel(const unsigned int* __restrict__ bits, const unsigned char* __restrict__ issame, int64_t n, int pass,
                 TarFars fars, TarState* st) {
  __shared__ unsigned int sh[kTarMaxFar][256];
  __shared__ unsigned int s_prefix[kTarMaxFar];
  __shared__ bool is_last;
  const unsigned int n_slot = st->n_slot;
  if (n_slot == 0) return;                     // every selection resolved (the same for all blocks)
  for (int i = threadIdx.x; i < kTarMaxFar * 256; i += kTarThreads) sh[i >> 8][i & 255] = 0u;
  if (threadIdx.x < kTarMaxFar) s_prefix[threadIdx.x] = st->slot_prefix[threadIdx.x];
  __syncthreads();
  const unsigned int shift = pass * 8;
  const unsigned int hi_mask = pass == 3 ? 0u : (0xffffffffu << (shift + 8));
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * kTarThreads;
  const int64_t first = (int64_t)blockIdx.x * kTarThreads + threadIdx.x;
  const int64_t n_iter = (n + stride - 1) / stride;                    // the same for every thread: match is warp-convergent
  unsigned int gen = 0, imp = 0, nan = 0;
  for (int64_t it = 0; it < n_iter; ++it) {
    const int64_t i = first + it * stride;
    unsigned int d = 0x10000u + (unsigned int)lane;                    // not counted: a digit of its own
    if (i < n) {
      const unsigned int key = tar_key(bits[i]);
      const bool g = issame[i] != 0;
      nan += key == 0u;
      gen += key != 0u && g;
      imp += key != 0u && !g;
      if (key != 0u && !g) {
        for (unsigned int s = 0; s < n_slot; ++s)
          if ((key & hi_mask) == s_prefix[s]) { d = (s << 8) | ((key >> shift) & 0xffu); break; }
      }
    }
    // impostor scores crowd into a few top bytes: lanes with the same (slot, digit) elect one to add their count
    const unsigned int peers = __match_any_sync(0xffffffffu, d);
    if (d < 0x10000u && lane == __ffs((int)peers) - 1) atomicAdd(&sh[d >> 8][d & 255u], (unsigned int)__popc(peers));
  }
  if (pass == 3) {
    for (int o = 16; o > 0; o >>= 1) {
      gen += __shfl_xor_sync(0xffffffffu, gen, o);
      imp += __shfl_xor_sync(0xffffffffu, imp, o);
      nan += __shfl_xor_sync(0xffffffffu, nan, o);
    }
    if (lane == 0) {
      atomicAdd(&st->n_gen, (unsigned long long)gen);
      atomicAdd(&st->n_imp, (unsigned long long)imp);
      atomicAdd(&st->n_nan, (unsigned long long)nan);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < (int)n_slot * 256; i += kTarThreads)
    if (sh[i >> 8][i & 255]) atomicAdd(&st->hist[i >> 8][i & 255], sh[i >> 8][i & 255]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(&st->blocks_done, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x == 0) tar_select(st, pass, fars);
  __syncthreads();
  for (int i = threadIdx.x; i < kTarMaxFar * 256; i += kTarThreads) st->hist[i >> 8][i & 255] = 0u;
}

// Accepted genuine / impostor pairs (score > threshold) for every FAR.
__global__ void __launch_bounds__(kTarThreads)
tar_accept_kernel(const unsigned int* __restrict__ bits, const unsigned char* __restrict__ issame, int64_t n, int n_far,
                  TarState* st) {
  __shared__ unsigned int s_thr[kTarMaxFar];
  if (threadIdx.x < kTarMaxFar) s_thr[threadIdx.x] = st->thr_key[threadIdx.x];
  __syncthreads();
  unsigned int ag[kTarMaxFar], ai[kTarMaxFar];
#pragma unroll
  for (int q = 0; q < kTarMaxFar; ++q) ag[q] = ai[q] = 0u;
  for (int64_t i = (int64_t)blockIdx.x * kTarThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kTarThreads) {
    const unsigned int key = tar_key(bits[i]);
    if (key == 0u) continue;
    const bool g = issame[i] != 0;
#pragma unroll
    for (int q = 0; q < kTarMaxFar; ++q) {
      const unsigned int acc = (q < n_far && key > s_thr[q]) ? 1u : 0u;
      ag[q] += g ? acc : 0u;
      ai[q] += g ? 0u : acc;
    }
  }
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < kTarMaxFar; ++q) {
    for (int o = 16; o > 0; o >>= 1) {
      ag[q] += __shfl_xor_sync(0xffffffffu, ag[q], o);
      ai[q] += __shfl_xor_sync(0xffffffffu, ai[q], o);
    }
    if (lane == 0 && q < n_far) {
      atomicAdd(&st->acc_gen[q], (unsigned long long)ag[q]);
      atomicAdd(&st->acc_imp[q], (unsigned long long)ai[q]);
    }
  }
}

// counts = [n_gen, n_imp, n_nan, acc_gen_0, acc_imp_0, acc_gen_1, ...]; thresholds as fp32
__global__ void tar_finish_kernel(const TarState* st, int n_far, int64_t* counts, unsigned int* thr_bits) {
  const int q = threadIdx.x;
  if (q == 0) {
    counts[0] = (int64_t)st->n_gen;
    counts[1] = (int64_t)st->n_imp;
    counts[2] = (int64_t)st->n_nan;
  }
  if (q < n_far) {
    counts[3 + 2 * q] = (int64_t)st->acc_gen[q];
    counts[4 + 2 * q] = (int64_t)st->acc_imp[q];
    const unsigned int key = st->thr_key[q];
    thr_bits[q] = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  }
}

}  // namespace pfc

using namespace pfc;

extern "C" {

int pfc_template_pool(const float* feats, const float* weights, const int64_t* order, const int64_t* media_start,
                      const int64_t* tmpl_start, int64_t n_templates, int emb, float* template_feats, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_template_pool");
  PFC_REQUIRE(n_templates >= 0 && emb > 0, PFC_E_ARG, "pfc_template_pool: bad size");
  PFC_REQUIRE(emb <= kPoolMaxEmb && n_templates < (1ll << 31), PFC_E_SHAPE, "pfc_template_pool: emb > 4096 or too many templates");
  if (n_templates == 0) return 0;
  PFC_REQUIRE(feats && order && media_start && tmpl_start && template_feats, PFC_E_ARG, "pfc_template_pool: null pointer");
  template_pool_kernel<<<(unsigned int)n_templates, kPoolThreads, 0, as_stream(stream)>>>(
      feats, weights, emb, order, media_start, tmpl_start, template_feats);
  PFC_LAUNCH_CHECK();
  return 0;
}

int pfc_pair_scores(const float* template_feats, int64_t n_templates, int emb, const int64_t* row1, const int64_t* row2,
                    int64_t n_pairs, float* scores, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_pair_scores");
  PFC_REQUIRE(n_templates >= 0 && emb > 0 && n_pairs >= 0, PFC_E_ARG, "pfc_pair_scores: bad size");
  if (n_pairs == 0) return 0;
  PFC_REQUIRE(template_feats && row1 && row2 && scores, PFC_E_ARG, "pfc_pair_scores: null pointer");
  const int64_t tiles = (n_pairs + kPairTile - 1) / kPairTile;
  PFC_REQUIRE(tiles < (1ll << 31), PFC_E_SHAPE, "pfc_pair_scores: too many pairs");
  pair_score_kernel<<<(unsigned int)tiles, kPairTile, 0, as_stream(stream)>>>(template_feats, n_templates, emb, row1, row2,
                                                                               n_pairs, scores);
  PFC_LAUNCH_CHECK();
  return 0;
}

size_t pfc_tar_at_far_workspace_bytes(int64_t n) {
  (void)n;
  return sizeof(TarState);
}

int pfc_tar_at_far(const float* scores, const unsigned char* issame, int64_t n, const double* fars_host, int n_far,
                   int64_t* counts, float* thresholds, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_tar_at_far");
  PFC_REQUIRE(scores && issame && fars_host && counts && thresholds && workspace && n > 0, PFC_E_ARG,
              "pfc_tar_at_far: bad argument");
  PFC_REQUIRE(n_far >= 1 && n_far <= kTarMaxFar, PFC_E_ARG, "pfc_tar_at_far: 1 to 8 FARs per call");
  PFC_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 8 == 0, PFC_E_ARG, "pfc_tar_at_far: workspace not 8-byte aligned");
  PFC_REQUIRE(n < (1ll << 31), PFC_E_SHAPE, "pfc_tar_at_far: more than 2^31 - 1 scores");
  PFC_REQUIRE(workspace_bytes >= pfc_tar_at_far_workspace_bytes(n), PFC_E_WORKSPACE, "pfc_tar_at_far: workspace too small");
  TarFars fars;
  fars.n = n_far;
  for (int q = 0; q < kTarMaxFar; ++q) {
    fars.f[q] = q < n_far ? fars_host[q] : 1.0;
    PFC_REQUIRE(fars.f[q] > 0.0 && fars.f[q] <= 1.0, PFC_E_ARG, "pfc_tar_at_far: a FAR outside (0, 1]");
  }
  cudaStream_t st = as_stream(stream);
  auto* state = reinterpret_cast<TarState*>(workspace);
  const auto* bits = reinterpret_cast<const unsigned int*>(scores);
  int64_t nb = (n + kTarThreads * 8 - 1) / (kTarThreads * 8);
  if (nb > 2 * sm_count()) nb = 2 * sm_count();
  tar_init_kernel<<<1, 256, 0, st>>>(state);
  PFC_LAUNCH_CHECK();
  for (int pass = 3; pass >= 0; --pass) {
    tar_radix_kernel<<<(int)nb, kTarThreads, 0, st>>>(bits, issame, n, pass, fars, state);
    PFC_LAUNCH_CHECK();
  }
  tar_accept_kernel<<<(int)nb, kTarThreads, 0, st>>>(bits, issame, n, n_far, state);
  PFC_LAUNCH_CHECK();
  tar_finish_kernel<<<1, 32, 0, st>>>(state, n_far, counts, reinterpret_cast<unsigned int*>(thresholds));
  PFC_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
