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
// TAR@FAR: scores map to order-preserving uint32 keys (tar_key in score_key.cuh: -0.0 folded onto +0.0, NaN counted
// and left out).  A 4 x 8-bit radix select over the impostor keys finds the (k+1)-th largest for up to 8 FARs at once:
// per pass, the unresolved selections with the same key prefix share one histogram (prefixes of one length are equal
// or disjoint, so each key lands in at most one), counted with warp-aggregated shared atomics; the last block to finish
// a pass picks the bins.  One counting pass then accepts score > threshold for every FAR.  No sort of the scores.
//
// ROC curve (sklearn.metrics.roc_curve with drop_intermediate): the TAR keys, complemented so that ascending order is
// descending score, are sorted with a stable 4 x 8-bit LSD radix sort that carries the class byte (per pass: a tile
// histogram, a scan of each digit's row over the tiles, a scatter ranked with match.any).  Reduce-then-scan passes over
// the sorted keys then cut it into runs of one key (tps = genuine up to the run's end, fps = its position + 1 - tps),
// apply sklearn's thinning stencil to the runs and compact the kept points in order.  Integer counts and scans only: the
// result does not depend on the schedule.
//
// K-fold verification accuracy (insightface's eval/verification.py evaluate / calculate_roc, the per-round LFW / CFP-FP
// / AgeDB test): one warp per pair fuses, normalises and takes the squared distance of the two rows with the fp64 sums
// pinned in the header, and bins the distance on the threshold grid by a binary search.  One CTA per fold then builds
// the fold's integer histogram of bins by class (shared atomics) and adds it into the all-pairs totals (integer global
// atomics); one CTA per fold scans its histogram and the totals into test and train counts, picks the first train
// maximum and writes its accuracy and test rates; a last pass takes the fold-order mean of the rates.  Integer counts,
// fixed-order sums: the result does not depend on the schedule.
#include "common.cuh"
#include "../../fedfr_b200/csrc/dot_chain.cuh"
#include "../../fedfr_b200/csrc/score_key.cuh"

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

constexpr int kRocThreads = 256;               // every ROC kernel runs 256 threads: one per digit where it works on digits
constexpr int kRocItems = 8;
constexpr int kRocTile = kRocThreads * kRocItems;
constexpr int kRocWarps = kRocThreads / 32;
constexpr int kRocColTiles = 32;               // tiles per block of the digit-offset scan

struct RocState {
  unsigned long long n_gen, n_imp, n_bad;      // finite genuine, finite impostor, NaN or +-inf scores
  unsigned int run_totals[2];                  // distinct keys (runs), genuine pairs (from the run scan)
  unsigned int n_keep;                         // runs kept by the thinning
};

// Sort key: tar_key complemented, so that ascending keys are descending scores.  Counts and positions fit 32 bits: n < 2^31.
__device__ __forceinline__ unsigned int roc_sort_key(unsigned int u) { return ~tar_key(u); }

__device__ __forceinline__ double roc_key_value(unsigned int sort_key) {
  const unsigned int key = ~sort_key;
  union { unsigned int u; float f; } v;
  v.u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  return (double)v.f;
}

// Exclusive prefix sum of v over the block's threads (blockDim = kRocThreads); the block's sum -> *total.
__device__ unsigned int roc_block_scan(unsigned int v, unsigned int* total) {
  __shared__ unsigned int warp_tot[kRocWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int y = __shfl_sync(0xffffffffu, x, lane >= o ? lane - o : lane);
    if (lane >= o) x += y;
  }
  if (lane == 31) warp_tot[w] = x;
  __syncthreads();
  unsigned int before = 0, all = 0;
  for (int i = 0; i < kRocWarps; ++i) {
    before += i < w ? warp_tot[i] : 0u;
    all += warp_tot[i];
  }
  __syncthreads();                             // warp_tot is rewritten by the next call
  *total = all;
  return before + x - v;
}

// One sort pass, step 1: hist[tile][digit] = count of `digit` at bit `shift` in this tile.  The first pass reads the scores
// (bits, issame) and counts the classes; later passes read the previous pass's keys.
__global__ void __launch_bounds__(kRocThreads)
roc_hist_kernel(const unsigned int* __restrict__ bits, const unsigned char* __restrict__ issame,
                const unsigned int* __restrict__ keys, int64_t n, int shift, unsigned int* __restrict__ hist, RocState* st) {
  __shared__ unsigned int h[256];
  const int lane = threadIdx.x & 31;
  h[threadIdx.x] = 0u;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kRocTile;
  unsigned int gen = 0, imp = 0, bad = 0;
  for (int r = 0; r < kRocItems; ++r) {
    const int64_t i = base + r * kRocThreads + threadIdx.x;
    unsigned int d = 0x100u + (unsigned int)lane;                      // past the end: a digit of its own, not counted
    if (i < n) {
      unsigned int key;
      if (bits) {
        const unsigned int u = bits[i];
        const bool finite = (u & 0x7fffffffu) < 0x7f800000u, g = issame[i] != 0;
        bad += !finite;
        gen += finite && g;
        imp += finite && !g;
        key = roc_sort_key(u);
      } else {
        key = keys[i];
      }
      d = (key >> shift) & 0xffu;
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, d);
    if (d < 0x100u && lane == __ffs((int)peers) - 1) atomicAdd(&h[d], (unsigned int)__popc(peers));
  }
  if (bits) {                                  // the same for the whole grid
    unsigned int t;
    roc_block_scan(gen, &t);
    if (threadIdx.x == 0) atomicAdd(&st->n_gen, (unsigned long long)t);
    roc_block_scan(imp, &t);
    if (threadIdx.x == 0) atomicAdd(&st->n_imp, (unsigned long long)t);
    roc_block_scan(bad, &t);
    if (threadIdx.x == 0) atomicAdd(&st->n_bad, (unsigned long long)t);
  }
  __syncthreads();
  hist[(int64_t)blockIdx.x * 256 + threadIdx.x] = h[threadIdx.x];
}

// Step 2: part[g][digit] = sum of hist[tile][digit] over the kRocColTiles tiles of group g.
__global__ void __launch_bounds__(kRocThreads)
roc_col_sum_kernel(const unsigned int* __restrict__ hist, int64_t n_tiles, unsigned int* __restrict__ part) {
  const int64_t t0 = (int64_t)blockIdx.x * kRocColTiles;
  const int64_t t1 = t0 + kRocColTiles < n_tiles ? t0 + kRocColTiles : n_tiles;
  unsigned int s = 0;
  for (int64_t t = t0; t < t1; ++t) s += hist[t * 256 + threadIdx.x];
  part[(int64_t)blockIdx.x * 256 + threadIdx.x] = s;
}

// Step 3 (one block, thread = digit): part[g][digit] = position of group g's first key with that digit in the output.
__global__ void __launch_bounds__(kRocThreads)
roc_col_scan_kernel(unsigned int* __restrict__ part, int64_t n_groups) {
  const int d = threadIdx.x;
  unsigned int run = 0;
  for (int64_t g = 0; g < n_groups; ++g) {
    const unsigned int c = part[g * 256 + d];
    part[g * 256 + d] = run;
    run += c;
  }
  unsigned int total;
  const unsigned int digit_base = roc_block_scan(run, &total);
  for (int64_t g = 0; g < n_groups; ++g) part[g * 256 + d] += digit_base;
}

// Step 4: hist[tile][digit] = position of the tile's first key with that digit in the output.
__global__ void __launch_bounds__(kRocThreads)
roc_col_apply_kernel(unsigned int* __restrict__ hist, int64_t n_tiles, const unsigned int* __restrict__ part) {
  const int64_t t0 = (int64_t)blockIdx.x * kRocColTiles;
  const int64_t t1 = t0 + kRocColTiles < n_tiles ? t0 + kRocColTiles : n_tiles;
  unsigned int run = part[(int64_t)blockIdx.x * 256 + threadIdx.x];
  for (int64_t t = t0; t < t1; ++t) {
    const unsigned int c = hist[t * 256 + threadIdx.x];
    hist[t * 256 + threadIdx.x] = run;
    run += c;
  }
}

// Step 5: stable scatter.  Warp w of a tile owns its keys w * 256 ... w * 256 + 255 in rounds of 32; within a round,
// lanes with one digit are ranked by match.any and their leader advances the warp's count of that digit.  Tile order is
// (warp, round, lane) = key order, so equal digits keep their order.
__global__ void __launch_bounds__(kRocThreads)
roc_scatter_kernel(const unsigned int* __restrict__ bits, const unsigned char* __restrict__ issame,
                   const unsigned int* __restrict__ keys_in, const unsigned char* __restrict__ cls_in, int64_t n, int shift,
                   const unsigned int* __restrict__ hist, unsigned int* __restrict__ keys_out,
                   unsigned char* __restrict__ cls_out) {
  __shared__ unsigned int cnt[kRocWarps][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < kRocWarps * 256; i += kRocThreads) cnt[i >> 8][i & 255] = 0u;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * kRocTile + w * (kRocItems * 32);
  unsigned int key[kRocItems], rank[kRocItems];
  unsigned char cls[kRocItems];
#pragma unroll
  for (int r = 0; r < kRocItems; ++r) {
    const int64_t i = base + r * 32 + lane;
    unsigned int d = 0x100u + (unsigned int)lane;
    key[r] = 0u;
    cls[r] = 0;
    if (i < n) {
      if (bits) {
        key[r] = roc_sort_key(bits[i]);
        cls[r] = issame[i] != 0;
      } else {
        key[r] = keys_in[i];
        cls[r] = cls_in[i];
      }
      d = (key[r] >> shift) & 0xffu;
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, d);
    const int leader = __ffs((int)peers) - 1;
    unsigned int before = 0;
    if (lane == leader && d < 0x100u) {
      before = cnt[w][d];
      cnt[w][d] = before + (unsigned int)__popc(peers);
    }
    before = __shfl_sync(0xffffffffu, before, leader);
    rank[r] = before + (unsigned int)__popc(peers & ((1u << lane) - 1u));
    __syncwarp();
  }
  __syncthreads();
  {                                            // thread = digit: warp counts -> output positions
    unsigned int run = hist[(int64_t)blockIdx.x * 256 + threadIdx.x];
    for (int v = 0; v < kRocWarps; ++v) {
      const unsigned int c = cnt[v][threadIdx.x];
      cnt[v][threadIdx.x] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kRocItems; ++r) {
    if (base + r * 32 + lane < n) {
      const unsigned int dst = cnt[w][(key[r] >> shift) & 0xffu] + rank[r];
      keys_out[dst] = key[r];
      cls_out[dst] = cls[r];
    }
  }
}

// Sorted key i closes a run of equal keys.
__device__ __forceinline__ bool roc_run_end(const unsigned int* __restrict__ keys, int64_t n, int64_t i) {
  return i == n - 1 || keys[i + 1] != keys[i];
}

// sums[tile] = {run ends, genuine} in this tile of the sorted keys (kRocItems consecutive keys per thread).
__global__ void __launch_bounds__(kRocThreads)
roc_run_count_kernel(const unsigned int* __restrict__ keys, const unsigned char* __restrict__ cls, int64_t n,
                     unsigned int* __restrict__ sums) {
  const int64_t i0 = (int64_t)blockIdx.x * kRocTile + threadIdx.x * kRocItems;
  unsigned int e = 0, g = 0;
  for (int k = 0; k < kRocItems; ++k) {
    const int64_t i = i0 + k;
    if (i < n) {
      e += roc_run_end(keys, n, i);
      g += cls[i];
    }
  }
  unsigned int te, tg;
  roc_block_scan(e, &te);
  roc_block_scan(g, &tg);
  if (threadIdx.x == 0) {
    sums[2 * (int64_t)blockIdx.x] = te;
    sums[2 * (int64_t)blockIdx.x + 1] = tg;
  }
}

// One block: exclusive scan, in place, of each of the `comps` interleaved columns of sums [n_tiles][comps]; column
// totals -> totals[comps].
__global__ void __launch_bounds__(kRocThreads)
roc_tile_scan_kernel(unsigned int* __restrict__ sums, int64_t n_tiles, int comps, unsigned int* __restrict__ totals) {
  for (int c = 0; c < comps; ++c) {
    unsigned int carry = 0;
    for (int64_t t0 = 0; t0 < n_tiles; t0 += kRocTile) {
      const int64_t ti = t0 + threadIdx.x * kRocItems;
      unsigned int s = 0;
      for (int k = 0; k < kRocItems; ++k)
        if (ti + k < n_tiles) s += sums[(ti + k) * comps + c];
      unsigned int tot;
      unsigned int run = carry + roc_block_scan(s, &tot);
      for (int k = 0; k < kRocItems; ++k)
        if (ti + k < n_tiles) {
          const unsigned int v = sums[(ti + k) * comps + c];
          sums[(ti + k) * comps + c] = run;
          run += v;
        }
      carry += tot;
    }
    if (threadIdx.x == 0) totals[c] = carry;
  }
}

// Run j of the sorted keys: tps[j] = genuine keys up to and including its last key, last[j] = that key's position.
__global__ void __launch_bounds__(kRocThreads)
roc_run_write_kernel(const unsigned int* __restrict__ keys, const unsigned char* __restrict__ cls, int64_t n,
                     const unsigned int* __restrict__ sums, unsigned int* __restrict__ tps, unsigned int* __restrict__ last) {
  const int64_t i0 = (int64_t)blockIdx.x * kRocTile + threadIdx.x * kRocItems;
  unsigned int e = 0, g = 0;
  for (int k = 0; k < kRocItems; ++k) {
    const int64_t i = i0 + k;
    if (i < n) {
      e += roc_run_end(keys, n, i);
      g += cls[i];
    }
  }
  unsigned int t;
  unsigned int j = sums[2 * (int64_t)blockIdx.x] + roc_block_scan(e, &t);
  unsigned int gen = sums[2 * (int64_t)blockIdx.x + 1] + roc_block_scan(g, &t);
  for (int k = 0; k < kRocItems; ++k) {
    const int64_t i = i0 + k;
    if (i < n) {
      gen += cls[i];
      if (roc_run_end(keys, n, i)) {
        tps[j] = gen;
        last[j] = (unsigned int)i;
        ++j;
      }
    }
  }
}

// sklearn's thinning (np.diff(fps, 2) or np.diff(tps, 2) nonzero): the first and the last of the m runs stay; an inner
// run stays iff the next run has another genuine count or another size.
__device__ __forceinline__ bool roc_keep(const unsigned int* __restrict__ tps, const unsigned int* __restrict__ last,
                                         unsigned int m, int64_t j) {
  if (j >= m) return false;
  if (j == 0 || j == m - 1) return true;
  return tps[j + 1] - tps[j] != tps[j] - tps[j - 1] || last[j + 1] - last[j] != last[j] - last[j - 1];
}

// sums[tile] = kept runs among this tile of kRocTile runs.
__global__ void __launch_bounds__(kRocThreads)
roc_keep_count_kernel(const unsigned int* __restrict__ tps, const unsigned int* __restrict__ last, const RocState* st,
                      unsigned int* __restrict__ sums) {
  const unsigned int m = st->run_totals[0];
  const int64_t j0 = (int64_t)blockIdx.x * kRocTile + threadIdx.x * kRocItems;
  unsigned int c = 0;
  for (int k = 0; k < kRocItems; ++k) c += roc_keep(tps, last, m, j0 + k);
  unsigned int t;
  roc_block_scan(c, &t);
  if (threadIdx.x == 0) sums[blockIdx.x] = t;
}

// The curve: point 0 is (0, 0) at +inf; kept run j becomes the next point, fpr = fps / n_imp, tpr = tps / n_gen.
__global__ void __launch_bounds__(kRocThreads)
roc_point_kernel(const unsigned int* __restrict__ keys, const unsigned int* __restrict__ tps,
                 const unsigned int* __restrict__ last, const RocState* st, const unsigned int* __restrict__ sums,
                 double* __restrict__ fpr, double* __restrict__ tpr, double* __restrict__ thresholds,
                 int64_t* __restrict__ n_points, int64_t* __restrict__ counts) {
  const unsigned int m = st->run_totals[0];
  const int64_t j0 = (int64_t)blockIdx.x * kRocTile + threadIdx.x * kRocItems;
  unsigned int c = 0;
  for (int k = 0; k < kRocItems; ++k) c += roc_keep(tps, last, m, j0 + k);
  unsigned int t;
  unsigned int p = 1 + sums[blockIdx.x] + roc_block_scan(c, &t);
  const double n_gen = (double)st->n_gen, n_imp = (double)st->n_imp;
  for (int k = 0; k < kRocItems; ++k) {
    const int64_t j = j0 + k;
    if (roc_keep(tps, last, m, j)) {
      const unsigned int tp = tps[j], fp = last[j] + 1 - tp;
      fpr[p] = (double)fp / n_imp;
      tpr[p] = (double)tp / n_gen;
      thresholds[p] = roc_key_value(keys[last[j]]);
      ++p;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    fpr[0] = 0.0;
    tpr[0] = 0.0;
    thresholds[0] = (double)INFINITY;
    *n_points = (int64_t)st->n_keep + 1;
    counts[0] = (int64_t)st->n_gen;
    counts[1] = (int64_t)st->n_imp;
    counts[2] = (int64_t)st->n_bad;
  }
}

// Workspace: the state, then 256-byte aligned arrays.
struct RocLayout {
  int64_t n_tiles, n_groups;
  size_t keys[2], cls[2], hist, part, sums, tps, last, bytes;
};

static RocLayout roc_layout(int64_t n) {
  RocLayout L;
  L.n_tiles = (n + kRocTile - 1) / kRocTile;
  L.n_groups = (L.n_tiles + kRocColTiles - 1) / kRocColTiles;
  size_t o = 0;
  auto take = [&o](size_t bytes) {
    const size_t at = o;
    o += (bytes + 255) & ~(size_t)255;
    return at;
  };
  take(sizeof(RocState));
  L.keys[0] = take(4 * (size_t)n);
  L.keys[1] = take(4 * (size_t)n);
  L.cls[0] = take((size_t)n);
  L.cls[1] = take((size_t)n);
  L.hist = take(4 * 256 * (size_t)L.n_tiles);
  L.part = take(4 * 256 * (size_t)L.n_groups);
  L.sums = take(4 * 2 * (size_t)L.n_tiles);
  L.tps = take(4 * (size_t)n);
  L.last = take(4 * (size_t)n);
  L.bytes = o;
  return L;
}

constexpr int kKfThreads = kRocThreads;        // the selection reuses roc_block_scan, which needs 256 threads
constexpr int kKfPairsPerBlock = kKfThreads / 32;
constexpr int kKfMaxEmb = 4096;
constexpr int kKfMaxThr = 16384;
constexpr int kKfWindow = 4096;                // histogram bins per class held in shared memory at once

// Fused value x_k of row r: emb + flip (one fp32 add), or emb alone.
__device__ __forceinline__ float kf_x(const float* __restrict__ emb, const float* __restrict__ flip, int64_t r, int E,
                                      int k) {
  const float e = emb[r * E + k];
  return flip ? __fadd_rn(e, flip[r * E + k]) : e;
}

// The pinned warp sum of the lanes' fp64 partials: xor butterfly over 16, 8, 4, 2, 1.  a + b == b + a in IEEE
// arithmetic, so every lane returns the same value.
__device__ __forceinline__ double kf_warp_sum(double s) {
  for (int o = 16; o > 0; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(0xffffffffu, s, o));
  return s;
}

// Pair p = rows 2p and 2p+1: dist[p], and bins[p] = the first j with (double)dist < thr[j] (T if none, so a NaN
// distance is never "same").  One warp per pair, grid-stride over the pairs.
__global__ void __launch_bounds__(kKfThreads)
kfold_dist_kernel(const float* __restrict__ emb, const float* __restrict__ flip, int64_t n_pairs, int E,
                  const double* __restrict__ thr, int T, float* __restrict__ dist, int* __restrict__ bins) {
  const int lane = threadIdx.x & 31;
  for (int64_t p = (int64_t)blockIdx.x * kKfPairsPerBlock + (threadIdx.x >> 5); p < n_pairs;
       p += (int64_t)gridDim.x * kKfPairsPerBlock) {
    const int64_t r1 = 2 * p, r2 = 2 * p + 1;
    double s1 = 0.0, s2 = 0.0;
    for (int k = lane; k < E; k += 32) {
      const double a = (double)kf_x(emb, flip, r1, E, k), b = (double)kf_x(emb, flip, r2, E, k);
      s1 = __dadd_rn(s1, __dmul_rn(a, a));
      s2 = __dadd_rn(s2, __dmul_rn(b, b));
    }
    float n1 = (float)sqrt(kf_warp_sum(s1)), n2 = (float)sqrt(kf_warp_sum(s2));
    if (n1 == 0.f) n1 = 1.f;
    if (n2 == 0.f) n2 = 1.f;
    double s = 0.0;
    for (int k = lane; k < E; k += 32) {
      const float d = kf_x(emb, flip, r1, E, k) / n1 - kf_x(emb, flip, r2, E, k) / n2;
      s = __dadd_rn(s, __dmul_rn((double)d, (double)d));
    }
    s = kf_warp_sum(s);
    if (lane == 0) {
      const float d = (float)s;
      int lo = 0, hi = T;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((double)d < thr[mid]) hi = mid;
        else lo = mid + 1;
      }
      dist[p] = d;
      bins[p] = lo;
    }
  }
}

// sklearn's KFold(F, shuffle=False): fold f tests pairs [lo, hi); the first P % F folds hold one pair more.
__device__ __forceinline__ void kf_fold_range(int64_t n_pairs, int64_t F, int64_t f, int64_t* lo, int64_t* hi) {
  const int64_t q = n_pairs / F, r = n_pairs % F;
  *lo = f * q + (f < r ? f : r);
  *hi = *lo + q + (f < r ? 1 : 0);
}

// One CTA per fold: hist[f][c][b] = test pairs of class c (0 genuine, 1 impostor) with bin b, b = 0 ... T; the same
// counts are added into totals[c][b].  Bins are counted kKfWindow at a time in shared memory.
__global__ void __launch_bounds__(kKfThreads)
kfold_hist_kernel(const int* __restrict__ bins, const unsigned char* __restrict__ issame, int64_t n_pairs, int64_t F,
                  int T, int* __restrict__ hist, int* __restrict__ totals) {
  __shared__ int sh[2][kKfWindow];
  const int64_t f = blockIdx.x;
  int64_t lo, hi;
  kf_fold_range(n_pairs, F, f, &lo, &hi);
  int* h = hist + f * 2 * (T + 1);
  for (int w0 = 0; w0 <= T; w0 += kKfWindow) {
    const int nw = T + 1 - w0 < kKfWindow ? T + 1 - w0 : kKfWindow;
    for (int i = threadIdx.x; i < 2 * kKfWindow; i += kKfThreads) sh[i / kKfWindow][i % kKfWindow] = 0;
    __syncthreads();
    for (int64_t p = lo + threadIdx.x; p < hi; p += kKfThreads) {
      const int b = bins[p] - w0;
      if (b >= 0 && b < nw) atomicAdd(&sh[issame[p] ? 0 : 1][b], 1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nw; i += kKfThreads)
      for (int c = 0; c < 2; ++c) {
        const int v = sh[c][i];
        h[c * (T + 1) + w0 + i] = v;
        if (v) atomicAdd(&totals[c * (T + 1) + w0 + i], v);
      }
    __syncthreads();                           // sh is cleared for the next window
  }
}

// Counts of one class at one threshold, as insightface's calculate_accuracy takes them.
__device__ __forceinline__ double kf_rate(unsigned int hit, unsigned int n) {
  return n ? (double)hit / (double)n : 0.0;
}

// One CTA per fold.  Thread t walks thresholds [t C, (t + 1) C) in order with the inclusive counts of bins <= j: test
// genuine / impostor from hist[f], all-pairs from totals; train = all - test (train = test when F = 1).  It writes the
// test rates rates[f][0 tpr, 1 fpr][j] and keeps its first maximum of the train tp + tn; thread 0 then takes the first
// maximum over the threads in order, which is the first over j.
__global__ void __launch_bounds__(kKfThreads)
kfold_select_kernel(const int* __restrict__ hist, const int* __restrict__ totals, int64_t F, int T,
                    const double* __restrict__ thr, double* __restrict__ rates, double* __restrict__ accuracy,
                    double* __restrict__ best_thr) {
  __shared__ unsigned int best_val[kKfThreads], best_j[kKfThreads], best_test[kKfThreads];
  const int64_t f = blockIdx.x;
  const int* hg = hist + f * 2 * (T + 1);
  const int* hi = hg + (T + 1);
  const int* tg = totals;
  const int* ti = totals + (T + 1);
  const int C = (T + kKfThreads - 1) / kKfThreads;
  const int j0 = threadIdx.x * C < T ? threadIdx.x * C : T;
  const int j1 = j0 + C < T ? j0 + C : T;
  unsigned int s[4] = {0u, 0u, 0u, 0u};
  for (int j = j0; j < j1; ++j) {
    s[0] += hg[j]; s[1] += hi[j]; s[2] += tg[j]; s[3] += ti[j];
  }
  unsigned int cum[4], all[4];
  for (int q = 0; q < 4; ++q) cum[q] = roc_block_scan(s[q], &all[q]);
  // class sizes: bins 0 ... T - 1 plus bin T (never "same")
  const unsigned int n_gen_te = all[0] + hg[T], n_imp_te = all[1] + hi[T], n_imp = all[3] + ti[T];
  const bool one_fold = F == 1;
  double* r_tpr = rates + f * 2 * (int64_t)T;
  double* r_fpr = r_tpr + T;
  unsigned int bv = 0u, bj = 0xffffffffu, bt = 0u;
  for (int j = j0; j < j1; ++j) {
    cum[0] += hg[j]; cum[1] += hi[j]; cum[2] += tg[j]; cum[3] += ti[j];
    const unsigned int tp = cum[0], fp = cum[1];                      // test: predicted same iff bin <= j
    const unsigned int tn = n_imp_te - fp;
    const unsigned int train = one_fold ? tp + tn : (cum[2] - tp) + ((n_imp - n_imp_te) - (cum[3] - fp));
    if (bj == 0xffffffffu || train > bv) { bv = train; bj = (unsigned int)j; bt = tp + tn; }
    r_tpr[j] = kf_rate(tp, n_gen_te);
    r_fpr[j] = kf_rate(fp, n_imp_te);
  }
  best_val[threadIdx.x] = bv;
  best_j[threadIdx.x] = bj;
  best_test[threadIdx.x] = bt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int w = -1;
    for (int t = 0; t < kKfThreads; ++t)
      if (best_j[t] != 0xffffffffu && (w < 0 || best_val[t] > best_val[w])) w = t;
    accuracy[f] = (double)best_test[w] / (double)(n_gen_te + n_imp_te);
    best_thr[f] = thr[best_j[w]];
  }
}

// tpr[j] = (rates[0][0][j] + rates[1][0][j] + ...) / F in fold order (np.mean(tprs, 0)); fpr the same.
__global__ void __launch_bounds__(kKfThreads)
kfold_mean_kernel(const double* __restrict__ rates, int64_t F, int T, double* __restrict__ tpr, double* __restrict__ fpr) {
  const int j = blockIdx.x * kKfThreads + threadIdx.x;
  if (j >= T) return;
  double st = 0.0, sf = 0.0;
  for (int64_t f = 0; f < F; ++f) {
    st = __dadd_rn(st, rates[f * 2 * T + j]);
    sf = __dadd_rn(sf, rates[f * 2 * T + T + j]);
  }
  tpr[j] = st / (double)F;
  fpr[j] = sf / (double)F;
}

struct KfoldLayout {
  size_t bins, hist, totals, rates, bytes;
};

static KfoldLayout kfold_layout(int64_t n_pairs, int T, int64_t F) {
  KfoldLayout L;
  size_t o = 0;
  auto take = [&o](size_t bytes) {
    const size_t at = o;
    o += (bytes + 255) & ~(size_t)255;
    return at;
  };
  L.bins = take(4 * (size_t)n_pairs);
  L.hist = take(4 * 2 * (size_t)F * (size_t)(T + 1));
  L.totals = take(4 * 2 * (size_t)(T + 1));
  L.rates = take(8 * 2 * (size_t)F * (size_t)T);
  L.bytes = o;
  return L;
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

size_t pfc_roc_curve_workspace_bytes(int64_t n) {
  return roc_layout(n > 0 ? n : 0).bytes;
}

int pfc_roc_curve(const float* scores, const unsigned char* issame, int64_t n, double* fpr, double* tpr, double* thresholds,
                  int64_t* n_points, int64_t* counts, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_roc_curve");
  PFC_REQUIRE(scores && issame && fpr && tpr && thresholds && n_points && counts && workspace && n > 0, PFC_E_ARG,
              "pfc_roc_curve: bad argument");
  PFC_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 8 == 0, PFC_E_ARG, "pfc_roc_curve: workspace not 8-byte aligned");
  PFC_REQUIRE(n < (1ll << 31), PFC_E_SHAPE, "pfc_roc_curve: more than 2^31 - 1 scores");
  PFC_REQUIRE(workspace_bytes >= pfc_roc_curve_workspace_bytes(n), PFC_E_WORKSPACE, "pfc_roc_curve: workspace too small");
  cudaStream_t st = as_stream(stream);
  const RocLayout L = roc_layout(n);
  char* ws = reinterpret_cast<char*>(workspace);
  auto* state = reinterpret_cast<RocState*>(ws);
  auto* hist = reinterpret_cast<unsigned int*>(ws + L.hist);
  auto* part = reinterpret_cast<unsigned int*>(ws + L.part);
  auto* sums = reinterpret_cast<unsigned int*>(ws + L.sums);
  auto* tps = reinterpret_cast<unsigned int*>(ws + L.tps);
  auto* last = reinterpret_cast<unsigned int*>(ws + L.last);
  const auto* bits = reinterpret_cast<const unsigned int*>(scores);
  const unsigned int nt = (unsigned int)L.n_tiles, ng = (unsigned int)L.n_groups;
  PFC_CUDA(cudaMemsetAsync(state, 0, sizeof(RocState), st));
  const unsigned int* keys = nullptr;
  const unsigned char* cls = nullptr;
  for (int pass = 0; pass < 4; ++pass) {       // LSD: digit 0 first; pass 0 reads the scores
    const int shift = 8 * pass;
    auto* keys_out = reinterpret_cast<unsigned int*>(ws + L.keys[pass & 1]);
    auto* cls_out = reinterpret_cast<unsigned char*>(ws + L.cls[pass & 1]);
    roc_hist_kernel<<<nt, kRocThreads, 0, st>>>(pass == 0 ? bits : nullptr, pass == 0 ? issame : nullptr, keys, n, shift,
                                                hist, state);
    PFC_LAUNCH_CHECK();
    roc_col_sum_kernel<<<ng, kRocThreads, 0, st>>>(hist, L.n_tiles, part);
    PFC_LAUNCH_CHECK();
    roc_col_scan_kernel<<<1, kRocThreads, 0, st>>>(part, L.n_groups);
    PFC_LAUNCH_CHECK();
    roc_col_apply_kernel<<<ng, kRocThreads, 0, st>>>(hist, L.n_tiles, part);
    PFC_LAUNCH_CHECK();
    roc_scatter_kernel<<<nt, kRocThreads, 0, st>>>(pass == 0 ? bits : nullptr, pass == 0 ? issame : nullptr, keys, cls, n,
                                                   shift, hist, keys_out, cls_out);
    PFC_LAUNCH_CHECK();
    keys = keys_out;
    cls = cls_out;
  }
  roc_run_count_kernel<<<nt, kRocThreads, 0, st>>>(keys, cls, n, sums);
  PFC_LAUNCH_CHECK();
  roc_tile_scan_kernel<<<1, kRocThreads, 0, st>>>(sums, L.n_tiles, 2, state->run_totals);
  PFC_LAUNCH_CHECK();
  roc_run_write_kernel<<<nt, kRocThreads, 0, st>>>(keys, cls, n, sums, tps, last);
  PFC_LAUNCH_CHECK();
  roc_keep_count_kernel<<<nt, kRocThreads, 0, st>>>(tps, last, state, sums);
  PFC_LAUNCH_CHECK();
  roc_tile_scan_kernel<<<1, kRocThreads, 0, st>>>(sums, L.n_tiles, 1, &state->n_keep);
  PFC_LAUNCH_CHECK();
  roc_point_kernel<<<nt, kRocThreads, 0, st>>>(keys, tps, last, state, sums, fpr, tpr, thresholds, n_points, counts);
  PFC_LAUNCH_CHECK();
  return 0;
}

size_t pfc_kfold_workspace_bytes(int64_t n_pairs, int n_thresholds, int64_t nfolds) {
  return kfold_layout(n_pairs > 0 ? n_pairs : 0, n_thresholds > 0 ? n_thresholds : 0, nfolds > 0 ? nfolds : 0).bytes;
}

int pfc_kfold_accuracy(const float* emb, const float* flip, const unsigned char* issame, int64_t n_pairs, int emb_dim,
                       const double* thr, int n_thresholds, int64_t nfolds, float* dist, double* accuracy, double* best_thr,
                       double* tpr, double* fpr, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_kfold_accuracy");
  PFC_REQUIRE(emb && issame && thr && dist && accuracy && best_thr && tpr && fpr && workspace, PFC_E_ARG,
              "pfc_kfold_accuracy: null pointer");
  PFC_REQUIRE(n_pairs > 0 && emb_dim > 0 && n_thresholds > 0 && nfolds >= 1 && nfolds <= n_pairs, PFC_E_ARG,
              "pfc_kfold_accuracy: bad size (need P >= 1, emb >= 1, T >= 1, 1 <= nfolds <= P)");
  PFC_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 8 == 0, PFC_E_ARG, "pfc_kfold_accuracy: workspace not 8-byte aligned");
  PFC_REQUIRE(emb_dim <= kKfMaxEmb && n_pairs < (1ll << 31) && n_thresholds <= kKfMaxThr, PFC_E_SHAPE,
              "pfc_kfold_accuracy: emb > 4096, P >= 2^31 or more than 16384 thresholds");
  PFC_REQUIRE(workspace_bytes >= pfc_kfold_workspace_bytes(n_pairs, n_thresholds, nfolds), PFC_E_WORKSPACE,
              "pfc_kfold_accuracy: workspace too small");
  cudaStream_t st = as_stream(stream);
  const KfoldLayout L = kfold_layout(n_pairs, n_thresholds, nfolds);
  char* ws = reinterpret_cast<char*>(workspace);
  auto* bins = reinterpret_cast<int*>(ws + L.bins);
  auto* hist = reinterpret_cast<int*>(ws + L.hist);
  auto* totals = reinterpret_cast<int*>(ws + L.totals);
  auto* rates = reinterpret_cast<double*>(ws + L.rates);
  PFC_CUDA(cudaMemsetAsync(totals, 0, 4 * 2 * (size_t)(n_thresholds + 1), st));
  int64_t nb = (n_pairs + kKfPairsPerBlock - 1) / kKfPairsPerBlock;
  if (nb > 16 * sm_count()) nb = 16 * sm_count();
  kfold_dist_kernel<<<(unsigned int)nb, kKfThreads, 0, st>>>(emb, flip, n_pairs, emb_dim, thr, n_thresholds, dist, bins);
  PFC_LAUNCH_CHECK();
  kfold_hist_kernel<<<(unsigned int)nfolds, kKfThreads, 0, st>>>(bins, issame, n_pairs, nfolds, n_thresholds, hist, totals);
  PFC_LAUNCH_CHECK();
  kfold_select_kernel<<<(unsigned int)nfolds, kKfThreads, 0, st>>>(hist, totals, nfolds, n_thresholds, thr, rates,
                                                                   accuracy, best_thr);
  PFC_LAUNCH_CHECK();
  kfold_mean_kernel<<<(unsigned int)((n_thresholds + kKfThreads - 1) / kKfThreads), kKfThreads, 0, st>>>(
      rates, nfolds, n_thresholds, tpr, fpr);
  PFC_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
