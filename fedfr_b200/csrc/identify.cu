// 1:N identification (the IJB-B / IJB-C search protocol of FedFR's ijbc_all.py rank-k and local_1n.py): the mate's
// rank and the top-1 match of every probe, with no [P, G] score matrix and no top-k list.  Every score is the 1:1 pair
// chain (dot_chain.cuh) and every key is TAR@FAR's (tar_key, score_key.cuh), so a 1:N score is bit-identical to
// pfc_pair_scores' score of the same two rows.  One thread per probe scores its mate with dot_chain; persistent CTAs
// then walk 64 x 64 (probe x gallery) tiles with the ROC histogram's exact tile loop (tile_chain), count per probe the
// gallery entries that beat the mate (integer atomics) and keep the packed (key, ~row) maximum (a 64-bit atomicMax).
// A last kernel turns the counts into ranks and decodes the top-1 row and score.  Integer counts and a maximum only:
// the result does not depend on the schedule.
#include "common.cuh"
#include "../../fedfr_b200/csrc/dot_chain.cuh"
#include "../../fedfr_b200/csrc/score_key.cuh"

namespace pfc {

constexpr int kIdThreads = 256;
constexpr int kIdMaxEmb = 4096;

struct IdentState {
  unsigned long long n_nan, n_bad;             // NaN scores over all (probe, gallery) pairs; mate rows outside [-1, G)
};

__device__ __forceinline__ unsigned int id_bits(float f) {
  union { float f; unsigned int u; } v;
  v.f = f;
  return v.u;
}

// The fp32 score of a tar_key (the inverse map; the key 0 of NaN gives the NaN 0xffffffff).
__device__ __forceinline__ float id_key_value(unsigned int key) {
  union { unsigned int u; float f; } v;
  v.u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  return v.f;
}

// A probe's mate row, or -1 when it has none (mate_row -1) or a row outside [0, G).
__device__ __forceinline__ int64_t id_mate(const int64_t* __restrict__ mate_row, int64_t p, int64_t G) {
  const int64_t m = mate_row[p];
  return m >= 0 && m < G ? m : -1;
}

// mate_score[p] = (float)dot_chain(0, probe[p], gallery[m_p], emb), one thread per probe: the same chain, in the same
// order, as the tile kernel's sum for that pair.  NaN without a mate; a row outside [-1, G) is counted in n_bad.
__global__ void __launch_bounds__(kIdThreads)
ident_mate_kernel(const float* __restrict__ probe, int64_t P, const float* __restrict__ gallery, int64_t G, int emb,
                  const int64_t* __restrict__ mate_row, float* __restrict__ mate_score, IdentState* st) {
  const int64_t p = (int64_t)blockIdx.x * kIdThreads + threadIdx.x;
  if (p >= P) return;
  const int64_t m = id_mate(mate_row, p, G);
  if (m < 0 && mate_row[p] != -1) atomicAdd(&st->n_bad, 1ull);
  mate_score[p] = m >= 0 ? (float)dot_chain(0.0, probe + p * emb, gallery + m * emb, emb) : nanf("");
}

// Persistent CTAs over 64 x 64 (probe x gallery) tiles, the sums by tile_chain.  Per pair: the key of its score; "beats"
// = key above the mate's key, or equal to it at a lower gallery row; the packed (key << 32 | ~row), whose maximum is
// the largest key at its first row.  The 16 threads of a probe row (one half warp) combine theirs with xor shuffles,
// then one integer atomicAdd (when nonzero) and one 64-bit atomicMax per row and tile.  No float atomics.
__global__ void __launch_bounds__(kChainThreads, 2)
ident_rank_kernel(const float* __restrict__ probe, int64_t P, const float* __restrict__ gallery, int64_t G, int emb,
                  const int64_t* __restrict__ mate_row, const float* __restrict__ mate_score, unsigned int* __restrict__ beats,
                  unsigned long long* __restrict__ top, IdentState* st) {
  __shared__ float As[kChainTile][kChainK + 1];
  __shared__ float Bs[kChainTile][kChainK + 1];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t n_tg = (G + kChainTile - 1) / kChainTile;
  const int64_t total = ((P + kChainTile - 1) / kChainTile) * n_tg;
  unsigned long long nan = 0;
  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int64_t i0 = (t / n_tg) * kChainTile;
    const int64_t j0 = (t % n_tg) * kChainTile;
    double acc[4][4];
    tile_chain(probe, P, i0, gallery, G, j0, emb, As, Bs, acc);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t p = i0 + ty + 16 * u;
      const bool p_ok = p < P;
      const int64_t m = p_ok ? id_mate(mate_row, p, G) : -1;
      const unsigned int mk = m >= 0 ? tar_key(id_bits(mate_score[p])) : 0u;
      unsigned int b = 0;
      unsigned long long best = 0ull;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int64_t g = j0 + tx + 16 * v;
        if (!p_ok || g >= G) continue;
        const unsigned int key = tar_key(id_bits((float)acc[u][v]));
        nan += key == 0u;
        b += m >= 0 && (key > mk || (key == mk && g < m));
        const unsigned long long packed = ((unsigned long long)key << 32) | (unsigned long long)(~(unsigned int)g);
        best = packed > best ? packed : best;
      }
      for (int o = 8; o > 0; o >>= 1) {
        b += __shfl_xor_sync(0xffffffffu, b, o);
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
      }
      if (tx == 0 && p_ok) {                   // column j0 < G: best holds at least one pair
        if (b) atomicAdd(beats + p, b);
        atomicMax(top + p, best);
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) nan += __shfl_xor_sync(0xffffffffu, nan, o);
  if ((tid & 31) == 0 && nan) atomicAdd(&st->n_nan, nan);
}

__global__ void __launch_bounds__(kIdThreads)
ident_finish_kernel(int64_t P, int64_t G, const int64_t* __restrict__ mate_row, const unsigned int* __restrict__ beats,
                    const unsigned long long* __restrict__ top, const IdentState* st, int64_t* __restrict__ rank,
                    int64_t* __restrict__ top1_row, float* __restrict__ top1_score, int64_t* __restrict__ counts) {
  const int64_t p = (int64_t)blockIdx.x * kIdThreads + threadIdx.x;
  if (p == 0) {
    counts[0] = (int64_t)st->n_nan;
    counts[1] = (int64_t)st->n_bad;
  }
  if (p >= P) return;
  rank[p] = id_mate(mate_row, p, G) >= 0 ? 1 + (int64_t)beats[p] : 0;
  const unsigned long long t = top[p];
  top1_row[p] = (int64_t)(~(unsigned int)t);
  top1_score[p] = id_key_value((unsigned int)(t >> 32));
}

struct IdentLayout {
  size_t beats, top, bytes;
};

static IdentLayout ident_layout(int64_t P) {
  IdentLayout L;
  size_t o = 0;
  auto take = [&o](size_t bytes) {
    const size_t at = o;
    o += (bytes + 255) & ~(size_t)255;
    return at;
  };
  take(sizeof(IdentState));
  L.beats = take(4 * (size_t)P);
  L.top = take(8 * (size_t)P);
  L.bytes = o;
  return L;
}


}  // namespace pfc

using namespace pfc;

extern "C" {

size_t pfc_identify_workspace_bytes(int64_t n_probe) {
  return ident_layout(n_probe > 0 ? n_probe : 0).bytes;
}

int pfc_identify(const float* probe, int64_t n_probe, const float* gallery, int64_t n_gallery, int emb,
                 const int64_t* mate_row, int64_t* rank, float* mate_score, int64_t* top1_row, float* top1_score,
                 int64_t* counts, void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = require_sm100()) return rc;
  NvtxScope nvtx_scope("pfc_identify");
  PFC_REQUIRE(probe && gallery && mate_row && rank && mate_score && top1_row && top1_score && counts && workspace, PFC_E_ARG,
              "pfc_identify: null pointer");
  PFC_REQUIRE(n_probe > 0 && n_gallery > 0 && emb > 0, PFC_E_ARG, "pfc_identify: bad size (need P >= 1, G >= 1, emb >= 1)");
  PFC_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 8 == 0, PFC_E_ARG, "pfc_identify: workspace not 8-byte aligned");
  PFC_REQUIRE(emb <= kIdMaxEmb && n_probe < (1ll << 31) && n_gallery < (1ll << 31), PFC_E_SHAPE,
              "pfc_identify: emb > 4096, P >= 2^31 or G >= 2^31");
  PFC_REQUIRE(workspace_bytes >= pfc_identify_workspace_bytes(n_probe), PFC_E_WORKSPACE, "pfc_identify: workspace too small");
  cudaStream_t st = as_stream(stream);
  const IdentLayout L = ident_layout(n_probe);
  char* ws = reinterpret_cast<char*>(workspace);
  auto* state = reinterpret_cast<IdentState*>(ws);
  auto* beats = reinterpret_cast<unsigned int*>(ws + L.beats);
  auto* top = reinterpret_cast<unsigned long long*>(ws + L.top);
  PFC_CUDA(cudaMemsetAsync(ws, 0, L.bytes, st));
  const unsigned int nb = (unsigned int)((n_probe + kIdThreads - 1) / kIdThreads);
  ident_mate_kernel<<<nb, kIdThreads, 0, st>>>(probe, n_probe, gallery, n_gallery, emb, mate_row, mate_score, state);
  PFC_LAUNCH_CHECK();
  const int64_t tiles = ((n_probe + kChainTile - 1) / kChainTile) * ((n_gallery + kChainTile - 1) / kChainTile);
  int64_t grid = 2 * (int64_t)sm_count();
  if (grid > tiles) grid = tiles;
  ident_rank_kernel<<<(unsigned int)grid, kChainThreads, 0, st>>>(probe, n_probe, gallery, n_gallery, emb, mate_row,
                                                                  mate_score, beats, top, state);
  PFC_LAUNCH_CHECK();
  ident_finish_kernel<<<nb, kIdThreads, 0, st>>>(n_probe, n_gallery, mate_row, beats, top, state, rank, top1_row,
                                                 top1_score, counts);
  PFC_LAUNCH_CHECK();
  return 0;
}


}  // extern "C"
