// Tensor-core path (sm_100a): TMA-fed tcgen05.mma kernels with TMEM accumulators.
//
//   logits2_kernel<MODE_PROB>   P = exp2(s2 (x.w_hat) - bound) tile by tile -> bf16 scratch, row sums and the target
//                               logit in the epilogue; optional normaliser warps produce w_hat of the next class chunk.
//                               The [Bt, Cs] logits never exist.            (partial_fc.py:127,137-147, losses.py:23-45)
//   logits2_kernel<MODE_STATS>  recompute flavour: online (max, sum-exp) only                    (same lines)
//   logits2_kernel<MODE_GRAD>   recompute flavour: G = s (softmax - onehot) / Bt -> bf16 chunk scratch   (partial_fc.py:150-166)
//   logits_kernel<...>          single-CTA variants of STATS / GRAD (tuning knob pfc_set_logits_pair(0))
//   dx2_kernel / dx_kernel      dx (+)= G . w_hat  (split over the class axis, fp32 partial slabs)        (autograd of :110)
//   dw_kernel                   dw = normalize_bwd(G^T . x), radial term from its own accumulator        (autograd of :110,127)
//   prob_prep / row_bound / reduce_dx_scaled: the per-row glue of the stored-probability backward
//
// Roles per CTA: epilogue warps (TMEM lane quadrants) + 1 TMA producer warp + 1 MMA issuer warp (+ normaliser warps);
// 128-byte-swizzled operand tiles, mbarrier pipelines (smem full/empty, TMEM full/empty), CTA pairs (cta_group::2) for
// the logits and dx kernels, an e-split CTA pair with a DSMEM exchange for dw.  Host side at the bottom: tensor maps,
// launch plans, CUDA-graph cache (one replay per phase).
#include "tc_common.cuh"
#include "rows_device.cuh"
#include <mutex>
#include <string.h>
#include <vector>

namespace pfc {

// ------------------------------------------------------------------------------------------------ tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::once_flag g_encode_once;

static EncodeTiledFn get_encode() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  return g_encode;
}

static int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dt, uint32_t esz, uint64_t rows, uint64_t cols,
                        uint64_t row_stride_elems, uint32_t box_rows, uint32_t box_cols) {
  EncodeTiledFn enc = get_encode();
  PFC_REQUIRE(enc != nullptr, PFC_E_ARCH, "cuTensorMapEncodeTiled is not available from the CUDA driver");
  PFC_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (row_stride_elems * esz) % 16 == 0, PFC_E_ARG,
              "TMA operand must be 16-byte aligned with a 16-byte multiple row pitch");
  PFC_REQUIRE(box_cols * esz == 128 && box_rows <= 256, PFC_E_ARG, "TMA box must be 128 bytes wide and at most 256 rows");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {row_stride_elems * esz};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PFC_REQUIRE(r == CUDA_SUCCESS, PFC_E_ARG, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu pitch=%llu box=%ux%u)", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)row_stride_elems, box_rows, box_cols);
  return 0;
}

int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems, uint32_t box_rows,
                      uint32_t box_cols) {
  return make_tmap_2d(out, base, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, rows, cols, row_stride_elems, box_rows, box_cols);
}

int make_tmap_f32_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems, uint32_t box_rows,
                     uint32_t box_cols) {
  return make_tmap_2d(out, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, rows, cols, row_stride_elems, box_rows, box_cols);
}

namespace tc {

constexpr int kThreads = 192;          // dx kernels: 4 epilogue warps + TMA warp + MMA warp
constexpr int kLogitsEpiWarps = 8;     // logits kernels: two warps per TMEM lane quadrant, each takes half of the tile's columns
constexpr int kLogitsThreads = (kLogitsEpiWarps + 2) * 32;
constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kChunkBytes = BM * BK * 2;      // one [128 x 64] bf16 K-major tile = 16 KB
constexpr int kBoxBytes = 64 * BK * 2;        // one [64 x 64] bf16 box = 8 KB

enum { MODE_STATS = 0, MODE_GRAD = 1, MODE_PROB = 2, MODE_HINGE = 3 };

struct LogitsParams {
  const int64_t* label;      // [n_rows] shard-local id or -1
  int n_rows;
  int n_classes;             // classes covered by this launch (chunk)
  int class_base;            // shard-local id of class 0 of this launch
  int emb;
  int n_rb, n_ct;            // row blocks, class tiles
  float s, m;
  int margin_kind;           // PFC_MARGIN_COSFACE / PFC_MARGIN_ARCFACE
  // MODE_STATS
  float* part_max;           // [gridDim.x, n_rows]   (log-e units)
  float* part_sum;
  float* target_logit;       // [n_rows]
  int accumulate_stats;      // 1: continue from the (max, sum) already in this CTA's slots (class-chunked forward)
  // normaliser warps (logits2_kernel<.., NORM = true>): normalize() of the NEXT class chunk rides under this chunk's MMAs
  const float* norm_w;       // fp32 rows (already offset to the chunk unless norm_index != NULL)
  const int64_t* norm_index;
  int64_t norm_rows;
  __nv_bfloat16* norm_out;   // [norm_rows, emb]
  float* norm_inv;           // [norm_rows]
  // MODE_GRAD
  const float* row_max;      // [n_rows]
  const float* row_sum;
  __nv_bfloat16* g;          // [n_rows, ldg]
  int64_t ldg;
  float g_scale;             // s / total_batch
  int prefetch;              // 1: TMA L2 prefetch of the next class tile
  // MODE_PROB (forward that keeps the unnormalised probabilities): P_ij = exp2(s2 cos_ij - row_bound_i) -> bf16 scratch
  const float* row_bound;    // [n_rows] log2 units: an upper bound of every logit of the row minus a fixed headroom
  float* target_cos;         // [n_rows] plain cosine at the target column (the backward's fp32 fix-up needs it)
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// Column sums of a 32x32 block held one row per lane, packed-add version: lane L returns sum over lanes r of h_r[L].
// Recursive halving: 31 shuffles; the adds are issued as f32x2 pairs.
__device__ __forceinline__ float warp_colsum32_x2(const float2 (&h)[16], int lane) {
  // h[q] = columns (2q, 2q+1).  Step 16 exchanges columns k <-> k+16, i.e. pairs q <-> q+8.
  float2 a[8];
  bool up = lane & 16;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float2 send = up ? h[q] : h[q + 8], keep = up ? h[q + 8] : h[q];
    float2 got;
    got.x = __shfl_xor_sync(0xffffffffu, send.x, 16);
    got.y = __shfl_xor_sync(0xffffffffu, send.y, 16);
    a[q] = __fadd2_rn(keep, got);
  }
  float2 b[4];
  up = lane & 8;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float2 send = up ? a[q] : a[q + 4], keep = up ? a[q + 4] : a[q];
    float2 got;
    got.x = __shfl_xor_sync(0xffffffffu, send.x, 8);
    got.y = __shfl_xor_sync(0xffffffffu, send.y, 8);
    b[q] = __fadd2_rn(keep, got);
  }
  float2 c[2];
  up = lane & 4;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const float2 send = up ? b[q] : b[q + 2], keep = up ? b[q + 2] : b[q];
    float2 got;
    got.x = __shfl_xor_sync(0xffffffffu, send.x, 4);
    got.y = __shfl_xor_sync(0xffffffffu, send.y, 4);
    c[q] = __fadd2_rn(keep, got);
  }
  up = lane & 2;
  {
    const float2 send = up ? c[0] : c[1], keep = up ? c[1] : c[0];
    float2 got;
    got.x = __shfl_xor_sync(0xffffffffu, send.x, 2);
    got.y = __shfl_xor_sync(0xffffffffu, send.y, 2);
    c[0] = __fadd2_rn(keep, got);
  }
  up = lane & 1;
  const float send = up ? c[0].x : c[0].y, keep = up ? c[0].y : c[0].x;
  return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

// Column sums of a 32x32 block held one row per lane: lane L returns sum over lanes r of h_r[L]
// (recursive halving: 31 shuffles instead of 32 five-step reductions).
__device__ __forceinline__ float warp_colsum32(const float (&h)[32], int lane) {
  float a[16];
  bool up = lane & 16;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float send = up ? h[k] : h[k + 16], keep = up ? h[k + 16] : h[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  up = lane & 8;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float send = up ? a[k] : a[k + 8], keep = up ? a[k + 8] : a[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  up = lane & 4;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float send = up ? a[k] : a[k + 4], keep = up ? a[k + 4] : a[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  up = lane & 2;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float send = up ? a[k] : a[k + 2], keep = up ? a[k + 2] : a[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  up = lane & 1;
  const float send = up ? a[0] : a[1], keep = up ? a[1] : a[0];
  return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

// same on fp32 bit patterns held in uint32 registers (the caller's TMEM load buffer, products written in place)
__device__ __forceinline__ float warp_colsum32_bits(const uint32_t (&h)[32], int lane) {
  float a[16];
  bool up = lane & 16;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float send = __uint_as_float(up ? h[k] : h[k + 16]), keep = __uint_as_float(up ? h[k + 16] : h[k]);
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  up = lane & 8;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float send = up ? a[k] : a[k + 8], keep = up ? a[k + 8] : a[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  up = lane & 4;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float send = up ? a[k] : a[k + 4], keep = up ? a[k + 4] : a[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  up = lane & 2;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const float send = up ? a[k] : a[k + 2], keep = up ? a[k + 2] : a[k];
    a[k] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  up = lane & 1;
  const float send = up ? a[0] : a[1], keep = up ? a[1] : a[0];
  return keep + __shfl_xor_sync(0xffffffffu, send, 1);
}

struct PipeState {
  int stage = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance(int n_stages) {
    if (++stage == n_stages) { stage = 0; phase ^= 1; }
  }
};

// ================================================================================================
// logits kernel: A = x_hat row block (stationary in smem), B = w_hat class tiles (streamed)
// ================================================================================================
template <int BN, int STAGES, int MODE>
__global__ void __launch_bounds__(kLogitsThreads, 1) logits_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                                                             const LogitsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int n_kb = p.emb / BK;
  uint8_t* smem_a = smem;                                  // n_kb chunks of [128 x 64]
  uint8_t* smem_b = smem + n_kb * kChunkBytes;             // STAGES tiles of [BN x 64]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + STAGES * BN * BK * 2);
  uint64_t* full = bars;                 // [STAGES]
  uint64_t* empty = bars + STAGES;       // [STAGES]
  uint64_t* tmem_full = bars + 2 * STAGES;      // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2; // [2]
  uint64_t* a_full = bars + 2 * STAGES + 4;
  uint64_t* a_empty = bars + 2 * STAGES + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 6);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t n_tiles = (int64_t)p.n_rb * p.n_ct;
  const int64_t t0 = n_tiles * blockIdx.x / gridDim.x, t1 = n_tiles * (blockIdx.x + 1) / gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], kLogitsEpiWarps); }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    fence_barrier_init();
  }
  constexpr int kProducerWarp = kLogitsEpiWarps, kMmaWarp = kLogitsEpiWarps + 1;
  if (warp == kProducerWarp && lane == 0) { prefetch_tmap(&tmap_x); prefetch_tmap(&tmap_w); }
  if (warp == kMmaWarp) tmem_alloc<2 * BN>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kProducerWarp) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      PipeState ps;
      int cur_rb = -1, a_loads = 0;
      for (int64_t t = t0; t < t1; ++t) {
        const int rb = (int)(t / p.n_ct), ct = (int)(t % p.n_ct);
        if (rb != cur_rb) {
          if (a_loads > 0) mbar_wait(a_empty, (a_loads - 1) & 1);      // MMAs of the previous row block are done
          mbar_arrive_expect_tx(a_full, n_kb * kChunkBytes);
          for (int kb = 0; kb < n_kb; ++kb) tma_load_2d(smem_a + kb * kChunkBytes, &tmap_x, a_full, kb * BK, rb * BM);
          cur_rb = rb;
          ++a_loads;
        }
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&empty[ps.stage], ps.phase ^ 1);
          mbar_arrive_expect_tx(&full[ps.stage], BN * BK * 2);
          tma_load_2d(smem_b + ps.stage * (BN * BK * 2), &tmap_w, &full[ps.stage], kb * BK, ct * BN);
          ps.advance(STAGES);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, false, false);
      PipeState ps;
      int cur_rb = -1, a_uses = 0;
      int64_t it = 0;
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const int rb = (int)(t / p.n_ct);
        if (rb != cur_rb) {
          mbar_wait(a_full, a_uses & 1);
          ++a_uses;
          cur_rb = rb;
        }
        const int acc = (int)(it & 1);
        const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&full[ps.stage], ps.phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + kb * kChunkBytes);
          const uint32_t b_addr = smem_u32(smem_b + ps.stage * (BN * BK * 2));
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            const uint64_t da = make_desc_sw128(a_addr + kk * 32, 0, 1024);
            const uint64_t db = make_desc_sw128(b_addr + kk * 32, 0, 1024);
            umma_bf16_ss(d_tmem, da, db, idesc, (kb | kk) != 0);
          }
          umma_commit(&empty[ps.stage]);      // frees the smem stage once these MMAs retire
          ps.advance(STAGES);
        }
        umma_commit(&tmem_full[acc]);
        const bool last_of_rb = (t + 1 == t1) || ((int)((t + 1) / p.n_ct) != rb);
        if (last_of_rb) umma_commit(a_empty);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 0..7), thread = row;
    // warp w reads TMEM lanes [32 (w & 3), +32) and the column half (w >> 2) of every tile
    const int quad = warp & 3, chalf = warp >> 2;
    constexpr int CH = BN / 2;
    const float s2 = p.s * kLog2e;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    int cur_rb = -1;
    constexpr int kNoLabel = -(1 << 30);
    int row = 0, my_label = kNoLabel;
    bool row_ok = false;
    float run_m = -INFINITY, run_l = 0.f;        // MODE_STATS (log2 units)
    float M2 = 0.f, rS = 0.f;                    // MODE_GRAD
    int64_t it = 0;
    for (int64_t t = t0; t < t1; ++t, ++it) {
      const int rb = (int)(t / p.n_ct), ct = (int)(t % p.n_ct);
      if (rb != cur_rb) {
        if (MODE == MODE_STATS && cur_rb >= 0 && row_ok) {
          p.part_max[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = run_m * kLn2;
          p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = run_l;
        }
        cur_rb = rb;
        row = rb * BM + quad * 32 + lane;
        row_ok = row < p.n_rows;
        my_label = kNoLabel;
        if (row_ok) {
          const int64_t y = p.label[row];
          if (y >= 0) my_label = (int)(y - p.class_base);          // relative to this launch; out of range never matches
        }
        run_m = -INFINITY; run_l = 0.f;
        if (MODE == MODE_STATS && p.accumulate_stats && row_ok) {
          const float l0 = p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row];
          if (l0 > 0.f) { run_l = l0; run_m = p.part_max[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] * kLog2e; }
        }
        if (MODE == MODE_GRAD && row_ok) { M2 = p.row_max[row] * kLog2e; rS = 1.0f / p.row_sum[row]; }
      }
      const int acc = (int)(it & 1);
      const uint32_t acc_phase = (uint32_t)((it >> 1) & 1);
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const int col0 = ct * BN;
      const bool tile_has_oob = col0 + BN > p.n_classes;
#pragma unroll 1
      for (int c = chalf * CH; c < (chalf + 1) * CH; c += 32) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + lane_base + acc * BN + c, v);
        tmem_ld_wait();
        const int cb = col0 + c;
        float z[32];
        const int hit = my_label - cb;                   // in [0,32) iff the target class is in this column group
        float c_hit = 0.f, slope = 1.f;                  // plain cosine / margin slope at the target
        if (hit >= 0 && hit < 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j) if (j == hit) {
            c_hit = __uint_as_float(v[j]);
            slope = margin_slope(c_hit, p.m, p.margin_kind);
            v[j] = __float_as_uint(margin_cos(c_hit, p.m, p.margin_kind));
            if (MODE == MODE_STATS) p.target_logit[row] = p.s * __uint_as_float(v[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) z[j] = __uint_as_float(v[j]) * s2;
        if (MODE == MODE_STATS) {
          if (tile_has_oob) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (cb + j >= p.n_classes) z[j] = -INFINITY;
          }
          float cm = z[0];
#pragma unroll
          for (int j = 1; j < 32; ++j) cm = fmaxf(cm, z[j]);
          if (cm > -INFINITY) {
            const float nm = fmaxf(run_m, cm);
            float sum = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) sum += fast_exp2(z[j] - nm);
            run_l = run_l * fast_exp2(run_m - nm) + sum;
            run_m = nm;
          }
        } else {
          uint32_t pk[16];
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            float g0 = fast_exp2(z[j] - M2) * rS, g1 = fast_exp2(z[j + 1] - M2) * rS;
            if (j == hit) g0 = (g0 - 1.0f) * slope;
            if (j + 1 == hit) g1 = (g1 - 1.0f) * slope;
            pk[j >> 1] = pack_bf16x2(g0 * p.g_scale, g1 * p.g_scale);
          }
          if (cb < p.ldg) {   // blocked scratch: [class block of 64][row block][128 rows][64 classes]; padded rows hold zeros
            uint4* dst = reinterpret_cast<uint4*>(p.g + ((int64_t)((cb >> 6) * p.n_rb + rb) * BM + quad * 32 + lane) * 64 + (cb & 32));
#pragma unroll
            for (int q = 0; q < 4; ++q) dst[q] = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
    if (MODE == MODE_STATS && cur_rb >= 0 && row_ok) {
      p.part_max[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = run_m * kLn2;
      p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = run_l;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc<2 * BN>(tmem_base);
}

// ================================================================================================
// logits kernel, CTA-pair version (cta_group::2): one tcgen05.mma of M = 256 covers two row blocks.
//   Each CTA of the pair keeps ITS 128-row x_hat block stationary in smem and receives only ITS 128-class half of every
//   256-class w_hat tile (16 KB per k-block instead of 32 KB): the L2 -> SM delivery per MMA is halved, which is what
//   bounds the single-CTA kernel (measured ~42 B/clk/SM).  The leader CTA (even cluster rank) issues the MMAs; its
//   tcgen05.commit is multicast to the barriers of both CTAs; every CTA runs its own epilogue on its own TMEM rows.
//   MODE_GRAD stores G through per-warp swizzled staging boxes and TMA stores into the blocked scratch.
// ================================================================================================
// extra HBM-streaming warps of the NORM variant.  MODE_PROB: 6 of them make a 512-thread CTA = 128 registers per thread,
// which its epilogue (two 32-column groups in flight + the packed bf16 staging) needs to stay spill-free; a setmaxnreg
// split (epilogue warpgroups up, the rest down) made ptxas spill in the reduced half and was dropped.
__host__ __device__ constexpr int norm_warps(int mode) { return mode == MODE_PROB ? 6 : 8; }
template <int STAGES, int MODE, bool NORM>
__global__ void __launch_bounds__(kLogitsThreads + (NORM ? norm_warps(MODE) * 32 : 0), 1)
    logits2_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                   const __grid_constant__ CUtensorMap tmap_g, const LogitsParams p) {
  constexpr int BN = 256;                 // classes per pair tile
  constexpr int BH = 128;                 // classes per CTA (its half of the B operand)
  constexpr int kBStage = BH * BK * 2;    // 16 KB
  constexpr int kGBox = 32 * 128;         // per-warp G staging: 32 rows x 64 classes bf16
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int n_kb = p.emb / BK;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + n_kb * kChunkBytes;
  uint8_t* smem_g = smem_b + STAGES * kBStage;                                   // [8 warps] staging (MODE_GRAD only)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_g + (MODE != MODE_STATS ? kLogitsEpiWarps * kGBox : 0));
  uint64_t* full = bars;                          // [STAGES]  used in the leader only (both CTAs' TMA bytes land here)
  uint64_t* empty = bars + STAGES;                // [STAGES]
  uint64_t* tmem_full = bars + 2 * STAGES;        // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;   // [2]      used in the leader only (arrivals from both CTAs)
  uint64_t* a_full = bars + 2 * STAGES + 4;       //          leader only
  uint64_t* a_empty = bars + 2 * STAGES + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 6);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int n_rp = (p.n_rb + 1) >> 1;                                 // row-block pairs
  const int64_t n_items = (int64_t)n_rp * p.n_ct;
  const int64_t t0 = n_items * pair / n_pairs, t1 = n_items * (pair + 1) / n_pairs;
  constexpr int kProducerWarp = kLogitsEpiWarps, kMmaWarp = kLogitsEpiWarps + 1;
  constexpr int kNormWarps = norm_warps(MODE);

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 2 * kLogitsEpiWarps); }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    fence_barrier_init();
  }
  if (warp == kProducerWarp && lane == 0) { prefetch_tmap(&tmap_x); prefetch_tmap(&tmap_w); if (MODE != MODE_STATS) prefetch_tmap(&tmap_g); }
  if (warp == kMmaWarp) tmem_alloc_2cta<2 * BN>(tmem_slot);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kProducerWarp) {
    // ------------------------------------------------------------------ TMA producer (both CTAs; bytes are credited to the leader)
    if (lane == 0) {
      PipeState ps;
      int cur_rp = -1, a_loads = 0;
      const uint32_t a_full_leader = mapa_u32(smem_u32(a_full), 0);
      for (int64_t t = t0; t < t1; ++t) {
        const int rp = (int)(t / p.n_ct), ct = (int)(t % p.n_ct);
        if (rp != cur_rp) {
          if (a_loads > 0) mbar_wait(a_empty, (a_loads - 1) & 1);
          if (leader) mbar_arrive_expect_tx(a_full, 2 * n_kb * kChunkBytes);
          const int rb = rp * 2 + (int)crank;
          for (int kb = 0; kb < n_kb; ++kb) tma_load_2d_2cta(smem_a + kb * kChunkBytes, &tmap_x, a_full_leader, kb * BK, rb * BM);
          cur_rp = rp;
          ++a_loads;
        }
        if (p.prefetch && t + 1 < t1) {                       // this CTA's half of the next class tile -> L2
          const int nct = (int)((t + 1) % p.n_ct);
          for (int kb = 0; kb < n_kb; ++kb) tma_prefetch_2d(&tmap_w, kb * BK, nct * BN + (int)crank * BH);
        }
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&empty[ps.stage], ps.phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full[ps.stage], 2 * kBStage);
          tma_load_2d_2cta(smem_b + ps.stage * kBStage, &tmap_w, mapa_u32(smem_u32(&full[ps.stage]), 0), kb * BK, ct * BN + (int)crank * BH);
          ps.advance(STAGES);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * BM, BN, false, false);
      PipeState ps;
      int cur_rp = -1, a_uses = 0;
      int64_t it = 0;
      for (int64_t t = t0; t < t1; ++t, ++it) {
        const int rp = (int)(t / p.n_ct);
        if (rp != cur_rp) {
          mbar_wait(a_full, a_uses & 1);
          ++a_uses;
          cur_rp = rp;
        }
        const int acc = (int)(it & 1);
        mbar_wait(&tmem_empty[acc], (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&full[ps.stage], ps.phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + kb * kChunkBytes);
          const uint32_t b_addr = smem_u32(smem_b + ps.stage * kBStage);
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            const uint64_t da = make_desc_sw128(a_addr + kk * 32, 0, 1024);
            const uint64_t db = make_desc_sw128(b_addr + kk * 32, 0, 1024);
            umma_bf16_ss_2cta(d_tmem, da, db, idesc, (kb | kk) != 0);
          }
          umma_commit_2cta(&empty[ps.stage], 3);
          ps.advance(STAGES);
        }
        umma_commit_2cta(&tmem_full[acc], 3);
        const bool last_of_rp = (t + 1 == t1) || ((int)((t + 1) / p.n_ct) != rp);
        if (last_of_rp) umma_commit_2cta(a_empty, 3);
      }
    }
  } else if (NORM && warp >= kLogitsEpiWarps + 2) {
    // ------------------------------------------------------------------ normaliser warps: pure HBM streaming (fp32 rows -> bf16 + 1/norm)
    normalize_rows_warp<4, 2, 2>(p.norm_w, p.norm_index, p.norm_rows, p.emb, p.norm_out, nullptr, p.norm_inv,
                              (int64_t)blockIdx.x * kNormWarps + (warp - (kLogitsEpiWarps + 2)), (int64_t)gridDim.x * kNormWarps, lane);
  } else {
    // ------------------------------------------------------------------ epilogue (8 warps per CTA), thread = row of THIS CTA's block
    const int quad = warp & 3, chalf = warp >> 2;
    constexpr int CH = BN / 2;
    const float s2 = p.s * kLog2e;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    constexpr int kNoLabel = -(1 << 30);
    uint8_t* gbuf = smem_g + warp * kGBox;
    int cur_rp = -1, rb = 0;
    int row = 0, my_label = kNoLabel;
    bool row_ok = false;
    float run_m = -INFINITY, run_l = 0.f;
    float M2 = 0.f, rS = 0.f;
    int64_t it = 0;
    for (int64_t t = t0; t < t1; ++t, ++it) {
      const int rp = (int)(t / p.n_ct), ct = (int)(t % p.n_ct);
      if (rp != cur_rp) {
        if (MODE != MODE_GRAD && cur_rp >= 0 && row_ok) {
          p.part_max[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = MODE == MODE_HINGE ? 0.f : (MODE == MODE_PROB ? M2 : run_m) * kLn2;
          p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = run_l;
        }
        cur_rp = rp;
        rb = rp * 2 + (int)crank;
        row = rb * BM + quad * 32 + lane;
        row_ok = row < p.n_rows;
        my_label = kNoLabel;
        if (row_ok && MODE != MODE_HINGE) {
          const int64_t y = p.label[row];
          if (y >= 0) my_label = (int)(y - p.class_base);
        }
        run_m = -INFINITY; run_l = 0.f;
        if (MODE == MODE_STATS && p.accumulate_stats && row_ok) {
          const float l0 = p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row];
          if (l0 > 0.f) { run_l = l0; run_m = p.part_max[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] * kLog2e; }
        }
        M2 = 0.f; rS = 0.f;
        if (MODE == MODE_GRAD && row_ok) { M2 = p.row_max[row] * kLog2e; rS = 1.0f / p.row_sum[row]; }
        if (MODE == MODE_PROB) {                           // rows past n_rows: exp2(-inf) = 0, nothing stored or summed
          M2 = row_ok ? p.row_bound[row] : INFINITY;
          if (p.accumulate_stats && row_ok) run_l = p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row];
        }
        if (MODE == MODE_HINGE && p.accumulate_stats && row_ok) run_l = p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row];
      }
      const int acc = (int)(it & 1);
      mbar_wait(&tmem_full[acc], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const int col0 = ct * BN;
      const bool tile_has_oob = col0 + BN > p.n_classes;
      // one 32-column group; the TMEM load of the next group is in flight while this one is processed
      auto process_group = [&](uint32_t (&v)[32], const int c) {
        const int cb = col0 + c;
        const int hit = my_label - cb;                       // in [0,32) iff this row's target class is in this column group
        const bool has_hit = hit >= 0 && hit < 32;
        float c_hit = 0.f, slope = 1.f;                      // plain cosine / margin slope at the target
        if (has_hit) {                                       // rare: fold the margin into the cosine
#pragma unroll
          for (int j = 0; j < 32; ++j) if (j == hit) {
            c_hit = __uint_as_float(v[j]);
            slope = margin_slope(c_hit, p.m, p.margin_kind);
            v[j] = __float_as_uint(margin_cos(c_hit, p.m, p.margin_kind));
            if (MODE != MODE_GRAD) p.target_logit[row] = p.s * __uint_as_float(v[j]);
            if (MODE == MODE_PROB) p.target_cos[row] = c_hit;
          }
        }
        if (MODE == MODE_HINGE) {
          // SpreadOut (server.py:48-63): H = relu(cos - margin) off the diagonal (x_hat == w_hat: row i, column j are classes),
          // sum of H^2 per row into this CTA's slot, H -> bf16 scratch for the gradient GEMM  dW_hat = 4 H . w_hat
          const float2 mv = make_float2(-p.m, -p.m), zero2 = make_float2(0.f, 0.f);
          float2 g[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float2 d = __fadd2_rn(make_float2(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), mv);
            g[q] = make_float2(fmaxf(d.x, zero2.x), fmaxf(d.y, zero2.y));
          }
          const int diag = row - (p.class_base + cb);                  // in [0, 32) iff this row's own column is in the group
          if ((diag >= 0 && diag < 32) || tile_has_oob || !row_ok) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              if (2 * q == diag || cb + 2 * q >= p.n_classes || !row_ok) g[q].x = 0.f;
              if (2 * q + 1 == diag || cb + 2 * q + 1 >= p.n_classes || !row_ok) g[q].y = 0.f;
            }
          }
          float2 sum = __fmul2_rn(g[0], g[0]);
#pragma unroll
          for (int q = 1; q < 16; ++q) sum = __ffma2_rn(g[q], g[q], sum);
          run_l += sum.x + sum.y;
          uint32_t pk[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) pk[q] = pack_bf16x2(g[q].x, g[q].y);
          const int half = (c >> 5) & 1;
          if (half == 0) {
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
          }
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(gbuf + sw128_off(lane, half * 4 + q)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
          if (half == 1) {
            fence_proxy_async_smem();
            __syncwarp();
            const int cbg = p.class_base + cb;
            if (lane == 0 && cbg < p.ldg && rb < p.n_rb) {
              tma_store_2d(&tmap_g, gbuf, 0, ((cbg >> 6) * p.n_rb + rb) * BM + quad * 32);
              tma_store_commit();
            }
          }
        } else if (MODE == MODE_PROB) {
          // P = exp2(s2 cos - bound): summed in fp32 (the softmax denominator, target included), stored as bf16 with the
          // target column zeroed -- the backward writes that one element from fp32 statistics (no p - 1 cancellation).
          const float2 s2v = make_float2(s2, s2), m2v = make_float2(-M2, -M2);
          float2 g[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float2 zz = __ffma2_rn(make_float2(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), s2v, m2v);
            g[q] = make_float2(fast_exp2(zz.x), fast_exp2(zz.y));
          }
          if (tile_has_oob) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              if (cb + 2 * q >= p.n_classes) g[q].x = 0.f;
              if (cb + 2 * q + 1 >= p.n_classes) g[q].y = 0.f;
            }
          }
          float2 sum = g[0];
#pragma unroll
          for (int q = 1; q < 16; ++q) sum = __fadd2_rn(sum, g[q]);
          run_l += sum.x + sum.y;
          if (has_hit) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              if (2 * q == hit) g[q].x = 0.f;
              if (2 * q + 1 == hit) g[q].y = 0.f;
            }
          }
          uint32_t pk[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) pk[q] = pack_bf16x2(g[q].x, g[q].y);
          const int half = (c >> 5) & 1;
          if (half == 0) {
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
          }
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(gbuf + sw128_off(lane, half * 4 + q)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
          if (half == 1) {
            fence_proxy_async_smem();
            __syncwarp();
            const int cbg = p.class_base + cb;               // the scratch spans the whole shard
            if (lane == 0 && cbg < p.ldg && rb < p.n_rb) {
              tma_store_2d(&tmap_g, gbuf, 0, ((cbg >> 6) * p.n_rb + rb) * BM + quad * 32);
              tma_store_commit();
            }
          }
        } else if (MODE == MODE_STATS) {
          if (tile_has_oob) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (cb + j >= p.n_classes) v[j] = __float_as_uint(-INFINITY);
          }
          // group max on the raw cosines (s > 0), three inputs per instruction
          float cm = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
#pragma unroll
          for (int j = 3; j < 31; j += 2) cm = fmax3(cm, __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
          cm = fmaxf(cm, __uint_as_float(v[31])) * s2;
          if (cm > -INFINITY) {
            const float nm = fmaxf(run_m, cm);
            const float2 s2v = make_float2(s2, s2), nmv = make_float2(-nm, -nm);
            float2 sum = make_float2(0.f, 0.f);
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const float2 zz = __ffma2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), s2v, nmv);
              sum = __fadd2_rn(sum, make_float2(fast_exp2(zz.x), fast_exp2(zz.y)));
            }
            run_l = run_l * fast_exp2(run_m - nm) + (sum.x + sum.y);
            run_m = nm;
          }
        } else {
          // G = (exp2(s2 cos - M2) * rS - onehot) * g_scale, packed two columns per instruction
          const float2 s2v = make_float2(s2, s2), m2v = make_float2(-M2, -M2);
          const float gs = rS * p.g_scale;
          const float2 gsv = make_float2(gs, gs);
          float2 g[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float2 zz = __ffma2_rn(make_float2(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), s2v, m2v);
            g[q] = __fmul2_rn(make_float2(fast_exp2(zz.x), fast_exp2(zz.y)), gsv);
          }
          if (has_hit) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              if (2 * q == hit) g[q].x = (g[q].x - p.g_scale) * slope;
              if (2 * q + 1 == hit) g[q].y = (g[q].y - p.g_scale) * slope;
            }
          }
          uint32_t pk[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) pk[q] = pack_bf16x2(g[q].x, g[q].y);
          // G -> swizzled staging box [32 rows x 64 classes]; one TMA store per 64 classes into the blocked scratch
          const int half = (c >> 5) & 1;
          if (half == 0) {
            if (lane == 0) tma_store_wait_read<0>();      // the previous store out of this warp's box has been read
            __syncwarp();
          }
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(gbuf + sw128_off(lane, half * 4 + q)) = make_uint4(pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
          if (half == 1) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0 && cb < p.ldg && rb < p.n_rb) {      // (a phantom row block of an odd pair has no scratch)
              tma_store_2d(&tmap_g, gbuf, 0, ((cb >> 6) * p.n_rb + rb) * BM + quad * 32);
              tma_store_commit();
            }
          }
        }
      };
      {
        constexpr int NG = CH / 32;
        static_assert(NG % 2 == 0, "two groups per pipeline round");
        const uint32_t t_base = tmem_base + lane_base + acc * BN + chalf * CH;
        uint32_t va[32], vb[32];
        tmem_ld_x32(t_base, va);
#pragma unroll
        for (int gi = 0; gi < NG; gi += 2) {
          tmem_ld_wait();
          tmem_ld_x32(t_base + (gi + 1) * 32, vb);
          process_group(va, chalf * CH + gi * 32);
          tmem_ld_wait();
          if (gi + 2 < NG) tmem_ld_x32(t_base + (gi + 2) * 32, va);
          process_group(vb, chalf * CH + (gi + 1) * 32);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {                                     // the accumulator lives in both CTAs; the leader's MMA warp waits for all 16 warps
        if (leader) mbar_arrive(&tmem_empty[acc]);
        else mbar_arrive_cluster_addr_relaxed(mapa_u32(smem_u32(&tmem_empty[acc]), 0));
      }
    }
    if (MODE != MODE_GRAD && cur_rp >= 0 && row_ok) {
      p.part_max[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = MODE == MODE_HINGE ? 0.f : (MODE == MODE_PROB ? M2 : run_m) * kLn2;
      p.part_sum[(int64_t)(blockIdx.x * 2 + chalf) * p.n_rows + row] = run_l;
    }
    if (MODE != MODE_STATS && lane == 0) tma_store_wait_all();
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == kMmaWarp) tmem_dealloc_2cta<2 * BN>(tmem_base);
}

// ================================================================================================
// dx kernel: D[128 rows x BN e] = sum over a class slice of G[rows, classes] * w_hat[classes, e]
//   A = G (K-major, K = classes), B = w_hat (MN-major: N = e contiguous, K = classes)
// ================================================================================================
// dx and dw run side by side and both walk the class axis upwards, reading the same G (or P) and w_hat tiles.  Each
// publishes the furthest class it has requested; whoever is more than `lead` classes ahead of the other waits, so the
// second reader of a tile finds it in L2 (the phase is HBM bound: a tile fetched twice costs as much as the dw write).
// Purely a pacing hint: the wait gives up after a bounded number of polls, and a finished kernel leaves its counter
// at the end of the class axis.
struct SweepSync {
  int* self;            // device counters (nullptr = not paced)
  const int* other;
  int lead;
};
__device__ __forceinline__ void sweep_pace(const SweepSync& sw, int pos) {
  if (sw.self == nullptr) return;
  atomicMax(sw.self, pos);
  int polls = 0;
  while (pos > *reinterpret_cast<const volatile int*>(sw.other) + sw.lead && ++polls < (1 << 14)) __nanosleep(200);
}

struct DxParams {
  SweepSync sweep;
  int n_rows, n_classes, emb;
  int n_rb, n_eh, ksplit;
  float* dx_part;          // [ksplit, n_rows, emb]
  int accumulate;
  int prefetch;            // > 0: TMA L2 prefetch distance in k-blocks
  int strided;             // 1: k-blocks ks, ks + ksplit, ... instead of a contiguous slice
};

template <int BN, int STAGES, int CS>
__global__ void __launch_bounds__(kThreads, 1) dx_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_w,
                                                         const DxParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kBBytes = (BN / 64) * kBoxBytes;
  constexpr int kStageBytes = kChunkBytes + kBBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * kStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // cluster = CS consecutive row blocks working on the same (e-half, class slice): they share the w_hat stream
  const uint32_t crank = CS > 1 ? cluster_ctarank() : 0;
  const int grp = blockIdx.x / CS;
  const int ks = grp % p.ksplit, eh = (grp / p.ksplit) % p.n_eh, rb = (grp / (p.ksplit * p.n_eh)) * CS + (int)crank;
  constexpr uint16_t kMask = (uint16_t)((1u << CS) - 1);
  const int n_kb_total = (p.n_classes + BK - 1) / BK;
  // k-blocks of this CTA: a contiguous slice, or (p.strided) every ksplit-th block so that all CTAs sweep the class axis
  // together -- in step with a dw kernel running beside it, whose reads of the same G / w_hat tiles then hit L2
  const int kstep = p.strided ? p.ksplit : 1;
  const int kb0 = p.strided ? ks : (int)((int64_t)n_kb_total * ks / p.ksplit);
  const int kb1 = p.strided ? n_kb_total : (int)((int64_t)n_kb_total * (ks + 1) / p.ksplit);

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], CS); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) { prefetch_tmap(&tmap_g); prefetch_tmap(&tmap_w); }
  if (warp == 5) tmem_alloc<BN>(tmem_slot);
  tc_fence_before();
  if (CS > 1) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      PipeState ps;
      int n_issued = 0;
      for (int kb = kb0; kb < kb1; kb += kstep) {
        if (p.prefetch && kb + p.prefetch * kstep < kb1) {  // k-block (kb + distance) -> L2 while the ring is still busy with kb
          const int pk = kb + p.prefetch * kstep;
          tma_prefetch_2d(&tmap_g, 0, (pk * p.n_rb + rb) * BM);
          if (CS == 1) {
#pragma unroll
            for (int nb = 0; nb < BN / 64; ++nb) tma_prefetch_2d(&tmap_w, eh * BN + nb * 64, pk * BK);
          } else {
            constexpr int kPer = (BN / 64) / CS;
#pragma unroll
            for (int q = 0; q < kPer; ++q) tma_prefetch_2d(&tmap_w, eh * BN + ((int)crank * kPer + q) * 64, pk * BK);
          }
        }
        if (crank == 0 && (n_issued++ & 3) == 0) sweep_pace(p.sweep, kb * BK);
        mbar_wait(&empty[ps.stage], ps.phase ^ 1);
        uint8_t* sa = smem + ps.stage * kStageBytes;
        uint8_t* sb = sa + kChunkBytes;
        mbar_arrive_expect_tx(&full[ps.stage], kStageBytes);
        tma_load_2d(sa, &tmap_g, &full[ps.stage], 0, (kb * p.n_rb + rb) * BM);      // one contiguous 16 KB block of the G scratch
        if (CS == 1) {
#pragma unroll
          for (int nb = 0; nb < BN / 64; ++nb) tma_load_2d(sb + nb * kBoxBytes, &tmap_w, &full[ps.stage], eh * BN + nb * 64, kb * BK);
        } else {                                  // this CTA fetches 1/CS of the w_hat boxes for the whole cluster
          constexpr int kPer = (BN / 64) / CS;
#pragma unroll
          for (int q = 0; q < kPer; ++q) {
            const int nb = (int)crank * kPer + q;
            tma_load_2d_mc(sb + nb * kBoxBytes, &tmap_w, &full[ps.stage], eh * BN + nb * 64, kb * BK, kMask);
          }
        }
        ps.advance(STAGES);
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, false, true);
      PipeState ps;
      for (int kb = kb0; kb < kb1; kb += kstep) {
        mbar_wait(&full[ps.stage], ps.phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + ps.stage * kStageBytes);
        const uint32_t b_addr = a_addr + kChunkBytes;
#pragma unroll
        for (int kk = 0; kk < BK / 16; ++kk) {
          const uint64_t da = make_desc_sw128(a_addr + kk * 32, 0, 1024);
          const uint64_t db = make_desc_sw128(b_addr + kk * 2048, kBoxBytes, 1024);
          umma_bf16_ss(tmem_base, da, db, idesc, (kb != kb0) || (kk != 0));
        }
        if (CS == 1) umma_commit(&empty[ps.stage]); else umma_commit_mc(&empty[ps.stage], kMask);
        ps.advance(STAGES);
      }
      umma_commit(tmem_full);
    }
  } else {
    const int row = rb * BM + threadIdx.x;
    const bool row_ok = row < p.n_rows;
    float* out = p.dx_part + ((int64_t)ks * p.n_rows + row) * p.emb + eh * BN;
    const bool have = kb1 > kb0;
    if (have) {
      mbar_wait(tmem_full, 0);
      tc_fence_after();
    }
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      uint32_t v[32];
      if (have) {
        tmem_ld_x32(tmem_base + lane_base + c, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0;
      }
      if (row_ok) {
        float4* o = reinterpret_cast<float4*>(out + c);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float4 r = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                                 __uint_as_float(v[4 * q + 3]));
          if (p.accumulate) { float4 old = o[q]; r.x += old.x; r.y += old.y; r.z += old.z; r.w += old.w; }
          o[q] = r;
        }
      }
    }
  }
  tc_fence_before();
  if (CS > 1) cluster_sync_all(); else __syncthreads();     // peers may still multicast into / arrive on this CTA
  if (warp == 5) tmem_dealloc<BN>(tmem_base);
}

// ================================================================================================
// dx kernel, CTA-pair version (cta_group::2), used when the gathered batch is a multiple of 512 rows.
//   A pair owns a row quad (4 row blocks = 512 rows), one e-half (N = 256) and a set of k-blocks (64 classes each).
//   Two accumulators live in TMEM for the whole kernel: acc 0 = row blocks (4q, 4q+1), acc 1 = (4q+2, 4q+3); CTA r of
//   the pair holds rows of blocks 4q + r and 4q + 2 + r.  Per k-block a CTA receives its two G boxes (2 x 16 KB) and
//   HALF of the w_hat tile (its 128 e-columns, 16 KB): 48 KB per 1024 MMA cycles, half of what the single-CTA kernel
//   needs -- that kernel is bound by L2 -> SM delivery -- and every w_hat byte is fetched once per row quad.
// ================================================================================================
template <int STAGES>
__global__ void __launch_bounds__(kThreads, 1) dx2_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_w,
                                                          const DxParams p) {
  constexpr int BN = 256;
  constexpr int kABytes = 2 * kChunkBytes;          // two G boxes [128 rows x 64 classes]
  constexpr int kBBytes = 2 * kBoxBytes;            // w_hat [64 classes x 128 e] = two boxes
  constexpr int kStageBytes = kABytes + kBBytes;    // 48 KB
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * kStageBytes);
  uint64_t* full = bars;                 // leader only: both CTAs' TMA bytes land here
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int pair = blockIdx.x >> 1;
  const int ks = pair % p.ksplit, eh = (pair / p.ksplit) % p.n_eh, quad = pair / (p.ksplit * p.n_eh);
  const int rb0 = quad * 4 + (int)crank, rb1 = rb0 + 2;
  const int n_kb_total = (p.n_classes + BK - 1) / BK;
  const int kstep = p.strided ? p.ksplit : 1;
  const int kb0 = p.strided ? ks : (int)((int64_t)n_kb_total * ks / p.ksplit);
  const int kb1 = p.strided ? n_kb_total : (int)((int64_t)n_kb_total * (ks + 1) / p.ksplit);

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) { prefetch_tmap(&tmap_g); prefetch_tmap(&tmap_w); }
  if (warp == 5) tmem_alloc_2cta<2 * BN>(tmem_slot);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      PipeState ps;
      int n_issued = 0;
      for (int kb = kb0; kb < kb1; kb += kstep, ++n_issued) {
        if (leader && (n_issued & 3) == 0) sweep_pace(p.sweep, kb * BK);
        mbar_wait(&empty[ps.stage], ps.phase ^ 1);
        uint8_t* sa = smem + ps.stage * kStageBytes;
        uint8_t* sb = sa + kABytes;
        const uint32_t full_leader = mapa_u32(smem_u32(&full[ps.stage]), 0);
        if (leader) mbar_arrive_expect_tx(&full[ps.stage], 2 * kStageBytes);
        tma_load_2d_2cta(sa, &tmap_g, full_leader, 0, (kb * p.n_rb + rb0) * BM);
        tma_load_2d_2cta(sa + kChunkBytes, &tmap_g, full_leader, 0, (kb * p.n_rb + rb1) * BM);
#pragma unroll
        for (int nb = 0; nb < 2; ++nb)
          tma_load_2d_2cta(sb + nb * kBoxBytes, &tmap_w, full_leader, eh * BN + (int)crank * 128 + nb * 64, kb * BK);
        ps.advance(STAGES);
      }
    }
  } else if (warp == 5) {
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * BM, BN, false, true);
      PipeState ps;
      for (int kb = kb0; kb < kb1; kb += kstep) {
        mbar_wait(&full[ps.stage], ps.phase);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + ps.stage * kStageBytes);
        const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
        for (int acc = 0; acc < 2; ++acc) {
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            const uint64_t da = make_desc_sw128(a_addr + acc * kChunkBytes + kk * 32, 0, 1024);
            const uint64_t db = make_desc_sw128(b_addr + kk * 2048, kBoxBytes, 1024);
            umma_bf16_ss_2cta(tmem_base + acc * BN, da, db, idesc, (kb != kb0) || (kk != 0));
          }
        }
        umma_commit_2cta(&empty[ps.stage], 3);
        ps.advance(STAGES);
      }
      umma_commit_2cta(tmem_full, 3);
    }
  } else {
    const bool have = kb1 > kb0;
    if (have) {
      mbar_wait(tmem_full, 0);
      tc_fence_after();
    }
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
#pragma unroll 1
    for (int acc = 0; acc < 2; ++acc) {
      const int row = (acc == 0 ? rb0 : rb1) * BM + threadIdx.x;
      const bool row_ok = row < p.n_rows;
      float* out = p.dx_part + ((int64_t)ks * p.n_rows + row) * p.emb + eh * BN;
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        uint32_t v[32];
        if (have) {
          tmem_ld_x32(tmem_base + lane_base + acc * BN + c, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0;
        }
        if (row_ok) {
          float4* o = reinterpret_cast<float4*>(out + c);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 r = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                                   __uint_as_float(v[4 * q + 3]));
            if (p.accumulate) { float4 old = o[q]; r.x += old.x; r.y += old.y; r.z += old.z; r.w += old.w; }
            o[q] = r;
          }
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 5) tmem_dealloc_2cta<2 * BN>(tmem_base);
}

__global__ void reduce_dx_kernel(const float4* __restrict__ part, int ksplit, int64_t n_vec, float4* __restrict__ dx) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    float4 a = part[i];
    for (int k = 1; k < ksplit; ++k) {
      const float4 b = part[(int64_t)k * n_vec + i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    dx[i] = a;
  }
}

// ================================================================================================
// dw kernel: D[128 classes x EN e] = G^T[classes, rows] * x_hat[rows, e-slice], epilogue = normalize backward
//   A = G^T (MN-major: M = classes contiguous in a G row), B = x_hat (MN-major: N = e contiguous), K = rows
//   (G is either the gradient scratch of logits_kernel<MODE_GRAD> or the stored probabilities of MODE_PROB, in which
//   case B is the row-scaled x_hat.)
//   Work item = (class tile, e-slice of EN = min(E, 256) columns): the accumulator is EN TMEM columns, two of them
//   are allocated so the epilogue of item k overlaps the MMAs of item k+1.
//   Epilogue = normalize backward,   dw_j[e] = (acc[e] - w_hat_j[e] * t_j) * inv_norm_j,   t_j = w_hat_j . acc_j:
//   two passes over the accumulator (dot, then output); thread = class row, so the dot is thread-local.
//     E <= 256: one item holds the whole row; a cluster of CS CTAs = CS class tiles in lock step sharing the x_hat
//               stream by TMA multicast.
//     E == 512: the row spans two e-slices.  A cluster of 2 CTAs owns ONE class tile, CTA r computes slice r; the G^T
//               tile is fetched once and multicast to both, and the two partial dots are exchanged through distributed
//               shared memory (st.shared::cluster + a cluster-scope mbarrier per warp) between the passes.
//   Each epilogue warp owns 32 classes: its w_hat rows arrive by its own TMA loads into swizzled smem (issued one
//   item ahead), the result leaves through swizzled staging boxes and its own TMA stores / reduce-adds.
// ================================================================================================
struct DwParams {
  SweepSync sweep;
  int n_rows, n_classes, emb;     // n_classes = classes in this launch
  int n_ct, n_rb;
  const float* inv_norm;          // [n_classes]
  int accumulate;
  int prefetch;                   // 1: TMA L2 prefetch of the next tile's G / w_hat boxes
  long long* dbg;                 // optional cycle counters of CTA 0 (developer instrumentation), else nullptr
};

__device__ __forceinline__ void st_cluster_f32(uint32_t cluster_addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(cluster_addr), "f"(v) : "memory");
}

constexpr int kDwEpiWarps = 8;                 // two warps per TMEM lane quadrant, each takes half of the slice's columns
constexpr int kDwThreads = (kDwEpiWarps + 2) * 32;

template <int EMB, int STAGES, int CS>
__global__ void __launch_bounds__(kDwThreads, 1) dw_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_x,
                                                           const __grid_constant__ CUtensorMap tmap_wh, const __grid_constant__ CUtensorMap tmap_dw,
                                                           const DwParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int EN = EMB < 256 ? EMB : 256;              // accumulator width = N of one MMA
  constexpr int NH = EMB / EN;                           // e-slices per class tile
  constexpr bool ES = NH == 2;                           // e-split cluster: both CTAs work on the same class tile
  static_assert(!ES || CS == 2, "the e-split arrangement is a cluster of two CTAs");
  constexpr int NBOX = EN / 64;                          // 64-wide boxes per e-slice
  constexpr int NCG = kDwEpiWarps / 4;                   // column groups (epilogue warps per lane quadrant)
  constexpr int CW = EN / NCG;                           // columns per epilogue warp
  constexpr int NG = CW / 32;                            // 32-column groups per epilogue warp (1, 2 or 4)
  constexpr int kContrib = (ES ? 2 : 1) * NCG;           // partial dots per class row: (cluster rank x) column group
  constexpr int kABytes = 2 * kBoxBytes;                 // 128 classes x 64 rows
  constexpr int kBBytes = NBOX * kBoxBytes;              // EN x 64 rows
  constexpr int kStageBytes = kABytes + kBBytes;
  constexpr int kWBox = 32 * 128;                        // w_hat box: 32 classes x 64 e bf16 = 4 KB = one fp32 staging box [32 x 32]
  constexpr int kWWarp = (NG + 1) / 2 * kWBox;           // per-warp w_hat columns (a warp with 32 columns still loads a 64-e box)
  constexpr int kSBox = NG == 1 ? 2 : 0;                 // extra staging boxes of the warps that own a single w_hat box
  uint8_t* smem_w = smem + STAGES * kStageBytes;         // [8 warps] w_hat boxes, reused as output staging
  uint8_t* smem_s = smem_w + kDwEpiWarps * kWWarp;       // [8 warps][kSBox] staging
  float* tpart = reinterpret_cast<float*>(smem_s + kDwEpiWarps * kSBox * kWBox);   // [2][kContrib][128] partial dots
  uint64_t* bars = reinterpret_cast<uint64_t*>(tpart + 2 * 8 * 128);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;               // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;          // [2]
  uint64_t* wfull = bars + 2 * STAGES + 4;               // [8 warps]
  uint64_t* tbar = bars + 2 * STAGES + 4 + kDwEpiWarps;  // [2][4 quadrants] all partial dots of the quadrant's rows have landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 12 + kDwEpiWarps);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_kb = (p.n_rows + BK - 1) / BK;
  const uint32_t crank = CS > 1 ? cluster_ctarank() : 0;
  const int n_clusters = gridDim.x / CS, cid = blockIdx.x / CS;
  constexpr uint16_t kMask = (uint16_t)((1u << CS) - 1);
  constexpr int kProducerWarp = kDwEpiWarps, kMmaWarp = kDwEpiWarps + 1;
  // ES:   item i -> class tile i * n_clusters + cid (both CTAs), e-slice = cluster rank.
  // else: item i -> class tile (i * n_clusters + cid) * CS + crank, the only e-slice.  Every CTA of a cluster runs the
  //       same number of items (tiles past n_ct are phantoms: TMA zero-fills their loads and clips their stores).
  auto tile_of = [&](int i) { return ES ? i * n_clusters + cid : (i * n_clusters + cid) * CS + (int)crank; };
  auto more = [&](int i) { return ES ? i * n_clusters + cid < p.n_ct : (i * n_clusters + cid) * CS < p.n_ct; };
  const int hs = ES ? (int)crank : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], CS); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], kDwEpiWarps); }
    for (int i = 0; i < kDwEpiWarps; ++i) mbar_init(&wfull[i], 1);
    for (int i = 0; i < 8; ++i) mbar_init(&tbar[i], kContrib);
    fence_barrier_init();
  }
  if (warp == kProducerWarp && lane == 0) { prefetch_tmap(&tmap_g); prefetch_tmap(&tmap_x); prefetch_tmap(&tmap_wh); prefetch_tmap(&tmap_dw); }
  if (warp == kMmaWarp) tmem_alloc<2 * EN>(tmem_slot);
  tc_fence_before();
  if (CS > 1) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kProducerWarp) {
    if (lane == 0) {
      PipeState ps;
      for (int i = 0; more(i); ++i) {
        const int ct = tile_of(i);
        if (crank == 0) sweep_pace(p.sweep, ct * BM);
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait_cluster(&empty[ps.stage], ps.phase ^ 1);
          uint8_t* sa = smem + ps.stage * kStageBytes;
          uint8_t* sb = sa + kABytes;
          mbar_arrive_expect_tx(&full[ps.stage], kStageBytes);
          // G scratch blocks (2 ct, kb / 2) and (2 ct + 1, kb / 2): 64 rows x 64 classes each, contiguous 8 KB
          if (ES) {                               // this CTA fetches class half `crank` for both CTAs of the cluster
            tma_load_2d_mc(sa + crank * kBoxBytes, &tmap_g, &full[ps.stage], 0, ((2 * ct + (int)crank) * p.n_rb + (kb >> 1)) * BM + (kb & 1) * 64, kMask);
#pragma unroll
            for (int nb = 0; nb < NBOX; ++nb) tma_load_2d(sb + nb * kBoxBytes, &tmap_x, &full[ps.stage], hs * EN + nb * 64, kb * BK);
          } else {
            tma_load_2d(sa, &tmap_g, &full[ps.stage], 0, ((2 * ct) * p.n_rb + (kb >> 1)) * BM + (kb & 1) * 64);
            tma_load_2d(sa + kBoxBytes, &tmap_g, &full[ps.stage], 0, ((2 * ct + 1) * p.n_rb + (kb >> 1)) * BM + (kb & 1) * 64);
            if (CS == 1) {
#pragma unroll
              for (int nb = 0; nb < NBOX; ++nb) tma_load_2d(sb + nb * kBoxBytes, &tmap_x, &full[ps.stage], nb * 64, kb * BK);
            } else {                              // 1/CS of the x_hat boxes, delivered to every CTA of the cluster
              constexpr int kPer = NBOX / CS > 0 ? NBOX / CS : 1;
#pragma unroll
              for (int q = 0; q < kPer; ++q) {
                const int nb = (int)crank * kPer + q;
                if (nb < NBOX) tma_load_2d_mc(sb + nb * kBoxBytes, &tmap_x, &full[ps.stage], nb * 64, kb * BK, kMask);
              }
            }
          }
          ps.advance(STAGES);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, EN, true, true);
      PipeState ps;
      long long t_we = 0, t_wf = 0, t_all = clock64();
      for (int it = 0; more(it); ++it) {
        const int acc = it & 1;
        long long c0 = clock64();
        mbar_wait_cluster(&tmem_empty[acc], (uint32_t)(((it >> 1) & 1) ^ 1));
        t_we += clock64() - c0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * EN;
        for (int kb = 0; kb < n_kb; ++kb) {
          c0 = clock64();
          mbar_wait_cluster(&full[ps.stage], ps.phase);
          t_wf += clock64() - c0;
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + ps.stage * kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            const uint64_t da = make_desc_sw128(a_addr + kk * 2048, kBoxBytes, 1024);
            const uint64_t db = make_desc_sw128(b_addr + kk * 2048, kBoxBytes, 1024);
            umma_bf16_ss(d_tmem, da, db, idesc, (kb | kk) != 0);
          }
          if (CS == 1) umma_commit(&empty[ps.stage]);
          else umma_commit_mc(&empty[ps.stage], kMask);
          ps.advance(STAGES);
        }
        umma_commit(&tmem_full[acc]);
      }
      if (p.dbg && blockIdx.x == 0) { p.dbg[0] = t_we; p.dbg[1] = t_wf; p.dbg[2] = clock64() - t_all; }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: warp (quad, chalf) owns classes [32 quad, +32) of
    // the tile and columns [chalf * CW, +CW) of the slice.  thread = class row.
    const int quad = warp & 3, chalf = warp >> 2;
    const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
    constexpr int kNW = (NG + 1) / 2;                     // w_hat boxes of this warp
    uint8_t* wbuf = smem_w + warp * kWWarp;
    uint8_t* sbuf = smem_s + warp * kSBox * kWBox;
    uint64_t* wbar = &wfull[warp];
    const uint32_t peer = crank ^ 1u;                     // the CTA holding the other e-slice of the same class tile
    const int contrib = (ES ? hs * NCG : 0) + chalf;
    const int e_warp = hs * EN + chalf * CW;              // first e column of this warp
    long long t_wfull = 0, t_ww = 0, t_ep = 0, t_p1 = 0, t_ex = 0, t_p2 = 0;
    auto issue_w = [&](int i) {                           // this warp's w_hat rows of item i (lane 0 only)
      const int cls0 = tile_of(i) * BM + quad * 32;
      mbar_arrive_expect_tx(wbar, kNW * kWBox);
#pragma unroll
      for (int nb = 0; nb < kNW; ++nb) tma_load_2d(wbuf + nb * kWBox, &tmap_wh, wbar, (e_warp & ~63) + nb * 64, cls0);
      if (more(i + 1)) {                                  // and the rows of the item after that -> L2, so this load only pays the L2 latency
        const int n0 = tile_of(i + 1) * BM + quad * 32;
#pragma unroll
        for (int nb = 0; nb < kNW; ++nb) tma_prefetch_2d(&tmap_wh, (e_warp & ~63) + nb * 64, n0);
      }
    };
    constexpr int kSub = NG == 1 ? 4 : 0;                 // 32-column warps read the upper / lower half of their 64-e box
    const int sub0 = NG == 1 ? ((e_warp >> 5) & 1) * kSub : 0;
    if (lane == 0 && more(0)) issue_w(0);
    for (int it = 0; more(it); ++it) {
      const int ct = tile_of(it);
      const int acc = it & 1;
      const int cls0 = ct * BM + quad * 32;
      const int cls = cls0 + lane;
      const bool ok = cls < p.n_classes;
      const float inv_n = ok ? p.inv_norm[cls] : 0.f;
      long long c0 = clock64();
      mbar_wait(&tmem_full[acc], (uint32_t)((it >> 1) & 1));
      t_wfull += clock64() - c0;
      c0 = clock64();
      mbar_wait(wbar, (uint32_t)(it & 1));
      t_ww += clock64() - c0;
      c0 = clock64();
      tc_fence_after();
      const uint32_t t_base = tmem_base + lane_base + acc * EN + chalf * CW;
      // ---- pass 1: partial dot t = w_hat_j . acc_j over this warp's columns (thread-local: lane = class row)
      float2 dot2 = make_float2(0.f, 0.f);
      {
        uint32_t va[32], vb[32];
        auto dot_group = [&](const uint32_t (&v)[32], int g) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 w16 = *reinterpret_cast<const uint4*>(wbuf + (g >> 1) * kWBox + sw128_off(lane, sub0 + (g & 1) * 4 + q));
            const uint32_t w4[4] = {w16.x, w16.y, w16.z, w16.w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
              dot2 = __ffma2_rn(make_float2(__uint_as_float(w4[k] << 16), __uint_as_float(w4[k] & 0xffff0000u)),
                                make_float2(__uint_as_float(v[q * 8 + 2 * k]), __uint_as_float(v[q * 8 + 2 * k + 1])), dot2);
          }
        };
        tmem_ld_x32(t_base, va);
#pragma unroll
        for (int g = 0; g < NG; g += 2) {
          tmem_ld_wait();
          if (g + 1 < NG) tmem_ld_x32(t_base + (g + 1) * 32, vb);
          dot_group(va, g);
          if (g + 1 < NG) {
            tmem_ld_wait();
            if (g + 2 < NG) tmem_ld_x32(t_base + (g + 2) * 32, va);
            dot_group(vb, g + 1);
          }
        }
      }
      t_p1 += clock64() - c0;
      // ---- exchange: every contributor (column half x cluster rank) publishes its partial to each CTA that needs it
      const int buf = it & 1;
      float* slot = tpart + (buf * 8 + contrib) * 128 + quad * 32 + lane;
      *slot = dot2.x + dot2.y;
      if (ES) st_cluster_f32(mapa_u32(smem_u32(slot), peer), dot2.x + dot2.y);
      __syncwarp();                                       // one release per warp covers the 32 lanes' stores (not 32 cluster fences)
      if (lane == 0) {
        mbar_arrive(&tbar[buf * 4 + quad]);
        if (ES) mbar_arrive_remote(&tbar[buf * 4 + quad], peer);
      }
      if (ES) mbar_wait_cluster(&tbar[buf * 4 + quad], (uint32_t)((it >> 1) & 1));
      else mbar_wait(&tbar[buf * 4 + quad], (uint32_t)((it >> 1) & 1));
      const float* all = tpart + buf * 8 * 128 + quad * 32 + lane;
      float t = all[0];                                   // fixed order: every warp (and both CTAs) get the same bits
#pragma unroll
      for (int c = 1; c < kContrib; ++c) t += all[c * 128];
      t_ex += clock64() - c0;
      const float c1 = ok ? -t * inv_n : 0.f;
      const float2 c1v = make_float2(c1, c1), inv2 = make_float2(inv_n, inv_n);
      // ---- pass 2: dw = acc * inv_norm - w_hat * (t * inv_norm); the w_hat boxes become the fp32 staging boxes
      uint4 wq[NG * 4];
#pragma unroll
      for (int g = 0; g < NG; ++g)
#pragma unroll
        for (int q = 0; q < 4; ++q) wq[g * 4 + q] = *reinterpret_cast<const uint4*>(wbuf + (g >> 1) * kWBox + sw128_off(lane, sub0 + (g & 1) * 4 + q));
      __syncwarp();                                       // every lane holds its w_hat row: the boxes are free
      {
        uint32_t va[32];
        auto out_group = [&](const uint32_t (&v)[32], int g) {
          uint8_t* orow = NG == 1 ? sbuf + (it & 1) * kWBox : wbuf + (g & (kNW - 1)) * kWBox;
          // the store issued two groups ago (same box) must have been read; stores are committed one group each
          if (lane == 0) {
            if (NG == 1) tma_store_wait_read<1>();
            else tma_store_wait_read<kNW - 1>();
          }
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 w8 = wq[g * 4 + q];
            const uint32_t w4[4] = {w8.x, w8.y, w8.z, w8.w};
            float2 r[4];
#pragma unroll
            for (int k = 0; k < 4; ++k)
              r[k] = __ffma2_rn(make_float2(__uint_as_float(w4[k] << 16), __uint_as_float(w4[k] & 0xffff0000u)), c1v,
                                __fmul2_rn(make_float2(__uint_as_float(v[q * 8 + 2 * k]), __uint_as_float(v[q * 8 + 2 * k + 1])), inv2));
            *reinterpret_cast<float4*>(orow + sw128_off(lane, 2 * q)) = make_float4(r[0].x, r[0].y, r[1].x, r[1].y);
            *reinterpret_cast<float4*>(orow + sw128_off(lane, 2 * q + 1)) = make_float4(r[2].x, r[2].y, r[3].x, r[3].y);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (p.accumulate) tma_reduce_add_2d(&tmap_dw, orow, e_warp + g * 32, cls0);
            else tma_store_2d(&tmap_dw, orow, e_warp + g * 32, cls0);
            tma_store_commit();
          }
        };
#pragma unroll
        for (int g = 0; g < NG; ++g) {                    // (one group in flight: the 16 w_hat registers leave no room for two)
          tmem_ld_x32(t_base + g * 32, va);
          tmem_ld_wait();
          out_group(va, g);
        }
      }
      t_p2 += clock64() - c0;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&tmem_empty[acc]);
        if (NG > 1) tma_store_wait_read<0>();             // the staging boxes are this warp's w_hat boxes: all reads done before the reload
        if (more(it + 1)) issue_w(it + 1);
      }
      __syncwarp();
      t_ep += clock64() - c0;
    }
    if (lane == 0) tma_store_wait_all();
    if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) { p.dbg[3] = t_wfull; p.dbg[4] = t_ww; p.dbg[5] = t_ep; p.dbg[6] = t_p1; p.dbg[7] = t_ex; p.dbg[8] = t_p2; }
  }
  tc_fence_before();
  if (CS > 1) cluster_sync_all(); else __syncthreads();     // peers may still multicast into / arrive on this CTA
  if (warp == kMmaWarp) tmem_dealloc<2 * EN>(tmem_base);
}

// ================================================================================================
// dw4 kernel (E = 512): the dw GEMM + normalize backward, TRANSPOSED, on a cluster of FOUR CTAs = two cta_group::2 pairs.
//   D^T[e, class] = sum_rows x_scaled[row, e] P[row, class]:   M = e, N = classes, K = rows.
//   pair h (cluster ranks 2h, 2h+1) owns e-slice h (256 of the 512 e); inside a pair CTA c supplies A = its 128 e-rows of
//   x_scaled^T and the N-half c of B = the P tile of class tile 2g + c (g = the cluster's item), and receives
//   D^T[its 128 e, all 256 classes] in TMEM (lane = e, column = class).
// Why (measured, profiles/README.md r02): every kernel here is bound by ONE per-SM resource, the 128 B/clk shared-memory /
// L1 data pipe, which TMA fills, tcgen05.mma operand reads, ld/st.shared AND every global load/store wavefront share.  In
// 128-byte slots per 4096-cycle item the e-split pair kernel above needs 3072 (fill) + 3072 (cta_group::1 operand reads)
// + 3584 (w_hat boxes, fp32 staging, TMA store) = 9728 -> 42 % of the tensor rate, which is what it measures.  Here:
//   * cta_group::2 halves the operand reads per CTA (2048 slots) and the B fill (1024 slots, 16 KB from L2 per CTA per
//     k-block);
//   * x_scaled^T, the M-side operand, is the SAME for every item: with Bt <= 512 its [512 rows x 128 e] slice (128 KB)
//     stays resident in shared memory (STAT, no fill at all); larger batches stream it (16 KB per k-block);
//   * lane = e means a warp's 32 lanes hold 32 CONSECUTIVE e of one class per register: dw leaves in full 128-byte
//     lines straight from registers (st.global, 1024 slots) and w_hat arrives the same way (64-byte lines, 1024 slots) --
//     no staging boxes, no shared-memory capacity for the epilogue, which is what makes the resident operand fit;
//   * the radial term t_j = w_hat_j . dW_hat_j is a sum over e = over lanes: a shuffle transpose-reduction per 32 x 32
//     block (warp_colsum32), then over the 4 lane quadrants (shared memory) and the 4 CTAs (DSMEM), fixed order.
//   Budget: 1024 + 2048 + ~2600 = ~5700 slots -> ~72 % (STAT), ~62 % streamed.
// Barriers: the two pairs load independently.  Both CTAs of a pair credit their TMA bytes to the leader's full barrier (the
// dx2 kernel's producer), the leader issues the MMAs and its tcgen05.commit releases the stage in both CTAs of the pair;
// the pairs of a cluster meet only in the radial-dot exchange.  (Sharing the P tile between the pairs by multicast coupled
// them through the stage barriers and measured slower: profiles/README.md r02.)
// ================================================================================================
struct Dw4Params {
  int n_rows, n_classes;
  int n_rb;                      // row blocks of the P / G scratch
  int n_tp;                      // pairs of class tiles = ceil(n_classes / 256)
  const float* inv_norm;         // [n_classes]
  const __nv_bfloat16* w_hat;    // [n_classes, 512]
  float* dw;                     // [n_classes, 512]
  int accumulate;
  long long* dbg;
};
constexpr int kDw4EpiWarps = 16;                 // warp (quad, cgp): e rows [32 quad, +32) of this CTA, classes [64 cgp, +64) of the item
constexpr int kDw4Threads = (kDw4EpiWarps + 2) * 32;
constexpr int kDw4E = 512;

template <bool STAT, int STAGES>
__global__ void __launch_bounds__(kDw4Threads, 1) dw4_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_x,
                                                             const Dw4Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kPBytes = 2 * kBoxBytes;                    // P half tile: 64 rows x 128 classes
  constexpr int kXBytes = 2 * kBoxBytes;                    // x_scaled: 64 rows x 128 e (this CTA's M rows)
  constexpr int kStageBytes = kPBytes + (STAT ? 0 : kXBytes);
  constexpr int kMaxKb = 8;                                 // STAT: n_rows <= 512
  uint8_t* smem_x = smem;                                   // STAT: [n_kb][2 boxes]
  uint8_t* smem_st = smem + (STAT ? kMaxKb * kXBytes : 0);
  float* part = reinterpret_cast<float*>(smem_st + STAGES * kStageBytes);     // [4 quadrants][256 classes]  partial dots of this CTA
  float* tsum = part + 4 * 256;                                                // [2][4 CTAs][256]            per-CTA sums, all CTAs
  float2* scal = reinterpret_cast<float2*>(tsum + 2 * 4 * 256);                // [256]                       (1/n_j, -t_j/n_j)
  uint64_t* bars = reinterpret_cast<uint64_t*>(scal + 256);
  uint64_t* full = bars;                          // [STAGES]  leader only: stage bytes of both CTAs of the pair
  uint64_t* empty = bars + STAGES;                // [STAGES]  the commit of the pair's leader
  uint64_t* tmem_full = bars + 2 * STAGES;        // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;   // [2]       leader only: epilogue warps of both CTAs
  uint64_t* tbar = bars + 2 * STAGES + 4;         // [2]       per-CTA sums of all four CTAs have landed
  uint64_t* x_full = bars + 2 * STAGES + 6;       // STAT, leader only: the resident x_scaled^T of both CTAs of the pair
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 7);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const int hs = (int)(crank >> 1), cpar = (int)(crank & 1);      // e-slice of the pair; N-half (class tile parity) inside the pair
  const bool leader = cpar == 0;
  const uint32_t leader_rank = crank & ~1u;
  const int n_clusters = gridDim.x >> 2, cid = blockIdx.x >> 2;
  const int n_kb = (p.n_rows + BK - 1) / BK;
  constexpr int kProducerWarp = kDw4EpiWarps, kMmaWarp = kDw4EpiWarps + 1;
  const uint16_t pair_mask = (uint16_t)(3u << (2 * hs));
  const int e_cta = hs * 256 + cpar * 128;                        // first e of this CTA's 128 M rows

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 2 * kDw4EpiWarps); mbar_init(&tbar[i], 4 * 8); }
    mbar_init(x_full, 1);
    fence_barrier_init();
  }
  if (warp == kProducerWarp && lane == 0) { prefetch_tmap(&tmap_g); prefetch_tmap(&tmap_x); }
  if (warp == kMmaWarp) tmem_alloc_2cta<512>(tmem_slot);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kProducerWarp) {
    if (lane == 0) {
      const uint32_t x_full_leader = mapa_u32(smem_u32(x_full), leader_rank);
      if (STAT) {
        if (leader) mbar_arrive_expect_tx(x_full, 2 * n_kb * kXBytes);
        for (int kb = 0; kb < n_kb; ++kb)
#pragma unroll
          for (int nb = 0; nb < 2; ++nb) tma_load_2d_2cta(smem_x + kb * kXBytes + nb * kBoxBytes, &tmap_x, x_full_leader, e_cta + nb * 64, kb * BK);
      }
      PipeState ps;
      for (int i = 0; i * n_clusters + cid < p.n_tp; ++i) {
        const int ct = 2 * (i * n_clusters + cid) + cpar;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait_cluster(&empty[ps.stage], ps.phase ^ 1);
          uint8_t* sp = smem_st + ps.stage * kStageBytes;
          const uint32_t full_leader = mapa_u32(smem_u32(&full[ps.stage]), leader_rank);
          if (leader) mbar_arrive_expect_tx(&full[ps.stage], 2 * kStageBytes);
#pragma unroll
          for (int hb = 0; hb < 2; ++hb)
            tma_load_2d_2cta(sp + hb * kBoxBytes, &tmap_g, full_leader, 0, ((2 * ct + hb) * p.n_rb + (kb >> 1)) * BM + (kb & 1) * 64);
          if (!STAT) {
#pragma unroll
            for (int nb = 0; nb < 2; ++nb) tma_load_2d_2cta(sp + kPBytes + nb * kBoxBytes, &tmap_x, full_leader, e_cta + nb * 64, kb * BK);
          }
          ps.advance(STAGES);
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * BM, 256, true, true);
      PipeState ps;
      long long t_we = 0, t_wf = 0, t_all = clock64();
      if (STAT) mbar_wait_cluster(x_full, 0);
      for (int it = 0; it * n_clusters + cid < p.n_tp; ++it) {
        const int acc = it & 1;
        long long c0 = clock64();
        mbar_wait_cluster(&tmem_empty[acc], (uint32_t)(((it >> 1) & 1) ^ 1));
        t_we += clock64() - c0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = 0; kb < n_kb; ++kb) {
          c0 = clock64();
          mbar_wait_cluster(&full[ps.stage], ps.phase);
          t_wf += clock64() - c0;
          tc_fence_after();
          const uint32_t p_addr = smem_u32(smem_st + ps.stage * kStageBytes);
          const uint32_t x_addr = STAT ? smem_u32(smem_x + kb * kXBytes) : p_addr + kPBytes;
#pragma unroll
          for (int kk = 0; kk < BK / 16; ++kk) {
            const uint64_t da = make_desc_sw128(x_addr + kk * 2048, kBoxBytes, 1024);     // A = x_scaled^T  (M = e, MN-major)
            const uint64_t db = make_desc_sw128(p_addr + kk * 2048, kBoxBytes, 1024);     // B = P           (N = classes, MN-major)
            umma_bf16_ss_2cta(d_tmem, da, db, idesc, (kb | kk) != 0);
          }
          umma_commit_2cta(&empty[ps.stage], pair_mask);
          ps.advance(STAGES);
        }
        umma_commit_2cta(&tmem_full[acc], pair_mask);
      }
      if (p.dbg && blockIdx.x == 0) { p.dbg[0] = t_we; p.dbg[1] = t_wf; p.dbg[2] = clock64() - t_all; }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: thread = e row, register = class
    // warp (quad, cgp): e rows [32 quad, +32) of this CTA, classes [64 cgp, +64) of the 256 of the item (tile cgp >> 1)
    const int quad = warp & 3, cgp = warp >> 2;
    const int tid = threadIdx.x;                            // < 256: also the class slot this thread sums / scales
    const int e_glob = e_cta + quad * 32 + lane;
    const uint32_t t_lane = (uint32_t)(quad * 32) << 16;
    const uint32_t tmem_leader_empty0 = mapa_u32(smem_u32(&tmem_empty[0]), leader_rank);
    const unsigned short* wbase = reinterpret_cast<const unsigned short*>(p.w_hat) + e_glob;
    unsigned t_wfull = 0, t_p1 = 0, t_ex = 0, t_p2 = 0;      // 32-bit cycle counters of CTA 0 / thread 0 (developer probe)
    for (int it = 0; it * n_clusters + cid < p.n_tp; ++it) {
      const int tp = it * n_clusters + cid;
      const int acc = it & 1, buf = it & 1;
      const int cls_w = 2 * tp * BM + cgp * 64;             // first class of this warp's 64
      // w_hat of this thread's e for its 64 classes, two bf16 per register (64-byte lines per warp and class)
      uint32_t wpk[32];
      const int n_ok = p.n_classes - cls_w;                 // classes of this group that exist (>= 64 for all but the last tiles)
      const unsigned short* wt = wbase + (int64_t)cls_w * kDw4E;
      if (n_ok >= 64) {
#pragma unroll
        for (int j = 0; j < 32; ++j) wpk[j] = (uint32_t)__ldg(wt + (2 * j) * kDw4E) | ((uint32_t)__ldg(wt + (2 * j + 1) * kDw4E) << 16);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t lo = 2 * j < n_ok ? (uint32_t)__ldg(wt + (2 * j) * kDw4E) : 0u;
          const uint32_t hi = 2 * j + 1 < n_ok ? (uint32_t)__ldg(wt + (2 * j + 1) * kDw4E) : 0u;
          wpk[j] = lo | (hi << 16);
        }
      }
      unsigned c0 = clock();
      mbar_wait(&tmem_full[acc], (uint32_t)((it >> 1) & 1));
      t_wfull += clock() - c0;
      c0 = clock();
      tc_fence_after();
      // ---- pass 1: per class, the sum over this warp's 32 e of w_hat * acc (a transpose-reduction across the lanes)
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + t_lane + acc * 256 + cgp * 64 + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const uint32_t w2 = wpk[c * 16 + (j >> 1)];
          const float2 pr = __fmul2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])),
                                       make_float2(__uint_as_float(w2 << 16), __uint_as_float(w2 & 0xffff0000u)));
          v[j] = __float_as_uint(pr.x);
          v[j + 1] = __float_as_uint(pr.y);
        }
        part[quad * 256 + cgp * 64 + c * 32 + lane] = warp_colsum32_bits(v, lane);
      }
      t_p1 += clock() - c0;
      c0 = clock();
      asm volatile("bar.sync 1, 512;" ::: "memory");
      // ---- the CTA's sum over its 128 e for class slot `tid`, published to all four CTAs (warps 0..7)
      if (tid < 256) {
        const float s4 = ((part[tid] + part[256 + tid]) + part[512 + tid]) + part[768 + tid];
        float* slot = tsum + (buf * 4 + (int)crank) * 256 + tid;
        const uint32_t slot_addr = smem_u32(slot);
#pragma unroll
        for (uint32_t r = 0; r < 4; ++r) {
          if (r == crank) *slot = s4;
          else st_cluster_f32(mapa_u32(slot_addr, r), s4);
        }
        __syncwarp();
        if (lane == 0) {
#pragma unroll
          for (uint32_t r = 0; r < 4; ++r) {
            if (r == crank) mbar_arrive(&tbar[buf]);
            else mbar_arrive_remote(&tbar[buf], r);
          }
        }
        mbar_wait_cluster(&tbar[buf], (uint32_t)((it >> 1) & 1));
        const float* ts = tsum + buf * 4 * 256 + tid;
        const float t = ((ts[0] + ts[256]) + ts[512]) + ts[768];          // fixed order: identical bits in all four CTAs
        const int cls = 2 * tp * BM + tid;
        const float inv = cls < p.n_classes ? __ldg(p.inv_norm + cls) : 0.f;
        scal[tid] = make_float2(inv, -t * inv);
      }
      asm volatile("bar.sync 1, 512;" ::: "memory");
      t_ex += clock() - c0;
      c0 = clock();
      // ---- pass 2: dw[class][e] = acc / n - w_hat (t / n): one full 128-byte line per warp and class, straight from registers
      const bool plain = n_ok >= 64 && !p.accumulate;      // the common case: no per-class predicates at all
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t v[32];
        tmem_ld_x32(tmem_base + t_lane + acc * 256 + cgp * 64 + c * 32, v);
        tmem_ld_wait();
        const float4* sc4 = reinterpret_cast<const float4*>(scal + cgp * 64 + c * 32);
        float* out = p.dw + (int64_t)(cls_w + c * 32) * kDw4E + e_glob;
        if (plain) {
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float4 sc = sc4[j >> 1];                   // (1/n_j, -t_j/n_j, 1/n_j+1, -t_j+1/n_j+1): same address in every lane
            const uint32_t w2 = wpk[c * 16 + (j >> 1)];
            const float2 r = __ffma2_rn(make_float2(__uint_as_float(w2 << 16), __uint_as_float(w2 & 0xffff0000u)), make_float2(sc.y, sc.w),
                                        __fmul2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), make_float2(sc.x, sc.z)));
            out[j * kDw4E] = r.x;
            out[(j + 1) * kDw4E] = r.y;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float4 sc = sc4[j >> 1];
            const uint32_t w2 = wpk[c * 16 + (j >> 1)];
            float2 r = __ffma2_rn(make_float2(__uint_as_float(w2 << 16), __uint_as_float(w2 & 0xffff0000u)), make_float2(sc.y, sc.w),
                                  __fmul2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), make_float2(sc.x, sc.z)));
            float* d = out + j * kDw4E;
            if (p.accumulate) {
              if (c * 32 + j < n_ok) r.x += d[0];
              if (c * 32 + j + 1 < n_ok) r.y += d[kDw4E];
            }
            if (c * 32 + j < n_ok) d[0] = r.x;
            if (c * 32 + j + 1 < n_ok) d[kDw4E] = r.y;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tmem_empty[acc]);
        else mbar_arrive_cluster_addr_relaxed(tmem_leader_empty0 + acc * 8);
      }
      t_p2 += clock() - c0;
    }
    if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) { p.dbg[3] = t_wfull; p.dbg[4] = 0; p.dbg[5] = t_p1 + t_ex + t_p2; p.dbg[6] = t_p1; p.dbg[7] = t_p1 + t_ex; p.dbg[8] = t_p1 + t_ex + t_p2; }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == kMmaWarp) tmem_dealloc_2cta<512>(tmem_base);
}

// ================================================================================================
// Stored-probability backward (MODE_PROB forward): the forward kept P_ij = exp2(s2 cos_ij - a_i) (bf16, blocked
// scratch, target column zero), so   G_ij = scale_i P_ij   with   scale_i = s / (S_i Bt)   (S_i = global sum of P_i.)
// and no logits are recomputed:
//     dx_i  = scale_i  sum_j P_ij w_hat_j                      (dx kernels on P, row scale in the slab reduction)
//     dwh_j = sum_i P_ij (scale_i x_hat_i)                      (dw kernel on P^T and the pre-scaled x_hat)
//     t_j   = w_hat_j . dwh_j                                    (dw epilogue, from its accumulator)
// The target element G_iy = s (p_iy - 1) slope / Bt is formed in fp32 from the row statistics and written into the
// scratch as v = (p_iy - 1) slope S_i by prob_prep_kernel (bf16 rounding of the difference, not of p_iy).
// ================================================================================================
constexpr float kProbHeadroom = 58.f;      // log2 units: P <= 2^58, so a row sum over < 2^30 classes stays below 2^88

// a_i = s2 |x_hat_i| (1 + 2^-7) - headroom.  |x.w_hat| <= |x| |w_hat| and bf16 rounding leaves |w_hat| <= 1 + 2^-8.
// range guard (flag = pinned host or device memory, may be null): flag[0] = 1 when s |x_i| of some row leaves the exponent
// window of the stored-probability path (or is not finite), flag[1] = 1 when a row sum came out 0 / non-finite in the
// backward.  Sticky plain stores; the host polls them without synchronising (PartialFC switches to the recomputing backward).
__global__ void __launch_bounds__(256) row_bound_kernel(const __nv_bfloat16* __restrict__ x, int64_t n_rows, int emb, float s2,
                                                        float* __restrict__ bound, int* __restrict__ range_flag, float limit_log2) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const uint32_t* p = reinterpret_cast<const uint32_t*>(x + r * emb);
  float ss = 0.f;
  for (int c = lane; c < emb / 2; c += 32) {
    const uint32_t u = p[c];
    const float a = __uint_as_float(u << 16), b = __uint_as_float(u & 0xffff0000u);
    ss = fmaf(a, a, fmaf(b, b, ss));
  }
  ss = warp_sum(ss);
  if (lane == 0) {
    bound[r] = s2 * sqrtf(ss) * 1.0078125f - kProbHeadroom;
    if (range_flag && !(s2 * sqrtf(ss) <= limit_log2)) *reinterpret_cast<volatile int*>(range_flag) = 1;
  }
}

// One warp per row: x_scaled_i = bf16(x_hat_i * scale_i), row_scale_i, and the target element of the row (if this
// shard owns it): scratch[i, y] = bf16((p_iy - 1) slope S_i).  With the target in place the dx / dw GEMMs and the radial
// term the dw epilogue takes from its accumulator need no further special case.
__global__ void __launch_bounds__(256) prob_prep_kernel(const __nv_bfloat16* __restrict__ x, const int64_t* __restrict__ label,
                                                        const float* __restrict__ row_sum, const float* __restrict__ row_bound,
                                                        const float* __restrict__ target_cos, int64_t n_rows, int emb, int n_rb, int64_t n_classes,
                                                        float s, float m, int margin_kind, float g_scale, __nv_bfloat16* __restrict__ x_scaled,
                                                        float* __restrict__ row_scale, __nv_bfloat16* __restrict__ scratch, int* __restrict__ range_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const float S = row_sum[r];
  const float sc = (S > 0.f && S < INFINITY) ? g_scale / S : 0.f;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(x + r * emb);
  uint32_t* dst = reinterpret_cast<uint32_t*>(x_scaled + r * emb);
  for (int c = lane; c < emb / 2; c += 32) {
    const uint32_t u = src[c];
    dst[c] = pack_bf16x2(__uint_as_float(u << 16) * sc, __uint_as_float(u & 0xffff0000u) * sc);
  }
  if (lane == 0) {
    row_scale[r] = sc;
    if (range_flag && sc == 0.f) *reinterpret_cast<volatile int*>(range_flag + 1) = 1;
    const int64_t y = label[r];
    if (y >= 0 && y < n_classes) {
      const float c = target_cos[r];
      const float pS = exp2f(s * kLog2e * margin_cos(c, m, margin_kind) - row_bound[r]);       // p_iy S_i
      const float v = (pS - S) * margin_slope(c, m, margin_kind);
      scratch[(((y >> 6) * n_rb + (r >> 7)) * BM + (r & 127)) * 64 + (y & 63)] = __float2bfloat16_rn(v);
    }
  }
}

// dx = row_scale_i * sum of the split-K slabs
__global__ void reduce_dx_scaled_kernel(const float4* __restrict__ part, int ksplit, int64_t n_vec, int vec_per_row, const float* __restrict__ row_scale,
                                        float4* __restrict__ dx) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec; i += (int64_t)gridDim.x * blockDim.x) {
    float4 a = part[i];
    for (int k = 1; k < ksplit; ++k) {
      const float4 b = part[(int64_t)k * n_vec + i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    const float sc = row_scale[i / vec_per_row];
    dx[i] = make_float4(a.x * sc, a.y * sc, a.z * sc, a.w * sc);
  }
}

}  // namespace tc

// ================================================================================================
// host launchers
// ================================================================================================
using namespace tc;

static int g_fwd_bn = 128;       // class-tile width of the logits kernels (128 or 256)

static int fwd_grid(int64_t n_rows, int64_t n_classes, int bn) {
  const int64_t n_rb = (n_rows + BM - 1) / BM, n_ct = (n_classes + bn - 1) / bn;
  const int64_t tiles = n_rb * n_ct;
  const int sms = sm_count();
  return (int)(tiles < sms ? tiles : sms);
}

template <int BN, int STAGES, int MODE>
static int launch_logits(const CUtensorMap& tx, const CUtensorMap& tw, const LogitsParams& p, int grid, cudaStream_t st) {
  const size_t smem = (size_t)(p.emb / BK) * kChunkBytes + (size_t)STAGES * BN * BK * 2 + 1024 + 256;
  auto kern = logits_kernel<BN, STAGES, MODE>;
  PFC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kLogitsThreads, smem, st>>>(tx, tw, p);
  PFC_LAUNCH_CHECK();
  return 0;
}

static int g_logits_pair = 1;      // 1: CTA-pair (cta_group::2) logits kernels, 0: single-CTA kernels

template <int STAGES, int MODE, bool NORM = false>
static int launch_logits2(const CUtensorMap& tx, const CUtensorMap& tw, const CUtensorMap& tg, const LogitsParams& p, int grid, cudaStream_t st) {
  const size_t smem = (size_t)(p.emb / BK) * kChunkBytes + (size_t)STAGES * 128 * BK * 2 + (MODE != MODE_STATS ? kLogitsEpiWarps * 4096 : 0) + 1024 + 256;
  auto kern = logits2_kernel<STAGES, MODE, NORM>;
  PFC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kLogitsThreads + (NORM ? norm_warps(MODE) * 32 : 0));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PFC_CUDA(cudaLaunchKernelEx(&cfg, kern, tx, tw, tg, p));
  PFC_LAUNCH_CHECK();
  return 0;
}

// grid of the pair kernels: one pair per two SMs, never more pairs than work items
static int pair_grid(int64_t n_rows, int64_t n_classes) {
  const int64_t n_rp = ((n_rows + BM - 1) / BM + 1) / 2, n_ct = (n_classes + 255) / 256;
  const int64_t items = n_rp * n_ct;
  const int64_t pairs = sm_count() / 2;
  return (int)(2 * (items < pairs ? items : pairs));
}

template <int MODE>
static int dispatch_logits(const CUtensorMap& tx, const CUtensorMap& tw, const LogitsParams& p, int bn, int grid, cudaStream_t st) {
  const int n_kb = p.emb / BK;
  if (bn == 256) {
    if (n_kb <= 4) return launch_logits<256, 4, MODE>(tx, tw, p, grid, st);
    return launch_logits<256, 3, MODE>(tx, tw, p, grid, st);
  }
  if (n_kb <= 4) return launch_logits<128, 8, MODE>(tx, tw, p, grid, st);
  return launch_logits<128, 5, MODE>(tx, tw, p, grid, st);
}

static bool tensor_emb_ok(int emb) { return emb == 64 || emb == 128 || emb == 256 || emb == 512; }

int tc_fwd_num_partials(int64_t n_rows, int64_t n_classes) {
  return 2 * (g_logits_pair ? pair_grid(n_rows, n_classes) : fwd_grid(n_rows, n_classes, g_fwd_bn));
}

int tc_fwd_stats(const void* x, const void* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind,
                 float* part_max, float* part_sum, float* target_logit, cudaStream_t st) {
  PFC_REQUIRE(tensor_emb_ok(emb), PFC_E_SHAPE, "tensor path supports emb in {64,128,256,512}, got %d (use PFC_PATH_CHECK)", emb);
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && n_classes < (1ll << 30) && n_rows < (1ll << 24), PFC_E_SHAPE, "pfc_fwd_stats: shape out of range");
  const int bn = g_logits_pair ? 256 : g_fwd_bn;
  CUtensorMap tx, tw;
  if (int rc = make_tmap_bf16_2d(&tx, x, n_rows, emb, emb, BM)) return rc;
  if (int rc = make_tmap_bf16_2d(&tw, w_hat, n_classes, emb, emb, g_logits_pair ? 128 : bn)) return rc;
  LogitsParams p{};
  p.label = label; p.n_rows = (int)n_rows; p.n_classes = (int)n_classes; p.class_base = 0; p.emb = emb;
  p.n_rb = (int)((n_rows + BM - 1) / BM); p.n_ct = (int)((n_classes + bn - 1) / bn);
  p.s = s; p.m = m; p.margin_kind = margin_kind; p.part_max = part_max; p.part_sum = part_sum; p.target_logit = target_logit;
  const int grid = g_logits_pair ? pair_grid(n_rows, n_classes) : fwd_grid(n_rows, n_classes, bn);
  PFC_CUDA(cudaMemsetAsync(part_sum, 0, sizeof(float) * (size_t)grid * 2 * n_rows, st));
  PFC_CUDA(cudaMemsetAsync(target_logit, 0, sizeof(float) * (size_t)n_rows, st));
  prof_begin(PH_FWD, st);
  int rc = g_logits_pair ? launch_logits2<4, MODE_STATS>(tx, tw, tw, p, grid, st) : dispatch_logits<MODE_STATS>(tx, tw, p, bn, grid, st);
  prof_end(PH_FWD, st);
  return rc;
}

// ---- backward chunking -------------------------------------------------------------------------
// The class axis is cut into chunks.  Per chunk: G kernel (recompute logits -> G scratch), then dx and dw consume the
// scratch.  With more than two chunks the three kernels run as three concurrent chains on disjoint SM subsets
// (G on the caller's stream, dx and dw on side streams, a ring of G buffers in between): the G kernel is bound by its
// epilogue issue slots, dx by L2 delivery and dw by the HBM write of dw, so they overlap well, and a chunk is consumed
// while it is still L2-resident.
struct BwdPlan {
  int64_t chunk;        // classes per chunk (multiple of 256)
  int64_t ldg;          // row pitch of the G scratch (elements)
  int n_chunks, ring;   // ring = G buffers
  bool pipelined;
  int sm_g, sm_dx, sm_dw;   // SMs (CTAs) per chain
  int ksplit, n_eh, dx_bn;
  bool dx_pair;             // CTA-pair dx kernel (row blocks a multiple of 4; the last one may be partial)
  size_t g_bytes, g_buf_bytes, dxp_bytes;
};

static int64_t g_chunk_budget_mb;                   // 0 = default
static int g_dx_pair = 1;                           // 1: CTA-pair dx kernel when the row count allows it
static int g_pipe = 1;                              // 1 = concurrent chains (see pfc_set_pipeline)
static int g_split[3] = {148, 48, 100};             // SMs for the G / dx / dw chains in pipelined mode
static int g_ring = 1;                              // G buffers; 1 = G alone on every SM, then dx || dw sweep the chunk in step

static BwdPlan make_bwd_plan(int64_t n_rows, int64_t n_classes, int emb) {
  BwdPlan pl{};
  const int64_t n_rb = (n_rows + BM - 1) / BM;
  const int64_t c_pad = (n_classes + 255) / 256 * 256;
  const int64_t row_bytes = n_rb * BM * 2;           // bytes of G scratch per class
  int64_t budget_seq = 512ll << 20, budget_pipe = 32ll << 20;
  if (g_chunk_budget_mb > 0) budget_seq = budget_pipe = g_chunk_budget_mb << 20;
  auto chunk_for = [&](int64_t budget) {
    int64_t c = budget / row_bytes / 256 * 256;
    if (c < 256) c = 256;
    if (c > c_pad) c = c_pad;
    return c;
  };
  int64_t chunk = chunk_for(budget_pipe);
  int64_t n_chunks = (n_classes + chunk - 1) / chunk;
  // ring == 1: G runs alone (it may use every SM), then dx and dw of the chunk run side by side on disjoint SMs
  const bool fits = g_ring == 1 ? (g_split[1] + g_split[2] <= sm_count() && g_split[0] <= sm_count())
                                : (g_split[0] + g_split[1] + g_split[2] <= sm_count());
  pl.pipelined = g_pipe && fits && (g_ring == 1 || n_chunks >= 4);
  if (pl.pipelined && g_ring == 1) budget_pipe = budget_seq;
  chunk = chunk_for(budget_pipe);
  n_chunks = (n_classes + chunk - 1) / chunk;
  if (!pl.pipelined) {
    chunk = chunk_for(budget_seq);
    n_chunks = (n_classes + chunk - 1) / chunk;
  }
  pl.chunk = chunk;
  pl.ldg = chunk;
  pl.n_chunks = (int)n_chunks;
  pl.ring = pl.pipelined ? g_ring : 1;
  pl.dx_bn = emb < 256 ? emb : 256;
  pl.n_eh = emb / pl.dx_bn;
  const int sms = sm_count();
  pl.sm_g = pl.pipelined ? g_split[0] : sms;
  pl.sm_dx = pl.pipelined ? g_split[1] : sms;
  pl.sm_dw = pl.pipelined ? g_split[2] : sms;
  pl.dx_pair = g_dx_pair && g_logits_pair && emb >= 256 && n_rb % 4 == 0;
  int64_t units = pl.dx_pair ? (n_rb / 4) * pl.n_eh * 2 : n_rb * pl.n_eh;      // CTAs per k-split
  int64_t ks = pl.sm_dx / units;
  if (ks < 1) ks = 1;
  const int64_t min_kb = ((chunk < n_classes ? chunk : n_classes) + BK - 1) / BK;
  if (ks > min_kb) ks = min_kb;
  if (ks > 64) ks = 64;
  pl.ksplit = (int)ks;
  pl.g_buf_bytes = (size_t)n_rb * BM * pl.ldg * 2;      // blocked: [ldg / 64][n_rb][128][64] bf16
  pl.g_bytes = pl.g_buf_bytes * pl.ring;
  pl.dxp_bytes = ((size_t)pl.ksplit * n_rows * emb * 4 + 1023) / 1024 * 1024;
  return pl;
}

size_t tc_bwd_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb) {
  BwdPlan pl = make_bwd_plan(n_rows, n_classes, emb);
  return pl.g_bytes + pl.dxp_bytes + 1024;
}

static int* g_range_flag[64];                       // per device: range-guard flag of the stored-probability path (tc_set_range_flag)
static float g_range_limit_nats = 80.f;
static int* range_flag_of_current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  return g_range_flag[dev];
}
static int g_prefetch[3] = {0, 0, 0};               // TMA L2 prefetch knobs: logits (0/1), dx (k-block distance), dw (0/1); measured slower, off
static long long* g_dbg = nullptr;                   // developer instrumentation buffer (device), see pfc_set_debug_buffer
static int g_dx_cluster = 2, g_dw_cluster = 2;      // cluster sizes (1, 2 or 4); tuning knobs

template <class Kern, class... Args>
static int launch_cluster_threads(Kern kern, int threads, int grid, int cs, size_t smem, cudaStream_t st, Args... args) {
  PFC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  PFC_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  PFC_LAUNCH_CHECK();
  return 0;
}
template <class Kern, class... Args>
static int launch_cluster(Kern kern, int grid, int cs, size_t smem, cudaStream_t st, Args... args) {
  return launch_cluster_threads(kern, kThreads, grid, cs, smem, st, args...);
}

template <int BN, int CS>
static int launch_dx_cs(const CUtensorMap& tg, const CUtensorMap& tw, const DxParams& p, int grid, cudaStream_t st) {
  constexpr int STAGES = BN == 256 ? 4 : 6;
  const size_t smem = (size_t)STAGES * (kChunkBytes + (BN / 64) * kBoxBytes) + 1024 + 256;
  return launch_cluster(dx_kernel<BN, STAGES, CS>, grid, CS, smem, st, tg, tw, p);
}

static int launch_dx2(const CUtensorMap& tg, const CUtensorMap& tw, const DxParams& p, int grid, cudaStream_t st) {
  constexpr int STAGES = 4;
  const size_t smem = (size_t)STAGES * (2 * kChunkBytes + 2 * kBoxBytes) + 1024 + 256;
  return launch_cluster(dx2_kernel<STAGES>, grid, 2, smem, st, tg, tw, p);
}

template <int BN>
static int launch_dx(const CUtensorMap& tg, const CUtensorMap& tw, const DxParams& p, int grid, int cs, cudaStream_t st) {
  if constexpr (BN == 256) {
    if (cs == 4) return launch_dx_cs<BN, 4>(tg, tw, p, grid, st);
    if (cs == 2) return launch_dx_cs<BN, 2>(tg, tw, p, grid, st);
  } else if constexpr (BN == 128) {
    if (cs == 2) return launch_dx_cs<BN, 2>(tg, tw, p, grid, st);
  }
  return launch_dx_cs<BN, 1>(tg, tw, p, grid, st);
}

template <int EMB, int CS>
static int launch_dw_cs(const CUtensorMap& tg, const CUtensorMap& tx, const CUtensorMap& twh, const CUtensorMap& tdw, const DwParams& p, int grid,
                        cudaStream_t st) {
  constexpr int EN = EMB < 256 ? EMB : 256;
  constexpr int kStage = 2 * kBoxBytes + (EN / 64) * kBoxBytes;
  constexpr int NG = EN / (kDwEpiWarps / 4) / 32;                // 32-column groups per epilogue warp
  constexpr int kEpi = kDwEpiWarps * ((NG + 1) / 2) * 4096 + (NG == 1 ? kDwEpiWarps * 2 * 4096 : 0);   // w_hat boxes (= staging) [+ staging]
  constexpr int kFixed = 8192 /* partial dots */ + 1024 /* alignment */ + 512 /* barriers */;
  constexpr int STAGES = (232448 - kFixed - kEpi) / kStage > 8 ? 8 : (232448 - kFixed - kEpi) / kStage;
  static_assert(STAGES >= 2, "dw kernel smem budget");
  const size_t smem = (size_t)STAGES * kStage + kEpi + kFixed;
  return launch_cluster_threads(dw_kernel<EMB, STAGES, CS>, kDwThreads, grid, CS, smem, st, tg, tx, twh, tdw, p);
}

template <int EMB>
static int launch_dw(const CUtensorMap& tg, const CUtensorMap& tx, const CUtensorMap& twh, const CUtensorMap& tdw, const DwParams& p, int n_ct,
                     int cs, int sms, cudaStream_t st) {
  if (EMB < 128) cs = 1;
  if (EMB == 128 && cs > 2) cs = 2;
  if (EMB > 256) cs = 2;                                   // e-split pair: one class tile per cluster, e-slice = cluster rank
  const int n_groups = EMB > 256 ? n_ct : (n_ct + cs - 1) / cs;
  int max_clusters = sms / cs;
  if (cs == 4) max_clusters = max_clusters * 9 / 10;     // GPCs of 18 SMs strand 2 SMs per GPC with 4-CTA clusters
  if (max_clusters < 1) max_clusters = 1;
  const int clusters = n_groups < max_clusters ? n_groups : max_clusters;
  const int grid = clusters * cs;
  if constexpr (EMB > 256) {
    return launch_dw_cs<EMB, 2>(tg, tx, twh, tdw, p, grid, st);
  } else {
    if constexpr (EMB >= 128) {
      if (cs == 4) { if constexpr (EMB >= 256) return launch_dw_cs<EMB, 4>(tg, tx, twh, tdw, p, grid, st); }
      if (cs == 2) return launch_dw_cs<EMB, 2>(tg, tx, twh, tdw, p, grid, st);
    }
    return launch_dw_cs<EMB, 1>(tg, tx, twh, tdw, p, grid, st);
  }
}

// dw kernel choice for E = 512 (pfc_set_dw4):  -1 (default) automatic: the 4-CTA-cluster transposed kernel from 2048
// gathered rows on -- there its shared-memory-pipe savings in the mainloop win (measured r02i: 0.72 vs 0.85 ms at
// Bt = 4096) --, the e-split pair kernel below that, where dw4's longer epilogue chain is not yet amortised by the K loop
// (1.73 vs 1.02 ms at Bt = 512);  0: never;  1: always.
static int g_dw4 = -1;
static bool dw4_chosen(int64_t n_rows, int emb) {
  if (emb != 512 || g_dw4 == 0) return false;
  return g_dw4 > 0 || n_rows >= 2048;
}
template <bool STAT, int STAGES>
static size_t dw4_smem_bytes() {
  return (size_t)(STAT ? 8 * 2 * kBoxBytes : 0) + (size_t)STAGES * (2 * kBoxBytes + (STAT ? 0 : 2 * kBoxBytes)) + 4 * 256 * 4 /* part */ +
         2 * 4 * 256 * 4 /* tsum */ + 256 * 8 /* scal */ + 512 /* barriers */ + 1024 /* alignment */;
}
constexpr int kDw4StagesStat = 5, kDw4StagesStream = 6;
static bool dw4_stationary(int64_t n_rows) { return n_rows <= 512; }
// clusters that can be resident at once (GPC packing of 4-CTA clusters leaves a few SMs unused); cached per variant
static int dw4_resident_clusters(bool stat) {
  static int cached[2] = {0, 0};
  if (cached[stat]) return cached[stat];
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(4 * 64);
  cfg.blockDim = dim3(kDw4Threads);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 4; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  cudaError_t e;
  if (stat) {
    cfg.dynamicSmemBytes = dw4_smem_bytes<true, kDw4StagesStat>();
    cudaFuncSetAttribute(dw4_kernel<true, kDw4StagesStat>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.dynamicSmemBytes);
    e = cudaOccupancyMaxActiveClusters(&n, dw4_kernel<true, kDw4StagesStat>, &cfg);
  } else {
    cfg.dynamicSmemBytes = dw4_smem_bytes<false, kDw4StagesStream>();
    cudaFuncSetAttribute(dw4_kernel<false, kDw4StagesStream>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.dynamicSmemBytes);
    e = cudaOccupancyMaxActiveClusters(&n, dw4_kernel<false, kDw4StagesStream>, &cfg);
  }
  if (e != cudaSuccess || n <= 0) { (void)cudaGetLastError(); n = sm_count() / 4 * 9 / 10; }
  cached[stat] = n;
  return n;
}

static int launch_dw4(const CUtensorMap& tg, const CUtensorMap& tx, const Dw4Params& p, int sms, cudaStream_t st) {
  const bool stat = dw4_stationary(p.n_rows);
  int clusters = sms / 4;
  const int cap = dw4_resident_clusters(stat);
  if (clusters > cap) clusters = cap;
  if (clusters > p.n_tp) clusters = p.n_tp;
  if (clusters < 1) clusters = 1;
  if (stat) return launch_cluster_threads(dw4_kernel<true, kDw4StagesStat>, kDw4Threads, clusters * 4, 4, dw4_smem_bytes<true, kDw4StagesStat>(), st, tg, tx, p);
  return launch_cluster_threads(dw4_kernel<false, kDw4StagesStream>, kDw4Threads, clusters * 4, 4, dw4_smem_bytes<false, kDw4StagesStream>(), st, tg, tx, p);
}

// side streams of the pipelined backward (per device)
static cudaStream_t g_side_stream[64][2];
static int side_streams(cudaStream_t* sx, cudaStream_t* sw) {
  int dev = 0;
  PFC_CUDA(cudaGetDevice(&dev));
  PFC_REQUIRE(dev >= 0 && dev < 64, PFC_E_ARG, "device index out of range");
  for (int i = 0; i < 2; ++i)
    if (!g_side_stream[dev][i]) PFC_CUDA(cudaStreamCreateWithFlags(&g_side_stream[dev][i], cudaStreamNonBlocking));
  *sx = g_side_stream[dev][0];
  *sw = g_side_stream[dev][1];
  return 0;
}

struct EventPool {          // edge markers of one enqueue; destroying a recorded event is deferred by the runtime
  std::vector<cudaEvent_t> ev;
  ~EventPool() { for (auto e : ev) cudaEventDestroy(e); }
  cudaEvent_t get() {
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    ev.push_back(e);
    return e;
  }
};
#define PFC_EDGE(from_stream, to_stream)                                  \
  do {                                                                    \
    cudaEvent_t edge_ev = pool.get();                                     \
    PFC_REQUIRE(edge_ev != nullptr, PFC_E_ARG, "cudaEventCreate failed"); \
    PFC_CUDA(cudaEventRecord(edge_ev, (from_stream)));                    \
    PFC_CUDA(cudaStreamWaitEvent((to_stream), edge_ev, 0));               \
  } while (0)

static int tc_bwd_enqueue(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_max, const float* row_sum,
                          int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
                          void* workspace, size_t workspace_bytes, cudaStream_t st) {
  PFC_REQUIRE(tensor_emb_ok(emb), PFC_E_SHAPE, "tensor path supports emb in {64,128,256,512}, got %d (use PFC_PATH_CHECK)", emb);
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && n_classes < (1ll << 30) && n_rows < (1ll << 24), PFC_E_SHAPE, "pfc_bwd: shape out of range");
  const BwdPlan pl = make_bwd_plan(n_rows, n_classes, emb);
  PFC_REQUIRE(workspace_bytes >= pl.g_bytes + pl.dxp_bytes, PFC_E_WORKSPACE, "pfc_bwd: workspace too small (%zu < %zu)",
              workspace_bytes, pl.g_bytes + pl.dxp_bytes);
  PFC_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, PFC_E_ARG, "pfc_bwd: workspace must be 1024-byte aligned");
  char* g_base = reinterpret_cast<char*>(workspace);
  float* dx_part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + pl.g_bytes);
  const auto* wh = reinterpret_cast<const __nv_bfloat16*>(w_hat);
  const int bn = g_logits_pair ? 256 : g_fwd_bn;
  const int n_rb = (int)((n_rows + BM - 1) / BM);
  CUtensorMap tx_k, tx_mn;
  if (int rc = make_tmap_bf16_2d(&tx_k, x, n_rows, emb, emb, BM)) return rc;       // logits: A K-major [128 x 64]
  if (int rc = make_tmap_bf16_2d(&tx_mn, x, n_rows, emb, emb, 64)) return rc;      // dw: B MN-major boxes [64 rows x 64 e]

  // chains: G on the caller's stream, dx and dw on side streams when pipelined
  cudaStream_t sG = st, sX = st, sW = st;
  EventPool pool;
  if (pl.pipelined) {
    if (int rc = side_streams(&sX, &sW)) return rc;
    PFC_EDGE(st, sX);
    PFC_EDGE(st, sW);
  }
  std::vector<cudaEvent_t> done_x(pl.n_chunks, nullptr), done_w(pl.n_chunks, nullptr);

  int chunk_idx = 0;
  for (int64_t c0 = 0; c0 < n_classes; c0 += pl.chunk, ++chunk_idx) {
    const int64_t cc = (n_classes - c0 < pl.chunk) ? n_classes - c0 : pl.chunk;
    auto* g = reinterpret_cast<__nv_bfloat16*>(g_base + (size_t)(chunk_idx % pl.ring) * pl.g_buf_bytes);
    // (1) G chunk
    if (pl.pipelined && chunk_idx >= pl.ring) {          // the ring slot is free once its consumers are done
      PFC_CUDA(cudaStreamWaitEvent(sG, done_x[chunk_idx - pl.ring], 0));
      PFC_CUDA(cudaStreamWaitEvent(sG, done_w[chunk_idx - pl.ring], 0));
    }
    CUtensorMap tw_k;
    if (int rc = make_tmap_bf16_2d(&tw_k, wh + c0 * emb, cc, emb, emb, g_logits_pair ? 128 : bn)) return rc;
    LogitsParams lp{};
    lp.label = label; lp.n_rows = (int)n_rows; lp.n_classes = (int)cc; lp.class_base = (int)c0; lp.emb = emb;
    lp.n_rb = n_rb; lp.n_ct = (int)((cc + bn - 1) / bn); lp.s = s; lp.m = m; lp.margin_kind = margin_kind;
    lp.row_max = row_max; lp.row_sum = row_sum; lp.g = g; lp.ldg = pl.ldg; lp.g_scale = s * inv_total_batch; lp.prefetch = g_prefetch[0];
    const uint64_t g_rows = (uint64_t)(pl.ldg / 64) * n_rb * BM;                              // rows of the blocked scratch viewed as [g_rows, 64]
    prof_begin(PH_GRAD, sG);
    if (g_logits_pair) {
      CUtensorMap tg_st;
      if (int rc = make_tmap_bf16_2d(&tg_st, g, g_rows, 64, 64, 32)) return rc;                // epilogue store boxes [32 rows x 64 classes]
      int grid = pair_grid(n_rows, cc);
      if (grid > pl.sm_g / 2 * 2) grid = pl.sm_g / 2 * 2;
      if (int rc = launch_logits2<4, MODE_GRAD>(tx_k, tw_k, tg_st, lp, grid, sG)) return rc;
    } else {
      int grid = fwd_grid(n_rows, cc, bn);
      if (grid > pl.sm_g) grid = pl.sm_g;
      if (int rc = dispatch_logits<MODE_GRAD>(tx_k, tw_k, lp, bn, grid, sG)) return rc;
    }
    prof_end(PH_GRAD, sG);
    if (pl.pipelined) {
      PFC_EDGE(sG, sX);
      PFC_CUDA(cudaStreamWaitEvent(sW, pool.ev.back(), 0));
    }
    // (2) dx partial slabs
    CUtensorMap tg_k, tw_mn, tg_mn;
    if (int rc = make_tmap_bf16_2d(&tg_k, g, g_rows, 64, 64, BM)) return rc;                  // A K-major [128 rows x 64 classes] = one block
    if (int rc = make_tmap_bf16_2d(&tw_mn, wh + c0 * emb, cc, emb, emb, 64)) return rc;     // B MN-major boxes [64 classes x 64 e]
    DxParams dp{};
    dp.n_rows = (int)n_rows; dp.n_classes = (int)cc; dp.emb = emb; dp.n_rb = n_rb; dp.n_eh = pl.n_eh; dp.ksplit = pl.ksplit;
    dp.dx_part = dx_part; dp.accumulate = chunk_idx > 0; dp.prefetch = g_prefetch[1]; dp.strided = pl.pipelined ? 1 : 0;
    int dcs = g_dx_cluster;
    if (pl.dx_bn < 128) dcs = 1;
    if (pl.dx_bn == 128 && dcs > 2) dcs = 2;
    const int n_rbg = (n_rb + dcs - 1) / dcs;
    const int dgrid = n_rbg * dcs * pl.n_eh * pl.ksplit;
    int rc = 0;
    prof_begin(PH_DX, sX);
    if (pl.dx_pair) rc = launch_dx2(tg_k, tw_mn, dp, (n_rb / 4) * pl.n_eh * pl.ksplit * 2, sX);
    else switch (pl.dx_bn) {
      case 256: rc = launch_dx<256>(tg_k, tw_mn, dp, dgrid, dcs, sX); break;
      case 128: rc = launch_dx<128>(tg_k, tw_mn, dp, dgrid, dcs, sX); break;
      default: rc = launch_dx<64>(tg_k, tw_mn, dp, dgrid, dcs, sX); break;
    }
    if (rc) return rc;
    prof_end(PH_DX, sX);
    if (pl.pipelined) {
      done_x[chunk_idx] = pool.get();
      PFC_REQUIRE(done_x[chunk_idx] != nullptr, PFC_E_ARG, "cudaEventCreate failed");
      PFC_CUDA(cudaEventRecord(done_x[chunk_idx], sX));
    }
    // (3) dw chunk
    if (int rc2 = make_tmap_bf16_2d(&tg_mn, g, g_rows, 64, 64, 64)) return rc2;              // A MN-major boxes [64 rows x 64 classes] = half a block
    DwParams wp{};
    wp.n_rows = (int)n_rows; wp.n_classes = (int)cc; wp.emb = emb; wp.n_ct = (int)((cc + BM - 1) / BM); wp.n_rb = n_rb;
    wp.inv_norm = inv_norm + c0; wp.accumulate = accumulate_dw; wp.dbg = g_dbg; wp.prefetch = g_prefetch[2];
    CUtensorMap twh_e, tdw_e;
    if (int rc3 = make_tmap_bf16_2d(&twh_e, wh + c0 * emb, cc, emb, emb, 32)) return rc3;      // epilogue: per-warp [32 classes x 64 e]
    if (int rc3 = make_tmap_f32_2d(&tdw_e, dw + c0 * emb, cc, emb, emb, 32)) return rc3;       // epilogue: per-warp [32 classes x 32 e] fp32
    prof_begin(PH_DW, sW);
    switch (emb) {
      case 512: rc = launch_dw<512>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
      case 256: rc = launch_dw<256>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
      case 128: rc = launch_dw<128>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
      default: rc = launch_dw<64>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
    }
    if (rc) return rc;
    prof_end(PH_DW, sW);
    if (pl.pipelined) {
      done_w[chunk_idx] = pool.get();
      PFC_REQUIRE(done_w[chunk_idx] != nullptr, PFC_E_ARG, "cudaEventCreate failed");
      PFC_CUDA(cudaEventRecord(done_w[chunk_idx], sW));
    }
  }
  if (pl.pipelined) {                                   // join: both side chains are in order, their last markers suffice
    PFC_CUDA(cudaStreamWaitEvent(st, done_x[pl.n_chunks - 1], 0));
    PFC_CUDA(cudaStreamWaitEvent(st, done_w[pl.n_chunks - 1], 0));
  }
  const int64_t n_vec = n_rows * emb / 4;
  int64_t blocks = (n_vec + 255) / 256;
  if (blocks > (int64_t)sm_count() * 4) blocks = (int64_t)sm_count() * 4;
  reduce_dx_kernel<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(dx_part), pl.ksplit, n_vec, reinterpret_cast<float4*>(dx));
  PFC_LAUNCH_CHECK();
  return 0;
}

// ---- step graphs -------------------------------------------------------------------------------
// The forward and the backward are fixed launch sequences for a given argument set.  Each is captured once into a CUDA
// graph on a library-owned stream and replayed on the caller's stream: one submission per phase instead of ~100
// launches, tensor-map encodes and attribute calls, and the concurrent branches (normalise || logits, dx || dw) become
// graph branches.  Entries are keyed on every argument and tuning knob; another pointer set captures another graph (LRU).
struct GraphEntry {
  unsigned char key[384];
  size_t key_len = 0;
  cudaGraphExec_t exec = nullptr;
  long long launches = 0;
  uint64_t stamp = 0;
};
constexpr int kGraphCache = 24;
static GraphEntry g_graphs[kGraphCache];
static uint64_t g_graph_clock = 0;
static int g_use_graph = 1;
static cudaStream_t g_capture_stream[64];
static std::mutex g_graph_mutex;

struct KeyBuilder {
  unsigned char buf[384];
  size_t len = 0;
  KeyBuilder() { memset(buf, 0, sizeof(buf)); }
  bool overflow = false;      // a key that does not fit must never alias another one: the caller then launches un-captured
  template <class T> KeyBuilder& add(const T& v) {
    if (len + sizeof(T) <= sizeof(buf)) { memcpy(buf + len, &v, sizeof(T)); len += sizeof(T); }
    else overflow = true;
    return *this;
  }
};

static bool graph_eligible(cudaStream_t st) {
  if (!g_use_graph || prof_enabled() || g_dbg != nullptr) return false;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread) (void)cudaStreamIsCapturing(st, &cap);
  return cap == cudaStreamCaptureStatusNone;
}

template <class Enqueue>
static int run_cached_graph(const KeyBuilder& kb, cudaStream_t st, Enqueue enqueue) {
  std::lock_guard<std::mutex> lock(g_graph_mutex);
  int device = 0;
  PFC_CUDA(cudaGetDevice(&device));
  PFC_REQUIRE(device >= 0 && device < 64, PFC_E_ARG, "device index out of range");
  GraphEntry* slot = nullptr;
  for (auto& e : g_graphs)
    if (e.exec && e.key_len == kb.len && memcmp(e.key, kb.buf, kb.len) == 0) { slot = &e; break; }
  if (!slot) {
    slot = &g_graphs[0];
    for (auto& e : g_graphs) {
      if (!e.exec) { slot = &e; break; }
      if (e.stamp < slot->stamp) slot = &e;
    }
    if (slot->exec) { cudaGraphExecDestroy(slot->exec); slot->exec = nullptr; }
    cudaStream_t& cs = g_capture_stream[device];
    if (!cs) PFC_CUDA(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
    const long long l0 = g_launch_count;
    PFC_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue(cs);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
    slot->launches = g_launch_count - l0;
    g_launch_count = l0;
    if (rc != 0) { if (graph) cudaGraphDestroy(graph); (void)cudaGetLastError(); return rc; }
    PFC_CUDA(ce);
    const cudaError_t ie = cudaGraphInstantiate(&slot->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) { slot->exec = nullptr; PFC_CUDA(ie); }
    memcpy(slot->key, kb.buf, sizeof(kb.buf));
    slot->key_len = kb.len;
  }
  slot->stamp = ++g_graph_clock;
  PFC_CUDA(cudaGraphLaunch(slot->exec, st));
  g_launch_count += slot->launches;
  return 0;
}

int tc_bwd(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_max, const float* row_sum,
           int64_t n_rows, int64_t n_classes, int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
           void* workspace, size_t workspace_bytes, cudaStream_t st) {
  auto enqueue = [&](cudaStream_t cs) {
    return tc_bwd_enqueue(x, w_hat, inv_norm, label, row_max, row_sum, n_rows, n_classes, emb, s, m, margin_kind, inv_total_batch, dx, dw, accumulate_dw,
                          workspace, workspace_bytes, cs);
  };
  if (!graph_eligible(st)) return enqueue(st);
  KeyBuilder kb;
  kb.add(1).add(x).add(w_hat).add(inv_norm).add(label).add(row_max).add(row_sum).add(dx).add(dw).add(workspace).add(n_rows).add(n_classes)
      .add(workspace_bytes).add(emb).add(accumulate_dw).add(s).add(m).add(margin_kind).add(inv_total_batch).add(g_fwd_bn).add(g_logits_pair)
      .add(g_dx_cluster).add(g_dw_cluster).add(make_bwd_plan(n_rows, n_classes, emb).chunk).add(g_pipe).add(g_ring).add(g_split[0])
      .add(g_split[1]).add(g_split[2]).add(g_prefetch[0]).add(g_prefetch[1]).add(g_prefetch[2]).add(g_dx_pair);
  if (kb.overflow) return enqueue(st);
  return run_cached_graph(kb, st, enqueue);
}

// ---- fused forward: normalise (HBM bound) || logits + stats (tensor bound) ---------------------
// The class axis is cut into chunks; normalize(k+1) runs on a side stream while the logits kernel works on chunk k, so
// the fp32 weight read hides behind the MMAs.  The logits kernel continues its per-CTA (max, sum) slots across chunks.
int launch_normalize_rows(const float* w, const int64_t* index, int64_t n_rows, int emb, __nv_bfloat16* ob, float* of, float* inv_norm,
                          int blocks_per_sm, cudaStream_t st);
static int g_fwd_chunks = 4;
static int g_norm_blocks_per_sm = 2;

// layout of the stored-probability workspace (MODE_PROB forward -> tc_bwd_prob)
struct ProbLayout {
  int n_rb;
  int64_t c_pad;                    // classes rounded up to the 256-class pair tile
  size_t off_bound, off_tcos, off_scale, off_xs, total;      // scratch (bf16, blocked [c_pad/64][n_rb][128][64]) sits at offset 0
};
static ProbLayout prob_layout(int64_t n_rows, int64_t n_classes, int emb) {
  ProbLayout L{};
  L.n_rb = (int)((n_rows + BM - 1) / BM);
  L.c_pad = (n_classes + 255) / 256 * 256;
  auto up = [](size_t v) { return (v + 1023) / 1024 * 1024; };
  size_t off = up((size_t)L.n_rb * BM * L.c_pad * 2);
  L.off_bound = off; off += up((size_t)n_rows * 4);
  L.off_tcos = off; off += up((size_t)n_rows * 4);
  L.off_scale = off; off += up((size_t)n_rows * 4);
  L.off_xs = off; off += up((size_t)n_rows * emb * 2);
  L.total = off;
  return L;
}
size_t tc_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb) { return prob_layout(n_rows, n_classes, emb).total; }

// w == nullptr: w_hat / inv_norm are already valid (normalised by PartialFC.step), only the logits kernels run.
// prob_ws != nullptr: MODE_PROB forward (probabilities kept for tc_bwd_prob), else MODE_STATS.
static int tc_normalize_fwd_enqueue(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes,
                                    int emb, float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum,
                                    float* target_logit, char* prob_ws, cudaStream_t st) {
  PFC_REQUIRE(tensor_emb_ok(emb), PFC_E_SHAPE, "tensor path supports emb in {64,128,256,512}, got %d (use PFC_PATH_CHECK)", emb);
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && n_classes < (1ll << 30) && n_rows < (1ll << 24), PFC_E_SHAPE, "pfc_normalize_fwd_stats: shape out of range");
  auto* wh = reinterpret_cast<__nv_bfloat16*>(w_hat);
  const int bn = g_logits_pair ? 256 : g_fwd_bn;
  PFC_REQUIRE(!prob_ws || g_logits_pair, PFC_E_ARG, "the stored-probability forward needs the CTA-pair logits kernels");
  int64_t n_chunks = (g_logits_pair && w) ? g_fwd_chunks : 1;          // the normaliser warps live in the CTA-pair kernel
  if (n_chunks > n_classes / 16384) n_chunks = n_classes / 16384;      // a chunk must keep every SM busy for a while
  if (n_chunks < 1) n_chunks = 1;
  const int64_t chunk = ((n_classes + n_chunks - 1) / n_chunks + 255) / 256 * 256;
  const int grid_full = g_logits_pair ? pair_grid(n_rows, n_classes) : fwd_grid(n_rows, n_classes, bn);
  PFC_CUDA(cudaMemsetAsync(part_sum, 0, sizeof(float) * (size_t)grid_full * 2 * n_rows, st));
  PFC_CUDA(cudaMemsetAsync(target_logit, 0, sizeof(float) * (size_t)n_rows, st));
  CUtensorMap tx, tg;
  if (int rc = make_tmap_bf16_2d(&tx, x, n_rows, emb, emb, BM)) return rc;
  const ProbLayout L = prob_layout(n_rows, n_classes, emb);
  float* row_bound = nullptr;
  float* target_cos = nullptr;
  if (prob_ws) {
    row_bound = reinterpret_cast<float*>(prob_ws + L.off_bound);
    target_cos = reinterpret_cast<float*>(prob_ws + L.off_tcos);
    const uint64_t g_rows = (uint64_t)(L.c_pad / 64) * L.n_rb * BM;                        // blocked scratch viewed as [g_rows, 64]
    if (int rc = make_tmap_bf16_2d(&tg, prob_ws, g_rows, 64, 64, 32)) return rc;            // epilogue store boxes [32 rows x 64 classes]
    row_bound_kernel<<<(int)((n_rows + 7) / 8), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), n_rows, emb, s * kLog2e, row_bound,
                                                              range_flag_of_current_device(), g_range_limit_nats * kLog2e);
    PFC_LAUNCH_CHECK();
  }
  auto chunk_len = [&](int64_t c0) { return (n_classes - c0 < chunk) ? n_classes - c0 : chunk; };
  // chunk 0 is normalised by the stand-alone kernel; chunk k+1 by the normaliser warps of the logits kernel of chunk k
  if (w) {
    prof_begin(PH_NORMALIZE, st);
    if (int rc = launch_normalize_rows(w, index, chunk_len(0), emb, wh, nullptr, inv_norm, 0, st)) return rc;
    prof_end(PH_NORMALIZE, st);
  }
  int k = 0;
  for (int64_t c0 = 0; c0 < n_classes; c0 += chunk, ++k) {
    const int64_t cc = chunk_len(c0);
    const int64_t n0 = c0 + chunk;                                     // first class of the next chunk
    const bool has_next = w && n0 < n_classes;
    CUtensorMap tw;
    if (int rc = make_tmap_bf16_2d(&tw, wh + c0 * emb, cc, emb, emb, g_logits_pair ? 128 : bn)) return rc;
    LogitsParams p{};
    p.label = label; p.n_rows = (int)n_rows; p.n_classes = (int)cc; p.class_base = (int)c0; p.emb = emb;
    p.n_rb = (int)((n_rows + BM - 1) / BM); p.n_ct = (int)((cc + bn - 1) / bn);
    p.s = s; p.m = m; p.margin_kind = margin_kind; p.part_max = part_max; p.part_sum = part_sum; p.target_logit = target_logit; p.accumulate_stats = k > 0; p.prefetch = g_prefetch[0];
    p.row_bound = row_bound; p.target_cos = target_cos; p.ldg = L.c_pad;
    if (has_next) {
      p.norm_w = index ? w : w + n0 * emb; p.norm_index = index ? index + n0 : nullptr; p.norm_rows = chunk_len(n0);
      p.norm_out = wh + n0 * emb; p.norm_inv = inv_norm + n0;
    }
    const int grid = g_logits_pair ? pair_grid(n_rows, cc) : fwd_grid(n_rows, cc, bn);
    prof_begin(PH_FWD, st);
    int rc;
    if (!g_logits_pair) rc = dispatch_logits<MODE_STATS>(tx, tw, p, bn, grid, st);
    else if (prob_ws) rc = has_next ? launch_logits2<4, MODE_PROB, true>(tx, tw, tg, p, grid, st) : launch_logits2<4, MODE_PROB>(tx, tw, tg, p, grid, st);
    else if (has_next) rc = launch_logits2<4, MODE_STATS, true>(tx, tw, tw, p, grid, st);
    else rc = launch_logits2<4, MODE_STATS>(tx, tw, tw, p, grid, st);
    if (rc) return rc;
    prof_end(PH_FWD, st);
  }
  return 0;
}

int tc_normalize_fwd(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                     float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum, float* target_logit, cudaStream_t st) {
  auto enqueue = [&](cudaStream_t cs) {
    return tc_normalize_fwd_enqueue(w, index, x, label, n_rows, n_classes, emb, s, m, margin_kind, w_hat, inv_norm, part_max, part_sum, target_logit, nullptr, cs);
  };
  if (!graph_eligible(st)) return enqueue(st);
  KeyBuilder kb;
  kb.add(2).add(w).add(index).add(x).add(label).add(n_rows).add(n_classes).add(emb).add(s).add(m).add(margin_kind).add(w_hat).add(inv_norm).add(part_max)
      .add(part_sum).add(target_logit).add(g_fwd_bn).add(g_logits_pair).add(g_fwd_chunks).add(g_norm_blocks_per_sm).add(g_prefetch[0]);
  if (kb.overflow) return enqueue(st);
  return run_cached_graph(kb, st, enqueue);
}

// ---- stored-probability path: forward keeps P, backward = per-row prep + (dx || dw) -------------
int tc_normalize_fwd_prob(const float* w, const int64_t* index, const void* x, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                          float s, float m, int margin_kind, void* w_hat, float* inv_norm, float* part_max, float* part_sum, float* target_logit,
                          void* prob_ws, size_t prob_ws_bytes, cudaStream_t st) {
  PFC_REQUIRE(prob_ws && prob_ws_bytes >= tc_prob_workspace_bytes(n_rows, n_classes, emb), PFC_E_WORKSPACE,
              "pfc_normalize_fwd_prob: probability workspace too small (%zu < %zu)", prob_ws_bytes, tc_prob_workspace_bytes(n_rows, n_classes, emb));
  PFC_REQUIRE((reinterpret_cast<uintptr_t>(prob_ws) & 1023) == 0, PFC_E_ARG, "pfc_normalize_fwd_prob: workspace must be 1024-byte aligned");
  auto enqueue = [&](cudaStream_t cs) {
    return tc_normalize_fwd_enqueue(w, index, x, label, n_rows, n_classes, emb, s, m, margin_kind, w_hat, inv_norm, part_max, part_sum, target_logit,
                                    reinterpret_cast<char*>(prob_ws), cs);
  };
  if (!graph_eligible(st)) return enqueue(st);
  KeyBuilder kb;
  kb.add(3).add(w).add(index).add(x).add(label).add(n_rows).add(n_classes).add(emb).add(s).add(m).add(margin_kind).add(w_hat).add(inv_norm).add(part_max)
      .add(part_sum).add(target_logit).add(prob_ws).add(g_fwd_bn).add(g_logits_pair).add(g_fwd_chunks).add(g_norm_blocks_per_sm).add(g_prefetch[0])
      .add(range_flag_of_current_device()).add(g_range_limit_nats);
  if (kb.overflow) return enqueue(st);
  return run_cached_graph(kb, st, enqueue);
}

struct ProbBwdPlan {
  bool dx_pair, side_by_side;
  int dx_bn, n_eh, ksplit, dcs, dx_ctas, sm_dw;
  size_t dxp_bytes;
};
static int g_prob_dx_sms = 0;            // 0 = choose from the shape; > 0: SM budget of the dx kernel (tuning knob)
static float g_prob_dw_rate = 0.42f;     // measured per-SM throughput of the dw kernel relative to the dx kernel
static float g_prob_dw4_rate = 0.65f;    // the same for the dw4 kernel at the shapes it is chosen for (r02i: 0.62 at Bt = 2048, 0.79 at 4096)
static int g_sweep_lead = 0;             // classes the faster of dx / dw may run ahead of the other (0 = not paced: measured no gain)

static ProbBwdPlan make_prob_bwd_plan(int64_t n_rows, int64_t n_classes, int emb) {
  ProbBwdPlan pl{};
  const int64_t n_rb = (n_rows + BM - 1) / BM;
  const int sms = sm_count();
  pl.dx_bn = emb < 256 ? emb : 256;
  pl.n_eh = emb / pl.dx_bn;
  pl.dx_pair = g_dx_pair && g_logits_pair && emb >= 256 && n_rb % 4 == 0;
  pl.dcs = g_dx_cluster;
  if (pl.dx_bn < 128) pl.dcs = 1;
  if (pl.dx_bn == 128 && pl.dcs > 2) pl.dcs = 2;
  const int64_t units = pl.dx_pair ? (n_rb / 4) * pl.n_eh * 2 : ((n_rb + pl.dcs - 1) / pl.dcs) * pl.dcs * pl.n_eh;   // CTAs per k-split
  const int64_t max_ks = (n_classes + BK - 1) / BK < 64 ? (n_classes + BK - 1) / BK : 64;
  // dx and dw run side by side on disjoint SMs; pick the k-split whose slower side finishes first
  int64_t best = 0;
  float best_t = 0.f;
  const float dw_rate = dw4_chosen(n_rows, emb) ? g_prob_dw4_rate : g_prob_dw_rate;
  for (int64_t ks = 1; ks <= max_ks && units * ks <= sms - 16; ++ks) {
    const float t_dx = 1.f / (float)(units * ks), t_dw = 1.f / (dw_rate * (float)(sms - units * ks));
    const float t = g_prob_dx_sms > 0 ? fabsf((float)(units * ks - g_prob_dx_sms)) : (t_dx > t_dw ? t_dx : t_dw);
    if (best == 0 || t < best_t) { best = ks; best_t = t; }
  }
  pl.side_by_side = best > 0;
  if (!pl.side_by_side) {                 // more dx units than SMs to spare: one kernel after the other, each on the whole GPU
    best = sms / units;
    if (best < 1) best = 1;
    if (best > max_ks) best = max_ks;
  }
  pl.ksplit = (int)best;
  pl.dx_ctas = (int)(units * best);
  pl.sm_dw = pl.side_by_side ? sms - pl.dx_ctas : sms;
  pl.dxp_bytes = ((size_t)pl.ksplit * n_rows * emb * 4 + 1023) / 1024 * 1024;
  return pl;
}

size_t tc_bwd_prob_workspace_bytes(int64_t n_rows, int64_t n_classes, int emb) {
  const ProbBwdPlan pl = make_prob_bwd_plan(n_rows, n_classes, emb);
  return pl.dxp_bytes + 1024;       // split-K slabs + the two sweep counters
}

static int tc_bwd_prob_enqueue(const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_sum, int64_t n_rows, int64_t n_classes,
                               int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw,
                               const void* x, char* prob_ws, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  PFC_REQUIRE(tensor_emb_ok(emb), PFC_E_SHAPE, "tensor path supports emb in {64,128,256,512}, got %d (use PFC_PATH_CHECK)", emb);
  PFC_REQUIRE(n_rows > 0 && n_classes > 0 && n_classes < (1ll << 30) && n_rows < (1ll << 24), PFC_E_SHAPE, "pfc_bwd_prob: shape out of range");
  const ProbLayout L = prob_layout(n_rows, n_classes, emb);
  const ProbBwdPlan pl = make_prob_bwd_plan(n_rows, n_classes, emb);
  PFC_REQUIRE(workspace_bytes >= pl.dxp_bytes + 1024, PFC_E_WORKSPACE, "pfc_bwd_prob: workspace too small (%zu < %zu)", workspace_bytes,
              pl.dxp_bytes + 1024);
  int* sweep_ctr = reinterpret_cast<int*>(reinterpret_cast<char*>(workspace) + pl.dxp_bytes);      // [0] dx, [1] dw
  PFC_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, PFC_E_ARG, "pfc_bwd_prob: workspace must be 1024-byte aligned");
  float* dx_part = reinterpret_cast<float*>(workspace);
  auto* scratch = reinterpret_cast<__nv_bfloat16*>(prob_ws);
  const float* row_bound = reinterpret_cast<const float*>(prob_ws + L.off_bound);
  const float* target_cos = reinterpret_cast<const float*>(prob_ws + L.off_tcos);
  float* row_scale = reinterpret_cast<float*>(prob_ws + L.off_scale);
  auto* xs = reinterpret_cast<__nv_bfloat16*>(prob_ws + L.off_xs);
  const auto* wh = reinterpret_cast<const __nv_bfloat16*>(w_hat);
  const int n_rb = L.n_rb;
  const float g_scale = s * inv_total_batch;

  // (1) per-row prep: scaled x_hat, row scales, target elements of the scratch
  prof_begin(PH_GRAD, st);
  prob_prep_kernel<<<(int)((n_rows + 7) / 8), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), label, row_sum, row_bound, target_cos, n_rows, emb,
                                                            n_rb, n_classes, s, m, margin_kind, g_scale, xs, row_scale, scratch,
                                                            range_flag_of_current_device());
  PFC_LAUNCH_CHECK();
  prof_end(PH_GRAD, st);

  // (2) dx || dw over the whole shard
  const uint64_t g_rows = (uint64_t)(L.c_pad / 64) * n_rb * BM;
  CUtensorMap tg_k, tw_mn, tg_mn, tx_mn, twh_e, tdw_e;
  if (int rc = make_tmap_bf16_2d(&tg_k, scratch, g_rows, 64, 64, BM)) return rc;           // dx A: [128 rows x 64 classes] blocks
  if (int rc = make_tmap_bf16_2d(&tw_mn, wh, n_classes, emb, emb, 64)) return rc;          // dx B: MN-major boxes [64 classes x 64 e]
  if (int rc = make_tmap_bf16_2d(&tg_mn, scratch, g_rows, 64, 64, 64)) return rc;          // dw A: [64 rows x 64 classes] boxes
  if (int rc = make_tmap_bf16_2d(&tx_mn, xs, n_rows, emb, emb, 64)) return rc;             // dw B: scaled x_hat, [64 rows x 64 e]
  if (int rc = make_tmap_bf16_2d(&twh_e, wh, n_classes, emb, emb, 32)) return rc;          // dw epilogue: per-warp [32 classes x 64 e]
  if (int rc = make_tmap_f32_2d(&tdw_e, dw, n_classes, emb, emb, 32)) return rc;           // dw epilogue: per-warp [32 classes x 32 e] fp32
  cudaStream_t sX = st, sW = st;
  EventPool pool;
  const bool paced = pl.side_by_side && g_sweep_lead > 0;
  if (paced) PFC_CUDA(cudaMemsetAsync(sweep_ctr, 0, 2 * sizeof(int), st));
  if (pl.side_by_side) {
    if (int rc = side_streams(&sX, &sW)) return rc;
    PFC_EDGE(st, sX);
    PFC_EDGE(st, sW);
  }
  DxParams dp{};
  if (paced) dp.sweep = SweepSync{sweep_ctr, sweep_ctr + 1, g_sweep_lead};
  dp.n_rows = (int)n_rows; dp.n_classes = (int)n_classes; dp.emb = emb; dp.n_rb = n_rb; dp.n_eh = pl.n_eh; dp.ksplit = pl.ksplit;
  dp.dx_part = dx_part; dp.accumulate = 0; dp.prefetch = g_prefetch[1]; dp.strided = pl.side_by_side ? 1 : 0;
  auto enqueue_dx = [&]() -> int {
    int rc = 0;
    prof_begin(PH_DX, sX);
    if (pl.dx_pair) rc = launch_dx2(tg_k, tw_mn, dp, pl.dx_ctas, sX);
    else switch (pl.dx_bn) {
      case 256: rc = launch_dx<256>(tg_k, tw_mn, dp, pl.dx_ctas, pl.dcs, sX); break;
      case 128: rc = launch_dx<128>(tg_k, tw_mn, dp, pl.dx_ctas, pl.dcs, sX); break;
      default: rc = launch_dx<64>(tg_k, tw_mn, dp, pl.dx_ctas, pl.dcs, sX); break;
    }
    if (rc) return rc;
    prof_end(PH_DX, sX);
    return 0;
  };
  const bool use_dw4 = dw4_chosen(n_rows, emb);
  auto enqueue_dw = [&]() -> int {
    int rc = 0;
    DwParams wp{};
    if (paced) wp.sweep = SweepSync{sweep_ctr + 1, sweep_ctr, g_sweep_lead};
    wp.n_rows = (int)n_rows; wp.n_classes = (int)n_classes; wp.emb = emb; wp.n_ct = (int)((n_classes + BM - 1) / BM); wp.n_rb = n_rb;
    wp.inv_norm = inv_norm; wp.accumulate = accumulate_dw; wp.dbg = g_dbg; wp.prefetch = g_prefetch[2];
    prof_begin(PH_DW, sW);
    if (use_dw4) {
      Dw4Params qp{};
      qp.n_rows = (int)n_rows; qp.n_classes = (int)n_classes; qp.n_rb = n_rb; qp.n_tp = (int)((n_classes + 255) / 256);
      qp.inv_norm = inv_norm; qp.w_hat = wh; qp.dw = dw; qp.accumulate = accumulate_dw; qp.dbg = g_dbg;
      rc = launch_dw4(tg_mn, tx_mn, qp, pl.sm_dw, sW);
    } else switch (emb) {
      case 512: rc = launch_dw<512>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
      case 256: rc = launch_dw<256>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
      case 128: rc = launch_dw<128>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
      default: rc = launch_dw<64>(tg_mn, tx_mn, twh_e, tdw_e, wp, wp.n_ct, g_dw_cluster, pl.sm_dw, sW); break;
    }
    if (rc) return rc;
    prof_end(PH_DW, sW);
    return 0;
  };
  // the 4-CTA clusters of dw4 are placed first (they need four free SMs of one GPC), the dx pairs fill what is left
  if (use_dw4) {
    if (int rc = enqueue_dw()) return rc;
    if (int rc = enqueue_dx()) return rc;
  } else {
    if (int rc = enqueue_dx()) return rc;
    if (int rc = enqueue_dw()) return rc;
  }
  if (pl.side_by_side) {
    PFC_EDGE(sX, st);
    PFC_EDGE(sW, st);
  }
  // (3) dx = row scale x sum of the split-K slabs
  const int64_t n_vec = n_rows * emb / 4;
  int64_t blocks = (n_vec + 255) / 256;
  if (blocks > (int64_t)sm_count() * 4) blocks = (int64_t)sm_count() * 4;
  reduce_dx_scaled_kernel<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(dx_part), pl.ksplit, n_vec, emb / 4, row_scale,
                                                       reinterpret_cast<float4*>(dx));
  PFC_LAUNCH_CHECK();
  return 0;
}

int tc_bwd_prob(const void* x, const void* w_hat, const float* inv_norm, const int64_t* label, const float* row_sum, int64_t n_rows, int64_t n_classes,
                int emb, float s, float m, int margin_kind, float inv_total_batch, float* dx, float* dw, int accumulate_dw, void* prob_ws,
                size_t prob_ws_bytes, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  PFC_REQUIRE(prob_ws && prob_ws_bytes >= tc_prob_workspace_bytes(n_rows, n_classes, emb), PFC_E_WORKSPACE, "pfc_bwd_prob: probability workspace too small");
  auto enqueue = [&](cudaStream_t cs) {
    return tc_bwd_prob_enqueue(w_hat, inv_norm, label, row_sum, n_rows, n_classes, emb, s, m, margin_kind, inv_total_batch, dx, dw, accumulate_dw, x,
                               reinterpret_cast<char*>(prob_ws), workspace, workspace_bytes, cs);
  };
  if (!graph_eligible(st)) return enqueue(st);
  KeyBuilder kb;
  kb.add(4).add(x).add(w_hat).add(inv_norm).add(label).add(row_sum).add(dx).add(dw).add(workspace).add(prob_ws).add(n_rows).add(n_classes)
      .add(workspace_bytes).add(emb).add(accumulate_dw).add(s).add(m).add(margin_kind).add(inv_total_batch).add(g_logits_pair).add(g_dx_cluster)
      .add(g_dw_cluster).add(g_prob_dx_sms).add(g_prob_dw_rate).add(g_sweep_lead).add(g_prefetch[1]).add(g_prefetch[2]).add(g_dx_pair)
      .add(range_flag_of_current_device()).add(g_dw4);
  if (kb.overflow) return enqueue(st);
  return run_cached_graph(kb, st, enqueue);
}

void tc_set_prob_split(int dx_sms, float dw_rate, int sweep_lead) {
  g_prob_dx_sms = dx_sms > 0 ? dx_sms : 0;
  if (dw_rate > 0.05f && dw_rate < 4.f) g_prob_dw_rate = dw_rate;
  if (sweep_lead >= 0) g_sweep_lead = sweep_lead;
}

// ---- SpreadOut (server.py:48-63) on the same kernel pair ---------------------------------------
// similarity = w_hat . w_hat^T is a logits GEMM with x_hat := w_hat; its epilogue (MODE_HINGE) keeps H = relu(sim - margin)
// off the diagonal as bf16 and sums H^2; the gradient w.r.t. the normalised rows is 4 H . w_hat (H is symmetric), which is
// the dx GEMM on that scratch.  The row-wise normalize backward and the loss reduction are O(N E) glue on the host side.
struct SpreadPlan {
  int n_rb, dx_bn, n_eh, dcs, ksplit, dx_grid;
  bool dx_pair;
  int64_t c_pad;
  size_t scratch_bytes, dxp_bytes;
};
static SpreadPlan make_spread_plan(int64_t n, int emb) {
  SpreadPlan pl{};
  pl.n_rb = (int)((n + BM - 1) / BM);
  pl.c_pad = (n + 255) / 256 * 256;
  pl.dx_bn = emb < 256 ? emb : 256;
  pl.n_eh = emb / pl.dx_bn;
  pl.dx_pair = g_dx_pair && emb >= 256 && pl.n_rb % 4 == 0;
  pl.dcs = g_dx_cluster;
  if (pl.dx_bn < 128) pl.dcs = 1;
  if (pl.dx_bn == 128 && pl.dcs > 2) pl.dcs = 2;
  const int64_t units = pl.dx_pair ? (int64_t)(pl.n_rb / 4) * pl.n_eh * 2 : (int64_t)((pl.n_rb + pl.dcs - 1) / pl.dcs) * pl.dcs * pl.n_eh;
  int64_t ks = sm_count() / units;
  const int64_t n_kb = (n + BK - 1) / BK;
  if (ks > n_kb) ks = n_kb;
  if (ks > 64) ks = 64;
  if (ks < 1) ks = 1;
  pl.ksplit = (int)ks;
  pl.dx_grid = (int)(units * ks);
  pl.scratch_bytes = ((size_t)pl.n_rb * BM * pl.c_pad * 2 + 1023) / 1024 * 1024;
  pl.dxp_bytes = ((size_t)pl.ksplit * n * emb * 4 + 1023) / 1024 * 1024;
  return pl;
}
size_t tc_spreadout_workspace_bytes(int64_t n, int emb) {
  const SpreadPlan pl = make_spread_plan(n, emb);
  return pl.scratch_bytes + pl.dxp_bytes;
}

int tc_spreadout(const void* w_hat, int64_t n, int emb, float margin, float* part_max, float* part_sum, float* hw_out, void* workspace,
                 size_t workspace_bytes, cudaStream_t st) {
  PFC_REQUIRE(tensor_emb_ok(emb), PFC_E_SHAPE, "tensor path supports emb in {64,128,256,512}, got %d", emb);
  PFC_REQUIRE(n > 0 && n < (1ll << 24), PFC_E_SHAPE, "pfc_spreadout: row count out of range");
  const SpreadPlan pl = make_spread_plan(n, emb);
  PFC_REQUIRE(workspace_bytes >= pl.scratch_bytes + pl.dxp_bytes, PFC_E_WORKSPACE, "pfc_spreadout: workspace too small (%zu < %zu)", workspace_bytes,
              pl.scratch_bytes + pl.dxp_bytes);
  PFC_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, PFC_E_ARG, "pfc_spreadout: workspace must be 1024-byte aligned");
  char* scratch = reinterpret_cast<char*>(workspace);
  float* dx_part = reinterpret_cast<float*>(scratch + pl.scratch_bytes);
  const uint64_t g_rows = (uint64_t)(pl.c_pad / 64) * pl.n_rb * BM;
  CUtensorMap tx, tw, tg_st, tg_k, tw_mn;
  if (int rc = make_tmap_bf16_2d(&tx, w_hat, n, emb, emb, BM)) return rc;
  if (int rc = make_tmap_bf16_2d(&tw, w_hat, n, emb, emb, 128)) return rc;
  if (int rc = make_tmap_bf16_2d(&tg_st, scratch, g_rows, 64, 64, 32)) return rc;
  if (int rc = make_tmap_bf16_2d(&tg_k, scratch, g_rows, 64, 64, BM)) return rc;
  if (int rc = make_tmap_bf16_2d(&tw_mn, w_hat, n, emb, emb, 64)) return rc;
  const int grid = pair_grid(n, n);
  PFC_CUDA(cudaMemsetAsync(part_sum, 0, sizeof(float) * (size_t)grid * 2 * n, st));
  LogitsParams p{};
  p.n_rows = (int)n; p.n_classes = (int)n; p.class_base = 0; p.emb = emb;
  p.n_rb = pl.n_rb; p.n_ct = (int)((n + 255) / 256); p.m = margin; p.part_max = part_max; p.part_sum = part_sum; p.ldg = pl.c_pad;
  if (int rc = launch_logits2<4, MODE_HINGE>(tx, tw, tg_st, p, grid, st)) return rc;
  DxParams dp{};
  dp.n_rows = (int)n; dp.n_classes = (int)n; dp.emb = emb; dp.n_rb = pl.n_rb; dp.n_eh = pl.n_eh; dp.ksplit = pl.ksplit;
  dp.dx_part = dx_part; dp.accumulate = 0; dp.prefetch = 0; dp.strided = 0;
  int rc = 0;
  if (pl.dx_pair) rc = launch_dx2(tg_k, tw_mn, dp, pl.dx_grid, st);
  else switch (pl.dx_bn) {
    case 256: rc = launch_dx<256>(tg_k, tw_mn, dp, pl.dx_grid, pl.dcs, st); break;
    case 128: rc = launch_dx<128>(tg_k, tw_mn, dp, pl.dx_grid, pl.dcs, st); break;
    default: rc = launch_dx<64>(tg_k, tw_mn, dp, pl.dx_grid, pl.dcs, st); break;
  }
  if (rc) return rc;
  const int64_t n_vec = n * emb / 4;
  int64_t blocks = (n_vec + 255) / 256;
  if (blocks > (int64_t)sm_count() * 4) blocks = (int64_t)sm_count() * 4;
  reduce_dx_kernel<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(dx_part), pl.ksplit, n_vec, reinterpret_cast<float4*>(hw_out));
  PFC_LAUNCH_CHECK();
  return 0;
}

void tc_set_fwd_overlap(int chunks, int norm_blocks_per_sm) {
  if (chunks >= 1 && chunks <= 64) g_fwd_chunks = chunks;
  if (norm_blocks_per_sm >= 1 && norm_blocks_per_sm <= 8) g_norm_blocks_per_sm = norm_blocks_per_sm;
}

int tc_set_range_flag(int* flag, float limit_nats) {
  int dev = 0;
  PFC_CUDA(cudaGetDevice(&dev));
  PFC_REQUIRE(dev >= 0 && dev < 64, PFC_E_ARG, "device index out of range");
  g_range_flag[dev] = flag;
  if (limit_nats > 0.f) g_range_limit_nats = limit_nats;
  return 0;
}
void tc_set_graph(int on) { g_use_graph = on ? 1 : 0; }
void tc_set_dw4(int on) { g_dw4 = on < 0 ? -1 : (on > 0 ? 1 : 0); }
void tc_set_dx_pair(int on) { g_dx_pair = on ? 1 : 0; }
void tc_set_prefetch(int logits, int dx, int dw) { g_prefetch[0] = logits; g_prefetch[1] = dx; g_prefetch[2] = dw; }
void tc_set_pipeline(int on, int sm_g, int sm_dx, int sm_dw, int ring) {
  g_pipe = on ? 1 : 0;
  if (sm_g > 0 && sm_dx > 0 && sm_dw > 0) { g_split[0] = sm_g; g_split[1] = sm_dx; g_split[2] = sm_dw; }
  if (ring >= 1 && ring <= 8) g_ring = ring;
}
void tc_set_chunk_mb(int mb) { g_chunk_budget_mb = mb > 0 ? mb : 0; }
void tc_set_fwd_bn(int bn) { g_fwd_bn = (bn == 256) ? 256 : 128; }
void tc_set_debug(long long* p) { g_dbg = p; }
void tc_set_logits_pair(int on) { g_logits_pair = on ? 1 : 0; }
void tc_set_clusters(int dx_cs, int dw_cs) {
  if (dx_cs == 1 || dx_cs == 2 || dx_cs == 4) g_dx_cluster = dx_cs;
  if (dw_cs == 1 || dw_cs == 2 || dw_cs == 4) g_dw_cluster = dw_cs;
}

}  // namespace pfc
