/* CPU oracle (plain C) for 1:N identification  --  TEST INFRASTRUCTURE ONLY.
 *
 * The checker, never the product: only tests/ and tools/ident_bench.py load the library built from this file
 * (oracle/identify_oracle.py compiles it with gcc -ffp-contract=off into a temporary directory on first use).
 * It restates csrc/identify.cu's pfc_identify bit for bit; the tests also check it against a stable numpy argsort. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>


/* 1:N identification (fedfr_b200.verify.mate_ranks; csrc/identify.cu pfc_identify), a literal loop over the definition in
 * include/fedfr_b200.h.  The score of a (probe, gallery) pair is oracle_pair_scores' chain (oracle_verify.c); keys are
 * pfc_tar_at_far's (order-preserving, -0.0 folded onto +0.0, NaN -> 0). */
static float ident_chain(const float* a, const float* b, int emb) {
  double tmp = 0.0;
  for (int k = 0; k < emb; ++k) {
    const float q = a[k] * b[k];
    tmp = tmp + (double)q;
  }
  return (float)tmp;
}

static uint32_t ident_key(float s) {
  union { float f; uint32_t u; } v;
  v.f = s;
  uint32_t u = v.u;
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0u;
  if ((u & 0x7fffffffu) == 0u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

static float ident_value(uint32_t key) {
  union { uint32_t u; float f; } v;
  v.u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  return v.f;
}

/* scores [P, G] of every (probe, gallery) pair, for the tests' independent numpy check. */
void oracle_score_matrix(const float* probe, int64_t P, const float* gallery, int64_t G, int emb, float* out) {
  for (int64_t p = 0; p < P; ++p)
    for (int64_t g = 0; g < G; ++g) out[p * G + g] = ident_chain(probe + p * (int64_t)emb, gallery + g * (int64_t)emb, emb);
}

/* rank, top1_row int64 [P]; mate_score, top1_score fp32 [P]; counts int64 [2] = {NaN scores, mate rows outside [-1, G)}. */
void oracle_identify(const float* probe, int64_t P, const float* gallery, int64_t G, int emb, const int64_t* mate_row,
                     int64_t* rank, float* mate_score, int64_t* top1_row, float* top1_score, int64_t* counts) {
  uint32_t* key = (uint32_t*)malloc((size_t)(G > 0 ? G : 1) * sizeof(uint32_t));
  float* s = (float*)malloc((size_t)(G > 0 ? G : 1) * sizeof(float));
  counts[0] = counts[1] = 0;
  for (int64_t p = 0; p < P; ++p) {
    for (int64_t g = 0; g < G; ++g) {
      s[g] = ident_chain(probe + p * (int64_t)emb, gallery + g * (int64_t)emb, emb);
      key[g] = ident_key(s[g]);
      counts[0] += key[g] == 0u;
    }
    const int64_t m = mate_row[p];
    if (m >= 0 && m < G) {
      int64_t r = 1;
      for (int64_t g = 0; g < G; ++g)
        if (key[g] > key[m] || (key[g] == key[m] && g < m)) ++r;
      rank[p] = r;
      mate_score[p] = s[m];
    } else {
      counts[1] += m != -1;
      rank[p] = 0;
      mate_score[p] = NAN;
    }
    int64_t best = 0;
    for (int64_t g = 1; g < G; ++g)
      if (key[g] > key[best]) best = g;
    top1_row[p] = best;
    top1_score[p] = ident_value(key[best]);
  }
  free(key);
  free(s);
}
