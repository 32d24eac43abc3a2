/* CPU oracle (plain C) for 1:1 template verification  --  TEST INFRASTRUCTURE ONLY.
 *
 * The checker, never the product: only tests/ and tools/verify_bench.py load the library built from this file
 * (oracle/verify_oracle.py compiles it with gcc -ffp-contract=off into a temporary directory on first use).
 * It restates csrc/verify.cu's arithmetic bit for bit; tests/test_verify.py checks it against a float64 numpy
 * restatement of the recipe. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

/* 1:1 template verification (fedfr_b200.verify; csrc/verify.cu), the arithmetic pinned step by step:
 *   x_i = feats_i, or fl32(feats_i * weights_i)
 *   images visited in ascending (template, media) order, ties in row order
 *   media = fp32 sum of its images in that order starting from the first, then / (float)count when count > 1
 *   template t = fp32 sum of its medias in ascending media id, starting from the first
 *   out_k = (float)((double)t_k / max(sqrt(sum_k (double)t_k * (double)t_k), 1e-12)), fp64 adds over ascending k
 * out [n, emb] and out_ids [n] must hold n rows; returns the number of templates T (rows 0..T-1, ids ascending). */
static const int64_t* g_pool_t;
static const int64_t* g_pool_m;

static int pool_cmp(const void* pa, const void* pb) {         /* (template, media, row); not reentrant: tests only */
  const int64_t a = *(const int64_t*)pa, b = *(const int64_t*)pb;
  if (g_pool_t[a] != g_pool_t[b]) return g_pool_t[a] < g_pool_t[b] ? -1 : 1;
  if (g_pool_m[a] != g_pool_m[b]) return g_pool_m[a] < g_pool_m[b] ? -1 : 1;
  return a < b ? -1 : (a > b);
}

int64_t oracle_template_pool(const float* feats, const int64_t* templates, const int64_t* medias, const float* weights,
                             int64_t n, int emb, float* out, int64_t* out_ids) {
  int64_t* idx = (int64_t*)malloc((size_t)(n > 0 ? n : 1) * sizeof(int64_t));
  float* media = (float*)malloc((size_t)emb * sizeof(float));
  float* t = (float*)malloc((size_t)emb * sizeof(float));
  int64_t n_t = 0;
  for (int64_t i = 0; i < n; ++i) idx[i] = i;
  g_pool_t = templates;
  g_pool_m = medias;
  qsort(idx, (size_t)n, sizeof(int64_t), pool_cmp);
  for (int64_t a = 0; a < n;) {                                /* one template: idx[a .. b) */
    int64_t b = a;
    while (b < n && templates[idx[b]] == templates[idx[a]]) ++b;
    int first_media = 1;
    for (int64_t c = a; c < b;) {                              /* one media: idx[c .. d) */
      int64_t d = c;
      while (d < b && medias[idx[d]] == medias[idx[c]]) ++d;
      for (int64_t i = c; i < d; ++i) {
        const float* f = feats + idx[i] * (int64_t)emb;
        for (int k = 0; k < emb; ++k) {
          const float x = weights ? f[k] * weights[idx[i]] : f[k];
          media[k] = i == c ? x : media[k] + x;
        }
      }
      if (d - c > 1)
        for (int k = 0; k < emb; ++k) media[k] = media[k] / (float)(d - c);
      for (int k = 0; k < emb; ++k) t[k] = first_media ? media[k] : t[k] + media[k];
      first_media = 0;
      c = d;
    }
    double ss = 0.0;
    for (int k = 0; k < emb; ++k) ss += (double)t[k] * (double)t[k];
    double nrm = sqrt(ss);
    if (!(nrm > 1e-12)) nrm = 1e-12;
    for (int k = 0; k < emb; ++k) out[n_t * (int64_t)emb + k] = (float)((double)t[k] / nrm);
    out_ids[n_t++] = templates[idx[a]];
    a = b;
  }
  free(idx);
  free(media);
  free(t);
  return n_t;
}

/* score[p] = (float)tmp, tmp = 0.0; tmp = tmp + (double)fl32(a_k * b_k) over ascending k, a / b = rows row1[p] / row2[p]
 * of tf [n_rows, emb] (the chain of oracle_roc_histogram).  Returns -1 if a row is out of range. */
int oracle_pair_scores(const float* tf, int64_t n_rows, int emb, const int64_t* row1, const int64_t* row2, int64_t n_pairs,
                       float* out) {
  for (int64_t p = 0; p < n_pairs; ++p) {
    if (row1[p] < 0 || row1[p] >= n_rows || row2[p] < 0 || row2[p] >= n_rows) return -1;
    const float* a = tf + row1[p] * (int64_t)emb;
    const float* b = tf + row2[p] * (int64_t)emb;
    double tmp = 0.0;
    for (int k = 0; k < emb; ++k) {
      const float q = a[k] * b[k];
      tmp = tmp + (double)q;
    }
    out[p] = (float)tmp;
  }
  return 0;
}
