/* fedfr_b200 -- developer / tuning hooks of libfedfr_b200.so.
 *
 * NOT part of the reference-facing surface (include/fedfr_b200.h): nothing here replaces a reference interface.  These
 * entries expose launch accounting, per-phase timing, NVTX ranges and the tuning knobs that bench.py / tools/ use to
 * sweep kernel configurations.  All of them are process-global, none is needed for correct results, and their defaults
 * are what the product ships with.  Every function returns 0 on success (pfc_launch_count returns the count). */
#ifndef FEDFR_B200_DEV_H_
#define FEDFR_B200_DEV_H_
#ifdef __cplusplus
extern "C" {
#endif

/* kernels launched by this library so far (bench.py reports the difference over its timed region as gpu_launches) */
long long pfc_launch_count(void);

/* per-phase device timing: CUDA events around the phases (normalize, forward, prep/grad, dx, dw) on their launch streams.
 * enable(1) also turns CUDA-graph replay off so that the events bracket real launches; collect() synchronises, returns the
 * summed milliseconds and span counts of the five phases and resets. */
int pfc_profile_enable(int on);
int pfc_profile_collect(float* ms_out /* [5] */, int* count_out /* [5] */);

/* NVTX ranges around every compute entry of the library (default: environment variable FEDFR_NVTX) */
int pfc_set_nvtx(int on);

/* device buffer of 16 int64 cycle counters written by CTA 0 of the dw kernels (tools/dw_probe.py); NULL = off */
int pfc_set_debug_buffer(void* dev_ptr);

/* ---- tuning knobs (defaults in brackets) ---- */
int pfc_set_graph(int on);                                  /* [1] replay forward / backward as cached CUDA graphs */
int pfc_set_logits_pair(int on);                            /* [1] cta_group::2 logits kernels; 0 = single-CTA kernels */
int pfc_set_logits_tile(int bn);                            /* [128] class-tile width of the single-CTA logits kernels (128 / 256) */
int pfc_set_dx_pair(int on);                                /* [1] cta_group::2 dx kernel when ceil(Bt / 128) % 4 == 0, E >= 256 and
                                                               pfc_set_logits_pair is on (the last row block may be partial) */
int pfc_set_dw4(int mode);                                  /* [-1] E = 512 dw kernel: -1 auto (4-CTA-cluster kernel from 2048 gathered rows on),
                                                               0 e-split pair kernel, > 0 4-CTA-cluster kernel */
int pfc_set_clusters(int dx_cluster, int dw_cluster);       /* [2, 2] cluster sizes of the single-CTA dx / dw kernels (1, 2, 4) */
int pfc_set_fwd_overlap(int chunks, int norm_blocks_per_sm);/* [4, 2] class chunks of the fused forward; normalise blocks per SM */
int pfc_set_prefetch(int logits, int dx_distance, int dw);  /* [0, 0, 0] TMA L2 prefetch ahead of the shared-memory rings */
int pfc_set_prob_split(int dx_sms, float dw_rate, int sweep_lead);  /* [0 = from the shape, 0.42, 0] dx / dw SM split of the backward */
int pfc_set_pipeline(int on, int sm_g, int sm_dx, int sm_dw, int ring);  /* recompute backward: concurrent G / dx / dw chains */
int pfc_set_chunk_mb(int mb);                               /* [0 = default] bf16 G scratch per chunk of the recompute backward, MiB */
int pfc_set_roc_mode(int mode);                             /* ROC histogram kernel: 0 exact chain for every pair, 1 two-tier */

#ifdef __cplusplus
}
#endif
#endif  /* FEDFR_B200_DEV_H_ */
