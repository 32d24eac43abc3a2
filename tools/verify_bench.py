"""Time 1:1 template verification (fedfr_b200.verify) at the IJB-C shape and write one JSON file.

    python tools/verify_bench.py --out OUT_DIR [--reps 20] [--seed 0]

Data: oracle.verify_oracle.ijbc_like, seeded synthetic arrays of the IJB-C 1:1 shape (227,630 images, 23,124 templates,
15,658,489 pairs grouped by p1, 19,557 genuine), E = 512.  Each stage is timed with CUDA events over `reps` calls after
a warm-up call: pooling (index plumbing included), pair scores (the pfc_pair_scores kernel alone, rows precomputed, and
the public call with its id lookup), TAR@FAR at the six IJB-C FARs (public call, with the read-back of its counts), and
the ROC curve (the pfc_roc_curve chain alone, buffers preallocated, and the public call with its read-back and copies).
The 47 MB of template features stay in the 126 MB L2 between passes, as they would in use.  Counted work: bytes the
pair kernel must read from L2 (every p2 row once per pair, every p1 row once per run of equal p1 in a 128-pair tile),
and fp32->fp64 conversions (P * E).  Baseline: the float64 numpy restatement on the host cores in the same run (the
pair scores on a seeded 1 M-pair sample, reported with its rate) and sklearn.metrics.roc_curve on all the scores.  The
ROC curve must equal sklearn's array for array.  Prints the card name and power limit and writes OUT_DIR/verify_bench.json.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
from sklearn.metrics import auc, roc_curve

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fedfr_b200 as F  # noqa: E402
from fedfr_b200 import _native as N  # noqa: E402
from fedfr_b200 import verify as V  # noqa: E402
from oracle import verify_oracle as O  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def cuda_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def numpy_pool(feats, templates, medias):
    """float64 numpy restatement of the recipe, vectorised: sort, media means, template sums, normalise."""
    order = np.lexsort((medias, templates))
    t, m, x = templates[order], medias[order], feats[order].astype(np.float64)
    cut = np.flatnonzero((np.diff(t) != 0) | (np.diff(m) != 0)) + 1
    starts = np.concatenate([[0], cut])
    media = np.add.reduceat(x, starts, axis=0) / np.diff(np.concatenate([starts, [t.size]]))[:, None]
    mt = t[starts]
    tcut = np.concatenate([[0], np.flatnonzero(np.diff(mt) != 0) + 1])
    tf = np.add.reduceat(media, tcut, axis=0)
    return tf / np.maximum(np.linalg.norm(tf, axis=1, keepdims=True), 1e-12), mt[tcut]


def numpy_scores(tf, r1, r2, chunk=1 << 16):
    out = np.empty(r1.size)
    for c in range(0, r1.size, chunk):
        out[c:c + chunk] = np.einsum("pk,pk->p", tf[r1[c:c + chunk]], tf[r2[c:c + chunk]])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("verify_bench: no CUDA device (a CPU run measures nothing)")
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda:0")
    gpu = card()
    print("[verify_bench]", gpu, flush=True)

    feats, t, m, p1, p2, y = O.ijbc_like(args.seed)
    P, E = p1.size, feats.shape[1]
    fd, td, md = (torch.from_numpy(a).to(dev) for a in (feats, t, m))
    p1d, p2d, yd = (torch.from_numpy(a).to(dev) for a in (p1, p2, y))

    ms_pool = cuda_ms(lambda: F.template_features(fd, td, md), args.reps)
    tf, ids = F.template_features(fd, td, md)
    r1, r2 = V.pair_rows(ids, p1d, p2d)
    scores = torch.empty(P, dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def kernel():
        N.check(N.lib.pfc_pair_scores(N.ptr(tf), tf.shape[0], E, N.ptr(r1), N.ptr(r2), P, N.ptr(scores), stream), "pfc_pair_scores")
    ms_pair_kernel = cuda_ms(kernel, args.reps)
    ms_pair_call = cuda_ms(lambda: F.pair_scores(tf, ids, p1d, p2d), args.reps)
    fars = V.DEFAULT_FARS
    ms_tar = cuda_ms(lambda: F.tar_at_far(scores, yd, fars), args.reps)
    result = F.tar_at_far(scores, yd, fars)
    exact = result == O.tar_at_far(scores.cpu().numpy(), y, fars)

    ws = torch.empty(int(N.lib.pfc_roc_curve_workspace_bytes(P)), dtype=torch.uint8, device=dev)
    curve_bufs = [torch.empty(P + 1, dtype=torch.float64, device=dev) for _ in range(3)]
    roc_out = torch.empty(4, dtype=torch.int64, device=dev)
    y8 = yd.to(torch.uint8)

    def roc_abi():
        N.check(N.lib.pfc_roc_curve(N.ptr(scores), N.ptr(y8), P, *(N.ptr(b) for b in curve_bufs), N.ptr(roc_out[3:]),
                                    N.ptr(roc_out), N.ptr(ws), ws.numel(), stream), "pfc_roc_curve")
    ms_roc_abi = cuda_ms(roc_abi, args.reps)
    ms_roc_call = cuda_ms(lambda: F.roc_curve(scores, yd), args.reps)
    curve = [c.cpu().numpy() for c in F.roc_curve(scores, yd)]

    # counted work of the pair kernel
    r1h = r1.cpu().numpy()
    tile = np.arange(P) // 128
    runs = int(np.count_nonzero((np.diff(r1h) != 0) | (np.diff(tile) != 0))) + 1
    l2_bytes = (P + runs) * E * 4
    conversions = P * E

    # host baseline: the float64 numpy restatement
    t0 = time.perf_counter()
    tf64, ids64 = numpy_pool(feats, t, m)
    s_np_pool = time.perf_counter() - t0
    sample = np.sort(np.random.default_rng(args.seed).choice(P, 1_000_000, replace=False))
    t0 = time.perf_counter()
    s64 = numpy_scores(tf64, np.searchsorted(ids64, p1[sample]), np.searchsorted(ids64, p2[sample]))
    s_np_pairs_sample = time.perf_counter() - t0
    s_all = scores.cpu().numpy()
    t0 = time.perf_counter()
    O.tar_at_far(s_all, y, fars)
    s_np_tar = time.perf_counter() - t0
    t0 = time.perf_counter()
    sk = roc_curve(y, s_all)
    s_sk_roc = time.perf_counter() - t0
    roc_exact = all(np.array_equal(a, b) for a, b in zip(curve, sk))
    max_dev = float(np.abs(s_all[sample] - s64).max())

    rec = {
        "tool": "verify_bench", "gpu": gpu, "shape": {"images": int(feats.shape[0]), "templates": int(ids.numel()), "pairs": int(P),
                                                      "genuine": int(y.sum()), "emb": int(E), "p1_runs_per_128_tiles": runs},
        "reps": args.reps,
        "ms": {"template_features": round(ms_pool, 4), "pair_scores_kernel": round(ms_pair_kernel, 4),
               "pair_scores_call": round(ms_pair_call, 4), "tar_at_far_6_fars": round(ms_tar, 4),
               "roc_curve_abi": round(ms_roc_abi, 4), "roc_curve_call": round(ms_roc_call, 4)},
        "pair_kernel": {"pairs_per_s": P / (ms_pair_kernel * 1e-3), "l2_bytes": l2_bytes,
                        "l2_bytes_per_s": l2_bytes / (ms_pair_kernel * 1e-3), "f2f_conversions": conversions,
                        "f2f_per_s": conversions / (ms_pair_kernel * 1e-3),
                        "f2f_per_clk_per_sm_at_max_clock": None},
        "tar_at_far": [{"far_target": f, "tar": tar, "far": far, "threshold": thr} for f, tar, far, thr in result],
        "tar_at_far_exact_vs_numpy": exact,
        "roc_curve": {"points": int(curve[0].size), "exact_vs_sklearn": roc_exact, "auc": auc(curve[0], curve[1]),
                      "sklearn_host_s": round(s_sk_roc, 3),
                      "tar_at_far_nearest": [{"far_target": f, "tar": tar, "far": far}
                                             for f, tar, far in F.tar_at_far_nearest(curve[0], curve[1], fars)]},
        "numpy_host": {"template_features_s": round(s_np_pool, 3), "pair_scores_sample": int(sample.size),
                       "pair_scores_sample_s": round(s_np_pairs_sample, 3),
                       "pair_scores_pairs_per_s": sample.size / s_np_pairs_sample, "tar_at_far_s": round(s_np_tar, 3),
                       "cpu_count": os.cpu_count(), "max_abs_diff_vs_float64": max_dev},
    }
    try:                                                  # F2F per clock per SM, at the card's maximum SM clock
        mhz = float(gpu.split(",")[2].strip().split()[0])
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        rec["pair_kernel"]["f2f_per_clk_per_sm_at_max_clock"] = conversions / (ms_pair_kernel * 1e-3) / (mhz * 1e6) / sms
    except (IndexError, ValueError):
        pass
    with open(os.path.join(args.out, "verify_bench.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))
    assert exact, "TAR@FAR differs from the numpy definition"
    assert roc_exact, "the ROC curve differs from sklearn.metrics.roc_curve"


if __name__ == "__main__":
    main()
