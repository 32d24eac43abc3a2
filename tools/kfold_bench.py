#!/usr/bin/env python
"""The per-round small-set test's K-fold accuracy (insightface's eval/verification.py test() -> evaluate() ->
calculate_roc, 10 folds on np.arange(0, 4, 0.01)) on two paths:

  gpu    fedfr_b200.kfold_accuracy on CUDA tensors (pfc_kfold_accuracy: four launches, no host synchronisation);
  host   the numpy + sklearn recipe verbatim (tests/kfold_oracle.py), on numpy arrays already on the host, as FedFR
         runs it once the embeddings have been copied back.

The GPU path is timed with CUDA events over --steps calls after --warmup calls, at the LFW shape (6,000 pairs) and at
1,000,000 pairs (E = 512, with flipped embeddings: 2 x 4 GB of fp32 rows, read once from HBM per call).  The host
recipe is timed with a wall clock over --host-runs runs at the LFW shape only.  The same seeded data feeds both, and
the run reports whether the GPU's outputs equal the recipe's: exactly on the GPU's distances, and on the recipe's own
float32 distances (with the number of pairs within 1e-6 of a grid threshold, which may bin differently).  The card's
name and power limit are read in the same run.  Prints one JSON object (and writes it to --out).

usage: python tools/kfold_bench.py [--steps 50] [--warmup 5] [--host-runs 3] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

E = 512
SHAPES = [6000, 1_000_000]                            # pairs: LFW / AgeDB-30, and a large synthetic set


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def make_data(P, dev):
    """Seeded embeddings on the device: the second row of a pair mixes the first with noise, genuine pairs more."""
    g = torch.Generator(device=dev).manual_seed(P)
    y = torch.rand(P, generator=g, device=dev) < 0.5
    base = torch.randn(P, E, generator=g, device=dev)
    other = torch.randn(P, E, generator=g, device=dev)
    mix = torch.where(y, 0.3 + 0.6 * torch.rand(P, generator=g, device=dev), 0.4 * torch.rand(P, generator=g, device=dev))
    emb = torch.empty(2 * P, E, device=dev)
    emb[0::2] = base
    emb[1::2] = mix[:, None] * base + (1 - mix[:, None]) * other
    del base, other
    flip = emb + 0.3 * torch.randn(2 * P, E, generator=g, device=dev)
    return emb, flip, y


def time_gpu(F, emb, flip, y, steps, warmup):
    for _ in range(warmup):
        out = F.kfold_accuracy(emb, y, flipped=flip)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = F.kfold_accuracy(emb, y, flipped=flip)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, out


def main():
    import __graft_entry__ as G
    import kfold_oracle as KO
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--host-runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    G.build()
    import fedfr_b200 as F
    dev = torch.device("cuda:0")
    result = {"card": card(), "steps": a.steps, "warmup": a.warmup, "E": E, "nfolds": 10, "thresholds": "np.arange(0, 4, 0.01)",
              "rows": []}
    for P in SHAPES:
        emb, flip, y = make_data(P, dev)
        gpu_ms, (acc, best, tpr, fpr) = time_gpu(F, emb, flip, y, a.steps, a.warmup)
        row = {"pairs": P, "gpu_ms_per_call": round(gpu_ms, 4),
               "hbm_bytes_read": 2 * emb.numel() * 4, "accuracy_mean": float(acc.mean()),
               "accuracy_std": float(acc.std(correction=0))}
        if P == SHAPES[0]:
            e, fl, yy = emb.cpu().numpy(), flip.cpu().numpy(), y.cpu().numpy()
            host = []
            for _ in range(a.host_runs):
                h0 = time.perf_counter()
                r_acc, r_best, r_tpr, r_fpr, r_dist = KO.insightface_kfold(e, yy, fl, 10, KO.GRID)
                host.append((time.perf_counter() - h0) * 1e3)
            row["host_recipe_ms_per_call"] = round(min(host), 1)
            row["host_recipe_ms_runs"] = [round(h, 1) for h in host]
            row["gpu_speedup_vs_host_recipe"] = round(min(host) / gpu_ms, 1)
            got = [t.cpu().numpy() for t in (acc, best, tpr, fpr)]
            dist = KO.pinned_dist(e, fl)
            k_tpr, k_fpr, k_acc, k_best = KO.roc_from_dist(KO.GRID, dist, yy, 10)
            row["equal_to_recipe_on_kernel_distances"] = all(
                np.array_equal(g, w) for g, w in zip(got, (k_acc, k_best, k_tpr, k_fpr)))
            near = lambda d: (np.abs(np.asarray(d, np.float64)[:, None] - KO.GRID[None, :]) <= 1e-6).any(1)   # noqa: E731
            row["pairs_within_1e-6_of_a_threshold"] = int((near(dist) | near(r_dist)).sum())
            row["same_bins_as_recipe"] = bool(np.array_equal(KO.pinned_bins(dist, KO.GRID), KO.pinned_bins(r_dist, KO.GRID)))
            row["equal_to_recipe_on_its_own_distances"] = all(
                np.array_equal(g, w) for g, w in zip(got, (r_acc, r_best, r_tpr, r_fpr)))
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
        del emb, flip, y
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
