#!/usr/bin/env python
"""1:N identification (fedfr_b200.mate_ranks: exact mate ranks and top-1 matches, no score matrix) on the GPU, against
the host recipe of an ijbc_all.py-style 1:N section (np.dot for the score matrix, then np.argsort per probe).

Shapes (E = 512, L2-normalised rows):
  ijbc_g1, ijbc_g2   seeded synthetic data of the IJB-C 1:N shape (oracle/identify_oracle.py ijbc_1n_like): 19,593
                     probe templates against the 1,772- and 1,759-subject galleries;
  10k_x_100k         10,000 probes against a 100,000-entry gallery.
Per shape, CUDA events over --steps calls after --warmup calls time the pfc_identify chain alone (memset + three
launches on preallocated buffers) and the public call (subject -> mate-row lookup, duplicate check, the chain, the NaN
count read back).  At the IJB-C shape the host recipe is timed with a wall clock (one run per gallery) and its ranks
and top-1 rows are compared with the GPU's: the host's float32 np.dot differs from the exact chain in the last bits, so
probes whose mate ties or nearly ties another entry may rank differently; the count of those is reported.  The card's
name and power limit are read in the same run.  Prints one JSON object (and writes it to --out).

usage: python tools/ident_bench.py [--steps 20] [--warmup 3] [--out PATH]"""
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

E = 512


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def chain_call(N, x, y, m):
    """pfc_identify on preallocated outputs and workspace -> a closure that launches it once."""
    P = x.shape[0]
    dev = x.device
    rank, top1 = (torch.empty(P, dtype=torch.int64, device=dev) for _ in range(2))
    ms, ts = (torch.empty(P, dtype=torch.float32, device=dev) for _ in range(2))
    counts = torch.empty(2, dtype=torch.int64, device=dev)
    ws = torch.empty(int(N.lib.pfc_identify_workspace_bytes(P)), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def run():
        N.check(N.lib.pfc_identify(N.ptr(x), P, N.ptr(y), y.shape[0], E, N.ptr(m), N.ptr(rank), N.ptr(ms), N.ptr(top1),
                                   N.ptr(ts), N.ptr(counts), N.ptr(ws), ws.numel(), stream), "pfc_identify")
    return run


def host_recipe(probe, gallery, mate_row):
    """The host recipe: float32 score matrix, stable argsort of each row by descending score."""
    S = np.dot(probe, gallery.T)
    order = np.argsort(-S, axis=1, kind="stable")
    rank = np.zeros(probe.shape[0], np.int64)
    mated = np.flatnonzero(mate_row >= 0)
    rank[mated] = np.argmax(order[mated] == mate_row[mated, None], axis=1) + 1
    return rank, order[:, 0]


def main():
    import __graft_entry__ as G
    from oracle import identify_oracle as IO
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    G.build()
    import fedfr_b200 as F
    from fedfr_b200 import _native as N
    from fedfr_b200.verify import mate_rows
    dev = torch.device("cuda:0")
    result = {"card": card(), "steps": a.steps, "warmup": a.warmup, "E": E, "rows": []}

    probe, p_subj, g1, g2 = IO.ijbc_1n_like(seed=0)
    shapes = [("ijbc_g1", probe, p_subj) + g1, ("ijbc_g2", probe, p_subj) + g2]
    g = torch.Generator(device=dev).manual_seed(7)
    big_g = torch.nn.functional.normalize(torch.randn(100_000, E, generator=g, device=dev), dim=1)
    big_subj = torch.arange(100_000, device=dev) * 3 + 1
    big_mate = torch.randint(0, 100_000, (10_000,), generator=g, device=dev)
    big_p = torch.nn.functional.normalize(big_g[big_mate] + 0.12 * torch.randn(10_000, E, generator=g, device=dev), dim=1)
    big_psubj = torch.where(torch.rand(10_000, generator=g, device=dev) < 0.5, big_subj[big_mate], -big_mate - 1)
    shapes.append(("10k_x_100k", big_p, big_psubj, big_g, big_subj))

    for name, pf, ps, gf, gs in shapes:
        x, xs, y, ys = (torch.as_tensor(t).to(dev).contiguous() for t in (pf, ps, gf, gs))
        m = mate_rows(xs, ys)
        P, Gn = x.shape[0], y.shape[0]
        chain_ms = timed(chain_call(N, x, y, m), a.steps, a.warmup)
        public_ms = timed(lambda: F.mate_ranks(x, xs, y, ys), a.steps, a.warmup)
        rank, ms, top1, ts = F.mate_ranks(x, xs, y, ys)
        pairs = P * Gn
        row = {"shape": name, "probes": P, "gallery": Gn, "mated": int((rank > 0).sum()),
               "chain_ms_per_call": round(chain_ms, 4), "public_ms_per_call": round(public_ms, 4),
               "pairs_per_s_chain": round(pairs / (chain_ms * 1e-3), 1),
               "rank1": float(F.cmc(rank, 1)[0]),
               "tpir_at_fpir_rank1": F.tpir_at_fpir(rank, ms, ts, (1e-2, 1e-1))}
        if name.startswith("ijbc"):
            pn, gn, mn = x.cpu().numpy(), y.cpu().numpy(), m.cpu().numpy()
            h0 = time.perf_counter()
            h_rank, h_top1 = host_recipe(pn, gn, mn)
            row["host_recipe_ms"] = round((time.perf_counter() - h0) * 1e3, 1)
            row["gpu_speedup_vs_host_recipe"] = round(row["host_recipe_ms"] / public_ms, 1)
            g_rank, g_top1 = rank.cpu().numpy(), top1.cpu().numpy()
            row["host_rank_disagreements"] = int((h_rank != g_rank).sum())
            row["host_top1_disagreements"] = int((h_top1 != g_top1).sum())
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
