#!/usr/bin/env python
"""One step of the personalised head (client.py:382,393: the converter, BCE_module's cosine head, 10 * BCE_loss, and the
backward) on three paths, at FedFR's shapes:

  reference  client.BCE_module.forward (client.py:45-58) and losses.BCE_loss (losses.py:4-15) written out in eager
             PyTorch fp32: two normalisations, the matmul, the [B, C + 1] bool scatter, masked g_func / margin writes,
             the bias, and the loss's in-place masked edits (each boolean mask waits for the device);
  unfused    fedfr_b200.BCE_module (one forward and one backward launch) with the reference's BCE_loss on its logits;
  fused      fedfr_b200.BCE_module.loss (pfc_bce_loss_fwd / pfc_bce_loss_bwd: no logits, no host synchronisation).

For each path: CUDA-event time per step over --steps steps after --warmup steps, the host wall time per step over the
same window (ending in a device synchronise), and the GPU operations per step counted by torch.profiler in a separate
short run.  The card's name and power limit are read in the same run.  Prints one JSON object (and writes it to --out).

usage: python tools/bce_bench.py [--steps 500] [--warmup 50] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(256, 100, 512, 3), (64, 300, 512, 3)]      # (B, C, E, t): a client batch, a client's identities, E = 512
M, R = 0.4, 30.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def reference_bce_loss(logits, gts, lam=0.7, r=30.0):
    logits[gts] = (lam / r) * torch.log(1 + torch.exp(-1 * logits[gts]) + 1e-8)
    logits[~gts] = ((1 - lam) / r) * torch.log(1 + torch.exp(1 * logits[~gts]) + 1e-8)
    return torch.mean(torch.sum(logits, dim=1))


class ReferenceHead(object):
    """client.BCE_module's forward in eager PyTorch (parameters shared with the fedfr_b200 module under test)."""

    def __init__(self, mod):
        self.mod = mod

    def __call__(self, x, labels):
        import torch.nn.functional as F
        mod, C = self.mod, self.mod.n_class
        feat = mod.converter(x)
        cosine = torch.matmul(F.normalize(feat), F.normalize(mod.weight).t())
        tmp = labels.clone()
        tmp[tmp >= C] = C
        gt = torch.zeros(labels.shape[0], C + 1, dtype=torch.bool, device=x.device)
        gt[torch.arange(labels.shape[0], device=x.device), tmp] = True
        gt = gt[:, :-1]
        logits = torch.zeros_like(cosine)
        logits[gt] = mod.r * (mod.g_func(cosine[gt]) - mod.m)
        logits[~gt] = mod.r * (mod.g_func(cosine[~gt]) + mod.m)
        return logits + mod.bias[None, :], gt


def main():
    import __graft_entry__ as G
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    G.build()
    import fedfr_b200
    dev = torch.device("cuda:0")
    result = {"card": card(), "steps": a.steps, "warmup": a.warmup, "rows": []}
    for B, C, E, t in SHAPES:
        g = torch.Generator().manual_seed(B * C)
        mod = fedfr_b200.BCE_module(E, C, 1, m=M, r=R, t=t).to(dev)
        with torch.no_grad():
            mod.weight.copy_(torch.randn(C, E, generator=g) * 0.01)
            mod.bias.copy_(torch.randn(C, generator=g) * 0.1)
        x0 = torch.randn(B, E, generator=g).to(dev)
        y = torch.randint(0, C + C // 3, (B,), generator=g).to(dev)
        ref = ReferenceHead(mod)
        paths = {"reference": lambda x: 10 * reference_bce_loss(*ref(x, y)),
                 "unfused": lambda x: 10 * reference_bce_loss(*mod(x, y)),
                 "fused": lambda x: 10 * mod.loss(x, y)}
        row = {"B": B, "C": C, "E": E, "t": t}
        for name, fn in paths.items():
            x = x0.clone().requires_grad_(True)

            def step():
                mod.zero_grad(set_to_none=True)
                x.grad = None
                loss = fn(x)
                loss.backward()
                return loss

            for _ in range(a.warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0 = time.perf_counter()
            e0.record()
            for _ in range(a.steps):
                loss = step()
            e1.record()
            torch.cuda.synchronize()
            host_ms = (time.perf_counter() - h0) * 1e3 / a.steps
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    step()
                torch.cuda.synchronize()
            n_ops = sum(1 for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA) / 5
            row[name] = {"cuda_event_ms_per_step": round(e0.elapsed_time(e1) / a.steps, 4), "host_wall_ms_per_step": round(host_ms, 4),
                         "gpu_ops_per_step": n_ops, "loss": float(loss)}
        row["fused_speedup_vs_reference"] = round(row["reference"]["host_wall_ms_per_step"] / row["fused"]["host_wall_ms_per_step"], 2)
        row["fused_speedup_vs_unfused"] = round(row["unfused"]["host_wall_ms_per_step"] / row["fused"]["host_wall_ms_per_step"], 2)
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
