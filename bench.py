#!/usr/bin/env python
"""bench.py -- PartialFC CosFace fwd+bwd throughput (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5                     # this repo's CUDA path
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1     # the reference algorithm on host cores
    torchrun ... bench.py --gpus N ...                                 # class-sharded, one rank per GPU

A "step" is one ``PartialFC.forward_backward`` (prepare -> return: weight normalisation, logits GEMM +
CosFace + softmax statistics, loss, backward to the feature gradient and the centre-shard gradient, all
collectives) on a batch of 512 synthetic 512-d embeddings per GPU against 1M classes sharded over the N
GPUs (BASELINE.json configs[2]).  ``optimizer.step()`` / ``update()`` are outside the step (SURVEY 8d).

Prints ONE JSON line (rank 0).  value = whole-job samples/s with inputs resident in HBM; e2e = the same
through the public API with pinned HOST inputs and a device->host read of the result inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# Rank 0 prints ONE JSON line on stdout.  NCCL writes its version banner to file descriptor 1 when a communicator is
# created, so everything but that line is sent to stderr: fd 1 is pointed at fd 2 for the whole run and the JSON line is
# written to the saved original stdout.
_REAL_STDOUT = None


def _quiet_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)

WORKLOADS = {
    # name: (batch per GPU, classes (global), emb, sample_rate)
    "c3": (512, 1_000_000, 512, 1.0),
    "c2": (512, 100_000, 512, 1.0),
    "c4": (512, 2_000_000, 512, 0.1),
}
METRIC = "PartialFC CosFace fwd+bwd samples/s"
S, M = 64.0, 0.4
# --dump-outputs keeps the files small enough to compare two builds (64 MB at most): a fixed sample of the outputs that are
# too large to store whole -- rows of the class-shard gradient (split over the ranks), elements of the averaged model (c5)
DUMP_ROWS = 8192
DUMP_ELEMS = 4 << 20


def sample_index(n, k, seed=0):
    """Sorted indices of a fixed, seeded sample of k of 0..n-1 (all of them when n <= k), as an int64 tensor."""
    import numpy as np
    import torch
    if n <= k:
        return torch.arange(n)
    return torch.from_numpy(np.sort(np.random.default_rng(seed).choice(n, k, replace=False)))


def dump_outputs(path, arrays):
    """Each tensor of ``arrays`` (name -> tensor) as path/<name>.npy: float32, float64 for integer data."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(path, name + ".npy"), (t.float() if t.is_floating_point() else t.double()).numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML every ~5 ms while the timed region runs."""

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.mx, self.stop_flag, self.err = index, [], set(), None, False, None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            uuid = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            except Exception:
                pass
            h = None
            if uuid:
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
                except Exception:
                    h = None
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.nv, self.h = nv, h
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception as e:           # noqa: BLE001
            self.err = repr(e)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv, h = self.nv, self.h
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception as e:       # noqa: BLE001
                self.err = repr(e)
                return
            time.sleep(0.005)

    def stop(self):
        self.stop_flag = True
        if self.err and not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["nvml unavailable: " + self.err]}
        self.t.join(timeout=1.0)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons), "samples": len(sm)}


def oracle_step_time(B, C_sample, E, steps, warmup, threads):
    """Reference algorithm (oracle port of partial_fc.py:130-176 + losses.py:23-29) on the host cores."""
    import torch
    from oracle import partial_fc_oracle as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(100)
    x = torch.nn.functional.normalize(torch.randn(B, E, generator=g))
    y = torch.randint(0, C_sample, (B,), generator=g)
    w = torch.randn(C_sample, E, generator=g) * 0.01
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.forward_backward([x], [y], [w], C_sample, S, M)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return sum(times) / len(times)


def reference_cpu_steps(B, C, E, sr, steps, warmup, threads):
    """Per-step seconds of the reference's CPU path for one (B, C, sr) configuration at world size 1: the UNMODIFIED
    ``partial_fc.PartialFC.forward_backward`` (baseline/_ref, copied by build() from /root/reference) when it is present,
    else the oracle port.  Returns (times, kind)."""
    from oracle import reference_runner as R
    if R.available():
        times, _ = R.time_steps("cpu", B, C, E, sr, S, M, steps, warmup, threads=threads)
        return times, "reference"
    Cs = int(C * sr) if sr < 1 else C
    t = oracle_step_time(B, Cs, E, steps, warmup, threads)
    return [t] * steps, "port"


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, same metric and
    config (rank 0 only; the other ranks exit without work).  N = 1: the full configuration, every one of the --steps
    timed.  N > 1: one rank's batch (B rows) of the B*N-row job against all classes -- the CPU cost is linear in rows, so
    whole-job samples/s is the same number; the sample is stated in the line."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    if args.workload == "c5":
        raise SystemExit("--impl reference times the PartialFC path (c2/c3/c4); the FedAvg CPU baseline is the cpu_baseline of --workload c5")
    B, C, E, sr = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    times, kind = reference_cpu_steps(B, C, E, sr, args.steps, args.warmup, threads)
    t = sum(times) / len(times)
    ms = t * 1e3
    val = B / t
    what = "unmodified partial_fc.PartialFC.forward_backward + losses.CosFace (baseline/_ref) on CPU, gloo world size 1" if kind == "reference" \
        else "oracle port of PartialFC.forward_backward (the reference files are not on this box)"
    sample = f"{what}; B={B}, all {C} classes, sample_rate={sr}, every step at full size"
    if args.gpus > 1:
        sample += f"; one rank's {B} rows of the {B * args.gpus}-row global batch per step (cost is linear in rows: same samples/s)"
    cpu = {"value": val, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind, "sample": sample}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: class-sharded PartialFC CosFace fwd+bwd, B={B}/GPU, {C} classes over {args.gpus} GPU(s), E={E}, "
                                   f"sample_rate={sr}, s={S}, m={M}"},
            "cpu_baseline": cpu, "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


def iresnet50_shapes():
    """(name, shape, is_float) with the layout of the reference's iresnet50 state_dict (backbones/iresnet.py:60-204, layers 3,4,14,3):
    475 tensors, 43,629,071 elements, 79 of them int64 num_batches_tracked scalars (SURVEY 8a row a9)."""
    out = []

    def bn(p, c):
        out.extend([(p + ".weight", (c,), True), (p + ".bias", (c,), True), (p + ".running_mean", (c,), True), (p + ".running_var", (c,), True),
                    (p + ".num_batches_tracked", (), False)])
    out.append(("conv1.weight", (64, 3, 3, 3), True))
    bn("bn1", 64)
    out.append(("prelu.weight", (64,), True))
    inpl = 64
    for li, (planes, blocks) in enumerate(zip((64, 128, 256, 512), (3, 4, 14, 3)), 1):
        for b in range(blocks):
            p = f"layer{li}.{b}"
            bn(p + ".bn1", inpl)
            out.append((p + ".conv1.weight", (planes, inpl, 3, 3), True))
            bn(p + ".bn2", planes)
            out.append((p + ".prelu.weight", (planes,), True))
            out.append((p + ".conv2.weight", (planes, planes, 3, 3), True))
            bn(p + ".bn3", planes)
            if b == 0:
                out.append((p + ".downsample.0.weight", (planes, inpl, 1, 1), True))
                bn(p + ".downsample.1", planes)
            inpl = planes
    bn("bn2", 512)
    out.append(("fc.weight", (512, 512 * 7 * 7), True))
    out.append(("fc.bias", (512,), True))
    bn("features", 512)
    out.append(("converter.weight", (512, 512), True))        # the transformation layer (client.py:29-36), BASELINE configs[4]
    out.append(("converter.bias", (512,), True))
    return out


def run_fedavg(args):
    """--workload c5: server.py FedPavg over 40 client state_dicts (iresnet50 + transformation layer), BASELINE configs[4].
    value = algorithmic GB/s ((K+1) * N * 4 bytes per call) of the public ``FedPavg`` call with the clients resident in HBM as
    ``FlatStateDict``s (one flat buffer per client, ``fedfr_b200.flatten_state_dict``); the plain dict-of-477-tensors call is
    timed beside it.  Clients are sharded over the ranks (K/W each) and the partial sums meet in one all-reduce."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import __graft_entry__ as G
    G.build()
    import fedfr_b200
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    K = 40
    shapes = iresnet50_shapes()
    mine = list(range(rank, K, world))
    torch.manual_seed(100)
    base = {n: (torch.randn(sh, device=dev) if f else torch.zeros(sh, dtype=torch.int64, device=dev)) for n, sh, f in shapes}
    gens = {i: torch.Generator(device=dev).manual_seed(1000 + i) for i in mine}          # client i is the same tensor on any rank layout
    models = [{n: (v + 0.01 * torch.randn(v.shape, device=dev, generator=gens[i])) if v.dtype == torch.float32 else v + i for n, v in base.items()}
              for i in mine]
    flats = [fedfr_b200.flatten_state_dict(m) for m in models]
    weights = [6000 + 37 * i for i in mine]
    n_elem = sum(v.numel() for v in base.values())
    alg_bytes = (K + 1) * n_elem * 4.0

    def call(clients):
        if world == 1:
            return fedfr_b200.FedPavg(clients, weights)
        return fedfr_b200.FedPavg_sharded(clients, weights)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    for _ in range(max(args.warmup, 3)):
        call(flats)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    from fedfr_b200 import _native as N
    last = [None]

    def call_flats():
        last[0] = call(flats)

    l0 = N.lib.pfc_launch_count()
    ms = timed(call_flats, args.steps)
    launches = N.lib.pfc_launch_count() - l0
    if args.dump_outputs and rank == 0:          # the averaged model is the same on every rank
        # a sample of the model's tensors laid end to end (key order), gathered tensor by tensor: no copy of the whole model
        vals = list(last[0].values())
        starts = np.cumsum([0] + [v.numel() for v in vals])
        idx = sample_index(int(starts[-1]), DUMP_ELEMS)
        cut = np.searchsorted(idx.numpy(), starts)
        picked = [v.reshape(-1)[(idx[a:b] - int(s)).to(dev)] for v, s, a, b in zip(vals, starts, cut[:-1], cut[1:]) if b > a]
        dump_outputs(args.dump_outputs, {"fedpavg_sample_index": idx, "fedpavg_sample": torch.cat(picked)})
        del vals, picked
    last[0] = None
    # the C-ABI call alone (table upload + the one kernel), re-launched from the tables the last call staged
    from fedfr_b200 import fedavg as FA
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(args.steps):
        FA.relaunch_last()
    k1.record()
    torch.cuda.synchronize()
    kernel_ms = k0.elapsed_time(k1) / args.steps
    clocks = sampler.stop() if sampler else None
    for _ in range(2):
        call(models)
    ms_dict = timed(lambda: call(models), max(args.steps // 2, 2))

    # parity (driver-visible: exit 3 on failure): W = 1 bit-exact against the reference's own loop order in torch fp32 on the
    # device (mul, then add, client order; 0 + first term) and flat == dict path; W > 1 against an fp64 sum, 1e-6, same bits on all ranks
    out = call(flats)
    out_d = call(models)
    names = [n for n, _, _ in shapes]
    probe = [max(names, key=lambda n: base[n].numel()), "conv1.weight", "bn1.num_batches_tracked", "converter.weight", "features.running_var"]
    tot_w = float(sum(6000 + 37 * i for i in range(K)))
    parity = {"keys_checked": probe, "world": world}
    ok = all(out[n].dtype == torch.float32 for n in names)
    if world == 1:
        wn = [w / tot_w for w in weights]
        exact = True
        for n in probe:
            ref = 0
            for wi, m in zip(wn, models):
                ref = ref + wi * m[n]                         # python_float * tensor, then add: server.py:31-32
            exact = exact and bool(torch.equal(out[n], ref)) and bool(torch.equal(out_d[n], ref))
        parity["bit_exact_vs_reference_order"] = exact
        ok = ok and exact
    else:
        worst = 0.0
        same = True
        for n in probe:
            part = torch.zeros_like(base[n], dtype=torch.float64)
            for i, m in zip(mine, models):
                part += ((6000 + 37 * i) / tot_w) * m[n].double()
            dist.all_reduce(part)
            worst = max(worst, float((out[n].double() - part).norm() / part.norm().clamp_min(1e-30)))
            g = [torch.empty_like(out[n]) for _ in range(world)]
            dist.all_gather(g, out[n].contiguous())
            same = same and all(bool(torch.equal(g[0], t)) for t in g)
        parity["max_rel_err_vs_fp64"] = worst
        parity["identical_on_all_ranks"] = same
        ok = ok and worst < 1e-6 and same
    if world > 1:
        flag = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item() > 0)
    parity["ok_all_ranks"] = ok
    del out, out_d

    # end to end: every client starts as a FlatStateDict in pinned HOST memory (where FedFR keeps the uploads, client.py:469),
    # one H2D copy per client buffer, result read back to the host; all K/W clients of this rank, K in total
    host_flats = [fedfr_b200.flatten_state_dict(m, device="cpu", pin_memory=True) for m in models]
    torch.cuda.synchronize()

    def e2e_call():
        o = call(host_flats)
        return o.flat_f32.cpu() if hasattr(o, "flat_f32") else {n: v.cpu() for n, v in o.items()}

    e2e_call()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e2e_call()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if not ok:
            sys.exit(3)
        return
    peaks = load_peaks()
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import reference_runner as R
        torch.set_num_threads(os.cpu_count() or 1)
        n_cpu = 8
        cm = [{n: v.cpu() for n, v in m.items()} for m in models[:n_cpu]]
        try:
            ref_fedpavg, _ = R.load_server_functions()
            kind, what = "reference", "unmodified server.FedPavg (baseline/_ref/server.py:25-34) on CPU tensors"
        except FileNotFoundError:
            from oracle import partial_fc_oracle as O
            ref_fedpavg, kind, what = (lambda ms_, ws_: O.fedpavg([{n: v.numpy() for n, v in m.items()} for m in ms_], ws_)), "port", "oracle port of server.FedPavg"
        t0 = time.perf_counter()
        ref_fedpavg(cm, weights[:n_cpu])
        t = time.perf_counter() - t0
        cpu = {"value": (n_cpu + 1) * n_elem * 4.0 / t / 1e9, "unit": "GB/s", "cores": torch.get_num_threads(), "kind": kind,
               "sample": f"{what}, {n_cpu} of the {K} clients (incl. its deepcopy of client 0)"}
    line = {"metric": "FedPavg weighted average, algorithmic GB/s ((K+1)*N*4 bytes)", "value": gbs, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"c5: FedPavg of {K} client state_dicts (iresnet50 475 tensors + transformation layer, {n_elem} elements each) held as "
                                   f"FlatStateDicts, clients sharded over {world} GPU(s)" + (", one all-reduce of the flat partial sum" if world > 1 else ""),
                       "l2": "inputs larger than L2 (7 GB of client tensors)"},
            "e2e": {"value": alg_bytes / e2e_s / 1e9, "unit": "GB/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": len(mine) * n_elem * 4, "d2h_bytes_per_step": n_elem * 4,
                    "sample": f"all {K} clients from pinned host memory ({len(mine)} per rank, one H2D copy per client buffer), result copied back"},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "fedavg_kernel (fedavg_weighted_sum call: table upload + one launch)",
                         "achieved": (len(mine) + 1) * n_elem * 4.0 / (kernel_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": (len(mine) + 1) * n_elem * 4.0 / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": None,
                         "ms_per_launch": kernel_ms, "peak_source": peaks["source"] + " copy bandwidth",
                         "note": "the peak is a COPY bandwidth (1 read : 1 write); this kernel reads K client buffers per buffer it writes, and an "
                                 "HBM stream with no read/write turnarounds can exceed the copy figure by a few percent (frac > 1 is not an error)"},
            "cpu_baseline": cpu, "parity": parity,
            "extras": {"dict_of_tensors_call_ms": ms_dict, "dict_of_tensors_call_gbs": alg_bytes / (ms_dict * 1e-3) / 1e9,
                       "note": "same call on plain state_dicts (K x 477 tensors): bound by per-tensor Python work"}}
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        sys.exit(3)


def run_ours(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as G
    G.build()
    import fedfr_b200
    from fedfr_b200 import _native as N

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    B, C, E, sr = WORKLOADS[args.workload]
    if args.logits_tile:
        N.check(N.lib.pfc_set_logits_tile(args.logits_tile), "pfc_set_logits_tile")
    if args.logits_pair >= 0:
        N.lib.pfc_set_logits_pair(args.logits_pair)
    if args.graph >= 0:
        N.lib.pfc_set_graph(args.graph)
    if args.chunk_mb:
        N.lib.pfc_set_chunk_mb(args.chunk_mb)
    if args.fwd_overlap:
        v = [int(t) for t in args.fwd_overlap.split(",")] + [0]
        N.lib.pfc_set_fwd_overlap(v[0], v[1])
    if args.prefetch:
        v = [int(t) for t in args.prefetch.split(",")]
        N.lib.pfc_set_prefetch(v[0], v[1], v[2])
    if args.dx_pair >= 0:
        N.lib.pfc_set_dx_pair(args.dx_pair)
    if args.dw4 >= 0:
        N.lib.pfc_set_dw4(args.dw4)
    if args.pipe:
        v = [int(t) for t in args.pipe.split(",")] + [0, 0, 0, 0]
        N.lib.pfc_set_pipeline(v[0], v[1], v[2], v[3], v[4])
    if args.prob_split:
        v = args.prob_split.split(",")
        N.lib.pfc_set_prob_split(int(v[0]), float(v[1]) if len(v) > 1 else 0.0, int(v[2]) if len(v) > 2 else -1)
    if args.dx_cluster or args.dw_cluster:
        N.lib.pfc_set_clusters(args.dx_cluster, args.dw_cluster)
    torch.manual_seed(100 + rank)
    head = fedfr_b200.PartialFC(rank, local_rank, world, B, False, fedfr_b200.CosFace(s=S, m=M), C, sample_rate=sr, embedding_size=E, prefix="/tmp")
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.1, momentum=0.9, weight_decay=5e-4)
    feats = torch.nn.functional.normalize(torch.randn(B, E, device=dev))
    label = torch.randint(0, C, (B,), device=dev)
    feats_h = feats.cpu().pin_memory()
    label_h = label.cpu().pin_memory()

    last = [None]

    def step_resident():
        head.sub_weight.grad = None                      # what optimizer.zero_grad(set_to_none=True) leaves behind
        last[0] = head.forward_backward(label, feats, opt)

    xg_h = torch.empty((B, E), dtype=torch.float32).pin_memory()
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()

    def step_e2e():
        head.sub_weight.grad = None
        f = feats_h.to(dev, non_blocking=True)           # H2D of this step's inputs from pinned host memory
        l = label_h.to(dev, non_blocking=True)
        xg, loss = head.forward_backward(l, f, opt)
        xg_h.copy_(xg, non_blocking=True)                # D2H of the step's results into pinned host memory ...
        loss_h.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()        # ... and the host waits for them every step
        return xg_h, float(loss_h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = N.lib.pfc_launch_count()
    ms_total = timed(step_resident, args.steps)
    launches = N.lib.pfc_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    ms_step = ms_total / args.steps
    if args.dump_outputs:                                # what the caller received from the last timed step
        x_grad, loss = last[0]
        grad = head.sub_weight.grad
        rows = sample_index(grad.shape[0], DUMP_ROWS // world)
        out = {"x_grad": x_grad, "loss": loss, "sub_weight_grad_rows": rows, "sub_weight_grad": grad[rows.to(dev)]}
        if head.index is not None:                       # the sampled classes (sample_rate < 1)
            out["index"] = head.index
        dump_outputs(args.dump_outputs, {(n + f"_rank{rank}" if world > 1 else n): t for n, t in out.items()})
        del x_grad, loss, grad, out
    last[0] = None

    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps) / args.steps

    # same copies, but the host reads step n's results while step n+1 is already enqueued (how a training loop that logs
    # the loss one step late behaves); reported next to the strict number, never instead of it
    pp_bufs = [(torch.empty((B, E), dtype=torch.float32).pin_memory(), torch.empty((), dtype=torch.float32).pin_memory()) for _ in range(2)]
    pp_evs = [torch.cuda.Event(), torch.cuda.Event()]
    pp_state = {"i": 0, "sink": 0.0}

    def step_e2e_lagged():
        i = pp_state["i"]
        head.sub_weight.grad = None
        f = feats_h.to(dev, non_blocking=True)
        l = label_h.to(dev, non_blocking=True)
        xg, loss = head.forward_backward(l, f, opt)
        pp_bufs[i & 1][0].copy_(xg, non_blocking=True)
        pp_bufs[i & 1][1].copy_(loss, non_blocking=True)
        pp_evs[i & 1].record()
        if i > 0:
            pp_evs[(i - 1) & 1].synchronize()
            pp_state["sink"] += float(pp_bufs[(i - 1) & 1][1])
        pp_state["i"] = i + 1

    for _ in range(2):
        step_e2e_lagged()
    ms_e2e_lagged = timed(step_e2e_lagged, args.steps) / args.steps

    # parity of this very configuration, on every rank (driver-visible: a failure makes the run exit 3): one more step,
    # checked against a chunked device-side restatement of partial_fc.py:127-174 (fedfr_b200/selfcheck.py) -- the
    # reference's fp32 arithmetic at 1e-2, the bf16-operand emulation row by row (max 1e-2, rms 1e-3), identical loss bits on all ranks
    parity = None
    if not args.no_parity:
        from fedfr_b200 import selfcheck
        head.sub_weight.grad = None
        xg_c, loss_c = head.forward_backward(label, feats, opt)
        parity = selfcheck.check_head_step(head, label, feats, xg_c, loss_c, **({} if head._ops.bwd_mode == "prob" else {"tol_rows": 2e-2, "tol_rows_rms": 1e-2}))
        del xg_c, loss_c
        torch.cuda.empty_cache()
        if not parity["ok_all_ranks"]:
            sys.stderr.write(f"[bench] PARITY FAILURE on rank {rank}: {json.dumps(parity)}\n")

    # the step either side of the path (SURVEY 8d: reported separately): optimizer.step() + update(), torch vs fused
    def opt_time(fn, n=5):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    def torch_opt():
        opt.step()
        head.update()

    def train_step_torch():
        head.sub_weight.grad = None
        head.forward_backward(label, feats, opt)
        opt.step()
        head.update()

    def train_step_fused():
        head.sub_weight.grad = None
        head.forward_backward(label, feats, opt)
        head.step(opt)

    step_resident()
    extras = {}
    try:
        opt_time(torch_opt, 2)
        extras["optimizer_step_update_torch_ms"] = opt_time(torch_opt)
        step_resident()
        opt_time(lambda: head.step(opt, prenormalize=False), 2)
        extras["optimizer_step_update_fused_ms"] = opt_time(lambda: head.step(opt, prenormalize=False))
        opt_time(train_step_torch, 2)
        extras["train_step_torch_optimizer_ms"] = opt_time(train_step_torch, 10)
        opt_time(train_step_fused, 2)
        extras["train_step_fused_optimizer_ms"] = opt_time(train_step_fused, 10)
    except Exception as e:           # noqa: BLE001  (extras never fail the bench line)
        extras["error"] = repr(e)
    head._prenorm = None
    # context: the reference's formulation (client.py:69-74 + losses.py:23-29 + F.cross_entropy, autograd) in stock PyTorch
    # eager fp32 on this same GPU, single rank only (it materialises the [B, C] logits: ~10 GB of temporaries at c3)
    if world == 1 and sr >= 1 and not args.no_cpu_baseline:
        try:
            F = torch.nn.functional
            w_ref = head.weight.detach().clone().requires_grad_(True)
            x_ref = feats.clone().requires_grad_(True)

            def torch_step():
                w_ref.grad = None
                x_ref.grad = None
                cosine = F.linear(x_ref, F.normalize(w_ref))
                onehot = torch.zeros_like(cosine).scatter_(1, label[:, None], M)
                F.cross_entropy((cosine - onehot) * S, label).backward()

            opt_time(torch_step, 2)
            extras["torch_eager_fp32_same_gpu_ms"] = opt_time(torch_step, 3)
            del w_ref, x_ref
            torch.cuda.empty_cache()
        except Exception as e:       # noqa: BLE001
            extras["torch_eager_error"] = repr(e)

    # the UNMODIFIED reference class on this same B200 in fp32 (real constructor, nccl group of one rank): context row
    if world == 1 and not args.no_cpu_baseline:
        try:
            from oracle import reference_runner as R
            if R.available():
                torch.cuda.empty_cache()
                tr, _ = R.time_steps(f"cuda:{local_rank}", B, C, E, sr, S, M, 3, 2)
                extras["reference_on_b200_ms"] = 1e3 * sum(tr) / len(tr)
                extras["reference_on_b200_note"] = "unmodified partial_fc.PartialFC.forward_backward (baseline/_ref), fp32, same GPU, wall clock around synchronised steps"
                torch.cuda.empty_cache()
        except Exception as e:       # noqa: BLE001
            extras["reference_on_b200_error"] = repr(e)

    # per-phase device times (events on the launch stream inside the library) for the roofline of the dominant kernel
    import ctypes as CT
    N.lib.pfc_profile_enable(1)
    prof_steps = min(args.steps, 5)
    for _ in range(prof_steps):
        step_resident()
    torch.cuda.synchronize()
    ms = (CT.c_float * 5)()
    cnt = (CT.c_int * 5)()
    N.lib.pfc_profile_collect(ms, cnt)
    N.lib.pfc_profile_enable(0)
    prob = head._ops.bwd_mode == "prob"
    names = (["normalize_rows(chunk 0)", "logits_prob(fwd, normalises the next chunk)", "prob_prep", "dx", "dw"] if prob else
             ["normalize_rows(chunk 0)", "logits_stats(fwd, normalises the next chunk)", "logits_grad(bwd)", "dx", "dw"])
    phase_ms = {n: ms[i] / prof_steps for i, n in enumerate(names)}
    phase_launches = {n: cnt[i] // prof_steps for i, n in enumerate(names)}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if parity is not None and not parity["ok_all_ranks"]:
            sys.exit(3)
        return

    peaks = load_peaks()
    Bt = B * world
    Cs = head.num_sample if sr < 1 else head.num_local
    gemm_flops = 2.0 * Bt * Cs * E                       # one GEMM of the three (SURVEY 8d: 6*Bt*Cs*E per step)
    gemm_phases = [names[1], "dx", "dw"] + ([] if prob else [names[2]])
    dom = max(gemm_phases, key=lambda n: phase_ms[n])
    dom_launches = max(phase_launches[dom], 1)
    dom_ms = phase_ms[dom]
    achieved = gemm_flops / (dom_ms * 1e-3) / 1e12
    # DRAM bytes of the dominant kernel per launch from the committed `ncu --set full` capture (profiles/traffic.json, c3 at N=1 only)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if world == 1 and args.workload == "c3" and os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get("prob" if prob else "recompute", {}).get(dom.split("(")[0])
        except Exception:                                 # noqa: BLE001
            traffic = None
    # HBM view of the whole step: bytes this design moves per step (DESIGN.md section 4), not the minimum any design needs.
    # Formula: every tensor counted once per kernel that touches it.  Measured (ncu --graph-profiling graph, the forward and
    # the backward graph each as one unit, profiles/traffic.json "step_graphs", c3 at N=1): 9.73 GB -- the P / w_hat tiles dx
    # and dw both read are fetched from DRAM once because the two kernels run side by side and share them through L2.
    design_bytes = (16.0 * Cs * E + 6.0 * Bt * Cs) if prob else (18.0 * Cs * E + 6.0 * Bt * Cs)
    measured_bytes = None
    if world == 1 and args.workload == "c3" and prob and os.path.exists(tpath):
        try:
            measured_bytes = json.load(open(tpath)).get("step_graphs", {}).get("step_total")
        except Exception:                                 # noqa: BLE001
            measured_bytes = None
    roof = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peaks["tflops_sustained"], "unit": "TFLOP/s",
            "frac": achieved / peaks["tflops_sustained"], "traffic": traffic,
            "peak_source": f"{peaks['source']} bf16 sustained (kernel timed inside the step loop); burst {peaks['tflops']}",
            "flops_per_launch": gemm_flops / dom_launches, "ms_per_launch": dom_ms / dom_launches, "launches_per_step": dom_launches,
            "note": "dx and dw run side by side on disjoint SM subsets (their phase times overlap); achieved = the kernel's GEMM FLOPs / its own duration",
            "phase_ms_per_step": phase_ms,
            "step_tflops": 6.0 * Bt * Cs * E / (ms_step * 1e-3) / 1e12 / 1.0,
            "step_frac_of_burst_peak_per_gpu": 6.0 * Bt * Cs * E / (ms_step * 1e-3) / 1e12 / peaks["tflops"],
            "step_hbm": {"design_bytes_per_step": design_bytes, "gbs": design_bytes / (ms_step * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"],
                         "frac": design_bytes / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "measured_dram_bytes_per_step": measured_bytes,
                         "measured_frac": None if not measured_bytes else measured_bytes / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"]},
            "backward": "stored probabilities (3 GEMMs)" if prob else "recompute (4 GEMMs)"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        times, kind = reference_cpu_steps(B, C, E, sr, 2, 1, threads)        # bounded sample: two full-size steps after one warm-up
        t = sum(times) / len(times)
        cpu = {"value": B / t, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
               "sample": ("unmodified partial_fc.PartialFC.forward_backward (baseline/_ref) on CPU" if kind == "reference" else "oracle port") +
                         f", B={B}, all {C} classes, sample_rate={sr}, 2 full-size steps after 1 warm-up"}

    line = {"metric": METRIC, "value": Bt / (ms_step * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.workload}: class-sharded PartialFC CosFace fwd+bwd, B={B}/GPU, {C} classes over {world} GPU(s), E={E}, "
                                   f"sample_rate={sr}, s={S}, m={M}",
                       "l2": "inputs larger than L2 (weight shard fp32+bf16 streamed every step)", "parallelism": f"class-shard x{world}"},
            "e2e": {"value": Bt / (ms_e2e * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": B * E * 4 + B * 8, "d2h_bytes_per_step": B * E * 4 + 4,
                    "ms_per_step": ms_e2e, "readback": "synchronous: the host waits for x_grad and the loss of every step before starting the next",
                    "lagged_readback": {"value": Bt / (ms_e2e_lagged * 1e-3), "ms_per_step": ms_e2e_lagged,
                                        "note": "same copies; step n is read back while step n+1 is already enqueued"}},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "parity": parity, "extras": extras}
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if parity is not None and not parity["ok_all_ranks"]:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS) + ["c5"])
    ap.add_argument("--logits-tile", type=int, default=0)
    ap.add_argument("--logits-pair", type=int, default=-1)
    ap.add_argument("--dx-cluster", type=int, default=0)
    ap.add_argument("--dw-cluster", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-timing parity self-check (developer runs under ncu)")
    ap.add_argument("--graph", type=int, default=-1, help="1/0: replay the backward as a cached CUDA graph (library default: 1)")
    ap.add_argument("--pipe", default="", help="backward chain pipeline: 'on,smG,smDx,smDw,ring' (e.g. 1,56,32,60,3) or 0")
    ap.add_argument("--fwd-overlap", default="", help="fused forward: 'chunks,normalize_blocks_per_sm' (e.g. 6,2)")
    ap.add_argument("--prefetch", default="", help="TMA L2 prefetch: 'logits,dx_distance,dw' (e.g. 1,6,1)")
    ap.add_argument("--dx-pair", type=int, default=-1, help="1/0: CTA-pair dx kernel")
    ap.add_argument("--dw4", type=int, default=-1, help="1/0: 4-CTA-cluster dw kernel (E = 512)")
    ap.add_argument("--prob-split", default="", help="stored-probability backward: 'dx_sms[,dw_rate[,sweep_lead]]' (SM budget of the dx kernel, dx/dw pacing)")
    ap.add_argument("--chunk-mb", type=int, default=0, help="bf16 G scratch per backward chunk in MiB (0 = library default)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step returned to DIR/<name>.npy (float32, integer data as float64; a fixed "
                         "sample of the large outputs, 64 MB at most) to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c5":
        run_fedavg(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
