"""Kernel-by-kernel bring-up on a real B200 (developer tool, not a test): every stage runs in its own
subprocess with a timeout so one trap/hang does not poison the rest.  Usage:

    python tools/gpu_bringup.py            # all stages
    python tools/gpu_bringup.py fwd_tc     # one stage
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAGES = ["rows", "sample", "fedavg", "check", "fwd_tc", "grad_tc", "bwd_tc", "bwd_tc_big", "step_tc"]


def _ref_math(x, w_hat, label, s, m):
    import torch
    z = (x.double() @ w_hat.double().t())
    rows = torch.nonzero(label >= 0, as_tuple=True)[0]
    z[rows, label[rows]] -= m
    z *= s
    return z


def stage_rows():
    import torch
    from fedfr_b200 import _native as N
    from fedfr_b200.ops_cuda import CudaOps
    dev = torch.device("cuda:0")
    ops = CudaOps(dev)
    w = torch.randn(1000, 512, device=dev) * 0.01
    w[3] = 0
    w_hat, inv = ops.normalize(w)
    ref = torch.nn.functional.normalize(w)
    print("normalize bf16 max err", float((w_hat.float() - ref).abs().max()), "inv err",
          float((inv[:3] - 1 / w[:3].norm(dim=1)).abs().max()), "zero row inv", float(inv[3]))
    ops_c = CudaOps(dev, N.PATH_CHECK)
    w_f, inv2 = ops_c.normalize(w)
    print("normalize f32 max err", float((w_f - ref).abs().max()))
    idx = torch.randperm(1000, device=dev)[:100].sort()[0]
    mom = torch.randn_like(w)
    sw, sm = ops.gather_rows2(w, mom, idx)
    print("gather exact", bool((sw == w[idx]).all() and (sm == mom[idx]).all()))
    w2, m2 = w.clone(), mom.clone()
    ops.scatter_rows2(w2, m2, idx, sw * 2, sm * 3)
    wr, mr = w.clone(), mom.clone()
    wr[idx] = sw * 2
    mr[idx] = sm * 3
    print("scatter exact", bool((w2 == wr).all() and (m2 == mr).all()))
    x = torch.randn(300, 512, device=dev)
    print("cast exact", bool((ops.cast_features(x) == x.to(torch.bfloat16)).all()))


def stage_sample():
    import torch
    from fedfr_b200.ops_cuda import CudaOps
    dev = torch.device("cuda:0")
    ops = CudaOps(dev)
    torch.manual_seed(0)
    for (nl, k, nlab, quant) in [(1000, 100, 64, 0), (250000, 25000, 4096, 0), (5000, 500, 512, 64), (300, 30, 64, 0), (77, 0, 16, 0),
                                 (100000, 10000, 512, 1024)]:
        lab = torch.randint(-1, nl, (nlab,), device=dev)
        if nl == 300:
            lab = (torch.randint(0, 60, (nlab,), device=dev) * 5)
        perm = torch.rand(nl, device=dev)
        if quant:
            perm = torch.floor(perm * quant) / quant       # force ties at the threshold
        # reference (torch CUDA ops, exactly partial_fc.py:94-104)
        tl = lab.clone()
        pos = torch.unique(tl[tl >= 0], sorted=True)
        p2 = perm.clone()
        if k - pos.numel() >= 0:
            p2[pos] = 2.0
            ref_idx = torch.topk(p2, k=k)[1].sort()[0]
        else:
            ref_idx = pos
        ref_lab = tl.clone()
        ref_lab[tl >= 0] = torch.searchsorted(ref_idx, tl[tl >= 0])
        mine_lab = lab.clone()
        idx = ops.sample(mine_lab, perm.clone(), k)
        ok_i = idx.shape == ref_idx.shape and bool((idx == ref_idx).all())
        ok_l = bool((mine_lab == ref_lab).all())
        print(f"sample nl={nl} k={k} nlab={nlab} quant={quant}: n_index={idx.numel()} (ref {ref_idx.numel()}) index_exact={ok_i} labels_exact={ok_l}")
        if not ok_i and idx.shape == ref_idx.shape:
            d = torch.nonzero(idx != ref_idx).flatten()
            print("   first diffs", d[:5].tolist(), idx[d[:5]].tolist(), ref_idx[d[:5]].tolist())


def stage_fedavg():
    import torch
    import fedfr_b200
    dev = torch.device("cuda:0")
    torch.manual_seed(1)
    K = 7
    shapes = {"a": (64, 3, 3, 3), "b": (64,), "c": (), "d": (1000, 513), "e": (5,)}
    models = []
    for i in range(K):
        sd = {k: torch.randn(v, device=dev) for k, v in shapes.items()}
        sd["cnt"] = torch.tensor(1000 * i + 3, device=dev)
        models.append(sd)
    weights = [6000 + 37 * i for i in range(K)]
    out = fedfr_b200.FedPavg(models, weights)
    wn = [w / sum(weights) for w in weights]
    for k in models[0]:
        tmp = 0
        for i in range(K):
            tmp += wn[i] * models[i][k]
        print("fedavg", k, tuple(out[k].shape), out[k].dtype, "bit-exact vs torch sequential:", bool((out[k] == tmp).all()))
    fcs = [torch.randn(600, 512, device=dev) for _ in range(K)]
    old = torch.randn(600, 512, device=dev)
    r = fedfr_b200.FedAvg_on_FC(old, fcs, weights, 0.7)
    aggr = fcs[0].clone() * wn[0]
    for i in range(1, K):
        aggr += fcs[i] * wn[i]
    ref = (1 - 0.7) * old + 0.7 * aggr
    print("fedavg_on_fc bit-exact:", bool((r == ref).all()), float((r - ref).abs().max()))


def _step_inputs(B, C, E, dev, seed=0):
    import torch
    torch.manual_seed(seed)
    x = torch.nn.functional.normalize(torch.randn(B, E, device=dev))
    w = torch.randn(C, E, device=dev) * 0.01
    label = torch.randint(0, C, (B,), device=dev)
    label[::7] = -1
    return x, w, label


def _check_fwd_bwd(path, B, C, E, s=64.0, m=0.4, inspect_g=False):
    import torch
    from fedfr_b200 import _native as N
    from fedfr_b200.ops_cuda import CudaOps
    dev = torch.device("cuda:0")
    ops = CudaOps(dev, path)
    x, w, label = _step_inputs(B, C, E, dev)
    w_hat, inv = ops.normalize(w)
    x_hat = ops.cast_features(x)
    xr, wr = x_hat.double(), w_hat.double()          # reference sees the same rounded operands
    z = _ref_math(xr, wr, label, s, m)
    M = z.max(dim=1)[0]
    S = torch.exp(z - M[:, None]).sum(dim=1)
    stats = ops.fwd_stats(x_hat, w_hat, label, s, m)
    torch.cuda.synchronize()
    rows = torch.nonzero(label >= 0, as_tuple=True)[0]
    tz = torch.zeros(B, dtype=torch.float64, device=dev)
    tz[rows] = z[rows, label[rows]]
    lse_ref = M + torch.log(S)
    lse = stats[:, 0].double() + torch.log(stats[:, 1].double())
    print(f"  fwd: max|lse err| {float((lse - lse_ref).abs().max()):.3e}  max|M err| {float((stats[:,0].double()-M).abs().max()):.3e} "
          f"max|target err| {float((stats[:,2].double()-tz).abs().max()):.3e}")
    row_max, row_sum, loss = ops.finalize(stats.unsqueeze(0))
    p = torch.exp(z - M[:, None]) / S[:, None]
    pt = torch.zeros(B, dtype=torch.float64, device=dev)
    pt[rows] = p[rows, label[rows]]
    loss_ref = -(pt.clamp_min(1e-30).log().mean())
    print(f"  loss {float(loss):.6f} ref {float(loss_ref):.6f}")
    g = p.clone()
    g[rows, label[rows]] -= 1
    g *= s / B
    dx_ref = g @ wr
    dwh = g.t() @ xr
    dw_ref = (dwh - wr * (wr * dwh).sum(1, keepdim=True)) * inv.double()[:, None]
    dw = torch.full((C, E), 7.0, device=dev)
    dx = ops.bwd(x_hat, w_hat, inv, label, row_max, row_sum, s, m, 1.0 / B, dw, False)
    torch.cuda.synchronize()

    def rel(a, b):
        return float((a.double() - b).norm() / b.norm())
    if inspect_g and path == N.PATH_TENSOR:
        ws = ops._ws["bwd"]
        off = (-ws.data_ptr()) % 1024
        ldg = (C + 255) // 256 * 256
        n_rb = (B + 127) // 128
        # blocked scratch: [ldg / 64][n_rb][128 rows][64 classes]
        gbuf = ws[off: off + n_rb * 128 * ldg * 2].view(torch.bfloat16).view(ldg // 64, n_rb, 128, 64)
        gbuf = gbuf.permute(1, 2, 0, 3).reshape(n_rb * 128, ldg)[:B, :C]
        print(f"  G: rel err {rel(gbuf, g):.3e}  max|G| ref {float(g.abs().max()):.3e}")
        g_used = gbuf.double()
        print(f"  dx vs G-from-kernel: {rel(dx, g_used @ wr):.3e}")
        dwh2 = g_used.t() @ xr
        dw2 = (dwh2 - wr * (wr * dwh2).sum(1, keepdim=True)) * inv.double()[:, None]
        print(f"  dw vs G-from-kernel: {rel(dw, dw2):.3e}")
    print(f"  bwd: dx rel err {rel(dx, dx_ref):.3e}   dw rel err {rel(dw, dw_ref):.3e}   (|dx| {float(dx_ref.norm()):.3e} |dw| {float(dw_ref.norm()):.3e})")
    if rel(dx, dx_ref) > 5e-2:
        print("  dx sample", dx[0, :6].tolist(), "\n  ref      ", dx_ref[0, :6].tolist())
    if rel(dw, dw_ref) > 5e-2:
        j = int(label[1]) if int(label[1]) >= 0 else int(label[2])
        print("  dw sample row", j, dw[j, :6].tolist(), "\n  ref      ", dw_ref[j, :6].tolist())
    # accumulate path
    dw_acc = torch.ones((C, E), device=dev)
    ops.bwd(x_hat, w_hat, inv, label, row_max, row_sum, s, m, 1.0 / B, dw_acc, True)
    torch.cuda.synchronize()
    print(f"  accumulate: rel err {rel(dw_acc - 1.0, dw_ref):.3e}")


def stage_check():
    from fedfr_b200 import _native as N
    for (B, C, E) in [(16, 200, 512), (100, 1000, 128), (130, 333, 64)]:
        print(f"check mode B={B} C={C} E={E}")
        _check_fwd_bwd(N.PATH_CHECK, B, C, E)


def stage_fwd_tc():
    import torch
    from fedfr_b200 import _native as N
    from fedfr_b200.ops_cuda import CudaOps
    dev = torch.device("cuda:0")
    for bn in (128, 256):
        N.check(N.lib.pfc_set_logits_tile(bn), "set tile")
        for (B, C, E) in [(128, 256, 64), (128, 512, 512), (100, 1000, 128), (512, 40000, 512), (300, 777, 256)]:
            ops = CudaOps(dev, N.PATH_TENSOR)
            x, w, label = _step_inputs(B, C, E, dev)
            w_hat, inv = ops.normalize(w)
            x_hat = ops.cast_features(x)
            z = _ref_math(x_hat, w_hat, label, 64.0, 0.4)
            M = z.max(dim=1)[0]
            S = torch.exp(z - M[:, None]).sum(dim=1)
            stats = ops.fwd_stats(x_hat, w_hat, label, 64.0, 0.4)
            torch.cuda.synchronize()
            lse = stats[:, 0].double() + torch.log(stats[:, 1].double())
            rows = torch.nonzero(label >= 0, as_tuple=True)[0]
            tz = torch.zeros(B, dtype=torch.float64, device=dev)
            tz[rows] = z[rows, label[rows]]
            print(f"fwd_tc bn={bn} B={B} C={C} E={E}: max|lse err| {float((lse - (M + torch.log(S))).abs().max()):.3e} "
                  f"max|M err| {float((stats[:,0].double()-M).abs().max()):.3e} max|tz err| {float((stats[:,2].double()-tz).abs().max()):.3e}", flush=True)


def stage_grad_tc():
    from fedfr_b200 import _native as N
    for (B, C, E) in [(128, 256, 64), (128, 512, 512), (100, 1000, 128)]:
        print(f"tensor path B={B} C={C} E={E}", flush=True)
        _check_fwd_bwd(N.PATH_TENSOR, B, C, E, inspect_g=True)


def stage_bwd_tc():
    from fedfr_b200 import _native as N
    for (B, C, E) in [(300, 777, 256), (512, 5000, 512), (256, 3000, 512)]:
        print(f"tensor path B={B} C={C} E={E}", flush=True)
        _check_fwd_bwd(N.PATH_TENSOR, B, C, E, inspect_g=True)


def stage_bwd_tc_big():
    from fedfr_b200 import _native as N
    N.lib.pfc_set_chunk_mb(16)                 # force several chunks
    try:
        print("tensor path B=512 C=40000 E=512 (multi-chunk)", flush=True)
        _check_fwd_bwd(N.PATH_TENSOR, 512, 40000, 512)
    finally:
        N.lib.pfc_set_chunk_mb(0)


def stage_step_tc():
    import __graft_entry__ as g
    g.smoke()


def main():
    if len(sys.argv) > 1 and sys.argv[1].startswith("--run="):
        globals()["stage_" + sys.argv[1][6:]]()
        return
    stages = sys.argv[1:] or STAGES
    for s in stages:
        print(f"===== {s} =====", flush=True)
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), f"--run={s}"], timeout=300, cwd=ROOT)
            print(f"===== {s}: exit {r.returncode}", flush=True)
        except subprocess.TimeoutExpired:
            print(f"===== {s}: TIMEOUT", flush=True)


if __name__ == "__main__":
    main()
