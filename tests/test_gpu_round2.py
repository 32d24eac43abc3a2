"""Round-2 GPU parity tests (through the C ABI): the tensor-core kernels held ROW BY ROW to an oracle that makes their bf16
operand roundings explicit, the per-GPU shapes of multi-rank jobs on one GPU, the every-step range guard, the FedAvg
corner cases (signed zero, unaligned views, more than 64 clients, flat state dicts) and the dense margin callables."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


def _head(pkg, B, C, E, s, m, w, margin="cosface", sample_rate=1.0, world=1, rank=0):
    mg = pkg.CosFace(s=s, m=m) if margin == "cosface" else pkg.ArcFace(s=s, m=m)
    head = pkg.PartialFC(rank, 0, world, B, False, mg, C, sample_rate=sample_rate, embedding_size=E, prefix="/tmp")
    if w is not None:
        head.weight.copy_(w.to(head.device))
    head.weight_mom.zero_()
    return head


@pytest.mark.parametrize("B,C,E,s,margin", [(512, 20000, 512, 64.0, "cosface"), (300, 5000, 256, 30.0, "arcface"), (130, 700, 128, 64.0, "cosface"),
                                             (1024, 9000, 512, 64.0, "cosface")])
def test_rows_vs_bf16_oracle(pkg, B, C, E, s, margin):
    """logits2 / dx2 / dw kernels against ``oracle.forward_backward_bf16`` fed the kernel's own bf16 ``w_hat``: every row of
    ``dx`` and ``dw`` within 1e-2 (2.5 bf16 ulp: a row dominated by one or two rounded elements), the rms over the rows within 1e-3 for target and non-target rows alike --
    a whole-tensor relative L2 (the 1e-2 bf16 tolerance, still asserted) would let a ~6 % error in every non-target row of
    ``dw`` through."""
    from fedfr_b200 import selfcheck as SC
    from oracle import partial_fc_oracle as O
    g = torch.Generator().manual_seed(B + C + E)
    w = torch.randn(C, E, generator=g) * 0.01
    y = torch.randint(0, C, (B,), generator=g)
    y[1] = y[0]
    x = torch.nn.functional.normalize(torch.randn(B, E, generator=g) + 2.0 * torch.nn.functional.normalize(w[y]) * (torch.arange(B) % 4 == 0)[:, None])
    m = 0.4 if margin == "cosface" else 0.5
    head = _head(pkg, B, C, E, s, m, w, margin)
    assert head._ops.bwd_mode == "prob"
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.1, momentum=0.9)
    xg, loss = head.forward_backward(y.to(head.device), x.to(head.device), opt)
    w_hat = head._norm[0].float().cpu()
    # normalize(): the kernel's bf16 operand is within one rounding of F.normalize
    wn = torch.nn.functional.normalize(w)
    assert float(((w_hat - wn).abs() / wn.abs().clamp_min(1e-6)).max()) <= 2.0 ** -8 * 1.01
    ref = O.forward_backward_bf16([x], [y], [w], C, s, m, margin=margin, w_hats=[w_hat])
    exact = O.forward_backward([x], [y], [w], C, s, m, margin=margin)
    assert abs(float(loss) - float(ref.loss)) < 1e-4 * float(ref.loss)
    tgt = torch.zeros(C, dtype=torch.bool)
    tgt[y] = True
    dw = head.sub_weight.grad.cpu()
    groups = {"dx": (xg.cpu(), ref.x_grad[0]), "dw target rows": (dw[tgt], ref.dw[0][tgt]), "dw other rows": (dw[~tgt], ref.dw[0][~tgt])}
    for name, (got, want) in groups.items():
        assert SC._rows_err(got, want) < 1e-2, (name, SC._rows_err(got, want))
        assert SC._rows_err(got, want, rms=True) < 1e-3, (name, SC._rows_err(got, want, rms=True))
    assert SC._rel(xg.cpu(), exact.x_grad[0]) < 1e-2 and SC._rel(dw, exact.dw[0]) < 1e-2


@pytest.mark.parametrize("B,C,sr", [(4096, 125_000, 1.0), (512, 1_000_000, 1.0), (4096, 250_000, 0.1)])
def test_selfcheck_at_job_shapes(pkg, B, C, sr):
    """The per-GPU shapes the scaling run times, on one GPU: W=8 of c3 (Bt=4096, Cs=125k), c3 at W=1, and c4's rank shard
    (250k classes, 25k sampled, gathered batch 4096).  fedfr_b200.selfcheck = the check bench.py runs after its timed loops."""
    from fedfr_b200 import selfcheck as SC
    torch.manual_seed(100)
    head = _head(pkg, B, C, 512, 64.0, 0.4, None, sample_rate=sr)
    dev = head.device
    x = torch.nn.functional.normalize(torch.randn(B, 512, device=dev))
    y = torch.randint(0, C, (B,), device=dev)
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.1, momentum=0.9)
    xg, loss = head.forward_backward(y, x, opt)
    out = SC.check_head_step(head, y, x, xg, loss)
    assert out["ok"], out
    # and the check is not vacuous: a 3 % error on the non-target rows of dw only (what a global norm cannot see) fails it
    rows = torch.arange(0, head.sub_weight.shape[0], 1009, device=dev)
    head.sub_weight.grad[rows] *= 1.03
    bad = SC.check_head_step(head, y, x, xg, loss)
    assert not bad["ok"] and bad["fp32"]["dw_rel"] < 1e-2, bad


def test_range_guard_every_step(pkg):
    """Features that are in range on the first call and leave it later: the device-side flag (checked every step) must
    switch the head to the recomputing backward within two steps -- not after up to 255 -- and results must match the oracle
    from then on."""
    from oracle import partial_fc_oracle as O
    B, C, E, s = 128, 3000, 256, 64.0
    g = torch.Generator().manual_seed(7)
    w = torch.randn(C, E, generator=g) * 0.01
    y = torch.randint(0, C, (B,), generator=g)
    x = torch.nn.functional.normalize(torch.randn(B, E, generator=g))
    head = _head(pkg, B, C, E, s, 0.4, w)
    dev = head.device
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.0)
    for _ in range(3):
        head.sub_weight.grad = None
        head.forward_backward(y.to(dev), x.to(dev), opt)
    assert head._ops.bwd_mode == "prob"
    big = x * 3.0                                                      # s |x| = 192 nats
    steps_to_switch = None
    for k in range(4):
        head.sub_weight.grad = None
        xg, loss = head.forward_backward(y.to(dev), big.to(dev), opt)
        if head._ops.bwd_mode == "recompute" and steps_to_switch is None:
            steps_to_switch = k
    assert steps_to_switch is not None and steps_to_switch <= 2, steps_to_switch
    ref = O.forward_backward([big], [y], [w], C, s, 0.4)
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    assert abs(float(loss) - float(ref.loss)) <= 3e-2 * float(ref.loss)
    assert rel(xg.cpu(), ref.x_grad[0]) < 3e-2 and rel(head.sub_weight.grad.cpu(), ref.dw[0]) < 3e-2
    head._ops.bwd_mode = "prob"                                        # shared per-device provider: leave it as found
    for slot in range(4):                                              # and the per-device flag pairs too: a pair raised
        head._ops.read_range_slot(slot)                                # here and never read would switch a later head


def test_fedavg_signed_zero_unaligned_and_many_clients(pkg):
    dev = torch.device("cuda:0")
    # FedPavg: tmp = 0; tmp += w * x (server.py:30-32) turns -0.0 into +0.0; FedAvg_on_FC (server.py:38) starts AT the first term
    a = torch.tensor([-0.0, 0.0, -0.0, 1.0, -0.0], device=dev)
    out = pkg.FedPavg([{"t": a}], [1.0])["t"]
    ref = 0 + 1.0 * a
    assert torch.equal(out.view(torch.int32), ref.view(torch.int32))
    fc = pkg.FedAvg_on_FC(a, [a.clone(), a.clone()], [1, 1], 1)
    ref_fc = a.clone() * 0.5
    ref_fc += a * 0.5
    assert torch.equal(fc.view(torch.int32), ref_fc.view(torch.int32))
    # views at odd offsets of a flat buffer (not 16-byte aligned) take the scalar path instead of failing
    g = torch.Generator(device=dev).manual_seed(1)
    flat = [torch.randn(4099, device=dev, generator=g) for _ in range(3)]
    models = [{"odd": f[1:1 + 2050], "even": f[2052:2052 + 2040]} for f in flat]
    got = pkg.FedPavg(models, [3, 2, 1])
    want = {k: 0 for k in models[0]}
    for wi, md in zip([3 / 6, 2 / 6, 1 / 6], models):
        for k in want:
            want[k] = want[k] + wi * md[k]
    for k in want:
        assert torch.equal(got[k], want[k]), k
    # K > 64 clients: several launches continue one running sum in client order -> still the reference's bits
    K = 150
    ms = [{"w": torch.randn(10007, device=dev, generator=g), "n": torch.tensor(i, device=dev)} for i in range(K)]
    ws = [1 + (i % 7) for i in range(K)]
    got = pkg.FedPavg(ms, ws)
    tot = float(sum(ws))
    want_w, want_n = 0, 0
    for wi, md in zip(ws, ms):
        want_w = want_w + (wi / tot) * md["w"]
        want_n = want_n + (wi / tot) * md["n"]
    assert torch.equal(got["w"], want_w) and torch.equal(got["n"], want_n)


def test_fedavg_flat_state_dicts(pkg):
    """FlatStateDict clients (one buffer per client) give the same bits as plain dicts, from the GPU and from pinned host
    memory, and the result loads into a module."""
    dev = torch.device("cuda:0")
    net = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3), torch.nn.BatchNorm2d(8), torch.nn.Linear(8, 5))
    K = 5
    sds = []
    for i in range(K):
        torch.manual_seed(i)
        sd = {k: (torch.randn_like(v) if v.is_floating_point() else torch.tensor(10 * i + 3)) for k, v in net.state_dict().items()}
        sds.append({k: v.to(dev) for k, v in sd.items()})
    w = [5, 4, 3, 2, 1]
    plain = pkg.FedPavg(sds, w)
    flats = [pkg.flatten_state_dict(sd) for sd in sds]
    assert all(isinstance(f, dict) and f.layout is flats[0].layout for f in flats)
    got = pkg.FedPavg(flats, w)
    host = pkg.FedPavg([pkg.flatten_state_dict(sd, device="cpu", pin_memory=True) for sd in sds], w)
    assert list(got.keys()) == list(plain.keys())
    for k in plain:
        assert got[k].dtype == torch.float32 and torch.equal(got[k], plain[k]) and torch.equal(host[k], plain[k]), k
    net.to(dev).load_state_dict(got)                                        # int64 counter truncated back, server.py:333
    flats[0]["0.weight"] = torch.zeros_like(flats[0]["0.weight"])           # a replaced entry drops the client to the dict path
    again = pkg.FedPavg(flats, w)
    assert not torch.equal(again["0.weight"], plain["0.weight"]) and torch.equal(again["2.bias"], plain["2.bias"])


@pytest.mark.parametrize("kind", ["cosface", "arcface"])
def test_margin_callables_on_dense_logits(pkg, kind):
    """losses.CosFace / losses.ArcFace called on materialised logits (client.py:430, --loss ArcFace): the reference's
    arithmetic incl. its in-place edits of ``cosine`` and -1 labels."""
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(2)
    cos = (torch.rand(37, 211, generator=g) * 1.9 - 0.95)
    lab = torch.randint(0, 211, (37,), generator=g)
    lab[3] = -1
    s, m = 30.0, 0.45
    ref_in = cos.clone()
    idx = torch.where(lab != -1)[0]
    m_hot = torch.zeros(idx.numel(), 211).scatter_(1, lab[idx, None], m)
    if kind == "cosface":                                                  # losses.py:23-29
        ref_in[idx] -= m_hot
        ref_out = ref_in * s
    else:                                                                  # losses.py:38-45
        ref_in.acos_()
        ref_in[idx] += m_hot
        ref_in.cos_().mul_(s)
        ref_out = ref_in
    c = cos.to(dev)
    out = (pkg.CosFace(s, m) if kind == "cosface" else pkg.ArcFace(s, m))(c, lab.to(dev))
    assert torch.allclose(out.cpu(), ref_out, rtol=1e-5, atol=2e-5)
    assert torch.allclose(c.cpu(), ref_in, rtol=1e-5, atol=2e-5)           # the input is edited in place like the reference's
    if kind == "arcface":
        assert out.data_ptr() == c.data_ptr()
