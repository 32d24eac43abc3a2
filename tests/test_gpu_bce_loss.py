"""``BCE_module.loss`` on the B200: the personalised head's ``losses.BCE_loss`` fused into the head
(``pfc_bce_loss_fwd`` / ``pfc_bce_loss_bwd``).

- The golden of the unmodified reference classes (tests/golden/bce_head.npz), to the suite's 1e-4.
- The shapes of test_bce_head.test_gpu_matches_reference_formulation against fp64 autograd of ``reference_head`` +
  ``bce_loss``, by norm and row by row, with the loss's ``r_loss`` apart from the head's ``r`` and an upstream gradient
  other than 1.
- The C entries on NaN-filled outputs with guard elements, row by row against the restatement (test_bce_loss.check_case):
  the emulator's cases, FedFR's shapes, every label rule, zero rows, overflowing exps, NULL pointers, empty batches and
  every error code; cosine and inverse norms bit-identical to ``pfc_bce_head_fwd``'s.
- The fused path against the unfused one (the reference's ``BCE_loss`` on ``BCE_module``'s logits), two runs bit for
  bit, and forward plus backward under ``torch.cuda.set_sync_debug_mode("error")``, which the unfused path fails."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
import bce_loss_oracle as BL  # noqa: E402
from test_bce_head import _load_module, bce_loss, reference_head, rel  # noqa: E402
from test_bce_loss import EMU_CASES, check_case, check_empty, check_error_codes  # noqa: E402

TOL = 1e-4
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


@pytest.fixture(scope="module")
def golden():
    import numpy as np
    z = np.load(os.path.join(HERE, "golden", "bce_head.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


@pytest.fixture(scope="module")
def lib(pkg):
    from fedfr_b200 import _native as N
    return N.lib


def rows_close(got, want, tol):
    """Each row within tol of its own norm, with a floor of tol times the largest row norm (rows that cancel to ~0)."""
    got, want = got.double().cpu(), want.double().cpu()
    err = (got - want).norm(dim=1)
    floor = tol * float(want.norm(dim=1).max())
    bad = err > tol * want.norm(dim=1) + floor
    assert not bool(bad.any()), (int(bad.nonzero()[0, 0]), float((err / (want.norm(dim=1) + floor)).max()))


def _module(pkg, C, E, r, t, weight, bias):
    mod = pkg.BCE_module(E, C, 1, r=r, t=t).to(DEV)
    with torch.no_grad():
        mod.weight.copy_(weight)
        mod.bias.copy_(bias)
    return mod


# ----------------------------------------------------------------------------------------------- the module
@pytest.mark.gpu
def test_gpu_loss_matches_reference_golden(pkg, golden):
    mod = _load_module(pkg, golden, DEV)
    x = golden["x"].detach().clone().to(DEV).requires_grad_(True)
    loss = 10 * mod.loss(x, golden["y"].to(DEV))
    loss.backward()
    assert abs(float(loss.detach()) - float(golden["loss"])) < TOL * abs(float(golden["loss"]))
    assert rel(x.grad, golden["dx"]) < TOL
    for k, p in mod.named_parameters():
        assert rel(p.grad, golden["grad/" + k]) < TOL, k


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,E,t,detach,r,lam,r_loss,grad_out", [(256, 100, 512, 3, False, 30.0, 0.7, 30.0, 10.0),
                                                                  (64, 300, 512, 3, True, 30.0, 0.7, 30.0, 10.0),
                                                                  (7, 3, 33, 2, False, 50.0, 0.55, 20.0, -0.37),
                                                                  (5, 1, 1024, 4, False, 12.0, 0.7, 30.0, 2.5)])
def test_gpu_loss_matches_reference_formulation(pkg, B, C, E, t, detach, r, lam, r_loss, grad_out):
    g = torch.Generator().manual_seed(B + C)
    feat = torch.randn(B, E, generator=g) * 2
    weight = torch.randn(C, E, generator=g) * 0.01
    bias = torch.randn(C, generator=g) * 0.1
    y = torch.randint(0, C + C // 3 + 1, (B,), generator=g)
    fr, wr, br = (v.double().requires_grad_(True) for v in (feat, weight, bias))
    lr, gr = reference_head(fr, wr, br, y, 0.4, r, t)
    ref = bce_loss(lr, gr, r=r_loss, lam=lam)
    (grad_out * ref).backward()

    mod = _module(pkg, C, E, r, t, weight, bias)
    x = feat.to(DEV).requires_grad_(not detach)
    loss = mod.loss(x, y.to(DEV), lam=lam, r_loss=r_loss)           # identity converter: feat == x
    (grad_out * loss).backward()
    assert abs(float(loss.detach()) - float(ref.detach())) < TOL * abs(float(ref.detach()))
    assert rel(mod.weight.grad, wr.grad) < TOL and rel(mod.bias.grad, br.grad) < TOL
    rows_close(mod.weight.grad, wr.grad, TOL)
    if detach:
        assert x.grad is None
    else:
        assert rel(x.grad, fr.grad) < TOL
        rows_close(x.grad, fr.grad, TOL)
    dconv = fr.grad.t() @ feat.double()
    assert rel(mod.converter[0].weight.grad, dconv) < TOL
    rows_close(mod.converter[0].weight.grad, dconv, TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,E", [(256, 100, 512), (64, 300, 512), (300, 257, 128)])
def test_gpu_fused_equals_unfused(pkg, B, C, E):
    """10 * BCE_module.loss against 10 * losses.BCE_loss on BCE_module's logits (client.py:382,393 today), same inputs."""
    g = torch.Generator().manual_seed(B * C)
    x0 = torch.randn(B, E, generator=g)
    y = torch.randint(-2, C + 3, (B,), generator=g).to(DEV)
    mod = _module(pkg, C, E, 30.0, 3, torch.randn(C, E, generator=g) * 0.01, torch.randn(C, generator=g) * 0.1)
    grads = []
    for fused in (True, False):
        mod.zero_grad()
        x = x0.to(DEV).requires_grad_(True)
        loss = 10 * (mod.loss(x, y) if fused else BL.reference_bce_loss(*mod(x, y)))
        loss.backward()
        grads.append([loss.detach(), x.grad] + [p.grad.clone() for p in mod.parameters()])
    for i, (a, b) in enumerate(zip(*grads)):
        assert rel(a, b) < 1e-5, i
        if a.dim() == 2:
            rows_close(a, b, 1e-4)
    print("fused vs unfused, max |diff| per output:", [float((a - b).abs().max()) for a, b in zip(*grads)])


@pytest.mark.gpu
def test_gpu_loss_is_deterministic(pkg):
    """Two runs of the same step give the same bits: loss, dx, and every parameter gradient."""
    g = torch.Generator().manual_seed(11)
    B, C, E = 300, 600, 512
    x0, y = torch.randn(B, E, generator=g).to(DEV), torch.randint(0, C, (B,), generator=g).to(DEV)
    mod = _module(pkg, C, E, 30.0, 3, torch.randn(C, E, generator=g) * 0.01, torch.randn(C, generator=g) * 0.1)
    runs = []
    for _ in range(2):
        mod.zero_grad()
        x = x0.clone().requires_grad_(True)
        loss = 10 * mod.loss(x, y)
        loss.backward()
        runs.append([loss.detach().clone(), x.grad] + [p.grad.clone() for p in mod.parameters()])
    for a, b in zip(*runs):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.gpu
def test_gpu_loss_never_synchronises(pkg):
    """Forward and backward of 10 * BCE_module.loss run under set_sync_debug_mode("error"); the reference formulation
    (BCE_loss's boolean-mask edits on the logits) raises there."""
    g = torch.Generator().manual_seed(5)
    B, C, E = 64, 300, 512
    x0, y = torch.randn(B, E, generator=g).to(DEV), torch.randint(0, C, (B,), generator=g).to(DEV)
    mod = _module(pkg, C, E, 30.0, 3, torch.randn(C, E, generator=g) * 0.01, torch.randn(C, generator=g) * 0.1)
    (10 * mod.loss(x0.clone().requires_grad_(True), y)).backward()           # first call: lazy set-up outside the check
    torch.cuda.synchronize()
    mod.zero_grad()
    x = x0.clone().requires_grad_(True)
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss = 10 * mod.loss(x, y)
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert x.grad is not None and mod.weight.grad is not None and bool(torch.isfinite(loss))
    torch.cuda.set_sync_debug_mode("error")
    try:
        with pytest.raises(RuntimeError):
            BL.reference_bce_loss(*mod(x0, y))
    finally:
        torch.cuda.set_sync_debug_mode(0)


@pytest.mark.gpu
def test_gpu_loss_in_cuda_graph(pkg):
    """The forward captured in a CUDA graph and replayed between eager calls on the same stream gives the eager loss's
    bits every time: each call zeroes a ticket of its own, so the captured kernel and the eager ones share no counter."""
    g = torch.Generator().manual_seed(9)
    B, C, E = 256, 100, 512
    x, y = torch.randn(B, E, generator=g).to(DEV), torch.randint(0, C, (B,), generator=g).to(DEV)
    mod = _module(pkg, C, E, 30.0, 3, torch.randn(C, E, generator=g) * 0.01, torch.randn(C, generator=g) * 0.1)
    with torch.no_grad():
        want = mod.loss(x, y).clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            mod.loss(x, y)                                         # warm-up on the capture stream
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            captured = mod.loss(x, y)
        for _ in range(3):
            graph.replay()
            eager = mod.loss(x, y)
            assert torch.equal(captured.view(torch.int32), want.view(torch.int32))
            assert torch.equal(eager.view(torch.int32), want.view(torch.int32))


@pytest.mark.gpu
def test_gpu_loss_empty_batch(pkg):
    mod = pkg.BCE_module(64, 5).to(DEV)
    loss = mod.loss(torch.zeros(0, 64, device=DEV), torch.zeros(0, dtype=torch.long, device=DEV))
    assert bool(torch.isnan(loss))
    loss.backward()
    assert float(mod.weight.grad.abs().max()) == 0.0 and float(mod.bias.grad.abs().max()) == 0.0


# ----------------------------------------------------------------------------------------------- the C entries
@pytest.mark.gpu
@pytest.mark.parametrize("B,C,E,t,r,lam,r_loss,grad_out", EMU_CASES + [(256, 100, 512, 3, 30.0, 0.7, 30.0, 10.0),
                                                                        (64, 300, 512, 3, 30.0, 0.7, 30.0, 10.0),
                                                                        (257, 513, 1024, 3, 30.0, 0.7, 30.0, 10.0),
                                                                        (1000, 3000, 128, 2, 50.0, 0.7, 30.0, -1.5)])
def test_gpu_abi_matches_restatement(lib, B, C, E, t, r, lam, r_loss, grad_out):
    check_case(lib, DEV, B, C, E, t, r, lam, r_loss, grad_out, seed=B * 1009 + C * 31 + E)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["overflow", "bias NULL", "dfeat NULL", "dbias NULL"])
def test_gpu_abi_variants(lib, what):
    """Overflowing exps give the restatement's inf loss and NaN rows; NULL bias, dfeat and dbias follow the head's rules."""
    check_case(lib, DEV, 300, 257, 512, 3, 30.0, 0.7, 30.0, 10.0, seed=7, overflow=what == "overflow",
               bias_on=what != "bias NULL", need_dfeat=what != "dfeat NULL", need_dbias=what != "dbias NULL")


@pytest.mark.gpu
def test_gpu_abi_empty(lib):
    check_empty(lib, DEV)


@pytest.mark.gpu
def test_gpu_abi_error_codes(lib):
    check_error_codes(lib, DEV)
    torch.cuda.synchronize()
