"""The personalised head's loss fused into the head (``BCE_module.loss``; ``pfc_bce_loss_fwd`` / ``pfc_bce_loss_bwd`` in
csrc/bce_head.cu) without a GPU.

- The fp64 restatement (tests/bce_loss_oracle.py) reproduces the golden of the unmodified ``client.BCE_module`` +
  ``losses.BCE_loss`` + ``loss.backward()`` (tests/golden/bce_head.npz), and equals fp64 autograd of the reference
  formulation with the loss's scale ``r_loss`` apart from the head's ``r`` and an upstream gradient other than 1.
- ``BCE_module.loss``'s host logic (converter, autograd glue, NULL gradients) runs on the oracle-backed ops.
- The emulated build of bce_head.cu (tests/emu/cuda_emu.h, ``_build_abi`` of test_kernel_emulation.py) is called through
  the C entries with NaN-filled outputs followed by NaN guard elements, and held to the restatement row by row: B and C
  across the 256-class chunks, emb across the 32-lane slices up to 1024, t = 2, 3, 4, every label rule, zero feature and
  class rows, overflowing exps, empty batches, and every error code.  Its cosine and inverse norms must be the bits of
  the emulated ``pfc_bce_head_fwd``.  The emulated tests run again under AddressSanitizer with the reverse schedule.

Mutations these tests catch (each applied alone):
- ``pos_coef`` and ``neg_coef`` swapped in ``bce_term`` (lam for 1 - lam): every case of
  test_emulated_loss_matches_restatement and test_emulated_loss_variants fails (13 tests);
- ``*s.grad_out`` read as 1 in ``bce_loss_dz`` (the upstream gradient ignored): every emulated case whose grad_out is
  not 1 fails (11 tests);
- the head's ``r`` passed for ``r_loss`` in ``BCE_module.loss``: test_module_loss_scales_and_detached_features fails
  (r = 64, r_loss = 12)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import bce_loss_oracle as BL  # noqa: E402
from test_bce_head import _load_module, bce_loss, reference_head, rel  # noqa: E402
from test_gpu_bce_head_edges import _cpu_case, restate_bwd, restate_fwd  # noqa: E402
from test_kernel_emulation import _build_abi  # noqa: E402

E_ARG, E_SHAPE = -1, -2
M = 0.4
GUARD = 17


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


@pytest.fixture(scope="module")
def golden():
    z = np.load(os.path.join(HERE, "golden", "bce_head.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


# ----------------------------------------------------------------------------------------------- restatement
def test_restatement_matches_reference_golden(golden):
    """10 * BCE_loss on the unmodified reference head: the loss and every gradient of the golden, to 1e-5."""
    sd = {k[3:]: v.double() for k, v in golden.items() if k.startswith("sd/")}
    x = golden["x"].double()
    feat = x @ sd["converter.0.weight"].t() + sd["converter.0.bias"]
    R = BL.restate(feat, sd["weight"], sd["bias"], golden["y"], M, 30.0, 3, *BL.coefs(0.7, 30.0), grad_out=10.0)
    assert abs(10 * float(R["loss"]) - float(golden["loss"])) <= 1e-5 * abs(float(golden["loss"]))
    assert rel(R["dfeat"] @ sd["converter.0.weight"], golden["dx"]) < 1e-5
    assert rel(R["dweight"], golden["grad/weight"]) < 1e-5 and rel(R["dbias"], golden["grad/bias"]) < 1e-5
    assert rel(R["dfeat"].t() @ x, golden["grad/converter.0.weight"]) < 1e-5
    assert rel(R["dfeat"].sum(dim=0), golden["grad/converter.0.bias"]) < 1e-5


@pytest.mark.parametrize("B,C,E,t,r,lam,r_loss,grad_out", [(9, 7, 16, 3, 30.0, 0.7, 30.0, 1.0), (6, 5, 33, 2, 50.0, 0.75, 32.0, 10.0),
                                                           (8, 4, 5, 4, 12.0, 0.5, 16.0, -0.37), (7, 9, 12, 3, 30.0, 0.7, 45.0, 10.0)])
def test_restatement_is_autograd_of_the_reference(B, C, E, t, r, lam, r_loss, grad_out):
    """fp64: grad_out * bce_loss(reference_head(...), r=r_loss, lam) differentiated by autograd equals the restatement,
    row by row, with a zero feature row and rows whose norm is below eps (their gradient is d / eps)."""
    feat, weight, bias, y = _cpu_case(B, C, E, B * C + E)
    fr, wr, br = (v.clone().requires_grad_(True) for v in (feat, weight, bias))
    lr, gr = reference_head(fr, wr, br, y, M, r, t)
    loss = bce_loss(lr, gr, r=r_loss, lam=lam)
    (grad_out * loss).backward()
    R = BL.restate(feat, weight, bias, y, M, r, t, lam / r_loss, (1 - lam) / r_loss, grad_out=grad_out)
    # the restatement rounds the coefficients to fp32 as the reference does; autograd here ran with the doubles, which
    # are the same numbers for lam / r_loss = 0.75 / 32 and 0.5 / 16 and differ by up to 2^-24 relative otherwise
    tol = 1e-10 if BL.coefs(lam, r_loss) == (lam / r_loss, (1 - lam) / r_loss) else 1e-6
    loss = float(loss.detach())
    assert abs(float(R["loss"]) - loss) <= tol * abs(loss)
    for got, want in ((R["dfeat"], fr.grad), (R["dweight"], wr.grad)):
        for i in range(want.shape[0]):
            assert float((got[i] - want[i]).abs().max()) <= tol * (float(want[i].abs().max()) + 1e-300), i
    assert float((R["dbias"] - br.grad).abs().max()) <= tol * float(br.grad.abs().max())


def test_restatement_overflow_and_empty_batch():
    """An exp beyond fp32's range gives an infinite loss and NaN gradients, as the fp32 reference does; B = 0 gives a NaN
    loss (torch's mean of nothing)."""
    z = torch.tensor([[100.0, -100.0, 3.0], [-95.0, 1.0, 0.5]], dtype=torch.float64)
    gt = torch.tensor([[False, False, True], [True, False, False]])
    loss, row, dz = BL.loss_from_logits(z, gt, *BL.coefs())
    assert float(loss) == float("inf") and torch.isinf(row).all()
    assert torch.isnan(dz).tolist() == [[True, False, False], [True, False, False]]
    z32 = z.float().requires_grad_(True)                  # the reference, in fp32, agrees
    ref = BL.reference_bce_loss(z32, gt)
    ref.backward()
    assert torch.isinf(ref) and torch.equal(torch.isnan(z32.grad), torch.isnan(dz))
    loss0, row0, dz0 = BL.loss_from_logits(torch.zeros(0, 3, dtype=torch.float64), torch.zeros(0, 3, dtype=torch.bool), 0.1, 0.2)
    assert torch.isnan(loss0) and row0.numel() == 0 and dz0.numel() == 0
    assert torch.isnan(BL.reference_bce_loss(torch.zeros(0, 3), torch.zeros(0, 3, dtype=torch.bool)))


# ----------------------------------------------------------------------------------------------- module host logic
def test_module_loss_host_logic_cpu(pkg, golden):
    """10 * BCE_module.loss(x, y) on the oracle-backed ops gives the golden's loss and every gradient; forward still
    returns the golden's (logits, gt)."""
    ops = BL.OracleBceLossOps()
    mod = _load_module(pkg, golden, ops=ops)
    x = golden["x"].detach().clone().requires_grad_(True)
    loss = 10 * mod.loss(x, golden["y"])
    assert loss.dim() == 0 and loss.dtype == torch.float32
    loss.backward()
    assert abs(float(loss.detach()) - float(golden["loss"])) < 1e-5 * abs(float(golden["loss"]))
    assert rel(x.grad, golden["dx"]) < 1e-5
    for k, p in mod.named_parameters():
        assert rel(p.grad, golden["grad/" + k]) < 1e-5, k
    assert ops.calls == [(True, True)]
    logits, gts = mod(golden["x"], golden["y"])
    assert torch.equal(gts, golden["gt"]) and rel(logits.detach(), golden["logits"]) < 1e-5


def test_module_loss_scales_and_detached_features(pkg):
    """lam and r_loss reach the loss apart from the head's r; features that need no gradient (a frozen converter on
    detached input, client.py:94-95 with the converter fixed) ask the backward for no dfeat."""
    g = torch.Generator().manual_seed(3)
    x, y = torch.randn(6, 16, generator=g), torch.tensor([1, 7, 4, 0, -2, 3])
    ops = BL.OracleBceLossOps()
    mod = pkg.BCE_module(16, 5, r=64.0, t=2, _ops=ops)
    with torch.no_grad():
        mod.weight.copy_(torch.randn(5, 16, generator=g))
        mod.bias.copy_(torch.randn(5, generator=g))
    mod.converter.requires_grad_(False)
    loss = mod.loss(x.detach(), y, lam=0.55, r_loss=12.0)
    loss.backward()
    assert ops.calls == [(False, True)] and mod.converter[0].weight.grad is None and mod.weight.grad is not None
    R = BL.restate(x.double(), mod.weight.detach().double(), mod.bias.detach().double(), y, M, 64.0, 2, 0.55 / 12.0, 0.45 / 12.0)
    assert abs(float(loss) - float(R["loss"])) < 1e-5 * float(R["loss"])
    assert rel(mod.weight.grad, R["dweight"]) < 1e-5 and rel(mod.bias.grad, R["dbias"]) < 1e-5
    logits, gts = mod(x, y)
    assert abs(float(loss) - float(bce_loss(logits.detach(), gts, r=12.0, lam=0.55))) < 1e-5 * float(loss)


def test_module_loss_needs_cuda(pkg):
    with pytest.raises(RuntimeError):
        pkg.BCE_module(16, 5).loss(torch.randn(3, 16), torch.tensor([1, 2, 3]))


# ----------------------------------------------------------------------------------------------- emulated kernels
@pytest.fixture(scope="module")
def emu(pkg, tmp_path_factory):
    """The emulated bce_head.cu with the product's ctypes signatures."""
    from fedfr_b200 import _native as N
    lib = _build_abi("bce_head", str(tmp_path_factory.mktemp("bce_loss_emu")))
    for name in ("pfc_bce_head_fwd", "pfc_bce_head_bwd", "pfc_bce_loss_fwd", "pfc_bce_loss_bwd"):
        f = getattr(lib, name)
        f.restype, f.argtypes = N.SIGNATURES[name]
    return lib


def _ptr(t):
    return None if t is None else t.data_ptr()


def _on(a, dev):
    return None if a is None else torch.from_numpy(a).to(dev)


def _stream(dev):
    """the launch stream: the emulated build ignores it"""
    return torch.cuda.current_stream().cuda_stream if torch.device(dev).type == "cuda" else None


def _nan(n, dev):
    """n NaN fp32 elements followed by GUARD NaN guards: (whole buffer, the leading n)."""
    buf = torch.full((n + GUARD,), float("nan"), dtype=torch.float32, device=dev)
    return buf, buf[:n]


def make_case(B, C, E, seed, overflow=False):
    """fp32 rows and labels with every label rule (in range, >= C, -1, -2, -(C + 1), -(C + 2)), a zero feature row and a
    zero class row where B, C >= 3.  overflow: a class with bias +150 (exp(z) overflows on the rows where it is negative)
    and one with bias -150 that some row has as its target (exp(-z) overflows there)."""
    g = torch.Generator().manual_seed(seed)
    feat = torch.randn(B, E, generator=g) * 2
    weight = torch.randn(C, E, generator=g) * 0.01
    bias = torch.randn(C, generator=g) * 0.1
    y = torch.randint(0, max(C, 1), (B,), generator=g)
    special = [C, C + 3, -1, -2, -(C + 1), -(C + 2)][:max(B - 1, 0)]
    y[1:1 + len(special)] = torch.tensor(special, dtype=torch.long)
    if B >= 3:
        feat[B - 1] = 0.0
    if C >= 3:
        weight[C - 1] = 0.0
    if overflow and C >= 2 and B >= 2:
        bias[0] = 150.0
        bias[1] = -150.0
        y[0] = 1
    return feat.numpy(), weight.numpy(), bias.numpy(), y.numpy()


def run_abi(lib, dev, feat, weight, bias, y, t, r, lam, r_loss, grad_out, need_dfeat=True, need_dbias=True):
    """pfc_bce_loss_fwd then pfc_bce_loss_bwd on `dev` (the emulated build: "cpu"), as BCE_module.loss marshals them,
    into NaN-filled outputs with NaN guards; the ticket must come back 0 and no guard may change.  -> numpy outputs."""
    B, E = feat.shape
    C = weight.shape[0]
    pc, nc = lam / r_loss, (1 - lam) / r_loss
    f, w, b, lab = _on(feat, dev), _on(weight, dev), _on(bias, dev), _on(y, dev)
    bufs = {k: _nan(n, dev) for k, n in (("loss", 1), ("row_loss", B), ("cosine", B * C), ("inv_nf", B), ("inv_nw", C),
                                         ("dfeat", B * E), ("dweight", C * E), ("dbias", C))}
    v = {k: inner for k, (_, inner) in bufs.items()}
    ticket = torch.zeros(1, dtype=torch.int32, device=dev)
    rc = lib.pfc_bce_loss_fwd(_ptr(f), _ptr(w), _ptr(b), _ptr(lab), B, C, E, M, r, float(t), pc, nc, _ptr(v["loss"]),
                              _ptr(v["row_loss"]), _ptr(ticket), _ptr(v["cosine"]), _ptr(v["inv_nf"]), _ptr(v["inv_nw"]),
                              _stream(dev))
    assert rc == 0
    go = torch.tensor([grad_out], dtype=torch.float32, device=dev)
    rc = lib.pfc_bce_loss_bwd(_ptr(f), _ptr(w), _ptr(b), _ptr(lab), _ptr(v["cosine"]), _ptr(v["inv_nf"]), _ptr(v["inv_nw"]),
                              _ptr(go), B, C, E, M, r, float(t), pc, nc, _ptr(v["dfeat"]) if need_dfeat else None,
                              _ptr(v["dweight"]), _ptr(v["dbias"]) if need_dbias else None, _stream(dev))
    assert rc == 0
    assert int(ticket.cpu()[0]) == 0, "the ticket must come back 0"
    assert all(bool(torch.isnan(whole[-GUARD:]).all()) for whole, _ in bufs.values()), "a store past the end of an output"
    out = {k: t_.cpu().numpy() for k, t_ in v.items()}
    out["cosine"] = out["cosine"].reshape(B, C)
    out["dfeat"], out["dweight"] = out["dfeat"].reshape(B, E), out["dweight"].reshape(C, E)
    return out


def restate_from_kernel(feat, weight, bias, y, got, t, r, lam, r_loss, grad_out):
    """fp64 from the kernel's own fp32 cosine and inverse norms (so only the loss's and the backward's arithmetic is
    compared): per-row loss, d z, and the backward of test_gpu_bce_head_edges.restate_bwd."""
    f, w = torch.from_numpy(feat), torch.from_numpy(weight)
    b = None if bias is None else torch.from_numpy(bias)
    cos = torch.from_numpy(got["cosine"])
    ref = restate_fwd(f, w, b, torch.from_numpy(y), cos, t, m=M, r=r)
    loss, row, dz = BL.loss_from_logits(ref["logits"], ref["gt"], lam / r_loss, (1 - lam) / r_loss, grad_out)
    g = restate_bwd(f, w, cos, torch.from_numpy(got["inv_nf"]), torch.from_numpy(got["inv_nw"]), dz, t, r=r)
    g.update(loss=loss, row_loss=row, dz=dz, fwd=ref)
    return g


def check_rows(got, want, parts, inv, tol, what):
    """Every row of a gradient against the restatement, relative to the size of the two terms it is the difference of
    (inv |acc| and inv |mine inv radial|); rows that are NaN in the restatement must be NaN in the kernel."""
    got = torch.from_numpy(np.asarray(got)).double()
    nan_want = torch.isnan(want).any(dim=1)
    assert torch.equal(torch.isnan(got).any(dim=1), nan_want), what + ": NaN rows differ"
    assert bool(torch.isnan(got[nan_want]).all()), what + ": a NaN row is only partly NaN"
    acc, rad = parts
    scale = inv.double() * (acc.norm(dim=1) + rad.norm(dim=1))
    err = (got - want).norm(dim=1)
    ok = ~nan_want
    ratio = err[ok] / (scale[ok] + 1e-30)
    assert bool((ratio <= tol).all()), (what, float(ratio.max()), int(ratio.argmax()))
    return float(ratio.max()) if ratio.numel() else 0.0


def check_case(lib, dev, B, C, E, t, r, lam, r_loss, grad_out, seed, overflow=False, bias_on=True, need_dfeat=True,
               need_dbias=True):
    """One case through run_abi, held to the restatement row by row.  -> the outputs."""
    feat, weight, bias, y = make_case(B, C, E, seed, overflow)
    bias = bias if bias_on else None
    got = run_abi(lib, dev, feat, weight, bias, y, t, r, lam, r_loss, grad_out, need_dfeat, need_dbias)

    # cosine and both inverse norms: the bits pfc_bce_head_fwd computes for the same inputs
    head = {k: torch.full((n,), float("nan"), device=dev) for k, n in (("logits", B * C), ("cosine", B * C), ("inv_nf", B),
                                                                        ("inv_nw", C))}
    gt = torch.zeros(B * C, dtype=torch.uint8, device=dev)
    assert lib.pfc_bce_head_fwd(_ptr(_on(feat, dev)), _ptr(_on(weight, dev)), _ptr(_on(bias, dev)), _ptr(_on(y, dev)), B, C, E,
                                M, r, float(t), _ptr(head["logits"]), _ptr(gt), _ptr(head["cosine"]), _ptr(head["inv_nf"]),
                                _ptr(head["inv_nw"]), _stream(dev)) == 0
    head = {k: v.cpu().numpy() for k, v in head.items()}
    assert np.array_equal(got["cosine"].reshape(-1).view(np.uint32), head["cosine"].view(np.uint32))
    assert np.array_equal(got["inv_nf"].view(np.uint32), head["inv_nf"].view(np.uint32))
    assert np.array_equal(got["inv_nw"].view(np.uint32), head["inv_nw"].view(np.uint32))

    # the loss: row sums against fp64 of the kernel's cosine, the mean bit for bit from the kernel's row sums
    R = restate_from_kernel(feat, weight, bias, y, got, t, r, lam, r_loss, grad_out)
    row = torch.from_numpy(got["row_loss"]).double()
    assert torch.equal(torch.isinf(row), torch.isinf(R["row_loss"])) and not bool(torch.isnan(row).any())
    fin = torch.isfinite(R["row_loss"])
    # fp32 rounds 1 + exp(-|z|) to 1 once exp(-|z|) < 2^-24: the term is then exactly 0 where fp64 keeps ~coef e, an
    # absolute error of at most coef 2^-24 (plus as much from the rounding of + 1e-8) per term
    absorbed = C * max(lam, 1 - lam) / r_loss * 2.0 ** -22
    row_err = ((row - R["row_loss"]).abs() / (2e-5 * R["row_loss"].abs() + absorbed))[fin]
    assert bool((row_err <= 1).all()), float(row_err.max())
    s = np.float32(0)
    for v in got["row_loss"]:
        s = np.float32(s + v)
    assert np.float32(s / np.float32(B)).view(np.uint32) == got["loss"][0].view(np.uint32)
    if overflow:
        assert got["loss"][0] == np.inf
    else:
        assert abs(float(got["loss"][0]) - float(R["loss"])) <= 2e-5 * abs(float(R["loss"])) + absorbed
        # and against the restatement from the fp64 inputs (the kernel's cosine error included), at the suite's 1e-4
        X = BL.restate(torch.from_numpy(feat).double(), torch.from_numpy(weight).double(),
                       None if bias is None else torch.from_numpy(bias).double(), torch.from_numpy(y), M, r, t,
                       lam / r_loss, (1 - lam) / r_loss, grad_out)
        assert abs(float(got["loss"][0]) - float(X["loss"])) <= 1e-4 * abs(float(X["loss"])) + absorbed
        assert rel(got["dweight"], X["dweight"]) < 1e-4
        if need_dfeat:
            assert rel(got["dfeat"], X["dfeat"]) < 1e-4

    # the gradients, row by row
    errs = {"row_loss err/bound": float(row_err.max()) if row_err.numel() else 0.0}
    errs["dweight"] = check_rows(got["dweight"], R["dweight"], R["dweight parts"], torch.from_numpy(got["inv_nw"]), 1e-4, "dweight")
    if need_dfeat:
        errs["dfeat"] = check_rows(got["dfeat"], R["dfeat"], R["dfeat parts"], torch.from_numpy(got["inv_nf"]), 1e-4, "dfeat")
    else:
        assert np.isnan(got["dfeat"]).all(), "dfeat == NULL: nothing may be written"
    if need_dbias:
        db = torch.from_numpy(got["dbias"]).double()
        assert torch.equal(torch.isnan(db), torch.isnan(R["dbias"]))
        ok = ~torch.isnan(R["dbias"])
        scale = R["dz"].abs().sum(dim=0)[ok]
        assert bool(((db[ok] - R["dbias"][ok]).abs() <= 1e-5 * scale + 1e-30).all())
    else:
        assert np.isnan(got["dbias"]).all(), "dbias == NULL: nothing may be written"
    if overflow:
        assert np.isnan(got["dfeat"][0]).all() and np.isnan(got["dbias"][:2]).all()
    print("B=%d C=%d E=%d t=%s r=%s grad_out=%s" % (B, C, E, t, r, grad_out), errs)
    return got


# B and C across the 256-class chunks of the forward and the 256-row chunks of the backward, emb across 32-lane slices
# and up to 1024, t = 2, 3, 4; r, lam, r_loss and grad_out vary so that mixing up the two scales or dropping the
# upstream gradient fails
EMU_CASES = [
    (1, 1, 1, 2, 30.0, 0.7, 30.0, 1.0),
    (7, 257, 33, 3, 50.0, 0.7, 30.0, 10.0),
    (257, 7, 512, 4, 30.0, 0.7, 30.0, 10.0),
    (255, 7, 33, 2, 12.0, 0.55, 20.0, -0.37),
    (7, 256, 1, 3, 30.0, 0.7, 30.0, 10.0),
    (256, 7, 1, 3, 30.0, 0.7, 45.0, 2.5),
    (1, 255, 1024, 4, 50.0, 0.7, 30.0, 10.0),
    (7, 1, 1024, 2, 30.0, 0.7, 30.0, 1.0),
    (256, 1, 512, 3, 30.0, 0.7, 30.0, 10.0),
]


@pytest.mark.parametrize("B,C,E,t,r,lam,r_loss,grad_out", EMU_CASES)
def test_emulated_loss_matches_restatement(emu, B, C, E, t, r, lam, r_loss, grad_out):
    check_case(emu, "cpu", B, C, E, t, r, lam, r_loss, grad_out, seed=B * 1009 + C * 31 + E)


@pytest.mark.parametrize("what", ["overflow", "bias NULL", "dfeat NULL", "dbias NULL"])
def test_emulated_loss_variants(emu, what):
    """Overflowing exps give the restatement's inf loss and NaN rows; NULL bias, dfeat and dbias follow the head's rules."""
    check_case(emu, "cpu", 20, 260, 64, 3, 30.0, 0.7, 30.0, 10.0, seed=7, overflow=what == "overflow", bias_on=what != "bias NULL",
                   need_dfeat=what != "dfeat NULL", need_dbias=what != "dbias NULL")


def check_empty(lib, dev):
    """B = 0: NaN loss, zero dweight and dbias.  C = 0: zero loss and row sums, the feature norms, zero dfeat."""
    E = 8
    w = np.random.default_rng(0).standard_normal((3, E)).astype(np.float32)
    got = run_abi(lib, dev, np.zeros((0, E), np.float32), w, np.zeros(3, np.float32), np.zeros(0, np.int64), 3, 30.0, 0.7,
                  30.0, 10.0)
    assert np.isnan(got["loss"][0]) and (got["dweight"] == 0).all() and (got["dbias"] == 0).all()
    f = np.random.default_rng(1).standard_normal((4, E)).astype(np.float32)
    got = run_abi(lib, dev, f, np.zeros((0, E), np.float32), np.zeros(0, np.float32), np.arange(4, dtype=np.int64), 3, 30.0,
                  0.7, 30.0, 10.0)
    assert got["loss"][0] == 0 and (got["row_loss"] == 0).all() and (got["dfeat"] == 0).all()
    np.testing.assert_allclose(got["inv_nf"], 1 / np.linalg.norm(f.astype(np.float64), axis=1), rtol=1e-6)


def check_error_codes(lib, dev):
    """Bad sizes, NULL pointers and emb > 1024 are refused before any launch (PFC_E_ARG, PFC_E_SHAPE), and nothing is
    written; an empty batch needs only loss and ticket."""
    f = torch.zeros(64, device=dev)
    lab = torch.zeros(4, dtype=torch.int64, device=dev)
    tk = torch.zeros(1, dtype=torch.int32, device=dev)
    out = torch.full((64,), 7.0, device=dev)
    st = _stream(dev)

    def fwd(feat=f, weight=f, label=lab, B=2, C=2, E=8, loss=out, row=out, ticket=tk, cos=out, inf=out, inw=out):
        return lib.pfc_bce_loss_fwd(_ptr(feat), _ptr(weight), None, _ptr(label), B, C, E, M, 30.0, 3.0, 0.1, 0.2, _ptr(loss),
                                    _ptr(row), _ptr(ticket), _ptr(cos), _ptr(inf), _ptr(inw), st)

    def bwd(feat=f, weight=f, label=lab, go=f, B=2, C=2, E=8, dw=out):
        return lib.pfc_bce_loss_bwd(_ptr(feat), _ptr(weight), None, _ptr(label), _ptr(f), _ptr(f), _ptr(f), _ptr(go), B, C, E, M,
                                    30.0, 3.0, 0.1, 0.2, _ptr(out), _ptr(dw), _ptr(out), st)

    assert fwd(B=-1) == E_ARG and fwd(C=-1) == E_ARG and fwd(E=0) == E_ARG and fwd(E=1025) == E_SHAPE
    assert fwd(B=1 << 31) == E_SHAPE
    for k in ("feat", "weight", "label", "loss", "row", "ticket", "cos", "inf", "inw"):
        assert fwd(**{k: None}) == E_ARG, k
    assert fwd(B=0, loss=None) == E_ARG
    assert bwd(B=-1) == E_ARG and bwd(C=-1) == E_ARG and bwd(E=0) == E_ARG and bwd(E=1025) == E_SHAPE
    assert bwd(B=1 << 30, C=1 << 30) == E_SHAPE
    for k in ("feat", "weight", "label", "go", "dw"):
        assert bwd(**{k: None}) == E_ARG, k
    assert bool((out == 7.0).all()) and int(tk.cpu()[0]) == 0
    loss = torch.zeros(1, device=dev)
    assert fwd(B=0, feat=None, label=None, row=None, cos=None, inf=None, loss=loss) == 0
    assert bool(torch.isnan(loss.cpu()[0])) and int(tk.cpu()[0]) == 0


def test_emulated_loss_empty(emu):
    check_empty(emu, "cpu")


def test_emulated_loss_error_codes(emu):
    check_error_codes(emu, "cpu")


@pytest.mark.skipif(os.environ.get("EMU_ASAN") == "1", reason="this IS the sanitizer child")
def test_emulated_loss_under_address_sanitizer():
    """Every emulated test above once more in a child whose emulated build is compiled with -fsanitize=address and runs
    threads and blocks in descending order (EMU_SCHEDULE=reverse): an out-of-bounds access aborts the child, a result
    that depends on the schedule differs."""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not available")
    env = dict(os.environ, LD_PRELOAD=asan, EMU_ASAN="1", EMU_SCHEDULE="reverse",
               ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "emulated"], env=env, capture_output=True, text=True, cwd=ROOT, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0 and "AddressSanitizer" not in r.stdout + r.stderr.replace(
        "ASan doesn't fully support makecontext/swapcontext", ""), tail
