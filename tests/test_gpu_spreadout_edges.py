"""SpreadOut's tensor-core kernels at the edges of their dispatch, row by row.

``pfc_spreadout`` runs ``logits2_kernel<MODE_HINGE>`` with ``x_hat := w_hat`` (its epilogue masks the diagonal, the
padded columns and rows, stores H = relu(S - margin) as bf16 and sums H^2 per row), then the dx GEMM on that scratch
(``dx2`` or ``dx<256|128|64>``, chosen with a cluster size and a K split by ``make_spread_plan``) and
``reduce_dx_kernel``.  The aggregate bounds of ``test_spreadout.py`` cannot see a dropped class tile, a wrong last row
block or a K-split slice left out of the sum; here every row is held to an fp64 restatement with the kernels' operand
roundings (the library's own bf16 ``w_hat``, bf16 H), so that only the order of summation differs.

The workspace is filled with 0xFF bytes (NaN in bf16: an H element the dx GEMM reads but the hinge epilogue did not
write turns the row into NaN even where TMA pads with zeros, NaN * 0 = NaN).  ``part_max`` / ``part_sum`` get sentinel
rows past the count ``pfc_spreadout_num_partials`` documents, ``hw_out`` guard rows past the last row, and the
workspace slack on either side of the aligned window stays as filled: none of them may change."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from test_gpu_kernel_edges import _guarded, _same_bits, knobs  # noqa: E402
from test_spreadout import _centres  # noqa: E402

SMS = 148                  # B200
BM, BK = 128, 64           # row block and k-block of the kernels (csrc/tc_kernels.cu)
EXTRA_PARTIALS = SMS       # sentinel rows past the documented count: more than a 148-SM device can launch CTAs
ZERO_MARGIN = 1.01         # bf16 rounding can lift the cosine of two equal unit rows to (1 + 2^-9)^2 < 1.004
GRAD_OUT = 3.0
# per-row loss: each slot sums H^2 of up to ceil(n / 32) column groups in fp32, a relative error of at most
# ceil(n / 32) 2^-24 = 7.5e-5 at n = 40 000 (typically its square root), and S itself is an fp32 sum of E bf16 products
LOSS_ROW_TOL = 1e-4
ROWS_MAX, ROWS_RMS = 1e-2, 1e-3    # selfcheck.check_head_step: bf16(H) may round the other way where S differs in fp32


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------------ plan mirror
def pair_items(n):
    """(class tiles, [(t0, t1) items of each CTA pair]) of ``logits2_kernel`` on an [n, n] problem (``pair_grid``)."""
    n_rp, n_ct = (cdiv(n, BM) + 1) // 2, cdiv(n, 256)
    items = n_rp * n_ct
    pairs = min(items, SMS // 2)
    return n_ct, [(items * p // pairs, items * (p + 1) // pairs) for p in range(pairs)]


def spread_plan(n, emb, dx_pair=1, dx_cluster=2):
    """``make_spread_plan`` on a 148-SM device.  Only used to choose and label cases."""
    n_rb = cdiv(n, BM)
    dx_bn = min(emb, 256)
    n_eh = emb // dx_bn
    pair = bool(dx_pair) and emb >= 256 and n_rb % 4 == 0
    dcs = 1 if dx_bn < 128 else min(dx_cluster, 2) if dx_bn == 128 else dx_cluster
    units = n_rb // 4 * n_eh * 2 if pair else cdiv(n_rb, dcs) * dcs * n_eh
    n_kb = cdiv(n, BK)
    return {"kernel": "dx2" if pair else "dx<%d>" % dx_bn, "clamped": not pair and dcs != dx_cluster,
            "ksplit": max(1, min(SMS // units, n_kb, 64)), "n_kb": n_kb, "n_rb": n_rb}


def plan_features(n, emb, settings=None):
    settings = settings or {}
    pl = spread_plan(n, emb, settings.get("dx_pair", (1,))[0], settings.get("clusters", (2, 2))[0])
    f = {pl["kernel"]}
    if pl["clamped"]:
        f.add("cluster clamp")
    if pl["ksplit"] == 1:
        f.add("ksplit 1")
    if pl["ksplit"] == pl["n_kb"]:
        f.add("ksplit n_kb")
    if 1 < pl["ksplit"] < pl["n_kb"]:
        f.add("1 < ksplit < n_kb")
    if pl["n_rb"] % 2:
        f.add("odd n_rb")
    if 1 <= n % 256 <= 128:
        f.add("last tile half empty")
    if n % 64:
        f.add("n % 64 != 0")
    n_ct, ranges = pair_items(n)
    if any(t1 - t0 >= 2 and t0 // n_ct != (t1 - 1) // n_ct for t0, t1 in ranges):
        f.add("pair crosses row pairs")
    return f


REQUIRED = {"dx2", "dx<256>", "dx<128>", "dx<64>", "cluster clamp", "ksplit 1", "ksplit n_kb", "1 < ksplit < n_kb", "odd n_rb",
            "last tile half empty", "n % 64 != 0", "pair crosses row pairs"}

# (n, E); the comments say what a 148-SM device runs
SHAPES = [
    (1, 512),          # one row: only the diagonal, everything 0
    (2, 64),           # dx<64>, cluster 2 -> 1
    (3, 128),          # dx<128>
    (127, 256),        # dx<256>, ksplit = n_kb = 2, phantom second row block
    (128, 512),        # one full row block
    (129, 512),        # one row past a block: n_rb = 2
    (255, 64),
    (256, 128),        # one full class tile
    (257, 256),        # one class past a tile: odd n_rb, the second CTA's half of the last tile is empty
    (383, 512),
    (512, 512),        # dx2, ksplit = n_kb = 8
    (1000, 256),       # dx2 with a ragged last block, ksplit = n_kb = 16
    (6000, 512),       # FedFR's public classes: odd n_rb, ksplit 1, pairs over several items across row pairs
    (6144, 512),       # dx2, ksplit 3
    (40000, 512),      # tools/spreadout_bench.py
]
MARGINS = [0.7, 0.4, 0.0, -0.5, ZERO_MARGIN]      # 0.7: the reference default; < 0 makes H dense and the padded masks visible
DIRECT = [(n, e, m) for n, e in SHAPES for m in MARGINS]

# (id, knob settings, n, E), all at margin -0.5
VARIANTS = [("dx_pair_0_n%d" % n, {"dx_pair": (0,)}, n, 512) for n in (512, 6144)] + [
    ("clusters_%d_e%d" % (c, e), {"clusters": (c, c)}, 300, e) for e in (128, 256, 512) for c in (1, 2, 4)] + [
    # the single-CTA logits kernels of the head: the hinge GEMM still runs on the CTA-pair kernel, with its own count
    ("logits_pair_0_tile%d_n%d" % (t, n), {"logits_pair": (0,), "logits_tile": (t,)}, n, 256) for t in (128, 256) for n in (100, 300)]

# (n, E, margin, mode) of SpreadOut_Module.  n = 5 is the smallest make_fc input whose exact FC.grad is not 0: at n = 2 and 3
# every pair over the margin is two equal rows, whose cosine is stationary, so the exact gradient vanishes and a relative
# error against it means nothing (test_direct holds those shapes row by row)
MODULE = [(5, 64, 0.7, "mean"), (129, 512, -0.5, "sum"), (383, 512, 0.4, "mean"), (1000, 256, 0.0, "sum"), (6000, 512, 0.4, "sum"),
          (6000, 512, -0.5, "mean"), (6144, 512, 0.7, "sum")]


def make_fc(n, e):
    """Clustered centres (``test_spreadout._centres``) with exact duplicates of row 0 in the first row, across the first
    row-block and class-tile boundaries and in the last row block (S = 1 off the diagonal must count), and the last row
    antipodal to row 0."""
    fc = _centres(n, e, 7 * n + e)
    for i in (1, 128, 256, n - 2):
        if 1 <= i <= n - 2 or (n == 2 and i == 1):
            fc[i] = fc[0]
    if n >= 3:
        fc[n - 1] = -fc[0]
    return fc


# ------------------------------------------------------------------------------------------------ reference
def reference(w, w_hat, inv_norm, margin, mean=False, grad_out=1.0, bf16_h=True, chunk=2048):
    """fp64 restatement of ``pfc_spreadout`` and of the glue in ``spreadout.py``, in row chunks (n = 40 000 fits):
    S = w_hat w_hat^T, H = relu(S - margin) with H_ii = 0 (by index, not by value), rows_i = sum_j H_ij^2,
    hw = bf16(H) w_hat (``bf16_h``) or H w_hat; loss = scale sum_i rows_i and
    FC.grad = grad_out (g - u (u . g)) inv_norm with g = 4 scale hw, u = w inv_norm (the normalize backward).
    ``w`` [n, E] are the rows of FC, ``w_hat`` / ``inv_norm`` the operands (the library's, or exact ones)."""
    wh = w_hat.double()
    n = wh.shape[0]
    rows = torch.empty(n, dtype=torch.float64, device=wh.device)
    hw = torch.empty_like(wh)
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        h = (wh[r0:r1] @ wh.t() - margin).clamp_min_(0.0)
        i = torch.arange(r0, r1, device=wh.device)
        h[i - r0, i] = 0.0
        rows[r0:r1] = (h * h).sum(dim=1)
        if bf16_h:
            h = h.float().to(torch.bfloat16).double()
        hw[r0:r1] = h @ wh
    scale = 1.0 / (n * (n - 1)) if mean and n > 1 else 1.0
    inv = inv_norm.double()[:, None]
    u = w.double() * inv
    g = hw * (4.0 * scale)
    grad = (g - u * (u * g).sum(dim=1, keepdim=True)) * inv * grad_out
    return {"rows": rows, "loss": rows.sum() * scale, "hw": hw, "grad": grad}


def exact_reference(fc, margin, mean=False, grad_out=1.0, chunk=2048):
    """``reference`` with fp64 operands and no bf16 anywhere: what autograd of the reference formulation gives."""
    w = fc.double()
    norm = w.norm(dim=1).clamp_min(1e-12)
    return reference(w, w / norm[:, None], 1.0 / norm, margin, mean, grad_out, bf16_h=False, chunk=chunk)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


@pytest.mark.parametrize("n,e,margin,mode", [(40, 64, 0.7, "sum"), (40, 64, 0.0, "mean"), (33, 32, -0.5, "sum"), (2, 16, 0.4, "mean"),
                                             (1, 8, -0.5, "sum")])
def test_exact_reference_is_autograd_of_the_oracle(n, e, margin, mode):
    """The restatement the GPU rows are held to is pinned to the reference formulation (``oracle.spreadout_loss``,
    itself pinned to the unmodified class by ``test_spreadout``): fp64 loss and autograd gradient, chunked in 7 rows."""
    from oracle import partial_fc_oracle as O
    fc = make_fc(n, e).double().requires_grad_(True)
    loss = O.spreadout_loss(fc, margin, mode)
    (GRAD_OUT * loss).backward()
    ref = exact_reference(fc.detach(), margin, mode == "mean", GRAD_OUT, chunk=7)
    assert abs(float(ref["loss"]) - loss.item()) <= 1e-12 * max(abs(loss.item()), 1e-300)
    assert float((ref["grad"] - fc.grad).abs().max()) <= 1e-12 * (1.0 + float(fc.grad.abs().max()))   # n = 2: the gradient is 0


@pytest.mark.parametrize("n,e,margin", [(300, 256, 0.4), (300, 64, -0.5)])
def test_emulated_reference_differs_by_bf16_rounding_only(n, e, margin):
    """With bf16 operands and bf16 H the restatement moves by what bf16 rounding explains, and no more."""
    fc = make_fc(n, e)
    inv = 1.0 / fc.norm(dim=1).clamp_min(1e-12)
    emu = reference(fc, (fc * inv[:, None]).to(torch.bfloat16), inv, margin, grad_out=GRAD_OUT, chunk=64)
    exact = exact_reference(fc, margin, grad_out=GRAD_OUT)
    assert abs(float(emu["loss"] - exact["loss"])) <= 1e-2 * float(exact["loss"])
    assert _rel(emu["grad"], exact["grad"]) < 2e-2


def test_case_matrix_reaches_every_branch():
    """The shapes and knob variants reach every branch of ``make_spread_plan`` and every edge of the hinge GEMM's schedule
    on a 148-SM device (the mirror above; it chooses cases, the library decides)."""
    seen = set()
    for n, e in SHAPES:
        seen |= plan_features(n, e)
    for _vid, settings, n, e in VARIANTS:
        seen |= plan_features(n, e, settings)
    assert REQUIRED <= seen, REQUIRED - seen
    assert [spread_plan(n, e)["kernel"] for n, e in [(512, 512), (1000, 256), (6144, 512)]] == ["dx2"] * 3
    assert spread_plan(6144, 512)["ksplit"] == 3 and spread_plan(6000, 512)["ksplit"] == 1


def test_partial_count_ignores_the_head_knobs():
    """The hinge GEMM always runs on the CTA-pair kernel: its partial count may not follow the head's logits knobs."""
    import __graft_entry__ as g
    g.build()
    from fedfr_b200 import _native as N
    assert N.lib.pfc_spreadout_num_partials(0, 512) == 0
    shapes = [(n, 256) for n in (1, 100, 128, 129, 300, 640, 1920, 6000, 40000)]
    want = [N.lib.pfc_spreadout_num_partials(n, e) for n, e in shapes]
    assert all(c >= 2 and c % 2 == 0 for c in want)
    for settings in ({"logits_pair": (0,)}, {"logits_pair": (0,), "logits_tile": (256,)}, {"logits_tile": (256,)}):
        with knobs(**settings):
            assert [N.lib.pfc_spreadout_num_partials(n, e) for n, e in shapes] == want, settings


# ------------------------------------------------------------------------------------------------ GPU driver
@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


@pytest.fixture
def defaults(pkg):
    with knobs():
        yield


def normalize(w):
    """The library's bf16 ``w_hat`` and fp32 ``inv_norm`` of the rows of ``w`` (as ``spreadout.py`` makes them)."""
    from fedfr_b200 import _native as N
    n, e = w.shape
    w_hat = torch.empty((n, e), dtype=torch.bfloat16, device=w.device)
    inv_norm = torch.empty(n, dtype=torch.float32, device=w.device)
    N.check(N.lib.pfc_normalize_rows(N.ptr(w), None, n, e, N.ptr(w_hat), None, N.ptr(inv_norm), torch.cuda.current_stream().cuda_stream),
            "pfc_normalize_rows")
    return w_hat, inv_norm


class Buffers:
    """The outputs and workspace of one ``pfc_spreadout`` call, with sentinels: ``part`` [2, count + EXTRA_PARTIALS, n] and
    the workspace filled with 0xFF bytes, ``hw`` followed by random guard rows."""

    def __init__(self, n, e, dev):
        from fedfr_b200 import _native as N
        self.n, self.e = n, e
        self.n_part = N.lib.pfc_spreadout_num_partials(n, e)
        self.part = torch.empty((2, self.n_part + EXTRA_PARTIALS, n), dtype=torch.float32, device=dev)
        self.part.view(torch.uint8).fill_(0xFF)
        self.hw, self.tail, self.tail_want = _guarded(n, e, torch.Generator(device=dev).manual_seed(n))
        self.nbytes = N.lib.pfc_spreadout_workspace_bytes(n, e)
        self.ws = torch.full((self.nbytes + 2048,), 0xFF, dtype=torch.uint8, device=dev)
        self.off = (-self.ws.data_ptr()) % 1024

    def call(self, w_hat, margin, n=None, e=None, ws_bytes=None, ws_shift=0, null_w_hat=False):
        from fedfr_b200 import _native as N
        return N.lib.pfc_spreadout(None if null_w_hat else N.ptr(w_hat), self.n if n is None else n, self.e if e is None else e, float(margin),
                                   N.ptr(self.part[0]), N.ptr(self.part[1]), N.ptr(self.hw), self.ws.data_ptr() + self.off + ws_shift,
                                   self.nbytes if ws_bytes is None else ws_bytes, torch.cuda.current_stream().cuda_stream)

    def untouched(self):
        """Every byte outside what the call may write still holds what was put there."""
        extra = self.part[:, self.n_part:]
        slack = torch.cat([self.ws[:self.off], self.ws[self.off + self.nbytes:]])
        return {"partial rows past the count": bool((extra.contiguous().view(torch.uint8) == 0xFF).all()),
                "hw_out guard rows": _same_bits(self.tail, self.tail_want),
                "workspace slack": bool((slack == 0xFF).all())}


def edge_groups(n):
    """Row sets held to the max-row bound on their own: the last row block, the last class tile (rows are classes too)
    and the rows within +-1 of every 128-row boundary (which includes the 256-class tile boundaries)."""
    near = sorted({i for b in range(BM, n, BM) for i in (b - 1, b, b + 1) if 0 <= i < n})
    return {"last row block": torch.arange((n - 1) // BM * BM, n), "last class tile": torch.arange((n - 1) // 256 * 256, n),
            "rows at 128 / 256 boundaries": torch.tensor(near, dtype=torch.long)}


def check_rows(name, got, want, errs):
    """``selfcheck.check_head_step``'s row criteria on all rows, and the max-row bound on each edge group alone."""
    from fedfr_b200 import selfcheck as SC
    errs[name] = (SC._rows_err(got, want), SC._rows_err(got, want, rms=True))
    assert errs[name][0] <= ROWS_MAX and errs[name][1] <= ROWS_RMS, (name, errs)
    for group, idx in edge_groups(got.shape[0]).items():
        if len(idx):
            idx = idx.to(got.device)
            errs[name + ", " + group] = SC._rows_err(got[idx], want[idx])
            assert errs[name + ", " + group] <= ROWS_MAX, (name, group, errs)


def check_loss_rows(got, want, errs):
    """Per-row loss: exactly 0 where the reference row is 0, within LOSS_ROW_TOL elsewhere."""
    zero = want == 0
    assert bool((got[zero] == 0).all()), ("rows with no pair over the margin", int((got[zero] != 0).sum()))
    errs["loss rows"] = float(((got - want).abs() / want)[~zero].max()) if bool((~zero).any()) else 0.0
    assert errs["loss rows"] <= LOSS_ROW_TOL, errs
    return zero


def run_direct(n, e, margin):
    """``pfc_normalize_rows`` then ``pfc_spreadout`` as ``spreadout.py`` calls them, on sentinel buffers; every row checked.
    Returns the measured errors."""
    from fedfr_b200 import _native as N
    w = make_fc(n, e).cuda()
    w_hat, inv_norm = normalize(w)
    b = Buffers(n, e, w.device)
    N.check(b.call(w_hat, margin), "pfc_spreadout")
    torch.cuda.synchronize()
    untouched = b.untouched()
    assert all(untouched.values()), untouched
    rows = b.part[1, :b.n_part].double().sum(dim=0)
    assert bool(torch.isfinite(rows).all()) and bool(torch.isfinite(b.hw).all())
    ref = reference(w, w_hat, inv_norm, margin)
    errs = {}
    zero = check_loss_rows(rows, ref["rows"], errs)
    assert bool((b.hw[zero] == 0).all())
    if margin >= 1:
        assert bool(zero.all()) and not bool(b.hw.any())
    elif n > 1:
        assert not bool(zero.all())
        check_rows("hw_out", b.hw, ref["hw"], errs)
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("n,e,margin", DIRECT)
def test_direct(defaults, n, e, margin):
    print("errors", run_direct(n, e, margin))


@pytest.mark.gpu
@pytest.mark.parametrize("vid,settings,n,e", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_knob_variant(defaults, vid, settings, n, e):
    with knobs(**settings):
        print("errors", run_direct(n, e, -0.5))


@pytest.mark.gpu
@pytest.mark.parametrize("n,e,margin,mode", MODULE)
def test_module(defaults, pkg, n, e, margin, mode):
    """``SpreadOut_Module`` end to end with ``grad_out`` != 1: every row of ``FC.grad`` against the emulated reference, and
    the loss and ``FC.grad`` against autograd of the reference formulation in fp64 (the bounds of ``test_spreadout``)."""
    from oracle import partial_fc_oracle as O
    fc = make_fc(n, e)
    mod = pkg.SpreadOut_Module(fc.clone().cuda(), margin=margin, mode=mode)
    loss = mod()
    (GRAD_OUT * loss).backward()
    torch.cuda.synchronize()
    w = fc.cuda()
    w_hat, inv_norm = normalize(w)
    ref = reference(w, w_hat, inv_norm, margin, mode == "mean", GRAD_OUT)
    errs = {"loss": abs(loss.item() - float(ref["loss"])) / float(ref["loss"])}
    assert errs["loss"] <= LOSS_ROW_TOL, errs
    assert bool(torch.isfinite(mod.FC.grad).all())
    check_rows("FC.grad", mod.FC.grad, ref["grad"], errs)
    ref_fc = fc.double().requires_grad_(True)
    exact = O.spreadout_loss(ref_fc, margin, mode)
    (GRAD_OUT * exact).backward()
    errs["exact"] = (abs(loss.item() - exact.item()) / exact.item(), _rel(mod.FC.grad.cpu(), ref_fc.grad))
    assert errs["exact"][0] <= 1e-2 and errs["exact"][1] < 2e-2, errs
    print("errors", errs)


# ------------------------------------------------------------------------------------------------ ABI errors
@pytest.mark.gpu
@pytest.mark.parametrize("what", ["emb 33", "n 0", "n 2^24", "workspace one byte short", "workspace misaligned", "null w_hat"])
def test_abi_errors(defaults, what):
    """Each bad argument is refused with its code before anything is enqueued: no launch, no byte of any buffer changed."""
    from fedfr_b200 import _native as N
    n, e = 300, 256
    w_hat, _ = normalize(make_fc(n, e).cuda())
    b = Buffers(n, e, w_hat.device)
    hw0 = b.hw.clone()
    args, want = {"emb 33": ({"e": 33}, -2), "n 0": ({"n": 0}, -1), "n 2^24": ({"n": 1 << 24}, -2),
                  "workspace one byte short": ({"ws_bytes": b.nbytes - 1}, -4), "workspace misaligned": ({"ws_shift": 512}, -1),
                  "null w_hat": ({"null_w_hat": True}, -1)}[what]
    torch.cuda.synchronize()
    launches = N.lib.pfc_launch_count()
    assert b.call(w_hat, 0.4, **args) == want
    torch.cuda.synchronize()
    assert N.lib.pfc_launch_count() == launches
    assert bool((b.part.view(torch.uint8) == 0xFF).all()) and bool((b.ws == 0xFF).all()) and _same_bits(b.hw, hw0)
    assert all(b.untouched().values())
