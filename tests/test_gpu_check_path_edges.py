"""Check mode (``PFC_PATH_CHECK``: ``normalize_rows``' fp32 branch, ``csrc/simt_check.cu``, ``csrc/stats.cu``) at the edges of
its backward chunks, tiles, class splits and embedding sizes, row by row.

Check mode is the head's fp32 cross-check of the tensor-core kernels and the only path for embedding sizes other than
64 / 128 / 256 / 512.  ``simt_bwd`` walks the classes in chunks of ``check_chunk(Bt, Cs)`` columns (a 64 MiB fp32 G
scratch, at least one 64-column tile, at most 65,535 tiles: ``grad_logits_kernel`` puts the class tiles on gridDim.y);
only chunks after the first accumulate into dx and offset the class base, ``w_hat``, ``inv_norm`` and ``dw``.

Each case drives the head through ``run_shards`` (W virtual ranks, the provider calls of ``PartialFC.forward_backward``)
with every library scratch filled with 0xFF bytes and guard rows after ``dx`` and ``dw``, and holds the loss and every row
of ``dx`` / ``dw`` to an fp64 restatement that uses the library's own fp32 ``w_hat`` and ``inv_norm``, so that only the
order of summation differs (``restate``, itself pinned to fp64 autograd of partial_fc.py + losses.py and to the golden
steps by the CPU tests below)."""
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from test_gpu_kernel_edges import _guarded, _same_bits, knobs, run_shards, shard_geometry  # noqa: E402

S, M_COS, M_ARC = 64.0, 0.4, 0.5
S_CPU = 30.0
EPS = 1e-12                        # F.normalize default (partial_fc.py:127)
U = 2.0 ** -24                     # fp32 unit roundoff
# Fixed per-row criteria of the softmax gradient (selfcheck._rows_err: per-row relative error, floor 1 % of the rms row
# norm), ten times tighter than the bf16 criteria of selfcheck.check_head_step.  The fp32 chains are: a cosine of E fma in
# k order (tile_gemm), expf (2 ulp), one division by the row sum, and the dx / dwh GEMMs of up to Cs (Bt) fma; the
# cosine's rounding is amplified by s = 64 in p = exp(s cos - M) / S, which is what dominates the measured error.
LOSS_TOL = 1e-5
ROWS_MAX, ROWS_RMS = 1e-3, 1e-4


def check_chunk(n_rows, n_classes):
    """Mirror of ``check_chunk`` in csrc/simt_check.cu (chooses cases; the library decides)."""
    chunk = (64 << 20) // (n_rows * 4) // 64 * 64
    chunk = min(max(chunk, 64), 65535 * 64)
    return min(chunk, (n_classes + 63) // 64 * 64)


def chunk_starts(n_rows, n_classes):
    return list(range(0, n_classes, check_chunk(n_rows, n_classes)))


def clamped_inv():
    """fp32 1 / eps: the inv_norm of a row whose norm was clamped (a correctly rounded division, as on the device)."""
    return float(torch.tensor([1.0], dtype=torch.float32) / torch.tensor([EPS], dtype=torch.float32))


# ------------------------------------------------------------------------------------------------ restatement
def restate(x, y, w_hat, inv_norm, clamped, s, m, kind):
    """fp64 step over all C classes of all ranks: x [Bt, E], y [Bt] global labels, w_hat [C, E] / inv_norm [C] the
    normalised rows and their inverse norms, ``clamped`` [C] bool the rows whose norm was clamped to eps.
    z = s margin(x w_hat^T), p = softmax(z), loss = mean(-log max(p_y, 1e-30)),
    G = s (p - onehot) / Bt (target column times the margin slope), dx = G w_hat, dwh = G^T x,
    dw = (dwh - w_hat (w_hat . dwh)) inv_norm, without the radial term on clamped rows (the norm is then a constant).
    Returns dict(loss, dx [Bt, E], dw [C, E]) in fp64."""
    from fedfr_b200 import selfcheck as SC
    X, Wh = x.double(), w_hat.double()
    Bt = X.shape[0]
    z = X @ Wh.t()
    rows = torch.arange(Bt, device=X.device)
    mc, slope = SC._margin(z[rows, y], m, kind)
    z = z * s
    z[rows, y] = mc * s
    lse = torch.logsumexp(z, dim=1)
    logp = z[rows, y] - lse
    loss = torch.minimum(-logp, torch.full_like(logp, -math.log(1e-30))).mean()
    G = torch.exp(z - lse[:, None]).mul_(s / Bt)
    G[rows, y] = (G[rows, y] - s / Bt) * slope
    dx = G @ Wh
    dwh = G.t() @ X
    del G, z
    rad = (Wh * dwh).sum(dim=1, keepdim=True)
    rad[clamped.to(rad.device)] = 0.0
    dw = (dwh - Wh * rad) * inv_norm.double()[:, None]
    return {"loss": loss, "dx": dx, "dw": dw}


def autograd_reference(x, y, w, s, m, kind):
    """fp64 autograd of the reference formulation: partial_fc.py:127 (F.normalize, linear), losses.py:23-29 (CosFace) or
    :38-45 (ArcFace, acos / cos over the whole matrix), partial_fc.py:140-162 (softmax, -log max(p_y, 1e-30), mean)."""
    xr, wr = x.double().requires_grad_(True), w.double().requires_grad_(True)
    cos = xr @ F.normalize(wr).t()
    onehot = F.one_hot(y, w.shape[0]).double()
    if kind == 0:
        logits = (cos - m * onehot) * s
    else:
        logits = torch.cos(torch.acos(cos) + m * onehot) * s
    p = torch.softmax(logits, dim=1)
    loss = -(p.gather(1, y[:, None]).clamp_min(1e-30).log()).mean()
    loss.backward()
    return loss.detach(), xr.grad, wr.grad


def exact_operands(w):
    n = w.double().norm(dim=1)
    nc = n.clamp_min(EPS)
    return w.double() / nc[:, None], 1.0 / nc, n < EPS


def _cpu_inputs(Bt, C, E, seed, special_rows=True):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(C, E, generator=g, dtype=torch.float64) * 0.01
    y = torch.randint(0, C, (Bt,), generator=g)
    x = F.normalize(torch.randn(Bt, E, generator=g, dtype=torch.float64) + 2.0 * F.normalize(w[y]) * (torch.arange(Bt) % 4 == 0)[:, None])
    if special_rows:
        w[1] = 0.0
        w[2] = F.normalize(w[2], dim=0) * 0.9e-12
        y[:2] = torch.tensor([1, 2])
    return x, y, w


@pytest.mark.parametrize("Bt,C,E,kind", [(40, 70, 20, 0), (33, 65, 132, 1), (7, 5, 4, 0), (64, 130, 100, 1)])
def test_restatement_is_autograd_of_the_reference(Bt, C, E, kind):
    """The restatement equals fp64 autograd of partial_fc.py + losses.py, including a zero weight row and one with
    0 < |w| < eps (autograd of F.normalize gives it d / eps, no radial term).  s = 30 keeps every p_y above the 1e-30
    floor, where autograd of the clamped loss and partial_fc.py's hand-written gradient part (the golden steps pin that)."""
    x, y, w = _cpu_inputs(Bt, C, E, Bt + C + E)
    m = M_COS if kind == 0 else M_ARC
    loss, gx, gw = autograd_reference(x, y, w, S_CPU, m, kind)
    ref = restate(x, y, *exact_operands(w), S_CPU, m, kind)
    assert abs(float(ref["loss"]) - float(loss)) <= 1e-10 * float(loss)
    assert float((ref["dx"] - gx).abs().max()) <= 1e-11 * float(gx.abs().max())
    for r in range(C):                                       # the clamped row's gradient is ~1e12 times the others
        assert float((ref["dw"][r] - gw[r]).abs().max()) <= 1e-11 * (float(gw[r].abs().max()) + 1e-300), r


def test_radial_term_on_a_clamped_row_is_not_autograd():
    """The formula the kernels used before (radial term on every row) differs from autograd on a row with 0 < |w| < eps
    by far more than rounding (by w_hat (w_hat . d) / eps, |w_hat| = |w| / eps), and agrees on a zero row: the deviation
    the clamped-row cases on the device look for."""
    x, y, w = _cpu_inputs(40, 70, 20, 5)
    _, _, gw = autograd_reference(x, y, w, S_CPU, M_COS, 0)
    w_hat, inv, clamped = exact_operands(w)
    old = restate(x, y, w_hat, inv, torch.zeros_like(clamped), S_CPU, M_COS, 0)
    assert float((old["dw"][1] - gw[1]).abs().max()) <= 1e-11 * float(gw[1].abs().max())
    assert float((old["dw"][2] - gw[2]).norm() / gw[2].norm()) > 1e-3


@pytest.mark.parametrize("name", ["w1_sr1_small", "w1_sr1_s30", "w2_sr1_ragged", "w1_arc_small"])
def test_restatement_matches_golden_steps(name):
    """... and reproduces the unmodified reference's stored steps (loss, x_grad of every rank, dw of every shard)."""
    from golden_util import Case
    case = Case(name)
    cfg = case.cfg
    W = cfg["world_size"]
    x, y, w = torch.cat(case.features), torch.cat(case.labels), torch.cat(case.weights)
    kind = 1 if cfg.get("loss", "cosface") == "arcface" else 0
    ref = restate(x, y, *exact_operands(w), cfg["s"], cfg["m"], kind)
    B = x.shape[0] // W
    for r in range(W):
        want_loss = float(case.get(r, 0, "loss"))
        assert abs(float(ref["loss"]) - want_loss) <= 1e-5 * abs(want_loss)
        n_loc, c0 = shard_geometry(cfg["num_classes"], W, r)
        for got, key in ((ref["dx"][r * B:(r + 1) * B] * W, "x_grad"), (ref["dw"][c0:c0 + n_loc], "dw")):
            want = torch.from_numpy(case.get(r, 0, key)).double()
            assert float((got - want).abs().max()) <= 1e-5 * float(want.abs().max()), (r, key)


def test_chunk_mirror():
    """The case matrix reaches what it claims: 1, 2 and 3 backward chunks, the 64-column floor and the grid cap."""
    assert chunk_starts(64, 1000) == [0]
    assert chunk_starts(4096, 8192) == [0, 4096]
    assert chunk_starts(4096, 10000) == [0, 4096, 8192]
    assert chunk_starts(270000, 200) == [0, 64, 128, 192]
    assert chunk_starts(4, 4194305) == [0, 4194240]          # uncapped, 4,194,304 columns would need gridDim.y = 65,536


@pytest.mark.parametrize("Bt,C,E,kind", [(300, 3001, 128, 0), (300, 5001, 1024, 0), (256, 6100, 1024, 1), (4096, 8192, 64, 1)])
def test_dw_groups_see_every_ordinary_row(Bt, C, E, kind):
    """With the clamped rows in the inputs (the weight_rows cases and the public entries), flipping the sign of the
    ordinary target rows, of the ordinary other rows, or of one ordinary row at a chunk edge fails its group: the clamped
    rows' ~1e11 larger gradients do not set the floor of any group that holds ordinary rows."""
    x, y, w = make_inputs(Bt, C, E, 1, 11, weight_rows=True, device="cpu")
    w_hat, inv, clamped = exact_operands(w.double())
    ref = restate(x, y, w_hat, inv, clamped, S, M_COS if kind == 0 else M_ARC, kind)["dw"]
    tgt = torch.zeros(C, dtype=torch.bool)
    tgt[y] = True
    edge = torch.zeros(C, dtype=torch.bool)
    for b in chunk_starts(Bt, C):
        edge[max(b - 1, 0): b + 2] = True
    errs = dw_group_errors(ref, ref, y, clamped, edge)
    assert max(max(e) if isinstance(e, tuple) else e for e in errs.values()) == 0.0
    assert errs["clamped rows, each to its own norm"] == (0.0, 0.0)
    for name, sel in (("target rows", tgt & ~clamped), ("other rows", ~tgt & ~clamped)):
        bad = ref.clone()
        bad[sel] *= -1
        assert min(dw_group_errors(bad, ref, y, clamped, edge)[name]) > 1.0, name
    bad = ref.clone()
    r = int(torch.nonzero(edge & ~clamped)[-1])
    bad[r] *= -1
    assert dw_group_errors(bad, ref, y, clamped, edge)["chunk-edge rows"] > ROWS_MAX
    bad = ref.clone()
    bad[clamped] *= 1.01
    assert min(dw_group_errors(bad, ref, y, clamped, edge)["clamped rows, each to its own norm"]) > ROWS_MAX


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


def make_inputs(Bt, C, E, W, seed, weight_rows=False, device="cuda"):
    """Unit features, a quarter pulled toward their class and every eighth at a target cosine in [0.9, 0.999]; labels at
    the first and last class of every shard and at c0 - 1, c0, c0 + 1 of every backward chunk, one duplicated.
    ``weight_rows``: a zero weight row and one with 0 < |w| < eps, both labelled."""
    g = torch.Generator(device=device).manual_seed(seed)
    w = torch.randn(C, E, generator=g, device=device) * 0.01
    y = torch.randint(0, C, (Bt,), generator=g, device=device)
    special = []
    for r in range(W):
        n_loc, c0 = shard_geometry(C, W, r)
        special += [c0, c0 + n_loc - 1]
        for b in chunk_starts(Bt, n_loc)[1:]:
            special += [c0 + b - 1, c0 + b, c0 + b + 1]
    if weight_rows:
        zr, cr = C // 3 + 5, C // 2 + 3          # away from the chunk starts, whose labels are ordinary rows
        w[zr] = 0.0
        w[cr] = F.normalize(w[cr], dim=0) * 0.9e-12
        special = [zr, cr] + special
    special = [c for c in special if 0 <= c < C][:Bt]
    pos = torch.randperm(Bt, generator=g, device=device)
    y[pos[:len(special)]] = torch.tensor(special, dtype=y.dtype, device=device)
    if Bt > len(special) + 1:
        y[pos[len(special)]] = y[pos[0]]
    wy = F.normalize(w[y])
    x = F.normalize(torch.randn(Bt, E, generator=g, device=device) + 2.0 * wy * (torch.arange(Bt, device=device) % 4 == 0)[:, None])
    hi = torch.nonzero(torch.arange(Bt, device=device) % 8 == 1).flatten()
    if len(hi) and E > 1:
        c = torch.linspace(0.9, 0.999, len(hi), device=device)[:, None]
        n = torch.randn(len(hi), E, generator=g, device=device)
        n = F.normalize(n - (n * wy[hi]).sum(dim=1, keepdim=True) * wy[hi])
        x[hi] = F.normalize(c * wy[hi] + (1 - c * c).sqrt() * n)
    if weight_rows:                      # the clamped row's samples at cosine 0.6: a radial term of O(1) if one were applied
        at = torch.nonzero(y == cr).flatten()
        n = torch.randn(len(at), E, generator=g, device=device)
        n = F.normalize(n - (n * wy[at]).sum(dim=1, keepdim=True) * wy[at])
        x[at] = 0.6 * wy[at] + 0.8 * n
    return x, y, w


def check_normalize(w, w_hat, inv_norm, errs):
    """The two outputs of ``normalize``, each against what its own chain allows.

    ``inv_norm`` within the chain bound of 1 / max(|w|, eps): the sum of squares is a chain of L = 4 ceil(E / 128) + 5
    roundings of positive terms (each lane's float4s, then the warp tree), relative error <= L u; sqrt halves it and adds
    u / 2, the reciprocal another u / 2.

    ``w_hat`` is not held to one ulp of the fp64 normalisation w / |w|: it is w / fl(norm), and the fp32 norm itself can
    be several ulp off (the chain above), so no correct kernel meets that bound at every emb.  It is held instead to
    w * inv_norm with the kernel's own inv_norm: w_hat = fl(w / norm) is one rounding from w / norm, and inv_norm =
    fl(1 / norm) is one rounding from 1 / norm, so |w_hat - w inv_norm| <= 2u / (1 - u) |w inv_norm| = 1.19e-7.  This
    is a rigorous bound, not a fit: measured maxima reach 0.99 of it, as two roundings in opposite directions can."""
    E = w.shape[1]
    q = w.double() * inv_norm.double()[:, None]
    errs["w_hat / (w inv_norm) - 1"] = float(((w_hat.double() - q).abs() / q.abs().clamp_min(1e-300))[q != 0].max()) if bool((q != 0).any()) else 0.0
    assert bool((w_hat[q == 0] == 0).all())
    assert errs["w_hat / (w inv_norm) - 1"] <= 2 * U / (1 - U), errs
    L = 4 * -(-E // 128) + 5
    ref = 1.0 / w.double().norm(dim=1).clamp_min(EPS)
    errs["inv_norm rel"] = float(((inv_norm.double() - ref).abs() / ref).max())
    assert errs["inv_norm rel"] <= (L / 2 + 1.5) * U, (errs, L)


def check_rows(name, got, want, errs):
    from fedfr_b200 import selfcheck as SC
    errs[name] = (SC._rows_err(got, want), SC._rows_err(got, want, rms=True))
    assert errs[name][0] <= ROWS_MAX and errs[name][1] <= ROWS_RMS, (name, errs)


def dw_group_errors(dw, ref, y, clamped, edge=None):
    """Per-row errors of ``dw`` by group.  A row whose norm was clamped gets dwh / eps, about 1e11 times an ordinary row:
    inside a group it would lift ``selfcheck._rows_err``'s floor (1 % of the group's rms row norm) above every ordinary
    row.  So the clamped rows (zero and 0 < |w| < eps) form their own group, each held to its own norm, and the target,
    other and chunk-edge groups hold only ordinary rows.  Returns {group: (max, rms)} (the edge group: max only)."""
    from fedfr_b200 import selfcheck as SC
    tgt = torch.zeros(dw.shape[0], dtype=torch.bool, device=dw.device)
    tgt[y] = True
    ok = ~clamped.to(dw.device)
    errs = {}
    for name, sel in (("target rows", tgt & ok), ("other rows", ~tgt & ok)):
        errs[name] = (SC._rows_err(dw[sel], ref[sel]), SC._rows_err(dw[sel], ref[sel], rms=True))
    if bool((~ok).any()):
        r = ref[~ok].double()
        e = (dw[~ok].double() - r).norm(dim=1) / r.norm(dim=1).clamp_min(1e-300)
        errs["clamped rows, each to its own norm"] = (float(e.max()), float(e.pow(2).mean().sqrt()))
    if edge is not None:
        errs["chunk-edge rows"] = SC._rows_err(dw[edge & ok], ref[edge & ok])
    return errs


def check_dw(prefix, dw, ref, y, clamped, errs, edge=None):
    for name, e in dw_group_errors(dw, ref, y, clamped, edge).items():
        errs[prefix + " " + name] = e
        emax, erms = e if isinstance(e, tuple) else (e, 0.0)
        assert emax <= ROWS_MAX and erms <= ROWS_RMS, (prefix + " " + name, errs)


def run_case(Bt, C, E, W=1, kind=0, accumulate=False, weight_rows=False, seed=None):
    """Warm-up call, 0xFF-filled scratch and guard rows, the checked call, then every row against ``restate``."""
    from fedfr_b200 import _native as N
    from fedfr_b200.ops_cuda import CudaOps
    dev = torch.device("cuda:0")
    m = M_COS if kind == 0 else M_ARC
    x, y, w = make_inputs(Bt, C, E, W, seed if seed is not None else Bt * 7 + C + E + W, weight_rows)
    provs = [CudaOps(dev, N.PATH_CHECK) for _ in range(W)]
    gen = torch.Generator(device=dev).manual_seed(7)
    guards, dw_out = [], []
    for r, o in enumerate(provs):
        dx, tail, want = _guarded(Bt, E, gen)
        o._ws[("dx", (Bt, E), torch.float32)] = dx
        guards.append((tail, want))
        dw, tail, want = _guarded(shard_geometry(C, W, r)[0], E, gen)
        dw_out.append(dw)
        guards.append((tail, want))
    dw_init = None
    if accumulate:
        dw_init = [torch.randn(d.shape, generator=gen, device=dev) * 1e-3 for d in dw_out]
    run_shards(lambda r: provs[r], x, y, C, W, S, m, kind, accumulate, dw_init, w=w, dw_out=dw_out)
    for o in provs:
        for v in o._ws.values():
            if isinstance(v, torch.Tensor):
                v.view(torch.uint8).fill_(0xFF)
    out = run_shards(lambda r: provs[r], x, y, C, W, S, m, kind, accumulate, dw_init, w=w, dw_out=dw_out)
    torch.cuda.synchronize()
    assert torch.isfinite(out["loss"]) and bool(torch.isfinite(out["dx"]).all())
    assert all(bool(torch.isfinite(d).all()) for d in out["dw"])
    for tail, want in guards:
        assert _same_bits(tail, want), "a kernel wrote past the last row / class"
    inv = torch.cat([o._ws[("inv_norm", (shard_geometry(C, W, r)[0],), torch.float32)] for r, o in enumerate(provs)])
    w_hat = torch.cat(out["w_hat"])
    errs = {}
    check_normalize(w, w_hat, inv, errs)
    clamped = inv == clamped_inv()
    assert int(clamped.sum()) == (1 if weight_rows else 0) + int((w.norm(dim=1) == 0).sum())
    ref = restate(x, y, w_hat, inv, clamped, S, m, kind)
    errs["loss"] = abs(float(out["loss"]) - float(ref["loss"])) / float(ref["loss"])
    assert errs["loss"] <= LOSS_TOL, errs
    dw = torch.cat([d - dw_init[r] if accumulate else d for r, d in enumerate(out["dw"])])
    check_rows("dx", out["dx"], ref["dx"], errs)
    # the classes at every backward-chunk boundary of every shard are also held to the max criterion by themselves
    edge = torch.zeros(C, dtype=torch.bool, device=dev)
    for r in range(W):
        n_loc, c0 = shard_geometry(C, W, r)
        for b in chunk_starts(Bt, n_loc):
            edge[c0 + max(b - 1, 0): c0 + b + 2] = True
        edge[c0 + n_loc - 1] = True
    check_dw("dw", dw, ref["dw"], y, clamped, errs, edge)
    assert ("dw clamped rows, each to its own norm" in errs) == weight_rows
    print("errors", name_of(Bt, C, E, W, kind, accumulate, weight_rows), errs)
    return errs


def name_of(*args):
    return "Bt=%d C=%d E=%d W=%d kind=%d accumulate=%s weight_rows=%s" % args


# (Bt, C, E, W, kind, weight_rows); the comments say what check_chunk / the grids give
CASES = {
    "one_chunk": (64, 1000, 128, 1, 0, False),
    "two_chunks": (4096, 8192, 64, 1, 0, False),              # chunk 4096
    "three_chunks_ragged_arc": (4096, 10000, 128, 1, 1, False),   # 4096, 4096, 1808
    "column_floor": (270000, 200, 64, 1, 0, False),           # chunk 64: 4 chunks, the last of 8 columns; finalize's thread stride
    "grid_limit": (4, 4194305, 64, 1, 0, False),              # chunk capped at 65,535 tiles: 4,194,240 + 65
    "e4": (100, 3000, 4, 1, 0, False),                        # normalize_rows<1, 1>, one k step with a 12-wide tail
    "e20": (100, 3000, 20, 1, 1, False),                      # TK tail of 4
    "e100": (100, 3000, 100, 1, 0, False),
    "e132": (100, 3000, 132, 1, 1, False),                    # normalize_rows<2, 1>
    "e260": (100, 3000, 260, 1, 0, False),                    # normalize_rows<4, 1>
    "e1020": (100, 3000, 1020, 1, 0, False),                  # normalize_rows<8, 1>, TK tail of 12
    "e1024_arc": (100, 3000, 1024, 1, 1, False),
    "e2048": (100, 3000, 2048, 1, 0, False),                  # normalize_rows<16, 1>
    "bt1": (1, 1000, 128, 1, 0, False),
    "bt63": (63, 1000, 128, 1, 1, False),
    "bt64": (64, 1000, 128, 1, 0, False),
    "bt65": (65, 1000, 128, 1, 0, False),
    "bt129": (129, 1000, 128, 1, 1, False),
    "cs37": (65, 37, 128, 1, 0, False),                       # below one class tile
    "cs1985": (65, 31 * 64 + 1, 128, 1, 0, False),            # 32 tiles, 32 splits, last tile of 1
    "cs2048": (65, 32 * 64, 128, 1, 1, False),
    "cs2112": (65, 33 * 64, 128, 1, 0, False),                # 33 tiles over 32 splits
    "cs100003": (129, 100003, 128, 1, 0, False),              # 1563 tiles over 32 splits, ragged
    "w3_ragged": (300, 10001, 128, 3, 0, False),              # -1 labels through fwd_stats, merge and finalize
    "w3_bt1500_arc": (1500, 3001, 64, 3, 1, False),           # Bt > 1024
    "weight_rows": (300, 3001, 128, 1, 0, True),
    "weight_rows_arc_chunks": (4096, 8192, 64, 1, 1, True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_check_edge_case(defaults, name):
    Bt, C, E, W, kind, weight_rows = CASES[name]
    run_case(Bt, C, E, W, kind, weight_rows=weight_rows)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["two_chunks", "three_chunks_ragged_arc", "w3_ragged"])
def test_check_edge_case_accumulate(defaults, name):
    """``accumulate_dw = 1`` on multi-chunk shards: got - dw_init row by row."""
    Bt, C, E, W, kind, weight_rows = CASES[name]
    run_case(Bt, C, E, W, kind, accumulate=True, weight_rows=weight_rows)


@pytest.mark.gpu
@pytest.mark.parametrize("emb", [2052, 6])
def test_unsupported_emb_is_refused(defaults, emb):
    """``normalize_rows`` takes multiples of 4 up to 2048: anything else is PFC_E_SHAPE, and nothing is written."""
    from fedfr_b200 import _native as N
    w = torch.randn(10, emb, device="cuda")
    w_hat = torch.full((10, emb), 7.0, device="cuda")
    inv = torch.full((10,), 7.0, device="cuda")
    rc = N.lib.pfc_normalize_rows(N.ptr(w), None, 10, emb, None, N.ptr(w_hat), N.ptr(inv), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == -2
    assert bool((w_hat == 7.0).all()) and bool((inv == 7.0).all())


@pytest.mark.gpu
def test_partial_fc_check_mode_step(defaults, pkg):
    """One ``PartialFC(check_mode=True)`` step at emb 1024: loss, every row of x_grad and sub_weight.grad."""
    from fedfr_b200 import _native as N
    from fedfr_b200.ops_cuda import CudaOps
    B, C, E = 300, 5001, 1024
    head = pkg.PartialFC(0, 0, 1, B, False, pkg.CosFace(s=S, m=M_COS), C, embedding_size=E, prefix="/tmp", check_mode=True)
    dev = head.device
    x, y, w = make_inputs(B, C, E, 1, 11, weight_rows=True)
    with torch.no_grad():
        head.weight.copy_(w)
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.1, momentum=0.9)
    xg, loss = head.forward_backward(y, x, opt)
    torch.cuda.synchronize()
    w_hat, inv = CudaOps(dev, N.PATH_CHECK).normalize(w)
    errs = {}
    check_normalize(w, w_hat, inv, errs)
    clamped = inv == clamped_inv()
    ref = restate(x, y, w_hat, inv, clamped, S, M_COS, 0)
    errs["loss"] = abs(float(loss) - float(ref["loss"])) / float(ref["loss"])
    assert errs["loss"] <= LOSS_TOL, errs
    check_rows("dx", xg, ref["dx"], errs)
    check_dw("dw", head.sub_weight.grad, ref["dw"], y, clamped, errs)
    print("errors PartialFC", errs)


@pytest.mark.gpu
def test_margin_softmax_head_check_mode(defaults, pkg):
    """``MarginSoftmaxHead(check_mode=True)`` forward / backward at emb 1024 with ArcFace: loss, every row of x.grad
    (through the normalisation of x) and fc.grad."""
    from fedfr_b200 import _native as N
    from fedfr_b200.ops_cuda import CudaOps
    B, C, E = 256, 6100, 1024
    dev = torch.device("cuda:0")
    x, y, w = make_inputs(B, C, E, 1, 12, weight_rows=True)
    x = x * 3.0
    head = pkg.MarginSoftmaxHead(C, pkg.ArcFace(S, M_ARC), E, check_mode=True).to(dev)
    head.fc.data.copy_(w)
    xa = x.clone().requires_grad_(True)
    loss = head(xa, y)
    loss.backward()
    torch.cuda.synchronize()
    norm = x.norm(dim=1, keepdim=True).clamp_min(EPS)
    xu = x / norm                                            # the operand the head hands the kernels (dense_head.py)
    w_hat, inv = CudaOps(dev, N.PATH_CHECK).normalize(w)
    clamped = inv == clamped_inv()
    ref = restate(xu, y, w_hat, inv, clamped, S, M_ARC, 1)
    xu64, n64 = xu.double(), norm.double()
    dx_ref = (ref["dx"] - xu64 * (xu64 * ref["dx"]).sum(dim=1, keepdim=True)) / n64
    errs = {"loss": abs(loss.item() - float(ref["loss"])) / float(ref["loss"])}
    assert errs["loss"] <= LOSS_TOL, errs
    check_rows("x.grad", xa.grad, dx_ref, errs)
    check_dw("fc.grad", head.fc.grad, ref["dw"], y, clamped, errs)
    print("errors MarginSoftmaxHead", errs)
