"""The tensor-core kernels of the head at the edges of their dispatch: every kernel choice ``make_prob_bwd_plan`` /
``dw4_chosen`` / the chunked fused forward can make, partial row blocks and class tiles, forward-chunk boundaries, -1 labels
of multi-rank shards, ``accumulate_dw``, and the variants the ``pfc_set_*`` knobs select.

Each case drives the provider exactly as ``PartialFC.forward_backward`` does, for W virtual ranks on one device
(``run_shards``), and holds EVERY row of ``dx`` and ``dw`` to ``selfcheck.reference_step(emulate=True)`` -- the fp64
restatement with the tensor path's operand roundings written out, so that only summation order differs -- with the
criteria of ``selfcheck.check_head_step`` (max over rows <= 1e-2, rms <= 1e-3 for dx, target and non-target dw rows), and
also on each edge group by itself.  The library's scratch is filled with NaN bytes and ``dw`` / ``dx`` are followed by
guard rows, so an element a kernel forgets to write, or a store past the last row or class, fails the case."""
import contextlib
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

S, M_COS, M_ARC = 64.0, 0.4, 0.5
GUARD_ROWS = 131
BM = 128                       # row block / class tile of the kernels (csrc/tc_kernels.cu BM)
FWD_CHUNK_MIN = 16384          # a forward class chunk keeps every SM busy: at most n_classes / 16384 chunks


# ------------------------------------------------------------------------------------------------ knobs
def _restore_defaults(lib):
    """The shipped values of every pfc_set_* tuning knob (include/fedfr_b200_dev.h)."""
    lib.pfc_set_graph(1)
    lib.pfc_set_logits_pair(1)
    lib.pfc_set_logits_tile(128)
    lib.pfc_set_dx_pair(1)
    lib.pfc_set_dw4(-1)
    lib.pfc_set_clusters(2, 2)
    lib.pfc_set_fwd_overlap(4, 2)
    lib.pfc_set_prefetch(0, 0, 0)
    lib.pfc_set_prob_split(0, 0.42, 0)
    lib.pfc_set_pipeline(1, 148, 48, 100, 1)
    lib.pfc_set_chunk_mb(0)


@contextlib.contextmanager
def knobs(ops_list=(), **settings):
    """Set process-global tuning knobs, e.g. ``knobs(dw4=(1,), clusters=(4, 4))``; every knob goes back to its shipped
    default afterwards, and the ``bwd_mode`` of the given providers to what it was.  A leaked knob would silently change
    what every later test measures."""
    from fedfr_b200 import _native as N
    assert torch.backends.cuda.matmul.allow_tf32 is False, "the reference GEMMs must run in full fp32"
    modes = [(o, o.bwd_mode) for o in ops_list]
    try:
        for name, args in settings.items():
            N.check(getattr(N.lib, "pfc_set_" + name)(*args), "pfc_set_" + name)
        yield
    finally:
        _restore_defaults(N.lib)
        for o, mode in modes:
            o.bwd_mode = mode


# ------------------------------------------------------------------------------------------------ shard driver
def shard_geometry(C, W, r):
    """(num_local, class_start) of rank r: the reference's ragged class split (partial_fc.py ctor)."""
    return C // W + int(r < C % W), C // W * r + min(r, C % W)


def run_shards(make_ops, x, y, C, W, s, m, kind, accumulate=False, dw_init=None, *, w, dw_out=None):
    """One ``PartialFC.forward_backward`` step of W ranks on one device, through exactly the provider calls the head
    makes: per rank ``remap_labels`` and ``normalize_fwd_stats`` (``normalize`` + ``fwd_stats`` for a provider without
    the fused call), one ``finalize`` of the stacked [W, Bt, 3] statistics, then ``bwd`` per rank.

    ``make_ops(r)`` -> the provider of rank r; ``x`` [Bt, E] fp32 gathered features, ``y`` [Bt] global labels, ``w`` [C, E]
    the classes of all ranks.  ``accumulate``: ``bwd`` adds to ``dw_init`` (list of per-rank [Cs_r, E]).  ``dw_out``:
    per-rank tensors to receive ``dw`` (default: fresh ones); without ``accumulate`` they are first filled with 0xFF
    bytes (NaN), as an unwritten ``torch.empty`` might hold.
    Returns dict(loss, dx = sum over ranks of dx_r [Bt, E], dw = [per-rank dw], w_hat = [per-rank operand])."""
    assert w.shape[0] == C
    Bt, E = x.shape
    ops = [make_ops(r) for r in range(W)]
    stats, per_rank = [], []
    for r in range(W):
        o = ops[r]
        n_loc, c0 = shard_geometry(C, W, r)
        x_hat = o.cast_features(x)
        if hasattr(o, "remap_labels_"):         # as PartialFC: in place, in a label buffer with a stable address
            label = o.remap_labels_(o._persist("total_label", tuple(y.shape), y.dtype).copy_(y), c0, n_loc)
        else:
            label = o.remap_labels(y, c0, n_loc)
        sub_w = w[c0:c0 + n_loc]
        if hasattr(o, "normalize_fwd_stats"):
            w_hat, inv_norm, st = o.normalize_fwd_stats(sub_w, x_hat, label, s, m, kind)
        else:
            w_hat, inv_norm = o.normalize(sub_w)
            st = o.fwd_stats(x_hat, w_hat, label, s, m, kind)
        stats.append(st.clone())
        per_rank.append((label, x_hat, w_hat, inv_norm))
    row_max, row_sum, loss = ops[0].finalize(torch.stack(stats))
    dx_sum, dws, w_hats = None, [], []
    for r in range(W):
        o = ops[r]
        label, x_hat, w_hat, inv_norm = per_rank[r]
        dw = dw_out[r] if dw_out is not None else torch.empty((w_hat.shape[0], E), dtype=torch.float32, device=x.device)
        if accumulate:
            dw.copy_(dw_init[r])
        elif dw_out is not None:
            dw.view(torch.uint8).fill_(0xFF)
        dx = o.bwd(x_hat, w_hat, inv_norm, label, row_max, row_sum, s, m, 1.0 / Bt, dw, accumulate, kind)
        dx_sum = dx.clone() if dx_sum is None else dx_sum + dx
        dws.append(dw)
        w_hats.append(w_hat.clone())
    return {"loss": loss.clone(), "dx": dx_sum, "dw": dws, "w_hat": w_hats}


def test_run_shards_matches_two_rank_reference_golden():
    """The driver, given the CPU oracle as its provider, reproduces the unmodified reference's 2-rank ragged-shard step."""
    from golden_util import Case
    from oracle_ops import OracleOps
    case = Case("w2_sr1_ragged")
    cfg = case.cfg
    W = cfg["world_size"]
    x, y, w = torch.cat(case.features), torch.cat(case.labels), torch.cat(case.weights)
    out = run_shards(lambda r: OracleOps(), x, y, cfg["num_classes"], W, cfg["s"], cfg["m"], 0, w=w)
    B = x.shape[0] // W
    for r in range(W):
        assert abs(float(out["loss"]) - float(case.get(r, 0, "loss"))) <= 1e-5 * abs(float(case.get(r, 0, "loss")))
        for got, want in ((out["dx"][r * B:(r + 1) * B] * W, case.get(r, 0, "x_grad")), (out["dw"][r], case.get(r, 0, "dw"))):
            want = torch.from_numpy(want)
            assert float((got.double() - want.double()).abs().max()) <= 1e-5 * float(want.abs().max()), r
    # and accumulate=True adds to what is there
    init = [torch.randn_like(d) for d in out["dw"]]
    again = run_shards(lambda r: OracleOps(), x, y, cfg["num_classes"], W, cfg["s"], cfg["m"], 0, accumulate=True, dw_init=init, w=w)
    for r in range(W):
        assert torch.allclose(again["dw"][r] - init[r], out["dw"][r], rtol=0, atol=1e-6)


# ------------------------------------------------------------------------------------------------ inputs and checks
def fwd_chunk_starts(cs, chunks=4):
    """First class of every forward chunk of a shard of ``cs`` classes (tc_normalize_fwd_enqueue)."""
    n = max(1, min(chunks, cs // FWD_CHUNK_MIN))
    chunk = ((cs + n - 1) // n + 255) // 256 * 256
    return list(range(0, cs, chunk))


def make_inputs(Bt, C, E, W, seed, chunks=4, device="cuda"):
    """Unit features, a quarter of the rows pulled toward their class; duplicate labels; in every shard labels at its
    first and last class and at each forward-chunk boundary +-1."""
    g = torch.Generator(device=device).manual_seed(seed)
    w = torch.randn(C, E, generator=g, device=device) * 0.01
    y = torch.randint(0, C, (Bt,), generator=g, device=device)
    special = []
    for r in range(W):
        n_loc, c0 = shard_geometry(C, W, r)
        special += [c0, c0 + n_loc - 1]
        for b in fwd_chunk_starts(n_loc, chunks)[1:]:
            special += [c0 + b - 1, c0 + b, c0 + b + 1]
    if Bt >= 3:
        y[1] = y[0]                                                 # duplicate labels, one of them in the last row block
        y[Bt - 1] = y[0]
        special = special[: Bt - 3]
        pos = 2 + torch.randperm(Bt - 3, generator=g, device=device)[: len(special)]
        y[pos] = torch.tensor(special, dtype=y.dtype, device=device)
    pull = (torch.arange(Bt, device=device) % 4 == 0)[:, None]
    x = torch.nn.functional.normalize(torch.randn(Bt, E, generator=g, device=device) + 2.0 * torch.nn.functional.normalize(w[y]) * pull)
    return x, y, w


def _poison(ops_list):
    """Every library workspace of the providers -> 0xFF bytes (NaN in bf16 and fp32); the replayed graphs keep the addresses."""
    for o in ops_list:
        for v in o._ws.values():
            if isinstance(v, torch.Tensor):
                v.view(torch.uint8).fill_(0xFF)


def _guarded(rows, E, gen):
    """(the leading ``rows`` rows of a larger buffer, its tail, the sentinel written there)"""
    buf = torch.empty((rows + GUARD_ROWS, E), dtype=torch.float32, device=gen.device)
    tail = torch.randn((GUARD_ROWS, E), generator=gen, device=gen.device)
    buf[rows:] = tail
    return buf[:rows], buf[rows:], tail


def _same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def reference_recompute(x, y, w, w_hat, s, m, kind):
    """(dx, dw) in fp64 with the operand roundings of the recomputing backward (``tc_bwd``), which differ from those of
    the stored-probability path that ``reference_step(emulate=True)`` restates: G_ij = bf16(p_ij s / Bt) with the
    target element bf16((p_iy - 1) slope s / Bt), and the unscaled bf16 x_hat.  Against the stored-probability
    restatement a dw row dominated by one sample would differ by one independent bf16 rounding of that sample's
    features (rms ~2e-3 per row), which the 1e-3 rms criterion cannot tell from a real error.  One class block: the
    recompute cases are small."""
    from fedfr_b200 import selfcheck as SC
    Bt = x.shape[0]
    xb, wb = x.to(torch.bfloat16).double(), w_hat.double()
    rows = torch.arange(Bt, device=x.device)
    z = xb @ wb.t()
    mc_t, slope = SC._margin(z[rows, y], m, kind)
    z[rows, y] = mc_t
    s2 = s * SC.LOG2E
    P = torch.exp2(z * s2 - s2 * z.max(dim=1, keepdim=True).values)
    gs = s / Bt
    G = P * (gs / P.sum(dim=1, keepdim=True))
    G[rows, y] = (G[rows, y] - gs) * slope
    G = G.float().to(torch.bfloat16).double()
    dwh = G.t() @ xb
    inv_n = (1.0 / w.norm(dim=1, keepdim=True).clamp_min(1e-12)).double()
    return G @ wb, (dwh - wb * (wb * dwh).sum(dim=1, keepdim=True)) * inv_n


def check_against_reference(out, x, y, w, C, W, s, m, kind, dw_base=None, chunks=4, recompute=False):
    """Row-by-row comparison with ``reference_step(emulate=True)`` (criteria of ``check_head_step``), the same max-row
    criterion on each edge group alone, and the exact fp32-operand reference at 1e-2 relative L2.  ``dw_base``: per-rank
    contents ``dw`` held before an accumulating call (subtracted).  ``recompute``: the rows are held to
    ``reference_recompute`` instead.  Returns the measured errors."""
    from fedfr_b200 import selfcheck as SC
    Bt, E = x.shape
    w_hat = torch.cat(out["w_hat"])
    ref = SC.reference_step(x, y, w, s, m, kind, w_hat=w_hat, emulate=True, dw_rows=None)
    if recompute:
        ref["dx_total"], ref["dw"] = reference_recompute(x, y, w, w_hat, s, m, kind)
    exact = SC.reference_step(x, y, w, s, m, kind, emulate=False, dw_rows=None)
    dw_got = torch.cat([d - dw_base[r] if dw_base is not None else d for r, d in enumerate(out["dw"])])
    errs = {"loss": abs(float(out["loss"]) - float(ref["loss"])) / abs(float(ref["loss"]))}
    assert errs["loss"] < 1e-4, errs
    tgt = torch.zeros(C, dtype=torch.bool, device=x.device)
    tgt[y] = True
    dx, dx_ref = out["dx"], ref["dx_total"]
    groups = {"dx": (dx, dx_ref), "dw target rows": (dw_got[tgt], ref["dw"][tgt]), "dw other rows": (dw_got[~tgt], ref["dw"][~tgt])}
    for name, (got, want) in groups.items():
        errs[name] = (SC._rows_err(got, want), SC._rows_err(got, want, rms=True))
        assert errs[name][0] <= 1e-2 and errs[name][1] <= 1e-3, (name, errs)
    # edge groups, each by itself: the rows of the last row block, the last class tile pair of each shard, the classes
    # within +-1 of every forward-chunk boundary (split into target / non-target rows, as above)
    last_rb = slice((Bt - 1) // BM * BM, Bt)
    errs["dx last row block"] = SC._rows_err(dx[last_rb], dx_ref[last_rb])
    assert errs["dx last row block"] <= 1e-2, errs
    edge = torch.zeros(C, dtype=torch.bool, device=x.device)
    for r in range(W):
        n_loc, c0 = shard_geometry(C, W, r)
        edge[c0 + (n_loc - 1) // 256 * 256: c0 + n_loc] = True
        for b in fwd_chunk_starts(n_loc, chunks)[1:]:
            edge[c0 + b - 1: c0 + b + 2] = True
    for name, sel in (("dw edge target rows", edge & tgt), ("dw edge other rows", edge & ~tgt)):
        errs[name] = SC._rows_err(dw_got[sel], ref["dw"][sel])
        assert errs[name] <= 1e-2, (name, errs)
    errs["fp32"] = (abs(float(out["loss"]) - float(exact["loss"])) / abs(float(exact["loss"])), SC._rel(dx, exact["dx_total"]), SC._rel(dw_got, exact["dw"]))
    assert max(errs["fp32"]) < 1e-2, errs
    return errs


def run_case(Bt, C, E, W=1, kind=0, accumulate=False, chunks=4, recompute=False, prepare=None, seed=None):
    """Warm-up call (allocates the providers' buffers, captures the graphs), NaN-poisoned scratch and guard rows, the
    checked call, then the reference comparison.  Returns (outputs, errors, inputs)."""
    from fedfr_b200.ops_cuda import CudaOps
    dev = torch.device("cuda:0")
    m = M_COS if kind == 0 else M_ARC
    x, y, w = make_inputs(Bt, C, E, W, seed if seed is not None else Bt * 7 + C + E + W, chunks)
    provs = [CudaOps(dev) for _ in range(W)]
    if prepare is not None:
        prepare(provs)
    gen = torch.Generator(device=dev).manual_seed(7)
    guards, dw_out = [], []
    for r, o in enumerate(provs):
        dx, tail, want = _guarded(Bt, E, gen)               # the provider's dx scratch, ("dx", (Bt, E), fp32)
        o._ws[("dx", (Bt, E), torch.float32)] = dx
        guards.append((tail, want))
        dw, tail, want = _guarded(shard_geometry(C, W, r)[0], E, gen)
        dw_out.append(dw)
        guards.append((tail, want))
    dw_init = None
    if accumulate:
        first = run_shards(lambda r: provs[r], x, y, C, W, S, m, kind, w=w)
        dw_init = [torch.randn(d.shape, generator=gen, device=dev) * d.norm(dim=1, keepdim=True) / E ** 0.5 for d in first["dw"]]
    run_shards(lambda r: provs[r], x, y, C, W, S, m, kind, accumulate, dw_init, w=w, dw_out=dw_out)
    _poison(provs)                                          # the checked call replays the graphs of the warm-up call
    out = run_shards(lambda r: provs[r], x, y, C, W, S, m, kind, accumulate, dw_init, w=w, dw_out=dw_out)
    torch.cuda.synchronize()
    assert torch.isfinite(out["loss"]) and bool(torch.isfinite(out["dx"]).all())
    assert all(bool(torch.isfinite(d).all()) for d in out["dw"])
    for tail, want in guards:
        assert _same_bits(tail, want), "a kernel wrote past the last row / class"
    errs = check_against_reference(out, x, y, w, C, W, S, m, kind, dw_base=dw_init, chunks=chunks, recompute=recompute)
    return out, errs, (x, y, w, provs)


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


@pytest.fixture
def defaults(pkg):
    """Every test of this module starts and ends with the shipped knob values, and raises none of the per-device range
    flags of the stored-probability path (s |x| out of its window, a row sum of 0): every input here is in range."""
    from fedfr_b200 import ops_cuda
    with knobs():
        yield
    torch.cuda.synchronize()
    flags = ops_cuda._RANGE_FLAGS.get(0)
    raised = flags is not None and bool(flags.any())
    if raised:
        flags.zero_()
    assert not raised, "a case raised a range flag of the stored-probability path"


# ------------------------------------------------------------------------------------------------ case matrix
# (Bt, C, E, W, kind): what each reaches with the shipped knobs on a 148-SM B200
CASES = {
    "one_row": (1, 65, 64, 1, 0),                        # one row, partial tiles everywhere
    "row_past_block": (129, 257, 128, 1, 0),             # one row past a block, one class past a tile
    "dx2_ragged_e512": (500, 3001, 512, 1, 0),           # dx2 with a ragged last block; E=512 pair dw, 8 k-blocks, last partial
    "dx2_ragged_arc_e256": (900, 1000, 256, 1, 1),       # dx2 ragged (n_rb = 8), E=256 dw
    "pair_dw_2047": (2047, 20000, 512, 1, 0),            # last Bt of the pair dw kernel
    "dw4_2048": (2048, 20000, 512, 1, 0),                # first Bt of dw4
    "dw4_2049_arc": (2049, 257, 512, 1, 1),              # dw4, Bt % 64 = 1, single-CTA dx; second item holds 1 class
    "dw4_idle_clusters": (2500, 65, 512, 1, 0),          # dw4 with Cs below one tile
    "dw4_two_chunks": (3000, 40001, 512, 1, 0),          # dw4, Cs % 256 = 65, 2 forward chunks, dx2 ragged
    "four_chunks_arc": (4096, 65537, 512, 1, 1),         # 4 forward chunks (last ragged), dw4 + dx2
    "w8_shard": (4160, 100003, 512, 8, 0),               # per-GPU W = 8 shape: 7/8 of the labels -1 on each shard
    "w4_arc_dx2": (500, 30001, 512, 4, 1),               # -1 labels through dx2-ragged and the pair dw kernel
    "sequential_bwd": (20480, 5000, 512, 1, 0),          # dx needs more CTAs than SMs - 16: dx, then dw
    "e256_large_bt": (2100, 3000, 256, 1, 0),            # E < 512 at large Bt
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_edge_case(defaults, name):
    Bt, C, E, W, kind = CASES[name]
    run_case(Bt, C, E, W, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["row_past_block", "dx2_ragged_e512", "dw4_2049_arc", "dw4_idle_clusters", "dw4_two_chunks"])
def test_edge_case_accumulate(defaults, name):
    """``accumulate_dw = 1`` (``sub_weight.grad`` already exists): got - dw_init row by row."""
    Bt, C, E, W, kind = CASES[name]
    run_case(Bt, C, E, W, kind, accumulate=True)


# ------------------------------------------------------------------------------------------------ knob variants
# (id, knob settings, Bt, C, E, kind, bwd_mode)
VARIANTS = [
    ("dw4_0_bt4096", {"dw4": (0,)}, 4096, 20000, 512, 0, "prob"),
    ("dw4_forced_bt3000", {"dw4": (1,)}, 3000, 40001, 512, 0, "prob"),
    ("dw4_forced_stat_bt129", {"dw4": (1,)}, 129, 257, 512, 0, "prob"),
    ("dw4_forced_stat_bt500_arc", {"dw4": (1,)}, 500, 3001, 512, 1, "prob"),
    ("dw4_forced_stat_bt500", {"dw4": (1,)}, 500, 3001, 512, 0, "prob"),
    ("dx_pair_0_bt512", {"dx_pair": (0,)}, 512, 3001, 512, 0, "prob"),
    ("dx_pair_0_bt4096", {"dx_pair": (0,)}, 4096, 20000, 512, 0, "prob"),
] + [("clusters_%d_e%d" % (c, e), {"clusters": (c, c)}, 300, 3001, e, 0, "prob") for e in (256, 128) for c in (1, 2, 4)] + [
    ("fwd_chunks_%d" % k, {"fwd_overlap": (k, 2)}, 512, 65537, 512, 0, "prob") for k in (1, 2, 8)] + [
    ("prob_split_%d" % k, {"prob_split": (k, 0.42, 0)}, 1024, 20000, 512, 0, "prob") for k in (16, 100)] + [
    ("recompute_chunk1_pipe%d" % p, {"chunk_mb": (1,), "pipeline": (p, 0, 0, 0, 0)}, 500, 20000, 512, 0, "recompute") for p in (0, 1)] + [
    ("recompute_single_cta_tile%d" % t, {"logits_pair": (0,), "logits_tile": (t,)}, 500, 20000, 512, 0, "recompute") for t in (128, 256)]


@pytest.mark.gpu
@pytest.mark.parametrize("vid,settings,Bt,C,E,kind,mode", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_knob_variant(defaults, vid, settings, Bt, C, E, kind, mode):
    chunks = settings.get("fwd_overlap", (4,))[0]
    holder = []

    def prepare(provs):
        holder.extend(provs)
        for o in provs:
            o.bwd_mode = mode
    with knobs(**settings):
        try:
            run_case(Bt, C, E, 1, kind, chunks=chunks, recompute=mode == "recompute", prepare=prepare)
        finally:
            for o in holder:
                o.bwd_mode = "prob"
        if "logits_pair" in settings:
            # the stored-probability forward needs the CTA-pair kernels: it must refuse, not return numbers
            from fedfr_b200.ops_cuda import CudaOps
            o = CudaOps(torch.device("cuda:0"))
            x, y, w = make_inputs(Bt, C, E, 1, 1)
            with pytest.raises(RuntimeError):
                o.normalize_fwd_stats(w, o.cast_features(x), y, S, M_COS, 0, bwd_mode="prob")


@pytest.mark.gpu
def test_graph_off_is_bit_identical(defaults):
    """Kernel-by-kernel launches run the same kernels with the same geometry as the replayed graphs: same bits."""
    on, _, (x, y, w, _p) = run_case(3000, 40001, 512)
    with knobs(graph=(0,)):
        off, _, _ = run_case(3000, 40001, 512)
    assert _same_bits(on["loss"], off["loss"]) and _same_bits(on["dx"], off["dx"])
    assert all(_same_bits(a, b) for a, b in zip(on["dw"], off["dw"]))


# ------------------------------------------------------------------------------------------------ multi-step head
@pytest.mark.gpu
def test_multi_step_head(defaults, pkg):
    """Real ``PartialFC`` steps at a dw4 shape with fresh features and labels every step: graph replay with new contents,
    the None / zeroed / existing ``.grad`` flow, ``optimizer.step()``, then ``head.step(opt)`` and its prenormalised
    forward (``fwd_stats`` with w == NULL).  Every row of ``dx`` and ``dw`` is checked before each update."""
    from fedfr_b200 import selfcheck as SC
    B, C, E = 2100, 50000, 512
    head = pkg.PartialFC(0, 0, 1, B, False, pkg.CosFace(s=S, m=M_COS), C, embedding_size=E, prefix="/tmp")
    dev = head.device
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.1, momentum=0.9, weight_decay=5e-4)
    with knobs([head._ops]):
        for step in range(6):
            x, y, _ = make_inputs(B, C, E, 1, 1000 + step)
            with torch.no_grad():                                  # the pulled rows follow the current weights
                x = torch.nn.functional.normalize(x + 2.0 * torch.nn.functional.normalize(head.weight[y]) * (torch.arange(B, device=dev) % 4 == 0)[:, None])
            if step == 1:
                opt.zero_grad(set_to_none=False)                   # zeroed .grad: the accumulating backward onto zeros
            else:
                opt.zero_grad()
            prenormalized = head._prenorm is not None
            assert prenormalized == (step >= 4)
            xg, loss = head.forward_backward(y, x, opt)
            out = SC.check_head_step(head, y, x, xg, loss, dw_stride=1)
            assert out["ok"], (step, out)
            if step < 3:
                opt.step()
            else:
                head.step(opt)
