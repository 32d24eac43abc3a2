"""The cosine head of FedFR's personalised branch (``csrc/bce_head.cu``) at the edges of its grid stride, its 256-row
chunks, its embedding slices, exponents, labels and degenerate rows, element by element.

``pfc_bce_head_fwd`` is one warp per (row, class) pair, grid-strided over at most 148 x 16 blocks of 8 warps;
``pfc_bce_head_bwd`` is one CTA per feature row and one per class row, each streaming the other operand in chunks of
``kBceChunk = 256`` rows, with ``kBceMaxKpt = 8`` slices of 128 embedding columns per thread (emb <= 1024).

Every output buffer is filled with 0xFF bytes first and followed by guard elements that must keep their bits.  Each
output is held to an fp64 restatement that starts from the kernel's own operands (the fp32 inputs; for the epilogue and
the backward the kernel's fp32 ``cosine`` and inverse norms), with a per-element bound derived from the fp32 chain that
produced it (``bound_*``).  The restatement is pinned to fp64 autograd of ``test_bce_head.reference_head`` on the CPU."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from test_bce_head import bce_loss, reference_head  # noqa: E402
from test_gpu_kernel_edges import _same_bits  # noqa: E402

M, R = 0.4, 30.0
EPS = 1e-12
U = 2.0 ** -24                 # fp32 unit roundoff
GUARD = 97
POW_ULP = 8                    # powf: CUDA documents at most 4 ulp; twice that


def target_col(labels, C):
    from oracle import bce_head_oracle as O
    return O.target_col(labels, C)


# ------------------------------------------------------------------------------------------------ restatement
def restate_fwd(feat, weight, bias, labels, cosine, t, m=M, r=R):
    """fp64: (cos from the fp32 inputs, inverse norms, logits from the KERNEL's fp32 cosine, gt).
    cos = f.w / (max(|f|, eps) max(|w|, eps)), u = max((cos + 1) / 2, 0), g = 2 u^t - 1,
    logit = r (g -+ m) + bias_c, gt = (c == target column of the row's label)."""
    f, w = feat.double(), weight.double()
    inf = 1.0 / f.norm(dim=1).clamp_min(EPS)
    inw = 1.0 / w.norm(dim=1).clamp_min(EPS)
    cos = (f @ w.t()) * inf[:, None] * inw[None, :]
    col = target_col(labels.cpu(), weight.shape[0]).to(feat.device)
    gt = torch.zeros(cos.shape, dtype=torch.bool, device=feat.device)
    rows = torch.nonzero(col >= 0, as_tuple=True)[0]
    gt[rows, col[rows]] = True
    u = ((cosine.double() + 1) / 2).clamp_min(0)
    g = 2 * u.pow(t) - 1
    logits = r * torch.where(gt, g - m, g + m)
    if bias is not None:
        logits = logits + bias.double()[None, :]
    return {"cos": cos, "inv_nf": inf, "inv_nw": inw, "logits": logits, "gt": gt, "u": u, "g": g}


def restate_bwd(feat, weight, cosine, inv_nf, inv_nw, dlogits, t, r=R):
    """fp64 backward from the kernel's operands: dcos = dz r t u^(t-1) (u from the fp32 cosine, clamped at 0),
    dfeat_b = inv_f (sum_c dcos inv_w_c w_c - f_b inv_f sum_c dcos cos), likewise dweight_c over the feature rows, and no
    radial term on a row whose norm was clamped (inv == 1 / eps in fp32); dbias_c = sum_b dz.  Also returns the
    magnitudes the bounds need."""
    f, w, cs = feat.double(), weight.double(), cosine.double()
    ifn, iwn = inv_nf.double(), inv_nw.double()
    dz = dlogits.double()
    u = ((cs + 1) / 2).clamp_min(0)
    dcos = dz * (r * t) * u.pow(t - 1)
    cl = float(torch.tensor([1.0]) / torch.tensor([EPS], dtype=torch.float32))
    out = {}
    for name, d, mine, other, i_me, i_other in (("dfeat", dcos, f, w, ifn, iwn), ("dweight", dcos.t(), w, f, iwn, ifn)):
        sd = d * i_other[None, :]
        acc = sd @ other
        radial = (d * (cs if name == "dfeat" else cs.t())).sum(dim=1)
        radial = torch.where(i_me.float() >= cl, torch.zeros_like(radial), radial)
        out[name] = i_me[:, None] * (acc - mine * i_me[:, None] * radial[:, None])
        out[name + " |acc|"] = sd.abs() @ other.abs()
        out[name + " |radial|"] = (d * (cs if name == "dfeat" else cs.t())).abs().sum(dim=1)
        out[name + " parts"] = (acc, mine * i_me[:, None] * radial[:, None])
    out["dbias"] = dz.sum(dim=0)
    out["dbias |sum|"] = dz.abs().sum(dim=0)
    return out


# ------------------------------------------------------------------------------------------------ bounds
def chain(n, lanes):
    """Roundings on the longest path of a sum of n terms split over `lanes` sequential partial sums and then a tree:
    ceil(n / lanes) in each partial sum plus log2(lanes) tree levels."""
    return -(-n // lanes) + max(lanes - 1, 0).bit_length()


def bound_cos(f, w, E, ref):
    """|cos32 - cos64|.  fw, ff, ww: each lane runs ceil(E / 32) fma, then a 5-level warp tree: L = chain(E, 32) roundings,
    |error| <= L u sum |products|.  inv = 1 / max(sqrt(ff), eps) adds u / 2 (sqrt) and u / 2 (division) to L u / 2; cos =
    fw inf inw two more roundings.  So |d cos| <= L u sum|f_k w_k| inf inw + (L + 4) u |cos| (1 % for second order)."""
    L = chain(E, 32)
    A = (f.double().abs() @ w.double().abs().t()) * ref["inv_nf"][:, None] * ref["inv_nw"][None, :]
    return 1.01 * U * (L * A + (L + 4) * ref["cos"].abs()) + 1e-30


def bound_inv(E):
    """Relative bound of the inverse norms: L u / 2 (sum of squares, halved by sqrt) + u / 2 + u / 2."""
    return 1.01 * U * (chain(E, 32) / 2 + 1)


def bound_logits(ref, t, bias):
    """|z32 - z64| given the same fp32 cosine: cs + 1 rounds once (u |cs + 1|; times 1/2 is exact), which moves u^t by
    t u^(t-1) u |cs + 1| / 2; the power is exact for t = 1, 1 or 2 roundings for t = 2, 3, powf (POW_ULP) otherwise; then
    2 p - 1, g -+ m, r (.) and + bias round once each, relative to their results."""
    u, g = ref["u"], ref["g"]
    p = u.pow(t)
    n_pow = {1: 0, 2: 1, 3: 2}.get(t, POW_ULP)
    gm = torch.where(ref["gt"], g - M, g + M)
    err_g = 2 * (t * u.pow(t - 1) * (2 * u) * U / 2 + n_pow * U * p) + U * g.abs()
    return 1.01 * (R * (err_g + U * gm.abs()) + U * R * gm.abs() + U * ref["logits"].abs()) + 1e-30


def bound_grad(ref, name, n_other, t):
    """|d32 - d64| per element.  s_d = dz (r t) u^(t-1) inv_other: r t, the product with dz, with the power (0-2 roundings
    or powf) and with inv_other, plus |t - 1| times u's one rounding: D = (4 + POW_ULP + |t - 1|) u relative.  acc runs
    n_other sequential fma per thread: (n_other + D / u) u sum|s_d o_k|.  radial: ceil(n_other / 128) fma per thread then the
    warp and 4-warp trees (7 levels), with the same D.  out = inv (acc - mine inv radial): four more roundings, relative to
    |acc| and |mine inv radial|, and the final result."""
    D = 4 + POW_ULP + abs(t - 1)
    inv = ref["inv"][:, None]
    acc, rad_part = ref[name + " parts"]
    e_acc = (n_other + D) * U * ref[name + " |acc|"]
    e_rad = (chain(n_other, 128) + 2 + D) * U * ref[name + " |radial|"][:, None] * ref["mine_inv"]
    return 1.01 * (inv * (e_acc + e_rad + 2 * U * (acc.abs() + rad_part.abs())) + U * ref[name].abs()) + 1e-30


# ------------------------------------------------------------------------------------------------ CPU pin
def _cpu_case(B, C, E, seed):
    g = torch.Generator().manual_seed(seed)
    feat = torch.randn(B, E, generator=g, dtype=torch.float64) * 2
    weight = torch.randn(C, E, generator=g, dtype=torch.float64) * 0.01
    bias = torch.randn(C, generator=g, dtype=torch.float64) * 0.1
    y = torch.randint(0, C + C // 3 + 1, (B,), generator=g)
    feat[0] = weight[1] * 3                                  # same direction as a class row
    feat[2] = 0.0
    feat[3] = F.normalize(feat[3], dim=0) * 0.9e-12          # 0 < |f| < eps
    weight[2] = F.normalize(weight[2], dim=0) * 0.9e-12
    return feat, weight, bias, y


@pytest.mark.parametrize("B,C,E,t", [(9, 7, 16, 3), (6, 5, 33, 1), (8, 4, 5, 2.5), (7, 9, 12, 4), (5, 6, 8, 2)])
def test_restatement_is_autograd_of_the_reference(B, C, E, t):
    """With exact fp64 operands the restatement equals fp64 autograd of ``reference_head`` (client.py:47-57) under
    ``bce_loss`` (losses.py:4-15): logits, gt, and the gradients of feat, weight and bias -- including a zero feature row
    and rows with 0 < |v| < eps, whose gradient autograd gives as d / eps with no radial term."""
    feat, weight, bias, y = _cpu_case(B, C, E, B * C + E)
    fr, wr, br = (v.clone().requires_grad_(True) for v in (feat, weight, bias))
    lr, gr = reference_head(fr, wr, br, y, M, R, t)
    loss = bce_loss(lr, gr)
    loss.backward()
    lg = lr.detach().clone().requires_grad_(True)
    bce_loss(lg, gr).backward()
    ref = restate_fwd(feat, weight, bias, y, (F.normalize(feat) @ F.normalize(weight).t()), t)
    assert torch.equal(ref["gt"], gr)
    assert float((ref["logits"] - lr.detach()).abs().max()) <= 1e-12 * R
    g = restate_bwd(feat, weight, ref["cos"], ref["inv_nf"], ref["inv_nw"], lg.grad, t)
    for got, want in ((g["dfeat"], fr.grad), (g["dweight"], wr.grad)):
        for i in range(want.shape[0]):
            assert float((got[i] - want[i]).abs().max()) <= 1e-10 * (float(want[i].abs().max()) + 1e-300), i
    assert float((g["dbias"] - br.grad).abs().max()) <= 1e-12


def test_negative_labels_pick_python_columns():
    """-2 selects column C - 1, -(C + 1) column 0; -1, -(C + 2) and labels >= C select none (client.py:48-52)."""
    C = 5
    col = target_col(torch.tensor([3, C, C + 4, -1, -2, -(C + 1), -(C + 2)]), C)
    assert col.tolist() == [3, -1, -1, -1, C - 1, 0, -1]


# ------------------------------------------------------------------------------------------------ GPU driver
@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


def _buf(n, dtype, dev, gen):
    """(the leading n elements of a 0xFF-filled buffer, its guard tail, the guard's contents)"""
    b = torch.empty(n + GUARD, dtype=dtype, device=dev)
    b.view(torch.uint8).fill_(0xFF)
    tail = torch.randint(0, 256, (GUARD,), generator=gen, device=dev).to(dtype)
    b[n:] = tail
    return b[:n], b[n:], tail


def below_minus_one_scale():
    """A scale a whose one-hot row a e_0 has an fp32 cosine below -1 against its negation in the forward kernel.  For a row
    with one non-zero element every sum of the kernel is exact but the first product: fw = -fl(a^2) = -ww, and
    inv = fl(1 / fl(sqrt(ww))), so cos = fl(fl(-ww inv) inv), which this search evaluates with the same IEEE fp32
    operations (correctly rounded products, sqrt and division, as nvcc emits them by default)."""
    one = torch.tensor(1.0, dtype=torch.float32)
    for a in torch.linspace(0.01, 0.02, 2001, dtype=torch.float32):
        ww = a * a
        inv = one / torch.sqrt(ww)
        if float((-ww * inv) * inv) < -1.0:
            return float(a)
    raise AssertionError("no fp32 scale in [0.01, 0.02] rounds the antipodal cosine below -1")


def test_antipodal_pair_rounds_below_minus_one():
    """The antipodal pair of ``make_case`` has fp32 cosine < -1 (and the equal pair > 1): without the clamp of
    (cos + 1) / 2 at 0, powf at a non-integer t would return NaN for it."""
    a = torch.tensor(below_minus_one_scale(), dtype=torch.float32)
    inv = torch.tensor(1.0) / torch.sqrt(a * a)
    assert float((-(a * a) * inv) * inv) < -1.0 and float(((a * a) * inv) * inv) > 1.0


def make_case(B, C, E, seed, dev):
    """Random rows, labels with every rule (in range, >= C, -1, -2, -(C + 1), -(C + 2), duplicates), and degenerate rows:
    a feature row equal to class row C // 2 and one antipodal to it (that class row is one-hot, scaled so that the
    antipodal cosine rounds below -1 in fp32: ``below_minus_one_scale``), a zero row, one with 0 < |f| < eps, and a
    class row with 0 < |w| < eps."""
    g = torch.Generator(device=dev).manual_seed(seed)
    feat = torch.randn(B, E, generator=g, device=dev) * 2
    weight = torch.randn(C, E, generator=g, device=dev) * 0.01
    bias = torch.randn(C, generator=g, device=dev) * 0.1
    y = torch.randint(0, C, (B,), generator=g, device=dev)
    special = [C, C + 3, -1, -2, -(C + 1), -(C + 2)]
    y[1: 1 + min(len(special), max(B - 1, 0))] = torch.tensor(special[:max(B - 1, 0)], device=dev)
    if B > 8:
        y[7] = y[0]                                          # duplicate
    j = C // 2
    weight[j] = 0.0
    weight[j, 0] = below_minus_one_scale()
    rows = {0: lambda: weight[j].clone(), 3: lambda: -weight[j], 5: lambda: torch.zeros(E, device=dev),
            6: lambda: F.normalize(feat[6], dim=0) * 0.9e-12}
    for i, v in rows.items():
        if i < B:
            feat[i] = v()
    if C >= 3:
        weight[C - 1] = F.normalize(weight[C - 1], dim=0) * 0.9e-12
    return feat, weight, bias, y


def run_case(B, C, E, t, seed=None, bias_on=True, dfeat_on=True, dbias_on=True, dl="random"):
    from fedfr_b200 import _native as N
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(99)
    feat, weight, bias, y = make_case(B, C, E, seed if seed is not None else B * 131 + C * 7 + E, dev)
    st = torch.cuda.current_stream().cuda_stream
    logits, lt, lw = _buf(B * C, torch.float32, dev, gen)
    cosine, ct, cw = _buf(B * C, torch.float32, dev, gen)
    gt, gtt, gtw = _buf(B * C, torch.uint8, dev, gen)
    inf, it, iw = _buf(B, torch.float32, dev, gen)
    inw, jt, jw = _buf(C, torch.float32, dev, gen)
    rc = N.lib.pfc_bce_head_fwd(N.ptr(feat), N.ptr(weight), N.ptr(bias) if bias_on else None, N.ptr(y), B, C, E, M, R, float(t),
                                N.ptr(logits), N.ptr(gt), N.ptr(cosine), N.ptr(inf), N.ptr(inw), st)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(gtt, gtw), "a store past the end of gt"
    for tail, want in ((lt, lw), (ct, cw), (it, iw), (jt, jw)):
        assert _same_bits(tail, want), "a store past the end"
    logits, cosine, gt = logits.view(B, C), cosine.view(B, C), gt.view(B, C)
    if B > 3:                            # the equal and antipodal pairs: the clamp of (cos + 1) / 2 at 0 is exercised
        assert float(cosine[0, C // 2]) > 1.0 and float(cosine[3, C // 2]) < -1.0, (float(cosine[0, C // 2]), float(cosine[3, C // 2]))
    b = bias if bias_on else None
    ref = restate_fwd(feat, weight, b, y, cosine, t)
    errs = {}
    assert torch.equal(gt.bool(), ref["gt"]), "gt"
    for name, got, want, bound in (("cosine", cosine, ref["cos"], bound_cos(feat, weight, E, ref)),
                                   ("logits", logits, ref["logits"], bound_logits(ref, t, b)),
                                   ("inv_nf", inf, ref["inv_nf"], bound_inv(E) * ref["inv_nf"]),
                                   ("inv_nw", inw, ref["inv_nw"], bound_inv(E) * ref["inv_nw"])):
        assert bool(torch.isfinite(got).all()), name
        ratio = (got.double() - want).abs() / bound
        errs[name + " err/bound"] = float(ratio.max())
        assert errs[name + " err/bound"] <= 1.0, (name, errs)
    # backward
    if dl == "bce":
        lg = logits.detach().clone().requires_grad_(True)
        bce_loss(lg, gt.bool()).backward()
        dlog = lg.grad.contiguous()
    else:
        dlog = torch.randn(B, C, generator=gen, device=dev)
    dfeat, ft, fw = _buf(B * E, torch.float32, dev, gen)
    dweight, wt, ww = _buf(C * E, torch.float32, dev, gen)
    dbias, bt, bw = _buf(C, torch.float32, dev, gen)
    rc = N.lib.pfc_bce_head_bwd(N.ptr(feat), N.ptr(weight), N.ptr(cosine), N.ptr(inf), N.ptr(inw), N.ptr(dlog), B, C, E, R, float(t),
                                N.ptr(dfeat) if dfeat_on else None, N.ptr(dweight), N.ptr(dbias) if dbias_on else None, st)
    assert rc == 0
    torch.cuda.synchronize()
    for tail, want in ((ft, fw), (wt, ww), (bt, bw)):
        assert _same_bits(tail, want), "a store past the end"
    g = restate_bwd(feat, weight, cosine, inf, inw, dlog, t)
    checks = [("dweight", dweight.view(C, E), weight, inw, B)]
    if dfeat_on:
        checks.append(("dfeat", dfeat.view(B, E), feat, inf, C))
    else:
        assert bool((dfeat.view(torch.int32) == -1).all()), "dfeat == NULL: nothing may be written"
    for name, got, mine, inv, n_other in checks:
        g["inv"] = inv.double()
        g["mine_inv"] = mine.double().abs() * inv.double()[:, None]
        assert bool(torch.isfinite(got).all()), name
        ratio = (got.double() - g[name]).abs() / bound_grad(g, name, n_other, t)
        errs[name + " err/bound"] = float(ratio.max())
        assert errs[name + " err/bound"] <= 1.0, (name, errs)
    if dbias_on:
        bound = 1.01 * (chain(B, 128) + 2) * U * g["dbias |sum|"] + 1e-30
        errs["dbias err/bound"] = float(((dbias.double() - g["dbias"]).abs() / bound).max())
        assert errs["dbias err/bound"] <= 1.0, errs
    else:
        assert bool((dbias.view(torch.int32) == -1).all()), "dbias == NULL: nothing may be written"
    print("errors B=%d C=%d E=%d t=%s" % (B, C, E, t), errs)
    return errs


CHUNK = [(1, 513), (513, 1), (255, 257), (256, 256), (257, 255), (513, 513), (1, 1), (255, 1), (1, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,C", CHUNK)
def test_chunking(pkg, B, C):
    """Both roles across 0, 1 and 2 chunk boundaries of 256 rows."""
    run_case(B, C, 128, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,E", [(148, 128, 64), (5, 3789, 64), (1000, 3000, 128)])
def test_forward_grid_stride(pkg, B, C, E):
    """18,944 pairs = 148 x 16 blocks x 8 warps, one pair more (warp 0 takes a second), and a large case."""
    run_case(B, C, E, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("E", [1, 31, 33, 128, 129, 897, 1024])
def test_emb(pkg, E):
    run_case(64, 100, E, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("t", [1, 2, 3, 4, 2.5])
def test_exponent(pkg, t):
    """pow_small's special cases and powf in both directions; at t = 2.5 the antipodal pair's cosine may round below -1."""
    run_case(100, 300, 128, t)


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["bias NULL", "dfeat NULL", "dbias NULL", "BCE_loss gradient"])
def test_null_pointers_and_loss(pkg, what):
    run_case(300, 257, 512, 3, bias_on=what != "bias NULL", dfeat_on=what != "dfeat NULL", dbias_on=what != "dbias NULL",
             dl="bce" if what == "BCE_loss gradient" else "random")


@pytest.mark.gpu
def test_emb_1025_is_refused(pkg):
    """The backward holds at most 8 slices of 128 columns per thread: emb 1025 is PFC_E_SHAPE, nothing written."""
    from fedfr_b200 import _native as N
    dev = torch.device("cuda:0")
    B, C, E = 4, 3, 1025
    feat, weight = torch.randn(B, E, device=dev), torch.randn(C, E, device=dev)
    cosine, dl = torch.zeros(B, C, device=dev), torch.ones(B, C, device=dev)
    inf, inw = torch.ones(B, device=dev), torch.ones(C, device=dev)
    outs = [torch.full((n,), 7.0, device=dev) for n in (B * E, C * E, C)]
    rc = N.lib.pfc_bce_head_bwd(N.ptr(feat), N.ptr(weight), N.ptr(cosine), N.ptr(inf), N.ptr(inw), N.ptr(dl), B, C, E, R, 3.0,
                                N.ptr(outs[0]), N.ptr(outs[1]), N.ptr(outs[2]), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == -2
    assert all(bool((o == 7.0).all()) for o in outs)
