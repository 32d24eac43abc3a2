"""The exact ROC curve on the B200 (csrc/verify.cu pfc_roc_curve through fedfr_b200.verify.roc_curve): equal array for
array to sklearn.metrics.roc_curve and to the numpy restatement on counts, at the edge cases of test_roc_curve.py, at
sizes of many sort tiles, and on IJB-C-sized scores from template_features and pair_scores, with the insightface TAR
table read the same way from both curves."""
import os
import sys

import numpy as np
import pytest
import torch
from sklearn.metrics import auc
from sklearn.metrics import roc_curve as sk_roc_curve

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import roc_curve_oracle as RO  # noqa: E402
from test_roc_curve import KINDS, PAD, assert_same_curve, insightface_readout, make_case  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def F():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


def abi_roc(s, y):
    """pfc_roc_curve on the device with NaN-filled outputs of n + 1 + PAD entries -> (counts, n_points, fpr, tpr,
    thresholds) on the host, full length."""
    from fedfr_b200 import _native as N
    dev = torch.device("cuda:0")
    sd = torch.from_numpy(np.ascontiguousarray(s, np.float32)).to(dev)
    yd = torch.from_numpy(np.ascontiguousarray(y, np.uint8)).to(dev)
    n = sd.numel()
    ws = torch.empty(int(N.lib.pfc_roc_curve_workspace_bytes(n)), dtype=torch.uint8, device=dev)
    fpr, tpr, thr = (torch.full((n + 1 + PAD,), float("nan"), dtype=torch.float64, device=dev) for _ in range(3))
    out = torch.full((4,), -5, dtype=torch.int64, device=dev)
    N.check(N.lib.pfc_roc_curve(N.ptr(sd), N.ptr(yd), n, N.ptr(fpr), N.ptr(tpr), N.ptr(thr), N.ptr(out[3:]), N.ptr(out),
                                N.ptr(ws), ws.numel(), torch.cuda.current_stream(dev).cuda_stream), "pfc_roc_curve")
    o = out.cpu().numpy()
    return o[:3], int(o[3]), fpr.cpu().numpy(), tpr.cpu().numpy(), thr.cpu().numpy()


def large_case(kind, n):
    rng = np.random.default_rng(n + len(kind))
    y = rng.random(n) < 0.05
    s = (rng.standard_normal(n) * 0.2 + 0.5 * y).astype(np.float32)
    if kind == "ties":
        s = (np.round(s * 1024) / 1024).astype(np.float32)
    elif kind == "zeros":
        s = (np.round(s * 16) / 16).astype(np.float32)
        z = s == 0
        s[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(-0.0), np.float32(0.0))
    elif kind == "one_genuine":
        y = np.zeros(n, bool)
        y[n // 3] = True
    elif kind == "mostly_genuine":
        y = rng.random(n) < 0.9
    return s, y


def check_public(F, s, y):
    """roc_curve from numpy and from CUDA tensors: float64 CUDA tensors of the curve's length, equal to sklearn."""
    got = F.roc_curve(s, y)
    assert all(t.is_cuda and t.dtype == torch.float64 for t in got)
    got = [t.cpu().numpy() for t in got]
    assert_same_curve(got, s, y)
    again = F.roc_curve(torch.from_numpy(s).cuda(), torch.from_numpy(y).cuda())
    assert all(np.array_equal(a.cpu().numpy(), b) for a, b in zip(again, got))
    return got


@pytest.mark.parametrize("kind", KINDS)
def test_roc_curve_equals_sklearn(F, kind):
    s, y = make_case(kind)
    counts, k, fpr, tpr, thr = abi_roc(s, y)
    assert counts.tolist() == [int(y.sum()), int((~y).sum()), 0]
    assert np.isnan(fpr[k:]).all() and np.isnan(tpr[k:]).all() and np.isnan(thr[k:]).all()
    assert_same_curve((fpr[:k], tpr[:k], thr[:k]), s, y)
    check_public(F, s, y)


@pytest.mark.parametrize("kind", ["random", "ties", "zeros", "one_genuine", "mostly_genuine"])
@pytest.mark.parametrize("n", [70_001, 3_000_000])
def test_roc_curve_large(F, kind, n):
    """Thousands of sort tiles and more than one block of the digit-offset scan; two calls give the same bits."""
    s, y = large_case(kind, n)
    counts, k, fpr, tpr, thr = abi_roc(s, y)
    assert np.isnan(fpr[k:]).all()
    assert_same_curve((fpr[:k], tpr[:k], thr[:k]), s, y)
    _, k2, fpr2, tpr2, thr2 = abi_roc(s, y)
    assert k2 == k and all(np.array_equal(a[:k], b[:k]) for a, b in ((fpr, fpr2), (tpr, tpr2), (thr, thr2)))


def test_roc_curve_errors(F):
    s, y = make_case("random")
    for bad in (np.nan, np.inf, -np.inf):
        s2 = s.copy()
        s2[9] = bad
        with pytest.raises(ValueError, match="NaN or infinite"):
            F.roc_curve(s2, y)
    with pytest.raises(ValueError, match="genuine and impostor"):
        F.roc_curve(s[~y], y[~y])
    with pytest.raises(ValueError, match="genuine and impostor"):
        F.roc_curve(s[y], y[y])
    with pytest.raises(ValueError, match="one issame flag"):
        F.roc_curve(s, y[1:])
    with pytest.raises(ValueError, match="no scores"):
        F.roc_curve(s[:0], y[:0])


def test_ijbc_size(F):
    """IJB-C-shaped scores (15,658,489 pairs, 19,557 genuine) from template_features and pair_scores: the curve equals
    sklearn's array for array, and the TAR table read from it equals the one read from sklearn's curve."""
    from oracle import verify_oracle as O
    feats, t, m, p1, p2, y = O.ijbc_like(0)
    assert p1.size == 15_658_489 and int(y.sum()) == 19_557
    tf, ids = F.template_features(feats, t, m)
    scores = F.pair_scores(tf, ids, p1, p2)
    fpr, tpr, thr = F.roc_curve(scores, y)
    s = scores.cpu().numpy()
    want = sk_roc_curve(y, s)
    got = [fpr.cpu().numpy(), tpr.cpu().numpy(), thr.cpu().numpy()]
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    assert all(np.array_equal(g, o) for g, o in zip(got, RO.roc_curve(s, y)))
    assert auc(got[0], got[1]) == auc(want[0], want[1])
    table = F.tar_at_far_nearest(fpr, tpr)
    assert table == insightface_readout(want[0], want[1], F.verify.DEFAULT_FARS)
