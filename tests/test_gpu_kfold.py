"""The K-fold verification accuracy on the B200 (csrc/verify.cu pfc_kfold_accuracy through
fedfr_b200.verify.kfold_accuracy): the cases of test_kfold.py against the same two restatements, LFW-, CFP-FP- and
AgeDB-30-shaped seeded runs against insightface's recipe, the same bits from two calls, and a call under
``torch.cuda.set_sync_debug_mode("error")``."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import kfold_oracle as KO  # noqa: E402
from test_kfold import KINDS, PAD, check_outputs, make_case, same_bits  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def F():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


def abi_kfold(emb, flip, issame, nfolds, thr):
    """pfc_kfold_accuracy on the device with NaN-filled outputs PAD entries longer than they need -> (dist, accuracy,
    best_thr, tpr, fpr) on the host, cut to their lengths after checking the tails."""
    from fedfr_b200 import _native as N
    dev = torch.device("cuda:0")
    e = torch.from_numpy(np.ascontiguousarray(emb, np.float32)).to(dev)
    fl = None if flip is None else torch.from_numpy(np.ascontiguousarray(flip, np.float32)).to(dev)
    y = torch.from_numpy(np.ascontiguousarray(issame, np.uint8)).to(dev)
    t = torch.from_numpy(np.ascontiguousarray(thr, np.float64)).to(dev)
    P, T = y.numel(), t.numel()
    ws = torch.full((int(N.lib.pfc_kfold_workspace_bytes(P, T, nfolds)),), 0xFF, dtype=torch.uint8, device=dev)
    dist = torch.full((P + PAD,), float("nan"), dtype=torch.float32, device=dev)
    acc, best = (torch.full((nfolds + PAD,), float("nan"), dtype=torch.float64, device=dev) for _ in range(2))
    tpr, fpr = (torch.full((T + PAD,), float("nan"), dtype=torch.float64, device=dev) for _ in range(2))
    N.check(N.lib.pfc_kfold_accuracy(N.ptr(e), N.ptr(fl), N.ptr(y), P, e.shape[1], N.ptr(t), T, nfolds, N.ptr(dist),
                                     N.ptr(acc), N.ptr(best), N.ptr(tpr), N.ptr(fpr), N.ptr(ws), ws.numel(),
                                     torch.cuda.current_stream(dev).cuda_stream), "pfc_kfold_accuracy")
    out = []
    for a, n in ((dist, P), (acc, nfolds), (best, nfolds), (tpr, T), (fpr, T)):
        h = a.cpu().numpy()
        assert np.isnan(h[n:]).all(), "a store past the output"
        out.append(h[:n])
    return out


def check_public(F, emb, flip, y, nfolds, thr, want):
    """kfold_accuracy from numpy and from CUDA tensors: float64 CUDA tensors equal to the ABI's outputs."""
    for args in ((emb, flip, y), tuple(None if a is None else torch.from_numpy(np.asarray(a)).cuda() for a in (emb, flip, y))):
        got = F.kfold_accuracy(args[0], args[2], flipped=args[1], nfolds=nfolds, thresholds=thr)
        assert all(g.is_cuda and g.dtype == torch.float64 for g in got)
        for g, w in zip(got, want[1:]):
            assert np.array_equal(g.cpu().numpy(), w)


@pytest.mark.parametrize("kind", KINDS)
def test_kfold_equals_recipe(F, kind):
    emb, flip, y, nfolds, thr = make_case(kind)
    got = abi_kfold(emb, flip, y, nfolds, thr)
    check_outputs(got, emb, flip, y, nfolds, thr)
    check_public(F, emb, flip, y, nfolds, thr, got)


def benchmark_like(name):
    """Seeded embeddings of a verification set's shape: LFW and AgeDB-30 have 6,000 pairs, CFP-FP 7,000; E = 512, half
    genuine, with flipped embeddings."""
    P = {"lfw": 6000, "cfp_fp": 7000, "agedb_30": 6000}[name]
    rng = np.random.default_rng(len(name) * 1000 + P)
    E = 512
    y = np.arange(P) // 300 % 2 == 0                      # the .bin files alternate blocks of 300 same / different pairs
    base = rng.standard_normal((P, E)).astype(np.float32)
    other = rng.standard_normal((P, E)).astype(np.float32)
    mix = np.where(y, rng.uniform(0.3, 0.9, P), rng.uniform(0.0, 0.4, P))[:, None].astype(np.float32)
    emb = np.empty((2 * P, E), np.float32)
    emb[0::2], emb[1::2] = base, (mix * base + (1 - mix) * other).astype(np.float32)
    flip = (emb + 0.3 * rng.standard_normal(emb.shape)).astype(np.float32)
    return emb, flip, y


@pytest.mark.parametrize("name", ["lfw", "cfp_fp", "agedb_30"])
def test_kfold_benchmark_shapes(F, name):
    """insightface's evaluate(): 10 folds on np.arange(0, 4, 0.01); the outputs equal the recipe's, and the mean and
    std of the accuracy are test()'s acc2 and std2."""
    emb, flip, y = benchmark_like(name)
    got = abi_kfold(emb, flip, y, 10, KO.GRID)
    n_band = check_outputs(got, emb, flip, y, 10, KO.GRID)
    assert n_band <= y.size // 500
    acc, best, tpr, fpr = F.kfold_accuracy(torch.from_numpy(emb).cuda(), torch.from_numpy(y).cuda(),
                                           flipped=torch.from_numpy(flip).cuda())
    assert np.array_equal(acc.cpu().numpy(), got[1])
    assert abs(float(acc.mean()) - np.mean(got[1])) < 1e-15 and abs(float(acc.std(correction=0)) - np.std(got[1])) < 1e-15
    assert 0.5 < float(acc.mean()) < 1.0


def test_kfold_two_calls_same_bits(F):
    emb, flip, y = benchmark_like("lfw")
    a, b = abi_kfold(emb, flip, y, 10, KO.GRID), abi_kfold(emb, flip, y, 10, KO.GRID)
    assert all(same_bits(u, v) for u, v in zip(a, b))


def test_kfold_does_not_synchronise(F):
    """CUDA-tensor inputs and the default grid: no call waits for the device."""
    emb, flip, y = benchmark_like("agedb_30")
    e, fl, yy = (torch.from_numpy(a).cuda() for a in (emb, flip, y))
    want = [t.cpu().numpy() for t in F.kfold_accuracy(e, yy, flipped=fl)]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = F.kfold_accuracy(e, yy, flipped=fl)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert all(np.array_equal(g.cpu().numpy(), w) for g, w in zip(got, want))


def test_kfold_errors(F):
    emb, flip, y, _, _ = make_case("random")
    with pytest.raises(ValueError, match="one issame flag"):
        F.kfold_accuracy(emb, y[1:])
    with pytest.raises(ValueError, match="nfolds"):
        F.kfold_accuracy(emb, y, nfolds=y.size + 1)
    with pytest.raises(ValueError, match="ascending"):
        F.kfold_accuracy(emb, y, thresholds=torch.tensor([0.5, 0.25], dtype=torch.float64, device="cuda"))
    with pytest.raises(RuntimeError, match="emb > 4096"):
        F.kfold_accuracy(np.zeros((4, 4097), np.float32), np.zeros(2, bool), nfolds=2)
    with pytest.raises(RuntimeError, match="16384"):
        F.kfold_accuracy(emb, y, thresholds=np.arange(16385) / 4096.0)
