"""The K-fold verification accuracy (csrc/verify.cu pfc_kfold_accuracy, fedfr_b200.verify.kfold_accuracy) without a GPU.

The emulated build of verify.cu (tests/emu/cuda_emu.h, ``_build_abi`` of test_kernel_emulation.py) must give:
- distances equal bit for bit to the pinned restatement (tests/kfold_oracle.py, (b));
- accuracy, best thresholds, tpr and fpr equal element for element to insightface's recipe ((a)) and to (b), both fed
  the kernel's distances;
- the same outputs as the recipe on its own float32 distances, except where a pair lies within 1e-6 of a grid
  threshold (such pairs are counted; every other pair must fall in the same bin).
Cases: uneven folds, F = 1, 2, 10 and P, distances exactly on grid values, train-accuracy ties, folds without genuine
or without impostor pairs, zero and NaN rows, with and without flipped embeddings, the 4,000-point grid and a custom
grid, E = 512, 33 and 1, and an LFW-shaped run.  Outputs start as NaN and are longer than the call may write."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import kfold_oracle as KO  # noqa: E402
from test_kernel_emulation import _build_abi  # noqa: E402

E_ARG, E_SHAPE, E_WS = -1, -2, -4
PAD = 3                                                   # NaN entries past what the ABI may write
BAND = 1e-6                                               # a pair this close to a threshold may bin differently


def make_case(kind, seed=0):
    """(emb fp32 [2P, E], flip fp32 [2P, E] or None, issame bool [P], nfolds, thresholds) for one case."""
    rng = np.random.default_rng(seed + 17 * len(kind))
    P, E, F, thr, with_flip = 403, 64, 10, KO.GRID, True
    if kind == "lfw":
        P, E = 6000, 512
    elif kind in ("e512", "e33", "e1"):
        E = int(kind[1:])
    elif kind == "noflip":
        with_flip = False
    elif kind == "grid4000":
        thr = np.arange(0, 4, 0.001)
    elif kind == "custom_grid":                           # unevenly spaced, below 0 and past 4
        thr = np.unique(np.r_[-0.5, rng.uniform(0, 4, 35), 4.5])
    y = rng.random(P) < 0.5
    # the second row mixes the first with noise, genuine pairs more of it: the distances of both classes overlap
    base = rng.standard_normal((P, E)).astype(np.float32)
    other = rng.standard_normal((P, E)).astype(np.float32)
    mix = np.where(y, rng.uniform(0.25, 0.9, P), rng.uniform(0.0, 0.45, P))[:, None].astype(np.float32)
    second = (mix * base + (1 - mix) * other).astype(np.float32)
    emb = np.empty((2 * P, E), np.float32)
    emb[0::2], emb[1::2] = base, second
    flip = (emb + 0.3 * rng.standard_normal(emb.shape)).astype(np.float32) if with_flip else None
    if kind == "on_grid":                                 # d = 0, 2 and 4 exactly: equal, orthogonal, opposite rows
        for p in range(0, P, 7):
            e0, e1 = np.zeros(E, np.float32), np.zeros(E, np.float32)
            e0[p % E] = 3.0
            e1[(p + 1) % E] = 0.5
            emb[2 * p] = e0
            emb[2 * p + 1] = (e0, e1, -e0)[(p // 7) % 3]
            flip[2 * p], flip[2 * p + 1] = emb[2 * p], emb[2 * p + 1]
        assert (thr == 2.0).any() and thr[0] == 0.0
    elif kind == "ties":                                  # two clusters far apart: a plateau of equal train accuracy
        d = np.where(y, 0.205, 1.705)
        emb[0::2] = 0
        emb[1::2] = 0
        emb[0::2, 0] = 1
        emb[1::2, 0] = 1 - d / 2
        emb[1::2, 1] = np.sqrt(1 - (1 - d / 2) ** 2)
        flip = None
    elif kind == "one_class_folds":                       # fold 0 has no genuine pair, fold 1 no impostor
        y[:41] = False
        y[41:81] = True
    elif kind == "zero_nan":
        emb[[4, 9, 30]] = 0
        flip[[4, 9, 30]] = 0                              # zero rows after fusion: norm 1
        emb[[17, 60]] = np.nan
    elif kind == "uneven":
        P2 = 997                                          # 997 = 10 * 99 + 7
        emb, flip, y = emb[:2 * P2], flip[:2 * P2], y[:P2]
    elif kind.startswith("folds_"):
        F = {"folds_1": 1, "folds_2": 2, "folds_P": 61}[kind]
        emb, flip, y = emb[:122], flip[:122], y[:61]
    return np.ascontiguousarray(emb), flip, y, F, np.asarray(thr, np.float64)


KINDS = ["random", "uneven", "folds_1", "folds_2", "folds_P", "on_grid", "ties", "one_class_folds", "zero_nan", "noflip",
         "grid4000", "custom_grid", "e512", "e33", "e1"]


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import __graft_entry__ as g
    g.build()                                             # the product library, for its ctypes signatures
    from fedfr_b200 import _native as N
    emu = _build_abi("verify", str(tmp_path_factory.mktemp("kfold_emu")))
    for name in ("pfc_kfold_workspace_bytes", "pfc_kfold_accuracy"):
        f = getattr(emu, name)
        f.restype, f.argtypes = N.SIGNATURES[name]
    return emu


def emu_kfold(lib, emb, flip, issame, nfolds, thr):
    """pfc_kfold_accuracy on the emulated build -> (dist, accuracy, best_thr, tpr, fpr), each NaN-initialised and PAD
    entries longer than its output."""
    e = np.ascontiguousarray(emb, np.float32)
    fl = None if flip is None else np.ascontiguousarray(flip, np.float32)
    y = np.ascontiguousarray(issame, np.uint8)
    t = np.ascontiguousarray(thr, np.float64)
    P, T = y.size, t.size
    ws = np.zeros(lib.pfc_kfold_workspace_bytes(P, T, nfolds) // 8 + 1, np.uint64)
    ws.view(np.uint8)[:] = 0xFF                           # the call must not read workspace it did not write
    dist = np.full(P + PAD, np.nan, np.float32)
    acc, best = np.full(nfolds + PAD, np.nan), np.full(nfolds + PAD, np.nan)
    tpr, fpr = np.full(T + PAD, np.nan), np.full(T + PAD, np.nan)
    rc = lib.pfc_kfold_accuracy(e.ctypes.data, None if fl is None else fl.ctypes.data, y.ctypes.data, P, e.shape[1],
                                t.ctypes.data, T, nfolds, dist.ctypes.data, acc.ctypes.data, best.ctypes.data,
                                tpr.ctypes.data, fpr.ctypes.data, ws.ctypes.data, ws.nbytes, None)
    assert rc == 0
    for a, n in ((dist, P), (acc, nfolds), (best, nfolds), (tpr, T), (fpr, T)):
        assert np.isnan(a[n:]).all(), "a store past the output"
    return dist[:P], acc[:nfolds], best[:nfolds], tpr[:T], fpr[:T]


def same_bits(a, b):
    """Equal element for element, NaN where the other is NaN, and the same bits elsewhere."""
    a, b = np.asarray(a), np.asarray(b)
    nan = np.isnan(a)
    return a.shape == b.shape and np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan], b[~nan]) and \
        np.array_equal(np.signbit(a[~nan]), np.signbit(b[~nan]))


def check_outputs(got, emb, flip, y, F, thr):
    """The kernel's outputs against (b) and (a) on the kernel's distances, and against (a) on its own distances.
    -> the number of pairs within BAND of a threshold."""
    dist, acc, best, tpr, fpr = got
    assert same_bits(dist, KO.pinned_dist(emb, flip))
    assert np.array_equal(KO.pinned_bins(dist, thr), KO.pinned_bins(KO.pinned_dist(emb, flip), thr))
    r_tpr, r_fpr, r_acc, r_best = KO.roc_from_dist(thr, dist, y, F)
    for want in (KO.pinned_from_dist(dist, y, F, thr), (r_acc, r_best, r_tpr, r_fpr)):
        for g, w in zip((acc, best, tpr, fpr), want):
            assert g.dtype == np.float64 and np.array_equal(g, w)
    if np.isnan(emb).any() or (flip is not None and np.isnan(flip).any()):
        return 0                                          # sklearn's normalize refuses NaN rows
    r_acc, r_best, r_tpr, r_fpr, r_dist = KO.insightface_kfold(emb, y, flip, F, thr)
    near = lambda d: (np.abs(np.asarray(d, np.float64)[:, None] - thr[None, :]) <= BAND).any(1)   # noqa: E731
    band = near(dist) | near(r_dist)
    kb, rb = KO.pinned_bins(dist, thr), KO.pinned_bins(r_dist, thr)
    assert np.array_equal(kb[~band], rb[~band])
    if np.array_equal(kb, rb):
        for g, w in zip((acc, best, tpr, fpr), (r_acc, r_best, r_tpr, r_fpr)):
            assert np.array_equal(g, w)
    return int(band.sum())


@pytest.mark.parametrize("kind", KINDS)
def test_emulated_kfold_equals_recipe(lib, kind):
    emb, flip, y, F, thr = make_case(kind)
    got = emu_kfold(lib, emb, flip, y, F, thr)
    n_band = check_outputs(got, emb, flip, y, F, thr)
    if kind not in ("on_grid", "e1"):                     # there pairs sit on thresholds by design (E = 1: d = 0 or 4)
        assert n_band <= max(2, y.size // 500)


def test_emulated_kfold_lfw_shape(lib):
    """6,000 pairs of E = 512 with flipped embeddings, 10 folds on the default grid: evaluate()'s LFW call."""
    emb, flip, y, F, thr = make_case("lfw")
    got = emu_kfold(lib, emb, flip, y, F, thr)
    check_outputs(got, emb, flip, y, F, thr)
    assert 0.5 < got[1].mean() < 1.0


def test_emulated_kfold_edges(lib):
    """The edge cases do what they were built to do."""
    emb, flip, y, F, thr = make_case("on_grid")
    dist, acc, best, tpr, fpr = emu_kfold(lib, emb, flip, y, F, thr)
    on = np.arange(0, y.size, 7)
    assert set(np.unique(dist[on]).tolist()) == {0.0, 2.0, 4.0}
    b = KO.pinned_bins(dist, thr)
    assert (b[on][dist[on] == 0] == 1).all()             # d = 0 is not < 0: first "same" at thr[1]
    assert (thr[b[on][dist[on] == 2]] > 2).all() and (thr[b[on][dist[on] == 2] - 1] == 2).all()
    assert (b[on][dist[on] == 4] == thr.size).all()       # beyond the grid: never "same"

    emb, flip, y, F, thr = make_case("ties")
    dist, acc, best, tpr, fpr = emu_kfold(lib, emb, flip, y, F, thr)
    assert (acc == 1.0).all()                             # a plateau from 0.21 to 1.70; the first threshold wins
    first = thr[np.searchsorted(thr, dist[y].astype(np.float64).max(), side="right")]
    assert (best == first).all() and first < 0.22

    emb, flip, y, F, thr = make_case("one_class_folds")
    dist, acc, best, tpr, fpr = emu_kfold(lib, emb, flip, y, F, thr)
    assert y[:41].sum() == 0 and y[41:81].all()
    assert np.isfinite(tpr).all() and np.isfinite(fpr).all()

    emb, flip, y, F, thr = make_case("zero_nan")
    dist, *_ = emu_kfold(lib, emb, flip, y, F, thr)
    assert np.isnan(dist[[8, 30]]).all() and np.isfinite(np.delete(dist, [8, 30])).all()
    assert abs(dist[2] - 1) < 1e-6                        # rows 4 and 5: a zero row against a unit row
    assert (KO.pinned_bins(dist, thr)[[8, 30]] == thr.size).all()


def test_emulated_kfold_uneven_folds_are_sklearns(lib):
    """P = 997, F = 10: the first seven test blocks hold 100 pairs, the last three 99 (sklearn's KFold)."""
    from sklearn.model_selection import KFold
    got = [(int(te[0]), int(te[-1]) + 1) for _, te in KFold(10).split(np.arange(997))]
    assert KO.fold_ranges(997, 10) == got and got[6] == (600, 700) and got[7] == (700, 799)


def test_emulated_kfold_is_schedule_free(lib):
    """Two calls give the same bits (the reverse-schedule child below runs every case once more)."""
    emb, flip, y, F, thr = make_case("random")
    a, b = emu_kfold(lib, emb, flip, y, F, thr), emu_kfold(lib, emb, flip, y, F, thr)
    assert all(same_bits(u, v) for u, v in zip(a, b))


def test_c_abi_error_codes_kfold(lib):
    P, E, T, F = 8, 4, 5, 2
    emb, y, thr = np.zeros((2 * P, E), np.float32), np.zeros(P, np.uint8), np.arange(T, dtype=np.float64)
    out = np.zeros(64)
    ws = np.zeros(lib.pfc_kfold_workspace_bytes(P, T, P) // 8 + 1, np.uint64)
    p = lambda a: a.ctypes.data                                               # noqa: E731

    def call(e=p(emb), fl=None, iss=p(y), n=P, emb_dim=E, t=p(thr), nt=T, nf=F, dist=p(out), acc=p(out), w=p(ws),
             wb=ws.nbytes):
        return lib.pfc_kfold_accuracy(e, fl, iss, n, emb_dim, t, nt, nf, dist, acc, p(out), p(out), p(out), w, wb, None)
    assert lib.pfc_kfold_workspace_bytes(P, T, P) > lib.pfc_kfold_workspace_bytes(P, T, F)
    assert call() == 0 and call(fl=p(emb)) == 0
    assert call(e=None) == E_ARG and call(iss=None) == E_ARG and call(t=None) == E_ARG
    assert call(dist=None) == E_ARG and call(acc=None) == E_ARG and call(w=None) == E_ARG
    assert call(n=0) == E_ARG and call(n=-1) == E_ARG and call(emb_dim=0) == E_ARG and call(nt=0) == E_ARG
    assert call(nf=0) == E_ARG and call(nf=P + 1) == E_ARG and call(nf=P) == 0
    assert call(w=p(ws) + 4) == E_ARG                                         # misaligned workspace
    assert call(emb_dim=4097) == E_SHAPE and call(n=2 ** 31) == E_SHAPE and call(nt=16385) == E_SHAPE
    assert call(wb=lib.pfc_kfold_workspace_bytes(P, T, F) - 1) == E_WS
    assert lib.pfc_kfold_workspace_bytes(0, 0, 0) == lib.pfc_kfold_workspace_bytes(-3, -1, -2)
    assert lib.pfc_kfold_workspace_bytes(6000, 400, 10) >= 4 * 6000 + 24 * 10 * 400


def test_kfold_input_errors():
    """Every check comes before any device work, so the ValueErrors are raised on a machine without a GPU too."""
    from fedfr_b200.verify import kfold_accuracy, kfold_thresholds
    emb, y = np.zeros((10, 4), np.float32), np.zeros(5, bool)
    with pytest.raises(ValueError, match="even number of rows"):
        kfold_accuracy(emb[:9], y)
    with pytest.raises(ValueError, match="even number of rows"):
        kfold_accuracy(emb[:, 0], y)
    with pytest.raises(ValueError, match="shape of embeddings"):
        kfold_accuracy(emb, y, flipped=emb[:8])
    with pytest.raises(ValueError, match="one issame flag per pair"):
        kfold_accuracy(emb, y[:4])
    for nf in (0, 6, -1):
        with pytest.raises(ValueError, match="nfolds"):
            kfold_accuracy(emb, y, nfolds=nf)
    for bad, msg in (([[0.1, 0.2]], "1-D"), ([], "1-D"), ([0.1, np.nan], "finite"), ([0.1, np.inf], "finite"),
                     ([0.1, 0.1, 0.3], "ascending"), ([0.3, 0.2], "ascending")):
        with pytest.raises(ValueError, match=msg):
            kfold_accuracy(emb, y, nfolds=5, thresholds=bad)
    assert np.array_equal(kfold_thresholds(), np.arange(0, 4, 0.01))
    assert np.array_equal(kfold_thresholds([0, 1.5]), [0.0, 1.5])


@pytest.mark.skipif(os.environ.get("EMU_ASAN") == "1", reason="this IS the sanitizer child")
def test_kfold_emulation_under_address_sanitizer():
    """Every emulated test above once more in a child whose emulated build is compiled with -fsanitize=address and runs
    threads and blocks in descending order (EMU_SCHEDULE=reverse), as test_roc_curve.py does: an out-of-bounds access
    aborts the child, a result that depends on the schedule differs."""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not available")
    env = dict(os.environ, LD_PRELOAD=asan, EMU_ASAN="1", EMU_SCHEDULE="reverse",
               ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "emulated or c_abi"], env=env, capture_output=True, text=True, cwd=ROOT, timeout=2400)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0 and "AddressSanitizer" not in r.stdout + r.stderr.replace(
        "ASan doesn't fully support makecontext/swapcontext", ""), tail
    assert " passed" in r.stdout, tail
