"""The exact ROC curve (csrc/verify.cu pfc_roc_curve, fedfr_b200.verify.roc_curve / tar_at_far_nearest) without a GPU.

The emulated build of verify.cu (tests/emu/cuda_emu.h, ``_build_abi`` of test_kernel_emulation.py) must return
``sklearn.metrics.roc_curve`` and the numpy restatement on counts (tests/roc_curve_oracle.py) array for array, at the
edges of the definition and of the radix sort: ties, ±0.0, keys that differ in one radix digit only, n = 2 and 3, one
genuine pair, mostly genuine pairs, scores at ±1, and several sort tiles.  Output buffers start as NaN and are longer
than the curve, so an unwritten point or a store past the curve's end fails."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from sklearn.metrics import auc
from sklearn.metrics import roc_curve as sk_roc_curve

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import roc_curve_oracle as RO  # noqa: E402
from test_kernel_emulation import _build_abi  # noqa: E402

E_ARG, E_SHAPE, E_WS = -1, -2, -4
PAD = 5                                                  # NaN entries past the n + 1 the ABI may use


def key_scores(keys):
    """uint32 keys (order-preserving, see roc_curve_oracle.score_key) -> the fp32 scores they are the keys of."""
    return RO.key_value(np.asarray(keys, dtype=np.uint32))


def make_case(kind, seed=0):
    """(scores fp32, issame bool) for one edge case of the curve."""
    rng = np.random.default_rng(seed + len(kind))
    n = 1500
    y = rng.random(n) < 0.15
    s = (rng.standard_normal(n) * 0.2 + 0.45 * y).astype(np.float32)
    if kind == "distinct":                               # three sort tiles, every score different
        n = 5000
        s = np.unique(rng.standard_normal(3 * n).astype(np.float32))[:n]
        rng.shuffle(s)
        y = rng.random(n) < 0.3
    elif kind == "ties":                                 # scores rounded to 1/8: ties at every threshold, two tiles
        n = 3000
        y = rng.random(n) < 0.3
        s = (np.round((rng.standard_normal(n) * 0.3 + 0.3 * y) * 8) / 8).astype(np.float32)
    elif kind == "equal":
        s = np.full(n, 0.25, np.float32)
    elif kind == "zeros":                                # -0.0 and +0.0 mixed, in both classes
        s = (np.round(s * 2) / 2).astype(np.float32)
        z = s == 0
        s[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(-0.0), np.float32(0.0))
        assert np.signbit(s[z]).any() and (~np.signbit(s[z])).any()
    elif kind == "low_digit":                            # keys differ only in their lowest byte
        s = key_scores(0xBF3A7100 + rng.integers(0, 256, n))
    elif kind == "high_digit":                           # keys differ only in their highest byte (both signs)
        s = key_scores((rng.integers(1, 255, n).astype(np.uint32) << 24) | 0x5A5A5A)
    elif kind == "n2":
        s, y = np.array([0.5, 0.25], np.float32), np.array([False, True])
    elif kind == "n2_tied":
        s, y = np.array([0.5, 0.5], np.float32), np.array([True, False])
    elif kind == "n3":
        s, y = np.array([0.1, 0.7, 0.1], np.float32), np.array([True, False, False])
    elif kind == "one_genuine":
        y = np.zeros(n, bool)
        y[rng.integers(0, n)] = True
    elif kind == "mostly_genuine":
        y = rng.random(n) < 0.9
    elif kind == "pm_one":                               # scores at exactly -1 and +1, in both classes
        s = np.clip(s * 6, -1, 1).astype(np.float32)
        assert (s == 1).sum() > 10 and (s == -1).sum() > 10
    if not y.any() or y.all():
        y[0] = not y[0]
    return np.ascontiguousarray(s, np.float32), y


KINDS = ["random", "distinct", "ties", "equal", "zeros", "low_digit", "high_digit", "n2", "n2_tied", "n3", "one_genuine",
         "mostly_genuine", "pm_one"]


def insightface_readout(fpr, tpr, x_labels):
    """The TAR table of the insightface IJB scripts (FedFR's ijbc_all.py), verbatim in its lookup."""
    fpr, tpr = np.flipud(fpr), np.flipud(tpr)
    out = []
    for x in x_labels:
        _, min_index = min(list(zip(abs(fpr - x), range(len(fpr)))))
        out.append((float(x), float(tpr[min_index]), float(fpr[min_index])))
    return out


def assert_same_curve(got, s, y):
    want = sk_roc_curve(y, s)
    ora = RO.roc_curve(s, y)
    for g, w, o in zip(got, want, ora):
        assert g.dtype == np.float64 and g.shape == w.shape
        assert np.array_equal(g, w) and np.array_equal(g, o)
    assert auc(got[0], got[1]) == auc(want[0], want[1])


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import __graft_entry__ as g
    g.build()                                            # the product library, for its ctypes signatures
    from fedfr_b200 import _native as N
    emu = _build_abi("verify", str(tmp_path_factory.mktemp("roc_curve_emu")))
    for name in ("pfc_roc_curve_workspace_bytes", "pfc_roc_curve"):
        f = getattr(emu, name)
        f.restype, f.argtypes = N.SIGNATURES[name]
    return emu


def emu_roc(lib, scores, issame):
    """pfc_roc_curve on the emulated build -> (counts, n_points, fpr, tpr, thresholds); the outputs keep their full
    NaN-initialised length n + 1 + PAD."""
    s = np.ascontiguousarray(scores, np.float32)
    y = np.ascontiguousarray(issame, np.uint8)
    ws = np.zeros(lib.pfc_roc_curve_workspace_bytes(s.size) // 8 + 1, np.uint64)
    fpr, tpr, thr = (np.full(s.size + 1 + PAD, np.nan) for _ in range(3))
    n_points, counts = np.full(1, -5, np.int64), np.full(3, -5, np.int64)
    rc = lib.pfc_roc_curve(s.ctypes.data, y.ctypes.data, s.size, fpr.ctypes.data, tpr.ctypes.data, thr.ctypes.data,
                           n_points.ctypes.data, counts.ctypes.data, ws.ctypes.data, ws.nbytes, None)
    assert rc == 0
    return counts, int(n_points[0]), fpr, tpr, thr


@pytest.mark.parametrize("kind", KINDS)
def test_emulated_roc_curve_equals_sklearn(lib, kind):
    from fedfr_b200.verify import curve_length
    s, y = make_case(kind)
    counts, k, fpr, tpr, thr = emu_roc(lib, s, y)
    assert counts.tolist() == [int(y.sum()), int((~y).sum()), 0]
    assert curve_length(counts, k) == k and 2 <= k <= s.size + 1
    assert np.isnan(fpr[k:]).all() and np.isnan(tpr[k:]).all() and np.isnan(thr[k:]).all()
    assert_same_curve((fpr[:k], tpr[:k], thr[:k]), s, y)


def test_emulated_roc_curve_thins(lib):
    """Mostly impostor scores at distinct values: the thinning drops most points, as sklearn's does."""
    s, y = make_case("distinct")
    _, k, fpr, tpr, thr = emu_roc(lib, s, y)
    assert k < np.unique(s).size // 2
    assert_same_curve((fpr[:k], tpr[:k], thr[:k]), s, y)


def test_emulated_roc_curve_two_offset_groups(lib):
    """33 sort tiles: the digit offsets are scanned in two groups of up to 32 tiles."""
    rng = np.random.default_rng(3)
    n = 66_000
    y = rng.random(n) < 0.2
    s = (np.round(rng.standard_normal(n) * 64) / 64).astype(np.float32)
    _, k, fpr, tpr, thr = emu_roc(lib, s, y)
    assert np.isnan(fpr[k:]).all()
    assert_same_curve((fpr[:k], tpr[:k], thr[:k]), s, y)


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_emulated_roc_curve_nonfinite_scores(lib, bad):
    from fedfr_b200.verify import curve_length
    s, y = make_case("random")
    s[[3, 700]] = bad
    counts, k, _, _, _ = emu_roc(lib, s, y)
    assert counts[2] == 2 and counts[0] + counts[1] == s.size - 2
    with pytest.raises(ValueError, match="NaN or infinite"):
        curve_length(counts, k)
    with pytest.raises(ValueError):
        sk_roc_curve(y, s)                                # sklearn refuses them too


@pytest.mark.parametrize("cls", [True, False])
def test_emulated_roc_curve_one_class(lib, cls):
    from fedfr_b200.verify import curve_length
    s, _ = make_case("random")
    y = np.full(s.size, cls)
    counts, k, _, _, _ = emu_roc(lib, s, y)
    assert counts.tolist() == ([s.size, 0, 0] if cls else [0, s.size, 0])
    with pytest.raises(ValueError, match="genuine and impostor"):
        curve_length(counts, k)


def test_c_abi_error_codes_roc_curve(lib):
    s, y = np.zeros(8, np.float32), np.zeros(8, np.uint8)
    out = np.zeros(16)
    i64 = np.zeros(4, np.int64)
    ws = np.zeros(lib.pfc_roc_curve_workspace_bytes(8) // 8 + 1, np.uint64)
    p = lambda a: a.ctypes.data                                               # noqa: E731

    def roc(scores=p(s), issame=p(y), n=8, fpr=p(out), n_points=p(i64), w=p(ws), wb=ws.nbytes):
        return lib.pfc_roc_curve(scores, issame, n, fpr, p(out), p(out), n_points, p(i64), w, wb, None)
    assert roc() == 0
    assert roc(scores=None) == E_ARG and roc(issame=None) == E_ARG and roc(fpr=None) == E_ARG
    assert roc(n_points=None) == E_ARG and roc(w=None) == E_ARG
    assert roc(n=0) == E_ARG and roc(n=-1) == E_ARG
    assert roc(w=p(ws) + 4) == E_ARG                                          # misaligned workspace
    assert roc(n=2 ** 31) == E_SHAPE
    assert roc(wb=lib.pfc_roc_curve_workspace_bytes(8) - 1) == E_WS
    assert lib.pfc_roc_curve_workspace_bytes(0) == lib.pfc_roc_curve_workspace_bytes(-3) > 0
    assert lib.pfc_roc_curve_workspace_bytes(10 ** 6) > 18 * 10 ** 6


def test_roc_curve_input_errors():
    """Length checks come before any device work, so they raise ValueError on a machine without a GPU too."""
    from fedfr_b200.verify import curve_length, roc_curve
    with pytest.raises(ValueError, match="one issame flag per score"):
        roc_curve(np.zeros(4, np.float32), np.zeros(3, bool))
    with pytest.raises(ValueError, match="no scores"):
        roc_curve(np.zeros(0, np.float32), np.zeros(0, bool))
    with pytest.raises(ValueError, match="NaN or infinite"):
        curve_length([5, 5, 1], 4)
    with pytest.raises(ValueError, match="got 0 and 5"):
        curve_length([0, 5, 0], 2)
    with pytest.raises(ValueError, match="got 5 and 0"):
        curve_length([5, 0, 0], 2)
    assert curve_length([1, 1, 0], 3) == 3


@pytest.mark.parametrize("kind", ["random", "ties", "one_genuine", "mostly_genuine", "zeros"])
def test_tar_at_far_nearest_equals_insightface_readout(kind):
    from fedfr_b200.verify import DEFAULT_FARS, tar_at_far_nearest
    s, y = make_case(kind)
    fpr, tpr, _ = sk_roc_curve(y, s)
    fars = list(DEFAULT_FARS) + [0.3, 0.5, 1.0]
    assert tar_at_far_nearest(fpr, tpr, fars) == insightface_readout(fpr, tpr, fars)
    assert tar_at_far_nearest(torch.from_numpy(fpr), torch.from_numpy(tpr), fars) == insightface_readout(fpr, tpr, fars)


def test_tar_at_far_nearest_far_halfway_between_points():
    """16 impostors: every fpr is k / 16, so the midpoint of two neighbouring fprs is exactly as far from both.  The
    scripts take the first index of the minimum in the flipped curve (the larger fpr and tpr)."""
    from fedfr_b200.verify import tar_at_far_nearest
    rng = np.random.default_rng(5)
    s = rng.permutation(np.arange(40, dtype=np.float32) / 40)
    y = np.zeros(40, bool)
    y[np.argsort(s)[rng.choice(40, 24, replace=False)]] = True
    fpr, tpr, _ = sk_roc_curve(y, s)
    assert int((~y).sum()) == 16
    u = np.unique(fpr)
    mids = (u[1:] + u[:-1]) / 2
    assert np.array_equal(mids - u[:-1], u[1:] - mids)                   # exact ties
    got = tar_at_far_nearest(fpr, tpr, mids)
    assert got == insightface_readout(fpr, tpr, mids)
    assert all(far == u[q + 1] for q, (_, _, far) in enumerate(got))    # the tie goes to the larger fpr
    with pytest.raises(ValueError):
        tar_at_far_nearest(fpr, tpr[:-1])
    with pytest.raises(ValueError):
        tar_at_far_nearest([], [])


@pytest.mark.skipif(os.environ.get("EMU_ASAN") == "1", reason="this IS the sanitizer child")
def test_roc_curve_emulation_under_address_sanitizer():
    """Every emulated test above once more in a child whose emulated build is compiled with -fsanitize=address and runs
    threads and blocks in descending order (EMU_SCHEDULE=reverse), as test_verify.py does: an out-of-bounds access
    aborts the child, a result that depends on the schedule differs."""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not available")
    env = dict(os.environ, LD_PRELOAD=asan, EMU_ASAN="1", EMU_SCHEDULE="reverse",
               ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "emulated or c_abi"], env=env, capture_output=True, text=True, cwd=ROOT, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0 and "AddressSanitizer" not in r.stdout + r.stderr.replace(
        "ASan doesn't fully support makecontext/swapcontext", ""), tail
    assert " passed" in r.stdout, tail
