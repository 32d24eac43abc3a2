"""1:1 template verification (csrc/verify.cu, fedfr_b200/verify.py) without a GPU.

The C oracle (oracle/oracle_verify.c) is checked against a float64 numpy restatement of the recipe; the whole C-ABI of
verify.cu, built on the CPU execution-model emulator (tests/emu/cuda_emu.h, ``_build_abi`` of test_kernel_emulation.py),
must then reproduce the oracle's pooled features and scores bit for bit and the numpy definition of TAR@FAR exactly.
The index plumbing of the Python wrapper (``pool_index``, ``pair_rows``, ``tar_from_counts``) runs here on CPU tensors."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
from test_kernel_emulation import _build_abi  # noqa: E402

E_ARG, E_SHAPE, E_WS = -1, -2, -4


def make_images(seed, n_templates, emb, weighted=False, zero_template=False):
    """Synthetic IJB-style images: sparse and negative int64 template ids, 1-3 medias of 1-4 images each, template 0 a
    single image, a media id shared by templates 1 and 2, rows shuffled.  -> feats, templates, medias, weights."""
    rng = np.random.default_rng(seed)
    ids = np.unique(rng.integers(-2 ** 62, 2 ** 62, n_templates * 2))[:n_templates]
    rng.shuffle(ids)
    t, m = [], []
    for r, tid in enumerate(ids):
        n_media = 1 if r == 0 else int(rng.integers(1, 4))
        media_ids = rng.choice(np.arange(-40, 40), n_media, replace=False)
        if r in (1, 2):
            media_ids[0] = 777
        for mid in media_ids:
            k = 1 if r == 0 else int(rng.integers(1, 5))
            t += [tid] * k
            m += [mid] * k
    t, m = np.array(t, np.int64), np.array(m, np.int64)
    perm = rng.permutation(t.size)
    t, m = t[perm], m[perm]
    feats = (rng.standard_normal((t.size, emb)) * rng.uniform(0.5, 3.0, (t.size, 1))).astype(np.float32)
    w = rng.uniform(0.0, 2.0, t.size).astype(np.float32) if weighted else None
    if zero_template:
        if w is None:
            w = np.ones(t.size, np.float32)
        w[t == ids[3]] = 0.0
    return feats, t, m, w


def make_pairs(seed, ids, n_pairs):
    """Pair list grouped by p1 (runs of one p1, as IJB-C's), with a self pair."""
    rng = np.random.default_rng(seed)
    p1 = np.repeat(rng.choice(ids, max(1, n_pairs // 37)), 37)[:n_pairs]
    p2 = rng.choice(ids, p1.size)
    p2[0] = p1[0]
    return p1, p2


def make_scores(kind, seed, n=3000):
    """(scores fp32, issame bool) for the TAR@FAR edge cases."""
    rng = np.random.default_rng(seed)
    issame = rng.random(n) < 0.15
    s = (rng.standard_normal(n) * 0.2 + 0.45 * issame).astype(np.float32)
    if kind == "ties":                                   # coarse values: genuine and impostor ties at every threshold
        s = (np.round(s * 8) / 8).astype(np.float32)
    elif kind == "equal":                                # every impostor the same score
        s[~issame] = np.float32(0.25)
        s[np.nonzero(issame)[0][::3]] = np.float32(0.25)   # genuine pairs tied with them
    elif kind == "zeros":                                # -0.0 and +0.0 mixed, around the thresholds
        s = (np.round(s * 2) / 2).astype(np.float32)
        z = s == 0
        s[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(-0.0), np.float32(0.0))
    elif kind == "extremes":
        s[rng.integers(0, n, 20)] = np.float32(-np.inf)
        s[rng.integers(0, n, 20)] = np.float32(np.inf)
        s[rng.integers(0, n, 20)] = np.float32(-1e-40)
    return s, issame


FAR_SETS = [(1e-6, 1e-3, 1e-2, 1e-1, 0.5, 1.0), (0.9999, 0.37, 1.0 / 3, 2.0 ** -20)]


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import __graft_entry__ as g
    g.build()                                            # the C oracle and the product library (for its ctypes signatures)
    from fedfr_b200 import _native as N
    emu = _build_abi("verify", str(tmp_path_factory.mktemp("verify_emu")))
    for name in ("pfc_template_pool", "pfc_pair_scores", "pfc_tar_at_far_workspace_bytes", "pfc_tar_at_far"):
        f = getattr(emu, name)
        f.restype, f.argtypes = N.SIGNATURES[name]
    return emu


@pytest.fixture(scope="module")
def O():
    import __graft_entry__ as g
    g.build()
    from oracle import verify_oracle
    return verify_oracle


def emu_pool(lib, feats, templates, medias, weights=None):
    from fedfr_b200.verify import pool_index
    ids, order, media_start, tmpl_start = (x.numpy() for x in pool_index(torch.from_numpy(templates), torch.from_numpy(medias)))
    out = np.full((ids.size, feats.shape[1]), np.nan, np.float32)
    rc = lib.pfc_template_pool(feats.ctypes.data, None if weights is None else weights.ctypes.data, order.ctypes.data,
                               media_start.ctypes.data, tmpl_start.ctypes.data, ids.size, feats.shape[1], out.ctypes.data, None)
    assert rc == 0
    return out, ids


def emu_scores(lib, tf, r1, r2):
    r1, r2 = np.ascontiguousarray(r1, np.int64), np.ascontiguousarray(r2, np.int64)
    out = np.full(r1.size, 7.0, np.float32)
    assert lib.pfc_pair_scores(tf.ctypes.data, tf.shape[0], tf.shape[1], r1.ctypes.data, r2.ctypes.data, r1.size, out.ctypes.data, None) == 0
    return out


def emu_tar(lib, scores, issame, fars):
    from fedfr_b200.verify import tar_from_counts
    s = np.ascontiguousarray(scores, np.float32)
    y = np.ascontiguousarray(issame, np.uint8)
    f = np.asarray(fars, np.float64)
    ws = np.zeros(lib.pfc_tar_at_far_workspace_bytes(s.size) // 8 + 1, np.uint64)
    counts = np.full(3 + 2 * f.size, -5, np.int64)
    thr = np.full(f.size, np.nan, np.float32)
    rc = lib.pfc_tar_at_far(s.ctypes.data, y.ctypes.data, s.size, f.ctypes.data, f.size, counts.ctypes.data, thr.ctypes.data,
                            ws.ctypes.data, ws.nbytes, None)
    assert rc == 0
    return counts, thr, lambda: tar_from_counts(counts, thr, fars)


@pytest.mark.parametrize("weighted", [False, True])
def test_oracle_matches_float64_recipe(O, weighted):
    feats, t, m, w = make_images(1 + weighted, 30, 96, weighted=weighted)
    got, ids = O.template_pool(feats, t, m, w)
    want, want_ids = O.recipe_float64(feats, t, m, w)
    assert np.array_equal(ids, want_ids)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)
    p1, p2 = make_pairs(3, ids, 200)
    r1, r2 = np.searchsorted(ids, p1), np.searchsorted(ids, p2)
    np.testing.assert_allclose(O.pair_scores(got, r1, r2), np.einsum("pk,pk->p", want[r1], want[r2]), rtol=0, atol=1e-6)


@pytest.mark.parametrize("emb,weighted,zero_template,n_t", [(80, False, False, 12), (80, True, True, 9), (512, True, False, 5),
                                                            (33, False, True, 7)])
def test_emulated_pool_and_scores_match_oracle_bit_for_bit(lib, O, emb, weighted, zero_template, n_t):
    feats, t, m, w = make_images(emb + n_t, n_t, emb, weighted, zero_template)
    got, ids = emu_pool(lib, feats, t, m, w)
    want, want_ids = O.template_pool(feats, t, m, w)
    assert np.array_equal(ids, want_ids)
    assert np.array_equal(bits(got), bits(want))
    if zero_template:
        assert not got[np.searchsorted(ids, t[w == 0][0])].any()
    p1, p2 = make_pairs(emb, ids, 300)
    r1, r2 = np.searchsorted(ids, p1), np.searchsorted(ids, p2)
    assert np.array_equal(bits(emu_scores(lib, got, r1, r2)), bits(O.pair_scores(want, r1, r2)))


def test_emulated_scores_rows_out_of_range_are_nan(lib):
    tf = np.random.default_rng(0).standard_normal((4, 40)).astype(np.float32)
    out = emu_scores(lib, tf, [0, 4, 1, -1, 2], [1, 0, 7, 0, 2])
    assert np.isnan(out[[1, 2, 3]]).all() and not np.isnan(out[[0, 4]]).any()


@pytest.mark.parametrize("kind", ["random", "ties", "equal", "zeros", "extremes"])
@pytest.mark.parametrize("fars", FAR_SETS)
def test_emulated_tar_at_far_is_exact(lib, O, kind, fars):
    s, y = make_scores(kind, len(kind), 2500)
    counts, thr, result = emu_tar(lib, s, y, fars)
    assert counts[0] == y.sum() and counts[1] == (~y).sum() and counts[2] == 0
    assert result() == O.tar_at_far(s, y, fars)
    assert not np.signbit(thr[thr == 0]).any()               # the threshold key of -0.0 is that of +0.0


def test_emulated_tar_at_far_errors(lib):
    s, y = make_scores("random", 5, 600)
    s[17] = np.nan
    counts, _, result = emu_tar(lib, s, y, (0.1,))
    assert counts[2] == 1 and counts[0] + counts[1] == s.size - 1
    with pytest.raises(ValueError, match="NaN"):
        result()
    _, _, result = emu_tar(lib, s[~y & ~np.isnan(s)], y[~y & ~np.isnan(s)], (0.1,))
    with pytest.raises(ValueError, match="genuine"):
        result()


def test_pair_rows_unknown_id():
    from fedfr_b200.verify import pair_rows
    ids = torch.tensor([-5, 3, 2 ** 40])
    r1, r2 = pair_rows(ids, torch.tensor([3, -5]), torch.tensor([2 ** 40, 3]))
    assert r1.tolist() == [1, 0] and r2.tolist() == [2, 1]
    with pytest.raises(ValueError, match="unknown template id 4"):
        pair_rows(ids, torch.tensor([3, 4]), torch.tensor([3, 3]))
    with pytest.raises(ValueError, match="unknown template id 99"):
        pair_rows(ids, torch.tensor([3]), torch.tensor([99]))
    with pytest.raises(ValueError, match="sorted"):
        pair_rows(torch.tensor([3, -5]), torch.tensor([3]), torch.tensor([3]))


def test_c_abi_error_codes(lib):
    f = np.zeros((4, 8), np.float32)
    i64 = np.zeros(8, np.int64)
    p = lambda a: a.ctypes.data                                               # noqa: E731
    assert lib.pfc_template_pool(p(f), None, p(i64), p(i64), p(i64), 1, 0, p(f), None) == E_ARG
    assert lib.pfc_template_pool(p(f), None, p(i64), p(i64), p(i64), -1, 8, p(f), None) == E_ARG
    assert lib.pfc_template_pool(p(f), None, None, p(i64), p(i64), 1, 8, p(f), None) == E_ARG
    assert lib.pfc_template_pool(p(f), None, p(i64), p(i64), p(i64), 1, 4097, p(f), None) == E_SHAPE
    assert lib.pfc_template_pool(None, None, None, None, None, 0, 8, None, None) == 0       # no templates: nothing to do
    assert lib.pfc_pair_scores(p(f), 4, 8, p(i64), None, 2, p(f), None) == E_ARG
    assert lib.pfc_pair_scores(p(f), 4, 8, p(i64), p(i64), -1, p(f), None) == E_ARG
    assert lib.pfc_pair_scores(p(f), 4, 0, p(i64), p(i64), 2, p(f), None) == E_ARG
    assert lib.pfc_pair_scores(None, 4, 8, None, None, 0, None, None) == 0

    s, y = np.zeros(8, np.float32), np.zeros(8, np.uint8)
    ws = np.zeros(lib.pfc_tar_at_far_workspace_bytes(8) // 8 + 1, np.uint64)
    counts, thr = np.zeros(32, np.int64), np.zeros(16, np.float32)

    def tar(fars=(0.1,), n=8, n_far=None, w=ws.ctypes.data, wb=ws.nbytes, scores=p(s)):
        fa = np.asarray(fars, np.float64)
        return lib.pfc_tar_at_far(scores, p(y), n, fa.ctypes.data, len(fars) if n_far is None else n_far, p(counts), p(thr), w, wb, None)
    assert tar() == 0
    assert tar(scores=None) == E_ARG and tar(n=0) == E_ARG
    assert tar(fars=(0.0,)) == E_ARG and tar(fars=(1.5,)) == E_ARG and tar(fars=(float("nan"),)) == E_ARG
    assert tar(fars=(0.1,) * 9) == E_ARG and tar(n_far=0) == E_ARG
    assert tar(wb=8) == E_WS
    assert tar(w=ws.ctypes.data + 4) == E_ARG                                 # misaligned workspace
    assert tar(n=2 ** 31) == E_SHAPE


@pytest.mark.skipif(os.environ.get("EMU_ASAN") == "1", reason="this IS the sanitizer child")
def test_verify_emulation_under_address_sanitizer():
    """Every emulated test above once more in a child whose emulated build is compiled with -fsanitize=address and runs
    threads and blocks in descending order (EMU_SCHEDULE=reverse), as test_kernel_emulation.py does for its kernels:
    an out-of-bounds access aborts the child, a missing barrier changes a result."""
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
