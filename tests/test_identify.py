"""1:N identification (csrc/identify.cu pfc_identify, fedfr_b200.verify mate_ranks / cmc / tpir_at_fpir) without a GPU.

The emulated build of identify.cu (tests/emu/cuda_emu.h plus its 64-bit additions in tests/emu/cuda_emu_u64.h, built the
way ``_build_abi`` of test_kernel_emulation.py builds a translation unit) must give every output equal bit for bit to
the literal C loop over the definition (``oracle_identify``, oracle/oracle_identify.c), and its ranks and top-1 rows
equal to the mate's position and element 0 of ``np.argsort(-S, axis=1, kind="stable")`` on the oracle's score rows.
Cases: P and G across the 64-row tile edges (1, 63, 64, 65, 200), E = 512, 80, 33 and 1, more tiles than resident CTAs,
integer features with many equal scores across tiles, duplicate gallery rows with the mate before and after its
duplicate, all scores equal, zero (and negative-zero) rows, probes without a mate, a gallery of one, NaN rows, and mate
rows outside [-1, G).  Outputs start as sentinels and are longer than the call may write; the workspace starts as 0xFF.
``cmc`` and the s' of ``tpir_at_fpir`` are checked against numpy restatements."""
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
from oracle import identify_oracle as IO  # noqa: E402
from oracle import verify_oracle as VO  # noqa: E402
from test_kernel_emulation import SAN_FLAGS, _transform_launches  # noqa: E402

E_ARG, E_SHAPE, E_WS = -1, -2, -4
PAD = 3                                                   # sentinel entries past what the ABI may write
SENT_I, SENT_F = -7, np.float32(-1234.5)


def make_case(kind, seed=0):
    """(probe fp32 [P, E], gallery fp32 [G, E], mate_row int64 [P]) for one case."""
    rng = np.random.default_rng(seed + 31 * len(kind))
    P, G, E = 65, 65, 64
    if kind.startswith("pg_"):
        P, G = (int(v) for v in kind[3:].split("x"))
    elif kind.startswith("e"):
        E = int(kind[1:])
    elif kind == "many_tiles":                            # 3 x 5 = 15 tiles over 4 resident CTAs
        P, G = 130, 300
    elif kind == "gallery_of_one":
        P, G = 40, 1
    gallery = rng.standard_normal((G, E)).astype(np.float32)
    gallery /= np.linalg.norm(gallery, axis=1, keepdims=True)
    mate = rng.integers(0, G, P)
    probe = (gallery[mate] + 0.9 * rng.standard_normal((P, E))).astype(np.float32)
    mate_row = np.where(rng.random(P) < 0.7, mate, -1).astype(np.int64)
    if kind == "ties":                                    # small integers: many equal scores, spread over the tiles
        G, E = 200, 33
        gallery = rng.integers(-1, 2, (G, E)).astype(np.float32)
        probe = rng.integers(-1, 2, (P, E)).astype(np.float32)
        mate_row = np.where(rng.random(P) < 0.8, rng.integers(0, G, P), -1).astype(np.int64)
    elif kind == "duplicates":                            # row 70 repeats row 5, row 130 repeats row 100
        G = 200
        gallery = rng.standard_normal((G, E)).astype(np.float32)
        gallery[70], gallery[130] = gallery[5], gallery[100]
        probe = np.repeat(gallery[[5, 5, 100, 100, 70, 130]], 11, axis=0)[:P]
        probe = (probe + 0.01 * rng.standard_normal(probe.shape)).astype(np.float32)
        mate_row = np.tile(np.array([5, 70, 100, 130, 70, 130]), 11)[:P].astype(np.int64)
    elif kind == "all_equal":
        gallery[:] = gallery[0]
        probe[:] = probe[0]
        mate_row = np.where(np.arange(P) % 5 == 0, -1, np.arange(P) % G).astype(np.int64)
    elif kind == "zero_rows":                             # score 0 (from +0.0 and -0.0 features) is one key
        gallery[[3, 40, 64]] = 0.0
        gallery[[10, 63]] = -0.0
        probe[[0, 7]] = 0.0
        probe[9] = -0.0
        mate_row[[0, 1, 2, 9]] = [3, 10, 40, 63]
    elif kind == "no_mate":
        mate_row[:] = -1
    elif kind == "nan_rows":
        probe[[4, 20]] = np.nan
        gallery[[7]] = np.nan
        mate_row[[4, 5, 6]] = [1, 7, -1]
    elif kind == "bad_mate":
        mate_row[[1, 2, 3]] = [G, -2, 2 ** 40]
    return np.ascontiguousarray(probe), np.ascontiguousarray(gallery), mate_row


KINDS = (["pg_%dx%d" % (p, g) for p, g in [(1, 1), (1, 200), (63, 65), (64, 64), (65, 63), (200, 1), (200, 200)]] +
         ["e512", "e80", "e33", "e1", "many_tiles", "ties", "duplicates", "all_equal", "zero_rows", "no_mate",
          "gallery_of_one", "nan_rows", "bad_mate"])


def build_verify_emu(tmp):
    """identify.cu, kernels and extern "C" entries, on the emulator: test_kernel_emulation's ``_build_abi`` with
    cuda_emu_u64.h included after cuda_emu.h."""
    import ctypes as C
    src = open(os.path.join(ROOT, "fedfr_b200", "csrc", "identify.cu")).read()
    body = _transform_launches(src.replace('#include "common.cuh"', '#include "cuda_emu.h"\n#include "cuda_emu_u64.h"', 1))
    assert "<<<" not in body and "cuda_emu_u64.h" in body
    cpp, so = os.path.join(tmp, "identify_emu.cpp"), os.path.join(tmp, "identify_emu.so")
    with open(cpp, "w") as f:
        f.write(body)
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas"] + SAN_FLAGS +
                       ["-I", os.path.join(HERE, "emu"), cpp, "-o", so], capture_output=True, text=True)
    assert r.returncode == 0, "\n".join(l for l in r.stderr.splitlines() if "error" in l)[:1500]
    return C.CDLL(so)


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import __graft_entry__ as g
    g.build()                                             # the product library, for its ctypes signatures
    from fedfr_b200 import _native as N
    emu = build_verify_emu(str(tmp_path_factory.mktemp("ident_emu")))
    for name in ("pfc_identify_workspace_bytes", "pfc_identify"):
        f = getattr(emu, name)
        f.restype, f.argtypes = N.SIGNATURES[name]
    return emu


def emu_identify(lib, probe, gallery, mate_row):
    """pfc_identify on the emulated build -> (rank, mate_score, top1_row, top1_score, counts)."""
    x = np.ascontiguousarray(probe, np.float32)
    y = np.ascontiguousarray(gallery, np.float32)
    m = np.ascontiguousarray(mate_row, np.int64)
    P, G = x.shape[0], y.shape[0]
    ws = np.zeros(lib.pfc_identify_workspace_bytes(P) // 8 + 1, np.uint64)
    ws.view(np.uint8)[:] = 0xFF
    rank, top1_row, counts = np.full(P + PAD, SENT_I, np.int64), np.full(P + PAD, SENT_I, np.int64), np.full(2 + PAD, SENT_I, np.int64)
    mate_score, top1_score = np.full(P + PAD, SENT_F, np.float32), np.full(P + PAD, SENT_F, np.float32)
    rc = lib.pfc_identify(x.ctypes.data, P, y.ctypes.data, G, x.shape[1], m.ctypes.data, rank.ctypes.data,
                          mate_score.ctypes.data, top1_row.ctypes.data, top1_score.ctypes.data, counts.ctypes.data,
                          ws.ctypes.data, ws.nbytes, None)
    assert rc == 0
    for a, n, s in ((rank, P, SENT_I), (top1_row, P, SENT_I), (counts, 2, SENT_I), (mate_score, P, SENT_F), (top1_score, P, SENT_F)):
        assert (a[n:] == s).all(), "a store past the output"
    return rank[:P], mate_score[:P], top1_row[:P], top1_score[:P], counts[:2]


def same_bits(a, b):
    """Equal element for element: NaN where the other is NaN, the same bits elsewhere."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype.kind != "f":
        return np.array_equal(a, b)
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32))


def check_outputs(got, probe, gallery, mate_row):
    """Every output against oracle_identify bit for bit; rank and top1_row against the numpy argsort."""
    want = IO.identify(probe, gallery, mate_row)
    for name, g, w in zip(("rank", "mate_score", "top1_row", "top1_score", "counts"), got, want):
        assert same_bits(g, w), name
    S = IO.score_matrix(probe, gallery)
    valid = (mate_row >= 0) & (mate_row < gallery.shape[0])
    rank, top1 = IO.argsort_ranks(S, np.where(valid, mate_row, -1))
    assert np.array_equal(got[0], rank) and np.array_equal(got[2], top1)
    return want


@pytest.mark.parametrize("kind", KINDS)
def test_emulated_identify_equals_oracle(lib, kind):
    probe, gallery, mate_row = make_case(kind)
    got = emu_identify(lib, probe, gallery, mate_row)
    check_outputs(got, probe, gallery, mate_row)


def test_emulated_identify_edges(lib):
    """The edge cases do what they were built to do."""
    probe, gallery, mate_row = make_case("ties")
    rank, ms, top1, ts, counts = emu_identify(lib, probe, gallery, mate_row)
    S = IO.score_matrix(probe, gallery)
    mated = np.flatnonzero(mate_row >= 0)
    assert sum(int((S[p] == S[p, mate_row[p]])[:mate_row[p]].sum()) for p in mated) > 50   # ties before the mate
    # top-1 ties whose rows lie in different 64-column tiles
    assert any(np.unique(np.flatnonzero(S[p] == S[p].max()) // 64).size > 1 for p in range(S.shape[0]))

    probe, gallery, mate_row = make_case("duplicates")
    rank, *_ = emu_identify(lib, probe, gallery, mate_row)
    S = IO.score_matrix(probe, gallery)
    assert (S[:, 5] == S[:, 70]).all() and (S[:, 100] == S[:, 130]).all()
    first, second = np.isin(mate_row, (5, 100)), np.isin(mate_row, (70, 130))
    assert first.any() and second.any()
    # the duplicate after the mate does not beat it; the one before does
    before = np.array([int((S[p] > S[p, mate_row[p]]).sum()) for p in range(mate_row.size)])
    assert np.array_equal(rank[first], 1 + before[first]) and np.array_equal(rank[second], 2 + before[second])

    probe, gallery, mate_row = make_case("all_equal")
    rank, ms, top1, ts, counts = emu_identify(lib, probe, gallery, mate_row)
    mated = mate_row >= 0
    assert np.array_equal(rank[mated], 1 + mate_row[mated]) and (rank[~mated] == 0).all() and (top1 == 0).all()

    probe, gallery, mate_row = make_case("zero_rows")
    rank, ms, top1, ts, counts = emu_identify(lib, probe, gallery, mate_row)
    assert (ms[[0, 9]] == 0).all() and not np.signbit(ts[[0, 7, 9]]).any() and (top1[[0, 7, 9]] == 0).all()
    assert rank[0] == 4 and rank[9] == 64                 # every score of a zero probe is 0: the rows before the mate tie

    probe, gallery, mate_row = make_case("no_mate")
    rank, ms, top1, ts, counts = emu_identify(lib, probe, gallery, mate_row)
    assert (rank == 0).all() and np.isnan(ms).all() and np.isfinite(ts).all()

    probe, gallery, mate_row = make_case("nan_rows")
    rank, ms, top1, ts, counts = emu_identify(lib, probe, gallery, mate_row)
    G = gallery.shape[0]
    assert counts[0] == 2 * G + (probe.shape[0] - 2) and counts[1] == 0
    assert np.isnan(ts[[4, 20]]).all() and (top1[[4, 20]] == 0).all() and np.isnan(ms[[4, 5]]).all()
    assert rank[5] == G                                   # a NaN mate: every number beats it, then the NaN rows before it

    probe, gallery, mate_row = make_case("bad_mate")
    rank, ms, top1, ts, counts = emu_identify(lib, probe, gallery, mate_row)
    assert counts[1] == 3 and (rank[1:4] == 0).all() and np.isnan(ms[1:4]).all()


def test_emulated_identify_is_schedule_free(lib):
    """Two calls give the same bits (the reverse-schedule child below runs every case once more)."""
    probe, gallery, mate_row = make_case("ties")
    a, b = emu_identify(lib, probe, gallery, mate_row), emu_identify(lib, probe, gallery, mate_row)
    assert all(same_bits(u, v) for u, v in zip(a, b))


def test_c_abi_error_codes_identify(lib):
    P, G, E = 8, 5, 4
    x, y, m = np.zeros((P, E), np.float32), np.zeros((G, E), np.float32), np.full(P, -1, np.int64)
    out = np.zeros(64, np.int64)
    ws = np.zeros(lib.pfc_identify_workspace_bytes(P) // 8 + 1, np.uint64)
    p = lambda a: a.ctypes.data                                               # noqa: E731

    def call(x_=p(x), n=P, y_=p(y), g=G, e=E, m_=p(m), rk=p(out), ms=p(out), t1=p(out), ts=p(out), c=p(out), w=p(ws),
             wb=ws.nbytes):
        return lib.pfc_identify(x_, n, y_, g, e, m_, rk, ms, t1, ts, c, w, wb, None)
    assert call() == 0
    for kw in ("x_", "y_", "m_", "rk", "ms", "t1", "ts", "c", "w"):
        assert call(**{kw: None}) == E_ARG, kw
    assert call(n=0) == E_ARG and call(n=-1) == E_ARG and call(g=0) == E_ARG and call(g=-1) == E_ARG
    assert call(e=0) == E_ARG and call(e=-4) == E_ARG
    assert call(w=p(ws) + 4) == E_ARG                                         # misaligned workspace
    assert call(e=4097) == E_SHAPE and call(n=2 ** 31) == E_SHAPE and call(g=2 ** 31) == E_SHAPE
    assert call(wb=lib.pfc_identify_workspace_bytes(P) - 1) == E_WS
    assert lib.pfc_identify_workspace_bytes(0) == lib.pfc_identify_workspace_bytes(-3)
    assert lib.pfc_identify_workspace_bytes(19593) >= 12 * 19593


def test_mate_rows_on_host():
    from fedfr_b200.verify import mate_rows
    g = torch.tensor([50, -3, 2 ** 40, 7])
    p = torch.tensor([7, 8, -3, 2 ** 40, 50, -4, 2 ** 41])
    assert mate_rows(p, g).tolist() == [3, -1, 1, 2, 0, -1, -1]
    with pytest.raises(ValueError, match="subject 7 occurs more than once"):
        mate_rows(p, torch.tensor([7, 1, 7]))


def cmc_numpy(rank, max_rank):
    rank = np.asarray(rank)
    mated = rank > 0
    return np.array([int((mated & (rank <= r)).sum()) / int(mated.sum()) for r in range(1, max_rank + 1)])


def s_prime_numpy(rank, mate_score, top1_score, max_rank):
    """The definition's s': mate_score for mated probes within rank R, -inf for other mated probes, top-1 otherwise."""
    rank = np.asarray(rank)
    return np.where(rank > 0, np.where(rank <= max_rank, mate_score, np.float32(-np.inf)), top1_score).astype(np.float32)


def test_cmc_equals_numpy():
    rng = np.random.default_rng(5)
    rank = np.where(rng.random(5000) < 0.3, 0, rng.integers(1, 40, 5000))
    from fedfr_b200.verify import cmc
    for R in (1, 5, 20, 45):
        got = cmc(torch.from_numpy(rank), R)
        assert got.dtype == torch.float64 and np.array_equal(got.numpy(), cmc_numpy(rank, R))
    with pytest.raises(ValueError, match="mated"):
        cmc(torch.zeros(4, dtype=torch.int64))
    with pytest.raises(ValueError, match="max_rank"):
        cmc(torch.ones(4, dtype=torch.int64), 0)


def test_tpir_input_errors():
    """The checks come before any device work."""
    from fedfr_b200.verify import tpir_at_fpir
    s = torch.zeros(4)
    with pytest.raises(ValueError, match="mated and non-mated"):
        tpir_at_fpir(torch.tensor([1, 2, 3, 1]), s, s)
    with pytest.raises(ValueError, match="mated and non-mated"):
        tpir_at_fpir(torch.zeros(4, dtype=torch.int64), s, s)
    with pytest.raises(ValueError, match="one entry per probe"):
        tpir_at_fpir(torch.tensor([1, 0, 3]), s, s)
    with pytest.raises(ValueError, match="max_rank"):
        tpir_at_fpir(torch.tensor([1, 0, 3, 0]), s, s, max_rank=0)


def test_tpir_s_prime_is_the_definition():
    """tar_at_far over s' equals the rank-and-threshold reading of TPIR@FPIR for every input, infinities included
    (numpy restatement of both sides on the oracle's outputs)."""
    probe, gallery, mate_row = make_case("ties")
    rank, ms, top1, ts, _ = IO.identify(probe, gallery, mate_row)
    ts = ts.copy()
    ts[:3] = [np.inf, -np.inf, 0.0]
    for R in (1, 3, 1000):
        sp = s_prime_numpy(rank, ms, ts, R)
        mated = rank > 0
        for f, tpir, fpir, thr in VO.tar_at_far(sp, mated, (1e-2, 0.1, 0.5, 1.0)):
            direct = int(((rank >= 1) & (rank <= R) & (ms > np.float32(thr))).sum()) / int(mated.sum())
            assert tpir == direct


@pytest.mark.skipif(os.environ.get("EMU_ASAN") == "1", reason="this IS the sanitizer child")
def test_identify_emulation_under_address_sanitizer():
    """Every emulated test above once more in a child whose emulated build is compiled with -fsanitize=address and runs
    threads and blocks in descending order (EMU_SCHEDULE=reverse), as test_kfold.py does: an out-of-bounds access
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
