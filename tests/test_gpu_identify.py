"""1:N identification on the B200 (csrc/identify.cu pfc_identify through fedfr_b200.verify mate_ranks / cmc /
tpir_at_fpir): the cases of test_identify.py against the same oracle and numpy argsort, the IJB-C 1:N shape (both
galleries) against the oracle on a seeded sample of probes, mate scores equal to ``pair_scores`` bit for bit, the same
bits from two calls, CUDA-tensor and numpy inputs, and CMC / TPIR@FPIR against numpy restatements."""
import os
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
from test_identify import KINDS, PAD, SENT_F, SENT_I, check_outputs, cmc_numpy, make_case, s_prime_numpy, same_bits  # noqa: E402
from test_verify import FAR_SETS  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def F():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


def abi_identify(probe, gallery, mate_row):
    """pfc_identify on the device with sentinel-filled outputs PAD entries longer than they need and a 0xFF workspace
    -> (rank, mate_score, top1_row, top1_score, counts) on the host, cut to their lengths after checking the tails."""
    from fedfr_b200 import _native as N
    dev = torch.device("cuda:0")
    x = torch.from_numpy(np.ascontiguousarray(probe, np.float32)).to(dev)
    y = torch.from_numpy(np.ascontiguousarray(gallery, np.float32)).to(dev)
    m = torch.from_numpy(np.ascontiguousarray(mate_row, np.int64)).to(dev)
    P, G = x.shape[0], y.shape[0]
    ws = torch.full((int(N.lib.pfc_identify_workspace_bytes(P)),), 0xFF, dtype=torch.uint8, device=dev)
    rank, top1_row = (torch.full((P + PAD,), SENT_I, dtype=torch.int64, device=dev) for _ in range(2))
    counts = torch.full((2 + PAD,), SENT_I, dtype=torch.int64, device=dev)
    mate_score, top1_score = (torch.full((P + PAD,), float(SENT_F), dtype=torch.float32, device=dev) for _ in range(2))
    N.check(N.lib.pfc_identify(N.ptr(x), P, N.ptr(y), G, x.shape[1], N.ptr(m), N.ptr(rank), N.ptr(mate_score),
                               N.ptr(top1_row), N.ptr(top1_score), N.ptr(counts), N.ptr(ws), ws.numel(),
                               torch.cuda.current_stream(dev).cuda_stream), "pfc_identify")
    out = []
    for a, n, s in ((rank, P, SENT_I), (mate_score, P, SENT_F), (top1_row, P, SENT_I), (top1_score, P, SENT_F),
                    (counts, 2, SENT_I)):
        h = a.cpu().numpy()
        assert (h[n:] == s).all(), "a store past the output"
        out.append(h[:n])
    return out


def subjects(mate_row, G, seed=0):
    """Sparse int64 subject ids: gallery row g has subject ids[g]; a probe's subject is its mate's, or an id no gallery
    row has."""
    rng = np.random.default_rng(seed)
    ids = rng.choice(2 ** 40, G + mate_row.size, replace=False).astype(np.int64) - 2 ** 39
    g_subj = ids[:G]
    p_subj = np.where(mate_row >= 0, g_subj[np.clip(mate_row, 0, G - 1)], ids[G:])
    return p_subj, g_subj


def check_public(F, probe, gallery, mate_row, want):
    """mate_ranks from numpy and from CUDA tensors: CUDA tensors equal to the ABI's outputs."""
    p_subj, g_subj = subjects(mate_row, gallery.shape[0])
    for args in ((probe, p_subj, gallery, g_subj), tuple(torch.from_numpy(a).cuda() for a in (probe, p_subj, gallery, g_subj))):
        got = F.mate_ranks(*args)
        assert all(g.is_cuda for g in got)
        assert [g.dtype for g in got] == [torch.int64, torch.float32, torch.int64, torch.float32]
        for g, w in zip(got, want[:4]):
            assert same_bits(g.cpu().numpy(), w)


@pytest.mark.parametrize("kind", KINDS)
def test_identify_equals_oracle(F, kind):
    probe, gallery, mate_row = make_case(kind)
    got = abi_identify(probe, gallery, mate_row)
    check_outputs(got, probe, gallery, mate_row)
    if kind == "nan_rows":
        p_subj, g_subj = subjects(mate_row, gallery.shape[0])
        with pytest.raises(ValueError, match="NaN"):
            F.mate_ranks(probe, p_subj, gallery, g_subj)
    elif kind != "bad_mate":
        check_public(F, probe, gallery, mate_row, got)


@pytest.fixture(scope="module")
def ijbc():
    return IO.ijbc_1n_like(seed=0)


def ijbc_rows(probe_subj, g_subj):
    order = np.argsort(g_subj)
    pos = np.clip(np.searchsorted(g_subj[order], probe_subj), 0, g_subj.size - 1)
    return np.where(g_subj[order][pos] == probe_subj, order[pos], -1).astype(np.int64)


@pytest.mark.parametrize("gallery", ["g1", "g2"])
def test_identify_ijbc_shape(F, ijbc, gallery):
    """19,593 probes against a full IJB-C-sized gallery: a seeded sample of 500 probes equals the oracle and the numpy
    argsort; every mate score equals pair_scores on the same rows bit for bit; CMC and TPIR@FPIR equal numpy
    restatements on the outputs."""
    probe, p_subj, g1, g2 = ijbc
    g_feats, g_subj = g1 if gallery == "g1" else g2
    x, ps, y, gs = (torch.from_numpy(a).cuda() for a in (probe, p_subj, g_feats, g_subj))
    rank, ms, top1, ts = (t.cpu().numpy() for t in F.mate_ranks(x, ps, y, gs))
    mate_row = ijbc_rows(p_subj, g_subj)
    assert np.array_equal(rank > 0, mate_row >= 0) and 0.4 < (mate_row >= 0).mean() < 0.6
    sample = np.sort(np.random.default_rng(1).choice(probe.shape[0], 500, replace=False))
    want = check_outputs([rank[sample], ms[sample], top1[sample], ts[sample], np.zeros(2, np.int64)],
                         probe[sample], g_feats, mate_row[sample])
    assert int(want[4][0]) == 0

    # mate scores are pair_scores of the same two rows (probe and gallery stacked into one template matrix)
    mated = np.flatnonzero(mate_row >= 0)
    tf = torch.cat([x, y])
    ids = torch.arange(tf.shape[0], device="cuda")
    pair = F.pair_scores(tf, ids, torch.from_numpy(mated).cuda(), torch.from_numpy(probe.shape[0] + mate_row[mated]).cuda())
    assert same_bits(pair.cpu().numpy(), ms[mated])

    r = torch.from_numpy(rank).cuda()
    assert (rank[mated] == 1).mean() > 0.5
    for R in (1, 5, 20):
        assert np.array_equal(F.cmc(r, R).cpu().numpy(), cmc_numpy(rank, R))
    for R in (1, 10):
        for fpirs in FAR_SETS:
            got = F.tpir_at_fpir(r, torch.from_numpy(ms).cuda(), torch.from_numpy(ts).cuda(), fpirs, max_rank=R)
            assert got == VO.tar_at_far(s_prime_numpy(rank, ms, ts, R), rank > 0, fpirs)


def test_identify_two_calls_same_bits(F, ijbc):
    probe, p_subj, (g_feats, g_subj), _ = ijbc
    args = [torch.from_numpy(a).cuda() for a in (probe, p_subj, g_feats, g_subj)]
    a, b = F.mate_ranks(*args), F.mate_ranks(*args)
    assert all(same_bits(u.cpu().numpy(), v.cpu().numpy()) for u, v in zip(a, b))


def test_identify_errors(F):
    probe, gallery, mate_row = make_case("pg_63x65")
    p_subj, g_subj = subjects(mate_row, gallery.shape[0])
    g_dup = g_subj.copy()
    g_dup[40] = g_dup[3]
    with pytest.raises(ValueError, match="more than once"):
        F.mate_ranks(probe, p_subj, gallery, g_dup)
    with pytest.raises(ValueError, match="one subject per"):
        F.mate_ranks(probe, p_subj[1:], gallery, g_subj)
    with pytest.raises(ValueError, match="one E"):
        F.mate_ranks(probe, p_subj, gallery[:, 1:], g_subj)
    with pytest.raises(RuntimeError, match="emb > 4096"):
        F.mate_ranks(np.zeros((2, 4097), np.float32), [1, 2], np.zeros((2, 4097), np.float32), [1, 3])
    rank = F.mate_ranks(probe, p_subj, gallery, g_subj)[0]
    with pytest.raises(ValueError, match="mated and non-mated"):
        F.tpir_at_fpir(rank[rank > 0], torch.zeros(int((rank > 0).sum()), device="cuda"),
                       torch.zeros(int((rank > 0).sum()), device="cuda"))
