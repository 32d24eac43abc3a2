"""1:1 template verification on the B200 (csrc/verify.cu through fedfr_b200.verify): pooled template features and pair
scores bit-identical to oracle/oracle_verify.c, TAR@FAR exactly the numpy definition, at the edge cases and at IJB-C size."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_verify import FAR_SETS, bits, make_images, make_pairs, make_scores  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    from oracle import verify_oracle
    return fedfr_b200, verify_oracle


@pytest.mark.parametrize("emb", [512, 80])
@pytest.mark.parametrize("weighted,zero_template", [(False, False), (True, False), (True, True), (False, True)])
def test_pool_and_scores_bit_identical_to_oracle(env, emb, weighted, zero_template):
    F, O = env
    feats, t, m, w = make_images(emb * 7 + weighted + 2 * zero_template, 300, emb, weighted, zero_template)
    got, ids = F.template_features(feats, t, m, w)
    want, want_ids = O.template_pool(feats, t, m, w)
    assert got.is_cuda and np.array_equal(ids.cpu().numpy(), want_ids)
    assert np.array_equal(bits(got.cpu().numpy()), bits(want))
    if zero_template:
        assert not got[int(np.searchsorted(want_ids, t[w == 0][0]))].any()
    p1, p2 = make_pairs(emb, want_ids, 20000)
    scores = F.pair_scores(got, ids, p1, p2)
    r1, r2 = np.searchsorted(want_ids, p1), np.searchsorted(want_ids, p2)
    assert np.array_equal(bits(scores.cpu().numpy()), bits(O.pair_scores(want, r1, r2)))
    # the same pairs ungrouped (shuffled): the same scores
    perm = np.random.default_rng(0).permutation(p1.size)
    assert np.array_equal(F.pair_scores(got, ids, p1[perm], p2[perm]).cpu().numpy(), scores.cpu().numpy()[perm])


def test_torch_inputs_on_the_device(env):
    F, O = env
    feats, t, m, w = make_images(5, 50, 128, True)
    dev = torch.device("cuda:0")
    got, ids = F.template_features(torch.from_numpy(feats).to(dev), torch.from_numpy(t).to(dev), torch.from_numpy(m).to(dev),
                                   torch.from_numpy(w).to(dev))
    want, _ = O.template_pool(feats, t, m, w)
    assert np.array_equal(bits(got.cpu().numpy()), bits(want))


@pytest.mark.parametrize("kind", ["random", "ties", "equal", "zeros", "extremes"])
@pytest.mark.parametrize("fars", FAR_SETS)
def test_tar_at_far_exact(env, kind, fars):
    F, O = env
    s, y = make_scores(kind, 11 + len(kind), 200_000)
    assert F.tar_at_far(s, y, fars) == O.tar_at_far(s, y, fars)
    got = F.tar_at_far(torch.from_numpy(s).cuda(), torch.from_numpy(y).cuda(), fars)
    assert got == O.tar_at_far(s, y, fars)


def test_tar_at_far_more_than_eight_fars_and_k0(env):
    F, O = env
    s, y = make_scores("random", 3, 50_000)
    fars = [10.0 ** -e for e in range(1, 8)] + [0.25, 0.5, 1.0]
    got = F.tar_at_far(s, y, fars)
    assert got == O.tar_at_far(s, y, fars)
    assert got[6][3] == float(s[~y].max())                     # k = 0: the largest impostor; no impostor accepted
    assert got[6][2] == 0.0 and got[-1][3] == float("-inf") and got[-1][1] == 1.0


def test_errors(env):
    F, _ = env
    s, y = make_scores("random", 4, 1000)
    s2 = s.copy()
    s2[10] = np.nan
    with pytest.raises(ValueError, match="NaN"):
        F.tar_at_far(s2, y)
    with pytest.raises(ValueError, match="genuine"):
        F.tar_at_far(s[~y], y[~y])
    with pytest.raises(ValueError, match="genuine"):
        F.tar_at_far(s[y], y[y])
    with pytest.raises(ValueError):
        F.tar_at_far(s, y, (0.0,))
    feats, t, m, _ = make_images(9, 20, 64)
    tf, ids = F.template_features(feats, t, m)
    bad = int(ids.max()) + 1
    with pytest.raises(ValueError, match="unknown template id %d" % bad):
        F.pair_scores(tf, ids, [int(ids[0])], [bad])


def test_ijbc_size(env):
    """One run at the IJB-C 1:1 shape (227,630 images, 23,124 templates, 15,658,489 pairs, 19,557 genuine): pooled
    features and a seeded sample of 100k scores bit-identical to the C oracle, every TAR@FAR point exact."""
    F, O = env
    feats, t, m, p1, p2, y = O.ijbc_like(0)
    tf, ids = F.template_features(feats, t, m)
    want, want_ids = O.template_pool(feats, t, m)
    assert np.array_equal(bits(tf.cpu().numpy()), bits(want))
    scores = F.pair_scores(tf, ids, p1, p2)
    sample = np.random.default_rng(1).choice(p1.size, 100_000, replace=False)
    r1, r2 = np.searchsorted(want_ids, p1[sample]), np.searchsorted(want_ids, p2[sample])
    assert np.array_equal(bits(scores.cpu().numpy()[sample]), bits(O.pair_scores(want, r1, r2)))
    got = F.tar_at_far(scores, y)
    assert got == O.tar_at_far(scores.cpu().numpy(), y, (1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1))
