"""The ROC curve of ``fedfr_b200.verify.roc_curve`` restated in numpy on counts -- TEST INFRASTRUCTURE ONLY.

The second oracle next to ``sklearn.metrics.roc_curve`` (the definition of include/fedfr_b200.h, steps 1-4): distinct
order-preserving keys of the fp32 scores with -0.0 folded onto +0.0, exact genuine / impostor counts per key in
descending key order, sklearn's thinning stated on those counts, and one float64 division per rate.  No float sort."""
import numpy as np


def score_key(scores):
    """fp32 scores -> order-preserving uint32 keys (the TAR kernels' ``tar_key``), -0.0 and +0.0 one key."""
    u = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32).copy()
    u[(u & 0x7FFFFFFF) == 0] = 0
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def key_value(keys):
    keys = np.asarray(keys, dtype=np.uint32)
    return np.where(keys & 0x80000000, keys & 0x7FFFFFFF, ~keys).astype(np.uint32).view(np.float32)


def roc_curve(scores, issame):
    """-> (fpr, tpr, thresholds) float64; ValueError for a NaN or infinite score or a missing class."""
    s = np.asarray(scores, dtype=np.float32).reshape(-1)
    y = np.asarray(issame).reshape(-1) != 0
    if not np.isfinite(s).all():
        raise ValueError("NaN or infinite score")
    if y.all() or not y.any():
        raise ValueError("needs genuine and impostor pairs")
    keys, inv = np.unique(score_key(s), return_inverse=True)            # ascending keys
    g = np.bincount(inv[y], minlength=keys.size)[::-1]                   # descending keys from here on
    i = np.bincount(inv[~y], minlength=keys.size)[::-1]
    keys = keys[::-1]
    keep = np.ones(keys.size, dtype=bool)
    keep[1:-1] = (g[2:] != g[1:-1]) | (i[2:] != i[1:-1])                  # empty with at most 2 keys
    tps, fps = np.cumsum(g)[keep], np.cumsum(i)[keep]
    fpr = np.r_[0.0, fps.astype(np.float64) / float(i.sum())]
    tpr = np.r_[0.0, tps.astype(np.float64) / float(g.sum())]
    return fpr, tpr, np.r_[np.inf, key_value(keys[keep]).astype(np.float64)]
