"""The K-fold verification accuracy of ``fedfr_b200.verify.kfold_accuracy`` restated twice -- TEST INFRASTRUCTURE ONLY.

(a) ``insightface_*``: insightface's eval/verification.py (vendored by FedFR) verbatim in numpy + sklearn: ``test()``'s
    flip fusion and ``sklearn.preprocessing.normalize``, then ``evaluate``'s pair split and ``calculate_roc`` /
    ``calculate_accuracy`` with ``KFold`` (``LFold`` for one fold).  ``roc_from_dist`` is its fold loop on given
    distances, so that it can be fed the kernel's.
(b) ``pinned_*``: the definition of include/fedfr_b200.h in numpy fp64, with the kernel's summation order (32 lane
    partials over k = l, l + 32, ..., then the xor butterfly), so that its distances are the kernel's bit for bit; then
    the same counts, folds and rates stated on bins."""
import numpy as np
import sklearn.preprocessing
from sklearn.model_selection import KFold

GRID = np.arange(0, 4, 0.01)                                  # evaluate()'s grid for the accuracy


# ---- (a) insightface, verbatim ------------------------------------------------------------------------------------

class LFold:
    def __init__(self, n_splits=2, shuffle=False):
        self.n_splits = n_splits
        if self.n_splits > 1:
            self.k_fold = KFold(n_splits=n_splits, shuffle=shuffle)

    def split(self, indices):
        if self.n_splits > 1:
            return self.k_fold.split(indices)
        else:
            return [(indices, indices)]


def calculate_accuracy(threshold, dist, actual_issame):
    predict_issame = np.less(dist, threshold)
    tp = np.sum(np.logical_and(predict_issame, actual_issame))
    fp = np.sum(np.logical_and(predict_issame, np.logical_not(actual_issame)))
    tn = np.sum(np.logical_and(np.logical_not(predict_issame), np.logical_not(actual_issame)))
    fn = np.sum(np.logical_and(np.logical_not(predict_issame), actual_issame))

    tpr = 0 if (tp + fn == 0) else float(tp) / float(tp + fn)
    fpr = 0 if (fp + tn == 0) else float(fp) / float(fp + tn)
    acc = float(tp + tn) / dist.size
    return tpr, fpr, acc


def roc_from_dist(thresholds, dist, actual_issame, nrof_folds=10):
    """calculate_roc's fold loop (pca = 0) on given distances -> (tpr, fpr, accuracy, best_thresholds)."""
    nrof_pairs = len(actual_issame)
    nrof_thresholds = len(thresholds)
    k_fold = LFold(n_splits=nrof_folds, shuffle=False)

    tprs = np.zeros((nrof_folds, nrof_thresholds))
    fprs = np.zeros((nrof_folds, nrof_thresholds))
    accuracy = np.zeros((nrof_folds))
    best = np.zeros((nrof_folds))
    indices = np.arange(nrof_pairs)

    for fold_idx, (train_set, test_set) in enumerate(k_fold.split(indices)):
        # Find the best threshold for the fold
        acc_train = np.zeros((nrof_thresholds))
        for threshold_idx, threshold in enumerate(thresholds):
            _, _, acc_train[threshold_idx] = calculate_accuracy(threshold, dist[train_set], actual_issame[train_set])
        best_threshold_index = np.argmax(acc_train)
        for threshold_idx, threshold in enumerate(thresholds):
            tprs[fold_idx, threshold_idx], fprs[fold_idx, threshold_idx], _ = calculate_accuracy(
                threshold, dist[test_set], actual_issame[test_set])
        _, _, accuracy[fold_idx] = calculate_accuracy(thresholds[best_threshold_index], dist[test_set],
                                                      actual_issame[test_set])
        best[fold_idx] = thresholds[best_threshold_index]

    tpr = np.mean(tprs, 0)
    fpr = np.mean(fprs, 0)
    return tpr, fpr, accuracy, best


def insightface_embeddings(emb, flip=None):
    """test(): embeddings_list[0] + embeddings_list[1] (or the first alone), sklearn.preprocessing.normalize."""
    embeddings = emb.copy() if flip is None else emb + flip
    return sklearn.preprocessing.normalize(embeddings)


def insightface_dist(embeddings):
    """evaluate() / calculate_roc(): embeddings[0::2] vs [1::2], np.sum(np.square(diff), 1)."""
    embeddings1 = embeddings[0::2]
    embeddings2 = embeddings[1::2]
    diff = np.subtract(embeddings1, embeddings2)
    return np.sum(np.square(diff), 1)


def insightface_kfold(emb, issame, flip=None, nfolds=10, thresholds=GRID):
    """The whole recipe -> (accuracy, best_thresholds, tpr, fpr, dist)."""
    dist = insightface_dist(insightface_embeddings(emb, flip))
    tpr, fpr, acc, best = roc_from_dist(thresholds, dist, np.asarray(issame), nfolds)
    return acc, best, tpr, fpr, dist


# ---- (b) the pinned definition ------------------------------------------------------------------------------------

def lane_sum(sq):
    """fp64 [n, E] -> fp64 [n]: lane l adds k = l, l + 32, ... in order, then s_l + s_(l^o) for o = 16, 8, 4, 2, 1."""
    n, e = sq.shape
    m = -(-e // 32)
    pad = np.zeros((n, m * 32))
    pad[:, :e] = sq
    pad = pad.reshape(n, m, 32)
    s = np.zeros((n, 32))
    for i in range(m):
        s = s + pad[:, i, :]
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        s = s + s[:, lanes ^ o]
    return s[:, 0]


def pinned_dist(emb, flip=None):
    x = np.asarray(emb, np.float32) if flip is None else np.asarray(emb, np.float32) + np.asarray(flip, np.float32)
    x64 = x.astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        nrm = np.sqrt(lane_sum(x64 * x64)).astype(np.float32)
        nrm[nrm == 0] = 1
        xh = x / nrm[:, None]
        d = (xh[0::2] - xh[1::2]).astype(np.float64)
        return lane_sum(d * d).astype(np.float32)


def fold_ranges(n_pairs, nfolds):
    q, r = divmod(n_pairs, nfolds)
    lo = [f * q + min(f, r) for f in range(nfolds)]
    return [(a, a + q + (f < r)) for f, a in enumerate(lo)]


def pinned_bins(dist, thresholds):
    """b = #{j : !(dist < thr_j)}; NaN -> T."""
    d = np.asarray(dist, np.float32).astype(np.float64)
    b = np.searchsorted(thresholds, d, side="right")
    b[np.isnan(d)] = len(thresholds)
    return b


def pinned_from_dist(dist, issame, nfolds, thresholds):
    """Steps 4-7 on counts -> (accuracy, best_thresholds, tpr, fpr)."""
    y = np.asarray(issame) != 0
    T = len(thresholds)
    b = pinned_bins(dist, thresholds)
    cum = lambda sel: np.cumsum(np.bincount(b[sel], minlength=T + 1)[:T])           # noqa: E731  pairs with bin <= j
    all_g, all_i = cum(y), cum(~y)
    acc, best, rt, rf = [], [], [], []
    for lo, hi in fold_ranges(len(y), nfolds):
        te = np.zeros(len(y), bool)
        te[lo:hi] = True
        tp, fp = cum(te & y), cum(te & ~y)
        n_g, n_i = int((te & y).sum()), int((te & ~y).sum())
        tn = n_i - fp
        if nfolds == 1:
            train = tp + tn
        else:
            train = (all_g - tp) + ((int((~y).sum()) - n_i) - (all_i - fp))
        j = int(np.argmax(train))
        acc.append(float(tp[j] + tn[j]) / (hi - lo))
        best.append(thresholds[j])
        rt.append(tp / n_g if n_g else np.zeros(T))
        rf.append(fp / n_i if n_i else np.zeros(T))
    st, sf = np.zeros(T), np.zeros(T)
    for f in range(nfolds):
        st, sf = st + rt[f], sf + rf[f]
    return np.array(acc), np.array(best), st / nfolds, sf / nfolds
