"""1:1 template verification on the sm_100a kernels -- the IJB-B / IJB-C protocol of FedFR's ``ijbc_all.py`` /
``ijbc_conti.py``, on arrays: image features with template and media ids, a template pair list, genuine flags.

    template_feats, template_ids = template_features(feats, templates, medias, weights)
    scores = pair_scores(template_feats, template_ids, p1, p2)
    for far_target, tar, far, threshold in tar_at_far(scores, issame): ...
    fpr, tpr, thresholds = roc_curve(scores, issame)            # sklearn.metrics.roc_curve, element for element
    for far_target, tar, far in tar_at_far_nearest(fpr, tpr): ...   # the insightface IJB scripts' TAR table
    acc, best_thr, tpr, fpr = kfold_accuracy(emb, issame, flipped)  # the per-round LFW / CFP-FP / AgeDB K-fold test
    rank, mate_score, top1_row, top1_score = mate_ranks(probe_feats, probe_subjects, gallery_feats, gallery_subjects)
    cmc(rank, max_rank=20)                                          # 1:N identification: rank-1 ... rank-20 rates
    for fpir_target, tpir, fpir, threshold in tpir_at_fpir(rank, mate_score, top1_score): ...

The arithmetic is this repository's definition, pinned step by step (``include/fedfr_b200.h``, ``csrc/verify.cu``,
``csrc/identify.cu``) so that a plain C restatement reproduces every feature and score bit for bit; it follows the usual insightface recipe (media
mean, template sum, L2 normalise, cosine).  Inputs are CUDA tensors or numpy arrays; nothing runs on the CPU except
index plumbing on the device (sorting ids into a CSR, id -> row lookup) and the final division of two counts.
"""
import numpy as np
import torch

from . import _native as N

DEFAULT_FARS = (1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1)
_MAX_FARS_PER_CALL = 8


def _device(t):
    if isinstance(t, torch.Tensor) and t.is_cuda:
        return t.device
    return torch.device("cuda", torch.cuda.current_device())


def _on(t, dtype, device):
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t))
    return torch.as_tensor(t).to(device=device, dtype=dtype).contiguous()


def _stream(device):
    return torch.cuda.current_stream(device).cuda_stream


def pool_index(templates, medias):
    """CSR of the images in ascending (template, media, row) order, from int64 id tensors on any device:
    -> (template_ids [T], order [n], media_start [n_media + 1], tmpl_start [T + 1])."""
    template_ids, t_inv = torch.unique(templates, return_inverse=True)
    media_ids, m_inv = torch.unique(medias, return_inverse=True)
    key = t_inv * media_ids.numel() + m_inv
    key_sorted, order = torch.sort(key, stable=True)
    _, counts = torch.unique_consecutive(key_sorted, return_counts=True)
    media_start = torch.cat([counts.new_zeros(1), counts.cumsum(0)])
    media_tmpl = key_sorted[media_start[:-1]] // media_ids.numel()
    tmpl_start = torch.searchsorted(media_tmpl, torch.arange(template_ids.numel() + 1, device=key.device))
    return template_ids, order, media_start, tmpl_start


def template_features(feats, templates, medias, weights=None):
    """Pool image features into L2-normalised template features.

    feats fp32 [n, E]; templates, medias int64 [n] (arbitrary ids; a media is a (template, media) pair, so one media id
    may occur in several templates); weights fp32 [n] or None (a per-image scale such as a detector score).  Each media
    is the mean of its images, each template the sum of its medias (ascending media id), then normalised.
    -> (template_feats fp32 [T, E], template_ids int64 [T], sorted unique), on the GPU."""
    device = _device(feats)
    f = _on(feats, torch.float32, device)
    t = _on(templates, torch.int64, device).reshape(-1)
    m = _on(medias, torch.int64, device).reshape(-1)
    w = None if weights is None else _on(weights, torch.float32, device).reshape(-1)
    if f.dim() != 2 or f.shape[0] == 0 or f.shape[1] == 0:
        raise ValueError("feats must be a non-empty [n, E] array")
    n, emb = f.shape
    if t.numel() != n or m.numel() != n or (w is not None and w.numel() != n):
        raise ValueError("templates, medias and weights need one entry per image row")
    template_ids, order, media_start, tmpl_start = pool_index(t, m)
    out = torch.empty(template_ids.numel(), emb, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        N.check(N.lib.pfc_template_pool(N.ptr(f), N.ptr(w), N.ptr(order), N.ptr(media_start), N.ptr(tmpl_start),
                                        template_ids.numel(), emb, N.ptr(out), _stream(device)), "pfc_template_pool")
    return out, template_ids


def pair_rows(template_ids, p1, p2):
    """Template ids -> rows of ``template_ids`` (sorted unique), by binary search on the ids' device.  ValueError for an
    id that is not there."""
    if template_ids.numel() == 0 or bool((template_ids[1:] <= template_ids[:-1]).any()):
        raise ValueError("template_ids must be non-empty, sorted and unique (as template_features returns them)")
    rows = []
    for p in (p1, p2):
        r = torch.searchsorted(template_ids, p).clamp_(max=template_ids.numel() - 1)
        missing = template_ids[r] != p
        if bool(missing.any()):
            raise ValueError("unknown template id %d in the pair list" % int(p[missing.nonzero()[0, 0]]))
        rows.append(r)
    return rows


def pair_scores(template_feats, template_ids, p1, p2):
    """Cosine of each template pair: ``sum_k (double)fl32(a_k * b_k)`` over ascending k, rounded to fp32 (the chain of
    the ROC histogram).  template_feats fp32 [T, E] and template_ids int64 [T] as template_features returns them;
    p1, p2 int64 [P] template ids.  Pair lists grouped by p1 (as IJB-C's is) read each p1 row once per 128 pairs.
    -> scores fp32 [P] on the GPU."""
    device = _device(template_feats)
    tf = _on(template_feats, torch.float32, device)
    ids = _on(template_ids, torch.int64, device).reshape(-1)
    a = _on(p1, torch.int64, device).reshape(-1)
    b = _on(p2, torch.int64, device).reshape(-1)
    if tf.dim() != 2 or tf.shape[0] != ids.numel():
        raise ValueError("template_feats [T, E] needs one id per row")
    if a.numel() != b.numel():
        raise ValueError("p1 and p2 must have the same length")
    out = torch.empty(a.numel(), dtype=torch.float32, device=device)
    if a.numel() == 0:
        return out
    r1, r2 = pair_rows(ids, a, b)
    with torch.cuda.device(device):
        N.check(N.lib.pfc_pair_scores(N.ptr(tf), tf.shape[0], tf.shape[1], N.ptr(r1), N.ptr(r2), a.numel(), N.ptr(out),
                                      _stream(device)), "pfc_pair_scores")
    return out


def tar_from_counts(counts, thresholds, fars):
    """(counts [3 + 2 n_far] of pfc_tar_at_far, thresholds [n_far]) -> [(far_target, tar, far, threshold)]."""
    counts = [int(c) for c in counts]
    n_gen, n_imp, n_nan = counts[:3]
    if n_nan:
        raise ValueError("%d scores are NaN" % n_nan)
    if n_gen == 0 or n_imp == 0:
        raise ValueError("tar_at_far needs genuine and impostor pairs (got %d and %d)" % (n_gen, n_imp))
    return [(float(f), counts[3 + 2 * q] / n_gen, counts[4 + 2 * q] / n_imp, float(thresholds[q])) for q, f in enumerate(fars)]


def tar_at_far(scores, issame, fars=DEFAULT_FARS):
    """Exact TAR at each target FAR from the full score distribution (no sort, no binning).

    With n_imp impostor pairs and k = floor(f * n_imp), the threshold is the (k+1)-th largest impostor score (-inf when
    k >= n_imp) and a pair is accepted iff its score is above it, so ties at the threshold are rejected and the achieved
    far = accepted impostors / n_imp is at most f: the best operating point with FAR <= f.  -0.0 and +0.0 are one
    value.  The sklearn-based IJB scripts instead read the nearest point of a thinned ROC curve: that read-out is
    ``tar_at_far_nearest(*roc_curve(scores, issame)[:2])``.  scores fp32 [P], issame bool [P]; fars in (0, 1].  A NaN
    score, or no genuine or no impostor pair, raises ValueError.  -> [(far_target, tar, far, threshold)]."""
    device = _device(scores)
    s = _on(scores, torch.float32, device).reshape(-1)
    y = (_on(issame, torch.int64, device).reshape(-1) != 0).to(torch.uint8)
    fars = [float(f) for f in fars]
    if s.numel() != y.numel():
        raise ValueError("one issame flag per score")
    if s.numel() == 0:
        raise ValueError("tar_at_far needs genuine and impostor pairs (got no scores)")
    if not fars or not all(0.0 < f <= 1.0 for f in fars):
        raise ValueError("FARs must lie in (0, 1]")
    ws = torch.empty(int(N.lib.pfc_tar_at_far_workspace_bytes(s.numel())), dtype=torch.uint8, device=device)
    result = []
    for c0 in range(0, len(fars), _MAX_FARS_PER_CALL):
        chunk = fars[c0:c0 + _MAX_FARS_PER_CALL]
        f_host = np.asarray(chunk, dtype=np.float64)
        counts = torch.empty(3 + 2 * len(chunk), dtype=torch.int64, device=device)
        thr = torch.empty(len(chunk), dtype=torch.float32, device=device)
        with torch.cuda.device(device):
            N.check(N.lib.pfc_tar_at_far(N.ptr(s), N.ptr(y), s.numel(), f_host.ctypes.data, len(chunk), N.ptr(counts),
                                         N.ptr(thr), N.ptr(ws), ws.numel(), _stream(device)), "pfc_tar_at_far")
        result += tar_from_counts(counts.cpu().tolist(), thr.cpu().tolist(), chunk)
    return result


def _numel(t):
    return t.numel() if isinstance(t, torch.Tensor) else np.asarray(t).size


def curve_length(counts, n_points):
    """(counts [3] of pfc_roc_curve, n_points) -> n_points, or ValueError for NaN / inf scores or a missing class."""
    n_gen, n_imp, n_nonfinite = (int(c) for c in counts)
    if n_nonfinite:
        raise ValueError("%d scores are NaN or infinite" % n_nonfinite)
    if n_gen == 0 or n_imp == 0:
        raise ValueError("roc_curve needs genuine and impostor pairs (got %d and %d)" % (n_gen, n_imp))
    return int(n_points)


def roc_curve(scores, issame):
    """The ROC curve of the scores, equal element for element to ``sklearn.metrics.roc_curve(issame, scores)`` (with
    its default ``drop_intermediate=True``), computed on the GPU by a radix sort of the scores and integer scans.

    -0.0 and +0.0 are one value.  sklearn raises for NaN or infinite scores, and so does this.  Where sklearn only warns
    and returns NaN rates (no genuine or no impostor pair), this raises ValueError.  The definition on counts is in
    ``include/fedfr_b200.h``.  ``sklearn.metrics.auc(fpr, tpr)`` on the result gives the IJB scripts' AUC, and
    ``tar_at_far_nearest(fpr, tpr)`` their TAR table.  scores fp32 [P], issame bool [P], CUDA tensors or numpy arrays.
    -> (fpr, tpr, thresholds), float64 CUDA tensors of the curve's length; thresholds[0] = +inf."""
    if _numel(scores) != _numel(issame):
        raise ValueError("one issame flag per score")
    if _numel(scores) == 0:
        raise ValueError("roc_curve needs genuine and impostor pairs (got no scores)")
    device = _device(scores)
    s = _on(scores, torch.float32, device).reshape(-1)
    y = (_on(issame, torch.int64, device).reshape(-1) != 0).to(torch.uint8)
    n = s.numel()
    ws = torch.empty(int(N.lib.pfc_roc_curve_workspace_bytes(n)), dtype=torch.uint8, device=device)
    fpr, tpr, thr = (torch.empty(n + 1, dtype=torch.float64, device=device) for _ in range(3))
    out = torch.empty(4, dtype=torch.int64, device=device)                  # counts [3], n_points
    with torch.cuda.device(device):
        N.check(N.lib.pfc_roc_curve(N.ptr(s), N.ptr(y), n, N.ptr(fpr), N.ptr(tpr), N.ptr(thr), N.ptr(out[3:]), N.ptr(out),
                                    N.ptr(ws), ws.numel(), _stream(device)), "pfc_roc_curve")
    host = out.cpu().tolist()
    k = curve_length(host[:3], host[3])
    return fpr[:k].clone(), tpr[:k].clone(), thr[:k].clone()


def tar_at_far_nearest(fpr, tpr, fars=DEFAULT_FARS):
    """TAR at each target FAR as the insightface IJB-B / IJB-C scripts print it (FedFR's ``ijbc_all.py`` and
    ``ijbc_conti.py``): on the curve flipped end to end (largest tpr first at an equal fpr), the point whose fpr is
    nearest to f, the first one on a tie.  Its FAR may lie above f; ``tar_at_far`` stays the exact FAR <= f operating
    point.  fpr, tpr as ``roc_curve`` returns them (or sklearn's), tensors or numpy arrays; the lookup runs on the host.
    -> [(far_target, tar, far_at_point)]."""
    f = np.flipud(np.asarray(torch.as_tensor(fpr).cpu(), dtype=np.float64))
    t = np.flipud(np.asarray(torch.as_tensor(tpr).cpu(), dtype=np.float64))
    if f.size == 0 or f.shape != t.shape:
        raise ValueError("fpr and tpr must be non-empty and of one length")
    out = []
    for far in fars:
        i = int(np.argmin(np.abs(f - float(far))))
        out.append((float(far), float(t[i]), float(f[i])))
    return out


def kfold_thresholds(thresholds=None):
    """The threshold grid as a validated float64 numpy array: ``np.arange(0, 4, 0.01)`` (insightface's ``evaluate``)
    when None.  ValueError unless it is 1-D, non-empty, finite and strictly ascending.  A CUDA tensor is copied to the
    host to be checked, which waits for the device."""
    if thresholds is None:
        return np.arange(0, 4, 0.01)
    if isinstance(thresholds, torch.Tensor):
        thresholds = thresholds.detach().cpu().numpy()
    t = np.asarray(thresholds, dtype=np.float64)
    if t.ndim != 1 or t.size == 0:
        raise ValueError("thresholds must be a non-empty 1-D array")
    if not np.isfinite(t).all():
        raise ValueError("thresholds must be finite")
    if not (t[1:] > t[:-1]).all():
        raise ValueError("thresholds must be strictly ascending")
    return np.ascontiguousarray(t)


def kfold_accuracy(embeddings, issame, flipped=None, nfolds=10, thresholds=None):
    """The K-fold verification accuracy of the per-round LFW / CFP-FP / AgeDB test (insightface's
    ``eval/verification.py``: ``test()``'s flip fusion and normalisation, then ``evaluate`` / ``calculate_roc``), exact
    on integer counts.

    embeddings fp32 [2P, E] (rows 2p and 2p+1 are pair p); flipped fp32 [2P, E] (the embeddings of the flipped images,
    added to ``embeddings`` before normalising) or None; issame bool [P]; folds are sklearn's ``KFold(nfolds)`` without
    shuffling (nfolds = 1: train = test = all pairs); thresholds float64 [T], strictly ascending, default
    ``np.arange(0, 4, 0.01)``.  CUDA tensors or numpy arrays.  A pair is predicted "same" at threshold t iff its squared
    distance is < t.  The definition, with its pinned fp64 sums, is in ``include/fedfr_b200.h``: on the same distances,
    every output equals the numpy recipe's element for element.  Nothing is copied back to the host, so the call does not
    wait for the device (unless ``thresholds`` is a CUDA tensor, which is checked on the host).

    -> (accuracy [nfolds], best_thresholds [nfolds], tpr [T], fpr [T]), float64 CUDA tensors.  ``test()``'s
    ``acc2, std2`` are ``accuracy.mean(), accuracy.std(correction=0)`` (np.std's ddof=0; torch's default is 1)."""
    shape = tuple(embeddings.shape) if isinstance(embeddings, torch.Tensor) else np.shape(embeddings)
    if len(shape) != 2 or shape[0] % 2 or shape[1] == 0:
        raise ValueError("embeddings must be [2P, E]: an even number of rows, pair p in rows 2p and 2p+1")
    if flipped is not None and (tuple(flipped.shape) if isinstance(flipped, torch.Tensor) else np.shape(flipped)) != shape:
        raise ValueError("flipped must have the shape of embeddings")
    n_pairs = shape[0] // 2
    if _numel(issame) != n_pairs:
        raise ValueError("one issame flag per pair (%d pairs, got %d flags)" % (n_pairs, _numel(issame)))
    nfolds = int(nfolds)
    if not 1 <= nfolds <= n_pairs:
        raise ValueError("nfolds must lie in [1, %d] (the number of pairs), got %d" % (n_pairs, nfolds))
    thr_host = kfold_thresholds(thresholds)
    device = _device(embeddings)
    e = _on(embeddings, torch.float32, device)
    fl = None if flipped is None else _on(flipped, torch.float32, device)
    y = (_on(issame, torch.int64, device).reshape(-1) != 0).to(torch.uint8)
    thr = torch.from_numpy(thr_host).pin_memory().to(device, non_blocking=True)
    n_thr = thr.numel()
    ws = torch.empty(int(N.lib.pfc_kfold_workspace_bytes(n_pairs, n_thr, nfolds)), dtype=torch.uint8, device=device)
    dist = torch.empty(n_pairs, dtype=torch.float32, device=device)
    acc, best = (torch.empty(nfolds, dtype=torch.float64, device=device) for _ in range(2))
    tpr, fpr = (torch.empty(n_thr, dtype=torch.float64, device=device) for _ in range(2))
    with torch.cuda.device(device):
        N.check(N.lib.pfc_kfold_accuracy(N.ptr(e), N.ptr(fl), N.ptr(y), n_pairs, e.shape[1], N.ptr(thr), n_thr, nfolds,
                                         N.ptr(dist), N.ptr(acc), N.ptr(best), N.ptr(tpr), N.ptr(fpr), N.ptr(ws),
                                         ws.numel(), _stream(device)), "pfc_kfold_accuracy")
    return acc, best, tpr, fpr


def mate_rows(probe_subjects, gallery_subjects):
    """Gallery row of each probe's subject, -1 when the subject is not in the gallery, by a sort and a binary search on
    the device.  ValueError when a subject occurs twice in the gallery (1:N here takes one entry per subject)."""
    g_sorted, g_order = torch.sort(gallery_subjects)
    if bool((g_sorted[1:] == g_sorted[:-1]).any()):
        dup = int(g_sorted[1:][g_sorted[1:] == g_sorted[:-1]][0])
        raise ValueError("gallery subject %d occurs more than once: the gallery needs one entry per subject" % dup)
    r = torch.searchsorted(g_sorted, probe_subjects).clamp_(max=g_sorted.numel() - 1)
    return torch.where(g_sorted[r] == probe_subjects, g_order[r], torch.full_like(r, -1))


def mate_ranks(probe_feats, probe_subjects, gallery_feats, gallery_subjects):
    """1:N identification (the IJB-B / IJB-C search protocol): for every probe, the rank of its mate in the gallery and
    the gallery's top-1 match, exact, without a [P, G] score matrix.

    probe_feats fp32 [P, E], gallery_feats fp32 [G, E] (used as given: normally ``template_features`` output);
    probe_subjects int64 [P], gallery_subjects int64 [G] (one gallery entry per subject); CUDA tensors or numpy arrays.
    A probe is mated when its subject is in the gallery.  Every score is the ``pair_scores`` chain, so it equals
    ``pair_scores`` on the same two rows bit for bit.  rank = the mate's 1-based position in
    ``np.argsort(-scores, kind="stable")`` (gallery order breaks ties; -0.0 == +0.0), 0 for a non-mated probe;
    mate_score = its score (NaN when non-mated); top1_row / top1_score = the first gallery row with the largest score
    and that score.  The definition is in ``include/fedfr_b200.h``.  Raises ValueError for duplicate gallery subjects
    and for NaN scores (the check reads two counts back, which waits for the device).

    IJB-C, once per gallery (G1, G2), with subjects from the protocol's template -> subject table::

        feats_t, ids_t = template_features(img_feats, templates, medias, faceness)
        probe_rows = torch.searchsorted(ids_t, probe_template_ids)     # the G1 / G2 template ids likewise
        rank, mate_score, top1_row, top1_score = mate_ranks(feats_t[probe_rows], probe_subjects,
                                                            feats_t[g1_rows], g1_subjects)
        rank1 = cmc(rank, 1)[0]; tpir_fpir = tpir_at_fpir(rank, mate_score, top1_score)

    -> (rank int64 [P], mate_score fp32 [P], top1_row int64 [P], top1_score fp32 [P]), CUDA tensors."""
    device = _device(probe_feats)
    x = _on(probe_feats, torch.float32, device)
    y = _on(gallery_feats, torch.float32, device)
    ps = _on(probe_subjects, torch.int64, device).reshape(-1)
    gs = _on(gallery_subjects, torch.int64, device).reshape(-1)
    if x.dim() != 2 or y.dim() != 2 or x.shape[0] == 0 or y.shape[0] == 0 or x.shape[1] == 0 or x.shape[1] != y.shape[1]:
        raise ValueError("probe_feats [P, E] and gallery_feats [G, E] must be non-empty with one E")
    if ps.numel() != x.shape[0] or gs.numel() != y.shape[0]:
        raise ValueError("one subject per probe row and per gallery row")
    m = mate_rows(ps, gs)
    P = x.shape[0]
    rank, top1_row, counts = (torch.empty(n, dtype=torch.int64, device=device) for n in (P, P, 2))
    mate_score, top1_score = (torch.empty(P, dtype=torch.float32, device=device) for _ in range(2))
    ws = torch.empty(int(N.lib.pfc_identify_workspace_bytes(P)), dtype=torch.uint8, device=device)
    with torch.cuda.device(device):
        N.check(N.lib.pfc_identify(N.ptr(x), P, N.ptr(y), y.shape[0], x.shape[1], N.ptr(m), N.ptr(rank),
                                   N.ptr(mate_score), N.ptr(top1_row), N.ptr(top1_score), N.ptr(counts), N.ptr(ws),
                                   ws.numel(), _stream(device)), "pfc_identify")
    n_nan = int(counts[0])
    if n_nan:
        raise ValueError("%d probe-gallery scores are NaN" % n_nan)
    return rank, mate_score, top1_row, top1_score


def cmc(rank, max_rank=20):
    """Cumulative match characteristic from ``mate_ranks``' ranks: cmc[r-1] = #{mated probes with rank <= r} / n_mated
    for r = 1 ... max_rank (non-mated probes, rank 0, are left out).  ValueError without a mated probe.
    -> float64 [max_rank] on the ranks' device."""
    r = torch.as_tensor(rank).reshape(-1)
    max_rank = int(max_rank)
    if max_rank < 1:
        raise ValueError("max_rank must be >= 1")
    mated = r > 0
    n_mated = int(mated.sum())
    if n_mated == 0:
        raise ValueError("cmc needs mated probes (got none)")
    hits = torch.bincount(torch.where(mated, r.clamp(max=max_rank + 1), 0), minlength=max_rank + 2)[1:max_rank + 1]
    hits = hits.cumsum(0).to(torch.float64)
    return hits / torch.full_like(hits, n_mated)        # an IEEE division each (CUDA divides by a scalar as a product)


def tpir_at_fpir(rank, mate_score, top1_score, fpirs=(1e-2, 1e-1), max_rank=1):
    """TPIR at each target FPIR, at rank ``max_rank``, from ``mate_ranks``' outputs.  A non-mated probe's score is its
    top-1 score; a mated probe's is its mate's score when rank <= max_rank, else -inf.  The result is exactly
    ``tar_at_far`` of those scores with mated = genuine: the threshold is the (k+1)-th largest non-mated top-1 score,
    k = floor(f * n_nonmated), and a mated probe counts iff its mate is within rank ``max_rank`` and scores above it.
    ValueError without a mated or without a non-mated probe.  -> [(fpir_target, tpir, fpir, threshold)]."""
    r = torch.as_tensor(rank).reshape(-1)
    if int(max_rank) < 1:
        raise ValueError("max_rank must be >= 1")
    if not r.numel() == _numel(mate_score) == _numel(top1_score):
        raise ValueError("rank, mate_score and top1_score need one entry per probe")
    n_mated = int((r > 0).sum())
    if n_mated == 0 or n_mated == r.numel():
        raise ValueError("tpir_at_fpir needs mated and non-mated probes (got %d and %d)" % (n_mated, r.numel() - n_mated))
    device = r.device if r.is_cuda else _device(mate_score)
    r = r.to(device)
    ms = _on(mate_score, torch.float32, device).reshape(-1)
    ts = _on(top1_score, torch.float32, device).reshape(-1)
    mated = r > 0
    s = torch.where(mated, torch.where(r <= int(max_rank), ms, torch.full_like(ms, float("-inf"))), ts)
    return tar_at_far(s, mated, fpirs)
