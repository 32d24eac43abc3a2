"""1:1 template verification restated on the CPU  --  TEST INFRASTRUCTURE ONLY, like everything under oracle/.

``template_pool`` and ``pair_scores`` are the ctypes face of ``oracle_template_pool`` / ``oracle_pair_scores`` in
``oracle/oracle_verify.c`` (the bit-exact restatement of ``csrc/verify.cu``), compiled with gcc ``-ffp-contract=off`` on
first use into a temporary directory, so the source tree is never written.  ``recipe_float64`` is the insightface IJB 1:1
recipe in float64 numpy (media mean, template sum, L2 normalise, cosine), the independent check of that arithmetic at a
tolerance.  ``tar_at_far`` is the definition of ``fedfr_b200.verify.tar_at_far`` as a numpy sort.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_verify.c")
_FLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off"]
_lib_cache = None


def _lib():
    global _lib_cache
    if _lib_cache is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src + " ".join(_FLAGS).encode()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "fedfr_oracle_verify_%s_%d.so" % (tag, os.getuid()))
        if not os.path.exists(so):
            tmp = "%s.tmp.%d" % (so, os.getpid())
            subprocess.check_call(["gcc"] + _FLAGS + [_SRC, "-lm", "-o", tmp])
            os.replace(tmp, so)                                  # concurrent builders: the last rename wins, same bytes
        lib = C.CDLL(so)
        lib.oracle_template_pool.restype = C.c_int64
        lib.oracle_template_pool.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
        lib.oracle_pair_scores.restype = C.c_int
        lib.oracle_pair_scores.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        _lib_cache = lib
    return _lib_cache


def template_pool(feats, templates, medias, weights=None):
    """-> (template_feats fp32 [T, E], template_ids int64 [T] ascending)."""
    feats = np.ascontiguousarray(feats, dtype=np.float32)
    templates = np.ascontiguousarray(templates, dtype=np.int64)
    medias = np.ascontiguousarray(medias, dtype=np.int64)
    w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float32)
    n, emb = feats.shape
    out = np.empty((max(n, 1), emb), dtype=np.float32)
    ids = np.empty(max(n, 1), dtype=np.int64)
    t = _lib().oracle_template_pool(feats.ctypes.data, templates.ctypes.data, medias.ctypes.data,
                                    None if w is None else w.ctypes.data, n, emb, out.ctypes.data, ids.ctypes.data)
    return out[:t].copy(), ids[:t].copy()


def pair_scores(template_feats, row1, row2):
    tf = np.ascontiguousarray(template_feats, dtype=np.float32)
    r1 = np.ascontiguousarray(row1, dtype=np.int64)
    r2 = np.ascontiguousarray(row2, dtype=np.int64)
    out = np.empty(r1.shape[0], dtype=np.float32)
    rc = _lib().oracle_pair_scores(tf.ctypes.data, tf.shape[0], tf.shape[1], r1.ctypes.data, r2.ctypes.data, r1.shape[0],
                                   out.ctypes.data)
    if rc != 0:
        raise ValueError("row index out of range")
    return out


def recipe_float64(feats, templates, medias, weights=None):
    """-> (template_feats float64 [T, E], ids): single-image medias as they are, other medias averaged, templates summed,
    then L2-normalised."""
    x = np.asarray(feats, dtype=np.float64)
    if weights is not None:
        x = x * np.asarray(weights, dtype=np.float64)[:, None]
    ids = np.unique(templates)
    out = np.zeros((ids.size, x.shape[1]))
    for r, t in enumerate(ids):
        sel = templates == t
        for m in np.unique(medias[sel]):
            out[r] += x[sel & (medias == m)].mean(axis=0)
    return out / np.maximum(np.linalg.norm(out, axis=1, keepdims=True), 1e-12), ids


def tar_at_far(scores, issame, fars):
    """[(far_target, tar, far, threshold)]: threshold = (k+1)-th largest impostor score, k = floor(f * n_imp), -inf when
    k >= n_imp; accepted iff score > threshold."""
    scores = np.asarray(scores, dtype=np.float32)
    issame = np.asarray(issame, dtype=bool)
    gen, imp = scores[issame], scores[~issame]
    desc = np.sort(imp)[::-1]
    out = []
    for f in fars:
        k = int(np.floor(float(f) * imp.size))
        tau = np.float32(desc[k]) if k < imp.size else np.float32(-np.inf)
        out.append((float(f), int((gen > tau).sum()) / gen.size, int((imp > tau).sum()) / imp.size, float(tau)))
    return out


IJBC_SHAPE = dict(images=227_630, templates=23_124, pairs=15_658_489, genuine=19_557)


def ijbc_like(seed=0, emb=512, images=IJBC_SHAPE["images"], templates=IJBC_SHAPE["templates"], pairs=IJBC_SHAPE["pairs"],
              genuine=IJBC_SHAPE["genuine"]):
    """Seeded synthetic data of the IJB-C 1:1 shape: every template has images (about 10 on average, in 1-4 medias of a
    few images), four templates per subject, sparse int64 template ids, and a pair list grouped by p1 with `genuine`
    same-subject pairs.  -> feats fp32 [n, E], templates, medias int64 [n], p1, p2 int64 [P], issame bool [P]."""
    rng = np.random.default_rng(seed)
    ids = np.sort(rng.choice(2 ** 40, templates, replace=False)).astype(np.int64) - 2 ** 39
    t_idx = np.concatenate([np.arange(templates), rng.integers(0, templates, images - templates)])
    rng.shuffle(t_idx)
    medias = t_idx * 4 + rng.integers(0, 4, images)
    subject = t_idx // 4
    centres = rng.standard_normal((templates // 4 + 1, emb), dtype=np.float32)
    feats = centres[subject]
    feats += 1.6 * rng.standard_normal((images, emb), dtype=np.float32)
    a = rng.integers(0, templates // 4, genuine) * 4
    off = rng.integers(0, 6, genuine)                                    # one of the 6 pairs of a subject's 4 templates
    first = np.array([0, 0, 0, 1, 1, 2])[off]
    second = np.array([1, 2, 3, 2, 3, 3])[off]
    g1, g2 = a + first, a + second
    i1 = rng.integers(0, templates, pairs - genuine)
    i2 = rng.integers(0, templates, pairs - genuine)
    same = i1 // 4 == i2 // 4
    i2[same] = (i2[same] + 4) % templates
    r1, r2 = np.concatenate([g1, i1]), np.concatenate([g2, i2])
    order = np.argsort(r1, kind="stable")                                # grouped by p1
    r1, r2 = r1[order], r2[order]
    return feats, ids[t_idx], medias, ids[r1], ids[r2], (r1 // 4) == (r2 // 4)
