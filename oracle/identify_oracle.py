"""1:N identification restated on the CPU  --  TEST INFRASTRUCTURE ONLY, like everything under oracle/.

``identify`` and ``score_matrix`` are the ctypes face of ``oracle_identify`` / ``oracle_score_matrix`` in
``oracle/oracle_identify.c`` (a literal loop over the definition of ``csrc/identify.cu``'s ``pfc_identify``), compiled with
gcc ``-ffp-contract=off`` on first use into a temporary directory, so the source tree is never written.
``argsort_ranks`` is the independent numpy check of ``identify``: the mate's position and element 0 of
``np.argsort(-S, axis=1, kind="stable")``.  ``ijbc_1n_like`` generates seeded data of the IJB-C 1:N shape.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_identify.c")
_FLAGS = ["-O2", "-fPIC", "-shared", "-ffp-contract=off"]
_lib_cache = None


def _lib():
    global _lib_cache
    if _lib_cache is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src + " ".join(_FLAGS).encode()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "fedfr_oracle_identify_%s_%d.so" % (tag, os.getuid()))
        if not os.path.exists(so):
            tmp = "%s.tmp.%d" % (so, os.getpid())
            subprocess.check_call(["gcc"] + _FLAGS + [_SRC, "-lm", "-o", tmp])
            os.replace(tmp, so)                                  # concurrent builders: the last rename wins, same bytes
        lib = C.CDLL(so)
        lib.oracle_score_matrix.restype = None
        lib.oracle_score_matrix.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
        lib.oracle_identify.restype = None
        lib.oracle_identify.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int] + [C.c_void_p] * 6
        _lib_cache = lib
    return _lib_cache


def score_matrix(probe, gallery):
    """-> S fp32 [P, G], every (probe, gallery) score by the oracle_pair_scores chain."""
    a = np.ascontiguousarray(probe, dtype=np.float32)
    b = np.ascontiguousarray(gallery, dtype=np.float32)
    out = np.empty((a.shape[0], b.shape[0]), dtype=np.float32)
    _lib().oracle_score_matrix(a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], a.shape[1], out.ctypes.data)
    return out


def identify(probe, gallery, mate_row):
    """The 1:N definition of include/fedfr_b200.h, looped literally.  -> (rank int64 [P], mate_score fp32 [P],
    top1_row int64 [P], top1_score fp32 [P], counts int64 [2] = {NaN scores, mate rows outside [-1, G)})."""
    a = np.ascontiguousarray(probe, dtype=np.float32)
    b = np.ascontiguousarray(gallery, dtype=np.float32)
    m = np.ascontiguousarray(mate_row, dtype=np.int64)
    P = a.shape[0]
    rank, top1_row, counts = np.empty(P, np.int64), np.empty(P, np.int64), np.empty(2, np.int64)
    mate_score, top1_score = np.empty(P, np.float32), np.empty(P, np.float32)
    _lib().oracle_identify(a.ctypes.data, P, b.ctypes.data, b.shape[0], a.shape[1], m.ctypes.data, rank.ctypes.data,
                           mate_score.ctypes.data, top1_row.ctypes.data, top1_score.ctypes.data, counts.ctypes.data)
    return rank, mate_score, top1_row, top1_score, counts


def argsort_ranks(S, mate_row):
    """The mate's 1-based position in np.argsort(-S_p, kind="stable") (0 without a mate) and element 0 of that order.
    -> (rank int64 [P], top1_row int64 [P])."""
    order = np.argsort(-np.asarray(S, dtype=np.float32), axis=1, kind="stable")
    mate_row = np.asarray(mate_row, dtype=np.int64)
    rank = np.zeros(order.shape[0], np.int64)
    mated = np.flatnonzero(mate_row >= 0)
    rank[mated] = np.argmax(order[mated] == mate_row[mated, None], axis=1) + 1
    return rank, order[:, 0].astype(np.int64)


IJBC_1N_SHAPE = dict(probes=19_593, g1=1_772, g2=1_759)


def ijbc_1n_like(seed=0, emb=512, probes=IJBC_1N_SHAPE["probes"], g1=IJBC_1N_SHAPE["g1"], g2=IJBC_1N_SHAPE["g2"]):
    """Seeded synthetic data of the IJB-C 1:N shape: two galleries of one L2-normalised template per subject (the G1
    and G2 subjects are disjoint) and probe templates of subjects drawn from both, so each probe is mated in one
    gallery and non-mated in the other.  Subject ids are sparse int64.
    -> probe_feats fp32 [P, E], probe_subjects int64 [P], (g1_feats, g1_subjects), (g2_feats, g2_subjects)."""
    rng = np.random.default_rng(seed)
    n_subj = g1 + g2
    ids = rng.choice(2 ** 40, n_subj, replace=False).astype(np.int64) - 2 ** 39
    centres = rng.standard_normal((n_subj, emb), dtype=np.float32)

    def unit(x):
        return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)

    gallery = unit(centres + 0.8 * rng.standard_normal((n_subj, emb), dtype=np.float32))
    subj = rng.integers(0, n_subj, probes)
    probe = unit(centres[subj] + 4.0 * rng.standard_normal((probes, emb), dtype=np.float32))   # rank-1 about 0.8
    return probe, ids[subj], (gallery[:g1], ids[:g1]), (gallery[g1:], ids[g1:])
