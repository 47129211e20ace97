"""float64 numpy restatement of filtered relation ranking and top-k relations of a node pair for the DistMult decoder.

Semantics as in ``gripnet_b200/ranking.py`` (pinned here independently of it).  Relation queries ``(s, ?, t)``: every
relation ``r'`` is a candidate with pre-sigmoid score ``S(r') = sum_k z[s,k] z[t,k] w[r',k]``; a filter is a set of
directed triples ``(s, r', t)`` (duplicates count once); the rank of ``(s, r, t)`` is the OGB rule
``1 + (opt + pess) / 2`` over ``N = {r' != r : (s, r', t) not in filter}``; top-k by descending score, ties by smaller
relation id, padded with id -1 / NaN (``k`` may exceed ``R``).  Per-relation MRR / Hits@k: ``ranking.rank_metrics``.
"""
import numpy as np


def relation_scores(z, w, src, dst):
    """float64 ``[Q, R]``: the score of every relation of every pair ``(src[i], dst[i])``."""
    z = np.asarray(z, dtype=np.float64)
    w = np.asarray(w, dtype=np.float64)
    p = z[np.asarray(src)] * z[np.asarray(dst)]
    return p @ w.T


def pair_filter_index(edge_lists):
    """``{(s, t): sorted unique relations r}`` of the triples of a sequence of ``(edge_index, edge_type)`` lists."""
    rows = {}
    for ei, et in edge_lists:
        ei, et = np.asarray(ei), np.asarray(et)
        for s, r, t in zip(ei[0].tolist(), et.tolist(), ei[1].tolist()):
            rows.setdefault((s, t), set()).add(r)
    return {key: np.array(sorted(v), dtype=np.int64) for key, v in rows.items()}


def _relation_negatives(R, filt, s, t, r=None):
    keep = np.ones(R, dtype=bool)
    f = filt.get((s, t))
    if f is not None:
        keep[f] = False
    if r is not None:
        keep[r] = False
    return keep


def filtered_relation_ranks(z, w, edge_index, edge_type, filter_edges=(), tol=None):
    """Filtered OGB relation rank of every triple (float64 ``[E]``) against all relations of its pair.  With ``tol``
    (per-triple tolerances ``delta``), returns ``(lo, hi)`` as ``filtered_ranks`` does."""
    ei, et = np.asarray(edge_index), np.asarray(edge_type)
    filt = pair_filter_index(filter_edges)
    z64, w64 = np.asarray(z, dtype=np.float64), np.asarray(w, dtype=np.float64)
    R = w64.shape[0]
    ranks, lo, hi = (np.empty(ei.shape[1]) for _ in range(3))
    for e in range(ei.shape[1]):
        s, r, t = int(ei[0, e]), int(et[e]), int(ei[1, e])
        row = w64 @ (z64[s] * z64[t])
        v, sr = row[_relation_negatives(R, filt, s, t, r)], row[r]
        ranks[e] = 1.0 + (np.sum(v > sr) + np.sum(v >= sr)) / 2.0
        if tol is not None:
            d = float(np.asarray(tol).reshape(-1)[e])
            lo[e] = 1.0 + np.sum(v > sr + d)
            hi[e] = 1.0 + np.sum(v >= sr - d)
    return (lo, hi) if tol is not None else ranks


def topk_relations(z, w, src, dst, k, filter_edges=()):
    """``(scores float64 [Q, k] pre-sigmoid, ids int64 [Q, k])``: the ``k`` best admissible relations of every pair,
    descending score, ties by smaller relation id; id -1 / NaN where fewer than ``k`` are admissible."""
    filt = pair_filter_index(filter_edges)
    src, dst = np.asarray(src).reshape(-1), np.asarray(dst).reshape(-1)
    S = relation_scores(z, w, src, dst)
    R = S.shape[1]
    out_s = np.full((src.size, k), np.nan)
    out_i = np.full((src.size, k), -1, dtype=np.int64)
    for i in range(src.size):
        cand = np.nonzero(_relation_negatives(R, filt, int(src[i]), int(dst[i])))[0]
        cand = cand[np.lexsort((cand, -S[i, cand]))]              # descending score, then ascending id
        m = min(k, cand.size)
        out_i[i, :m] = cand[:m]
        out_s[i, :m] = S[i, cand[:m]]
    return out_s, out_i
