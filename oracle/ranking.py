"""float64 numpy restatement of filtered candidate ranking and top-k link prediction of the DistMult decoder.

Semantics as in ``gripnet_b200/ranking.py`` (pinned here independently of it): pre-sigmoid scores
``S(s, r, c) = sum_k z[s,k] w[r,k] z[c,k]`` for every candidate ``c``; a filter is a set of directed triples; tail
queries only; OGB rank ``1 + (opt + pess) / 2`` over ``N = {c != t : (s, r, c) not in filter}``; per-relation MRR and
Hits@k (NaN for a relation without edges); top-k by descending score, ties by smaller id, padded with id -1 / NaN.
"""
import numpy as np


def scores(z, w, node, rel):
    """float64 ``[Q, n]``: the score of every candidate of every query ``(node[i], rel[i])``."""
    z = np.asarray(z, dtype=np.float64)
    w = np.asarray(w, dtype=np.float64)
    q = z[np.asarray(node)] * w[np.asarray(rel)]
    return q @ z.T


def filter_index(edge_lists):
    """``{(s, r): sorted unique candidates c}`` of the triples of a sequence of ``(edge_index [2, E], edge_type [E])``
    lists."""
    rows = {}
    for ei, et in edge_lists:
        ei, et = np.asarray(ei), np.asarray(et)
        for s, r, c in zip(ei[0].tolist(), et.tolist(), ei[1].tolist()):
            rows.setdefault((s, r), set()).add(c)
    return {key: np.array(sorted(v), dtype=np.int64) for key, v in rows.items()}


def _negatives(n, filt, s, r, t=None):
    keep = np.ones(n, dtype=bool)
    f = filt.get((s, r))
    if f is not None:
        keep[f] = False
    if t is not None:
        keep[t] = False
    return keep


def filtered_ranks(z, w, edge_index, edge_type, filter_edges=(), tol=None):
    """Filtered OGB rank of every edge (float64 ``[E]``).  With ``tol`` (per-edge tolerances ``delta``), returns
    ``(lo, hi)`` instead: the ranks obtained when every negative within ``delta`` of the target score is counted as
    not beating it (``lo``) and as beating it (``hi``)."""
    ei, et = np.asarray(edge_index), np.asarray(edge_type)
    filt = filter_index(filter_edges)
    z64, w64 = np.asarray(z, dtype=np.float64), np.asarray(w, dtype=np.float64)
    n = z64.shape[0]
    ranks, lo, hi = (np.empty(ei.shape[1]) for _ in range(3))
    for e in range(ei.shape[1]):
        s, r, t = int(ei[0, e]), int(et[e]), int(ei[1, e])
        row = (z64[s] * w64[r]) @ z64.T
        v, st = row[_negatives(n, filt, s, r, t)], row[t]
        ranks[e] = 1.0 + (np.sum(v > st) + np.sum(v >= st)) / 2.0
        if tol is not None:
            d = float(np.asarray(tol).reshape(-1)[e])
            lo[e] = 1.0 + np.sum(v > st + d)
            hi[e] = 1.0 + np.sum(v >= st - d)
    return (lo, hi) if tol is not None else ranks


def rank_metrics(ranks, edge_type, num_relations, hits=(1, 3, 10)):
    """float64 ``[1 + len(hits), R]``: MRR and Hits@k per relation; NaN for a relation without edges."""
    ranks, et = np.asarray(ranks, dtype=np.float64), np.asarray(edge_type)
    out = np.full((1 + len(hits), num_relations), np.nan)
    for r in range(num_relations):
        rk = ranks[et == r]
        if rk.size:
            out[0, r] = np.mean(1.0 / rk)
            for i, k in enumerate(hits):
                out[1 + i, r] = np.mean(rk <= k)
    return out


def topk(z, w, node, rel, k, filter_edges=()):
    """``(scores float64 [Q, k] pre-sigmoid, ids int64 [Q, k])``: the ``k`` best admissible candidates of every
    query, descending score, ties by smaller id; id -1 / NaN where fewer than ``k`` are admissible."""
    filt = filter_index(filter_edges)
    node, rel = np.asarray(node).reshape(-1), np.asarray(rel).reshape(-1)
    S = scores(z, w, node, rel)
    n = S.shape[1]
    out_s = np.full((node.size, k), np.nan)
    out_i = np.full((node.size, k), -1, dtype=np.int64)
    for i in range(node.size):
        s, r = int(node[i]), int(rel[i])
        cand = np.nonzero(_negatives(n, filt, s, r))[0]
        cand = cand[np.lexsort((cand, -S[i, cand]))]              # descending score, then ascending id
        m = min(k, cand.size)
        out_i[i, :m] = cand[:m]
        out_s[i, :m] = S[i, cand[:m]]
    return out_s, out_i
