"""float64 numpy restatement of the top-k new pairs of a relation for the DistMult decoder.

Semantics as in ``gripnet_b200/ranking.py`` (pinned here independently of it).  Pair queries ``(?, r, ?)``: every
unordered pair ``{s, t}`` with ``s < t`` is a candidate with pre-sigmoid score ``S(s, t) = sum_k z[s,k] w[r,k] z[t,k]``;
the pair is filtered for ``r`` when ``(s, r, t)`` or ``(t, r, s)`` is a filter triple; top-k by descending score,
ties by smaller ``s`` then smaller ``t`` (the pair id ``s * n + t``), padded with ids -1 / NaN.
"""
import numpy as np


def pair_scores(z, w, r):
    """float64 ``[n, n]``: ``S(s, t)`` of relation ``r`` for every ordered pair (symmetric)."""
    z = np.asarray(z, dtype=np.float64)
    w = np.asarray(w, dtype=np.float64)
    return (z * w[int(r)]) @ z.T


def symmetric_filter(edge_lists):
    """The filter triples of a sequence of ``(edge_index, edge_type)`` lists as a set of ``(min(s, t), r, max(s, t))``:
    both directions of a pair meet in one entry."""
    out = set()
    for ei, et in edge_lists:
        ei, et = np.asarray(ei), np.asarray(et)
        for s, r, t in zip(ei[0].tolist(), et.tolist(), ei[1].tolist()):
            out.add((min(s, t), r, max(s, t)))
    return out


def topk_pairs(z, w, rel, k, filter_edges=()):
    """``(scores float64 [Q, k] pre-sigmoid, src int64 [Q, k], dst int64 [Q, k])``: the ``k`` best admissible
    unordered pairs of every relation ``rel[i]``, ``src < dst``, descending score, ties by smaller ``src`` then
    smaller ``dst``; ids -1 / NaN where fewer than ``k`` are admissible."""
    filt = symmetric_filter(filter_edges)
    rel = np.asarray(rel, dtype=np.int64).reshape(-1)
    n = np.asarray(z).shape[0]
    su, tu = np.triu_indices(n, k=1)                     # every s < t, in ascending pair id s * n + t
    out_s = np.full((rel.size, k), np.nan)
    out_a = np.full((rel.size, k), -1, dtype=np.int64)
    out_b = np.full((rel.size, k), -1, dtype=np.int64)
    for i, r in enumerate(rel.tolist()):
        S = pair_scores(z, w, r)[su, tu]
        keep = np.array([(a, r, b) not in filt for a, b in zip(su.tolist(), tu.tolist())], dtype=bool)
        a, b, v = su[keep], tu[keep], S[keep]
        order = np.lexsort((b, a, -v))                   # descending score, then ascending s, then ascending t
        m = min(k, order.size)
        out_a[i, :m], out_b[i, :m], out_s[i, :m] = a[order[:m]], b[order[:m]], v[order[:m]]
    return out_s, out_a, out_b
