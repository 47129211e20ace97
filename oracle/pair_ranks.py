"""float64 numpy restatement of the filtered pair ranks of a relation for the DistMult decoder.

Semantics as in ``gripnet_b200/ranking.py`` (pinned here independently of it).  The triple ``(s, r, t)`` is the query
``(?, r, ?)`` with answer ``{s, t}``; its OGB rank ``1 + (opt + pess) / 2`` is taken over the unordered pairs
``a < b`` of ``r`` other than ``{s, t}`` that the filter does not hold in either direction (the candidates, scores and
filter of ``pair_ranking.topk_pairs``); a self pair ``s == t`` has no rank (NaN).
"""
import numpy as np

from .pair_ranking import pair_scores, symmetric_filter


def filtered_pair_ranks(z, w, edge_index, edge_type, filter_edges=(), tol=None):
    """Filtered OGB pair rank of every triple (float64 ``[E]``): ``(s, r, t)`` is the query ``(?, r, ?)`` with answer
    ``{min(s, t), max(s, t)}``, ranked among the unfiltered pairs ``a < b`` of ``r`` other than itself.  NaN for a
    self-pair ``s == t``.  With ``tol`` (per-triple tolerances ``delta``), returns ``(lo, hi)`` as
    ``ranking.filtered_ranks`` does."""
    ei, et = np.asarray(edge_index), np.asarray(edge_type)
    filt = symmetric_filter(filter_edges)
    n = np.asarray(z).shape[0]
    su, tu = np.triu_indices(n, k=1)
    ranks, lo, hi = (np.full(ei.shape[1], np.nan) for _ in range(3))
    for r in np.unique(et).tolist():
        S = pair_scores(z, w, r)[su, tu]
        keep = np.array([(a, r, b) not in filt for a, b in zip(su.tolist(), tu.tolist())], dtype=bool)
        for e in np.nonzero(et == r)[0].tolist():
            a, b = sorted((int(ei[0, e]), int(ei[1, e])))
            if a == b:
                continue
            target = a * n - a * (a + 1) // 2 + (b - a - 1)            # position of (a, b) in the triu order
            sel = keep.copy()
            sel[target] = False
            v, st = S[sel], S[target]
            ranks[e] = 1.0 + (np.sum(v > st) + np.sum(v >= st)) / 2.0
            if tol is not None:
                d = float(np.asarray(tol).reshape(-1)[e])
                lo[e] = 1.0 + np.sum(v > st + d)
                hi[e] = 1.0 + np.sum(v >= st - d)
    return (lo, hi) if tol is not None else ranks
