"""CPU: the float64 relation-ranking oracle (oracle/relation_ranking.py: relation_scores, filtered_relation_ranks,
topk_relations) against a hand-worked example, a per-relation brute force and the tail oracle's scores."""
import numpy as np
import pytest

from oracle import ranking as orank
from oracle import relation_ranking as orel

# Hand-worked graph: n = 4, D = 1, R = 5 (relation 4 has no query triple).  S(s, r', t) = z[s] * z[t] * w[r']:
#   pair (0, 1), and its mirror (1, 0): S = [2, 4, 4, -2, 1]      pair (2, 2): S = [9, 18, 18, -9, 4.5]
#   pair (0, 3):                        S = [-2, -4, -4, 2, -1]
HREL_Z = np.array([[2.0], [1.0], [3.0], [-1.0]])
HREL_W = np.array([[1.0], [2.0], [2.0], [-1.0], [0.5]])
HREL_TEST = (np.array([[0, 0, 2, 0], [1, 1, 2, 3]]), np.array([0, 1, 3, 2]))
# (0, 1, 1): the second test triple's relation; (2, r, 2) for r != 3: every other relation of the self pair;
# (0, 0, 3) twice: a duplicated filter triple
HREL_TRAIN = (np.array([[0, 2, 2, 2, 2, 0, 0], [1, 2, 2, 2, 2, 3, 3]]), np.array([1, 0, 1, 2, 4, 0, 0]))
HREL_FILTER = (HREL_TRAIN, HREL_TEST)
# e0 (0,0,1): the target is in the filter; r' = 1 filtered; r' = 2 beats it, r' = 3 / 4 do not       -> 1 + (1+1)/2
# e1 (0,1,1): r' = 0 filtered (a test triple); r' = 2 ties the target                                 -> 1 + (0+1)/2
# e2 (2,3,2): self pair s == t, every other relation filtered                                           -> 1
# e3 (0,2,3): r' = 1 ties the target, r' = 3 and 4 beat it, r' = 0 filtered (twice)                    -> 1 + (2+3)/2
HREL_RANKS = [2.0, 1.5, 1.0, 3.5]
HREL_RAW_RANKS = [3.0, 1.5, 5.0, 4.5]          # no filter: r' = 1 now beats e0, everything beats e2, r' = 0 beats e3
HREL_PAIRS = ([0, 2, 0, 1], [1, 2, 3, 0])
HREL_TOPK_IDS = [[2, 4, 3, -1, -1, -1],         # k = 6 > R = 5: every row padded
                 [-1, -1, -1, -1, -1, -1],      # every relation of the self pair is filtered
                 [3, 4, 1, -1, -1, -1],
                 [1, 2, 0, 4, 3, -1]]           # mirror pair (1, 0): nothing filtered; the 1 / 2 tie -> smaller id
HREL_TOPK_SCORES = [[4.0, 1.0, -2.0], [], [2.0, -1.0, -4.0], [4.0, 4.0, 2.0, 1.0, -2.0]]


def _brute_ranks(z, w, ei, et, triples):
    R, d = w.shape
    out = []
    for e in range(ei.shape[1]):
        s, r, t = int(ei[0, e]), int(et[e]), int(ei[1, e])

        def score(q):
            acc = 0.0
            for k in range(d):
                acc += float(z[s, k]) * float(z[t, k]) * float(w[q, k])
            return acc

        sr = score(r)
        opt = pess = 0
        for q in range(R):
            if q == r or (s, q, t) in triples:
                continue
            sc = score(q)
            opt += sc > sr
            pess += sc >= sr
        out.append(1.0 + (opt + pess) / 2.0)
    return np.array(out)


def _triples(lists):
    return {(int(s), int(r), int(t)) for ei, et in lists for s, t, r in zip(ei[0], ei[1], et)}


def test_hand_example_relation_ranks():
    np.testing.assert_array_equal(orel.filtered_relation_ranks(HREL_Z, HREL_W, *HREL_TEST, HREL_FILTER), HREL_RANKS)
    np.testing.assert_array_equal(orel.filtered_relation_ranks(HREL_Z, HREL_W, *HREL_TEST), HREL_RAW_RANKS)


def test_hand_example_relation_metrics():
    m = orank.rank_metrics(HREL_RANKS, HREL_TEST[1], 5, hits=(1, 3))
    np.testing.assert_allclose(m[:, :4], [[0.5, 2 / 3, 2 / 7, 1.0], [0, 0, 0, 1], [1, 1, 0, 1]], rtol=0, atol=1e-15)
    assert np.isnan(m[:, 4]).all()


def test_hand_example_topk_relations():
    s, i = orel.topk_relations(HREL_Z, HREL_W, *HREL_PAIRS, 6, HREL_FILTER)
    np.testing.assert_array_equal(i, HREL_TOPK_IDS)
    for q, want in enumerate(HREL_TOPK_SCORES):
        np.testing.assert_array_equal(s[q, :len(want)], want)
        assert np.isnan(s[q, len(want):]).all()
    s, i = orel.topk_relations(HREL_Z, HREL_W, [0], [1], 2)          # no filter: the 2-way tie goes to the smaller id
    np.testing.assert_array_equal(i, [[1, 2]])
    np.testing.assert_array_equal(s, [[4.0, 4.0]])


def test_single_relation():
    """R = 1: no other relation to beat the target, so every rank is 1; k > R pads."""
    w = np.array([[1.0]])
    test = (np.array([[0, 2], [1, 2]]), np.array([0, 0]))
    np.testing.assert_array_equal(orel.filtered_relation_ranks(HREL_Z, w, *test), [1.0, 1.0])
    np.testing.assert_array_equal(orel.filtered_relation_ranks(HREL_Z, w, *test, (test,)), [1.0, 1.0])
    s, i = orel.topk_relations(HREL_Z, w, [0], [1], 3)
    np.testing.assert_array_equal(i, [[0, -1, -1]])
    assert s[0, 0] == 2.0 and np.isnan(s[0, 1:]).all()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_relation_oracle_matches_brute_force_and_tail_scores(seed):
    rs = np.random.RandomState(seed)
    n, d, R = 6, 3, 7
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float64)           # integer scores: plenty of exact ties
    w = rs.randint(-1, 2, size=(R, d)).astype(np.float64)
    e = 30
    test = (rs.randint(0, n, size=(2, e)), rs.randint(0, R, size=e))
    train = (rs.randint(0, n, size=(2, 60)), rs.randint(0, R, size=60))
    lists = (train, test)
    trip = _triples(lists)
    want = _brute_ranks(z, w, test[0], test[1], trip)
    np.testing.assert_array_equal(orel.filtered_relation_ranks(z, w, *test, lists), want)
    lo, hi = orel.filtered_relation_ranks(z, w, *test, lists, tol=np.full(e, 0.5))
    assert (lo <= want).all() and (want <= hi).all()
    # relation scores of (s, ?, t) are the tail scores of (s, r, ?) read at column t
    src, dst = test[0]
    rel_s = orel.relation_scores(z, w, src, dst)
    for r in range(R):
        tail = orank.scores(z, w, src, np.full(e, r))
        np.testing.assert_allclose(rel_s[:, r], tail[np.arange(e), dst], rtol=1e-15, atol=0)
    # top-k: brute-force order of the admissible relations
    s, ids = orel.topk_relations(z, w, src, dst, 5, lists)
    for q in range(e):
        cand = sorted((r for r in range(R) if (int(src[q]), r, int(dst[q])) not in trip),
                      key=lambda r: (-rel_s[q, r], r))[:5]
        assert ids[q, :len(cand)].tolist() == cand
        assert (ids[q, len(cand):] == -1).all()
