"""CPU: the float64 ranking oracle (oracle/ranking.py) against a per-candidate brute force and a hand-worked example."""
import numpy as np
import pytest

from oracle import ranking as orank

# Hand-worked graph: n = 5, D = 1, R = 3 (relation 2 has no edges).  S(s, r, c) = z[s] * w[r] * z[c]:
#   query (0, 0): S = [4, 2, 2, 6, 0]      query (2, 1): S = [-2, -1, -1, -3, 0]      query (4, 0): S = 0 everywhere
HAND_Z = np.array([[2.0], [1.0], [1.0], [3.0], [0.0]])
HAND_W = np.array([[1.0], [-1.0], [0.5]])
HAND_TEST = (np.array([[0, 0, 2, 4], [1, 3, 1, 0]]), np.array([0, 0, 1, 0]))
HAND_TRAIN = (np.array([[0, 0], [3, 3]]), np.array([0, 0]))       # (0, 0, 3) twice: a duplicated filter edge
HAND_FILTER = (HAND_TRAIN, HAND_TEST)
# e0 (0,0,1): target in the filter, filtered c = 3 outscores it, c = 2 ties it, c == s (0) beats it -> 1 + (1+2)/2
# e1 (0,0,3): nothing admissible reaches 6                                                             -> 1
# e2 (2,1,1): c == s (2) ties the target, c = 4 beats it                                               -> 1 + (1+2)/2
# e3 (4,0,0): all four admissible candidates tie the target                                            -> 1 + (0+4)/2
HAND_RANKS = [2.5, 1.0, 2.5, 3.0]
HAND_RAW_RANKS = [3.5, 1.0, 2.5, 3.0]            # no filter: c = 3 now beats e0's target


def _brute_ranks(z, w, ei, et, triples):
    n, d = z.shape
    out = []
    for e in range(ei.shape[1]):
        s, r, t = int(ei[0, e]), int(et[e]), int(ei[1, e])

        def score(c):
            acc = 0.0
            for k in range(d):
                acc += float(z[s, k]) * float(w[r, k]) * float(z[c, k])
            return acc

        st = score(t)
        opt = pess = 0
        for c in range(n):
            if c == t or (s, r, c) in triples:
                continue
            sc = score(c)
            opt += sc > st
            pess += sc >= st
        out.append(1.0 + (opt + pess) / 2.0)
    return np.array(out)


def _triples(lists):
    return {(int(s), int(r), int(c)) for ei, et in lists for s, c, r in zip(ei[0], ei[1], et)}


def test_hand_example_ranks():
    np.testing.assert_array_equal(orank.filtered_ranks(HAND_Z, HAND_W, *HAND_TEST, HAND_FILTER), HAND_RANKS)
    np.testing.assert_array_equal(orank.filtered_ranks(HAND_Z, HAND_W, *HAND_TEST), HAND_RAW_RANKS)


def test_hand_example_metrics():
    m = orank.rank_metrics(HAND_RANKS, HAND_TEST[1], 3, hits=(1, 3))
    np.testing.assert_allclose(m[:, 0], [(1 / 2.5 + 1 + 1 / 3) / 3, 1 / 3, 1.0], rtol=0, atol=1e-15)
    np.testing.assert_allclose(m[:, 1], [0.4, 0.0, 1.0], rtol=0, atol=1e-15)
    assert np.isnan(m[:, 2]).all()


def test_hand_example_topk():
    s, i = orank.topk(HAND_Z, HAND_W, [0, 2, 4], [0, 1, 0], 4, HAND_FILTER)
    np.testing.assert_array_equal(i, [[0, 2, 4, -1], [4, 2, 0, 3], [1, 2, 3, 4]])
    np.testing.assert_array_equal(s[0, :3], [4.0, 2.0, 0.0])
    assert np.isnan(s[0, 3])
    np.testing.assert_array_equal(s[1], [0.0, -1.0, -2.0, -3.0])
    s, i = orank.topk(HAND_Z, HAND_W, [0], [0], 3)                   # no filter: the 2-way tie goes to the smaller id
    np.testing.assert_array_equal(i, [[3, 0, 1]])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_matches_brute_force(seed):
    rs = np.random.RandomState(seed)
    n, d, r = 9, 3, 3
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float64)           # integer scores: plenty of exact ties
    w = rs.randint(-1, 2, size=(r, d)).astype(np.float64)
    e = 30
    test = (rs.randint(0, n, size=(2, e)), rs.randint(0, r, size=e))
    train = (rs.randint(0, n, size=(2, 40)), rs.randint(0, r, size=40))
    lists = (train, test)
    want = _brute_ranks(z, w, test[0], test[1], _triples(lists))
    np.testing.assert_array_equal(orank.filtered_ranks(z, w, *test, lists), want)
    # the ambiguity band brackets the rank
    lo, hi = orank.filtered_ranks(z, w, *test, lists, tol=np.full(e, 0.5))
    assert (lo <= want).all() and (want <= hi).all()
    # top-k: brute-force order of the admissible candidates
    trip = _triples(lists)
    node, rel = test[0][0], test[1]
    s, ids = orank.topk(z, w, node, rel, 5, lists)
    full = orank.scores(z, w, node, rel)
    for q in range(e):
        cand = sorted((c for c in range(n) if (int(node[q]), int(rel[q]), c) not in trip),
                      key=lambda c: (-full[q, c], c))[:5]
        assert ids[q, :len(cand)].tolist() == cand
        assert (ids[q, len(cand):] == -1).all()
