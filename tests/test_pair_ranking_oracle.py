"""CPU: the float64 pair-ranking oracle (oracle/pair_ranking.py: topk_pairs) against a hand-worked example and an
itertools.combinations brute force with a directed filter read in both directions."""
import itertools

import numpy as np
import pytest

from oracle import pair_ranking as opair

# Hand-worked graph: n = 4, D = 1, R = 2.  S(s, r, t) = z[s] * w[r] * z[t]:
#   r = 0: {0,1} = 2, {0,2} = 4, {0,3} = -2, {1,2} = 2, {1,3} = -1, {2,3} = -2
#   r = 1: {0,1} = -2, {0,2} = -4, {0,3} = 2, {1,2} = -2, {1,3} = 1, {2,3} = 2
HPAIR_Z = np.array([[2.0], [1.0], [2.0], [-1.0]])
HPAIR_W = np.array([[1.0], [-1.0]])
# (2, 0, 0): only the flipped direction of {0, 2} under r = 0; (1, 1, 3): {1, 3} under r = 1; (2, 1, 2): a self
# pair, never a candidate; (3, 0, 1), listed twice: {1, 3} under r = 0
HPAIR_FILTER = ((np.array([[2, 1, 2], [0, 3, 2]]), np.array([0, 1, 1])),
                (np.array([[3, 3], [1, 1]]), np.array([0, 0])))
HPAIR_REL = [0, 1, 0]                                       # a duplicated query
# r = 0: {0,2} and {1,3} filtered; the 2 / 2 tie goes to s = 0, the -2 / -2 tie to s = 0; k = 6 > 4 admissible
# r = 1: {1,3} filtered; the 2 / 2 tie goes to s = 0, the -2 / -2 tie to s = 0
HPAIR_SRC = [[0, 1, 0, 2, -1, -1], [0, 2, 0, 1, 0, -1], [0, 1, 0, 2, -1, -1]]
HPAIR_DST = [[1, 2, 3, 3, -1, -1], [3, 3, 1, 2, 2, -1], [1, 2, 3, 3, -1, -1]]
HPAIR_SCORES = [[2.0, 2.0, -2.0, -2.0], [2.0, 2.0, -2.0, -2.0, -4.0], [2.0, 2.0, -2.0, -2.0]]


def _check_hand(s, a, b):
    np.testing.assert_array_equal(a, HPAIR_SRC)
    np.testing.assert_array_equal(b, HPAIR_DST)
    for q, want in enumerate(HPAIR_SCORES):
        np.testing.assert_array_equal(s[q, :len(want)], want)
        assert np.isnan(s[q, len(want):]).all()


def test_hand_example_topk_pairs():
    _check_hand(*opair.topk_pairs(HPAIR_Z, HPAIR_W, HPAIR_REL, 6, HPAIR_FILTER))
    s, a, b = opair.topk_pairs(HPAIR_Z, HPAIR_W, [0], 2)     # no filter: {0,2} first, then the {0,1} / {1,2} tie
    np.testing.assert_array_equal(a, [[0, 0]])
    np.testing.assert_array_equal(b, [[2, 1]])
    np.testing.assert_array_equal(s, [[4.0, 2.0]])


def test_fewer_than_two_nodes_pads():
    s, a, b = opair.topk_pairs(HPAIR_Z[:1], HPAIR_W, [0, 1], 3)
    assert (a == -1).all() and (b == -1).all() and np.isnan(s).all()
    s, a, b = opair.topk_pairs(HPAIR_Z[:2], HPAIR_W, [1], 3)
    assert a.tolist() == [[0, -1, -1]] and b.tolist() == [[1, -1, -1]] and s[0, 0] == -2.0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_pair_oracle_matches_brute_force(seed):
    rs = np.random.RandomState(seed)
    n, d, R = 9, 3, 4
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float64)           # integer scores: plenty of exact ties
    w = rs.randint(-1, 2, size=(R, d)).astype(np.float64)
    lists = ((rs.randint(0, n, size=(2, 40)), rs.randint(0, R, size=40)),
             (rs.randint(0, n, size=(2, 10)), rs.randint(0, R, size=10)))
    trip = {(int(s), int(r), int(t)) for ei, et in lists for s, t, r in zip(ei[0], ei[1], et)}
    rel = [0, 3, 1, 3, 2]
    k = 20
    s, a, b = opair.topk_pairs(z, w, rel, k, lists)
    for q, r in enumerate(rel):
        def score(p):
            return sum(float(z[p[0], j]) * float(w[r, j]) * float(z[p[1], j]) for j in range(d))

        cand = [p for p in itertools.combinations(range(n), 2) if (p[0], r, p[1]) not in trip and
                (p[1], r, p[0]) not in trip]
        cand = sorted(cand, key=lambda p: (-score(p), p[0], p[1]))[:k]
        assert list(zip(a[q, :len(cand)].tolist(), b[q, :len(cand)].tolist())) == cand
        assert [s[q, i] for i in range(len(cand))] == [score(p) for p in cand]
        assert (a[q, len(cand):] == -1).all() and (b[q, len(cand):] == -1).all()
    # the filter is read in both directions: flipping every filter triple changes nothing
    flipped = tuple((ei[::-1].copy(), et) for ei, et in lists)
    s2, a2, b2 = opair.topk_pairs(z, w, rel, k, flipped)
    np.testing.assert_array_equal(a2, a)
    np.testing.assert_array_equal(b2, b)
    np.testing.assert_array_equal(s2, s)
    # and a filter of one direction only excludes the pair
    _, a3, b3 = opair.topk_pairs(z, w, [rel[0]], k)
    one = (np.array([[int(b3[0, 0])], [int(a3[0, 0])]]), np.array([rel[0]]))     # (t, r, s) of the best pair
    _, a4, b4 = opair.topk_pairs(z, w, [rel[0]], k, (one,))
    assert (int(a3[0, 0]), int(b3[0, 0])) not in set(zip(a4[0].tolist(), b4[0].tolist()))
    assert (a4[0, :k - 1] == a3[0, 1:]).all() and (b4[0, :k - 1] == b3[0, 1:]).all()
