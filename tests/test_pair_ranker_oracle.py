"""CPU: the float64 pair-rank oracle (oracle/pair_ranks.py: filtered_pair_ranks) against a hand-worked example and
an itertools.combinations brute force with a directed filter read in both directions."""
import itertools

import numpy as np
import pytest

from oracle import pair_ranks as opr
from test_pair_ranking_oracle import HPAIR_FILTER, HPAIR_W, HPAIR_Z

# Query triples of the hand-worked graph of test_pair_ranking_oracle (n = 4, D = 1, R = 2):
#   r = 0: {0,1} = 2, {0,2} = 4, {0,3} = -2, {1,2} = 2, {1,3} = -1, {2,3} = -2; filter: {0,2}, {1,3}
#   r = 1: {0,1} = -2, {0,2} = -4, {0,3} = 2, {1,2} = -2, {1,3} = 1, {2,3} = 2; filter: {1,3} (and the self pair 2-2)
# (0,0,1) and its mirror (1,0,0); (2,0,0) and (1,1,3) are filter triples; (2,1,2) is a self pair.
HRANK_EI = np.array([[0, 1, 2, 3, 2, 1, 0], [1, 0, 0, 2, 2, 3, 2]])
HRANK_ET = np.array([0, 0, 0, 0, 1, 1, 1])
# filtered, e.g. (3,0,2): S = -2 against {0,1} = 2, {0,3} = -2, {1,2} = 2 -> opt 2, pess 3, rank 3.5
HRANK_FILTERED = [1.5, 1.5, 1.0, 3.5, np.nan, 3.0, 5.0]
# raw, e.g. (0,0,1): S = 2 against 4, -2, 2, -1, -2 -> opt 1, pess 2, rank 2.5
HRANK_RAW = [2.5, 2.5, 1.0, 5.5, np.nan, 3.0, 6.0]


def test_hand_example_pair_ranks():
    got = opr.filtered_pair_ranks(HPAIR_Z, HPAIR_W, HRANK_EI, HRANK_ET, HPAIR_FILTER)
    np.testing.assert_array_equal(got, HRANK_FILTERED)
    np.testing.assert_array_equal(opr.filtered_pair_ranks(HPAIR_Z, HPAIR_W, HRANK_EI, HRANK_ET), HRANK_RAW)
    lo, hi = opr.filtered_pair_ranks(HPAIR_Z, HPAIR_W, HRANK_EI, HRANK_ET, HPAIR_FILTER, tol=np.full(7, 0.5))
    np.testing.assert_array_equal(lo, [1.0, 1.0, 1.0, 3.0, np.nan, 3.0, 5.0])      # ties counted as below
    np.testing.assert_array_equal(hi, [2.0, 2.0, 1.0, 4.0, np.nan, 3.0, 5.0])      # ties counted as above


def _brute(z, w, ei, et, lists):
    trip = {(int(s), int(r), int(t)) for l_ei, l_et in lists for s, t, r in zip(l_ei[0], l_ei[1], l_et)}
    n, d = z.shape
    out = []
    for s, t, r in zip(ei[0].tolist(), ei[1].tolist(), et.tolist()):
        if s == t:
            out.append(np.nan)
            continue

        def score(p):
            return sum(float(z[p[0], j]) * float(w[r, j]) * float(z[p[1], j]) for j in range(d))

        st = score((min(s, t), max(s, t)))
        neg = [score(p) for p in itertools.combinations(range(n), 2)
               if set(p) != {s, t} and (p[0], r, p[1]) not in trip and (p[1], r, p[0]) not in trip]
        out.append(1.0 + (sum(v > st for v in neg) + sum(v >= st for v in neg)) / 2.0)
    return np.array(out)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_pair_rank_oracle_matches_brute_force(seed):
    rs = np.random.RandomState(seed)
    n, d, R = 9, 3, 4
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float64)           # integer scores: plenty of exact ties
    w = rs.randint(-1, 2, size=(R, d)).astype(np.float64)
    lists = ((rs.randint(0, n, size=(2, 30)), rs.randint(0, R, size=30)),)
    # queries: half of them filter triples (targets inside the filter), the rest random, their mirrors, self pairs
    q = np.concatenate([lists[0][0][:, :8], rs.randint(0, n, size=(2, 12)), [[4, 5], [4, 5]]], axis=1)
    qt = np.concatenate([lists[0][1][:8], rs.randint(0, R, size=12), [1, 2]])
    ei, et = np.concatenate([q, q[::-1]], axis=1), np.concatenate([qt, qt])
    got = opr.filtered_pair_ranks(z, w, ei, et, lists)
    np.testing.assert_array_equal(got, _brute(z, w, ei, et, lists))
    np.testing.assert_array_equal(got[:qt.size], got[qt.size:])                    # mirrored triples
    assert np.isnan(got[ei[0] == ei[1]]).all() and not np.isnan(got[ei[0] != ei[1]]).any()
    np.testing.assert_array_equal(opr.filtered_pair_ranks(z, w, ei, et), _brute(z, w, ei, et, ()))
    # the filter is read in both directions: flipping every filter triple changes nothing
    flipped = tuple((l_ei[::-1].copy(), l_et) for l_ei, l_et in lists)
    np.testing.assert_array_equal(opr.filtered_pair_ranks(z, w, ei, et, flipped), got)
