"""GPU: filtered pair ranks (gripnet_b200.ranking.PairRanker) against the float64 oracle
(oracle/pair_ranks.py: filtered_pair_ranks) and against topk_pairs."""
import numpy as np
import pytest
import torch

from oracle import pair_ranking as opair
from oracle import pair_ranks as opr
from oracle import ranking as oracle_ranking
from test_gpu_pair_ranking import _integer_fixture, _lists_t, _pose_split, _strided, _t

pytestmark = pytest.mark.gpu


def _bits(x):
    """Bitwise view (NaN-aware equality)."""
    return x.contiguous().view(torch.int32 if x.dtype == torch.float32 else torch.int64)


def _queries(rs, n, r, lists, count):
    """Triples of both directions, duplicated, half of them filter triples (targets in the filter), the
    one-direction filter pairs of relation 0 queried the other way round, and two self pairs."""
    (tr_ei, tr_et), (fl_ei, fl_et) = lists
    pick = rs.randint(0, tr_et.size, size=count)
    rand = rs.randint(0, n, size=(2, count))
    ei = np.concatenate([tr_ei[:, pick], rand, fl_ei[::-1], [[0, n - 1], [0, n - 1]]], axis=1)
    et = np.concatenate([tr_et[pick], rs.randint(0, r, size=count), fl_et, [1, 2]])
    ei = np.concatenate([ei, ei[::-1], ei[:, :3]], axis=1)
    et = np.concatenate([et, et, et[:3]])
    return ei, et


def _metrics_oracle(ranks, et, r, hits):
    keep = ~np.isnan(ranks)
    return oracle_ranking.rank_metrics(ranks[keep], et[keep], r, hits)


@pytest.mark.parametrize("d", [1, 7, 80])
@pytest.mark.parametrize("n", [2, 3, 40, 700])
def test_exact_integer_fixture(n, d):
    """Bit for bit against the oracle on exact integer scores (many ties), strided z, filter present and absent."""
    import gripnet_b200 as gb
    r = 3
    z, w, lists = _integer_fixture(n * 17 + d, n, d, r)
    rs = np.random.RandomState(n + d)
    ei, et = _queries(rs, n, r, lists, 24)
    zt, wt = _strided(z), _t(w, torch.float32)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    for f, fl in ((filt, lists), (None, ())):
        ranker = gb.PairRanker(_t(ei), _t(et), n, r, filter=f)
        got = ranker.ranks(zt, wt).cpu().numpy()
        want = opr.filtered_pair_ranks(z, w, ei, et, fl)
        np.testing.assert_array_equal(got, want.astype(np.float32))
        assert np.isnan(got[ei[0] == ei[1]]).all()
        assert ranker.n_groups == np.unique(et[ei[0] != ei[1]]).size
        hits = (1, 3, 10)
        m = ranker.metrics(zt, wt, hits=hits).cpu().numpy()
        np.testing.assert_allclose(m, _metrics_oracle(got.astype(np.float64), et, r, hits), rtol=1e-12)


def test_ranks_of_topk_pairs_are_one_to_k():
    """Gaussian scores: the k = 256 best new pairs of topk_pairs under a filter F rank 1, 2, ..., 256 under F, so
    both paths score every pair with the same fp32 arithmetic."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    n, d, r, k = 300, 37, 4, 256
    rs = np.random.RandomState(8)
    z, w = rs.randn(n, d).astype(np.float32), rs.randn(r, d).astype(np.float32)
    lists = ((rs.randint(0, n, size=(2, 3000)), rs.randint(0, r, size=3000)),)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    zt, wt = _strided(z), _t(w, torch.float32)
    for rel in (0, 3):
        s, a, b = ranking.topk_pairs(zt, wt, _t([rel]), k, filter=filt, sigmoid=False)
        assert torch.unique(s).numel() == k
        ei = torch.cat([torch.stack([a[0], b[0]]), torch.stack([b[0], a[0]])], dim=1)
        et = torch.full((2 * k,), rel, dtype=torch.int64, device=ei.device)
        ranks = gb.PairRanker(ei, et, n, r, filter=filt).ranks(zt, wt)
        want = torch.arange(1, k + 1, dtype=torch.float32, device=ei.device)
        assert torch.equal(ranks, torch.cat([want, want]))


def test_counter_paths_and_empty_relations():
    """One relation with 10^5 triples (counters in global memory), one with a single triple, the others empty."""
    import gripnet_b200 as gb
    n, d, r = 300, 7, 5
    z, w, lists = _integer_fixture(4, n, d, r)
    rs = np.random.RandomState(9)
    base = rs.randint(0, n, size=(2, 400))
    base = base[:, base[0] != base[1]]
    want_base = opr.filtered_pair_ranks(z, w, base, np.full(base.shape[1], 2), lists)
    idx = rs.randint(0, base.shape[1], size=100_000)
    one = np.array([[17], [5]])
    ei = np.concatenate([base[:, idx], one], axis=1)
    et = np.concatenate([np.full(idx.size, 2), [4]])
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    ranker = gb.PairRanker(_t(ei), _t(et), n, r, filter=filt)
    assert ranker.n_groups == 2
    got = ranker.ranks(zt, wt).cpu().numpy()
    np.testing.assert_array_equal(got[:-1], want_base[idx].astype(np.float32))
    np.testing.assert_array_equal(got[-1:], opr.filtered_pair_ranks(z, w, one, [4], lists).astype(np.float32))
    staged = gb.PairRanker(_t(base), _t(np.full(base.shape[1], 2)), n, r, filter=filt).ranks(zt, wt)
    np.testing.assert_array_equal(staged.cpu().numpy(), want_base.astype(np.float32))
    m = ranker.metrics(zt, wt, hits=(1, 10)).cpu().numpy()
    assert np.isnan(m[:, [0, 1, 3]]).all() and not np.isnan(m[:, [2, 4]]).any()
    np.testing.assert_allclose(m, _metrics_oracle(got.astype(np.float64), et, r, (1, 10)), rtol=1e-12)


def _pose(graph_fn):
    g = graph_fn()
    train, test = _pose_split(g)
    n, r, d = g["n_d"], g["n_rel"], 80
    rs = np.random.RandomState(3)
    z = (rs.randn(n, d) / np.sqrt(d)).astype(np.float32)
    w = rs.randn(r, d).astype(np.float32)
    return dict(z=z, w=w, lists=(train, test), test=test, n=n, r=r, zt=_t(z, torch.float32),
                wt=_t(w, torch.float32))


@pytest.fixture(scope="module")
def pose0():
    """pose-0 shape (n = 645, R = 16), D = 80, filter = train + test of a 90/10 split."""
    import synthdata
    return _pose(synthdata.pose_graph)


@pytest.fixture(scope="module")
def pose2():
    """pose-2 shape (n = 645, R = 1 097), as pose0."""
    import synthdata
    return _pose(synthdata.pose2_graph)


def _check_pose(p, n_sample):
    """The whole test split and its mirror are ranked; a sample falls inside the fp32 band of the float64 oracle,
    and mirrored triples get bitwise-equal ranks."""
    import gripnet_b200 as gb
    ei, et = p["test"]
    e = et.size
    filt = gb.EdgeFilter(_lists_t(p["lists"]), p["n"], p["r"])
    both = np.concatenate([ei, ei[::-1]], axis=1)
    ranker = gb.PairRanker(_t(both), _t(np.concatenate([et, et])), p["n"], p["r"], filter=filt)
    got = ranker.ranks(p["zt"], p["wt"])
    assert torch.equal(_bits(got[:e]), _bits(got[e:]))
    got = got[:e].cpu().numpy()
    assert np.isnan(got[ei[0] == ei[1]]).all() and not np.isnan(got[ei[0] != ei[1]]).any()
    sample = np.random.RandomState(2).choice(e, n_sample, replace=False)
    sei, set_ = ei[:, sample], et[sample]
    scale = np.array([np.abs(opair.pair_scores(p["z"], p["w"], rr)).max() for rr in set_])
    lo, hi = opr.filtered_pair_ranks(p["z"], p["w"], sei, set_, p["lists"], tol=1e-5 * scale)
    g = got[sample]
    ok = ~np.isnan(lo)
    assert ((g[ok] >= lo[ok]) & (g[ok] <= hi[ok])).all()
    assert np.isnan(g[~ok]).all()


def test_pose0_sampled_triples_in_oracle_band(pose0):
    _check_pose(pose0, 48)


def test_pose2_sampled_triples_in_oracle_band(pose2):
    _check_pose(pose2, 24)


def test_determinism_and_cuda_graph_replay(pose0):
    import gripnet_b200 as gb
    p = pose0
    ei, et = p["test"]
    filt = gb.EdgeFilter(_lists_t(p["lists"]), p["n"], p["r"])
    ranker = gb.PairRanker(_t(ei), _t(et), p["n"], p["r"], filter=filt)
    first = ranker.ranks(p["zt"], p["wt"]).clone()
    assert torch.equal(_bits(first), _bits(ranker.ranks(p["zt"], p["wt"])))
    hits = (1, 10, 100)
    m_first = ranker.metrics(p["zt"], p["wt"], hits=hits)
    assert torch.equal(_bits(m_first), _bits(ranker.metrics(p["zt"], p["wt"], hits=hits)))
    zbuf = p["zt"].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ranker.metrics(zbuf, p["wt"], hits=hits)                                  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        rec = ranker.metrics(zbuf, p["wt"], hits=hits)
    zbuf.mul_(-0.5).add_(0.01)                                                    # new embeddings, same buffer
    graph.replay()
    torch.cuda.synchronize()
    eager = ranker.metrics(zbuf.clone(), p["wt"], hits=hits)
    assert torch.equal(_bits(rec), _bits(eager))
    assert not torch.equal(_bits(rec), _bits(m_first))


def test_input_checks():
    import gripnet_b200 as gb
    n, r = 40, 6
    z, w, lists = _integer_fixture(1, n, 7, r)
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    ei, et = _t([[0, 1], [2, 3]]), _t([0, 5])
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    ranker = gb.PairRanker(ei, et, n, r, filter=filt)
    assert ranker.ranks(zt, wt).shape == (2,)
    empty = gb.PairRanker(_t(np.zeros((2, 0))), _t(np.zeros(0)), n, r, filter=filt)
    assert empty.ranks(zt, wt).shape == (0,) and empty.n_groups == 0
    with pytest.raises(RuntimeError):
        ranker.ranks(zt.cpu(), wt.cpu())                                          # wrong device
    with pytest.raises(RuntimeError):
        gb.PairRanker(ei.cpu(), et.cpu(), n, r)                                   # CPU triples
    with pytest.raises(RuntimeError):
        gb.PairRanker(ei, et, 46341, r)                                           # 46341^2 >= 2^31
    with pytest.raises(RuntimeError):
        gb.PairRanker(ei, et, n, r, filter=gb.EdgeFilter(_lists_t(lists), n, r + 1))   # filter of another graph
    with pytest.raises(RuntimeError):
        gb.PairRanker(ei, et, n + 1, r, filter=filt)                              # node count of another graph
    with pytest.raises(IndexError):
        gb.PairRanker(ei, _t([0, r]), n, r)                                       # relation out of range
    with pytest.raises(RuntimeError):
        ranker.ranks(zt[:-1], wt)                                                 # z of another graph
    for bad in (torch.empty(3, device=zt.device), torch.empty(2, dtype=torch.float64, device=zt.device),
                torch.empty(4, device=zt.device)[::2], torch.empty(2)):
        with pytest.raises(RuntimeError):
            ranker.ranks(zt, wt, out=bad)                                         # bad out
    with pytest.raises(RuntimeError):
        ranker.metrics(zt, wt, out=torch.empty((4, r), device=zt.device))         # float32 metrics out
