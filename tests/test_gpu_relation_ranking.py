"""GPU: filtered relation ranking, per-relation MRR / Hits@k and top-k relations of a node pair
(gripnet_b200.RelationRanker, ranking.topk_relations) against the float64 oracle (oracle/relation_ranking.py)."""
import numpy as np
import pytest
import torch

from oracle import ranking as orank
from oracle import relation_ranking as orel

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _t(a, dtype=torch.int64):
    return torch.as_tensor(np.asarray(a), dtype=dtype, device=_dev())


def _lists_t(lists):
    return [(_t(ei), _t(et)) for ei, et in lists]


def _mirror(lst):
    return lst[0][::-1].copy(), lst[1]


def _integer_fixture(seed, n, r, e_test, e_train):
    """z in {-2..2}, w in {-1, 0, 1}: every fp32 score is an exact small integer on the FFMA and 3xTF32 paths.
    Relation r-1 has no query triple; a few pairs carry many filtered relations (padded top-k rows)."""
    rs = np.random.RandomState(seed)
    d = 16
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float32)
    w = rs.randint(-1, 2, size=(r, d)).astype(np.float32)
    test = (rs.randint(0, n, size=(2, e_test)), rs.randint(0, r - 1, size=e_test))
    train = (rs.randint(0, n, size=(2, e_train)), rs.randint(0, r, size=e_train))
    hubs = rs.randint(0, 5, size=4 * r)                                    # pairs of test edges 0..4, many relations
    dense = (test[0][:, hubs], rs.randint(0, r, size=hubs.size))
    train = (np.concatenate([train[0], dense[0], train[0][:, :50]], axis=1),
             np.concatenate([train[1], dense[1], train[1][:50]]))           # + duplicated triples
    return z, w, test, (train, test)


def _pose_split(g, seed=7):
    ei, et = g["dd_edge_index"].numpy(), g["dd_edge_type"].numpy()
    perm = np.random.RandomState(seed).permutation(ei.shape[1])
    cut = int(0.9 * perm.size)
    tr, te = np.sort(perm[:cut]), np.sort(perm[cut:])
    return (ei[:, tr], et[tr]), (ei[:, te], et[te])


def _delta(z, w, src, dst, chunk=4096):
    """1e-5 * max |S_row| of every pair's relation row (the fp32 ambiguity band)."""
    out = np.empty(len(src))
    for a in range(0, len(src), chunk):
        out[a:a + chunk] = 1e-5 * np.abs(orel.relation_scores(z, w, src[a:a + chunk], dst[a:a + chunk])).max(axis=1)
    return out


def _restrict(lists, src, dst, n):
    """The filter triples of the pairs (src, dst) only (the oracle reads no other pair)."""
    keys = np.unique(np.asarray(src, dtype=np.int64) * n + dst)
    out = []
    for ei, et in lists:
        keep = np.isin(ei[0].astype(np.int64) * n + ei[1], keys)
        out.append((ei[:, keep], et[keep]))
    return out


@pytest.mark.parametrize("n,r,e_test,k_list", [(40, 7, 300, (1, 3, 7, 10)),          # FFMA products
                                               (200, 31, 20000, (1, 10, 31, 40))])   # >= 4096 pairs: 3xTF32
def test_exact_integer_fixture(n, r, e_test, k_list):
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    z, w, test, lists = _integer_fixture(0, n, r, e_test, 3 * e_test)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    ranker = gb.RelationRanker(_t(test[0]), _t(test[1]), n, r, filter=filt)
    assert (ranker.n_groups >= 4096) == (e_test > 4096)
    assert ranker.n_groups == np.unique(test[0][0] * n + test[0][1]).size
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    got = ranker.ranks(zt, wt).cpu().numpy()
    want = orel.filtered_relation_ranks(z, w, *test, lists)
    np.testing.assert_array_equal(got, want)
    m = ranker.metrics(zt, wt, hits=(1, 3, 10)).cpu().numpy()
    mw = orank.rank_metrics(want, test[1], r, hits=(1, 3, 10))
    np.testing.assert_array_equal(m[1:], mw[1:])                          # Hits@k: exact counts
    np.testing.assert_allclose(m[0], mw[0], rtol=1e-14, atol=0)           # MRR: float64 sums in another order
    assert np.isnan(m[:, r - 1]).all()                                    # the relation without query triples
    raw = gb.RelationRanker(_t(test[0]), _t(test[1]), n, r).ranks(zt, wt).cpu().numpy()
    np.testing.assert_array_equal(raw, orel.filtered_relation_ranks(z, w, *test))
    src, dst = test[0]                                                    # >= 4096 rows: 3xTF32 in the second case
    for k in k_list:                                                      # k >= R - |filter row|: padded rows
        s, ids = ranking.topk_relations(zt, wt, _t(src), _t(dst), k, filter=filt, sigmoid=False)
        ws_, wi = orel.topk_relations(z, w, src, dst, k, lists)
        np.testing.assert_array_equal(ids.cpu().numpy(), wi)
        np.testing.assert_array_equal(s.cpu().numpy(), ws_.astype(np.float32))
    assert (ids.cpu().numpy() == -1).any()
    # sigmoid on the returned scores only; unfiltered selection
    s, ids = ranking.topk_relations(zt, wt, _t(src), _t(dst), 5)
    ws_, wi = orel.topk_relations(z, w, src, dst, 5)
    np.testing.assert_array_equal(ids.cpu().numpy(), wi)
    np.testing.assert_allclose(s.cpu().numpy(), 1.0 / (1.0 + np.exp(-ws_)), rtol=1e-6)


def test_hand_example_on_device():
    """The hand-worked example of the CPU oracle test (D = 1: the FFMA product), literal ranks and top-k."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    from test_relation_ranking_oracle import (HREL_FILTER, HREL_PAIRS, HREL_RANKS, HREL_RAW_RANKS, HREL_TEST,
                                              HREL_TOPK_IDS, HREL_TOPK_SCORES, HREL_W, HREL_Z)
    zt, wt = _t(HREL_Z, torch.float32), _t(HREL_W, torch.float32)
    filt = gb.EdgeFilter(_lists_t(HREL_FILTER), 4, 5)
    ranker = gb.RelationRanker(_t(HREL_TEST[0]), _t(HREL_TEST[1]), 4, 5, filter=filt)
    assert ranker.n_groups == 3
    assert ranker.ranks(zt, wt).cpu().tolist() == HREL_RANKS
    assert gb.RelationRanker(_t(HREL_TEST[0]), _t(HREL_TEST[1]), 4, 5).ranks(zt, wt).cpu().tolist() == HREL_RAW_RANKS
    m = ranker.metrics(zt, wt, hits=(1, 3)).cpu().numpy()
    np.testing.assert_allclose(m[:, :4], [[0.5, 2 / 3, 2 / 7, 1.0], [0, 0, 0, 1], [1, 1, 0, 1]], rtol=0, atol=1e-15)
    assert np.isnan(m[:, 4]).all()
    s, ids = ranking.topk_relations(zt, wt, *HREL_PAIRS, 6, filter=filt, sigmoid=False)
    assert ids.cpu().tolist() == HREL_TOPK_IDS
    for q, want in enumerate(HREL_TOPK_SCORES):
        assert s[q, :len(want)].cpu().tolist() == want and torch.isnan(s[q, len(want):]).all()
    s, ids = ranking.topk_relations(zt, wt[:1], [0], [1], 3, sigmoid=False)    # R = 1, k > R
    assert ids.cpu().tolist() == [[0, -1, -1]] and s[0, 0].item() == 2.0 and torch.isnan(s[0, 1:]).all()
    r1 = gb.RelationRanker(_t([[0, 2], [1, 2]]), _t([0, 0]), 4, 1)
    assert r1.ranks(zt, wt[:1]).cpu().tolist() == [1.0, 1.0]


def _pose(graph_fn):
    import gripnet_b200 as gb
    g = graph_fn()
    train, test = _pose_split(g)
    n, r, d = g["n_d"], g["n_rel"], 80
    rs = np.random.RandomState(3)
    z = (rs.randn(n, d) / np.sqrt(d)).astype(np.float32)
    w = rs.randn(r, d).astype(np.float32)
    lists = (train, test)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    ranker = gb.RelationRanker(_t(test[0]), _t(test[1]), n, r, filter=filt)
    return dict(z=z, w=w, test=test, lists=lists, filt=filt, ranker=ranker, n=n, r=r,
                zt=_t(z, torch.float32), wt=_t(w, torch.float32))


@pytest.fixture(scope="module")
def pose0():
    """pose-0 shape (n = 645, R = 16, 400 k directed edges), D = 80, 90/10 split, filter = train + test."""
    import synthdata
    return _pose(synthdata.pose_graph)


@pytest.fixture(scope="module")
def pose2():
    """pose-2 shape (n = 645, R = 1 097, 8.3 M directed edges over 63 473 drug pairs), as pose0."""
    import synthdata
    return _pose(synthdata.pose2_graph)


def _check_shape(p, n_sample, seed):
    """Ranks of a sample of the test triples inside the oracle's fp32 band; top-k (k = 10) of every test pair returns
    no filtered relation, is sorted, and its scores are the scores of the returned ids."""
    from gripnet_b200 import ranking
    z, w, n, r = p["z"], p["w"], p["n"], p["r"]
    test = p["test"]
    got = p["ranker"].ranks(p["zt"], p["wt"]).cpu().numpy().astype(np.float64)
    pick = np.sort(np.random.RandomState(seed).choice(test[1].size, n_sample, replace=False))
    sub = (test[0][:, pick], test[1][pick])
    lists = _restrict(p["lists"], sub[0][0], sub[0][1], n)
    lo, hi = orel.filtered_relation_ranks(z, w, *sub, lists, tol=_delta(z, w, sub[0][0], sub[0][1]))
    g = got[pick]
    assert (g >= lo).all() and (g <= hi).all(), np.nonzero((g < lo) | (g > hi))[0][:10]
    m = p["ranker"].metrics(p["zt"], p["wt"]).cpu().numpy()
    np.testing.assert_allclose(m, orank.rank_metrics(got, test[1], r), rtol=1e-12)
    # top-k over every distinct test pair
    keys = np.unique(test[0][0].astype(np.int64) * n + test[0][1])
    src, dst = keys // n, keys % n
    s, ids = ranking.topk_relations(p["zt"], p["wt"], _t(src), _t(dst), 10, filter=p["filt"], sigmoid=False)
    s, ids = s.cpu().numpy().astype(np.float64), ids.cpu().numpy()
    trip = np.concatenate([(ei[0].astype(np.int64) * n + ei[1]) * r + et for ei, et in p["lists"]])
    ok = ids >= 0
    assert not np.isin(((src * n + dst)[:, None] * r + ids)[ok], trip).any()      # no filtered relation returned
    assert (np.diff(np.where(ok, s, -np.inf), axis=1) <= 0).all()
    q = np.random.RandomState(seed + 1).choice(keys.size, 2000, replace=False)
    full = orel.relation_scores(z, w, src[q], dst[q])
    delta = _delta(z, w, src[q], dst[q])[:, None]
    sq, iq, okq = s[q], ids[q], ok[q]
    assert (np.abs(sq - np.take_along_axis(full, np.maximum(iq, 0), axis=1))[okq] <=
            np.broadcast_to(delta + 1e-30, sq.shape)[okq]).all()
    ws_, wi = orel.topk_relations(z, w, src[q], dst[q], 10, _restrict(p["lists"], src[q], dst[q], n))
    np.testing.assert_array_equal(wi == -1, ~okq)
    some = okq.any(axis=1)
    last = np.where(okq, sq, np.inf).min(axis=1)[some]
    assert (last >= np.nanmin(ws_[some], axis=1) - delta[some, 0]).all()
    return got


def test_pose0_ranks_within_fp32_band(pose0):
    assert pose0["ranker"].n_groups >= 4096                                # one chunk on the tensor cores
    _check_shape(pose0, 4000, 0)


def test_pose0_ranks_run_on_tensor_cores_and_the_shared_count(pose0):
    """One chunk of pair rows: one query-row launch, the product on gn_tc_gemm, one launch of the count kernel that
    tail queries use too, and no filter lookup per call (each pair's filter row is found at construction)."""
    p = pose0
    assert p["filt"] is p["ranker"].filter and p["ranker"].n_groups >= 4096
    p["ranker"].ranks(p["zt"], p["wt"])
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        p["ranker"].ranks(p["zt"], p["wt"])
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("tc_gemm_kernel" in x for x in names), sorted(set(names))
    assert sum("rank_rows_kernel" in x for x in names) == 1, sorted(set(names))
    assert sum("rank_count_kernel" in x for x in names) == 1, sorted(set(names))
    assert not any("rank_lookup_kernel" in x or "rank_rel_pairs" in x for x in names), sorted(set(names))


def test_pose2_ranks_within_fp32_band(pose2):
    """1 097-wide rows: several chunks, and top-k radix selection over more than 256 admissible relations."""
    from gripnet_b200 import ranking
    lds, rows = ranking._chunk_rows(pose2["r"], pose2["ranker"].n_groups)
    assert lds == 1100 and rows < pose2["ranker"].n_groups
    _check_shape(pose2, 3000, 1)


def test_pose0_mirror_pairs_rank_alike(pose0):
    """(s, t) and (t, s) have bitwise equal rows P, the same product path (one chunk) and, under a symmetric filter,
    the same filtered relations: each test triple and its mirror get identical ranks."""
    import gripnet_b200 as gb
    p = pose0
    test, mir = p["test"], _mirror(p["test"])
    both = (np.concatenate([test[0], mir[0]], axis=1), np.concatenate([test[1], mir[1]]))
    filt = gb.EdgeFilter(_lists_t(p["lists"] + (mir,)), p["n"], p["r"])
    ranker = gb.RelationRanker(_t(both[0]), _t(both[1]), p["n"], p["r"], filter=filt)
    from gripnet_b200 import ranking
    assert ranking._chunk_rows(p["r"], ranker.n_groups)[1] >= ranker.n_groups
    got = ranker.ranks(p["zt"], p["wt"]).cpu().numpy()
    e = test[1].size
    np.testing.assert_array_equal(got[:e], got[e:])


def test_chunking_matches_one_chunk(pose0, monkeypatch):
    """Four chunks of >= 4096 pairs each (the same tensor-core product path) give the ranks and top-k of one."""
    from gripnet_b200 import ranking
    p = pose0
    one = p["ranker"].ranks(p["zt"], p["wt"]).clone()
    src, dst = _t(p["test"][0][0][:20000]), _t(p["test"][0][1][:20000])
    s1, i1 = ranking.topk_relations(p["zt"], p["wt"], src, dst, 10, filter=p["filt"])
    g = p["ranker"].n_groups
    lds, _ = ranking._chunk_rows(p["r"], g)
    monkeypatch.setattr(ranking, "CHUNK_BYTES", 4 * lds * ((g + 3) // 4))
    assert ranking._chunk_rows(p["r"], g)[1] < g and g - 3 * ((g + 3) // 4) >= 4096
    assert torch.equal(p["ranker"].ranks(p["zt"], p["wt"]), one)
    monkeypatch.setattr(ranking, "CHUNK_BYTES", 4 * lds * 5000)
    s4, i4 = ranking.topk_relations(p["zt"], p["wt"], src, dst, 10, filter=p["filt"])
    assert torch.equal(i4, i1)
    torch.testing.assert_close(s4, s1, rtol=0, atol=0, equal_nan=True)


def test_metrics_capture_and_determinism(pose0):
    p = pose0
    zt, wt = p["zt"], p["wt"]
    ranker = p["ranker"]
    a = ranker.metrics(zt, wt).clone()
    b = ranker.metrics(zt, wt).clone()
    assert torch.equal(a, b)
    zbuf = zt.clone()
    rec = torch.empty_like(a)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ranker.metrics(zbuf, wt, out=rec)                               # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ranker.metrics(zbuf, wt, out=rec)
    zbuf.mul_(-0.5).add_(0.01)                                           # new embeddings, same buffer
    graph.replay()
    torch.cuda.synchronize()
    eager = ranker.metrics(zbuf.clone(), wt)
    assert torch.equal(rec, eager)
    assert not torch.equal(rec, a)


def test_decoder_topk_relations(pose0):
    from gripnet_b200 import multiRelaInnerProductDecoder, ranking
    p = pose0
    dec = multiRelaInnerProductDecoder(p["z"].shape[1], p["r"]).to(_dev())
    with torch.no_grad():
        dec.weight.copy_(p["wt"])
    src, dst = _t(p["test"][0][0][:500]), _t(p["test"][0][1][:500])
    s, ids = dec.topk_relations(p["zt"], src, dst, 8, filter=p["filt"])
    s0, ids0 = ranking.topk_relations(p["zt"], p["wt"], src, dst, 8, filter=p["filt"], sigmoid=False)
    assert torch.equal(ids, ids0)
    torch.testing.assert_close(s, torch.sigmoid(s0), rtol=1e-6, atol=0, equal_nan=True)


def test_empty_queries_and_input_checks():
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    z, w, test, lists = _integer_fixture(1, 40, 6, 200, 400)
    n, r = z.shape[0], w.shape[0]
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    empty = gb.RelationRanker(_t(np.zeros((2, 0))), _t(np.zeros(0)), n, r, filter=filt)
    assert empty.n_groups == 0 and empty.ranks(zt, wt).numel() == 0
    assert torch.isnan(empty.metrics(zt, wt)).all()
    s, ids = ranking.topk_relations(zt, wt, _t(np.zeros(0)), _t(np.zeros(0)), 4, filter=filt)
    assert s.shape == (0, 4) and ids.shape == (0, 4)
    with pytest.raises(IndexError):
        gb.RelationRanker(_t([[0, n], [1, 2]]), _t([0, 0]), n, r)
    with pytest.raises(IndexError):
        gb.RelationRanker(_t([[0], [1]]), _t([r]), n, r)
    with pytest.raises(RuntimeError):
        gb.RelationRanker(_t([[0, 1, 2]]), _t([0, 0, 0]), n, r)                    # edge_index not [2, E]
    with pytest.raises(RuntimeError):
        gb.RelationRanker(_t([[0, 1], [1, 2]]), _t([0]), n, r)                    # edge_type not [E]
    with pytest.raises(RuntimeError):
        gb.RelationRanker(torch.as_tensor(test[0]), torch.as_tensor(test[1]), n, r)   # CPU tensors
    with pytest.raises(IndexError):
        ranking.topk_relations(zt, wt, _t([0, n]), _t([0, 0]), 3)
    with pytest.raises(IndexError):
        ranking.topk_relations(zt, wt, _t([0]), _t([-1]), 3)
    with pytest.raises(RuntimeError):
        ranking.topk_relations(zt, wt, _t([0, 1]), _t([0]), 3)                     # unequal lengths
    with pytest.raises(RuntimeError):
        ranking.topk_relations(zt, wt, _t([0], torch.int32), _t([0], torch.int32), 3)
    with pytest.raises(RuntimeError):
        ranking.topk_relations(zt.cpu(), wt.cpu(), [0], [0], 3)
    for k in (0, 257, 2.5):
        with pytest.raises(RuntimeError):
            ranking.topk_relations(zt, wt, _t([0]), _t([0]), k)
    other = gb.EdgeFilter(_lists_t(lists), n, r + 1)
    with pytest.raises(RuntimeError):
        gb.RelationRanker(_t(test[0]), _t(test[1]), n, r, filter=other)           # filter of another graph
    with pytest.raises(RuntimeError):
        ranking.topk_relations(zt, wt, _t([0]), _t([1]), 3, filter=other)
    ranker = gb.RelationRanker(_t(test[0]), _t(test[1]), n, r, filter=filt)
    with pytest.raises(RuntimeError):
        ranker.ranks(zt, wt[:, :-1])                                    # D mismatch
    with pytest.raises(RuntimeError):
        ranker.ranks(zt[:-1], wt)                                       # node count
    with pytest.raises(RuntimeError):
        ranker.ranks(zt, wt[:-1])                                       # relation count
    with pytest.raises(RuntimeError):
        ranker.metrics(zt, wt, hits=tuple(range(1, 11)))                # more thresholds than the kernel takes
