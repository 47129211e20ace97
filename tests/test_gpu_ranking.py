"""GPU: filtered candidate ranking, per-relation MRR / Hits@k and top-k of the DistMult decoder (gripnet_b200.ranking)
against the float64 oracle (oracle/ranking.py)."""
import numpy as np
import pytest
import torch

from oracle import ranking as orank

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _t(a, dtype=torch.int64):
    return torch.as_tensor(np.asarray(a), dtype=dtype, device=_dev())


def _lists_t(lists):
    return [(_t(ei), _t(et)) for ei, et in lists]


def _integer_fixture(seed, n=40, d=16, r=4, e_test=300, e_train=900):
    """z in {-2..2}, w in {-1, 0, 1}: every fp32 score is an exact small integer on the FFMA and 3xTF32 paths."""
    rs = np.random.RandomState(seed)
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float32)
    w = rs.randint(-1, 2, size=(r, d)).astype(np.float32)
    test = (rs.randint(0, n, size=(2, e_test)), rs.randint(0, r - 1, size=e_test))      # relation r-1: no test edge
    train = (rs.randint(0, n, size=(2, e_train)), rs.randint(0, r, size=e_train))
    train = (np.concatenate([train[0], train[0][:, :50]], axis=1), np.concatenate([train[1], train[1][:50]]))  # dups
    return z, w, test, (train, test)


def _pose_split(g, seed=7):
    ei, et = g["dd_edge_index"].numpy(), g["dd_edge_type"].numpy()
    perm = np.random.RandomState(seed).permutation(ei.shape[1])
    cut = int(0.9 * perm.size)
    tr, te = np.sort(perm[:cut]), np.sort(perm[cut:])
    return (ei[:, tr], et[tr]), (ei[:, te], et[te])


def _delta(z, w, node, rel, chunk=4096):
    """1e-5 * max |S_row| of every query row (the fp32 ambiguity band)."""
    out = np.empty(len(node))
    for a in range(0, len(node), chunk):
        out[a:a + chunk] = 1e-5 * np.abs(orank.scores(z, w, node[a:a + chunk], rel[a:a + chunk])).max(axis=1)
    return out


def _check_band(got, z, w, test, lists):
    lo, hi = orank.filtered_ranks(z, w, *test, lists, tol=_delta(z, w, test[0][0], test[1]))
    assert (got >= lo).all() and (got <= hi).all(), np.nonzero((got < lo) | (got > hi))[0][:10]


@pytest.mark.parametrize("n,r,e_test,n_q", [(40, 4, 300, 120),          # FFMA products
                                             (200, 31, 20000, 5000)])    # >= 4096 rows a chunk: 3xTF32 products
def test_exact_integer_fixture(n, r, e_test, n_q):
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    z, w, test, lists = _integer_fixture(0, n=n, r=r, e_test=e_test, e_train=3 * e_test)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    ranker = gb.LinkRanker(_t(test[0]), _t(test[1]), n, r, filter=filt)
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    got = ranker.ranks(zt, wt).cpu().numpy()
    want = orank.filtered_ranks(z, w, *test, lists)
    np.testing.assert_array_equal(got, want)
    m = ranker.metrics(zt, wt, hits=(1, 3, 10)).cpu().numpy()
    mw = orank.rank_metrics(want, test[1], r, hits=(1, 3, 10))
    np.testing.assert_array_equal(m[1:], mw[1:])                          # Hits@k: exact counts
    np.testing.assert_allclose(m[0], mw[0], rtol=1e-14, atol=0)           # MRR: float64 sums in another order
    assert np.isnan(m[:, r - 1]).all()                                    # the relation without edges
    node, rel = test[0][0][:n_q], test[1][:n_q]
    for k in (1, 7, n - 2):                                               # n - 2 > n - |filter row|: padded rows
        s, ids = ranking.topk(zt, wt, _t(node), _t(rel), k, filter=filt, sigmoid=False)
        ws_, wi = orank.topk(z, w, node, rel, k, lists)
        np.testing.assert_array_equal(ids.cpu().numpy(), wi)
        np.testing.assert_array_equal(s.cpu().numpy(), ws_.astype(np.float32))
    assert (ids.cpu().numpy() == -1).any()
    # sigmoid on the returned scores only; unfiltered selection
    s, ids = ranking.topk(zt, wt, _t(node), _t(rel), 5)
    ws_, wi = orank.topk(z, w, node, rel, 5)
    np.testing.assert_array_equal(ids.cpu().numpy(), wi)
    np.testing.assert_allclose(s.cpu().numpy(), 1.0 / (1.0 + np.exp(-ws_)), rtol=1e-6)


def test_hand_example_on_device():
    """The hand-worked example of the CPU oracle test (D = 1: the FFMA product), literal ranks and top-k."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    from test_ranking_oracle import HAND_FILTER, HAND_RANKS, HAND_RAW_RANKS, HAND_TEST, HAND_W, HAND_Z
    zt, wt = _t(HAND_Z, torch.float32), _t(HAND_W, torch.float32)
    filt = gb.EdgeFilter(_lists_t(HAND_FILTER), 5, 3)
    got = gb.LinkRanker(_t(HAND_TEST[0]), _t(HAND_TEST[1]), 5, 3, filter=filt).ranks(zt, wt)
    assert got.cpu().tolist() == HAND_RANKS
    assert gb.LinkRanker(_t(HAND_TEST[0]), _t(HAND_TEST[1]), 5, 3).ranks(zt, wt).cpu().tolist() == HAND_RAW_RANKS
    s, ids = ranking.topk(zt, wt, [0, 2, 4], [0, 1, 0], 4, filter=filt, sigmoid=False)
    assert ids.cpu().tolist() == [[0, 2, 4, -1], [4, 2, 0, 3], [1, 2, 3, 4]]
    assert s[1].cpu().tolist() == [0.0, -1.0, -2.0, -3.0] and torch.isnan(s[0, 3])


@pytest.fixture(scope="module")
def pose0():
    """pose-0 shape (n = 645, R = 16, 400 k directed edges), D = 80, 90/10 split, filter = train + test."""
    import gripnet_b200 as gb
    import synthdata
    g = synthdata.pose_graph()
    train, test = _pose_split(g)
    n, r, d = g["n_d"], g["n_rel"], 80
    rs = np.random.RandomState(3)
    z = (rs.randn(n, d) / np.sqrt(d)).astype(np.float32)
    w = rs.randn(r, d).astype(np.float32)
    lists = (train, test)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    ranker = gb.LinkRanker(_t(test[0]), _t(test[1]), n, r, filter=filt)
    return dict(z=z, w=w, test=test, lists=lists, filt=filt, ranker=ranker, n=n, r=r)


def test_pose0_ranks_within_fp32_band(pose0):
    p = pose0
    zt, wt = _t(p["z"], torch.float32), _t(p["w"], torch.float32)
    assert p["ranker"].n_groups >= 4096
    got = p["ranker"].ranks(zt, wt).cpu().numpy().astype(np.float64)
    _check_band(got, p["z"], p["w"], p["test"], p["lists"])
    m = p["ranker"].metrics(zt, wt).cpu().numpy()
    np.testing.assert_allclose(m, orank.rank_metrics(got, p["test"][1], p["r"]), rtol=1e-12)


def test_pose0_product_runs_on_tensor_cores(pose0):
    """A chunk of >= 4096 query rows goes through gn_tc_gemm (kernel names of the profiler's launch list)."""
    p = pose0
    zt, wt = _t(p["z"], torch.float32), _t(p["w"], torch.float32)
    p["ranker"].ranks(zt, wt)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        p["ranker"].ranks(zt, wt)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("tc_gemm_kernel" in x for x in names), sorted(set(names))
    assert any("rank_count_kernel" in x for x in names)


def test_pose0_topk(pose0):
    from gripnet_b200 import ranking
    p = pose0
    z, w = p["z"], p["w"]
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    node, rel = p["test"][0][0][:3000], p["test"][1][:3000]
    k = 10
    s, ids = ranking.topk(zt, wt, _t(node), _t(rel), k, filter=p["filt"], sigmoid=False)
    s, ids = s.cpu().numpy().astype(np.float64), ids.cpu().numpy()
    ws_, wi = orank.topk(z, w, node, rel, k, p["lists"])
    delta = _delta(z, w, node, rel)[:, None]
    assert (ids >= 0).all()                                              # 645 candidates: no row is padded
    assert (np.diff(s, axis=1) <= 0).all()
    full = orank.scores(z, w, node, rel)
    assert (np.abs(s - np.take_along_axis(full, ids, axis=1)) <= delta + 1e-30).all()   # scores of the returned ids
    assert (s[:, -1] >= ws_[:, -1] - delta[:, 0]).all()
    fidx = orank.filter_index(p["lists"])
    for q in range(len(node)):
        f = fidx.get((int(node[q]), int(rel[q])))
        if f is not None:
            assert not np.isin(ids[q], f).any()
    # the decoder method: the same selection with its own weight, sigmoid applied
    from gripnet_b200 import multiRelaInnerProductDecoder
    dec = multiRelaInnerProductDecoder(z.shape[1], p["r"]).to(_dev())
    with torch.no_grad():
        dec.weight.copy_(wt)
    s2, ids2 = dec.topk(zt, _t(node), _t(rel), k, filter=p["filt"])
    assert torch.equal(ids2.cpu(), torch.from_numpy(ids))
    np.testing.assert_allclose(s2.cpu().numpy(), 1.0 / (1.0 + np.exp(-s)), rtol=1e-6)


def test_long_rows_strided_and_odd_widths():
    """n = 50 000 (a row does not fit shared memory), D = 32 from a column slice of a wider buffer; D = 30."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    rs = np.random.RandomState(11)
    for n, d, strided in ((50000, 32, True), (3000, 30, False), (700, 30, True)):
        r = 3
        big = rs.randn(n, d + 12).astype(np.float32)
        z = big[:, 5:5 + d] if strided else big[:, :d].copy()
        w = rs.randn(r, d).astype(np.float32)
        e = 300
        test = (rs.randint(0, n, size=(2, e)), rs.randint(0, r, size=e))
        hubs = rs.randint(0, 4, size=4000)                  # a few (s, r) rows with long filter rows
        train = (np.stack([test[0][0][hubs], rs.randint(0, n, size=4000)]), test[1][hubs])
        lists = (train, test)
        zt_big = _t(big, torch.float32)
        zt = zt_big[:, 5:5 + d] if strided else zt_big[:, :d].contiguous()
        wt = _t(w, torch.float32)
        filt = gb.EdgeFilter(_lists_t(lists), n, r)
        got = gb.LinkRanker(_t(test[0]), _t(test[1]), n, r, filter=filt).ranks(zt, wt).cpu().numpy()
        _check_band(got.astype(np.float64), z, w, test, lists)
        node, rel = test[0][0][:40], test[1][:40]
        s, ids = ranking.topk(zt, wt, _t(node), _t(rel), 256, filter=filt, sigmoid=False)
        ws_, wi = orank.topk(z, w, node, rel, 256, lists)
        delta = _delta(z, w, node, rel)[:, None]
        s, ids = s.cpu().numpy().astype(np.float64), ids.cpu().numpy()
        pad = wi == -1                                      # rows whose filter leaves fewer than 256 candidates
        np.testing.assert_array_equal(ids == -1, pad)
        assert np.isnan(s[pad]).all()
        s, ws_ = np.where(pad, -1e30, s), np.where(pad, -1e30, ws_)
        assert (np.diff(s, axis=1) <= 0).all()
        ok = ~pad
        assert (np.abs(s - ws_)[ok] <= np.broadcast_to(2 * delta + 1e-30, s.shape)[ok]).all()


def test_empty_relation_and_no_queries():
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    z, w, test, lists = _integer_fixture(1)
    n, r = z.shape[0], w.shape[0]
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    empty = gb.LinkRanker(_t(np.zeros((2, 0))), _t(np.zeros(0)), n, r)
    assert empty.ranks(zt, wt).numel() == 0
    assert torch.isnan(empty.metrics(zt, wt)).all()
    s, ids = ranking.topk(zt, wt, _t(np.zeros(0)), _t(np.zeros(0)), 4)
    assert s.shape == (0, 4) and ids.shape == (0, 4)


def test_metrics_capture_and_determinism(pose0):
    p = pose0
    zt, wt = _t(p["z"], torch.float32), _t(p["w"], torch.float32)
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


def test_input_checks():
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    z, w, test, lists = _integer_fixture(2)
    n, r = z.shape[0], w.shape[0]
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    with pytest.raises(IndexError):
        gb.LinkRanker(_t([[0, n], [1, 2]]), _t([0, 0]), n, r)
    with pytest.raises(IndexError):
        gb.EdgeFilter([(_t([[0], [1]]), _t([r]))], n, r)
    with pytest.raises(IndexError):
        ranking.topk(zt, wt, _t([0, n]), _t([0, 0]), 3)
    with pytest.raises(IndexError):
        ranking.topk(zt, wt, _t([0]), _t([-1]), 3)
    with pytest.raises(RuntimeError):
        gb.LinkRanker(torch.as_tensor(test[0]), torch.as_tensor(test[1]), n, r)      # CPU tensors
    with pytest.raises(RuntimeError):
        ranking.topk(zt.cpu(), wt.cpu(), [0], [0], 3)
    for k in (0, 257, 2.5):
        with pytest.raises(RuntimeError):
            ranking.topk(zt, wt, _t([0]), _t([0]), k)
    ranker = gb.LinkRanker(_t(test[0]), _t(test[1]), n, r)
    with pytest.raises(RuntimeError):
        ranker.ranks(zt, wt[:, :-1])                                    # D mismatch
    with pytest.raises(RuntimeError):
        ranking.topk(zt, wt[:, :-1], _t([0]), _t([0]), 3)
    with pytest.raises(RuntimeError):
        ranker.ranks(zt[:-1], wt)                                       # node count
    with pytest.raises(RuntimeError):
        ranker.metrics(zt, wt, hits=tuple(range(1, 11)))                # more thresholds than the kernel takes
