"""GPU: top-k new pairs of a relation (gripnet_b200.ranking.topk_pairs, multiRelaInnerProductDecoder.topk_pairs)
against the float64 oracle (oracle/pair_ranking.py)."""
import numpy as np
import pytest
import torch

from oracle import pair_ranking as opair

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _t(a, dtype=torch.int64):
    return torch.as_tensor(np.asarray(a), dtype=dtype, device=_dev())


def _lists_t(lists):
    return [(_t(ei), _t(et)) for ei, et in lists]


def _strided(z):
    """z as a row view of a wider buffer (row stride D + 5)."""
    n, d = z.shape
    buf = torch.full((n, d + 5), float("nan"), dtype=torch.float32, device=_dev())
    buf[:, 2:2 + d] = _t(z, torch.float32)
    return buf[:, 2:2 + d]


def _integer_fixture(seed, n, d, r):
    """z in {-2..2}, w in {-1, 0, 1}: every fp32 score is an exact small integer (many exact ties).  The filter
    holds random triples in one direction and, for relation 0, a few pairs only in the flipped direction."""
    rs = np.random.RandomState(seed)
    z = rs.randint(-2, 3, size=(n, d)).astype(np.float32)
    w = rs.randint(-1, 2, size=(r, d)).astype(np.float32)
    e = max(4, n * 3)
    train = (rs.randint(0, n, size=(2, e)), rs.randint(0, r, size=e))
    flip = rs.randint(0, n, size=(2, 8))
    lists = (train, (np.concatenate([flip, flip[:, :2]], axis=1), np.zeros(10, dtype=np.int64)))
    return z, w, lists


def _assert_exact(got, want):
    s, a, b = (x.cpu().numpy() for x in got)
    ws_, wa, wb = want
    np.testing.assert_array_equal(a, wa)
    np.testing.assert_array_equal(b, wb)
    np.testing.assert_array_equal(s, ws_.astype(np.float32))


@pytest.mark.parametrize("n,d,k", [(2, 1, 1), (3, 7, 7), (40, 7, 256), (40, 80, 7), (40, 1, 256),
                                   (700, 80, 256), (700, 1, 7), (700, 7, 1)])
def test_exact_integer_fixture(n, d, k):
    """Bit for bit against the oracle, ids and tie order included, on a strided z and duplicated relations."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    r = 3
    z, w, lists = _integer_fixture(n * 31 + d, n, d, r)
    zt, wt = _strided(z), _t(w, torch.float32)
    assert zt.stride(0) == d + 5
    rel = [0, 2, 1, 0]
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    got = ranking.topk_pairs(zt, wt, _t(rel), k, filter=filt, sigmoid=False)
    _assert_exact(got, opair.topk_pairs(z, w, rel, k, lists))
    s, a, b = (x.cpu().numpy() for x in got)
    ok = a >= 0
    assert (a[ok] < b[ok]).all() and np.array_equal(ok, b >= 0)
    for x in (s, a, b):
        np.testing.assert_array_equal(x[0], x[3])                    # duplicated query
    raw = ranking.topk_pairs(zt.contiguous(), wt, _t(rel), k, sigmoid=False)
    _assert_exact(raw, opair.topk_pairs(z, w, rel, k))


def test_all_scores_equal_give_the_smallest_pair_ids():
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    n, d, r, k = 150, 5, 2, 256
    z, w = np.ones((n, d), np.float32), np.ones((r, d), np.float32)
    filt_list = (np.array([[0, 3, 1], [5, 0, 2]]), np.array([1, 1, 0]))   # r = 1: {0,5}, {0,3}; r = 0: {1,2}
    filt = gb.EdgeFilter(_lists_t([filt_list]), n, r)
    s, a, b = ranking.topk_pairs(_t(z, torch.float32), _t(w, torch.float32), _t([1, 0]), k, filter=filt,
                                 sigmoid=False)
    su, tu = np.triu_indices(n, k=1)
    for q, drop in enumerate(({(0, 5), (0, 3)}, {(1, 2)})):
        keep = [(x, y) for x, y in zip(su.tolist(), tu.tolist()) if (x, y) not in drop][:k]
        assert list(zip(a[q].tolist(), b[q].tolist())) == keep
    assert (s == float(d)).all()


def test_scores_rising_along_rows_force_compactions():
    """S(s, t) = s * t: every tile of a row block beats all earlier ones, so every tile refills the candidate
    buffer and is cut again."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    n = 700
    z = np.stack([np.arange(n), np.ones(n)], axis=1).astype(np.float32)
    w = np.array([[1.0, 0.0], [-1.0, 0.0]], np.float32)
    lists = ((np.array([[699, 697], [698, 699]]), np.array([0, 0])),)     # the two best pairs of r = 0
    filt = gb.EdgeFilter(_lists_t(lists), n, 2)
    for k in (1, 100, 256):
        got = ranking.topk_pairs(_t(z, torch.float32), _t(w, torch.float32), _t([0, 1]), k, filter=filt,
                                 sigmoid=False)
        _assert_exact(got, opair.topk_pairs(z, w, [0, 1], k, lists))
    assert got[1][0, 0].item() == 697 and got[2][0, 0].item() == 698          # 697 * 698 > 696 * 699


def test_one_direction_filter_excludes_the_pair():
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    n, d, r, k = 60, 7, 2, 20
    rs = np.random.RandomState(5)
    z, w = rs.randn(n, d).astype(np.float32), rs.randn(r, d).astype(np.float32)
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    s0, a0, b0 = ranking.topk_pairs(zt, wt, _t([1]), k, sigmoid=False)
    x, y = int(a0[0, 0]), int(b0[0, 0])
    for trip in ((y, x), (x, y)):                                        # (t, r, s) alone, then (s, r, t) alone
        filt = gb.EdgeFilter(_lists_t([(np.array([[trip[0]], [trip[1]]]), np.array([1]))]), n, r)
        s1, a1, b1 = ranking.topk_pairs(zt, wt, _t([1]), k, filter=filt, sigmoid=False)
        assert torch.equal(a1[0, :k - 1], a0[0, 1:]) and torch.equal(b1[0, :k - 1], b0[0, 1:])
        assert torch.equal(s1[0, :k - 1], s0[0, 1:])


def test_padding():
    """k above the admissible pairs, and n < 2 (no pair at all)."""
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    from test_pair_ranking_oracle import HPAIR_DST, HPAIR_FILTER, HPAIR_REL, HPAIR_SCORES, HPAIR_SRC, HPAIR_W, HPAIR_Z
    zt, wt = _t(HPAIR_Z, torch.float32), _t(HPAIR_W, torch.float32)
    filt = gb.EdgeFilter(_lists_t(HPAIR_FILTER), 4, 2)
    s, a, b = ranking.topk_pairs(zt, wt, _t(HPAIR_REL), 6, filter=filt, sigmoid=False)
    assert a.cpu().tolist() == HPAIR_SRC and b.cpu().tolist() == HPAIR_DST
    for q, want in enumerate(HPAIR_SCORES):
        assert s[q, :len(want)].cpu().tolist() == want and torch.isnan(s[q, len(want):]).all()
    s, a, b = ranking.topk_pairs(zt[:1], wt, _t([0, 1]), 5)
    assert (a == -1).all() and (b == -1).all() and torch.isnan(s).all()
    s, a, b = ranking.topk_pairs(zt[:2], wt, _t([1]), 3, sigmoid=True)
    assert a.cpu().tolist() == [[0, -1, -1]] and b.cpu().tolist() == [[1, -1, -1]]
    assert abs(s[0, 0].item() - 1.0 / (1.0 + np.exp(2.0))) < 1e-7 and torch.isnan(s[0, 1:]).all()


def _pose_split(g, seed=7):
    ei, et = g["dd_edge_index"].numpy(), g["dd_edge_type"].numpy()
    perm = np.random.RandomState(seed).permutation(ei.shape[1])
    cut = int(0.9 * perm.size)
    tr, te = np.sort(perm[:cut]), np.sort(perm[cut:])
    return (ei[:, tr], et[tr]), (ei[:, te], et[te])


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
    return dict(z=z, w=w, lists=lists, filt=filt, n=n, r=r, zt=_t(z, torch.float32), wt=_t(w, torch.float32))


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


def _check_tie_aware(p, rels, k):
    """Every slot admissible and distinct, src < dst, scores non-increasing and within the fp32 band of their exact
    value, and no admissible pair whose exact score beats the k-th by more than twice the band is missing."""
    from gripnet_b200 import ranking
    z, w, n = p["z"], p["w"], p["n"]
    s, a, b = ranking.topk_pairs(p["zt"], p["wt"], _t(rels), k, filter=p["filt"], sigmoid=False)
    s, a, b = s.cpu().numpy().astype(np.float64), a.cpu().numpy(), b.cpu().numpy()
    assert (a >= 0).all() and (a < b).all() and (b < n).all()
    assert (np.diff(s, axis=1) <= 0).all()
    su, tu = np.triu_indices(n, k=1)
    for q, r in enumerate(rels):
        exact = opair.pair_scores(z, w, r)
        adm = np.ones((n, n), dtype=bool)
        for ei, et in p["lists"]:
            sel = et == r
            adm[ei[0][sel], ei[1][sel]] = False
            adm[ei[1][sel], ei[0][sel]] = False
        delta = 1e-5 * np.abs(exact[su, tu]).max()
        assert adm[a[q], b[q]].all()                                         # nothing filtered returned
        assert np.unique(a[q] * n + b[q]).size == k                          # distinct
        assert (np.abs(s[q] - exact[a[q], b[q]]) <= delta).all()
        kth = exact[a[q, -1], b[q, -1]]
        must = (exact[su, tu] > kth + 2 * delta) & adm[su, tu]
        got = set((a[q] * n + b[q]).tolist())
        assert set((su[must] * n + tu[must]).tolist()) <= got


@pytest.mark.parametrize("k", [10, 100])
def test_pose0_all_relations_tie_aware(pose0, k):
    _check_tie_aware(pose0, list(range(pose0["r"])), k)


def test_pose2_sampled_relations_tie_aware(pose2):
    rels = np.sort(np.random.RandomState(11).choice(pose2["r"], 16, replace=False)).tolist()
    _check_tie_aware(pose2, rels, 10)
    _check_tie_aware(pose2, rels[:4], 100)


def test_determinism_and_cuda_graph_replay(pose0):
    from gripnet_b200 import ranking
    p = pose0
    rel = _t(np.arange(p["r"]))
    first = ranking.topk_pairs(p["zt"], p["wt"], rel, 50, filter=p["filt"])      # also builds the filter's view
    second = ranking.topk_pairs(p["zt"], p["wt"], rel, 50, filter=p["filt"])
    for x, y in zip(first, second):
        assert torch.equal(x, y)
    zbuf = p["zt"].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ranking.topk_pairs(zbuf, p["wt"], rel, 50, filter=p["filt"])            # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        rec = ranking.topk_pairs(zbuf, p["wt"], rel, 50, filter=p["filt"])
    zbuf.mul_(-0.5).add_(0.01)                                                  # new embeddings, same buffer
    graph.replay()
    torch.cuda.synchronize()
    eager = ranking.topk_pairs(zbuf.clone(), p["wt"], rel, 50, filter=p["filt"])
    for x, y in zip(rec, eager):
        assert torch.equal(x, y)
    assert not torch.equal(rec[0], first[0])


def test_decoder_topk_pairs(pose0):
    from gripnet_b200 import multiRelaInnerProductDecoder, ranking
    p = pose0
    dec = multiRelaInnerProductDecoder(p["z"].shape[1], p["r"]).to(_dev())
    with torch.no_grad():
        dec.weight.copy_(p["wt"])
    rel = _t([3, 0, 3, 15])
    s, a, b = dec.topk_pairs(p["zt"], rel, 8, filter=p["filt"])
    s0, a0, b0 = ranking.topk_pairs(p["zt"], p["wt"], rel, 8, filter=p["filt"], sigmoid=False)
    assert torch.equal(a, a0) and torch.equal(b, b0)
    torch.testing.assert_close(s, torch.sigmoid(s0), rtol=1e-6, atol=0)


def test_empty_queries_and_input_checks():
    import gripnet_b200 as gb
    from gripnet_b200 import ranking
    n, r = 40, 6
    z, w, lists = _integer_fixture(1, n, 7, r)
    zt, wt = _t(z, torch.float32), _t(w, torch.float32)
    filt = gb.EdgeFilter(_lists_t(lists), n, r)
    s, a, b = ranking.topk_pairs(zt, wt, _t(np.zeros(0)), 4, filter=filt)
    assert s.shape == (0, 4) and a.shape == (0, 4) and b.shape == (0, 4)
    for k in (0, 257, 2.5, True):
        with pytest.raises(RuntimeError):
            ranking.topk_pairs(zt, wt, _t([0]), k)
    with pytest.raises(IndexError):
        ranking.topk_pairs(zt, wt, _t([0, r]), 3)
    with pytest.raises(IndexError):
        ranking.topk_pairs(zt, wt, _t([-1]), 3)
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(zt, wt, _t([0], torch.int32), 3)
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(zt, wt[:, :-1], _t([0]), 3)                       # width mismatch
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(zt.cpu(), wt.cpu(), [0], 3)                       # CPU tensors
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(zt, wt, torch.zeros(1, dtype=torch.int64), 3)     # CPU query list
    big = torch.zeros((46341, 1), dtype=torch.float32, device=_dev())        # 46341^2 >= 2^31
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(big, wt[:, :1], _t([0]), 3)
    other = gb.EdgeFilter(_lists_t(lists), n, r + 1)
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(zt, wt, _t([0]), 3, filter=other)                 # filter of another graph
    with pytest.raises(RuntimeError):
        ranking.topk_pairs(zt[:-1], wt, _t([0]), 3, filter=filt)             # node count of another graph
