"""GPU: each C-ABI kernel against a float64 restatement of the same op on CPU.

Tolerance: 1e-5 relative (max|a-b| / max|b| per tensor) — north_star's fp32 bar.
"""
import numpy as np
import pytest
import torch

from golden_util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _dev():
    return torch.device("cuda:0")


def _rand_csr(rs, n_rows, n_cols, lens):
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    nnz = int(rowptr[-1])
    col = rs.randint(0, n_cols, size=nnz).astype(np.int32)
    val = rs.uniform(-1, 1, size=nnz).astype(np.float32)
    return rowptr, col, val


def _dense_ref(rowptr, col, val, x, n_rows):
    out = np.zeros((n_rows, x.shape[1]))
    rows = np.repeat(np.arange(n_rows), np.diff(rowptr))
    g = x[col].astype(np.float64)
    if val is not None:
        g = g * val[:, None].astype(np.float64)
    np.add.at(out, rows, g)
    return out


@pytest.mark.parametrize("F", [1, 3, 4, 16, 20, 32, 64, 80, 128, 200])
@pytest.mark.parametrize("chunk_len", [32, 256])
def test_spmm_widths_and_row_split(F, chunk_len):
    from gripnet_b200 import ops
    from gripnet_b200.graph import Csr
    rs = np.random.RandomState(F * 7 + chunk_len)
    n_rows, n_cols = 300, 500
    lens = rs.randint(0, 40, n_rows)
    lens[[3, 50, 299]] = [1500, 0, 700]                       # hub rows -> several chunks, one empty row
    rowptr, col, val = _rand_csr(rs, n_rows, n_cols, lens)
    x = rs.randn(n_cols, F).astype(np.float32)
    bias = rs.randn(F).astype(np.float32)
    scale = rs.uniform(0.5, 2, n_rows).astype(np.float32)
    add = rs.randn(n_rows, F).astype(np.float32)
    d = _dev()
    csr = Csr(torch.from_numpy(rowptr).to(d), torch.from_numpy(col).to(d), torch.from_numpy(val).to(d), n_rows,
              n_cols, len(col), chunk_len=chunk_len)
    xt, bt, st, at = (torch.from_numpy(a).to(d) for a in (x, bias, scale, add))
    ref = _dense_ref(rowptr, col, val, x, n_rows)
    out = torch.empty(n_rows, F, device=d)
    ops.spmm(csr, ops.M(xt), ops.M(out), F)
    assert rel_err(out, ref) < TOL
    out2 = torch.empty(n_rows, F, device=d)
    ops.spmm(csr, ops.M(xt), ops.M(out2), F, row_scale=st, bias=bt, addend=ops.M(at), relu=True)
    ref2 = np.maximum(scale[:, None] * ref + bias + add, 0)
    assert rel_err(out2, ref2) < TOL
    # determinism: identical bits on a second run (fixed summation order, no data atomics)
    out3 = torch.empty(n_rows, F, device=d)
    ops.spmm(csr, ops.M(xt), ops.M(out3), F, row_scale=st, bias=bt, addend=ops.M(at), relu=True)
    assert torch.equal(out2, out3)
    assert int(csr.row_counter.abs().sum()) == 0              # counters re-armed


def test_spmm_strided_slices_and_unit_values():
    from gripnet_b200 import ops
    from gripnet_b200.graph import Csr
    rs = np.random.RandomState(0)
    n_rows, n_cols, F = 257, 100, 16
    lens = rs.randint(0, 9, n_rows)
    rowptr, col, _ = _rand_csr(rs, n_rows, n_cols, lens)
    d = _dev()
    csr = Csr(torch.from_numpy(rowptr).to(d), torch.from_numpy(col).to(d), None, n_rows, n_cols, len(col))
    xbig = torch.randn(n_cols, 48, device=d)
    obig = torch.full((n_rows, 64), 7.0, device=d)
    ops.spmm(csr, ops.M(xbig, 16, F), ops.M(obig, 32, F), F)
    ref = _dense_ref(rowptr, col, None, xbig[:, 16:32].cpu().numpy(), n_rows)
    assert rel_err(obig[:, 32:48], ref) < TOL
    assert bool((obig[:, :32] == 7).all()) and bool((obig[:, 48:] == 7).all())   # neighbours untouched
    # in-place accumulate (addend aliases out), as the RGCN root term does
    base = torch.randn(n_rows, F, device=d)
    acc = base.clone()
    ops.spmm(csr, ops.M(xbig, 16, F), ops.M(acc), F, addend=ops.M(acc))
    assert rel_err(acc, ref + base.cpu().numpy()) < TOL


def _sgemm_ref(ta, tb, A, B):
    a = A.T if ta else A
    b = B.T if tb else B
    return a.astype(np.float64) @ b.astype(np.float64)


@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("m,n,k", [(1, 1, 1), (65, 17, 33), (300, 16, 32), (129, 130, 70), (48, 32, 5000)])
def test_sgemm_shapes(ta, tb, m, n, k):
    from gripnet_b200 import ops
    rs = np.random.RandomState(m + n + k)
    A = rs.randn(*((k, m) if ta else (m, k))).astype(np.float32)
    B = rs.randn(*((n, k) if tb else (k, n))).astype(np.float32)
    d = _dev()
    At, Bt = torch.from_numpy(A).to(d), torch.from_numpy(B).to(d)
    C = torch.empty(m, n, device=d)
    ops.sgemm(ta, tb, m, n, k, At.data_ptr(), A.shape[1], Bt.data_ptr(), B.shape[1], C.data_ptr(), n, d)
    assert rel_err(C, _sgemm_ref(ta, tb, A, B)) < TOL


def test_sgemm_epilogue_batch_and_gather():
    from gripnet_b200 import ops
    rs = np.random.RandomState(1)
    d = _dev()
    m, n, k = 70, 24, 40
    A, B = rs.randn(m, k).astype(np.float32), rs.randn(k, n).astype(np.float32)
    C0, add, mask = (rs.randn(m, n).astype(np.float32) for _ in range(3))
    At, Bt, addt, maskt = (torch.from_numpy(a).to(d) for a in (A, B, add, mask))
    C = torch.from_numpy(C0).to(d)
    ops.sgemm(0, 0, m, n, k, At.data_ptr(), k, Bt.data_ptr(), n, C.data_ptr(), n, d, alpha=0.5, accumulate=True,
              addend=ops.M(addt), mask=ops.M(maskt))
    ref = np.where(mask > 0, 0.5 * (A.astype(np.float64) @ B) + C0 + add, 0)
    assert rel_err(C, ref) < TOL
    # row gather on A, both layouts
    rows = rs.randint(0, m, size=55).astype(np.int64)
    rt = torch.from_numpy(rows).to(d)
    C = torch.empty(55, n, device=d)
    ops.sgemm(0, 0, 55, n, k, At.data_ptr(), k, Bt.data_ptr(), n, C.data_ptr(), n, d, a_rows=rt)
    assert rel_err(C, A[rows].astype(np.float64) @ B) < TOL
    G = rs.randn(55, n).astype(np.float32)
    Gt = torch.from_numpy(G).to(d)
    C = torch.empty(k, n, device=d)
    ops.sgemm(1, 0, k, n, 55, At.data_ptr(), k, Gt.data_ptr(), n, C.data_ptr(), n, d, a_rows=rt)
    assert rel_err(C, A[rows].astype(np.float64).T @ G) < TOL
    # batched with shared A, and batch-reduce
    r = 5
    W = rs.randn(r, k, n).astype(np.float32)
    Wt = torch.from_numpy(W).to(d)
    Y = torch.empty(m, r, n, device=d)
    ops.sgemm(0, 0, m, n, k, At.data_ptr(), k, Wt.data_ptr(), n, Y.data_ptr(), r * n, d, batch=r, sa=0, sb=k * n,
              sc=n)
    assert rel_err(Y, np.einsum("mk,rkn->mrn", A.astype(np.float64), W)) < TOL
    dX = torch.zeros(m, k, device=d)
    ops.sgemm(0, 1, m, k, n, Y.data_ptr(), r * n, Wt.data_ptr(), n, dX.data_ptr(), k, d, batch=r, sa=n, sb=k * n,
              sc=0, batch_reduce=True)
    assert rel_err(dX, np.einsum("mrn,rkn->mk", Y.cpu().numpy().astype(np.float64), W)) < TOL


def test_distmult_forward_backward():
    from gripnet_b200 import ops
    rs = np.random.RandomState(2)
    d = _dev()
    for D, n, r, e in [(80, 64, 5, 3000), (20, 30, 3, 100), (7, 10, 2, 50), (160, 40, 4, 500), (288, 20, 3, 200),
                       (128, 100, 6, 5000), (48, 7, 1, 33), (96, 300, 40, 20000)]:
        z = torch.randn(n, D, dtype=torch.float64)
        w = torch.randn(r, D, dtype=torch.float64)
        ei = torch.from_numpy(rs.randint(0, n, (2, e)))
        et = torch.from_numpy(rs.randint(0, r, e))
        for sig in (True, False):
            zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
            s = (zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1)
            ref = torch.sigmoid(s) if sig else s
            gvec = torch.linspace(-1, 1, e, dtype=torch.float64)
            (ref * gvec).sum().backward()
            zc = z.float().to(d).requires_grad_(True)
            wc = w.float().to(d).requires_grad_(True)
            out = ops.DistMult.apply(zc, wc, ei.to(d), et.to(d), sig)
            (out * gvec.float().to(d)).sum().backward()
            assert rel_err(out, ref) < TOL, (D, sig)
            assert rel_err(zc.grad, zr.grad) < TOL, (D, sig)
            assert rel_err(wc.grad, wr.grad) < TOL, (D, sig)


@pytest.mark.parametrize("D", [80, 160])
@pytest.mark.parametrize("n", [645, 3000])
def test_distmult_pose_sized_and_pair(n, D):
    """Pose-sized decoder call (n = 645 drugs x D = 80, 400 k edges) and a larger table, against float64;
    the fused pos/neg pair against two single calls (scores bit-identical; the pair adds the two lists' T
    before the products with w / z, two single calls add afterwards: gradients agree to rounding).
    Both kernel families: D = 80 takes the batch forms (32 edges / entries per warp step, every float4 width up
    to 128), D = 160 the per-edge / per-entry forms."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(n)
    d = _dev()
    r, e = 16, 400_000
    z = torch.randn(n, D, dtype=torch.float64) * 0.3
    w = torch.randn(r, D, dtype=torch.float64)
    ei = torch.from_numpy(rs.randint(0, n, (2, e)))
    ni = torch.from_numpy(rs.randint(0, n, (2, e)))
    et = torch.from_numpy(np.sort(rs.randint(0, r, e)))
    zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
    pos_ref = torch.sigmoid((zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1))
    neg_ref = torch.sigmoid((zr[ni[0]] * zr[ni[1]] * wr[et]).sum(1))
    gp = torch.linspace(-1, 1, e, dtype=torch.float64)
    gn = torch.linspace(0.5, -0.5, e, dtype=torch.float64)
    ((pos_ref * gp).sum() + (neg_ref * gn).sum()).backward()
    eid, nid, etd = ei.to(d), ni.to(d), et.to(d)
    res = []
    for pair in (False, True):
        zc = z.float().to(d).requires_grad_(True)
        wc = w.float().to(d).requires_grad_(True)
        if pair:
            pos, neg = ops.DistMultPair.apply(zc, wc, eid, nid, etd, True)
        else:
            pos, neg = ops.DistMult.apply(zc, wc, eid, etd, True), ops.DistMult.apply(zc, wc, nid, etd, True)
        ((pos * gp.float().to(d)).sum() + (neg * gn.float().to(d)).sum()).backward()
        torch.cuda.synchronize()
        assert rel_err(pos, pos_ref) < TOL and rel_err(neg, neg_ref) < TOL
        assert rel_err(zc.grad, zr.grad) < TOL and rel_err(wc.grad, wr.grad) < TOL
        res.append((pos.detach(), neg.detach(), zc.grad.clone(), wc.grad.clone()))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    assert rel_err(res[1][2], res[0][2]) < 1e-6 and rel_err(res[1][3], res[0][3]) < 1e-6


def test_distmult_short_rows_with_hub_rows():
    """(node, relation) rows that are short on average (the pose-2 regime: ~6 entries here, chunk length 32) with
    two hub rows split over ~190 chunks each, which finish through the partial / last-arrival path; against
    float64, and bit-identical run to run."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(17)
    d = _dev()
    n, D, r, e, hub = 2000, 80, 4, 20000, 6000
    src = np.r_[rs.randint(0, n, e), np.full(hub, 7)]
    dst = np.r_[rs.randint(0, n, e), rs.randint(0, n, hub)]
    et = np.r_[rs.randint(0, r, e), np.full(hub, 1)]
    order = np.argsort(et, kind="stable")
    ei = torch.from_numpy(np.stack([src, dst])[:, order].copy())
    et = torch.from_numpy(et[order].copy())
    z = torch.randn(n, D, dtype=torch.float64) * 0.3
    w = torch.randn(r, D, dtype=torch.float64)
    zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ref = torch.sigmoid((zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1))
    gvec = torch.linspace(-1, 1, ei.size(1), dtype=torch.float64)
    (ref * gvec).sum().backward()
    grads = []
    for _ in range(2):
        zc, wc = z.float().to(d).requires_grad_(True), w.float().to(d).requires_grad_(True)
        out = ops.DistMult.apply(zc, wc, ei.to(d), et.to(d), True)
        (out * gvec.float().to(d)).sum().backward()
        assert rel_err(out, ref) < TOL
        assert rel_err(zc.grad, zr.grad) < TOL and rel_err(wc.grad, wr.grad) < TOL
        grads.append((zc.grad.clone(), wc.grad.clone()))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])


def test_distmult_backward_deterministic_and_hub_rows():
    from gripnet_b200 import ops
    rs = np.random.RandomState(3)
    d = _dev()
    n, D, r, e = 20, 80, 3, 60_000                   # ~6000 entries per node -> many chunks per row
    z = torch.randn(n, D, device=d)
    w = torch.randn(r, D, device=d)
    ei = torch.from_numpy(rs.randint(0, n, (2, e))).to(d)
    et = torch.from_numpy(rs.randint(0, r, e)).to(d)
    grads = []
    for _ in range(2):
        zc, wc = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
        ops.DistMult.apply(zc, wc, ei, et, True).sum().backward()
        grads.append((zc.grad.clone(), wc.grad.clone()))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])
    z64 = z.double().cpu().requires_grad_(True)
    w64 = w.double().cpu().requires_grad_(True)
    torch.sigmoid((z64[ei[0].cpu()] * z64[ei[1].cpu()] * w64[et.cpu()]).sum(1)).sum().backward()
    assert rel_err(grads[0][0], z64.grad) < TOL and rel_err(grads[0][1], w64.grad) < TOL


def test_multiclass_decoder():
    from gripnet_b200 import ops
    d = _dev()
    rs = np.random.RandomState(4)
    for n, D, C, m in [(50, 288, 8, 30), (40, 32, 5, 60), (10, 7, 3, 4)]:
        z = torch.randn(n, D, dtype=torch.float64)
        w = torch.randn(D, C, dtype=torch.float64) / np.sqrt(D)   # keeps the softmax out of saturation
        idx = torch.from_numpy(rs.randint(0, n, m))          # duplicates allowed
        for sm in (True, False):
            zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
            ref = zr[idx] @ wr
            ref = torch.softmax(ref, 1) if sm else ref
            gm = torch.linspace(-1, 1, m * C, dtype=torch.float64).view(m, C)
            (ref * gm).sum().backward()
            zc = z.float().to(d).requires_grad_(True)
            wc = w.float().to(d).requires_grad_(True)
            out = ops.MultiClass.apply(zc, wc, idx.to(d), sm)
            (out * gm.float().to(d)).sum().backward()
            assert rel_err(out, ref) < TOL and rel_err(zc.grad, zr.grad) < TOL and rel_err(wc.grad, wr.grad) < TOL


def test_losses_and_elementwise():
    import gripnet_b200 as gb
    from gripnet_b200 import ops, _lib
    d = _dev()
    pos = torch.rand(5000, dtype=torch.float64) * 0.98 + 0.01
    neg = torch.rand(4000, dtype=torch.float64) * 0.98 + 0.01
    pr, nr = pos.clone().requires_grad_(True), neg.clone().requires_grad_(True)
    ref = -torch.log(pr + 1e-13).mean() - torch.log(1 - nr + 1e-13).mean()
    (ref * 1.7).backward()
    pc, nc = pos.float().to(d).requires_grad_(True), neg.float().to(d).requires_grad_(True)
    loss = gb.link_prediction_loss(pc, nc)
    (loss * 1.7).backward()
    assert rel_err(loss, ref) < TOL and rel_err(pc.grad, pr.grad) < TOL and rel_err(nc.grad, nr.grad) < TOL
    score = torch.softmax(torch.randn(300, 6, dtype=torch.float64), 1)
    lab = torch.randint(0, 6, (300,))
    sr = score.clone().requires_grad_(True)
    ref = -torch.log(sr[torch.arange(300), lab] + 1e-13).mean()
    ref.backward()
    sc = score.float().to(d).requires_grad_(True)
    loss = gb.node_classification_loss(sc, lab.to(d))
    loss.backward()
    assert rel_err(loss, ref) < TOL and rel_err(sc.grad, sr.grad) < TOL
    # column sums (bias gradient), several widths incl. > 256
    for n, F in [(1, 3), (1000, 16), (5000, 48), (777, 300)]:
        x = torch.randn(n, F + 5, device=d)
        out = torch.empty(F, device=d)
        ops.colsum(ops.M(x, 2, F), out)
        assert rel_err(out, x[:, 2:2 + F].double().sum(0).cpu()) < TOL
    # strided maps
    a = torch.randn(33, 20, device=d)
    o = torch.zeros(33, 50, device=d)
    ops.map2d(_lib.EW_ABS, ops.M(a), ops.M(o, 8, 20))
    assert torch.equal(o[:, 8:28], a.abs()) and float(o[:, :8].abs().sum()) == 0
    ops.map2d(_lib.EW_ADD, ops.M(a), ops.M(o, 8, 20))
    assert torch.allclose(o[:, 8:28], a.abs() + a)
    y = torch.randn(33, 20, device=d)
    r = torch.empty(33, 20, device=d)
    ops.relu_bwd(ops.M(a), ops.M(y), ops.M(r))
    assert torch.equal(r, torch.where(y > 0, a, torch.zeros_like(a)))


def test_distmult_pair_edge_cases():
    """Same tensor as positive AND negative list (one shared structure: the two walks must not race), an
    in-place rewrite of the indices between forward and backward (must raise, not mis-pair), out-of-range
    ids (IndexError like the reference's indexing), empty edge lists."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(9)
    d = _dev()
    n, D, r, e = 50, 80, 4, 20_000
    z = torch.randn(n, D, dtype=torch.float64) * 0.3
    w = torch.randn(r, D, dtype=torch.float64)
    ei = torch.from_numpy(rs.randint(0, n, (2, e)))
    et = torch.from_numpy(np.sort(rs.randint(0, r, e)))
    zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ref = torch.sigmoid((zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1))
    (ref.sum() * 2).backward()
    zc, wc = z.float().to(d).requires_grad_(True), w.float().to(d).requires_grad_(True)
    eid, etd = ei.to(d), et.to(d)
    pos, neg = ops.DistMultPair.apply(zc, wc, eid, eid, etd, True)
    (pos.sum() + neg.sum()).backward()
    assert torch.equal(pos, neg) and rel_err(pos, ref) < TOL
    assert rel_err(zc.grad, zr.grad) < TOL and rel_err(wc.grad, wr.grad) < TOL
    # in-place rewrite between forward and backward
    zc2 = z.float().to(d).requires_grad_(True)
    buf = eid.clone()
    out = ops.DistMult.apply(zc2, wc.detach(), buf, etd, True)
    buf.copy_(eid.flip(1))
    with pytest.raises(RuntimeError, match="modified in place"):
        out.sum().backward()
    # out-of-range ids
    bad = eid.clone()
    bad[0, 5] = n
    with pytest.raises(IndexError):
        ops.DistMult.apply(zc.detach(), wc.detach(), bad, etd, True)
    bad_t = etd.clone()
    bad_t[-1] = r
    with pytest.raises(IndexError):
        ops.DistMult.apply(zc.detach(), wc.detach(), eid, bad_t, True)
    with pytest.raises(IndexError):
        ops.MultiClass.apply(zc.detach(), torch.randn(D, 3, device=d), torch.tensor([0, n], device=d), True)
    with pytest.raises(IndexError):
        ops.NodeClassLoss.apply(torch.rand(4, 3, device=d), torch.tensor([0, 1, 2, 3], device=d))
    # empty lists
    z0 = z.float().to(d).requires_grad_(True)
    empty = torch.zeros((2, 0), dtype=torch.int64, device=d)
    o = ops.DistMult.apply(z0, wc.detach().requires_grad_(True), empty, torch.zeros(0, dtype=torch.int64, device=d), True)
    assert o.numel() == 0
    o.sum().backward()
    assert float(z0.grad.abs().sum()) == 0.0


def test_mean3_matches_the_reference_expression():
    """(z + z1 + emb) / 3 of GripNet-freebase-d.py:160-161: same association order and a true division, as the
    reference evaluates it on the CPU (torch's CUDA kernel multiplies by the rounded reciprocal instead: equal to
    1 ulp), gradient g / 3 on all three inputs."""
    from gripnet_b200 import ops
    d = _dev()
    a, b, c = (torch.randn(1000, 128, device=d, requires_grad=True) for _ in range(3))
    out = ops.mean3(a, b, c)
    ref = ((a.detach().cpu() + b.detach().cpu()) + c.detach().cpu()) / 3
    assert torch.equal(out.detach().cpu(), ref)
    assert rel_err(out, (a + b + c) / 3) < 1e-6
    g = torch.randn_like(out)
    out.backward(g)
    for t in (a, b, c):
        assert rel_err(t.grad, (g / 3)) < 1e-6
