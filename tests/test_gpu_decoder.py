"""GPU: every kernel instantiation of the DistMult decoder (``csrc/decoder.cu``) and every layout of ``z`` it is
reached with, against a float64 restatement of the decoder on the CPU.

``gn_distmult_fwd``, ``gn_distmult_bwd_pairs`` and ``gn_distmult_grads`` pick an instantiation from the width ``D``,
the row stride of ``z`` and its 16-byte alignment.  Each case below names the instantiations it reaches, checks
through the profiler that they ran, and the last test checks that the cases together reach every instantiation the
file compiles.  Also: gradients of one input only, a relation slice on one GPU, non-finite rows no edge references,
row strides at the 32-bit byte boundary of the batch forms, run-to-run and captured-graph bit equality, and the
multi-class decoder.

Tolerance: 1e-5 relative (max|a-b| / max|b| per tensor), as in test_gpu_kernels.py.
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from golden_util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5

# every instantiation csrc/decoder.cu compiles (its GN_*_CASE lists)
FWD_KERNELS = {f"distmult_fwd_batch_kernel<{n}>" for n in (1, 2, 3, 4)} | {
    f"distmult_fwd_kernel<{l},{v}>" for l, v in ((8, 4), (32, 4), (4, 1), (8, 1), (32, 1))}
WALK_KERNELS = {f"pair_walk_batch_kernel<{n}>" for n in (1, 2, 3, 4)} | {"pair_walk_kernel<4,1,1>"} | {
    f"pair_walk_kernel<{l},{v},{n}>" for l, v in ((32, 4), (4, 1), (32, 1)) for n in (2, 4, 5, 8)}
GRAD_KERNELS = {"distmult_grads_vec_kernel", "distmult_grads_kernel"}
ALL_KERNELS = FWD_KERNELS | WALK_KERNELS | GRAD_KERNELS

# instantiations each width reaches with a contiguous z: (forward, walk per column block, gradients per block)
CONTIGUOUS = {
    4: ("distmult_fwd_batch_kernel<1>", ["pair_walk_batch_kernel<1>"], ["distmult_grads_vec_kernel"]),
    48: ("distmult_fwd_batch_kernel<2>", ["pair_walk_batch_kernel<2>"], ["distmult_grads_vec_kernel"]),
    80: ("distmult_fwd_batch_kernel<3>", ["pair_walk_batch_kernel<3>"], ["distmult_grads_vec_kernel"]),
    128: ("distmult_fwd_batch_kernel<4>", ["pair_walk_batch_kernel<4>"], ["distmult_grads_vec_kernel"]),
    132: ("distmult_fwd_kernel<8,4>", ["pair_walk_kernel<32,4,2>"], ["distmult_grads_kernel"]),
    260: ("distmult_fwd_kernel<32,4>", ["pair_walk_kernel<32,4,4>"], ["distmult_grads_kernel"]),
    516: ("distmult_fwd_kernel<32,4>", ["pair_walk_kernel<32,4,5>"], ["distmult_grads_kernel"]),
    1024: ("distmult_fwd_kernel<32,4>", ["pair_walk_kernel<32,4,8>"], ["distmult_grads_kernel"]),
    3: ("distmult_fwd_kernel<4,1>", ["pair_walk_kernel<4,1,1>"], ["distmult_grads_kernel"]),
    7: ("distmult_fwd_kernel<4,1>", ["pair_walk_kernel<4,1,2>"], ["distmult_grads_kernel"]),
    13: ("distmult_fwd_kernel<4,1>", ["pair_walk_kernel<4,1,4>"], ["distmult_grads_kernel"]),
    19: ("distmult_fwd_kernel<4,1>", ["pair_walk_kernel<4,1,5>"], ["distmult_grads_kernel"]),
    29: ("distmult_fwd_kernel<4,1>", ["pair_walk_kernel<4,1,8>"], ["distmult_grads_kernel"]),
    33: ("distmult_fwd_kernel<8,1>", ["pair_walk_kernel<32,1,2>"], ["distmult_grads_kernel"]),
    65: ("distmult_fwd_kernel<32,1>", ["pair_walk_kernel<32,1,4>"], ["distmult_grads_kernel"]),
    150: ("distmult_fwd_kernel<32,1>", ["pair_walk_kernel<32,1,5>"], ["distmult_grads_kernel"]),
    250: ("distmult_fwd_kernel<32,1>", ["pair_walk_kernel<32,1,8>"], ["distmult_grads_kernel"]),
    # wider than one pass of the backward: column blocks of 256 (scalar rows) or 1024 (float4 rows)
    258: ("distmult_fwd_kernel<32,1>", ["pair_walk_kernel<32,1,8>", "pair_walk_kernel<4,1,1>"],
          ["distmult_grads_kernel", "distmult_grads_kernel"]),
    1028: ("distmult_fwd_kernel<32,4>", ["pair_walk_kernel<32,4,8>", "pair_walk_batch_kernel<1>"],
           ["distmult_grads_kernel", "distmult_grads_kernel"]),
}
LAYOUTS = ("contiguous", "offset4", "offset1", "stride_d5")



def _dev():
    return torch.device("cuda:0")


def _layout(x, kind):
    """A float32 CUDA leaf with x's values whose rows are laid out as `kind`:
    contiguous; a column view at offset 4 of a wider buffer (16-byte aligned, row stride != D); offset 1
    (misaligned); offset 0 with row stride D + 5 (not a multiple of 4)."""
    n, d = x.shape
    if kind == "contiguous":
        v = x.float().to(_dev())
    else:
        c0, ld = {"offset4": (4, d + 8), "offset1": (1, d + 8), "stride_d5": (0, d + 5)}[kind]
        buf = torch.full((n, ld), float("nan"), device=_dev())      # columns outside the view must not be read
        buf[:, c0:c0 + d] = x.float().to(_dev())
        v = buf[:, c0:c0 + d]
    return v.detach().requires_grad_(True)


def _plan(d, ldz, aligned):
    """Instantiations the dispatch of decoder.cu picks (a restatement of its rules, column blocks included)."""
    v4 = d % 4 == 0 and ldz % 4 == 0 and aligned and (d > 128 or ldz < 2 ** 30)
    if v4 and d <= 128:
        fwd = f"distmult_fwd_batch_kernel<{(d // 4 + 7) // 8}>"
    else:
        units = d // 4 if v4 else d
        fwd = f"distmult_fwd_kernel<{4 if units <= 32 else 8 if units <= 64 else 32},{4 if v4 else 1}>"
    walks, grads = [], []
    blk = 1024 if (d % 4 == 0 and ldz % 4 == 0 and aligned) else 256
    for c0 in range(0, d, blk):
        w = min(blk, d - c0)
        b4 = w % 4 == 0 and ldz % 4 == 0 and aligned and (w > 128 or ldz < 2 ** 30)
        if b4 and w <= 128:
            walks.append(f"pair_walk_batch_kernel<{(w // 4 + 7) // 8}>")
        else:
            units = w // 4 if b4 else w
            lpe = 4 if units <= 32 else 32
            need = -(-units // lpe)
            nv = 1 if need <= 1 else 2 if need <= 2 else 4 if need <= 4 else 5 if need <= 5 else 8
            walks.append(f"pair_walk_kernel<{lpe},{4 if b4 else 1},{nv}>")
        vec = w == d and d % 4 == 0 and d <= 128 and ldz % 4 == 0 and aligned      # (float4 kernel: whole rows of w)
        grads.append("distmult_grads_vec_kernel" if vec else "distmult_grads_kernel")
    return fwd, walks, grads


def _kernel_names(fn):
    """Run fn under the profiler; the decoder kernels that ran, spelled like the keys above."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r"((?:distmult_fwd|pair_walk|distmult_grads)\w*kernel)(<[^>]*>)?", e.name)
        if m:
            names.add(m.group(1) + re.sub(r"\s", "", m.group(2) or ""))
    return names


def _graph(rs, n, r, e, hub, shuffled):
    """e random edges plus `hub` edges of node 1 under relation 0 (one pair row split over several chunks) and pair
    rows of lengths 1-5 (nodes n - 1 ... n - 5, relation r - 1), relation-sorted or shuffled."""
    src = [rs.randint(0, n, e), np.full(hub, 1)]
    dst = [rs.randint(0, n, e), rs.randint(0, n, hub)]
    ty = [rs.randint(0, r, e), np.zeros(hub, np.int64)]
    for k in range(1, 6):
        src.append(np.full(k, n - k))
        dst.append(rs.randint(1, n, k))
        ty.append(np.full(k, r - 1))
    src, dst, ty = np.concatenate(src), np.concatenate(dst), np.concatenate(ty)
    order = rs.permutation(len(ty)) if shuffled else np.argsort(ty, kind="stable")
    return torch.from_numpy(np.stack([src, dst])[:, order].copy()), torch.from_numpy(ty[order].copy())


def _reference(z, w, ei, et, sig, gvec, need=(True, True)):
    zr, wr = z.clone().requires_grad_(need[0]), w.clone().requires_grad_(need[1])
    s = (zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1)
    ref = torch.sigmoid(s) if sig else s
    (ref * gvec).sum().backward()
    return ref.detach(), zr.grad, wr.grad


def _run(z, w, ei, et, sig, gvec):
    from gripnet_b200 import ops
    out = ops.DistMult.apply(z, w, ei.to(_dev()), et.to(_dev()), sig)
    (out * gvec.float().to(_dev())).sum().backward()
    return out


def _matrix_case(D, layout, seed):
    from gripnet_b200 import graph
    rs = np.random.RandomState(seed)
    e = 1500 if D <= 300 else 600
    for n, r, shuffled, sig in ((90, 5, False, True), (300, 40, True, False)):
        ei, et = _graph(rs, n, r, e, hub=2500, shuffled=shuffled)
        z = torch.randn(n, D, dtype=torch.float64) * 0.3
        w = torch.randn(r, D, dtype=torch.float64)
        gvec = torch.linspace(-1, 1, et.numel(), dtype=torch.float64)
        ref, dz_ref, dw_ref = _reference(z, w, ei, et, sig, gvec)
        zc, wc = _layout(z, layout), w.float().to(_dev()).requires_grad_(True)
        out = _run(zc, wc, ei, et, sig, gvec)
        ps = graph.pair_struct(ei.to(_dev()), et.to(_dev()), n, r)
        assert ps.csr.n_chunks > ps.csr.n_rows                     # the split-row finish ran
        assert rel_err(out, ref) < TOL, (D, layout, sig)
        assert rel_err(zc.grad, dz_ref) < TOL, (D, layout, sig)
        assert rel_err(wc.grad, dw_ref) < TOL, (D, layout, sig)
    return _plan(D, zc.stride(0), zc.data_ptr() % 16 == 0)


MATRIX = {f"matrix:{lay}": [(D, lay, D * 7 + LAYOUTS.index(lay)) for D in sorted(CONTIGUOUS)] for lay in LAYOUTS}
MATRIX["wide"] = [(300, "offset1", 301)]


def _profile_all():
    """The decoder kernels each profiled group of cases launches: {group: sorted names}."""
    got = {key: _kernel_names(lambda: [_matrix_case(*c) for c in cases]) for key, cases in MATRIX.items()}
    if _enough_memory():
        for ldz in STRIDES:
            got[f"stride:{ldz}"] = _kernel_names(lambda: _stride_case(ldz))
    return {k: sorted(v) for k, v in got.items()}


@pytest.fixture(scope="module")
def profiled():
    """Kernel names per group of cases, recorded by torch.profiler in a process of its own: a profiler session in
    the test process itself can leave sessions of later test modules without kernel records."""
    env = dict(os.environ)
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=env, capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return {k: set(v) for k, v in json.loads(res.stdout.strip().splitlines()[-1]).items()}


def _matrix(key, profiled):
    """The cases of group `key` against float64; each case's instantiations must be among those the group ran."""
    plans = {(D, lay): _matrix_case(D, lay, seed) for D, lay, seed in MATRIX[key]}
    ran = profiled[key]
    for case, (fwd, walks, grads) in plans.items():
        assert {fwd, *walks, *grads} <= ran, (case, sorted({fwd, *walks, *grads} - ran), sorted(ran))
    return plans


@pytest.mark.parametrize("layout", LAYOUTS)
def test_distmult_instantiation_matrix(layout, profiled):
    """Forward, dz and dw against float64 for every width class and layout of z: relation-sorted edges with the
    sigmoid (uniform-relation batches, n = 90 < 96 nodes: one dw slab, 5 relations) and shuffled edges without it
    (mixed batches, n = 300: several slabs, 40 relations: 8 sub-rows per node in the float4 dz)."""
    plans = _matrix(f"matrix:{layout}", profiled)
    if layout == "contiguous":
        assert {D: p for (D, _), p in plans.items()} == CONTIGUOUS


def test_distmult_misaligned_wide_view(profiled):
    """z[:, 1:301]: 300 misaligned columns, two column blocks (256 + 44) in the backward."""
    (got,) = _matrix("wide", profiled).values()
    assert got == ("distmult_fwd_kernel<32,1>", ["pair_walk_kernel<32,1,8>", "pair_walk_kernel<32,1,2>"],
                   ["distmult_grads_kernel", "distmult_grads_kernel"])


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("which", ["z", "w"])
@pytest.mark.parametrize("D", [80, 29])
def test_distmult_gradient_of_one_input(pair, which, D):
    """Only z or only w requires grad: the dz-only and dw-only launches of both gradient kernels."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(40 + D)
    n, r = 200, 6
    ei, et = _graph(rs, n, r, 3000, hub=2000, shuffled=True)
    ni = torch.from_numpy(rs.randint(0, n, ei.shape))
    z = torch.randn(n, D, dtype=torch.float64) * 0.3
    w = torch.randn(r, D, dtype=torch.float64)
    need = (which == "z", which == "w")
    gp = torch.linspace(-1, 1, et.numel(), dtype=torch.float64)
    gn = torch.linspace(0.5, -0.5, et.numel(), dtype=torch.float64)
    zr, wr = z.clone().requires_grad_(need[0]), w.clone().requires_grad_(need[1])
    pos_ref = torch.sigmoid((zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1))
    neg_ref = torch.sigmoid((zr[ni[0]] * zr[ni[1]] * wr[et]).sum(1))
    loss_ref = (pos_ref * gp).sum() + ((neg_ref * gn).sum() if pair else 0)
    loss_ref.backward()
    zc = z.float().to(_dev()).requires_grad_(need[0])
    wc = w.float().to(_dev()).requires_grad_(need[1])
    d = _dev()

    def step():
        if pair:
            pos, neg = ops.DistMultPair.apply(zc, wc, ei.to(d), ni.to(d), et.to(d), True)
            ((pos * gp.float().to(d)).sum() + (neg * gn.float().to(d)).sum()).backward()
        else:
            pos = ops.DistMult.apply(zc, wc, ei.to(d), et.to(d), True)
            (pos * gp.float().to(d)).sum().backward()

    step()
    if need[0]:
        assert wc.grad is None and rel_err(zc.grad, zr.grad) < TOL
    else:
        assert zc.grad is None and rel_err(wc.grad, wr.grad) < TOL


@pytest.mark.parametrize("D", [80, 250])
def test_distmult_pair_relation_slice(D):
    """DistMultPair over relations [rel_lo, rel_lo + n_rel_local) of R with shifted edge types: dz and the slice of
    dw against float64, the other rows of dw exactly zero."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(50 + D)
    n, R, lo, nl = 150, 9, 3, 4
    ei, et = _graph(rs, n, nl, 2000, hub=1500, shuffled=False)
    ni = torch.from_numpy(rs.randint(0, n, ei.shape))
    z = torch.randn(n, D, dtype=torch.float64) * 0.3
    w = torch.randn(R, D, dtype=torch.float64)
    gp = torch.linspace(-1, 1, et.numel(), dtype=torch.float64)
    gn = torch.linspace(0.5, -0.5, et.numel(), dtype=torch.float64)
    zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
    etg = et + lo
    pos_ref = torch.sigmoid((zr[ei[0]] * zr[ei[1]] * wr[etg]).sum(1))
    neg_ref = torch.sigmoid((zr[ni[0]] * zr[ni[1]] * wr[etg]).sum(1))
    ((pos_ref * gp).sum() + (neg_ref * gn).sum()).backward()
    d = _dev()
    zc, wc = z.float().to(d).requires_grad_(True), w.float().to(d).requires_grad_(True)
    pos, neg = ops.DistMultPair.apply(zc, wc, ei.to(d), ni.to(d), et.to(d), True, lo, nl)
    ((pos * gp.float().to(d)).sum() + (neg * gn.float().to(d)).sum()).backward()
    assert rel_err(pos, pos_ref) < TOL and rel_err(neg, neg_ref) < TOL
    assert rel_err(zc.grad, zr.grad) < TOL
    assert rel_err(wc.grad[lo:lo + nl], wr.grad[lo:lo + nl]) < TOL
    outside = torch.cat([wc.grad[:lo], wc.grad[lo + nl:]])
    assert torch.equal(outside, torch.zeros_like(outside))


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("D", [7, 29, 80, 160, 250])
def test_distmult_nonfinite_unreferenced_rows(D, pair):
    """z rows of nodes no edge references (node 0 among them) hold +Inf, -Inf and NaN, and w holds an Inf row for a
    relation no edge uses.  They cannot change any score or gradient of the reference: every result is finite and
    matches float64 on the same data with those rows zeroed, and their own dz / dw rows are exactly zero."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(60 + D)
    n, r = 120, 6
    poisoned = np.array([0, 11, 57, 119])
    live = np.setdiff1d(np.arange(n), poisoned)
    e = 3000
    src = np.r_[live[rs.randint(0, len(live), e)], np.full(1200, live[3])]
    dst = np.r_[live[rs.randint(0, len(live), e)], live[rs.randint(0, len(live), 1200)]]
    ty = np.r_[rs.randint(0, r - 1, e), np.zeros(1200, np.int64)]          # relation r - 1: unused
    order = np.argsort(ty, kind="stable")
    ei = torch.from_numpy(np.stack([src, dst])[:, order].copy())
    et = torch.from_numpy(ty[order].copy())
    ni = torch.from_numpy(live[rs.randint(0, len(live), (2, et.numel()))])
    z = torch.randn(n, D, dtype=torch.float64) * 0.3
    w = torch.randn(r, D, dtype=torch.float64)
    z[poisoned] = 0.0
    w[r - 1] = 0.0
    gp = torch.linspace(-1, 1, et.numel(), dtype=torch.float64)
    gn = torch.linspace(0.5, -0.5, et.numel(), dtype=torch.float64)
    zr, wr = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
    pos_ref = torch.sigmoid((zr[ei[0]] * zr[ei[1]] * wr[et]).sum(1))
    neg_ref = torch.sigmoid((zr[ni[0]] * zr[ni[1]] * wr[et]).sum(1))
    ((pos_ref * gp).sum() + ((neg_ref * gn).sum() if pair else 0)).backward()
    zp, wp = z.float().clone(), w.float().clone()
    zp[0], zp[11], zp[57], zp[119] = float("inf"), float("-inf"), float("nan"), float("nan")
    zp[57, ::2] = float("inf")
    wp[r - 1] = float("inf")
    d = _dev()
    zc, wc = zp.to(d).requires_grad_(True), wp.to(d).requires_grad_(True)
    if pair:
        pos, neg = ops.DistMultPair.apply(zc, wc, ei.to(d), ni.to(d), et.to(d), True)
        ((pos * gp.float().to(d)).sum() + (neg * gn.float().to(d)).sum()).backward()
        assert torch.isfinite(neg).all() and rel_err(neg, neg_ref) < TOL
    else:
        pos = ops.DistMult.apply(zc, wc, ei.to(d), et.to(d), True)
        (pos * gp.float().to(d)).sum().backward()
    assert torch.isfinite(pos).all() and rel_err(pos, pos_ref) < TOL
    assert torch.isfinite(zc.grad).all() and torch.isfinite(wc.grad).all()
    assert rel_err(zc.grad, zr.grad) < TOL and rel_err(wc.grad, wr.grad) < TOL
    assert torch.equal(zc.grad[poisoned], torch.zeros(len(poisoned), D, device=d))
    assert torch.equal(wc.grad[r - 1], torch.zeros(D, device=d))


STRIDES = {
    2 ** 30 - 4: {"distmult_fwd_batch_kernel<3>", "pair_walk_batch_kernel<3>", "distmult_grads_vec_kernel"},
    2 ** 30: {"distmult_fwd_kernel<32,1>", "pair_walk_kernel<32,1,4>", "distmult_grads_vec_kernel"},
}


def _enough_memory():
    return torch.cuda.mem_get_info()[0] >= 10 * 2 ** 30


def _stride_case(ldz):
    D, r = 80, 3
    rs = np.random.RandomState(70)
    z = torch.randn(2, D, dtype=torch.float64) * 0.3
    w = torch.randn(r, D, dtype=torch.float64)
    ei = torch.from_numpy(rs.randint(0, 2, (2, 300)))
    et = torch.from_numpy(np.sort(rs.randint(0, r, 300)))
    gvec = torch.linspace(-1, 1, 300, dtype=torch.float64)
    ref, dz_ref, dw_ref = _reference(z, w, ei, et, True, gvec)
    buf = torch.empty(ldz + D, device=_dev())
    zv = buf.as_strided((2, D), (ldz, 1))
    zv.copy_(z.float())
    zc = zv.detach().requires_grad_(True)
    assert zc.stride(0) == ldz
    wc = w.float().to(_dev()).requires_grad_(True)
    out = _run(zc, wc, ei, et, True, gvec)
    assert rel_err(out, ref) < TOL
    assert rel_err(zc.grad, dz_ref) < TOL and rel_err(wc.grad, dw_ref) < TOL
    del zc, zv, buf, out
    torch.cuda.empty_cache()


@pytest.mark.parametrize("ldz", sorted(STRIDES))
def test_distmult_row_stride_at_the_32bit_boundary(ldz, profiled):
    """Two rows of z, ldz floats apart: just below 2^30 the batch forms step rows with a 32-bit byte stride (row 1
    at byte 2^32 - 16); at 2^30 they cannot, and the per-edge / per-entry forms take over.  About 4 GiB each."""
    if not _enough_memory():
        pytest.skip("needs 10 GiB of free device memory")
    _stride_case(ldz)
    ran = profiled.get(f"stride:{ldz}", set())
    assert STRIDES[ldz] <= ran, sorted(ran)


@pytest.mark.parametrize("D", [29, 250])
def test_distmult_deterministic_and_captured(D):
    """Per-entry widths with hub rows: two eager runs give bit-identical gradients, and the forward + backward
    captured in a CUDA graph — whose (node, relation) structure is built inside the capture with the inexact chunk
    bound — replays to the same bits."""
    from gripnet_b200 import graph, ops
    rs = np.random.RandomState(80 + D)
    n, r = 400, 7
    ei, et = _graph(rs, n, r, 4000, hub=3000, shuffled=True)
    d = _dev()
    z = (torch.randn(n, D, dtype=torch.float64) * 0.3).float().to(d)
    w = torch.randn(r, D, dtype=torch.float64).float().to(d)
    gvec = torch.linspace(-1, 1, et.numel()).to(d)
    eid, etd = ei.to(d), et.to(d)

    def step(zc, wc, idx, ty):
        out = ops.DistMult.apply(zc, wc, idx, ty, True)
        (out * gvec).sum().backward()
        return out

    runs = []
    for _ in range(2):
        zc, wc = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
        out = step(zc, wc, eid, etd)
        runs.append((out.detach(), zc.grad, wc.grad))
    assert all(torch.equal(a, b) for a, b in zip(runs[0], runs[1]))
    zc, wc = z.clone().requires_grad_(True), w.clone().requires_grad_(True)
    eid2, etd2 = eid.clone(), etd.clone()          # not in the structure cache: built inside the capture
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):                          # warm-up on the capture stream
            zc.grad = wc.grad = None
            step(zc, wc, eid, etd)
    torch.cuda.current_stream().wait_stream(s)
    zc.grad = wc.grad = None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step(zc, wc, eid2, etd2)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    ps, exact = graph.pair_struct(eid2, etd2, n, r), graph.pair_struct(eid, etd, n, r)
    assert ps.csr.n_chunks > exact.csr.n_chunks > exact.csr.n_rows    # the inexact chunk bound, split rows
    assert torch.equal(out, runs[0][0])
    assert torch.equal(zc.grad, runs[0][1]) and torch.equal(wc.grad, runs[0][2])


@pytest.mark.parametrize("C", [1, 31, 33, 1000])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_multiclass_decoder_widths_and_layouts(C, layout):
    """softmax(z[node_list] W) for C up to 1000 (the softmax kernels loop over columns past 32), every z layout, a
    node list with duplicates, both gradients and each one alone."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(C + LAYOUTS.index(layout))
    n, D, m = 70, 48, 150
    z = torch.randn(n, D, dtype=torch.float64)
    w = torch.randn(D, C, dtype=torch.float64) / np.sqrt(D)
    idx = torch.from_numpy(np.r_[rs.randint(0, n, m - 10), np.full(10, 3)])
    gm = torch.from_numpy(rs.uniform(-1, 1, (m, C)))     # O(1) spread within a row: no cancellation in gy - <y, gy>
    for sm in (True, False):
        for need in ((True, True), (True, False), (False, True)):
            zr, wr = z.clone().requires_grad_(need[0]), w.clone().requires_grad_(need[1])
            ref = zr[idx] @ wr
            ref = torch.softmax(ref, 1) if sm else ref
            (ref * gm).sum().backward()
            zc = _layout(z, layout).requires_grad_(need[0])
            wc = w.float().to(_dev()).requires_grad_(need[1])
            out = ops.MultiClass.apply(zc, wc, idx.to(_dev()), sm)
            (out * gm.float().to(_dev())).sum().backward()
            assert rel_err(out, ref) < TOL, (C, layout, sm)
            if need[0]:
                assert rel_err(zc.grad, zr.grad) < TOL, (C, layout, sm)
            else:
                assert zc.grad is None
            if need[1]:
                assert rel_err(wc.grad, wr.grad) < TOL, (C, layout, sm)
            else:
                assert wc.grad is None


def test_every_instantiation_ran(profiled):
    """The cases above reach every instantiation of the decoder: one added to decoder.cu needs a case here."""
    seen = set().union(*profiled.values())
    assert seen >= ALL_KERNELS, sorted(ALL_KERNELS - seen)
    assert seen <= ALL_KERNELS, sorted(seen - ALL_KERNELS)


if __name__ == "__main__":          # the `profiled` fixture's child process
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    print(json.dumps(_profile_all()))
