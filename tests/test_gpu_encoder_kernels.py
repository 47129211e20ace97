"""GPU: every kernel instantiation of the encoder side (``csrc/spmm.cu``, ``csrc/gemm.cu``, ``csrc/elementwise.cu``)
and every operand layout and epilogue it is reached with, against float64 restatements on the CPU.

``gn_spmm`` picks ``spmm_kernel<LPE, VEC>`` per column panel from the width, the row strides and the 16-byte alignment
of its operands; ``gn_sgemm`` picks one of five CTA tiles, a reduction split and a split-reduce kernel from the output
shape.  Each case below restates those rules (``_spmm_plan``, ``_gemm_plan``), checks through the profiler that the
instances it expects ran, and the last test checks that the cases together ran exactly the instances the three files
compile.  The GCN / RGCN layer stacks run at node counts on both sides of the thresholds that route their products
(FFMA tiles at M = 1024, ``gn_tc_gemm`` at M >= 4096, ``gn_tc_tn`` at 2^15 rows) against a sparse float64 restatement.

Tolerance: 1e-5 relative (max|a-b| / max|b| per tensor), as in test_gpu_kernels.py; the loss gradients, whose
entries span many orders of magnitude, per element (and exactly 0 where the reference is 0).
"""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-5

# every instance the three files compile (cuobjdump -elf of their objects, demangled)
TILES = {0: "64,64,4,4,16", 1: "128,32,4,4,16", 2: "128,16,2,4,16", 3: "32,32,2,2,16", 4: "32,32,2,2,64"}
SPMM_KERNELS = {f"spmm_kernel<{l},{v}>" for l in (1, 2, 4, 8, 16, 32) for v in (1, 4)}
GEMM_KERNELS = {f"sgemm_kernel<{a},{b},{t}>" for a in (0, 1) for b in (0, 1) for t in TILES.values()} | {
    "splitk_reduce_kernel<1>", "splitk_reduce_kernel<32>"}
EW_KERNELS = {f"map2d{v}_kernel<{op}>" for v in ("", "_vec") for op in range(4)} | {
    "relu_bwd_kernel", "relu_bwd_vec_kernel", "abs_bwd_kernel", "abs_bwd_vec_kernel", "axpby_kernel", "mean3_kernel",
    "colsum_partial_kernel", "colsum_final_kernel"} | {
    f"{l}_loss_{s}_kernel" for l in ("lp", "nc") for s in ("partial", "final", "bwd")}
ALL_KERNELS = SPMM_KERNELS | GEMM_KERNELS | EW_KERNELS
TC_KERNELS = {"tc_gemm_kernel", "tc_tn_kernel"}   # routing targets of the layer stacks (own shape tests elsewhere)

_NAME = re.compile(r"\b((?:spmm|sgemm|splitk_reduce|map2d|map2d_vec|relu_bwd|relu_bwd_vec|abs_bwd|abs_bwd_vec|axpby|"
                   r"mean3|colsum_partial|colsum_final|lp_loss_partial|lp_loss_final|lp_loss_bwd|nc_loss_partial|"
                   r"nc_loss_final|nc_loss_bwd|tc_gemm|tc_tn)_kernel)(<[^>]*>)?")


def kernel_name(raw):
    """A kernel record's name spelled like the sets above, or None: template arguments without blanks, bools as 0/1
    (the profiler prints ``false``/``true``, cu++filt ``(bool)0``), no ``(int)`` casts; tc kernels without them."""
    m = _NAME.search(raw)
    if not m:
        return None
    if m.group(1) in ("tc_gemm_kernel", "tc_tn_kernel"):
        return m.group(1)
    args = re.sub(r"\s", "", m.group(2) or "")
    args = re.sub(r"\((?:bool|int)\)", "", args).replace("false", "0").replace("true", "1")
    return m.group(1) + args


def _dev():
    return torch.device("cuda:0")


def _kernel_names(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {n for n in (kernel_name(e.name) for e in prof.events()) if n}


def _bits(t):
    return t.contiguous().view(torch.int32)


# layouts of a [n, F] operand: (first column, row stride) inside a wider buffer; the other columns must not be read
# (NaN) or written (sentinel)
LAYOUTS = ("contiguous", "offset4", "offset1", "stride_f5")


def _place(a, layout, fill):
    """float32 device buffer holding `a` (numpy [n, F]) at `layout`; returns (buffer, first column)."""
    n, f = a.shape
    c0, ld = {"contiguous": (0, f), "offset4": (4, f + 8), "offset1": (1, f + 8), "stride_f5": (0, f + 5)}[layout]
    buf = torch.full((n, ld), fill, dtype=torch.float32, device=_dev())
    buf[:, c0:c0 + f] = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(_dev())
    return buf, c0


def _outside(buf, c0, f):
    return torch.cat([buf[:, :c0], buf[:, c0 + f:]], 1)


# ------------------------------------------------------------------------------------------------------------ SpMM
def _pow2_ceil(x):
    p = 1
    while p < x:
        p <<= 1
    return p


def _spmm_plan(F, ldx, ldo, aligned):
    """Instances gn_spmm launches, one per column panel: float4 rows in panels of 128 columns when F and both row
    strides are multiples of 4 and every operand is 16-byte aligned, else scalar rows in panels of 32."""
    vec4 = F % 4 == 0 and ldx % 4 == 0 and ldo % 4 == 0 and aligned
    panel = 128 if vec4 else 32
    return [f"spmm_kernel<{_pow2_ceil((min(panel, F - f0)) // (4 if vec4 else 1))},{4 if vec4 else 1}>"
            for f0 in range(0, F, panel)]


SPMM_WIDTHS = (1, 2, 3, 4, 5, 8, 12, 13, 24, 29, 31, 36, 64, 70, 128, 129, 260)


def _spmm_lens(rs, kind):
    """(row lengths, chunk_len, exact) of the test structures:
    one_chunk: every row within one 32-entry chunk (GN_CSR_ROW_IS_CHUNK), empty rows and rows of exactly 32;
    hub32 / hub256: hub rows of ~280 / ~310 chunks (sum_partials loops several times per slot at every LPE), rows of
    2 chunks, empty rows and rows of length 1; inexact: the hub rows with an upper bound for n_chunks."""
    if kind == "one_chunk":
        lens = rs.randint(0, 33, 300)
        lens[[7, 8, 9]] = [0, 1, 32]
        return lens, 32, True
    lens = rs.randint(0, 40, 200)
    lens[[4, 5, 150]] = [0, 1, 33]
    lens[3] = 9000 if kind != "hub256" else 80000
    lens[199] = 2000
    return lens, {"hub32": 32, "hub256": 256, "inexact": 64}[kind], kind != "inexact"


def _csr(rowptr, col, val, n_rows, n_cols, chunk_len, exact):
    from gripnet_b200.graph import Csr
    d = _dev()
    return Csr(torch.from_numpy(rowptr).to(d), torch.from_numpy(col).to(d),
               None if val is None else torch.from_numpy(val).to(d), n_rows, n_cols, len(col), exact=exact,
               chunk_len=chunk_len)


def _spmm_struct(rs, kind, n_ref):
    lens, chunk_len, exact = _spmm_lens(rs, kind)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = rs.randint(0, n_ref, int(rowptr[-1])).astype(np.int32)
    val = rs.uniform(-1, 1, len(col)).astype(np.float32)
    return rowptr, col, val, chunk_len, exact


def _check_structure(csr, kind):
    from gripnet_b200 import _lib
    if kind == "one_chunk":
        assert csr.flags == _lib.CSR_ROW_IS_CHUNK and csr.n_chunks == csr.n_rows
    elif kind == "inexact":
        assert csr.flags == 0 and csr.n_chunks > int(csr.chunk_ptr[csr.n_rows]) > csr.n_rows
    else:
        assert csr.flags == 0 and csr.n_chunks > csr.n_rows + 200


SPMM_SENTINEL = -1234.5


def _spmm_case(F, layout):
    """Every structure and epilogue at width F with x and out laid out as `layout`: values plain and None,
    row_scale + bias + a separate addend (twice: bit-identical), and addend aliasing out with ReLU.  Rows of x that
    no entry references hold +Inf / -Inf / NaN."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(F * 11 + LAYOUTS.index(layout))
    n_cols = 400
    x = rs.randn(n_cols, F).astype(np.float32)
    x[n_cols - 3], x[n_cols - 2], x[n_cols - 1] = np.inf, -np.inf, np.nan
    x64 = x.astype(np.float64)
    x64[n_cols - 3:] = 0.0
    xbuf, cx = _place(x, layout, float("nan"))
    X = ops.M(xbuf, cx, F)
    bias = rs.randn(F).astype(np.float32)
    bias_t = torch.from_numpy(bias).to(_dev())
    plan = None
    for kind in ("one_chunk", "hub32", "hub256", "inexact"):
        rowptr, col, val, chunk_len, exact = _spmm_struct(rs, kind, n_cols - 3)
        n_rows = len(rowptr) - 1
        a64 = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(n_rows, n_cols))
        a1 = sp.csr_matrix((np.ones(len(col)), col, rowptr), shape=(n_rows, n_cols))
        ref, ref1 = a64 @ x64, a1 @ x64
        scale = rs.uniform(0.5, 2, n_rows).astype(np.float32)
        add = rs.randn(n_rows, F).astype(np.float32)
        base = rs.randn(n_rows, F).astype(np.float32)
        scale_t, add_t = torch.from_numpy(scale).to(_dev()), torch.from_numpy(add).to(_dev())
        csr = _csr(rowptr, col, val, n_rows, n_cols, chunk_len, exact)
        csr1 = _csr(rowptr, col, None, n_rows, n_cols, chunk_len, exact)
        _check_structure(csr, kind)
        epi = scale[:, None].astype(np.float64) * ref + bias + add
        results = []
        for name, c, kw, init, want in (
                ("val", csr, {}, None, ref),
                ("unit", csr1, {}, None, ref1),
                ("scale_bias_addend", csr, dict(row_scale=scale_t, bias=bias_t, addend=ops.M(add_t)), None, epi),
                ("scale_bias_addend", csr, dict(row_scale=scale_t, bias=bias_t, addend=ops.M(add_t)), None, epi),
                ("in_place_relu", csr, dict(row_scale=scale_t, bias=bias_t, relu=True), base,
                 np.maximum(epi - add + base, 0.0))):
            obuf, co = _place(np.zeros((n_rows, F)) if init is None else init, layout, SPMM_SENTINEL)
            O = ops.M(obuf, co, F)
            if name == "in_place_relu":
                kw = dict(kw, addend=O)
            ops.spmm(c, X, O, F, **kw)
            out = obuf[:, co:co + F]
            assert bool(torch.isfinite(out).all()), (F, layout, kind, name)
            assert rel_err(out, want) < TOL, (F, layout, kind, name)
            assert bool((_outside(obuf, co, F) == SPMM_SENTINEL).all()), (F, layout, kind, name)
            results.append(out.clone())
            p = _spmm_plan(F, xbuf.stride(0), obuf.stride(0), cx % 4 == 0 and co % 4 == 0)
            assert plan is None or p == plan
            plan = p
        assert torch.equal(_bits(results[2]), _bits(results[3])), (F, layout, kind)      # run to run
        assert int(csr.row_counter.abs().sum()) == 0 and int(csr1.row_counter.abs().sum()) == 0
    return set(plan), set()


def _scratch_case(kind, F):
    """gn_spmm called directly with `partial` of exactly 2 (n_chunks - n_rows) rows of min(F, 128) floats and a
    canary tail that must come back bit-identical.  "50+2": a row of 50 chunks and one of 2 (52 chunks, 2 rows: the
    second row owns slots 98 and 99, past the [n_chunks, F] the header once documented)."""
    from gripnet_b200 import _lib, ops
    from gripnet_b200.graph import _stream
    rs = np.random.RandomState(F + len(kind))
    n_cols = 300
    if kind == "50+2":
        lens, chunk_len = np.array([50 * 32, 40]), 32
    else:
        lens, chunk_len, _ = _spmm_lens(rs, "hub32")
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    col = rs.randint(0, n_cols, int(rowptr[-1])).astype(np.int32)
    val = rs.uniform(-1, 1, len(col)).astype(np.float32)
    csr = _csr(rowptr, col, val, len(lens), n_cols, chunk_len, True)
    if kind == "50+2":
        assert (csr.n_rows, csr.n_chunks) == (2, 52)
    need = 2 * (csr.n_chunks - csr.n_rows) * min(F, 128)
    canary = torch.arange(4096, dtype=torch.int32, device=_dev()) * 7919 - 2 ** 30
    buf = torch.full((need + 4096,), float("nan"), device=_dev())
    buf[need:] = canary.view(torch.float32)
    x = rs.randn(n_cols, F).astype(np.float32)
    xt = torch.from_numpy(x).to(_dev())
    out = torch.empty(len(lens), F, device=_dev())
    _lib.check(_lib.load().gn_spmm(csr.ref, xt.data_ptr(), F, F, None, None, None, 0, 0, out.data_ptr(), F,
                                   buf.data_ptr(), _stream()), "gn_spmm")
    ref = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(len(lens), n_cols)) @ x.astype(np.float64)
    assert rel_err(out, ref) < TOL
    assert torch.equal(_bits(buf[need:]), canary)
    # the Python wrapper sizes the scratch the same way
    assert csr.partial(min(F, 128)).numel() == need
    ops.spmm(csr, ops.M(xt), ops.M(out), F)
    assert rel_err(out, ref) < TOL
    return set(_spmm_plan(F, F, F, True)), set()


# ------------------------------------------------------------------------------------------------------- FFMA GEMM
def _cdiv(a, b):
    return -(-a // b)


def _gemm_plan(M, N, K, batch=1, batch_reduce=False, split=True):
    """(tile config, reduction slices, split-reduce kernel or None) of gn_sgemm: a restatement of make_plan and of
    the reduce-kernel choice.  `split`: a workspace is passed."""
    if M >= 1024:
        cfg = 2 if N <= 16 else 1 if N <= 32 else 0
    elif M <= 32 or N <= 32 or M * N <= 16384:
        cfg = 3
    else:
        cfg = 0
    bk = 16
    if cfg == 3 and K >= 256:
        cfg, bk = 4, 64
    bm, bn = {0: (64, 64), 1: (128, 32), 2: (128, 16), 3: (32, 32), 4: (32, 32)}[cfg]
    kt = _cdiv(K, bk)
    indep = 1 if batch_reduce else batch
    iters = (batch if batch_reduce else 1) * kt
    tiles = _cdiv(M, bm) * _cdiv(N, bn) * indep
    splits = 1
    if split and K > 0 and iters >= 4 and tiles < 296:
        want = (3 * 148 if bk >= 64 else 296) // tiles
        cap = iters if bk >= 64 else iters // 2
        splits = max(1, min(want, cap, 3 * 148))
    per = _cdiv(max(iters, 1), splits)
    splits = _cdiv(max(iters, 1), per)
    reduce = None
    if splits > 1:
        reduce = "splitk_reduce_kernel<32>" if splits >= 16 and M * N * indep <= 8192 else "splitk_reduce_kernel<1>"
    return cfg, splits, reduce


def _gemm_names(ta, tb, plan):
    cfg, _, reduce = plan
    return {f"sgemm_kernel<{int(ta)},{int(tb)},{TILES[cfg]}>"} | ({reduce} if reduce else set())


def _sgemm(ta, tb, M, N, K, A, lda, B, ldb, C, ldc, batch=1, sa=0, sb=0, sc=0, br=False, alpha=1.0, acc=False,
           add=None, mask=None, rows=None, split=True):
    """lib.gn_sgemm on raw pointers (A, B, C: ints; add / mask: (ptr, ld)); split: pass a workspace of exactly
    gn_sgemm_workspace_bytes.  Returns the instances it must have launched."""
    from gripnet_b200 import _lib
    from gripnet_b200.graph import _stream
    lib = _lib.load()
    nbytes = int(lib.gn_sgemm_workspace_bytes(M, N, K, batch, int(br))) if split else 0
    plan = _gemm_plan(M, N, K, batch, br, nbytes > 0)
    indep = 1 if br else batch
    assert nbytes == (4 * indep * plan[1] * M * N if plan[1] > 1 else 0)      # the [batch][splits][M][N] workspace
    ws = torch.empty(nbytes // 4, device=_dev()) if nbytes else None
    _lib.check(lib.gn_sgemm(int(ta), int(tb), M, N, K, A, lda, B, ldb, C, ldc, batch, sa, sb, sc, int(br),
                            float(alpha), int(acc), add[0] if add else None, add[1] if add else 0,
                            mask[0] if mask else None, mask[1] if mask else 0,
                            None if rows is None else rows.data_ptr(), 1 if split else 0,
                            None if ws is None else ws.data_ptr(), nbytes, _stream()), "gn_sgemm")
    return _gemm_names(ta, tb, plan)


def _f32(rs, *shape):
    return rs.randn(*shape).astype(np.float32)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(_dev())


# (M, N, K): both sides of M = 1024, N at the 16 / 32 tile widths and +-1, K at a multiple of 16 and +-1,
# K at the 256 threshold of the deep k-tile, M * N on both sides of 16384
GEMM_SHAPES = (
    (1023, 16, 64), (1024, 16, 64), (1025, 15, 63), (4097, 16, 65),          # cfg 3 just below, cfg 2
    (1024, 32, 48), (1025, 17, 31), (4097, 31, 100), (1024, 33, 47),         # cfg 1, cfg 0 at N = 33
    (33, 31, 17), (1, 1, 1), (64, 64, 255),                                  # cfg 3
    (32, 33, 300), (31, 32, 256), (48, 16, 5000),                            # cfg 4 (5000: 79 slices, reduce<32>)
    (200, 100, 48), (129, 129, 64), (128, 128, 16))                          # cfg 0 (M * N > 16384); 16384: cfg 3


def _gemm_case(ta, tb, M, N, K):
    """op(A) op(B) against float64 with the split on (workspace) and off (NULL), each run twice bit-identical."""
    rs = np.random.RandomState(M * 3 + N * 5 + K + 2 * ta + tb)
    A = _f32(rs, *((K, M) if ta else (M, K)))
    B = _f32(rs, *((N, K) if tb else (K, N)))
    ref = (A.T if ta else A).astype(np.float64) @ (B.T if tb else B).astype(np.float64)
    At, Bt = _t(A), _t(B)
    names, runs = set(), {}
    for split in (False, True):
        for rep in range(2):
            C = torch.full((M, N), float("nan"), device=_dev())
            names |= _sgemm(ta, tb, M, N, K, At.data_ptr(), A.shape[1], Bt.data_ptr(), B.shape[1], C.data_ptr(), N,
                            split=split)
            assert rel_err(C, ref) < TOL, (ta, tb, M, N, K, split)
            runs[split, rep] = C
        assert torch.equal(_bits(runs[split, 0]), _bits(runs[split, 1])), (ta, tb, M, N, K, split)
    return names, set()


def _mask_values(rs, shape):
    """A ReLU mask with +0, -0, negative, NaN and positive entries: only the positive ones keep the output."""
    m = rs.uniform(0.1, 2, shape).astype(np.float32)
    flat = m.reshape(-1)
    flat[0::7], flat[1::7], flat[2::7], flat[3::7] = 0.0, -0.0, np.nan, -1.5
    return m


def _gemm_epilogue_case(M, N, K, layout):
    """alpha, accumulate, addend and mask together, in the GEMM kernel (no split) and in the split-reduce kernel,
    with C, addend and mask at `layout`.  The float4 epilogue is taken only without the split, by the tiles whose
    threads own 4 columns (cfg 0 / 1 / 2) and with C, addend and mask aligned ("contiguous" here); cfg 3 / 4 (2
    columns per thread), the split-reduce kernel (one output per thread) and the other layouts are scalar."""
    rs = np.random.RandomState(M + N + K + LAYOUTS.index(layout))
    A, B = _f32(rs, M, K), _f32(rs, K, N)
    C0, add, mask = _f32(rs, M, N), _f32(rs, M, N), _mask_values(rs, (M, N))
    keep = mask > 0
    ref = np.where(keep, 0.75 * (A.astype(np.float64) @ B) + C0 + add, 0.0)
    At, Bt = _t(A), _t(B)
    addb, ca = _place(add, layout, float("nan"))
    maskb, cm = _place(mask, layout, float("nan"))
    names = set()
    for split in (False, True):
        cb, cc = _place(C0, layout, SPMM_SENTINEL)
        names |= _sgemm(0, 0, M, N, K, At.data_ptr(), K, Bt.data_ptr(), N, cb.data_ptr() + 4 * cc, cb.stride(0),
                        alpha=0.75, acc=True, add=(addb.data_ptr() + 4 * ca, addb.stride(0)),
                        mask=(maskb.data_ptr() + 4 * cm, maskb.stride(0)), split=split)
        out = cb[:, cc:cc + N]
        assert rel_err(out, ref) < TOL, (M, N, K, layout, split)
        assert bool((_bits(out)[torch.from_numpy(~keep).to(_dev())] == 0).all())     # +0 wherever the mask is not > 0
        assert bool((_outside(cb, cc, N) == SPMM_SENTINEL).all())
    return names, set()


def _gemm_batch_case(kind):
    rs = np.random.RandomState(len(kind))
    d = _dev()
    names = set()
    if kind.startswith("indep"):
        # independent batch entries with the split: workspace [batch][splits][M][N], slice zb of the grid
        M, N, K, b = {"indep_r32": (40, 24, 3000, 3), "indep_r1": (1030, 16, 160, 3)}[kind]
        A, B = _f32(rs, b, M, K), _f32(rs, b, K, N)
        ref = np.einsum("bmk,bkn->bmn", A.astype(np.float64), B)
        At, Bt = _t(A), _t(B)
        for split in (False, True):
            C = torch.full((b, M, N), float("nan"), device=d)
            names |= _sgemm(0, 0, M, N, K, At.data_ptr(), K, Bt.data_ptr(), N, C.data_ptr(), N, batch=b,
                            sa=M * K, sb=K * N, sc=M * N, split=split)
            assert rel_err(C, ref) < TOL, (kind, split)
        assert _gemm_plan(M, N, K, b)[1] > 1
    elif kind == "shared_a":
        # the RGCN dW fallback: dW[r] = H^T dY[:, r, :], one H for every relation (sa = 0), transposed A
        n, k, f, r = 3000, 13, 7, 4
        h, dy = _f32(rs, n, k), _f32(rs, n, r * f)
        ref = np.einsum("nk,nrf->rkf", h.astype(np.float64), dy.reshape(n, r, f))
        ht, dyt = _t(h), _t(dy)
        for split in (False, True):
            C = torch.full((r, k, f), float("nan"), device=d)
            names |= _sgemm(1, 0, k, f, n, ht.data_ptr(), k, dyt.data_ptr(), r * f, C.data_ptr(), f, batch=r,
                            sa=0, sb=f, sc=k * f, split=split)
            assert rel_err(C, ref) < TOL, (kind, split)
    elif kind.startswith("reduce"):
        # the RGCN dH: dH = mask(dH + sum_r dY[:, r, :] W[r]^T), batch_reduce + accumulate + mask with the split
        n, k, f, r = {"reduce_pose": (645, 48, 16, 8), "reduce_odd": (2500, 13, 21, 3)}[kind]
        dy, w, d0, mask = _f32(rs, n, r * f), _f32(rs, r, k, f), _f32(rs, n, k), _mask_values(rs, (n, k))
        ref = np.where(mask > 0, np.einsum("nrf,rkf->nk", dy.reshape(n, r, f).astype(np.float64), w) + d0, 0.0)
        assert _gemm_plan(n, k, f, r, True)[1] > 1
        mt, dyt, wt = _t(mask), _t(dy), _t(w)
        for split in (False, True):
            C = _t(d0.copy())
            names |= _sgemm(0, 1, n, k, f, dyt.data_ptr(), r * f, wt.data_ptr(), f, C.data_ptr(), k, batch=r,
                            sa=f, sb=k * f, sc=0, br=True, acc=True, mask=(mt.data_ptr(), k), split=split)
            assert rel_err(C, ref) < TOL, (kind, split)
    elif kind == "batched_epilogue":
        # independent batch entries share ONE addend and ONE mask (they are not offset by the batch entry)
        M, N, K, b = 64, 20, 700, 3
        A, B = _f32(rs, b, M, K), _f32(rs, b, K, N)
        add, mask = _f32(rs, M, N), _mask_values(rs, (M, N))
        ref = np.where(mask > 0, np.einsum("bmk,bkn->bmn", A.astype(np.float64), B) + add, 0.0)
        at, mt, At, Bt = _t(add), _t(mask), _t(A), _t(B)
        for split in (False, True):
            C = torch.full((b, M, N), float("nan"), device=d)
            names |= _sgemm(0, 0, M, N, K, At.data_ptr(), K, Bt.data_ptr(), N, C.data_ptr(), N, batch=b,
                            sa=M * K, sb=K * N, sc=M * N, add=(at.data_ptr(), N), mask=(mt.data_ptr(), N),
                            split=split)
            assert rel_err(C, ref) < TOL, (kind, split)
    return names, set()


def _gemm_rows_case(ta):
    """a_rows (a gather of the stored A's rows, duplicates included), both layouts, split and unsplit."""
    rs = np.random.RandomState(90 + ta)
    rows = rs.randint(0, 300, 2000 if ta else 1100)
    rows[:10] = rows[10]                                  # duplicates
    if ta:
        A, B = _f32(rs, 300, 24), _f32(rs, 2000, 16)
        ref = A[rows].astype(np.float64).T @ B
        M, N, K, lda = 24, 16, 2000, 24
    else:
        A, B = _f32(rs, 300, 40), _f32(rs, 40, 16)
        ref = A[rows].astype(np.float64) @ B
        M, N, K, lda = 1100, 16, 40, 40
    rt, At, Bt = _t(rows.astype(np.int64)), _t(A), _t(B)
    names = set()
    for split in (False, True):
        C = torch.full((M, N), float("nan"), device=_dev())
        names |= _sgemm(ta, 0, M, N, K, At.data_ptr(), lda, Bt.data_ptr(), N, C.data_ptr(), N, rows=rt,
                        split=split)
        assert rel_err(C, ref) < TOL, (ta, split)
    return names, set()


def _gemm_empty_k_case():
    """K == 0 with NULL A and B: the output is the epilogue of a zero product."""
    rs = np.random.RandomState(5)
    M, N = 50, 20
    C0, add, mask = _f32(rs, M, N), _f32(rs, M, N), _mask_values(rs, (M, N))
    C, addt, maskt = _t(C0.copy()), _t(add), _t(mask)
    names = _sgemm(0, 0, M, N, 0, None, 1, None, 1, C.data_ptr(), N, alpha=2.0, acc=True,
                   add=(addt.data_ptr(), N), mask=(maskt.data_ptr(), N))
    assert torch.equal(C.cpu(), torch.from_numpy(np.where(mask > 0, C0 + add, 0.0).astype(np.float32)))
    C = torch.full((M, N), float("nan"), device=_dev())
    names |= _sgemm(1, 1, M, N, 0, None, 1, None, 1, C.data_ptr(), N)
    assert torch.equal(C, torch.zeros_like(C))
    return names, set()


# ---------------------------------------------------------------------------------------------------- elementwise
def _map2d_case():
    """All four ops through both kernels; EW_ADD accumulates into a strided dst; columns beside dst untouched."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(11)
    n, names = 1000, set()
    for op in range(4):
        for vec in (True, False):
            F = 16 if vec else 13
            s, d0 = _f32(rs, n, F), _f32(rs, n, F)
            sb, cs = _place(s, "contiguous" if vec else "offset1", float("nan"))
            db, cd = _place(d0, "offset4" if vec else "stride_f5", SPMM_SENTINEL)
            ops.map2d(op, ops.M(sb, cs, F), ops.M(db, cd, F))
            s64 = s.astype(np.float64)
            want = [s64, np.abs(s64), np.maximum(s64, 0.0), d0 + s64][op]
            out = db[:, cd:cd + F]
            if op == 3:
                assert rel_err(out, want) < TOL
            else:
                assert torch.equal(out.cpu(), torch.from_numpy(want.astype(np.float32)))
            assert bool((_outside(db, cd, F) == SPMM_SENTINEL).all())
            names.add(f"map2d{'_vec' if vec else ''}_kernel<{op}>")
    return names, set()


def _special_t(rs, n, F):
    t = _f32(rs, n, F)
    specials = np.array([0.0, -0.0, 1e-40, -1e-40, 1e-45, -1e-45, np.inf, -np.inf], np.float32)
    t.reshape(-1)[: 8 * 50] = np.tile(specials, 50)
    return t


def _bwd_case():
    """relu_bwd and abs_bwd through both kernels; abs_bwd at scale 1 and 0.5 with t = +-0, +-denormal, +-Inf."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(12)
    n, names = 700, set()
    for vec in (True, False):
        F = 8 if vec else 7
        g = _f32(rs, n, F)
        y = _special_t(rs, n, F)
        gb, cg = _place(g, "contiguous" if vec else "offset1", float("nan"))
        yb, cy = _place(y, "offset4" if vec else "stride_f5", float("nan"))
        out = torch.full((n, F), float("nan"), device=_dev())
        ops.relu_bwd(ops.M(gb, cg, F), ops.M(yb, cy, F), ops.M(out))
        assert torch.equal(out.cpu(), torch.from_numpy(np.where(y > 0, g, np.float32(0))))
        names.add("relu_bwd_vec_kernel" if vec else "relu_bwd_kernel")
        for scale in (1.0, 0.5):
            out = torch.full((n, F), float("nan"), device=_dev())
            ops.abs_bwd(ops.M(gb, cg, F), ops.M(yb, cy, F), ops.M(out), scale)
            want = (g.astype(np.float64) * np.sign(y.astype(np.float64)) * scale).astype(np.float32)
            assert torch.equal(out.cpu(), torch.from_numpy(want)), (vec, scale)
            names.add("abs_bwd_vec_kernel" if vec else "abs_bwd_kernel")
    return names, set()


def _axpby_mean3_case():
    """axpby with b == NULL and with b aliasing dst (as the interGraph tail calls it), on strided views; mean3 on
    strided views, bit-equal to ((a + b) + c) / 3 evaluated on the CPU."""
    from gripnet_b200 import ops
    rs = np.random.RandomState(13)
    n, F = 900, 21
    a, d0 = _f32(rs, n, F), _f32(rs, n, F)
    ab, ca = _place(a, "offset1", float("nan"))
    db, cd = _place(d0, "stride_f5", SPMM_SENTINEL)
    ops.axpby(ops.M(ab, ca, F), 0.3, None, 0.0, ops.M(db, cd, F))
    assert rel_err(db[:, cd:cd + F], 0.3 * a.astype(np.float64)) < TOL
    db, cd = _place(d0, "stride_f5", SPMM_SENTINEL)
    D = ops.M(db, cd, F)
    ops.axpby(ops.M(ab, ca, F), 0.5, D, -1.25, D)
    assert rel_err(db[:, cd:cd + F], 0.5 * a.astype(np.float64) - 1.25 * d0) < TOL
    assert bool((_outside(db, cd, F) == SPMM_SENTINEL).all())
    xs = [_place(_f32(rs, n, F), lay, float("nan")) for lay in ("offset1", "offset4", "stride_f5")]
    views = [b[:, c:c + F] for b, c in xs]
    out = ops.mean3(*views)
    v = [t.cpu() for t in views]
    assert torch.equal(out.cpu(), ((v[0] + v[1]) + v[2]) / 3)
    return {"axpby_kernel", "mean3_kernel"}, set()


COLSUM_F = (1, 7, 48, 255, 256, 257, 513)
COLSUM_N = (0, 1, 255, 592 * 256 + 1, 600_000)


def _colsum_case(F):
    """Column sums of a misaligned strided view across the cols_per_pass / row_lanes boundaries and past 256 rows
    per block (n > 592 * 256)."""
    from gripnet_b200 import ops
    g = torch.Generator(device=_dev()).manual_seed(F)
    names = set()
    for n in COLSUM_N:
        buf = torch.randn(n, F + 1, device=_dev(), generator=g)
        out = torch.full((F,), float("nan"), device=_dev())
        ops.colsum(ops.M(buf, 1, F), out)
        want = buf[:, 1:].cpu().numpy().sum(0, dtype=np.float64)
        if n == 0:
            assert torch.equal(out, torch.zeros_like(out))
        else:
            assert rel_err(out, want) < TOL, (F, n)
            names |= {"colsum_partial_kernel", "colsum_final_kernel"}
        del buf
    return names, set()


def _probs(rs, n):
    p = rs.uniform(0.01, 0.99, n).astype(np.float32)
    k = min(n, 6)
    p[:k] = np.array([0.0, 1e-7, 1e-30, 1.0, np.float32(1) - np.float32(6e-8), 0.5], np.float32)[:k]
    return p


def _elem_rel_err(a, b):
    """Largest per-element relative error |a - b| / |b|; inf unless a is exactly 0 wherever b is.  The gradients of
    the losses span ~12 orders of magnitude within one tensor (p + eps at 1e-13 next to p ~ 0.5), so a per-tensor
    max-relative error would see only the largest entries."""
    a = torch.as_tensor(a).detach().to("cpu", torch.float64)
    b = torch.as_tensor(b).detach().to("cpu", torch.float64)
    if a.shape != b.shape:
        return float("inf")
    if b.numel() == 0:
        return 0.0
    zero = b == 0
    if bool((a[zero] != 0).any()):
        return float("inf")
    return float(((a - b).abs()[~zero] / b.abs()[~zero]).max()) if bool((~zero).any()) else 0.0


def _check_grad(got, want, what):
    """got against float64 per element; and the check itself must reject `want` with its tail zeroed (a backward
    that wrote only the first grid pass) or with one bulk entry off by 1e-4 of its value."""
    assert _elem_rel_err(got, want) < TOL, what
    n = want.numel()
    if n > 10:
        w32 = want.float().flatten()
        tail, bulk = w32.clone(), w32.clone()
        tail[n // 2:] = 0.0
        bulk[n - 1] *= 1 + 1e-4
        assert _elem_rel_err(tail.view_as(want), want) > TOL and _elem_rel_err(bulk.view_as(want), want) > TOL


def _loss_case():
    """Link-prediction and node-classification losses, forward and backward: past the 296-block grid-stride cap,
    with no positives or no negatives, probabilities at and near 0 and 1; against float64 with the same eps."""
    from gripnet_b200 import ops
    eps = ops.EPS
    rs = np.random.RandomState(14)
    d = _dev()
    for n_pos, n_neg in ((400_000, 350_000), (0, 5000), (5000, 0), (1, 1)):
        pos, neg = _probs(rs, n_pos), _probs(rs, n_neg)
        pr, nr = torch.from_numpy(pos).double().requires_grad_(True), torch.from_numpy(neg).double().requires_grad_(True)
        ref = torch.zeros((), dtype=torch.float64)
        if n_pos:
            ref = ref - torch.log(pr + eps).mean()
        if n_neg:
            ref = ref - torch.log(1 - nr + eps).mean()
        (ref * 1.7).backward()
        pc, nc = _t(pos).requires_grad_(True), _t(neg).requires_grad_(True)
        loss = ops.LinkPredLoss.apply(pc, nc)
        (loss * 1.7).backward()
        assert rel_err(loss, ref) < TOL, (n_pos, n_neg)
        _check_grad(pc.grad, pr.grad if n_pos else torch.zeros(0), ("pos", n_pos, n_neg))
        _check_grad(nc.grad, nr.grad if n_neg else torch.zeros(0), ("neg", n_pos, n_neg))
    for n, C in ((400_000, 3), (1, 5)):
        score = rs.dirichlet(np.ones(C), n).astype(np.float32)
        lab = rs.randint(0, C, n)
        k = min(n, 4)
        score[np.arange(k), lab[:k]] = np.array([0.0, 1e-7, 1.0, np.float32(1) - np.float32(6e-8)], np.float32)[:k]
        sr = torch.from_numpy(score).double().requires_grad_(True)
        ref = -torch.log(sr[torch.arange(n), torch.from_numpy(lab)] + eps).mean()
        (ref * 0.6).backward()
        sc = _t(score).requires_grad_(True)
        loss = ops.NodeClassLoss.apply(sc, _t(lab.astype(np.int64)))
        (loss * 0.6).backward()
        assert rel_err(loss, ref) < TOL, (n, C)
        _check_grad(sc.grad, sr.grad, ("score", n, C))            # non-label entries: exactly 0
    return {f"{l}_loss_{s}_kernel" for l in ("lp", "nc") for s in ("partial", "final", "bwd")}, set()


# ----------------------------------------------------------------------------------------------- layer stacks
STACK_NODES = (700, 2500, 6000, 40_000)
STACK_WIDTHS = {"aligned": (16, 32, 16), "odd": (13, 21, 7)}
STACK_VARIANTS = (("gcn", "plain"), ("gcn", "catout_weighted"), ("rgcn", "plain"), ("rgcn", "catout"))
N_REL, N_BASE = 3, 2


def _stack_graph(n, seed):
    """~6 random in-edges per node without self-loops, plus 600 into node 5 (a row split over chunks), relation-
    sorted for the RGCN: (edge_index [2, E], edge_type, range_list, edge_weight) on the CPU."""
    rs = np.random.RandomState(seed)
    e = 6 * n
    src = np.r_[rs.randint(0, n, e), rs.randint(6, n, 600)]
    dst = np.r_[rs.randint(0, n, e), np.full(600, 5)]
    dst = np.where(src == dst, (dst + 1) % n, dst)
    et = rs.randint(0, N_REL, len(src))
    order = np.argsort(et, kind="stable")
    src, dst, et = src[order], dst[order], et[order]
    ends = np.cumsum(np.bincount(et, minlength=N_REL))
    rl = np.stack([np.r_[0, ends[:-1]], ends], 1)
    w = rs.uniform(0.5, 1.5, len(src))
    return (torch.from_numpy(np.stack([src, dst])), torch.from_numpy(et), torch.from_numpy(rl), torch.from_numpy(w))


class _Relu(torch.autograd.Function):
    """ReLU whose backward mask follows the kernel's output where the float64 pre-activation lies within 1e-5 of
    its largest magnitude of 0 (float32 rounding may put such an entry on either side)."""

    @staticmethod
    def forward(ctx, z, h32):
        keep = z > 0
        if h32 is not None:
            near = z.abs() < 1e-5 * float(z.abs().max())
            keep = torch.where(near, h32 > 0, keep)
        ctx.save_for_backward(keep)
        return z.clamp_min(0.0)

    @staticmethod
    def backward(ctx, g):
        (keep,) = ctx.saved_tensors
        return g * keep, None


def _stack_ref(kind, x, params, ei, et, rl, w, catout, h32=None):
    """Float64 restatement of homoGraph on an edge list (index_add_, no n x n matrix): GCN with the symmetric
    normalisation of A + I (in-degree by target, weighted), RGCN with one mean over all in-edges plus the root term;
    ReLU after every layer; optional concat of x and every layer's output."""
    n = x.size(0)
    src, dst = ei[0], ei[1]
    outs, h = [x], x
    if kind == "gcn":
        w = torch.ones(src.numel(), dtype=torch.float64) if w is None else w
        deg = torch.ones(n, dtype=torch.float64).index_add_(0, dst, w)
        dis = deg.rsqrt()
        norm = dis[src] * w * dis[dst]
        for l, (W, b) in enumerate(params):
            y = h @ W
            z = torch.zeros(n, W.size(1), dtype=torch.float64).index_add_(0, dst, norm[:, None] * y[src])
            z = z + (dis * dis)[:, None] * y + b
            h = _Relu.apply(z, None if h32 is None else h32[l])
            outs.append(h)
    else:
        cnt = torch.zeros(n, dtype=torch.float64).index_add_(0, dst, torch.ones(src.numel(), dtype=torch.float64))
        inv = 1.0 / cnt.clamp_min(1.0)
        rel = torch.repeat_interleave(torch.arange(len(rl)), rl[:, 1] - rl[:, 0])
        assert torch.equal(rel, et)
        for l, (basis, att, root) in enumerate(params):
            wr = torch.einsum("rb,bkf->rkf", att, basis)
            y = torch.einsum("nk,rkf->nrf", h, wr)
            z = torch.zeros(n, root.size(1), dtype=torch.float64).index_add_(0, dst, y[src, rel])
            z = z * inv[:, None] + h @ root
            h = _Relu.apply(z, None if h32 is None else h32[l])
            outs.append(h)
    return torch.cat(outs, 1) if catout else h


def _stack_model(kind, dims, seed):
    import gripnet_b200 as gb
    torch.manual_seed(seed)
    m = gb.homoGraph(list(dims), multi_relational=kind == "rgcn", n_rela=N_REL, n_base=N_BASE)
    if kind == "gcn":
        with torch.no_grad():
            for c in m.conv_list:
                c.bias.normal_(std=0.1)
    return m


def _stack_params(kind, m):
    if kind == "gcn":
        return [(c.weight, c.bias) for c in m.conv_list]
    return [(c.basis, c.att, c.root) for c in m.conv_list]


def _stack_routing(kind, n, dims, aligned):
    """(instances of the three files expected, tensor-core kernels expected, tensor-core kernels excluded): a
    restatement of the routing of ops.sgemm (gn_tc_gemm for plain products of >= 4096 aligned rows and k >= 16),
    weight_grad (gn_tc_tn from 2^15 aligned rows, and for every aligned relational dW) and rel_transform."""
    def tc(m, k):
        return aligned and m >= 4096 and k >= 16

    want = set()
    for k, f in zip(dims[:-1], dims[1:]):
        if kind == "gcn":
            if not tc(n, k):
                want |= _gemm_names(0, 0, _gemm_plan(n, f, k))                       # X W
            if not (aligned and n >= 1 << 15):
                want |= _gemm_names(1, 0, _gemm_plan(k, f, n))                       # dW = H^T dY
            if not tc(n, f):
                want |= _gemm_names(0, 1, _gemm_plan(n, k, f))                       # dH = dY W^T
        else:
            want |= _gemm_names(0, 0, _gemm_plan(N_REL, k * f, N_BASE))              # W[r] = att basis
            if not tc(n, k):
                want |= _gemm_names(0, 0, _gemm_plan(n, f, k))                       # X root
            if not aligned:
                want |= _gemm_names(0, 0, _gemm_plan(n, f, k, N_REL))                # X W[r], batched
                want |= _gemm_names(1, 0, _gemm_plan(k, f, n, N_REL))                # dW[r], batched split fallback
            want |= _gemm_names(1, 0, _gemm_plan(k, f, n))                           # droot
            want |= _gemm_names(0, 1, _gemm_plan(N_REL, N_BASE, k * f))              # datt
            want |= _gemm_names(1, 0, _gemm_plan(N_BASE, k * f, N_REL))              # dbasis
            if not tc(n, f):
                want |= _gemm_names(0, 1, _gemm_plan(n, k, f))                       # dZ root^T
            want |= _gemm_names(0, 1, _gemm_plan(n, k, f, N_REL, True))              # + sum_r dY_r W_r^T, masked
    if kind == "gcn":
        tc_gemm, tc_tn = aligned and n >= 4096, aligned and n >= 1 << 15
    else:
        tc_gemm = tc_tn = aligned
    on = {name for name, b in (("tc_gemm_kernel", tc_gemm), ("tc_tn_kernel", tc_tn)) if b}
    return want, on, TC_KERNELS - on


def _stack_case(kind, variant, n, widths):
    """One homoGraph stack: forward, dx and every parameter gradient against float64, and its routing."""
    from gripnet_b200 import graph as G
    from gripnet_b200 import ops
    d = _dev()
    dims = STACK_WIDTHS[widths]
    catout, weighted = "catout" in variant, "weighted" in variant
    seed = n + len(variant) + dims[0]
    ei, et, rl, w = _stack_graph(n, seed)
    model = _stack_model(kind, dims, seed).to(d)
    x64 = torch.randn(n, dims[0], dtype=torch.float64, generator=torch.Generator().manual_seed(seed))
    x = x64.float().to(d).requires_grad_(True)
    eid = ei.to(d)
    kw = dict(edge_type=et.to(d), range_list=rl) if kind == "rgcn" else \
        dict(edge_weight=w.float().to(d) if weighted else None)
    out = model(x, eid, if_catout=catout, **kw)
    gout = torch.randn(out.shape, dtype=torch.float64, generator=torch.Generator().manual_seed(seed + 1))
    (out * gout.float().to(d)).sum().backward()
    params = _stack_params(kind, model)
    if catout:
        offs = np.cumsum(dims)
        h32 = [out.detach()[:, offs[l]:offs[l + 1]].cpu() for l in range(len(dims) - 1)]
    else:
        # the first layer's kernel output: the same launches as the stack's first layer, as a stack of its own
        p0 = [t.detach() for t in params[0]]
        if kind == "gcn":
            h1 = ops.GcnStack.apply(x.detach(), model.conv_list[0]._graph, (True,), False, *p0)
        else:
            h1 = ops.RgcnStack.apply(x.detach(), G.rgcn_graph(eid, rl, n, N_REL), (True,), False, *p0, None)
        h32 = [h1.cpu(), out.detach().cpu()]
    p64 = [[t.detach().double().cpu().requires_grad_(True) for t in layer] for layer in params]
    xr = x64.clone().requires_grad_(True)
    ref = _stack_ref(kind, xr, p64, ei, et, rl, w if weighted else None, catout, [h.double() for h in h32])
    (ref * gout).sum().backward()
    case = (kind, variant, n, widths)
    assert rel_err(out, ref) < TOL, case
    assert rel_err(x.grad, xr.grad) < TOL, case
    for layer, ref_layer in zip(params, p64):
        for t, r in zip(layer, ref_layer):
            assert rel_err(t.grad, r.grad) < TOL, (case, tuple(t.shape))
    want, on, off = _stack_routing(kind, n, dims, widths == "aligned")
    return want | on, off


# -------------------------------------------------------------------------------------------- profiled groups
GROUPS = {f"spmm:{lay}": [(_spmm_case, (F, lay)) for F in SPMM_WIDTHS] for lay in LAYOUTS}
GROUPS["spmm:scratch"] = [(_scratch_case, (k, F)) for k in ("50+2", "hub") for F in (29, 260)]
GROUPS.update({f"gemm:{ta}{tb}": [(_gemm_case, (ta, tb) + s) for s in GEMM_SHAPES] for ta in (0, 1) for tb in (0, 1)})
# cfg 1, 2 and 0 (float4 epilogue when contiguous and unsplit), cfg 4 with reduce<1>, cfg 4 with reduce<32>
GROUPS["gemm:epilogue"] = [(_gemm_epilogue_case, s + (lay,))
                           for s in ((1100, 24, 96), (1100, 16, 96), (200, 100, 96), (40, 20, 600), (32, 16, 4000))
                           for lay in ("contiguous", "offset1", "stride_f5")]
GROUPS["gemm:batch"] = [(_gemm_batch_case, (k,)) for k in ("indep_r32", "indep_r1", "shared_a", "reduce_pose",
                                                           "reduce_odd", "batched_epilogue")]
GROUPS["gemm:rows_and_empty"] = [(_gemm_rows_case, (0,)), (_gemm_rows_case, (1,)), (_gemm_empty_k_case, ())]
GROUPS["ew:map2d"] = [(_map2d_case, ())]
GROUPS["ew:bwd"] = [(_bwd_case, ())]
GROUPS["ew:axpby_mean3"] = [(_axpby_mean3_case, ())]
GROUPS["ew:colsum"] = [(_colsum_case, (F,)) for F in COLSUM_F]
GROUPS["ew:loss"] = [(_loss_case, ())]
GROUPS.update({f"stack:{k}:{v}:{n}:{w}": [(_stack_case, (k, v, n, w))]
               for k, v in STACK_VARIANTS for n in STACK_NODES for w in STACK_WIDTHS})


def _profile_all():
    """Kernel names per profiled group: {group: sorted names}."""
    out = {}
    for key, cases in GROUPS.items():
        out[key] = sorted(_kernel_names(lambda: [fn(*args) for fn, args in cases]))
        torch.cuda.empty_cache()
    return out


@pytest.fixture(scope="module")
def profiled():
    """Kernel names per group of cases, recorded by torch.profiler in a process of its own (a profiler session in
    the test process can leave the sessions of later test modules without kernel records)."""
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], env=dict(os.environ), capture_output=True,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return {k: set(v) for k, v in json.loads(res.stdout.strip().splitlines()[-1]).items()}


def _run_group(key, profiled, exact=False):
    """The cases of group `key` against float64; each case's expected instances must be among those the group ran,
    its excluded ones absent.  exact: the group launches nothing of the three files but what its cases expect."""
    ran, expected = profiled[key], set()
    for fn, args in GROUPS[key]:
        want, absent = fn(*args)
        assert want <= ran, (key, args, sorted(want - ran), sorted(ran))
        assert not (absent & ran), (key, args, sorted(absent & ran))
        expected |= want
    if exact:
        assert ran - TC_KERNELS == expected, (key, sorted(ran ^ expected))


@pytest.mark.parametrize("layout", LAYOUTS)
def test_spmm_instance_matrix(layout, profiled):
    """Widths reaching all 12 spmm_kernel instances and both panel loops (128 + 128 + 4 float4 columns, 32 + 32 + 6
    scalar ones), x and out at `layout`, four chunk structures, five epilogues, non-finite unreferenced rows."""
    _run_group(f"spmm:{layout}", profiled, exact=True)
    if layout == "contiguous":
        assert {F: _spmm_plan(F, F, F, True) for F in (8, 24, 70, 260)} == {
            8: ["spmm_kernel<2,4>"], 24: ["spmm_kernel<8,4>"],
            70: ["spmm_kernel<32,1>", "spmm_kernel<32,1>", "spmm_kernel<8,1>"],
            260: ["spmm_kernel<32,4>", "spmm_kernel<32,4>", "spmm_kernel<1,4>"]}


def test_spmm_partial_scratch_bound(profiled):
    """The split-row scratch is 2 (n_chunks - n_rows) rows of min(F, 128) floats; nothing past it is written."""
    _run_group("spmm:scratch", profiled, exact=True)


@pytest.mark.parametrize("trans", ["00", "01", "10", "11"])
def test_sgemm_tile_matrix(trans, profiled):
    """All five tiles at one transpose pair, split and unsplit, at tile edges."""
    _run_group(f"gemm:{trans}", profiled, exact=True)
    ta, tb = int(trans[0]), int(trans[1])
    tiles = set()
    for M, N, K in GEMM_SHAPES:
        tiles |= _gemm_names(ta, tb, _gemm_plan(M, N, K))
    assert {n for n in tiles if n.startswith("sgemm")} == {f"sgemm_kernel<{ta},{tb},{t}>" for t in TILES.values()}


def test_sgemm_epilogue_paths(profiled):
    """alpha / accumulate / addend / mask in the GEMM kernel (float4 epilogue for cfg 0, 1 and 2 with aligned C,
    scalar otherwise) and in both split-reduce kernels."""
    _run_group("gemm:epilogue", profiled, exact=True)


def test_sgemm_batching(profiled):
    """Independent batches with the split, shared A, the RGCN's batch_reduce + accumulate + mask, and the batched
    epilogue contract: every batch entry adds the same addend and uses the same mask."""
    _run_group("gemm:batch", profiled, exact=True)


def test_sgemm_row_gather_and_empty_reduction(profiled):
    _run_group("gemm:rows_and_empty", profiled, exact=True)


@pytest.mark.parametrize("group", ["map2d", "bwd", "axpby_mean3", "colsum", "loss"])
def test_elementwise(group, profiled):
    _run_group(f"ew:{group}", profiled, exact=True)


def test_index_validation_ends_with_its_tensor():
    """A validated index tensor that is freed leaves no entry behind: a new tensor of the same shape in its recycled
    storage (the caching allocator hands the block straight back) is checked again and its bad id raises."""
    from gripnet_b200 import graph
    good = torch.zeros(64, dtype=torch.int64, device=_dev())
    graph.validate_index(good, 10, "ids")
    del good
    bad = torch.full((64,), 10, dtype=torch.int64, device=_dev())
    with pytest.raises(IndexError):
        graph.validate_index(bad, 10, "ids")


def test_stack_reference_matches_dense64():
    """The sparse float64 restatement used below against oracle/dense64 at a small n."""
    import gripnet_b200 as gb
    from oracle import dense64
    n = 60
    ei, et, rl, w = _stack_graph(n, 3)
    x = torch.randn(n, 13, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    for kind, catout, weighted in (("gcn", False, False), ("gcn", True, True), ("rgcn", True, False)):
        m = gb.homoGraph([13, 21, 7], multi_relational=kind == "rgcn", n_rela=N_REL, n_base=N_BASE)
        p = {k: v.detach().double() for k, v in m.state_dict().items()}
        params = [[p[f"conv_list.{l}.{k}"] for k in (("weight", "bias") if kind == "gcn" else ("basis", "att", "root"))]
                  for l in range(2)]
        if kind == "gcn":
            for l in range(2):
                params[l][1] = torch.randn(21 if l == 0 else 7, dtype=torch.float64) * 0.1
                p[f"conv_list.{l}.bias"] = params[l][1]
        ref = _stack_ref(kind, x, params, ei, et, rl, w if weighted else None, catout)
        dense = dense64.homo(p, x, ei, w if weighted else None, rl, catout, kind == "rgcn")
        assert rel_err(ref, dense) < 1e-12, (kind, catout, weighted)


@pytest.mark.parametrize("widths", list(STACK_WIDTHS))
@pytest.mark.parametrize("n", STACK_NODES)
@pytest.mark.parametrize("kind,variant", STACK_VARIANTS)
def test_layer_stack_routing(kind, variant, n, widths, profiled):
    """homoGraph stacks at node counts across M = 1024, 4096 and 2^15: forward and every gradient against float64,
    and the products routed as the dispatch rules say (FFMA tiles 1 / 2 at 2 500 rows, tc_gemm only for aligned
    operands from 4096 rows, tc_tn from 2^15 rows, the batched split FFMA dW for the odd RGCN)."""
    _run_group(f"stack:{kind}:{variant}:{n}:{widths}", profiled)
    want, on, off = _stack_routing(kind, n, STACK_WIDTHS[widths], widths == "aligned")
    if kind == "gcn" and n == 2500:
        assert {f"sgemm_kernel<0,0,{TILES[1]}>", f"sgemm_kernel<0,0,{TILES[2]}>"} <= want
    if n == 6000 and kind == "gcn":
        assert ("tc_gemm_kernel" in on) == (widths == "aligned")
    if n == 40_000 and widths == "aligned":
        assert "tc_tn_kernel" in on
    if kind == "rgcn" and widths == "odd":
        plan = _gemm_plan(21, 7, n, N_REL)
        assert plan[1] > 1 and _gemm_names(1, 0, plan) <= want


def test_every_instance_ran(profiled):
    """The cases above reach every instance of spmm.cu, gemm.cu and elementwise.cu, and nothing else of them: one
    added to those files needs a case here."""
    seen = set().union(*profiled.values()) - TC_KERNELS
    assert seen >= ALL_KERNELS, sorted(ALL_KERNELS - seen)
    assert seen <= ALL_KERNELS, sorted(seen - ALL_KERNELS)
    assert len(ALL_KERNELS) == 56


if __name__ == "__main__":          # the `profiled` fixture's child process
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    print(json.dumps(_profile_all()))
