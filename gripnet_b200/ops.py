"""``torch.autograd.Function`` wrappers over the C ABI (``include/gripnet_b200.h``).

Each Function covers a whole module-level stage (a stack of GCN / RGCN layers, a
decoder, a loss) so that intermediate tensors the reference materialises — the
``[E,F]`` message tensors, ``[E,D]`` decoder gathers, zero-padded inter-graph
inputs, ``torch.cat`` copies — never exist, and so that ReLU masks / concat-slice
gradients are fused into the producing kernels' epilogues.

PyTorch is used for device memory (``torch.empty``) and streams only; every
arithmetic step is a kernel of ``libgripnet_b200.so``.
"""
import weakref

import torch

from . import _lib, streams
from .graph import _ptr, _stream, _ws, require_cuda, validate_index

EPS = 1e-13  # reference gripnet/utils.py:10


class M:
    """A row-major fp32 matrix view: (tensor kept alive, pointer, leading dim, rows, cols)."""
    __slots__ = ("t", "ptr", "ld", "n", "f")

    def __init__(self, t, col0=0, width=None):
        assert t.dim() == 2 and t.stride(1) == 1 and t.dtype == torch.float32
        self.t = t
        self.n = t.size(0)
        self.f = t.size(1) - col0 if width is None else width
        self.ld = t.stride(0) if t.size(0) > 1 else max(t.size(1), 1)
        self.ptr = t.data_ptr() + 4 * col0


def _as_rows(x, name):
    """fp32 CUDA matrix with unit column stride (copy only if needed)."""
    require_cuda(x, name)
    if x.dtype != torch.float32:
        raise RuntimeError(f"gripnet_b200: {name} must be float32")
    if x.dim() != 2:
        raise RuntimeError(f"gripnet_b200: {name} must be 2-D")
    if x.stride(1) != 1 or (x.size(0) > 1 and x.stride(0) < x.size(1)):
        x = x.contiguous()
    return x


def _new(n, f, like):
    return torch.empty((n, f), dtype=torch.float32, device=like.device)


class Slot:
    """Rows of a matrix that may have to be all-gathered before a SpMM reads them.

    Single GPU: a plain ``[n, f]`` matrix (``full`` is the matrix itself).  Partitioned run
    (``parallel.py``): ``full`` is the ``[world*B, f]`` gather buffer, ``m`` views this rank's slot, so
    the producing kernel writes in place and ``gather()`` completes the buffer with one in-place
    NCCL all-gather (gathered row index == global node id)."""
    __slots__ = ("m", "full", "dctx", "halo")

    def __init__(self, m, full=None, dctx=None, halo=None):
        """``Slot(m)`` wraps an existing local matrix that needs no gather; ``alloc`` makes a new slot."""
        self.m, self.full = m, m if full is None else full
        self.dctx, self.halo = dctx, halo

    @classmethod
    def alloc(cls, n_local, f, like, dctx=None, block=None, halo=None):
        if dctx is None:
            return cls(M(_new(n_local, f, like)))
        if halo is not None:
            # halo-packed operand (graph.HaloPlan): own rows first, then only the referenced rows of each peer
            buf = dctx.slot_buffer(halo.rows, f, like, uniform=False)
            return cls(M(buf[:n_local]), M(buf), dctx, halo)
        buf = dctx.slot_buffer(dctx.world * block, f, like)
        return cls(M(buf[dctx.rank * block: dctx.rank * block + n_local]), M(buf), dctx)

    def gather(self):
        if self.dctx is not None:
            if self.halo is not None:
                self.dctx.halo_gather(self.full.t, self.halo)
            else:
                self.dctx.all_gather_slots(self.full.t)
        return self.full


def _reduce(dctx, t):
    """Partial sums of a replicated parameter's gradient -> all-reduce (no-op on one GPU)."""
    if dctx is not None:
        dctx.reduce_param_grad_(t)
    return t


# ----------------------------------------------------------------------------
# thin kernel wrappers
# ----------------------------------------------------------------------------
def spmm(csr, x, out, F, row_scale=None, bias=None, addend=None, relu=False):
    lib = _lib.load()
    partial = csr.partial(min(F, 128))
    _lib.check(lib.gn_spmm(csr.ref, x.ptr, x.ld, F, _ptr(row_scale), _ptr(bias),
                           addend.ptr if addend is not None else None, addend.ld if addend is not None else 0,
                           int(relu), out.ptr, out.ld, _ptr(partial), _stream()), "gn_spmm")


# dense-transform dispatch: tall products (M >= _TC_MIN_M) go to the tcgen05 3xTF32 kernel, the rest to the
# CUDA-core kernel
_TC_MIN_M = 4096


def _tc_eligible(ta, m, n, k, a_ptr, lda, c_ptr, ldc, batch, alpha, accumulate, addend, mask, a_rows):
    if ta or batch != 1 or a_rows is not None or accumulate or alpha != 1.0:
        return False
    if m < _TC_MIN_M or k < 16:
        return False
    if k % 4 or lda % 4 or ldc % 4 or a_ptr % 16 or c_ptr % 16 or k > 4096:
        return False
    for e in (addend, mask):
        if e is not None and (e.ld % 4 or e.ptr % 16):
            return False
    return True


def sgemm(ta, tb, m, n, k, a_ptr, lda, b_ptr, ldb, c_ptr, ldc, device, batch=1, sa=0, sb=0, sc=0, batch_reduce=False,
          alpha=1.0, accumulate=False, addend=None, mask=None, a_rows=None, split_k=True):
    """C = epilogue(alpha * op(A) op(B)).  Tall plain products go to the tcgen05 3xTF32 kernel
    (``gn_tc_gemm``); everything else to the FFMA kernel, where the library splits the reduction over
    CTAs when the output alone cannot fill the GPU (deterministic slice-order sum through ``ws``)."""
    lib = _lib.load()
    if m > 0 and n > 0 and k > 0 and _tc_eligible(ta, m, n, k, a_ptr, lda, c_ptr, ldc, batch, alpha, accumulate,
                                                  addend, mask, a_rows):
        nbytes = int(lib.gn_tc_gemm_workspace_bytes(m, n, k))
        if nbytes:
            img = _ws(nbytes, device)
            _lib.check(lib.gn_tc_gemm(int(tb), m, n, k, a_ptr, lda, b_ptr, ldb, c_ptr, ldc,
                                      addend.ptr if addend is not None else None,
                                      addend.ld if addend is not None else 0,
                                      mask.ptr if mask is not None else None, mask.ld if mask is not None else 0,
                                      _ptr(img), nbytes, _stream()), "gn_tc_gemm")
            return
    ws, ws_bytes = None, 0
    if split_k:
        ws_bytes = int(lib.gn_sgemm_workspace_bytes(m, n, k, batch, int(batch_reduce)))
        if ws_bytes:
            ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=device)
            streams.keep(ws)
    _lib.check(lib.gn_sgemm(int(ta), int(tb), m, n, k, a_ptr, lda, b_ptr, ldb, c_ptr, ldc, batch, sa, sb, sc,
                            int(batch_reduce), float(alpha), int(accumulate),
                            addend.ptr if addend is not None else None, addend.ld if addend is not None else 0,
                            mask.ptr if mask is not None else None, mask.ld if mask is not None else 0,
                            _ptr(a_rows), 1 if ws is not None else 0, _ptr(ws), ws_bytes, _stream()), "gn_sgemm")


# relation transform Y[:, r, :] = X W[r]: tensor cores whenever the 3xTF32 kernel's alignment rules hold
def _rel_tc_ok(k, ldx, ldy, x_ptr, y_ptr):
    return k % 4 == 0 and ldx % 4 == 0 and ldy % 4 == 0 and x_ptr % 16 == 0 and y_ptr % 16 == 0


def rel_transform(x, w, y, r, k, f, device, image=None):
    """``x``: M view [n, k]; ``w``: contiguous [r, k, f] tensor; ``y``: M view [n, r*f].  ``image``: the tensor-core
    operand image of ``w`` for ``n`` rows when a ``RelPrologue`` already built it."""
    lib = _lib.load()
    n = x.n
    if n == 0:
        return
    if _rel_tc_ok(k, x.ld, y.ld, x.ptr, y.ptr):
        if image is not None:
            _lib.check(lib.gn_tc_gemm_rel_image(n, r, f, k, x.ptr, x.ld, _ptr(image), image.numel(), y.ptr, y.ld,
                                                _stream()), "gn_tc_gemm_rel_image")
            return
        nbytes = int(lib.gn_tc_gemm_rel_workspace_bytes(n, r, f, k))
        if nbytes:
            img = _ws(nbytes, device)
            _lib.check(lib.gn_tc_gemm_rel(n, r, f, k, x.ptr, x.ld, w.data_ptr(), y.ptr, y.ld, _ptr(img), nbytes,
                                          _stream()), "gn_tc_gemm_rel")
            return
    sgemm(False, False, n, f, k, x.ptr, x.ld, w.data_ptr(), f, y.ptr, y.ld, device, batch=r, sa=0, sb=k * f, sc=f)


def rel_weights(basis, att):
    """``W[r] = sum_b att[r, b] basis[b]`` (``layers.py:172-173``) as a contiguous [r, k, f] tensor."""
    nb, k, f = basis.shape
    r = att.size(0)
    bs, at = basis.contiguous(), att.contiguous()
    w = torch.empty((r, k, f), dtype=torch.float32, device=basis.device)
    sgemm(False, False, r, k * f, nb, at.data_ptr(), nb, bs.data_ptr(), k * f, w.data_ptr(), k * f, basis.device)
    return w


class RelPrologue:
    """Everything of an RGCN stack's forward that depends on the PARAMETERS only — ``W[r]`` of every layer and its
    tensor-core operand image for ``n_rows`` input rows — launched on a background branch.  A training step creates it
    before its first kernel (``homoGraph.prologue``), so these launches are roots of the captured graph instead of
    sitting on the dependency chain between the previous supervertex and the relational layer.  ``RgcnStack.forward``
    picks the entries up by parameter identity + version and joins the branch."""

    _pending = {}

    def __init__(self, layers, n_rows):
        """``layers``: [(basis, att), ...] parameters of the stack."""
        lib = _lib.load()
        self.branch = streams.Branch(background=True)
        self.entries = []
        flat = [t for pair in layers for t in pair]
        with self.branch(*flat):
            for basis, att in layers:
                w = rel_weights(basis.detach(), att.detach())
                nb, k, f = basis.shape
                r = att.size(0)
                image = None
                nbytes = int(lib.gn_tc_gemm_rel_workspace_bytes(n_rows, r, f, k)) if k % 4 == 0 else 0
                if nbytes and n_rows > 0:
                    image = _ws(nbytes, basis.device)
                    _lib.check(lib.gn_tc_rel_image(n_rows, r, f, k, w.data_ptr(), _ptr(image), nbytes, _stream()),
                               "gn_tc_rel_image")
                key = (basis.data_ptr(), att.data_ptr())
                entry = (self.branch, basis._version, att._version, int(n_rows), w, image)
                RelPrologue._pending.pop(key, None)
                RelPrologue._pending[key] = entry
                self.entries.append(key)
        while len(RelPrologue._pending) > 16:               # entries nobody took (their branch joins when dropped)
            RelPrologue._pending.pop(next(iter(RelPrologue._pending)))

    @staticmethod
    def take(basis, att, n_rows):
        """``(w, image)`` prepared for these parameters (branch joined), or None."""
        e = RelPrologue._pending.pop((basis.data_ptr(), att.data_ptr()), None)
        if e is None:
            return None
        branch, vb, va, rows, w, image = e
        branch.join()
        if vb != basis._version or va != att._version:
            return None                                  # parameters changed since the prologue: recompute
        return w, (image if rows == int(n_rows) else None)


# weight gradients C = A^T B (reduction over the node rows): tensor cores when the reduction is long enough to be a
# stream of the operands (or covers all relations at once), the split-K FFMA kernel otherwise
_TC_TN_MIN_ROWS = 1 << 15


def weight_grad(a, b, out, device, c_inner=0, c_stride=0, force_tc=False):
    """``out = a^T b`` — ``a``: M [n, Mo], ``b``: M [n, No]; ``out``: contiguous [Mo, No] tensor, or with
    ``c_inner`` the ``[No / c_inner][Mo][c_inner]`` relational layout.  Returns False when the tensor path does
    not apply (the caller then runs its FFMA product)."""
    lib = _lib.load()
    n, mo, no = a.n, a.f, b.f
    ok = n > 0 and mo % 4 == 0 and no % 4 == 0 and a.ld % 4 == 0 and b.ld % 4 == 0 and \
        a.ptr % 16 == 0 and b.ptr % 16 == 0 and (force_tc or n >= _TC_TN_MIN_ROWS)
    if not ok:
        return False
    nbytes = int(lib.gn_tc_tn_workspace_bytes(n, mo, no))
    if not nbytes:
        return False
    ws = _ws(nbytes, device)
    _lib.check(lib.gn_tc_tn(a.ptr, a.ld, b.ptr, b.ld, n, mo, no, out.data_ptr(), no, int(c_inner), int(c_stride),
                            _ptr(ws), nbytes, _stream()), "gn_tc_tn")
    return True


def map2d(op, src, dst):
    _lib.check(_lib.load().gn_map2d(op, src.ptr, src.ld, dst.ptr, dst.ld, src.n, src.f, _stream()), "gn_map2d")


def relu_bwd(g, y, dst):
    _lib.check(_lib.load().gn_relu_bwd(g.ptr, g.ld, y.ptr, y.ld, dst.ptr, dst.ld, g.n, g.f, _stream()), "gn_relu_bwd")


def colsum(x, out):
    lib = _lib.load()
    ws = _ws(lib.gn_colsum_workspace_bytes(x.n, x.f), out.device)
    _lib.check(lib.gn_colsum(x.ptr, x.ld, x.n, x.f, _ptr(out), _ptr(ws), ws.numel(), _stream()), "gn_colsum")


# ----------------------------------------------------------------------------
# layer stacks: one autograd node per stack of GCN / RGCN layers.  With ``catout`` every H_l (H_0 = x) is a column
# slice of one [n, sum(dims)] buffer, the stack's output; without it each H_l is a tensor of its own and H_L is the
# output.
# ----------------------------------------------------------------------------
def _views(dims, catout, ts):
    """M views of H_0 .. H_L, or of their gradients: the column slices of ``ts[0]`` with ``catout``, else ``ts``."""
    if catout:
        offs = [sum(dims[:i]) for i in range(len(dims))]
        return [M(ts[0], offs[i], dims[i]) for i in range(len(dims))]
    return [M(t) for t in ts]


def _stack_input(x0, n_rows, nodes, catout, out_dims):
    """``(x0, dims, buf, outs)``: the checked input, the widths of H_0 .. H_L, the catout buffer (or None) and the
    views of the H_l that exist yet: all of them with ``catout``, else H_0 alone (the layer loop appends the rest)."""
    x0 = _as_rows(x0, "x")
    if x0.size(0) != n_rows:
        raise RuntimeError(f"x has {x0.size(0)} rows but the graph has {n_rows} {nodes}")
    dims = [x0.size(1)] + out_dims
    if not catout:
        return x0, dims, None, [M(x0)]
    buf = _new(n_rows, sum(dims), x0)
    return x0, dims, buf, _views(dims, True, [buf])


def _stack_save(ctx, graph, relu_flags, catout, dims, params, n_per, buf, outs, saved):
    """Keeps what ``_stack_backward`` reads (``saved``: the same number of tensors for every layer, layer by layer)
    and returns the stack's output.  ``n_per``: parameters per layer, the bias last."""
    ctx.graph, ctx.relu_flags, ctx.catout, ctx.dims = graph, relu_flags, catout, dims
    ctx.has_bias = [b is not None for b in params[n_per - 1::n_per]]
    ctx.param_refs = [None if p is None else weakref.ref(p) for p in params]
    # outputs/intermediates go through save_for_backward (no ctx <-> output reference cycle)
    acts = [buf] if catout else [o.t for o in outs]
    ctx.n_acts = len(acts)
    ctx.save_for_backward(*acts, *saved)
    return buf if catout else outs[-1].t


def _stack_backward(ctx, grad_out, n_per, n_dst, n_src, block, halo, layer_bwd):
    """Backward of a layer stack, layer L down to 1, with ``n_per`` parameters per layer (the bias last).

    Decided here for both stacks: which dZ_l lives in a gatherable slot, the bias gradient, and the slot dH_{l-1} is
    produced into (``n_dst`` / ``n_src`` local rows, ``block`` rows per rank, halo plan ``halo``) together with the
    concat-slice ``addend`` and the ReLU ``mask`` of layer l-1 applied to it.
    ``layer_bwd(saved, need, dz, h_prev, dprev, addend, mask, br)`` launches the rest of one layer: the SpMM backward
    from the slot ``dz``; the other parameter gradients flagged in ``need`` on the branch ``br``, returned in
    parameter order; and, when ``dprev`` is not None, dH_{l-1} into ``dprev.m``.  ``saved``: the layer's tensors
    kept by ``_stack_save``; ``h_prev``: the view of H_{l-1}."""
    graph, relu_flags, catout, dims = ctx.graph, ctx.relu_flags, ctx.catout, ctx.dims
    n_layers = len(relu_flags)
    saved = ctx.saved_tensors
    outs, per_layer = _views(dims, catout, saved[: ctx.n_acts]), saved[ctx.n_acts:]
    g = _as_rows(grad_out, "grad")
    dev = g.device
    dctx = getattr(graph, "ctx", None)
    gs = _views(dims, catout, [g])
    dh = gs[-1]
    grads = [None] * (n_per * n_layers)
    need_db = [ctx.has_bias[i] and ctx.needs_input_grad[4 + n_per * i + n_per - 1] for i in range(n_layers)]
    dz_slot = None            # set when `dh` already is a masked dZ living in a gatherable slot
    dx0 = None
    # bias / weight gradients leave the dependency chain dZ -> dY -> dH_{l-1}: side stream (a partitioned
    # run all-reduces them on the caller's stream right away unless the reduction is deferred)
    side = dctx is None or dctx.defer_grad_reduce
    br = streams.Branch(enabled=side, background=True)
    # bias sums on a branch of their own: ready before the SpMM, never queued behind a weight GEMM
    br_b = streams.Branch(enabled=side, background=True) if any(need_db) else None
    for l in range(n_layers, 0, -1):
        f, k = dims[l], dims[l - 1]
        p = n_per * (l - 1)                   # the layer's first parameter
        h_prev = outs[l - 1]
        if dz_slot is not None:
            dz = dz_slot
        elif relu_flags[l - 1]:
            dz = Slot.alloc(n_dst, f, g, dctx, block, halo)
            relu_bwd(dh, outs[l], dz.m)
        elif dctx is not None:
            dz = Slot.alloc(n_dst, f, g, dctx, block, halo)
            map2d(_lib.EW_COPY, dh, dz.m)
        else:
            dz = Slot(dh)
        if need_db[l - 1]:
            db = torch.empty(f, dtype=torch.float32, device=dev)
            with br_b(dz.m.t):
                colsum(dz.m, db)
            grads[p + n_per - 1] = _reduce(dctx, db)
        dprev = addend = mask = None
        if l > 1 or ctx.needs_input_grad[0]:
            addend = gs[l - 1] if catout else None
            mask = h_prev if (l > 1 and relu_flags[l - 2]) else None
            # when dH_{l-1} is the next layer's dZ it is produced straight into that layer's gather slot
            dprev = Slot.alloc(n_src, k, g, dctx if mask is not None else None, block, halo)
        s = len(per_layer) // n_layers
        grads[p: p + n_per - 1] = layer_bwd(per_layer[s * (l - 1): s * l], ctx.needs_input_grad[4 + p: 3 + p + n_per],
                                            dz, h_prev, dprev, addend, mask, br)
        dz_slot = dprev if mask is not None else None
        if dprev is not None:
            dh = dprev.m
            if l == 1:
                dx0 = dprev.m.t
    defer = _only_stored(ctx, dctx)
    if br_b is not None:
        br_b.join(deferrable=defer)
    br.join(deferrable=defer)
    return (dx0, None, None, None) + tuple(grads)


def _only_stored(ctx, dctx):
    """May the parameter-gradient branch of this backward stay un-joined until the backward pass ends?"""
    if dctx is not None and not dctx.defer_grad_reduce:
        return False                      # the gradients are all-reduced right away
    params = [None if r is None else r() for r in ctx.param_refs]
    return streams.grads_only_stored(params, ctx.needs_input_grad[4:])


# ----------------------------------------------------------------------------
# GCN stack:  H_l = act_l( A_hat (H_{l-1} W_l) + b_l ),  optional concat of all H_l
#   reference: myGCN.forward (layers.py:71-100) inside homoGraph.forward (:252-318)
#   and interGraph.forward (:362-370, rectangular A_hat)
# ----------------------------------------------------------------------------
class GcnStack(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x0, graph, relu_flags, catout, *params):
        n_layers = len(relu_flags)
        weights = [params[2 * l] for l in range(n_layers)]
        biases = [params[2 * l + 1] for l in range(n_layers)]
        if catout and graph.n_src != graph.n_dst:
            raise RuntimeError("if_catout needs a square graph")
        x0, dims, buf, outs = _stack_input(x0, graph.n_src, "source nodes", catout, [w.size(1) for w in weights])
        for l, w in enumerate(weights):
            require_cuda(w, "weight", torch.float32)
            if w.size(0) != dims[l]:
                raise RuntimeError(f"layer {l}: weight expects {w.size(0)} input features, got {dims[l]}")
        dev = x0.device
        dctx = getattr(graph, "ctx", None)
        b_src = graph.b_src if dctx is not None else None
        br = streams.Branch()                  # no collective is ever issued inside a branch
        for l in range(n_layers):
            w = weights[l].contiguous()
            k, f = dims[l], dims[l + 1]
            y = Slot.alloc(graph.n_src, f, x0, dctx, b_src, getattr(graph, "fwd_halo", None))
            xin = M(x0) if l == 0 else outs[l]
            sgemm(False, False, graph.n_src, f, k, xin.ptr, xin.ld, w.data_ptr(), f, y.m.ptr, y.m.ld, dev)
            if l == 0 and catout:
                with br(x0):                     # the concat copy of H_0 is off the chain (layer 0 reads x0 itself);
                    map2d(_lib.EW_COPY, M(x0), outs[0])   # forked behind the first transform: the chain starts first
            if not catout:
                outs.append(M(_new(graph.n_dst, f, x0)))
            b = biases[l].contiguous() if biases[l] is not None else None
            spmm(graph.fwd, y.gather(), outs[l + 1], f, bias=b, relu=relu_flags[l])
        br.join()
        return _stack_save(ctx, graph, relu_flags, catout, dims, params, 2, buf, outs,
                           [w.contiguous() for w in weights])

    @staticmethod
    def backward(ctx, grad_out):
        graph = ctx.graph
        dctx = getattr(graph, "ctx", None)

        def layer(saved, need, dz, h_prev, dprev, addend, mask, br):
            (w,) = saved
            k, f, dev = h_prev.f, dz.m.f, dz.m.t.device
            dy = M(_new(graph.n_src, f, dz.m.t))
            spmm(graph.bwd, dz.gather(), dy, f)
            dw = None
            if need[0]:
                dw = torch.empty((k, f), dtype=torch.float32, device=dev)
                # dW = H_{l-1}^T dY : reduction over the node dimension -> deterministic split-K
                with br(dy.t, h_prev.t):
                    if not weight_grad(h_prev, dy, dw, dev):
                        sgemm(True, False, k, f, graph.n_src, h_prev.ptr, h_prev.ld, dy.ptr, dy.ld, dw.data_ptr(),
                              f, dev)
                dw = _reduce(dctx, dw)
            if dprev is not None:
                # dH_{l-1} = dY W^T (+ concat-slice grad) (masked by ReLU of layer l-1)
                sgemm(False, True, graph.n_src, k, f, dy.ptr, dy.ld, w.data_ptr(), f, dprev.m.ptr, dprev.m.ld, dev,
                      addend=addend, mask=mask)
            return (dw,)

        return _stack_backward(ctx, grad_out, 2, graph.n_dst, graph.n_src, graph.b_dst if dctx is not None else None,
                               getattr(graph, "bwd_halo", None), layer)


# ----------------------------------------------------------------------------
# RGCN stack: H_l = relu( mean_{e->i} H_{l-1}[src_e] W_{r(e)} + H_{l-1} root (+ b) )
#   reference: myRGCN (layers.py:165-197) inside homoGraph.forward (:268-309)
# ----------------------------------------------------------------------------
class RgcnStack(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x0, graph, relu_flags, catout, *params):
        n_layers = len(relu_flags)
        basis = [params[4 * l] for l in range(n_layers)]
        att = [params[4 * l + 1] for l in range(n_layers)]
        root = [params[4 * l + 2] for l in range(n_layers)]
        bias = [params[4 * l + 3] for l in range(n_layers)]
        n, r = graph.n_nodes, graph.n_rel
        x0, dims, buf, outs = _stack_input(x0, n, "nodes", catout, [rt.size(1) for rt in root])
        dev = x0.device
        dctx = getattr(graph, "ctx", None)
        blk = graph.b if dctx is not None else None
        saved = []                             # (w, basis, att, root) of every layer
        br = streams.Branch()                  # no collective is ever issued inside a branch
        if catout:
            with br(x0):
                map2d(_lib.EW_COPY, M(x0), outs[0])
        for l in range(n_layers):
            k, f = dims[l], dims[l + 1]
            if att[l].size(0) != r:
                raise RuntimeError("att rows must equal the number of relations of the graph")
            bs, at, rt = basis[l].contiguous(), att[l].contiguous(), root[l].contiguous()
            n_in = n if dctx is None else dctx.world * blk           # rows of the (gathered) layer input
            # W[r] = sum_b att[r,b] basis[b]   (layers.py:172-173) — from the step's prologue when there is one
            pre = RelPrologue.take(basis[l], att[l], n_in)
            w, image = pre if pre is not None else (rel_weights(bs, at), None)
            xin = M(x0) if l == 0 else outs[l]
            if not catout:
                outs.append(M(_new(n, f, x0)))
            hl = outs[l + 1]
            # root term X root (layers.py:193), next to the relation transforms; the segmented mean
            # accumulates onto it
            with br(xin.t, rt, hl.t):
                sgemm(False, False, n, f, k, xin.ptr, xin.ld, rt.data_ptr(), f, hl.ptr, hl.ld, dev)
            # Y[:, r, :] = X W[r] for every relation at once (transform-then-gather), on the tensor cores.
            # Partitioned run: the NARROW layer input (k floats per node) is what crosses NVLink, and every
            # rank transforms all the gathered rows itself — R*f/k times fewer bytes exchanged than gathering Y
            if dctx is not None:
                xs = Slot.alloc(n, k, x0, dctx, blk)
                map2d(_lib.EW_COPY, xin, xs.m)
                xall = xs.gather()
            else:
                xall = xin
            yfull = _new(xall.n, r * f, x0)
            rel_transform(xall, w, M(yfull), r, k, f, dev, image=image if xall.n == n_in else None)
            b = bias[l].contiguous() if bias[l] is not None else None
            br.join()
            spmm(graph.fwd, M(yfull.view(yfull.size(0) * r, f)), hl, f, row_scale=graph.inv_cnt, bias=b, addend=hl,
                 relu=relu_flags[l])
            saved += (w, bs, at, rt)
        br.join()
        return _stack_save(ctx, graph, relu_flags, catout, dims, params, 4, buf, outs, saved)

    @staticmethod
    def backward(ctx, grad_out):
        graph = ctx.graph
        n, r = graph.n_nodes, graph.n_rel
        dctx = getattr(graph, "ctx", None)

        def layer(saved, need, dzs, h_prev, dprev, addend, mask, br):
            w, bs, at, rt = saved
            dz = dzs.m
            k, f, nb, dev = h_prev.f, dz.f, bs.size(0), dz.t.device
            # dY[(j,r)] = sum_{e: src=j, rel=r} dZ[dst_e] / c_dst   (transpose CSR, atomic-free)
            dy = torch.empty((n * r, f), dtype=torch.float32, device=dev)
            spmm(graph.bwd, dzs.gather(), M(dy), f)
            dbasis = datt = droot = None
            if need[2]:
                droot = torch.empty((k, f), dtype=torch.float32, device=dev)
                with br(dz.t, h_prev.t):
                    sgemm(True, False, k, f, n, h_prev.ptr, h_prev.ld, dz.ptr, dz.ld, droot.data_ptr(), f, dev)
                droot = _reduce(dctx, droot)
            if need[0] or need[1]:
                # dW[r] = H_{l-1}^T dY[:, r, :]
                dw = torch.empty((r, k, f), dtype=torch.float32, device=dev)
                datt = torch.empty((r, nb), dtype=torch.float32, device=dev) if need[1] else None
                dbasis = torch.empty((nb, k, f), dtype=torch.float32, device=dev) if need[0] else None
                with br(dy, h_prev.t, dw, bs, at):
                    # dW[r] = X^T dY[:, r, :] for all relations at once: one TN product on the tensor cores
                    if not weight_grad(h_prev, M(dy.view(n, r * f)), dw, dev, c_inner=f, c_stride=k * f,
                                       force_tc=True):
                        sgemm(True, False, k, f, n, h_prev.ptr, h_prev.ld, dy.data_ptr(), r * f, dw.data_ptr(), f,
                              dev, batch=r, sa=0, sb=f, sc=k * f)
                    if datt is not None:
                        sgemm(False, True, r, nb, k * f, dw.data_ptr(), k * f, bs.data_ptr(), k * f, datt.data_ptr(),
                              nb, dev)
                    if dbasis is not None:
                        sgemm(True, False, nb, k * f, r, at.data_ptr(), nb, dw.data_ptr(), k * f, dbasis.data_ptr(),
                              k * f, dev)
                if datt is not None:
                    datt = _reduce(dctx, datt)
                if dbasis is not None:
                    dbasis = _reduce(dctx, dbasis)
            if dprev is not None:
                # dH_{l-1} = dZ root^T (+ concat grad), then += sum_r dY[:, r, :] W[r]^T, then ReLU mask
                d = dprev.m
                sgemm(False, True, n, k, f, dz.ptr, dz.ld, rt.data_ptr(), f, d.ptr, d.ld, dev, addend=addend)
                sgemm(False, True, n, k, f, dy.data_ptr(), r * f, w.data_ptr(), f, d.ptr, d.ld, dev,
                      batch=r, sa=f, sb=k * f, sc=0, batch_reduce=True, accumulate=True, mask=mask)
            return dbasis, datt, droot

        # the partitioned relational graph has no halo plan: its layer inputs and dZ are gathered as whole blocks
        return _stack_backward(ctx, grad_out, 4, n, n, graph.b if dctx is not None else None, None, layer)


# ----------------------------------------------------------------------------
# interGraph tail: cat([h, |t|]) / (h+|t|)/2 / (h+relu(t D))/2   (layers.py:375-384)
# ----------------------------------------------------------------------------
def axpby(a, alpha, b, beta, dst):
    _lib.check(_lib.load().gn_axpby(a.ptr, a.ld, float(alpha), b.ptr if b is not None else None,
                                    b.ld if b is not None else 0, float(beta), dst.ptr, dst.ld, a.n, a.f,
                                    _stream()), "gn_axpby")


class Mean3(torch.autograd.Function):
    """``(a + b + c) / 3`` (``GripNet-freebase-d.py:160-161``) as one kernel; backward ``g / 3`` once, shared."""

    @staticmethod
    def forward(ctx, a, b, c):
        a, b, c = _as_rows(a, "a"), _as_rows(b, "b"), _as_rows(c, "c")
        if a.shape != b.shape or a.shape != c.shape:
            raise RuntimeError("mean3: the three inputs must have the same shape")
        out = _new(a.size(0), a.size(1), a)
        ma, mb, mc, mo = M(a), M(b), M(c), M(out)
        _lib.check(_lib.load().gn_mean3(ma.ptr, ma.ld, mb.ptr, mb.ld, mc.ptr, mc.ld, mo.ptr, mo.ld, ma.n, ma.f,
                                        _stream()), "gn_mean3")
        return out

    @staticmethod
    def backward(ctx, g):
        g = _as_rows(g, "grad")
        dg = _new(g.size(0), g.size(1), g)
        axpby(M(g), 1.0 / 3.0, None, 0.0, M(dg))
        return dg, dg, dg


def mean3(a, b, c):
    return Mean3.apply(a, b, c)


def abs_bwd(g, t, dst, scale):
    _lib.check(_lib.load().gn_abs_bwd(g.ptr, g.ld, t.ptr, t.ld, dst.ptr, dst.ld, g.n, g.f, float(scale),
                                      _stream()), "gn_abs_bwd")


class InterTail(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, target_feat, target_feat_down, mod, dctx=None):
        ctx.dctx = dctx
        h = _as_rows(h, "h")
        t = _as_rows(target_feat, "target_feat")
        n, f, ft = h.size(0), h.size(1), t.size(1)
        if t.size(0) != n:
            raise RuntimeError("target_feat rows must equal the number of target nodes")
        dev = h.device
        ctx.shapes = (n, f, ft)
        if mod == "cat":
            out = _new(n, f + ft, h)
            map2d(_lib.EW_COPY, M(h), M(out, 0, f))
            map2d(_lib.EW_ABS, M(t), M(out, f, ft))
            ctx.kind = 0
            ctx.save_for_backward(t)
            return out
        out = _new(n, f, h)
        if f == ft:
            map2d(_lib.EW_ABS, M(t), M(out))
            ctx.kind = 1
            ctx.save_for_backward(t)
        else:
            d = _as_rows(target_feat_down, "target_feat_down")
            u = _new(n, f, h)
            sgemm(False, False, n, f, ft, t.data_ptr(), t.stride(0), d.data_ptr(), d.stride(0), u.data_ptr(), f, dev)
            map2d(_lib.EW_RELU, M(u), M(out))
            ctx.kind = 2
            ctx.save_for_backward(t, d, u)
        axpby(M(h), 0.5, M(out), 0.5, M(out))
        return out

    @staticmethod
    def backward(ctx, grad):
        n, f, ft = ctx.shapes
        g = _as_rows(grad, "grad")
        dev = g.device
        if ctx.kind == 0:
            (t,) = ctx.saved_tensors
            dt = _new(n, ft, g)
            abs_bwd(M(g, f, ft), M(t), M(dt), 1.0)
            return g[:, :f], dt, None, None, None
        dh = _new(n, f, g)
        axpby(M(g), 0.5, None, 0.0, M(dh))
        if ctx.kind == 1:
            (t,) = ctx.saved_tensors
            dt = _new(n, ft, g)
            abs_bwd(M(g), M(t), M(dt), 0.5)
            return dh, dt, None, None, None
        t, d, u = ctx.saved_tensors
        du = _new(n, f, g)
        relu_bwd(M(dh), M(u), M(du))                      # 0.5 * g where t D > 0
        dt = _new(n, ft, g)
        sgemm(False, True, n, ft, f, du.data_ptr(), f, d.data_ptr(), d.stride(0), dt.data_ptr(), ft, dev)
        dd = torch.empty((ft, f), dtype=torch.float32, device=dev)
        sgemm(True, False, ft, f, n, t.data_ptr(), t.stride(0), du.data_ptr(), f, dd.data_ptr(), f, dev)
        return dh, dt, _reduce(ctx.dctx, dd), None, None


# ----------------------------------------------------------------------------
# DistMult decoder  (decoder.py:19-23)
# ----------------------------------------------------------------------------
def _distmult_check(z, weight, edge_index, edge_type):
    z = _as_rows(z, "z")
    w = _as_rows(weight, "weight").contiguous()
    require_cuda(edge_index, "edge_index", torch.int64)
    require_cuda(edge_type, "edge_type", torch.int64)
    if edge_index.dim() != 2 or edge_index.size(0) != 2 or edge_type.numel() != edge_index.size(1):
        raise RuntimeError("edge_index must be [2,E] and edge_type [E]")
    if w.size(1) != z.size(1):
        raise RuntimeError("decoder weight width must equal the embedding width")
    validate_index(edge_index, z.size(0), "edge_index")          # the reference raises IndexError here too
    validate_index(edge_type, w.size(0), "edge_type")
    return z, w, edge_index.contiguous(), edge_type.contiguous()


def _ldz(z):
    return z.stride(0) if z.size(0) > 1 else z.size(1)


def _distmult_fwd(z, w, ei, et, sigmoid):
    e = ei.size(1)
    out = torch.empty(e, dtype=torch.float32, device=z.device)
    _lib.check(_lib.load().gn_distmult_fwd(z.data_ptr(), _ldz(z), z.size(1), w.data_ptr(),
                                           _ptr(ei[0]) if e else None, _ptr(ei[1]) if e else None,
                                           _ptr(et) if e else None, e, int(sigmoid), _ptr(out), _stream()),
               "gn_distmult_fwd")
    return out


def _distmult_coef(g, out, sigmoid):
    e = out.numel()
    coef = torch.empty(max(e, 1), dtype=torch.float32, device=out.device)
    _lib.check(_lib.load().gn_distmult_coef(_ptr(g), _ptr(out), e, int(sigmoid), _ptr(coef), _stream()),
               "gn_distmult_coef")
    return coef


def _pair_walk(ps, coef, z):
    """T[n, r, :] = sum over the pair row (n, r) of coef[e] * z[other]  (one gather pass, atomic-free)."""
    d = z.size(1)
    t = torch.empty((ps.csr.n_rows, d), dtype=torch.float32, device=z.device)
    part = ps.csr.partial(d)
    _lib.check(_lib.load().gn_distmult_bwd_pairs(ps.csr.ref, _ptr(ps.ent_other), _ptr(ps.ent_eid), _ptr(coef),
                                                 z.data_ptr(), _ldz(z), d, t.data_ptr(), _ptr(part), _stream()),
               "gn_distmult_bwd_pairs")
    return t


def _distmult_grads(t, t2, z, w, need_z, need_w):
    n, d, r = z.size(0), z.size(1), w.size(0)
    dz = torch.empty((n, d), dtype=torch.float32, device=z.device) if need_z else None
    dw = torch.empty_like(w) if need_w else None
    if need_z or need_w:
        lib = _lib.load()
        ws = _ws(lib.gn_distmult_grads_workspace_bytes(n, r, d), z.device)
        _lib.check(lib.gn_distmult_grads(t.data_ptr(), _ptr(t2), n, r, d, z.data_ptr(), _ldz(z), w.data_ptr(),
                                         _ptr(dz), d, _ptr(dw), _ptr(ws), ws.numel(), _stream()), "gn_distmult_grads")
    return dz, dw


def _check_versions(tensors, versions, what):
    """The backward's index structures are keyed on the LIVE index tensors: an in-place rewrite between
    forward and backward (e.g. ``sampler.sample(out=buf)``) would silently pair the saved scores with
    another edge list."""
    for t, v in zip(tensors, versions):
        if t._version != v:
            raise RuntimeError(f"gripnet_b200: {what} was modified in place between forward and backward")


class DistMult(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, weight, edge_index, edge_type, sigmoid):
        from .graph import pair_struct
        z, w, ei, et = _distmult_check(z, weight, edge_index, edge_type)
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]      # (grad mode is off inside forward)
        br = streams.Branch()
        if need:      # the (node, relation) structure depends on the indices only: built next to the scores
            with br(edge_index, edge_type):
                pair_struct(edge_index, edge_type, z.size(0), w.size(0))
        out = _distmult_fwd(z, w, ei, et, sigmoid)
        br.join()
        ctx.sigmoid = bool(sigmoid)
        ctx.key_tensors = (edge_index, edge_type)
        ctx.key_versions = (edge_index._version, edge_type._version)
        ctx.save_for_backward(z, w, out)
        return out

    @staticmethod
    def backward(ctx, grad):
        from .graph import pair_struct
        z, w, out = ctx.saved_tensors
        _check_versions(ctx.key_tensors, ctx.key_versions, "edge_index / edge_type")
        coef = _distmult_coef(grad.contiguous(), out, ctx.sigmoid)
        ps = pair_struct(ctx.key_tensors[0], ctx.key_tensors[1], z.size(0), w.size(0))
        t = _pair_walk(ps, coef, z)
        dz, dw = _distmult_grads(t, None, z, w, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        return dz, dw, None, None, None


class DistMultPair(torch.autograd.Function):
    """Positive and negative edge lists of one training step scored together
    (``GripNet-pose.py:133-138`` calls the decoder twice on the same ``z`` and ``edge_type``).

    Forward: the two lists are independent, so they run on two streams, next to the build of their
    (node, relation) structures (the negatives' one is rebuilt on the device every step).  Backward: ONE
    gather pass per list (``gn_distmult_bwd_pairs``, concurrently) and one kernel that forms
    ``dz = sum_r (T_pos + T_neg)[n,r] .* w[r]`` and ``dw = 1/2 sum_n z[n] .* (T_pos + T_neg)[n,r]``.

    ``rel_lo`` / ``n_rel_local`` (partitioned runs): the edge lists of this call only hold relations
    ``[rel_lo, rel_lo + n_rel_local)`` and ``edge_type`` is already SHIFTED by ``rel_lo`` — a rank's slice of
    a relation-major list covers a few relations, and the (node, relation) structures, ``T`` and the gradient
    kernel then span ``n_rel_local`` relations instead of all of them; the other rows of ``dw`` are zero.
    """

    @staticmethod
    def forward(ctx, z, weight, pos_index, neg_index, edge_type, sigmoid, rel_lo=0, n_rel_local=None,
                struct_branch=None):
        from .graph import pair_struct
        w_full = _as_rows(weight, "weight").contiguous()
        r_loc = w_full.size(0) if n_rel_local is None else int(n_rel_local)
        if rel_lo < 0 or rel_lo + r_loc > w_full.size(0):
            raise RuntimeError("relation slice out of range")
        w_loc = w_full[rel_lo: rel_lo + r_loc]
        z, w, pi, et = _distmult_check(z, w_loc, pos_index, edge_type)
        _, _, ni, _ = _distmult_check(z, w_loc, neg_index, edge_type)
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]      # (grad mode is off inside forward)
        # the structures are read by the BACKWARD only: their branch (the caller's `struct_branch`, forked earlier in
        # the step, or the one forked here) is joined at the top of backward(), so the scores never wait for the sort
        br = streams.Branch()
        br_s = struct_branch if struct_branch is not None else streams.Branch(background=True)
        if need:
            with br_s(pos_index, neg_index, edge_type):
                pair_struct(neg_index, edge_type, z.size(0), r_loc)      # (cache hits when the caller built them)
                pair_struct(pos_index, edge_type, z.size(0), r_loc)      # cached after the first step
        with br(z, w, ni, et):
            neg = _distmult_fwd(z, w, ni, et, sigmoid)
        pos = _distmult_fwd(z, w, pi, et, sigmoid)
        br.join()
        if need and br_s._parent is None:
            ctx.struct_branch = br_s
        else:
            ctx.struct_branch = None
            br_s.join()
        ctx.sigmoid = bool(sigmoid)
        ctx.keys = (pos_index, neg_index, edge_type)
        ctx.key_versions = tuple(t._version for t in ctx.keys)
        ctx.rel = (int(rel_lo), r_loc, w_full.size(0))
        ctx.save_for_backward(z, w, pos, neg)
        return pos, neg

    @staticmethod
    def backward(ctx, g_pos, g_neg):
        from .graph import pair_struct
        z, w, pos, neg = ctx.saved_tensors
        pos_key, neg_key, et_key = ctx.keys
        _check_versions(ctx.keys, ctx.key_versions, "pos / neg edge_index or edge_type")
        rel_lo, r, r_full = ctx.rel
        n = z.size(0)
        if ctx.struct_branch is not None:
            ctx.struct_branch.join()
            ctx.struct_branch = None
        ps_p = pair_struct(pos_key, et_key, n, r)
        ps_n = pair_struct(neg_key, et_key, n, r)
        g_pos, g_neg = g_pos.contiguous(), g_neg.contiguous()
        # one structure serves both lists when they are the same tensor: its arrival counters cannot be
        # shared by two concurrent walks, so that case runs on one stream
        br = streams.Branch(enabled=ps_p is not ps_n)
        with br(g_neg, neg, z):
            coef_n = _distmult_coef(g_neg, neg, ctx.sigmoid)
            t_n = _pair_walk(ps_n, coef_n, z)
        coef_p = _distmult_coef(g_pos, pos, ctx.sigmoid)
        t_p = _pair_walk(ps_p, coef_p, z)
        br.join()
        dz, dw = _distmult_grads(t_p, t_n, z, w, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        if dw is not None and r != r_full:                    # relations outside this rank's slice: zero rows
            dw_full = torch.empty((r_full, w.size(1)), dtype=torch.float32, device=w.device)
            _lib.check(_lib.load().gn_zero(dw_full.data_ptr(), dw_full.numel() * 4, _stream()), "gn_zero")
            map2d(_lib.EW_COPY, M(dw), M(dw_full[rel_lo: rel_lo + r]))
            dw = dw_full
        return dz, dw, None, None, None, None, None, None, None


# ----------------------------------------------------------------------------
# multi-class decoder  softmax(z[node_list] W)   (decoder.py:38-45)
# ----------------------------------------------------------------------------
class MultiClass(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z, weight, node_list, softmax):
        lib = _lib.load()
        z = _as_rows(z, "z")
        w = _as_rows(weight, "weight").contiguous()
        require_cuda(node_list, "node_list", torch.int64)
        if w.size(0) != z.size(1):
            raise RuntimeError("decoder weight rows must equal the embedding width")
        validate_index(node_list, z.size(0), "node_list")
        idx = node_list.contiguous().view(-1)
        m, d, c = idx.numel(), z.size(1), w.size(1)
        dev = z.device
        logits = torch.empty((m, c), dtype=torch.float32, device=dev)
        sgemm(False, False, m, c, d, z.data_ptr(), z.stride(0) if z.size(0) > 1 else d, w.data_ptr(), c,
              logits.data_ptr(), c, dev, a_rows=idx)
        if softmax:
            out = torch.empty_like(logits)
            _lib.check(lib.gn_softmax_fwd(_ptr(logits), m, c, _ptr(out), _stream()), "gn_softmax_fwd")
        else:
            out = logits
        ctx.softmax = bool(softmax)
        ctx.key_tensor = node_list
        ctx.save_for_backward(z, w, out, idx)
        return out

    @staticmethod
    def backward(ctx, grad):
        from .graph import index_struct
        lib = _lib.load()
        z, w, out, idx = ctx.saved_tensors
        n, d, c, m = z.size(0), z.size(1), w.size(1), idx.numel()
        dev = z.device
        g = grad.contiguous()
        ldz = z.stride(0) if n > 1 else d
        if ctx.softmax:
            gl = torch.empty_like(g)
            _lib.check(lib.gn_softmax_bwd(_ptr(out), _ptr(g), m, c, _ptr(gl), _stream()), "gn_softmax_bwd")
        else:
            gl = g
        dz = dw = None
        if ctx.needs_input_grad[1]:
            dw = torch.empty((d, c), dtype=torch.float32, device=dev)
            sgemm(True, False, d, c, m, z.data_ptr(), ldz, gl.data_ptr(), c, dw.data_ptr(), c, dev, a_rows=idx)
        if ctx.needs_input_grad[0]:
            grows = torch.empty((max(m, 1), d), dtype=torch.float32, device=dev)
            sgemm(False, True, m, d, c, gl.data_ptr(), c, w.data_ptr(), c, grows.data_ptr(), d, dev)
            st = index_struct(ctx.key_tensor, n)
            dz = torch.empty((n, d), dtype=torch.float32, device=dev)
            spmm(st.csr, M(grows), M(dz), d)
        return dz, dw, None, None


# ----------------------------------------------------------------------------
# fused losses  (GripNet-pose.py:140-142, GripNet-aminer.py:133)
# ----------------------------------------------------------------------------
class LinkPredLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, neg):
        lib = _lib.load()
        pos = require_cuda(pos, "pos_score", torch.float32).contiguous()
        neg = require_cuda(neg, "neg_score", torch.float32).contiguous()
        dev = pos.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        n = max(pos.numel(), neg.numel())
        ws = _ws(lib.gn_loss_workspace_bytes(n), dev)
        _lib.check(lib.gn_lp_loss_fwd(_ptr(pos), pos.numel(), _ptr(neg), neg.numel(), EPS, _ptr(loss), _ptr(ws),
                                      ws.numel(), _stream()), "gn_lp_loss_fwd")
        ctx.save_for_backward(pos, neg)
        return loss.view(())

    @staticmethod
    def backward(ctx, grad):
        lib = _lib.load()
        pos, neg = ctx.saved_tensors
        g = grad.contiguous().view(1)
        gp, gn_ = torch.empty_like(pos), torch.empty_like(neg)
        _lib.check(lib.gn_lp_loss_bwd(_ptr(pos), pos.numel(), _ptr(neg), neg.numel(), EPS, _ptr(g), _ptr(gp),
                                      _ptr(gn_), _stream()), "gn_lp_loss_bwd")
        return gp, gn_


class NodeClassLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, score, labels):
        lib = _lib.load()
        score = _as_rows(score, "score").contiguous()
        labels = require_cuda(labels, "labels", torch.int64).contiguous()
        if labels.numel() != score.size(0):
            raise RuntimeError("labels must have one entry per score row")
        validate_index(labels, score.size(1), "labels")
        dev = score.device
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        ws = _ws(lib.gn_loss_workspace_bytes(score.size(0)), dev)
        _lib.check(lib.gn_nc_loss_fwd(_ptr(score), score.size(0), score.size(1), _ptr(labels), EPS, _ptr(loss),
                                      _ptr(ws), ws.numel(), _stream()), "gn_nc_loss_fwd")
        ctx.save_for_backward(score, labels)
        return loss.view(())

    @staticmethod
    def backward(ctx, grad):
        lib = _lib.load()
        score, labels = ctx.saved_tensors
        g = grad.contiguous().view(1)
        gs = torch.empty_like(score)
        _lib.check(lib.gn_nc_loss_bwd(_ptr(score), score.size(0), score.size(1), _ptr(labels), EPS, _ptr(g),
                                      _ptr(gs), _stream()), "gn_nc_loss_bwd")
        return gs, None


# ----------------------------------------------------------------------------
# plain dense product with autograd (encoder.RGCN's input projection)
# ----------------------------------------------------------------------------
class MatMul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w):
        x = _as_rows(x, "x")
        w = _as_rows(w, "w").contiguous()
        out = _new(x.size(0), w.size(1), x)
        sgemm(False, False, x.size(0), w.size(1), x.size(1), x.data_ptr(), M(x).ld, w.data_ptr(), w.size(1),
              out.data_ptr(), w.size(1), x.device)
        ctx.save_for_backward(x, w)
        return out

    @staticmethod
    def backward(ctx, grad):
        x, w = ctx.saved_tensors
        g = _as_rows(grad, "grad")
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = _new(x.size(0), x.size(1), x)
            sgemm(False, True, x.size(0), x.size(1), w.size(1), g.data_ptr(), M(g).ld, w.data_ptr(), w.size(1),
                  dx.data_ptr(), x.size(1), x.device)
        if ctx.needs_input_grad[1]:
            dw = _new(w.size(0), w.size(1), x)
            sgemm(True, False, w.size(0), w.size(1), x.size(0), x.data_ptr(), M(x).ld, g.data_ptr(), M(g).ld,
                  dw.data_ptr(), w.size(1), x.device)
        return dx, dw


def matmul(x, w):
    return MatMul.apply(x, w)
