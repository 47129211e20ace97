"""Device-resident graph structures built by the K1 preprocessing kernels.

``edge_index`` (int64 ``[2,E]``) is turned once into a destination-sorted CSR and
its transpose (stable counting sort => bit-exact edge order), with the GCN
symmetric normalisation precomputed, and cached per tensor identity — the
counterpart of ``myGCN.cached_result`` (reference ``gripnet/layers.py:83-90``).
All arrays live in HBM as int32 / fp32 tensors owned by these objects.
"""
import ctypes as C
import os
import weakref
from collections import OrderedDict

import torch

from . import _lib, streams

_SM_COUNT = 148


def _stream():
    """The CUDA stream every kernel launch goes to: the active side branch (``streams.py``) or
    torch's current stream."""
    s = streams.override()
    return (s if s is not None else torch.cuda.current_stream()).cuda_stream


def _host_int(t):
    """One device int -> host (a build-time sync).  Inside a side branch the producing kernels are not
    ordered before a copy on torch's current stream, so that stream is drained first."""
    s = streams.override()
    if s is not None:
        s.synchronize()
    return int(t.item())


def _ptr(t):
    return None if t is None else t.data_ptr()


def require_cuda(t, name, dtype=None):
    if not torch.is_tensor(t):
        raise TypeError(f"{name} must be a tensor")
    if not t.is_cuda:
        raise RuntimeError(f"gripnet_b200: {name} must be a CUDA tensor (no CPU fallback exists)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"gripnet_b200: {name} must be {dtype}, got {t.dtype}")
    return t


def _ws(nbytes, device):
    t = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
    streams.keep(t)          # scratch of a side-stream launch lives until the branch joins
    return t


def pick_chunk_len(nnz):
    """Entries per warp-chunk: enough chunks to fill 148 SMs x 32 warps, within [32, 1024]."""
    target = max(1, nnz // (_SM_COUNT * 32))
    c = 32
    while c * 2 <= target and c < 1024:
        c *= 2
    return c


class Csr:
    """Device CSR + row-split chunk list (mirror of ``gn_csr``)."""

    def __init__(self, rowptr, col, val, n_rows, n_cols, nnz_bound, exact=True, chunk_len=None):
        lib = _lib.load()
        dev = rowptr.device
        self.rowptr, self.col, self.val = rowptr, col, val
        self.n_rows, self.n_cols = int(n_rows), int(n_cols)
        self.nnz = int(nnz_bound)
        self.chunk_len = int(chunk_len or pick_chunk_len(self.nnz))
        cap = self.n_rows + self.nnz // self.chunk_len + 1
        self.chunk_ptr = torch.empty(self.n_rows + 1, dtype=torch.int32, device=dev)
        self.chunk_row = torch.empty(cap, dtype=torch.int32, device=dev)
        self.chunk_beg = torch.empty(cap, dtype=torch.int32, device=dev)
        self.row_counter = torch.empty(max(self.n_rows, 1), dtype=torch.int32, device=dev)   # zeroed by the kernel
        ws = _ws(lib.gn_build_chunks_workspace_bytes(self.n_rows), dev)
        _lib.check(lib.gn_build_chunks(_ptr(rowptr), self.n_rows, self.chunk_len, _ptr(self.chunk_ptr),
                                       _ptr(self.chunk_row), _ptr(self.chunk_beg), cap, _ptr(self.row_counter),
                                       _ptr(ws), ws.numel(), _stream()), "gn_build_chunks")
        if exact:   # one host read at graph-build time (never inside a captured step)
            self.n_chunks = _host_int(self.chunk_ptr[self.n_rows]) if self.n_rows > 0 else 0
        else:
            self.n_chunks = cap - 1 if self.n_rows > 0 else 0
        # every row fits one chunk (known exactly): kernels read the row bounds straight from rowptr
        self.flags = _lib.CSR_ROW_IS_CHUNK if (exact and self.n_chunks == self.n_rows) else 0
        self.c = _lib.GnCsr(self.n_rows, self.n_cols, self.nnz, self.chunk_len, self.n_chunks, self.flags,
                            _ptr(rowptr), _ptr(col), _ptr(val), _ptr(self.chunk_ptr), _ptr(self.chunk_row),
                            _ptr(self.chunk_beg), _ptr(self.row_counter))
        self.ref = C.byref(self.c)

    @property
    def extra_chunks(self):
        return max(0, self.n_chunks - self.n_rows)

    def partial(self, width):
        """Scratch for rows split over several chunks (2 slots per extra chunk), or None."""
        if self.extra_chunks == 0:
            return None
        t = torch.empty(2 * self.extra_chunks * int(width), dtype=torch.float32, device=self.rowptr.device)
        streams.keep(t)
        return t


class GcnGraph:
    """dst-sorted CSR (forward) + src-sorted CSR (backward) with GCN normalisation."""

    def __init__(self, edge_index, n_src, n_dst, edge_weight=None, improved=False, bipartite=False,
                 want_aug=False):
        lib = _lib.load()
        require_cuda(edge_index, "edge_index", torch.int64)
        if edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise RuntimeError("edge_index must have shape [2, E]")
        dev = edge_index.device
        E = int(edge_index.size(1))
        if E + n_dst >= 2 ** 31 or n_src >= 2 ** 31:
            raise RuntimeError("gripnet_b200: graph exceeds the int32 index space (N, E + N must be < 2^31)")
        ei = edge_index.contiguous()
        w = None
        if edge_weight is not None:
            w = require_cuda(edge_weight, "edge_weight").to(torch.float32).contiguous()
            if w.numel() != E:
                raise RuntimeError("edge_weight must have one entry per edge")
        if E > 0:
            lo, hi0, hi1 = int(ei.min()), int(ei[0].max()), int(ei[1].max())
            if lo < 0 or hi0 >= n_src or hi1 >= n_dst:
                raise IndexError("edge_index out of range for the given node counts")
        self.n_src, self.n_dst, self.n_edges, self.bipartite = int(n_src), int(n_dst), E, bool(bipartite)
        cap = E + (0 if bipartite else n_dst)
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        rowptr = torch.empty(n_dst + 1, **i32)
        col = torch.empty(max(cap, 1), **i32)
        val = torch.empty(max(cap, 1), **f32)
        perm = torch.empty(max(cap, 1), **i32)
        rowptr_t = torch.empty(n_src + 1, **i32)
        col_t = torch.empty(max(cap, 1), **i32)
        val_t = torch.empty(max(cap, 1), **f32)
        perm_t = torch.empty(max(cap, 1), **i32)
        self.deg = torch.empty(n_dst, **f32)
        self.indeg = torch.empty(n_dst, **i32)
        counts = torch.zeros(4, **i32)
        aug_idx = aug_norm = None
        if want_aug and not bipartite:
            aug_idx = torch.empty(2, max(cap, 1), dtype=torch.int64, device=dev)
            aug_norm = torch.empty(max(cap, 1), **f32)
        ws = _ws(lib.gn_gcn_prep_workspace_bytes(E, n_src, n_dst), dev)
        fill = 2.0 if improved else 1.0
        _lib.check(lib.gn_gcn_prep(
            _ptr(ei[0]) if E else None, _ptr(ei[1]) if E else None, _ptr(w), E, n_src, n_dst, int(bipartite), fill,
            _ptr(aug_idx[0]) if aug_idx is not None else None, _ptr(aug_idx[1]) if aug_idx is not None else None,
            _ptr(aug_norm), _ptr(rowptr), _ptr(col), _ptr(val), _ptr(perm), _ptr(rowptr_t), _ptr(col_t),
            _ptr(val_t), _ptr(perm_t), _ptr(self.deg), _ptr(self.indeg), _ptr(counts), _ptr(ws), ws.numel(),
            _stream()), "gn_gcn_prep")
        self.nnz = _host_int(counts[0])            # E' (one host read, at graph-build time)
        self.perm, self.perm_t = perm[: self.nnz], perm_t[: self.nnz]
        self.fwd = Csr(rowptr, col, val, n_dst, n_src, self.nnz)
        self.bwd = Csr(rowptr_t, col_t, val_t, n_src, n_dst, self.nnz)
        if aug_idx is not None:
            self.aug_edge_index = aug_idx[:, : self.nnz]
            self.aug_norm = aug_norm[: self.nnz]
        else:
            self.aug_edge_index = self.aug_norm = None


class RgcnGraph:
    """Relation-aware CSR pair for myRGCN (joint mean over all in-edges)."""

    def __init__(self, edge_index, range_list, n_nodes, n_rel):
        lib = _lib.load()
        require_cuda(edge_index, "edge_index", torch.int64)
        dev = edge_index.device
        E = int(edge_index.size(1))
        rl = torch.as_tensor(range_list).to(torch.int64)
        rl_host = rl.cpu()
        if rl_host.dim() != 2 or rl_host.size(1) != 2 or rl_host.size(0) != n_rel:
            raise RuntimeError("range_list must have shape [num_relations, 2]")
        # the reference concatenates the per-relation slices and scatters them at
        # edge_index[1] positionally (layers.py:178-189): only an ascending partition
        # of [0, E) is meaningful there, anything else mis-sizes its scatter.
        flat = rl_host.flatten().tolist()
        ok = flat[0] == 0 and flat[-1] == E and all(flat[2 * r + 1] == flat[2 * r + 2] for r in range(n_rel - 1)) \
            and all(flat[2 * r] <= flat[2 * r + 1] for r in range(n_rel))
        if not ok:
            raise RuntimeError("range_list must partition [0, E) into ascending contiguous [start, end) slices")
        if n_nodes * n_rel >= 2 ** 31 or E >= 2 ** 31:
            raise RuntimeError("gripnet_b200: num_nodes * num_relations must be < 2^31")
        ei = edge_index.contiguous()
        if E > 0 and (int(ei.min()) < 0 or int(ei.max()) >= n_nodes):
            raise IndexError("edge_index out of range")
        rl_dev = rl.to(dev).contiguous()
        self.n_nodes, self.n_rel, self.n_edges = int(n_nodes), int(n_rel), E
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        rowptr = torch.empty(n_nodes + 1, **i32)
        col = torch.empty(max(E, 1), **i32)
        self.perm = torch.empty(max(E, 1), **i32)
        self.inv_cnt = torch.empty(n_nodes, **f32)
        rowptr_t = torch.empty(n_nodes * n_rel + 1, **i32)
        col_t = torch.empty(max(E, 1), **i32)
        val_t = torch.empty(max(E, 1), **f32)
        self.perm_t = torch.empty(max(E, 1), **i32)
        ws = _ws(lib.gn_rgcn_prep_workspace_bytes(E, n_nodes, n_rel), dev)
        _lib.check(lib.gn_rgcn_prep(_ptr(ei[0]) if E else None, _ptr(ei[1]) if E else None, E, _ptr(rl_dev), n_nodes,
                                    n_rel, _ptr(rowptr), _ptr(col), _ptr(self.perm), _ptr(self.inv_cnt),
                                    _ptr(rowptr_t), _ptr(col_t), _ptr(val_t), _ptr(self.perm_t), _ptr(ws),
                                    ws.numel(), _stream()), "gn_rgcn_prep")
        self.fwd = Csr(rowptr, col, None, n_nodes, n_nodes * n_rel, E)
        self.bwd = Csr(rowptr_t, col_t, val_t, n_nodes * n_rel, n_nodes, E)


def slice_csr(csr, r0, r1, n_cols):
    """Rows ``[r0, r1)`` of a device CSR as a stand-alone ``Csr`` (own chunk list).

    ``col`` / ``val`` are copies of the corresponding slices of the global arrays (so the global
    arrays can be freed) and ``rowptr`` is rebased by a kernel: bit-identical to slicing."""
    lib = _lib.load()
    n_local = int(r1 - r0)
    dev = csr.rowptr.device
    rowptr = torch.empty(n_local + 1, dtype=torch.int32, device=dev)
    _lib.check(lib.gn_rowptr_slice(_ptr(csr.rowptr), int(r0), n_local, _ptr(rowptr), _stream()), "gn_rowptr_slice")
    a, b = (int(v) for v in csr.rowptr[[r0, r1]].tolist())          # two host reads at graph-build time
    col = csr.col[a:b].clone() if b > a else torch.empty(1, dtype=torch.int32, device=dev)
    val = None
    if csr.val is not None:
        val = csr.val[a:b].clone() if b > a else torch.empty(1, dtype=torch.float32, device=dev)
    return Csr(rowptr, col, val, n_local, n_cols, b - a)


def filter_edges(edge_index, edge_weight, by_src, lo, hi, chunk=1 << 26):
    """Order-preserving selection of the edges whose source (``by_src``) or destination lies in
    ``[lo, hi)`` (``gn_edge_filter``; long lists go chunk by chunk).  Two passes: count every chunk, ONE
    host read of the counts, then scatter into exactly sized outputs.
    Returns ``(edge_index_local int64 [2, n], edge_weight_local or None)``."""
    lib = _lib.load()
    dev = edge_index.device
    ei = edge_index.contiguous()
    E = int(ei.size(1))
    w = None if edge_weight is None else edge_weight.to(torch.float32).contiguous()
    spans = [(a, min(E, a + chunk)) for a in range(0, E, chunk)]
    counts = torch.zeros(max(len(spans), 1), dtype=torch.int32, device=dev)
    ws = _ws(lib.gn_edge_filter_workspace_bytes(min(E, chunk)), dev)
    for i, (a, b) in enumerate(spans):
        _lib.check(lib.gn_edge_filter(_ptr(ei[0, a:]), _ptr(ei[1, a:]), None, b - a, int(by_src), int(lo), int(hi),
                                      None, None, None, None, 0, _ptr(counts[i:]), _ptr(ws), ws.numel(), _stream()),
                   "gn_edge_filter")
    host = [int(v) for v in counts.tolist()]                      # one host read at graph-build time
    total = sum(host)
    out = torch.empty((2, max(total, 1)), dtype=torch.int64, device=dev)
    out_w = torch.empty(max(total, 1), dtype=torch.float32, device=dev) if w is not None else None
    scratch = torch.zeros(1, dtype=torch.int32, device=dev)
    off = 0
    for (a, b), c in zip(spans, host):
        if c:
            _lib.check(lib.gn_edge_filter(_ptr(ei[0, a:]), _ptr(ei[1, a:]), _ptr(w[a:]) if w is not None else None,
                                          b - a, int(by_src), int(lo), int(hi), _ptr(out[0, off:]), _ptr(out[1, off:]),
                                          _ptr(out_w[off:]) if out_w is not None else None, None, 0, _ptr(scratch),
                                          _ptr(ws), ws.numel(), _stream()), "gn_edge_filter")
        off += c
    return out[:, :total], (out_w[:total] if out_w is not None else None)


def part_structure(shard, weight, key_row, row0, n_rows, with_loops, fill, want_deg):
    """Rows ``[row0, row0 + n_rows)`` of the CSR keyed by row ``key_row`` of ``shard`` (int64 ``[2, e]``, every
    key inside the block; ``gn_gcn_part_structure``) -> ``(rowptr, col, val, deg, dis, nnz)``; ``val`` still
    holds the per-entry weights (``part_values`` turns them into the GCN coefficients)."""
    lib = _lib.load()
    dev = shard.device
    i32 = dict(dtype=torch.int32, device=dev)
    f32 = dict(dtype=torch.float32, device=dev)
    e = int(shard.size(1))
    cap = max(e + (n_rows if with_loops else 0), 1)
    rowptr = torch.empty(max(n_rows, 1) + 1, **i32)
    col, val = torch.empty(cap, **i32), torch.empty(cap, **f32)
    deg = torch.empty(max(n_rows, 1), **f32) if want_deg else None
    dis = torch.empty(max(n_rows, 1), **f32) if want_deg else None
    counts = torch.zeros(4, **i32)
    if n_rows <= 0:
        rowptr.zero_()
        return rowptr, col, val, deg, dis, 0
    ws = _ws(lib.gn_gcn_part_workspace_bytes(e, n_rows), dev)
    _lib.check(lib.gn_gcn_part_structure(
        _ptr(shard[key_row]) if e else None, _ptr(shard[1 - key_row]) if e else None, _ptr(weight), e, int(row0),
        int(n_rows), int(with_loops), float(fill), _ptr(rowptr), _ptr(col), _ptr(val), _ptr(deg), _ptr(dis),
        _ptr(counts), _ptr(ws), ws.numel(), _stream()), "gn_gcn_part_structure")
    return rowptr, col, val, deg, dis, _host_int(counts[0])


def part_values(rowptr, col, val, n_rows, row0, dis_src, dis_dst, transpose):
    """``val <- (dis_src[source] * w) * dis_dst[target]`` with GLOBAL ``deg^-1/2`` vectors (``gn_gcn_part_values``)."""
    if n_rows > 0:
        _lib.check(_lib.load().gn_gcn_part_values(_ptr(rowptr), _ptr(col), int(n_rows), int(row0), _ptr(dis_src),
                                                  _ptr(dis_dst), int(bool(transpose)), _ptr(val), _stream()),
                   "gn_gcn_part_values")


HALO_MODE = os.environ.get("GRIPNET_B200_HALO", "auto")      # "auto" | "off" | "force"
HALO_THRESHOLD = 0.6        # pack when every rank references < 60 % of the remote rows


class HaloPlan:
    """Halo-packed operand layout of one partitioned CSR (``parallel.DistContext.halo_gather``).

    The gathered operand of this rank becomes ``[own block (B rows) | rows of peer 0 it references | peer 1 | ...]``;
    ``need[q]`` are the (sorted, unique) global columns of peer q's block this rank's rows reference, the CSR's
    column indices are remapped IN PLACE to the packed positions, and the lists are exchanged once so that every
    rank knows which of its rows each peer wants (``send_idx[p]``) and where they land there (``dst_row[p]``).
    Built collectively; ``None`` from ``build`` means the full slot all-gather stays (dense references)."""

    @staticmethod
    def build(csr, ctx, block, n_cols_global, r0, r1):
        import torch.distributed as dist
        if HALO_MODE == "off" or ctx.world == 1:
            return None
        dev = csr.col.device
        world, rank = ctx.world, ctx.rank
        cols = csr.col[: csr.nnz].long()
        seen = torch.zeros(world * block, dtype=torch.bool, device=dev)
        if csr.nnz > 0:
            seen[cols] = True
        seen[rank * block:(rank + 1) * block] = False
        need = [seen[q * block:(q + 1) * block].nonzero().view(-1).to(torch.int32) for q in range(world)]   # local ids in q
        counts = torch.tensor([int(t.numel()) for t in need], dtype=torch.int64, device=dev)
        total = int(counts.sum())
        stats = torch.tensor([total], dtype=torch.int64, device=dev)
        dist.all_reduce(stats, op=dist.ReduceOp.MAX, group=ctx.group)
        max_total = int(stats.item())
        if HALO_MODE != "force" and max_total >= HALO_THRESHOLD * (world - 1) * block:
            return None
        plan = HaloPlan()
        plan.block, plan.world, plan.rank = block, world, rank
        plan.rows = block + max_total                       # symmetric buffer size: the largest packed operand
        plan.recv_counts = [int(c) for c in counts.tolist()]
        offs, off = [], block
        for q in range(world):
            offs.append(off)
            off += plan.recv_counts[q]
        plan.recv_off = offs
        # column remap: own block -> [0, B), a referenced remote column -> its packed position
        lut = torch.full((world * block,), -1, dtype=torch.int32, device=dev)
        lut[rank * block:(rank + 1) * block] = torch.arange(block, dtype=torch.int32, device=dev)
        for q in range(world):
            if q != rank and plan.recv_counts[q]:
                lut[q * block + need[q].long()] = offs[q] + torch.arange(plan.recv_counts[q], dtype=torch.int32, device=dev)
        if csr.nnz > 0:
            csr.col[: csr.nnz] = lut[cols]
        # tell every peer which of ITS rows this rank wants, and where they go
        send_counts = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_to_all_single(send_counts, counts, group=ctx.group)
        dst_rows = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_to_all_single(dst_rows, torch.tensor(offs, dtype=torch.int64, device=dev), group=ctx.group)
        plan.send_counts = [int(c) for c in send_counts.tolist()]
        plan.dst_row = [int(c) for c in dst_rows.tolist()]
        flat_need = torch.cat(need) if total else torch.empty(0, dtype=torch.int32, device=dev)
        flat_send = torch.empty(sum(plan.send_counts), dtype=torch.int32, device=dev)
        dist.all_to_all_single(flat_send, flat_need, output_split_sizes=plan.send_counts,
                               input_split_sizes=plan.recv_counts, group=ctx.group)
        plan.send_idx = list(flat_send.split(plan.send_counts))          # local row ids, per destination peer
        plan.send_flat = flat_send
        plan.fraction = max_total / float(max((world - 1) * block, 1))
        return plan


class DistGcnGraph:
    """This rank's rows of a destination-partitioned GCN graph (``parallel.py``), built from this rank's
    edges ONLY: the edges whose destination lies in its block give the rows of the dst-sorted CSR
    (``fwd``: local TARGET rows, columns = global source ids — the gathered operand has ``world * b_src``
    rows), the edges whose source lies in its block give the rows of the transpose CSR (``bwd``: local
    SOURCE rows, columns = global target ids).  No rank sorts or stores the global CSR; the only global
    quantity is the ``deg^-1/2`` vector (one float per node), all-gathered once at build time.  Rows are
    bit-identical to the matching rows of the single-GPU ``GcnGraph``.
    ``n_src`` / ``n_dst`` are the LOCAL row counts the layer stacks see."""

    def __init__(self, edge_index, spec, edge_weight=None, improved=False, bipartite=False):
        import torch.distributed as dist
        ctx = spec.ctx
        dev = edge_index.device
        self.ctx, self.bipartite = ctx, bool(bipartite)
        self.n_src_global, self.n_dst_global = spec.n_src, spec.n_dst
        self.b_src, self.b_dst = ctx.block(spec.n_src), ctx.block(spec.n_dst)
        s0, s1 = ctx.bounds(spec.n_src)
        d0, d1 = ctx.bounds(spec.n_dst)
        self.src_bounds, self.dst_bounds = (s0, s1), (d0, d1)
        self.n_src, self.n_dst = s1 - s0, d1 - d0
        if spec.n_src >= 2 ** 31 or spec.n_dst >= 2 ** 31:
            raise RuntimeError("gripnet_b200: node counts must be < 2^31")
        if spec.shards is None:
            require_cuda(edge_index, "edge_index", torch.int64)
            if edge_index.dim() != 2 or edge_index.size(0) != 2:
                raise RuntimeError("edge_index must have shape [2, E]")
            self.n_edges = int(edge_index.size(1))
            if self.n_edges > 0:
                lo, hi0, hi1 = int(edge_index.min()), int(edge_index[0].max()), int(edge_index[1].max())
                if lo < 0 or hi0 >= spec.n_src or hi1 >= spec.n_dst:
                    raise IndexError("edge_index out of range for the given node counts")
            by_dst, w_dst = filter_edges(edge_index, edge_weight, False, d0, d1)
            by_src, w_src = filter_edges(edge_index, edge_weight, True, s0, s1)
        else:                       # the caller streamed the generator / loader through filter_edges itself
            (by_dst, w_dst), (by_src, w_src) = spec.shards
            self.n_edges = int(spec.n_edges_global)
        fill = 2.0 if improved else 1.0
        with_loops = 0 if bipartite else 1
        f32 = dict(dtype=torch.float32, device=dev)
        rowptr, col, val, deg, dis, nnz = part_structure(by_dst.contiguous(), w_dst, 1, d0, self.n_dst, with_loops,
                                                         fill, True)
        # the one global quantity: deg^-1/2 of every target node (block-padded so index == global node id)
        dis_all = torch.zeros(ctx.world * self.b_dst, **f32)
        dis_all[ctx.rank * self.b_dst: ctx.rank * self.b_dst + self.n_dst].copy_(dis[: self.n_dst])
        if ctx.world > 1:
            streams.effective_stream().synchronize()
            dist.all_gather_into_tensor(dis_all, dis_all[ctx.rank * self.b_dst:(ctx.rank + 1) * self.b_dst].clone(),
                                        group=ctx.group)
        dis_src = None if bipartite else dis_all
        part_values(rowptr, col, val, self.n_dst, d0, dis_src, dis_all, False)
        self.fwd = Csr(rowptr, col, val, self.n_dst, ctx.world * self.b_src, nnz)
        rowptr_t, col_t, val_t, _, _, nnz_t = part_structure(by_src.contiguous(), w_src, 0, s0, self.n_src,
                                                             with_loops, fill, False)
        part_values(rowptr_t, col_t, val_t, self.n_src, s0, dis_src, dis_all, True)
        self.bwd = Csr(rowptr_t, col_t, val_t, self.n_src, ctx.world * self.b_dst, nnz_t)
        # halo-packed operands where the rows reference only part of the remote blocks (power-law graphs)
        self.fwd_halo = HaloPlan.build(self.fwd, ctx, self.b_src, spec.n_src, s0, s1)
        self.bwd_halo = HaloPlan.build(self.bwd, ctx, self.b_dst, spec.n_dst, d0, d1)
        self.nnz = nnz
        self.deg = deg[: self.n_dst]
        self.indeg = (rowptr[1: self.n_dst + 1] - rowptr[: self.n_dst]).to(torch.int32)
        # share of the operand rows this rank's forward rows actually reference (halo statistics): with the
        # uniformly random / hashed R-MAT graphs of the benchmarks it is ~1, which is why the exchange is a full
        # slot all-gather rather than a packed halo
        self._halo = None

    def halo_fraction(self):
        """Fraction of the REMOTE operand rows referenced by this rank's forward rows (one pass, cached)."""
        if self.fwd_halo is not None:
            return self.fwd_halo.fraction
        if self._halo is None:
            n_cols = self.ctx.world * self.b_src
            seen = torch.zeros(n_cols, dtype=torch.bool, device=self.fwd.col.device)
            if self.fwd.nnz > 0:
                seen[self.fwd.col[: self.fwd.nnz].long()] = True
            s0, s1 = self.src_bounds
            remote = int(seen.sum()) - int(seen[s0:s1].sum())
            total_remote = max(self.n_src_global - (s1 - s0), 1)
            self._halo = remote / total_remote
        return self._halo


class DistRgcnGraph:
    """This rank's rows of a destination-partitioned multi-relational graph."""

    def __init__(self, edge_index, range_list, spec, n_rel):
        ctx = spec.ctx
        n = spec.n_dst
        g = RgcnGraph(edge_index, range_list, n, n_rel)
        self.ctx, self.n_rel, self.n_edges = ctx, int(n_rel), g.n_edges
        self.n_global, self.b = n, ctx.block(n)
        r0, r1 = ctx.bounds(n)
        self.bounds = (r0, r1)
        self.n_nodes = r1 - r0
        self.inv_cnt = g.inv_cnt[r0:r1].clone()
        self.fwd = slice_csr(g.fwd, r0, r1, ctx.world * self.b * n_rel)
        self.bwd = slice_csr(g.bwd, r0 * n_rel, r1 * n_rel, ctx.world * self.b)


class PairStruct:
    """(node, relation) pair CSR of an edge list — rows = ``node * n_rel + rel``, entries = (other endpoint,
    edge id) — for the one-gather-pass DistMult backward (``gn_pair_prep`` / ``gn_distmult_bwd_pairs``)."""

    def __init__(self, edge_index, edge_type, n_nodes, n_rel, exact):
        lib = _lib.load()
        dev = edge_index.device
        E = int(edge_index.size(1))
        if 2 * E >= 2 ** 31 or n_nodes * n_rel >= 2 ** 31:
            raise RuntimeError("gripnet_b200: 2*E and num_nodes * num_relations must be < 2^31")
        ei = edge_index.contiguous()
        et = edge_type.contiguous()
        self.edge_index, self.edge_type = ei, et
        self.n_nodes, self.n_rel = int(n_nodes), int(n_rel)
        i32 = dict(dtype=torch.int32, device=dev)
        n_rows = n_nodes * n_rel
        rowptr = torch.empty(n_rows + 1, **i32)
        self.ent_other = torch.empty(max(2 * E, 1), **i32)
        self.ent_eid = torch.empty(max(2 * E, 1), **i32)
        ws = _ws(lib.gn_pair_prep_workspace_bytes(E), dev)
        _lib.check(lib.gn_pair_prep(_ptr(ei[0]) if E else None, _ptr(ei[1]) if E else None, _ptr(et) if E else None,
                                    E, n_nodes, n_rel, _ptr(rowptr), _ptr(self.ent_other), _ptr(self.ent_eid),
                                    _ptr(ws), ws.numel(), _stream()), "gn_pair_prep")
        self.csr = Csr(rowptr, self.ent_other, None, n_rows, n_nodes, 2 * E, exact=exact)


class IndexStruct:
    """CSR of an index list: row n lists the positions i with index[i] == n."""

    def __init__(self, index, n_nodes, exact=True):
        lib = _lib.load()
        dev = index.device
        n = int(index.numel())
        idx = index.contiguous()
        if n > 0 and exact and (int(idx.min()) < 0 or int(idx.max()) >= n_nodes):
            raise IndexError("node_list out of range")
        rowptr = torch.empty(n_nodes + 1, dtype=torch.int32, device=dev)
        self.perm = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        ws = _ws(lib.gn_index_prep_workspace_bytes(n, n_nodes), dev)
        _lib.check(lib.gn_index_prep(_ptr(idx) if n else None, n, n_nodes, _ptr(rowptr), _ptr(self.perm), _ptr(ws),
                                     ws.numel(), _stream()), "gn_index_prep")
        self.csr = Csr(rowptr, self.perm, None, n_nodes, max(n, 1), n, exact=exact)


# --------------------------------------------------------------------------
# structure cache, keyed by tensor identity (the cache entry keeps the key
# tensors alive, so their storage cannot be recycled under a stale entry)
# --------------------------------------------------------------------------
class _Cache:
    def __init__(self, capacity=16):
        self.capacity = capacity
        self.store = OrderedDict()

    @staticmethod
    def tkey(t):
        if t is None:
            return None
        return (t.data_ptr(), tuple(t.shape), tuple(t.stride()), t._version, str(t.dtype))

    def get(self, key, tensors, build):
        hit = self.store.get(key)
        if hit is not None:
            self.store.move_to_end(key)
            return hit[0]
        obj = build()
        self.store[key] = (obj, tensors)
        while len(self.store) > self.capacity:
            self.store.popitem(last=False)
        return obj

    def clear(self):
        self.store.clear()


_cache = _Cache()


def clear_cache():
    _cache.clear()


def _capturing():
    return torch.cuda.is_current_stream_capturing()


# --------------------------------------------------------------------------
# index validation for the decoder paths (the kernels address  z + src[e]*ldz,  w + etype[e]*D,
# score[i*C + label[i]]  directly: an out-of-range id would be a silent out-of-bounds device read where
# the reference raises IndexError).  One host check (min / max) per (tensor identity, version, bound),
# remembered in an LRU; skipped while a CUDA graph is being captured (the eager warm-up iterations that
# precede every capture have validated the same buffers).  An entry lives only as long as the tensor it was
# made for: a later tensor placed in the recycled storage with the same shape would have the same key.
# --------------------------------------------------------------------------
_validated = OrderedDict()
_VALIDATED_CAPACITY = 256


def mark_valid(t, hi):
    """Record that every entry of ``t`` lies in ``[0, hi)`` (producers that guarantee it by construction,
    e.g. the device negative sampler, call this instead of paying the host check)."""
    key = (_Cache.tkey(t), int(hi))
    ref = _validated.get(key)
    if ref is None or ref() is not t:
        _validated[key] = weakref.ref(t, lambda r, k=key: _validated.pop(k) if _validated.get(k) is r else None)
    _validated.move_to_end(key)
    while len(_validated) > _VALIDATED_CAPACITY:
        _validated.popitem(last=False)


def validate_index(t, hi, name):
    """Raise IndexError unless every entry of the int64 CUDA tensor ``t`` lies in ``[0, hi)``."""
    if t is None or t.numel() == 0:
        return
    key = (_Cache.tkey(t), int(hi))
    ref = _validated.get(key)
    if ref is not None and ref() is not None:
        _validated.move_to_end(key)
        return
    if _capturing():
        return
    s = streams.override()
    if s is not None:
        s.synchronize()
    lo, mx = torch.aminmax(t)
    lo, mx = int(lo.item()), int(mx.item())
    if lo < 0 or mx >= hi:
        raise IndexError(f"gripnet_b200: {name} holds ids in [{lo}, {mx}] but the valid range is [0, {int(hi)})")
    mark_valid(t, hi)


def gcn_graph(edge_index, n_src, n_dst, edge_weight=None, improved=False, bipartite=False, want_aug=False):
    from . import parallel
    spec = parallel.lookup(edge_index)
    if spec is not None:          # destination-partitioned edge list: node counts come from the registry
        key = ("dgcn", _Cache.tkey(edge_index), _Cache.tkey(edge_weight), improved, bipartite, spec.ctx.rank)
        return _cache.get(key, (edge_index, edge_weight),
                          lambda: DistGcnGraph(edge_index, spec, edge_weight, improved, bipartite))
    key = ("gcn", _Cache.tkey(edge_index), _Cache.tkey(edge_weight), n_src, n_dst, improved, bipartite, want_aug)
    return _cache.get(key, (edge_index, edge_weight),
                      lambda: GcnGraph(edge_index, n_src, n_dst, edge_weight, improved, bipartite, want_aug))


def _range_key(range_list):
    """Cache key of a ``range_list`` given as a tensor, ndarray or nested list (the reference passes an
    ndarray-backed tensor, utils.py:141-148): tensors by identity + version, anything else by value."""
    if torch.is_tensor(range_list):
        return _Cache.tkey(range_list)
    return tuple(int(v) for v in torch.as_tensor(range_list).flatten().tolist())


def rgcn_graph(edge_index, range_list, n_nodes, n_rel):
    from . import parallel
    spec = parallel.lookup(edge_index)
    if spec is not None:
        key = ("drgcn", _Cache.tkey(edge_index), _range_key(range_list), n_rel, spec.ctx.rank)
        return _cache.get(key, (edge_index, range_list),
                          lambda: DistRgcnGraph(edge_index, range_list, spec, n_rel))
    key = ("rgcn", _Cache.tkey(edge_index), _range_key(range_list), n_nodes, n_rel)
    return _cache.get(key, (edge_index, range_list), lambda: RgcnGraph(edge_index, range_list, n_nodes, n_rel))


def pair_struct(edge_index, edge_type, n_nodes, n_rel):
    key = ("pair", _Cache.tkey(edge_index), _Cache.tkey(edge_type), n_nodes, n_rel)
    exact = not _capturing()
    return _cache.get(key, (edge_index, edge_type),
                      lambda: PairStruct(edge_index, edge_type, n_nodes, n_rel, exact))


def index_struct(index, n_nodes):
    key = ("index", _Cache.tkey(index), n_nodes)
    exact = not _capturing()
    return _cache.get(key, (index,), lambda: IndexStruct(index, n_nodes, exact))
