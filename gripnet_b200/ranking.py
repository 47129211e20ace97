"""Filtered candidate ranking (MRR, Hits@k) and top-k link prediction for the DistMult decoder.

The evaluation of the training scripts scores each positive against one sampled negative
(``GripNet-pose.py:148-164``).  The other standard protocol of multi-relational link prediction ranks every test
edge ``(s, r, t)`` against ALL candidate tails ``c``, skipping the candidates that are known positives (the
"filtered" setting), and reports MRR and Hits@k; and a trained model is asked for the most likely partners ``c`` of
a query ``(s, r)``.  Both score every candidate, ``S(c) = sum_k z[s,k] w[r,k] z[c,k]``: here as rows of the dense
product ``Q . z^T`` with ``Q[g] = z[s_g] .* w[r_g]`` (tensor cores for tall chunks), around which the kernels of
``csrc/rank.cu`` group the queries, count the filtered ranks, reduce them per relation and select the top k.

Semantics (``include/gripnet_b200.h``, K16):

* ranking and selection use the PRE-sigmoid score (the sigmoid saturates to 1.0f in fp32 and would create ties the
  model does not have); every candidate ``c in [0, n)`` is scored, ``c == s`` included;
* a filter is a set of directed known-positive triples ``(s, r, c)`` (duplicates count once);
* only tail queries ``(s, r, ?)`` are ranked; edge lists that hold both directions of every pair (the pose lists)
  rank the head through the mirrored edge;
* rank (OGB rule): with ``N = {c != t : (s, r, c) not in the filter}``, ``opt = #{c in N : S(c) > S(t)}``,
  ``pess = #{c in N : S(c) >= S(t)}``, ``rank = 1 + (opt + pess) / 2``; ``S(t)`` comes from the same computed row
  as every ``S(c)``;
* top-k: descending pre-sigmoid score, ties by smaller candidate id; id ``-1`` / score NaN pad a query with fewer
  than ``k`` admissible candidates.

Relation queries ``(s, ?, t)`` of a directed pair (``RelationRanker``, ``topk_relations``) score every relation
``r' in [0, R)`` as one row of ``S = P . W^T`` with ``P[g] = z[s_g] .* z[t_g]`` and ``W`` the decoder weight:

* ``S(r') = sum_k z[s,k] z[t,k] w[r',k]``, pre-sigmoid, as above;
* the filter is the same ``EdgeFilter`` (directed triples ``(s, r', t)``, duplicates count once);
* rank of a query triple ``(s, r, t)``: with ``N = {r' != r : (s, r', t) not in the filter}``,
  ``opt = #{r' in N : S(r') > S(r)}``, ``pess = #{r' in N : S(r') >= S(r)}``, ``rank = 1 + (opt + pess) / 2``;
  ``S(r)`` comes from the same computed row as every ``S(r')``;
* metrics: float64 ``[1 + len(hits), R]`` as for ``LinkRanker``, grouped by the relation of the query triple (NaN
  for a relation without query triples);
* top-k over relations: descending pre-sigmoid score, ties by smaller relation id; id ``-1`` / score NaN pad a pair
  with fewer than ``k`` admissible relations (``k`` may exceed ``R``); ``sigmoid`` applies to the returned scores;
* ``P`` is bitwise symmetric (fp32 products commute): ``(s, t)`` and ``(t, s)`` give identical score rows whenever
  both rows take the same product path (the same chunk, hence the same dense-product kernel).

Pair queries ``(?, r, ?)`` of a relation (``topk_pairs``: "which new drug pairs does the model predict for side effect
``r``?") score every unordered node pair; the kernels score tiles of the triangle and keep only the best keys, so the
``[n, n]`` score matrix of a relation is never written:

* candidates are the unordered pairs ``{s, t}`` with ``s < t``: DistMult is symmetric in ``s`` and ``t``, so ``(s, t)``
  and ``(t, s)`` are one prediction, and a self-pair is not an interaction; there is no ordered or self-pair mode;
* ``S(s, t) = sum_k z[s,k] w[r,k] z[t,k]``, pre-sigmoid, as above;
* the filter is the same ``EdgeFilter``: ``{s, t}`` is excluded for ``r`` when ``(s, r, t)`` OR ``(t, r, s)`` is in it;
* order: descending pre-sigmoid score, ties by the smaller ``s``, then the smaller ``t`` (the smaller pair id
  ``s * n + t``); ids ``-1`` / score NaN pad a query with fewer than ``k`` admissible pairs (e.g. ``n < 2``);
  ``sigmoid`` applies to the returned scores;
* ``1 <= k <= 256`` and ``n * n < 2^31`` (the pair id is the low word of the 64-bit selection key); the work grows as
  ``Q * n^2 * D``;
* pair ranking (``PairRanker``): each triple ``(s, r, t)`` of a list is the query ``(?, r, ?)`` with answer
  ``{s, t}``, canonicalised to ``(min(s, t), r, max(s, t))`` (so ``(s, r, t)`` and ``(t, r, s)`` get one rank); the
  candidates are those of ``topk_pairs``; with ``N = {a < b : {a, b} != {s, t}, {a, b} not filtered for r}``,
  ``opt = #{N : S > S(s, t)}``, ``pess = #{N : S >= S(s, t)}``, ``rank = 1 + (opt + pess) / 2``; the target is
  left out of ``N`` whether or not the filter holds it;
* every pair score, the target's and each candidate's, is the one fp32 sequence ``q_f = z[a,f] * w[r,f]`` (rounded),
  ``acc = fmaf(q_f, z[b,f], acc)`` for ``f = 0 .. D-1`` with ``a < b``: a target never ties or beats itself through
  two code paths, and the ranker's scores equal those ``topk_pairs`` selects on (+0 / -0 aside, which compare equal);
* a self-pair triple ``s == t`` is no candidate of any query: its rank is NaN and ``metrics`` leaves it out;
* ranks are exact in float32 while ``n (n - 1) / 2 < 2^23`` (``n <= 4096``) and round to the nearest float32 beyond;
  counts are int32 (``n * n < 2^31``).

Single GPU: a partitioned ``z`` is gathered by the caller first (``parallel.all_gather_rows``).
"""
import ctypes
import operator

import torch

from . import _lib, ops
from .graph import _host_int, _ptr, _stream, _ws, require_cuda, validate_index

# bytes of one chunk of score rows: a few tens of MB, well inside the B200's 126 MB L2
CHUNK_BYTES = 48 << 20
MAX_K = 256


def _edge_list(edge_index, edge_type, num_nodes, num_relations, name):
    require_cuda(edge_index, f"{name} edge_index", torch.int64)
    require_cuda(edge_type, f"{name} edge_type", torch.int64)
    if edge_index.dim() != 2 or edge_index.size(0) != 2 or edge_type.dim() != 1 or \
            edge_type.numel() != edge_index.size(1):
        raise RuntimeError(f"gripnet_b200: {name} edge_index must be [2, E] and edge_type [E]")
    validate_index(edge_index, num_nodes, f"{name} edge_index")
    validate_index(edge_type, num_relations, f"{name} edge_type")
    return edge_index.contiguous(), edge_type.contiguous()


def _sizes(num_nodes, num_relations):
    n, r = int(num_nodes), int(num_relations)
    if n <= 0 or r <= 0:
        raise RuntimeError("gripnet_b200: num_nodes and num_relations must be positive")
    if n * r >= 2 ** 31:
        raise RuntimeError("gripnet_b200: num_nodes * num_relations must be < 2^31")
    return n, r


class _Grouped:
    """``gn_rank_csr`` of one edge list: rows ``s * R + r``, entries (dst, edge id) sorted by dst."""

    def __init__(self, ei, et, n, r, groups):
        lib = _lib.load()
        dev = ei.device
        e = int(ei.size(1))
        if e >= 2 ** 31:
            raise RuntimeError("gripnet_b200: edge lists must hold < 2^31 edges")
        i32 = dict(dtype=torch.int32, device=dev)
        self.rowptr = torch.empty(n * r + 1, **i32)
        self.dst = torch.empty(max(e, 1), **i32)
        self.eid = torch.empty(max(e, 1), **i32)
        self.group_row = torch.empty(n * r, **i32) if groups else None
        count = torch.zeros(1, **i32) if groups else None
        ws = _ws(lib.gn_rank_csr_workspace_bytes(e, n, r), dev)
        _lib.check(lib.gn_rank_csr(_ptr(ei[0]) if e else None, _ptr(ei[1]) if e else None, _ptr(et) if e else None, e,
                                   n, r, _ptr(self.rowptr), _ptr(self.dst), _ptr(self.eid), _ptr(self.group_row),
                                   _ptr(count), _ptr(ws), ws.numel(), _stream()), "gn_rank_csr")
        self.n_groups = _host_int(count[0]) if groups else 0          # the one host read, at build time


class _Paired:
    """``gn_rank_pair_csr`` of one edge list: rows are the distinct directed pairs ``(s, t)`` in ``(src, dst)`` order,
    entries (relation, edge id) sorted by relation inside a row."""

    def __init__(self, ei, et, n, r):
        lib = _lib.load()
        dev = ei.device
        e = int(ei.size(1))
        if e >= 2 ** 31:
            raise RuntimeError("gripnet_b200: edge lists must hold < 2^31 edges")
        i32 = dict(dtype=torch.int32, device=dev)
        self.rowptr = torch.empty(e + 1, **i32)
        self.src = torch.empty(max(e, 1), **i32)
        self.dst = torch.empty(max(e, 1), **i32)
        self.rel = torch.empty(max(e, 1), **i32)
        self.eid = torch.empty(max(e, 1), **i32)
        count = torch.zeros(1, **i32)
        ws = _ws(lib.gn_rank_pair_csr_workspace_bytes(e), dev)
        _lib.check(lib.gn_rank_pair_csr(_ptr(ei[0]) if e else None, _ptr(ei[1]) if e else None, _ptr(et) if e else None,
                                        e, n, r, _ptr(self.rowptr), _ptr(self.src), _ptr(self.dst), _ptr(self.rel),
                                        _ptr(self.eid), _ptr(count), _ptr(ws), ws.numel(), _stream()),
                   "gn_rank_pair_csr")
        self.n_pairs = _host_int(count[0])                             # the one host read, at build time

    def lookup(self, count, pair_src=None, pair_dst=None, src=None, dst=None):
        """int32 ``[count]``: the row of every query pair in this structure, -1 where it holds no such pair."""
        dev = self.rowptr.device
        row = torch.empty(max(count, 1), dtype=torch.int32, device=dev)
        _lib.check(_lib.load().gn_rank_pair_lookup(_ptr(self.src), _ptr(self.dst), self.n_pairs, _ptr(pair_src),
                                                   _ptr(pair_dst), _ptr(src), _ptr(dst), count, _ptr(row), _stream()),
                   "gn_rank_pair_lookup")
        return row


class EdgeFilter:
    """The known-positive triples ``(s, r, c)`` of one or more edge lists (e.g. train + test), grouped by ``(s, r)``
    and sorted by ``c``.  ``edge_lists``: a sequence of ``(edge_index int64 [2, E], edge_type int64 [E])`` on one
    CUDA device.  Built once; reusable by any number of rankers and top-k calls of the same graph.  The first
    relation query that uses the filter (``RelationRanker``, ``topk_relations``) also builds its pair-grouped view
    from the same edge lists (the filter keeps references to them) and caches it here; the first pair query
    (``topk_pairs``) likewise builds and caches a symmetrised view."""

    def __init__(self, edge_lists, num_nodes, num_relations):
        self.num_nodes, self.num_relations = _sizes(num_nodes, num_relations)
        lists = [_edge_list(ei, et, self.num_nodes, self.num_relations, "filter") for ei, et in edge_lists]
        if not lists:
            raise RuntimeError("gripnet_b200: EdgeFilter needs at least one edge list")
        self.device = lists[0][0].device
        if any(ei.device != self.device for ei, _ in lists):
            raise RuntimeError("gripnet_b200: the filter's edge lists must be on one device")
        ei = torch.cat([l[0] for l in lists], dim=1) if len(lists) > 1 else lists[0][0]
        et = torch.cat([l[1] for l in lists]) if len(lists) > 1 else lists[0][1]
        self.n_edges = int(ei.size(1))
        self._g = _Grouped(ei, et, self.num_nodes, self.num_relations, groups=False)
        self._lists = lists
        self._p = None
        self._s = None

    def _check(self, n, r, device):
        if (n, r) != (self.num_nodes, self.num_relations) or device != self.device:
            raise RuntimeError("gripnet_b200: the filter was built for another graph (node / relation count or device)")
        return self._g

    def _pairs(self, n, r, device):
        """The pair-grouped view (``_Paired``) of the filter's triples, built on first use."""
        self._check(n, r, device)
        if self._p is None:
            lists = self._lists
            ei = torch.cat([l[0] for l in lists], dim=1) if len(lists) > 1 else lists[0][0]
            et = torch.cat([l[1] for l in lists]) if len(lists) > 1 else lists[0][1]
            self._p = _Paired(ei, et, self.num_nodes, self.num_relations)
        return self._p

    def _symmetric(self, n, r, device):
        """The grouped view (``_Grouped``) of the filter's triples and their flipped copies, built on first use: row
        ``s * R + r`` holds every ``t`` with ``(s, r, t)`` or ``(t, r, s)`` in the filter, sorted."""
        self._check(n, r, device)
        if self._s is None:
            ei = torch.cat([l[0] for l in self._lists] + [l[0].flip(0) for l in self._lists], dim=1)
            et = torch.cat([l[1] for l in self._lists] * 2)
            self._s = _Grouped(ei, et, self.num_nodes, self.num_relations, groups=False)
        return self._s


def _embeddings(z, weight, n=None, r=None):
    z = ops._as_rows(z.detach(), "z")
    w = ops._as_rows(weight.detach(), "weight").contiguous()
    if w.device != z.device:
        raise RuntimeError("gripnet_b200: z and weight must be on one device")
    if w.size(1) != z.size(1):
        raise RuntimeError(f"gripnet_b200: decoder weight width {w.size(1)} != embedding width {z.size(1)}")
    if n is not None and z.size(0) != n:
        raise RuntimeError(f"gripnet_b200: z has {z.size(0)} rows but the graph has {n} nodes")
    if r is not None and w.size(0) != r:
        raise RuntimeError(f"gripnet_b200: weight has {w.size(0)} rows but the graph has {r} relations")
    if z.size(1) == 0:
        raise RuntimeError("gripnet_b200: embedding width must be positive")
    return z, w


def _chunk_rows(n, total):
    lds = (n + 3) // 4 * 4               # a multiple of 4 floats: tall chunks qualify for the tensor-core product
    return lds, max(1, min(int(total), CHUNK_BYTES // (4 * lds)))


def _pair_scores(z, w, p, s, rows, lds, pair_src=None, pair_dst=None, src=None, dst=None):
    """``S[0:rows] = (z[s_i] .* z[t_i]) . w^T`` for one chunk of pairs."""
    lib = _lib.load()
    d = z.size(1)
    _lib.check(lib.gn_rank_pair_rows(z.data_ptr(), ops._ldz(z), d, _ptr(pair_src), _ptr(pair_dst), _ptr(src),
                                     _ptr(dst), rows, p.data_ptr(), d, _stream()), "gn_rank_pair_rows")
    ops.sgemm(False, True, rows, w.size(0), d, p.data_ptr(), d, w.data_ptr(), d, s.data_ptr(), lds, z.device)


def _relation_index(et, num_relations, device):
    """``gn_index_prep`` of the edge types: the edges of each relation, walked in a fixed order by the per-relation
    reduction."""
    lib = _lib.load()
    e = int(et.numel())
    rowptr = torch.empty(num_relations + 1, dtype=torch.int32, device=device)
    perm = torch.empty(max(e, 1), dtype=torch.int32, device=device)
    ws = _ws(lib.gn_index_prep_workspace_bytes(e, num_relations), device)
    _lib.check(lib.gn_index_prep(_ptr(et) if e else None, e, num_relations, _ptr(rowptr), _ptr(perm), _ptr(ws),
                                 ws.numel(), _stream()), "gn_index_prep")
    return rowptr, perm


class _Ranker:
    """What ``LinkRanker``, ``RelationRanker`` and ``PairRanker`` share: the output checks of ``ranks`` and the
    per-relation reduction of ``metrics``.  Subclasses set ``num_relations``, ``device``, ``n_edges``,
    ``_rel_rowptr``, ``_rel_perm`` (the edges of relation ``r`` are ``_rel_perm[_rel_rowptr[r]:_rel_rowptr[r + 1]]``
    for ``r < R``) and define ``ranks``."""

    def _rank_out(self, out):
        if out is None:
            return torch.empty(self.n_edges, dtype=torch.float32, device=self.device)
        if out.shape != (self.n_edges,) or out.dtype != torch.float32 or not out.is_contiguous() or \
                out.device != self.device:
            raise RuntimeError("gripnet_b200: out must be a contiguous float32 [E] tensor on the ranker's device")
        return out

    def metrics(self, z, weight, hits=(1, 3, 10), out=None):
        """float64 ``[1 + len(hits), R]``: row 0 the MRR, row 1 + i the Hits@``hits[i]`` of each relation (NaN for
        a relation without edges)."""
        lib = _lib.load()
        hits = [int(h) for h in hits]
        if len(hits) > int(lib.gn_rank_max_hits()) or any(h < 1 for h in hits):
            raise RuntimeError(f"gripnet_b200: hits must be at most {int(lib.gn_rank_max_hits())} thresholds >= 1")
        rows = 1 + len(hits)
        if out is None:
            out = torch.empty((rows, self.num_relations), dtype=torch.float64, device=self.device)
        elif out.shape != (rows, self.num_relations) or out.dtype != torch.float64 or not out.is_contiguous() or \
                out.device != self.device:
            raise RuntimeError("gripnet_b200: out must be a contiguous float64 [1 + len(hits), R] tensor on the "
                               "ranker's device")
        rank = self.ranks(z, weight)
        hk = (ctypes.c_int32 * max(len(hits), 1))(*hits)
        _lib.check(lib.gn_rank_metrics(_ptr(rank), _ptr(self._rel_rowptr), _ptr(self._rel_perm), self.num_relations,
                                       hk, len(hits), out.data_ptr(), _stream()), "gn_rank_metrics")
        return out


def _score_rows(z, w, q, s, rows, lds, group_row=None, node=None, rel=None):
    """``S[0:rows] = (z[s_i] .* w[r_i]) . z^T`` for one chunk of queries."""
    lib = _lib.load()
    d = z.size(1)
    _lib.check(lib.gn_rank_query_rows(z.data_ptr(), ops._ldz(z), d, w.data_ptr(), w.size(0), _ptr(group_row),
                                      _ptr(node), _ptr(rel), rows, q.data_ptr(), d, _stream()), "gn_rank_query_rows")
    ops.sgemm(False, True, rows, z.size(0), d, q.data_ptr(), d, z.data_ptr(), ops._ldz(z), s.data_ptr(), lds, z.device)


class LinkRanker(_Ranker):
    """Filtered ranks of the edges of one list against all candidate tails, and their per-relation MRR / Hits@k.

    ``edge_index`` int64 ``[2, E]`` / ``edge_type`` int64 ``[E]``: the edges to rank (e.g. the test split);
    ``filter``: an ``EdgeFilter`` of the known positives to skip (None: raw ranks).  The query structure is built once
    here (one device->host read, the number of distinct ``(s, r)`` queries); ``ranks`` / ``metrics`` then read nothing
    back and branch on no device value, so they can be captured in a CUDA graph and replayed every epoch.  One GPU:
    gather a partitioned ``z`` first (``parallel.all_gather_rows``)."""

    def __init__(self, edge_index, edge_type, num_nodes, num_relations, filter=None):
        self.num_nodes, self.num_relations = _sizes(num_nodes, num_relations)
        ei, et = _edge_list(edge_index, edge_type, self.num_nodes, self.num_relations, "query")
        self.device = ei.device
        self.n_edges = int(ei.size(1))
        self.filter = filter
        self._f = filter._check(self.num_nodes, self.num_relations, self.device) if filter is not None else None
        self._q = _Grouped(ei, et, self.num_nodes, self.num_relations, groups=True)
        self._rel_rowptr, self._rel_perm = _relation_index(et, self.num_relations, self.device)

    @property
    def n_groups(self):
        """Number of distinct ``(s, r)`` queries of the list."""
        return self._q.n_groups

    def ranks(self, z, weight, out=None):
        """float32 ``[E]``: the filtered rank of every edge, in the list's order."""
        lib = _lib.load()
        z, w = _embeddings(z, weight, self.num_nodes, self.num_relations)
        if z.device != self.device:
            raise RuntimeError("gripnet_b200: z is not on the ranker's device")
        out = self._rank_out(out)
        g_total = self._q.n_groups
        if g_total == 0:
            return out
        n, d = self.num_nodes, z.size(1)
        lds, rows = _chunk_rows(n, g_total)
        q = torch.empty((rows, d), dtype=torch.float32, device=self.device)
        s = torch.empty((rows, lds), dtype=torch.float32, device=self.device)
        fr, fd = (self._f.rowptr, self._f.dst) if self._f is not None else (None, None)
        for g0 in range(0, g_total, rows):
            cnt = min(rows, g_total - g0)
            grp = self._q.group_row[g0:]
            _score_rows(z, w, q, s, cnt, lds, group_row=grp)
            _lib.check(lib.gn_rank_count(s.data_ptr(), lds, n, _ptr(grp), cnt, _ptr(self._q.rowptr), _ptr(self._q.dst),
                                         _ptr(self._q.eid), _ptr(fr), _ptr(fd), out.data_ptr(), _stream()),
                       "gn_rank_count")
        return out


class RelationRanker(_Ranker):
    """Filtered ranks of the triples of one list against all ``R`` relations of their pair, and their per-relation
    MRR / Hits@k.

    ``edge_index`` int64 ``[2, E]`` / ``edge_type`` int64 ``[E]``: the triples ``(s, r, t)`` to rank (e.g. the test
    split), each the query ``(s, ?, t)`` with answer ``r``; ``filter``: an ``EdgeFilter`` of the known triples to
    skip (None: raw ranks).  The pair-grouped query structure and each pair's filter row are built once here (one
    device->host read, the number of distinct directed pairs); ``ranks`` / ``metrics`` then read nothing back and
    branch on no device value, so they can be captured in a CUDA graph.  One GPU: gather a partitioned ``z`` first."""

    def __init__(self, edge_index, edge_type, num_nodes, num_relations, filter=None):
        self.num_nodes, self.num_relations = _sizes(num_nodes, num_relations)
        ei, et = _edge_list(edge_index, edge_type, self.num_nodes, self.num_relations, "query")
        self.device = ei.device
        self.n_edges = int(ei.size(1))
        self.filter = filter
        self._f = filter._pairs(self.num_nodes, self.num_relations, self.device) if filter is not None else None
        self._q = _Paired(ei, et, self.num_nodes, self.num_relations)
        self._f_row = None
        if self._f is not None:
            self._f_row = self._f.lookup(self._q.n_pairs, pair_src=self._q.src, pair_dst=self._q.dst)
        self._rel_rowptr, self._rel_perm = _relation_index(et, self.num_relations, self.device)

    @property
    def n_groups(self):
        """Number of distinct directed pairs ``(s, t)`` of the list."""
        return self._q.n_pairs

    def ranks(self, z, weight, out=None):
        """float32 ``[E]``: the filtered relation rank of every triple, in the list's order."""
        lib = _lib.load()
        z, w = _embeddings(z, weight, self.num_nodes, self.num_relations)
        if z.device != self.device:
            raise RuntimeError("gripnet_b200: z is not on the ranker's device")
        out = self._rank_out(out)
        g_total = self._q.n_pairs
        if g_total == 0:
            return out
        r, d = self.num_relations, z.size(1)
        lds, rows = _chunk_rows(r, g_total)
        p = torch.empty((rows, d), dtype=torch.float32, device=self.device)
        s = torch.empty((rows, lds), dtype=torch.float32, device=self.device)
        fr, fd = (self._f.rowptr, self._f.rel) if self._f is not None else (None, None)
        for g0 in range(0, g_total, rows):
            cnt = min(rows, g_total - g0)
            _pair_scores(z, w, p, s, cnt, lds, pair_src=self._q.src[g0:], pair_dst=self._q.dst[g0:])
            _lib.check(lib.gn_rank_pair_count(s.data_ptr(), lds, r, cnt, _ptr(self._q.rowptr[g0:]), _ptr(self._q.rel),
                                              _ptr(self._q.eid),
                                              _ptr(self._f_row[g0:]) if self._f_row is not None else None, _ptr(fr),
                                              _ptr(fd), out.data_ptr(), _stream()), "gn_rank_pair_count")
        return out


class PairRanker(_Ranker):
    """Filtered ranks of the triples of one list among all unordered pairs of their relation, and their per-relation
    MRR / Hits@k.

    ``edge_index`` int64 ``[2, E]`` / ``edge_type`` int64 ``[E]``: the triples ``(s, r, t)`` to rank (e.g. the test
    split), each the query ``(?, r, ?)`` with answer ``{s, t}``; ``filter``: an ``EdgeFilter`` of the known triples,
    read in both directions (None: raw ranks).  ``(s, r, t)`` and ``(t, r, s)`` get the same rank; a self-pair
    triple ``s == t`` is no candidate, so its rank is NaN and ``metrics`` leaves it out.  Needs ``n * n < 2^31``;
    ranks are exact in float32 while ``n (n - 1) / 2 < 2^23`` (``n <= 4096``) and round to the nearest float32
    beyond.  Construction does the host reads (the filter's symmetrised view, the relation index, whether each
    target pair is filtered); ``ranks`` / ``metrics`` then read nothing back and branch on no device value, so they
    can be captured in a CUDA graph.  One GPU: gather a partitioned ``z`` first."""

    def __init__(self, edge_index, edge_type, num_nodes, num_relations, filter=None):
        lib = _lib.load()
        self.num_nodes, self.num_relations = _sizes(num_nodes, num_relations)
        n, r = self.num_nodes, self.num_relations
        if n * n >= 2 ** 31:
            raise RuntimeError(f"gripnet_b200: PairRanker needs num_nodes^2 < 2^31, got {n} nodes")
        ei, et = _edge_list(edge_index, edge_type, n, r, "query")
        self.device = ei.device
        self.n_edges = int(ei.size(1))
        self.filter = filter
        self._f = filter._symmetric(n, r, self.device) if filter is not None else None
        self._ei, self._et = ei, et
        # relation index over R + 1 keys: a self-pair triple takes key R, so metrics (rows 0 .. R - 1) skip it
        key = torch.where(ei[0] == ei[1], torch.full_like(et, r), et)
        self._rel_rowptr, self._rel_perm = _relation_index(key, r + 1, self.device)
        counts = self._rel_rowptr[:r + 1].cpu()                         # the one host read of the index
        self._n_queries = int(counts[r])
        self._groups = torch.nonzero(counts[1:] > counts[:-1]).view(-1).to(torch.int32).to(self.device)
        self._t_filtered = None
        if self._f is not None and self._n_queries > 0:
            self._t_filtered = torch.empty(self._n_queries, dtype=torch.int32, device=self.device)
            _lib.check(lib.gn_rank_rel_pairs_targets(_ptr(ei[0]), _ptr(ei[1]), _ptr(et), _ptr(self._rel_perm),
                                                     self._n_queries, r, _ptr(self._f.rowptr), _ptr(self._f.dst),
                                                     _ptr(self._t_filtered), _stream()), "gn_rank_rel_pairs_targets")
        self._ws_bytes = int(lib.gn_rank_rel_pairs_rank_workspace_bytes(self._n_queries, r))

    @property
    def n_groups(self):
        """Number of distinct relations with rankable (non-self-pair) triples."""
        return int(self._groups.numel())

    def ranks(self, z, weight, out=None):
        """float32 ``[E]``: the filtered pair rank of every triple, in the list's order (NaN for a self-pair)."""
        lib = _lib.load()
        z, w = _embeddings(z, weight, self.num_nodes, self.num_relations)
        if z.device != self.device:
            raise RuntimeError("gripnet_b200: z is not on the ranker's device")
        out = self._rank_out(out)
        if self.n_edges == 0:
            return out
        r = self.num_relations
        ws = _ws(self._ws_bytes, self.device)
        fr, fd = (self._f.rowptr, self._f.dst) if self._f is not None else (None, None)
        ei, et = self._ei, self._et
        _lib.check(lib.gn_rank_rel_pairs_count(z.data_ptr(), ops._ldz(z), z.size(1), w.data_ptr(), r, self.num_nodes,
                                               _ptr(ei[0]), _ptr(ei[1]), _ptr(et), _ptr(self._rel_rowptr),
                                               _ptr(self._rel_perm), self._n_queries, _ptr(self._groups),
                                               self.n_groups, _ptr(fr), _ptr(fd), _ptr(ws), ws.numel(), _stream()),
                   "gn_rank_rel_pairs_count")
        _lib.check(lib.gn_rank_rel_pairs_finish(_ptr(ws), ws.numel(), r, _ptr(self._rel_rowptr), _ptr(self._rel_perm),
                                                self._n_queries, _ptr(self._t_filtered), out.data_ptr(), _stream()),
                   "gn_rank_rel_pairs_finish")
        return out


def _k_arg(k):
    try:
        k_ok = not isinstance(k, bool) and 1 <= operator.index(k) <= MAX_K
    except TypeError:
        k_ok = False
    if not k_ok:
        raise RuntimeError(f"gripnet_b200: k must be an integer in [1, {MAX_K}], got {k!r}")
    return operator.index(k)


def _query_lists(a, b, names, bounds, dev):
    """Two equally long int64 CUDA index lists, flattened and range-checked."""
    a = a if torch.is_tensor(a) else torch.as_tensor(a, dtype=torch.int64, device=dev)
    b = b if torch.is_tensor(b) else torch.as_tensor(b, dtype=torch.int64, device=dev)
    require_cuda(a, names[0], torch.int64)
    require_cuda(b, names[1], torch.int64)
    a, b = a.contiguous().view(-1), b.contiguous().view(-1)
    if a.numel() != b.numel():
        raise RuntimeError(f"gripnet_b200: {names[0]} and {names[1]} must have the same length")
    validate_index(a, bounds[0], names[0])
    validate_index(b, bounds[1], names[1])
    return a, b


def topk(z, weight, node, rel, k, filter=None, sigmoid=True):
    """The ``k`` (1..256) most likely tails ``c`` of every query ``(node[i], rel[i])`` with ``(node[i], rel[i], c)``
    not in ``filter``: ``(scores float32 [Q, k], ids int64 [Q, k])``, descending pre-sigmoid score, ties by smaller
    id; scores after the sigmoid when ``sigmoid``; id -1 / score NaN where fewer than ``k`` candidates are left."""
    lib = _lib.load()
    z, w = _embeddings(z, weight)
    n, r = _sizes(z.size(0), w.size(0))
    dev = z.device
    k = _k_arg(k)
    node, rel = _query_lists(node, rel, ("node", "rel"), (n, r), dev)
    f = filter._check(n, r, dev) if filter is not None else None
    nq = node.numel()
    scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    if nq == 0:
        return scores, ids
    lds, rows = _chunk_rows(n, nq)
    q = torch.empty((rows, z.size(1)), dtype=torch.float32, device=dev)
    s = torch.empty((rows, lds), dtype=torch.float32, device=dev)
    for q0 in range(0, nq, rows):
        cnt = min(rows, nq - q0)
        _score_rows(z, w, q, s, cnt, lds, node=node[q0:], rel=rel[q0:])
        _lib.check(lib.gn_rank_topk(s.data_ptr(), lds, n, r, _ptr(node[q0:]), _ptr(rel[q0:]), cnt,
                                    _ptr(f.rowptr) if f is not None else None, _ptr(f.dst) if f is not None else None,
                                    k, int(bool(sigmoid)), _ptr(scores[q0:]), _ptr(ids[q0:]), _stream()),
                   "gn_rank_topk")
    return scores, ids


def topk_relations(z, weight, src, dst, k, filter=None, sigmoid=True):
    """The ``k`` (1..256) most likely relations ``r`` of every directed pair ``(src[i], dst[i])`` with
    ``(src[i], r, dst[i])`` not in ``filter``: ``(scores float32 [Q, k], ids int64 [Q, k])``, descending pre-sigmoid
    score, ties by smaller relation id; scores after the sigmoid when ``sigmoid``; id -1 / score NaN where fewer than
    ``k`` relations are left (``k`` may exceed ``R``)."""
    lib = _lib.load()
    z, w = _embeddings(z, weight)
    n, r = _sizes(z.size(0), w.size(0))
    dev = z.device
    k = _k_arg(k)
    src, dst = _query_lists(src, dst, ("src", "dst"), (n, n), dev)
    f = filter._pairs(n, r, dev) if filter is not None else None
    nq = src.numel()
    scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    if nq == 0:
        return scores, ids
    f_row = f.lookup(nq, src=src, dst=dst) if f is not None else None
    lds, rows = _chunk_rows(r, nq)
    p = torch.empty((rows, z.size(1)), dtype=torch.float32, device=dev)
    s = torch.empty((rows, lds), dtype=torch.float32, device=dev)
    for q0 in range(0, nq, rows):
        cnt = min(rows, nq - q0)
        _pair_scores(z, w, p, s, cnt, lds, src=src[q0:], dst=dst[q0:])
        _lib.check(lib.gn_rank_pair_topk(s.data_ptr(), lds, r, cnt, _ptr(f_row[q0:]) if f is not None else None,
                                         _ptr(f.rowptr) if f is not None else None,
                                         _ptr(f.rel) if f is not None else None, k, int(bool(sigmoid)),
                                         _ptr(scores[q0:]), _ptr(ids[q0:]), _stream()), "gn_rank_pair_topk")
    return scores, ids


def topk_pairs(z, weight, rel, k, filter=None, sigmoid=True):
    """The ``k`` (1..256) most likely unordered pairs ``{s, t}``, ``s < t``, of every relation query ``rel[i]`` with
    neither ``(s, rel[i], t)`` nor ``(t, rel[i], s)`` in ``filter``: ``(scores float32 [Q, k], src int64 [Q, k],
    dst int64 [Q, k])`` with ``src < dst``, descending pre-sigmoid score, ties by smaller ``src`` then smaller
    ``dst``; scores after the sigmoid when ``sigmoid``; ids -1 / score NaN where fewer than ``k`` pairs are left.
    ``rel`` may repeat a relation.  Needs ``n * n < 2^31``.  After the filter's symmetrised view exists (first use),
    a call reads nothing back to the host and can be captured in a CUDA graph."""
    lib = _lib.load()
    z, w = _embeddings(z, weight)
    n, r = _sizes(z.size(0), w.size(0))
    if n * n >= 2 ** 31:
        raise RuntimeError(f"gripnet_b200: topk_pairs needs num_nodes^2 < 2^31 (pair ids), got {n} nodes")
    dev = z.device
    k = _k_arg(k)
    rel = rel if torch.is_tensor(rel) else torch.as_tensor(rel, dtype=torch.int64, device=dev)
    require_cuda(rel, "rel", torch.int64)
    rel = rel.contiguous().view(-1)
    validate_index(rel, r, "rel")
    f = filter._symmetric(n, r, dev) if filter is not None else None
    nq = rel.numel()
    scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
    src = torch.empty((nq, k), dtype=torch.int64, device=dev)
    dst = torch.empty((nq, k), dtype=torch.int64, device=dev)
    if nq == 0:
        return scores, src, dst
    ws = _ws(lib.gn_rank_rel_pairs_workspace_bytes(nq, n, k), dev)
    _lib.check(lib.gn_rank_rel_pairs_select(z.data_ptr(), ops._ldz(z), z.size(1), w.data_ptr(), r, n, _ptr(rel), nq,
                                            _ptr(f.rowptr) if f is not None else None,
                                            _ptr(f.dst) if f is not None else None, k, _ptr(ws), ws.numel(),
                                            _stream()), "gn_rank_rel_pairs_select")
    _lib.check(lib.gn_rank_rel_pairs_merge(_ptr(ws), ws.numel(), n, nq, k, int(bool(sigmoid)), _ptr(scores), _ptr(src),
                                           _ptr(dst), _stream()), "gn_rank_rel_pairs_merge")
    return scores, src, dst
