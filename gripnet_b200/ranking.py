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


def _edge_count(ei):
    e = int(ei.size(-1))
    if e >= 2 ** 31:
        raise RuntimeError("gripnet_b200: edge lists must hold < 2^31 edges")
    return e


def _ptr_at(t, i):
    """Address of ``t[i]`` (None for None) without building a view: the chunk loops run once per chunk."""
    return None if t is None else t.data_ptr() + i * t.element_size()


class _Grouped:
    """``gn_rank_csr`` of one edge list, the dense view pair queries read at any row: rows ``s * R + r``, entries
    (dst, edge id) sorted by dst."""

    def __init__(self, ei, et, n, r):
        lib = _lib.load()
        dev = ei.device
        e = _edge_count(ei)
        i32 = dict(dtype=torch.int32, device=dev)
        self.rowptr = torch.empty(n * r + 1, **i32)
        self.dst = torch.empty(max(e, 1), **i32)
        self.eid = torch.empty(max(e, 1), **i32)
        ws = _ws(lib.gn_rank_csr_workspace_bytes(e), dev)
        _lib.check(lib.gn_rank_csr(_ptr(ei[0]) if e else None, _ptr(ei[1]) if e else None, _ptr(et) if e else None, e,
                                   n, r, _ptr(self.rowptr), _ptr(self.dst), _ptr(self.eid), _ptr(ws), ws.numel(),
                                   _stream()), "gn_rank_csr")


class _KeyGroups:
    """``gn_rank_group`` of the columns ``(a, b, c)`` of one edge list: rows ("groups") are the distinct key pairs
    ``(a, b)`` in ascending order, entries (``c``, edge id) sorted by ``c`` inside a row."""

    def __init__(self, a, b, c, sizes):
        lib = _lib.load()
        dev = a.device
        e = _edge_count(a)
        i32 = dict(dtype=torch.int32, device=dev)
        self.rowptr = torch.empty(e + 1, **i32)
        self.a, self.b, self.c, self.eid = (torch.empty(max(e, 1), **i32) for _ in range(4))
        count = torch.zeros(1, **i32)
        ws = _ws(lib.gn_rank_group_workspace_bytes(e), dev)
        _lib.check(lib.gn_rank_group(_ptr(a) if e else None, _ptr(b) if e else None, _ptr(c) if e else None, e,
                                     *sizes, _ptr(self.rowptr), _ptr(self.a), _ptr(self.b), _ptr(self.c),
                                     _ptr(self.eid), _ptr(count), _ptr(ws), ws.numel(), _stream()), "gn_rank_group")
        self.n_groups = _host_int(count[0])                             # the one host read, at build time

    def lookup(self, count, a32=None, b32=None, a64=None, b64=None):
        """int32 ``[count]``: the row of every query key pair in this structure, -1 where it holds no such pair."""
        row = torch.empty(max(count, 1), dtype=torch.int32, device=self.rowptr.device)
        _lib.check(_lib.load().gn_rank_lookup(_ptr(self.a), _ptr(self.b), self.n_groups, _ptr(a32), _ptr(b32),
                                              _ptr(a64), _ptr(b64), count, _ptr(row), _stream()), "gn_rank_lookup")
        return row


# Tail queries (s, r, ?) group a triple list by (src, rel) with candidates dst and score the rows z[s] .* w[r]
# against z; relation queries (s, ?, t) group it by (src, dst) with candidates rel and score z[s] .* z[t] against w.
def _columns(view, ei, et, n, r):
    """The key columns ``(a, b)``, the candidate column ``c`` and their sizes of a triple list."""
    if view == "tail":
        return (ei[0], et, ei[1]), (n, r, n)
    return (ei[0], ei[1], et), (n, n, r)


def _tables(view, z, w):
    """``y`` of the query rows ``z[a] .* y[b]`` and the candidate table."""
    return (w, z) if view == "tail" else (z, w)


class EdgeFilter:
    """The known-positive triples ``(s, r, c)`` of one or more edge lists (e.g. train + test), grouped by ``(s, r)``
    and sorted by ``c``.  ``edge_lists``: a sequence of ``(edge_index int64 [2, E], edge_type int64 [E])`` on one
    CUDA device.  Built once; reusable by any number of rankers and top-k calls of the same graph.  The first
    relation query that uses the filter (``RelationRanker``, ``topk_relations``) also builds its pair-grouped view
    from the same triples (the filter keeps them) and caches it here; the first pair query (``topk_pairs``,
    ``PairRanker``) likewise builds and caches a symmetrised view."""

    def __init__(self, edge_lists, num_nodes, num_relations):
        self.num_nodes, self.num_relations = _sizes(num_nodes, num_relations)
        lists = [_edge_list(ei, et, self.num_nodes, self.num_relations, "filter") for ei, et in edge_lists]
        if not lists:
            raise RuntimeError("gripnet_b200: EdgeFilter needs at least one edge list")
        self.device = lists[0][0].device
        if any(ei.device != self.device for ei, _ in lists):
            raise RuntimeError("gripnet_b200: the filter's edge lists must be on one device")
        self._ei = torch.cat([l[0] for l in lists], dim=1) if len(lists) > 1 else lists[0][0]
        self._et = torch.cat([l[1] for l in lists]) if len(lists) > 1 else lists[0][1]
        self.n_edges = int(self._ei.size(1))
        self._views = {}
        self._view("tail", self.num_nodes, self.num_relations, self.device)

    def _view(self, view, n, r, device):
        """The filter's triples grouped for one query kind, built on first use: ``"tail"`` and ``"relation"`` as
        ``_KeyGroups`` of ``_columns``; ``"symmetric"``, the ``_Grouped`` view of the triples and their flipped copies
        (row ``s * R + r`` holds every ``t`` with ``(s, r, t)`` or ``(t, r, s)`` in the filter, sorted)."""
        if (n, r) != (self.num_nodes, self.num_relations) or device != self.device:
            raise RuntimeError("gripnet_b200: the filter was built for another graph (node / relation count or device)")
        if view not in self._views:
            ei, et = self._ei, self._et
            if view == "symmetric":
                self._views[view] = _Grouped(torch.cat([ei, ei.flip(0)], dim=1), torch.cat([et, et]), n, r)
            else:
                cols, sizes = _columns(view, ei, et, n, r)
                self._views[view] = _KeyGroups(*cols, sizes)
        return self._views[view]


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


def _score_chunks(z, y, cand, total, a32=None, b32=None, a64=None, b64=None):
    """Score rows ``S[i] = (z[a_i] .* y[b_i]) . cand^T`` of the queries ``i < total``, one chunk at a time: yields
    ``(i0, cnt, S, lds)`` with the rows of queries ``i0 .. i0 + cnt - 1`` in ``S[0:cnt]`` (one buffer for all)."""
    lib = _lib.load()
    d, m = z.size(1), cand.size(0)
    lds, rows = _chunk_rows(m, total)
    q = torch.empty((rows, d), dtype=torch.float32, device=z.device)
    s = torch.empty((rows, lds), dtype=torch.float32, device=z.device)
    for i0 in range(0, total, rows):
        cnt = min(rows, total - i0)
        _lib.check(lib.gn_rank_rows(z.data_ptr(), ops._ldz(z), y.data_ptr(), ops._ldz(y), d, _ptr_at(a32, i0),
                                    _ptr_at(b32, i0), _ptr_at(a64, i0), _ptr_at(b64, i0), cnt, q.data_ptr(), d,
                                    _stream()), "gn_rank_rows")
        ops.sgemm(False, True, cnt, m, d, q.data_ptr(), d, cand.data_ptr(), ops._ldz(cand), s.data_ptr(), lds,
                  z.device)
        yield i0, cnt, s, lds


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
    """What ``LinkRanker``, ``RelationRanker`` and ``PairRanker`` share: the checked triple list, the prologue and
    output checks of ``ranks`` and the per-relation reduction of ``metrics``.  Subclasses set ``_rel_rowptr``,
    ``_rel_perm`` (the edges of relation ``r`` are ``_rel_perm[_rel_rowptr[r]:_rel_rowptr[r + 1]]`` for ``r < R``)
    and define ``_rank(z, w, out)``, called for a non-empty list."""

    def __init__(self, edge_index, edge_type, num_nodes, num_relations, filter):
        self.num_nodes, self.num_relations = _sizes(num_nodes, num_relations)
        self._ei, self._et = _edge_list(edge_index, edge_type, self.num_nodes, self.num_relations, "query")
        self.device = self._ei.device
        self.n_edges = int(self._ei.size(1))
        self.filter = filter

    def ranks(self, z, weight, out=None):
        """float32 ``[E]``: the filtered rank of every triple against the candidates of the ranker's query kind, in
        the list's order."""
        z, w = _embeddings(z, weight, self.num_nodes, self.num_relations)
        if z.device != self.device:
            raise RuntimeError("gripnet_b200: z is not on the ranker's device")
        if out is None:
            out = torch.empty(self.n_edges, dtype=torch.float32, device=self.device)
        elif out.shape != (self.n_edges,) or out.dtype != torch.float32 or not out.is_contiguous() or \
                out.device != self.device:
            raise RuntimeError("gripnet_b200: out must be a contiguous float32 [E] tensor on the ranker's device")
        if self.n_edges > 0:
            self._rank(z, w, out)
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


class _GroupRanker(_Ranker):
    """``LinkRanker`` and ``RelationRanker``: the list grouped by its key pairs (``_columns`` of the class's
    ``_VIEW``), the filter row of every group found once here, and one loop over chunks of score rows that counts
    the ranks of each group's triples."""

    def __init__(self, edge_index, edge_type, num_nodes, num_relations, filter=None):
        super().__init__(edge_index, edge_type, num_nodes, num_relations, filter)
        n, r = self.num_nodes, self.num_relations
        self._f = filter._view(self._VIEW, n, r, self.device) if filter is not None else None
        cols, sizes = _columns(self._VIEW, self._ei, self._et, n, r)
        self._q = _KeyGroups(*cols, sizes)
        self._f_row = self._f.lookup(self._q.n_groups, a32=self._q.a, b32=self._q.b) if self._f is not None else None
        self._rel_rowptr, self._rel_perm = _relation_index(self._et, r, self.device)

    def _rank(self, z, w, out):
        lib = _lib.load()
        y, cand = _tables(self._VIEW, z, w)
        q = self._q
        fr, fc = (self._f.rowptr, self._f.c) if self._f is not None else (None, None)
        for g0, cnt, s, lds in _score_chunks(z, y, cand, q.n_groups, a32=q.a, b32=q.b):
            _lib.check(lib.gn_rank_count(s.data_ptr(), lds, cand.size(0), cnt, _ptr_at(q.rowptr, g0), _ptr(q.c),
                                         _ptr(q.eid), _ptr_at(self._f_row, g0), _ptr(fr), _ptr(fc), out.data_ptr(),
                                         _stream()), "gn_rank_count")


class LinkRanker(_GroupRanker):
    """Filtered ranks of the edges of one list against all candidate tails, and their per-relation MRR / Hits@k.

    ``edge_index`` int64 ``[2, E]`` / ``edge_type`` int64 ``[E]``: the edges to rank (e.g. the test split);
    ``filter``: an ``EdgeFilter`` of the known positives to skip (None: raw ranks).  The query structure and each
    query's filter row are built once here (one device->host read, the number of distinct ``(s, r)`` queries);
    ``ranks`` / ``metrics`` then read nothing back and branch on no device value, so they can be captured in a CUDA
    graph and replayed every epoch.  One GPU: gather a partitioned ``z`` first (``parallel.all_gather_rows``)."""

    _VIEW = "tail"

    @property
    def n_groups(self):
        """Number of distinct ``(s, r)`` queries of the list."""
        return self._q.n_groups


class RelationRanker(_GroupRanker):
    """Filtered ranks of the triples of one list against all ``R`` relations of their pair, and their per-relation
    MRR / Hits@k.

    ``edge_index`` int64 ``[2, E]`` / ``edge_type`` int64 ``[E]``: the triples ``(s, r, t)`` to rank (e.g. the test
    split), each the query ``(s, ?, t)`` with answer ``r``; ``filter``: an ``EdgeFilter`` of the known triples to
    skip (None: raw ranks).  The pair-grouped query structure and each pair's filter row are built once here (one
    device->host read, the number of distinct directed pairs); ``ranks`` / ``metrics`` then read nothing back and
    branch on no device value, so they can be captured in a CUDA graph.  One GPU: gather a partitioned ``z`` first."""

    _VIEW = "relation"

    @property
    def n_groups(self):
        """Number of distinct directed pairs ``(s, t)`` of the list."""
        return self._q.n_groups


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
        super().__init__(edge_index, edge_type, num_nodes, num_relations, filter)
        lib = _lib.load()
        n, r = self.num_nodes, self.num_relations
        if n * n >= 2 ** 31:
            raise RuntimeError(f"gripnet_b200: PairRanker needs num_nodes^2 < 2^31, got {n} nodes")
        ei, et = self._ei, self._et
        self._f = filter._view("symmetric", n, r, self.device) if filter is not None else None
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

    def _rank(self, z, w, out):
        lib = _lib.load()
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


def _k_arg(k):
    try:
        k_ok = not isinstance(k, bool) and 1 <= operator.index(k) <= MAX_K
    except TypeError:
        k_ok = False
    if not k_ok:
        raise RuntimeError(f"gripnet_b200: k must be an integer in [1, {MAX_K}], got {k!r}")
    return operator.index(k)


def _query_list(a, name, bound, dev):
    """An int64 CUDA index list, flattened and range-checked."""
    a = a if torch.is_tensor(a) else torch.as_tensor(a, dtype=torch.int64, device=dev)
    require_cuda(a, name, torch.int64)
    a = a.contiguous().view(-1)
    validate_index(a, bound, name)
    return a


def _query_lists(a, b, names, bounds, dev):
    """Two equally long int64 CUDA index lists, flattened and range-checked."""
    a, b = _query_list(a, names[0], bounds[0], dev), _query_list(b, names[1], bounds[1], dev)
    if a.numel() != b.numel():
        raise RuntimeError(f"gripnet_b200: {names[0]} and {names[1]} must have the same length")
    return a, b


def _topk(view, z, w, a, b, k, filter, sigmoid):
    """``topk`` / ``topk_relations`` after their argument checks: the top ``k`` candidates of the query rows
    ``z[a_i] .* y[b_i]``, the filter row of ``(a_i, b_i)`` skipped."""
    lib = _lib.load()
    dev = z.device
    f = filter._view(view, z.size(0), w.size(0), dev) if filter is not None else None
    y, cand = _tables(view, z, w)
    nq = a.numel()
    scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    if nq == 0:
        return scores, ids
    f_row = f.lookup(nq, a64=a, b64=b) if f is not None else None
    fr, fc = (f.rowptr, f.c) if f is not None else (None, None)
    for q0, cnt, s, lds in _score_chunks(z, y, cand, nq, a64=a, b64=b):
        _lib.check(lib.gn_rank_topk(s.data_ptr(), lds, cand.size(0), cnt, _ptr_at(f_row, q0), _ptr(fr), _ptr(fc), k,
                                    int(bool(sigmoid)), _ptr_at(scores, q0 * k), _ptr_at(ids, q0 * k), _stream()),
                   "gn_rank_topk")
    return scores, ids


def topk(z, weight, node, rel, k, filter=None, sigmoid=True):
    """The ``k`` (1..256) most likely tails ``c`` of every query ``(node[i], rel[i])`` with ``(node[i], rel[i], c)``
    not in ``filter``: ``(scores float32 [Q, k], ids int64 [Q, k])``, descending pre-sigmoid score, ties by smaller
    id; scores after the sigmoid when ``sigmoid``; id -1 / score NaN where fewer than ``k`` candidates are left."""
    z, w = _embeddings(z, weight)
    n, r = _sizes(z.size(0), w.size(0))
    k = _k_arg(k)
    node, rel = _query_lists(node, rel, ("node", "rel"), (n, r), z.device)
    return _topk("tail", z, w, node, rel, k, filter, sigmoid)


def topk_relations(z, weight, src, dst, k, filter=None, sigmoid=True):
    """The ``k`` (1..256) most likely relations ``r`` of every directed pair ``(src[i], dst[i])`` with
    ``(src[i], r, dst[i])`` not in ``filter``: ``(scores float32 [Q, k], ids int64 [Q, k])``, descending pre-sigmoid
    score, ties by smaller relation id; scores after the sigmoid when ``sigmoid``; id -1 / score NaN where fewer than
    ``k`` relations are left (``k`` may exceed ``R``)."""
    z, w = _embeddings(z, weight)
    n, r = _sizes(z.size(0), w.size(0))
    k = _k_arg(k)
    src, dst = _query_lists(src, dst, ("src", "dst"), (n, n), z.device)
    return _topk("relation", z, w, src, dst, k, filter, sigmoid)


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
    rel = _query_list(rel, "rel", r, dev)
    f = filter._view("symmetric", n, r, dev) if filter is not None else None
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
