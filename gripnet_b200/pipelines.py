"""The reference training scripts' model wiring, as reusable containers.

``PoseModel`` = ``GripNet-pose.py:73-99`` (``Model(gg, gd, dd, dmt)``) + the
forward/loss part of its ``train()`` (``:117-142``); ``AminerModel`` =
``GripNet-aminer.py:83-108,124-133``; ``FreebaseDModel`` =
``GripNet-freebase-d.py:78-137,151-166``.  Submodule names match the scripts, so
a ``state_dict`` saved by the reference scripts loads unchanged.
Used by ``bench.py``, ``__graft_entry__.smoke()`` and the parity tests.
"""
import torch
from torch.nn import Module, Parameter

from . import parallel
from .decoder import multiClassInnerProductDecoder, multiRelaInnerProductDecoder
from . import graph as G
from . import ops, streams
from .layers import homoGraph, interGraph
from .losses import link_prediction_loss, node_classification_loss


class PoseModel(Module):
    def __init__(self, n_g, n_d, n_rel, gg=(32, 16, 16), gd=(16, 32), dd_out=32, n_base=32):
        super().__init__()
        dd = [sum(gd), dd_out]
        self.gg = homoGraph(list(gg), start_graph=True, in_dim=n_g)
        self.gd = interGraph(sum(gg), gd[0], n_d, target_feat_dim=gd[1])
        self.dd = homoGraph(dd, multi_relational=True, n_rela=n_rel, n_base=n_base)
        self.dmt = multiRelaInnerProductDecoder(sum(dd), n_rel)

    def embed(self, data, after_first=None):
        z = self.gg(None, data["gg_edge_index"], edge_weight=data.get("gg_edge_weight"), if_catout=True)
        if after_first is not None:
            after_first()
        z = self.gd(z, data["gd_edge_index"], mod="cat", if_relu=True)
        return self.dd(z, data["dd_edge_index"], edge_type=data["dd_edge_type"],
                       range_list=data["dd_range_list"], if_catout=True)

    def forward(self, data, neg_edge_index=None):
        """Returns (loss, z, pos_score, neg_score) for one training step's forward.

        Partitioned run (``data`` from ``shard_pose``): ``z`` holds this rank's drug rows, the scores
        are those of this rank's slice of the edge lists, the loss is the global mean — or, with
        ``DistContext(defer_grad_reduce=True)``, this rank's SHARE of it (same backward); the global value
        is then in ``dctx.loss_value`` after ``dctx.reduce_gradients(...)``."""
        dctx = data.get("dist")
        if dctx is not None:
            dctx.begin_step()
        if dctx is None:
            pos, et = data["dd_edge_index"], data["dd_edge_type"]
            neg = data["neg_edge_index"] if neg_edge_index is None else neg_edge_index
            n_dec = self.gd.n_target
        else:
            # this rank's slice of the relation-major lists covers relations [rel_lo, rel_lo + rel_n) only
            pos, et = data["dd_edge_index_local"], data["dd_edge_type_shifted"]
            neg = data["neg_edge_index_local"] if neg_edge_index is None else neg_edge_index
            n_dec = dctx.world * dctx.block(data["n_d_global"])
            rel_lo, rel_n = data["dd_rel_lo"], data["dd_rel_n"]
        # the decoder backward's (node, relation) structures depend on the edge lists only — the negatives' one is
        # rebuilt every step (GripNet-pose.py:131 resamples them).  The build is forked BEFORE the first kernel of the
        # step on a background-priority stream: its ~15 small kernels are roots of the captured graph, fill SM slots
        # the dependency chain leaves idle, and are joined where they are consumed (the decoder's backward).  Forked
        # behind the first supervertex instead, the build ends ~30 us after the loss is ready and the backward waits
        # for it (profiles/r02_v19_*).
        prep = streams.Branch(background=True)
        if torch.is_grad_enabled():
            with prep(pos, neg, et):
                G.pair_struct(neg, et, n_dec, self.dmt.num_et if dctx is None else rel_n)
                G.pair_struct(pos, et, n_dec, self.dmt.num_et if dctx is None else rel_n)

        def after_first():
            # W[r] / image of the relational layer: needed ~30 us after the first supervertex, so they are forked
            # behind it (two fewer launches ahead of the chain's first kernel)
            self.dd.prologue(n_dec)

        z = self.embed(data, after_first=after_first)
        # `prep` is NOT joined here: only the decoder's backward reads the structures (it joins the branch)
        if dctx is None:
            pos_score, neg_score = self.dmt.score_pair(z, pos, neg, et, struct_branch=prep)
            return link_prediction_loss(pos_score, neg_score), z, pos_score, neg_score
        z_full = parallel.all_gather_rows(z, dctx, data["n_d_global"])
        pos_score, neg_score = self.dmt.score_pair(z_full, pos, neg, et, rel_lo=rel_lo, n_rel_local=rel_n,
                                                   struct_branch=prep)
        loss = parallel.global_mean_loss(link_prediction_loss(pos_score, neg_score), pos_score.numel(),
                                         data["e_dd_global"], dctx)
        return loss, z, pos_score, neg_score


class AminerModel(Module):
    def __init__(self, n_p, n_a, n_class, pp=(128, 64, 64), pa=(64, 64), aa_hid=(128, 32)):
        super().__init__()
        aa = [sum(pa)] + list(aa_hid)
        self.pp = homoGraph(list(pp), start_graph=True, in_dim=n_p)
        self.pa = interGraph(sum(pp), pa[0], n_a, target_feat_dim=pa[1])
        self.aa = homoGraph(aa)
        self.mcip = multiClassInnerProductDecoder(sum(aa), n_class)

    def forward(self, data):
        z = self.pp(None, data["pp_edge_index"], edge_weight=data.get("pp_edge_weight"), if_catout=True)
        z = self.pa(z, data["pa_edge_index"], if_relu=True, mod="cat")
        z = self.aa(z, data["aa_edge_index"], edge_weight=data.get("aa_edge_weight"), if_catout=True)
        score = self.mcip(z, data["train_node_idx"])
        return node_classification_loss(score, data["train_node_class"]), z, score


class FreebaseDModel(Module):
    def __init__(self, n_p, n_q, n_a, n_class, pp=(256, 128, 128), pa=(128, 128), aa_out=32):
        super().__init__()
        self.pp = homoGraph(list(pp), start_graph=True, in_dim=n_p)
        self.pa = interGraph(sum(pp), pa[0], n_a, target_feat_dim=pa[1], if_one_external=False)
        self.qq = homoGraph(list(pp), start_graph=True, in_dim=n_q)
        self.qa = interGraph(sum(pp), pa[0], n_a, target_feat_dim=pa[1], if_one_external=False)
        self.aa_embeddings = Parameter(torch.randn(n_a, pa[1]))
        self.aa = homoGraph([pa[1], aa_out])
        self.mcip = multiClassInnerProductDecoder(aa_out, n_class)

    def forward(self, data):
        z = self.pa(self.pp(None, data["pp_edge_index"], if_catout=True), data["pa_edge_index"], mod="add",
                    if_relu=True)
        z1 = self.qa(self.qq(None, data["qq_edge_index"], if_catout=True), data["qa_edge_index"], mod="add",
                     if_relu=True)
        z = self.aa(ops.mean3(z, z1, self.aa_embeddings), data["aa_edge_index"])    # freebase-d.py:160-164
        score = self.mcip(z, data["train_node_idx"])
        return node_classification_loss(score, data["train_node_class"]), z, score


class ChainModel(Module):
    """Three-supervertex chain A -> B -> C for node classification on C (BASELINE config 5: the
    aminer wiring, ``GripNet-aminer.py:103-108``, extended by one more supervertex).  Widths default
    to the F=64 hidden size of SURVEY.md §8d."""

    def __init__(self, n_a, n_b, n_c, n_class, hid=64, out=32):
        super().__init__()
        self.aa = homoGraph([hid, hid, hid], start_graph=True, in_dim=n_a)                    # -> 3*hid
        self.ab = interGraph(3 * hid, hid, n_b, target_feat_dim=hid)                          # -> 2*hid
        self.bb = homoGraph([2 * hid, hid, hid])                                              # -> 4*hid
        self.bc = interGraph(4 * hid, hid, n_c, target_feat_dim=hid)                          # -> 2*hid
        self.cc = homoGraph([2 * hid, hid, out])                                              # -> 3*hid + out
        self.mcip = multiClassInnerProductDecoder(3 * hid + out, n_class)

    def forward(self, data):
        if data.get("dist") is not None:
            data["dist"].begin_step()
        z = self.aa(None, data["aa_edge_index"], if_catout=True)
        z = self.ab(z, data["ab_edge_index"], if_relu=True, mod="cat")
        z = self.bb(z, data["bb_edge_index"], if_catout=True)
        z = self.bc(z, data["bc_edge_index"], if_relu=True, mod="cat")
        z = self.cc(z, data["cc_edge_index"], if_catout=True)
        score = self.mcip(z, data["train_node_idx"])          # local ids of this rank's labelled nodes
        loss = node_classification_loss(score, data["train_node_class"])
        dctx = data.get("dist")
        if dctx is not None:
            loss = parallel.global_mean_loss(loss, score.size(0), data["n_train_global"], dctx)
        return loss, z, score


def chain_edges_per_epoch(g):
    """Input edges traversed by one forward of ``ChainModel`` (2 GCN layers per supervertex)."""
    c = g.get("edge_counts")
    if c is None:
        c = {k: g[k + "_edge_index"].shape[1] for k in ("aa", "ab", "bb", "bc", "cc")}
    return 2 * c["aa"] + c["ab"] + 2 * c["bb"] + c["bc"] + 2 * c["cc"]


# ----------------------------------------------------------------------------------------------
# destination-partitioned runs (parallel.py): every rank holds the GLOBAL edge lists (registered as
# partitioned), its own rows of the row-partitioned parameters and its slice of the decoder lists
# ----------------------------------------------------------------------------------------------
def shard_pose(g, dctx, device):
    """Per-rank ``data`` dict for ``PoseModel`` built with LOCAL node counts."""
    d = to_device(g, device)
    n_g, n_d = g["n_g"], g["n_d"]
    parallel.distribute_edges(d["gg_edge_index"], dctx, n_g)
    parallel.distribute_edges(d["gd_edge_index"], dctx, n_g, n_d)
    parallel.distribute_edges(d["dd_edge_index"], dctx, n_d)
    e = g["dd_edge_index"].shape[1]
    e0, e1 = dctx.edge_slice(e)
    et_loc = g["dd_edge_type"][e0:e1]
    rel_lo = int(et_loc.min()) if e1 > e0 else 0
    rel_n = (int(et_loc.max()) - rel_lo + 1) if e1 > e0 else 1
    d.update({
        "dd_rel_lo": rel_lo, "dd_rel_n": rel_n,
        "dd_edge_type_shifted": (d["dd_edge_type"][e0:e1] - rel_lo).contiguous(),
        "dist": dctx, "n_g_global": n_g, "n_d_global": n_d, "e_dd_global": e,
        "n_g": dctx.local_count(n_g), "n_d": dctx.local_count(n_d), "edge_slice": (e0, e1),
        "dd_edge_index_local": d["dd_edge_index"][:, e0:e1].contiguous(),
        "dd_edge_type_local": d["dd_edge_type"][e0:e1].contiguous(),
        "neg_edge_index_local": d["neg_edge_index"][:, e0:e1].contiguous(),
    })
    return d


def shard_pose_params(flat, g, dctx):
    """Rows of the row-partitioned parameters owned by this rank; everything else is replicated."""
    out = dict(flat)
    out["gg.embedding"] = dctx.shard_rows(flat["gg.embedding"], g["n_g"]).clone()
    out["gd.target_feat"] = dctx.shard_rows(flat["gd.target_feat"], g["n_d"]).clone()
    return out


ROW_PARTITIONED = {"gg.embedding": "n_g", "gd.target_feat": "n_d",
                   "aa.embedding": "n_a", "ab.target_feat": "n_b", "bc.target_feat": "n_c"}


def shard_chain(g, dctx, device):
    """Per-rank ``data`` dict for ``ChainModel`` (labelled nodes of C are handled by their owner rank)."""
    d = to_device(g, device)
    n_a, n_b, n_c = g["n_a"], g["n_b"], g["n_c"]
    parallel.distribute_edges(d["aa_edge_index"], dctx, n_a)
    parallel.distribute_edges(d["ab_edge_index"], dctx, n_a, n_b)
    parallel.distribute_edges(d["bb_edge_index"], dctx, n_b)
    parallel.distribute_edges(d["bc_edge_index"], dctx, n_b, n_c)
    parallel.distribute_edges(d["cc_edge_index"], dctx, n_c)
    r0, r1 = dctx.bounds(n_c)
    idx, cls = d["train_node_idx"], d["train_node_class"]
    mine = ((idx >= r0) & (idx < r1)).nonzero().view(-1)
    d.update({"dist": dctx, "n_train_global": int(idx.numel()),
              "n_a": dctx.local_count(n_a), "n_b": dctx.local_count(n_b), "n_c": r1 - r0,
              "train_node_idx": (idx[mine] - r0).contiguous(), "train_node_class": cls[mine].contiguous()})
    return d


def shard_chain_streamed(make_graph, dctx, device):
    """Per-rank ``data`` dict for ``ChainModel`` WITHOUT any rank holding a global edge list: ``make_graph``
    (``synthdata.chain_full`` / ``chain_small``) streams every intra-supervertex graph chunk by chunk through
    sinks that keep only the edges touching this rank's block (``graph.filter_edges``) and registers the two
    shards (by destination -> forward CSR rows, by source -> transpose CSR rows) with
    ``parallel.distribute_edge_shards``.  Every rank consumes the generator's random stream identically, so the
    union of the shards is exactly the graph the single-GPU run sees."""
    from .graph import filter_edges

    def homo_sink(name, n, e_directed, half_chunks):
        r0, r1 = dctx.bounds(n)
        a_parts, b_parts = [], []
        for chunk in half_chunks:                          # global list = [half, flip(half)]
            a_parts.append(filter_edges(chunk, None, False, r0, r1)[0])      # half, destination in the block
            b_parts.append(filter_edges(chunk, None, True, r0, r1)[0])       # half, source in the block
            del chunk
        a, b = torch.cat(a_parts, dim=1), torch.cat(b_parts, dim=1)
        by_dst = torch.cat([a, b.flip(0)], dim=1).contiguous()
        by_src = torch.cat([b, a.flip(0)], dim=1).contiguous()
        return parallel.distribute_edge_shards(by_dst, by_src, dctx, n, n, n_edges_global=e_directed)

    def bip_sink(name, ns, nt, ei):
        s0, s1 = dctx.bounds(ns)
        t0, t1 = dctx.bounds(nt)
        by_dst = filter_edges(ei, None, False, t0, t1)[0].contiguous()
        by_src = filter_edges(ei, None, True, s0, s1)[0].contiguous()
        return parallel.distribute_edge_shards(by_dst, by_src, dctx, ns, nt, n_edges_global=ei.size(1))

    g = make_graph(device, homo_sink=homo_sink, bip_sink=bip_sink)
    n_a, n_b, n_c = g["n_a"], g["n_b"], g["n_c"]
    r0, r1 = dctx.bounds(n_c)
    idx, cls = g["train_node_idx"], g["train_node_class"]
    mine = ((idx >= r0) & (idx < r1)).nonzero().view(-1)
    d = dict(g)
    d.update({"dist": dctx, "n_train_global": int(idx.numel()), "n_a_global": n_a, "n_b_global": n_b,
              "n_c_global": n_c, "n_a": dctx.local_count(n_a), "n_b": dctx.local_count(n_b), "n_c": r1 - r0,
              "train_node_idx": (idx[mine] - r0).contiguous(), "train_node_class": cls[mine].contiguous()})
    return d


def to_device(data, device):
    """Tensors of a graph dict on ``device``, CONTIGUOUS: an edge list that arrives as a strided view (numpy fancy
    indexing returns Fortran-ordered index arrays) would be re-packed by every decoder call of every step
    (``r02_final_launches_pose2.csv``: a 133 MB strided copy, 62 us per step at pose-2 size)."""
    return {k: (v.to(device).contiguous() if torch.is_tensor(v) else v) for k, v in data.items()}


def load_flat_params(model, flat):
    """Load a flat {"gg.embedding": ..., "dmt.weight": ...} dict (oracle / reference naming)."""
    sd = model.state_dict()
    missing = set(sd.keys()) ^ set(flat.keys())
    if missing:
        raise KeyError(f"parameter name mismatch: {sorted(missing)}")
    model.load_state_dict({k: torch.as_tensor(v) for k, v in flat.items()})
    return model
