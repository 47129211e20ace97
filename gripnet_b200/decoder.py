"""Drop-in ``gripnet.decoder`` on the CUDA path (reference ``gripnet/decoder.py``)."""
import math

import torch
from torch.nn import Module, Parameter

from . import ops, ranking
from .parallel import replicated


class multiRelaInnerProductDecoder(Module):
    """DistMult link decoder ``sigmoid(sum_k z[s,k] z[d,k] w[r,k])`` (``decoder.py:10-26``).

    One fused gather-multiply-reduce kernel; nothing of size ``[E, in_dim]`` is
    materialised, so the reference's activation checkpointing
    (``GripNet-pose.py:133-135``) is unnecessary.  The backward is atomic-free.
    """

    def __init__(self, in_dim, num_et):
        super().__init__()
        self.num_et, self.in_dim = num_et, in_dim
        self.weight = Parameter(torch.empty(num_et, in_dim))
        self.dist_ctx = None          # set to a parallel.DistContext when edge lists are partitioned over ranks
        self.reset_parameters()

    def forward(self, z, edge_index, edge_type, sigmoid=True):
        return ops.DistMult.apply(z, replicated(self.weight, self.dist_ctx), edge_index, edge_type, bool(sigmoid))

    def score_pair(self, z, pos_edge_index, neg_edge_index, edge_type, sigmoid=True, rel_lo=0, n_rel_local=None,
                   struct_branch=None):
        """``(forward(z, pos, et), forward(z, neg, et))`` of one training step
        (``GripNet-pose.py:133-138``) as one autograd node whose two halves run concurrently.
        ``rel_lo`` / ``n_rel_local``: see ``ops.DistMultPair`` (edge lists that only hold a slice of the relations,
        ``edge_type`` shifted by ``rel_lo``).  ``struct_branch``: a ``streams.Branch`` on which the caller already
        started the build of the backward's (node, relation) structures; the decoder's backward joins it."""
        return ops.DistMultPair.apply(z, replicated(self.weight, self.dist_ctx), pos_edge_index, neg_edge_index,
                                      edge_type, bool(sigmoid), int(rel_lo), n_rel_local, struct_branch)

    def topk(self, z, node, rel, k, filter=None, sigmoid=True):
        """The ``k`` most likely tails of every query ``(node[i], rel[i])`` under this decoder's weight, skipping the
        known positives of ``filter`` (a ``ranking.EdgeFilter``): ``(scores [Q, k], ids int64 [Q, k])`` —
        ``ranking.topk``.  No gradient flows through it."""
        return ranking.topk(z, self.weight, node, rel, k, filter=filter, sigmoid=sigmoid)

    def topk_relations(self, z, src, dst, k, filter=None, sigmoid=True):
        """The ``k`` most likely relations of every directed pair ``(src[i], dst[i])`` under this decoder's weight,
        skipping the known triples of ``filter``: ``(scores [Q, k], relation ids int64 [Q, k])`` —
        ``ranking.topk_relations``.  No gradient flows through it."""
        return ranking.topk_relations(z, self.weight, src, dst, k, filter=filter, sigmoid=sigmoid)

    def topk_pairs(self, z, rel, k, filter=None, sigmoid=True):
        """The ``k`` most likely new unordered pairs ``{s, t}`` (``s < t``) of every relation ``rel[i]`` under this
        decoder's weight, skipping the pairs ``filter`` holds in either direction: ``(scores [Q, k], src int64 [Q, k],
        dst int64 [Q, k])`` — ``ranking.topk_pairs``.  No gradient flows through it."""
        return ranking.topk_pairs(z, self.weight, rel, k, filter=filter, sigmoid=sigmoid)

    def reset_parameters(self):
        with torch.no_grad():
            self.weight.normal_(std=1.0 / math.sqrt(self.in_dim))          # decoder.py:25-26


class multiClassInnerProductDecoder(Module):
    """``softmax(z[node_list] W)`` (``decoder.py:29-50``): row-gather GEMM + softmax kernels."""

    def __init__(self, in_dim, num_class):
        super().__init__()
        self.num_class, self.in_dim = num_class, in_dim
        self.weight = Parameter(torch.empty(in_dim, num_class))
        self.dist_ctx = None          # set to a parallel.DistContext when node lists are partitioned over ranks
        self.reset_parameters()

    def forward(self, z, node_list, softmax=True):
        if not torch.is_tensor(node_list):
            node_list = torch.as_tensor(node_list, dtype=torch.int64, device=z.device)
        return ops.MultiClass.apply(z, replicated(self.weight, self.dist_ctx), node_list, bool(softmax))

    def reset_parameters(self):
        bound = math.sqrt(6.0 / (self.in_dim + self.num_class))            # decoder.py:47-49
        with torch.no_grad():
            self.weight.uniform_(-bound, bound)
