"""Drop-in for the live classes of track_mm/mmgcn_models.py: ``GraphConvolution`` (:8-39), ``GCNII_lyc`` (:342-394)
and ``MMGCN`` (:485-646) with the reference's constructor arguments, forward signatures and state_dict keys.

The reference materialises a dense [3N,3N] adjacency (98 % zeros) on the host side of a python double loop and runs
64 dense (3N)^2 x 200 products.  Here ``create_big_adj`` is kernel K7 (block adjacency, ``BlockAdjacency``) and every
propagation is a block product + one GEMM whose epilogue is the GCNII update, the ReLU and the next layer's dropout (K8).
The attention classes of the reference file that MMGCNModule never calls are not rebuilt.
"""
import math

import torch
from torch import nn

from .. import ops, ops_mmgcn
from ..ops_mmgcn import BlockLayout
from .mmgcn_utils import lengths_graph


def _fresh_seed():
    return int(torch.empty((), dtype=torch.int64).random_().item()) & (2 ** 62 - 1)


class BlockAdjacency:
    """What ``create_big_adj`` returns here: the flat non-zero values (a differentiable tensor) + their layout."""

    def __init__(self, values, layout):
        self.values, self.layout = values, layout

    def to_dense(self):
        return self.layout.dense(self.values)


def _need_block(adj):
    if not isinstance(adj, BlockAdjacency):
        raise TypeError("adj must come from MMGCN.create_big_adj of this package (a BlockAdjacency); "
                        "a dense [3N,3N] matrix is never materialised on the GPU path")
    return adj


class GraphConvolution(nn.Module):
    def __init__(self, in_features, out_features, residual=False, variant=False):
        super().__init__()
        self.variant = variant
        self.in_features = 2 * in_features if variant else in_features
        self.out_features = out_features
        self.residual = residual
        self.weight = nn.Parameter(torch.empty(self.in_features, self.out_features))
        self.reset_parameters()

    def reset_parameters(self):
        stdv = 1.0 / math.sqrt(self.out_features)
        self.weight.data.uniform_(-stdv, stdv)

    def forward(self, input, adj, h0, lamda, alpha, l):
        if not self.variant or self.residual:
            raise NotImplementedError("MMGCNModule only builds variant=True, residual=False (track_mm/mmgcn.py:76-80)")
        adj = _need_block(adj)
        theta = math.log(lamda / l + 1)
        return ops_mmgcn.gcnii_layer(input, adj.values, h0, self.weight, adj.layout, theta, alpha, relu=False)


class GCNII_lyc(nn.Module):
    def __init__(self, nfeat, nlayers, nhidden, nclass, dropout, lamda, alpha, variant, return_feature, use_residue,
                 new_graph=False):
        super().__init__()
        if not (variant and return_feature):
            raise NotImplementedError("MMGCNModule only builds variant=True, return_feature=True (track_mm/mmgcn.py:76-80)")
        self.return_feature, self.use_residue, self.new_graph = return_feature, use_residue, new_graph
        self.convs = nn.ModuleList([GraphConvolution(nhidden, nhidden, variant=variant) for _ in range(nlayers)])
        self.fcs = nn.ModuleList([nn.Linear(nfeat, nhidden)])
        self.dropout, self.alpha, self.lamda = dropout, alpha, lamda

    def forward(self, x, dia_len, topicLabel, adj=None):
        if adj is None:
            raise NotImplementedError("the reference's MMGCN always passes create_big_adj's result (mmgcn_models.py:570)")
        adj = _need_block(adj)
        p = self.dropout if self.training else 0.0
        seed = _fresh_seed()
        if p > 0:
            x = ops.dropout(x, p, seed)
        fc = self.fcs[0]
        h = ops_mmgcn.gcnii_stack(x, adj.values, fc.weight, fc.bias, [c.weight for c in self.convs], adj.layout,
                                  self.lamda, self.alpha, p, ops_mmgcn.site_seed(seed, 1, ops.SEED_DEV))
        return torch.cat([x, h], dim=-1) if self.use_residue else h


class MMGCN(nn.Module):
    def __init__(self, a_dim, v_dim, l_dim, n_dim, nlayers, nhidden, nclass, dropout, lamda, alpha, variant,
                 return_feature, use_residue, new_graph='full', n_speakers=2, modals=['a', 'v', 't'], use_speaker=True,
                 use_modal=False):
        super().__init__()
        if use_modal or not return_feature:
            raise NotImplementedError("MMGCNModule builds use_modal=False, return_feature=True (track_mm/mmgcn.py:76-80)")
        self.return_feature, self.use_residue, self.new_graph = return_feature, use_residue, new_graph
        self.graph_net = GCNII_lyc(nfeat=n_dim, nlayers=nlayers, nhidden=nhidden, nclass=nclass, dropout=dropout,
                                   lamda=lamda, alpha=alpha, variant=variant, return_feature=return_feature,
                                   use_residue=use_residue)
        # dead in the reference's forward, kept for state_dict compatibility (mmgcn_models.py:498-514)
        self.a_fc = nn.Linear(a_dim, n_dim)
        self.v_fc = nn.Linear(v_dim, n_dim)
        self.l_fc = nn.Linear(l_dim, n_dim)
        self.feature_fc = nn.Linear(n_dim * 3 + nhidden * 3, nhidden) if use_residue else nn.Linear(nhidden * 3, nhidden)
        self.final_fc = nn.Linear(nhidden, nclass)
        self.modal_embeddings = nn.Embedding(3, n_dim)
        self.speaker_embeddings = nn.Embedding(n_speakers, n_dim)
        self.a_spk_embs = nn.Embedding(n_speakers, n_dim)
        self.v_spk_embs = nn.Embedding(n_speakers, n_dim)
        self.l_spk_embs = nn.Embedding(n_speakers, n_dim)
        self.dropout, self.alpha, self.lamda = dropout, alpha, lamda
        self.modals, self.use_speaker, self.use_modal = modals, use_speaker, use_modal

    def _present(self, a, v, l):
        return [x for x, k in ((a, 'a'), (v, 'v'), (l, 't')) if k in self.modals]

    def create_big_adj(self, a, v, l, dia_len, modals, graph=None):
        feats = [x for x, k in ((a, 'a'), (v, 'v'), (l, 't')) if k in modals]
        if len(feats) < 2:
            raise NotImplementedError("the reference returns NotImplementedError for a single modality (:596-597)")
        g = graph if graph is not None else lengths_graph(dia_len, feats[0].device)
        layout = BlockLayout(g, len(feats), dia_len)
        return BlockAdjacency(ops_mmgcn.big_adj(torch.cat(feats, 0), layout), layout)

    def forward(self, a, v, l, dia_len, qmask, graph=None):
        """a, v, l: packed [N, n_dim]; qmask: seq-first one-hot speakers [Lmax, B, n_speakers] -> [N, M*(n_dim+nhidden)]"""
        dev = next(x.device for x in (a, v, l) if torch.is_tensor(x))
        g = graph if graph is not None else lengths_graph(dia_len, dev)
        if self.use_speaker and 't' in self.modals:
            rows = ops_mmgcn.node_rows(g, qmask.size(0), seq_first=True)
            l, _ = ops_mmgcn.speaker_embed_add(l, qmask, rows, self.speaker_embeddings.weight)
        feats = self._present(a, v, l)
        if len(feats) < 2:
            raise NotImplementedError("the reference returns NotImplementedError for a single modality (:562-563)")
        layout = BlockLayout(g, len(feats), dia_len)
        features = torch.cat(feats, 0)
        adj = BlockAdjacency(ops_mmgcn.big_adj(features, layout), layout)
        out = self.graph_net(features, None, qmask, adj)
        N = g.N
        return torch.cat([out[m * N:(m + 1) * N] for m in range(len(feats))], dim=-1)
