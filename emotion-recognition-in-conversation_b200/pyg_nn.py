"""Drop-in replacements for the torch_geometric.nn layers the reference imports.

  RGCNConv, TransformerConv   track_mm/cogmen.py:23,65-66
  GraphConv                   track_mm/dgcn_models.py:6,42
Same constructor arguments, same forward signatures, same parameter names/shapes (so a reference
state_dict loads unchanged), PyG-2.x semantics (SURVEY.md 8a rows a6-a8) -- but every forward and
backward runs in libercgraph kernels: one dense transform (K2) followed by one deterministic
gather over the packed CSR (K3) or the fused edge-attention kernel (K4).  CUDA only.
"""
import math

import torch
from torch import nn

from . import ops
from .graph import graph_from_edge_index


def _glorot(t):
    a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        t.uniform_(-a, a)


class RGCNConv(nn.Module):
    """out_i = sum_r mean_{j in N_r(i)} x_j W_r + x_i W_root + b  (PyG RGCNConv, aggr='mean', no bases).

    Computed transform-first: Y = x @ [W_0 | ... | W_{R-1} | W_root] (one GEMM), then
    out_i = sum_e inv_cnt[e] * Y[src_e, type_e] + Y[i, root] + b (one gather).
    """

    def __init__(self, in_channels, out_channels, num_relations):
        super().__init__()
        self.in_channels, self.out_channels, self.num_relations = in_channels, out_channels, num_relations
        self.weight = nn.Parameter(torch.empty(num_relations, in_channels, out_channels))
        self.root = nn.Parameter(torch.empty(in_channels, out_channels))
        self.bias = nn.Parameter(torch.zeros(out_channels))
        _glorot(self.weight)
        _glorot(self.root)

    def forward(self, x, edge_index, edge_type):
        R, H = self.num_relations, self.out_channels
        g = graph_from_edge_index(edge_index, edge_type, x.size(0), R)
        census = g.relation_slots()
        if g.num_relations is not None and g.num_relations > R:
            # The graph numbers more relation ids than this layer has weights: the reference builds GNN with the DEFAULT
            # n_speakers = 2 whatever the data set (cogmen.py:114), so MELD batches (9 speakers, ids up to 161) meet an
            # 8-relation RGCNConv.  PyG loops ``for i in range(num_relations)`` and never selects ids >= R: those edges
            # carry no message.  Same here: ids >= R get slot -1, which every gather kernel skips.
            if census is not None:
                ids = [i for i in census[0] if i < R]
            else:
                ids = list(range(R))
            P = len(ids)
            if P == 0:                                   # no edge of this batch has a relation the layer knows
                return ops.matmul_kn(x, self.root, self.bias)
            table = torch.full((g.num_relations,), -1, dtype=torch.int32)
            table[torch.tensor(ids, dtype=torch.int64)] = torch.arange(P, dtype=torch.int32)
            rel_slot = table.to(x.device, non_blocking=True)
            sel = torch.tensor(ids, dtype=torch.int64, device=x.device)
            wrel = self.weight.index_select(0, sel)
            wcat = torch.cat([wrel.permute(1, 0, 2).reshape(self.in_channels, P * H), self.root], dim=1)
            y = ops.matmul_kn(x, wcat)
            return ops.gather(y, g, H, R, w=g.mean_weight(), bias=self.bias, root_off=P * H, rel_slot=rel_slot, n_slots=P)
        if census is not None and g.num_relations == R and len(census[0]) < R:
            # only the relation ids that occur in this batch are transformed and gathered (one-speaker MOSEI batches use
            # 2 of the 8 ids): Y is [N, (P+1)*H]; the other weights get an exactly-zero gradient, as in the reference
            ids, rel_slot = census
            P = len(ids)
            sel = g.relation_sel()
            wrel = self.weight.index_select(0, sel)
            wcat = torch.cat([wrel.permute(1, 0, 2).reshape(self.in_channels, P * H), self.root], dim=1)
            y = ops.matmul_kn(x, wcat)
            return ops.gather(y, g, H, R, w=g.mean_weight(), bias=self.bias, root_off=P * H, rel_slot=rel_slot, n_slots=P)
        wcat = torch.cat([self.weight.permute(1, 0, 2).reshape(self.in_channels, R * H), self.root], dim=1)
        y = ops.matmul_kn(x, wcat)
        return ops.gather(y, g, H, R, w=g.mean_weight(), bias=self.bias, root_off=R * H)


class TransformerConv(nn.Module):
    """PyG TransformerConv(in, out, heads=1, concat=True), beta=False, dropout=0, root_weight=True."""

    def __init__(self, in_channels, out_channels, heads=1, concat=True):
        super().__init__()
        if heads != 1:
            raise NotImplementedError("the reference only uses heads=1 (track_mm/cogmen.py:66)")
        self.in_channels, self.out_channels, self.heads, self.concat = in_channels, out_channels, heads, concat
        self.lin_key = nn.Linear(in_channels, out_channels)
        self.lin_query = nn.Linear(in_channels, out_channels)
        self.lin_value = nn.Linear(in_channels, out_channels)
        self.lin_skip = nn.Linear(in_channels, out_channels)

    def forward(self, x, edge_index):
        H = self.out_channels
        g = graph_from_edge_index(edge_index, None, x.size(0), 1)
        w = torch.cat([self.lin_query.weight, self.lin_key.weight, self.lin_value.weight, self.lin_skip.weight], 0)
        b = torch.cat([self.lin_query.bias, self.lin_key.bias, self.lin_value.bias, self.lin_skip.bias], 0)
        qkvs = ops.linear(x, w, b)
        return ops.edge_attention(qkvs, g, H, 1.0 / math.sqrt(H))


class GraphConv(nn.Module):
    """out_i = lin_rel(sum_j x_j) + lin_root(x_i)  (PyG GraphConv, aggr='add').

    By linearity lin_rel(sum_j x_j) = sum_j lin_rel.W x_j, so this is again transform-then-gather:
    Y = x @ [W_rel^T | W_root^T], out_i = sum_j Y[j, :H] + Y[i, H:] + b_rel.
    """

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin_rel = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_root = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x, edge_index):
        H = self.out_channels
        g = graph_from_edge_index(edge_index, None, x.size(0), 1)
        w = torch.cat([self.lin_rel.weight, self.lin_root.weight], 0)       # [2H, in]
        y = ops.linear(x, w)
        return ops.gather(y, g, H, 1, w=None, bias=self.lin_rel.bias, root_off=H, use_types=False)
