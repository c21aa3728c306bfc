"""Drop-in for track_mm/dgcn_models.py (reference :10-170): SeqContext, GCN, batch_graphify, edge_perms,
EdgeAtt, Classifier with the reference's constructor arguments, forward signatures and state_dict keys.

Kernel mapping:
  SeqContext   packed 2-layer BiLSTM / BiGRU = hoisted input GEMM (K2) + register-resident recurrence (K6 / K6b) :10-33
  EdgeAtt      u = x W^T (K2) + per-source window softmax (K5); no B*L python loop                  :121-152
  batch_graphify  K1 packed CSR + EdgeAtt weights as edge_norm (canonical edge order)                :51-92
  GCN          vendored RGCNConv(edge_norm) = basis GEMM + relation GEMM + gather (K2,K3); GraphConv :36-48
  Classifier   Linear+ReLU(+Dropout) fused epilogue, Linear; ``emotion_att`` is dead in the reference :155-170
"""
import torch
from torch import nn

from .. import ops
from ..graph import build_graph, speakers_from_edge_dict
from ..models.rgcn import RGCNConv
from ..pyg_nn import GraphConv
from .cogmen_utils import edge_perms  # noqa: F401  (same function in the reference, dgcn_models.py:95-118)


def _fresh_seed():
    return int(torch.empty((), dtype=torch.int64).random_().item())


def birnn_forward(rnn, x2d, graph, a_rows, training):
    """Multi-layer bidirectional nn.LSTM or nn.GRU over the dialogues of ``graph`` (packed-sequence semantics): per layer one
    hoisted input GEMM for all utterances and both directions (K2) + the recurrence kernel (K6 LSTM, K6b GRU)."""
    gru = isinstance(rnn, nn.GRU)
    assert gru or isinstance(rnn, nn.LSTM), type(rnn)
    h = x2d
    for layer in range(rnn.num_layers):
        sfx = "_l%d" % layer
        w_ih = torch.cat([getattr(rnn, "weight_ih" + sfx), getattr(rnn, "weight_ih" + sfx + "_reverse")], 0)
        b_ih = (getattr(rnn, "bias_ih" + sfx), getattr(rnn, "bias_ih" + sfx + "_reverse"))
        b_hh = (getattr(rnn, "bias_hh" + sfx), getattr(rnn, "bias_hh" + sfx + "_reverse"))
        rows = a_rows if layer == 0 else None
        if gru:           # b_hn is scaled by the reset gate, so b_hh stays out of the hoisted GEMM
            gx = ops.linear(h, w_ih, torch.cat(b_ih, 0), a_rows=rows)
        else:
            gx = ops.linear(h, w_ih, torch.cat([b_ih[0] + b_hh[0], b_ih[1] + b_hh[1]], 0), a_rows=rows)
        # W_hh is stacked after the input transform: autograd runs the later node first, so W_hh's gradient is complete
        # before the input transform's weight-gradient GEMM (what the train step's early gradient bucket waits for)
        w_hh = torch.stack([getattr(rnn, "weight_hh" + sfx), getattr(rnn, "weight_hh" + sfx + "_reverse")], 0)
        if gru:
            h = ops.gru_layer(gx, w_hh, torch.stack(b_hh, 0), graph)
        else:
            h = ops.lstm_layer(gx, w_hh, graph)
        if training and rnn.dropout > 0 and layer + 1 < rnn.num_layers:
            h = ops.dropout(h, rnn.dropout, _fresh_seed())
    return h


class SeqContext(nn.Module):
    def __init__(self, u_dim, g_dim, dropout=0.4, rnn_type="lstm"):
        super().__init__()
        self.input_size, self.hidden_dim = u_dim, g_dim
        if rnn_type == "lstm":
            self.rnn = nn.LSTM(u_dim, g_dim // 2, dropout=dropout, bidirectional=True, num_layers=2, batch_first=True)
        elif rnn_type == "gru":
            self.rnn = nn.GRU(u_dim, g_dim // 2, dropout=dropout, bidirectional=True, num_layers=2, batch_first=True)
        else:
            raise ValueError("rnn_type must be 'lstm' or 'gru', got %r" % (rnn_type,))

    def packed_forward(self, x2d, graph, a_rows=None):
        """x2d: [rows, u_dim]; a_rows maps packed node -> row of x2d (None = already packed). -> [N, g_dim]"""
        return birnn_forward(self.rnn, x2d, graph, a_rows, self.training)

    def forward(self, text_len_tensor, text_tensor):
        """Reference signature: -> zero-padded [B, max(L), g_dim] like pad_packed_sequence."""
        B, Lmax, D = text_tensor.shape
        spk = torch.zeros((B, Lmax), dtype=torch.int64, device=text_tensor.device)
        g = build_graph(text_len_tensor, spk, 0, 0, 1, device=text_tensor.device, reference_layout=False, mean_weight=False)
        h = self.packed_forward(text_tensor.reshape(B * Lmax, D), g, a_rows=g.pad_row)
        return ops.unpack_rows(h, g, int(text_len_tensor.max()))


class EdgeAtt(nn.Module):
    def __init__(self, g_dim, wp, wf):
        super().__init__()
        self.wp, self.wf = wp, wf
        self.weight = nn.Parameter(torch.zeros((g_dim, g_dim)).float(), requires_grad=True)
        var = 2.0 / (self.weight.size(0) + self.weight.size(1))
        self.weight.data.normal_(0, var)                     # the reference passes var as the std (:129-130)

    def edge_weights(self, x_packed, graph):
        """nu[e] for every edge in canonical (by-destination) order; x_packed [N, g_dim]."""
        u = ops.linear(x_packed, self.weight)                # u_k = W x_k  (:136-137)
        return ops.edge_att(x_packed, u, graph)

    def forward(self, node_features, text_len_tensor, edge_ind):
        """Reference signature: list of B tensors [Lmax, 110] with alpha[j, k] (row = source j)."""
        B, Lmax, D = node_features.shape
        dev = node_features.device
        spk = torch.zeros((B, Lmax), dtype=torch.int64, device=dev)
        g = build_graph(text_len_tensor, spk, self.wp, self.wf, 1, device=dev, mean_weight=False)
        x = ops.pack_rows(node_features, g)
        nu = self.edge_weights(x, g)
        src, dst = g.edge_index[0], g.edge_index[1]
        d = g.node_dlg.long()[src]
        off = g.node_off.long()[d]
        dense = torch.zeros((B, Lmax, 110), dtype=nu.dtype, device=dev)
        dense = dense.index_put((d, src - off, dst - off), nu)
        return [dense[i] for i in range(B)]


class GCN(nn.Module):
    def __init__(self, g_dim, h1_dim, h2_dim, n_speakers):
        super().__init__()
        self.num_relations = 2 * n_speakers ** 2
        self.conv1 = RGCNConv(g_dim, h1_dim, self.num_relations, num_bases=30)
        self.conv2 = GraphConv(h1_dim, h2_dim)

    def forward(self, node_features, edge_index, edge_norm, edge_type):
        x = self.conv1(node_features, edge_index, edge_type, edge_norm=edge_norm)
        return self.conv2(x, edge_index)


def batch_graphify(features, lengths, speaker_tensor, wp, wf, edge_type_to_idx, att_model):
    """-> (node_features [N,D], edge_index [2,E], edge_norm [E] (differentiable), edge_type [E], edge_index_lengths [B])."""
    n_speakers = speakers_from_edge_dict(edge_type_to_idx)
    g = build_graph(lengths, speaker_tensor, wp, wf, n_speakers, device=features.device, mean_weight=False)
    node_features = ops.pack_rows(features, g)
    edge_norm = att_model.edge_weights(node_features, g)
    g.attach()
    return node_features, g.edge_index, edge_norm, g.edge_type, g.edge_index_lengths


class MaskedEmotionAtt(nn.Module):
    """Dead in the reference (Classifier.forward never calls it, :163-170); kept for its state_dict keys."""

    def __init__(self, input_dim):
        super().__init__()
        self.lin = nn.Linear(input_dim, input_dim)


class Classifier(nn.Module):
    def __init__(self, input_dim, hidden_size, tag_size, dropout, loss_weights=True):
        super().__init__()
        self.emotion_att = MaskedEmotionAtt(input_dim)
        self.lin1 = nn.Linear(input_dim, hidden_size)
        self.drop = nn.Dropout(dropout)
        self.lin2 = nn.Linear(hidden_size, tag_size)

    def forward(self, h, text_len_tensor=None):
        p = self.drop.p if self.training else 0.0
        return ops.mlp_head(h, self.lin1.weight, self.lin1.bias, self.lin2.weight, self.lin2.bias, p,
                            _fresh_seed() if p > 0 else 0)
