"""Drop-in for ``DGCNModule`` of track_mm/dgcnv2.py (reference :54-181; declare-lab DialogueGCN): same constructor, forward
signature ``(input_tensor [L,B,D], speaker_tensor one-hot [L,B,n], attention_mask [B,L], text_length)`` (seq-first, one-hot
speakers: dgcnv2.py:44-45), return values (logits [N,C] of the real utterances, features [N,2*hidden]) and state_dict keys.
Base models: 'LSTM' (the default, dgcnv2.py:31: unpacked 2-layer BiLSTM over the padded batch), 'GRU' (the same with a 2-layer
BiGRU, K6b) and 'None' (a Linear).  'DialogRNN' is not rebuilt: no reference output pins the DialogueRNN classes."""
import torch
from torch import nn

from .. import ops, ops_mmgcn
from ..graph import build_graph, standard_edge_dict
from .dgcn_models import birnn_forward
from .dgcnv2_models import MaskedEdgeAttention, GraphNetwork
from .mmgcn_utils import lengths_graph


class DGCNModule(nn.Module):
    def __init__(self, base_model, input_size=100, hidden_size=100, n_speakers=2, window_past=10, window_future=10, n_classes=7,
                 listener_state=False, context_attention="general", dropout_rec=0.5, dropout=0.4, nodal_attention=True, avec=False):
        super().__init__()
        self.base_model, self.avec, self.n_speakers = base_model, avec, n_speakers
        graph_hidden_size, max_seq_len = 100, 110
        if base_model == "LSTM":
            self.lstm = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=2, bidirectional=True, dropout=dropout)
        elif base_model == "GRU":
            self.gru = nn.GRU(input_size=input_size, hidden_size=hidden_size, num_layers=2, bidirectional=True, dropout=dropout)
        elif base_model == "None":
            self.base_linear = nn.Linear(input_size, 2 * hidden_size)
        elif base_model == "DialogRNN":
            raise NotImplementedError("base_model='DialogRNN' is not implemented: the DialogueRNN classes of dgcnv2_models.py are "
                                      "not rebuilt, as no reference output pins them; use 'LSTM', 'GRU' or 'None'")
        else:
            raise NotImplementedError("Base model must be one of DialogRNN/LSTM/GRU")
        if avec:
            raise NotImplementedError("avec regression head is not used by the trainer (dgcnv2.py:186-193)")
        self.window_past, self.window_future = window_past, window_future
        self.att_model = MaskedEdgeAttention(2 * hidden_size, max_seq_len)
        self.att_model.window = (window_past, window_future)
        self.nodal_attention = nodal_attention
        self.graph_net = GraphNetwork(2 * hidden_size, n_classes, 2 * n_speakers ** 2, max_seq_len, graph_hidden_size, dropout)
        self.edge_type_mapping = standard_edge_dict(n_speakers)

    def forward(self, input_tensor, speaker_tensor, attention_mask=None, text_length=None, **kwargs):
        Lmax, B, D = input_tensor.shape
        dev = input_tensor.device
        lens = torch.as_tensor(text_length).to(torch.int64).cpu()
        ids = speaker_tensor.argmax(-1).t().contiguous()                       # [B, Lmax] speaker ids (padding = 0)
        g = build_graph(lens, ids, self.window_past, self.window_future, self.n_speakers, device=dev, mean_weight=False)
        gf = lengths_graph(torch.full((B,), Lmax, dtype=torch.int64), dev)     # every dialogue as a full-length sequence
        rows_full = ops_mmgcn.node_rows(gf, Lmax, seq_first=True)
        x2d = input_tensor.reshape(Lmax * B, D)
        if self.base_model in ("LSTM", "GRU"):                                 # unpacked: runs over the padding, dgcnv2.py:151
            rnn = self.lstm if self.base_model == "LSTM" else self.gru
            emo = birnn_forward(rnn, x2d, gf, rows_full, self.training)
        else:
            emo = ops.linear(x2d, self.base_linear.weight, self.base_linear.bias, a_rows=rows_full)
        edge_norm = self.att_model.edge_weights(emo, g, Lmax)                  # [E], canonical by-destination order
        features = ops.pack_rows(emo.view(B, Lmax, -1), g)                     # the real utterances [N, 2*hidden]
        g.attach()
        gfull = build_graph(lens, torch.zeros(g.N, dtype=torch.int64, device=dev), -1, -1, 1, device=dev, reference_layout=False,
                            mean_weight=False)                                  # nodal attention: all pairs of a dialogue
        logits = self.graph_net.packed_logits(features, g.edge_index, edge_norm, g.edge_type, gfull, self.nodal_attention)
        g.check_inputs()
        return logits, features
