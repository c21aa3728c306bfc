"""Drop-in for ``DGCNModule`` of track_mm/dgcnv2.py (reference :54-181; declare-lab DialogueGCN): same constructor, forward
signature ``(input_tensor [L,B,D], speaker_tensor one-hot [L,B,n], attention_mask [B,L], text_length)`` (seq-first, one-hot
speakers: dgcnv2.py:44-45), return values (logits [N,C] of the real utterances, features [N,2*hidden]) and state_dict keys.
Base models: 'LSTM' (the default, dgcnv2.py:31: unpacked 2-layer BiLSTM over the padded batch), 'GRU' (the same with a 2-layer
BiGRU, K6b) and 'None' (a Linear).  'DialogRNN' is not rebuilt: no reference output pins the DialogueRNN classes.
``forward_packed`` takes the batch-first padded rows instead (the entry of train_step.Dgcnv2TrainStep): same values, with the
base's layer-0 input transform on the tensor-core GEMMs."""
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
        gf, gfull = length_graphs(lens, Lmax, dev)
        rows_full = ops_mmgcn.node_rows(gf, Lmax, seq_first=True)
        emo = self._base(input_tensor.reshape(Lmax * B, D), gf, rows_full)    # unpacked: runs over the padding, dgcnv2.py:151
        logits, features = self._graph_head(emo, g, gfull, B, Lmax)
        g.check_inputs()
        return logits, features

    def forward_packed(self, x_rows, speaker_ids, lengths, lmax, graphs=None):
        """Resident-data entry point: x_rows [B * lmax, D] = the batch-first padded input [B, lmax, D] viewed as rows (zero
        padding, 16-byte aligned rows, as synth.padded_batch lays it out), speaker_ids [N] the packed speaker ids of the real
        utterances, lengths [B] the dialogue lengths, lmax the padded length (>= the longest dialogue, <= max_seq_len; it may
        exceed this batch's longest dialogue, so that every shard of a batch split over GPUs pads to the global length).
        Same values as ``forward`` on the seq-first [lmax, B, D] batch.  The base's layer-0 input transform is a plain
        product on the rows (no row gather): it runs on the tensor-core kernels, and the rows get no gradient.
        graphs: optional prebuilt (g, gf, gfull) -- the window graph (build_graph over speaker_ids, mean_weight=False), the
        full-length graph and the fully connected per-dialogue graph (``length_graphs(lengths, lmax)``).  K1's input flags
        are NOT read here (that would wait for the host): call ``g.check_inputs()`` after the step, as the train step's
        ``check()`` does."""
        lmax = int(lmax)
        if not 1 <= lmax <= self.att_model.max_seq_len:
            raise ValueError("forward_packed: lmax must lie in [1, %d] (max_seq_len), got %d" % (self.att_model.max_seq_len, lmax))
        dev = x_rows.device
        if graphs is None:
            lens = torch.as_tensor(lengths).to(torch.int64).cpu()
            if int(lens.max()) > lmax:
                raise ValueError("forward_packed: a dialogue of length %d exceeds lmax %d" % (int(lens.max()), lmax))
            g = build_graph(lens, speaker_ids, self.window_past, self.window_future, self.n_speakers, device=dev,
                            mean_weight=False)
            gf, gfull = length_graphs(lens, lmax, dev)
        else:
            g, gf, gfull = graphs
        if x_rows.dim() != 2 or x_rows.size(0) != gf.B * lmax:
            raise ValueError("forward_packed: x_rows must be [B * lmax, D] = [%d, D], got %s" % (gf.B * lmax, tuple(x_rows.shape)))
        emo = self._base(x_rows, gf, None)
        return self._graph_head(emo, g, gfull, gf.B, lmax)

    def _base(self, x2d, gf, a_rows):
        """The base model over every dialogue of ``gf`` at full length -> dialogue-major rows [B * Lmax, 2 * hidden]."""
        if self.base_model in ("LSTM", "GRU"):
            rnn = self.lstm if self.base_model == "LSTM" else self.gru
            return birnn_forward(rnn, x2d, gf, a_rows, self.training)
        return ops.linear(x2d, self.base_linear.weight, self.base_linear.bias, a_rows=a_rows)

    def _graph_head(self, emo, g, gfull, B, Lmax):
        """Everything after the base: K11 edge weights over all Lmax positions, the real utterances' rows, GraphNetwork."""
        edge_norm = self.att_model.edge_weights(emo, g, Lmax)                  # [E], canonical by-destination order
        features = ops.pack_rows(emo.view(B, Lmax, -1), g)                     # the real utterances [N, 2*hidden]
        g.attach()
        logits = self.graph_net.packed_logits(features, g.edge_index, edge_norm, g.edge_type, gfull, self.nodal_attention)
        return logits, features


def length_graphs(lengths, lmax, device):
    """The two graphs of a batch that depend on its lengths alone: (gf, gfull) = every dialogue as a full-length ``lmax``
    sequence (the base runs over the padding) and the fully connected graph of each dialogue (nodal attention).
    lengths: CPU int64 [B]."""
    gf = lengths_graph(torch.full((lengths.numel(),), int(lmax), dtype=torch.int64), device)
    gfull = build_graph(lengths, torch.zeros(int(lengths.sum()), dtype=torch.int64, device=device), -1, -1, 1, device=device,
                        reference_layout=False, mean_weight=False)
    return gf, gfull
