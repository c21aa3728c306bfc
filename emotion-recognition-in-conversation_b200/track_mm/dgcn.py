"""Drop-in for ``DGCNModule`` of track_mm/dgcn.py (reference :53-93): same constructor, forward signature,
return values (logits [N,C], graph_out [N,100]) and state_dict keys.  The node features stay PACKED from the
BiLSTM to the classifier (the reference pads after the LSTM and re-packs in batch_graphify)."""
import torch
from torch import nn

from .. import ops
from ..graph import build_graph, standard_edge_dict
from .dgcn_models import SeqContext, Classifier, GCN, EdgeAtt, batch_graphify  # noqa: F401

# class weights of the 6-way IEMOCAP setting, dgcn.py:109-110
LOSS_WEIGHTS = [1 / 0.086747, 1 / 0.144406, 1 / 0.227883, 1 / 0.160585, 1 / 0.127711, 1 / 0.252668]


class DGCNModule(nn.Module):
    def __init__(self, n_speakers, input_size=100, hidden_size=200, context=[10, 10], dropout=0.4, n_classes=4):
        super().__init__()
        h1_dim = h2_dim = hc_dim = 100
        self.wp, self.wf = context
        self.rnn = SeqContext(input_size, hidden_size, dropout)
        self.edge_att = EdgeAtt(hidden_size, self.wp, self.wf)
        self.gcn = GCN(hidden_size, h1_dim, h2_dim, n_speakers=n_speakers)
        self.clf = Classifier(hidden_size + h2_dim, hc_dim, n_classes, dropout=dropout)
        self.n_speakers = n_speakers
        self.edge_type_to_idx = standard_edge_dict(n_speakers)

    def forward(self, input_tensor, speaker_tensor, text_length, **kwargs):
        B, Lmax, D = input_tensor.shape
        g = build_graph(text_length, speaker_tensor, self.wp, self.wf, self.n_speakers, device=input_tensor.device,
                        mean_weight=False)
        features = self.rnn.packed_forward(input_tensor.reshape(B * Lmax, D), g, a_rows=g.pad_row)
        edge_norm = self.edge_att.edge_weights(features, g)
        g.attach()
        graph_out = self.gcn(features, g.edge_index, edge_norm, g.edge_type)
        logits = self.clf(torch.cat([features, graph_out], dim=-1), text_length)
        g.check_inputs()          # K1's input-error flags (length > padded width, speaker id out of range) -> ValueError
        return logits, graph_out

    def forward_packed(self, x_packed, speaker_packed, text_length, graph=None):
        """Resident-data entry point: utterance rows already packed [N, hidden_all] (16-byte aligned rows, as
        collate.DeviceCollate / synth.packed_batch lay them out), packed speakers [N].  Same values as ``forward``.
        The BiLSTM's layer-0 input transform is a plain product on the packed rows (no row gather), so it runs on the
        tensor-core kernels; the rows get no gradient.  K1's input flags are NOT read here (that would wait for the
        host): call ``graph.check_inputs()`` after the step, as the train step's ``check()`` does."""
        g = graph if graph is not None else build_graph(text_length, speaker_packed, self.wp, self.wf, self.n_speakers,
                                                        device=x_packed.device, mean_weight=False)
        features = self.rnn.packed_forward(x_packed, g)
        edge_norm = self.edge_att.edge_weights(features, g)
        g.attach()
        graph_out = self.gcn(features, g.edge_index, edge_norm, g.edge_type)
        logits = self.clf(torch.cat([features, graph_out], dim=-1), text_length)
        return logits, graph_out
