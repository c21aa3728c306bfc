"""Drop-in for ``MMGCNModule`` of track_mm/mmgcn.py (reference :56-122): same constructor, forward signature, return
values (logits [N,C], None) and state_dict keys (the dead ``att_model`` / ``gatedatt`` parameters included).

Kernel mapping:
  linear_a / linear_v   K2 with the seq-first padded->packed row gather fused in (simple_batch_graphify, :99-110)
  linear_l + lstm_l     K2 + K6 over ALL Lmax positions of every dialogue -- the reference runs the LSTM UNPACKED
                        over the zero padding (:113-114), so the reverse direction starts in the padding
  graph_model           K7 block adjacency + K8 x 64 (mmgcn_models.py)
  dropout_ / ReLU / smax_fc   one elementwise kernel + K2 (:116-119)
"""
import torch
from torch import nn

from .. import ops, ops_mmgcn
from ..graph import build_graph, standard_edge_dict
from .dgcn_models import birnn_forward
from .mmgcn_models import MMGCN, _fresh_seed
from .mmgcn_utils import simple_batch_graphify, lengths_graph  # noqa: F401


class _DeadParams(nn.Module):
    """Parameters the reference instantiates but never uses in forward; only their state_dict keys matter."""

    def __init__(self, spec):
        super().__init__()
        for name, shape in spec:
            mod = self
            *path, leaf = name.split(".")
            for part in path:
                if not hasattr(mod, part):
                    setattr(mod, part, nn.Module())
                mod = getattr(mod, part)
            mod.register_parameter(leaf, nn.Parameter(torch.zeros(shape)))


def _att_model_spec(d, max_seq_len):
    return [("scalar.weight", (max_seq_len, d)), ("matchatt.transform.weight", (d, d)), ("matchatt.transform.bias", (d,)),
            ("simpleatt.scalar.weight", (1, d)), ("att.weight", (2 * d,)), ("att.w_k.weight", (d, d)), ("att.w_k.bias", (d,)),
            ("att.w_q.weight", (d, d)), ("att.w_q.bias", (d,)), ("att.proj.weight", (d, d)), ("att.proj.bias", (d,))]


def _gatedatt_spec(mem, cand):
    s = []
    for k in ("l", "v", "a"):
        s += [("transform_%s.weight" % k, (cand, mem)), ("transform_%s.bias" % k, (cand,))]
    for k in ("av", "al", "vl"):
        s += [("transform_%s.weight" % k, (1, 3 * mem)), ("transform_%s.bias" % k, (1,))]
    return s


class MMGCNModule(nn.Module):
    def __init__(self, hidden_text=100, D_e=100, graph_hidden_size=200, n_speakers=2, max_seq_len=200, window_past=10,
                 window_future=10, n_classes=7, nodal_attention=True, hidden_visual=512, hidden_audio=100, modals='atv'):
        super().__init__()
        self.modals = modals
        self.linear_l = nn.Linear(hidden_text, 200)
        self.lstm_l = nn.LSTM(200, 100, 2, bidirectional=True, dropout=0.4)
        self.linear_a = nn.Linear(hidden_audio, 200)
        self.linear_v = nn.Linear(hidden_visual, 200)
        self.window_past, self.window_future = window_past, window_future
        self.att_model = _DeadParams(_att_model_spec(2 * D_e, max_seq_len))
        self.nodal_attention = nodal_attention
        self.graph_model = MMGCN(a_dim=2 * D_e, v_dim=2 * D_e, l_dim=2 * D_e, n_dim=2 * D_e, nlayers=64,
                                 nhidden=graph_hidden_size, nclass=n_classes, dropout=0.4, lamda=0.5, alpha=0.1,
                                 variant=True, return_feature=True, use_residue=True, n_speakers=n_speakers,
                                 modals=self.modals, use_speaker=True, use_modal=False)
        self.edge_type_mapping = standard_edge_dict(n_speakers)
        self.gatedatt = _DeadParams(_gatedatt_spec(2 * D_e + graph_hidden_size, graph_hidden_size))
        self.dropout_ = nn.Dropout(0.4)
        self.smax_fc = nn.Linear(400 * len(self.modals), n_classes)

    def forward(self, text_feature=None, audio_feature=None, visual_feature=None, speaker_tensor=None, text_length=None,
                graph=None, full_graph=None, **kwargs):
        """graph / full_graph (optional): lengths_graph(text_length) and lengths_graph([Lmax] * B), built once by a caller
        that runs many batches of the same lengths (train_step.MmgcnTrainStep).  With both given and text_length on the
        host, the forward copies nothing from the host and never waits for the device."""
        ref = text_feature if text_feature is not None else (audio_feature if audio_feature is not None else visual_feature)
        Lmax, B = ref.shape[0], ref.shape[1]
        dev = ref.device
        g = graph if graph is not None else lengths_graph(text_length, dev)  # the real utterances, dialogue-major
        rows_seq = ops_mmgcn.node_rows(g, Lmax, seq_first=True)              # packed node -> row of a [Lmax*B, *] tensor
        fa = fv = fl = []
        if 'a' in self.modals:
            fa = ops.linear(audio_feature.reshape(Lmax * B, -1), self.linear_a.weight, self.linear_a.bias, a_rows=rows_seq)
        if 'v' in self.modals:
            fv = ops.linear(visual_feature.reshape(Lmax * B, -1), self.linear_v.weight, self.linear_v.bias, a_rows=rows_seq)
        if 't' in self.modals:
            # every dialogue as a length-Lmax sequence (padding rows = linear_l(0) = its bias), dialogue-major
            gf = full_graph if full_graph is not None else lengths_graph(torch.full((B,), Lmax, dtype=torch.int64), dev)
            rows_full = ops_mmgcn.node_rows(gf, Lmax, seq_first=True)
            t200 = ops.linear(text_feature.reshape(Lmax * B, -1), self.linear_l.weight, self.linear_l.bias, a_rows=rows_full)
            emo = birnn_forward(self.lstm_l, t200, gf, None, self.training)  # [B*Lmax, 200]
            fl = ops.pack_rows(emo.view(B, Lmax, -1), g, seq_first=False)
        feat = self.graph_model(fa, fv, fl, text_length, speaker_tensor, graph=g)
        p = self.dropout_.p if self.training else 0.0
        feat = ops_mmgcn.relu_dropout(feat, p, _fresh_seed())
        return ops.linear(feat, self.smax_fc.weight, self.smax_fc.bias), None
