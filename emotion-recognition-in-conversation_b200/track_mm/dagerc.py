"""Drop-in for ``DAGERCModule`` of track_mm/dagerc.py (reference :73-198): same constructor, forward signature, return
values (logits [B,Lmax,C], None) and state_dict keys (dead ``fcs`` / ``attentive_node_features`` included).

Kernel mapping:
  get_adj_v1 / get_s_mask   K9: closed-form predecessor ranges, integer kernel (the reference: python O(B L^2))
  fc1 + ReLU                K2 epilogue
  4 x (GAT + 2 GRUCell per utterance)   K2 (hoisted input transforms) + K10 persistent layer kernel
  out_mlp                   K2 with fused ReLU / dropout epilogues

``compute_padding=True`` (default) reproduces the reference exactly: every dialogue is run for all Lmax positions
(padded rows are zero features with speaker 0, dagerc.py:157-165), so the returned [B,Lmax,C] logits match at padded
positions too.  ``compute_padding=False`` runs only the real utterances (the DAG is causal, so real positions are
unaffected) and returns zeros at padded positions, which the loss masks anyway (dagerc.py:223-226).
"""
import torch
from torch import nn

from .. import ops, ops_dagerc
from ..graph import build_graph
from .dagerc_models import GAT_dialoggcn_v1, attentive_node_features


def _fresh_seed():
    return int(torch.empty((), dtype=torch.int64).random_().item()) & (2 ** 62 - 1)


def _speaker_ids(speakers, device=None):
    """[B,L,n] one-hot (tensor or nested lists, as the reference passes them) or [B,L] ids -> int64 ids [B,L]."""
    s = speakers if torch.is_tensor(speakers) else torch.tensor(speakers)
    if device is not None:
        s = s.to(device)
    return s.argmax(-1) if s.dim() == 3 else s.long()


def speaker_count(speakers):
    """The speaker count the DAG-ERC graph is built with: the one-hot width, or 2 for [B,L] ids."""
    return max(int(speakers.size(-1)) if speakers.dim() == 3 else 2, 1)


class DAGERCModule(nn.Module):
    def __init__(self, emb_dim=100, dropout=0.2, n_classes=7, gnn_layers=4, compute_padding=True):
        super().__init__()
        self.rel_attn = True
        self.nodal_att_type = None
        self.dropout = nn.Dropout(dropout)
        hidden_dim = 300
        self.gnn_layers = gnn_layers
        self.gather = nn.ModuleList([GAT_dialoggcn_v1(hidden_dim) for _ in range(gnn_layers)])
        self.grus_c = nn.ModuleList([nn.GRUCell(hidden_dim, hidden_dim) for _ in range(gnn_layers)])
        self.grus_p = nn.ModuleList([nn.GRUCell(hidden_dim, hidden_dim) for _ in range(gnn_layers)])
        self.fcs = nn.ModuleList([nn.Linear(hidden_dim * 2, hidden_dim) for _ in range(gnn_layers)])   # dead (:178-179)
        self.fc1 = nn.Linear(emb_dim, hidden_dim)
        self.windowp = 1
        in_dim = hidden_dim * (gnn_layers + 1) + emb_dim
        self.out_mlp = nn.Sequential(nn.Linear(in_dim, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, hidden_dim), nn.ReLU(),
                                     nn.Dropout(dropout), nn.Linear(hidden_dim, n_classes))
        self.attentive_node_features = attentive_node_features(in_dim)
        self.compute_padding = compute_padding

    # ---- reference-layout helpers (dense); the fused path does not use them
    def get_adj_v1(self, speakers, max_dialog_len):
        ids = _speaker_ids(speakers, self.fc1.weight.device)[:, :max_dialog_len]
        return ops_dagerc.dense_masks(ids, self.windowp)[0]

    def get_s_mask(self, speakers, max_dialog_len):
        ids = _speaker_ids(speakers, self.fc1.weight.device)[:, :max_dialog_len]
        sm = ops_dagerc.dense_masks(ids, self.windowp)[1]
        return sm, torch.nn.functional.one_hot(sm, 2).float()

    def graph_lengths(self, text_length, Lmax):
        """CPU int64 dialogue lengths the graph is built over: every dialogue padded to Lmax when compute_padding."""
        if self.compute_padding:
            return torch.full((text_length.numel(),), int(Lmax), dtype=torch.int64)
        return text_length.cpu().to(torch.int64)

    def forward(self, input_tensor, text_length, speaker_tensor, graph=None, dag=None, **kwargs):
        """graph / dag (optional): the K1 graph over graph_lengths() with the speaker ids, and its DagStructure, built by a
        caller that keeps the batch's sizes on the host (train_step.DagercTrainStep).  With both given, the forward copies
        nothing from the host and never waits for the device."""
        B, Lmax, emb = input_tensor.shape
        dev = input_tensor.device
        if graph is None or dag is None:
            lengths = self.graph_lengths(text_length, Lmax)
        if graph is None:
            graph = build_graph(lengths, _speaker_ids(speaker_tensor, dev), 0, 0, speaker_count(speaker_tensor), device=dev,
                                reference_layout=False, mean_weight=False)
        g = graph
        if dag is None:
            dag = ops_dagerc.DagStructure(g, lengths, self.windowp)
        flat = input_tensor.reshape(B * Lmax, emb)
        a_rows = None if self.compute_padding else g.pad_row
        H0 = ops.linear(flat, self.fc1.weight, self.fc1.bias, act=ops.ACT_RELU, a_rows=a_rows)
        x = flat if self.compute_padding else ops.pack_rows(input_tensor, g)
        H = [H0]
        for l in range(self.gnn_layers):
            H.append(ops_dagerc.dag_layer(H[l], self.gather[l], self.grus_c[l], self.grus_p[l], dag))
        H.append(x)
        feat = self.attentive_node_features(torch.cat(H, dim=1), text_length, self.nodal_att_type)
        l0, l2, drop, l5 = self.out_mlp[0], self.out_mlp[2], self.out_mlp[4], self.out_mlp[5]
        h = ops.linear(feat, l0.weight, l0.bias, act=ops.ACT_RELU)
        if self.training and drop.p > 0:
            h = ops.linear(h, l2.weight, l2.bias, act=ops.ACT_RELU_DROPOUT, drop_p=drop.p, seed=_fresh_seed())
        else:
            h = ops.linear(h, l2.weight, l2.bias, act=ops.ACT_RELU)
        logits = ops.linear(h, l5.weight, l5.bias)
        if self.compute_padding:
            return logits.view(B, Lmax, -1), None
        return ops.unpack_rows(logits, g, Lmax), None
