"""CPU (PyTorch) restatement of the declare-lab sequence classifiers that track_mm/dgcnv2_models.py vendors:
``MatchingAttention`` ('general' / 'general2' with a mask), ``LSTMModel``, ``GRUModel`` and ``DialogRNNModel``, with the
reference's module trees and parameter names, so state_dicts load both ways with erc_b200.track_mm.dgcnv2_models.  The att2
head is the reference's loop over positions (one matching attention per position), ``_reverse_seq`` its flip / pad_sequence
loop; the DialogueRNN is oracle/dialogue_rnn_oracle.DialogueRNN.  Runs in fp32 or fp64.
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  No reference output pins these classes: parity is unpinned."""
import torch
from torch import nn
import torch.nn.functional as F
from torch.nn.utils.rnn import pad_sequence

from .dialogue_rnn_oracle import DialogueRNN


class MatchingAttention(nn.Module):
    def __init__(self, mem_dim, cand_dim, alpha_dim=None, att_type="general"):
        super().__init__()
        assert att_type in ("general", "general2"), att_type
        self.mem_dim, self.cand_dim, self.att_type = mem_dim, cand_dim, att_type
        self.transform = nn.Linear(cand_dim, mem_dim, bias=att_type == "general2")

    def forward(self, M, x, mask=None):
        if mask is None:
            mask = torch.ones(M.size(1), M.size(0), dtype=M.dtype, device=M.device)
        M_ = M.permute(1, 2, 0)                                           # [B, D, L]
        x_ = self.transform(x).unsqueeze(1)                               # [B, 1, D]
        if self.att_type == "general":
            alpha = F.softmax(torch.bmm(x_, M_), dim=2)
        else:
            mask_ = mask.unsqueeze(2).repeat(1, 1, self.mem_dim).transpose(1, 2)
            M_ = M_ * mask_
            alpha_ = torch.bmm(x_, M_) * mask.unsqueeze(1)
            alpha_ = torch.tanh(alpha_)
            alpha_ = F.softmax(alpha_, dim=2)
            alpha_masked = alpha_ * mask.unsqueeze(1)
            alpha_sum = torch.sum(alpha_masked, dim=2, keepdim=True)
            alpha = alpha_masked / alpha_sum
        attn_pool = torch.bmm(alpha, M.transpose(0, 1))[:, 0, :]
        return attn_pool, alpha


def _head(m, emotions, umask, att2):
    if att2:
        att_emotions, alpha = [], []
        for t in emotions:
            att_em, alpha_ = m.matchatt(emotions, t, mask=umask)
            att_emotions.append(att_em.unsqueeze(0))
            alpha.append(alpha_[:, 0, :])
        hidden = F.relu(m.linear(torch.cat(att_emotions, dim=0)))
    else:
        alpha = []
        hidden = F.relu(m.linear(emotions))
    hidden = m.dropout(hidden)
    return F.log_softmax(m.smax_fc(hidden), 2), alpha


class LSTMModel(nn.Module):
    def __init__(self, D_m, D_e, D_h, n_classes=7, dropout=0.5):
        super().__init__()
        self.n_classes = n_classes
        self.dropout = nn.Dropout(dropout)
        self.lstm = nn.LSTM(input_size=D_m, hidden_size=D_e, num_layers=2, bidirectional=True, dropout=dropout)
        self.matchatt = MatchingAttention(2 * D_e, 2 * D_e, att_type="general2")
        self.linear = nn.Linear(2 * D_e, D_h)
        self.smax_fc = nn.Linear(D_h, n_classes)

    def forward(self, U, qmask, umask, att2=True):
        emotions, _ = self.lstm(U)
        log_prob, alpha = _head(self, emotions, umask, att2)
        return log_prob, alpha, [], []


class GRUModel(nn.Module):
    def __init__(self, D_m, D_e, D_h, n_classes=7, dropout=0.5):
        super().__init__()
        self.n_classes = n_classes
        self.dropout = nn.Dropout(dropout)
        self.gru = nn.GRU(input_size=D_m, hidden_size=D_e, num_layers=2, bidirectional=True, dropout=dropout)
        self.matchatt = MatchingAttention(2 * D_e, 2 * D_e, att_type="general2")
        self.linear = nn.Linear(2 * D_e, D_h)
        self.smax_fc = nn.Linear(D_h, n_classes)

    def forward(self, U, qmask, umask, att2=True):
        emotions, _ = self.gru(U)
        log_prob, alpha = _head(self, emotions, umask, att2)
        return log_prob, alpha, [], []


class DialogRNNModel(nn.Module):
    def __init__(self, D_m, D_g, D_p, D_e, D_h, D_a=100, n_classes=7, listener_state=False, context_attention="simple",
                 dropout_rec=0.5, dropout=0.5):
        super().__init__()
        self.dropout = nn.Dropout(dropout)
        self.dropout_rec = nn.Dropout(dropout + 0.15)
        self.dialog_rnn_f = DialogueRNN(D_m, D_g, D_p, D_e, listener_state, context_attention, D_a, dropout_rec)
        self.dialog_rnn_r = DialogueRNN(D_m, D_g, D_p, D_e, listener_state, context_attention, D_a, dropout_rec)
        self.linear = nn.Linear(2 * D_e, 2 * D_h)
        self.smax_fc = nn.Linear(2 * D_h, n_classes)
        self.matchatt = MatchingAttention(2 * D_e, 2 * D_e, att_type="general2")

    def _reverse_seq(self, X, mask):
        X_ = X.transpose(0, 1)
        mask_sum = torch.sum(mask, 1).int()
        xfs = []
        for x, c in zip(X_, mask_sum):
            xfs.append(torch.flip(x[:c], [0]))
        return pad_sequence(xfs)

    def forward(self, U, qmask, umask, att2=True):
        emotions_f, alpha_f = self.dialog_rnn_f(U, qmask)
        emotions_f = self.dropout_rec(emotions_f)
        rev_U = self._reverse_seq(U, umask)
        rev_qmask = self._reverse_seq(qmask, umask)
        emotions_b, alpha_b = self.dialog_rnn_r(rev_U, rev_qmask)
        emotions_b = self._reverse_seq(emotions_b, umask)
        emotions_b = self.dropout_rec(emotions_b)
        emotions = torch.cat([emotions_f, emotions_b], dim=-1)
        log_prob, alpha = _head(self, emotions, umask, att2)
        return log_prob, alpha, alpha_f, alpha_b
