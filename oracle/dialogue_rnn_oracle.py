"""CPU (PyTorch) restatement of the declare-lab DialogueRNN that track_mm/dgcnv2_models.py:235-348 vendors: ``SimpleAttention``,
``MatchingAttention`` ('general'), ``DialogueRNNCell`` and ``DialogueRNN`` (listener_state=False), with the reference's module
tree and parameter names, so state_dicts load both ways with erc_b200.track_mm.dgcnv2_models.DialogueRNN.  Runs in fp32 or
fp64.  ``DialogueRNN.forward(U, qmask, masks=(mg, mq, me))`` replaces the cell's nn.Dropout by explicit [L*B, D_x] keep/scale
masks (row t*B + b), the layout of ops.dropout(torch.ones(L*B, D_x), p, seed); the party mask is applied to every party's
candidate state, as the reference's dropout is.
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  No reference output pins these classes: parity is unpinned."""
import torch
from torch import nn
import torch.nn.functional as F


class SimpleAttention(nn.Module):
    def __init__(self, input_dim):
        super().__init__()
        self.input_dim = input_dim
        self.scalar = nn.Linear(input_dim, 1, bias=False)

    def forward(self, M, x=None):
        scale = self.scalar(M)                                    # [seq, B, 1]
        alpha = F.softmax(scale, dim=0).permute(1, 2, 0)          # [B, 1, seq]
        attn_pool = torch.bmm(alpha, M.transpose(0, 1))[:, 0, :]
        return attn_pool, alpha


class MatchingAttention(nn.Module):
    def __init__(self, mem_dim, cand_dim, alpha_dim=None, att_type="general"):
        super().__init__()
        assert att_type == "general", att_type
        self.mem_dim, self.cand_dim, self.att_type = mem_dim, cand_dim, att_type
        self.transform = nn.Linear(cand_dim, mem_dim, bias=False)

    def forward(self, M, x, mask=None):
        M_ = M.permute(1, 2, 0)                                   # [B, mem_dim, seq]
        x_ = self.transform(x).unsqueeze(1)                       # [B, 1, mem_dim]
        alpha = F.softmax(torch.bmm(x_, M_), dim=2)               # [B, 1, seq]
        attn_pool = torch.bmm(alpha, M.transpose(0, 1))[:, 0, :]
        return attn_pool, alpha


class DialogueRNNCell(nn.Module):
    def __init__(self, D_m, D_g, D_p, D_e, listener_state=False, context_attention="simple", D_a=100, dropout=0.5):
        super().__init__()
        assert not listener_state
        self.D_m, self.D_g, self.D_p, self.D_e = D_m, D_g, D_p, D_e
        self.g_cell = nn.GRUCell(D_m + D_p, D_g)
        self.p_cell = nn.GRUCell(D_m + D_g, D_p)
        self.e_cell = nn.GRUCell(D_p, D_e)
        self.dropout = nn.Dropout(dropout)
        self.attention = SimpleAttention(D_g) if context_attention == "simple" else MatchingAttention(D_g, D_m, D_a, context_attention)

    @staticmethod
    def _select_parties(X, indices):
        return X[torch.arange(X.size(0), device=X.device), indices]

    def forward(self, U, qmask, g_hist, q0, e0, drop=None):
        drop = drop or (self.dropout, self.dropout, self.dropout)
        qm_idx = torch.argmax(qmask, 1)
        q0_sel = self._select_parties(q0, qm_idx)
        g_ = self.g_cell(torch.cat([U, q0_sel], dim=1),
                         torch.zeros(U.size(0), self.D_g, dtype=U.dtype, device=U.device) if g_hist.size(0) == 0 else g_hist[-1])
        g_ = drop[0](g_)
        if g_hist.size(0) == 0:
            c_ = torch.zeros(U.size(0), self.D_g, dtype=U.dtype, device=U.device)
            alpha = None
        else:
            c_, alpha = self.attention(g_hist, U)
        U_c_ = torch.cat([U, c_], dim=1).unsqueeze(1).expand(-1, qmask.size(1), -1)
        qs_ = self.p_cell(U_c_.contiguous().view(-1, self.D_m + self.D_g), q0.view(-1, self.D_p)).view(U.size(0), qmask.size(1), self.D_p)
        qs_ = drop[1](qs_)
        qmask_ = qmask.unsqueeze(2)
        q_ = q0 * (1 - qmask_) + qs_ * qmask_
        e0 = torch.zeros(qmask.size(0), self.D_e, dtype=U.dtype, device=U.device) if e0.size(0) == 0 else e0
        e_ = self.e_cell(self._select_parties(q_, qm_idx), e0)
        e_ = drop[2](e_)
        return g_, q_, e_, alpha


class DialogueRNN(nn.Module):
    def __init__(self, D_m, D_g, D_p, D_e, listener_state=False, context_attention="simple", D_a=100, dropout=0.5):
        super().__init__()
        self.D_m, self.D_g, self.D_p, self.D_e = D_m, D_g, D_p, D_e
        self.dropout = nn.Dropout(dropout)
        self.dialogue_cell = DialogueRNNCell(D_m, D_g, D_p, D_e, listener_state, context_attention, D_a, dropout)

    def forward(self, U, qmask, masks=None):
        B = U.size(1)
        g_hist = torch.zeros(0, dtype=U.dtype, device=U.device)
        q_ = torch.zeros(qmask.size(1), qmask.size(2), self.D_p, dtype=U.dtype, device=U.device)
        e_ = torch.zeros(0, dtype=U.dtype, device=U.device)
        e = e_
        alpha = []
        for t, (u_, qmask_) in enumerate(zip(U, qmask)):
            drop = None
            if masks is not None:
                mg, mq, me = (m[t * B:(t + 1) * B].to(U.dtype) for m in masks)
                drop = (lambda x: x * mg, lambda x: x * mq.unsqueeze(1), lambda x: x * me)
            g_, q_, e_, alpha_ = self.dialogue_cell(u_, qmask_, g_hist, q_, e_, drop)
            g_hist = torch.cat([g_hist, g_.unsqueeze(0)], 0)
            e = torch.cat([e, e_.unsqueeze(0)], 0)
            if alpha_ is not None:
                alpha.append(alpha_[:, 0, :])
        return e, alpha
