"""Drop-in for track_mm/dgcnv2_models.py (SURVEY.md 8f-2): the DialogueGCN part (reference :517-773) -- ``MatchingAttention``
('general2'), ``MaskedEdgeAttention`` ('attn1'), ``edge_perms``, ``batch_graphify`` and ``GraphNetwork`` --, the DialogueRNN
recurrence (:235-348) -- ``SimpleAttention``, ``DialogueRNNCell``, ``DialogueRNN`` -- and the declare-lab sequence classifiers
``LSTMModel``, ``GRUModel`` and ``DialogRNNModel`` with ``MatchingAttention.forward(M, x, mask)``, with the reference's
constructor arguments, signatures and state_dict keys.

Kernel mapping
  MaskedEdgeAttention.scalar (Linear 2D -> 110)   K2 over the dialogue-major full-length rows
  softmax over the sequence axis, mask, renorm    K11 (csrc/dgcnv2.cu): closed form per source node, edge order = packed CSR
  edge_perms / batch_graphify                     K1
  GraphNetwork.conv1 / conv2                      vendored RGCNConv(edge_norm, 30 bases) / GraphConv: K2 + K3
  nodal MatchingAttention over each dialogue      transform = K2, then the generic K4 kernels with the tanh option on the
                                                  fully connected per-dialogue graph (K1 with window -1 / -1)
  linear -> ReLU -> dropout -> smax_fc            ops.mlp_head
  DialogueRNN (all L steps, all dialogues)        the U columns of g_cell / p_cell and the 'general' transform: one K2 GEMM
                                                  over all L*B rows; the three GRUCells, the attention over the global-state
                                                  history and the party-state update: K12 (csrc/dialogue_rnn.cu), one
                                                  persistent kernel forward and one backward
  MatchingAttention.forward(M, x, mask)           transform = K2, then K13 (csrc/seq_attn.cu): 'general' / masked 'general2'
                                                  attention of one query per dialogue, forward and backward
  LSTMModel / GRUModel                            2-layer BiLSTM / BiGRU over the unpacked batch (birnn_forward: K2 + K6 / K6b)
  DialogRNNModel                                  DialogueRNN (K12) forward and over the reversed dialogues (_reverse_seq:
                                                  ercg_reverse_seq, its backward the same permutation); dropout_rec =
                                                  ops.dropout
  att2 head of the three (the per-position loop)  K13 with Q = L: all positions of all dialogues in one launch
  linear -> ReLU -> dropout -> smax_fc            ops.mlp_head, then ercg_log_softmax_fwd / bwd
The unused attention variants of the file (Attention 'mlp', MatchingAttention 'dot' / 'concat') are parameter holders or
NotImplementedError: DGCNModule with 'attn1' and nodal 'general2' never executes them.  DialogueRNN runs stand-alone and
inside DialogRNNModel; DGCNModule("DialogRNN") still raises NotImplementedError.
"""
import torch
from torch import nn

from .. import ops, ops_dgcnv2
from ..graph import build_graph, speakers_from_edge_dict
from ..models.rgcn import RGCNConv
from ..pyg_nn import GraphConv
from .cogmen_utils import edge_perms  # noqa: F401  (same function in the reference, dgcnv2_models.py:612-635)
from .dgcn_models import _fresh_seed, birnn_forward
from .mmgcn_utils import lengths_graph


class MatchingAttention(nn.Module):
    def __init__(self, mem_dim, cand_dim, alpha_dim=None, att_type="general"):
        super().__init__()
        if att_type not in ("general", "general2"):
            raise NotImplementedError("att_type %r: only 'general' (DialogueRNN's context attention) and 'general2' (the "
                                      "DialogueGCN path, dgcnv2_models.py:531,761) are instantiated" % (att_type,))
        self.mem_dim, self.cand_dim, self.att_type = mem_dim, cand_dim, att_type
        self.transform = nn.Linear(cand_dim, mem_dim, bias=att_type == "general2")

    def pooled(self, emotions, graph_full):
        """All nodes at once: out_t = sum_j softmax_j(tanh(<transform(e_t), e_j>)) e_j over node t's own dialogue."""
        xt = ops.linear(emotions, self.transform.weight, self.transform.bias)
        return ops.matching_attention(xt, emotions, graph_full)

    def forward(self, M, x, mask=None):
        """Reference signature: M [L,B,mem_dim] (seq-first), x [B,cand_dim], mask [B,L] float or None -> (pool [B,mem_dim],
        alpha [B,1,L]); one query per dialogue on K13.  'general' ignores the mask; 'general2' with mask None uses all ones,
        and a dialogue whose mask is all zero gets NaN, as in the reference."""
        dev = self.transform.weight.device
        if M.dim() != 3 or x.dim() != 2 or M.size(2) != self.mem_dim or x.size(1) != self.cand_dim or x.size(0) != M.size(1):
            raise ValueError("M [L, B, %d] and x [B, %d] expected, got %s and %s" % (self.mem_dim, self.cand_dim, tuple(M.shape),
                                                                                 tuple(x.shape)))
        _check_mask(mask, M.size(1), M.size(0), dev)
        _check_cuda_f32(dev, M=M, x=x)
        L, B, _ = M.shape
        pool, alpha = ops_dgcnv2.match_attention(M, ops.linear(x, self.transform.weight, self.transform.bias), mask, self.att_type)
        return pool, alpha.view(B, 1, L)

    def all_positions(self, M, mask=None):
        """The att2 loop of the sequence classifiers in one K13 launch: query t of dialogue b is transform(M[t, b]) against all
        of M[:, b] -> (pool [L,B,mem_dim] = the stacked forward(M, M[t], mask)[0], alpha [L,B,L]: alpha[t] = forward(...)[1][:, 0])."""
        L, B, D = M.shape
        xq = ops.linear(M.reshape(L * B, D), self.transform.weight, self.transform.bias).view(L, B, D)
        return ops_dgcnv2.match_attention(M, xq, mask, self.att_type)


class SimpleAttention(nn.Module):
    """Parameter holder of the 'simple' context attention: alpha = softmax over the history of
    scalar(M); DialogueRNN runs it inside K12."""

    def __init__(self, input_dim):
        super().__init__()
        self.input_dim = input_dim
        self.scalar = nn.Linear(input_dim, 1, bias=False)

    def forward(self, M, x=None):
        raise NotImplementedError("SimpleAttention.forward: DialogueRNN evaluates the attention of every step inside K12")


class DialogueRNNCell(nn.Module):
    """One step of DialogueRNN (dgcnv2_models.py:235-313).  Holds the reference's parameters; the recurrence over all steps
    runs in DialogueRNN.forward (K12)."""

    def __init__(self, D_m, D_g, D_p, D_e, listener_state=False, context_attention="simple", D_a=100, dropout=0.5):
        super().__init__()
        if listener_state:
            raise NotImplementedError("DialogueRNNCell(listener_state=True) is not implemented")
        if context_attention not in ("simple", "general"):
            raise NotImplementedError("context_attention %r: only 'simple' and 'general' are implemented" % (context_attention,))
        self.D_m, self.D_g, self.D_p, self.D_e = D_m, D_g, D_p, D_e
        self.listener_state, self.context_attention = listener_state, context_attention
        self.g_cell = nn.GRUCell(D_m + D_p, D_g)
        self.p_cell = nn.GRUCell(D_m + D_g, D_p)
        self.e_cell = nn.GRUCell(D_p, D_e)
        self.dropout = nn.Dropout(dropout)
        if context_attention == "simple":
            self.attention = SimpleAttention(D_g)
        else:
            self.attention = MatchingAttention(D_g, D_m, D_a, context_attention)

    def forward(self, U, qmask, g_hist, q0, e0):
        raise NotImplementedError("DialogueRNNCell.forward (one step): use DialogueRNN.forward(U, qmask) -- all steps of all "
                                  "dialogues in one K12 launch per direction")


class DialogueRNN(nn.Module):
    """dgcnv2_models.py:316-348.  forward(U [L,B,D_m], qmask [L,B,P]) -> (e [L,B,D_e], alpha: L-1 tensors [B, t]).
    Every dialogue runs all L steps (no lengths, as in the reference).  The party cell is evaluated for the speaker
    (first argmax of the qmask row) only, which equals the reference's blend over all parties when each qmask row has at
    most one non-zero entry (one-hot or all-zero rows)."""

    def __init__(self, D_m, D_g, D_p, D_e, listener_state=False, context_attention="simple", D_a=100, dropout=0.5):
        super().__init__()
        self.D_m, self.D_g, self.D_p, self.D_e = D_m, D_g, D_p, D_e
        self.dropout = nn.Dropout(dropout)          # owned but never applied by the reference's forward
        self.dialogue_cell = DialogueRNNCell(D_m, D_g, D_p, D_e, listener_state, context_attention, D_a, dropout)

    def forward(self, U, qmask):
        cell = self.dialogue_cell
        if U.dim() != 3 or qmask.dim() != 3:
            raise ValueError("U [L, B, D_m] and qmask [L, B, P] must be 3-D, got %s and %s" % (tuple(U.shape), tuple(qmask.shape)))
        if U.size(2) != self.D_m or qmask.shape[:2] != U.shape[:2]:
            raise ValueError("shape mismatch: U %s (D_m = %d), qmask %s" % (tuple(U.shape), self.D_m, tuple(qmask.shape)))
        dev = cell.g_cell.weight_hh.device
        if U.device != dev or qmask.device != dev or dev.type != "cuda":
            raise ValueError("U (%s), qmask (%s) and the parameters (%s) must be on the same CUDA device" % (U.device, qmask.device, dev))
        if U.dtype != torch.float32:
            raise ValueError("U must be float32, got %s" % U.dtype)
        p = cell.dropout.p if self.training else 0.0
        seeds = (_fresh_seed(), _fresh_seed(), _fresh_seed()) if p > 0 else (0, 0, 0)
        att = cell.attention.scalar.weight if cell.context_attention == "simple" else cell.attention.transform.weight
        return ops_dgcnv2.dialogue_rnn(U, qmask, cell.g_cell, cell.p_cell, cell.e_cell, att, cell.context_attention, p, seeds)


class MaskedEdgeAttention(nn.Module):
    def __init__(self, input_dim, max_seq_len):
        super().__init__()
        self.input_dim, self.max_seq_len = input_dim, max_seq_len
        self.scalar = nn.Linear(input_dim, max_seq_len, bias=False)
        self.matchatt = MatchingAttention(input_dim, input_dim, att_type="general2")       # dead in 'attn1' (keys kept)
        self.simpleatt = nn.Module()
        self.simpleatt.scalar = nn.Linear(input_dim, 1, bias=False)
        self.att = nn.Module()                                                             # Attention(score_function='mlp'): dead
        self.att.weight = nn.Parameter(torch.zeros(2 * input_dim))
        self.att.w_k, self.att.w_q, self.att.proj = (nn.Linear(input_dim, input_dim) for _ in range(3))
        self.window = (10, 10)                     # set by DGCNModule / batch_graphify (window_past, window_future)

    def edge_weights(self, m_rows, graph, Lmax):
        """m_rows [B*Lmax, 2D]: dialogue-major, all Lmax positions of every dialogue (padding included -- the reference's
        softmax runs over them, dgcnv2_models.py:544) -> edge_norm [E] in the packed by-destination order."""
        if Lmax > self.max_seq_len:
            raise IndexError("dialogue longer than max_seq_len=%d (the reference indexes a [B,%d,L] mask, dgcnv2_models.py:546-557)"
                             % (self.max_seq_len, self.max_seq_len))
        S = ops.linear(m_rows, self.scalar.weight)
        return ops_dgcnv2.masked_edge_att(S, graph, Lmax, self.window[0], self.window[1])

    def forward(self, M, lengths, edge_ind):
        """Reference signature: M [L,B,2D] -> dense scores [B, max_seq_len, L] (non-zero on the window edges only).  The edges
        are the window graph of ``self.window`` (what batch_graphify passes in ``edge_ind``)."""
        L, B, D = M.shape
        dev = M.device
        lens = torch.as_tensor(lengths).to(torch.int64).cpu()
        g = build_graph(lens, torch.zeros((B, L), dtype=torch.int64, device=dev), self.window[0], self.window[1], 1, device=dev,
                        mean_weight=False)
        nu = self.edge_weights(M.transpose(0, 1).reshape(B * L, D), g, L)
        scores = torch.zeros((B, self.max_seq_len, L), dtype=torch.float32, device=dev)
        ei = g.edge_index
        off = g.node_off.long()
        b = g.node_dlg.long()[ei[0]]
        scores[b, ei[0] - off[b], ei[1] - off[b]] = nu          # API-compat scatter (ATen); the module path never builds this
        return scores


def batch_graphify(features, qmask, lengths, window_past, window_future, edge_type_mapping, att_model):
    """Reference signature (dgcnv2_models.py:638-690): features [L,B,D] seq-first, qmask one-hot [L,B,n] ->
    (node_features [N,D], edge_index [2,E], edge_norm [E], edge_type [E], edge_index_lengths list).
    Edges come back in canonical (dialogue, destination, source) order."""
    n_speakers = speakers_from_edge_dict(edge_type_mapping)
    L, B, D = features.shape
    dev = features.device
    ids = qmask.argmax(-1).t().contiguous()
    g = build_graph(torch.as_tensor(lengths), ids, window_past, window_future, n_speakers, device=dev, mean_weight=False)
    att_model.window = (window_past, window_future)
    rows = features.transpose(0, 1).reshape(B * L, D)
    edge_norm = att_model.edge_weights(rows, g, L)
    node_features = ops.pack_rows(features, g, seq_first=True)
    g.attach()
    return node_features, g.edge_index, edge_norm, g.edge_type, [int(v) for v in g.edge_index_lengths.tolist()]


class GraphNetwork(nn.Module):
    def __init__(self, num_features, num_classes, num_relations, max_seq_len, hidden_size=64, dropout=0.5):
        super().__init__()
        self.conv1 = RGCNConv(num_features, hidden_size, num_relations, num_bases=30)
        self.conv2 = GraphConv(hidden_size, hidden_size)
        self.matchatt = MatchingAttention(num_features + hidden_size, num_features + hidden_size, att_type="general2")
        self.linear = nn.Linear(num_features + hidden_size, hidden_size)
        self.dropout = nn.Dropout(dropout)
        self.smax_fc = nn.Linear(hidden_size, num_classes)

    def packed_logits(self, x, edge_index, edge_norm, edge_type, graph_full, nodal_attn=True):
        """-> logits [N, C] on the packed nodes."""
        out = self.conv1(x, edge_index, edge_type, edge_norm=edge_norm)
        out = self.conv2(out, edge_index)
        emotions = torch.cat([x, out], dim=-1)
        if nodal_attn:
            emotions = self.matchatt.pooled(emotions, graph_full)
        p = self.dropout.p if self.training else 0.0
        return ops.mlp_head(emotions, self.linear.weight, self.linear.bias, self.smax_fc.weight, self.smax_fc.bias, p,
                            _fresh_seed() if p > 0 else 0)

    def forward(self, x, edge_index, edge_norm, edge_type, seq_lengths, umask, nodal_attn, avec):
        """Reference signature -> logits [max_len, B, C] (seq-first, zero at the padded positions; the reference leaves the
        classifier's output for zero rows there and DGCNModule drops them through the attention mask)."""
        if avec:
            raise NotImplementedError("avec regression head is not used by DGCNModule (dgcnv2.py:63)")
        lens = torch.as_tensor(seq_lengths).to(torch.int64).cpu()
        gfull = build_graph(lens, torch.zeros(int(lens.sum()), dtype=torch.int64, device=x.device), -1, -1, 1, device=x.device,
                            reference_layout=False, mean_weight=False)
        logits = self.packed_logits(x, edge_index, edge_norm, edge_type, gfull, nodal_attn)
        return ops.unpack_rows(logits, gfull, int(lens.max()), seq_first=True)


# ------------------------------------------------------------------------------------------- sequence classifiers
def _check_cuda_f32(dev, **tensors):
    for name, t in tensors.items():
        if t.device != dev or dev.type != "cuda":
            raise ValueError("%s (%s) and the parameters (%s) must be on the same CUDA device" % (name, t.device, dev))
        if t.dtype != torch.float32:
            raise ValueError("%s must be float32, got %s" % (name, t.dtype))


def _check_mask(mask, B, L, dev):
    if mask is None:
        return
    if mask.dim() != 2 or tuple(mask.shape) != (B, L):
        raise ValueError("mask must be [B, L] = [%d, %d], got %s" % (B, L, tuple(mask.shape)))
    if mask.device != dev:
        raise ValueError("mask (%s) and the parameters (%s) must be on the same CUDA device" % (mask.device, dev))


def _check_seq_inputs(m, U, qmask, umask, D_m):
    """U [L,B,D_m] float32, qmask [L,B,P], umask [B,L] on the parameters' CUDA device."""
    dev = m.linear.weight.device
    if U.dim() != 3 or U.size(2) != D_m:
        raise ValueError("U must be [L, B, %d], got %s" % (D_m, tuple(U.shape)))
    if qmask.dim() != 3 or qmask.shape[:2] != U.shape[:2]:
        raise ValueError("qmask must be [L, B, P] with U's L, B = %s, got %s" % (tuple(U.shape[:2]), tuple(qmask.shape)))
    if umask is None:
        raise ValueError("umask [B, L] is required")
    _check_mask(umask, U.size(1), U.size(0), dev)
    _check_cuda_f32(dev, U=U)
    if qmask.device != dev:
        raise ValueError("qmask (%s) and the parameters (%s) must be on the same CUDA device" % (qmask.device, dev))


def _classify(m, emotions, umask, att2):
    """The shared head of LSTMModel / GRUModel / DialogRNNModel: att2 = masked 'general2' MatchingAttention of every
    position over its dialogue (K13), then relu(linear) -> dropout -> smax_fc (ops.mlp_head) -> log_softmax over the classes.
    -> (log_prob [L,B,C], alpha: L tensors [B,L] with att2, else [])."""
    L, B, D = emotions.shape
    alpha = []
    if att2:
        emotions, a = m.matchatt.all_positions(emotions, umask)
        alpha = list(a.unbind(0))
    p = m.dropout.p if m.training else 0.0
    logits = ops.mlp_head(emotions.reshape(L * B, D), m.linear.weight, m.linear.bias, m.smax_fc.weight, m.smax_fc.bias, p,
                          _fresh_seed() if p > 0 else 0)
    return ops_dgcnv2.log_softmax(logits).view(L, B, -1), alpha


class LSTMModel(nn.Module):
    """declare-lab LSTMModel: a 2-layer bidirectional nn.LSTM over the unpacked batch (every dialogue runs all L steps;
    hoisted input GEMM + K6 through birnn_forward), then the head of ``_classify``.  forward(U [L,B,D_m], qmask [L,B,P],
    umask [B,L], att2=True) -> (log_prob [L,B,n_classes], alpha, [], []); padded positions get outputs too."""
    rnn_type = nn.LSTM

    def __init__(self, D_m, D_e, D_h, n_classes=7, dropout=0.5):
        super().__init__()
        self.n_classes = n_classes
        self.dropout = nn.Dropout(dropout)
        setattr(self, self._rnn_name(), self.rnn_type(input_size=D_m, hidden_size=D_e, num_layers=2, bidirectional=True,
                                                      dropout=dropout))
        self.matchatt = MatchingAttention(2 * D_e, 2 * D_e, att_type="general2")
        self.linear = nn.Linear(2 * D_e, D_h)
        self.smax_fc = nn.Linear(D_h, n_classes)

    @classmethod
    def _rnn_name(cls):
        return "lstm" if cls.rnn_type is nn.LSTM else "gru"

    def forward(self, U, qmask, umask, att2=True):
        rnn = getattr(self, self._rnn_name())
        _check_seq_inputs(self, U, qmask, umask, rnn.input_size)
        L, B, D_m = U.shape
        dev = U.device
        gf = lengths_graph(torch.full((B,), L, dtype=torch.int64), dev)
        h = birnn_forward(rnn, ops.pack_rows(U, gf, seq_first=True), gf, None, self.training)     # dialogue-major rows
        emotions = ops.unpack_rows(h, gf, L, seq_first=True)
        log_prob, alpha = _classify(self, emotions, umask, att2)
        return log_prob, alpha, [], []


class GRUModel(LSTMModel):
    """declare-lab GRUModel: LSTMModel with ``gru = nn.GRU(...)`` (K6b)."""
    rnn_type = nn.GRU


class DialogRNNModel(nn.Module):
    """declare-lab DialogRNNModel: a forward and a reversed DialogueRNN (K12 each), ``dropout_rec`` (p = dropout + 0.15, the
    declare-lab value) on both, their concatenation, then the head of ``_classify``.  forward(U [L,B,D_m], qmask [L,B,P],
    umask [B,L], att2=True) -> (log_prob [L,B,n_classes], alpha or [], alpha_f, alpha_b).  The reversed direction reads each
    dialogue's first int(sum(umask[b])) rows in reverse order (``_reverse_seq``); the longest such count must equal L (the
    reference's concatenation fails otherwise: ValueError here).
    K12's limits hold: D_g, D_p, D_e <= 256, P <= 16, at most one non-zero entry per qmask row, listener_state=False,
    context_attention 'simple' or 'general'."""

    def __init__(self, D_m, D_g, D_p, D_e, D_h, D_a=100, n_classes=7, listener_state=False, context_attention="simple",
                 dropout_rec=0.5, dropout=0.5):
        super().__init__()
        self.D_m, self.D_g, self.D_p, self.D_e, self.D_h, self.n_classes = D_m, D_g, D_p, D_e, D_h, n_classes
        self.dropout = nn.Dropout(dropout)
        self.dropout_rec = nn.Dropout(dropout + 0.15)
        self.dialog_rnn_f = DialogueRNN(D_m, D_g, D_p, D_e, listener_state, context_attention, D_a, dropout_rec)
        self.dialog_rnn_r = DialogueRNN(D_m, D_g, D_p, D_e, listener_state, context_attention, D_a, dropout_rec)
        self.linear = nn.Linear(2 * D_e, 2 * D_h)
        self.smax_fc = nn.Linear(2 * D_h, n_classes)
        self.matchatt = MatchingAttention(2 * D_e, 2 * D_e, att_type="general2")

    @staticmethod
    def _counts(mask):
        return mask.sum(1).int()                      # the reference's torch.sum(mask, 1).int()

    def _reverse_seq(self, X, mask, counts=None):
        """pad_sequence([flip(X[:c_b, b]) for each b]), c_b = int(sum(mask[b])): [max c_b, B, D]."""
        counts = self._counts(mask) if counts is None else counts
        Lout = int(counts.max()) if counts.numel() else 0
        return ops_dgcnv2.reverse_seq(X, counts, max(Lout, 0))

    def _drop_rec(self, x):
        p = self.dropout_rec.p if self.training else 0.0
        return ops.dropout(x, p, _fresh_seed()) if p > 0 else x

    def forward(self, U, qmask, umask, att2=True):
        _check_seq_inputs(self, U, qmask, umask, self.D_m)
        L, B, _ = U.shape
        counts = self._counts(umask)
        maxc = int(counts.max()) if B else L
        if maxc != L:
            raise ValueError("the longest dialogue in umask has %d positions, U has L = %d: the forward and reversed "
                             "directions cannot be concatenated" % (maxc, L))
        emotions_f, alpha_f = self.dialog_rnn_f(U, qmask)
        emotions_f = self._drop_rec(emotions_f)
        rev_U = self._reverse_seq(U, umask, counts)
        rev_qmask = self._reverse_seq(qmask, umask, counts)
        emotions_b, alpha_b = self.dialog_rnn_r(rev_U, rev_qmask)
        emotions_b = self._drop_rec(self._reverse_seq(emotions_b, umask, counts))
        emotions = torch.cat([emotions_f, emotions_b], dim=-1)
        log_prob, alpha = _classify(self, emotions, umask, att2)
        return log_prob, alpha, alpha_f, alpha_b
