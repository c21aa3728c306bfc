"""torch.autograd wrappers for K11 (MaskedEdgeAttention 'attn1' in closed form, csrc/dgcnv2.cu), K12 (the DialogueRNN
recurrence, csrc/dialogue_rnn.cu), K13 (dense masked MatchingAttention) with the sequence reversal (csrc/seq_attn.cu), and the
log-softmax of the sequence classifiers (csrc/norm_loss.cu); include/ercgraph.h."""
import ctypes

import torch

from . import ops
from ._lib import lib, check, DialogueRnnArgs
from .ops import _p, _stream, _rows


class _MaskedEdgeAtt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, S, graph, Lmax, wp, wf):
        S, ldS = _rows(S)
        N = graph.N
        nu = torch.empty(graph.E, dtype=torch.float32, device=S.device)
        stat = torch.empty((N, 2), dtype=torch.float32, device=S.device)
        check(lib().ercg_masked_edge_att_fwd(_p(S), ldS, _p(graph.node_off), _p(graph.node_dlg), _p(graph.t_rowptr), _p(graph.t_eid),
                                             int(Lmax), int(wp), int(wf), _p(nu), _p(stat), N, _stream()), "ercg_masked_edge_att_fwd")
        ctx.graph, ctx.Lmax, ctx.wp, ctx.wf = graph, int(Lmax), int(wp), int(wf)
        ctx.save_for_backward(S, nu, stat)
        return nu

    @staticmethod
    def backward(ctx, dnu):
        S, nu, stat = ctx.saved_tensors
        g = ctx.graph
        dS = torch.zeros_like(S)                       # columns of positions beyond a dialogue's length stay zero
        check(lib().ercg_masked_edge_att_bwd(_p(S), S.stride(0), _p(g.node_off), _p(g.node_dlg), _p(g.t_rowptr), _p(g.t_eid),
                                             ctx.Lmax, ctx.wp, ctx.wf, _p(nu), _p(dnu.contiguous()), _p(stat), _p(dS), dS.stride(0),
                                             g.N, _stream()), "ercg_masked_edge_att_bwd")
        return dS, None, None, None, None


def masked_edge_att(S, graph, Lmax, wp, wf):
    """S [B*Lmax, >= Lmax'] (dialogue-major full-length rows x max_seq_len columns) -> edge weights in by-destination order."""
    Lmax = int(Lmax)
    if S.dim() != 2 or S.size(0) != graph.B * Lmax or S.size(1) < Lmax:
        raise ValueError("masked_edge_att: S must be [B * Lmax, >= Lmax] = [%d, >= %d], got %s"
                         % (graph.B * Lmax, Lmax, tuple(S.shape)))
    return _MaskedEdgeAtt.apply(S, graph, Lmax, wp, wf)


# ------------------------------------------------------------------------------------------- K12 DialogueRNN
class _DialogueRnn(torch.autograd.Function):
    """The sequential part of DialogueRNN (csrc/dialogue_rnn.cu).  pre [L*B, 3Dg+3Dp (+Dg)] = the hoisted U-dependent input
    gates of g_cell and p_cell (+ the 'general' query W_a U_t); w [1, Dg] = the 'simple' attention weight (None for
    'general').  -> (e [L*B, De], alpha packed: step t >= 1 is the [B, t] block at offset B*t*(t-1)/2)."""

    @staticmethod
    def forward(ctx, pre, w, qmask, Wgq, Whh_g, bhh_g, Wpc, Whh_p, bhh_p, Wih_e, Whh_e, bih_e, bhh_e, dims, drop_p, seeds):
        L, B, Dg, Dp, De, P = dims
        LB, dev = L * B, pre.device
        f32 = dict(dtype=torch.float32, device=dev)
        general = w is None
        xq, ldxq = (pre[:, 3 * (Dg + Dp):], pre.stride(0)) if general else (w.contiguous(), 0)
        wts = [x.contiguous() for x in (Wgq, Whh_g, bhh_g, Wpc, Whh_p, bhh_p, Wih_e, Whh_e, bih_e, bhh_e)]
        out = dict(e=torch.empty((LB, De), **f32), g=torch.empty((LB, Dg), **f32), c=torch.empty((LB, Dg), **f32),
                   qprev=torch.empty((LB, Dp), **f32), qcur=torch.empty((LB, Dp), **f32),
                   gates_g=torch.empty((LB, 4 * Dg), **f32), gates_p=torch.empty((LB, 4 * Dp), **f32),
                   gates_e=torch.empty((LB, 4 * De), **f32), alpha=torch.empty(max(B * L * (L - 1) // 2, 1), **f32),
                   qstate=torch.empty(max(B * P * Dp, 1), **f32))
        a = _drnn_args(dims, drop_p, seeds, qmask, pre, xq, ldxq, wts, out)
        check(lib().ercg_dialogue_rnn_fwd(ctypes.byref(a), _stream()), "ercg_dialogue_rnn_fwd")
        ctx.dims, ctx.drop_p, ctx.seeds, ctx.general, ctx.ldxq = dims, drop_p, seeds, general, ldxq
        ctx.names = list(out)
        ctx.save_for_backward(pre, xq, qmask, *wts, *out.values())
        ctx.mark_non_differentiable(out["alpha"])
        return out["e"], out["alpha"]

    @staticmethod
    def backward(ctx, de, _dalpha):
        L, B, Dg, Dp, De, P = ctx.dims
        pre, xq, qmask, *rest = ctx.saved_tensors
        wts, out = rest[:10], dict(zip(ctx.names, rest[10:]))
        LB, dev = L * B, pre.device
        f32 = dict(dtype=torch.float32, device=dev)
        W6 = 3 * (Dg + Dp)
        dpre = torch.empty((LB, W6 + Dg if ctx.general else W6), **f32)
        dxq = dpre[:, W6:] if ctx.general else torch.empty((LB, Dg), **f32)
        grads = dict(dgh=torch.empty((LB, 3 * Dg), **f32), dph=torch.empty((LB, 3 * Dp), **f32),
                     dei=torch.empty((LB, 3 * De), **f32), deh=torch.empty((LB, 3 * De), **f32),
                     dG=torch.empty((LB, Dg), **f32), dQ=torch.empty(max(B * P * Dp, 1), **f32),
                     dEh=torch.empty((max(B, 1), De), **f32), dc=torch.empty((max(B, 1), Dg), **f32))
        a = _drnn_args(ctx.dims, ctx.drop_p, ctx.seeds, qmask, pre, xq, ctx.ldxq, wts, out)
        de = de.contiguous()
        a.de, a.dpre, a.lddpre, a.dxq, a.lddxq = _p(de), _p(dpre), dpre.stride(0), _p(dxq), dpre.stride(0) if ctx.general else Dg
        for k, v in grads.items():
            setattr(a, k, _p(v))
        check(lib().ercg_dialogue_rnn_bwd(ctypes.byref(a), _stream()), "ercg_dialogue_rnn_bwd")
        dgh, dph, dei, deh = grads["dgh"], grads["dph"], grads["dei"], grads["deh"]
        g, e, qprev, qcur, c = out["g"], out["e"], out["qprev"], out["qcur"], out["c"]
        G3 = 3 * Dg
        return (dpre, None if ctx.general else ops.colsum(dxq).view(1, Dg), None,
                ops.gemm_tn(dpre[:, :G3], qprev), ops.gemm_tn(dgh[B:], g[:LB - B]), ops.colsum(dgh),
                ops.gemm_tn(dpre[:, G3:W6], c), ops.gemm_tn(dph, qprev), ops.colsum(dph),
                ops.gemm_tn(dei, qcur), ops.gemm_tn(deh[B:], e[:LB - B]), ops.colsum(dei), ops.colsum(deh),
                None, None, None)


def _drnn_args(dims, drop_p, seeds, qmask, pre, xq, ldxq, wts, out):
    a = DialogueRnnArgs()
    a.L, a.B, a.Dg, a.Dp, a.De, a.P = dims
    a.drop_p, a.reserved = float(drop_p), 0
    a.seed_g, a.seed_q, a.seed_e = (int(s) & (2 ** 64 - 1) for s in seeds)
    a.qmask, a.pre, a.ldpre, a.xq, a.ldxq = _p(qmask), _p(pre), pre.stride(0), _p(xq), ldxq
    for k, v in zip(("Wgq", "Whh_g", "bhh_g", "Wpc", "Whh_p", "bhh_p", "Wih_e", "Whh_e", "bih_e", "bhh_e"), wts):
        setattr(a, k, _p(v))
    for k, v in out.items():
        setattr(a, k, _p(v))
    return a


def dialogue_rnn(U, qmask, g_cell, p_cell, e_cell, att_weight, att_type, drop_p=0.0, seeds=(0, 0, 0)):
    """DialogueRNN.forward (dgcnv2_models.py:314-348, listener_state=False): U [L,B,Dm], qmask [L,B,P] (seq-first; each row
    with at most one non-zero entry, see include/ercgraph.h K12) -> (e [L,B,De], alpha: list of L-1 tensors [B, t]).
    g_cell / p_cell / e_cell are the nn.GRUCell holders, att_weight the attention's transform.weight [Dg,Dm] ('general')
    or scalar.weight [1,Dg] ('simple').  The element (t*B + b, u) of each cell's dropout keeps iff
    hash_uniform(seed_x, (t*B + b) * D_x + u) >= drop_p: ops.dropout(torch.ones(L*B, D_x), drop_p, seed_x) is that mask."""
    L, B, Dm = U.shape
    P = qmask.size(2)
    Dg, Dp, De = g_cell.weight_hh.size(1), p_cell.weight_hh.size(1), e_cell.weight_hh.size(1)
    general = att_type == "general"
    blocks = [g_cell.weight_ih[:, :Dm], p_cell.weight_ih[:, :Dm]] + ([att_weight] if general else [])
    biases = [g_cell.bias_ih, p_cell.bias_ih] + ([g_cell.bias_ih.new_zeros(Dg)] if general else [])
    pre = ops.linear(U.reshape(L * B, Dm), torch.cat(blocks, 0), torch.cat(biases, 0))
    qm = qmask.reshape(L * B, P).to(torch.float32).contiguous()
    e, alpha = _DialogueRnn.apply(pre, None if general else att_weight, qm, g_cell.weight_ih[:, Dm:], g_cell.weight_hh,
                                  g_cell.bias_hh, p_cell.weight_ih[:, Dm:], p_cell.weight_hh, p_cell.bias_hh, e_cell.weight_ih,
                                  e_cell.weight_hh, e_cell.bias_ih, e_cell.bias_hh, (L, B, Dg, Dp, De, P), float(drop_p),
                                  tuple(int(s) for s in seeds))
    return e.view(L, B, De), [alpha[B * t * (t - 1) // 2:B * t * (t + 1) // 2].view(B, t) for t in range(1, L)]


# ------------------------------------------------------------------------------------------- K13 dense MatchingAttention
MATCH_KINDS = {"general": 0, "general2": 1}


class _MatchAtt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, M, xq, mask, kind, L, B, Q):
        M, ldm = _rows(M)
        xq, ldq = _rows(xq)
        D, dev = M.size(1), M.device
        pool = torch.empty((Q * B, D), dtype=torch.float32, device=dev)
        alpha = torch.empty((Q, B, L), dtype=torch.float32, device=dev)
        score = torch.empty((Q, B, L), dtype=torch.float32, device=dev)
        check(lib().ercg_match_att_fwd(_p(M), ldm, L, B, D, Q, _p(xq), ldq, _p(mask), kind, _p(pool), D, _p(alpha), _p(score),
                                       _stream()), "ercg_match_att_fwd")
        ctx.dims = (kind, L, B, Q, ldm, ldq)
        ctx.save_for_backward(M, xq, mask, alpha, score)
        ctx.mark_non_differentiable(alpha)
        return pool, alpha

    @staticmethod
    def backward(ctx, dpool, _dalpha):
        M, xq, mask, alpha, score = ctx.saved_tensors
        kind, L, B, Q, ldm, ldq = ctx.dims
        dpool, lddp = _rows(dpool)
        D, dev = M.size(1), M.device
        w = torch.empty((Q, B, L), dtype=torch.float32, device=dev)
        dxq = torch.empty((Q * B, D), dtype=torch.float32, device=dev)
        dM = torch.empty((L * B, D), dtype=torch.float32, device=dev)
        check(lib().ercg_match_att_bwd(_p(M), ldm, L, B, D, Q, _p(xq), ldq, _p(mask), kind, _p(alpha), _p(score), _p(dpool),
                                       lddp, _p(w), _p(dxq), D, _p(dM), D, _stream()), "ercg_match_att_bwd")
        return dM, dxq, None, None, None, None, None


def match_attention(M, xq, mask, att_type):
    """MatchingAttention over B dialogues (K13): M [L, B, D] memory (seq-first), xq [Q, B, D] or [B, D] (Q = 1) transformed
    queries, mask [B, L] float or None (ignored for 'general') -> (pool [Q, B, D] (or [B, D]), alpha [Q, B, L]); alpha is not
    differentiable.  Q = L with xq = transform(M) is the att2 loop over every position."""
    L, B, D = M.shape
    squeeze = xq.dim() == 2
    xq3 = xq.unsqueeze(0) if squeeze else xq
    Q = xq3.size(0)
    kind = MATCH_KINDS[att_type]
    m = None
    if kind == 1 and mask is not None:
        m = mask.to(torch.float32).contiguous()
    pool, alpha = _MatchAtt.apply(M.reshape(L * B, D), xq3.reshape(Q * B, D), m, kind, L, B, Q)
    return (pool.view(B, D) if squeeze else pool.view(Q, B, D)), alpha


# ------------------------------------------------------------------------------------------- sequence reversal, log-softmax
class _ReverseSeq(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, counts, Lout):
        Lin, B, D = x.shape
        x2, ldx = _rows(x.reshape(Lin * B, D))
        out = torch.empty((Lout, B, D), dtype=torch.float32, device=x.device)
        check(lib().ercg_reverse_seq(_p(x2), ldx, Lin, B, D, _p(counts), _p(out), D, Lout, _stream()), "ercg_reverse_seq")
        ctx.save_for_backward(counts)
        ctx.Lin = Lin
        return out

    @staticmethod
    def backward(ctx, dout):
        (counts,) = ctx.saved_tensors
        Lout, B, D = dout.shape
        dout = dout.contiguous()
        dx = torch.empty((ctx.Lin, B, D), dtype=torch.float32, device=dout.device)
        check(lib().ercg_reverse_seq(_p(dout), D, Lout, B, D, _p(counts), _p(dx), D, ctx.Lin, _stream()), "ercg_reverse_seq")
        return dx, None, None


def reverse_seq(x, counts, Lout):
    """x [L, B, D] -> [Lout, B, D]: the first counts[b] rows of dialogue b in reverse order, zero rows after them
    (pad_sequence of flip(x[:c_b]) when Lout = max c_b).  counts: int32 CUDA tensor [B]."""
    return _ReverseSeq.apply(x.to(torch.float32), counts, int(Lout))


class _LogSoftmax(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x, ldx = _rows(x)
        R, C = x.shape
        y = torch.empty((R, C), dtype=torch.float32, device=x.device)
        check(lib().ercg_log_softmax_fwd(_p(x), ldx, _p(y), C, R, C, _stream()), "ercg_log_softmax_fwd")
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy, lddy = _rows(dy)
        R, C = y.shape
        dx = torch.empty((R, C), dtype=torch.float32, device=y.device)
        check(lib().ercg_log_softmax_bwd(_p(y), C, _p(dy), lddy, _p(dx), C, R, C, _stream()), "ercg_log_softmax_bwd")
        return dx


def log_softmax(x):
    """F.log_softmax(x, dim=-1) for a 2-D fp32 CUDA tensor [rows, C]."""
    return _LogSoftmax.apply(x)
