"""torch.autograd wrappers for the DAG-ERC kernels (K9 predecessor structure, K10 persistent layer kernel;
include/ercgraph.h).  PyTorch only owns buffers; no CPU / ATen fallback."""
import ctypes

import torch

from ._lib import lib, check, DagLayer
from . import ops
from .ops import _p, _stream, _rows, _ws


class DagStructure:
    """get_adj_v1 / get_s_mask (track_mm/dagerc.py:109-154) for a batch of PACKED dialogues, as index arrays."""

    __slots__ = ("graph", "lo", "cnt", "eoff", "E", "order", "Tmax", "windowp")

    def __init__(self, graph, lengths_cpu, windowp=1, e_cap=None, order=None):
        """e_cap (optional): an upper bound on the predecessor count E, such as sum_d L_d (L_d - 1) / 2 (utterance i has at
        most i predecessors); the attention-weight array is sized to it and E is not read back.  order (optional): the
        dialogues by descending length (stable), int32 on the device.  With both, nothing waits for the device or copies
        from the host."""
        self.graph, self.windowp = graph, int(windowp)
        N, dev = graph.N, graph.device
        self.lo = torch.empty(N, dtype=torch.int32, device=dev)
        self.cnt = torch.empty(N, dtype=torch.int32, device=dev)
        self.eoff = torch.empty(N, dtype=torch.int64, device=dev)
        total = torch.empty(1, dtype=torch.int64, device=dev)
        ws = _ws(lib().ercg_dag_build_workspace_bytes(N), dev)
        check(lib().ercg_dag_build(_p(graph.node_off), _p(graph.node_dlg), _p(graph.spk), N, self.windowp, _p(self.lo),
                                   _p(self.cnt), _p(self.eoff), _p(total), _p(ws), ws.numel(), _stream()), "ercg_dag_build")
        lengths_cpu = lengths_cpu.cpu().to(torch.int64)
        self.order = order if order is not None else dag_order(lengths_cpu, dev)
        self.Tmax = int(lengths_cpu.max()) if lengths_cpu.numel() else 0
        # size of the attention-weight array (the kernels index it through eoff): without e_cap, the one host sync
        self.E = int(e_cap) if e_cap is not None else int(total.item())


def dag_order(lengths_cpu, device):
    """The dialogues by descending length (stable), int32 on ``device``: DagStructure.order."""
    return torch.argsort(lengths_cpu.cpu().to(torch.int64), descending=True, stable=True).to(torch.int32).to(device)


def dag_edge_capacity(lengths_cpu):
    """sum_d L_d (L_d - 1) / 2: no DAG over these dialogues has more predecessor edges."""
    L = lengths_cpu.cpu().to(torch.int64)
    return int((L * (L - 1) // 2).sum())


def dense_masks(spk_padded, windowp=1):
    """Reference layout from padded speaker ids [B,Lmax]: (adj [B,L,L] fp32, s_mask [B,L,L] int64)."""
    spk = spk_padded.to(torch.int32).contiguous()
    B, L = spk.shape
    adj = torch.empty((B, L, L), dtype=torch.float32, device=spk.device)
    sm = torch.empty((B, L, L), dtype=torch.int64, device=spk.device)
    check(lib().ercg_dag_dense_masks(_p(spk), B, L, int(windowp), _p(adj), _p(sm), _stream()), "ercg_dag_dense_masks")
    return adj, sm


def _args(dag, D, tensors):
    g = dag.graph
    a = DagLayer()
    a.B, a.D, a.Tmax, a.reserved = g.B, D, dag.Tmax, 0
    a.node_off, a.order, a.spk, a.lo, a.eoff = _p(g.node_off), _p(dag.order), _p(g.spk), _p(dag.lo), _p(dag.eoff)
    for k, v in tensors.items():
        setattr(a, k, _p(v))
    return a


class _DagLayer(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Hin, gat_w, gat_b, Wr0, Wr1, c_wih, c_whh, c_bih, c_bhh, p_wih, p_whh, p_bih, p_bhh, dag):
        Hin, _ = _rows(Hin)
        if Hin.stride(0) != Hin.size(1):
            Hin = Hin.contiguous()
        N, D = Hin.shape
        dev = Hin.device
        wcat = torch.cat([c_wih, p_whh], 0)                       # [6D, D]: everything that multiplies H[l]_i
        bcat = torch.cat([c_bih, p_bhh], 0)
        pre = ops.gemm_nn(Hin, wcat.t().contiguous(), bcat)       # hoisted out of the recurrence
        f32 = dict(dtype=torch.float32, device=dev)
        t = dict(wk=gat_w.reshape(-1)[D:].contiguous(), Wr0=Wr0.contiguous(), Wr1=Wr1.contiguous(), Whh_c=c_whh.contiguous(),
                 bhh_c=c_bhh.contiguous(), Wih_p=p_wih.contiguous(), bih_p=p_bih.contiguous(), Hin=Hin, pre=pre,
                 H1=torch.empty((N, D), **f32), a=torch.zeros(N, **f32), S=torch.empty((N, 2 * D), **f32),
                 M=torch.empty((N, D), **f32), alpha=torch.empty(max(dag.E, 1), **f32), gc=torch.empty((N, 3 * D), **f32),
                 hnc=torch.empty((N, D), **f32), gp=torch.empty((N, 3 * D), **f32))
        args = _args(dag, D, t)
        check(lib().ercg_dag_layer_fwd(ctypes.byref(args), _stream()), "ercg_dag_layer_fwd")
        ctx.dag, ctx.names = dag, list(t)
        ctx.save_for_backward(wcat, *t.values())
        return t["H1"]

    @staticmethod
    def backward(ctx, dH1):
        dag = ctx.dag
        wcat, *vals = ctx.saved_tensors
        t = dict(zip(ctx.names, vals))
        Hin = t["Hin"]
        N, D = Hin.shape
        f32 = dict(dtype=torch.float32, device=Hin.device)
        t.update(dH1=dH1.contiguous().clone(), dpre=torch.empty((N, 6 * D), **f32), dGseq=torch.empty((N, 6 * D), **f32),
                 dM=torch.empty((N, D), **f32), dS=torch.zeros((N, 2 * D), **f32), dHdir=torch.empty((N, D), **f32),
                 ga=torch.zeros(N, **f32))
        args = _args(dag, D, t)
        check(lib().ercg_dag_layer_bwd(ctypes.byref(args), _stream()), "ercg_dag_layer_bwd")
        dpre, dG, dM = t["dpre"], t["dGseq"], t["dM"]
        dHin = ops.gemm_nn(dpre, wcat.contiguous()).add_(t["dHdir"])
        dwcat = ops.gemm_tn(dpre, Hin)                           # [6D, D]
        dbcat = ops.colsum(dpre)
        dwseq = ops.gemm_tn(dG, t["M"])                          # [6D, D]
        dbseq = ops.colsum(dG)
        dwr = ops.gemm_tn(dM, t["S"])                            # [D, 2D]
        dgat = torch.zeros((1, 2 * D), **f32)                    # w_q part and bias: exactly zero (softmax shift)
        dgat[:, D:] = ops.gemm_tn(t["ga"].view(N, 1), t["H1"])
        D3 = 3 * D
        return (dHin, dgat, torch.zeros(1, **f32), dwr[:, :D].contiguous(), dwr[:, D:].contiguous(), dwcat[:D3], dwseq[:D3], dbcat[:D3], dbseq[:D3],
                dwseq[D3:], dwcat[D3:], dbseq[D3:], dbcat[D3:], None)


def dag_layer(Hin, gat, gru_c, gru_p, dag):
    """One GNN layer of DAGERCModule.forward: H[l] [N,D] -> H[l+1] [N,D]."""
    return _DagLayer.apply(Hin, gat.linear.weight, gat.linear.bias, gat.Wr0.weight, gat.Wr1.weight, gru_c.weight_ih, gru_c.weight_hh,
                           gru_c.bias_ih, gru_c.bias_hh, gru_p.weight_ih, gru_p.weight_hh, gru_p.bias_ih, gru_p.bias_hh, dag)


# ------------------------------------------------------------------------------------------- stand-alone GAT step
class _GatStep(torch.autograd.Function):
    """(alpha [B,N], S01 [B,2D]) = attention of B queries over N context rows (ercg_dag_gat_fwd); the Wr0 / Wr1 mix is a
    dense transform on S01 applied by the caller (ops.linear), so its weight gradients come from the GEMM kernels."""

    @staticmethod
    def forward(ctx, Q, K, V, adj, s_mask, w_linear, b_linear):
        B, N, D = K.shape
        Q, K, V = Q.contiguous(), K.contiguous(), V.contiguous()
        adj = adj.to(torch.float32).contiguous()
        s_mask = s_mask.to(torch.float32).contiguous()
        w = w_linear.reshape(-1).contiguous()
        alpha = torch.empty((B, N), dtype=torch.float32, device=K.device)
        S01 = torch.empty((B, 2 * D), dtype=torch.float32, device=K.device)
        check(lib().ercg_dag_gat_fwd(_p(Q), D, _p(K), N * D, D, _p(V), N * D, D, _p(adj), _p(s_mask), N, _p(w),
                                     _p(b_linear.contiguous()), _p(alpha), _p(S01), B, N, D, _stream()), "ercg_dag_gat_fwd")
        ctx.save_for_backward(Q, K, V, s_mask, w, alpha)
        ctx.wshape = w_linear.shape
        return alpha, S01

    @staticmethod
    def backward(ctx, dalpha, dS01):
        Q, K, V, s_mask, w, alpha = ctx.saved_tensors
        B, N, D = K.shape
        dev = K.device
        dS01 = dS01.contiguous() if dS01 is not None else torch.zeros((B, 2 * D), dtype=torch.float32, device=dev)
        dalpha = dalpha.contiguous() if dalpha is not None else None
        de = torch.empty((B, N), dtype=torch.float32, device=dev)
        dQ = torch.empty((B, D), dtype=torch.float32, device=dev)
        dK = torch.empty((B, N, D), dtype=torch.float32, device=dev)
        dV = torch.empty((B, N, D), dtype=torch.float32, device=dev)
        check(lib().ercg_dag_gat_bwd(_p(V), N * D, D, _p(s_mask), N, _p(w), _p(alpha), _p(dalpha), _p(dS01), _p(de), _p(dQ),
                                     _p(dK), _p(dV), B, N, D, _stream()), "ercg_dag_gat_bwd")
        # Linear(2D,1): dw = [sum_b (sum_n de) Q_b | sum_{b,n} de K_{b,n}], db = sum de  -- transposed products through K2
        de_col = de.reshape(B * N, 1)
        ones = torch.ones((N, 1), dtype=torch.float32, device=dev)
        rs = ops.gemm_nn(de, ones)                                          # [B,1] row sums of de
        dwq = ops.gemm_tn(rs, Q)                                            # [1,D]
        dwk = ops.gemm_tn(de_col, K.reshape(B * N, D))                      # [1,D]
        dw = torch.cat([dwq, dwk], 1).reshape(ctx.wshape)
        db = ops.colsum(de_col)
        return dQ, dK, dV, None, None, dw, db


def gat_step(Q, K, V, adj, s_mask, w_linear, b_linear):
    return _GatStep.apply(Q, K, V, adj, s_mask, w_linear, b_linear)
