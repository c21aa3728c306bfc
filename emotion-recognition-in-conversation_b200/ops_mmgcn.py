"""torch.autograd wrappers for the MMGCN kernels (K7 block adjacency, K8 GCNII layers; include/ercgraph.h).

The reference builds a dense [3N,3N] adjacency (track_mm/mmgcn_models.py:582-646) and multiplies it 64 times
(:373-394).  Here the adjacency is a flat fp32 tensor holding only the non-zero blocks (``BlockLayout``) and every
product with it is a block kernel.  As in ops.py, PyTorch only owns buffers; there is no CPU / ATen fallback.
"""
import math

import torch

from ._lib import lib, check
from . import ops
from .ops import _p, _stream, _rows


class BlockLayout:
    """Where the non-zeros of the reference's dense adjacency live (see csrc/mmgcn.cu)."""

    __slots__ = ("graph", "B", "N", "M", "SB", "blk_off", "nflat")

    def __init__(self, graph, M, lengths_cpu=None):
        self.graph, self.B, self.N, self.M = graph, graph.B, graph.N, int(M)
        self.blk_off = torch.empty(self.B + 1, dtype=torch.int64, device=graph.device)
        check(lib().ercg_mmgcn_block_offsets(_p(graph.node_off), self.B, _p(self.blk_off), _stream()),
              "ercg_mmgcn_block_offsets")
        if lengths_cpu is not None and not lengths_cpu.is_cuda:
            self.SB = int((lengths_cpu.to(torch.int64) ** 2).sum())
        else:
            self.SB = int(self.blk_off[-1].item())
        self.nflat = self.M * self.SB + self.M * (self.M - 1) * self.N

    def args(self):
        g = self.graph
        return _p(g.node_off), _p(g.node_dlg), _p(self.blk_off), self.N, self.SB, self.M

    def dense(self, flat):
        """Expand a flat block array into the reference's dense [M*N, M*N] matrix (tests / debugging only)."""
        M, N = self.M, self.N
        out = torch.zeros((M * N, M * N), dtype=flat.dtype, device=flat.device)
        off = self.graph.node_off.tolist()
        boff = self.blk_off.tolist()
        for m in range(M):
            for d in range(self.B):
                s, L = off[d], off[d + 1] - off[d]
                out[m * N + s:m * N + s + L, m * N + s:m * N + s + L] = \
                    flat[m * self.SB + boff[d]: m * self.SB + boff[d] + L * L].view(L, L)
            for n in range(M):
                if n == m:
                    continue
                slot = n if n < m else n - 1
                base = M * self.SB + (m * (M - 1) + slot) * N
                idx = torch.arange(N, device=flat.device)
                out[m * N + idx, n * N + idx] = flat[base:base + N]
        return out


# ------------------------------------------------------------------------------------------- K7 adjacency
class _BigAdj(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, layout):
        feats, ldx = _rows(feats)
        rows, D = feats.shape
        assert rows == layout.M * layout.N, (feats.shape, layout.M, layout.N)
        dev = feats.device
        xhat = torch.empty((rows, D), dtype=torch.float32, device=dev)
        rinv = torch.empty(rows, dtype=torch.float32, device=dev)
        dinv = torch.empty(rows, dtype=torch.float32, device=dev)
        cs = torch.empty(layout.nflat, dtype=torch.float32, device=dev)
        ahat = torch.empty(layout.nflat, dtype=torch.float32, device=dev)
        a = layout.args()
        check(lib().ercg_mmgcn_adj_fwd(_p(feats), ldx, a[0], a[1], a[2], a[3], a[4], a[5], D, _p(xhat), D, _p(rinv), _p(cs),
                                       _p(ahat), _p(dinv), _stream()), "ercg_mmgcn_adj_fwd")
        ctx.layout, ctx.D = layout, D
        ctx.save_for_backward(xhat, rinv, cs, dinv)
        return ahat

    @staticmethod
    def backward(ctx, G):
        xhat, rinv, cs, dinv = ctx.saved_tensors
        layout, D = ctx.layout, ctx.D
        G = G.contiguous()
        rows = xhat.size(0)
        ddeg = torch.empty(rows, dtype=torch.float32, device=G.device)
        dx = torch.empty((rows, D), dtype=torch.float32, device=G.device)
        a = layout.args()
        check(lib().ercg_mmgcn_adj_bwd(_p(G), _p(cs), _p(dinv), _p(xhat), D, _p(rinv), a[0], a[1], a[2], a[3], a[4], a[5], D,
                                       _p(ddeg), _p(dx), D, _stream()), "ercg_mmgcn_adj_bwd")
        return dx, None


def big_adj(feats, layout):
    """create_big_adj: feats [M*N, D] (modality-major) -> flat normalised block adjacency (differentiable)."""
    return _BigAdj.apply(feats, layout)


# ------------------------------------------------------------------------------------------- raw block products
def spmm(ahat, h, layout, transpose=False, out=None, acc_src=None, acc_dst=None):
    h, ldh = _rows(h)
    rows, H = h.shape
    if out is None:
        out = torch.empty((rows, H), dtype=torch.float32, device=h.device)
    lds = ldd = 0
    if acc_dst is not None:
        lds, ldd = acc_src.stride(0), acc_dst.stride(0)
    a = layout.args()
    check(lib().ercg_mmgcn_spmm(_p(ahat), 1 if transpose else 0, _p(h), ldh, _p(out), out.stride(0), a[0], a[1], a[2], a[3],
                                a[4], a[5], H, _p(acc_src), lds, _p(acc_dst), ldd, _stream()), "ercg_mmgcn_spmm")
    return out


def sddmm(dhi, h, layout, G, accumulate):
    h, ldh = _rows(h)
    a = layout.args()
    check(lib().ercg_mmgcn_sddmm(_p(dhi), dhi.stride(0), _p(h), ldh, a[0], a[1], a[2], a[3], a[4], a[5], h.size(1), _p(G),
                                 1 if accumulate else 0, _stream()), "ercg_mmgcn_sddmm")
    return G


def _layer_fwd(hi, h0, W, theta, alpha, relu, p, seed, seed_dev=None):
    M, H = hi.shape
    out = torch.empty((M, H), dtype=torch.float32, device=hi.device)
    args = (_p(hi), hi.stride(0), _p(h0), h0.stride(0), _p(W), W.stride(0), _p(out), H, M, H, float(theta), float(alpha),
            1 if relu else 0, float(p), int(seed) & (2 ** 64 - 1))
    if seed_dev is None:
        check(lib().ercg_gcnii_layer_fwd(*args, _stream()), "ercg_gcnii_layer_fwd")
    else:
        check(lib().ercg_gcnii_layer_fwd_dev(*args, _p(seed_dev), _stream()), "ercg_gcnii_layer_fwd_dev")
    return out


# Seeds of the dropout sites of the GCNII stack (the input dropout, h0's dropout, the 64 layers' output dropouts).  With
# host seeds only, site k draws from seed + k, as before.  With a device word (ops.SEED_DEV: a step counter that grows by
# 1 per step) site k at step s would then draw the mask site k + 1 drew at step s - 1, so the sites are spaced 2^32 apart.
SITE_STRIDE = 1 << 32


def site_seed(seed, k, seed_dev):
    return seed + k * (1 if seed_dev is None else SITE_STRIDE)


def _layer_bwd_input(dZ, W, theta, alpha):
    M, H = dZ.shape
    Wt = W.t().contiguous()                                    # [H, 2H], O(parameters) re-layout
    dS = torch.empty((M, 2 * H), dtype=torch.float32, device=dZ.device)
    check(lib().ercg_gcnii_layer_bwd_input(_p(dZ), dZ.stride(0), _p(Wt), 2 * H, _p(dS), 2 * H, M, H, float(theta),
                                           float(alpha), _stream()), "ercg_gcnii_layer_bwd_input")
    return dS


def _layer_wgrad(hi, h0, dZ, theta):
    return torch.cat([ops.gemm_tn(hi, dZ), ops.gemm_tn(h0, dZ)], 0).mul_(theta)      # [2H, H], O(parameters)


# ------------------------------------------------------------------------------------------- K8 one layer
class _GcniiLayer(torch.autograd.Function):
    """GraphConvolution.forward (variant=True, residual=False), optionally with the caller's ReLU fused."""

    @staticmethod
    def forward(ctx, h, ahat, h0, W, layout, theta, alpha, relu):
        h, _ = _rows(h)
        h0, _ = _rows(h0)
        hi = spmm(ahat, h, layout)
        out = _layer_fwd(hi, h0, W.contiguous(), theta, alpha, relu, 0.0, 0)
        ctx.layout, ctx.theta, ctx.alpha, ctx.relu = layout, theta, alpha, relu
        ctx.save_for_backward(h, ahat, h0, W, hi, out if relu else None)
        return out

    @staticmethod
    def backward(ctx, dout):
        h, ahat, h0, W, hi, out = ctx.saved_tensors
        layout, theta, alpha = ctx.layout, ctx.theta, ctx.alpha
        H = h.size(1)
        dout, _ = _rows(dout)
        dZ = ops.mask_pos(dout, out, 1.0) if ctx.relu else dout
        dW = _layer_wgrad(hi, h0, dZ, theta)
        dS = _layer_bwd_input(dZ, W.contiguous(), theta, alpha)
        G = torch.empty(layout.nflat, dtype=torch.float32, device=h.device)
        sddmm(dS[:, :H], h, layout, G, accumulate=False)
        dh = spmm(ahat, dS[:, :H], layout, transpose=True)
        return dh, G, dS[:, H:].contiguous(), dW, None, None, None, None


def gcnii_layer(h, ahat, h0, W, layout, theta, alpha, relu=False):
    return _GcniiLayer.apply(h, ahat, h0, W, layout, float(theta), float(alpha), bool(relu))


# ------------------------------------------------------------------------------------------- K8 the 64-layer stack
class _GcniiStack(torch.autograd.Function):
    """GCNII_lyc.forward (mmgcn_models.py:373-394) from the (already dropped-out) input x to the last layer's
    (dropped-out) output: h0 = relu(fc(x)); h_l = dropout(relu(GraphConvolution_l(h_{l-1}, adj, h0))).

    One Function for the whole stack so that the gradient w.r.t. the adjacency (64 block outer products) and w.r.t.
    h0 (64 contributions) are accumulated inside the kernels instead of by 128 autograd adds."""

    @staticmethod
    def forward(ctx, x, ahat, fc_w, fc_b, layout, lamda, alpha, p, seed, *Ws):
        x, _ = _rows(x)
        seed_dev = ops.SEED_DEV                                  # the backward reads the same device word
        h0 = ops.gemm_nn(x, fc_w.t().contiguous(), fc_b, act=ops.ACT_RELU)
        h = h0
        if p > 0:
            h = torch.empty_like(h0)
            ops._dropout_call(h0, h, p, seed, seed_dev)
        saved = [h]
        his = []
        for l, W in enumerate(Ws, start=1):
            theta = math.log(lamda / l + 1)
            hi = spmm(ahat, h, layout)
            h = _layer_fwd(hi, h0, W.contiguous(), theta, alpha, True, p, site_seed(seed, l, seed_dev), seed_dev)
            his.append(hi)
            saved.append(h)
        ctx.layout, ctx.lamda, ctx.alpha, ctx.p, ctx.seed, ctx.nl = layout, lamda, alpha, p, seed, len(Ws)
        ctx.seed_dev = seed_dev
        ctx.save_for_backward(x, ahat, fc_w, h0, *Ws, *his, *saved)
        return h

    @staticmethod
    def backward(ctx, dh):
        nl, layout, alpha, p = ctx.nl, ctx.layout, ctx.alpha, ctx.p
        t = ctx.saved_tensors
        x, ahat, fc_w, h0 = t[:4]
        Ws, his, hs = t[4:4 + nl], t[4 + nl:4 + 2 * nl], t[4 + 2 * nl:]
        H = h0.size(1)
        dev = h0.device
        scale = 1.0 / (1.0 - p)
        dh, _ = _rows(dh)
        G = torch.empty(layout.nflat, dtype=torch.float32, device=dev)
        dh0 = torch.zeros_like(h0)
        dWs = [None] * nl
        for l in range(nl, 0, -1):
            theta = math.log(ctx.lamda / l + 1)
            dZ = ops.mask_pos(dh, hs[l], scale)                  # relu + this layer's output dropout
            dWs[l - 1] = _layer_wgrad(his[l - 1], h0, dZ, theta)
            dS = _layer_bwd_input(dZ, Ws[l - 1].contiguous(), theta, alpha)
            sddmm(dS[:, :H], hs[l - 1], layout, G, accumulate=(l != nl))
            dh = spmm(ahat, dS[:, :H], layout, transpose=True, acc_src=dS[:, H:], acc_dst=dh0)
        if nl == 0:
            G.zero_()
        if p > 0:                                                # hs[0] = dropout(h0): same counter-hash mask
            d0 = torch.empty_like(dh)
            ops._dropout_call(dh, d0, p, ctx.seed, ctx.seed_dev)
            dh = d0
        dh0.add_(dh)
        dpre = ops.mask_pos(dh0, h0, 1.0)
        dfc_w = ops.gemm_tn(dpre, x)                             # [out, in]
        dfc_b = ops.colsum(dpre)
        dx = ops.gemm_nn(dpre, fc_w.contiguous()) if ctx.needs_input_grad[0] else None
        return (dx, G, dfc_w, dfc_b, None, None, None, None, None) + tuple(dWs)


def gcnii_stack(x, ahat, fc_w, fc_b, weights, layout, lamda, alpha, p, seed):
    return _GcniiStack.apply(x, ahat, fc_w, fc_b, layout, float(lamda), float(alpha), float(p), int(seed), *weights)


# ------------------------------------------------------------------------------------------- helpers
def node_rows(graph, Lmax, seq_first):
    rows = torch.empty(graph.N, dtype=torch.int32, device=graph.device)
    check(lib().ercg_node_rows(_p(graph.node_off), _p(graph.node_dlg), graph.N, graph.B, int(Lmax), 1 if seq_first else 0,
                               _p(rows), _stream()), "ercg_node_rows")
    return rows


class _SpeakerEmbedAdd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, qmask, rows, emb):
        x, ldx = _rows(x)
        N, D = x.shape
        n_spk = qmask.size(-1)
        q = qmask.reshape(-1, n_spk).contiguous().float()
        emb_c = emb.contiguous()
        out = torch.empty((N, D), dtype=torch.float32, device=x.device)
        ids = torch.empty(N, dtype=torch.int32, device=x.device)
        onehot = torch.empty((N, n_spk), dtype=torch.float32, device=x.device)
        check(lib().ercg_speaker_embed_add(_p(x), ldx, _p(q), n_spk, _p(rows), _p(emb_c), D, _p(out), D, _p(ids), _p(onehot),
                                           N, D, _stream()), "ercg_speaker_embed_add")
        ctx.save_for_backward(onehot)
        ctx.mark_non_differentiable(ids)
        return out, ids

    @staticmethod
    def backward(ctx, dout, _dids):
        (onehot,) = ctx.saved_tensors
        dout = dout.contiguous()
        return dout, None, None, ops.gemm_tn(onehot, dout)


def speaker_embed_add(x, qmask, rows, emb):
    """x[i] + emb[argmax(qmask[rows[i]])]  (mmgcn_models.py:540-545) -> (out, speaker ids)."""
    return _SpeakerEmbedAdd.apply(x, qmask, rows, emb)


class _ReluDropout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p, seed):
        x = x.contiguous()
        out = torch.empty_like(x)
        if ops.SEED_DEV is None:
            check(lib().ercg_relu_dropout(_p(x), _p(out), x.numel(), p, seed & (2 ** 64 - 1), _stream()), "ercg_relu_dropout")
        else:
            check(lib().ercg_relu_dropout_dev(_p(x), _p(out), x.numel(), p, seed & (2 ** 64 - 1), _p(ops.SEED_DEV), _stream()),
                  "ercg_relu_dropout_dev")
        ctx.p = p
        ctx.save_for_backward(out)
        return out

    @staticmethod
    def backward(ctx, dout):
        (out,) = ctx.saved_tensors
        shape = out.shape
        d = ops.mask_pos(dout.contiguous().reshape(-1, shape[-1]), out.reshape(-1, shape[-1]), 1.0 / (1.0 - ctx.p))
        return d.reshape(shape), None, None


def relu_dropout(x, p, seed):
    return _ReluDropout.apply(x, float(p), int(seed))
