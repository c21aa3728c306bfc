"""torch.autograd wrappers around the C ABI (include/ercgraph.h).

Every forward/backward here is one or more calls into libercgraph.so on the current CUDA stream;
PyTorch only owns the buffers.  Nothing in this file computes on the CPU or through ATen kernels
except O(parameters) re-layouts of weights (transposes / concatenations of <= 600 KB tensors).
"""
import torch

from ._lib import lib, check, ACT_NONE, ACT_RELU, ACT_RELU_DROPOUT, ACT_MASK_POS  # noqa: F401  (ACT_* re-exported as ops.ACT_*)


def _p(t):
    return None if t is None else t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    """Raw handle of torch's current CUDA stream (the C-level getter is ~10x cheaper than building a Stream object,
    and this is called once per kernel launch)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _rows(t):
    """2-D fp32 CUDA tensor with unit inner stride -> (tensor, leading dimension)."""
    assert t.is_cuda and t.dtype == torch.float32 and t.dim() == 2, (t.device, t.dtype, t.shape)
    if t.stride(1) != 1 or (t.size(0) > 1 and t.stride(0) < t.size(1)):
        t = t.contiguous()
    return t, (t.stride(0) if t.size(0) > 1 else max(t.size(1), t.stride(0)))


# ------------------------------------------------------------------------------------------- raw calls
# Dense-transform engine: "tc" = tcgen05 3xTF32 tensor-core kernels where the operands qualify (16-byte aligned rows,
# no row gather, enough rows to fill a tile), exact-fp32 SIMT kernels otherwise; "simt" forces the SIMT kernels.
# Both meet the 1e-5 fp32 parity bound; this is a kernel choice inside one CUDA library, not a backend dispatch.
import os as _os
GEMM_ENGINE = _os.environ.get("ERCG_GEMM", "tc")
TC_MIN_ROWS = 256


def _tag_set(t, name, value):
    """Attach a by-product of the kernel that produced ``t`` (its column sums, "already masked") to the tensor object.
    The tag records the tensor's version counter: if anything writes into ``t`` afterwards (e.g. the autograd engine
    accumulating a second gradient in place) the version moves on and the tag is ignored."""
    setattr(t, name, (value, t._version))


def _tag_get(t, name):
    tag = getattr(t, name, None)
    if tag is None or tag[1] != t._version:
        return None
    return tag[0]


# Optional device word added to every dropout seed (see ercg_gemm_nn's seed_dev): a train step captured in a CUDA graph
# points this at its device step counter so that each replay draws a fresh mask.  None = host seeds only.
SEED_DEV = None


def gemm_nn(A, Bm, bias=None, act=ACT_NONE, a_rows=None, M=None, aux=None, aux_scale=1.0, drop_p=0.0, seed=0, out=None,
            want_colsum=False):
    """C = act(A[a_rows] @ Bm + bias).  ``want_colsum``: when the tensor-core kernel runs a plain product with N <= 128 it
    also reduces the column sums of C (from the tiles in shared memory) and hangs them on the result (``C._ercg_colsum``)
    for ops.colsum -- the bias gradient of the upstream layer costs no extra pass over C."""
    A, lda = _rows(A)
    Bm, ldb = _rows(Bm)
    K, N = Bm.shape
    assert A.size(1) == K, (A.shape, Bm.shape)
    if M is None:
        M = a_rows.numel() if a_rows is not None else A.size(0)
    C = out if out is not None else torch.empty((M, N), dtype=torch.float32, device=A.device)
    ldaux = 0
    if aux is not None:
        aux, ldaux = _rows(aux)
    ldc = C.stride(0) if M > 1 else N
    if (GEMM_ENGINE == "tc" and a_rows is None and M >= TC_MIN_ROWS and K > 0
            and lib().ercg_gemm_nn_tc_supported(_p(A), lda, _p(C), ldc, M, N, K)):
        ws = _ws(lib().ercg_gemm_nn_tc_workspace_bytes(N, K), A.device)
        cs = None
        if want_colsum and N <= 128 and bias is None and act == ACT_NONE and out is None:
            cs = torch.empty(N, dtype=torch.float32, device=A.device)
        check(lib().ercg_gemm_nn_tc(_p(A), lda, _p(Bm), ldb, _p(bias), _p(C), ldc, M, N, K, act, _p(aux), ldaux,
                                    float(aux_scale), float(drop_p), int(seed) & (2 ** 64 - 1), _p(SEED_DEV), _p(cs), _p(ws),
                                    ws.numel(), _stream()), "ercg_gemm_nn_tc")
        if cs is not None:
            _tag_set(C, "_ercg_colsum", cs)
        return C
    check(lib().ercg_gemm_nn(_p(A), lda, _p(a_rows), _p(Bm), ldb, _p(bias), _p(C), C.stride(0) if M > 1 else N, M, N, K,
                             act, _p(aux), ldaux, float(aux_scale), float(drop_p), int(seed) & (2 ** 64 - 1), _p(SEED_DEV),
                             _stream()), "ercg_gemm_nn")
    return C


def gemm_tn(A, Bm, a_rows=None, M=None):
    """A[M,K1]^T @ B[M,N1] -> [K1,N1]"""
    A, lda = _rows(A)
    Bm, ldb = _rows(Bm)
    if M is None:
        M = Bm.size(0)
    K1, N1 = A.size(1), Bm.size(1)
    C = torch.empty((K1, N1), dtype=torch.float32, device=A.device)
    if (GEMM_ENGINE == "tc" and a_rows is None and M >= 4 * TC_MIN_ROWS
            and lib().ercg_gemm_tn_tc_supported(_p(A), lda, _p(Bm), ldb, M, K1, N1)):
        ws = _ws(lib().ercg_gemm_tn_tc_workspace_bytes(M, K1, N1), A.device)
        check(lib().ercg_gemm_tn_tc(_p(A), lda, _p(Bm), ldb, _p(C), N1, M, K1, N1, _p(ws), ws.numel(), _stream()),
              "ercg_gemm_tn_tc")
        return C
    nbytes = lib().ercg_gemm_tn_workspace_bytes(M, K1, N1)
    ws = _ws(nbytes, A.device)
    check(lib().ercg_gemm_tn(_p(A), lda, _p(a_rows), _p(Bm), ldb, _p(C), N1, M, K1, N1, _p(ws), ws.numel(), _stream()),
          "ercg_gemm_tn")
    return C


def colsum(A):
    pre = _tag_get(A, "_ercg_colsum")            # column sums emitted by the kernel that produced A (see _Attn.backward)
    if pre is not None and pre.numel() == A.size(1):
        return pre
    A, lda = _rows(A)
    M, N = A.shape
    out = torch.empty(N, dtype=torch.float32, device=A.device)
    ws = _ws(lib().ercg_colsum_workspace_bytes(M, N), A.device)
    check(lib().ercg_colsum(_p(A), lda, M, N, _p(out), _p(ws), ws.numel(), _stream()), "ercg_colsum")
    return out


# ------------------------------------------------------------------------------------------- Linear
class _LinearAct(torch.autograd.Function):
    """C = act(A[a_rows] @ Bm + bias); Bm is [K,N] (already transposed weight)."""

    @staticmethod
    def forward(ctx, A, Bm, bias, act, a_rows, drop_p, seed):
        C = gemm_nn(A, Bm, bias, act=act, a_rows=a_rows, drop_p=drop_p, seed=seed)
        ctx.act, ctx.drop_p, ctx.has_bias = act, drop_p, bias is not None
        ctx.a_rows = a_rows
        ctx.save_for_backward(A, Bm, C if act != ACT_NONE else None)
        return C

    @staticmethod
    def backward(ctx, dC):
        A, Bm, C = ctx.saved_tensors
        dC = dC.contiguous()
        if ctx.act != ACT_NONE:
            scale = 1.0 / (1.0 - ctx.drop_p) if ctx.act == ACT_RELU_DROPOUT else 1.0
            dZ = mask_pos(dC, C, scale)
        else:
            dZ = dC
        dA = dB = dbias = None
        if ctx.needs_input_grad[0]:
            assert ctx.a_rows is None, "input gradient through a row gather is not needed by any reference path"
            dA = gemm_nn(dZ, Bm.t().contiguous(), want_colsum=True)
        if ctx.needs_input_grad[1]:
            dB = gemm_tn(A, dZ, a_rows=ctx.a_rows, M=dZ.size(0))
        if ctx.has_bias and ctx.needs_input_grad[2]:
            dbias = colsum(dZ)
        return dA, dB, dbias, None, None, None, None


def mask_pos(x, ref, scale=1.0):
    """x * (ref > 0 ? scale : 0) -- relu / relu+dropout backward.  Implemented with the GEMM epilogue
    (identity contraction is wasteful), so use the dedicated elementwise entry point instead."""
    x, ldx = _rows(x)
    ref, ldr = _rows(ref)
    out = torch.empty_like(x)
    check(lib().ercg_mask_pos(_p(x), ldx, _p(ref), ldr, float(scale), _p(out), out.stride(0), x.size(0), x.size(1), _stream()),
          "ercg_mask_pos")
    return out


class _MlpHead(torch.autograd.Function):
    """logits = Linear3(dropout(relu(Linear0(x))))  --  ``Linear -> ReLU -> Dropout -> Linear(H, C)``, the classifier of
    cogmen.py:116-122 and dgcn_models.py:158-167, as ONE autograd node.

    The hidden activation never leaves this node, so its backward can be one pass over it (ercg_cls_tail_bwd: the masked /
    dropout-scaled gradient of Linear0's pre-activation, dW3, db3 and db0 together) without any contract between two
    autograd nodes: no other consumer, hook or retain_grad can ever see -- or add to -- the intermediate gradient."""

    @staticmethod
    def forward(ctx, x, W0, b0, W3, b3, drop_p, seed):
        act = ACT_RELU_DROPOUT if drop_p > 0 else ACT_RELU
        h = gemm_nn(x, W0.t().contiguous(), b0, act=act, drop_p=drop_p, seed=seed)
        logits = gemm_nn(h, W3.t().contiguous(), b3)
        ctx.scale = 1.0 / (1.0 - drop_p) if drop_p > 0 else 1.0
        ctx.save_for_backward(x, W0, h, W3)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        x, W0, h, W3 = ctx.saved_tensors
        N, K = h.shape
        C = W3.size(0)
        dlogits = dlogits.contiguous()
        dev = h.device
        dZ = torch.empty((N, K), dtype=torch.float32, device=dev)
        dW3 = torch.empty((C, K), dtype=torch.float32, device=dev)
        db3 = torch.empty(C, dtype=torch.float32, device=dev)
        db0 = torch.empty(K, dtype=torch.float32, device=dev)
        ws = _ws(lib().ercg_cls_tail_bwd_workspace_bytes(K, C), dev)
        check(lib().ercg_cls_tail_bwd(_p(h), h.stride(0), _p(dlogits), _p(W3.contiguous()), float(ctx.scale), _p(dZ), K, _p(dW3),
                                      _p(db3), _p(db0), N, K, C, _p(ws), ws.numel(), _stream()), "ercg_cls_tail_bwd")
        dx = gemm_nn(dZ, W0.contiguous(), want_colsum=True) if ctx.needs_input_grad[0] else None
        dW0 = gemm_tn(dZ, x) if ctx.needs_input_grad[1] else None
        return dx, dW0, db0, dW3, db3, None, None


def mlp_head(x, W0, b0, W3, b3, drop_p=0.0, seed=0):
    """``Linear(W0,b0) -> ReLU -> Dropout(drop_p) -> Linear(W3,b3)`` (nn.Linear weight layout [out,in]); pass drop_p = 0 in
    eval mode.  Shapes the fused backward kernel does not cover go through two ordinary ops.linear nodes."""
    K, C = W0.size(0), W3.size(0)
    if b0 is None or b3 is None or (K & 3) or K > 128 or C > 8:
        act = ACT_RELU_DROPOUT if drop_p > 0 else ACT_RELU
        return linear(linear(x, W0, b0, act=act, drop_p=drop_p, seed=seed), W3, b3)
    return _MlpHead.apply(x, W0, b0, W3, b3, float(drop_p), int(seed))


class _LinearBf16In(torch.autograd.Function):
    """y = x @ Bm + bias with the input rows x STORED in bf16 (bf16 input-feature mode, include/ercgraph.h): tensor-core
    kernels with a bf16 streamed operand for the forward and the weight gradient; x itself gets no gradient."""

    @staticmethod
    def forward(ctx, x, Bm, bias):
        assert x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1
        M, K = x.shape
        lda = x.stride(0) if M > 1 else max(K, x.stride(0))
        if not lib().ercg_gemm_bf16a_supported(_p(x), lda, M, K):
            raise ValueError("bf16 input rows must be 16-byte aligned with a row pitch that is a multiple of 8 elements "
                             "(got pitch %d): store them with synth.to_bf16_rows / a padded pitch" % lda)
        Bm, ldb = _rows(Bm)
        N = Bm.size(1)
        C = torch.empty((M, N), dtype=torch.float32, device=x.device)
        ws = _ws(lib().ercg_gemm_nn_tc_workspace_bytes(N, K), x.device)
        check(lib().ercg_gemm_nn_tc_bf16a(_p(x), lda, _p(Bm), ldb, _p(bias), _p(C), N, M, N, K, _p(ws), ws.numel(), _stream()),
              "ercg_gemm_nn_tc_bf16a")
        ctx.save_for_backward(x)
        ctx.lda, ctx.has_bias = lda, bias is not None
        return C

    @staticmethod
    def backward(ctx, dC):
        (x,) = ctx.saved_tensors
        dC, ldb = _rows(dC.contiguous())
        M, K = x.shape
        N = dC.size(1)
        dB = dbias = None
        if ctx.needs_input_grad[1]:
            dB = torch.empty((K, N), dtype=torch.float32, device=x.device)
            ws = _ws(lib().ercg_gemm_tn_tc_workspace_bytes(M, K, N), x.device)
            check(lib().ercg_gemm_tn_tc_bf16a(_p(x), ctx.lda, _p(dC), ldb, _p(dB), N, M, K, N, _p(ws), ws.numel(), _stream()),
                  "ercg_gemm_tn_tc_bf16a")
        if ctx.has_bias and ctx.needs_input_grad[2]:
            dbias = colsum(dC)
        return None, dB, dbias


def linear(x, weight, bias=None, act=ACT_NONE, a_rows=None, drop_p=0.0, seed=0):
    """nn.Linear semantics (weight [out,in]) on 2-D row-major input.  bf16 input rows select the bf16 input-feature mode."""
    if x.dtype == torch.bfloat16:
        assert act == ACT_NONE and a_rows is None, "bf16 input rows: plain projection only"
        return _LinearBf16In.apply(x, weight.t().contiguous(), bias)
    return _LinearAct.apply(x, weight.t().contiguous(), bias, act, a_rows, drop_p, seed)


def matmul_kn(x, w_kn, bias=None, act=ACT_NONE, a_rows=None):
    """x @ w_kn (+bias) with w_kn already [K,N]."""
    return _LinearAct.apply(x, w_kn if w_kn.is_contiguous() else w_kn.contiguous(), bias, act, a_rows, 0.0, 0)


# ------------------------------------------------------------------------------------------- K3 gather
class _Gather(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Y, w, bias, graph, H, R, root_off, use_types, rel_slot):
        Y, ldy = _rows(Y)
        N = Y.size(0)
        out = torch.empty((N, H), dtype=torch.float32, device=Y.device)
        # (a CTA-tiled forward that stages all relation slots of the window in shared memory was measured SLOWER than this
        # warp-per-node kernel -- 0.59 vs 0.55 ms at 2^20 nodes: 1200-byte rows make the tile 50 KB -- and was dropped)
        check(lib().ercg_gather_fwd(_p(Y), ldy, _p(graph.rowptr), _p(graph.col), _p(graph.etype) if use_types else None,
                                    _p(rel_slot), _p(w), root_off, _p(bias), _p(out), H, N, H, _stream()), "ercg_gather_fwd")
        ctx.graph, ctx.H, ctx.R, ctx.root_off, ctx.use_types, ctx.rel_slot = graph, H, R, root_off, use_types, rel_slot
        ctx.has_bias = bias is not None
        ctx.w_grad = w is not None and w.requires_grad
        ctx.save_for_backward(Y if ctx.w_grad else None, w)
        ctx.ycols = Y.size(1)
        return out

    @staticmethod
    def backward(ctx, dout):
        Y, w = ctx.saved_tensors
        g, H, R = ctx.graph, ctx.H, ctx.R
        dout, ldo = _rows(dout)
        if (ldo & 3) or (dout.data_ptr() & 15):
            # the gradient of a column slice of a wider concatenation -- DialogueGCN's [features | graph out] at g = 2 (mod 4),
            # dgcnv2's [features | graph out] at odd hidden sizes -- has rows only 8-byte aligned; the gather kernels read
            # 16-byte chunks, so such a gradient is repacked once ([N, H], H = the graph width of 100)
            dout = dout.clone(memory_format=torch.contiguous_format)
            ldo = dout.stride(0)
        N = dout.size(0)
        dY = torch.empty((N, ctx.ycols), dtype=torch.float32, device=dout.device)
        dw = torch.empty(g.E, dtype=torch.float32, device=dout.device) if ctx.w_grad else None
        ldy = Y.stride(0) if Y is not None else 0
        win = _window(g, H) if dw is None else None
        if win is not None:          # K1 window graph, no edge-weight gradient: CTA-tiled kernel (out-neighbours [j-wp, j+wf])
            n_slots = (ctx.ycols - (H if ctx.root_off >= 0 else 0)) // H
            check(lib().ercg_gather_window_bwd(_p(dout), ldo, _p(g.t_rowptr), _p(g.t_col),
                                               _p(g.t_etype) if ctx.use_types else None, _p(g.t_eid), _p(ctx.rel_slot), _p(w),
                                               n_slots, ctx.root_off, _p(dY), ctx.ycols, N, H, win[1], win[0], _stream()),
                  "ercg_gather_window_bwd")
            dbias = colsum(dout) if ctx.has_bias else None
            return dY, dw, dbias, None, None, None, None, None, None
        check(lib().ercg_gather_bwd(_p(dout), ldo, _p(Y), ldy, _p(g.t_rowptr), _p(g.t_col),
                                    _p(g.t_etype) if ctx.use_types else None, _p(g.t_eid), _p(ctx.rel_slot), _p(w), R,
                                    ctx.root_off, _p(dY), ctx.ycols, _p(dw), N, H, _stream()), "ercg_gather_bwd")
        dbias = colsum(dout) if ctx.has_bias else None
        return dY, dw, dbias, None, None, None, None, None, None


def gather(Y, graph, H, R, w=None, bias=None, root_off=-1, use_types=True, rel_slot=None, n_slots=None):
    """out[k] = sum_e w[e] * Y[col[e], slot(e)*H:+H] (+ Y[k, root_off:+H]) (+ bias), slot(e) = etype[e], or
    rel_slot[etype[e]] when Y only holds the ``n_slots`` relation ids that occur in the graph (K1's relation census)."""
    slots = R if rel_slot is None else n_slots
    assert Y.size(1) == (slots * H + (H if root_off >= 0 else 0)), (Y.shape, R, slots, H, root_off)
    return _Gather.apply(Y, w, bias, graph, H, R, root_off, use_types, rel_slot)


# ------------------------------------------------------------------------------------------- K4 attention
def _window(graph, H):
    """(wf, wp) when ``graph`` is a K1 window graph the tiled attention kernels support, else None."""
    wp, wf = getattr(graph, "wp", None), getattr(graph, "wf", None)
    if wp is None or wf is None or getattr(graph, "perm", None) is not None:
        return None
    if wp < 0 or wf < 0 or not lib().ercg_attn_window_supported(H, wf, wp):
        return None
    return wf, wp


class _Attn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkvs, graph, H, scale):
        qkvs, ld = _rows(qkvs)
        N = qkvs.size(0)
        out = torch.empty((N, H), dtype=torch.float32, device=qkvs.device)
        alpha = torch.empty(graph.E, dtype=torch.float32, device=qkvs.device)
        b = qkvs.data_ptr()
        win = _window(graph, H)
        if win is not None:      # in-neighbours of node k: [k - wf, k + wp]
            check(lib().ercg_attn_window_fwd(b, b + 4 * H, b + 8 * H, b + 12 * H, ld, _p(graph.rowptr), _p(graph.col), scale,
                                             _p(out), H, _p(alpha), N, H, win[0], win[1], _stream()), "ercg_attn_window_fwd")
        else:
            check(lib().ercg_attn_fwd(b, b + 4 * H, b + 8 * H, b + 12 * H, ld, _p(graph.rowptr), _p(graph.col), scale,
                                      _p(out), H, _p(alpha), None, N, H, _stream()), "ercg_attn_fwd")
        ctx.graph, ctx.H, ctx.scale, ctx.win = graph, H, scale, win
        ctx.save_for_backward(qkvs, alpha)
        return out

    @staticmethod
    def backward(ctx, dout):
        qkvs, alpha = ctx.saved_tensors
        g, H, scale, win = ctx.graph, ctx.H, ctx.scale, ctx.win
        dout, ldo = _rows(dout)
        N, ld = qkvs.size(0), qkvs.stride(0)
        d = torch.empty((N, 4 * H), dtype=torch.float32, device=dout.device)
        dsig = torch.empty(g.E, dtype=torch.float32, device=dout.device)
        b, db = qkvs.data_ptr(), d.data_ptr()
        if win is not None:
            tiles = int(lib().ercg_attn_window_tiles(N))
            part = torch.empty((2, tiles, 2 * H), dtype=torch.float32, device=dout.device)   # per-CTA column sums
            check(lib().ercg_attn_window_bwd_dst(_p(dout), ldo, b + 4 * H, b + 8 * H, ld, _p(g.rowptr), _p(g.col), _p(alpha),
                                                 scale, db, db + 12 * H, 4 * H, _p(dsig), _p(part[0]), N, H, win[0], win[1],
                                                 _stream()), "ercg_attn_window_bwd_dst")
            # out-neighbours of node j: [j - wp, j + wf]
            check(lib().ercg_attn_window_bwd_src(_p(dout), ldo, b, ld, _p(g.t_rowptr), _p(g.t_col), _p(g.t_eid), _p(alpha),
                                                 _p(dsig), scale, db + 4 * H, db + 8 * H, 4 * H, _p(part[1]), N, H, win[1],
                                                 win[0], _stream()), "ercg_attn_window_bwd_src")
            # bias gradient of the fused q|k|v|skip Linear = column sums of d: finished from the per-CTA partials and handed
            # to the consumer (ops.colsum) on the tensor itself, so the 4H-wide gradient is not read a second time
            cs_dst, cs_src = colsum(part[0]), colsum(part[1])                               # (dq | ds), (dk | dv)
            _tag_set(d, "_ercg_colsum", torch.cat([cs_dst[:H], cs_src, cs_dst[H:]]))
            return d, None, None, None
        check(lib().ercg_attn_bwd_dst(_p(dout), ldo, b + 4 * H, b + 8 * H, ld, _p(g.rowptr), _p(g.col), _p(alpha), scale,
                                      db, db + 12 * H, 4 * H, _p(dsig), None, N, H, _stream()), "ercg_attn_bwd_dst")
        check(lib().ercg_attn_bwd_src(_p(dout), ldo, b, ld, _p(g.t_rowptr), _p(g.t_col), _p(g.t_eid), _p(alpha), _p(dsig),
                                      scale, db + 4 * H, db + 8 * H, 4 * H, N, H, _stream()), "ercg_attn_bwd_src")
        return d, None, None, None


def edge_attention(qkvs, graph, H, scale):
    """qkvs = [q | k | v | skip] (each H wide); TransformerConv(heads=1) message+aggregate+skip."""
    assert qkvs.size(1) == 4 * H
    return _Attn.apply(qkvs, graph, H, float(scale))


class _MatchAttn(torch.autograd.Function):
    """out_t = sum_j softmax_j(tanh(<xt_t, e_j>)) e_j over the in-edges of t (generic K4 kernels with the tanh option)."""

    @staticmethod
    def forward(ctx, xe, graph, H):
        """xe = [xt | e] ([N, 2H]): queries and keys = values side by side (one row stride)."""
        xe, ld = _rows(xe)
        N = xe.size(0)
        out = torch.empty((N, H), dtype=torch.float32, device=xe.device)
        alpha = torch.empty(graph.E, dtype=torch.float32, device=xe.device)
        dact = torch.empty(graph.E, dtype=torch.float32, device=xe.device)
        b = xe.data_ptr()
        check(lib().ercg_attn_fwd(b, b + 4 * H, b + 4 * H, None, ld, _p(graph.rowptr), _p(graph.col), 1.0, _p(out), H, _p(alpha),
                                  _p(dact), N, H, _stream()), "ercg_attn_fwd")
        ctx.graph, ctx.H = graph, H
        ctx.save_for_backward(xe, alpha, dact)
        return out

    @staticmethod
    def backward(ctx, dout):
        xe, alpha, dact = ctx.saved_tensors
        g, H = ctx.graph, ctx.H
        dout, ldo = _rows(dout)
        N, ld = xe.size(0), xe.stride(0)
        d = torch.empty((N, 3 * H), dtype=torch.float32, device=dout.device)           # [dq | dk | dv]
        dsig = torch.empty(g.E, dtype=torch.float32, device=dout.device)
        b, db = xe.data_ptr(), d.data_ptr()
        check(lib().ercg_attn_bwd_dst(_p(dout), ldo, b + 4 * H, b + 4 * H, ld, _p(g.rowptr), _p(g.col), _p(alpha), 1.0, db, None,
                                      3 * H, _p(dsig), _p(dact), N, H, _stream()), "ercg_attn_bwd_dst")
        check(lib().ercg_attn_bwd_src(_p(dout), ldo, b, ld, _p(g.t_rowptr), _p(g.t_col), _p(g.t_eid), _p(alpha), _p(dsig), 1.0,
                                      db + 4 * H, db + 8 * H, 3 * H, N, H, _stream()), "ercg_attn_bwd_src")
        return torch.cat([d[:, :H], d[:, H:2 * H] + d[:, 2 * H:]], 1), None, None      # e is both key and value


def matching_attention(xt, e, graph):
    """Nodal MatchingAttention 'general2' (dgcnv2_models.py:119-148) on packed nodes: for node t of a dialogue,
    alpha = softmax over the dialogue's nodes j of tanh(<xt_t, e_j>), out_t = sum_j alpha e_j.  ``graph`` = the fully connected
    per-dialogue graph (window -1 / -1); xt = transform(e).  (The reference's masked softmax + renormalisation over the valid
    positions of the padded dialogue is exactly the softmax over the dialogue's own nodes.)"""
    H = e.size(1)
    return _MatchAttn.apply(torch.cat([xt, e], 1), graph, H)


# ------------------------------------------------------------------------------------------- K5 EdgeAtt
class _EdgeAtt(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, u, graph):
        x, ldx = _rows(x)
        u, ldu = _rows(u)
        N, H = x.shape
        nu = torch.empty(graph.E, dtype=torch.float32, device=x.device)
        check(lib().ercg_edgeatt_fwd(_p(x), ldx, _p(u), ldu, _p(graph.t_rowptr), _p(graph.t_col), _p(graph.t_eid), _p(nu),
                                     N, H, _stream()), "ercg_edgeatt_fwd")
        ctx.graph = graph
        ctx.save_for_backward(x, u, nu)
        return nu

    @staticmethod
    def backward(ctx, dnu):
        x, u, nu = ctx.saved_tensors
        g = ctx.graph
        N, H = x.shape
        dnu = dnu.contiguous()
        dsig = torch.empty_like(nu)
        dx = torch.empty((N, H), dtype=torch.float32, device=x.device)
        du = torch.empty((N, H), dtype=torch.float32, device=x.device)
        check(lib().ercg_edgeatt_bwd_src(_p(dnu), _p(nu), _p(u), u.stride(0), _p(g.t_rowptr), _p(g.t_col), _p(g.t_eid),
                                         _p(dsig), _p(dx), H, N, H, _stream()), "ercg_edgeatt_bwd_src")
        check(lib().ercg_edgeatt_bwd_dst(_p(dsig), _p(x), x.stride(0), _p(g.rowptr), _p(g.col), _p(du), H, N, H, _stream()),
              "ercg_edgeatt_bwd_dst")
        return dx, du, None


def edge_att(x, u, graph):
    """nu[j->k] = softmax over the out-edges of j of <x_j, u_k>, in by-destination edge order."""
    return _EdgeAtt.apply(x, u, graph)


# ------------------------------------------------------------------------------------------- BN + LeakyReLU
class _BnAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, mean, var, eps, slope, use_batch_stats, count, stat_sync):
        x, ldx = _rows(x)
        N, H = x.shape
        out = torch.empty((N, H), dtype=torch.float32, device=x.device)
        check(lib().ercg_bn_act_fwd(_p(x), ldx, _p(mean), _p(var), eps, _p(gamma), _p(beta), slope, _p(out), H, N, H, _stream()),
              "ercg_bn_act_fwd")
        ctx.eps, ctx.slope, ctx.use_batch_stats, ctx.count, ctx.stat_sync = eps, slope, use_batch_stats, count, stat_sync
        ctx.save_for_backward(x, gamma, beta, mean, var)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, gamma, beta, mean, var = ctx.saved_tensors
        dout, ldo = _rows(dout)
        N, H = x.shape
        ldx = x.stride(0)
        sums = torch.empty(2 * H, dtype=torch.float32, device=x.device)
        ws = _ws(lib().ercg_bn_workspace_bytes(N, H), x.device)
        sync = ctx.stat_sync if ctx.use_batch_stats else None
        comm = getattr(getattr(sync, "__self__", None), "reduce", None)      # StatSync.grads -> its Reducer -> PeerComm
        comm = getattr(comm, "comm", None)
        if comm is not None and 2 * H <= 8 * 128:
            # reduction and exchange over peer memory in one kernel: this rank's sums (dbeta | dgamma) and the global ones
            local = sums
            sums = torch.empty(2 * H, dtype=torch.float32, device=x.device)
            check(lib().ercg_p2p_bn_act_bwd_reduce(comm.regions.data_ptr(), comm.rank, comm.world, _p(dout), ldo, _p(x), ldx, _p(mean),
                                                   _p(var), ctx.eps, _p(gamma), _p(beta), ctx.slope, _p(local), _p(sums), N, H,
                                                   _p(ws), ws.numel(), comm.max_bytes, _stream()), "ercg_p2p_bn_act_bwd_reduce")
        else:
            check(lib().ercg_bn_act_bwd_reduce(_p(dout), ldo, _p(x), ldx, _p(mean), _p(var), ctx.eps, _p(gamma), _p(beta), ctx.slope,
                                               _p(sums), N, H, _p(ws), ws.numel(), _stream()), "ercg_bn_act_bwd_reduce")
            local = sums
            if sync is not None:
                sums = sync(sums.clone())              # all-reduce(sum) of (sum dy, sum dy*xhat) across ranks
        dx = torch.empty((N, H), dtype=torch.float32, device=x.device)
        check(lib().ercg_bn_act_bwd_apply(_p(dout), ldo, _p(x), ldx, _p(mean), _p(var), ctx.eps, _p(gamma), _p(beta), ctx.slope,
                                          _p(sums), float(ctx.count), 1 if ctx.use_batch_stats else 0, _p(dx), H, N, H,
                                          _stream()), "ercg_bn_act_bwd_apply")
        return dx, local[H:], local[:H], None, None, None, None, None, None, None


def bn_stats(x):
    """(mean[H], biased var[H]) over the rows of x."""
    x, ldx = _rows(x)
    N, H = x.shape
    mean = torch.empty(H, dtype=torch.float32, device=x.device)
    var = torch.empty(H, dtype=torch.float32, device=x.device)
    ws = _ws(lib().ercg_bn_workspace_bytes(N, H), x.device)
    check(lib().ercg_bn_stats(_p(x), ldx, N, H, _p(mean), _p(var), _p(ws), ws.numel(), _stream()), "ercg_bn_stats")
    return mean, var


def bn_stats_sync(x, comm, count_global, bn=None):
    """Data-parallel BatchNorm statistics fused with their exchange (ercg_p2p_bn_stats): (mean[H], biased var[H]) over the rows
    of ALL ranks, the same on every rank; ``bn`` (an nn.BatchNorm1d in train mode) also gets its running statistics updated.
    ``comm``: p2p.PeerComm; collective -- every rank of the communicator calls it at the same point of its stream."""
    x, ldx = _rows(x)
    N, H = x.shape
    mean = torch.empty(H, dtype=torch.float32, device=x.device)
    var = torch.empty(H, dtype=torch.float32, device=x.device)
    ws = _ws(lib().ercg_bn_workspace_bytes(N, H), x.device)
    run = bn is not None and bn.track_running_stats
    check(lib().ercg_p2p_bn_stats(comm.regions.data_ptr(), comm.rank, comm.world, _p(x), ldx, N, H, float(count_global), _p(mean),
                                  _p(var), _p(bn.running_mean) if run else None, _p(bn.running_var) if run else None,
                                  _p(bn.num_batches_tracked) if run else None,
                                  (float(bn.momentum) if bn.momentum is not None else -1.0) if run else 0.0,
                                  _p(ws), ws.numel(), comm.max_bytes, _stream()), "ercg_p2p_bn_stats")
    return mean, var


def bn_running_update(bn, mean, var, count):
    """Train-mode bookkeeping of nn.BatchNorm1d (num_batches_tracked, running_mean, running_var) in ONE launch."""
    check(lib().ercg_bn_running_update(_p(mean), _p(var), _p(bn.running_mean), _p(bn.running_var), _p(bn.num_batches_tracked),
                                       float(bn.momentum) if bn.momentum is not None else -1.0, float(count),
                                       mean.numel(), _stream()), "ercg_bn_running_update")


def bn_leaky_relu(x, gamma, beta, mean, var, eps, slope, use_batch_stats, count=None, stat_sync=None):
    return _BnAct.apply(x, gamma, beta, mean, var, float(eps), float(slope), bool(use_batch_stats),
                        float(count if count is not None else x.size(0)), stat_sync)


# ------------------------------------------------------------------------------------------- cross entropy
class _CrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, class_weight, reduce_sync, denom, num_out):
        logits, ld = _rows(logits)
        N, C = logits.shape
        nd = torch.empty(2, dtype=torch.float32, device=logits.device)
        dl = torch.empty((N, C), dtype=torch.float32, device=logits.device)
        ws = _ws(lib().ercg_ce_workspace_bytes(N), logits.device)
        check(lib().ercg_ce_fwd(_p(logits), ld, _p(labels), _p(class_weight), _p(nd), _p(dl), C, N, C, _p(ws), ws.numel(),
                                _stream()), "ercg_ce_fwd")
        if num_out is not None:
            num_out.copy_(nd[:1])                      # local numerator rides along with the gradient all-reduce
        if denom is not None:
            nd[1:].fill_(float(denom))                 # host-known global normaliser (utterance count): no collective needed
        if reduce_sync is not None:
            nd = reduce_sync(nd)                       # global numerator / denominator across ranks
        ctx.save_for_backward(dl, nd)
        return nd[0] / nd[1]

    @staticmethod
    def backward(ctx, g):
        dl, nd = ctx.saved_tensors
        out = dl.clone()
        g = g.contiguous().reshape(1)
        check(lib().ercg_scale_by_ratio(_p(out), out.numel(), _p(g), nd.data_ptr() + 4, _stream()), "ercg_scale_by_ratio")
        return out, None, None, None, None, None


def cross_entropy(logits, labels, class_weight=None, reduce_sync=None, denom=None, num_out=None):
    """F.cross_entropy(logits, labels, weight=class_weight) with mean reduction.

    Data-parallel use: ``reduce_sync`` all-reduces (numerator, denominator) so every rank sees the global mean; or, with no
    collective at all, ``denom`` = the host-known GLOBAL sum of weights (the utterance count for unweighted CE) makes the
    returned value this rank's share of the global mean (gradients are then exact after the summed gradient all-reduce)
    and ``num_out`` (a 1-element device tensor, e.g. a ride-along slot of FlatAdam) receives the local numerator."""
    assert labels.dtype == torch.int64 and labels.is_cuda
    return _CrossEntropy.apply(logits, labels.contiguous(), class_weight, reduce_sync, denom, num_out)


# ------------------------------------------------------------------------------------------- pack rows
class _PackRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, padded, graph, seq_first):
        shape = padded.shape
        D = shape[-1]
        flat = padded.reshape(-1, D)
        flat, ld = _rows(flat)
        B = graph.B
        Lmax = shape[0] if seq_first else shape[1]
        out = torch.empty((graph.N, D), dtype=torch.float32, device=padded.device)
        check(lib().ercg_pack_rows(_p(flat), ld, Lmax, B, 1 if seq_first else 0, _p(graph.node_off), _p(graph.node_dlg),
                                   _p(out), D, graph.N, D, _stream()), "ercg_pack_rows")
        ctx.graph, ctx.seq_first, ctx.shape, ctx.Lmax = graph, seq_first, shape, Lmax
        return out

    @staticmethod
    def backward(ctx, dout):
        g = ctx.graph
        dout, ldp = _rows(dout)
        D = ctx.shape[-1]
        dpad = torch.zeros(ctx.shape, dtype=torch.float32, device=dout.device)
        check(lib().ercg_unpack_rows(_p(dout), ldp, _p(g.node_off), _p(g.node_dlg), _p(dpad), D, ctx.Lmax, g.B,
                                     1 if ctx.seq_first else 0, g.N, D, _stream()), "ercg_unpack_rows")
        return dpad, None, None


def pack_rows(padded, graph, seq_first=False):
    """[B,Lmax,D] (or [Lmax,B,D] when seq_first) -> packed [N,D], dialogue-major."""
    return _PackRows.apply(padded, graph, seq_first)


# ------------------------------------------------------------------------------------------- K6 LSTM
class _LstmLayer(torch.autograd.Function):
    """One bidirectional layer on packed rows: gx [N, 8*Hd] (input transform already applied) -> out [N, 2*Hd]."""

    @staticmethod
    def forward(ctx, gx, whh, graph):
        gx, ldgx = _rows(gx)
        whh = whh.contiguous()
        N, Hd = gx.size(0), whh.size(2)
        dev = gx.device
        out = torch.empty((N, 2 * Hd), dtype=torch.float32, device=dev)
        gates = torch.empty((N, 8 * Hd), dtype=torch.float32, device=dev)
        cells = torch.empty((N, 2 * Hd), dtype=torch.float32, device=dev)
        hprev = torch.empty((N, 2 * Hd), dtype=torch.float32, device=dev)
        check(lib().ercg_lstm_fwd(_p(gx), ldgx, _p(whh), _p(graph.node_off), graph.B, Hd, _p(out), 2 * Hd, _p(gates), _p(cells),
                                  _p(hprev), _stream()), "ercg_lstm_fwd")
        ctx.graph, ctx.Hd = graph, Hd
        ctx.save_for_backward(whh, gates, cells, hprev)
        return out

    @staticmethod
    def backward(ctx, dout):
        whh, gates, cells, hprev = ctx.saved_tensors
        g, Hd = ctx.graph, ctx.Hd
        dout, ldo = _rows(dout)
        N = dout.size(0)
        dgx = torch.empty((N, 8 * Hd), dtype=torch.float32, device=dout.device)
        check(lib().ercg_lstm_bwd(_p(dout), ldo, _p(gates), _p(cells), _p(whh), _p(g.node_off), g.B, Hd, _p(dgx), 8 * Hd,
                                  _stream()), "ercg_lstm_bwd")
        dwhh = None
        if ctx.needs_input_grad[1]:
            dwhh = torch.stack([gemm_tn(dgx[:, d * 4 * Hd:(d + 1) * 4 * Hd], hprev[:, d * Hd:(d + 1) * Hd]) for d in range(2)])
        return dgx, dwhh, None


def lstm_layer(gx, whh, graph):
    return _LstmLayer.apply(gx, whh, graph)


# ------------------------------------------------------------------------------------------- K6b GRU
class _GruLayer(torch.autograd.Function):
    """One bidirectional nn.GRU layer on packed rows: gx [N, 6*Hd] (= x W_ih^T + b_ih, both directions), whh [2, 3*Hd, Hd],
    bhh [2, 3*Hd] -> out [N, 2*Hd].  b_hh is applied inside the recurrence (b_hn is scaled by the reset gate)."""

    @staticmethod
    def forward(ctx, gx, whh, bhh, graph):
        gx, ldgx = _rows(gx)
        whh, bhh = whh.contiguous(), bhh.contiguous()
        N, Hd = gx.size(0), whh.size(2)
        assert gx.size(1) == 6 * Hd and whh.shape == (2, 3 * Hd, Hd) and bhh.shape == (2, 3 * Hd), (gx.shape, whh.shape, bhh.shape)
        dev = gx.device
        out = torch.empty((N, 2 * Hd), dtype=torch.float32, device=dev)
        gates = torch.empty((N, 8 * Hd), dtype=torch.float32, device=dev)
        hprev = torch.empty((N, 2 * Hd), dtype=torch.float32, device=dev)
        check(lib().ercg_gru_fwd(_p(gx), ldgx, _p(whh), _p(bhh), _p(graph.node_off), graph.B, Hd, _p(out), 2 * Hd, _p(gates),
                                 _p(hprev), _stream()), "ercg_gru_fwd")
        ctx.graph, ctx.Hd = graph, Hd
        ctx.save_for_backward(whh, gates, hprev)
        return out

    @staticmethod
    def backward(ctx, dout):
        whh, gates, hprev = ctx.saved_tensors
        g, Hd = ctx.graph, ctx.Hd
        dout, ldo = _rows(dout)
        N = dout.size(0)
        dgx = torch.empty((N, 6 * Hd), dtype=torch.float32, device=dout.device)
        dgh = torch.empty((N, 6 * Hd), dtype=torch.float32, device=dout.device)
        check(lib().ercg_gru_bwd(_p(dout), ldo, _p(gates), _p(hprev), _p(whh), _p(g.node_off), g.B, Hd, _p(dgx), 6 * Hd,
                                 _p(dgh), 6 * Hd, _stream()), "ercg_gru_bwd")
        dwhh = dbhh = None
        if ctx.needs_input_grad[1]:
            dwhh = torch.stack([gemm_tn(dgh[:, d * 3 * Hd:(d + 1) * 3 * Hd], hprev[:, d * Hd:(d + 1) * Hd]) for d in range(2)])
        if ctx.needs_input_grad[2]:
            dbhh = colsum(dgh).view(2, 3 * Hd)
        return dgx, dwhh, dbhh, None


def gru_layer(gx, whh, bhh, graph):
    return _GruLayer.apply(gx, whh, bhh, graph)


def _dropout_call(x, out, p, seed, seed_dev):
    if seed_dev is None:
        check(lib().ercg_dropout(_p(x), _p(out), x.numel(), p, seed & (2 ** 64 - 1), _stream()), "ercg_dropout")
    else:
        check(lib().ercg_dropout_dev(_p(x), _p(out), x.numel(), p, seed & (2 ** 64 - 1), _p(seed_dev), _stream()),
              "ercg_dropout_dev")


class _Dropout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p, seed):
        x = x.contiguous()
        out = torch.empty_like(x)
        ctx.p, ctx.seed, ctx.seed_dev = p, seed, SEED_DEV       # the backward reads the same device word
        _dropout_call(x, out, p, seed, ctx.seed_dev)
        return out

    @staticmethod
    def backward(ctx, dout):
        dout = dout.contiguous()
        dx = torch.empty_like(dout)
        _dropout_call(dout, dx, ctx.p, ctx.seed, ctx.seed_dev)
        return dx, None, None


def dropout(x, p, seed):
    return _Dropout.apply(x, float(p), int(seed))


def unpack_rows(packed, graph, Lmax, seq_first=False):
    """packed [N,D] -> zero-padded [B,Lmax,D] (pad_packed_sequence layout); autograd via pack_rows' kernels."""
    return _UnpackRows.apply(packed, graph, Lmax, seq_first)


class _UnpackRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, packed, graph, Lmax, seq_first):
        packed, ldp = _rows(packed)
        D = packed.size(1)
        shape = (Lmax, graph.B, D) if seq_first else (graph.B, Lmax, D)
        out = torch.zeros(shape, dtype=torch.float32, device=packed.device)
        check(lib().ercg_unpack_rows(_p(packed), ldp, _p(graph.node_off), _p(graph.node_dlg), _p(out), D, Lmax, graph.B,
                                     1 if seq_first else 0, graph.N, D, _stream()), "ercg_unpack_rows")
        ctx.graph, ctx.seq_first, ctx.Lmax, ctx.D = graph, seq_first, Lmax, D
        return out

    @staticmethod
    def backward(ctx, dout):
        g = ctx.graph
        dout = dout.contiguous()
        flat = dout.reshape(-1, ctx.D)
        dp = torch.empty((g.N, ctx.D), dtype=torch.float32, device=dout.device)
        check(lib().ercg_pack_rows(_p(flat), ctx.D, ctx.Lmax, g.B, 1 if ctx.seq_first else 0, _p(g.node_off), _p(g.node_dlg),
                                   _p(dp), ctx.D, g.N, ctx.D, _stream()), "ercg_pack_rows")
        return dp, None, None, None
