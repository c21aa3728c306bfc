"""K6c, the cluster-resident LSTM / GRU recurrence (csrc/rnn_cluster.cu) that ercg_lstm_* / ercg_gru_* run for hidden sizes
101..384 per direction: one layer, SeqContext, the DialogueGCN DGCNModule and the dgcnv2 DGCNModule at those sizes, against
torch.nn.LSTM / nn.GRU and the oracles on the CPU in fp32 and fp64.

Every tensor is measured against its own scale (parity_check with zero_floor_frac=1e-12), so a small recurrent-weight
gradient cannot hide under the largest gradient of the model."""
import copy

import pytest
import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

from conftest import parity_check
from oracle import dgcnv2_oracle, seeded
from oracle import modules as om
from oracle.make_golden import DGCNV2_SEED
from test_gpu_gru import GruDgcnv2Oracle

OWN_SCALE = 1e-12
CELLS = {"lstm": nn.LSTM, "gru": nn.GRU}


def _padded(lengths, D, gen):
    B, Lmax = len(lengths), max(lengths)
    mask = torch.arange(Lmax)[None, :] < torch.tensor(lengths)[:, None]
    return torch.randn(B, Lmax, D, generator=gen) * mask[..., None], mask


def _torch_rnn(rnn, x_pad, lengths, R_pad, dtype):
    """torch's module over the packed batch on the CPU in ``dtype``, loss sum(out * R):
    -> (padded output, dx_pad, {parameter name: gradient})."""
    ref = copy.deepcopy(rnn).to(dtype)
    x = x_pad.to(dtype, copy=True).requires_grad_(True)
    packed = pack_padded_sequence(x, torch.tensor(lengths), batch_first=True, enforce_sorted=False)
    out, _ = pad_packed_sequence(ref(packed)[0], batch_first=True, total_length=x.size(1))
    (out * R_pad.to(dtype)).sum().backward()
    return out.detach(), x.grad, {k: p.grad.numpy() for k, p in ref.named_parameters()}


def _layer(cell, Hd, D, seed):
    """One bidirectional layer with random weights and random non-zero biases of order 0.3 (large enough that a b_hn
    folded into the hoisted GEMM, outside the GRU's reset gate, fails the comparison)."""
    rnn = CELLS[cell](D, Hd, num_layers=1, bidirectional=True, batch_first=True)
    seeded.fill_by_name(rnn, seed)
    seeded.fill_by_name(rnn, seed + 1, scale=8.0, only=lambda k: k.startswith("bias"))
    assert all(float(p.detach().abs().min()) > 0 for k, p in rnn.named_parameters() if k.startswith("bias"))
    return rnn


def _run_layer(rnn, x_pad, mask, lengths, R_pad):
    """hoisted ops.linear + ops.lstm_layer / ops.gru_layer (dgcn_models.birnn_forward) on the GPU, loss sum(out * R)."""
    from erc_b200.track_mm.dgcn_models import birnn_forward
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    dev = torch.device("cuda")
    m = copy.deepcopy(rnn).to(dev)
    g = lengths_graph(torch.tensor(lengths), dev)
    x = x_pad[mask].to(dev).requires_grad_(True)
    out = birnn_forward(m, x, g, None, False)
    (out * R_pad[mask].to(dev)).sum().backward()
    return {"out": out.detach(), "dx": x.grad, **{k: p.grad for k, p in m.named_parameters()}}


def _check_layer(case, cell, Hd, lengths, seed):
    gen = torch.Generator().manual_seed(seed)
    D = 40
    x_pad, mask = _padded(lengths, D, gen)
    R_pad = torch.randn(len(lengths), max(lengths), 2 * Hd, generator=gen) * mask[..., None]
    rnn = _layer(cell, Hd, D, seed)
    refs = []
    for dt in (torch.float32, torch.float64):
        out, dx, grads = _torch_rnn(rnn, x_pad, lengths, R_pad, dt)
        refs.append({"out": out[mask].numpy(), "dx": dx[mask].numpy(), **grads})
    got = _run_layer(rnn, x_pad, mask, lengths, R_pad)
    assert len(got) == 10
    parity_check(case, got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", ["lstm", "gru"])
@pytest.mark.parametrize("Hd", [101, 128, 150, 256, 384])
def test_layer_vs_torch_on_packed_sequences(cell, Hd):
    """400 dialogues, lengths 1..110 with 1 and 110 included: the output, dx and all eight parameter gradients."""
    import erc_b200  # noqa: F401
    gen = torch.Generator().manual_seed(300 + Hd)
    lengths = [1, 110] + torch.randint(1, 111, (398,), generator=gen).tolist()
    _check_layer("%s/layer/Hd%d" % (cell, Hd), cell, Hd, lengths, 11 + Hd)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", ["lstm", "gru"])
def test_layer_many_dialogues(cell):
    """2999 IEMOCAP-shaped dialogues at Hd = 128: every cluster runs many dialogues on each of its lanes, and the count is
    odd, so it is not a multiple of the (even) number of clusters."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    lengths = synth.iemocap_lengths(2999, torch.Generator().manual_seed(8)).tolist()
    _check_layer("%s/layer/many" % cell, cell, 128, lengths, 5)


@pytest.mark.gpu
@pytest.mark.parametrize("cell", ["lstm", "gru"])
@pytest.mark.parametrize("g_dim", [300, 512])
def test_seqcontext_vs_torch(cell, g_dim):
    """SeqContext(100, g_dim, rnn_type=cell) -> zero-padded [B, max L, g_dim] and its parameter gradients, against the
    torch module over the packed batch with the same state_dict (Hd = 150 and 256, two layers)."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    from erc_b200.track_mm.dgcn_models import SeqContext
    gen = torch.Generator().manual_seed(g_dim)
    lengths = [1] + synth.iemocap_lengths(23, gen).tolist()
    D = 100
    x_pad, mask = _padded(lengths, D, gen)
    R_pad = torch.randn(len(lengths), max(lengths), g_dim, generator=gen) * mask[..., None]
    m = SeqContext(D, g_dim, dropout=0.4, rnn_type=cell).eval()
    seeded.fill_by_name(m, 29)
    rnn = CELLS[cell](D, g_dim // 2, num_layers=2, bidirectional=True, batch_first=True, dropout=0.4).eval()
    rnn.load_state_dict({k[len("rnn."):]: v for k, v in m.state_dict().items()})
    refs = []
    for dt in (torch.float32, torch.float64):
        out, _, grads = _torch_rnn(rnn, x_pad, lengths, R_pad, dt)
        refs.append({"out": out.numpy(), **{"rnn." + k: v for k, v in grads.items()}})
    m = m.cuda()
    out = m(torch.tensor(lengths), x_pad.cuda())
    assert out.shape == (len(lengths), max(lengths), g_dim)
    (out * R_pad.cuda()).sum().backward()
    got = {"out": out, **{k: p.grad for k, p in m.named_parameters()}}
    assert len(got) == 17
    parity_check("%s/seqcontext/%d" % (cell, g_dim), got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
def test_dialoguegcn_hidden_300_vs_oracle():
    """DialogueGCN DGCNModule(2, input_size=1380, hidden_size=300) (BiLSTM Hd = 150) on an IEMOCAP-shaped batch of 16
    dialogues with class weights, against DgcnOracle(hidden_size=300) in fp32 and fp64: logits, graph output and every
    live gradient."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops, synth
    from erc_b200.track_mm.dgcn import DGCNModule, LOSS_WEIGHTS
    b = synth.config2(seed=4, B=16)
    x, spk, lens, y = b["input_tensor"], b["speaker_tensor"], b["text_length"], b["label"]
    w = torch.tensor(LOSS_WEIGHTS)
    torch.manual_seed(4)
    o = om.DgcnOracle(2, input_size=1380, hidden_size=300, n_classes=6, dropout=0.0)
    res = []
    for dt in (torch.float32, torch.float64):
        oo = copy.deepcopy(o).to(dt).train()
        ol, og = oo(x.to(dt), spk, lens)
        F.cross_entropy(ol, y, weight=w.to(dt)).backward()
        res.append(({"logits": ol.detach().numpy(), "graph_out": og.detach().numpy()},
                    {k: p.grad.numpy() for k, p in oo.named_parameters() if p.grad is not None}))
    assert any(k.startswith("rnn.") for k in res[0][1])
    m = DGCNModule(2, input_size=1380, hidden_size=300, n_classes=6).cuda()
    missing, unexpected = m.load_state_dict(o.state_dict(), strict=False)
    assert not unexpected and all(k.startswith("clf.emotion_att") for k in missing)
    m.rnn.rnn.dropout = 0.0
    m.clf.drop.p = 0.0
    m.train()
    logits, graph_out = m(x.cuda(), spk.cuda(), lens)
    ops.cross_entropy(logits, y.cuda(), w.cuda()).backward()
    parity_check("dgcn/hidden300/outputs", {"logits": logits, "graph_out": graph_out}, res[0][0], res[1][0],
                 zero_floor_frac=OWN_SCALE)
    grads = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None}
    assert set(res[0][1]) <= set(grads), sorted(set(res[0][1]) - set(grads))
    parity_check("dgcn/hidden300/grads", {k: grads[k] for k in res[0][1]}, res[0][1], res[1][1],
                 zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("base", ["LSTM", "GRU"])
def test_dgcnv2_hidden_128_vs_oracle(base):
    """dgcnv2 DGCNModule(base, hidden_size=128) on the IEMOCAP-shaped batch of 16 dialogues (inputs 1380 wide, window
    10/10, class weights) against Dgcnv2Oracle / the GRU-base oracle in fp32 and fp64: logits, features and every live
    gradient."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops, synth
    from erc_b200.train_mm import DGCN_LOSS_WEIGHTS
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    lengths = [int(v) for v in synth.iemocap_lengths(16, torch.Generator().manual_seed(3))]
    b = dgcnv2_oracle.inputs(lengths, 1380, 2, 6, seed=5)
    w = torch.tensor(DGCN_LOSS_WEIGHTS)
    if base == "LSTM":
        o = dgcnv2_oracle.Dgcnv2Oracle(1380, hidden_size=128, n_classes=6, dropout=0.0)
    else:
        o = GruDgcnv2Oracle(1380, hidden_size=128, n_classes=6, dropout=0.0)
    seeded.fill_by_name(o, DGCNV2_SEED)
    res = []
    for dt in (torch.float32, torch.float64):
        oo = copy.deepcopy(o).to(dt).train()
        lg, ft = oo(b["input_tensor"].to(dt), b["speaker_tensor"].to(dt), b["attention_mask"], b["text_length"])
        F.cross_entropy(lg, b["label"], weight=w.to(dt)).backward()
        res.append(({"logits": lg.detach().numpy(), "features": ft.detach().numpy()},
                    {k: p.grad.numpy() for k, p in oo.named_parameters() if p.grad is not None}))
    assert any(k.startswith(base.lower() + ".") for k in res[0][1])
    m = DGCNModule(base, input_size=1380, hidden_size=128, n_speakers=2, n_classes=6, dropout=0.0)
    m.graph_net.dropout.p = 0.0
    seeded.fill_by_name(m, DGCNV2_SEED)
    m = m.cuda().train()
    logits, feats = m(input_tensor=b["input_tensor"].cuda(), speaker_tensor=b["speaker_tensor"].cuda(),
                      attention_mask=b["attention_mask"].cuda(), text_length=b["text_length"])
    ops.cross_entropy(logits, b["label"].cuda(), w.cuda()).backward()
    parity_check("dgcnv2_%s/hidden128/outputs" % base, {"logits": logits, "features": feats}, res[0][0], res[1][0],
                 zero_floor_frac=OWN_SCALE)
    grads = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None}
    assert set(res[0][1]) <= set(grads), sorted(set(res[0][1]) - set(grads))
    parity_check("dgcnv2_%s/hidden128/grads" % base, {k: grads[k] for k in res[0][1]}, res[0][1], res[1][1],
                 zero_floor_frac=OWN_SCALE)


def _layer_args(cell, Hd, lengths, seed):
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(seed)
    G = 4 if cell == "lstm" else 3
    N = int(sum(lengths))
    gx = torch.randn(N, 2 * G * Hd, device=dev, generator=gen)
    whh = torch.randn(2, G * Hd, Hd, device=dev, generator=gen) / Hd ** 0.5
    bhh = torch.randn(2, G * Hd, device=dev, generator=gen) * 0.3
    R = torch.randn(N, 2 * Hd, device=dev, generator=gen)
    return gx, whh, bhh, R, lengths_graph(torch.tensor(lengths), dev)


def _fwd_bwd(cell, gx, whh, bhh, R, g):
    from erc_b200 import ops
    gx, whh, bhh = (t.detach().requires_grad_(True) for t in (gx, whh, bhh))
    out = ops.lstm_layer(gx, whh, g) if cell == "lstm" else ops.gru_layer(gx, whh, bhh, g)
    inputs = [gx, whh] if cell == "lstm" else [gx, whh, bhh]
    return [out.detach()] + list(torch.autograd.grad(out, inputs, R))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", ["lstm", "gru"])
@pytest.mark.parametrize("Hd", [128, 384])
def test_bit_reproducible_grid_independent_and_graph_capturable(cell, Hd):
    """Two forward + backward runs are bit-identical; the first 37 dialogues run alone (a smaller grid) give the same
    bits for their rows; a CUDA-graph capture of the layer, forward and backward, replays the eager result bit for bit."""
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    gen = torch.Generator().manual_seed(Hd)
    lengths = [1, 110] + torch.randint(1, 111, (598,), generator=gen).tolist()
    gx, whh, bhh, R, g = _layer_args(cell, Hd, lengths, Hd)
    a = _fwd_bwd(cell, gx, whh, bhh, R, g)
    b = _fwd_bwd(cell, gx, whh, bhh, R, g)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    assert all(torch.isfinite(u).all() for u in a)

    n = int(sum(lengths[:37]))
    sub = _fwd_bwd(cell, gx[:n], whh, bhh, R[:n], lengths_graph(torch.tensor(lengths[:37]), gx.device))
    assert torch.equal(sub[0], a[0][:n]) and torch.equal(sub[1], a[1][:n])

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _fwd_bwd(cell, gx, whh, bhh, R, g)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c = _fwd_bwd(cell, gx, whh, bhh, R, g)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(a, c))


@pytest.mark.gpu
def test_hidden_sizes_above_384_raise():
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200._lib import ErcgError
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    dev = torch.device("cuda")
    g = lengths_graph(torch.tensor([3, 5]), dev)
    for Hd in (385, 512):
        with pytest.raises(ErcgError):
            ops.lstm_layer(torch.randn(8, 8 * Hd, device=dev), torch.randn(2, 4 * Hd, Hd, device=dev), g)
        with pytest.raises(ErcgError):
            ops.gru_layer(torch.randn(8, 6 * Hd, device=dev), torch.randn(2, 3 * Hd, Hd, device=dev),
                          torch.randn(2, 3 * Hd, device=dev), g)
    torch.cuda.synchronize()


@pytest.mark.parametrize("Hd", [101, 256, 384])
def test_entry_points_accept_an_empty_batch_and_reject_negative_at_new_sizes(Hd):
    """B = 0 is a no-op that touches no pointer; B < 0 is an argument error (checked before any launch)."""
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    for B, want in ((0, 0), (-1, -1)):
        assert lib().ercg_lstm_fwd(None, 0, None, None, B, Hd, None, 0, None, None, None, None) == want
        assert lib().ercg_lstm_bwd(None, 0, None, None, None, None, B, Hd, None, 0, None) == want
        assert lib().ercg_gru_fwd(None, 0, None, None, None, B, Hd, None, 0, None, None, None) == want
        assert lib().ercg_gru_bwd(None, 0, None, None, None, None, B, Hd, None, 0, None, 0, None) == want
