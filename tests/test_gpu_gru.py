"""K6b, the bidirectional GRU context encoder (csrc/gru.cu): ops.gru_layer, SeqContext(rnn_type="gru"), the dgcnv2
DGCNModule("GRU") and the train_mm launcher, against torch.nn.GRU on the CPU in fp32 and fp64.

Every tensor is measured against its own scale (parity_check with zero_floor_frac=1e-12), so a small recurrent-weight
gradient cannot hide under the largest gradient of the model."""
import copy
import os

import pytest
import torch
import torch.nn.functional as F
from torch import nn
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

from conftest import parity_check
from oracle import dgcnv2_oracle, seeded
from oracle.make_golden import DGCNV2_SEED

OWN_SCALE = 1e-12


class GruDgcnv2Oracle(dgcnv2_oracle.Dgcnv2Oracle):
    """The declare-lab DialogueGCN with base_model="GRU": ``self.gru = nn.GRU(input_size, hidden_size, num_layers=2,
    bidirectional=True, dropout=dropout)`` run unpacked over the seq-first padded batch, like the LSTM base.  Everything
    after the base is Dgcnv2Oracle's, which runs ``self.base_linear(input_tensor)`` for any base other than 'LSTM'."""

    def __init__(self, input_size, hidden_size=100, dropout=0.0, **kw):
        super().__init__(input_size, hidden_size, dropout=dropout, base_model="None", **kw)
        del self.base_linear
        self.base_model = "GRU"
        self.gru = nn.GRU(input_size=input_size, hidden_size=hidden_size, num_layers=2, bidirectional=True, dropout=dropout)

    def base_linear(self, x):
        return self.gru(x)[0]


def _padded(lengths, D, gen):
    B, Lmax = len(lengths), max(lengths)
    mask = torch.arange(Lmax)[None, :] < torch.tensor(lengths)[:, None]
    x = torch.randn(B, Lmax, D, generator=gen) * mask[..., None]
    return x, mask


def _torch_gru(rnn, x_pad, lengths, R_pad, dtype):
    """torch's nn.GRU over the packed batch on the CPU in ``dtype``, loss sum(out * R):
    -> (padded output, dx_pad, {parameter name: gradient})."""
    ref = copy.deepcopy(rnn).to(dtype)
    x = x_pad.to(dtype, copy=True).requires_grad_(True)
    packed = pack_padded_sequence(x, torch.tensor(lengths), batch_first=True, enforce_sorted=False)
    out, _ = pad_packed_sequence(ref(packed)[0], batch_first=True, total_length=x.size(1))
    (out * R_pad.to(dtype)).sum().backward()
    return out.detach(), x.grad, {k: p.grad.numpy() for k, p in ref.named_parameters()}


@pytest.mark.gpu
@pytest.mark.parametrize("Hd", [8, 24, 100])
def test_gru_layer_vs_torch_on_packed_sequences(Hd):
    """One bidirectional layer, hoisted ops.linear + ops.gru_layer, 400 dialogues (more than the 148 CTAs per direction,
    so every CTA runs several dialogues), lengths 1 and 110 included, random non-zero biases (a b_hn folded into the
    hoisted GEMM fails): the output, dx and all eight parameter gradients."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    gen = torch.Generator().manual_seed(100 + Hd)
    lengths = [1, 110] + torch.randint(1, 111, (398,), generator=gen).tolist()
    D = 40
    x_pad, mask = _padded(lengths, D, gen)
    R_pad = torch.randn(len(lengths), max(lengths), 2 * Hd, generator=gen) * mask[..., None]
    rnn = nn.GRU(D, Hd, num_layers=1, bidirectional=True, batch_first=True)
    seeded.fill_by_name(rnn, 7 + Hd)
    refs = []
    for dt in (torch.float32, torch.float64):
        out, dx, grads = _torch_gru(rnn, x_pad, lengths, R_pad, dt)
        refs.append({"out": out[mask].numpy(), "dx": dx[mask].numpy(), **grads})

    dev = torch.device("cuda")
    m = copy.deepcopy(rnn).to(dev)
    g = lengths_graph(torch.tensor(lengths), dev)
    x = x_pad[mask].to(dev).requires_grad_(True)
    gx = ops.linear(x, torch.cat([m.weight_ih_l0, m.weight_ih_l0_reverse]), torch.cat([m.bias_ih_l0, m.bias_ih_l0_reverse]))
    out = ops.gru_layer(gx, torch.stack([m.weight_hh_l0, m.weight_hh_l0_reverse]),
                        torch.stack([m.bias_hh_l0, m.bias_hh_l0_reverse]), g)
    (out * R_pad[mask].to(dev)).sum().backward()
    got = {"out": out, "dx": x.grad, **{k: p.grad for k, p in m.named_parameters()}}
    assert len(got) == 10
    parity_check("gru/layer/Hd%d" % Hd, got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
def test_seqcontext_gru_vs_torch_on_packed_sequences():
    """SeqContext(rnn_type="gru").forward(text_len_tensor, text_tensor) -> zero-padded [B, max L, g_dim] and its parameter
    gradients, against nn.GRU over the packed batch with the same state_dict."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    from erc_b200.track_mm.dgcn_models import SeqContext
    gen = torch.Generator().manual_seed(21)
    lengths = [1] + synth.iemocap_lengths(23, gen).tolist()
    D, g_dim = 100, 200
    x_pad, mask = _padded(lengths, D, gen)
    R_pad = torch.randn(len(lengths), max(lengths), g_dim, generator=gen) * mask[..., None]
    m = SeqContext(D, g_dim, dropout=0.4, rnn_type="gru").eval()
    seeded.fill_by_name(m, 23)
    rnn = nn.GRU(D, g_dim // 2, num_layers=2, bidirectional=True, batch_first=True, dropout=0.4).eval()
    rnn.load_state_dict({k[len("rnn."):]: v for k, v in m.state_dict().items()})
    refs = []
    for dt in (torch.float32, torch.float64):
        out, _, grads = _torch_gru(rnn, x_pad, lengths, R_pad, dt)
        refs.append({"out": out.numpy(), **{"rnn." + k: v for k, v in grads.items()}})

    m = m.cuda()
    out = m(torch.tensor(lengths), x_pad.cuda())
    assert out.shape == (len(lengths), max(lengths), g_dim)
    (out * R_pad.cuda()).sum().backward()
    got = {"out": out, **{k: p.grad for k, p in m.named_parameters()}}
    assert len(got) == 17
    parity_check("gru/seqcontext", got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


def test_gru_modules_state_dict_keys_and_rejected_bases():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcn_models import SeqContext
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    keys = list(nn.GRU(100, 100, num_layers=2, bidirectional=True).state_dict())
    assert len(keys) == 16 and keys[-1] == "bias_hh_l1_reverse"
    assert list(SeqContext(100, 200, rnn_type="gru").state_dict()) == ["rnn." + k for k in keys]
    m = DGCNModule("GRU", input_size=100, n_classes=6)
    assert [k for k in m.state_dict() if k.startswith("gru.")] == ["gru." + k for k in keys]
    assert set(GruDgcnv2Oracle(100, n_classes=6).state_dict()) <= set(m.state_dict())
    with pytest.raises(ValueError):
        SeqContext(100, 200, rnn_type="rnn")
    with pytest.raises(NotImplementedError):
        DGCNModule("DialogRNN", input_size=100)


def test_gru_entry_points_accept_an_empty_batch_and_reject_bad_sizes():
    """B = 0 is a no-op that touches no pointer; B < 0 is an argument error (checked before any launch)."""
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    assert lib().ercg_gru_fwd(None, 0, None, None, None, 0, 100, None, 0, None, None, None) == 0
    assert lib().ercg_gru_bwd(None, 0, None, None, None, None, 0, 100, None, 0, None, 0, None) == 0
    assert lib().ercg_gru_fwd(None, 0, None, None, None, -1, 100, None, 0, None, None, None) == -1
    assert lib().ercg_gru_bwd(None, 0, None, None, None, None, -1, 100, None, 0, None, 0, None) == -1


@pytest.mark.gpu
def test_gru_layer_unsupported_hidden_size_raises():
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200._lib import ErcgError
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    dev = torch.device("cuda")
    g = lengths_graph(torch.tensor([3, 5]), dev)
    for Hd in (50, 12):
        gx = torch.randn(8, 6 * Hd, device=dev)
        whh = torch.randn(2, 3 * Hd, Hd, device=dev)
        bhh = torch.randn(2, 3 * Hd, device=dev)
        with pytest.raises(ErcgError):
            ops.gru_layer(gx, whh, bhh, g)
    torch.cuda.synchronize()
    out = ops.gru_layer(torch.zeros(8, 48, device=dev), torch.zeros(2, 24, 8, device=dev), torch.zeros(2, 24, device=dev), g)
    torch.cuda.synchronize()
    assert torch.equal(out, torch.zeros(8, 16, device=dev))     # zero pre-activations: n = 0, z = 1/2, h stays 0


def _run(m, b):
    from erc_b200 import ops
    from erc_b200.train_mm import DGCN_LOSS_WEIGHTS
    logits, feats = m(input_tensor=b["input_tensor"].cuda(), speaker_tensor=b["speaker_tensor"].cuda(),
                      attention_mask=b["attention_mask"].cuda(), text_length=b["text_length"])
    loss = ops.cross_entropy(logits, b["label"].cuda(), torch.tensor(DGCN_LOSS_WEIGHTS).cuda())
    loss.backward()
    return logits, feats, loss


@pytest.mark.gpu
def test_dgcnv2_gru_base_iemocap_shape_vs_oracle():
    """DGCNModule("GRU") on the IEMOCAP-shaped batch of 16 dialogues (inputs 1380 wide, window 10/10, class weights)
    against the GRU-based DialogueGCN oracle in fp32 and fp64: logits, features and every live gradient."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    from erc_b200.train_mm import DGCN_LOSS_WEIGHTS
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    lengths = [int(v) for v in synth.iemocap_lengths(16, torch.Generator().manual_seed(3))]
    b = dgcnv2_oracle.inputs(lengths, 1380, 2, 6, seed=5)
    w = torch.tensor(DGCN_LOSS_WEIGHTS)
    o = GruDgcnv2Oracle(1380, n_classes=6, dropout=0.0)
    seeded.fill_by_name(o, DGCNV2_SEED)
    res = []
    for dt in (torch.float32, torch.float64):
        oo = copy.deepcopy(o).to(dt).train()
        lg, ft = oo(b["input_tensor"].to(dt), b["speaker_tensor"].to(dt), b["attention_mask"], b["text_length"])
        F.cross_entropy(lg, b["label"], weight=w.to(dt)).backward()
        res.append(({"logits": lg.detach().numpy(), "features": ft.detach().numpy()},
                    {k: p.grad.numpy() for k, p in oo.named_parameters() if p.grad is not None}))
    assert any(k.startswith("gru.") for k in res[0][1])
    m = DGCNModule("GRU", input_size=1380, hidden_size=100, n_speakers=2, n_classes=6, dropout=0.0)
    m.graph_net.dropout.p = 0.0
    seeded.fill_by_name(m, DGCNV2_SEED)
    m = m.cuda().train()
    logits, feats, loss = _run(m, b)
    parity_check("dgcnv2_gru/iemocap16/outputs", {"logits": logits, "features": feats}, res[0][0], res[1][0],
                 zero_floor_frac=OWN_SCALE)
    grads = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None}
    assert set(res[0][1]) <= set(grads), sorted(set(res[0][1]) - set(grads))
    grads = {k: grads[k] for k in res[0][1]}
    parity_check("dgcnv2_gru/iemocap16/grads", grads, res[0][1], res[1][1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
def test_gru_training_mode_dropout_and_eval_determinism():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcn_models import SeqContext
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    b = dgcnv2_oracle.inputs([6, 3, 11], 24, 2, 6, seed=2)
    torch.manual_seed(0)
    m = DGCNModule("GRU", input_size=24, n_classes=6).cuda().train()          # dropout 0.4 between the GRU layers
    logits, feats, loss = _run(m, b)
    assert torch.isfinite(loss) and logits.shape == (20, 6) and feats.shape == (20, 200)
    grads = {k: p.grad for k, p in m.named_parameters() if p.grad is not None}
    assert any(k.startswith("gru.") for k in grads) and all(torch.isfinite(v).all() for v in grads.values())
    m.eval()
    with torch.no_grad():
        e1 = m(b["input_tensor"].cuda(), b["speaker_tensor"].cuda(), b["attention_mask"].cuda(), b["text_length"])
        e2 = m(b["input_tensor"].cuda(), b["speaker_tensor"].cuda(), b["attention_mask"].cuda(), b["text_length"])
    assert torch.equal(e1[0], e2[0]) and torch.equal(e1[1], e2[1])

    gen = torch.Generator().manual_seed(4)
    lengths = [6, 3, 11]
    x, _ = _padded(lengths, 24, gen)
    x, lens = x.cuda(), torch.tensor(lengths)
    with torch.no_grad():
        for p, differ in ((0.4, True), (0.0, False)):
            sc = SeqContext(24, 200, dropout=p, rnn_type="gru").cuda()
            ev = sc.eval()(lens, x)
            assert torch.equal(ev, sc(lens, x))
            tr = sc.train()(lens, x)
            assert torch.isfinite(tr).all()
            assert (not torch.equal(tr, ev)) == differ, p


@pytest.mark.gpu
def test_train_mm_dgcnv2_gru_base_synthetic_epochs(tmp_path):
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import main, build_model
    lines = []
    out = main(["--module=dgcnv2", "--base_model=GRU", "--modality=atv", "--epoch=3", "--train_dialogues=24",
                "--test_dialogues=8", "--train.batch_size=8", "--save_dir=" + str(tmp_path), "--lr=0.001",
                "--dataset=iemocap-cogmen-6", "--max_len=40"], log=lambda *a: lines.append(" ".join(str(x) for x in a)))
    h = out["history"]
    assert out["params"]["base_model"] == "GRU"
    assert len(h) == 3 and all(torch.isfinite(torch.tensor(r["train_Lall"])) for r in h)
    assert h[-1]["train_Lall"] < h[0]["train_Lall"]
    for name in ("best_model.ckpt", "last_model.ckpt"):
        sd = torch.load(os.path.join(str(tmp_path), name))
        assert any(k.startswith("gru.") for k in sd)
        fresh = build_model(out["params"], torch.device("cuda"))
        fresh.load_state_dict(sd, strict=True)
    assert any(l.startswith("Best Results") for l in lines)
