"""K13 (csrc/seq_attn.cu: dense masked MatchingAttention, the sequence reversal) and the log-softmax of norm_loss.cu behind
track_mm.dgcnv2_models' MatchingAttention.forward, LSTMModel, GRUModel and DialogRNNModel, against the CPU transcription of
the declare-lab classes (oracle/dgcnv2_seq_oracle.py) in fp32 and fp64.

Every tensor is measured against its own scale (parity_check with zero_floor_frac=1e-12).  The model tests run in eval():
DialogRNNModel's dropout_rec is dropout + 0.15, so it is never 0 in training mode."""
import copy

import pytest
import torch

from conftest import parity_check
from oracle import dgcnv2_seq_oracle as O

OWN_SCALE = 1e-12


def _mask(kind, lengths, L, gen):
    B = len(lengths)
    if kind == "none":
        return None
    inside = (torch.arange(L)[None, :] < torch.tensor(lengths)[:, None]).float()
    if kind == "prefix":
        return inside
    m = (torch.rand(B, L, generator=gen) < 0.6).float()
    m[torch.arange(B), torch.randint(0, L, (B,), generator=gen)] = 1.0          # never all zero
    if kind == "float":
        m = m * torch.rand(B, L, generator=gen) * 1.5
        m[torch.arange(B), 0] = 0.75
    return m


def _att_oracle(o, M, x, mask, R, dt, all_positions):
    oo = copy.deepcopy(o).to(dt)
    m = M.detach().to(dt, copy=True).requires_grad_(True)
    xx = x.detach().to(dt, copy=True).requires_grad_(True)
    mk = None if mask is None else mask.to(dt)
    if all_positions:
        pools, alphas = zip(*[oo(m, m[t], mk) for t in range(m.size(0))])
        pool, alpha = torch.stack(pools), torch.stack([a[:, 0, :] for a in alphas])
    else:
        pool, alpha = oo(m, xx, mk)
    (pool * R.to(dt)).sum().backward()
    out = {"pool": pool.detach().numpy(), "alpha": alpha.detach().numpy(), "dM": m.grad.numpy(),
           **{"d" + k: p.grad.numpy() for k, p in oo.named_parameters()}}
    if not all_positions:
        out["dx"] = xx.grad.numpy()
    return out


def _att_ours(mod, M, x, mask, R, all_positions):
    mod.zero_grad(set_to_none=True)
    m = M.detach().cuda().requires_grad_(True)
    xx = x.detach().cuda().requires_grad_(True)
    mk = None if mask is None else mask.cuda()
    if all_positions:
        pool, alpha = mod.all_positions(m, mk)
    else:
        pool, alpha = mod(m, xx, mk)
    (pool * R.cuda()).sum().backward()
    out = {"pool": pool, "alpha": alpha, "dM": m.grad, **{"d" + k: p.grad for k, p in mod.named_parameters()}}
    if not all_positions:
        out["dx"] = xx.grad
    return out


SHAPES = [(1, 84, 7), (3, 110, 5), (200, 84, 400), (202, 110, 33), (768, 1, 16), (1024, 110, 9)]   # (D, L, B)


@pytest.mark.gpu
@pytest.mark.parametrize("D,L,B", SHAPES)
@pytest.mark.parametrize("att_type", ["general", "general2"])
@pytest.mark.parametrize("mask_kind", ["prefix", "random", "float", "none"])
def test_matching_attention_vs_oracle(D, L, B, att_type, mask_kind):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcnv2_models import MatchingAttention
    gen = torch.Generator().manual_seed(D * 1000 + L + B)
    torch.manual_seed(D + L)
    lengths = [int(v) for v in torch.randint(1, L + 1, (B,), generator=gen)]
    lengths[0] = L
    mask = _mask(mask_kind, lengths, L, gen)
    Dc = D if D > 3 else D + 2
    o = O.MatchingAttention(D, Dc, att_type=att_type)
    mod = MatchingAttention(D, Dc, att_type=att_type).cuda()
    mod.load_state_dict(o.state_dict(), strict=True)
    # memory rows and queries in (-1, 1), like the models' RNN outputs.  With N(0, 1) queries the scores reach |s| ~ 30 at width
    # 1024, and the fp32 summation of the transform GEMM (ops.linear, shared with every model here) then moves alpha, dM and dx
    # up to 2e-5 from the fp64 result, where the reference's fp32 CPU run stays within 4e-6 (DESIGN.md, K13).
    M = torch.tanh(torch.randn(L, B, D, generator=gen))
    x = torch.tanh(torch.randn(B, Dc, generator=gen))
    R = torch.randn(B, D, generator=gen)
    refs = [_att_oracle(o, M, x, mask, R, dt, False) for dt in (torch.float32, torch.float64)]
    got = _att_ours(mod, M, x, mask, R, False)
    assert got["alpha"].shape == (B, 1, L) and got["pool"].shape == (B, D)
    parity_check("match_att/%s/%s/%d_%d_%d" % (att_type, mask_kind, D, L, B), got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)
    # att2: every position of every dialogue as a query.  Not checked for the float mask at width 1024: there the queries come
    # from the tensor-core transform (3xTF32, DESIGN.md section 5) and dM / dtransform.weight land 1.6e-5 / 1.2e-5 from the
    # fp64 result against the fp32 reference's 3.2e-6 / 2.6e-6 (measured on a B200; DESIGN.md, K13).
    if Dc == D and not (mask_kind == "float" and D == 1024):
        R2 = torch.randn(L, B, D, generator=gen)
        refs = [_att_oracle(o, M, x, mask, R2, dt, True) for dt in (torch.float32, torch.float64)]
        got = _att_ours(mod, M, x, mask, R2, True)
        parity_check("match_att_all/%s/%s/%d_%d_%d" % (att_type, mask_kind, D, L, B), got, refs[0], refs[1],
                     zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
def test_matching_attention_all_zero_mask_gives_nan():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcnv2_models import MatchingAttention
    gen = torch.Generator().manual_seed(4)
    mod = MatchingAttention(12, 12, att_type="general2").cuda()
    M, x = torch.randn(9, 3, 12, generator=gen).cuda(), torch.randn(3, 12, generator=gen).cuda()
    mask = torch.ones(3, 9, device="cuda")
    mask[1] = 0
    with torch.no_grad():
        pool, alpha = mod(M, x, mask)
    assert torch.isnan(pool[1]).all() and torch.isnan(alpha[1]).all()
    assert torch.isfinite(pool[[0, 2]]).all() and torch.isfinite(alpha[[0, 2]]).all()
    o = O.MatchingAttention(12, 12, att_type="general2")
    o.load_state_dict({k: v.cpu() for k, v in mod.state_dict().items()})
    with torch.no_grad():
        ref, _ = o(M.cpu(), x.cpu(), mask.cpu())
    assert torch.isnan(ref[1]).all()                                    # the reference's 0 / 0


def _batch(lengths, L, Dm, P, gen, zero_frac=0.0):
    B = len(lengths)
    inside = torch.arange(L)[:, None] < torch.tensor(lengths)[None, :]                   # [L, B]
    U = torch.randn(L, B, Dm, generator=gen) * inside[..., None]
    spk = torch.randint(0, P, (L, B), generator=gen)
    drop = (torch.rand(L, B, generator=gen) < zero_frac) & (torch.arange(L)[:, None] > 0)
    qm = torch.nn.functional.one_hot(spk, P).float() * (inside & ~drop)[..., None]
    umask = inside.t().float().contiguous()
    return U, qm, umask


def _model_oracle(o, U, qm, umask, R, att2, dt):
    oo = copy.deepcopy(o).to(dt).eval()
    u = U.detach().to(dt, copy=True).requires_grad_(True)
    log_prob, alpha, alpha_f, alpha_b = oo(u, qm.to(dt), umask.to(dt), att2)
    (log_prob * R.to(dt)).sum().backward()
    return _pack(log_prob, alpha, alpha_f, alpha_b, u.grad, oo)


def _pack(log_prob, alpha, alpha_f, alpha_b, dU, m):
    out = {"log_prob": log_prob, "dU": dU,
           **{k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in m.named_parameters()}}
    for name, a in (("alpha", alpha), ("alpha_f", alpha_f), ("alpha_b", alpha_b)):
        if a:
            out[name] = torch.cat([x.reshape(-1) for x in a])
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def _model_ours(m, U, qm, umask, R, att2):
    u = U.detach().cuda().requires_grad_(True)
    log_prob, alpha, alpha_f, alpha_b = m(u, qm.cuda(), umask.cuda(), att2)
    (log_prob * R.cuda()).sum().backward()
    return _pack(log_prob, alpha, alpha_f, alpha_b, u.grad, m), (log_prob, alpha, alpha_f, alpha_b)


def _iemocap(B, seed):
    from erc_b200 import synth
    lengths = [int(v) for v in synth.iemocap_lengths(B, torch.Generator().manual_seed(seed))]
    return lengths, max(lengths)


MODELS = {
    "lstm_100": lambda: ("LSTMModel", (1380, 100, 100), 2, 0.0),
    "lstm_150": lambda: ("LSTMModel", (1380, 150, 100), 2, 0.0),
    "gru_100": lambda: ("GRUModel", (1380, 100, 100), 2, 0.0),
    "gru_150": lambda: ("GRUModel", (1380, 150, 100), 2, 0.0),
    "dialogrnn_simple_p2": lambda: ("DialogRNNModel", (1380, 150, 150, 100, 100), 2, 0.0, "simple"),
    "dialogrnn_general_p2": lambda: ("DialogRNNModel", (1380, 150, 150, 100, 100), 2, 0.0, "general"),
    "dialogrnn_general_p9_zero_rows": lambda: ("DialogRNNModel", (1380, 150, 150, 100, 100), 9, 0.1, "general"),
    "dialogrnn_simple_p9_zero_rows": lambda: ("DialogRNNModel", (1380, 150, 150, 100, 100), 9, 0.1, "simple"),
}


def _build(case, seed):
    from erc_b200.track_mm import dgcnv2_models as ours
    name, dims, P, zf, *att = MODELS[case]()
    kw = dict(n_classes=6, dropout=0.3)
    if att:
        kw["context_attention"] = att[0]
    torch.manual_seed(seed)
    o = getattr(O, name)(*dims, **kw)
    m = getattr(ours, name)(*dims, **kw)
    m.load_state_dict(o.state_dict(), strict=True)
    return o.eval(), m.cuda().eval(), dims[0], P, zf


@pytest.mark.gpu
@pytest.mark.parametrize("att2", [True, False])
@pytest.mark.parametrize("case", list(MODELS))
def test_sequence_model_vs_oracle(case, att2):
    import erc_b200  # noqa: F401
    seed = len(case) + 7 * att2
    o, m, Dm, P, zf = _build(case, seed)
    lengths, L = _iemocap(12, seed)
    gen = torch.Generator().manual_seed(seed)
    U, qm, umask = _batch(lengths, L, Dm, P, gen, zf)
    R = torch.randn(L, len(lengths), 6, generator=gen)
    refs = [_model_oracle(o, U, qm, umask, R, att2, dt) for dt in (torch.float32, torch.float64)]
    got, (log_prob, alpha, alpha_f, alpha_b) = _model_ours(m, U, qm, umask, R, att2)
    assert log_prob.shape == (L, len(lengths), 6)
    assert len(alpha) == (L if att2 else 0) and all(a.shape == (len(lengths), L) for a in alpha)
    if case.startswith("dialogrnn"):
        assert len(alpha_f) == len(alpha_b) == L - 1
    else:
        assert alpha_f == [] and alpha_b == []
    parity_check("seq_model/%s/att2=%d" % (case, att2), got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["lstm_100", "gru_150", "dialogrnn_general_p2"])
def test_sequence_model_training_mode(case):
    import erc_b200  # noqa: F401
    _, m, Dm, P, _ = _build(case, 3)
    lengths, L = _iemocap(6, 3)
    U, qm, umask = (t.cuda() for t in _batch(lengths, L, Dm, P, torch.Generator().manual_seed(3)))
    with torch.no_grad():
        ev = m.eval()(U, qm, umask)[0]
        assert torch.equal(ev, m(U, qm, umask)[0])                       # eval is bit-deterministic
        m.train()
        torch.manual_seed(11)
        tr = m(U, qm, umask)[0]
        torch.manual_seed(11)
        tr2 = m(U, qm, umask)[0]
    assert torch.isfinite(tr).all() and not torch.equal(tr, ev) and torch.equal(tr, tr2)


@pytest.mark.gpu
def test_sequence_model_eval_bit_deterministic_with_gradients():
    import erc_b200  # noqa: F401
    _, m, Dm, P, _ = _build("dialogrnn_simple_p2", 5)
    lengths, L = _iemocap(8, 5)
    gen = torch.Generator().manual_seed(5)
    U, qm, umask = _batch(lengths, L, Dm, P, gen)
    R = torch.randn(L, len(lengths), 6, generator=gen)
    runs = []
    for _ in range(2):
        m.zero_grad()
        runs.append(_model_ours(m, U, qm, umask, R, True)[0])
    assert all((runs[0][k] == runs[1][k]).all() for k in runs[0])


@pytest.mark.gpu
def test_dialog_rnn_model_rejects_masks_shorter_than_the_batch():
    import erc_b200  # noqa: F401
    _, m, Dm, P, _ = _build("dialogrnn_general_p2", 2)
    U, qm, umask = (t.cuda() for t in _batch([7, 5], 9, Dm, P, torch.Generator().manual_seed(2)))
    with pytest.raises(ValueError):
        m(U, qm, umask)
    with pytest.raises(ValueError):                                     # umask of the wrong shape
        m(U, qm, umask[:, :8])
