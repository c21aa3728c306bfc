"""K12, the DialogueRNN recurrence (csrc/dialogue_rnn.cu): ops_dgcnv2.dialogue_rnn and track_mm.dgcnv2_models.DialogueRNN
against the CPU transcription of the declare-lab classes (oracle/dialogue_rnn_oracle.py) in fp32 and fp64.

Every tensor is measured against its own scale (parity_check with zero_floor_frac=1e-12): e, alpha, dU and all 13
parameter gradients of the loss sum(e * R)."""
import copy
import ctypes

import pytest
import torch

from conftest import parity_check
from oracle import dialogue_rnn_oracle as O

OWN_SCALE = 1e-12


def _qmask(lengths, L, P, gen, zero_frac=0.0):
    """[L, B, P] one-hot speaker rows inside each dialogue, all-zero after its length; ``zero_frac`` of the rows inside a
    dialogue (never its first) are all-zero as well."""
    B = len(lengths)
    spk = torch.randint(0, P, (L, B), generator=gen)
    qm = torch.nn.functional.one_hot(spk, P).float()
    inside = torch.arange(L)[:, None] < torch.tensor(lengths)[None, :]
    drop = (torch.rand(L, B, generator=gen) < zero_frac) & (torch.arange(L)[:, None] > 0)
    return qm * (inside & ~drop)[..., None]


def _oracle_run(o, U, qm, R, dt, masks=None):
    oo = copy.deepcopy(o).to(dt)
    u = U.detach().to(dt, copy=True).requires_grad_(True)
    e, alpha = oo(u, qm.to(dt), masks)
    (e * R.to(dt)).sum().backward()
    # with L = 1 the attention is never evaluated: its weight has no .grad (mathematically zero)
    out = {"e": e.detach().numpy(), "dU": u.grad.numpy(),
           **{k: (p.grad if p.grad is not None else torch.zeros_like(p)).numpy() for k, p in oo.named_parameters()}}
    if alpha:
        out["alpha"] = torch.cat([a.reshape(-1) for a in alpha]).detach().numpy()
    return out


def _ours(m, U, qm, R, drop_p=None, seeds=(0, 0, 0)):
    """Module forward (eval) or, with drop_p, the op with explicit seeds; loss sum(e * R)."""
    from erc_b200 import ops_dgcnv2
    u = U.detach().cuda().requires_grad_(True)
    if drop_p is None:
        e, alpha = m(u, qm.cuda())
    else:
        c = m.dialogue_cell
        att = c.attention.scalar.weight if c.context_attention == "simple" else c.attention.transform.weight
        e, alpha = ops_dgcnv2.dialogue_rnn(u, qm.cuda(), c.g_cell, c.p_cell, c.e_cell, att, c.context_attention, drop_p, seeds)
    (e * R.cuda()).sum().backward()
    out = {"e": e, "dU": u.grad, **{k: p.grad for k, p in m.named_parameters()}}
    if alpha:
        out["alpha"] = torch.cat([a.reshape(-1) for a in alpha])
    return out, alpha


def _setup(lengths, L, Dm, Dg, Dp, De, P, att, seed, zero_frac=0.0):
    from erc_b200.track_mm.dgcnv2_models import DialogueRNN
    gen = torch.Generator().manual_seed(seed)
    B = len(lengths)
    torch.manual_seed(seed)
    o = O.DialogueRNN(Dm, Dg, Dp, De, context_attention=att, dropout=0.5).eval()
    U = torch.randn(L, B, Dm, generator=gen)
    qm = _qmask(lengths, L, P, gen, zero_frac)
    R = torch.randn(L, B, De, generator=gen)
    m = DialogueRNN(Dm, Dg, Dp, De, context_attention=att, dropout=0.5)
    m.load_state_dict(o.state_dict(), strict=True)
    return o, m.cuda().eval(), U, qm, R


def _iemocap(B, seed):
    from erc_b200 import synth
    lengths = [int(v) for v in synth.iemocap_lengths(B, torch.Generator().manual_seed(seed))]
    return lengths, max(lengths)


CASES = {
    "iemocap16_general": lambda: (*_iemocap(16, 3), 1380, 150, 150, 100, 2, "general", 0.0),
    "b400_p9_zero_rows": lambda: ([60] * 400, 60, 100, 100, 100, 100, 9, "general", 0.1),
    "odd_widths_simple": lambda: ([9, 4, 12, 1, 7], 12, 40, 33, 17, 5, 3, "simple", 0.0),
    "top_of_range": lambda: ([20, 13, 6, 20], 20, 64, 256, 256, 256, 4, "general", 0.0),
    "one_step": lambda: ([1, 1, 1], 1, 24, 16, 8, 12, 2, "general", 0.0),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_dialogue_rnn_vs_oracle(case):
    import erc_b200  # noqa: F401
    lengths, L, Dm, Dg, Dp, De, P, att, zf = CASES[case]()
    o, m, U, qm, R = _setup(lengths, L, Dm, Dg, Dp, De, P, att, seed=len(case), zero_frac=zf)
    refs = [_oracle_run(o, U, qm, R, dt) for dt in (torch.float32, torch.float64)]
    got, alpha = _ours(m, U, qm, R)
    assert len(alpha) == L - 1 and all(a.shape == (len(lengths), t + 1) for t, a in enumerate(alpha))
    assert len(got) == len(refs[0]) == 15 + (L > 1)
    parity_check("dialogue_rnn/" + case, got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
def test_dialogue_rnn_empty_batch():
    import erc_b200  # noqa: F401
    o, m, U, qm, R = _setup([], 5, 24, 16, 8, 12, 2, "general", seed=1)
    got, alpha = _ours(m, U, qm, R)
    assert got["e"].shape == (5, 0, 12) and got["dU"].shape == (5, 0, 24)
    assert len(alpha) == 4 and all(a.shape == (0, t + 1) for t, a in enumerate(alpha))
    assert all(torch.count_nonzero(v) == 0 for k, v in got.items() if k not in ("e", "dU", "alpha"))


@pytest.mark.gpu
@pytest.mark.parametrize("att", ["general", "simple"])
def test_dialogue_rnn_dropout_matches_oracle_with_the_same_masks(att):
    """p = 0.5 with explicit seeds: the oracle fed ops.dropout(ones, p, seed) as its three masks gives the same outputs
    and gradients."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    lengths, L = [14, 9, 3, 14, 11, 6], 14
    o, m, U, qm, R = _setup(lengths, L, 48, 40, 30, 20, 3, att, seed=9)
    seeds = (101, 202, 303)
    LB = L * len(lengths)
    masks = [ops.dropout(torch.ones(LB, d, device="cuda"), 0.5, s).cpu() for d, s in zip((40, 30, 20), seeds)]
    refs = [_oracle_run(o, U, qm, R, dt, masks) for dt in (torch.float32, torch.float64)]
    got, _ = _ours(m, U, qm, R, drop_p=0.5, seeds=seeds)
    parity_check("dialogue_rnn/dropout/" + att, got, refs[0], refs[1], zero_floor_frac=OWN_SCALE)


@pytest.mark.gpu
def test_dialogue_rnn_training_mode():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcnv2_models import DialogueRNN
    gen = torch.Generator().manual_seed(5)
    U = torch.randn(10, 4, 32, generator=gen).cuda()
    qm = _qmask([10, 7, 10, 2], 10, 2, gen).cuda()
    torch.manual_seed(0)
    m = DialogueRNN(32, 24, 20, 16, context_attention="general", dropout=0.5).cuda()
    with torch.no_grad():
        ev = m.eval()(U, qm)[0]
        tr = m.train()(U, qm)[0]
        assert torch.isfinite(tr).all() and not torch.equal(tr, ev)
        m.dialogue_cell.dropout.p = 0.0
        assert torch.equal(m.train()(U, qm)[0], ev)


def _fwd_bwd(m, U, qm, R, seeds):
    from erc_b200 import ops_dgcnv2
    c = m.dialogue_cell
    u = U.detach().requires_grad_(True)
    params = list(m.parameters())
    e, alpha = ops_dgcnv2.dialogue_rnn(u, qm, c.g_cell, c.p_cell, c.e_cell, c.attention.transform.weight, "general", 0.5, seeds)
    grads = torch.autograd.grad((e * R).sum(), [u] + params)
    return [e.detach(), torch.cat([a.reshape(-1) for a in alpha]), *grads]


@pytest.mark.gpu
def test_dialogue_rnn_bit_reproducible_and_graph_capturable():
    import erc_b200  # noqa: F401
    lengths, L = [30, 17, 30, 8, 22, 30, 5], 30
    o, m, U, qm, R = _setup(lengths, L, 72, 150, 150, 100, 2, "general", seed=13)
    U, qm, R = U.cuda(), qm.cuda(), R.cuda()
    seeds = (7, 8, 9)
    a = _fwd_bwd(m, U, qm, R, seeds)
    assert all(torch.equal(x, y) for x, y in zip(a, _fwd_bwd(m, U, qm, R, seeds)))
    assert all(torch.isfinite(x).all() for x in a)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _fwd_bwd(m, U, qm, R, seeds)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c = _fwd_bwd(m, U, qm, R, seeds)
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(a, c))


@pytest.mark.gpu
def test_dialogue_rnn_op_rejects_out_of_range_sizes():
    import erc_b200  # noqa: F401
    from erc_b200._lib import ErcgError
    from erc_b200.track_mm.dgcnv2_models import DialogueRNN
    gen = torch.Generator().manual_seed(2)
    for dims, P in (((8, 257, 4, 4), 2), ((8, 4, 4, 257), 2), ((8, 4, 4, 4), 17)):
        m = DialogueRNN(*dims, context_attention="general").cuda().eval()
        U = torch.randn(3, 2, 8, generator=gen).cuda()
        qm = _qmask([3, 3], 3, P, gen).cuda()
        with pytest.raises(ErcgError):
            m(U, qm)
    torch.cuda.synchronize()


def test_dialogue_rnn_state_dict_and_rejected_configurations():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcnv2_models import DialogueRNN, DialogueRNNCell, MatchingAttention
    for att, last in (("simple", ("dialogue_cell.attention.scalar.weight", (1, 150))),
                      ("general", ("dialogue_cell.attention.transform.weight", (150, 1380)))):
        m, o = DialogueRNN(1380, 150, 150, 100, context_attention=att), O.DialogueRNN(1380, 150, 150, 100, context_attention=att)
        a = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
        assert a == [(k, tuple(v.shape)) for k, v in o.state_dict().items()] and len(a) == 13 and a[-1] == last
        m.load_state_dict(o.state_dict(), strict=True)
        o.load_state_dict(m.state_dict(), strict=True)
    with pytest.raises(NotImplementedError):
        DialogueRNN(10, 8, 8, 8, listener_state=True)
    for att in ("dot", "concat", "general2"):
        with pytest.raises(NotImplementedError):
            DialogueRNN(10, 8, 8, 8, context_attention=att)
    for att in ("dot", "concat"):
        with pytest.raises(NotImplementedError):
            MatchingAttention(8, 10, att_type=att)
    assert MatchingAttention(8, 10, att_type="general").transform.bias is None
    assert MatchingAttention(8, 10, att_type="general2").transform.bias is not None
    cell = DialogueRNNCell(10, 8, 8, 8)
    with pytest.raises(NotImplementedError):
        cell(None, None, None, None, None)
    m = DialogueRNN(10, 8, 8, 8)
    for U, qm in ((torch.zeros(3, 2, 10), torch.zeros(3, 2)), (torch.zeros(3, 2, 11), torch.zeros(3, 2, 2)),
                  (torch.zeros(3, 2, 10), torch.zeros(4, 2, 2)), (torch.zeros(3, 2, 10), torch.zeros(3, 2, 2))):
        with pytest.raises(ValueError):       # wrong rank, width, length, or not on the parameters' CUDA device
            m(U, qm)


def test_dialogue_rnn_entry_points_check_sizes_on_the_host():
    """Widths outside 1..256, P outside 1..16, negative sizes and drop_p outside [0, 1) return ERCG_EINVAL before any
    launch; B == 0 or L == 0 is a no-op that touches no pointer."""
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib, DialogueRnnArgs

    def call(**kw):
        a = DialogueRnnArgs()
        a.L, a.B, a.Dg, a.Dp, a.De, a.P = 4, 2, 150, 150, 100, 2
        for k, v in kw.items():
            setattr(a, k, v)
        return lib().ercg_dialogue_rnn_fwd(ctypes.byref(a), None), lib().ercg_dialogue_rnn_bwd(ctypes.byref(a), None)

    for kw in (dict(Dg=0), dict(Dp=257), dict(De=0), dict(De=257), dict(P=17), dict(P=0), dict(L=-1), dict(B=-1),
               dict(drop_p=1.0), dict(drop_p=-0.1), {}):
        assert call(**kw) == (-1, -1), kw                     # the last: valid sizes, null pointers
    assert call(B=0) == (0, 0) and call(L=0) == (0, 0)
