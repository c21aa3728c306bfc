"""CPU checks of the sequence classifiers of track_mm/dgcnv2_models.py: the oracle (oracle/dgcnv2_seq_oracle.py) against the
real declare-lab classes when the reference tree is present, state_dict layouts, the refusals that stay pinned, and the
host-side size checks of the new entry points (K13, the sequence reversal, log-softmax)."""
import copy
import ctypes

import pytest
import torch

from oracle import dgcnv2_seq_oracle as O
from oracle import ref_loader


def _batch(lengths, L, Dm, P, gen):
    B = len(lengths)
    inside = torch.arange(L)[:, None] < torch.tensor(lengths)[None, :]
    U = torch.randn(L, B, Dm, generator=gen, dtype=torch.float64) * inside[..., None]
    qm = torch.nn.functional.one_hot(torch.randint(0, P, (L, B), generator=gen), P).double() * inside[..., None]
    return U, qm, inside.t().double().contiguous()


def _run(m, U, qm, umask, att2):
    u = U.clone().requires_grad_(True)
    log_prob, alpha, alpha_f, alpha_b = m(u, qm, umask, att2)
    log_prob.sum().backward()
    return [log_prob.detach(), u.grad, *[a.detach() for a in alpha + alpha_f + alpha_b],
            *[p.grad for _, p in sorted(m.named_parameters()) if p.grad is not None]]


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not found (ERC_REFERENCE_ROOT): the oracle is checked "
                                                       "against the real declare-lab classes only where they exist")
@pytest.mark.parametrize("name,args", [("LSTMModel", (20, 8, 6)), ("GRUModel", (20, 8, 6)),
                                       ("DialogRNNModel", (20, 12, 10, 8, 6))])
@pytest.mark.parametrize("att2", [True, False])
def test_oracle_equals_the_reference_classes(name, args, att2):
    ref = ref_loader.load_dgcnv2().dgcnv2_models
    torch.manual_seed(0)
    r = getattr(ref, name)(*args, n_classes=5, dropout=0.0).double().eval()
    o = getattr(O, name)(*args, n_classes=5, dropout=0.0).double().eval()
    assert set(r.state_dict()) == set(o.state_dict())
    o.load_state_dict(r.state_dict(), strict=True)
    U, qm, umask = _batch([7, 4, 7, 2], 7, 20, 2, torch.Generator().manual_seed(1))
    for a, b in zip(_run(r, U, qm, umask, att2), _run(o, U, qm, umask, att2)):
        assert torch.equal(a, b)
    for att_type in ("general", "general2"):
        ra, oa = ref.MatchingAttention(8, 6, att_type=att_type).double(), O.MatchingAttention(8, 6, att_type=att_type).double()
        oa.load_state_dict(ra.state_dict(), strict=True)
        M, x = torch.randn(5, 3, 8, dtype=torch.float64), torch.randn(3, 6, dtype=torch.float64)
        for mask in (None, umask[:3, :5], torch.rand(3, 5, dtype=torch.float64)):
            assert all(torch.equal(p, q) for p, q in zip(ra(M, x, mask), oa(M, x, mask)))


def test_state_dicts_match_the_oracle_and_refusals_stay():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm import dgcnv2_models as ours
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    for name, args in (("LSTMModel", (1380, 100, 100)), ("GRUModel", (1380, 150, 100)),
                       ("DialogRNNModel", (1380, 150, 150, 100, 100))):
        for kw in ({}, {"context_attention": "general"}) if name == "DialogRNNModel" else ({},):
            m, o = getattr(ours, name)(*args, **kw), getattr(O, name)(*args, **kw)
            assert [(k, v.shape) for k, v in m.state_dict().items()] == [(k, v.shape) for k, v in o.state_dict().items()]
            m.load_state_dict(o.state_dict(), strict=True)
    d = ours.DialogRNNModel(10, 8, 8, 8, 4, dropout=0.2)
    assert d.dropout.p == 0.2 and abs(d.dropout_rec.p - 0.35) < 1e-12
    with pytest.raises(NotImplementedError):
        DGCNModule("DialogRNN")
    with pytest.raises(NotImplementedError):
        ours.DialogRNNModel(10, 8, 8, 8, 4, listener_state=True)
    for att in ("dot", "concat"):
        with pytest.raises(NotImplementedError):
            ours.MatchingAttention(8, 8, att_type=att)
    with pytest.raises(NotImplementedError):
        ours.DialogueRNNCell(10, 8, 8, 8)(None, None, None, None, None)


def test_models_check_their_inputs_before_any_launch():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm import dgcnv2_models as ours
    ma = ours.MatchingAttention(8, 6, att_type="general2")
    for M, x, mask in ((torch.zeros(5, 3, 8), torch.zeros(3, 6), None),                 # parameters not on a CUDA device
                       (torch.zeros(5, 3, 7), torch.zeros(3, 6), None), (torch.zeros(5, 3, 8), torch.zeros(2, 6), None),
                       (torch.zeros(5, 3, 8), torch.zeros(3, 6), torch.ones(3, 4))):
        with pytest.raises(ValueError):
            ma(M, x, mask)
    m = ours.LSTMModel(10, 8, 6)
    for U, qm, um in ((torch.zeros(4, 2, 10), torch.zeros(4, 2, 2), torch.ones(2, 4)),
                      (torch.zeros(4, 2, 11), torch.zeros(4, 2, 2), torch.ones(2, 4)),
                      (torch.zeros(4, 2, 10), torch.zeros(3, 2, 2), torch.ones(2, 4)),
                      (torch.zeros(4, 2, 10), torch.zeros(4, 2, 2), torch.ones(4, 2)),
                      (torch.zeros(4, 2, 10), torch.zeros(4, 2, 2), None)):
        with pytest.raises(ValueError):
            m(U, qm, um)


def test_entry_points_check_sizes_on_the_host():
    """Invalid sizes return ERCG_EINVAL (-1) before touching a pointer; B == 0 (rows == 0) returns 0."""
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    f, b = lib().ercg_match_att_fwd, lib().ercg_match_att_bwd

    def call(L=4, B=2, D=8, Q=4, ldm=None, ldq=None, kind=1):
        ldm = D if ldm is None else ldm
        ldq = D if ldq is None else ldq
        return (f(None, ldm, L, B, D, Q, None, ldq, None, kind, None, D, None, None, None),
                b(None, ldm, L, B, D, Q, None, ldq, None, kind, None, None, None, D, None, None, D, None, D, None))

    for kw in (dict(D=0), dict(D=1025), dict(L=0), dict(L=4097), dict(Q=0), dict(Q=4097), dict(B=-1), dict(kind=2),
               dict(kind=-1), dict(ldm=7), dict(ldq=7), {}):
        assert call(**kw) == (-1, -1), kw                                   # the last: valid sizes, null pointers
    for kw in (dict(B=0), dict(B=0, D=1, L=1, Q=1), dict(B=0, D=1024, L=4096, Q=4096), dict(B=0, kind=0)):
        assert call(**kw) == (0, 0), kw
    rev = lib().ercg_reverse_seq
    assert rev(None, 8, 4, 2, 8, None, None, 8, 4, None) == -1
    assert rev(None, 8, -1, 2, 8, None, None, 8, 4, None) == -1 and rev(None, 7, 4, 2, 8, None, None, 8, 4, None) == -1
    assert rev(None, 8, 4, 0, 8, None, None, 8, 4, None) == 0 and rev(None, 8, 4, 2, 8, None, None, 8, 0, None) == 0
    lf, lb = lib().ercg_log_softmax_fwd, lib().ercg_log_softmax_bwd
    assert lf(None, 7, None, 7, 3, 7, None) == -1 and lf(None, 7, None, 7, 3, 0, None) == -1 and lf(None, 7, None, 7, -1, 7, None) == -1
    assert lf(None, 7, None, 7, 0, 7, None) == 0
    assert lb(None, 7, None, 7, None, 7, 3, 7, None) == -1 and lb(None, 7, None, 7, None, 7, 0, 7, None) == 0


def test_oracle_general2_formula():
    """The oracle's 'general2' is the formula of the spec for a float mask, and an all-zero mask row gives NaN."""
    gen = torch.Generator().manual_seed(3)
    o = O.MatchingAttention(6, 6, att_type="general2").double()
    M, x = torch.randn(5, 2, 6, generator=gen, dtype=torch.float64), torch.randn(2, 6, generator=gen, dtype=torch.float64)
    mask = torch.rand(2, 5, generator=gen, dtype=torch.float64)
    pool, alpha = o(M, x, mask)
    xq = o.transform(x)
    for b in range(2):
        m = mask[b]
        s = m * ((m[:, None] * M[:, b]) @ xq[b])
        p = torch.softmax(torch.tanh(s), 0)
        a = p * m / (p * m).sum()
        assert torch.allclose(alpha[b, 0], a, atol=1e-14) and torch.allclose(pool[b], a @ M[:, b], atol=1e-13)
    mask[1] = 0
    assert torch.isnan(o(M, x, mask)[0][1]).all()
