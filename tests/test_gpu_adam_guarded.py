"""ercg_adam_step_guarded: with its device flag at 0 it is ercg_adam_step bit for bit (Adam / AdamW, with and without the
clip, vectorised and scalar paths); with the flag non-zero it leaves p, m, v and the step counter untouched.  The flag here is
an ordinary device int -- no peer, no time-out."""
import pytest
import torch


def _state(n, off, dev, seed):
    gen = torch.Generator(device=dev).manual_seed(seed)
    mk = lambda scale=1.0: (torch.randn(n + off, device=dev, generator=gen) * scale)[off:]   # off = 1: not 16-byte aligned
    p, g, m = mk(), mk(0.1), mk(0.01)
    v = mk(0.01).square()
    return p, g, m, v


def _step(fn, p, g, m, v, step, sumsq, decoupled, extra=()):
    from erc_b200._lib import lib
    from erc_b200.ops import _p, _stream
    return getattr(lib(), fn)(_p(p), _p(g), _p(m), _p(v), p.numel(), 1e-3, 0.9, 0.999, 1e-8, 1e-2 if decoupled else 1e-4,
                              1 if decoupled else 0, 0.5, _p(sumsq), 0.05 if sumsq is not None else 0.0, _p(step), _stream(),
                              *extra)


@pytest.mark.gpu
@pytest.mark.parametrize("off", [0, 1])
@pytest.mark.parametrize("decoupled", [False, True], ids=["adam", "adamw"])
@pytest.mark.parametrize("clip", [False, True], ids=["noclip", "clip"])
def test_guarded_step_with_zero_flag_equals_adam_step(decoupled, clip, off):
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    from erc_b200.ops import _p, _ws, _stream
    dev = torch.device("cuda", 0)
    n = 4 * 65536 + 3
    ref = _state(n, off, dev, 11)
    got = [t.clone() for t in ref]
    got = [torch.cat([torch.zeros(off, device=dev), t])[off:] for t in got]    # same alignment as ref
    step_ref = torch.full((1,), 4, dtype=torch.int64, device=dev)
    step_got = step_ref.clone()
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    sumsq = None
    if clip:
        sumsq = torch.zeros(1, device=dev)
        ws = _ws(lib().ercg_sumsq_workspace_bytes(n), dev)
        assert lib().ercg_sumsq(_p(ref[1]), n, _p(sumsq), _p(ws), ws.numel(), _stream()) == 0
    for _ in range(3):
        assert _step("ercg_adam_step", *ref, step_ref, sumsq, decoupled) == 0
        assert _step("ercg_adam_step_guarded", *got, step_got, sumsq, decoupled, (_p(flag),)) == 0
    torch.cuda.synchronize()
    assert int(step_ref.item()) == int(step_got.item()) == 7
    for a, b, name in zip(ref, got, "pgmv"):
        assert torch.equal(a, b), name
    assert not torch.equal(ref[0], _state(n, off, dev, 11)[0])           # the steps did move the parameters


@pytest.mark.gpu
@pytest.mark.parametrize("flag_value", [1, -6])                         # -6 = ERCG_P2P_ETIMEOUT, what a timed-out exchange leaves
@pytest.mark.parametrize("clip", [False, True], ids=["noclip", "clip"])
def test_guarded_step_with_nonzero_flag_changes_nothing(flag_value, clip):
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    from erc_b200.ops import _p
    dev = torch.device("cuda", 0)
    n = 4 * 4096 + 1
    state = _state(n, 0, dev, 12)
    before = [t.clone() for t in state]
    step = torch.full((1,), 9, dtype=torch.int64, device=dev)
    flag = torch.full((1,), flag_value, dtype=torch.int32, device=dev)
    sumsq = torch.ones(1, device=dev) if clip else None
    for decoupled in (False, True):
        assert _step("ercg_adam_step_guarded", *state, step, sumsq, decoupled, (_p(flag),)) == 0
    torch.cuda.synchronize()
    assert int(step.item()) == 9
    for a, b, name in zip(state, before, "pgmv"):
        assert torch.equal(a, b), name
    # a NULL flag is an argument error, not an unguarded step
    rc = _step("ercg_adam_step_guarded", *state, step, sumsq, False, (None,))
    assert rc != 0 and lib().ercg_strerror(rc)


@pytest.mark.gpu
def test_flat_adam_uses_the_guarded_step_when_given_a_flag():
    import erc_b200  # noqa: F401
    from erc_b200.optim import FlatAdam
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    ws = [torch.nn.Parameter(torch.randn(37, 5, device=dev)) for _ in range(2)]
    opt = FlatAdam(ws, lr=1e-2)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    opt.skip_if_nonzero = flag.data_ptr()
    start = [w.detach().clone() for w in ws]
    for w in ws:
        w.grad = torch.ones_like(w)
    opt.step()
    moved = [w.detach().clone() for w in ws]
    assert not any(torch.equal(m, s) for m, s in zip(moved, start)) and int(opt.step_dev.item()) == 1
    flag.fill_(1)
    opt.step()
    torch.cuda.synchronize()
    assert int(opt.step_dev.item()) == 1 and all(torch.equal(w.detach(), m) for w, m in zip(ws, moved))
