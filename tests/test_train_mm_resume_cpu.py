"""Checkpoint state handling on CPU tensors: FlatAdam's torch.optim-form state (torch_state_dict / load_state_dict) against
torch.optim.Adam / AdamW, and train_mm's --load / --resume helpers on the reference trainer's checkpoint layout
({'models': {'model': sd}, 'optims': ..., 'others': ..., 'thtensor': ..., 'nptensor': ...}) for all five modules.
FlatAdam only lays out its flat buffers here (attach() after a backward); nothing calls a kernel."""
import pytest
import torch

MODULES = ("cogmen", "dgcn", "dgcnv2", "mmgcn", "dagerc")


def _net(seed):
    torch.manual_seed(seed)
    net = torch.nn.Sequential(torch.nn.Linear(7, 6), torch.nn.Tanh(), torch.nn.Linear(6, 3))
    dead = torch.nn.Parameter(torch.ones(5))                 # never gets a gradient, like the reference's dead encoder
    return list(net.parameters()) + [dead], net


NAMES = ["0.weight", "0.bias", "2.weight", "2.bias", "dead"]


def _backward(net, seed):
    for p in net.parameters():
        p.grad = None
    x = torch.randn(4, 7, generator=torch.Generator().manual_seed(seed))
    net(x).square().sum().backward()


def _torch_optim(decoupled, params):
    cls = torch.optim.AdamW if decoupled else torch.optim.Adam
    return cls(params, lr=3e-3, weight_decay=1e-2)


def _flat(decoupled, params):
    from erc_b200.optim import FlatAdam
    return FlatAdam(params, lr=3e-3, weight_decay=1e-2, decoupled=decoupled)


def _trained_torch(decoupled, steps=3, named=False):
    """A torch.optim optimizer after ``steps`` steps (the last parameter never has a gradient)."""
    params, net = _net(0)
    opt = _torch_optim(decoupled, list(zip(NAMES, params)) if named else params)
    for s in range(steps):
        _backward(net, s)
        opt.step()
    return opt, params, net


def _attached_flat(decoupled, seed=0):
    import erc_b200  # noqa: F401
    params, net = _net(seed)
    flat = _flat(decoupled, params)
    _backward(net, 0)
    return flat.attach(), params, net


def _same(a, b, path="sd"):
    """Exact equality of nested state dicts: keys, types, tensor dtypes / shapes / devices / values."""
    assert type(a) is type(b), (path, type(a), type(b))
    if isinstance(a, dict):
        assert list(a) == list(b), (path, list(a), list(b))
        for k in a:
            _same(a[k], b[k], "%s[%r]" % (path, k))
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, "%s[%d]" % (path, i))
    elif isinstance(a, torch.Tensor):
        assert (a.dtype, a.shape, a.device) == (b.dtype, b.shape, b.device), (path, a.dtype, b.dtype, a.shape, b.shape)
        assert torch.equal(a, b), path
    else:
        assert a == b, (path, a, b)


@pytest.mark.parametrize("decoupled", [False, True])
@pytest.mark.parametrize("named", [False, True])
def test_torch_state_dict_is_torch_optims(decoupled, named):
    ref, _, _ = _trained_torch(decoupled, named=named)
    want = ref.state_dict()
    flat, _, _ = _attached_flat(decoupled)
    for i, p in enumerate(flat.live):                        # the same moments and step in the flat buffers
        k, off = p.numel(), flat.offsets[i]
        flat.m[off:off + k].copy_(want["state"][i]["exp_avg"].reshape(-1))
        flat.v[off:off + k].copy_(want["state"][i]["exp_avg_sq"].reshape(-1))
    flat.step_dev.fill_(3)
    got = flat.torch_state_dict(NAMES if named else None)
    assert 4 not in got["state"]                             # the parameter without a gradient has no state
    _same(got, want)


def test_torch_state_dict_before_the_first_step_is_empty():
    import erc_b200  # noqa: F401
    params, _ = _net(0)
    assert _flat(False, params).torch_state_dict()["state"] == {}
    flat, _, _ = _attached_flat(False)
    assert flat.torch_state_dict()["state"] == {}


@pytest.mark.parametrize("decoupled", [False, True])
@pytest.mark.parametrize("before_attach", [True, False])
def test_torch_form_round_trips_exactly(decoupled, before_attach):
    # torch form -> FlatAdam -> torch form
    ref, _, _ = _trained_torch(decoupled, named=True)
    want = ref.state_dict()
    params, net = _net(1)
    flat = _flat(decoupled, params)
    flat.lr = 99.0                                           # hyper-parameters come from the loaded state
    if before_attach:
        flat.load_state_dict(want, NAMES)
        _same(flat.torch_state_dict(NAMES), want)           # the kept state is already visible in torch form
    _backward(net, 0)
    flat.attach()
    if not before_attach:
        flat.load_state_dict(want, NAMES)
    assert flat.lr == 3e-3 and flat.decoupled == decoupled
    _same(flat.torch_state_dict(NAMES), want)
    # FlatAdam -> torch form -> FlatAdam: the flat buffers (padding included) come back bit for bit
    params2, net2 = _net(2)
    other = _flat(decoupled, params2)
    other.load_state_dict(flat.torch_state_dict())           # by index
    _backward(net2, 0)
    other.attach()
    assert other.n == flat.n and torch.equal(other.m, flat.m) and torch.equal(other.v, flat.v)
    assert int(other.step_dev) == int(flat.step_dev) == 3


def test_flat_form_still_loads():
    flat, _, _ = _attached_flat(True)
    flat.m.uniform_()
    flat.v.uniform_()
    flat.step_dev.fill_(11)
    sd = flat.state_dict()
    params, net = _net(3)
    other = _flat(False, params)
    other.load_state_dict(sd)
    _backward(net, 0)
    other.attach()
    assert torch.equal(other.m, flat.m) and torch.equal(other.v, flat.v) and int(other.step_dev) == 11 and other.decoupled


@pytest.mark.parametrize("decoupled", [False, True])
def test_torch_optim_continues_from_the_exported_state(decoupled):
    """torch.optim.Adam.load_state_dict(flat.torch_state_dict()) + one step == one step from the original torch state."""
    ref, params, net = _trained_torch(decoupled)
    flat, _, _ = _attached_flat(decoupled)
    flat.load_state_dict(ref.state_dict())
    params2, net2 = _net(0)
    with torch.no_grad():
        for a, b in zip(params2, params):
            a.copy_(b)
    again = _torch_optim(decoupled, params2)
    again.load_state_dict(flat.torch_state_dict())
    for n_, o in ((net, ref), (net2, again)):
        _backward(n_, 7)
        o.step()
    for a, b in zip(params2, params):
        assert torch.equal(a, b)


def _state_of(decoupled=False):
    ref, _, _ = _trained_torch(decoupled, named=True)
    return ref.state_dict()


@pytest.mark.parametrize("before_attach", [True, False])
def test_state_for_a_parameter_without_gradient_is_refused(before_attach):
    sd = _state_of()
    sd["state"][4] = {"step": torch.tensor(3.0), "exp_avg": torch.zeros(5), "exp_avg_sq": torch.zeros(5)}
    params, net = _net(0)
    flat = _flat(False, params)
    with pytest.raises(ValueError, match="receive no gradient: dead"):
        if before_attach:
            flat.load_state_dict(sd, NAMES)
        _backward(net, 0)
        flat.attach()
        flat.load_state_dict(sd, NAMES)


@pytest.mark.parametrize("before_attach", [True, False])
def test_live_parameter_without_state_is_refused(before_attach):
    sd = _state_of()
    del sd["state"][1]
    params, net = _net(0)
    flat = _flat(False, params)
    with pytest.raises(ValueError, match=r"no state for parameters that receive a gradient: 0\.bias"):
        if before_attach:
            flat.load_state_dict(sd, NAMES)
        _backward(net, 0)
        flat.attach()
        flat.load_state_dict(sd, NAMES)


def test_no_state_at_all_is_a_fresh_start():
    sd = _state_of()
    sd["state"] = {}
    flat, _, _ = _attached_flat(False)
    flat.m.fill_(1.0)
    flat.step_dev.fill_(5)
    flat.load_state_dict(sd, NAMES)
    assert int(flat.step_dev) == 0 and not flat.m.any() and flat.torch_state_dict()["state"] == {}


def test_shape_mismatch_is_refused():
    sd = _state_of()
    sd["state"][2]["exp_avg"] = torch.zeros(3, 5)
    params, _ = _net(0)
    with pytest.raises(ValueError, match=r"shapes differ: 2\.weight: exp_avg \(3, 5\)"):
        _flat(False, params).load_state_dict(sd, NAMES)
    sd = _state_of()
    sd["param_groups"][0]["param_names"] = ["0.weight", "0.bias", "2.bias", "2.weight", "dead"]    # names say otherwise
    with pytest.raises(ValueError, match="shapes differ"):
        _flat(False, params).load_state_dict(sd, NAMES)
    sd = _state_of()
    sd["param_groups"][0]["params"].append(5)                # by index: the parameter count must match
    del sd["param_groups"][0]["param_names"]
    with pytest.raises(ValueError, match="6 parameters, this optimizer 5"):
        _flat(False, params).load_state_dict(sd)


def test_unequal_steps_are_refused():
    sd = _state_of()
    sd["state"][3]["step"] = torch.tensor(2.0)
    params, _ = _net(0)
    with pytest.raises(ValueError, match="step differs between parameters.*2.bias=2"):
        _flat(False, params).load_state_dict(sd, NAMES)


def test_state_for_an_unknown_name_is_refused():
    sd = _state_of()
    sd["param_groups"][0]["param_names"][1] = "gone.bias"
    params, _ = _net(0)
    with pytest.raises(ValueError, match="does not have: gone.bias"):
        _flat(False, params).load_state_dict(sd, NAMES)


# ------------------------------------------------------------------------------------------------ train_mm helpers
def _params(module, *extra):
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import parse_args, resolve_params
    return resolve_params(parse_args(["--module=" + module, "--dataset=iemocap-cogmen-6"] + list(extra)))


def _reference_module(module):
    """The module as the reference builds it (COGMEN with its dead TransformerEncoder), weights randomised."""
    from erc_b200.train_mm import build_model
    m = build_model(dict(_params(module), dead_encoder=True), torch.device("cpu"))
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        for t in m.state_dict().values():
            if t.is_floating_point():
                t.copy_(torch.randn(t.shape, generator=g))
    return m


def _lumo(ref, optim_sd=None):
    """A checkpoint in the reference trainer's layout, saved by an accelerate-wrapped model (``module.`` keys)."""
    return {"models": {"model": {"module." + k: v.clone() for k, v in ref.state_dict().items()}},
            "optims": {"optim": optim_sd} if optim_sd is not None else {}, "others": {}, "thtensor": {}, "nptensor": {}}


@pytest.mark.parametrize("module", MODULES)
def test_load_reads_a_reference_checkpoint(module):
    from erc_b200.train_mm import build_model, load_model_weights
    ref = _reference_module(module)
    ours = build_model(_params(module), torch.device("cpu"))
    lines = []
    ignored = load_model_weights(ours, _lumo(ref), log=lines.append)
    want = ref.state_dict()
    for k, v in ours.state_dict().items():
        assert torch.equal(v, want[k]), k
    dead = [k for k in want if k.startswith("rnn.0.")]
    assert ignored == dead and (module == "cogmen") == bool(dead)
    assert bool(lines) == bool(dead) and all(k in lines[0] for k in dead)
    # the plain state_dict layout loads the same way
    fresh = build_model(_params(module), torch.device("cpu"))
    load_model_weights(fresh, ours.state_dict(), log=lines.append)
    assert all(torch.equal(v, want[k]) for k, v in fresh.state_dict().items())


def test_load_needs_every_key_of_the_module():
    from erc_b200.train_mm import build_model, load_model_weights
    ck = _lumo(_reference_module("dgcn"))
    key = next(iter(ck["models"]["model"]))
    del ck["models"]["model"][key]
    with pytest.raises(SystemExit, match="lacks 1 of the module's keys: " + key[len("module."):]):
        load_model_weights(build_model(_params("dgcn"), torch.device("cpu")), ck)


def _reference_adam_state(ref, live_names, step=4):
    """torch.optim.Adam's state_dict over the reference module's parameters() (no param_names, as torch.optim writes it
    for a plain parameter list), with state for ``live_names`` only."""
    params = list(ref.parameters())
    opt = torch.optim.Adam(params, lr=3e-4)
    g = torch.Generator().manual_seed(9)
    for name, p in ref.named_parameters():
        if name in live_names:
            opt.state[p] = {"step": torch.tensor(float(step)), "exp_avg": torch.randn(p.shape, generator=g),
                            "exp_avg_sq": torch.rand(p.shape, generator=g)}
    return opt.state_dict()


@pytest.mark.parametrize("module", ["cogmen", "dagerc"])
def test_reference_optimizer_state_maps_by_the_reference_parameter_list(module):
    from erc_b200.optim import FlatAdam
    from erc_b200.train_mm import build_model, load_reference_optim
    p = _params(module)
    ref = _reference_module(module)
    ours = build_model(p, torch.device("cpu"))
    names = [k for k, _ in ours.named_parameters()]
    sd = _reference_adam_state(ref, set(names))
    flat = FlatAdam(ours.parameters(), lr=1.0)
    lines = []
    assert load_reference_optim(flat, _lumo(ref, sd), p, names, log=lines.append) and not lines
    for t in ours.parameters():
        t.grad = torch.zeros_like(t)
    flat.attach()
    by_name = dict(zip([k for k, _ in ref.named_parameters()], range(len(sd["param_groups"][0]["params"]))))
    got = flat.torch_state_dict(names)
    assert flat.lr == 3e-4 and int(flat.step_dev) == 4 and len(got["state"]) == len(names)
    for i, name in enumerate(names):
        assert torch.equal(got["state"][i]["exp_avg"], sd["state"][by_name[name]]["exp_avg"]), name
        assert torch.equal(got["state"][i]["exp_avg_sq"], sd["state"][by_name[name]]["exp_avg_sq"]), name


def test_unmappable_reference_optimizer_state_loads_weights_only():
    from erc_b200.optim import FlatAdam
    from erc_b200.train_mm import build_model, load_reference_optim
    p = _params("cogmen")
    ref = _reference_module("cogmen")
    ours = build_model(p, torch.device("cpu"))
    names = [k for k, _ in ours.named_parameters()]
    sd = _reference_adam_state(ref, set(names))
    sd["param_groups"][0]["params"] = sd["param_groups"][0]["params"][:-1]      # one index short of the module's list
    flat = FlatAdam(ours.parameters(), lr=1.0)
    lines = []
    assert not load_reference_optim(flat, _lumo(ref, sd), p, names, log=lines.append)
    assert "weights only" in lines[0] and flat.lr == 1.0
    lines.clear()
    assert not load_reference_optim(flat, _lumo(ref), p, names, log=lines.append)
    assert "no optimizer state" in lines[0]


def test_resume_refuses_another_run():
    from erc_b200.train_mm import check_resumable, run_params
    p = _params("dgcn")
    ck = {"models": {"model": {}}, "optims": {}, "others": {"train_mm": {"params": run_params(p, 1)}}, "thtensor": {},
          "nptensor": {}}
    check_resumable(ck, p, 1, "x.ckpt")
    with pytest.raises(SystemExit, match=r"batch_size=4 \(checkpoint: 32\)"):
        check_resumable(ck, _params("dgcn", "--train.batch_size=4"), 1, "x.ckpt")
    with pytest.raises(SystemExit, match=r"world=2 \(checkpoint: 1\)"):
        check_resumable(ck, p, 2, "x.ckpt")
    with pytest.raises(SystemExit, match="module='mmgcn'"):
        check_resumable(ck, _params("mmgcn"), 1, "x.ckpt")
    with pytest.raises(SystemExit, match="plain state_dict"):
        check_resumable({"w": torch.zeros(1)}, p, 1, "x.ckpt")


def test_checkpoint_options_are_checked():
    with pytest.raises(SystemExit, match="ckpt_layout"):
        _params("dgcn", "--ckpt_layout=lumo")
    with pytest.raises(SystemExit, match="exclude each other"):
        _params("dgcn", "--resume=a.ckpt", "--load=b.ckpt")
    p = _params("dgcn")
    assert p["ckpt_layout"] == "state_dict" and p["resume"] is None and p["load"] is None
