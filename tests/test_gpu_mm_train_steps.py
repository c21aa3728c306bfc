"""MMGCN and DAG-ERC as one captured train step each: the device-seeded GCNII / ReLU-dropout entries, MmgcnTrainStep and
DagercTrainStep against train_mm's module path (module forward + ops.cross_entropy + FlatAdam), replay against eager, fresh
and non-colliding dropout masks per replay, a batch sharded by dialogue against the whole batch, and the peer-memory payload
of each step (mmgcn.py:141-157, dagerc.py:217-237)."""
import copy
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

from conftest import ROOT, check_grads, rel_err

pytestmark = pytest.mark.gpu

C = 6
MMGCN_DIMS = dict(text=768, audio=100, visual=512)         # SURVEY.md config 3
DAG_EMB = 1380                                               # SURVEY.md config 4


# ------------------------------------------------------------------------------------------ batches and models
def _mmgcn_batch(seed, B=16):
    """Seq-first padded text / audio / visual (zero padding), one-hot speakers [Lmax, B, 2], packed labels [N]."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    gen = torch.Generator().manual_seed(seed)
    lens = synth.iemocap_lengths(B, gen)
    Lmax, N = int(lens.max()), int(lens.sum())
    mask = (torch.arange(Lmax)[:, None] < lens[None, :]).float()[..., None]          # [Lmax, B, 1]
    feats = {k: torch.randn(Lmax, B, d, generator=gen) * mask for k, d in MMGCN_DIMS.items()}
    spk = torch.nn.functional.one_hot(torch.randint(0, 2, (Lmax, B), generator=gen), 2).float() * mask
    return dict(lengths=lens, spk=spk, label=torch.randint(0, C, (N,), generator=gen), **feats)


def _mmgcn(seed, dropout=True):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.mmgcn import MMGCNModule
    torch.manual_seed(seed)
    m = MMGCNModule(hidden_text=768, hidden_visual=512, hidden_audio=100, n_speakers=2, n_classes=C).cuda()
    m.train()
    if not dropout:
        m.lstm_l.dropout = 0.0
        m.graph_model.graph_net.dropout = 0.0
        m.dropout_.p = 0.0
    return m


def _mm_feats(b, cols=None, lmax=None):
    """(text, audio, visual) on the GPU, optionally the dialogues ``cols`` padded to ``lmax``."""
    out = []
    for k in ("text", "audio", "visual"):
        t = b[k]
        if cols is not None:
            t = t[:lmax, cols]
        out.append(t.contiguous().cuda())
    return tuple(out)


def _dag_batch(seed, B=16):
    """Batch-first padded input_tensor [B, Lmax, 1380], one-hot speakers [B, Lmax, 2], labels [B, Lmax] (-100 at padding)."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    gen = torch.Generator().manual_seed(seed)
    lens = synth.iemocap_lengths(B, gen)
    Lmax = int(lens.max())
    mask = torch.arange(Lmax)[None, :] < lens[:, None]
    x = torch.randn(B, Lmax, DAG_EMB, generator=gen) * mask[..., None]
    spk = torch.nn.functional.one_hot(torch.randint(0, 2, (B, Lmax), generator=gen), 2).float() * mask[..., None]
    y = torch.randint(0, C, (B, Lmax), generator=gen).masked_fill(~mask, -100)
    return dict(lengths=lens, x=x, spk=spk, label=y, mask=mask)


def _dagerc(seed, dropout=0.0):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dagerc import DAGERCModule
    torch.manual_seed(seed)
    m = DAGERCModule(emb_dim=DAG_EMB, dropout=dropout, gnn_layers=4, n_classes=C).cuda()
    m.train()
    return m


def _grads(m):
    return {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters() if p.grad is not None}


def _params(m):
    return {k: p.detach().cpu().clone() for k, p in m.named_parameters()}


# ------------------------------------------------------------------------------------------ device-seeded entries
def test_device_seeded_gcnii_and_relu_dropout_equal_the_host_seeded_entries():
    import erc_b200  # noqa: F401
    from erc_b200 import ops, ops_mmgcn
    from erc_b200._lib import lib
    gen = torch.Generator(device="cuda").manual_seed(0)
    M, H, p, seed = 2411, 200, 0.4, 0x1234_5678_9ABC
    hi, h0 = torch.randn(M, H, device="cuda", generator=gen), torch.randn(M, H, device="cuda", generator=gen)
    W = torch.randn(2 * H, H, device="cuda", generator=gen) * 0.05
    word = torch.zeros(1, dtype=torch.int64, device="cuda")
    for w in (0, 1, 7, 1 << 33):
        word.fill_(w)
        got = ops_mmgcn._layer_fwd(hi, h0, W, 0.3, 0.1, True, p, seed, word)
        assert torch.equal(got, ops_mmgcn._layer_fwd(hi, h0, W, 0.3, 0.1, True, p, seed + w))
        if w:
            assert not torch.equal(got, ops_mmgcn._layer_fwd(hi, h0, W, 0.3, 0.1, True, p, seed))
    n = 1_000_003
    x = torch.randn(n, device="cuda", generator=gen)

    def relu_drop(s, wd=None):
        out = torch.empty_like(x)
        if wd is None:
            assert lib().ercg_relu_dropout(x.data_ptr(), out.data_ptr(), n, p, s & (2 ** 64 - 1), None) == 0
        else:
            assert lib().ercg_relu_dropout_dev(x.data_ptr(), out.data_ptr(), n, p, s, wd.data_ptr(), None) == 0
        return out

    for w in (0, 1, 123456789):
        word.fill_(w)
        assert torch.equal(relu_drop(seed, word), relu_drop(seed + w))
    # through GCNII_lyc (input dropout + the stack): the forward stores the word on ctx, so the backward re-applies the
    # forward's masks whether or not ops.SEED_DEV is still set when it runs
    from erc_b200.track_mm.mmgcn_models import BlockAdjacency, BlockLayout, GCNII_lyc
    from erc_b200.track_mm.mmgcn_utils import lengths_graph
    lens = torch.tensor([40, 35, 25])
    layout = BlockLayout(lengths_graph(lens, "cuda"), 3, lens)
    feats = torch.randn(300, H, device="cuda", generator=gen)
    ahat = ops_mmgcn.big_adj(feats, layout).detach()
    dout = torch.randn(300, 2 * H, device="cuda", generator=gen)

    def run(w, keep_during_backward):
        torch.manual_seed(5)
        g = GCNII_lyc(nfeat=H, nlayers=3, nhidden=H, nclass=C, dropout=p, lamda=0.5, alpha=0.1, variant=True,
                      return_feature=True, use_residue=True).cuda().train()
        xr = feats.clone().requires_grad_()
        if w is not None:
            word.fill_(w)
            ops.SEED_DEV = word
        try:
            torch.manual_seed(11)                               # the host seed GCNII_lyc draws
            out = g(xr, None, None, BlockAdjacency(ahat, layout))
            if not keep_during_backward:
                ops.SEED_DEV = None
            out.backward(dout)
        finally:
            ops.SEED_DEV = None
        return out.detach(), xr.grad, {k: q.grad for k, q in g.named_parameters() if q.grad is not None}

    o_host, _, _ = run(None, False)
    o0, _, _ = run(0, False)
    assert torch.equal(o0[:, :H], o_host[:, :H])               # word 0: the input dropout's mask is the host path's
    o5, gx5, gw5 = run(5, False)
    o5b, gx5b, gw5b = run(5, True)
    assert not torch.equal(o5, o0) and torch.equal(o5, o5b) and torch.equal(gx5, gx5b)
    assert all(torch.equal(gw5[k], gw5b[k]) for k in gw5)
    dropped = (o5[:, :H] == 0) & (feats != 0)                  # the input dropout zeroed these: no gradient reaches them
    assert bool(dropped.any()) and float(gx5[dropped].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------ eager step vs module path
def _mm_module_arm(m, b, steps):
    """train_mm's MMGCN step: MMGCNModule.forward on the padded batch + ops.cross_entropy + FlatAdam (mmgcn.py's Adam)."""
    from erc_b200 import ops
    from erc_b200.optim import FlatAdam
    opt = FlatAdam(m.parameters(), lr=3e-4, weight_decay=3e-5)
    t, a, v = _mm_feats(b)
    q, y = b["spk"].cuda(), b["label"].cuda()
    out = []
    for _ in range(steps):
        loss = ops.cross_entropy(m(text_feature=t, audio_feature=a, visual_feature=v, speaker_tensor=q,
                                   text_length=b["lengths"])[0], y)
        opt.zero_grad()
        loss.backward()
        out.append((float(loss), _grads(m)))
        opt.step()
    return out


def _dag_module_arm(m, b, steps, max_norm=5.0):
    """train_mm's DAG-ERC step: DAGERCModule.forward, logits[attention_mask] + ops.cross_entropy + FlatAdam (AdamW + clip)."""
    from erc_b200 import ops
    from erc_b200.optim import FlatAdam
    opt = FlatAdam(m.parameters(), lr=1e-3, weight_decay=1e-2, decoupled=True, max_norm=max_norm)
    x, q, mask = b["x"].cuda(), b["spk"].cuda(), b["mask"].cuda()
    y = b["label"].cuda()[mask]
    out = []
    for _ in range(steps):
        logits = m(input_tensor=x, text_length=b["lengths"], speaker_tensor=q)[0][mask]
        loss = ops.cross_entropy(logits, y)
        opt.zero_grad()
        loss.backward()
        out.append((float(loss), _grads(m)))
        opt.step()
    return out


def _assert_same_run(step_run, module_run, tol=1e-6):
    for (l1, g1), (l0, g0) in zip(step_run, module_run):
        assert abs(l1 - l0) <= tol * abs(l0), (l1, l0)
        assert set(g1) == set(g0)
        for k in g0:
            assert rel_err(g1[k], g0[k], floor=1e-2 * max(float(v.abs().max()) for v in g0.values())) <= tol, k


@pytest.mark.parametrize("which", ["mmgcn", "dagerc"])
def test_eager_step_equals_the_module_path(which):
    from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep
    steps = 3
    if which == "mmgcn":
        b = _mmgcn_batch(0)
        m0, m1 = _mmgcn(1, dropout=False), _mmgcn(1, dropout=False)
        want = _mm_module_arm(m0, b, steps)
        ts = MmgcnTrainStep(m1, b["lengths"])
        args = (_mm_feats(b), b["spk"].cuda(), b["label"].cuda())
    else:
        b = _dag_batch(0)
        m0, m1 = _dagerc(1), _dagerc(1)
        want = _dag_module_arm(m0, b, steps)
        ts = DagercTrainStep(m1, b["lengths"])
        args = (b["x"].cuda(), b["spk"].cuda(), b["label"].cuda())
    got = []
    for _ in range(steps):
        loss = float(ts.step(*args))
        got.append((loss, _grads(m1)))
    ts.check()
    _assert_same_run(got, want)
    p0, p1 = _params(m0), _params(m1)
    for k in p0:
        assert rel_err(p1[k], p0[k]) <= 1e-6, k
    assert got[-1][0] < got[0][0]


# ------------------------------------------------------------------------------------------ replay vs eager
def _refill(args, new):
    for a, n in zip(args, new):
        if isinstance(a, tuple):
            _refill(a, n)
        elif a is not None:
            a.copy_(n)


@pytest.mark.parametrize("which", ["mmgcn", "dagerc"])
def test_replay_equals_eager_bit_for_bit(which):
    from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep
    if which == "mmgcn":
        b, b2 = _mmgcn_batch(0), _mmgcn_batch(0)
        gen = torch.Generator().manual_seed(9)                 # new features / speakers / labels, same lengths
        for k in ("text", "audio", "visual"):
            b2[k] = torch.randn(b2[k].shape, generator=gen) * (b2[k] != 0).any(-1, keepdim=True)
        b2["label"] = torch.randint(0, C, b2["label"].shape, generator=gen)
        m0 = _mmgcn(3, dropout=False)
        mk = (lambda m: MmgcnTrainStep(m, b["lengths"]))
        mkargs = (lambda bb: (_mm_feats(bb), bb["spk"].cuda(), bb["label"].cuda()))
    else:
        b, b2 = _dag_batch(0), _dag_batch(0)
        gen = torch.Generator().manual_seed(9)
        b2["x"] = torch.randn(b2["x"].shape, generator=gen) * b2["mask"][..., None]
        b2["label"] = torch.randint(0, C, b2["label"].shape, generator=gen).masked_fill(~b2["mask"], -100)
        b2["spk"] = b2["spk"].flip(-1) * b2["mask"][..., None]
        m0 = _dagerc(3)
        mk = (lambda m: DagercTrainStep(m, b["lengths"]))
        mkargs = (lambda bb: (bb["x"].cuda(), bb["spk"].cuda(), bb["label"].cuda()))
    m1 = copy.deepcopy(m0)
    args0, args1 = mkargs(b), mkargs(b)
    ts0 = mk(m0)
    losses0 = [float(ts0.step(*args0)) for _ in range(5)]
    ts1 = mk(m1).capture(*args1, warmup=2)
    losses1 = [float(ts1.replay()) for _ in range(3)]
    assert losses1 == losses0[2:]
    for (k, p), q in zip(m0.named_parameters(), m1.parameters()):
        assert torch.equal(p, q), k
    assert int(ts1.opt.step_dev.item()) == 5
    new = mkargs(b2)
    _refill(args1, new)
    _refill(args0, new)
    for _ in range(2):
        assert float(ts1.replay()) == float(ts0.step(*args0))
    ts1.check()
    assert float(ts1.step(*args1)) == float(ts0.step(*args0))          # an eager step between replays
    assert float(ts1.replay()) == float(ts0.step(*args0)) == float(ts1.global_loss())
    for (k, p), q in zip(m0.named_parameters(), m1.parameters()):
        assert torch.equal(p, q), k


# ------------------------------------------------------------------------------------------ dropout in the captured step
@pytest.mark.parametrize("which", ["mmgcn", "dagerc"])
def test_replay_draws_fresh_masks_and_equals_eager_steps_with_the_same_counter(which):
    from erc_b200 import ops
    from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep
    if which == "mmgcn":
        b = _mmgcn_batch(2)
        args = (_mm_feats(b), b["spk"].cuda(), b["label"].cuda())
        mkm, mk = (lambda s: _mmgcn(s)), (lambda m, **kw: MmgcnTrainStep(m, b["lengths"], **kw))
    else:
        b = _dag_batch(2)
        args = (b["x"].cuda(), b["spk"].cuda(), b["label"].cuda())
        mkm, mk = (lambda s: _dagerc(s, dropout=0.2)), (lambda m, **kw: DagercTrainStep(m, b["lengths"], **kw))
    ts = mk(mkm(4), lr=0.0).capture(*args)                   # lr 0: only the masks change from replay to replay
    losses = [float(ts.replay()) for _ in range(4)]
    assert len(set(losses)) == 4 and all(l == l for l in losses)
    ma = mkm(6)
    mb = copy.deepcopy(ma)
    warm = 3
    tsa = mk(ma)
    torch.manual_seed(7)
    tsa.capture(*args, warmup=warm)
    replays = [float(tsa.replay()) for _ in range(3)]
    torch.manual_seed(7)
    tsb = mk(mb)
    for _ in range(warm):
        tsb.step(*args)
    at_capture = torch.get_rng_state()                       # the host seeds the recorded step drew
    eager = []
    for _ in range(3):
        torch.set_rng_state(at_capture)
        ops.SEED_DEV = tsb.opt.step_dev
        try:
            eager.append(float(tsb.step(*args)))
        finally:
            ops.SEED_DEV = None
    assert replays == eager and len(set(replays)) == 3
    for (k, p), q in zip(ma.named_parameters(), mb.parameters()):
        assert torch.equal(p, q), k


def test_no_mmgcn_dropout_site_reuses_another_sites_mask_a_step_later(monkeypatch):
    """Each dropout site draws its mask from (site seed + step counter).  Two sites of one size whose seeds lie within the
    number of steps of each other would swap masks from one replay to the next (site k at step s + 1 = site k + 1 at step
    s): the seeds the captured step's sites use (recorded from an eager step with the device word set, the code the
    capture records) are at least 2^32 apart."""
    from erc_b200 import ops, ops_mmgcn
    from erc_b200.train_step import MmgcnTrainStep
    b = _mmgcn_batch(4)
    args = (_mm_feats(b), b["spk"].cuda(), b["label"].cuda())
    ts = MmgcnTrainStep(_mmgcn(8), b["lengths"])
    ts.step(*args)
    sites = []
    real_drop, real_layer = ops._dropout_call, ops_mmgcn._layer_fwd

    def drop(x, out, p, seed, seed_dev):
        if seed_dev is not None and p > 0:
            sites.append(("dropout", x.numel(), seed))
        return real_drop(x, out, p, seed, seed_dev)

    def layer(hi, h0, W, theta, alpha, relu, p, seed, seed_dev=None):
        if seed_dev is not None and p > 0:
            sites.append(("gcnii", hi.numel(), seed))
        return real_layer(hi, h0, W, theta, alpha, relu, p, seed, seed_dev)

    monkeypatch.setattr(ops, "_dropout_call", drop)
    monkeypatch.setattr(ops_mmgcn, "_layer_fwd", layer)
    ops.SEED_DEV = ts.opt.step_dev
    try:
        ts.step(*args)
    finally:
        ops.SEED_DEV = None
    fwd = sites
    kinds = {k for k, _, _ in fwd}
    assert kinds == {"dropout", "gcnii"} and sum(k == "gcnii" for k, _, _ in fwd) == 64, [(k, n) for k, n, _ in fwd]
    seeds = {}
    for _, n, s in fwd:
        seeds.setdefault(n, set()).add(s % 2 ** 64)          # a backward re-draw repeats its forward's seed
    for n, ss in seeds.items():
        ss = sorted(ss)
        gaps = [(b - a) for a, b in zip(ss, ss[1:])] + [(ss[0] - ss[-1]) % 2 ** 64] if len(ss) > 1 else []
        assert all(g >= 1 << 32 for g in gaps), (n, min(gaps))


# ------------------------------------------------------------------------------------------ sharded == whole
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dialogues(lengths, rank, world):
    from erc_b200.dist import shard_dialogues
    return shard_dialogues(lengths, world)[rank]


def _mm_packed_rows(lengths, idx):
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(lengths, 0)])
    return torch.cat([torch.arange(int(off[d]), int(off[d + 1])) for d in idx.tolist()])


def _run_mm(ts, b, idx, global_pad, steps):
    lens = b["lengths"] if idx is None else b["lengths"][idx]
    lmax = int(b["lengths"].max()) if global_pad or idx is None else int(lens.max())
    if idx is None:
        feats, spk, y = _mm_feats(b), b["spk"].cuda(), b["label"].cuda()
    else:
        feats = _mm_feats(b, idx, lmax)
        spk = b["spk"][:lmax, idx].contiguous().cuda()
        y = b["label"][_mm_packed_rows(b["lengths"], idx)].contiguous().cuda()
    return [float(ts.step(feats, spk, y)) for _ in range(steps)]


def _run_dag(ts, b, idx, steps):
    if idx is None:
        x, spk, y = b["x"], b["spk"], b["label"]
    else:
        L = int(b["lengths"][idx].max())
        x, spk, y = b["x"][idx, :L], b["spk"][idx, :L], b["label"][idx, :L]
    x, spk, y = x.contiguous().cuda(), spk.contiguous().cuda(), y.contiguous().cuda()
    return [float(ts.step(x, spk, y)) for _ in range(steps)]


def _reduced_grads(ts, m):
    slot = {id(p): v for p, v in zip(ts.opt.live, ts.opt.g_views)}
    return {k: slot[id(p)].detach().cpu().clone() for k, p in m.named_parameters() if id(p) in slot}


def _make(which, lengths, world=1, group=None, lmax=None, max_norm=None):
    from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep
    if which.startswith("mmgcn"):
        m = _mmgcn(3, dropout=False)
        return m, MmgcnTrainStep(m, lengths, lmax=lmax, world=world, group=group, transport="nccl" if world > 1 else "auto")
    m = _dagerc(3)
    return m, DagercTrainStep(m, lengths, max_norm=max_norm, world=world, group=group,
                              transport="nccl" if world > 1 else "auto")


DAG_MAX_NORM = 0.05                                          # below the gradient norm of every step: the clip engages


def _sharded_worker(rank, world, port, out_dir, which, steps):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import erc_b200  # noqa: F401
    b = _mmgcn_batch(0) if which.startswith("mmgcn") else _dag_batch(0)
    idx = _dialogues(b["lengths"], rank, world)
    glob = which == "mmgcn"
    lmax = int(b["lengths"].max()) if glob else None
    m, ts = _make(which, b["lengths"][idx], world, dist.group.WORLD, lmax=lmax, max_norm=DAG_MAX_NORM)
    assert ts.transport == "torch.distributed"
    losses, grads = [], None
    for _ in range(steps):
        if which.startswith("mmgcn"):
            _run_mm(ts, b, idx, glob, 1)
        else:
            _run_dag(ts, b, idx, 1)
        losses.append(float(ts.global_loss()))
        grads = grads or _reduced_grads(ts, m)
    ts.check()
    torch.save({"losses": losses, "grads": grads, "params": _params(m)}, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


def _assert_within_travel(got, m, steps, lr):
    """Adam's first updates are sign-like (lr * m / (sqrt(v) + eps)): an element whose gradient is within fp32 rounding of
    zero may move by up to 2 lr on one side only.  Held to half the distance the steps can travel and 1 % of it on
    average, as the DialogueGCN step's test holds them."""
    travel = steps * lr
    for k, p in m.named_parameters():
        d = (got[k] - p.detach().cpu()).abs()
        assert float(d.max()) <= 0.5 * travel and float(d.mean()) <= 1e-2 * travel, (k, float(d.max()), float(d.mean()))


@pytest.mark.parametrize("which", ["mmgcn", "mmgcn_shard_padding", "dagerc"])
def test_two_ranks_on_one_gpu_equal_one_rank_on_the_whole_batch(tmp_path, which):
    """The batch sharded by dialogue over 2 ranks (two processes on this GPU over gloo, eager) against one rank on the whole
    batch, 3 steps, dropout off: the global loss of every step (1e-6), the all-reduced gradient of the first step (1e-5:
    the shards' GEMMs sum over other row sets) and the parameters after 3 steps.  MMGCN pads every shard to the global
    Lmax; padded to its own Lmax instead, a shard's reverse text LSTM starts elsewhere and the step differs.  DAG-ERC
    clips (max_norm below the gradient norm); its whole-batch run also equals clip_grad_norm_ + torch.optim.AdamW applied
    to the same gradients."""
    steps = 3
    mp.spawn(_sharded_worker, args=(2, _free_port(), str(tmp_path), which, steps), nprocs=2, join=True)
    b = _mmgcn_batch(0) if which.startswith("mmgcn") else _dag_batch(0)
    m, ts = _make(which, b["lengths"], max_norm=DAG_MAX_NORM)
    ref = copy.deepcopy(m)
    whole, grads, all_grads = [], None, []
    for _ in range(steps):
        if which.startswith("mmgcn"):
            _run_mm(ts, b, None, True, 1)
        else:
            _run_dag(ts, b, None, 1)
        whole.append(float(ts.global_loss()))
        all_grads.append(_reduced_grads(ts, m))
        grads = grads or all_grads[-1]
    got = [torch.load(str(tmp_path / ("rank%d.pt" % r))) for r in range(2)]
    if which == "mmgcn_shard_padding":
        # the loss, a mean over every utterance, moves by about an ulp; the text encoder's gradients move visibly
        scale = max(float(v.abs().max()) for v in grads.values())
        worst = max(rel_err(got[0]["grads"][k], grads[k], floor=1e-2 * scale) for k in grads)
        print("per-shard padding: first-step loss %.7f vs whole batch %.7f, worst first-step gradient rel err %.2e"
              % (got[0]["losses"][0], whole[0], worst))
        assert worst > 1e-4
        return
    lr = 3e-4 if which == "mmgcn" else 1e-3
    for r in range(2):
        for a, c in zip(got[r]["losses"], whole):
            assert abs(a - c) <= 1e-6 * abs(c), (r, got[r]["losses"], whole)
        worst_g = check_grads(got[r]["grads"], grads, 1e-5)
        print("%s rank %d: losses %s vs %s, first-step gradient rel err %.2e" % (which, r, got[r]["losses"], whole, worst_g))
        _assert_within_travel(got[r]["params"], m, steps, lr)
    if which == "dagerc":
        live = [(k, p) for k, p in ref.named_parameters() if k in grads]
        norms = [float(torch.sqrt(sum((g[k].double() ** 2).sum() for k, _ in live))) for g in all_grads]
        assert min(norms) > DAG_MAX_NORM, norms
        opt = torch.optim.AdamW([p for _, p in live], lr=1e-3, weight_decay=1e-2)
        for g in all_grads:
            for k, p in live:
                p.grad = g[k].to(p.device)
            torch.nn.utils.clip_grad_norm_([p for _, p in live], DAG_MAX_NORM)
            opt.step()
        for k, p in live:
            assert rel_err(dict(m.named_parameters())[k].detach().cpu(), p.detach().cpu()) <= 1e-6, k


# ------------------------------------------------------------------------------------------ peer-memory payload
@pytest.mark.parametrize("which", ["mmgcn", "dagerc"])
def test_step_communicator_size_carries_the_first_step_all_reduce(which):
    """Two peer-memory endpoints of the size the step creates (PeerComm.simulate: the same kernels and flag protocol as
    across GPUs, on two streams of this GPU) all-reduce a buffer as long as the step's flat gradient (over 16 MB)."""
    from erc_b200.p2p import PeerComm
    if which == "mmgcn":
        b = _mmgcn_batch(0)
        m, ts = _make("mmgcn", b["lengths"])
        _run_mm(ts, b, None, True, 1)
    else:
        b = _dag_batch(0)
        m, ts = _make("dagerc", b["lengths"], max_norm=5.0)
        _run_dag(ts, b, None, 1)
    n = ts.opt.flat_g.numel()
    assert 4 * n > 16 << 20 and ts.comm_bytes >= 4 * n
    comms = PeerComm.simulate(2, "cuda:0", max_bytes=ts.comm_bytes)
    gen = torch.Generator(device="cuda").manual_seed(1)
    xs = [torch.randn(n, device="cuda", generator=gen) for _ in range(2)]
    want = xs[0] + xs[1]
    streams = [torch.cuda.Stream() for _ in range(2)]
    torch.cuda.synchronize()
    for r in range(2):
        with torch.cuda.stream(streams[r]):
            comms[r].all_reduce(xs[r])
    torch.cuda.synchronize()
    assert all(torch.equal(x, want) for x in xs) and all(c.status() == 0 for c in comms)
    for c in comms:
        c.close()
