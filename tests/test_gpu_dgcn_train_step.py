"""DialogueGCN as one captured train step: ercg_dropout_dev (the BiLSTM's inter-layer dropout with a device seed word),
DGCNModule.forward_packed against forward, and train_step.DgcnTrainStep against the eager module path (train_mm's step:
forward on the padded batch + ops.cross_entropy + FlatAdam), replay against eager, fresh dropout masks per replay, and a
batch sharded by dialogue against the whole batch (dgcn.py:117-134)."""
import copy
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

from conftest import ROOT, check_grads, parity_check, rel_err

pytestmark = pytest.mark.gpu

D, C = 1380, 6


def _batch(seed, B):
    """A config-2-shaped batch (synth.config2: IEMOCAP lengths, width 1380, 2 speakers, 6 classes) in both layouts."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    b = synth.config2(seed=seed, B=B)
    mask = torch.arange(b["input_tensor"].size(1))[None, :] < b["text_length"][:, None]
    b["x_packed"] = b["input_tensor"][mask].contiguous()            # [N, 1380]: 5520-byte rows, 16-byte aligned
    b["speaker_packed"] = b["speaker_tensor"][mask].contiguous()
    return b


def _model(seed, dropout=0.4):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcn import DGCNModule
    torch.manual_seed(seed)
    m = DGCNModule(2, input_size=D, hidden_size=200, n_classes=C, dropout=dropout).cuda()
    m.train()
    return m


def _cuda(b, *keys):
    return [b[k].cuda() for k in keys]


def _weights():
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    return torch.tensor(LOSS_WEIGHTS, device="cuda")


# ------------------------------------------------------------------------------------------ ercg_dropout_dev
def test_dropout_dev_equals_host_seed_dropout_and_backward_reapplies_the_mask():
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200._lib import lib
    gen = torch.Generator(device="cuda").manual_seed(0)
    n, p, seed = 1_000_003, 0.4, 0x1234_5678_9ABC
    x = torch.randn(n, device="cuda", generator=gen)

    def host(t, s):
        out = torch.empty_like(t)
        assert lib().ercg_dropout(t.data_ptr(), out.data_ptr(), n, p, s & (2 ** 64 - 1), None) == 0
        return out

    def dev(t, s, word):
        out = torch.empty_like(t)
        w = torch.tensor([word], dtype=torch.int64, device="cuda")
        assert lib().ercg_dropout_dev(t.data_ptr(), out.data_ptr(), n, p, s, w.data_ptr(), None) == 0
        return out

    assert torch.equal(dev(x, seed, 0), host(x, seed))
    for word in (1, 7, 123456789):
        got = dev(x, seed, word)
        assert torch.equal(got, host(x, seed + word)) and not torch.equal(got, host(x, seed))
    kept = float((host(x, seed) != 0).float().mean())
    assert abs(kept - (1 - p)) < 3e-3
    # through ops.dropout: with SEED_DEV set the forward and the backward use the same word, hence the same mask
    word = torch.tensor([41], dtype=torch.int64, device="cuda")
    g = torch.randn(n, device="cuda", generator=gen)
    xr = x.clone().requires_grad_()
    ops.SEED_DEV = word
    try:
        y = ops.dropout(xr, p, seed)
    finally:
        ops.SEED_DEV = None
    y.backward(g)
    assert torch.equal(y.detach(), host(x, seed + 41)) and torch.equal(xr.grad, host(g, seed + 41))
    # bad arguments: ERCG_EINVAL before any launch
    w = torch.zeros(1, dtype=torch.int64, device="cuda")
    out = torch.empty_like(x)
    f = lib().ercg_dropout_dev
    assert f(x.data_ptr(), out.data_ptr(), n, p, seed, None, None) == -1
    assert f(x.data_ptr(), out.data_ptr(), -1, p, seed, w.data_ptr(), None) == -1
    assert f(x.data_ptr(), out.data_ptr(), n, 1.0, seed, w.data_ptr(), None) == -1
    assert f(x.data_ptr(), out.data_ptr(), n, -0.1, seed, w.data_ptr(), None) == -1
    assert f(x.data_ptr(), out.data_ptr(), 0, p, seed, w.data_ptr(), None) == 0


# ------------------------------------------------------------------------------------------ forward_packed
def _both_paths(m0, b, seed):
    from erc_b200 import ops
    m1 = copy.deepcopy(m0)
    w = _weights()
    lens, y = b["text_length"], b["label"].cuda()
    torch.manual_seed(100 + seed)
    l0, g0 = m0(b["input_tensor"].cuda(), b["speaker_tensor"].cuda(), lens)
    ops.cross_entropy(l0, y, w).backward()
    torch.manual_seed(100 + seed)                                    # same host seeds: same dropout masks
    l1, g1 = m1.forward_packed(b["x_packed"].cuda(), b["speaker_packed"].cuda(), lens)
    ops.cross_entropy(l1, y, w).backward()
    grads = [{k: p.grad.cpu() for k, p in m.named_parameters() if p.grad is not None} for m in (m0, m1)]
    return (l0, g0, grads[0]), (l1, g1, grads[1])


@pytest.mark.parametrize("seed,B", [(0, 32), (1, 360)])
def test_forward_packed_equals_forward(seed, B):
    """Same logits, graph_out and parameter gradients as ``forward``.  The packed input transform runs on the tensor-core
    kernels (N >= TC_MIN_ROWS), forward's on the SIMT row gather: both within the fp32 bar of each other, or the packed
    path no further from the fp64 oracle than the module path's own fp32 result is (conftest.parity_check, forward's
    result in the role of the fp32 reference).  At the config-2 size also with dropout on (the same host seeds give the
    same masks), to the plain 1e-5 bar."""
    import torch.nn.functional as F
    from erc_b200 import ops
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    from oracle import modules as om
    b = _batch(seed, B)
    N = b["x_packed"].size(0)
    assert N >= ops.TC_MIN_ROWS and (B < 100 or N >= 16384), N
    if B == 32:
        (l0, g0, gr0), (l1, g1, gr1) = _both_paths(_model(seed), b, seed)
        assert rel_err(l1, l0) < 1e-5 and rel_err(g1, g0) < 1e-5
        print("dropout on, N = %d: worst gradient rel err %.2e" % (N, check_grads(gr1, gr0, 1e-5)))
    m = _no_dropout(_model(seed))
    o = om.DgcnOracle(2, input_size=D, hidden_size=200, n_classes=C, dropout=0.0).double()
    om.load_live(o, {k: v.detach().cpu().double() for k, v in m.state_dict().items()})
    o.train()
    ol, og = o(b["input_tensor"].double(), b["speaker_tensor"], b["text_length"])
    F.cross_entropy(ol, b["label"], weight=torch.tensor(LOSS_WEIGHTS, dtype=torch.float64)).backward()
    (l0, g0, gr0), (l1, g1, gr1) = _both_paths(m, b, seed)
    parity_check("dgcn/forward_packed/N%d/outputs" % N, {"logits": l1, "graph_out": g1}, {"logits": l0, "graph_out": g0},
                 {"logits": ol.detach(), "graph_out": og.detach()})
    recs = parity_check("dgcn/forward_packed/N%d/grads" % N, gr1, gr0,
                        {k: p.grad for k, p in o.named_parameters() if p.grad is not None})
    print("dropout off, N = %d: worst gradient rel err vs forward %.2e" % (N, max(r["e_vs_ref32"] for r in recs)))


# ------------------------------------------------------------------------------------------ DgcnTrainStep, world 1
def _arm_a(m, b, steps, lr=3e-4):
    """train_mm's DialogueGCN step: forward on the padded batch + class-weighted ops.cross_entropy + FlatAdam."""
    from erc_b200 import ops
    from erc_b200.optim import FlatAdam
    opt = FlatAdam(m.parameters(), lr=lr, weight_decay=0.0)
    w = _weights()
    xp, spk, y = b["input_tensor"].cuda(), b["speaker_tensor"].cuda(), b["label"].cuda()
    losses = []
    for _ in range(steps):
        loss = ops.cross_entropy(m(xp, spk, b["text_length"])[0], y, w)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    return losses


def _no_dropout(m):
    m.rnn.rnn.dropout = 0.0
    m.clf.drop.p = 0.0
    return m


def test_train_step_matches_the_module_path_and_replay_equals_eager():
    from erc_b200.train_step import DgcnTrainStep
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    b = _batch(0, 32)
    N = int(b["text_length"].sum())
    g2 = torch.Generator().manual_seed(9)                            # new features / labels / speakers, same lengths
    x2, y2 = torch.randn(N, D, generator=g2), torch.randint(0, C, (N,), generator=g2)
    s2 = torch.randint(0, 2, (N,), generator=g2)
    m0 = _no_dropout(_model(3))
    m1 = copy.deepcopy(m0)
    x, spk, y = _cuda(b, "x_packed", "speaker_packed", "label")
    # eager steps through the train-step object
    ts0 = DgcnTrainStep(m0, b["text_length"], class_weight=LOSS_WEIGHTS)
    losses0 = [float(ts0.step(x, spk, y)) for _ in range(5)]
    ts0.check()
    assert float(ts0.global_loss()) == losses0[-1]
    # the same five steps: two eager warm-up steps inside capture(), then three replays
    ts1 = DgcnTrainStep(m1, b["text_length"], class_weight=LOSS_WEIGHTS).capture(x, spk, y, warmup=2)
    losses1 = [float(ts1.replay()) for _ in range(3)]
    assert losses1 == losses0[2:]
    for (k, p), q in zip(m0.named_parameters(), m1.parameters()):
        assert torch.equal(p, q), k
    assert int(ts1.opt.step_dev.item()) == 5 and float(ts1.global_loss()) == losses1[-1]
    # refill the static inputs in place with another batch of the same lengths: replay == eager, bit for bit
    x.copy_(x2.cuda())
    y.copy_(y2.cuda())
    spk.copy_(s2.cuda())
    for _ in range(2):
        assert float(ts1.replay()) == float(ts0.step(x, spk, y))
    ts1.check()
    # an eager step between replays: replay() still returns the graph's loss, global_loss() the last step's
    assert float(ts1.step(x, spk, y)) == float(ts0.step(x, spk, y))
    assert float(ts1.replay()) == float(ts0.step(x, spk, y)) == float(ts1.global_loss())
    for (k, p), q in zip(m0.named_parameters(), m1.parameters()):
        assert torch.equal(p, q), k
    # against train_mm's path (arm a): the losses of three steps agree to the fp32 bar.  The two paths compute the layer-0
    # input transform with different kernels (tensor-core vs SIMT row gather, ~1e-6 apart), and Adam's first updates are
    # lr * g / (|g| + eps), sign-like: an element whose gradient is within that noise of zero may move by up to 2 lr on one
    # side only.  So the parameters are held, as the COGMEN step's test holds them, to a small fraction of the distance
    # three steps can travel (3 lr), tightly on average.
    m3 = _no_dropout(_model(3))
    losses3 = _arm_a(m3, b, 3)
    for a, c in zip(losses0[:3], losses3):
        assert abs(a - c) <= 1e-5 * abs(c), (a, c)
    m4 = _no_dropout(_model(3))
    ts4 = DgcnTrainStep(m4, b["text_length"], class_weight=LOSS_WEIGHTS)
    x, spk, y = _cuda(b, "x_packed", "speaker_packed", "label")
    for _ in range(3):
        ts4.step(x, spk, y)
    travel = 3 * 3e-4
    for (k, p), q in zip(m4.named_parameters(), m3.parameters()):
        d = (p - q).abs()
        assert float(d.max()) <= 0.5 * travel and float(d.mean()) <= 1e-2 * travel, (k, float(d.max()), float(d.mean()))
    assert losses0[-1] < losses0[0]


# ------------------------------------------------------------------------------------------ dropout in the captured step
def test_replay_draws_fresh_masks_and_equals_eager_steps_with_the_same_counter():
    from erc_b200 import ops
    from erc_b200.train_step import DgcnTrainStep
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    b = _batch(2, 32)
    x, spk, y = _cuda(b, "x_packed", "speaker_packed", "label")
    # lr 0: the parameters stay, only the masks change from replay to replay.  The classifier's dropout is off, so only the
    # BiLSTM's inter-layer dropout (ops.dropout -> ercg_dropout_dev) can change the loss
    m = _model(4)
    m.clf.drop.p = 0.0
    ts = DgcnTrainStep(m, b["text_length"], lr=0.0, class_weight=LOSS_WEIGHTS).capture(x, spk, y)
    losses = [float(ts.replay()) for _ in range(4)]
    assert len(set(losses)) == 4 and all(l == l for l in losses)
    # replay k == eager step k of a second instance whose steps run with SEED_DEV at its own step counter (same value)
    # and the host seeds the capture drew
    ma = _model(6)
    mb = copy.deepcopy(ma)
    warm = 3
    tsa = DgcnTrainStep(ma, b["text_length"], class_weight=LOSS_WEIGHTS)
    torch.manual_seed(7)
    tsa.capture(x, spk, y, warmup=warm)
    replays = [float(tsa.replay()) for _ in range(3)]
    torch.manual_seed(7)
    tsb = DgcnTrainStep(mb, b["text_length"], class_weight=LOSS_WEIGHTS)
    for _ in range(warm):
        tsb.step(x, spk, y)
    at_capture = torch.get_rng_state()                 # the host seeds the recorded step drew
    eager = []
    for _ in range(3):
        torch.set_rng_state(at_capture)
        ops.SEED_DEV = tsb.opt.step_dev
        try:
            eager.append(float(tsb.step(x, spk, y)))
        finally:
            ops.SEED_DEV = None
    assert replays == eager and len(set(replays)) == 3
    for (k, p), q in zip(ma.named_parameters(), mb.parameters()):
        assert torch.equal(p, q), k


# ------------------------------------------------------------------------------------------ sharded == whole
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _shard(b, idx):
    """Rows of the dialogues ``idx`` (ascending) of a packed batch."""
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(b["text_length"], 0)])
    rows = torch.cat([torch.arange(int(off[d]), int(off[d + 1])) for d in idx.tolist()])
    return b["x_packed"][rows].contiguous(), b["speaker_packed"][rows].contiguous(), b["label"][rows].contiguous(), \
        b["text_length"][idx].contiguous()


def _reduced_grads(ts, m):
    """{name: the all-reduced gradient in the step's flat buffer} (valid right after a step)."""
    slot = {id(p): v for p, v in zip(ts.opt.live, ts.opt.g_views)}
    return {k: slot[id(p)].detach().cpu().clone() for k, p in m.named_parameters() if id(p) in slot}


def _assert_within_travel(got, m, steps, lr=3e-4):
    """Parameters after ``steps`` Adam steps from the same start, whose gradients agree to fp32 rounding: Adam's update
    lr * m / (sqrt(v) + eps) is sign-like, so an element whose gradient lies within that rounding of zero can move by up
    to 2 lr on one side only.  Held, as the COGMEN step's test holds them, to half the distance the steps can travel at
    most and to 1 % of it on average."""
    travel = steps * lr
    for k, p in m.named_parameters():
        d = (got[k] - p.detach().cpu()).abs()
        assert float(d.max()) <= 0.5 * travel and float(d.mean()) <= 1e-2 * travel, (k, float(d.max()), float(d.mean()))


def _sharded_worker(rank, world, port, out_dir, steps):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import erc_b200  # noqa: F401
    from erc_b200.dist import shard_dialogues
    from erc_b200.train_step import DgcnTrainStep
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    b = _batch(0, 32)
    x, spk, y, lens = _shard(b, shard_dialogues(b["text_length"], world)[rank])
    m = _no_dropout(_model(3))
    ts = DgcnTrainStep(m, lens, class_weight=LOSS_WEIGHTS, world=world, group=dist.group.WORLD, transport="nccl")
    assert ts.transport == "torch.distributed"
    x, spk, y = x.cuda(), spk.cuda(), y.cuda()
    losses, grads = [], None
    for _ in range(steps):
        ts.step(x, spk, y)
        losses.append(float(ts.global_loss()))
        grads = grads or _reduced_grads(ts, m)
    ts.check()
    torch.save({"losses": losses, "grads": grads, "params": {k: p.detach().cpu() for k, p in m.named_parameters()}},
               os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


def test_two_ranks_on_one_gpu_equal_one_rank_on_the_whole_batch(tmp_path):
    """The batch sharded by dialogue over 2 ranks (two processes on this GPU over gloo, torch.distributed transport, eager)
    takes the step of one rank on the whole batch: every step's loss is the global weighted mean (1e-6), the all-reduced
    gradient of the first step is the whole batch's gradient (the fp32 bar: the shards' weight-gradient GEMMs run over
    other row sets, hence other kernels and summation orders), and the parameters after 3 steps agree as Adam allows."""
    from erc_b200.train_step import DgcnTrainStep
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    steps = 3
    mp.spawn(_sharded_worker, args=(2, _free_port(), str(tmp_path), steps), nprocs=2, join=True)
    b = _batch(0, 32)
    m = _no_dropout(_model(3))
    ts = DgcnTrainStep(m, b["text_length"], class_weight=LOSS_WEIGHTS)
    x, spk, y = _cuda(b, "x_packed", "speaker_packed", "label")
    whole, grads = [], None
    for _ in range(steps):
        ts.step(x, spk, y)
        whole.append(float(ts.global_loss()))
        grads = grads or _reduced_grads(ts, m)
    for r in range(2):
        got = torch.load(str(tmp_path / ("rank%d.pt" % r)))
        for a, c in zip(got["losses"], whole):
            assert abs(a - c) <= 1e-6 * abs(c), (r, got["losses"], whole)
        worst_g = check_grads(got["grads"], grads, 1e-5)
        worst_p = max(rel_err(got["params"][k], p) for k, p in m.named_parameters())
        print("rank %d: losses %s vs %s, first-step gradient rel err %.2e, parameters after %d steps rel err %.2e"
              % (r, got["losses"], whole, worst_g, steps, worst_p))
        _assert_within_travel(got["params"], m, steps)


def test_sharded_capture_over_peer_memory_equals_the_whole_batch():
    """The same check on two GPUs under torch.distributed.run: peer-memory transport, captured step, replays."""
    import json
    import subprocess
    have = torch.cuda.device_count()
    if have < 2:
        print("skipped: the peer-memory sharded step needs 2 GPUs, %d visible" % have)
        pytest.skip("needs 2 GPUs, %d visible" % have)
    env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", "2",
                        os.path.join(ROOT, "tools", "bench_dgcn_step.py"), "--dist-check"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    print(line)
    assert line["transport"].startswith("peer memory")
    assert line["loss_rel_diff"] <= 1e-6 and line["grad_rel_err"] <= 1e-5, line
    travel = line["steps"] * 3e-4
    assert line["param_max_abs_diff"] <= 0.5 * travel and line["param_mean_abs_diff"] <= 1e-2 * travel, line


def test_dgcn_step_communicator_size_carries_the_first_step_all_reduce():
    """The first step all-reduces the whole flat gradient buffer (8.6 MB at width 1380) in one peer-memory call: two endpoints
    of the size the step creates (PeerComm.simulate: the same kernels and flag protocol as across GPUs, on two streams of
    this GPU) reduce a buffer of that length to the rank-ordered sum."""
    from erc_b200.p2p import PeerComm
    from erc_b200.train_step import DgcnTrainStep
    b = _batch(0, 32)
    ts = DgcnTrainStep(_model(3), b["text_length"])
    ts.step(*_cuda(b, "x_packed", "speaker_packed", "label"))
    n = ts.opt.flat_g.numel()
    assert 4 * n > 8 << 20
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
