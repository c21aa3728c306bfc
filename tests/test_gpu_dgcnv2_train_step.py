"""dgcnv2 (the declare-lab DialogueGCN, track_mm/dgcnv2.py) as one captured train step: DGCNModule.forward_packed against
forward for the LSTM, GRU and None bases, train_step.Dgcnv2TrainStep against train_mm's module path (forward on the
seq-first padded batch + class-weighted ops.cross_entropy + FlatAdam), replay against eager, fresh dropout masks per replay,
a batch sharded by dialogue (every shard padded to the global lmax) against the whole batch, and the argument checks of
the K11 edge attention."""
import copy
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp
from torch import nn

from conftest import ROOT, check_grads, parity_check, rel_err

pytestmark = pytest.mark.gpu

D, H, C = 1380, 100, 6
BASES = ("LSTM", "GRU", "None")


def _batch(seed, B):
    """A config-2-shaped batch (IEMOCAP lengths, width 1380, 2 speakers, 6 classes) in both layouts: seq-first with one-hot
    speakers (what ``forward`` takes) and batch-first rows [B * Lmax, D] with packed speaker ids (``forward_packed``)."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    b = synth.config2(seed=seed, B=B)
    x, spk, lens = b["input_tensor"], b["speaker_tensor"], b["text_length"]
    mask = torch.arange(x.size(1))[None, :] < lens[:, None]
    b["x_seq"] = x.transpose(0, 1).contiguous()
    b["spk_seq"] = nn.functional.one_hot(spk.t(), 2).float()
    b["x_rows"] = x.reshape(-1, D)                                  # 5520-byte rows: 16-byte aligned
    b["speaker_packed"] = spk[mask].contiguous()
    return b


def _model(seed, base="LSTM", dropout=0.4):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    torch.manual_seed(seed)
    m = DGCNModule(base, input_size=D, hidden_size=H, n_speakers=2, n_classes=C, dropout=dropout).cuda()
    m.train()
    return m


def _rnn(m):
    return {"LSTM": getattr(m, "lstm", None), "GRU": getattr(m, "gru", None)}.get(m.base_model)


def _no_dropout(m):
    if _rnn(m) is not None:
        _rnn(m).dropout = 0.0
    m.graph_net.dropout.p = 0.0
    return m


def _weights():
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    return torch.tensor(LOSS_WEIGHTS, device="cuda")


def _cuda(b, *keys):
    return [b[k].cuda() for k in keys]


def _grads(m):
    return {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters() if p.grad is not None}


# ------------------------------------------------------------------------------------------ forward_packed
_GEMM_K = {"ercg_gemm_nn_tc": 9, "ercg_gemm_tn_tc": 7, "ercg_gemm_nn": 10, "ercg_gemm_tn": 8}


def _gemm_label(name, args):
    """GEMM calls labelled by their contraction length (the layer-0 input transform is the one with K = D)."""
    k = _GEMM_K.get(name)
    return "%s/K=%d" % (name, args[k]) if k is not None else name


def _both_paths(m0, b, seed):
    from erc_b200 import _lib, ops
    m1 = copy.deepcopy(m0)
    w = _weights()
    lens, y = b["text_length"], b["label"].cuda()
    torch.manual_seed(100 + seed)
    with _lib.KernelTimer(_gemm_label) as kt0:
        l0, f0 = m0(b["x_seq"].cuda(), b["spk_seq"].cuda(), None, lens)
        ops.cross_entropy(l0, y, w).backward()
    torch.manual_seed(100 + seed)                                    # same host seeds: same dropout masks on the same rows
    with _lib.KernelTimer(_gemm_label) as kt1:
        l1, f1 = m1.forward_packed(b["x_rows"].cuda(), b["speaker_packed"].cuda(), lens, b["x_seq"].size(0))
        ops.cross_entropy(l1, y, w).backward()
    k0, k1 = kt0.summary(), kt1.summary()
    assert "ercg_gemm_nn/K=%d" % D in k0                             # forward: the SIMT row gather
    # forward_packed: the layer-0 product and its weight gradient on the tensor cores, nothing with K = D elsewhere
    assert "ercg_gemm_nn_tc/K=%d" % D in k1 and "ercg_gemm_tn_tc/K=%d" % D in k1, sorted(k1)
    assert "ercg_gemm_nn/K=%d" % D not in k1 and "ercg_gemm_tn/K=%d" % D not in k1, sorted(k1)
    return (l0, f0, _grads(m0)), (l1, f1, _grads(m1))


class _SeqRnn(nn.Module):
    """nn.GRU in the slot of the oracle's base Linear: [L, B, D] -> [L, B, 2h]."""

    def __init__(self, rnn):
        super().__init__()
        self.rnn = rnn

    def forward(self, x):
        return self.rnn(x)[0]


def _oracle64(m, b):
    """fp64 CPU restatement (oracle/dgcnv2_oracle.py; its base Linear slot holds an nn.GRU for the GRU base) of the
    module's logits, features and parameter gradients, names as the module's."""
    import torch.nn.functional as F
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    from oracle import dgcnv2_oracle, modules as om
    o = dgcnv2_oracle.Dgcnv2Oracle(D, hidden_size=H, n_classes=C, dropout=0.0,
                                   base_model="LSTM" if m.base_model == "LSTM" else "None")
    if m.base_model == "GRU":
        o.base_linear = _SeqRnn(nn.GRU(D, H, num_layers=2, bidirectional=True))
    o = o.double().train()
    to_o = {"gru.": "base_linear.rnn."}
    sd = {}
    for k, v in m.state_dict().items():
        for a, c in to_o.items():
            k = c + k[len(a):] if k.startswith(a) else k
        sd[k] = v.detach().cpu().double()
    om.load_live(o, sd)
    assert set(o.state_dict()) <= set(sd), sorted(set(o.state_dict()) - set(sd))
    lg, ft = o(b["x_seq"].double(), b["spk_seq"].double(), None, b["text_length"])
    F.cross_entropy(lg, b["label"], weight=torch.tensor(LOSS_WEIGHTS, dtype=torch.float64)).backward()
    grads = {}
    for k, p in o.named_parameters():
        if p.grad is not None:
            grads[k.replace("base_linear.rnn.", "gru.", 1) if k.startswith("base_linear.rnn.") else k] = p.grad
    return {"logits": lg.detach(), "features": ft.detach()}, grads


@pytest.mark.parametrize("base", BASES)
@pytest.mark.parametrize("seed,B", [(0, 32), (1, 300)])
def test_forward_packed_equals_forward(base, seed, B):
    """Same logits, features and parameter gradients as ``forward`` on the seq-first batch.  The packed layer-0 input
    transform runs on the tensor-core kernels, forward's on the SIMT row gather: each tensor within 1e-5 of forward's
    (relative to its own scale), or -- at a few hundred dialogues -- no further from the fp64 oracle than forward's own
    fp32 result is (conftest.parity_check).  The None base at 300 dialogues needs the second bar: there forward's own fp32
    gradients are up to 7e-4 from fp64 (no recurrence bounds the base's output), and the packed path's are as close.  At
    the config-2 size also with dropout on: the same host seeds draw the same masks, which sit on the same dialogue-major
    rows in both paths."""
    b = _batch(seed, B)
    if B == 32:
        (l0, f0, gr0), (l1, f1, gr1) = _both_paths(_model(seed, base), b, seed)
        parity_check("dgcnv2/forward_packed/%s/B%d/dropout/outputs" % (base, B), {"logits": l1, "features": f1},
                     {"logits": l0, "features": f0})
        parity_check("dgcnv2/forward_packed/%s/B%d/dropout/grads" % (base, B), gr1, gr0)
    m = _no_dropout(_model(seed, base))
    (l0, f0, gr0), (l1, f1, gr1) = _both_paths(m, b, seed)
    o_out, o_grads = _oracle64(m, b) if B > 32 else (None, None)
    parity_check("dgcnv2/forward_packed/%s/B%d/outputs" % (base, B), {"logits": l1, "features": f1},
                 {"logits": l0, "features": f0}, o_out)
    recs = parity_check("dgcnv2/forward_packed/%s/B%d/grads" % (base, B), gr1, gr0, o_grads)
    print("%s, B = %d: worst gradient rel err vs forward %.2e" % (base, B, max(r["e_vs_ref32"] for r in recs)))


def test_forward_packed_rejects_bad_lmax_and_rows():
    b = _batch(0, 4)
    m = _model(0)
    x, spk = _cuda(b, "x_rows", "speaker_packed")
    lens, L = b["text_length"], b["x_seq"].size(0)
    with pytest.raises(ValueError):
        m.forward_packed(x, spk, lens, L - 1)                       # shorter than the longest dialogue
    with pytest.raises(ValueError):
        m.forward_packed(torch.zeros(4 * 111, D, device="cuda"), spk, lens, 111)      # beyond max_seq_len
    with pytest.raises(ValueError):
        m.forward_packed(x[:-1], spk, lens, L)                      # not [B * lmax, D]


# ------------------------------------------------------------------------------------------ Dgcnv2TrainStep, world 1
def _arm_a(m, b, steps, lr=3e-4):
    """train_mm's dgcnv2 step: forward on the seq-first padded batch + class-weighted ops.cross_entropy + FlatAdam."""
    from erc_b200 import ops
    from erc_b200.optim import FlatAdam
    opt = FlatAdam(m.parameters(), lr=lr, weight_decay=0.0)
    w = _weights()
    xs, ss, y = b["x_seq"].cuda(), b["spk_seq"].cuda(), b["label"].cuda()
    losses = []
    for _ in range(steps):
        loss = ops.cross_entropy(m(xs, ss, None, b["text_length"])[0], y, w)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    return losses


def _step(m, lengths, **kw):
    from erc_b200.train_step import Dgcnv2TrainStep
    from erc_b200.track_mm.dgcn import LOSS_WEIGHTS
    return Dgcnv2TrainStep(m, lengths, class_weight=LOSS_WEIGHTS, **kw)


@pytest.mark.parametrize("base", BASES)
def test_eager_steps_match_the_module_path(base):
    """Three eager steps against train_mm's path: the losses to the fp32 bar, the parameters as Adam allows (its first
    updates are sign-like, lr * g / (|g| + eps): an element whose gradient lies within the two paths' GEMM rounding of zero
    may move by up to 2 lr on one side only), as the DialogueGCN step's test holds them."""
    b = _batch(0, 32)
    m3 = _no_dropout(_model(3, base))
    losses3 = _arm_a(m3, b, 3)
    m4 = _no_dropout(_model(3, base))
    ts = _step(m4, b["text_length"])
    x, spk, y = _cuda(b, "x_rows", "speaker_packed", "label")
    losses4 = [float(ts.step(x, spk, y)) for _ in range(3)]
    ts.check()
    for a, c in zip(losses4, losses3):
        assert abs(a - c) <= 1e-5 * abs(c), (losses4, losses3)
    travel = 3 * 3e-4
    for (k, p), q in zip(m4.named_parameters(), m3.parameters()):
        d = (p - q).abs()
        assert float(d.max()) <= 0.5 * travel and float(d.mean()) <= 1e-2 * travel, (k, float(d.max()), float(d.mean()))
    assert losses4[-1] < losses4[0]


@pytest.mark.parametrize("base", BASES)
def test_replay_equals_eager_bit_for_bit(base):
    b = _batch(0, 32)
    N = int(b["text_length"].sum())
    g2 = torch.Generator().manual_seed(9)                            # new features / labels / speakers, same lengths
    x2 = b["x_rows"].clone()
    mask = (torch.arange(b["x_seq"].size(0))[None, :] < b["text_length"][:, None]).reshape(-1)
    x2[mask] = torch.randn(N, D, generator=g2)
    y2, s2 = torch.randint(0, C, (N,), generator=g2), torch.randint(0, 2, (N,), generator=g2)
    m0 = _no_dropout(_model(3, base))
    m1 = copy.deepcopy(m0)
    x, spk, y = _cuda(b, "x_rows", "speaker_packed", "label")
    ts0 = _step(m0, b["text_length"])
    losses0 = [float(ts0.step(x, spk, y)) for _ in range(5)]
    ts0.check()
    assert float(ts0.global_loss()) == losses0[-1]
    # the same five steps: two eager warm-up steps inside capture(), then three replays
    ts1 = _step(m1, b["text_length"]).capture(x, spk, y, warmup=2)
    losses1 = [float(ts1.replay()) for _ in range(3)]
    assert losses1 == losses0[2:]
    for (k, p), q in zip(m0.named_parameters(), m1.parameters()):
        assert torch.equal(p, q), k
    assert int(ts1.opt.step_dev.item()) == 5 and float(ts1.global_loss()) == losses1[-1]
    # refill the static inputs in place with another batch of the same lengths
    x.copy_(x2.cuda())
    y.copy_(y2.cuda())
    spk.copy_(s2.cuda())
    for _ in range(2):
        assert float(ts1.replay()) == float(ts0.step(x, spk, y))
    ts1.check()
    assert float(ts1.step(x, spk, y)) == float(ts0.step(x, spk, y))
    assert float(ts1.replay()) == float(ts0.step(x, spk, y)) == float(ts1.global_loss())
    for (k, p), q in zip(m0.named_parameters(), m1.parameters()):
        assert torch.equal(p, q), k


def test_step_rejects_inputs_of_another_shape():
    b = _batch(0, 8)
    ts = _step(_model(0), b["text_length"])
    x, spk, y = _cuda(b, "x_rows", "speaker_packed", "label")
    for args in ((x[:-1], spk, y), (x, spk[:-1], y), (x, spk, y[:-1])):
        with pytest.raises(ValueError):
            ts.step(*args)


# ------------------------------------------------------------------------------------------ dropout in the captured step
@pytest.mark.parametrize("base,site", [("LSTM", "base"), ("LSTM", "head"), ("GRU", "base"), ("None", "head")])
def test_replay_draws_fresh_masks_and_equals_eager_steps_with_the_same_counter(base, site):
    """One dropout site on at a time (the base's inter-layer ops.dropout, or the GraphNetwork head's dropout in the GEMM
    epilogue): with lr 0 only the masks change between replays, so four replays give four losses -- no site replays a
    host-seeded mask.  Each replay equals an eager step of a second instance run with SEED_DEV at its own step counter
    and the host seeds the capture drew."""
    from erc_b200 import ops

    def model(seed):
        m = _model(seed, base)
        if site == "base":
            m.graph_net.dropout.p = 0.0
        else:
            if _rnn(m) is not None:
                _rnn(m).dropout = 0.0
        return m

    b = _batch(2, 32)
    x, spk, y = _cuda(b, "x_rows", "speaker_packed", "label")
    ts = _step(model(4), b["text_length"], lr=0.0).capture(x, spk, y)
    losses = [float(ts.replay()) for _ in range(4)]
    assert len(set(losses)) == 4 and all(l == l for l in losses), losses
    ma = model(6)
    mb = copy.deepcopy(ma)
    warm = 3
    tsa = _step(ma, b["text_length"])
    torch.manual_seed(7)
    tsa.capture(x, spk, y, warmup=warm)
    replays = [float(tsa.replay()) for _ in range(3)]
    torch.manual_seed(7)
    tsb = _step(mb, b["text_length"])
    for _ in range(warm):
        tsb.step(x, spk, y)
    at_capture = torch.get_rng_state()
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


def _shard(b, idx, lmax):
    """The dialogues ``idx`` (ascending) padded to ``lmax``: rows [len(idx) * lmax, D], packed speakers and labels."""
    lens = b["text_length"]
    x = b["input_tensor"][idx, :lmax]
    if x.size(1) < lmax:
        x = torch.nn.functional.pad(x, (0, 0, 0, lmax - x.size(1)))
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(lens, 0)])
    rows = torch.cat([torch.arange(int(off[d]), int(off[d + 1])) for d in idx.tolist()])
    return x.reshape(-1, D).contiguous(), b["speaker_packed"][rows].contiguous(), b["label"][rows].contiguous(), \
        lens[idx].contiguous()


def _reduced_grads(ts, m):
    """{name: the all-reduced gradient in the step's flat buffer} (valid right after a step)."""
    slot = {id(p): v for p, v in zip(ts.opt.live, ts.opt.g_views)}
    return {k: slot[id(p)].detach().cpu().clone() for k, p in m.named_parameters() if id(p) in slot}


def _sharded_worker(rank, world, port, out_dir, steps, global_pad):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import erc_b200  # noqa: F401
    from erc_b200.dist import shard_dialogues
    b = _batch(0, 32)
    idx = shard_dialogues(b["text_length"], world)[rank]
    L = int(b["text_length"].max())
    lmax = L if global_pad else int(b["text_length"][idx].max())
    x, spk, y, lens = _shard(b, idx, lmax)
    m = _no_dropout(_model(3))
    ts = _step(m, lens, lmax=lmax, world=world, group=dist.group.WORLD, transport="nccl")
    assert ts.transport == "torch.distributed"
    x, spk, y = x.cuda(), spk.cuda(), y.cuda()
    losses, grads = [], None
    for _ in range(steps):
        ts.step(x, spk, y)
        losses.append(float(ts.global_loss()))
        grads = grads or _reduced_grads(ts, m)
    ts.check()
    torch.save({"losses": losses, "grads": grads, "params": {k: p.detach().cpu() for k, p in m.named_parameters()},
                "longest": int(lens.max()), "lmax": lmax}, os.path.join(out_dir, "rank%d.pt" % rank))
    dist.destroy_process_group()


def _assert_within_travel(got, m, steps, lr=3e-4):
    travel = steps * lr
    for k, p in m.named_parameters():
        d = (got[k] - p.detach().cpu()).abs()
        assert float(d.max()) <= 0.5 * travel and float(d.mean()) <= 1e-2 * travel, (k, float(d.max()), float(d.mean()))


@pytest.mark.parametrize("padding", ["global", "per_shard"])
def test_two_ranks_on_one_gpu_equal_one_rank_on_the_whole_batch(tmp_path, padding):
    """The batch sharded by dialogue over 2 ranks (two processes on this GPU over gloo, torch.distributed transport, eager,
    dropout off) against one rank on the whole batch.  One shard's longest dialogue (82) is shorter than the batch's (88).
    Every shard padded to the global lmax: every step's loss is the global weighted mean (1e-6), the all-reduced gradient of
    the first step is the whole batch's (1e-5: the shards' GEMMs sum over other row sets) and the parameters after 3 Adam
    steps agree as Adam allows.  Padded to its own length instead, the shorter shard's reverse base starts elsewhere and its
    edge-attention softmax runs over fewer positions: the gradient differs visibly."""
    steps = 3
    mp.spawn(_sharded_worker, args=(2, _free_port(), str(tmp_path), steps, padding == "global"), nprocs=2, join=True)
    b = _batch(0, 32)
    m = _no_dropout(_model(3))
    ts = _step(m, b["text_length"])
    x, spk, y = _cuda(b, "x_rows", "speaker_packed", "label")
    whole, grads = [], None
    for _ in range(steps):
        ts.step(x, spk, y)
        whole.append(float(ts.global_loss()))
        grads = grads or _reduced_grads(ts, m)
    got = [torch.load(str(tmp_path / ("rank%d.pt" % r))) for r in range(2)]
    L = int(b["text_length"].max())
    assert min(g["longest"] for g in got) < L
    if padding == "per_shard":
        assert min(g["lmax"] for g in got) < L
        scale = max(float(v.abs().max()) for v in grads.values())
        worst = max(rel_err(got[0]["grads"][k], grads[k], floor=1e-2 * scale) for k in grads)
        print("per-shard padding: first-step loss %.7f vs whole batch %.7f, worst first-step gradient rel err %.2e"
              % (got[0]["losses"][0], whole[0], worst))
        assert worst > 1e-4
        return
    for r in range(2):
        assert got[r]["lmax"] == L
        for a, c in zip(got[r]["losses"], whole):
            assert abs(a - c) <= 1e-6 * abs(c), (r, got[r]["losses"], whole)
        worst_g = check_grads(got[r]["grads"], grads, 1e-5)
        print("rank %d: losses %s vs %s, first-step gradient rel err %.2e" % (r, got[r]["losses"], whole, worst_g))
        _assert_within_travel(got[r]["params"], m, steps)


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
                        os.path.join(ROOT, "tools", "bench_dgcnv2_step.py"), "--dist-check"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    print(line)
    assert line["transport"].startswith("peer memory")
    assert line["loss_rel_diff"] <= 1e-6 and line["grad_rel_err"] <= 1e-5, line
    travel = line["steps"] * 3e-4
    assert line["param_max_abs_diff"] <= 0.5 * travel and line["param_mean_abs_diff"] <= 1e-2 * travel, line


def test_step_communicator_size_carries_the_first_step_all_reduce():
    """The first step all-reduces the whole flat gradient buffer in one peer-memory call: two endpoints of the size the step
    creates (PeerComm.simulate: the same kernels and flag protocol as across GPUs, on two streams of this GPU) reduce a
    buffer of that length to the rank-ordered sum."""
    from erc_b200.p2p import PeerComm
    b = _batch(0, 32)
    ts = _step(_model(3), b["text_length"])
    ts.step(*_cuda(b, "x_rows", "speaker_packed", "label"))
    n = ts.opt.flat_g.numel()
    assert 4 * n <= ts.comm_bytes
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


# ------------------------------------------------------------------------------------------ K11 argument checks
def test_masked_edge_att_rejects_a_wrongly_shaped_score_matrix():
    """S must be [B * Lmax, >= Lmax]: a wrong row count or fewer than Lmax columns is a ValueError in Python, and the C
    entry points return ERCG_EINVAL for ldS < Lmax (or Lmax < 1) before any launch.  A valid S still gives the result."""
    from erc_b200 import ops_dgcnv2
    from erc_b200._lib import lib
    from erc_b200.graph import build_graph
    lens = torch.tensor([5, 3, 7])
    B, L = 3, 7
    g = build_graph(lens, torch.zeros(int(lens.sum()), dtype=torch.int64, device="cuda"), 2, 1, 1, device="cuda",
                    mean_weight=False)
    S = torch.randn(B * L, 110, device="cuda")
    nu = ops_dgcnv2.masked_edge_att(S, g, L, 2, 1)
    assert nu.shape == (g.E,) and bool(torch.isfinite(nu).all())
    for bad in (S[:-1], torch.randn(B * L + 1, 110, device="cuda"), S[:, :L - 1]):
        with pytest.raises(ValueError):
            ops_dgcnv2.masked_edge_att(bad, g, L, 2, 1)
    f32 = dict(dtype=torch.float32, device="cuda")
    nu2, stat = torch.empty(g.E, **f32), torch.empty((g.N, 2), **f32)
    dnu, dS = torch.ones(g.E, **f32), torch.zeros_like(S)
    p = lambda t: t.data_ptr()  # noqa: E731
    fwd = lambda ldS, Lm: lib().ercg_masked_edge_att_fwd(p(S), ldS, p(g.node_off), p(g.node_dlg), p(g.t_rowptr),  # noqa: E731
                                                         p(g.t_eid), Lm, 2, 1, p(nu2), p(stat), g.N, None)
    bwd = lambda ldS, Lm, ldd: lib().ercg_masked_edge_att_bwd(p(S), ldS, p(g.node_off), p(g.node_dlg),  # noqa: E731
                                                              p(g.t_rowptr), p(g.t_eid), Lm, 2, 1, p(nu2), p(dnu),
                                                              p(stat), p(dS), ldd, g.N, None)
    assert fwd(L - 1, L) == -1 and fwd(110, 0) == -1
    assert bwd(L - 1, L, 110) == -1 and bwd(110, L, L - 1) == -1 and bwd(110, 0, 110) == -1
    assert fwd(110, L) == 0
    torch.cuda.synchronize()
    assert torch.equal(nu2, nu)
