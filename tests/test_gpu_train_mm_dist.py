"""Data-parallel ``train_mm.py`` under ``torch.distributed.run`` against a one-process emulation of the same run on GPU 0.

The emulation trains the dealt batches (``deal_batches``) of every virtual rank in turn, each with its own CPU generator
state (the dropout seeds come from it, and MMGCN draws them in the test pass too), sums the per-rank flat gradients in rank
order (what the peer-memory all-reduce does), steps Adam with grad_scale = 1/W and keeps rank 0's BatchNorm running
statistics; its test pass evaluates batch i with virtual rank i % W.  Through peer memory the checkpoint must be the
emulation's bit for bit and the logged test metrics the emulation's; through NCCL (ERCG_P2P=0) within 1e-6 per tensor.
With one GPU, two ranks share cuda:0 over a gloo process group (a launcher script in the test's directory swaps the
backend; train_mm itself is unchanged), which checks everything but the transport, bit for bit."""
import json
import os
import re
import signal
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_err

MODULES = {"cogmen": ["--dataset=iemocap-cogmen-sbert-4"], "dgcn": ["--dataset=iemocap-cogmen-6"],
           "dgcnv2": ["--dataset=iemocap-cogmen-6", "--max_len=40"], "mmgcn": ["--dataset=iemocap-cogmen-6"],
           "dagerc": ["--dataset=iemocap-cogmen-6", "--max_len=24"]}
# 19 training dialogues in batches of 4 = 5 batches: the last round of 2 (and of 4) ranks is filled from the list's start;
# 9 test dialogues = 3 test batches, so the ranks evaluate unequal numbers of them (none at all on ranks 3, 4 of 4)
COMMON = ["--modality=atv", "--epoch=2", "--train_dialogues=19", "--test_dialogues=9", "--train.batch_size=4", "--lr=0.001"]


def _need_gpus(n):
    have = torch.cuda.device_count()
    if have < n:
        print("skipped: needs %d GPUs, %d visible" % (n, have))
        pytest.skip("needs %d GPUs, %d visible" % (n, have))


def _launch(world, argv, env_extra, script=None, timeout=900):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(world),
           script or os.path.join(ROOT, "train_mm.py")] + argv
    env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
    env.update(env_extra)
    proc = subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                            start_new_session=True)
    try:
        out, _ = proc.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(proc.pid, signal.SIGKILL)
        out, _ = proc.communicate()
        pytest.fail("torch.distributed.run did not finish in %d s:\n%s" % (timeout, out[-6000:]))
    if proc.returncode != 0:
        try:
            os.killpg(proc.pid, signal.SIGKILL)
        except ProcessLookupError:
            pass
        pytest.fail("torch.distributed.run exited with %d:\n%s" % (proc.returncode, out[-6000:]))
    return out


_EMULATED = {}


@torch.no_grad()
def _test_pass(tr, data, world, run_as):
    from sklearn import metrics
    from erc_b200 import ops
    tr.model.eval()
    bs = tr.p["batch_size"]
    res = []
    for i, s0 in enumerate(range(0, len(data), bs)):
        def ev():
            batch = tr.collate(data[s0:s0 + bs])
            logits = tr._logits(batch)
            ys = batch["label"]
            return float(ops.cross_entropy(logits, ys)), ys.cpu().tolist(), logits.argmax(-1).cpu().tolist()
        res.append(run_as(i % world, ev))
    tr.model.train()
    true, pred, lsum, n = [], [], 0.0, 0
    for ce, ys, ps in res:
        lsum += ce * len(ys)
        n += len(ys)
        true.extend(ys)
        pred.extend(ps)
    return {"Lall": lsum / n, "acc": metrics.accuracy_score(true, pred), "f1": metrics.f1_score(true, pred, average="weighted")}


def _emulate(module, world):
    """(state_dict, ["test Lall ... f1 ..." per epoch], best) of the run of ``world`` ranks, computed in this process."""
    key = (module, world)
    if key in _EMULATED:
        return _EMULATED[key]
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200.train_mm import Trainer, deal_batches, load_data, parse_args, resolve_params
    p = resolve_params(parse_args(["--module=" + module] + COMMON + MODULES[module]))
    train, test, _ = load_data(p)
    tr = Trainer(p)                                   # cuda:0, same seed and model initialisation as every rank
    opt = tr.optim
    opt.grad_scale = 1.0 / world
    rng = [torch.get_rng_state() for _ in range(world)]

    def run_as(r, fn):
        torch.set_rng_state(rng[r])
        out = fn()
        rng[r] = torch.get_rng_state()
        return out

    buffers = [b for _, b in tr.model.named_buffers()]
    lines, best = [], {}
    bs = p["batch_size"]
    for epoch in range(1, p["epoch"] + 1):
        order = np.random.default_rng(p["seed"] * 100003 + epoch).permutation(len(train))
        batches = [order[i:i + bs] for i in range(0, len(order), bs)]
        for dealt in deal_batches(len(batches), world):
            total = None
            for r, b in enumerate(dealt):
                keep = [t.clone() for t in buffers] if r > 0 else None    # only rank 0's running statistics count

                def fwd_bwd():
                    batch = tr.collate([train[j] for j in batches[b]])
                    loss = ops.cross_entropy(tr._logits(batch), batch["label"], tr.class_weight)
                    opt.zero_grad()
                    loss.backward()
                run_as(r, fwd_bwd)
                if keep is not None:
                    for t, k in zip(buffers, keep):
                        t.copy_(k)
                if opt.live is None:
                    opt.attach()
                opt.gather()
                g = opt.flat_g[:opt.n]
                total = g.clone() if total is None else total.add_(g)      # rank order, fp32, as ercg_p2p_allreduce adds
            opt.flat_g[:opt.n].copy_(total)
            opt.update()
        te = _test_pass(tr, test, world, run_as)
        lines.append("test Lall %.4f acc %.3f f1 %.3f" % (te["Lall"], te["acc"], te["f1"]))
        if te["f1"] >= best.get("f1", -1.0):
            best = {"f1": te["f1"], "acc": te["acc"], "epoch": epoch}
    torch.cuda.synchronize()
    sd = {k: v.detach().cpu().clone() for k, v in tr.model.state_dict().items()}
    _EMULATED[key] = (sd, lines, best)
    return _EMULATED[key]


GLOO_ON_ONE_GPU = """import os, sys
sys.path.insert(0, %r)
import torch.distributed as dist
_init = dist.init_process_group
dist.init_process_group = lambda backend, device_id=None, **kw: _init("gloo", **kw)
os.environ["LOCAL_RANK"] = "0"
import erc_b200
from erc_b200.train_mm import main
main()
"""


def _run_and_compare(module, world, transport, tmp_path):
    env, script = ({"ERCG_P2P": "0"}, None) if transport in ("nccl", "gloo") else ({}, None)
    if transport == "gloo":
        script = os.path.join(str(tmp_path), "gloo_on_one_gpu.py")
        with open(script, "w") as f:
            f.write(GLOO_ON_ONE_GPU % ROOT)
    save = os.path.join(str(tmp_path), "ckpt")
    out = _launch(world, ["--module=" + module] + COMMON + MODULES[module] + ["--save_dir=" + save], env, script)
    want_transport = "peer memory" if transport == "p2p" else "torch.distributed"
    assert re.search(r"gradient all-reduce of \d+ floats over %d GPUs through %s" % (world, want_transport), out), out[-3000:]
    got = torch.load(os.path.join(save, "last_model.ckpt"))
    sd, lines, best = _emulate(module, world)
    assert set(got) == set(sd)
    if transport in ("p2p", "gloo"):                   # rank-ordered sums (two ranks: any order is the same sum)
        diff = [k for k in sd if not torch.equal(got[k], sd[k])]
        assert not diff, diff
        logged = re.findall(r"test Lall \S+ acc \S+ f1 \S+", out)
        assert logged == lines, (logged, lines)
        res = json.loads(re.search(r"Best Results (\{.*\})", out).group(1))
        assert res == best, (res, best)
    else:
        worst = {k: rel_err(got[k].double(), sd[k].double()) for k in sd if sd[k].is_floating_point()}
        assert max(worst.values()) <= 1e-6, worst
        assert all(torch.equal(got[k], sd[k]) for k in sd if not sd[k].is_floating_point())


@pytest.mark.gpu
@pytest.mark.parametrize("transport", ["p2p", "nccl"])
@pytest.mark.parametrize("module", list(MODULES))
def test_two_gpus_match_the_emulation(module, transport, tmp_path):
    _need_gpus(2)
    _run_and_compare(module, 2, transport, tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("module", list(MODULES))
def test_two_ranks_on_one_gpu_match_the_emulation(module, tmp_path):
    _need_gpus(1)
    _run_and_compare(module, 2, "gloo", tmp_path)


@pytest.mark.gpu
def test_four_gpus_match_the_emulation(tmp_path):
    _need_gpus(4)
    _run_and_compare("cogmen", 4, "p2p", tmp_path)
