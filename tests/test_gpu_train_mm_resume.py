"""Resuming ``train_mm.py`` from a ``--ckpt_layout=reference`` checkpoint on an IEMOCAP-shaped synthetic set: a run of
2 epochs resumed up to 4 must end in the uninterrupted 4-epoch run's checkpoint bit for bit (weights, buffers, Adam moments,
step, every rank's CPU generator) and log the same test metrics, on one GPU and data-parallel; torch.optim.Adam continues
from the checkpoint's optimizer state as FlatAdam does; a checkpoint of another run is refused.  The eager path reduces
in a fixed order, so any difference is a bug, not noise."""
import os
import re
import signal
import subprocess
import sys

import pytest
import torch

from conftest import ROOT, rel_err

pytestmark = pytest.mark.gpu

MODULES = {"cogmen": ["--dataset=iemocap-cogmen-sbert-4"], "dgcn": ["--dataset=iemocap-cogmen-6"],
           "dgcnv2": ["--dataset=iemocap-cogmen-6", "--max_len=40"], "mmgcn": ["--dataset=iemocap-cogmen-6"],
           "dagerc": ["--dataset=iemocap-cogmen-6", "--max_len=24"]}
COMMON = ["--modality=atv", "--train_dialogues=24", "--test_dialogues=8", "--train.batch_size=8", "--lr=0.001",
          "--ckpt_layout=reference"]
METRICS = re.compile(r"test Lall \S+ acc \S+ f1 \S+")


def _main(module, save, *extra):
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import main
    lines = []
    main(["--module=" + module] + COMMON + MODULES[module] + ["--save_dir=" + save] + list(extra),
         log=lambda *a: lines.append(" ".join(str(x) for x in a)))
    return lines


def _load(d):
    return torch.load(os.path.join(d, "last_model.ckpt"), weights_only=True)


def _assert_same_checkpoint(a, b):
    """Every tensor bit for bit; the records equal except the measured throughput."""
    assert set(a) == set(b) == {"models", "optims", "others", "thtensor", "nptensor"}
    ma, mb = a["models"]["model"], b["models"]["model"]
    assert list(ma) == list(mb)
    diff = [k for k in ma if not torch.equal(ma[k], mb[k])]
    assert not diff, diff
    oa, ob = a["optims"]["optim"], b["optims"]["optim"]
    assert oa["param_groups"] == ob["param_groups"] and list(oa["state"]) == list(ob["state"]) and oa["state"]
    diff = [(i, k) for i in oa["state"] for k in ("step", "exp_avg", "exp_avg_sq")
            if not torch.equal(oa["state"][i][k], ob["state"][i][k])]
    assert not diff, diff
    ta, tb = a["others"]["train_mm"], b["others"]["train_mm"]
    assert ta["epoch"] == tb["epoch"] and ta["params"] == tb["params"] and ta["best"] == tb["best"]
    assert len(ta["rng"]) == len(tb["rng"]) and all(torch.equal(x, y) for x, y in zip(ta["rng"], tb["rng"]))
    strip = lambda h: [{k: v for k, v in r.items() if k != "utt_per_s"} for r in h]
    assert strip(ta["history"]) == strip(tb["history"])


_RUNS = {}


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """module -> directories of the uninterrupted 4-epoch run, the 2-epoch run and its resumption to epoch 4, with logs."""
    def get(module):
        if module not in _RUNS:
            base = str(tmp_path_factory.mktemp(module))
            full, two, resumed = (os.path.join(base, n) for n in ("full", "two", "resumed"))
            lines_full = _main(module, full, "--epoch=4")
            _main(module, two, "--epoch=2")
            lines_resumed = _main(module, resumed, "--epoch=4", "--resume=" + os.path.join(two, "last_model.ckpt"))
            _RUNS[module] = dict(full=full, two=two, resumed=resumed, lines_full=lines_full, lines_resumed=lines_resumed)
        return _RUNS[module]
    return get


@pytest.mark.parametrize("module", list(MODULES))
def test_resumed_run_is_the_uninterrupted_run(module, runs):
    r = runs(module)
    assert any(l.startswith("train_mm: resuming") for l in r["lines_resumed"])
    assert _load(r["two"])["others"]["train_mm"]["epoch"] == 2
    full, resumed = _load(r["full"]), _load(r["resumed"])
    assert full["others"]["train_mm"]["epoch"] == 4
    _assert_same_checkpoint(full, resumed)
    epochs_full = [METRICS.search(l).group(0) for l in r["lines_full"] if l.startswith("epoch ")]
    epochs_resumed = [METRICS.search(l).group(0) for l in r["lines_resumed"] if l.startswith("epoch ")]
    assert len(epochs_full) == 4 and epochs_resumed == epochs_full[2:]
    best = lambda lines: [l for l in lines if l.startswith("Best Results")]
    assert best(r["lines_full"]) == best(r["lines_resumed"])


@pytest.mark.parametrize("module", list(MODULES))
def test_torch_optim_continues_like_flat_adam(module, runs):
    """The 2-epoch checkpoint into a fresh module + torch.optim.Adam (AdamW + clip_grad_norm_(5) for DAG-ERC) and into
    one + FlatAdam; one step on the same batch: the parameters agree to FlatAdam's bar against torch.optim
    (tests/test_gpu_train_step.py)."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops
    from erc_b200.train_mm import Trainer, load_data, parse_args, resolve_params
    ck = torch.load(os.path.join(runs(module)["two"], "last_model.ckpt"), weights_only=True)
    osd = ck["optims"]["optim"]
    p = resolve_params(parse_args(["--module=" + module] + COMMON + MODULES[module]))
    samples = load_data(p)[0][:p["batch_size"]]
    flat, ref = Trainer(p, log=lambda *a: None), Trainer(p, log=lambda *a: None)
    for tr in (flat, ref):
        tr.model.load_state_dict(ck["models"]["model"])
    step = int(next(iter(osd["state"].values()))["step"])     # read now: torch.optim steps the loaded tensor in place
    flat.optim.load_state_dict(osd, flat.param_names)
    cls = torch.optim.AdamW if p["optim"] == "AdamW" else torch.optim.Adam
    opt = cls(ref.model.parameters(), lr=p["lr"], weight_decay=p["weight_decay"])
    opt.load_state_dict(osd)
    for g in opt.param_groups:
        g.update(foreach=False, fused=False)                 # the single-tensor formulation of the bar's reference
    assert opt.param_groups[0]["lr"] == p["lr"] and len(opt.state) == len(osd["state"])
    for tr in (flat, ref):
        torch.manual_seed(7)                                 # the same dropout seeds in both models
        batch = tr.collate(samples)
        loss = ops.cross_entropy(tr._logits(batch), batch["label"], tr.class_weight)
        tr.optim.zero_grad()
        loss.backward()
    flat.optim.step()
    if module == "dagerc":
        torch.nn.utils.clip_grad_norm_(ref.model.parameters(), 5.0)
    opt.step()
    assert int(flat.optim.step_dev.item()) == step + 1 == 7          # 2 epochs of 3 batches, then this one
    before = ck["models"]["model"]
    moved = 0
    for (k, a), b in zip(flat.model.named_parameters(), ref.model.parameters()):
        assert rel_err(a, b) < 2e-6, k
        moved += not torch.equal(a.detach().cpu(), before[k])
    assert moved > 0


def test_load_evaluates_a_checkpoint(runs):
    """--load=<checkpoint> --epoch=0 --eval_first: the test pass of the loaded weights is the one the run logged last."""
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import main
    path = os.path.join(runs("dgcn")["full"], "last_model.ckpt")
    last = torch.load(path, weights_only=True)["others"]["train_mm"]["history"][-1]
    lines = []
    out = main(["--module=dgcn"] + COMMON + MODULES["dgcn"] + ["--epoch=0", "--eval_first=True", "--load=" + path],
               log=lambda *a: lines.append(a))
    assert out["history"] == []
    got = [a[1] for a in lines if a[0] == "eval_first:"][0]
    assert [float(got[k]) for k in ("Lall", "acc", "f1")] == [last["test_" + k] for k in ("Lall", "acc", "f1")]


def test_resume_refuses_another_run(runs, tmp_path):
    """Another batch size or module: SystemExit naming the parameter, nothing trained, nothing written."""
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import main
    ck = os.path.join(runs("dgcn")["two"], "last_model.ckpt")
    for module, extra, what in (("dgcn", ["--train.batch_size=4"], r"batch_size=4 \(checkpoint: 8\)"),
                                ("mmgcn", [], r"module='mmgcn' \(checkpoint: 'dgcn'\)")):
        lines, save = [], str(tmp_path / module)
        with pytest.raises(SystemExit, match=what):
            main(["--module=" + module] + COMMON + MODULES[module] + ["--epoch=4", "--resume=" + ck, "--save_dir=" + save]
                 + extra, log=lambda *a: lines.append(" ".join(str(x) for x in a)))
        assert not os.path.exists(save) and not any(l.startswith("epoch ") for l in lines)


# ------------------------------------------------------------------------------------------------ data-parallel
# 19 training dialogues in batches of 4 = 5 batches (the last round is filled from the list's start); 9 test dialogues =
# 3 test batches, so the ranks evaluate unequal numbers of them and MMGCN's ranks draw different numbers of dropout seeds
DIST = ["--modality=atv", "--train_dialogues=19", "--test_dialogues=9", "--train.batch_size=4", "--lr=0.001",
        "--ckpt_layout=reference"]

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


def _dist_resume(module, transport, tmp_path):
    env, script = {}, None
    if transport == "gloo":                                  # two ranks share cuda:0 over gloo
        env = {"ERCG_P2P": "0"}
        script = os.path.join(str(tmp_path), "gloo_on_one_gpu.py")
        with open(script, "w") as f:
            f.write(GLOO_ON_ONE_GPU % ROOT)
    argv = ["--module=" + module] + DIST + MODULES[module]
    full, two, resumed = (os.path.join(str(tmp_path), n) for n in ("full", "two", "resumed"))
    out_full = _launch(2, argv + ["--epoch=4", "--save_dir=" + full], env, script)
    _launch(2, argv + ["--epoch=2", "--save_dir=" + two], env, script)
    out_resumed = _launch(2, argv + ["--epoch=4", "--save_dir=" + resumed, "--resume=" + os.path.join(two, "last_model.ckpt")],
                          env, script)
    want = "peer memory" if transport == "p2p" else "torch.distributed"
    assert re.search(r"gradient all-reduce of \d+ floats over 2 GPUs through %s" % want, out_resumed), out_resumed[-3000:]
    a, b = _load(full), _load(resumed)
    assert a["others"]["train_mm"]["params"]["world"] == 2 and len(a["others"]["train_mm"]["rng"]) == 2
    _assert_same_checkpoint(a, b)
    logged = lambda out: [m.group(0) for m in METRICS.finditer(out)]
    assert len(logged(out_full)) == 4 and logged(out_resumed) == logged(out_full)[2:]
    return os.path.join(two, "last_model.ckpt")


@pytest.mark.parametrize("module", ["mmgcn", "cogmen"])
def test_two_ranks_on_one_gpu_resume_bit_for_bit(module, tmp_path):
    _need_gpus(1)
    ck = _dist_resume(module, "gloo", tmp_path)
    # one process cannot continue a run of two
    import erc_b200  # noqa: F401
    from erc_b200.train_mm import main
    lines = []
    with pytest.raises(SystemExit, match=r"world=1 \(checkpoint: 2\)"):
        main(["--module=" + module] + DIST + MODULES[module] + ["--epoch=4", "--resume=" + ck,
                                                                "--save_dir=" + str(tmp_path / "one")],
             log=lambda *a: lines.append(" ".join(str(x) for x in a)))
    assert not os.path.exists(str(tmp_path / "one")) and not any(l.startswith("epoch ") for l in lines)


def test_two_gpus_resume_bit_for_bit(tmp_path):
    _need_gpus(2)
    _dist_resume("mmgcn", "p2p", tmp_path)
