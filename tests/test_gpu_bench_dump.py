"""bench.py --dump-outputs on the GPU: the files hold what the last timed step (a CUDA-graph replay) returned, and --steps
sets how many steps that was."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                        "--total-utts", "4096", "--e2e-steps", "1", "--no-cpu-baseline", "--no-bf16-mode",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    import torch
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.cogmen import COGMENModule
    torch.manual_seed(0)                                    # bench.py builds its model right after the same call
    init = {n: p.detach().numpy().copy() for n, p in COGMENModule(1443, 100, 17, 2, 6).named_parameters()
            if not n.startswith("rnn.0.")}                  # the dead encoder is never updated
    runs = {}
    for steps in (2, 3):
        line, out = _bench(tmp_path / ("steps%d" % steps), steps)
        assert line["steps"] == steps and len(line["graph"]["step_ms"]) == steps
        assert set(out) == ({"loss", "buffer.gcn.bn.running_mean", "buffer.gcn.bn.running_var"} |
                            {"param." + n for n in init})
        for k, v in out.items():
            assert v.dtype == np.float32 and np.isfinite(v).all(), k
        for n, p in init.items():
            assert out["param." + n].shape == p.shape, n
        assert out["loss"].shape == (1,) and float(out["loss"][0]) == line["loss"]     # the loss of the last graph replay
        assert not np.array_equal(out["param.rnn.1.weight"], init["rnn.1.weight"])    # Adam has moved the projection
        runs[steps] = out
    # one more timed step: the loss and the parameters are those of a later step
    assert runs[2]["loss"][0] != runs[3]["loss"][0]
    assert not np.array_equal(runs[2]["param.rnn.1.weight"], runs[3]["param.rnn.1.weight"])
