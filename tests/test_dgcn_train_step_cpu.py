"""Host-side checks of the DialogueGCN train step's pieces that need no GPU: ercg_dropout_dev's argument checks through the
C ABI (they return before any launch), the new kernel's register / spill report, and the size of the step's communicators
against its flat gradient buffer."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT


def test_dropout_dev_rejects_bad_arguments_before_any_launch():
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    f = lib().ercg_dropout_dev
    word = 4096                                             # any non-null address: never dereferenced on these paths
    assert f(None, None, 8, 0.4, 1, None, None) == -1       # seed_dev NULL
    assert f(None, None, -1, 0.4, 1, word, None) == -1      # n < 0
    assert f(None, None, 8, 1.0, 1, word, None) == -1       # p outside [0, 1)
    assert f(None, None, 8, -0.5, 1, word, None) == -1
    assert f(None, None, 8, float("nan"), 1, word, None) == -1
    assert f(None, None, 8, 0.4, 1, word, None) == -1       # null x / out
    assert f(None, None, 0, 0.4, 1, word, None) == 0        # n == 0: nothing to do


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.isfile("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
def test_dropout_dev_kernel_does_not_spill(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    csrc = os.path.join(ROOT, "emotion-recognition-in-conversation_b200", "csrc")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                        "--expt-relaxed-constexpr", "-DERCG_BUILD", "-I", os.path.join(ROOT, "include"), "-Xptxas", "-v", "-c",
                        os.path.join(csrc, "lstm.cu"), "-o", str(tmp_path / "lstm.o")], capture_output=True, text=True, cwd=csrc)
    assert r.returncode == 0, r.stderr[-2000:]
    m = re.search(r"Function properties for \w*dropout_dev_kernel\w*\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads", r.stderr)
    assert m is not None, r.stderr[-2000:]
    assert m.groups() == ("0", "0", "0"), m.groups()


def test_dgcn_step_communicators_hold_the_whole_flat_gradient():
    """The first step (and every step without overlap) all-reduces the whole flat gradient buffer in one peer-memory call, so
    the communicators must hold it.  At the IEMOCAP atv width (1380) that buffer is larger than COGMEN's 8 MB."""
    import torch
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcn import DGCNModule
    from erc_b200.train_step import DgcnTrainStep
    torch.manual_seed(0)
    m = DGCNModule(2, input_size=1380, hidden_size=200, n_classes=6)
    ts = DgcnTrainStep(m, torch.tensor([40, 61, 17]))
    for k, p in m.named_parameters():
        if not k.startswith("clf.emotion_att"):
            p.grad = torch.zeros_like(p)
    ts._attach()
    nbytes = ts.opt.flat_g.numel() * 4
    assert nbytes > 8 << 20 and ts.comm_bytes >= nbytes, (nbytes, ts.comm_bytes)
