"""Host-side checks of the MMGCN and DAG-ERC train steps' pieces that need no GPU: the argument checks of
ercg_gcnii_layer_fwd_dev and ercg_relu_dropout_dev through the C ABI (they return before any launch), the new kernels'
register / spill report, the step constructors' argument checks, and the size of each step's communicators against its
flat gradient buffer."""
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT

WORD = 4096                                                  # any non-null address: never dereferenced on these paths
NAN = float("nan")


def test_relu_dropout_dev_rejects_bad_arguments_before_any_launch():
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    f = lib().ercg_relu_dropout_dev
    assert f(None, None, 8, 0.4, 1, None, None) == -1        # seed_dev NULL
    assert f(None, None, -1, 0.4, 1, WORD, None) == -1       # n < 0
    for p in (1.0, -0.5, NAN):                               # p outside [0, 1)
        assert f(None, None, 8, p, 1, WORD, None) == -1
    assert f(None, None, 8, 0.4, 1, WORD, None) == -1        # null x / out
    assert f(None, None, 0, 0.4, 1, WORD, None) == 0         # n == 0: nothing to do
    assert f(None, None, 0, 0.0, 1, WORD, None) == 0


def test_gcnii_layer_fwd_dev_rejects_what_the_host_seeded_entry_rejects():
    import erc_b200  # noqa: F401
    from erc_b200._lib import lib
    dev, host = lib().ercg_gcnii_layer_fwd_dev, lib().ercg_gcnii_layer_fwd
    H = 16

    def both(M, H, p, ptr=None, ld=H):
        args = (ptr, ld, ptr, ld, ptr, ld, ptr, ld, M, H, 0.5, 0.1, 1, p, 7)
        return dev(*args, WORD, None), host(*args, None)

    assert dev(None, H, None, H, None, H, None, H, 4, H, 0.5, 0.1, 1, 0.4, 7, None, None) == -1   # seed_dev NULL
    assert dev(None, H, None, H, None, H, None, H, 0, H, 0.5, 0.1, 1, 0.4, 7, None, None) == -1   # ... even when M == 0
    assert both(-1, H, 0.4) == (-1, -1)                     # M < 0
    for p in (1.0, -0.5, NAN):                               # p outside [0, 1)
        assert both(4, H, p, ptr=WORD) == (-1, -1)
    assert both(4, 12, 0.4, ptr=WORD) == (-1, -1)           # H % 8 != 0
    assert both(4, 0, 0.4, ptr=WORD) == (-1, -1)            # H <= 0
    assert both(4, H, 0.4) == (-1, -1)                      # null operands
    assert both(4, H, 0.4, ptr=WORD, ld=8) == (-1, -1)      # leading dimension < H
    assert both(0, H, 0.4) == (0, 0)                        # M == 0: nothing to do


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.isfile("/usr/local/cuda/bin/nvcc"), reason="needs nvcc")
@pytest.mark.parametrize("src,kernel", [("gemm_simt.cu", "gcnii_fwd_dev_kernel"), ("mmgcn.cu", "relu_dropout_dev_kernel")])
def test_device_seeded_kernels_do_not_spill(tmp_path, src, kernel):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    csrc = os.path.join(ROOT, "emotion-recognition-in-conversation_b200", "csrc")
    r = subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
                        "--expt-relaxed-constexpr", "-DERCG_BUILD", "-I", os.path.join(ROOT, "include"), "-Xptxas", "-v", "-c",
                        os.path.join(csrc, src), "-o", str(tmp_path / "k.o")], capture_output=True, text=True, cwd=csrc)
    assert r.returncode == 0, r.stderr[-2000:]
    m = re.search(r"Function properties for \w*%s\w*\s*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                  r"(\d+) bytes spill loads" % kernel, r.stderr)
    assert m is not None, r.stderr[-2000:]
    assert m.groups() == ("0", "0", "0"), m.groups()


def _mmgcn():
    import torch
    from erc_b200.track_mm.mmgcn import MMGCNModule
    torch.manual_seed(0)
    return MMGCNModule(hidden_text=768, hidden_visual=512, hidden_audio=100, n_speakers=2, n_classes=6)


def _dagerc():
    import torch
    from erc_b200.track_mm.dagerc import DAGERCModule
    torch.manual_seed(0)
    return DAGERCModule(emb_dim=1380, dropout=0.0, gnn_layers=4, n_classes=6)


def test_step_constructors_reject_bad_arguments():
    import torch
    import erc_b200  # noqa: F401
    from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep
    lens = torch.tensor([5, 9, 3])
    for cls, model in ((MmgcnTrainStep, _mmgcn()), (DagercTrainStep, _dagerc())):
        for bad in (torch.tensor([], dtype=torch.int64), torch.tensor([4, 0]), torch.tensor([4, -2]), torch.tensor([4.0, 2.0]),
                    torch.tensor([[4, 2]])):
            with pytest.raises(ValueError):
                cls(model, bad)
        for world in (0, -1, 1.5, True):
            with pytest.raises(ValueError):
                cls(model, lens, world=world)
        with pytest.raises(ValueError):
            cls(model, lens, transport="nvlink")
    with pytest.raises(ValueError):
        MmgcnTrainStep(_mmgcn(), lens, lmax=8)                # shorter than the longest dialogue
    assert MmgcnTrainStep(_mmgcn(), lens).lmax == 9 and MmgcnTrainStep(_mmgcn(), lens, lmax=12).lmax == 12
    for max_norm in (0.0, -1.0, NAN):
        with pytest.raises(ValueError):
            DagercTrainStep(_dagerc(), lens, max_norm=max_norm)
    ts = DagercTrainStep(_dagerc(), lens, max_norm=None)
    assert ts.opt.max_norm is None and ts.opt.decoupled
    ts = DagercTrainStep(_dagerc(), lens)
    assert ts.opt.max_norm == 5.0 and ts.opt.decoupled and (ts.opt.lr, ts.opt.weight_decay) == (1e-3, 1e-2)
    # compute_padding: the graph runs every dialogue over Lmax; utterance i has at most i predecessors
    assert ts.graph_lengths.tolist() == [9, 9, 9] and ts.e_cap == 3 * 36 and ts.sizes[0] == 27
    ts = MmgcnTrainStep(_mmgcn(), lens)
    assert not ts.opt.decoupled and (ts.opt.lr, ts.opt.weight_decay) == (3e-4, 3e-5)


@pytest.mark.parametrize("which", ["mmgcn", "dagerc"])
def test_step_communicators_hold_the_whole_flat_gradient(which):
    """The first step (and every step without overlap) all-reduces the whole flat gradient buffer in one peer-memory call, so
    the communicators must hold it.  At the IEMOCAP widths both buffers are larger than COGMEN's 8 MB."""
    import torch
    import erc_b200  # noqa: F401
    from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep
    if which == "mmgcn":
        m, cls = _mmgcn(), MmgcnTrainStep
        dead = ("att_model.", "gatedatt.", "graph_model.a_fc", "graph_model.v_fc", "graph_model.l_fc",
                "graph_model.feature_fc", "graph_model.final_fc", "graph_model.modal_embeddings", "graph_model.a_spk_embs",
                "graph_model.v_spk_embs", "graph_model.l_spk_embs")
    else:
        m, cls = _dagerc(), DagercTrainStep
        dead = ("fcs.", "attentive_node_features.")
    ts = cls(m, torch.tensor([40, 61, 17]))
    for k, p in m.named_parameters():
        if not k.startswith(dead):
            p.grad = torch.zeros_like(p)
    ts._attach()
    nbytes = ts.opt.flat_g.numel() * 4
    assert nbytes > 16 << 20 and ts.comm_bytes >= nbytes, (nbytes, ts.comm_bytes)
