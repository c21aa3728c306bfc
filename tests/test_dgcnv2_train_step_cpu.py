"""Host-side checks of the dgcnv2 train step that need no GPU: the constructor's argument checks, the late gradient bucket
of each base, the size of the step's communicators against its flat gradient buffer, and the argument checks of the K11
edge attention (Python and C ABI: both return before any launch)."""
import types

import pytest
import torch


def _model(base="LSTM"):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dgcnv2 import DGCNModule
    torch.manual_seed(0)
    return DGCNModule(base, input_size=1380, hidden_size=100, n_speakers=2, n_classes=6)


def test_constructor_rejects_bad_lengths_and_lmax():
    from erc_b200.train_step import Dgcnv2TrainStep
    m = _model()
    for bad in ([], [[3, 4]], [3, 0, 5], [2.0, 3.0]):
        with pytest.raises(ValueError):
            Dgcnv2TrainStep(m, torch.tensor(bad))
    with pytest.raises(ValueError):
        Dgcnv2TrainStep(m, torch.tensor([40, 61, 17]), lmax=60)          # shorter than the longest dialogue
    with pytest.raises(ValueError):
        Dgcnv2TrainStep(m, torch.tensor([40, 61, 17]), lmax=111)         # beyond max_seq_len (MaskedEdgeAttention's 110)
    with pytest.raises(ValueError):
        Dgcnv2TrainStep(m, torch.tensor([40, 111]))
    with pytest.raises(ValueError):
        Dgcnv2TrainStep(m, torch.tensor([40, 61]), world=0)
    with pytest.raises(ValueError):
        Dgcnv2TrainStep(m, torch.tensor([40, 61]), transport="mpi")
    ts = Dgcnv2TrainStep(m, torch.tensor([40, 61, 17]), lmax=110)
    assert ts.lmax == 110 and ts.sizes[0] == 118
    assert Dgcnv2TrainStep(m, torch.tensor([40, 61, 17])).lmax == 61


@pytest.mark.parametrize("base,late", [
    ("LSTM", {"lstm.%s_l0%s" % (n, d) for n in ("weight_ih", "bias_ih", "bias_hh") for d in ("", "_reverse")}),
    ("GRU", {"gru.%s_l0%s" % (n, d) for n in ("weight_ih", "bias_ih") for d in ("", "_reverse")}),
    ("None", {"base_linear.weight", "base_linear.bias"}),
])
def test_late_bucket_is_the_layer0_input_transform(base, late):
    from erc_b200.train_step import Dgcnv2TrainStep
    m = _model(base)
    ts = Dgcnv2TrainStep(m, torch.tensor([40, 61, 17]))
    ids = {id(p) for p in ts._late_params()}
    assert {k for k, p in m.named_parameters() if id(p) in ids} == late


def test_dgcnv2_step_communicators_hold_the_whole_flat_gradient():
    """The first step (and every step without overlap) all-reduces the whole flat gradient buffer in one peer-memory call,
    so the communicators must hold it."""
    from erc_b200.train_step import Dgcnv2TrainStep
    m = _model()
    ts = Dgcnv2TrainStep(m, torch.tensor([40, 61, 17]))
    for k, p in m.named_parameters():
        if not (k.startswith("att_model.") and not k.startswith("att_model.scalar")):
            p.grad = torch.zeros_like(p)
    ts._attach()
    nbytes = ts.opt.flat_g.numel() * 4
    assert ts.comm_bytes >= max(nbytes, 8 << 20), (nbytes, ts.comm_bytes)


def test_masked_edge_att_rejects_bad_shapes_before_any_launch():
    import erc_b200  # noqa: F401
    from erc_b200 import ops_dgcnv2
    from erc_b200._lib import lib
    g = types.SimpleNamespace(B=3)
    for S in (torch.zeros(3 * 7 - 1, 110), torch.zeros(3 * 7 + 1, 110), torch.zeros(3 * 7, 6), torch.zeros(21)):
        with pytest.raises(ValueError):
            ops_dgcnv2.masked_edge_att(S, g, 7, 10, 10)
    ptr = 4096                                                # any non-null address: never dereferenced on these paths
    fwd = lambda ldS, L: lib().ercg_masked_edge_att_fwd(ptr, ldS, ptr, ptr, ptr, ptr, L, 10, 10, ptr, ptr, 5, None)  # noqa: E731
    bwd = lambda ldS, L, ldd: lib().ercg_masked_edge_att_bwd(ptr, ldS, ptr, ptr, ptr, ptr, L, 10, 10, ptr, ptr, ptr,  # noqa: E731
                                                             ptr, ldd, 5, None)
    assert fwd(6, 7) == -1 and fwd(110, 0) == -1 and fwd(110, -1) == -1
    assert bwd(6, 7, 110) == -1 and bwd(110, 7, 6) == -1 and bwd(110, 0, 110) == -1
