"""oracle/ref_port.py (the timed CPU baseline of bench.py's reference arm) pinned against the outputs of the REAL reference
module stored in tests/golden, and -- when the reference's source tree is present (ref_loader.available()) -- the cogmen.py:114
quirk (GNN always built with n_speakers = 2) pinned for a 9-speaker (MELD-shaped) batch.  CPU only."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import graph_np, ref_loader, ref_port, modules as om
from conftest import rel_err, check_grads

TOL = 1e-5   # fp32 relative, max-norm per tensor (as in test_oracle_models.py)

needs_reference = pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")


def _batch(B, D, n_speakers, n_classes, seed, lo=3, hi=20):
    gen = torch.Generator().manual_seed(seed)
    lens = torch.randint(lo, hi, (B,), generator=gen)
    Lmax = int(lens.max())
    x = torch.randn(B, Lmax, D, generator=gen)
    spk = torch.randint(0, n_speakers, (B, Lmax), generator=gen)
    mask = torch.arange(Lmax)[None, :] < lens[:, None]
    return x * mask[..., None], spk * mask, lens, torch.randint(0, n_classes, (int(lens.sum()),), generator=gen)


def test_ref_port_is_logit_identical_to_the_reference_module(golden):
    """The outputs the reference's COGMENModule and batch_graphify produced for the stored fixtures (oracle/make_golden.py):
    logits, features, loss, every gradient, BatchNorm running statistics, eval-mode logits within the fp32 parity bars of
    test_oracle_models.py (the fixtures were computed on another CPU, whose matmul kernels may round differently); the
    same edges, relation ids and node features, exactly, for every stored graph case."""
    fx = golden("cogmen_small")
    D, C = fx["input_tensor"].shape[-1], fx["logits"].shape[1]
    port = ref_port.CogmenRefPort(D, n_classes=C, skip_dead_encoder=True)    # the encoder's output is dropped (cogmen.py:146-147)
    port.cls[2].p = 0.0                                                      # as in the fixture
    missing, unexpected = port.load_state_dict({k[6:]: torch.from_numpy(v) for k, v in fx.items() if k.startswith("param/")},
                                               strict=False)
    assert not unexpected and all(k.startswith("rnn.0.") for k in missing), (missing, unexpected)
    x, spk, lens, y = (torch.from_numpy(fx[k]) for k in ("input_tensor", "speaker_tensor", "text_length", "label"))
    port.train()
    logits, feats = port(x, spk, lens)
    loss = F.cross_entropy(logits, y)
    loss.backward()
    assert rel_err(logits, fx["logits"]) < TOL and rel_err(feats, fx["features"]) < TOL
    assert abs(float(loss.detach()) - float(fx["loss"])) < TOL * abs(float(fx["loss"]))
    grads = {k: p.grad.numpy() for k, p in port.named_parameters() if p.grad is not None}
    check_grads(grads, {k[5:]: v for k, v in fx.items() if k.startswith("grad/")}, 5 * TOL)
    assert rel_err(port.gcn.bn.running_mean, fx["bn_running_mean"]) < TOL
    assert rel_err(port.gcn.bn.running_var, fx["bn_running_var"]) < TOL
    port.eval()
    with torch.no_grad():
        assert rel_err(port(x, spk, lens)[0], fx["logits_eval"]) < TOL
    # graph construction: same edges, relation ids and per-dialogue edge counts as the reference's batch_graphify
    g = golden("graph")
    for i in range(int(g["n_graph_cases"])):
        n, wp, wf = (int(v) for v in g["g%d_meta" % i])
        rel_ids = {str(a) + str(b) + t: 2 * (a * n + b) + int(t) for a in range(n) for b in range(n) for t in "01"}
        nf, ei, et, el = ref_port.graphify_loop(torch.from_numpy(g["g%d_features" % i]), torch.from_numpy(g["g%d_lengths" % i]),
                                                torch.from_numpy(g["g%d_speakers" % i]), wp, wf, rel_ids)
        order = graph_np.canonical_order(ei.numpy())
        assert np.array_equal(nf.numpy(), g["g%d_node_features" % i]), i
        assert np.array_equal(ei.numpy()[:, order], g["g%d_edge_index" % i]), i
        assert np.array_equal(et.numpy()[order], g["g%d_edge_type" % i]), i
        assert np.array_equal(el.numpy(), g["g%d_edge_index_lengths" % i]), i


@needs_reference
def test_reference_builds_gnn_with_default_speaker_count_and_oracle_follows():
    """cogmen.py:114: ``GNN(hidden, hidden, hidden)`` -- 8 relations for every data set.  With 9 speakers (MELD) relation ids
    run to 161; ids >= 8 are never selected by PyG's per-relation loop, i.e. those edges carry no message."""
    ref = ref_loader.load()
    D, C = 36, 7
    torch.manual_seed(3)
    real = ref.cogmen.COGMENModule(D, 100, 17, 9, C)
    assert tuple(real.gcn.conv1.weight.shape) == (8, 100, 100) and len(real.edge_type_to_idx) == 162
    o = om.CogmenOracle(D, n_speakers=9, n_classes=C, dropout=0.0)
    assert om.load_live(o, real.state_dict()) and tuple(o.gcn.conv1.weight.shape) == (8, 100, 100)
    x, spk, lens, y = _batch(6, D, 9, C, seed=4)
    real.eval()
    o.eval()
    with torch.no_grad():
        a, _ = real(x, spk, lens)
        b, _ = o(x, spk, lens)
    assert float((a - b).abs().max()) <= 1e-5 * float(a.abs().max())


@needs_reference
def test_oracle_gat_step_equals_the_reference_class():
    """dagerc_oracle._Gat (the checker of the stand-alone CUDA GAT step) against the real GAT_dialoggcn_v1
    (dagerc_models.py:312-365): same state_dict, same outputs."""
    from oracle import dagerc_oracle
    ref = ref_loader.load()
    torch.manual_seed(11)
    real = ref.dagerc_models.GAT_dialoggcn_v1(48)
    o = dagerc_oracle._Gat(48)
    o.load_state_dict(real.state_dict(), strict=True)
    gen = torch.Generator().manual_seed(5)
    Q, K = torch.randn(4, 48, generator=gen), torch.randn(4, 9, 48, generator=gen)
    adj = (torch.rand(4, 9, generator=gen) < 0.5).float()
    sm = (torch.rand(4, 9, generator=gen) < 0.5).long()
    w0, s0 = real(Q, K, K, adj, sm)
    w1, s1 = o(Q, K, K, adj, sm)
    assert torch.equal(w0, w1) and torch.equal(s0, s1)
