"""DAG-ERC (SURVEY.md 8a rows a17-a19) through the drop-in module: K9 predecessor structure bit-exact against the
reference's get_adj_v1 / get_s_mask, K10 layer kernel + module against the reference-generated fixture and the CPU oracle."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import copy

from conftest import rel_err, parity_check
from oracle import dagerc_oracle, seeded
from oracle.make_golden import DAGERC_SEED, dagerc_inputs
from test_oracle_mmgcn import check_against_fixture

pytestmark = pytest.mark.gpu
TOL = 1e-5


def test_dense_masks_bit_exact_vs_reference_fixture(golden):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dagerc import DAGERCModule
    fx = golden("dagerc_small")
    m = DAGERCModule(emb_dim=fx["input_tensor"].shape[-1], dropout=0.0, n_classes=6).cuda()
    L = fx["input_tensor"].shape[1]
    adj = m.get_adj_v1(fx["speaker_tensor"].tolist(), L)           # nested lists, as the reference passes them
    sm, onehot = m.get_s_mask(torch.from_numpy(fx["speaker_tensor"]), L)
    assert adj.dtype == torch.float32 and sm.dtype == torch.int64
    assert np.array_equal(adj.cpu().numpy(), fx["adj"]) and np.array_equal(sm.cpu().numpy(), fx["s_mask"])
    assert onehot.shape == sm.shape + (2,)


@pytest.mark.parametrize("windowp", [1, 2])
def test_dag_structure_random_speakers(windowp):
    import erc_b200  # noqa: F401
    from erc_b200 import ops_dagerc
    from erc_b200.graph import build_graph
    gen = torch.Generator().manual_seed(3)
    lengths = torch.tensor([1, 17, 110, 2, 64, 5000 // 100])
    B, Lmax = lengths.numel(), int(lengths.max())
    spk = torch.randint(0, 3, (B, Lmax), generator=gen)
    g = build_graph(lengths, spk.cuda(), 0, 0, 3, reference_layout=False, mean_weight=False)
    dag = ops_dagerc.DagStructure(g, lengths, windowp)
    want = dagerc_oracle.adj_v1(spk.numpy(), windowp)
    lo, cnt, eoff = dag.lo.cpu().numpy(), dag.cnt.cpu().numpy(), dag.eoff.cpu().numpy()
    off = np.concatenate([[0], np.cumsum(lengths.numpy())])
    for b in range(B):
        for i in range(int(lengths[b])):
            row = want[b, i, :int(lengths[b])]
            nz = np.nonzero(row)[0]
            n = off[b] + i
            assert cnt[n] == len(nz)
            if len(nz):
                assert lo[n] == nz[0] and nz[-1] == i - 1 and len(nz) == i - nz[0]
    assert np.array_equal(eoff, np.concatenate([[0], np.cumsum(cnt)[:-1]])) and dag.E == int(cnt.sum())
    dense, sm = ops_dagerc.dense_masks(spk.cuda(), windowp)
    assert np.array_equal(dense.cpu().numpy(), want) and np.array_equal(sm.cpu().numpy(), dagerc_oracle.s_mask(spk.numpy()))


def _oracle_runs(emb, C, b):
    """DagercOracle (same name-seeded weights) in fp32 and in fp64 -> ((logits, grads) fp32, (logits, grads) fp64)."""
    o = dagerc_oracle.DagercOracle(emb, n_classes=C, dropout=0.0)
    seeded.fill_by_name(o, DAGERC_SEED)
    res = []
    for dt in (torch.float32, torch.float64):
        oo = copy.deepcopy(o).to(dt)
        oo.train()
        ol, _ = oo(b["input_tensor"].to(dt), b["text_length"], b["speaker_tensor"])
        F.cross_entropy(ol[b["attention_mask"].bool()], b["label"]).backward()
        res.append((ol.detach().numpy(), {k: p.grad.numpy() for k, p in oo.named_parameters() if p.grad is not None}))
    return res


def _run(m, b):
    from erc_b200 import ops
    logits, none = m(input_tensor=b["input_tensor"].cuda(), text_length=b["text_length"],
                     speaker_tensor=b["speaker_tensor"].cuda())
    assert none is None
    sel = logits[b["attention_mask"].cuda().bool()]                 # dagerc.py:223-226
    loss = ops.cross_entropy(sel, b["label"].cuda())
    loss.backward()
    return logits, loss


def test_dagerc_module_vs_reference_fixture(golden):
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dagerc import DAGERCModule
    fx = golden("dagerc_small")
    emb, C = fx["input_tensor"].shape[-1], fx["logits"].shape[-1]
    m = DAGERCModule(emb_dim=emb, dropout=0.0, n_classes=C, gnn_layers=4)
    seeded.fill_by_name(m, DAGERC_SEED)
    m = m.cuda()
    m.train()
    b = {k: torch.from_numpy(fx[k]) for k in ("input_tensor", "speaker_tensor", "text_length", "attention_mask", "label")}
    logits, loss = _run(m, b)
    assert logits.shape == fx["logits"].shape
    assert rel_err(logits, fx["logits"]) < TOL                      # padded positions included
    assert abs(float(loss.detach()) - float(fx["loss"])) < TOL * float(fx["loss"])
    grads = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None}
    live = set(str(k) for k in fx["live"])
    assert live <= set(grads), sorted(live - set(grads))
    worst = check_against_fixture(fx, {k: grads[k] for k in live}, 1e-4)
    print("dagerc fixture: worst grad rel err", worst)
    # the 1e-4 bar above, backed by data: against the fp64 oracle the kernels are no further off than the fp32 reference math
    (l32, g32), (l64, g64) = _oracle_runs(emb, C, b)
    parity_check("dagerc/fixture/logits", {"logits": logits}, {"logits": fx["logits"]}, {"logits": l64})
    parity_check("dagerc/fixture/grads", {k: grads[k] for k in g32}, g32, g64)
    # packed mode: same logits at the real positions, zeros at the padding, same gradients
    m2 = DAGERCModule(emb_dim=emb, dropout=0.0, n_classes=C, gnn_layers=4, compute_padding=False)
    seeded.fill_by_name(m2, DAGERC_SEED)
    m2 = m2.cuda()
    m2.train()
    logits2, loss2 = _run(m2, b)
    mask = b["attention_mask"].bool()
    assert rel_err(logits2[mask.cuda()], logits[mask.cuda()]) < 1e-6 and float(logits2[~mask.cuda()].abs().max()) == 0.0
    for k, p in m2.named_parameters():
        if p.grad is not None:
            assert rel_err(p.grad, grads[k], floor=1e-8) < 1e-5, k


def test_dagerc_config4_shape_vs_oracle():
    """BASELINE config 4: DAG-ERC 6-way, B=16 IEMOCAP-shaped dialogues, hidden_all 1380, 4 layers, dropout 0."""
    import erc_b200  # noqa: F401
    from erc_b200 import synth
    from erc_b200.track_mm.dagerc import DAGERCModule
    gen = torch.Generator().manual_seed(1)
    lengths = [int(v) for v in synth.iemocap_lengths(16, gen)]
    b = dagerc_inputs(lengths, 1380, 6, seed=11)
    (ol, want), (l64, want64) = _oracle_runs(1380, 6, b)
    ol = torch.from_numpy(ol)
    oloss = F.cross_entropy(ol[b["attention_mask"].bool()], b["label"])
    m = DAGERCModule(emb_dim=1380, dropout=0.0, n_classes=6, gnn_layers=4)
    seeded.fill_by_name(m, DAGERC_SEED)
    m = m.cuda()
    m.train()
    logits, loss = _run(m, b)
    assert rel_err(logits, ol.detach()) < TOL
    assert abs(float(loss.detach()) - float(oloss.detach())) < TOL * float(oloss.detach())
    got = {k: p.grad.cpu().numpy() for k, p in m.named_parameters() if p.grad is not None and k in want}
    parity_check("dagerc/config4/logits", {"logits": logits}, {"logits": ol}, {"logits": l64})
    parity_check("dagerc/config4/grads", got, want, want64)


def test_dagerc_dropout_training_step_runs():
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dagerc import DAGERCModule
    b = dagerc_inputs([5, 9, 1], 24, 6, seed=2)
    torch.manual_seed(0)
    m = DAGERCModule(emb_dim=24, dropout=0.3, n_classes=6, gnn_layers=2).cuda()
    m.train()
    logits, loss = _run(m, b)
    assert torch.isfinite(loss) and logits.shape == (3, 9, 6)
    assert all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)


@pytest.mark.parametrize("B,N,D", [(16, 37, 300), (3, 1, 300), (5, 110, 64)])
def test_gat_dialoggcn_v1_standalone_forward_backward_vs_oracle(B, N, D):
    """The class called on its own with the reference's signature forward(Q, K, V, adj, s_mask) -> (attn_weight [B,1,N],
    attn_sum [B,D]) (dagerc_models.py:326-365); oracle = dagerc_oracle._Gat (pinned to the real class in
    tests/test_oracle_ref_port.py).  Both outputs feed the loss, so the dalpha path of the backward kernel is live."""
    import erc_b200  # noqa: F401
    from erc_b200.track_mm.dagerc_models import GAT_dialoggcn_v1
    gen = torch.Generator().manual_seed(B * 1000 + N)
    o = dagerc_oracle._Gat(D)
    m = GAT_dialoggcn_v1(D)
    m.load_state_dict(o.state_dict(), strict=True)
    m = m.cuda()
    Q, K = torch.randn(B, D, generator=gen), torch.randn(B, N, D, generator=gen)
    adj = (torch.rand(B, N, generator=gen) < 0.6).float()
    adj[:, -1] = 1.0                                                 # the reference always has the previous utterance
    if B > 1:
        adj[1] = 0.0                                                 # ... except this degenerate row: all masked -> uniform weights
    sm = (torch.rand(B, N, generator=gen) < 0.5).long()
    gw, gs = torch.randn(B, 1, N, generator=gen), torch.randn(B, D, generator=gen)
    res = []
    for mod, dev, dt in ((o, "cpu", torch.float32), (copy.deepcopy(o).double(), "cpu", torch.float64), (m, "cuda", torch.float32)):
        q, k = Q.to(dev, dt).detach().clone().requires_grad_(), K.to(dev, dt).detach().clone().requires_grad_()
        w, s = mod(q, k, k, adj.to(dev, dt), sm.to(dev))
        assert w.shape == (B, 1, N) and s.shape == (B, D)
        ((w * gw.to(dev, dt)).sum() + (s * gs.to(dev, dt)).sum()).backward()
        out = {"attn_weight": w.detach().cpu().numpy(), "attn_sum": s.detach().cpu().numpy(),
               "dQ": q.grad.cpu().numpy(), "dK": k.grad.cpu().numpy()}
        out.update({"d" + n: p.grad.cpu().numpy() for n, p in mod.named_parameters()})
        res.append(out)
    parity_check("dagerc/gat_standalone/B%d_N%d_D%d" % (B, N, D), res[2], res[0], res[1])


def test_dag_layer_graph_capture_bit_equal_to_eager():
    """One K10 layer forward + backward captured in a CUDA graph and replayed: the output and every gradient are bit-equal
    to the eager run (the layer's launch set-up is done once per device, not inside the capture)."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops_dagerc
    from erc_b200.graph import build_graph
    from erc_b200.track_mm.dagerc_models import GAT_dialoggcn_v1
    gen = torch.Generator().manual_seed(7)
    lengths = torch.tensor([30, 17, 1, 44, 8])
    D, N = 300, int(lengths.sum())
    spk = torch.randint(0, 2, (lengths.numel(), int(lengths.max())), generator=gen)
    g = build_graph(lengths, spk.cuda(), 0, 0, 2, reference_layout=False, mean_weight=False)
    dag = ops_dagerc.DagStructure(g, lengths, 1)                   # holds the one host sync: built before the capture
    torch.manual_seed(7)
    gat, gru_c, gru_p = GAT_dialoggcn_v1(D).cuda(), torch.nn.GRUCell(D, D).cuda(), torch.nn.GRUCell(D, D).cuda()
    H = torch.randn(N, D, generator=gen).cuda().requires_grad_()
    dout = torch.randn(N, D, generator=gen).cuda()
    wrt = [H, *gat.parameters(), *gru_c.parameters(), *gru_p.parameters()]

    def fwd_bwd():
        out = ops_dagerc.dag_layer(H, gat, gru_c, gru_p, dag)
        return (out.detach(), *torch.autograd.grad(out, wrt, dout))

    a = fwd_bwd()
    assert all(torch.isfinite(x).all() for x in a)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fwd_bwd()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c = fwd_bwd()
    graph.replay()
    torch.cuda.synchronize()
    assert len(c) == len(wrt) + 1
    assert all(torch.equal(x, y) for x, y in zip(a, c))
