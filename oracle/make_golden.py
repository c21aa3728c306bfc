"""Generate tests/golden/*.npz by running the REAL reference code from /root/reference.

TEST INFRASTRUCTURE ONLY.  Run in the build container (the reference tree is
not shipped to the GPU box):  ``python -m oracle.make_golden``
The reference's third-party layers are the stand-ins of oracle/pyg_standin.py
(see oracle/ref_loader.py), so for RGCNConv/TransformerConv/GraphConv the
fixtures pin our reading of PyG, not PyG itself ("parity unpinned" there).
Everything else (edge_perms, batch_graphify, EdgeAtt, vendored RGCNConv, module
forward, autograd gradients) is the reference's own code.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

from . import ref_loader, graph_np, seeded

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

DGCN_CLASS_WEIGHTS = [1 / 0.086747, 1 / 0.144406, 1 / 0.227883, 1 / 0.160585, 1 / 0.127711, 1 / 0.252668]  # dgcn.py:109-110


def _edge_dict(n):
    d = {}
    for j in range(n):
        for k in range(n):
            d[str(j) + str(k) + "0"] = len(d)
            d[str(j) + str(k) + "1"] = len(d)
    return d


def _np(t):
    return t.detach().cpu().numpy()


def graph_fixtures(ref):
    out = {}
    perm_cases = [(1, 5, 5), (2, 5, 5), (6, 5, 5), (11, 5, 5), (12, 5, 5), (37, 5, 5), (110, 10, 10), (9, 0, 0),
                  (15, 2, 7), (15, 7, 2), (20, -1, 3), (20, 3, -1), (13, -1, -1), (8, 10, 10), (30, 0, 4)]
    out["perm_cases"] = np.array(perm_cases, dtype=np.int64)
    for i, (L, wp, wf) in enumerate(perm_cases):
        p = sorted(ref.cogmen_utils.edge_perms(L, wp, wf))
        p2 = sorted(ref.dgcn_models.edge_perms(L, wp, wf))
        assert p == p2
        out["perm_%d" % i] = np.array(p, dtype=np.int64).reshape(-1, 2)
    g = torch.Generator().manual_seed(7)
    cases = [dict(lengths=[7, 1, 12, 3, 25], n=2, wp=5, wf=5), dict(lengths=[4, 18, 2], n=2, wp=10, wf=10),
             dict(lengths=[9, 5, 16], n=3, wp=2, wf=4), dict(lengths=[6, 11], n=2, wp=-1, wf=2),
             dict(lengths=[10, 3], n=9, wp=3, wf=-1)]
    out["n_graph_cases"] = np.array(len(cases))
    for i, c in enumerate(cases):
        lens = torch.tensor(c["lengths"])
        B, Lmax = len(c["lengths"]), max(c["lengths"])
        spk = torch.randint(0, c["n"], (B, Lmax), generator=g)
        for b in range(B):
            spk[b, c["lengths"][b]:] = 0
        feats = torch.randn(B, Lmax, 3, generator=g)
        nf, ei, et, el = ref.cogmen_utils.batch_graphify(feats, lens, spk, c["wp"], c["wf"], _edge_dict(c["n"]))
        order = graph_np.canonical_order(_np(ei))
        out["g%d_meta" % i] = np.array([c["n"], c["wp"], c["wf"]], dtype=np.int64)
        out["g%d_lengths" % i] = _np(lens)
        out["g%d_speakers" % i] = _np(spk)
        out["g%d_features" % i] = _np(feats)
        out["g%d_node_features" % i] = _np(nf)
        out["g%d_edge_index" % i] = _np(ei)[:, order]
        out["g%d_edge_type" % i] = _np(et)[order]
        out["g%d_edge_index_lengths" % i] = _np(el)
    np.savez_compressed(os.path.join(OUT, "graph.npz"), **out)
    print("graph.npz", len(out), "arrays")


def _grads(module):
    return {k: _np(p.grad) for k, p in module.named_parameters() if p.grad is not None}


def cogmen_fixture(ref):
    torch.manual_seed(11)
    D, C = 36, 4
    lengths = [9, 1, 14, 6, 30]
    B, Lmax = len(lengths), max(lengths)
    m = ref.cogmen.COGMENModule(input_size=D, hidden_size=100, num_head=17, n_speakers=2, n_classes=C)
    m.cls[2].p = 0.0                      # dropout off for parity (SURVEY.md 8c "parity mode")
    with torch.no_grad():                 # non-trivial BN affine so its gradients are exercised
        m.gcn.bn.weight.uniform_(0.5, 1.5)
        m.gcn.bn.bias.uniform_(-0.5, 0.5)
        m.gcn.conv1.bias.uniform_(-0.1, 0.1)
    g = torch.Generator().manual_seed(12)
    x = torch.randn(B, Lmax, D, generator=g)
    spk = torch.randint(0, 2, (B, Lmax), generator=g)
    lens = torch.tensor(lengths)
    for b in range(B):
        x[b, lengths[b]:] = 0
        spk[b, lengths[b]:] = 0
    y = torch.randint(0, C, (sum(lengths),), generator=g)
    sd0 = {k: _np(v).copy() for k, v in m.state_dict().items() if not k.startswith("rnn.0")}
    m.train()
    logits, feats = m(input_tensor=x, speaker_tensor=spk, text_length=lens)
    loss = F.cross_entropy(logits, y)
    loss.backward()
    grads = _grads(m)
    assert not any(k.startswith("rnn.0") for k in grads), "dead encoder must have no grad"
    out = dict(input_tensor=_np(x), speaker_tensor=_np(spk), text_length=_np(lens), label=_np(y),
               logits=_np(logits), features=_np(feats), loss=_np(loss),
               bn_running_mean=_np(m.gcn.bn.running_mean), bn_running_var=_np(m.gcn.bn.running_var))
    m.eval()
    with torch.no_grad():
        out["logits_eval"] = _np(m(input_tensor=x, speaker_tensor=spk, text_length=lens)[0])
    for k, v in sd0.items():
        out["param/" + k] = v
    for k, v in grads.items():
        out["grad/" + k] = v
    _save_split("cogmen_small", out)
    print("cogmen_small.npz loss", float(loss), "live grads", len(grads))


def dgcn_fixture(ref):
    torch.manual_seed(21)
    D, C = 24, 6
    lengths = [12, 1, 23, 7]
    B, Lmax = len(lengths), max(lengths)
    m = ref.dgcn.DGCNModule(n_speakers=2, input_size=D, hidden_size=48, n_classes=C)   # 48 keeps the fixture small
    m.rnn.rnn.dropout = 0.0
    m.clf.drop.p = 0.0
    g = torch.Generator().manual_seed(22)
    x = torch.randn(B, Lmax, D, generator=g)
    spk = torch.randint(0, 2, (B, Lmax), generator=g)
    lens = torch.tensor(lengths)
    for b in range(B):
        x[b, lengths[b]:] = 0
        spk[b, lengths[b]:] = 0
    y = torch.randint(0, C, (sum(lengths),), generator=g)
    sd0 = {k: _np(v).copy() for k, v in m.state_dict().items()}
    m.train()
    # intermediate pins: EdgeAtt + graphify + vendored RGCN
    ctx = m.rnn(lens, x)
    feats, ei, en, et, el = ref.dgcn_models.batch_graphify(ctx, lens, spk, m.wp, m.wf, m.edge_type_to_idx, m.edge_att)
    order = graph_np.canonical_order(_np(ei))
    rg = m.gcn.conv1(feats, ei, et, edge_norm=en)
    logits, graph_out = m(input_tensor=x, speaker_tensor=spk, text_length=lens)
    w = torch.tensor(DGCN_CLASS_WEIGHTS)
    loss = F.cross_entropy(logits, y, weight=w)
    loss.backward()
    grads = _grads(m)
    out = dict(input_tensor=_np(x), speaker_tensor=_np(spk), text_length=_np(lens), label=_np(y),
               class_weights=_np(w), logits=_np(logits), graph_out=_np(graph_out), loss=_np(loss),
               context=_np(ctx), node_features=_np(feats), edge_index=_np(ei)[:, order], edge_type=_np(et)[order],
               edge_norm=_np(en)[order], edge_index_lengths=_np(el), rgcn_out=_np(rg))
    for k, v in sd0.items():
        out["param/" + k] = v
    for k, v in grads.items():
        out["grad/" + k] = v
    _save_split("dgcn_small", out)
    print("dgcn_small.npz loss", float(loss), "live grads", len(grads))


def _save_split(name, out):
    """name.npz without the gradients, name_grads.npz with them: each file stays under 1 MB."""
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **{k: v for k, v in out.items() if not k.startswith("grad/")})
    np.savez_compressed(os.path.join(OUT, name + "_grads.npz"), **{k: v for k, v in out.items() if k.startswith("grad/")})


def _store_grads(out, grads, big=4096):
    """Small gradients whole; large ones as a strided sample + max-abs + sum (oracle/seeded.py)."""
    for k, v in grads.items():
        if v.size <= big:
            out["grad/" + k] = v
        else:
            s, mx, tot = seeded.digest(v)
            out["gsample/" + k] = s
            out["gmax/" + k] = mx
            out["gsum/" + k] = tot


MMGCN_SEED, DAGERC_SEED = 31, 41


def mmgcn_inputs(lengths, dims, n_classes, seed):
    """Seq-first batch as ERCCollate builds it for MMGCN (batch_first=False, speaker_onehot=True; mmgcn.py:39-40)."""
    dt, da, dv = dims
    B, Lmax = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(seed)
    t = torch.randn(Lmax, B, dt, generator=g)
    a = torch.randn(Lmax, B, da, generator=g)
    v = torch.randn(Lmax, B, dv, generator=g)
    spk = torch.randint(0, 2, (Lmax, B), generator=g)
    for b, L in enumerate(lengths):
        t[L:, b] = 0
        a[L:, b] = 0
        v[L:, b] = 0
        spk[L:, b] = 0
    y = torch.randint(0, n_classes, (sum(lengths),), generator=g)
    return dict(text_feature=t, audio_feature=a, visual_feature=v, speaker_tensor=F.one_hot(spk, 2).float(),
                text_length=torch.tensor(lengths), label=y)


def mmgcn_fixture(ref):
    """Real MMGCNModule (mmgcn.py:56-122, 64 GCNII layers of width 200) on a tiny batch.  Weights are NOT stored:
    both sides call seeded.fill_by_name(module, MMGCN_SEED)."""
    dims, C, lengths = (24, 10, 12), 6, [5, 1, 9, 3]
    torch.manual_seed(0)
    m = ref.mmgcn.MMGCNModule(hidden_text=dims[0], hidden_audio=dims[1], hidden_visual=dims[2], n_speakers=2, n_classes=C,
                              modals="atv")
    seeded.fill_by_name(m, MMGCN_SEED)
    m.lstm_l.dropout = 0.0
    m.graph_model.graph_net.dropout = 0.0
    m.dropout_.p = 0.0
    m.train()
    b = mmgcn_inputs(lengths, dims, C, seed=32)
    # intermediate pins: packed per-modality features and the normalised adjacency (create_big_adj)
    with torch.no_grad():
        fa = ref.mmgcn_utils.simple_batch_graphify(m.linear_a(b["audio_feature"]), b["text_length"])[0]
        fv = ref.mmgcn_utils.simple_batch_graphify(m.linear_v(b["visual_feature"]), b["text_length"])[0]
        fl = ref.mmgcn_utils.simple_batch_graphify(m.lstm_l(m.linear_l(b["text_feature"]))[0], b["text_length"])[0]
        qm = torch.cat([b["speaker_tensor"][:x, i, :] for i, x in enumerate(lengths)], 0)
        fl = fl + m.graph_model.speaker_embeddings(qm.argmax(-1))
        adj = m.graph_model.create_big_adj(fa, fv, fl, b["text_length"], "atv")
    logits, _ = m(**{k: v for k, v in b.items() if k != "label"})
    loss = F.cross_entropy(logits, b["label"])
    loss.backward()
    grads = _grads(m)
    out = {k: _np(v) for k, v in b.items()}
    out.update(logits=_np(logits), loss=_np(loss), feat_a=_np(fa), feat_v=_np(fv), feat_l=_np(fl), adj=_np(adj),
               dims=np.array(dims), live=np.array(sorted(grads)))
    _store_grads(out, grads)
    np.savez_compressed(os.path.join(OUT, "mmgcn_small.npz"), **out)
    print("mmgcn_small.npz loss", float(loss), "live grads", len(grads), "max grad",
          max(float(np.abs(v).max()) for v in grads.values()))


def dagerc_inputs(lengths, emb, n_classes, seed):
    """Batch-first batch with one-hot speakers (dagerc.py:41-42); padded speaker id 0 (mmbase.py:420,431-432)."""
    B, Lmax = len(lengths), max(lengths)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, Lmax, emb, generator=g)
    spk = torch.randint(0, 2, (B, Lmax), generator=g)
    mask = torch.zeros(B, Lmax)
    for b, L in enumerate(lengths):
        x[b, L:] = 0
        spk[b, L:] = 0
        mask[b, :L] = 1
    y = torch.randint(0, n_classes, (sum(lengths),), generator=g)
    return dict(input_tensor=x, speaker_tensor=F.one_hot(spk, 2).float(), text_length=torch.tensor(lengths),
                attention_mask=mask, label=y)


def dagerc_fixture(ref):
    """Real DAGERCModule (dagerc.py:73-198: 4 layers, hidden 300).  Weights by seeded.fill_by_name."""
    emb, C, lengths = 20, 6, [7, 2, 11, 1]
    torch.manual_seed(0)
    m = ref.dagerc.DAGERCModule(emb_dim=emb, dropout=0.0, n_classes=C, gnn_layers=4)
    seeded.fill_by_name(m, DAGERC_SEED)
    m.train()
    b = dagerc_inputs(lengths, emb, C, seed=42)
    mx = max(lengths)
    adj = m.get_adj_v1(b["speaker_tensor"].tolist(), mx)
    s_mask, _ = m.get_s_mask(b["speaker_tensor"].tolist(), mx)
    logits, _ = m(input_tensor=b["input_tensor"], text_length=b["text_length"], speaker_tensor=b["speaker_tensor"])
    sel = logits[b["attention_mask"].bool()]
    loss = F.cross_entropy(sel, b["label"])          # dagerc.py:223-226
    loss.backward()
    grads = _grads(m)
    out = {k: _np(v) for k, v in b.items()}
    out.update(logits=_np(logits), loss=_np(loss), adj=_np(adj), s_mask=_np(s_mask), live=np.array(sorted(grads)))
    _store_grads(out, grads)
    np.savez_compressed(os.path.join(OUT, "dagerc_small.npz"), **out)
    print("dagerc_small.npz loss", float(loss), "live grads", len(grads), "max grad",
          max(float(np.abs(v).max()) for v in grads.values()))


DGCNV2_SEED = 53


def dgcnv2_fixture(ref):
    """Real dgcnv2.DGCNModule('LSTM') (dgcnv2.py:54-181) with MaskedEdgeAttention / GraphNetwork / nodal MatchingAttention of
    dgcnv2_models.py; dropout 0; weights by seeded.fill_by_name; class-weighted CE as in the trainer (dgcnv2.py:200-217)."""
    from oracle import dgcnv2_oracle
    r = ref_loader.load_dgcnv2()
    D, C, lengths = 36, 6, [9, 3, 14, 1, 6]
    torch.manual_seed(0)
    m = r.dgcnv2.DGCNModule("LSTM", input_size=D, hidden_size=100, n_speakers=2, n_classes=C, dropout=0.0)
    m.graph_net.dropout.p = 0.0
    seeded.fill_by_name(m, DGCNV2_SEED)
    m.train()
    b = dgcnv2_oracle.inputs(lengths, D, 2, C, seed=77)
    w = torch.tensor([1 / 0.086747, 1 / 0.144406, 1 / 0.227883, 1 / 0.160585, 1 / 0.127711, 1 / 0.252668])
    logits, feats = m(**{k: v for k, v in b.items() if k != "label"})
    loss = F.cross_entropy(logits, b["label"], weight=w)
    loss.backward()
    grads = _grads(m)
    out = {k: _np(v) for k, v in b.items()}
    out.update(logits=_np(logits), features=_np(feats), loss=_np(loss), class_weights=_np(w), live=np.array(sorted(grads)))
    _store_grads(out, grads)
    np.savez_compressed(os.path.join(OUT, "dgcnv2_small.npz"), **out)
    print("dgcnv2_small.npz loss", float(loss), "live grads", len(grads), sorted(grads)[:6])


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = ref_loader.load()
    which = sys.argv[1:] or ["graph", "cogmen", "dgcn", "mmgcn", "dagerc", "dgcnv2"]
    if "graph" in which:
        graph_fixtures(ref)
    if "cogmen" in which:
        cogmen_fixture(ref)
    if "dgcn" in which:
        dgcn_fixture(ref)
    if "mmgcn" in which:
        mmgcn_fixture(ref)
    if "dagerc" in which:
        dagerc_fixture(ref)
    if "dgcnv2" in which:
        dgcnv2_fixture(ref)


if __name__ == "__main__":
    main()
