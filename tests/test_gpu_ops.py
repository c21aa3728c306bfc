"""Kernel-level parity: every libercgraph op against a plain fp32/fp64 PyTorch CPU expression."""
import math

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import graph_np

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _graph(lengths, n=2, wp=5, wf=5, seed=0):
    import erc_b200
    from erc_b200.graph import build_graph
    rng = np.random.default_rng(seed)
    lengths = np.asarray(lengths)
    spk = rng.integers(0, n, size=int(lengths.sum()))
    g = build_graph(torch.as_tensor(lengths, dtype=torch.int64), torch.as_tensor(spk).cuda(), wp, wf, n)
    return g, graph_np.batch_graphify_np(lengths, spk, wp, wf, n)


@pytest.mark.parametrize("M,K,N", [(1, 1, 1), (37, 100, 100), (300, 1380, 100), (257, 1443, 100), (130, 100, 900),
                                   (64, 900, 100), (129, 100, 6), (200, 6, 100), (513, 200, 131),
                                   # skinny kernels (narrow side <= 16, >= 1024 rows): gemm_skinny.cuh
                                   (5000, 100, 6), (3000, 6, 100), (4097, 100, 7), (2048, 300, 16), (1500, 13, 10),
                                   (1025, 101, 3), (70001, 100, 6)])
def test_gemm_nn_tn_colsum(M, K, N):
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(M * 7 + K)
    A, B, bias = torch.randn(M, K, generator=g), torch.randn(K, N, generator=g), torch.randn(N, generator=g)
    want = A.double() @ B.double() + bias.double()
    got = ops.gemm_nn(A.cuda(), B.cuda(), bias.cuda())
    assert rel_err(got, want) < TOL
    got = ops.gemm_nn(A.cuda(), B.cuda(), bias.cuda(), act=ops.ACT_RELU)
    assert rel_err(got, want.clamp(min=0)) < TOL
    dC = torch.randn(M, N, generator=g)
    assert rel_err(ops.gemm_tn(A.cuda(), dC.cuda()), A.double().t() @ dC.double()) < TOL
    assert rel_err(ops.colsum(dC.cuda()), dC.double().sum(0)) < TOL
    aux = torch.randn(M, N, generator=g)
    assert rel_err(ops.mask_pos(dC.cuda(), aux.cuda(), 2.0), torch.where(aux > 0, dC * 2.0, torch.zeros(()))) < 1e-7


@pytest.mark.parametrize("M,N", [(1024, 100), (70001, 100), (33000, 200), (5000, 6), (40000, 6), (2049, 10), (3000, 7), (999, 100)])
def test_column_sums_flat_stream_and_fallbacks(M, N):
    """ercg_colsum: flat float4 / float2 streams for contiguous matrices (col_stream.cuh), row-block kernels otherwise;
    bit-reproducible (two runs equal) and within 1e-5 of fp64."""
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(M + N)
    A = torch.randn(M, N, generator=g) + 0.3
    a, b = ops.colsum(A.cuda()), ops.colsum(A.cuda())
    assert torch.equal(a, b)
    scale = float(A.double().abs().sum(0).max())
    assert float((a.cpu().double() - A.double().sum(0)).abs().max()) < TOL * scale
    strided = torch.randn(M, N + 4, generator=g).cuda()[:, :N]          # row pitch != width: row-block path
    assert float((ops.colsum(strided).cpu().double() - strided.cpu().double().sum(0)).abs().max()) < TOL * scale * 2


def test_gemm_row_gather_and_unaligned_lda():
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(3)
    A = torch.randn(500, 1443, generator=g)               # 1443 floats per row: rows are not 16-byte aligned
    B = torch.randn(1443, 100, generator=g)
    rows = torch.randint(0, 500, (333,), generator=g).int()
    want = A[rows.long()].double() @ B.double()
    got = ops.gemm_nn(A.cuda(), B.cuda(), a_rows=rows.cuda())
    assert rel_err(got, want) < TOL
    dC = torch.randn(333, 100, generator=g)
    got = ops.gemm_tn(A.cuda(), dC.cuda(), a_rows=rows.cuda(), M=333)
    assert rel_err(got, A[rows.long()].double().t() @ dC.double()) < TOL


def test_gemm_large_split_reduction_is_deterministic():
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(4)
    A, dC = torch.randn(40_000, 200, generator=g).cuda(), torch.randn(40_000, 100, generator=g).cuda()
    r1, r2 = ops.gemm_tn(A, dC), ops.gemm_tn(A, dC)
    assert torch.equal(r1, r2)
    assert rel_err(r1, A.double().cpu().t() @ dC.double().cpu()) < TOL


def test_dropout_epilogue_statistics_and_backward():
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(5)
    x = torch.randn(4096, 100, generator=g).cuda().requires_grad_()
    w = torch.randn(100, 100, generator=g).cuda().requires_grad_()
    h = ops.linear(x, w, None, act=ops.ACT_RELU_DROPOUT, drop_p=0.5, seed=1234)
    ref = torch.relu(x.detach() @ w.detach().t())
    kept = h != 0
    frac = float(kept.sum()) / float((ref > 0).sum())
    assert 0.48 < frac < 0.52
    assert rel_err(h[kept], (ref * 2.0)[kept]) < TOL
    h2 = ops.linear(x, w, None, act=ops.ACT_RELU_DROPOUT, drop_p=0.5, seed=1234)
    assert torch.equal(h, h2)                               # same seed => same mask
    h.sum().backward()
    mask = kept.float() * 2.0
    assert rel_err(x.grad, mask @ w.detach()) < TOL
    assert rel_err(w.grad, mask.t() @ x.detach()) < TOL


@pytest.mark.parametrize("H,R,wp,wf", [(100, 8, 5, 5), (100, 8, 10, 10), (200, 8, 10, 10), (100, 2, -1, -1)])
def test_gather_fwd_bwd(H, R, wp, wf):
    import erc_b200
    from erc_b200 import ops
    n = 2 if R == 8 else 1
    g, b = _graph([7, 1, 23, 60, 4], n=n, wp=wp, wf=wf)
    N, E = b["N"], b["E"]
    gen = torch.Generator().manual_seed(H + R)
    Y = torch.randn(N, (R + 1) * H, generator=gen)
    w = torch.rand(E, generator=gen) + 0.1
    bias = torch.randn(H, generator=gen)
    src, dst, et = (torch.from_numpy(b[k]).long() for k in ("col", "edge_index", "etype"))
    dst = dst[1]
    Yd, wd = Y.double().requires_grad_(), w.double().requires_grad_()
    msg = Yd.view(N, R + 1, H)[src, et] * wd[:, None]
    want = torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, msg) + Yd[:, R * H:] + bias.double()
    dout = torch.randn(N, H, generator=gen)
    want.backward(dout.double())
    Yc, wc, bc = Y.cuda().requires_grad_(), w.cuda().requires_grad_(), bias.cuda().requires_grad_()
    got = ops.gather(Yc, g, H, R, w=wc, bias=bc, root_off=R * H)
    got.backward(dout.cuda())
    assert rel_err(got, want) < TOL
    assert rel_err(Yc.grad, Yd.grad) < TOL
    assert rel_err(wc.grad, wd.grad) < TOL
    assert rel_err(bc.grad, dout.double().sum(0)) < TOL


def test_gather_compact_relation_slots_equals_full_layout():
    """One speaker id out of n=2 (relation ids {6,7} only): Y restricted to the slots K1's census reports, addressed
    through rel_slot, gives the same output, dY (per present slot) and dw as the full 8-slot layout."""
    import erc_b200
    from erc_b200 import ops
    from erc_b200.graph import build_graph
    H, R = 100, 8
    lens = torch.tensor([7, 1, 23, 60, 4])
    spk = torch.ones(5, 60, dtype=torch.int64)
    g = build_graph(lens, spk.cuda(), 5, 5, 2)
    ids, rel_slot = g.relation_slots()
    assert ids == [6, 7]
    P = len(ids)
    gen = torch.Generator().manual_seed(11)
    Yfull = torch.randn(g.N, (R + 1) * H, generator=gen)
    w = torch.rand(g.E, generator=gen) + 0.1
    dout = torch.randn(g.N, H, generator=gen).cuda()
    cols = torch.cat([torch.arange(r * H, (r + 1) * H) for r in ids] + [torch.arange(R * H, (R + 1) * H)])
    Yf, wf_ = Yfull.cuda().requires_grad_(), w.cuda().requires_grad_()
    a = ops.gather(Yf, g, H, R, w=wf_, root_off=R * H)
    a.backward(dout)
    Yc, wc = Yfull[:, cols].contiguous().cuda().requires_grad_(), w.cuda().requires_grad_()
    b = ops.gather(Yc, g, H, R, w=wc, root_off=P * H, rel_slot=rel_slot, n_slots=P)
    b.backward(dout)
    assert torch.equal(a, b)
    assert torch.equal(Yf.grad[:, cols.cuda()], Yc.grad)
    mask = torch.ones((R + 1) * H, dtype=torch.bool)
    mask[cols] = False
    assert float(Yf.grad[:, mask.cuda()].abs().max()) == 0.0
    assert torch.equal(wf_.grad, wc.grad)


@pytest.mark.parametrize("wp,wf", [(5, 5), (-1, -1), (2, 40), (10, 10), (16, 15), (0, 3), (0, 0)])
def test_edge_attention_fwd_bwd(wp, wf):
    import erc_b200
    from erc_b200 import ops
    H = 100
    g, b = _graph([9, 1, 50, 75, 3], wp=wp, wf=wf, seed=2)     # wp=wf=-1 gives rows longer than 32 edges
    N = b["N"]
    gen = torch.Generator().manual_seed(11)
    qkvs = torch.randn(N, 4 * H, generator=gen)
    src, dst = torch.from_numpy(b["edge_index"][0]), torch.from_numpy(b["edge_index"][1])
    x = qkvs.double().requires_grad_()
    q, k, v, s = x[:, :H], x[:, H:2 * H], x[:, 2 * H:3 * H], x[:, 3 * H:]
    sc = (q[dst] * k[src]).sum(-1) / math.sqrt(H)
    mx = torch.full((N,), -1e300, dtype=torch.float64).scatter_reduce(0, dst, sc, reduce="amax")
    ex = (sc - mx[dst]).exp()
    alpha = ex / (torch.zeros(N, dtype=torch.float64).index_add(0, dst, ex) + 1e-16)[dst]
    want = torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, alpha[:, None] * v[src]) + s
    dout = torch.randn(N, H, generator=gen)
    want.backward(dout.double())
    xc = qkvs.cuda().requires_grad_()
    got = ops.edge_attention(xc, g, H, 1.0 / math.sqrt(H))
    got.backward(dout.cuda())
    assert rel_err(got, want) < TOL
    assert rel_err(xc.grad, x.grad) < TOL


def test_edge_att_source_softmax_fwd_bwd():
    import erc_b200
    from erc_b200 import ops
    H = 200
    g, b = _graph([12, 1, 40, 110], wp=10, wf=10, seed=3)
    N, E = b["N"], b["E"]
    gen = torch.Generator().manual_seed(13)
    x, u = torch.randn(N, H, generator=gen) * 0.3, torch.randn(N, H, generator=gen) * 0.3
    src, dst = torch.from_numpy(b["edge_index"][0]), torch.from_numpy(b["edge_index"][1])
    xd, ud = x.double().requires_grad_(), u.double().requires_grad_()
    sc = (xd[src] * ud[dst]).sum(-1)
    mx = torch.full((N,), -1e300, dtype=torch.float64).scatter_reduce(0, src, sc, reduce="amax")
    ex = (sc - mx[src]).exp()
    want = ex / torch.zeros(N, dtype=torch.float64).index_add(0, src, ex)[src]
    dnu = torch.randn(E, generator=gen)
    want.backward(dnu.double())
    xc, uc = x.cuda().requires_grad_(), u.cuda().requires_grad_()
    got = ops.edge_att(xc, uc, g)
    got.backward(dnu.cuda())
    assert rel_err(got, want) < TOL
    assert rel_err(xc.grad, xd.grad) < TOL
    assert rel_err(uc.grad, ud.grad) < TOL


@pytest.mark.parametrize("N", [1, 5, 1023, 5000])
def test_bn_leaky_relu_fwd_bwd(N):
    import erc_b200
    from erc_b200 import ops
    H = 100
    gen = torch.Generator().manual_seed(N)
    x = torch.randn(N, H, generator=gen) * 2 + 0.5
    gamma, beta = torch.rand(H, generator=gen) + 0.5, torch.randn(H, generator=gen)
    xd, gd, bd = x.double().requires_grad_(), gamma.double().requires_grad_(), beta.double().requires_grad_()
    mean, var = xd.mean(0), xd.var(0, unbiased=False)
    want = torch.nn.functional.leaky_relu((xd - mean) / (var + 1e-5).sqrt() * gd + bd, 0.01)
    dout = torch.randn(N, H, generator=gen)
    want.backward(dout.double())
    xc, gc, bc = x.cuda().requires_grad_(), gamma.cuda().requires_grad_(), beta.cuda().requires_grad_()
    m, v = ops.bn_stats(xc.detach())
    assert rel_err(m, mean.detach()) < TOL and rel_err(v, var.detach(), floor=1e-12) < TOL
    got = ops.bn_leaky_relu(xc, gc, bc, m, v, 1e-5, 0.01, True)
    got.backward(dout.cuda())
    assert rel_err(got, want) < TOL
    scale = float(xd.grad.abs().max())
    assert rel_err(xc.grad, xd.grad, floor=max(scale, 1e-3)) < 5 * TOL     # N=1: dx is exactly 0
    assert rel_err(gc.grad, gd.grad, floor=1e-3) < TOL and rel_err(bc.grad, bd.grad) < TOL


@pytest.mark.parametrize("momentum", [0.1, None])
def test_bn_running_update_matches_torch_batchnorm(momentum):
    """ercg_bn_running_update = the train-mode bookkeeping of nn.BatchNorm1d (num_batches_tracked, running_mean, running_var
    with the unbiased-variance factor), momentum=None (cumulative average) included."""
    import erc_b200
    from erc_b200 import ops
    H, gen = 100, torch.Generator().manual_seed(5)
    ref = torch.nn.BatchNorm1d(H, momentum=momentum).double().train()
    ours = torch.nn.BatchNorm1d(H, momentum=momentum).cuda().train()
    for n in (700, 33, 1500):
        x = torch.randn(n, H, generator=gen) * 3 + 1
        ref(x.double())
        m, v = ops.bn_stats(x.cuda())
        ops.bn_running_update(ours, m, v, float(n))
    assert int(ours.num_batches_tracked) == int(ref.num_batches_tracked) == 3
    assert rel_err(ours.running_mean, ref.running_mean) < TOL and rel_err(ours.running_var, ref.running_var) < TOL


def test_bn_sync_pack_unpack_equal_the_elementwise_expression():
    """The two kernels around the BatchNorm-statistics all-reduce (dist.StatSync.stats on CUDA) against the torch fp64
    expression they replace, bit for bit, with two simulated ranks."""
    import erc_b200
    from erc_b200._lib import lib, check
    H, gen = 100, torch.Generator().manual_seed(9)
    parts, bufs = [], []
    for n in (1234, 777):
        mean, var = torch.randn(H, generator=gen), torch.rand(H, generator=gen) + 0.1
        buf = torch.empty(2 * H + 2, dtype=torch.float64, device="cuda")
        mc, vc = mean.cuda(), var.cuda()
        check(lib().ercg_bn_sync_pack(mc.data_ptr(), vc.data_ptr(), float(n), H, buf.data_ptr(), None), "pack")
        want = torch.cat([mean.double() * n, (var.double() + mean.double() ** 2) * n, torch.tensor([float(n), 0.0], dtype=torch.float64)])
        assert torch.equal(buf.cpu(), want)
        bufs.append(buf)
        parts.append(want)
    tot = bufs[0] + bufs[1]                      # what the all-reduce delivers
    gm, gv = torch.empty(H, device="cuda"), torch.empty(H, device="cuda")
    check(lib().ercg_bn_sync_unpack(tot.data_ptr(), H, gm.data_ptr(), gv.data_ptr(), None), "unpack")
    w = parts[0] + parts[1]
    wm = w[:H] / w[2 * H]
    wv = (w[H:2 * H] / w[2 * H] - wm ** 2).clamp_(min=0)
    assert torch.equal(gm.cpu(), wm.float()) and torch.equal(gv.cpu(), wv.float())


@pytest.mark.parametrize("C,weighted", [(4, False), (6, True), (1, False), (7, True)])
def test_cross_entropy(C, weighted):
    import erc_b200
    from erc_b200 import ops
    gen = torch.Generator().manual_seed(C)
    N = 777
    z = torch.randn(N, C, generator=gen) * 3
    y = torch.randint(0, C, (N,), generator=gen)
    w = torch.rand(C, generator=gen) + 0.2 if weighted else None
    zd = z.double().requires_grad_()
    want = torch.nn.functional.cross_entropy(zd, y, weight=None if w is None else w.double())
    (want * 1.7).backward()
    zc = z.cuda().requires_grad_()
    got = ops.cross_entropy(zc, y.cuda(), None if w is None else w.cuda())
    (got * 1.7).backward()
    assert abs(float(got.detach()) - float(want.detach())) < TOL * max(abs(float(want.detach())), 1e-3)
    assert rel_err(zc.grad, zd.grad, floor=1e-8) < TOL


def test_pack_rows_roundtrip():
    import erc_b200
    from erc_b200 import ops
    g, b = _graph([5, 1, 9])
    gen = torch.Generator().manual_seed(1)
    for seq_first in (False, True):
        shape = (9, 3, 8) if seq_first else (3, 9, 8)
        pad = torch.randn(*shape, generator=gen).cuda().requires_grad_()
        got = ops.pack_rows(pad, g, seq_first)
        p = pad.detach().cpu()
        want = torch.cat([(p[:L, i] if seq_first else p[i, :L]) for i, L in enumerate([5, 1, 9])])
        assert torch.equal(got.cpu(), want)
        got.sum().backward()
        mask = torch.zeros(shape)
        for i, L in enumerate([5, 1, 9]):
            if seq_first:
                mask[:L, i] = 1
            else:
                mask[i, :L] = 1
        assert torch.equal(pad.grad.cpu(), mask)


def test_missing_library_fails_loudly(monkeypatch):
    import erc_b200
    from erc_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libercgraph.so")
    with pytest.raises(_lib.ErcgError):
        _lib.lib()


@pytest.mark.parametrize("copy_streams,chunk_bytes", [(1, 256 << 20), (2, 1 << 20), (3, 300_000)])
def test_device_feeder_double_buffering(copy_streams, chunk_bytes):
    """loader.DeviceFeeder: batches come out in submission order with the right contents while later copies are in
    flight; a third un-consumed submit is refused (depth 2)."""
    import erc_b200
    from erc_b200.loader import DeviceFeeder, pin
    dev = torch.device("cuda")
    feeder = DeviceFeeder(dev, depth=2, copy_streams=copy_streams, chunk_bytes=chunk_bytes)
    gen = torch.Generator().manual_seed(0)
    batches = [pin({"x": torch.randn(4096, 257, generator=gen), "spk": torch.randint(0, 2, (4096,), generator=gen)})
               for _ in range(5)]
    feeder.submit(batches[0])
    for i in range(5):
        if i + 1 < 5:
            feeder.submit(batches[i + 1])
        d = feeder.get()
        y = d["x"] * 2.0 + d["spk"][:, None].float()           # work on the current stream that reads the buffers
        feeder.release()
        want = batches[i]["x"] * 2.0 + batches[i]["spk"][:, None].float()
        assert torch.equal(y.cpu(), want)
    feeder.submit(batches[0])
    feeder.submit(batches[1])
    with pytest.raises(RuntimeError):
        feeder.submit(batches[2])
    assert feeder.h2d_bytes == 7 * (4096 * 257 * 4 + 4096 * 8)


def test_device_feeder_varying_shapes_with_compute_in_flight():
    """Every batch has its own Lmax (the reference collate pads per batch, mmbase.py:354-455) while earlier steps' kernels
    are still queued: buffers grow to a high-water mark and are handed out as views; a (re)allocation must not let the
    H2D copy overwrite a recycled block that queued kernels still read.  Heavy temporaries are freed on the compute
    stream right before each submit to give the caching allocator blocks to recycle."""
    import erc_b200
    from erc_b200.loader import DeviceFeeder, pin
    dev = torch.device("cuda")
    feeder = DeviceFeeder(dev, depth=2, copy_streams=2, chunk_bytes=1 << 20)
    gen = torch.Generator().manual_seed(1)
    shapes = [(64, 37, 300), (64, 80, 300), (64, 12, 300), (96, 110, 300), (8, 5, 300), (96, 110, 300), (64, 90, 300)]
    batches = [pin({"x": torch.randn(*sh, generator=gen), "len": torch.randint(1, sh[1] + 1, (sh[0],), generator=gen)})
               for sh in shapes]
    w = torch.randn(300, 300, generator=gen).cuda()
    results = []
    feeder.submit(batches[0])
    for i in range(len(batches)):
        tmp = torch.randn(96 * 110 * 300, device=dev)            # a block about the size of the largest buffer ...
        for _ in range(20):
            tmp = tmp * 1.0001 + 1.0                               # ... kept busy by queued kernels, then freed
        acc = tmp.sum()
        del tmp
        if i + 1 < len(batches):
            feeder.submit(batches[i + 1])
        d = feeder.get()
        assert d["x"].shape == batches[i]["x"].shape and d["x"].is_contiguous()
        y = (d["x"].reshape(-1, 300) @ w).sum() + d["len"].sum() + 0.0 * acc
        feeder.release()
        results.append(y)
    for i, y in enumerate(results):
        want = (batches[i]["x"].reshape(-1, 300).cuda() @ w).sum() + batches[i]["len"].sum().cuda()
        assert torch.allclose(y, want, rtol=1e-4), i
    assert len(feeder._store[0]) == 2 and feeder._store[0]["x"].numel() >= 96 * 110 * 300 * 4 or feeder._store[1]["x"].numel() >= 96 * 110 * 300 * 4


@pytest.mark.parametrize("wp,wf,n,one_speaker", [(5, 5, 2, False), (5, 5, 2, True), (10, 10, 2, False), (3, 8, 3, False)])
def test_gather_window_backward_is_bit_identical_to_generic(wp, wf, n, one_speaker):
    """CTA-tiled gather backward (window graphs) vs the generic warp-per-node kernel: same dY bit for bit, with and
    without the compact relation-slot table, across tile borders (N not a multiple of 32) and short dialogues."""
    import erc_b200
    from erc_b200 import _lib, ops
    from erc_b200.graph import build_graph
    H = 100
    rng = np.random.default_rng(wp * 100 + wf + n)
    lens = torch.as_tensor(rng.integers(1, 60, size=37))
    lens[3] = 1
    Lmax = int(lens.max())
    spk = torch.zeros(37, Lmax, dtype=torch.int64) if one_speaker else torch.as_tensor(rng.integers(0, n, size=(37, Lmax)))
    g = build_graph(lens, spk.cuda(), wp, wf, n)
    R = 2 * n * n
    census = g.relation_slots()
    variants = [(None, R)]
    if census is not None and len(census[0]) < R:
        variants.append((census[1], len(census[0])))
    gen = torch.Generator().manual_seed(5)
    dout = torch.randn(g.N, H, generator=gen).cuda()
    w = (torch.rand(g.E, generator=gen) + 0.1).cuda()
    lib, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
    for rel_slot, slots in variants:
        cols = (slots + 1) * H
        a = torch.full((g.N, cols), float("nan"), device="cuda")
        b = torch.full((g.N, cols), float("nan"), device="cuda")
        rs = None if rel_slot is None else rel_slot.data_ptr()
        _lib.check(lib.ercg_gather_bwd(dout.data_ptr(), H, None, 0, g.t_rowptr.data_ptr(), g.t_col.data_ptr(),
                                       g.t_etype.data_ptr(), g.t_eid.data_ptr(), rs, w.data_ptr(), R, slots * H,
                                       a.data_ptr(), cols, None, g.N, H, st), "ercg_gather_bwd")
        _lib.check(lib.ercg_gather_window_bwd(dout.data_ptr(), H, g.t_rowptr.data_ptr(), g.t_col.data_ptr(),
                                              g.t_etype.data_ptr(), g.t_eid.data_ptr(), rs, w.data_ptr(), slots, slots * H,
                                              b.data_ptr(), cols, g.N, H, wp, wf, st), "ercg_gather_window_bwd")
        torch.cuda.synchronize()
        assert not torch.isnan(b).any()
        assert torch.equal(a, b)


@pytest.mark.parametrize("N,C,p", [(37, 6, 0.0), (5000, 6, 0.5), (70001, 4, 0.5), (4096, 7, 0.0)])
def test_mlp_head_fused_backward(N, C, p):
    """Linear -> ReLU -> Dropout -> Linear as ONE autograd node (ops.mlp_head): the fused backward (one pass over the hidden
    activations) gives the same gradients as the chain of two ops.linear nodes (mask kernel, skinny GEMMs, column sums) and as
    fp64 autograd on the same dropout mask."""
    import erc_b200
    from erc_b200 import ops, _lib
    K = 100
    g = torch.Generator().manual_seed(N + C)
    x = torch.randn(N, K, generator=g).cuda().requires_grad_()
    W0, b0 = (torch.randn(K, K, generator=g) * 0.1).cuda().requires_grad_(), torch.randn(K, generator=g).cuda().requires_grad_()
    W3, b3 = (torch.randn(C, K, generator=g) * 0.1).cuda().requires_grad_(), torch.randn(C, generator=g).cuda().requires_grad_()
    dl = torch.randn(N, C, generator=g).cuda()
    act = ops.ACT_RELU_DROPOUT if p > 0 else ops.ACT_RELU
    scale = 1.0 / (1.0 - p) if p > 0 else 1.0

    def run(fused):
        for t in (x, W0, b0, W3, b3):
            t.grad = None
        if fused:
            out = ops.mlp_head(x, W0, b0, W3, b3, p, 77)
        else:
            out = ops.linear(ops.linear(x, W0, b0, act=act, drop_p=p, seed=77), W3, b3)
        n0 = _lib.launch_count()
        out.backward(dl)
        launches = _lib.launch_count() - n0
        return out.detach(), [t.grad.clone() for t in (x, W0, b0, W3, b3)], launches

    out_f, gf, lf = run(True)
    out_u, gu, lu = run(False)
    assert torch.equal(out_f, out_u)
    assert lf < lu                                   # fewer kernels, not just different ones
    # fp64 autograd with the mask the kernel drew (h > 0 after relu+dropout)
    h = ops.linear(x.detach(), W0.detach(), b0.detach(), act=act, drop_p=p, seed=77)
    mask = (h > 0).double() * scale
    xd, W0d, b0d, W3d, b3d = (t.detach().double().cpu().requires_grad_() for t in (x, W0, b0, W3, b3))
    hd = (xd @ W0d.t() + b0d) * mask.cpu()         # the mask IS relu' x dropout (no clamp: fp64 could flip a borderline sign)
    (hd @ W3d.t() + b3d).backward(dl.double().cpu())
    want = [t.grad for t in (xd, W0d, b0d, W3d, b3d)]
    for a, b, w in zip(gf, gu, want):
        assert rel_err(a, w) < 2e-5
        assert rel_err(a, b) < 2e-5


def test_mlp_head_input_with_a_second_consumer():
    """The node's input may have other consumers (COGMEN returns graph features next to the logits): the engine sums the
    gradients; nothing about the fused tail leaks out of the node."""
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(3)
    N, K, C = 4000, 100, 6
    x0 = torch.randn(N, K, generator=g).cuda().requires_grad_()
    Wp = (torch.randn(K, K, generator=g) * 0.1).cuda().requires_grad_()
    W0, b0 = (torch.randn(K, K, generator=g) * 0.1).cuda().requires_grad_(), torch.randn(K, generator=g).cuda().requires_grad_()
    W3, b3 = (torch.randn(C, K, generator=g) * 0.1).cuda().requires_grad_(), torch.randn(C, generator=g).cuda().requires_grad_()
    dl, extra = torch.randn(N, C, generator=g).cuda(), torch.randn(N, K, generator=g).cuda()
    f = ops.linear(x0, Wp)                                      # produced by one of our nodes, consumed twice
    ((ops.mlp_head(f, W0, b0, W3, b3, 0.5, 5) * dl).sum() + (f * extra).sum()).backward()
    h = ops.linear(f.detach(), W0.detach(), b0.detach(), act=ops.ACT_RELU_DROPOUT, drop_p=0.5, seed=5)
    mask = ((h > 0).double() * 2.0).cpu()
    d = [t.detach().double().cpu().requires_grad_() for t in (x0, Wp, W0, b0, W3, b3)]
    fd = d[0] @ d[1].t()
    ((((fd @ d[2].t() + d[3]) * mask) @ d[4].t() + d[5]) * dl.double().cpu()).sum().add((fd * extra.double().cpu()).sum()).backward()
    for a, w in zip((x0, Wp, W0, b0, W3, b3), d):
        assert rel_err(a.grad, w.grad) < 2e-5


def test_gradient_tags_do_not_survive_inplace_accumulation():
    """The by-products hung on gradient tensors (fused column sums) are tied to the tensor's version
    counter.  A feature tensor with TWO consumers makes the autograd engine add a second gradient to the tagged one; the
    bias gradient of the producing Linear must then be the column sums of the SUM, not the stale fused ones."""
    import erc_b200
    from erc_b200 import ops
    g = torch.Generator().manual_seed(9)
    N, K = 3000, 100
    x = torch.randn(N, K, generator=g).cuda()
    W0, b0 = (torch.randn(K, K, generator=g) * 0.1).cuda().requires_grad_(), torch.randn(K, generator=g).cuda().requires_grad_()
    W1 = (torch.randn(K, K, generator=g) * 0.1).cuda().requires_grad_()
    extra = torch.randn(N, K, generator=g).cuda()
    f = ops.linear(x, W0, b0)                       # feature tensor with two consumers
    y = ops.linear(f, W1)                           # consumer 1: its input gradient carries fused column sums
    loss = (y * y).sum() + (f * extra).sum()        # consumer 2: a plain ATen gradient added to it
    loss.backward()
    xd, W0d, b0d, W1d = x.double(), W0.detach().double().requires_grad_(), b0.detach().double().requires_grad_(), W1.detach().double()
    fd = xd @ W0d.t() + b0d
    ((fd @ W1d.t()) ** 2).sum().add((fd * extra.double()).sum()).backward()
    assert rel_err(b0.grad, b0d.grad) < 2e-5
    assert rel_err(W0.grad, W0d.grad) < 2e-5
    # and the tag helpers themselves
    t = torch.zeros(4, device="cuda")
    ops._tag_set(t, "_ercg_colsum", "payload")
    assert ops._tag_get(t, "_ercg_colsum") == "payload"
    t.add_(1.0)
    assert ops._tag_get(t, "_ercg_colsum") is None


@pytest.mark.parametrize("H,wp,wf,n", [(100, 5, 5, 2), (100, 10, 10, 2), (200, 4, 9, 3), (36, -1, -1, 2)])
def test_gather_forward_flat_mapping_is_bit_identical(H, wp, wf, n, monkeypatch):
    """gather_fwd_flat_kernel (thread per float4 chunk, all lanes busy) vs the warp-per-node kernel: same bits."""
    import erc_b200
    from erc_b200 import _lib
    from erc_b200.graph import build_graph
    rng = np.random.default_rng(H + wp + n)
    lens = torch.as_tensor(rng.integers(1, 50, size=41))
    spk = torch.as_tensor(rng.integers(0, n, size=(41, int(lens.max()))))
    g = build_graph(lens, spk.cuda(), wp, wf, n)
    R = 2 * n * n
    gen = torch.Generator().manual_seed(1)
    Y = torch.randn(g.N, (R + 1) * H, generator=gen).cuda()
    w = (torch.rand(g.E, generator=gen) + 0.1).cuda()
    bias = torch.randn(H, generator=gen).cuda()
    lib, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("ERCG_GATHER_FLAT", flag)
        o = torch.full((g.N, H), float("nan"), device="cuda")
        _lib.check(lib.ercg_gather_fwd(Y.data_ptr(), Y.stride(0), g.rowptr.data_ptr(), g.col.data_ptr(), g.etype.data_ptr(), None,
                                       w.data_ptr(), R * H, bias.data_ptr(), o.data_ptr(), H, g.N, H, st), "ercg_gather_fwd")
        torch.cuda.synchronize()
        outs.append(o)
    assert not torch.isnan(outs[0]).any() and torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("wp,wf,H", [(5, 5, 100), (0, 0, 100), (0, 3, 100), (3, 8, 100), (6, 6, 100), (12, 0, 100), (1, 11, 100),
                                     (5, 5, 36), (5, 5, 128), (2, 2, 4)])
def test_blocked_window_attention_matches_tile_kernels_and_fp64(wp, wf, H, monkeypatch):
    """attn_*_blk_kernel (register-blocked: 4 destinations share their candidate sources) against the round-1 tile kernels
    (ERCG_ATTN_BLK=0) and fp64, forward + backward + the fused bias-gradient column sums: many short dialogues (a tile spans
    several), single-utterance dialogues, N not a multiple of the 32-row tile, first / last tiles with clipped halos."""
    import erc_b200
    from erc_b200 import ops
    rng = np.random.default_rng(wp * 31 + wf * 7 + H)
    lens = [int(v) for v in rng.integers(1, 41, size=57)] + [1, 1, 2, 33, 64, 1]
    g, b = _graph(lens, wp=wp, wf=wf, seed=5)
    N = b["N"]
    gen = torch.Generator().manual_seed(H + wp)
    qkvs = torch.randn(N, 4 * H, generator=gen)
    dout = torch.randn(N, H, generator=gen)
    src, dst = torch.from_numpy(b["edge_index"][0]), torch.from_numpy(b["edge_index"][1])
    x = qkvs.double().requires_grad_()
    q, k, v, s = x[:, :H], x[:, H:2 * H], x[:, 2 * H:3 * H], x[:, 3 * H:]
    sc = (q[dst] * k[src]).sum(-1) / math.sqrt(H)
    mx = torch.full((N,), -1e300, dtype=torch.float64).scatter_reduce(0, dst, sc, reduce="amax")
    ex = (sc - mx[dst]).exp()
    alpha = ex / (torch.zeros(N, dtype=torch.float64).index_add(0, dst, ex) + 1e-16)[dst]
    want = torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, alpha[:, None] * v[src]) + s
    want.backward(dout.double())
    res = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("ERCG_ATTN_BLK", flag)
        xc = qkvs.cuda().requires_grad_()
        got = ops.edge_attention(xc, g, H, 1.0 / math.sqrt(H))
        (d,) = torch.autograd.grad(got, xc, dout.cuda())
        cs = ops._tag_get(d, "_ercg_colsum")
        assert cs is not None                                    # window path taken: column sums came with the gradient
        res[flag] = (got.detach(), d, cs)
        assert rel_err(got, want) < TOL and rel_err(d, x.grad) < TOL
        assert rel_err(cs, x.grad.sum(0)) < 1e-5
    assert rel_err(res["1"][0], res["0"][0]) < 2e-6 and rel_err(res["1"][1], res["0"][1]) < 2e-6
    assert not torch.isnan(res["1"][1]).any()


@pytest.mark.parametrize("n,wp,wf,one_speaker", [(2, 5, 5, True), (2, 5, 5, False), (1, 3, 7, True), (3, 0, 4, False), (2, 10, 0, False)])
def test_rgcn_transform_first_matches_fp64(n, wp, wf, one_speaker):
    """PyG RGCNConv on a K1 window graph, computed transform-first (GEMM + gather), against an fp64 evaluation of the
    layer's formula: output, input gradient, relation / root weight gradients (absent relations exactly zero), bias
    gradient.  At least 148 row tiles (the CTA-pair GEMM sizes), dialogues of length 1, windows clipped at both ends."""
    import erc_b200
    from erc_b200.graph import build_graph
    from erc_b200.pyg_nn import RGCNConv
    rng = np.random.default_rng(7 * n + wp + 3 * wf)
    lens = torch.as_tensor(np.concatenate([[1, 1, 2, 40, 3], rng.integers(1, 41, size=1100)]))
    spk = torch.as_tensor(rng.integers(0, 1 if one_speaker else n, size=(lens.numel(), int(lens.max()))))
    g = build_graph(lens, spk.cuda(), wp, wf, n)
    N, R, K, H = g.N, 2 * n * n, 100, 100
    assert N >= 148 * 128
    torch.manual_seed(3)
    conv = RGCNConv(K, H, R).cuda()
    with torch.no_grad():
        conv.bias.normal_()
    x0 = torch.randn(N, K, generator=torch.Generator().manual_seed(5)).cuda()
    dout = torch.randn(N, H, generator=torch.Generator().manual_seed(6)).cuda()
    edge_index, edge_type = g.attach(), g.edge_type
    x = x0.clone().requires_grad_()
    with erc_b200._lib.KernelTimer() as kt:
        out = conv(x, edge_index, edge_type)
        out.backward(dout)
    torch.cuda.synchronize()
    got = (out.detach(), x.grad, conv.weight.grad, conv.root.grad, conv.bias.grad)
    assert "ercg_gather_fwd" in set(kt.summary())
    # fp64 formula on the CPU
    src, dst, et = g.col.long().cpu(), edge_index[1].long().cpu(), g.etype.long().cpu()
    xd = x0.double().cpu().requires_grad_()
    Wd, rootd, bd = (t.detach().double().cpu().requires_grad_() for t in (conv.weight, conv.root, conv.bias))
    wmean = g.mean_weight().double().cpu()
    msg = torch.einsum("ek,ekh->eh", xd[src], Wd[et]) * wmean[:, None]
    want = torch.zeros(N, H, dtype=torch.float64).index_add(0, dst, msg) + xd @ rootd + bd
    want.backward(dout.double().cpu())
    refs = (want.detach(), xd.grad, Wd.grad, rootd.grad, bd.grad)
    for name, a, r in zip(("out", "dx", "dW", "droot", "dbias"), got, refs):
        assert rel_err(a, r) < TOL, (name, "transform-first vs fp64", rel_err(a, r))
    absent = [r_ for r_ in range(R) if not bool((et == r_).any())]
    for r_ in absent:
        assert float(got[2][r_].abs().max()) == 0.0
