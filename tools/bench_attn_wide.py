"""Micro-benchmark of the K4 / K5 warp-per-node attention kernels (csrc/attn.cu) at widths past H = 384 and at float2
chunks, forward + backward, against the reference's PyTorch formulation in eager mode on the same GPU.

    python tools/bench_attn_wide.py [--rounds 11] [--out result.json]

4096 IEMOCAP-shaped dialogues (synth.iemocap_lengths, seed 1; ~200 k utterances), fp32, TF32 off.
  * K5 EdgeAtt (DialogueGCN), g in {300 (float4 NC = 3), 302 (float2), 512, 768}: ops.edge_att(x, u) on
    the 10 / 10 window graph, gradients of x and u, against the oracle's formulation (oracle/modules.py EdgeAttOracle after
    its u = x W^T: gather both ends of every edge, per-source scatter softmax).
  * K4 nodal MatchingAttention 'general2' (dgcnv2), width in {356 (h = 128, float4 NC = 3), 358 (h = 129, float2), 868
    (h = 384)}: ops.matching_attention(xt, e) on the fully connected per-dialogue graph, gradients of xt and e, against the
    reference's loop over the 110 query positions of the padded [L, B, H] batch (dgcnv2_models.py attentive_node_features
    -> MatchingAttention 'general2': bmm, tanh, softmax, mask, renormalise, bmm).  The reference's M * mask product is
    left out: the padded rows are zero already, and autograd would keep one [B, H, L] copy of it per position.
Neither arm includes the Linear that produces u / xt.  The arms alternate within each round; the line reports the median
and the minimum per-call time over the rounds and the largest difference of our output from the reference's.
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import erc_b200  # noqa: E402,F401
from erc_b200 import ops, synth  # noqa: E402
from erc_b200.graph import build_graph  # noqa: E402
from bench_rnn import power_limit_w, timed  # noqa: E402


def edge_att_ref(x, u, src, n):
    score = (x.index_select(0, src[0]) * u.index_select(0, src[1])).sum(-1)
    smax = torch.full((n,), float("-inf"), device=x.device).scatter_reduce(0, src[0], score, reduce="amax", include_self=True)
    ex = (score - smax[src[0]]).exp()
    return ex / torch.zeros(n, device=x.device).index_add_(0, src[0], ex)[src[0]]


def matching_ref(xt_pad, e_pad, mask):
    """[L, B, H] queries and memory, [B, L] mask -> [L, B, H]: one MatchingAttention 'general2' call per position."""
    M_ = e_pad.permute(1, 2, 0)                     # B, H, L
    Mb = e_pad.transpose(0, 1)                      # B, L, H
    m = mask.unsqueeze(1)                           # B, 1, L
    out = []
    for t in range(xt_pad.size(0)):
        a = torch.tanh(torch.bmm(xt_pad[t].unsqueeze(1), M_) * m)
        a = F.softmax(a, dim=2) * m
        a = a / a.sum(2, keepdim=True)
        out.append(torch.bmm(a, Mb)[:, 0, :])
    return torch.stack(out, 0)


def run_arms(arms, rounds, warmup):
    reps = {}
    for k, fn in arms.items():
        for _ in range(warmup):
            fn()
        reps[k] = max(3, int(250.0 / max(timed(fn, 2), 1e-3)))
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))
    return ({k: round(statistics.median(v), 4) for k, v in samples.items()},
            {k: round(min(v), 4) for k, v in samples.items()}, reps)


def bench_edge_att(g_dim, lengths, spk, rounds, warmup, dev):
    graph = build_graph(lengths, spk, 10, 10, 2)
    N = int(lengths.sum())
    gen = torch.Generator(device=dev).manual_seed(g_dim)
    x = (torch.randn(N, g_dim, device=dev, generator=gen) * g_dim ** -0.25).requires_grad_()
    u = (torch.randn(N, g_dim, device=dev, generator=gen) * g_dim ** -0.25).requires_grad_()
    dst = torch.repeat_interleave(torch.arange(N, device=dev), graph.rowptr[1:] - graph.rowptr[:-1])
    src = (graph.col.long(), dst)                   # by-destination CSR order: the order ops.edge_att returns
    dnu = torch.randn(src[1].numel(), device=dev, generator=gen)
    arms = {"ops.edge_att": lambda: torch.autograd.grad(ops.edge_att(x, u, graph), [x, u], dnu),
            "reference": lambda: torch.autograd.grad(edge_att_ref(x, u, src, N), [x, u], dnu)}
    med, mn, reps = run_arms(arms, rounds, warmup)
    with torch.no_grad():
        a, b = ops.edge_att(x, u, graph), edge_att_ref(x, u, src, N)
        diff = float((a - b).abs().max() / b.abs().max())
    return {"kernel": "K5 edge_att", "width": g_dim, "utterances": N, "edges": int(dnu.numel()), "ms_median": med,
            "ms_min": mn, "reps_per_window": reps, "out_max_rel_diff": diff}


def bench_nodal(width, lengths, spk, rounds, warmup, dev):
    graph = build_graph(lengths, spk, -1, -1, 2)
    B, L, N = lengths.numel(), int(lengths.max()), int(lengths.sum())
    gen = torch.Generator(device=dev).manual_seed(width)
    mask = (torch.arange(L, device=dev)[None, :] < lengths.to(dev)[:, None]).float()          # B, L
    xt_pad = torch.randn(L, B, width, device=dev, generator=gen) * width ** -0.25 * mask.t()[..., None]
    e_pad = torch.randn(L, B, width, device=dev, generator=gen) * width ** -0.25 * mask.t()[..., None]
    dout_pad = torch.randn(L, B, width, device=dev, generator=gen) * mask.t()[..., None]
    sel = mask.t().bool()                                                                    # L, B
    pack = lambda t: t.transpose(0, 1)[sel.t()].contiguous()                                 # noqa: E731  dialogue-major
    xt, e, dout = pack(xt_pad).requires_grad_(), pack(e_pad).requires_grad_(), pack(dout_pad)
    xt_pad.requires_grad_()
    e_pad.requires_grad_()
    arms = {"ops.matching_attention": lambda: torch.autograd.grad(ops.matching_attention(xt, e, graph), [xt, e], dout),
            "reference": lambda: torch.autograd.grad(matching_ref(xt_pad, e_pad, mask), [xt_pad, e_pad], dout_pad)}
    med, mn, reps = run_arms(arms, rounds, warmup)
    with torch.no_grad():
        a, b = ops.matching_attention(xt, e, graph), pack(matching_ref(xt_pad, e_pad, mask))
        diff = float((a - b).abs().max() / b.abs().max())
    return {"kernel": "K4 matching_attention (tanh)", "width": width, "utterances": N, "edges": int(graph.col.numel()),
            "ms_median": med, "ms_min": mn, "reps_per_window": reps, "out_max_rel_diff": diff}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dialogues", type=int, default=4096)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_attn_wide: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda:0")
    lengths = synth.iemocap_lengths(args.dialogues, torch.Generator().manual_seed(1))
    spk = torch.randint(0, 2, (int(lengths.sum()),), generator=torch.Generator().manual_seed(2)).to(dev)
    res = [bench_edge_att(g, lengths, spk, args.rounds, args.warmup, dev) for g in (300, 302, 512, 768)]
    res += [bench_nodal(w, lengths, spk, args.rounds, args.warmup, dev) for w in (356, 358, 868)]
    line = json.dumps({"tool": "bench_attn_wide", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                       "torch": torch.__version__, "dialogues": args.dialogues,
                       "what": "forward + backward (input gradients), fp32, ms per call", "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
