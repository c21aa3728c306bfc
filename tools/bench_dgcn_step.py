"""Benchmark of one DialogueGCN train step (forward + weighted cross entropy + backward + Adam, dgcn.py:117-134), four arms:

  (a) module_eager   today's path, train_mm's step: DGCNModule.forward on the padded batch + ops.cross_entropy + FlatAdam
  (b) step_eager     train_step.DgcnTrainStep.step on the packed batch (K1 with host-known sizes, forward_packed)
  (c) step_replay    the same step captured once and replayed as one CUDA graph
  (d) oracle_eager   the oracle's DGCN formulation (oracle/modules.py: nn.LSTM over pack_padded_sequence, EdgeAtt, the vendored
                     RGCNConv, GraphConv, the classifier) + F.cross_entropy + torch.optim.Adam in eager PyTorch on the same GPU.
                     Its graph tensors (edge_index / edge_type) are built once on the host, outside the timed step.

    python tools/bench_dgcn_step.py [--rounds 11] [--out result.json]

Workloads: synth.config2 (32 IEMOCAP-shaped dialogues, width 1380, 2 speakers, 6 classes, dgcn.py's class weights) and 4096
IEMOCAP-shaped dialogues (~200 k utterances: the inputs alone are 1.1 GB packed, beyond the 126 MB L2).  Dropout 0.4 as in
training, lr 3e-4, fp32, TF32 off.  Every arm is warmed up, then the arms alternate within each of the rounds; a round times
``reps`` steps between CUDA events and ends in a synchronise.  The line reports the median (and minimum) ms per step and
utterances / s = N / median.  With >= 2 GPUs visible the large workload is also run sharded by dialogue over 2 / 4 / 8 GPUs
(step_replay, peer-memory transport) under torch.distributed.run (``--dist-time``); otherwise the record says it was not run.

``--dist-check`` (under torch.distributed.run): the config-2 batch sharded over the ranks, captured step through peer memory,
against one rank's eager step on the whole batch (3 steps, dropout off); rank 0 prints the differences as a JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import erc_b200  # noqa: E402,F401
from erc_b200 import ops, synth  # noqa: E402
from erc_b200.dist import shard_dialogues  # noqa: E402
from erc_b200.optim import FlatAdam  # noqa: E402
from erc_b200.track_mm.dgcn import DGCNModule, LOSS_WEIGHTS  # noqa: E402
from erc_b200.train_step import DgcnTrainStep  # noqa: E402
from bench_rnn import power_limit_w, timed  # noqa: E402

D, C, LR = 1380, 6, 3e-4


def workload(name, dev):
    """(lengths [B] CPU, padded x [B, Lmax, D], padded speakers, packed x [N, D], packed speakers, labels [N]) on ``dev``."""
    if name == "config2":
        b = synth.config2(seed=0)
        lengths, x_pad, spk_pad, y = b["text_length"], b["input_tensor"].to(dev), b["speaker_tensor"].to(dev), b["label"].to(dev)
    else:
        gen = torch.Generator().manual_seed(2)
        lengths = synth.iemocap_lengths(4096, gen)
        B, Lmax, N = lengths.numel(), int(lengths.max()), int(lengths.sum())
        g = torch.Generator(device=dev).manual_seed(2)
        mask = torch.arange(Lmax, device=dev)[None, :] < lengths.to(dev)[:, None]
        x_pad = torch.randn(B, Lmax, D, device=dev, generator=g) * mask[..., None]
        spk_pad = torch.randint(0, 2, (B, Lmax), device=dev, generator=g) * mask
        y = torch.randint(0, C, (N,), device=dev, generator=g)
    mask = torch.arange(x_pad.size(1), device=dev)[None, :] < lengths.to(dev)[:, None]
    return lengths, x_pad, spk_pad, x_pad[mask].contiguous(), spk_pad[mask].contiguous(), y


def model(dev, seed=0, dropout=0.4):
    torch.manual_seed(seed)
    m = DGCNModule(2, input_size=D, hidden_size=200, n_classes=C, dropout=dropout).to(dev)
    m.train()
    return m


def oracle_arm(m, lengths, x_pad, spk_pad, y, w, dev):
    from oracle import modules as om
    o = om.DgcnOracle(2, input_size=D, hidden_size=200, n_classes=C, dropout=0.4)
    om.load_live(o, {k: v.detach().cpu() for k, v in m.state_dict().items()})
    o = o.to(dev).train()
    _, ei, et = om._graph_tensors(lengths, spk_pad.cpu(), o.wp, o.wf, o.n_speakers)
    ei, et = ei.to(dev), et.to(dev)
    opt = torch.optim.Adam(o.parameters(), lr=LR)

    def step():
        with torch.device(dev):                      # the oracle allocates its scatter target without a device argument
            ctx = o.rnn(lengths, x_pad)
            feats = om.pack_nodes(ctx, lengths)
            graph_out = o.gcn(feats, ei, o.edge_att(feats, ei), et)
            logits = o.clf(torch.cat([feats, graph_out], -1))
            loss = torch.nn.functional.cross_entropy(logits, y, weight=w)
            opt.zero_grad()
            loss.backward()
            opt.step()
        return loss
    return step


def run_workload(name, rounds, dev):
    lengths, x_pad, spk_pad, x, spk, y = workload(name, dev)
    N = int(lengths.sum())
    w = torch.tensor(LOSS_WEIGHTS, device=dev)
    ma = model(dev)
    opt_a = FlatAdam(ma.parameters(), lr=LR)

    def arm_a():
        loss = ops.cross_entropy(ma(x_pad, spk_pad, lengths)[0], y, w)
        opt_a.zero_grad()
        loss.backward()
        opt_a.step()
        return loss

    tsb = DgcnTrainStep(model(dev), lengths, class_weight=LOSS_WEIGHTS)
    tsc = DgcnTrainStep(model(dev), lengths, class_weight=LOSS_WEIGHTS).capture(x, spk, y)
    arms = {"module_eager": arm_a, "step_eager": lambda: tsb.step(x, spk, y), "step_replay": tsc.replay,
            "oracle_eager": oracle_arm(ma, lengths, x_pad, spk_pad, y, w, dev)}
    reps = {}
    for k, fn in arms.items():
        for _ in range(3):
            fn()
        reps[k] = max(1, int(200.0 / max(timed(fn, 1), 1e-3)))
    tsc.check()
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))
    med = {k: statistics.median(v) for k, v in samples.items()}
    return {"workload": name, "dialogues": int(lengths.numel()), "utterances": N,
            "ms_median": {k: round(v, 3) for k, v in med.items()},
            "ms_min": {k: round(min(v), 3) for k, v in samples.items()},
            "utterances_per_s": {k: round(N / (v / 1e3)) for k, v in med.items()},
            "reps_per_window": reps}


# ------------------------------------------------------------------------------------------ under torch.distributed.run
def _dist_init():
    import torch.distributed as dist
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    return dist, rank, world, torch.device("cuda", torch.cuda.current_device())


def _rel(a, b, floor=1e-30):
    return float((a - b).abs().max() / max(float(b.abs().max()), floor))


def _reduced_grads(ts):
    return {id(p): v.detach().clone() for p, v in zip(ts.opt.live, ts.opt.g_views)}


def dist_check_main():
    """Step 1 eager (its all-reduced gradient is compared), steps 2-3 the capture's warm-up, step 4 a replay; the whole
    batch takes 4 eager steps on one rank.  Gradient error per tensor against 1e-2 x the largest gradient as the floor."""
    dist, rank, world, dev = _dist_init()
    b = synth.config2(seed=0)
    lengths = b["text_length"]
    mask = torch.arange(b["input_tensor"].size(1))[None, :] < lengths[:, None]
    x_all, spk_all, y_all = b["input_tensor"][mask], b["speaker_tensor"][mask], b["label"]
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(lengths, 0)])
    idx = shard_dialogues(lengths, world)[rank]
    rows = torch.cat([torch.arange(int(off[d]), int(off[d + 1])) for d in idx.tolist()])
    m = model(dev, seed=3, dropout=0.0)
    ts = DgcnTrainStep(m, lengths[idx], class_weight=LOSS_WEIGHTS, world=world, group=dist.group.WORLD, transport="p2p")
    x, spk, y = x_all[rows].contiguous().to(dev), spk_all[rows].contiguous().to(dev), y_all[rows].contiguous().to(dev)
    ts.step(x, spk, y)
    g_shard = _reduced_grads(ts)
    ts.capture(x, spk, y, warmup=2)
    ts.replay()
    loss = float(ts.global_loss())
    ts.check()
    whole = model(dev, seed=3, dropout=0.0)
    tw = DgcnTrainStep(whole, lengths, class_weight=LOSS_WEIGHTS)
    xw, sw, yw = x_all.contiguous().to(dev), spk_all.contiguous().to(dev), y_all.to(dev)
    tw.step(xw, sw, yw)
    g_whole = _reduced_grads(tw)
    for _ in range(3):
        tw.step(xw, sw, yw)
    want = float(tw.global_loss())
    gmax = max(float(v.abs().max()) for v in g_whole.values())
    pairs = [(id(p), id(q)) for p, q in zip(m.parameters(), whole.parameters()) if id(p) in g_shard]
    gerr = max(_rel(g_shard[a], g_whole[b], floor=1e-2 * gmax) for a, b in pairs)
    d = [(p - q).abs() for p, q in zip(m.parameters(), whole.parameters())]
    if rank == 0:
        print(json.dumps({"tool": "bench_dgcn_step --dist-check", "world": world, "transport": ts.transport, "steps": 4,
                          "loss": loss, "loss_whole": want, "loss_rel_diff": abs(loss - want) / abs(want), "grad_rel_err": gerr,
                          "param_max_abs_diff": max(float(t.max()) for t in d),
                          "param_mean_abs_diff": max(float(t.mean()) for t in d)}))
    dist.barrier()
    dist.destroy_process_group()


def dist_time_main(rounds):
    dist, rank, world, dev = _dist_init()
    lengths, _, _, x_all, spk_all, y_all = workload("iemocap_b4096", dev)
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(lengths, 0)])
    idx = shard_dialogues(lengths, world)[rank]
    rows = torch.cat([torch.arange(int(off[d]), int(off[d + 1])) for d in idx.tolist()]).to(dev)
    x, spk, y = x_all[rows].contiguous(), spk_all[rows].contiguous(), y_all[rows].contiguous()
    del x_all
    ts = DgcnTrainStep(model(dev), lengths[idx], class_weight=LOSS_WEIGHTS, world=world, group=dist.group.WORLD)
    ts.capture(x, spk, y)
    for _ in range(3):
        ts.replay()
    samples = []
    for _ in range(rounds):
        dist.barrier()
        samples.append(timed(ts.replay, 3))
    ts.check()
    med = torch.tensor([statistics.median(samples)], device=dev)
    dist.all_reduce(med, op=dist.ReduceOp.MAX)
    N = int(lengths.sum())
    if rank == 0:
        print(json.dumps({"world": world, "transport": ts.transport, "utterances": N, "ms_median_slowest_rank": round(float(med), 3),
                          "utterances_per_s": round(N / (float(med) / 1e3))}))
    dist.barrier()
    dist.destroy_process_group()


def scaling(rounds):
    have = torch.cuda.device_count()
    if have < 2:
        return {"run": False, "reason": "not run: %d GPU visible" % have}
    out = {"run": True, "workload": "iemocap_b4096", "arm": "step_replay", "results": []}
    for w in (2, 4, 8):
        if w > have:
            out["results"].append({"world": w, "run": False, "reason": "not run: %d GPUs visible" % have})
            continue
        env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(w),
                            os.path.abspath(__file__), "--dist-time", "--rounds", str(rounds)],
                           capture_output=True, text=True, timeout=1800, env=env)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        out["results"].append(json.loads(lines[-1]) if r.returncode == 0 and lines else
                              {"world": w, "error": (r.stdout + r.stderr)[-1500:]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--dist-check", action="store_true", help="(under torch.distributed.run) sharded == whole check")
    ap.add_argument("--dist-time", action="store_true", help="(under torch.distributed.run) time the sharded large workload")
    ap.add_argument("--workloads", default="config2,iemocap_b4096")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dgcn_step: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    if args.dist_check:
        return dist_check_main()
    if args.dist_time:
        return dist_time_main(args.rounds)
    dev = torch.device("cuda:0")
    res = []
    for name in args.workloads.split(","):
        res.append(run_workload(name, args.rounds, dev))
        print(json.dumps(res[-1]), file=sys.stderr)
        torch.cuda.empty_cache()
    line = json.dumps({"tool": "bench_dgcn_step", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                       "torch": torch.__version__, "what": "one DialogueGCN train step (forward, weighted CE, backward, Adam), "
                       "fp32, dropout 0.4, median of %d alternating rounds" % args.rounds,
                       "results": res, "strong_scaling": scaling(args.rounds)})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
