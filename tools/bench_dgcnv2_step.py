"""Benchmark of one dgcnv2 train step (the declare-lab DialogueGCN, track_mm/dgcnv2.py: forward + weighted cross entropy +
backward + Adam), three arms:

  (a) module_eager   train_mm's step: DGCNModule.forward on the seq-first padded batch + ops.cross_entropy + FlatAdam
  (b) step_eager     train_step.Dgcnv2TrainStep.step on the batch-first padded rows (K1 with host-known sizes,
                     forward_packed: the layer-0 input transform on the tensor-core GEMMs)
  (c) step_replay    the same step captured once and replayed as one CUDA graph

    python tools/bench_dgcnv2_step.py [--rounds 11] [--out result.json]

Workloads: synth.config2 (32 IEMOCAP-shaped dialogues, width 1380, 2 speakers, 6 classes, dgcn.py's class weights) and 4096
IEMOCAP-shaped dialogues (the padded inputs alone are 2.5 GB per layout, far beyond the 126 MB L2).  LSTM base (train_mm's
default), hidden 100, dropout 0.4 as in training, lr 3e-4, fp32, TF32 off.  Every arm is warmed up, then the arms alternate
within each of the rounds; a round times ``reps`` steps between CUDA events and ends in a synchronise.  The line reports the
median (and minimum) ms per step, utterances / s = N / median and the libercgraph launches of one eager step of (a) and
(b) (ATen copies / cats are not counted).  Strong scaling over several GPUs is not timed by this tool.

``--dist-check`` (under torch.distributed.run): the config-2 batch sharded over the ranks (each shard padded to the global
lmax), captured step through peer memory, against one rank's eager step on the whole batch (4 steps, dropout off); rank 0
prints the differences as a JSON line.
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import erc_b200  # noqa: E402,F401
from erc_b200 import _lib, ops, synth  # noqa: E402
from erc_b200.dist import shard_dialogues  # noqa: E402
from erc_b200.optim import FlatAdam  # noqa: E402
from erc_b200.track_mm.dgcn import LOSS_WEIGHTS  # noqa: E402
from erc_b200.track_mm.dgcnv2 import DGCNModule  # noqa: E402
from erc_b200.train_step import Dgcnv2TrainStep  # noqa: E402
from bench_rnn import power_limit_w, timed  # noqa: E402

D, H, C, LR = 1380, 100, 6, 3e-4


def workload(name, dev):
    """(lengths [B] CPU, batch-first padded x [B, Lmax, D], padded speaker ids [B, Lmax], labels [N]) on ``dev``."""
    if name == "config2":
        b = synth.config2(seed=0)
        return b["text_length"], b["input_tensor"].to(dev), b["speaker_tensor"].to(dev), b["label"].to(dev)
    gen = torch.Generator().manual_seed(2)
    lengths = synth.iemocap_lengths(4096, gen)
    B, Lmax, N = lengths.numel(), int(lengths.max()), int(lengths.sum())
    g = torch.Generator(device=dev).manual_seed(2)
    mask = torch.arange(Lmax, device=dev)[None, :] < lengths.to(dev)[:, None]
    x = torch.randn(B, Lmax, D, device=dev, generator=g) * mask[..., None]
    spk = torch.randint(0, 2, (B, Lmax), device=dev, generator=g) * mask
    return lengths, x, spk, torch.randint(0, C, (N,), device=dev, generator=g)


def model(dev, seed=0, dropout=0.4):
    torch.manual_seed(seed)
    m = DGCNModule("LSTM", input_size=D, hidden_size=H, n_speakers=2, n_classes=C, dropout=dropout).to(dev)
    m.train()
    return m


def layouts(lengths, x, spk):
    """(seq-first x [Lmax, B, D], seq-first one-hot speakers, rows [B * Lmax, D], packed speaker ids [N])."""
    mask = torch.arange(x.size(1), device=x.device)[None, :] < lengths.to(x.device)[:, None]
    x_seq = x.transpose(0, 1).contiguous()
    spk_seq = torch.nn.functional.one_hot(spk.t(), 2).float()
    return x_seq, spk_seq, x.reshape(-1, D), spk[mask].contiguous()


def run_workload(name, rounds, dev):
    lengths, x, spk, y = workload(name, dev)
    x_seq, spk_seq, x_rows, spk_packed = layouts(lengths, x, spk)
    N = int(lengths.sum())
    w = torch.tensor(LOSS_WEIGHTS, device=dev)
    ma = model(dev)
    opt_a = FlatAdam(ma.parameters(), lr=LR)

    def arm_a():
        loss = ops.cross_entropy(ma(x_seq, spk_seq, None, lengths)[0], y, w)
        opt_a.zero_grad()
        loss.backward()
        opt_a.step()
        return loss

    tsb = Dgcnv2TrainStep(model(dev), lengths, class_weight=LOSS_WEIGHTS)
    tsc = Dgcnv2TrainStep(model(dev), lengths, class_weight=LOSS_WEIGHTS).capture(x_rows, spk_packed, y)
    arms = {"module_eager": arm_a, "step_eager": lambda: tsb.step(x_rows, spk_packed, y), "step_replay": tsc.replay}
    reps, launches = {}, {}
    for k, fn in arms.items():
        for _ in range(3):
            fn()
        if k != "step_replay":
            torch.cuda.synchronize()
            before = _lib.launch_count()
            fn()
            torch.cuda.synchronize()
            launches[k] = _lib.launch_count() - before
        reps[k] = max(1, int(200.0 / max(timed(fn, 1), 1e-3)))
    tsb.check()
    tsc.check()
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))
    med = {k: statistics.median(v) for k, v in samples.items()}
    return {"workload": name, "dialogues": int(lengths.numel()), "utterances": N, "padded_length": int(lengths.max()),
            "ms_median": {k: round(v, 3) for k, v in med.items()},
            "ms_min": {k: round(min(v), 3) for k, v in samples.items()},
            "utterances_per_s": {k: round(N / (v / 1e3)) for k, v in med.items()},
            "libercgraph_launches_per_eager_step": launches, "reps_per_window": reps}


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
    lengths, x_all, spk_all, y_all = b["text_length"], b["input_tensor"], b["speaker_tensor"], b["label"]
    lmax = int(lengths.max())
    mask = torch.arange(lmax)[None, :] < lengths[:, None]
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(lengths, 0)])
    idx = shard_dialogues(lengths, world)[rank]
    rows = torch.cat([torch.arange(int(off[d]), int(off[d + 1])) for d in idx.tolist()])
    m = model(dev, seed=3, dropout=0.0)
    ts = Dgcnv2TrainStep(m, lengths[idx], lmax=lmax, class_weight=LOSS_WEIGHTS, world=world, group=dist.group.WORLD,
                         transport="p2p")
    x = x_all[idx].reshape(-1, D).contiguous().to(dev)                  # this shard, padded to the global lmax
    spk, y = spk_all[mask][rows].contiguous().to(dev), y_all[rows].contiguous().to(dev)
    ts.step(x, spk, y)
    g_shard = _reduced_grads(ts)
    ts.capture(x, spk, y, warmup=2)
    ts.replay()
    loss = float(ts.global_loss())
    ts.check()
    whole = model(dev, seed=3, dropout=0.0)
    tw = Dgcnv2TrainStep(whole, lengths, class_weight=LOSS_WEIGHTS)
    xw, sw, yw = x_all.reshape(-1, D).contiguous().to(dev), spk_all[mask].contiguous().to(dev), y_all.to(dev)
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
        print(json.dumps({"tool": "bench_dgcnv2_step --dist-check", "world": world, "transport": ts.transport, "steps": 4,
                          "shard_longest": [int(lengths[i].max()) for i in shard_dialogues(lengths, world)], "lmax": lmax,
                          "loss": loss, "loss_whole": want, "loss_rel_diff": abs(loss - want) / abs(want), "grad_rel_err": gerr,
                          "param_max_abs_diff": max(float(t.max()) for t in d),
                          "param_mean_abs_diff": max(float(t.mean()) for t in d)}))
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--dist-check", action="store_true", help="(under torch.distributed.run) sharded == whole check")
    ap.add_argument("--workloads", default="config2,iemocap_b4096")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dgcnv2_step: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    if args.dist_check:
        return dist_check_main()
    dev = torch.device("cuda:0")
    res = []
    for name in args.workloads.split(","):
        res.append(run_workload(name, args.rounds, dev))
        print(json.dumps(res[-1]), file=sys.stderr)
        torch.cuda.empty_cache()
    line = json.dumps({"tool": "bench_dgcnv2_step", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                       "torch": torch.__version__, "what": "one dgcnv2 train step (LSTM base; forward, weighted CE, backward, "
                       "Adam), fp32, dropout 0.4, median of %d alternating rounds" % args.rounds, "results": res,
                       "strong_scaling": "not measured: this tool times one GPU"})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
