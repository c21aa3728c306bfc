"""Benchmark of one MMGCN and one DAG-ERC train step (forward + cross entropy + backward + Adam / AdamW with clip;
mmgcn.py:141-157, dagerc.py:217-237), three arms per model:

  (a) module_eager   train_mm's step: the module's forward on the padded batch (DAG-ERC: logits[attention_mask]) +
                     ops.cross_entropy + FlatAdam
  (b) step_eager     train_step.MmgcnTrainStep / DagercTrainStep .step (graphs prebuilt or built with host-known sizes)
  (c) step_replay    the same step captured once and replayed as one CUDA graph

    python tools/bench_mm_steps.py [--rounds 11] [--out result.json]

Workloads: SURVEY.md config 3 (MMGCN, 16 IEMOCAP-shaped dialogues, text 768 / audio 100 / visual 512, 2 speakers), config 4
(DAG-ERC, 16 dialogues, width 1380, 4 GNN layers) and 512 dialogues of each (the padded inputs alone are ~0.3 GB per model,
beyond the 126 MB L2).  Dropout as train_mm trains them (MMGCN 0.4, DAG-ERC 0.0), 6 classes, fp32, TF32 off.  Every arm
is warmed up, then the arms alternate within each of the rounds; a round times ``reps`` steps between CUDA events and ends
in a synchronise.  The line reports the median (and minimum) ms per step, utterances / s = N / median and the kernel
launches of one eager step of (a) and (b) (libercgraph's launch counter: ATen copies / cats are not counted).
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
from erc_b200.optim import FlatAdam  # noqa: E402
from erc_b200.track_mm.dagerc import DAGERCModule  # noqa: E402
from erc_b200.track_mm.mmgcn import MMGCNModule  # noqa: E402
from erc_b200.train_step import DagercTrainStep, MmgcnTrainStep  # noqa: E402
from bench_rnn import power_limit_w, timed  # noqa: E402

C = 6
MM_DIMS = dict(text=768, audio=100, visual=512)
DAG_EMB = 1380


def lengths_of(B, seed):
    return synth.iemocap_lengths(B, torch.Generator().manual_seed(seed))


def mmgcn_workload(B, dev, seed=0):
    lens = lengths_of(B, seed)
    Lmax, N = int(lens.max()), int(lens.sum())
    g = torch.Generator(device=dev).manual_seed(seed)
    mask = (torch.arange(Lmax, device=dev)[:, None] < lens.to(dev)[None, :]).float()[..., None]
    feats = tuple(torch.randn(Lmax, B, d, device=dev, generator=g) * mask for d in MM_DIMS.values())
    spk = torch.nn.functional.one_hot(torch.randint(0, 2, (Lmax, B), device=dev, generator=g), 2).float() * mask
    y = torch.randint(0, C, (N,), device=dev, generator=g)
    return lens, feats, spk, y


def dagerc_workload(B, dev, seed=0):
    lens = lengths_of(B, seed)
    Lmax = int(lens.max())
    g = torch.Generator(device=dev).manual_seed(seed)
    mask = torch.arange(Lmax, device=dev)[None, :] < lens.to(dev)[:, None]
    x = torch.randn(B, Lmax, DAG_EMB, device=dev, generator=g) * mask[..., None]
    spk = torch.nn.functional.one_hot(torch.randint(0, 2, (B, Lmax), device=dev, generator=g), 2).float() * mask[..., None]
    y = torch.randint(0, C, (B, Lmax), device=dev, generator=g).masked_fill(~mask, -100)
    return lens, x, spk, y, mask


def mmgcn_model(dev, seed=0):
    torch.manual_seed(seed)
    return MMGCNModule(hidden_text=768, hidden_visual=512, hidden_audio=100, n_speakers=2, n_classes=C).to(dev).train()


def dagerc_model(dev, seed=0):
    torch.manual_seed(seed)
    return DAGERCModule(emb_dim=DAG_EMB, dropout=0.0, gnn_layers=4, n_classes=C).to(dev).train()


def mmgcn_arms(B, dev):
    lens, (t, a, v), spk, y = mmgcn_workload(B, dev)
    ma = mmgcn_model(dev)
    opt = FlatAdam(ma.parameters(), lr=3e-4, weight_decay=3e-5)

    def arm_a():
        loss = ops.cross_entropy(ma(text_feature=t, audio_feature=a, visual_feature=v, speaker_tensor=spk,
                                    text_length=lens)[0], y)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss
    tsb = MmgcnTrainStep(mmgcn_model(dev), lens)
    tsc = MmgcnTrainStep(mmgcn_model(dev), lens).capture((t, a, v), spk, y)
    return lens, {"module_eager": arm_a, "step_eager": lambda: tsb.step((t, a, v), spk, y), "step_replay": tsc.replay}, tsc


def dagerc_arms(B, dev):
    lens, x, spk, y, mask = dagerc_workload(B, dev)
    ma = dagerc_model(dev)
    opt = FlatAdam(ma.parameters(), lr=1e-3, weight_decay=1e-2, decoupled=True, max_norm=5.0)
    y_packed = y[mask]

    def arm_a():
        logits = ma(input_tensor=x, text_length=lens, speaker_tensor=spk)[0][mask]
        loss = ops.cross_entropy(logits, y_packed)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss
    tsb = DagercTrainStep(dagerc_model(dev), lens)
    tsc = DagercTrainStep(dagerc_model(dev), lens).capture(x, spk, y)
    return lens, {"module_eager": arm_a, "step_eager": lambda: tsb.step(x, spk, y), "step_replay": tsc.replay}, tsc


def run_workload(model, B, rounds, dev):
    lens, arms, tsc = (mmgcn_arms if model == "mmgcn" else dagerc_arms)(B, dev)
    N = int(lens.sum())
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
    tsc.check()
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))
    med = {k: statistics.median(v) for k, v in samples.items()}
    return {"model": model, "workload": "%s_b%d" % (model, B), "dialogues": B, "utterances": N,
            "padded_length": int(lens.max()), "ms_median": {k: round(v, 3) for k, v in med.items()},
            "ms_min": {k: round(min(v), 3) for k, v in samples.items()},
            "utterances_per_s": {k: round(N / (v / 1e3)) for k, v in med.items()},
            "libercgraph_launches_per_eager_step": launches, "reps_per_window": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--workloads", default="mmgcn:16,mmgcn:512,dagerc:16,dagerc:512",
                    help="comma-separated model:dialogues (model = mmgcn or dagerc)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mm_steps: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda:0")
    res = []
    for item in args.workloads.split(","):
        model, B = item.split(":")
        if model not in ("mmgcn", "dagerc"):
            raise SystemExit("bench_mm_steps: unknown model %r" % model)
        res.append(run_workload(model, int(B), args.rounds, dev))
        print(json.dumps(res[-1]), file=sys.stderr)
        torch.cuda.empty_cache()
    line = json.dumps({"tool": "bench_mm_steps", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                       "torch": torch.__version__, "what": "one MMGCN / DAG-ERC train step (forward, CE, backward, Adam / "
                       "AdamW + clip), fp32, median of %d alternating rounds" % args.rounds, "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
