"""Benchmark of DialogueRNN (K12, csrc/dialogue_rnn.cu) forward + backward against the reference's formulation -- the per-step
Python loop of DialogueRNN / DialogueRNNCell (oracle/dialogue_rnn_oracle.py, a transcription of the declare-lab classes) in
eager PyTorch on the same GPU.

    python tools/bench_dialogue_rnn.py [--rounds 11] [--out result.json]

D_m = 1380 (the IEMOCAP atv width train_mm builds), D_g / D_p / D_e = 150 / 150 / 100, context_attention 'general', P = 2,
eval mode (no dropout), fp32, TF32 off.  Two sizes: B = 32 IEMOCAP-like dialogues (synth.iemocap_lengths, seed 1) with L =
the longest of them, and B = 4096 at L = 110.  qmask rows are one-hot inside each dialogue and all-zero after it.  Both arms
compute e, dU and every parameter gradient of sum(e * R), including the hoisted input GEMM.  The arms alternate within each
round; the line reports the median and the minimum per-call time over the rounds and the largest difference of our e from
the reference's.
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import erc_b200  # noqa: E402,F401
from erc_b200 import synth  # noqa: E402
from erc_b200.track_mm.dgcnv2_models import DialogueRNN  # noqa: E402
from oracle import dialogue_rnn_oracle as O  # noqa: E402
from bench_rnn import power_limit_w, timed  # noqa: E402

DM, DG, DP, DE, P = 1380, 150, 150, 100, 2


def run_size(name, lengths, L, rounds, warmup, dev):
    B = len(lengths)
    gen = torch.Generator().manual_seed(B)
    torch.manual_seed(B)
    ref = O.DialogueRNN(DM, DG, DP, DE, context_attention="general").to(dev).eval()
    ours = DialogueRNN(DM, DG, DP, DE, context_attention="general").to(dev).eval()
    ours.load_state_dict(ref.state_dict(), strict=True)
    U = torch.randn(L, B, DM, generator=gen).to(dev).requires_grad_()
    spk = torch.randint(0, P, (L, B), generator=gen)
    inside = torch.arange(L)[:, None] < torch.tensor(lengths)[None, :]
    qm = (torch.nn.functional.one_hot(spk, P).float() * inside[..., None]).to(dev)
    R = torch.randn(L, B, DE, generator=gen).to(dev)

    def arm(m):
        params = list(m.parameters())
        return lambda: torch.autograd.grad(m(U, qm)[0], [U] + params, R)

    arms = {"ours": arm(ours), "reference_loop": arm(ref)}
    reps = {}
    for k, fn in arms.items():
        for _ in range(warmup):
            fn()
        reps[k] = max(1, int(250.0 / max(timed(fn, 1), 1e-3)))
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))
    with torch.no_grad():
        a, b = ours(U, qm)[0], ref(U, qm)[0]
        diff = float((a - b).abs().max() / b.abs().max())
    med = {k: round(statistics.median(v), 3) for k, v in samples.items()}
    return {"size": name, "B": B, "L": L, "ms_median": med, "ms_min": {k: round(min(v), 3) for k, v in samples.items()},
            "speedup_median": round(med["reference_loop"] / med["ours"], 2), "reps_per_window": reps,
            "e_max_rel_diff": diff}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dialogue_rnn: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda:0")
    small = [int(v) for v in synth.iemocap_lengths(32, torch.Generator().manual_seed(1))]
    res = [run_size("iemocap_b32", small, max(small), args.rounds, args.warmup, dev),
           run_size("b4096_l110", [110] * 4096, 110, args.rounds, args.warmup, dev)]
    line = json.dumps({"tool": "bench_dialogue_rnn", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                       "torch": torch.__version__, "widths": {"D_m": DM, "D_g": DG, "D_p": DP, "D_e": DE, "P": P},
                       "context_attention": "general",
                       "what": "forward + backward (dU and every parameter gradient), fp32, eval, ms per call", "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
