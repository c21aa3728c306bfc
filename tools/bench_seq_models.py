"""Benchmark of the declare-lab sequence classifiers of track_mm/dgcnv2_models.py -- the att2 matching attention (K13,
csrc/seq_attn.cu), LSTMModel, GRUModel and DialogRNNModel -- forward + backward against the reference's formulation
(oracle/dgcnv2_seq_oracle.py: the per-position loop of MatchingAttention calls, nn.LSTM / nn.GRU, the per-step DialogueRNN
loop, flip / pad_sequence) in eager PyTorch on the same GPU.

    python tools/bench_seq_models.py [--rounds 5] [--out result.json]

Widths: D_m = 1380 (IEMOCAP atv); LSTMModel / GRUModel D_e = 100, D_h = 100; DialogRNNModel D_g / D_p / D_e = 150 / 150 / 100,
D_h = 100, context_attention 'general', P = 2; the att2 attention alone at width 200 (= 2 D_e, the models' memory).  6 classes,
dropout 0 and eval mode (the reference's nn.LSTM / nn.GRU in training mode, which cuDNN's backward requires and which
computes the same with dropout 0), fp32, TF32 off, att2 on.  Two sizes: 32 and 4096 IEMOCAP-like dialogues (synth.iemocap_lengths,
seeds 1 and 2) with L = the longest of them; U is zero and qmask all-zero after each dialogue, umask the prefix mask.  Each
arm computes the outputs and the gradients of dU (the attention: dM) and every parameter of sum(out * R).  The arms
alternate within each round; the line reports the median and minimum per-call time over the rounds and the largest
difference of our output from the reference's (relative to its largest magnitude).
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
from erc_b200.track_mm import dgcnv2_models as ours_mod  # noqa: E402
from oracle import dgcnv2_seq_oracle as O  # noqa: E402
from bench_rnn import power_limit_w, timed  # noqa: E402

DM, C, P = 1380, 6, 2
MODELS = {"LSTMModel": ((DM, 100, 100), {}), "GRUModel": ((DM, 100, 100), {}),
          "DialogRNNModel": ((DM, 150, 150, 100, 100), {"context_attention": "general"})}


def _time_arms(arms, rounds, warmup):
    reps = {}
    for k, fn in arms.items():
        for _ in range(warmup):
            fn()
        reps[k] = max(1, int(250.0 / max(timed(fn, 1), 1e-3)))
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))
    med = {k: round(statistics.median(v), 3) for k, v in samples.items()}
    return {"ms_median": med, "ms_min": {k: round(min(v), 3) for k, v in samples.items()},
            "speedup_median": round(med["reference_loop"] / med["ours"], 2), "reps_per_window": reps}


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


def run_size(name, lengths, rounds, warmup, dev):
    B, L = len(lengths), max(lengths)
    gen = torch.Generator().manual_seed(B)
    inside = torch.arange(L)[:, None] < torch.tensor(lengths)[None, :]
    U = (torch.randn(L, B, DM, generator=gen) * inside[..., None]).to(dev).requires_grad_()
    qm = (torch.nn.functional.one_hot(torch.randint(0, P, (L, B), generator=gen), P).float() * inside[..., None]).to(dev)
    umask = inside.t().float().contiguous().to(dev)
    R = torch.randn(L, B, C, generator=gen).to(dev)
    out = []

    # the att2 attention alone: every position of every dialogue against its dialogue's memory
    torch.manual_seed(B)
    ref_att = O.MatchingAttention(200, 200, att_type="general2").to(dev)
    our_att = ours_mod.MatchingAttention(200, 200, att_type="general2").to(dev)
    our_att.load_state_dict(ref_att.state_dict(), strict=True)
    Mem = torch.tanh(torch.randn(L, B, 200, generator=gen)).to(dev).requires_grad_()
    R2 = torch.randn(L, B, 200, generator=gen).to(dev)

    def ref_all():
        return torch.stack([ref_att(Mem, Mem[t], umask)[0] for t in range(L)])

    def att_arm(fwd, m):
        params = list(m.parameters())
        return lambda: torch.autograd.grad(fwd(), [Mem] + params, R2)

    arms = {"ours": att_arm(lambda: our_att.all_positions(Mem, umask)[0], our_att), "reference_loop": att_arm(ref_all, ref_att)}
    rec = {"size": name, "B": B, "L": L, "what": "att2 MatchingAttention general2, width 200", **_time_arms(arms, rounds, warmup)}
    with torch.no_grad():
        rec["max_rel_diff"] = _rel(our_att.all_positions(Mem, umask)[0], ref_all())
    out.append(rec)
    del Mem, R2

    for mname, (dims, kw) in MODELS.items():
        torch.manual_seed(B)
        ref = getattr(O, mname)(*dims, n_classes=C, dropout=0.0, **kw).to(dev).eval()
        ours = getattr(ours_mod, mname)(*dims, n_classes=C, dropout=0.0, **kw).to(dev).eval()
        if mname != "DialogRNNModel":
            ref.train()                     # cuDNN's RNN backward needs training mode; with dropout 0 it computes what eval does
        ours.load_state_dict(ref.state_dict(), strict=True)

        def arm(m):
            params = list(m.parameters())
            return lambda: torch.autograd.grad(m(U, qm, umask)[0], [U] + params, R)

        arms = {"ours": arm(ours), "reference_loop": arm(ref)}
        rec = {"size": name, "B": B, "L": L, "what": mname, **_time_arms(arms, rounds, warmup)}
        with torch.no_grad():
            rec["max_rel_diff"] = _rel(ours(U, qm, umask)[0], ref(U, qm, umask)[0])
        out.append(rec)
        del ref, ours
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_seq_models: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda:0")
    res = []
    for name, B, seed in (("iemocap_b32", 32, 1), ("iemocap_b4096", 4096, 2)):
        lengths = [int(v) for v in synth.iemocap_lengths(B, torch.Generator().manual_seed(seed))]
        res += run_size(name, lengths, args.rounds, args.warmup, dev)
        print(json.dumps(res[-4:]), file=sys.stderr)
    line = json.dumps({"tool": "bench_seq_models", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                       "torch": torch.__version__, "what": "forward + backward (dU / dM and every parameter gradient), fp32, "
                       "eval, att2, ms per call", "results": res})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
