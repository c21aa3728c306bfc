"""Micro-benchmark of one bidirectional recurrent layer, forward + backward with every weight gradient and dx: the GRU
(K6b, ops.gru_layer) against the LSTM (K6, ops.lstm_layer), both as the models run them (hoisted input GEMM + recurrence,
dgcn_models.birnn_forward), and torch's cuDNN nn.GRU / nn.LSTM on the same packed sequences as a yardstick.

    python tools/bench_rnn.py [--Hd 100] [--D 200] [--rounds 11]

Two batches of IEMOCAP-shaped dialogues (synth.iemocap_lengths): 32 (BASELINE config 2, seed 0; its ~1.6 k utterances fit
in L2) and 4096 (~200 k utterances, every buffer of the layer far larger than L2).  D = 200 is the input width of the second
layer of the 2-layer stacks (2 x Hd).  The arms alternate within each round; the line reports the median and the minimum
per-call time over the rounds, the per-kernel times of the recurrence launches (CUDA events around each call, a separate
pass), the number of library launches per call, and the largest difference of the GRU output from cuDNN's (TF32 off, so
both are fp32).  Prints one JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
from torch import nn
from torch.nn.utils.rnn import PackedSequence, pack_padded_sequence, pad_packed_sequence

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import erc_b200  # noqa: E402,F401
from erc_b200 import _lib, ops, synth  # noqa: E402
from erc_b200.track_mm.dgcn_models import birnn_forward  # noqa: E402
from erc_b200.track_mm.mmgcn_utils import lengths_graph  # noqa: E402


def power_limit_w(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except (OSError, ValueError, subprocess.SubprocessError):
        return None


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def run_size(name, lengths, D, Hd, rounds, warmup, dev):
    B, N, Lmax = lengths.numel(), int(lengths.sum()), int(lengths.max())
    gen = torch.Generator(device=dev).manual_seed(B)
    mask = torch.arange(Lmax, device=dev)[None, :] < lengths.to(dev)[:, None]
    x_pad = torch.randn(B, Lmax, D, device=dev, generator=gen) * mask[..., None]
    R_pad = torch.randn(B, Lmax, 2 * Hd, device=dev, generator=gen) * mask[..., None]
    graph = lengths_graph(lengths, dev)
    x = x_pad[mask].requires_grad_()                      # packed, dialogue-major: the layout of the library
    R = R_pad[mask].contiguous()
    ps = pack_padded_sequence(x_pad, lengths, batch_first=True, enforce_sorted=False)
    xs = ps.data.detach().requires_grad_()                # cuDNN's packed (time-major) layout, a leaf for dx
    ps = PackedSequence(xs, ps.batch_sizes, ps.sorted_indices, ps.unsorted_indices)
    Rs = pack_padded_sequence(R_pad, lengths, batch_first=True, enforce_sorted=False).data
    torch.manual_seed(0)
    gru = nn.GRU(D, Hd, num_layers=1, bidirectional=True).to(dev)
    lstm = nn.LSTM(D, Hd, num_layers=1, bidirectional=True).to(dev)

    def ours(rnn):
        def step():
            out = birnn_forward(rnn, x, graph, None, False)
            return torch.autograd.grad(out, [x] + list(rnn.parameters()), R)
        return step

    def cudnn(rnn):
        def step():
            out = rnn(ps)[0].data
            return torch.autograd.grad(out, [xs] + list(rnn.parameters()), Rs)
        return step

    arms = {"ops.gru_layer": ours(gru), "ops.lstm_layer": ours(lstm), "cudnn_gru": cudnn(gru), "cudnn_lstm": cudnn(lstm)}
    reps = {}
    for k, fn in arms.items():                             # warm-up; pick a repeat count that fills ~0.25 s per window
        for _ in range(warmup):
            fn()
        reps[k] = max(3, int(250.0 / max(timed(fn, 2), 1e-3)))
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, reps[k]))

    launches = {}
    for k in ("ops.gru_layer", "ops.lstm_layer"):
        before = _lib.launch_count()
        arms[k]()
        launches[k] = _lib.launch_count() - before
    with _lib.KernelTimer() as kt:                         # per-launch times of the recurrence kernels, own pass
        for k in ("ops.gru_layer", "ops.lstm_layer"):
            for _ in range(reps[k]):
                arms[k]()
        per_kernel = {e: round(ms / c, 4) for e, (c, ms) in kt.summary().items()
                      if e in ("ercg_gru_fwd", "ercg_gru_bwd", "ercg_lstm_fwd", "ercg_lstm_bwd")}

    with torch.no_grad():                                  # same weights, same inputs: our GRU output against cuDNN's
        mine = ops.unpack_rows(birnn_forward(gru, x, graph, None, False), graph, Lmax)
        ref, _ = pad_packed_sequence(gru(ps)[0], batch_first=True, total_length=Lmax)
        diff = float((mine - ref).abs().max() / ref.abs().max())
    floats = N * (D + 6 * Hd + 8 * Hd + 2 * Hd + 2 * Hd + 12 * Hd)    # x, gx, saved gates, h_prev, out, dgx + dgh
    return {"name": name, "B": B, "utterances": N, "max_len": Lmax, "gru_working_set_mb": round(4 * floats / 2 ** 20, 1),
            "ms_median": {k: round(statistics.median(v), 4) for k, v in samples.items()},
            "ms_min": {k: round(min(v), 4) for k, v in samples.items()},
            "reps_per_window": reps, "kernel_ms_per_call": per_kernel, "library_launches_per_call": launches,
            "gru_out_max_rel_diff_vs_cudnn": diff}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--Hd", type=int, default=100)
    ap.add_argument("--D", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rnn: needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    sizes = [("config2_b32", synth.iemocap_lengths(32, torch.Generator().manual_seed(0))),
             ("b4096", synth.iemocap_lengths(4096, torch.Generator().manual_seed(1)))]
    res = [run_size(n, l, args.D, args.Hd, args.rounds, args.warmup, dev) for n, l in sizes]
    print(json.dumps({"tool": "bench_rnn", "gpu": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(0),
                      "torch": torch.__version__, "cudnn": torch.backends.cudnn.version(), "Hd": args.Hd, "D": args.D,
                      "what": "one bidirectional layer, forward + backward (dx and all weight gradients), ms per call",
                      "sizes": res}))


if __name__ == "__main__":
    main()
