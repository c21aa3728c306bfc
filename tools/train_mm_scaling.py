"""Epoch throughput of data-parallel ``train_mm.py`` at several GPU counts (reported, not asserted).

    python tools/train_mm_scaling.py --out train_mm_scaling.json [--gpus 1,2,8] [--modules cogmen,dgcn]

Every (module, GPU count) pair runs ``--repeats`` times, the pairs alternating within each repeat so that drift of the shared
machine hits them alike.  One run = ``python -m torch.distributed.run --standalone --nproc_per_node N train_mm.py`` on an
IEMOCAP-shaped synthetic data set (iemocap-cogmen-6 feature sizes, IEMOCAP-like dialogue lengths, per-GPU batch 32); the
first epoch is warm-up, the utt/s of the later epochs (utterances of all ranks over rank 0's epoch time, test pass excluded)
are recorded.  GPU counts above the visible devices are skipped."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(module, world, args):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node", str(world),
           os.path.join(ROOT, "train_mm.py"), "--module=" + module, "--dataset=iemocap-cogmen-6", "--modality=atv",
           "--epoch=%d" % args.epochs, "--train_dialogues=%d" % args.train_dialogues, "--test_dialogues=31",
           "--train.batch_size=32"]
    t0 = time.time()
    out = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
    if out.returncode != 0:
        raise SystemExit("%s at %d GPUs failed (%d):\n%s" % (module, world, out.returncode, out.stdout[-4000:]))
    rates = [float(x) for x in re.findall(r"\|\s+(\d+) utt/s", out.stdout)]
    transport = re.search(r"through (.*)$", out.stdout, flags=re.M)
    return {"module": module, "gpus": world, "utt_per_s_by_epoch": rates, "utt_per_s": statistics.median(rates[1:]),
            "transport": transport.group(1) if transport else None, "wall_s": round(time.time() - t0, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--modules", default="cogmen,dgcn")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--train_dialogues", type=int, default=2048)
    args = ap.parse_args()
    import torch
    visible = torch.cuda.device_count()
    gpus = [g for g in (int(x) for x in args.gpus.split(",")) if g <= visible]
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                               text=True).stdout.strip().splitlines()
    except OSError:
        power = None
    runs = []
    for rep in range(args.repeats):
        for module in args.modules.split(","):
            for world in gpus:
                r = run(module, world, args)
                r["repeat"] = rep
                runs.append(r)
                print(json.dumps(r), flush=True)
    summary = {}
    for module in args.modules.split(","):
        for world in gpus:
            xs = [r["utt_per_s"] for r in runs if r["module"] == module and r["gpus"] == world]
            summary["%s_%dgpu" % (module, world)] = {"median_utt_per_s": statistics.median(xs), "runs": xs}
    res = {"device": torch.cuda.get_device_name(0), "visible_gpus": visible, "nvidia_smi_name_power_limit": power,
           "train_dialogues": args.train_dialogues, "epochs": args.epochs, "summary": summary, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
