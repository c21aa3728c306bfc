#!/usr/bin/env python
"""bench.py -- COGMEN fwd+bwd utterances/sec on the BASELINE.json config-5 workload.

  python bench.py --gpus N --steps K --warmup W            our arm (libercgraph kernels)
  python bench.py --impl reference --gpus N ...            the reference's CPU path (oracle port), rank 0 only

Workload ("config.workload"): COGMEN train step (graphify + forward + cross entropy + backward + gradient all-reduce +
Adam, dropout on) on ~2^20 synthetic MOSEI-shaped utterances IN TOTAL (hidden_all = 768+640+35 = 1443, one speaker id,
dialogue lengths 1+Geometric(1/7) clipped to 40, 6 classes), whole dialogues sharded over the N GPUs, no data-path collective:
BASELINE.json configs[4] as written, i.e. STRONG scaling (the default).  With N > 1 the same run also measures the
weak-scaling point (2^20 utterances PER GPU) and reports it under "weak_scaling"; ``--scaling weak`` makes that the headline.
One "step" = one pass over a GPU's utterances as ONE batch.

``value``  = utterances / second with inputs resident in HBM, the step replayed as ONE CUDA graph (train_step.CogmenTrainStep:
             K1 + forward + backward + NCCL all-reduces + Adam captured once; ``--mode eager`` launches kernel by kernel).
``kernels`` / ``roofline`` = per-kernel CUDA-event times of the same steps run eagerly (events cannot bracket kernels inside
             a graph replay), K steps, inputs resident; ``eager`` holds that loop's own step time.
``e2e``    = the same step fed from pinned HOST buffers (H2D of the inputs and D2H of the loss inside the timed region).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "COGMEN fwd+bwd utterances/sec"
UNIT = "utterances/s"
HIDDEN = 1443
N_CLASSES = 6
WORKLOAD = "cogmen-train-step mosei-emo-sbert-fbank-6 shape (hidden_all=1443, 1 speaker id, window 5/5), ~2^20 utterances per step in total, whole dialogues sharded over the GPUs"


def measured_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full` capture of
    this workload: profiles/traffic.json {kernel label: {"bytes": ..., "utterances": ...}}."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return {}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled WHILE the timed region runs, through NVML in this process (nvidia_ml_py).

    An `nvidia-smi -lms 100` child was measured to perturb the run it observes: single steps of the 16 ms loop took
    100-290 ms whenever a poll landed in them (gpurun_out/bench_c4_1.json: step_ms).  Two NVML calls per 50 ms do not."""

    def __init__(self, index, period_s=0.05):
        super().__init__(daemon=True)
        self.index, self.period_s, self.samples, self.stop_flag, self.mark = index, period_s, [], False, 0
        self.sm_max = None
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except ValueError:
                    idx = self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                     ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                     ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
            while not self.stop_flag:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.samples.append((sm, [n for n, b in names if bits & b]))
                time.sleep(self.period_s)
        except Exception as e:          # no NVML: report that, never fail the bench
            self.err = repr(e)

    def finish(self):
        self.stop_flag = True
        self.join(timeout=1.0)
        sm, reasons = [], set()
        for clk, rs in self.samples[self.mark:]:
            sm.append(clk)
            reasons.update(rs)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max, "reasons": sorted(reasons),
               "samples": len(sm), "how": "NVML (nvidia_ml_py) polled every %d ms during the timed region" % int(self.period_s * 1e3)}
        if self.err:
            out["error"] = self.err
        return out


# --------------------------------------------------------------------------------------------- reference arm
def cpu_reference_rate(budget_s, steps=None, warmup=1, batch_dialogues=32, skip_dead_encoder=False, seed=0):
    """Times the reference's CPU COGMEN train step (oracle/ref_port.py, "port") on MOSEI-shaped batches of 32
    dialogues (the reference's batch size, cogmen.py:43-45).  Returns (utt/s, description, seconds per batch)."""
    from oracle import ref_port
    import importlib
    synth = importlib.import_module("erc_b200.synth")
    torch.set_num_threads(os.cpu_count() or 1)
    gen = torch.Generator().manual_seed(seed)
    model = ref_port.CogmenRefPort(HIDDEN, n_classes=N_CLASSES, skip_dead_encoder=skip_dead_encoder)
    model.train()
    optim = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-8)     # cogmen.py:50

    def batch():
        L = synth.mosei_lengths(batch_dialogues * 8, gen)[:batch_dialogues]
        return synth.padded_batch(L, HIDDEN, 2, N_CLASSES, gen, one_speaker=True)

    for _ in range(warmup):
        ref_port.train_step(model, optim, batch())
    utts, t_total, n = 0, 0.0, 0
    while True:
        b = batch()
        t0 = time.perf_counter()
        ref_port.train_step(model, optim, b)
        t_total += time.perf_counter() - t0
        utts += int(b["text_length"].sum())
        n += 1
        if (steps is not None and n >= steps) or (steps is None and (t_total >= budget_s or n >= 64)):
            break
    return utts / t_total, "%d batches x %d dialogues (%d utterances), MOSEI-shaped" % (n, batch_dialogues, utts), t_total / n


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import erc_b200  # noqa: F401  (synth only; no kernels run on this arm)
    cores = os.cpu_count() or 1
    # each "step" = a bounded sample of the workload: `bps` batches of 32 dialogues; sized so the run ends in minutes
    probe_rate, _, t_batch = cpu_reference_rate(0.0, steps=1, warmup=1)
    total_batches = max(1, int(150.0 / max(t_batch, 1e-3)))
    bps = max(1, min(16, total_batches // max(args.steps + args.warmup, 1)))
    from oracle import ref_port
    import importlib
    synth = importlib.import_module("erc_b200.synth")
    gen = torch.Generator().manual_seed(0)
    model = ref_port.CogmenRefPort(HIDDEN, n_classes=N_CLASSES)
    model.train()
    optim = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-8)

    def one_step():
        u = 0
        for _ in range(bps):
            L = synth.mosei_lengths(32 * 8, gen)[:32]
            b = synth.padded_batch(L, HIDDEN, 2, N_CLASSES, gen, one_speaker=True)
            ref_port.train_step(model, optim, b)
            u += int(L.sum())
        return u

    for _ in range(args.warmup):
        one_step()
    t0 = time.perf_counter()
    utts = sum(one_step() for _ in range(args.steps))
    dt = time.perf_counter() - t0
    value = utts / dt
    sample = "%d steps x %d batches x 32 dialogues (%d utterances) of the MOSEI-shaped workload; throughput is per-batch, linear in dialogues" % (
        args.steps, bps, utts)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "reference_batch": "32 dialogues/batch (cogmen.py:43-45)", "device": "cpu"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# --------------------------------------------------------------------------------------------- our arm
def kernel_label(name, args):
    try:
        if name == "ercg_gemm_nn":
            return "gemm_nn[K=%d,N=%d]" % (args[10], args[9])
        if name == "ercg_gemm_nn_tc":
            return "gemm_nn_tc[K=%d,N=%d]" % (args[9], args[8])
        if name == "ercg_gemm_tn_tc":
            return "gemm_tn_tc[K1=%d,N1=%d]" % (args[7], args[8])
        if name == "ercg_gemm_nn_tc_bf16a":
            return "gemm_nn_tc_bf16a[K=%d,N=%d]" % (args[9], args[8])
        if name == "ercg_gemm_tn_tc_bf16a":
            return "gemm_tn_tc_bf16a[K1=%d,N1=%d]" % (args[7], args[8])
        if name == "ercg_gemm_tn":
            return "gemm_tn[K1=%d,N1=%d]" % (args[8], args[9])
    except Exception:
        pass
    name = name.replace("attn_window_", "attn_")        # CTA-tiled window-graph variants of the same three kernels
    name = name.replace("gather_window_", "gather_")
    return name[5:] if name.startswith("ercg_") else name


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and allocate its pinned host buffers) on the NUMA node its GPU hangs off: with 8 ranks feeding 8 GPUs
    from one host, cross-socket pinned buffers halve the per-rank H2D rate.  Best effort; returns a description."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis else local_rank
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return "numa_node=-1 (single node or not reported)"
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return "node %d, %d cpus" % (node, len(allowed))
        return "node %d has no allowed cpus" % node
    except Exception as e:
        return "unavailable (%s)" % type(e).__name__


def run_ours(args):
    import gc
    import torch.distributed as dist
    import erc_b200  # noqa: F401
    from erc_b200 import _lib, synth
    from erc_b200.graph import graph_sizes
    from erc_b200.track_mm.cogmen import COGMENModule
    from erc_b200.dist import shard_dialogues
    from erc_b200.train_step import CogmenTrainStep
    from erc_b200.loader import DeviceFeeder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a GPU: libercgraph has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else "not bound (single rank)"
    ctl = None
    if args.watchdog_s > 0:
        import faulthandler
        faulthandler.dump_traceback_later(args.watchdog_s, exit=True)      # a hung collective must end the run with a traceback
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")      # NCCL collectives are captured into the step's CUDA graph
        dist.init_process_group("nccl", device_id=dev)
        ctl = dist.new_group(backend="gloo")              # control plane (barriers, max over ranks of the timings): host side
    _lib.lib()                                            # fail loudly now if the .so is missing
    ld = (HIDDEN + 3) // 4 * 4                            # 1444: rows 16-byte aligned in HBM

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=ctl)
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=ctl)
        return float(t.item())

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()                                  # before any warm-up: starting it later stalls rank 0's launch thread

    def step_outputs(loss, model, ts):
        """What a caller of the timed step receives after it (host copies): the loss (with world > 1 the global mean, not
        this rank's share), the parameters Adam updated (the dead encoder is never updated and is left out) and the
        floating-point buffers the step updates (BatchNorm running statistics)."""
        if world > 1:
            loss = ts.global_loss()
        out = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
        live = {id(p) for p in ts.opt.live}
        for name, p in model.named_parameters():
            if id(p) in live:
                out["param." + name] = p.detach().float().cpu().numpy()
        for name, b in model.named_buffers():
            if b.is_floating_point():
                out["buffer." + name] = b.detach().float().cpu().numpy()
        return out

    def measure(scaling, steps, with_kernels, with_e2e, in_dtype="f32", keep_outputs=False):
        """One workload (strong: args.total_utts in total; weak: per GPU) -> dict of measurements (same on every rank).
        in_dtype "bf16": the bf16 input-feature mode (features stored in bf16, row pitch 1448 elements; everything else fp32).
        keep_outputs: out["outputs"] = step_outputs() of the last timed step of the headline loop."""
        weak = scaling == "weak"
        lengths_all = synth.config5_lengths(args.total_utts * (world if weak else 1), seed=0)
        total_utts = int(lengths_all.sum())
        mine = shard_dialogues(lengths_all, world)[rank]
        lengths = lengths_all[mine].contiguous()
        N = int(lengths.sum())
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        x_store = torch.empty((N, ld), dtype=torch.float32, device=dev)
        x_store.normal_(generator=gen)
        if in_dtype == "bf16":
            x = synth.to_bf16_rows(x_store[:, :HIDDEN])          # [N, 1443] view of a [N, 1448] bf16 buffer
            x_store = x._base if x._base is not None else x
        else:
            x = x_store[:, :HIDDEN]
        spk = torch.zeros(N, dtype=torch.int64, device=dev)   # MOSEI: a single speaker id (mosei_feature.py:211)
        labels = torch.randint(0, N_CLASSES, (N,), device=dev, generator=gen)
        sizes = graph_sizes(lengths, 5, 5)
        torch.manual_seed(0)
        model = COGMENModule(HIDDEN, 100, 17, 2, N_CLASSES).to(dev)
        model.train()
        # cogmen.py:50: Adam(lr 1e-4, weight_decay 1e-8) -- here ercg_adam_step on the flat buffer of the live parameters
        data_group = dist.new_group(backend="nccl") if world > 1 else None     # the step's own communicator (captured in its graph)
        ts = CogmenTrainStep(model, lengths, speakers_present=(0,), lr=1e-4, weight_decay=1e-8, world=world,
                             global_utterances=total_utts, bn_sync=args.bn_sync, overlap=not args.no_overlap, group=data_group,
                             transport=args.transport)
        out = {"scaling": scaling, "utterances_per_step": total_utts, "utterances_rank0": N, "edges_rank0": sizes[1],
               "dialogues": int(lengths_all.numel()), "transport": ts.transport}

        # ---- eager steps (kernel by kernel): warm-up, then K steps with every C-ABI call bracketed by CUDA events
        loss = ts.step(x, spk, labels)
        gc.collect()
        gc.freeze()
        gc.disable()
        for _ in range(max(args.warmup, 3)):
            loss = ts.step(x, spk, labels)
        barrier()
        if args.profile_step:
            torch.cuda.profiler.start()
            ts.step(x, spk, labels)
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
            return {"profile_step": True, "utterances_per_step": total_utts}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        def time_eager():
            with _lib.KernelTimer(labeler=kernel_label):    # one more warm step WITH the event bracketing active (event pool)
                ts.step(x, spk, labels)
            barrier()
            launches0 = _lib.launch_count()
            timer = _lib.KernelTimer(labeler=kernel_label)
            with timer:
                barrier()
                e0.record()
                for _ in range(steps):
                    last = ts.step(x, spk, labels)
                e1.record()
                barrier()
            eager_ms = max_over_ranks(e0.elapsed_time(e1)) / steps
            out["eager"] = {"ms_per_step": eager_ms, "value": total_utts / (eager_ms / 1e3),
                            "launches_per_step": (_lib.launch_count() - launches0) / steps}
            out["ksum"] = timer.summary()
            out["step_kernel_ms"] = sum(t for _, t in out["ksum"].values()) / steps
            if keep_outputs:
                out["outputs"] = step_outputs(last, model, ts)
            return last

        if with_kernels or args.mode == "eager":
            loss = time_eager()

        # ---- the step as ONE CUDA graph
        graph_err = None
        if args.mode == "graph":
            try:
                launches0 = _lib.launch_count()
                ts.capture(x, spk, labels, warmup=2)
                barrier()
                for _ in range(max(args.warmup, 3)):
                    ts.replay()
                barrier()
                if sampler and scaling == args.scaling:
                    t_wait = time.perf_counter()
                    while not sampler.samples and time.perf_counter() - t_wait < 2.0:
                        time.sleep(0.01)
                    sampler.mark = len(sampler.samples)      # only samples taken from here on are reported
                mem_before = torch.cuda.memory_stats(dev)
                lc0 = _lib.launch_count()
                barrier()
                e0.record()
                marks = []
                for _ in range(steps):
                    loss = ts.replay()
                    marks.append(torch.cuda.Event(enable_timing=True))
                    marks[-1].record()
                e1.record()
                barrier()
                mem_after = torch.cuda.memory_stats(dev)
                ms = max_over_ranks(e0.elapsed_time(e1))
                out["graph"] = {"ms_per_step": ms / steps, "value": total_utts * steps / (ms / 1e3),
                                "step_ms": [round(a.elapsed_time(b), 3) for a, b in zip([e0] + marks[:-1], marks)],
                                "host_launches_in_timed_region": _lib.launch_count() - lc0,
                                "cuda_mallocs_in_timed_region": int(mem_after.get("num_device_alloc", 0) - mem_before.get("num_device_alloc", 0))}
                if keep_outputs:
                    out["outputs"] = step_outputs(loss, model, ts)
            except Exception as e:                             # report, and fall back to the eager numbers
                graph_err = "%s: %s" % (type(e).__name__, str(e)[:300])
                out["graph_error"] = graph_err
        if "graph" not in out and "eager" not in out:
            loss = time_eager()
        out["loss"] = float(loss.item()) if loss is not None else None
        if world > 1:
            out["loss_global"] = float(ts.global_loss().item())
            # Where does the time over (1-GPU time / N) go?  Every rank replays ITS shard as a stand-alone step (no collective,
            # no waiting for anybody) while all the others do the same, i.e. in the same power / thermal state as the
            # distributed run; the distributed step cannot be faster than the slowest of these.
            try:
                torch.manual_seed(0)
                solo_model = COGMENModule(HIDDEN, 100, 17, 2, N_CLASSES).to(dev)
                solo_model.train()
                solo = CogmenTrainStep(solo_model, lengths, speakers_present=(0,), lr=1e-4, weight_decay=1e-8, world=1)
                solo.capture(x, spk, labels, warmup=2)
                for _ in range(3):
                    solo.replay()
                barrier()
                e0.record()
                for _ in range(steps):
                    solo.replay()
                e1.record()
                torch.cuda.synchronize()
                mine_ms = e0.elapsed_time(e1) / steps
                all_ms = [None] * world
                dist.all_gather_object(all_ms, mine_ms, group=ctl)
                out["solo_ms_per_rank"] = [round(v, 4) for v in all_ms]
                del solo, solo_model
            except Exception as e:
                out["solo_error"] = "%s: %s" % (type(e).__name__, str(e)[:200])

        # ---- e2e: the step through the public API with HOST buffers; every step's inputs (features, speakers, labels) are
        # copied from pinned host memory inside the timed region (DeviceFeeder: double-buffered, on copy streams, so the H2D of
        # step i+1 overlaps the kernels of step i) and the loss is read back.  Eager steps: PCIe is the bound, not launches.
        if with_e2e:
            e2e_steps = max(1, args.e2e_steps)
            hx = torch.empty(tuple(x_store.shape), dtype=x_store.dtype, pin_memory=True)
            hx.copy_(x_store)
            host = {"x": hx, "spk": torch.zeros(N, dtype=torch.int64).pin_memory(), "label": labels.cpu().pin_memory()}
            feeder = DeviceFeeder(dev, depth=2, copy_streams=args.copy_streams)

            def e2e_run(n):
                feeder.submit(host)
                for i in range(n):
                    if i + 1 < n:
                        feeder.submit(host)                      # prefetch the next step's inputs
                    d = feeder.get()
                    loss_i = ts.step(d["x"][:, :HIDDEN], d["spk"], d["label"])
                    feeder.release()
                    float(loss_i.item())                         # D2H of the step's result

            # ceiling of the host->device path on this box: every rank copies its pinned feature buffer, nothing else running
            probe = torch.empty_like(x_store)
            barrier()
            e0.record()
            for _ in range(3):
                probe.copy_(hx, non_blocking=True)
            e1.record()
            barrier()
            h2d_probe_ms = max_over_ranks(e0.elapsed_time(e1)) / 3
            del probe
            e2e_run(2)
            barrier()
            b0 = feeder.h2d_bytes
            e0.record()
            e2e_run(e2e_steps)
            e1.record()
            barrier()
            e2e_ms = max_over_ranks(e0.elapsed_time(e1))
            h2d = (feeder.h2d_bytes - b0) // e2e_steps
            if world > 1:
                b = torch.tensor([h2d], dtype=torch.float64)
                dist.all_reduce(b, group=ctl)
                h2d = int(b.item())
            out["e2e"] = {"value": total_utts * e2e_steps / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                          "d2h_bytes_per_step": 4 * world, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                          "h2d_copy_only_ms": h2d_probe_ms,
                          "h2d_copy_only_gbs_all_ranks": round(world * hx.numel() * hx.element_size() / (h2d_probe_ms * 1e-3) / 1e9, 1),
                          "h2d_share_of_step": round(h2d_probe_ms / (e2e_ms / e2e_steps), 3),
                          "how": "pinned host buffers -> DeviceFeeder (double-buffered, %d copy streams) -> eager step -> loss.item(); "
                                 "all copies inside the timed region; host threads bound to the GPU's NUMA node: %s" % (args.copy_streams, numa)}
            del feeder, host, hx
        ts.check()                                             # K1's input-error flags of the last step, peer-collective timeouts
        if ts.comms:
            barrier()                                          # nobody may still be reading a region that is about to be freed
            for c in ts.comms:
                c.close()
        gc.enable()
        gc.unfreeze()
        out["x_bytes"] = x_store.numel() * x_store.element_size()
        out["N"], out["E"], out["n_dialogues_rank0"] = N, sizes[1], int(lengths.numel())
        del ts, model, x_store, x, spk, labels
        gc.collect()
        torch.cuda.empty_cache()
        return out

    head = measure(args.scaling, args.steps, with_kernels=True, with_e2e=True, keep_outputs=bool(args.dump_outputs))
    if args.profile_step:
        if rank == 0:
            emit(head)
        return
    outputs = head.pop("outputs", None)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    clocks = sampler.finish() if sampler else None
    other = None
    if world > 1 and not args.no_second_scaling:
        other = measure("weak" if args.scaling == "strong" else "strong", max(args.steps // 2, 3), with_kernels=False, with_e2e=False)
    bf16 = None
    if world == 1 and not args.no_bf16_mode:
        bf16 = measure(args.scaling, max(args.steps // 2, 3), with_kernels=True, with_e2e=True, in_dtype="bf16")

    if rank == 0:
        peak, peak_src = peaks()
        N, E = head["N"], head["E"]
        mode = "graph" if "graph" in head else "eager"
        best = head[mode]
        ksum = head["ksum"]
        per = {k: (c, tot / c) for k, (c, tot) in ksum.items()}          # kernel label -> (calls, avg ms)
        H, P = 100, 2          # row width; relation ids that occur (1 speaker id -> 2 of 8): Y / dY hold P + 1 slots
        nd = head["n_dialogues_rank0"]

        def alg_bytes(label):
            """Algorithmic (unique) HBM bytes of ONE launch on this rank (SURVEY.md 8d; weights ignored)."""
            if label.startswith("gemm_"):
                a, b = (int(v.split("=")[1]) for v in label[label.index("[") + 1:-1].split(","))
                if "bf16a" in label:
                    return N * (2 * a + 4 * b)            # the wide / streamed operand is stored in bf16
                return 4 * N * (a + b)
            return {
                "gather_fwd": 4 * H * P * N + 4 * H * N + 4 * H * N + 4 * (N + 1) + 9 * E,
                "gather_bwd": 4 * H * N + 4 * H * (P + 1) * N + 4 * (N + 1) + 13 * E,
                "attn_fwd": 5 * 4 * H * N + 4 * (N + 1) + 8 * E,
                "attn_bwd_dst": 5 * 4 * H * N + 4 * (N + 1) + 12 * E,
                "attn_bwd_src": 4 * 4 * H * N + 4 * (N + 1) + 16 * E,
                "attn_bwd": 8 * 4 * H * N + 8 * (N + 1) + 12 * E,
                "graphify_csr": 8 * nd + 8 * N + 8 * (N + 1) + 12 * N + E * (4 + 1 + 4 + 1 + 4 + 4 + 24),
                "bn_stats": 4 * H * N, "bn_act_fwd": 8 * H * N, "bn_act_bwd_reduce": 8 * H * N, "bn_act_bwd_apply": 12 * H * N,
                "mask_pos": 12 * H * N, "colsum": None, "ce_fwd": (4 * N_CLASSES * 2 + 8) * N,
                "cls_tail_bwd": (8 * H + 4 * N_CLASSES) * N,
            }.get(label)

        kernels = {}
        tr_all = measured_traffic()
        for label, (calls, avg_ms) in sorted(per.items(), key=lambda kv: -kv[1][0] * kv[1][1]):
            ab = alg_bytes(label)
            ent = {"calls_per_step": calls / args.steps, "avg_ms": round(avg_ms, 4)}
            if ab:
                gbs = ab / (avg_ms * 1e-3) / 1e9
                ent.update({"algorithmic_bytes": ab, "achieved_gbs": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peak, 4)})
            if label in tr_all and tr_all[label].get("utterances"):   # DRAM bytes per launch from the committed ncu capture
                ent["traffic"] = int(tr_all[label]["bytes"] * (N / float(tr_all[label]["utterances"])))
            kernels[label] = ent
        dom_label = max(ksum.items(), key=lambda kv: kv[1][1])[0]
        dom_calls, dom_ms = per[dom_label]
        dom_bytes = alg_bytes(dom_label) or 0
        tr = tr_all.get(dom_label)
        traffic = int(tr["bytes"] * (N / float(tr["utterances"]))) if tr and tr.get("utterances") else None
        roof = {"bound": "hbm", "kernel": dom_label, "achieved": dom_bytes / (dom_ms * 1e-3) / 1e9, "peak": peak,
                "unit": "GB/s", "frac": dom_bytes / (dom_ms * 1e-3) / 1e9 / peak, "traffic": traffic,
                "traffic_source": (tr or {}).get("source"), "peak_source": peak_src,
                "avg_launch_ms": dom_ms, "launches_timed": dom_calls, "algorithmic_bytes_per_launch": dom_bytes,
                "timed_in": "the eager loop (CUDA events around each C-ABI call on the launching stream); the headline loop replays the same kernels as one CUDA graph"}
        graph_kernels = {k: kernels[k] for k in ("gather_fwd", "gather_bwd", "attn_fwd", "attn_bwd_dst", "attn_bwd_src", "attn_bwd",
                                                 "graphify_csr") if k in kernels}
        launches_per_step = head["eager"]["launches_per_step"]
        line = {"metric": METRIC, "value": best["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": best["ms_per_step"], "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "utterances_per_step": head["utterances_per_step"], "dialogues": head["dialogues"],
                           "edges_per_step_rank0": E,
                           "parallelism": "dp%d (whole dialogues per GPU, %s scaling: %d utterances %s)" % (
                               world, args.scaling, args.total_utts, "per GPU" if args.scaling == "weak" else "in total"),
                           "l2": "inputs (%.2f GB/step/GPU) are larger than the 126 MB L2" % (head["x_bytes"] / 1e9),
                           "step": "one CUDA-graph replay per step" if mode == "graph" else "eager launches",
                           "bn_statistics": "global (all-reduced)" if (world > 1 and args.bn_sync == "global") else "per rank",
                           "collectives": head.get("transport", "none") if world > 1 else "none (one GPU)",
                           "dropout": "on (train mode)", "optimizer": "Adam inside the step (ercg_adam_step on the flat parameter buffer)",
                           "dead_encoder": "not executed (cogmen.py:146-147 discards its output)"},
                "roofline": roof, "graph_kernels": graph_kernels, "kernels": kernels,
                "eager": head.get("eager"), "graph": head.get("graph"),
                "kernel_time_share_of_eager_step": round(head["step_kernel_ms"] / head["eager"]["ms_per_step"], 4),
                "kernel_time_share_of_step": round(head["step_kernel_ms"] / best["ms_per_step"], 4),
                "e2e": head["e2e"],
                "gpu_launches": int(round(launches_per_step * args.steps)),
                "gpu_launches_how": "%d libercgraph kernel launches per step (counted in the eager loop) x %d steps%s" % (
                    int(round(launches_per_step)), args.steps, "; in the headline loop they are nodes of the replayed CUDA graph" if mode == "graph" else ""),
                "clocks": clocks, "loss": head["loss"]}
        if "graph_error" in head:
            line["graph_error"] = head["graph_error"]
        if "loss_global" in head:
            line["loss_global"] = head["loss_global"]
        if "solo_ms_per_rank" in head:
            sm = head["solo_ms_per_rank"]
            line["scaling_breakdown"] = {
                "solo_ms_per_rank": sm,
                "what": "each rank's own shard replayed as a stand-alone step (no collectives, no waiting), all ranks at once",
                "slowest_rank_solo_ms": max(sm), "fastest_rank_solo_ms": min(sm),
                "collectives_and_skew_ms": round(best["ms_per_step"] - max(sm), 4),
                "collectives_per_step": ("BN statistics (2H+1 doubles, forward) + their backward sums (2H floats) + flat gradients "
                                         "in two overlapped buckets" if args.bn_sync == "global"
                                         else "flat gradients in two overlapped buckets") +
                                        " (%s, nodes of the step's CUDA graph)" % head.get("transport", "torch.distributed")}
        if other is not None:
            ob = other.get("graph") or other.get("eager")
            line[other["scaling"] + "_scaling"] = {"value": ob["value"], "ms_per_step": ob["ms_per_step"],
                                                   "utterances_per_step": other["utterances_per_step"],
                                                   "mode": "graph" if "graph" in other else "eager", "unit": UNIT,
                                                   "solo_ms_per_rank": other.get("solo_ms_per_rank")}
        if bf16 is not None:
            bb = bf16.get("graph") or bf16.get("eager")
            bper = {k: (c, tot / c) for k, (c, tot) in bf16["ksum"].items()}
            bk = {}
            for label in ("gemm_nn_tc_bf16a[K=1443,N=100]", "gemm_tn_tc_bf16a[K1=1443,N1=100]"):
                if label in bper:
                    ab, ms_ = alg_bytes(label), bper[label][1]
                    bk[label] = {"avg_ms": round(ms_, 4), "algorithmic_bytes": ab, "achieved_gbs": round(ab / (ms_ * 1e-3) / 1e9, 1),
                                 "frac_of_hbm_peak": round(ab / (ms_ * 1e-3) / 1e9 / peak, 4)}
            line["bf16_input_mode"] = {
                "what": "utterance features stored in bf16 (row pitch 1448 elements); weights, activations, gradients, accumulation fp32",
                "value": bb["value"], "ms_per_step": bb["ms_per_step"], "unit": UNIT, "mode": "graph" if "graph" in bf16 else "eager",
                "e2e": bf16.get("e2e"), "kernels": bk, "loss": bf16["loss"],
                "tolerance": "equals the fp32 path run on the bf16-rounded features to the fp32 parity bars; vs the original features: "
                             "logits within 1e-2 relative (tests/test_gpu_bf16_mode.py)"}
        if world == 1 and not args.no_cpu_baseline:
            v, sample, _ = cpu_reference_rate(args.cpu_budget_s)
            v2, sample2, _ = cpu_reference_rate(args.cpu_budget_s / 2, skip_dead_encoder=True)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port", "sample": sample,
                                    "value_dead_encoder_skipped": v2}
        emit(line)
    if world > 1:
        # no NCCL teardown: destroying communicators whose kernels were captured in CUDA graphs was seen to hang
        # (gpurun_out/r02c_probe*.log); everything is synchronised, the line is out, leave through the gloo barrier
        torch.cuda.synchronize()
        dist.barrier(group=ctl)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """Writes each array as <directory>/<name>.npy, so that two builds run with the same arguments (hence the same inputs)
    can be compared output by output."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(directory, name + ".npy"), a)


def run_library_yardstick(args):
    """NOT the product path: times what a library gives for the two projection GEMMs of the workload on this box --
    cuBLAS through torch.matmul in exact fp32 (allow_tf32 off), in TF32 (10-bit mantissa: 1e-3 accuracy, outside the 1e-5 bar)
    and in bf16 -- next to libercgraph's split-precision tcgen05 kernels (VERDICT r1 item 8).  One JSON line."""
    import erc_b200  # noqa: F401
    from erc_b200 import ops, synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    M, K, N = args.total_utts, HIDDEN, 100
    ld = (K + 3) // 4 * 4
    xs = torch.randn((M, ld), device=dev)
    x = xs[:, :K]
    W = torch.randn((N, K), device=dev) / K ** 0.5
    dF = torch.randn((M, N), device=dev)
    xb = synth.to_bf16_rows(x)
    Wt = W.t().contiguous()

    def timeit(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ref_nn = (x[:4096].double() @ Wt.double())
    ref_tn = None
    out = {"shape": {"M": M, "K": K, "N": N}, "unit": "ms per launch", "nn": {}, "tn": {}}

    def err(y):
        return float((y[:4096].double() - ref_nn).abs().max() / ref_nn.abs().max())

    torch.backends.cuda.matmul.allow_tf32 = False
    out["nn"]["cublas_fp32"] = {"ms": timeit(lambda: torch.matmul(x, Wt)), "rel_err": err(torch.matmul(x, Wt))}
    out["tn"]["cublas_fp32"] = {"ms": timeit(lambda: torch.matmul(x.t(), dF))}
    torch.backends.cuda.matmul.allow_tf32 = True
    out["nn"]["cublas_tf32"] = {"ms": timeit(lambda: torch.matmul(x, Wt)), "rel_err": err(torch.matmul(x, Wt))}
    out["tn"]["cublas_tf32"] = {"ms": timeit(lambda: torch.matmul(x.t(), dF))}
    torch.backends.cuda.matmul.allow_tf32 = False
    Wb, dFb = Wt.to(torch.bfloat16), dF.to(torch.bfloat16)
    out["nn"]["cublas_bf16"] = {"ms": timeit(lambda: torch.matmul(xb, Wb)), "rel_err": err(torch.matmul(xb, Wb).float())}
    out["tn"]["cublas_bf16"] = {"ms": timeit(lambda: torch.matmul(xb.t(), dFb))}
    out["nn"]["libercgraph_fp32_split"] = {"ms": timeit(lambda: ops.gemm_nn(x, Wt)), "rel_err": err(ops.gemm_nn(x, Wt))}
    out["tn"]["libercgraph_fp32_split"] = {"ms": timeit(lambda: ops.gemm_tn(x, dF))}
    Wp = W.clone().requires_grad_()

    def bf_nn():
        return ops.linear(xb, Wp)

    y = bf_nn()
    out["nn"]["libercgraph_bf16_input"] = {"ms": timeit(bf_nn), "rel_err_vs_rounded_features": float(
        (y[:4096].double() - xb[:4096].double() @ Wt.double()).abs().max() / ref_nn.abs().max())}

    def bf_tn():
        (g,) = torch.autograd.grad(ops.linear(xb, Wp), Wp, dF)
        return g

    t_both = timeit(bf_tn)
    out["tn"]["libercgraph_bf16_input"] = {"ms": t_both - out["nn"]["libercgraph_bf16_input"]["ms"], "how": "forward+wgrad minus forward"}
    a = ops.gemm_tn(x, dF)[:64].double().cpu()
    r = (x[:, :64].double().t() @ dF.double()).cpu()
    out["tn"]["libercgraph_fp32_split"]["rel_err"] = float((a - r).abs().max() / r.abs().max())
    out["note"] = "cuBLAS fp32 = SIMT FFMA path; TF32 and bf16 do not meet the 1e-5 parity bar of BASELINE.json (rel_err column)"
    emit({"library_yardstick": out})


_REAL_STDOUT = None


def _quiet_stdout():
    """Libraries (NCCL prints its version banner to stdout) must not pollute the ONE JSON line: route fd 1 to stderr for
    the whole run and keep a private duplicate of the real stdout for the result."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--total-utts", type=int, default=1 << 20)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-budget-s", type=float, default=16.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--copy-streams", type=int, default=2, help="H2D copy streams of the e2e feeder (2: +3 %% over one)")
    ap.add_argument("--profile-step", action="store_true",
                    help="warm up, then run one step between cudaProfilerStart/Stop and exit (for ncu --profile-from-start off)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="strong (default, BASELINE configs[4]): --total-utts in total, sharded over the GPUs; weak: per GPU")
    ap.add_argument("--mode", default="graph", choices=["graph", "eager"], help="headline loop: CUDA-graph replay or eager launches")
    ap.add_argument("--bn-sync", default="global", choices=["global", "local"],
                    help="BatchNorm statistics across ranks: global = all-reduced (N-GPU == 1-GPU result), local = per rank (the reference's DDP)")
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N > 1: the step's all-reduces through libercgraph's peer-memory kernel (p2p), NCCL, or p2p when available")
    ap.add_argument("--no-overlap", action="store_true", help="one gradient all-reduce after backward instead of the two overlapped buckets")
    ap.add_argument("--watchdog-s", type=int, default=0, help="dump all Python stacks and exit if the run takes longer than this")
    ap.add_argument("--library-yardstick", action="store_true",
                    help="time cuBLAS (fp32 / TF32 / bf16) on the projection GEMM shapes next to libercgraph's kernels and exit")
    ap.add_argument("--no-bf16-mode", action="store_true", help="N = 1: skip the extra bf16 input-feature-mode measurement")
    ap.add_argument("--no-second-scaling", action="store_true", help="N > 1: skip the extra weak- (or strong-) scaling measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (loss.npy; param.<name>.npy: the parameters "
                         "Adam updated; buffer.<name>.npy: BatchNorm running statistics; float32) to DIR")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.library_yardstick or args.profile_step):
        ap.error("--dump-outputs needs the timed train step of our arm (not --impl reference, --library-yardstick "
                 "or --profile-step)")
    _quiet_stdout()
    if args.library_yardstick:
        run_library_yardstick(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
