"""``train_mm.py --module=<cogmen|dgcn|dgcnv2|mmgcn|dagerc> --dataset=... --modality=atv`` without lumo / accelerate
(SURVEY.md 8f-4; reference: train_mm.py:16-25 -> track_mm/<module>.main -> mmbase.main, mmbase.py:483-499).

What is kept from the reference
  * the command line: ``--key=value`` pairs, the same parameter names (module, dataset, modality, epoch, seed, device,
    n_classes, train.batch_size ...), the per-module defaults of the ``*Params`` classes (cogmen.py:36-52, dgcn.py:24-44,
    mmgcn.py:22-50, dagerc.py:25-66) and the data-set -> feature-size rules of ``MMBaseParams.iparams`` (mmbase.py:52-128);
  * the train / test steps (cogmen.py:179-195, dgcn.py:117-134, mmgcn.py:141-157, dagerc.py:217-237, mmbase.py:152-201):
    mean cross entropy (class-weighted for 6-way DialogueGCN, masked for DAG-ERC + clip_grad_norm_(5)), Adam / AdamW with the
    reference's learning rates, a test pass after every epoch (EvalCallback(test_per_epoch=1), mmbase.py:136) with accuracy,
    weighted / micro / macro F1, balanced accuracy and the confusion matrix (sklearn, mmbase.py:262-283), seed marking per
    epoch, ``best_model.ckpt`` / ``last_model.ckpt`` whose model keys are the reference modules' keys.
Checkpoints
  * ``--ckpt_layout=state_dict`` (default): each file is the model's plain ``state_dict``, written once per improvement /
    after the last epoch.  The reference's files are NOT this: mmbase.py:325-333 saves lumo's ``Trainer.state_dict()``.
  * ``--ckpt_layout=reference``: that layout (lumo/trainer/trainer.py:623-632), ``{'models': {'model': sd}, 'optims':
    {'optim': <torch.optim Adam / AdamW state_dict>}, 'others': {'train_mm': {epoch, best, history, run parameters, every
    rank's CPU generator state}}, 'thtensor': {}, 'nptensor': {}}``; ``last_model.ckpt`` is rewritten after every epoch.
  * ``--resume=<ckpt>`` continues a run from such a file (refused when a run-defining parameter differs);
    ``--load=<ckpt>`` starts from the weights alone, of either layout (a reference checkpoint included).
What is different
  * the model runs in libercgraph kernels; the batch is collated onto the device in the packed layout (collate.DeviceCollate);
    the optimizer is the flat-buffer Adam kernel (optim.FlatAdam);
  * ``mmdatasets`` (the reference's feature pickles) is not part of this repo: ``--data=<file>`` loads a pickle
    ``{"train": [sample, ...], "test": [...]}`` of samples in the reference's format (mmbase.py:374-384); without it a seeded
    synthetic data set of the data set's SHAPE is generated (``--train_dialogues``, ``--test_dialogues``).

Several GPUs (the reference's ``accelerate launch --num_processes N``, lumo/trainer/trainer.py:62-64,315-327)::

    python -m torch.distributed.run --standalone --nproc_per_node N train_mm.py --module=dgcn ...

One process per GPU (WORLD_SIZE / RANK / LOCAL_RANK; rank r runs on cuda:LOCAL_RANK, ``--device`` is ignored), with DDP's
semantics: ``--train.batch_size`` is the per-GPU batch, optimizer step s trains rank r on batch s*N + r of the epoch's list
(``deal_batches``), every rank takes the mean loss of its own batch and the update uses the average of the N gradients
(one all-reduce of the flat gradient buffer: libercgraph's peer-memory kernel, else NCCL), BatchNorm running statistics are
rank 0's.  The test pass is split over the ranks batch by batch and gathered back into the one-GPU order; only rank 0 logs
and writes checkpoints.  Without WORLD_SIZE (or with 1) nothing of this runs.
"""
import json
import math
import os
import pickle
import sys
import time

import numpy as np
import torch

MODULES = ("cogmen", "dgcn", "dgcnv2", "mmgcn", "dagerc")
CKPT_LAYOUTS = ("state_dict", "reference")
# the parameters a resumed run must share with the run that wrote the checkpoint (besides the number of processes)
RUN_KEYS = ("module", "dataset", "modality", "seed", "batch_size", "n_classes", "n_speakers", "optim")


# ------------------------------------------------------------------------------------------------ parameters
def parse_args(argv):
    """fire / lumo style: ``--key=value``, ``--key value``, ``--flag`` (= True); dotted keys kept as given."""
    out, i = {}, 0
    while i < len(argv):
        a = argv[i]
        if not a.startswith("--"):
            raise SystemExit("unexpected argument %r (expected --key=value)" % a)
        if "=" in a:
            k, v = a[2:].split("=", 1)
        elif i + 1 < len(argv) and not argv[i + 1].startswith("--"):
            k, v = a[2:], argv[i + 1]
            i += 1
        else:
            k, v = a[2:], "True"
        out[k.replace("-", "_")] = _coerce(v)
        i += 1
    return out


def _coerce(v):
    if v in ("True", "true"):
        return True
    if v in ("False", "false"):
        return False
    for cast in (int, float):
        try:
            return cast(v)
        except ValueError:
            pass
    return v


def resolve_params(args):
    """Defaults of <Module>Params + MMBaseParams.iparams (mmbase.py:52-128)."""
    module = args.get("module")
    if module not in MODULES:
        raise SystemExit("--module= one of %s" % (MODULES,))
    p = dict(seed=1, dataset="iemocap-cogmen-6", modality="atv", n_speakers=2, device=0, reimplement=False, data=None,
             train_dialogues=120, test_dialogues=31, save_dir=None, log_every=0, max_len=None, ckpt_layout="state_dict",
             resume=None, load=None)
    per_module = {
        "cogmen": dict(epoch=55, batch_size=32, optim="Adam", lr=1e-4, weight_decay=1e-8, num_heads=17),          # cogmen.py:36-52
        "dgcn": dict(epoch=55, batch_size=32, optim="Adam", lr=3e-4, weight_decay=0.0, loss_weights=True),        # dgcn.py:24-44
        "dgcnv2": dict(epoch=55, batch_size=32, optim="Adam", lr=3e-4, weight_decay=0.0, loss_weights=True, base_model="LSTM"),   # dgcnv2.py:20-45
        "mmgcn": dict(epoch=60, batch_size=16, optim="Adam", lr=3e-4, weight_decay=3e-5),                          # mmgcn.py:22-40
        "dagerc": dict(epoch=30, batch_size=8, optim="AdamW", lr=1e-3, weight_decay=1e-2, gnn_layers=4, dropout=0.0),   # dagerc.py:25-41
    }[module]
    p.update(per_module)
    p["module"] = module
    for k, v in args.items():
        k = {"train.batch_size": "batch_size", "optim.lr": "lr", "optim.weight_decay": "weight_decay"}.get(k, k)
        p[k] = v
    if p["ckpt_layout"] not in CKPT_LAYOUTS:
        raise SystemExit("--ckpt_layout= one of %s" % (CKPT_LAYOUTS,))
    if p["resume"] and p["load"]:
        raise SystemExit("--resume and --load exclude each other (--resume also loads the weights)")
    ds = p["dataset"]
    if "n_classes" not in p:
        tail = ds.rsplit("-", 1)[-1]
        p["n_classes"] = int(tail) if tail.isdigit() else 6
    ht, ha, hv = 100, 100, 100                                                                    # mmbase.py:45-47
    if "iemocap" in ds and "cogmen" in ds:
        ha, ht, hv = 100, 100, 512
    elif "meld" in ds:
        p["n_speakers"] = 9
        if "mmgcn" in ds:
            ha, ht, hv = 300, 600, 342
    elif "mosei" in ds:
        ht, ha, hv = 300, 74, 35
    if "pad80" in ds:
        ha = 80
    elif "fbank" in ds:
        ha = 640
    elif "is10" in ds:
        ha = 1584
    if "sbert" in ds or "robert" in ds:
        ht = 768
    if "tsn" in ds:
        hv = hv + 2048 if "v+" in ds else 2048
    p.update(hidden_text=ht, hidden_audio=ha, hidden_visual=hv)
    p["hidden_all"] = sum({"t": ht, "a": ha, "v": hv}[m] for m in set(p["modality"]))
    if module == "dagerc" and p["reimplement"] and "iemocap" in ds:                               # dagerc.py:45-50
        p.update(dropout=0.2, epoch=55, batch_size=16, lr=5e-4)
    p["batch_first"] = module not in ("mmgcn", "dgcnv2")                                          # mmgcn.py:39-40, dgcnv2.py:45
    p["speaker_onehot"] = module in ("mmgcn", "dagerc", "dgcnv2")                                 # mmgcn.py:39, dagerc.py:41, dgcnv2.py:44
    return p


# ------------------------------------------------------------------------------------------------ data
def synthetic_dataset(n_dialogues, p, seed, one_speaker=False):
    """Dialogues in the reference's sample format with the data set's feature sizes; IEMOCAP-like lengths
    (clamp(round(49 + 21 z), 8, 110)) or MOSEI-like (1 + Geometric(1/7) <= 40, one speaker id, mosei_feature.py:211)."""
    rng = np.random.default_rng(seed)
    mosei = "mosei" in p["dataset"]
    out = []
    for _ in range(n_dialogues):
        if mosei:
            L = int(min(40, rng.geometric(1.0 / 7.0)))
        else:
            L = int(np.clip(round(49 + 21 * rng.standard_normal()), 8, 110))
        if p.get("max_len"):
            L = min(L, int(p["max_len"]))
        spk = np.zeros(L, dtype=np.int64) if (mosei or one_speaker) else rng.integers(0, p["n_speakers"], size=L)
        label = rng.integers(0, p["n_classes"], size=L)
        # a learnable signal: the class shifts the first few text / audio dimensions
        t = rng.standard_normal((L, p["hidden_text"])).astype(np.float32)
        a = rng.standard_normal((L, p["hidden_audio"])).astype(np.float32)
        v = rng.standard_normal((L, p["hidden_visual"])).astype(np.float32)
        t[np.arange(L), label % p["hidden_text"]] += 3.0
        a[np.arange(L), label % p["hidden_audio"]] += 3.0
        out.append(({"text": list(t), "audio": list(a), "visual": list(v),
                     "speakers": [[1 if s == k else 0 for k in range(p["n_speakers"])] for s in spk],
                     "label": [int(x) for x in label]},))
    return out


def load_data(p):
    if p.get("data"):
        with open(p["data"], "rb") as f:
            d = pickle.load(f)
        wrap = lambda xs: [s if isinstance(s, tuple) else (s,) for s in xs]
        return wrap(d["train"]), wrap(d["test"]), "file %s" % p["data"]
    return (synthetic_dataset(p["train_dialogues"], p, 1000 + p["seed"]), synthetic_dataset(p["test_dialogues"], p, 2000 + p["seed"]),
            "synthetic (%s shape: t=%d a=%d v=%d)" % (p["dataset"], p["hidden_text"], p["hidden_audio"], p["hidden_visual"]))


# ------------------------------------------------------------------------------------------------ data parallelism
def init_distributed(p, log=print):
    """The torchrun environment (as bench.py reads it): WORLD_SIZE, RANK, LOCAL_RANK.  Returns (rank, world).  With
    WORLD_SIZE unset or 1 nothing is touched; otherwise p["device"] becomes LOCAL_RANK and the NCCL process group is
    initialised on that device (the caller destroys it)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return 0, 1
    import torch.distributed as dist
    rank, local = int(os.environ["RANK"]), int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        log("train_mm: %d processes; each runs on cuda:LOCAL_RANK, --device=%s is ignored" % (world, p["device"]))
    p["device"] = local
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world


def deal_batches(n_batches, world):
    """Per optimizer step, the index of the batch each rank trains on: step s takes batches s*W .. s*W+W-1 of the epoch's
    list and rank r the (s*W + r)-th (accelerate's BatchSamplerShard with split_batches=False).  A last round the list does
    not fill is completed with batches from its start (even_batches=True).  world = 1: [[0], [1], ...]."""
    steps = (n_batches + world - 1) // world
    return [[(s * world + r) % n_batches for r in range(world)] for s in range(steps)]


def shard_test_batches(n_batches, rank, world):
    """The test batches ``rank`` evaluates: r, r+W, r+2W, ... of the one-GPU batch list (each keeps its one-GPU composition
    and padding, which the unpacked reverse LSTMs of dgcnv2 / MMGCN run over)."""
    return list(range(rank, n_batches, world))


def restore_order(per_rank):
    """per_rank[r] = the results of rank r's batches (shard_test_batches) -> the results in the one-GPU batch order."""
    world = len(per_rank)
    return [per_rank[i % world][i // world] for i in range(sum(len(x) for x in per_rank))]


# ------------------------------------------------------------------------------------------------ trainer
DGCN_LOSS_WEIGHTS = [1 / 0.086747, 1 / 0.144406, 1 / 0.227883, 1 / 0.160585, 1 / 0.127711, 1 / 0.252668]      # dgcn.py:109-110


def build_model(p, dev):
    if p["module"] == "cogmen":
        from .track_mm.cogmen import COGMENModule
        m = COGMENModule(input_size=p["hidden_all"], hidden_size=100, num_head=p["num_heads"], n_speakers=p["n_speakers"],
                         n_classes=p["n_classes"], build_dead_encoder=bool(p.get("dead_encoder", False)))
    elif p["module"] == "dgcn":
        from .track_mm.dgcn import DGCNModule
        m = DGCNModule(input_size=p["hidden_all"], hidden_size=200, n_speakers=p["n_speakers"], n_classes=p["n_classes"])
    elif p["module"] == "dgcnv2":
        from .track_mm.dgcnv2 import DGCNModule as DGCNv2Module
        m = DGCNv2Module(base_model=p["base_model"], input_size=p["hidden_all"], hidden_size=100, n_speakers=p["n_speakers"],
                         n_classes=p["n_classes"], context_attention="general")                      # dgcnv2.py:188-195
    elif p["module"] == "mmgcn":
        from .track_mm.mmgcn import MMGCNModule
        m = MMGCNModule(hidden_text=p["hidden_text"], hidden_visual=p["hidden_visual"], hidden_audio=p["hidden_audio"],
                        n_speakers=p["n_speakers"], n_classes=p["n_classes"], modals=p["modality"])
    else:
        from .track_mm.dagerc import DAGERCModule
        m = DAGERCModule(emb_dim=p["hidden_all"], dropout=p["dropout"], gnn_layers=p["gnn_layers"], n_classes=p["n_classes"])
    return m.to(dev)


# ------------------------------------------------------------------------------------------------ checkpoints
def load_checkpoint(path):
    return torch.load(path, map_location="cpu", weights_only=True)


def is_reference_layout(ckpt):
    """The reference trainer's Trainer.state_dict() layout (lumo/trainer/trainer.py:623-632): {'models': {'model': sd},
    'optims': ..., 'others': ..., 'thtensor': ..., 'nptensor': ...}; anything else is a plain model state_dict."""
    return isinstance(ckpt, dict) and isinstance(ckpt.get("models"), dict) and "model" in ckpt["models"]


def load_model_weights(model, ckpt, log=print):
    """Weights and buffers of a checkpoint of either layout into ``model``.  A leading ``module.`` (DDP, accelerate) is
    stripped; every key of ``model`` must be present; keys ``model`` does not have (COGMEN's dead encoder in a build
    without it) are ignored and logged.  Returns the ignored keys."""
    sd = ckpt["models"]["model"] if is_reference_layout(ckpt) else ckpt
    sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in sd.items()}
    own = model.state_dict()
    missing = [k for k in own if k not in sd]
    if missing:
        raise SystemExit("train_mm: the checkpoint lacks %d of the module's keys: %s" % (len(missing), ", ".join(missing)))
    ignored = [k for k in sd if k not in own]
    if ignored:
        log("train_mm: ignoring %d checkpoint keys this build does not have: %s" % (len(ignored), ", ".join(ignored)))
    model.load_state_dict({k: sd[k] for k in own}, strict=True)
    return ignored


def reference_param_names(p):
    """Names of the reference module's parameters() in order -- what the indices of its torch.optim state count.  For
    COGMEN that list includes the dead TransformerEncoder, which this build leaves out unless --dead_encoder."""
    with torch.device("meta"):
        m = build_model(dict(p, dead_encoder=True), torch.device("meta"))
    return [k for k, _ in m.named_parameters()]


def load_reference_optim(optim, ckpt, p, names, log=print):
    """The Adam state of a reference-layout checkpoint train_mm did not write into ``optim`` (FlatAdam; ``names``: its
    parameters' names).  Without 'param_names' its indices are mapped to names through the reference module's parameter
    list.  Returns False, after saying so in the log, when the state cannot be mapped (the weights alone are loaded)."""
    optims = ckpt.get("optims") or {}
    sd = optims.get("optim", next(iter(optims.values())) if len(optims) == 1 else None)
    if not isinstance(sd, dict) or not sd.get("param_groups"):
        log("train_mm: the checkpoint holds no optimizer state; loading the weights only")
        return False
    g = sd["param_groups"]
    if len(g) == 1 and "param_names" not in g[0]:
        ref = reference_param_names(p)
        if len(g[0]["params"]) == len(ref):
            sd = dict(sd, param_groups=[dict(g[0], param_names=ref)])
    try:
        optim.load_state_dict(sd, names)
    except (ValueError, KeyError) as e:
        log("train_mm: the checkpoint's optimizer state does not map onto this module's parameters (%s); loading the "
            "weights only" % e)
        return False
    return True


def run_params(p, world):
    return dict({k: p[k] for k in RUN_KEYS}, world=world)


def check_resumable(ckpt, p, world, path):
    """SystemExit unless ``ckpt`` can continue this run: reference layout, and, when train_mm wrote it, the same
    run-defining parameters (RUN_KEYS and the number of processes)."""
    if not is_reference_layout(ckpt):
        raise SystemExit("train_mm: --resume=%s is a plain state_dict; resuming needs a checkpoint written with "
                         "--ckpt_layout=reference (--load reads the weights alone)" % path)
    mine = (ckpt.get("others") or {}).get("train_mm")
    if mine is None:
        return
    want = run_params(p, world)
    diff = ["%s=%r (checkpoint: %r)" % (k, want[k], mine["params"].get(k)) for k in want if mine["params"].get(k) != want[k]]
    if diff:
        raise SystemExit("train_mm: --resume=%s comes from a different run; it cannot continue with %s"
                         % (path, ", ".join(diff)))


def _plain(x):
    """numpy scalars (sklearn's metrics) -> Python numbers, so the checkpoint loads with torch.load(weights_only=True)."""
    if isinstance(x, dict):
        return {k: _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    return x.item() if isinstance(x, np.generic) else x


class Trainer:
    def __init__(self, p, rank=0, world=1, log=print):
        """rank / world from init_distributed; world > 1 needs the process group initialised."""
        from .collate import DeviceCollate
        from .optim import FlatAdam
        self.p = p
        self.rank, self.world, self.log = rank, world, log
        self.dev = torch.device("cuda", int(p["device"])) if p["device"] != "cpu" else None
        if self.dev is None or not torch.cuda.is_available():
            raise SystemExit("train_mm: the libercgraph modules need a CUDA device (there is no CPU path)")
        torch.cuda.set_device(self.dev)
        torch.manual_seed(p["seed"])
        self.model = build_model(p, self.dev)
        self.collate = DeviceCollate(p["modality"], p["batch_first"], p["speaker_onehot"], p["n_speakers"], device=self.dev)
        self.optim = FlatAdam(self.model.parameters(), lr=p["lr"], weight_decay=p["weight_decay"], decoupled=p["optim"] == "AdamW",
                              max_norm=5.0 if p["module"] == "dagerc" else None,                    # dagerc.py:229-231
                              extra_slots=2 if world > 1 else 0)           # this rank's loss and accuracy ride with the gradient
        self.comm = self.reduce = None
        if world > 1:
            import torch.distributed as dist
            for t in list(self.model.parameters()) + list(self.model.buffers()):
                dist.broadcast(t.data, 0)                  # rank 0's state everywhere, as DDP does when it wraps the model
            self.optim.grad_scale = 1.0 / world            # the Adam kernel averages the summed gradients (and the clip norm)
        self.class_weight = None
        if p["module"] in ("dgcn", "dgcnv2") and p.get("loss_weights") and p["n_classes"] == 6:
            self.class_weight = torch.tensor(DGCN_LOSS_WEIGHTS, device=self.dev)
        self.param_names = [k for k, _ in self.model.named_parameters()]     # the order of model.parameters()
        self.best, self.history, self.start_epoch = {}, [], 1

    def resume(self, ckpt, path):
        """--resume (after check_resumable): weights, buffers and Adam state; for a checkpoint train_mm wrote also the
        best record, the history, this rank's CPU generator and the epoch counter."""
        load_model_weights(self.model, ckpt, self.log)
        mine = (ckpt.get("others") or {}).get("train_mm")
        if mine is None:
            self.log("train_mm: %s was not written by train_mm: its weights and optimizer state are loaded, training starts "
                     "at epoch 1 and the run parameters cannot be checked" % path)
            load_reference_optim(self.optim, ckpt, self.p, self.param_names, self.log)
            return
        self.optim.load_state_dict(ckpt["optims"]["optim"], self.param_names)     # applied when the optimizer attaches
        self.best, self.history = mine["best"], list(mine["history"])
        torch.set_rng_state(mine["rng"][self.rank])
        self.start_epoch = int(mine["epoch"]) + 1
        self.log("train_mm: resuming %s after epoch %d" % (path, mine["epoch"]))

    def _logits(self, batch):
        m = self.p["module"]
        if m == "cogmen":
            return self.model(**batch.packed_kwargs())[0]
        if m == "dgcn":
            return self.model(input_tensor=batch["input_tensor"], speaker_tensor=batch["speaker_tensor"], text_length=batch["text_length"])[0]
        if m == "dgcnv2":
            return self.model(input_tensor=batch["input_tensor"], speaker_tensor=batch["speaker_tensor"],
                              attention_mask=batch["attention_mask"], text_length=batch["text_length"])[0]
        if m == "mmgcn":
            return self.model(text_feature=batch["text_feature"], audio_feature=batch["audio_feature"],
                              visual_feature=batch["visual_feature"], speaker_tensor=batch["speaker_tensor"],
                              text_length=batch["text_length"])[0]
        logits = self.model(input_tensor=batch["input_tensor"], text_length=batch["text_length"], speaker_tensor=batch["speaker_tensor"])[0]
        return logits[batch["attention_mask"].bool()]                                               # dagerc.py:223-226

    def train_step(self, samples):
        from . import ops
        batch = self.collate(samples)
        logits = self._logits(batch)
        loss = ops.cross_entropy(logits, batch["label"], self.class_weight)
        self.optim.zero_grad()
        loss.backward()
        if self.world > 1:
            return self._step_data_parallel(loss.detach(), logits, batch["label"])
        self.optim.step()
        with torch.no_grad():
            acc = (logits.argmax(-1) == batch["label"]).float().mean()
        return loss.detach(), acc

    def _step_data_parallel(self, loss, logits, labels):
        """gather -> all-reduce(sum) of the flat gradient buffer -> Adam with grad_scale = 1/W (DDP's averaged gradient;
        DAG-ERC's clip then acts on the norm of the average).  Returns the mean over the ranks of loss and accuracy, which
        ride in the buffer's two extra slots."""
        opt = self.optim
        if opt.live is None:
            self._attach_data_parallel()
        opt.gather()
        with torch.no_grad():
            acc = (logits.argmax(-1) == labels).float().mean()
            opt.extra.copy_(torch.stack([loss.float().reshape(()), acc]))
        self.reduce(opt.flat_g)
        opt.update()
        mean = opt.extra / self.world
        return mean[0], mean[1]

    def _attach_data_parallel(self):
        """After the first backward: the flat layout (must be the same on every rank, or the sum would mix parameters), then
        the communicator, collectively -- peer memory when every rank can open its peers, else NCCL."""
        import torch.distributed as dist
        from .p2p import PeerComm, Reducer
        opt = self.optim.attach()
        names = {id(t): k for k, t in self.model.named_parameters()}
        layout = [(names[id(t)], t.numel(), off) for t, off in zip(opt.live, opt.offsets)]
        layouts = [None] * self.world
        dist.all_gather_object(layouts, layout)
        bad = [r for r, lay in enumerate(layouts) if lay != layouts[0]]
        if bad:
            raise RuntimeError("train_mm: the parameters that received a gradient differ between rank 0 and rank(s) %s; "
                               "their flat gradient buffers cannot be summed" % bad)
        nbytes = opt.flat_g.numel() * opt.flat_g.element_size()
        comms = PeerComm.create(dist.group.WORLD, self.dev, max_bytes=nbytes)
        self.comm = comms[0] if comms else None
        self.reduce = Reducer(None, self.comm)
        if self.comm is not None:
            opt.skip_if_nonzero = self.comm.status_word()  # a timed-out exchange is never applied (ercg_adam_step_guarded)
        self.log("train_mm: gradient all-reduce of %d floats over %d GPUs through %s" % (opt.flat_g.numel(), self.world,
                                                                                          self.reduce.transport))

    def _check_exchange(self):
        """Raise on every rank if a peer-memory all-reduce timed out on any rank (no update was applied after it)."""
        import torch.distributed as dist
        from ._lib import ErcgError, lib
        status = [None] * self.world
        dist.all_gather_object(status, self.comm.status())
        bad = [(r, s) for r, s in enumerate(status) if s != 0]
        if bad:
            raise ErcgError("train_mm: peer-memory gradient all-reduce failed: %s" % ", ".join(
                "rank %d: %s (%d)" % (r, lib().ercg_strerror(s).decode(), s) for r, s in bad))

    @torch.no_grad()
    def test(self, data):
        """mmbase.py:180-201 + on_test_end :262-283."""
        from sklearn import metrics
        from . import ops
        if self.world > 1:
            import torch.distributed as dist
            for b in self.model.buffers():
                dist.broadcast(b, 0)                      # rank 0's BatchNorm running statistics (DDP broadcast_buffers)
        self.model.eval()
        bs = self.p["batch_size"]
        starts = list(range(0, len(data), bs))
        mine = []
        for i in shard_test_batches(len(starts), self.rank, self.world):
            batch = self.collate(data[starts[i]:starts[i] + bs])
            logits = self._logits(batch)
            ys = batch["label"]
            mine.append((float(ops.cross_entropy(logits, ys)), ys.cpu().tolist(), logits.argmax(-1).cpu().tolist()))
        self.model.train()
        results = mine
        if self.world > 1:
            per_rank = [None] * self.world
            dist.all_gather_object(per_rank, mine)
            results = restore_order(per_rank)
        true, pred, lsum, n = [], [], 0.0, 0
        for ce, ys, ps in results:
            lsum += ce * len(ys)
            n += len(ys)
            true.extend(ys)
            pred.extend(ps)
        return {"Lall": lsum / max(n, 1), "acc": metrics.accuracy_score(true, pred),
                "wa": metrics.balanced_accuracy_score(true, pred),
                "f1": metrics.f1_score(true, pred, average="weighted"), "mif1": metrics.f1_score(true, pred, average="micro"),
                "maf1": metrics.f1_score(true, pred, average="macro"),
                "cm": metrics.confusion_matrix(true, pred, labels=range(self.p["n_classes"])).tolist(), "C": n}

    def _rng_states(self):
        """The CPU generator state of every rank (the dropout seeds are drawn from it, by MMGCN in the test pass too, and
        the ranks evaluate unequal numbers of test batches), gathered on every rank."""
        st = torch.get_rng_state()
        if self.world == 1:
            return [st]
        import torch.distributed as dist
        out = [None] * self.world
        dist.all_gather_object(out, st)
        return out

    def save(self, name, epoch=None, rngs=None):
        """``state_dict`` layout: the model's state_dict (mmbase.py:325-333).  ``reference`` layout (``rngs`` from
        _rng_states): the reference trainer's Trainer.state_dict() with torch.optim's Adam state, plus what --resume
        needs under others.train_mm.  Written to a temporary file and renamed, so a kill never leaves a truncated file."""
        d = self.p.get("save_dir")
        if not d or self.rank != 0:
            return None
        os.makedirs(d, exist_ok=True)
        path = os.path.join(d, name)
        obj = {k: v.detach().cpu().clone() for k, v in self.model.state_dict().items()}
        if self.p["ckpt_layout"] == "reference":
            osd = self.optim.torch_state_dict(self.param_names)
            osd["state"] = {i: {k: v.detach().cpu() for k, v in st.items()} for i, st in osd["state"].items()}
            obj = {"models": {"model": obj}, "optims": {"optim": osd},
                   "others": {"train_mm": {"epoch": epoch, "best": _plain(self.best), "history": _plain(self.history),
                                           "params": run_params(self.p, self.world), "rng": rngs}},
                   "thtensor": {}, "nptensor": {}}
        tmp = path + ".tmp"
        torch.save(obj, tmp)
        os.replace(tmp, path)
        return path

    def train(self, train, test, log=print):
        p = self.p
        ref = p["ckpt_layout"] == "reference"
        self.model.train()
        history = self.history
        epoch = self.start_epoch - 1
        for epoch in range(self.start_epoch, int(p["epoch"]) + 1):
            rng = np.random.default_rng(p["seed"] * 100003 + epoch)                                  # rnd.mark(seed) per epoch, mmbase.py:207-208
            order = rng.permutation(len(train))
            t0 = time.perf_counter()
            lsum, asum, nb, utts = 0.0, 0.0, 0, 0
            batches = [order[i:i + p["batch_size"]] for i in range(0, len(order), p["batch_size"])]
            for dealt in deal_batches(len(batches), self.world):
                samples = [train[j] for j in batches[dealt[self.rank]]]
                loss, acc = self.train_step(samples)
                lsum += float(loss)
                asum += float(acc)
                nb += 1
                utts += sum(len(train[j][0]["text"]) for b in dealt for j in batches[b])     # the utterances of every rank
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if self.comm is not None:
                self._check_exchange()
            te = self.test(test)                                                                      # test_per_epoch = 1, mmbase.py:136
            rec = {"epoch": epoch, "train_Lall": lsum / nb, "train_Acc": asum / nb, "utt_per_s": utts / dt,
                   **{"test_" + k: v for k, v in te.items() if k != "cm"}}
            history.append(rec)
            rngs = self._rng_states() if ref else None                  # collective: before the rank-0-only writes
            if te["f1"] >= self.best.get("f1", -1.0):
                self.best = {"f1": te["f1"], "acc": te["acc"], "epoch": epoch, "cm": te["cm"]}
                self.save("best_model.ckpt", epoch, rngs)
            if ref:
                self.save("last_model.ckpt", epoch, rngs)              # every epoch: an interrupted run can be resumed
            log("epoch %3d  train Lall %.4f Acc %.3f  |  test Lall %.4f acc %.3f f1 %.3f  |  %.0f utt/s" % (
                epoch, rec["train_Lall"], rec["train_Acc"], te["Lall"], te["acc"], te["f1"], rec["utt_per_s"]))
        if not ref or self.start_epoch > int(p["epoch"]):
            self.save("last_model.ckpt", epoch, self._rng_states() if ref else None)
        return history


def main(argv=None, log=print):
    args = parse_args(list(sys.argv[1:] if argv is None else argv))
    p = resolve_params(args)
    rank, world = init_distributed(p, log)
    if rank != 0:
        log = lambda *a: None                                                                   # only rank 0 logs
    try:
        train, test, what = load_data(p)
        log("train_mm: module=%s dataset=%s modality=%s hidden_all=%d n_classes=%d n_speakers=%d | %s: %d / %d dialogues" % (
            p["module"], p["dataset"], p["modality"], p["hidden_all"], p["n_classes"], p["n_speakers"], what, len(train), len(test)))
        ckpt = None
        if p["resume"]:
            ckpt = load_checkpoint(p["resume"])                     # every rank reads it
            check_resumable(ckpt, p, world, p["resume"])
        tr = Trainer(p, rank, world, log=log)
        if ckpt is not None:
            tr.resume(ckpt, p["resume"])
        elif p["load"]:
            load_model_weights(tr.model, load_checkpoint(p["load"]), log)
            log("train_mm: weights loaded from %s" % p["load"])
        if p.get("eval_first"):
            log("eval_first:", {k: v for k, v in tr.test(test).items() if k != "cm"})
        hist = tr.train(train, test, log=log)
        log("Best Results", json.dumps({k: v for k, v in tr.best.items() if k != "cm"}))
        if tr.comm is not None:
            import torch.distributed as dist
            dist.barrier()                                 # no peer still reads this rank's region
            tr.comm.close()
        return {"params": p, "history": hist, "best": tr.best, "trainer": tr}
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
