"""The COGMEN, DialogueGCN, dgcnv2, MMGCN and DAG-ERC train steps as ONE replayable unit each (SURVEY.md 8e / 8f-3;
reference: CogmenTrainer.train_step, track_mm/cogmen.py:179-195, the DialogueGCN step, dgcn.py:117-134, dgcnv2's
(track_mm/dgcnv2.py), MMGCN's, mmgcn.py:141-157, and DAG-ERC's, dagerc.py:217-237, under accelerate/DDP,
lumo/trainer/trainer.py:62-64,315-327).

    graph build (K1) -> forward -> cross entropy -> backward -> gradient all-reduce -> [clip] -> Adam

* Nothing in the step touches the host: sizes and the possible relation ids come from the host-side batch description,
  the loss normaliser is host-known (COGMEN: the global utterance count) or reduced on the device (the other four), the
  optimizer's step counter and the dropout seed live on the device.  ``capture()`` records the step once into a
  CUDA graph (collectives included) and ``replay()`` relaunches it: ~50 kernel launches + autograd bookkeeping per step
  become one graph launch -- what makes 2^20 utterances split over 8 GPUs (1.7 ms of kernels per rank) scale.
* Collectives per step with world > 1: COGMEN's BatchNorm statistics (2H+1 doubles, forward), their backward sums (2H
  floats) -- both only in ``bn_sync="global"`` mode; ``"local"`` is the reference's DDP behaviour (per-rank statistics) --,
  the DialogueGCN / dgcnv2 / MMGCN / DAG-ERC loss (numerator, denominator: 2 floats, forward), and the flat gradient buffer.
  COGMEN's loss numerator rides in the tail of the gradient buffer; there is no separate loss collective.
* Transport: libercgraph's peer-memory kernels over NVLink (p2p.PeerComm: ercg_p2p_allreduce for the gradient buckets,
  ercg_p2p_bn_stats / ercg_p2p_bn_act_bwd_reduce = the BatchNorm reductions fused with their exchange) when every rank can set
  them up, else torch.distributed on ``group`` -- the results are the same to the last bit (rank-ordered sums).
* The gradient all-reduce is bucketed in two: everything except the parameters of the input transform is reduced on a side
  stream as soon as those gradients exist, under the input transform's weight-gradient GEMM (the longest kernel of the
  step); the input transform's own gradients follow on the main stream.
"""
import torch

from . import ops, ops_dagerc
from .graph import build_graph, graph_sizes, relation_ids_for_speakers
from .optim import FlatAdam

TRANSPORTS = ("auto", "p2p", "nccl")


def _lengths(lengths, who):
    """CPU int64 [B] dialogue lengths, B >= 1, every length >= 1 (ValueError otherwise)."""
    t = torch.as_tensor(lengths)
    if t.dim() != 1 or t.numel() == 0 or t.is_floating_point():
        raise ValueError("%s: lengths must be a non-empty 1-D integer tensor, got %s %s" % (who, t.dtype, tuple(t.shape)))
    t = t.to(torch.int64).cpu().contiguous()
    if int(t.min()) < 1:
        raise ValueError("%s: every dialogue length must be >= 1, got %d" % (who, int(t.min())))
    return t


class _FlatTrainStep:
    """What the train steps share: communicators, the flat optimizer layout with the two gradient buckets, the bucketed
    all-reduce + Adam tail, capture / replay and the deferred input check.  A subclass passes its FlatAdam and provides
    ``_forward_backward(x, spk, labels)`` (which ends in ``self._backward(loss)``), ``_late_params()`` (the parameters
    whose gradients come last: the input transform's) and ``global_loss()``."""

    def __init__(self, model, opt, comm_bytes, world, group, transport, overlap):
        """transport: "p2p" = peer-memory all-reduce kernels (ercg_p2p_allreduce, one NVSwitch node), "nccl" =
        torch.distributed on ``group``, "auto" = p2p when every rank can set it up, else torch.distributed.  opt: the step's
        FlatAdam.  comm_bytes: payload size of the peer-memory communicators; the first step, and every step without
        overlap, all-reduces the whole flat gradient buffer in one call, so it must hold that buffer."""
        from .p2p import PeerComm, Reducer
        name = type(self).__name__
        if isinstance(world, bool) or not isinstance(world, int) or world < 1:
            raise ValueError("%s: world must be an int >= 1, got %r" % (name, world))
        if transport not in TRANSPORTS:
            raise ValueError("%s: transport must be one of %s, got %r" % (name, ", ".join(TRANSPORTS), transport))
        self.model, self.world, self.group = model, world, group
        self.dev = next(model.parameters()).device
        comms = None
        if world > 1 and transport in ("auto", "p2p") and self.dev.type == "cuda":
            # two communicators: the early gradient bucket runs on a side stream next to the main stream's collectives
            comms = PeerComm.create(group, self.dev, max_bytes=comm_bytes, n=2)
            if comms is None and transport == "p2p":
                raise RuntimeError("%s: transport='p2p' but the peer-memory communicator could not be set up" % type(self).__name__)
        self.comms, self.comm_bytes = comms, comm_bytes
        self.reduce_main = Reducer(group, comms[0] if comms else None)
        self.reduce_side = Reducer(group, comms[1] if comms else None)
        self.opt = opt
        self.overlap = bool(overlap) and world > 1
        self.side = torch.cuda.Stream(device=self.dev) if self.overlap else None
        self._graph = None
        self._static = None
        self._graph_loss = None      # the captured step's loss (rewritten by every replay)
        self._last_loss = None       # the loss of the last step run, eager or replayed
        self._pending = 0
        self._n_early = None
        self._hooks = []
        self._late_ids = None

    # ------------------------------------------------------------------------------------------ one step, eager
    def _backward(self, loss):
        self.opt.zero_grad()
        self._pending = self._n_early if self._n_early is not None else -1
        loss.backward()

    def _late_first(self, p):
        # flat layout: gradients that exist EARLY in the backward first, the input transform's (computed last) at the end
        return 1 if id(p) in self._late_ids else 0

    def _attach(self):
        self._late_ids = {id(p) for p in self._late_params()}
        self.opt.attach(order=self._late_first)
        live = self.opt.live
        self._n_early = sum(1 for p in live if self._late_first(p) == 0)
        if self.overlap:
            for p in live[:self._n_early]:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._on_grad))

    def _on_grad(self, _p):
        """post-accumulate hook of every early parameter: when the last one has its gradient, reduce that bucket on the side
        stream while the main stream goes on to the input transform's weight gradient."""
        self._pending -= 1
        if self._pending != 0:
            return
        opt = self.opt
        opt.gather(0, self._n_early)
        ev = torch.cuda.Event()
        ev.record()
        self.side.wait_event(ev)
        with torch.cuda.stream(self.side):
            self.reduce_side(opt.span(0, self._n_early))

    def _first_step(self, loss):
        """Called once, right after the flat layout exists (before the first un-bucketed all-reduce)."""

    def step(self, x, spk, labels):
        """One eager step.  Returns the loss (device scalar): COGMEN, this rank's share of the global mean; DialogueGCN,
        the global weighted mean."""
        loss = self._forward_backward(x, spk, labels)
        if self.opt.live is None:
            self._attach()                                   # first step: decide the flat layout, then finish it un-bucketed
            self._first_step(loss)
            self.opt.gather()
            if self.world > 1:
                self.reduce_main(self.opt.flat_g)
            self.opt.update()
            self._last_loss = loss.detach()
            return self._last_loss
        opt = self.opt
        if self.world > 1:
            if self.overlap:
                opt.gather(self._n_early, None)
                self.reduce_main(opt.flat_g[opt.offsets[self._n_early]:])                    # late bucket + loss slots
                torch.cuda.current_stream(self.dev).wait_stream(self.side)
            else:
                opt.gather()
                self.reduce_main(opt.flat_g)
        else:
            opt.gather()
        opt.update()
        self._last_loss = loss.detach()
        return self._last_loss

    # ------------------------------------------------------------------------------------------ capture / replay
    def capture(self, x, spk, labels, warmup=3):
        """Record the step on the given STATIC input tensors (refill them in place between replays)."""
        self._static = (x, spk, labels)
        s = torch.cuda.Stream(device=self.dev)
        s.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(s):                           # warm-up on a side stream, as torch.cuda.graph requires
            for _ in range(max(warmup, 2)):                  # (first call attaches the flat buffers)
                self.step(x, spk, labels)
        torch.cuda.current_stream(self.dev).wait_stream(s)
        torch.cuda.synchronize(self.dev)
        ops.SEED_DEV = self.opt.step_dev                     # dropout seed = host seed + device step counter: fresh mask per replay
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._graph_loss = self.step(x, spk, labels)
        ops.SEED_DEV = None
        return self

    def replay(self):
        self._graph.replay()
        self._last_loss = self._graph_loss
        return self._graph_loss

    def check(self):
        """Raise if K1 flagged the batch of the last step (bad lengths / speaker ids / relation id outside the hint), or if
        a peer-memory collective timed out."""
        self._check_inputs()
        for c in self.comms or ():
            c.check()

    @property
    def transport(self):
        return self.reduce_main.transport


class _WindowGraphStep(_FlatTrainStep):
    """COGMEN and DialogueGCN: a K1 window graph (model.wp / model.wf) over the packed batch, rebuilt every step from the
    speaker ids, with its sizes and possible relation ids known on the host."""

    def __init__(self, model, lengths, speakers_present, opt, comm_bytes, world, group, transport, overlap):
        """lengths: CPU int64 [B] dialogue lengths of THIS rank's batch (a step re-run on new data of the same lengths reuses
        the capture; new lengths need a new capture).  speakers_present: the speaker ids the data set uses."""
        super().__init__(model, opt, comm_bytes, world, group, transport, overlap)
        self.lengths = lengths.to(torch.int64).cpu().contiguous()
        self.sizes = graph_sizes(self.lengths, model.wp, model.wf)
        self.lengths_dev = self.lengths.to(self.dev)
        self.rel_ids = relation_ids_for_speakers(speakers_present, model.n_speakers)

    def _check_inputs(self):
        self._last_graph.check_inputs()


class CogmenTrainStep(_WindowGraphStep):
    def __init__(self, model, lengths, speakers_present=(0,), lr=1e-4, weight_decay=1e-8, world=1, global_utterances=None,
                 bn_sync="global", overlap=True, group=None, transport="auto"):
        """See _WindowGraphStep.  global_utterances: the utterance count of the GLOBAL batch (the loss normaliser; default
        this rank's).  bn_sync: "global" = BatchNorm statistics over all ranks, "local" = per rank (the reference's DDP)."""
        from .dist import StatSync
        opt = FlatAdam(model.parameters(), lr=lr, weight_decay=weight_decay, extra_slots=1)
        # 8 MB holds the live gradient (1.1 MB at width 1443); the dead encoder's parameters never get one
        super().__init__(model, lengths, speakers_present, opt, 8 << 20, world, group, transport, overlap)
        self.global_utts = int(global_utterances if global_utterances is not None else self.sizes[0])
        if world > 1 and bn_sync == "global":
            model.gcn.stat_sync = StatSync(group=group, global_count=self.global_utts, reduce=self.reduce_main)
        self.loss_share = None

    def _forward_backward(self, x, spk, labels):
        m = self.model
        g = build_graph(self.lengths_dev, spk, m.wp, m.wf, m.n_speakers, device=self.dev, sizes=self.sizes,
                        relation_ids=self.rel_ids)
        logits, _ = m.forward_packed(x, spk, self.lengths_dev, graph=g)
        num_out = self.opt.extra if self.opt.live is not None else None
        loss = ops.cross_entropy(logits, labels, denom=self.global_utts if self.world > 1 else None, num_out=num_out)
        self._backward(loss)
        self._last_graph = g
        return loss

    def _late_params(self):
        proj = self.model.rnn[1]
        return proj.weight, proj.bias

    def _first_step(self, loss):
        if self.world > 1:                                   # the loss slot was not attached during the first forward
            self.opt.extra.copy_(loss.detach().reshape(1) * float(self.global_utts))

    def global_loss(self):
        """Global mean loss of the last step (valid after the gradient all-reduce; world == 1: the local loss)."""
        return self.opt.extra[0] / float(self.global_utts)


class DgcnTrainStep(_WindowGraphStep):
    def __init__(self, model, lengths, speakers_present=None, lr=3e-4, weight_decay=0.0, class_weight=None, world=1,
                 group=None, transport="auto", overlap=True):
        """DialogueGCN (track_mm.dgcn.DGCNModule) step.  See _WindowGraphStep.  speakers_present: default every speaker id of
        the model.  lr / weight_decay: dgcn.py's Adam defaults.  class_weight: the cross entropy's class weights
        (track_mm.dgcn.LOSS_WEIGHTS for the 6-way IEMOCAP setting, dgcn.py:109-110) or None.  The loss is the weighted mean
        over the GLOBAL batch: with world > 1 its (numerator, denominator) is all-reduced in the forward, so a batch sharded
        by dialogue takes the same step as one GPU on the whole batch."""
        if speakers_present is None:
            speakers_present = range(model.n_speakers)
        opt = FlatAdam(model.parameters(), lr=lr, weight_decay=weight_decay)
        # every parameter but the classifier's unused emotion_att gets a gradient: 8.6 MB at width 1380
        super().__init__(model, lengths, speakers_present, opt, max(8 << 20, opt.flat_bytes()), world, group, transport, overlap)
        self.class_weight = None
        if class_weight is not None:
            self.class_weight = torch.as_tensor(class_weight, dtype=torch.float32).to(self.dev).contiguous()

    def _forward_backward(self, x, spk, labels):
        m = self.model
        g = build_graph(self.lengths_dev, spk, m.wp, m.wf, m.n_speakers, device=self.dev, mean_weight=False, sizes=self.sizes,
                        relation_ids=self.rel_ids)
        logits, _ = m.forward_packed(x, spk, self.lengths_dev, graph=g)
        loss = ops.cross_entropy(logits, labels, self.class_weight, reduce_sync=self.reduce_main if self.world > 1 else None)
        self._backward(loss)
        self._last_graph = g
        return loss

    def _late_params(self):
        rnn = self.model.rnn.rnn
        return tuple(getattr(rnn, n + "_l0" + d) for n in ("weight_ih", "bias_ih", "bias_hh") for d in ("", "_reverse"))

    def global_loss(self):
        """Global weighted mean loss of the last step (eager or replayed)."""
        return self._last_loss


class MmgcnTrainStep(_FlatTrainStep):
    def __init__(self, model, lengths, lmax=None, lr=3e-4, weight_decay=3e-5, world=1, group=None, transport="auto",
                 overlap=True):
        """MMGCN (track_mm.mmgcn.MMGCNModule) step.  See _FlatTrainStep.  lengths: CPU [B] dialogue lengths of THIS rank's
        batch.  lmax: the padded length of the GLOBAL batch (default: this batch's longest dialogue).  The text LSTM runs
        unpacked over the padding (mmgcn.py:113-114), so the reverse direction of every dialogue depends on Lmax: a rank
        pads its shard to the global Lmax, and the shards then take the step one GPU takes on the whole batch.
        lr / weight_decay: mmgcn.py's Adam.  The loss is the mean cross entropy over the GLOBAL batch (numerator and
        denominator all-reduced in the forward when world > 1).

        step(feats, spk, labels): feats = (text, audio, visual), seq-first padded [lmax, B, D_m] (None for a modality the
        model does not use), spk: seq-first one-hot speakers [lmax, B, n_speakers], labels: packed int64 [N]."""
        self.lengths = _lengths(lengths, "MmgcnTrainStep")
        longest = int(self.lengths.max())
        self.lmax = longest if lmax is None else int(lmax)
        if self.lmax < longest:
            raise ValueError("MmgcnTrainStep: lmax %d is shorter than the longest dialogue (%d)" % (self.lmax, longest))
        opt = FlatAdam(model.parameters(), lr=lr, weight_decay=weight_decay)
        # every parameter but the dead attention / gating modules gets a gradient (64 GCNII weights [400, 200] among them);
        # flat_bytes() bounds it by all parameters: 27 MB at the IEMOCAP widths
        super().__init__(model, opt, max(8 << 20, opt.flat_bytes()), world, group, transport, overlap)
        self.graph = self.full_graph = None

    def _forward_backward(self, feats, spk, labels):
        if self.graph is None:
            # the graphs depend on the lengths alone: built once, by the first step (an eager one: capture() warms up first)
            from .track_mm.mmgcn_utils import lengths_graph
            self.graph = lengths_graph(self.lengths, self.dev)
            self.full_graph = lengths_graph(torch.full((self.lengths.numel(),), self.lmax, dtype=torch.int64), self.dev)
        text, audio, visual = feats
        ref = next(t for t in (text, audio, visual) if t is not None)
        if ref.size(0) != self.lmax or ref.size(1) != self.lengths.numel():
            raise ValueError("MmgcnTrainStep: features of shape %s, the step was built for [%d, %d, *]"
                             % (tuple(ref.shape), self.lmax, self.lengths.numel()))
        logits, _ = self.model(text, audio, visual, spk, self.lengths, graph=self.graph, full_graph=self.full_graph)
        loss = ops.cross_entropy(logits, labels, reduce_sync=self.reduce_main if self.world > 1 else None)
        self._backward(loss)
        return loss

    def _late_params(self):
        m = self.model
        return tuple(p for lin in (m.linear_a, m.linear_v, m.linear_l) for p in (lin.weight, lin.bias))

    def _check_inputs(self):
        self.graph.check_inputs()
        self.full_graph.check_inputs()

    def global_loss(self):
        """Global mean loss of the last step (eager or replayed)."""
        return self._last_loss


class Dgcnv2TrainStep(_FlatTrainStep):
    def __init__(self, model, lengths, lmax=None, speakers_present=None, lr=3e-4, weight_decay=0.0, class_weight=None, world=1,
                 group=None, transport="auto", overlap=True):
        """dgcnv2 (track_mm.dgcnv2.DGCNModule, base 'LSTM', 'GRU' or 'None') step.  See _FlatTrainStep.  lengths: CPU [B]
        dialogue lengths of THIS rank's batch.  lmax: the padded length of the GLOBAL batch (default: this batch's longest
        dialogue; at most max_seq_len = 110).  The unpacked reverse base starts in the padding (dgcnv2.py:151) and the edge
        attention's softmax runs over all padded positions (dgcnv2_models.py:544), so a rank pads its shard to the global
        lmax, and the shards then take the step one GPU takes on the whole batch.  speakers_present: the speaker ids the
        data set uses (default every speaker id of the model).  lr / weight_decay: train_mm's dgcnv2 Adam.  class_weight: the
        cross entropy's class weights (track_mm.dgcn.LOSS_WEIGHTS in the 6-way setting) or None.  The loss is the weighted
        mean over the GLOBAL batch (numerator and denominator all-reduced in the forward when world > 1).

        step(x_rows, speaker_ids, labels): x_rows [B * lmax, D] = the batch-first padded input viewed as rows (16-byte
        aligned), speaker_ids packed [N], labels packed int64 [N]."""
        self.lengths = _lengths(lengths, "Dgcnv2TrainStep")
        longest, cap = int(self.lengths.max()), model.att_model.max_seq_len
        self.lmax = longest if lmax is None else int(lmax)
        if self.lmax < longest:
            raise ValueError("Dgcnv2TrainStep: lmax %d is shorter than the longest dialogue (%d)" % (self.lmax, longest))
        if self.lmax > cap:
            raise ValueError("Dgcnv2TrainStep: lmax %d exceeds max_seq_len %d" % (self.lmax, cap))
        if speakers_present is None:
            speakers_present = range(model.n_speakers)
        opt = FlatAdam(model.parameters(), lr=lr, weight_decay=weight_decay)
        # every parameter but the edge attention's dead modules gets a gradient; flat_bytes() bounds it by all parameters
        super().__init__(model, opt, max(8 << 20, opt.flat_bytes()), world, group, transport, overlap)
        self.sizes = graph_sizes(self.lengths, model.window_past, model.window_future)
        self.lengths_dev = self.lengths.to(self.dev)
        self.rel_ids = relation_ids_for_speakers(speakers_present, model.n_speakers)
        self.class_weight = None
        if class_weight is not None:
            self.class_weight = torch.as_tensor(class_weight, dtype=torch.float32).to(self.dev).contiguous()
        self.gf = self.gfull = None

    def _forward_backward(self, x, spk, labels):
        from .track_mm.dgcnv2 import length_graphs
        m = self.model
        B, N = self.lengths.numel(), self.sizes[0]
        if x.dim() != 2 or x.size(0) != B * self.lmax or tuple(spk.shape) != (N,) or tuple(labels.shape) != (N,):
            raise ValueError("Dgcnv2TrainStep: x_rows %s, speaker_ids %s, labels %s; the step was built for [%d, D], [%d], [%d]"
                             % (tuple(x.shape), tuple(spk.shape), tuple(labels.shape), B * self.lmax, N, N))
        if self.gf is None:
            # these two depend on the lengths alone: built once, by the first step (an eager one: capture() warms up first)
            self.gf, self.gfull = length_graphs(self.lengths, self.lmax, self.dev)
        g = build_graph(self.lengths_dev, spk, m.window_past, m.window_future, m.n_speakers, device=self.dev, mean_weight=False,
                        sizes=self.sizes, relation_ids=self.rel_ids)
        logits, _ = m.forward_packed(x, spk, self.lengths_dev, self.lmax, graphs=(g, self.gf, self.gfull))
        loss = ops.cross_entropy(logits, labels, self.class_weight, reduce_sync=self.reduce_main if self.world > 1 else None)
        self._backward(loss)
        self._last_graph = g
        return loss

    def _late_params(self):
        m = self.model
        if m.base_model == "None":
            return m.base_linear.weight, m.base_linear.bias
        rnn = m.lstm if m.base_model == "LSTM" else m.gru
        # the LSTM's hoisted input transform folds in b_hh; the GRU applies b_hh inside the recurrence (dgcn_models.py:37-40)
        names = ("weight_ih", "bias_ih", "bias_hh") if m.base_model == "LSTM" else ("weight_ih", "bias_ih")
        return tuple(getattr(rnn, n + "_l0" + d) for n in names for d in ("", "_reverse"))

    def _check_inputs(self):
        self._last_graph.check_inputs()
        self.gf.check_inputs()
        self.gfull.check_inputs()

    def global_loss(self):
        """Global weighted mean loss of the last step (eager or replayed)."""
        return self._last_loss


class DagercTrainStep(_FlatTrainStep):
    def __init__(self, model, lengths, lr=1e-3, weight_decay=1e-2, max_norm=5.0, world=1, group=None, transport="auto",
                 overlap=True):
        """DAG-ERC (track_mm.dagerc.DAGERCModule) step.  See _FlatTrainStep.  lengths: CPU [B] dialogue lengths of THIS
        rank's batch.  The optimizer is dagerc.py's AdamW with clip_grad_norm_(params, max_norm) (max_norm None: no clip);
        the clip acts on the all-reduced gradient, the one a single GPU clips when it trains on the whole batch.  The loss
        is the mean cross entropy over the GLOBAL batch's real utterances, computed on the padded logits with the padding
        labelled -100 (no boolean indexing, so no wait for the device).  The DAG is causal, so the padding a rank adds
        changes none of its real utterances: the shards need no common padded length.

        step(x, spk, labels): x = batch-first padded input_tensor [B, Lmax, emb], spk = the speakers as DAGERCModule.forward
        takes them (one-hot [B, Lmax, n] or ids [B, Lmax]) on the device, labels int64 [B, Lmax] holding -100 at padding."""
        if max_norm is not None and not float(max_norm) > 0:
            raise ValueError("DagercTrainStep: max_norm must be > 0 or None, got %r" % (max_norm,))
        self.lengths = _lengths(lengths, "DagercTrainStep")
        opt = FlatAdam(model.parameters(), lr=lr, weight_decay=weight_decay, decoupled=True, max_norm=max_norm)
        # every parameter but the dead fcs / attentive_node_features gets a gradient (8 GRUCells of width 300 among them);
        # flat_bytes() bounds it by all parameters: 62 MB at width 1380, the dead [2880, 2880] transform included
        super().__init__(model, opt, max(8 << 20, opt.flat_bytes()), world, group, transport, overlap)
        self.Lmax = int(self.lengths.max())
        self.graph_lengths = model.graph_lengths(self.lengths, self.Lmax)
        self.graph_lengths_dev = self.graph_lengths.to(self.dev)
        self.sizes = graph_sizes(self.graph_lengths, 0, 0)
        self.order = ops_dagerc.dag_order(self.graph_lengths, self.dev)
        self.e_cap = ops_dagerc.dag_edge_capacity(self.graph_lengths)

    def _forward_backward(self, x, spk, labels):
        from .track_mm.dagerc import _speaker_ids, speaker_count
        m = self.model
        B, Lmax = self.lengths.numel(), self.Lmax
        if tuple(x.shape[:2]) != (B, Lmax) or tuple(labels.shape) != (B, Lmax):
            raise ValueError("DagercTrainStep: input %s / labels %s, the step was built for [%d, %d]"
                             % (tuple(x.shape), tuple(labels.shape), B, Lmax))
        n_spk = speaker_count(spk)
        # every relation id the speakers can form: K1 then takes the relation slots from the host, not from its census
        g = build_graph(self.graph_lengths_dev, _speaker_ids(spk), 0, 0, n_spk, device=self.dev, reference_layout=False,
                        mean_weight=False, sizes=self.sizes, relation_ids=relation_ids_for_speakers(range(n_spk), n_spk))
        dag = ops_dagerc.DagStructure(g, self.graph_lengths, m.windowp, e_cap=self.e_cap, order=self.order)
        logits, _ = m(x, self.lengths, spk, graph=g, dag=dag)
        loss = ops.cross_entropy(logits.reshape(B * Lmax, -1), labels.reshape(-1),
                                 reduce_sync=self.reduce_main if self.world > 1 else None)
        self._backward(loss)
        self._last_graph = g
        return loss

    def _late_params(self):
        return self.model.fc1.weight, self.model.fc1.bias

    def _check_inputs(self):
        self._last_graph.check_inputs()

    def global_loss(self):
        """Global mean loss of the last step (eager or replayed)."""
        return self._last_loss
