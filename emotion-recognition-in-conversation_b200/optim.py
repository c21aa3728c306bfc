"""Optimizer tail of the train steps (SURVEY.md 8f-3): Adam / AdamW (+ clip_grad_norm_) over ONE flat buffer.

  torch.optim.Adam(lr=1e-4, weight_decay=1e-8)          track_mm/cogmen.py:50,187-189; dgcn.py:41; mmgcn.py:34
  torch.optim.AdamW(...) + clip_grad_norm_(params, 5)    track_mm/dagerc.py:39,229-231

``FlatAdam`` keeps every LIVE parameter (one that actually receives a gradient: the reference modules carry dead ones,
SURVEY.md Appendix B) as a view into one flat fp32 buffer, with flat twins for the gradient and both moments.  A step is
  gather the per-parameter gradients into the flat gradient buffer  (one multi-tensor copy)
  [data-parallel: all-reduce that buffer -- erc_b200.dist]
  [clip: ercg_sumsq]
  ercg_adam_step                                          (ONE kernel for all parameters, step counter on the device)
so nothing in it needs host arithmetic and the whole train step can be captured in a CUDA graph.

Checkpoints: ``state_dict()`` is the flat form (the whole buffers); ``torch_state_dict()`` is torch.optim's per-parameter
form, which ``torch.optim.Adam.load_state_dict`` reads; ``load_state_dict()`` takes either.
"""
import torch

from ._lib import lib, check
from .ops import _p, _stream, _ws


ALIGN = 64      # every parameter starts on a 256-byte boundary of the flat buffers: the kernels read weights / biases as
                # float4 and through TMA


def _slot(numel):
    return (numel + ALIGN - 1) // ALIGN * ALIGN


def _step_tensor(step):
    """torch.optim's Adam 'step': a CPU scalar of the default float type (float64 only when that is the default)."""
    return torch.tensor(float(step), dtype=torch.float64 if torch.get_default_dtype() == torch.float64 else torch.float32)


class FlatAdam:
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, decoupled=False, max_norm=None,
                 extra_slots=0):
        """decoupled=False: torch.optim.Adam semantics (L2 term added to the gradient); True: torch.optim.AdamW.
        max_norm: clip_grad_norm_(params, max_norm) before the update (global L2 norm over the live gradients).
        extra_slots: floats appended to the flat GRADIENT buffer that ride along with the gradient all-reduce (loss
        numerators ...); they are not parameters and are not updated."""
        self.params = [p for p in params]
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        self.decoupled, self.max_norm, self.extra_slots = bool(decoupled), max_norm, int(extra_slots)
        self.live = None
        self.flat_p = self.flat_g = self.m = self.v = self.step_dev = None
        self.grad_scale = 1.0
        # device address of an int (a PeerComm's status word): when set, update() runs ercg_adam_step_guarded, which leaves
        # p, m, v and the step counter untouched while that int is non-zero
        self.skip_if_nonzero = None
        self._index = {id(p): i for i, p in enumerate(self.params)}
        self._pending = None            # state loaded before attach(): ("torch", {param index: state}) or ("flat", sd)
        self._names = None              # parameter names for error messages (from load_state_dict)

    # ---- one-time layout, decided after the first backward (only then is it known which parameters are live)
    def attach(self, order=None):
        live = [p for p in self.params if p.grad is not None]
        if not live:
            raise RuntimeError("FlatAdam.attach: no parameter has a gradient yet (call it after the first backward)")
        if order is not None:
            live = sorted(live, key=order)            # stable: lets a caller put early-available gradients first
        dev = live[0].device
        n = sum(_slot(p.numel()) for p in live)
        self.n = n
        self.flat_p = torch.zeros(n, dtype=torch.float32, device=dev)     # padding stays 0 under Adam (g = 0, p = 0)
        self.flat_g = torch.zeros(n + self.extra_slots, dtype=torch.float32, device=dev)
        self.m = torch.zeros(n, dtype=torch.float32, device=dev)
        self.v = torch.zeros(n, dtype=torch.float32, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self._sumsq = torch.zeros(1, dtype=torch.float32, device=dev)
        # the kernels need a CUDA device; on CPU tensors only the layout and the state conversion are usable
        self._sumsq_ws = _ws(lib().ercg_sumsq_workspace_bytes(n), dev) if dev.type == "cuda" else None
        self.offsets, self.g_views, off = [], [], 0
        with torch.no_grad():
            for p in live:
                k = p.numel()
                view = self.flat_p[off:off + k].view_as(p)
                view.copy_(p.data)
                p.data = view                          # the parameter now LIVES in the flat buffer (same Parameter object)
                self.g_views.append(self.flat_g[off:off + k].view_as(p))
                self.offsets.append(off)
                off += _slot(k)
        self.live = live
        self._live_ids = {id(p) for p in live}
        if self._pending is not None:                  # state loaded before the live set was known
            pending, self._pending = self._pending, None
            self._apply(*pending)
        return self

    def flat_bytes(self):
        """Bytes of the flat gradient buffer if every parameter were live: an upper bound known before the first backward
        (what a communicator that all-reduces that buffer has to hold)."""
        return 4 * (sum(_slot(p.numel()) for p in self.params) + self.extra_slots)

    @property
    def extra(self):
        """The ride-along slots at the tail of the flat gradient buffer."""
        return self.flat_g[self.n:]

    def gather(self, lo=0, hi=None):
        """Copy the gradients of live[lo:hi] into the flat gradient buffer (one multi-tensor copy launch)."""
        ps = self.live[lo:hi]
        grads = []
        for p in ps:
            if p.grad is None:
                raise RuntimeError("FlatAdam: a live parameter has no gradient in this step")
            grads.append(p.grad)
        torch._foreach_copy_(self.g_views[lo:hi], grads)

    def span(self, lo=0, hi=None):
        """Flat-gradient slice covering live[lo:hi] (for bucketed all-reduces)."""
        hi = len(self.live) if hi is None else hi
        a = self.offsets[lo] if lo < len(self.live) else self.n
        b = self.offsets[hi] if hi < len(self.live) else self.n
        return self.flat_g[a:b]

    def update(self):
        """clip (optional) + ONE Adam kernel over the flat buffers; bumps the device step counter."""
        sumsq = None
        if self.max_norm is not None:
            check(lib().ercg_sumsq(_p(self.flat_g), self.n, _p(self._sumsq), _p(self._sumsq_ws), self._sumsq_ws.numel(), _stream()),
                  "ercg_sumsq")
            sumsq = self._sumsq
        args = (_p(self.flat_p), _p(self.flat_g), _p(self.m), _p(self.v), self.n, self.lr, self.betas[0], self.betas[1], self.eps,
                self.weight_decay, 1 if self.decoupled else 0, float(self.grad_scale), _p(sumsq),
                float(self.max_norm if self.max_norm is not None else 0.0), _p(self.step_dev), _stream())
        if self.skip_if_nonzero is None:
            check(lib().ercg_adam_step(*args), "ercg_adam_step")
        else:
            check(lib().ercg_adam_step_guarded(*args, self.skip_if_nonzero), "ercg_adam_step_guarded")

    def step(self, allreduce=None):
        """gather -> [allreduce(flat gradient buffer)] -> update.  ``allreduce``: callable taking the flat tensor."""
        if self.live is None:
            self.attach()
        self.gather()
        if allreduce is not None:
            allreduce(self.flat_g)
        self.update()

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    def grad_norm(self):
        """Global L2 norm of the flat gradient buffer (device scalar; the value clip_grad_norm_ returns)."""
        check(lib().ercg_sumsq(_p(self.flat_g), self.n, _p(self._sumsq), _p(self._sumsq_ws), self._sumsq_ws.numel(), _stream()),
              "ercg_sumsq")
        return self._sumsq.sqrt() * self.grad_scale

    def state_dict(self):
        return {"step": int(self.step_dev.item()) if self.step_dev is not None else 0,
                "exp_avg": None if self.m is None else self.m.clone(), "exp_avg_sq": None if self.v is None else self.v.clone(),
                "hyper": dict(lr=self.lr, betas=self.betas, eps=self.eps, weight_decay=self.weight_decay, decoupled=self.decoupled,
                              max_norm=self.max_norm)}

    # ---- torch.optim's checkpoint form
    def torch_state_dict(self, names=None):
        """What torch.optim.Adam (AdamW when decoupled) returns from state_dict() for ``self.params``: state[i] =
        {'step', 'exp_avg', 'exp_avg_sq'} in parameter i's shape for every live parameter and none for the others, as
        torch gives none to a parameter that never had a gradient; the padding of the flat buffers is not exported.
        ``names`` (one per parameter) become the group's 'param_names'."""
        if names is not None and len(names) != len(self.params):
            raise ValueError("FlatAdam.torch_state_dict: %d names for %d parameters" % (len(names), len(self.params)))
        cls = torch.optim.AdamW if self.decoupled else torch.optim.Adam
        opt = cls(self.params if names is None else list(zip(names, self.params)), lr=self.lr, betas=self.betas, eps=self.eps,
                  weight_decay=self.weight_decay)
        for i, st in sorted(self._per_param_state().items()):
            opt.state[self.params[i]] = st
        return opt.state_dict()

    def _per_param_state(self):
        if self.live is None:
            if self._pending is None:
                return {}
            if self._pending[0] != "torch":
                raise RuntimeError("FlatAdam: a flat-form state loaded before attach() has no per-parameter form yet")
            return {i: dict(st) for i, st in self._pending[1].items()}
        step = int(self.step_dev.item())
        if step == 0:
            return {}
        out = {}
        for p, off in zip(self.live, self.offsets):
            k = p.numel()
            out[self._index[id(p)]] = {"step": _step_tensor(step), "exp_avg": self.m[off:off + k].view_as(p).clone(),
                                       "exp_avg_sq": self.v[off:off + k].view_as(p).clone()}
        return out

    def load_state_dict(self, sd, names=None):
        """Load a torch.optim Adam / AdamW state_dict (``torch_state_dict`` form) or a flat-form ``state_dict()``.
        Before attach() the state is kept and applied inside attach(), the first point where the live parameters and
        their offsets are known; after attach() it is applied at once.  A torch-form state is matched by the group's
        'param_names' when it has them and ``names`` (one per parameter of this optimizer) is given, else by index.
        Hyper-parameters come from the state, as in torch.optim; max_norm, grad_scale, extra_slots and skip_if_nonzero
        are not optimizer state and keep their values.  Raises ValueError, naming the parameters, when a parameter has
        state but receives no gradient, receives a gradient but has no state (unless none has state), a shape differs or
        the step is not the same for all parameters."""
        if names is not None and len(names) != len(self.params):
            raise ValueError("FlatAdam.load_state_dict: %d names for %d parameters" % (len(names), len(self.params)))
        if "param_groups" in sd:
            pending = ("torch", self._resolve_torch(sd, names))
            g = sd["param_groups"][0]
            hyper = dict(lr=g["lr"], betas=g["betas"], eps=g["eps"], weight_decay=g["weight_decay"],
                         decoupled=g.get("decoupled_weight_decay", self.decoupled))
        else:
            pending = ("flat", sd)
            hyper = sd["hyper"]
            self._names = list(names) if names is not None else None
        self.lr, self.betas, self.eps = float(hyper["lr"]), (float(hyper["betas"][0]), float(hyper["betas"][1])), float(hyper["eps"])
        self.weight_decay, self.decoupled = float(hyper["weight_decay"]), bool(hyper["decoupled"])
        if self.live is None:
            self._pending = pending
        else:
            self._pending = None
            self._apply(*pending)

    def _name(self, i):
        return self._names[i] if self._names is not None else "parameter %d" % i

    def _resolve_torch(self, sd, names):
        """torch-form state -> {index into self.params: {'step': int, 'exp_avg', 'exp_avg_sq'}} (names and shapes checked)."""
        groups = sd["param_groups"]
        if len(groups) != 1:
            raise ValueError("FlatAdam keeps one parameter group; the state has %d" % len(groups))
        g = groups[0]
        if g.get("amsgrad") or g.get("maximize"):
            raise ValueError("FlatAdam implements neither amsgrad nor maximize; the state uses them")
        ids, saved = list(g["params"]), g.get("param_names")
        if saved is not None and names is not None:
            where = {n: i for i, n in enumerate(names)}
            idx = [where.get(n) for n in saved]       # None: not a parameter of this optimizer
        else:
            if len(ids) != len(self.params):
                raise ValueError("FlatAdam.load_state_dict: the state's group has %d parameters, this optimizer %d"
                                 % (len(ids), len(self.params)))
            idx = list(range(len(ids)))
        self._names = list(names) if names is not None else (list(saved) if saved is not None else None)
        out, stray, bad_shape, steps = {}, [], [], {}
        for j, sid in enumerate(ids):
            st = sd["state"].get(sid)
            if st is None:
                continue
            i = idx[j]
            if i is None:
                stray.append(saved[j])
                continue
            shape = tuple(self.params[i].shape)
            for key in ("exp_avg", "exp_avg_sq"):
                if tuple(st[key].shape) != shape:
                    bad_shape.append("%s: %s %s, parameter %s" % (self._name(i), key, tuple(st[key].shape), shape))
            steps[self._name(i)] = int(float(st["step"]))
            # the step as a new tensor: torch.optim steps the loaded one in place when it shares this state dict
            out[i] = {"step": _step_tensor(steps[self._name(i)]), "exp_avg": st["exp_avg"], "exp_avg_sq": st["exp_avg_sq"]}
        if stray:
            raise ValueError("FlatAdam.load_state_dict: state for parameters this optimizer does not have: %s" % ", ".join(stray))
        if bad_shape:
            raise ValueError("FlatAdam.load_state_dict: shapes differ: %s" % "; ".join(bad_shape))
        if len(set(steps.values())) > 1:
            raise ValueError("FlatAdam.load_state_dict: the step differs between parameters (FlatAdam keeps one counter): %s"
                             % ", ".join("%s=%d" % kv for kv in steps.items()))
        return out

    def _apply(self, kind, payload):
        """Copy a loaded state into the flat buffers (after attach())."""
        if kind == "flat":
            if payload["exp_avg"] is None:
                self.m.zero_()
                self.v.zero_()
            else:
                if payload["exp_avg"].numel() != self.n or payload["exp_avg_sq"].numel() != self.n:
                    raise ValueError("FlatAdam.load_state_dict: the flat state holds %d floats, this layout %d"
                                     % (payload["exp_avg"].numel(), self.n))
                self.m.copy_(payload["exp_avg"])
                self.v.copy_(payload["exp_avg_sq"])
            self.step_dev.fill_(int(payload["step"]))
            return
        state = payload
        live = [self._index[id(p)] for p in self.live]
        not_live = sorted(set(state) - set(live))
        if not_live:
            raise ValueError("FlatAdam.load_state_dict: state for parameters that receive no gradient: %s"
                             % ", ".join(self._name(i) for i in not_live))
        no_state = [i for i in live if i not in state]
        if state and no_state:
            raise ValueError("FlatAdam.load_state_dict: no state for parameters that receive a gradient: %s"
                             % ", ".join(self._name(i) for i in no_state))
        self.m.zero_()
        self.v.zero_()
        step = 0
        for i, off in zip(live, self.offsets):
            if i in state:
                k = self.params[i].numel()
                self.m[off:off + k].copy_(state[i]["exp_avg"].reshape(-1))
                self.v[off:off + k].copy_(state[i]["exp_avg_sq"].reshape(-1))
                step = int(float(state[i]["step"]))
        self.step_dev.fill_(step)
