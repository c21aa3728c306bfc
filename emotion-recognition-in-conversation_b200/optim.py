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
"""
import torch

from ._lib import lib, check
from .ops import _p, _stream, _ws


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

    # ---- one-time layout, decided after the first backward (only then is it known which parameters are live)
    def attach(self, order=None):
        live = [p for p in self.params if p.grad is not None]
        if not live:
            raise RuntimeError("FlatAdam.attach: no parameter has a gradient yet (call it after the first backward)")
        if order is not None:
            live = sorted(live, key=order)            # stable: lets a caller put early-available gradients first
        dev = live[0].device
        ALIGN = 64                                     # every parameter starts on a 256-byte boundary of the flat buffers: the
        n = sum((p.numel() + ALIGN - 1) // ALIGN * ALIGN for p in live)    # kernels read weights / biases as float4 and through TMA
        self.n = n
        self.flat_p = torch.zeros(n, dtype=torch.float32, device=dev)     # padding stays 0 under Adam (g = 0, p = 0)
        self.flat_g = torch.zeros(n + self.extra_slots, dtype=torch.float32, device=dev)
        self.m = torch.zeros(n, dtype=torch.float32, device=dev)
        self.v = torch.zeros(n, dtype=torch.float32, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self._sumsq = torch.zeros(1, dtype=torch.float32, device=dev)
        self._sumsq_ws = _ws(lib().ercg_sumsq_workspace_bytes(n), dev)
        self.offsets, self.g_views, off = [], [], 0
        with torch.no_grad():
            for p in live:
                k = p.numel()
                view = self.flat_p[off:off + k].view_as(p)
                view.copy_(p.data)
                p.data = view                          # the parameter now LIVES in the flat buffer (same Parameter object)
                self.g_views.append(self.flat_g[off:off + k].view_as(p))
                self.offsets.append(off)
                off += (k + ALIGN - 1) // ALIGN * ALIGN
        self.live = live
        self._live_ids = {id(p) for p in live}
        return self

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
