import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    def load(name):
        # a fixture too large for one file keeps its gradients in <name>_grads.npz
        fx = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
        grads = os.path.join(GOLDEN, name + "_grads.npz")
        if os.path.isfile(grads):
            fx.update(np.load(grads))
        return fx
    return load


def rel_err(a, b, floor=1e-30):
    """max-norm relative error per tensor (SURVEY.md 8c parity mode).

    ``floor`` guards tensors that are mathematically zero (e.g. the gradient of a bias that feeds a
    train-mode BatchNorm, or of lin_key.bias under a softmax): there both sides are ~1e-11 noise.
    """
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    if hasattr(b, "detach"):
        b = b.detach().cpu().numpy()
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.size == 0:
        return 0.0
    den = max(np.abs(b).max(), floor)
    return float(np.abs(a - b).max() / den)


def check_grads(got, want, tol):
    """Every live gradient within ``tol`` relative (max-norm per tensor); tensors whose true value is
    zero are compared against 1e-2 x the largest gradient in the model instead of their own noise."""
    assert set(got) == set(want), (sorted(set(got) ^ set(want)))
    scale = max(float(np.abs(np.asarray(v)).max()) for v in want.values())
    worst = 0.0
    for k in want:
        e = rel_err(got[k], want[k], floor=1e-2 * scale)
        assert e < tol, (k, e)
        worst = max(worst, e)
    return worst


# ------------------------------------------------------------------------------------------ fp64-backed parity bars
# north_star asks for 1e-5 relative (max-norm per tensor) in fp32.  Wherever a bar above 1e-5 is used, it has to be
# backed by data: the same computation in fp64 (the oracle with .double()) is the truth, and the CUDA result may be
# no further from it than the reference's own fp32 result is (x PARITY_SLACK) -- i.e. the gap is fp32 reassociation
# noise of the reference itself, not an error of the kernels.  Every comparison is recorded (worst error per tensor)
# in gpurun_out/parity_r02.jsonl; a summary is committed under profiles/.
PARITY_TOL = 1e-5
# The tcgen05 GEMMs compute a split product (tf32 hi*hi + two bf16 correction terms, DESIGN.md section 5): 2^-20 per element
# where an exact-fp32 FFMA chain has 2^-24.  Both are far inside 1e-5 for ordinary tensors (see the recorded e_cuda_vs_fp64:
# 1e-6 .. 3e-6), but a few gradients are sums with heavy cancellation -- a bias upstream of a train-mode BatchNorm only
# acts through second-order paths -- and there EVERY fp32 implementation loses digits: the reference's own fp32 result is
# 5e-6 .. 1e-5 from the fp64 truth.  For those the bar is "within PARITY_SLACK x the fp32 reference's own distance".
PARITY_SLACK = 4.0
_PARITY_LOG = os.path.join(ROOT, "gpurun_out", "parity_r02.jsonl")


def _np64(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.asarray(a, dtype=np.float64)


def parity_check(case, got, ref32, ref64=None, tol=PARITY_TOL, zero_floor_frac=1e-2, slack=PARITY_SLACK):
    """got / ref32 / ref64: {name: array}.  Per tensor:
         e_ref   = |got - ref32| / max|ref32|            (what round 1 asserted)
         e_cuda  = |got - ref64| / max|ref64|,  e_f32 = |ref32 - ref64| / max|ref64|   (when ref64 is given)
       pass iff  e_ref <= tol                      (the north_star bar), or
                 e_cuda <= max(tol, slack * e_f32)   (no further from the fp64 truth than the fp32 reference is).
       Tensors that are mathematically zero are measured against ``zero_floor_frac`` x the largest tensor of the dict.
       Returns the list of records (also appended to gpurun_out/parity_r02.jsonl)."""
    import json
    assert set(got) == set(ref32), sorted(set(got) ^ set(ref32))
    scale = max(float(np.abs(_np64(v)).max()) for v in ref32.values()) if ref32 else 1.0
    floor = zero_floor_frac * scale
    recs, bad = [], []
    for k in sorted(ref32):
        g, r32 = _np64(got[k]), _np64(ref32[k])
        assert g.shape == r32.shape, (k, g.shape, r32.shape)
        rec = {"case": case, "tensor": k, "numel": int(g.size), "e_vs_ref32": rel_err(g, r32, floor=floor)}
        ok = rec["e_vs_ref32"] <= tol
        if ref64 is not None:
            r64 = _np64(ref64[k])
            rec["e_cuda_vs_fp64"] = rel_err(g, r64, floor=floor)
            rec["e_ref32_vs_fp64"] = rel_err(r32, r64, floor=floor)
            ok = ok or rec["e_cuda_vs_fp64"] <= max(tol, slack * rec["e_ref32_vs_fp64"])
        rec["ok"] = bool(ok)
        recs.append(rec)
        if not ok:
            bad.append(rec)
    try:
        os.makedirs(os.path.dirname(_PARITY_LOG), exist_ok=True)
        with open(_PARITY_LOG, "a") as f:
            for r in recs:
                f.write(json.dumps(r) + "\n")
    except OSError:
        pass
    assert not bad, bad
    return recs


def grads_of(module):
    return {k: p.grad.detach().cpu().numpy() for k, p in module.named_parameters() if p.grad is not None}
