"""bench.py pieces that do not need a GPU: the argument parser (its help text once crashed on a bare '%') and the labels the
per-kernel table and profiles/traffic.json are keyed by."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_help_prints_every_option():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-1000:]
    for opt in ("--gpus", "--steps", "--warmup", "--impl", "--scaling", "--transport", "--bn-sync", "--library-yardstick",
                "--dump-outputs"):
        assert opt in r.stdout, opt


def test_kernel_labels_match_the_traffic_table():
    b = _bench()
    # (A, lda, B, ldb, bias, C, ldc, M, N, K, ...)
    assert b.kernel_label("ercg_gemm_nn_tc", (0, 1444, 0, 100, 0, 0, 100, 1 << 20, 100, 1443)) == "gemm_nn_tc[K=1443,N=100]"
    # (A, lda, B, ldb, C, ldc, M, K1, N1, ...)
    assert b.kernel_label("ercg_gemm_tn_tc", (0, 1444, 0, 100, 0, 100, 1 << 20, 1443, 100)) == "gemm_tn_tc[K1=1443,N1=100]"
    assert b.kernel_label("ercg_attn_window_bwd_src", ()) == "attn_bwd_src"
    assert b.kernel_label("ercg_gather_window_bwd", ()) == "gather_bwd"
    assert b.kernel_label("ercg_p2p_allreduce", ()) == "p2p_allreduce"
    traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    for key in ("gemm_nn_tc[K=1443,N=100]", "gemm_tn_tc[K1=1443,N1=100]"):
        assert key in traffic, key


def test_dump_outputs_writes_one_npy_per_array_and_refuses_more_than_64_mb(tmp_path):
    import numpy as np
    import pytest
    b = _bench()
    arrays = {"loss": np.array([1.5], dtype=np.float32), "param.cls.0.weight": np.arange(6, dtype=np.float32).reshape(2, 3)}
    b.dump_outputs(str(tmp_path / "out"), arrays)
    assert sorted(os.listdir(tmp_path / "out")) == ["loss.npy", "param.cls.0.weight.npy"]
    for k, v in arrays.items():
        got = np.load(tmp_path / "out" / (k + ".npy"))
        assert got.dtype == v.dtype and np.array_equal(got, v)
    with pytest.raises(SystemExit):
        b.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(b.DUMP_LIMIT_BYTES // 4 + 1, dtype=np.float32)})
    assert not (tmp_path / "big").exists()


def test_dump_outputs_is_refused_where_no_train_step_is_timed(tmp_path):
    for extra in (["--impl", "reference"], ["--library-yardstick"], ["--profile-step"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "d")] + extra,
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr, (extra, r.stderr[-500:])
        assert not (tmp_path / "d").exists()
