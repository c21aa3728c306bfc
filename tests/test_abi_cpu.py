"""C-ABI checks that need no GPU: libercgraph.so loads, exports every function include/ercgraph.h declares, the ctypes
table of the host layer mirrors the header one to one (names and argument counts), and the host-only entry points
(error strings, closed-form graph sizes, workspace sizes) answer like the numpy oracle / the reference's edge_perms."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import graph_np

HEADER = os.path.join(ROOT, "include", "ercgraph.h")


def _declared():
    """{function name: number of parameters} parsed from the header (prototypes only, typedef'd structs skipped)."""
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//[^\n]*", " ", src)
    src = re.sub(r"typedef\s+struct[^{]*\{.*?\}\s*\w+\s*;", " ", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(?:int|int64_t|size_t|const\s+char\s*\*|unsigned\s+long\s+long)\s+(ercg_\w+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
    return out


def test_header_declares_the_expected_surface():
    d = _declared()
    for name in ("ercg_graphify_csr", "ercg_gemm_nn_tc", "ercg_gemm_tn_tc", "ercg_gather_fwd", "ercg_gather_bwd",
                 "ercg_attn_window_fwd", "ercg_edgeatt_fwd", "ercg_bn_act_fwd", "ercg_ce_fwd", "ercg_lstm_fwd",
                 "ercg_dag_layer_fwd", "ercg_strerror"):
        assert name in d, name
    assert len(d) >= 50


def test_library_exports_every_declared_symbol():
    import erc_b200
    from erc_b200 import _lib
    assert os.path.isfile(_lib.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    handle = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in _declared() if not hasattr(handle, n)]
    assert not missing, missing


def test_ctypes_table_mirrors_the_header():
    import erc_b200
    from erc_b200 import _lib
    d = _declared()
    assert set(_lib.SIGNATURES) == set(d), sorted(set(_lib.SIGNATURES) ^ set(d))
    bad = {n: (len(a), d[n]) for n, (_, a) in _lib.SIGNATURES.items() if len(a) != d[n]}
    assert not bad, bad
    fields = [f for f, _ in _lib.GraphOut._fields_]
    src = open(HEADER).read()
    body = re.search(r"typedef struct ercg_graph_out \{(.*?)\} ercg_graph_out;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", " ", body, flags=re.S)
    assert fields == re.findall(r"\*\s*(\w+)\s*;", body)


def test_launch_setup_only_in_common_cuh():
    """Shared-memory limits, residency queries and cluster / cooperative launches go through the helpers of
    csrc/common.cuh, so every kernel sets them up once per device, clears the error of a failed launch and counts it."""
    csrc = os.path.join(ROOT, "emotion-recognition-in-conversation_b200", "csrc")
    setup = re.compile(r"\b(cudaFuncSetAttribute|cudaOccupancyMaxActiveBlocksPerMultiprocessor|cudaOccupancyMaxActiveClusters|"
                       r"cudaLaunchKernelEx|cudaLaunchCooperativeKernel)\b|\[\s*kMaxDevices\s*\]")
    found = {}
    for name in sorted(os.listdir(csrc)):
        if not name.endswith((".cu", ".cuh")):
            continue
        src = open(os.path.join(csrc, name)).read()
        src = re.sub(r"//[^\n]*", " ", re.sub(r"/\*.*?\*/", " ", src, flags=re.S))
        found[name] = {m.group(0) for m in setup.finditer(src)}
    assert found["common.cuh"] >= {"cudaFuncSetAttribute", "cudaOccupancyMaxActiveClusters", "cudaLaunchKernelEx"}
    assert not {n: sorted(f) for n, f in found.items() if f and n != "common.cuh"}


def test_host_only_entry_points():
    import erc_b200
    from erc_b200 import _lib
    from erc_b200.graph import graph_sizes
    lib = _lib.lib()
    assert lib.ercg_version() > 0
    assert lib.ercg_strerror(0) and lib.ercg_strerror(-1) and lib.ercg_strerror(-12345)
    rng = np.random.default_rng(0)
    for wp, wf in ((5, 5), (10, 10), (-1, -1), (0, 3), (200, 1)):
        lengths = rng.integers(1, 111, size=40)
        spk = np.zeros((40, int(lengths.max())), dtype=np.int64)
        b = graph_np.batch_graphify_np(lengths, spk, wp, wf, 1)
        assert graph_sizes(torch.as_tensor(lengths), wp, wf) == (b["N"], b["E"])
    assert graph_sizes(torch.zeros(0, dtype=torch.int64), 5, 5) == (0, 0)
    assert lib.ercg_gemm_nn_tc_workspace_bytes(100, 1443) >= 2 * 100 * 1444 * 4
    assert lib.ercg_graphify_workspace_bytes(1000) >= 4 * 2 * 8


def test_edge_perms_matches_closed_form():
    """edge_perms keeps the reference's python signature and runs on the host (cogmen_utils.py:147-172)."""
    import erc_b200
    from erc_b200.track_mm.cogmen_utils import edge_perms
    for L, wp, wf in ((1, 5, 5), (7, 5, 5), (30, 10, 10), (12, -1, -1), (9, -1, 2), (9, 3, -1), (5, 0, 0)):
        got = sorted(edge_perms(L, wp, wf))
        P = L - 1 if wp < 0 else wp
        F = L - 1 if wf < 0 else wf
        want = sorted((j, k) for j in range(L) for k in range(max(0, j - P), min(L - 1, j + F) + 1))
        assert got == want, (L, wp, wf)
