"""ctypes binding of libercgraph.so (include/ercgraph.h).

The library is the product: there is NO fallback.  If the shared object is missing or a call
returns an error code this module raises -- it never routes to PyTorch or CPU code.
PyTorch is used only for device memory, streams and autograd bookkeeping around these calls.
"""
import ctypes
import os
from ctypes import c_int, c_int64, c_uint64, c_float, c_double, c_void_p, c_size_t, c_char_p, POINTER, Structure

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ERCG_LIB_PATH") or os.path.join(_HERE, "libercgraph.so")   # override: A/B kernel experiments only

ACT_NONE, ACT_RELU, ACT_RELU_DROPOUT, ACT_MASK_POS = 0, 1, 2, 3


class ErcgError(RuntimeError):
    pass


class GraphOut(Structure):
    _fields_ = [(n, c_void_p) for n in (
        "node_off", "edge_off", "rowptr", "col", "etype", "t_rowptr", "t_col", "t_etype", "t_eid", "spk",
        "node_dlg", "inv_cnt", "edge_index", "edge_type", "edge_index_lengths", "totals", "pad_row", "rel_info")]


class DagLayer(Structure):
    """ercg_dag_layer (include/ercgraph.h)."""
    _fields_ = ([(n, c_int) for n in ("B", "D", "Tmax", "reserved")] +
                [(n, c_void_p) for n in ("node_off", "order", "spk", "lo", "eoff", "wk", "Wr0", "Wr1", "Whh_c", "bhh_c",
                                         "Wih_p", "bih_p", "Hin", "pre", "H1", "a", "S", "M", "alpha", "gc", "hnc", "gp",
                                         "dH1", "dpre", "dGseq", "dM", "dS", "dHdir", "ga")])


class DialogueRnnArgs(Structure):
    """ercg_dialogue_rnn (include/ercgraph.h)."""
    _fields_ = ([(n, c_int) for n in ("L", "B", "Dg", "Dp", "De", "P")] + [("drop_p", c_float), ("reserved", c_int)] +
                [(n, c_uint64) for n in ("seed_g", "seed_q", "seed_e")] +
                [("qmask", c_void_p), ("pre", c_void_p), ("ldpre", c_int64), ("xq", c_void_p), ("ldxq", c_int64)] +
                [(n, c_void_p) for n in ("Wgq", "Whh_g", "bhh_g", "Wpc", "Whh_p", "bhh_p", "Wih_e", "Whh_e", "bih_e", "bhh_e",
                                         "e", "g", "c", "qprev", "qcur", "gates_g", "gates_p", "gates_e", "alpha", "qstate",
                                         "de", "dpre")] + [("lddpre", c_int64), ("dxq", c_void_p), ("lddxq", c_int64)] +
                [(n, c_void_p) for n in ("dgh", "dph", "dei", "deh", "dG", "dQ", "dEh", "dc")])


P, I, L, F, D, U64, SZ = c_void_p, c_int, c_int64, c_float, c_double, c_uint64, c_size_t

# name -> (restype, argtypes); mirrors include/ercgraph.h one to one
SIGNATURES = {
    "ercg_strerror": (c_char_p, [I]),
    "ercg_version": (I, []),
    "ercg_launch_count": (ctypes.c_ulonglong, []),
    "ercg_graphify_sizes_host": (I, [P, I, I, I, POINTER(L), POINTER(L)]),
    "ercg_graphify_count": (I, [P, I, I, I, I, P, P]),
    "ercg_graphify_workspace_bytes": (SZ, [I]),
    "ercg_graphify_csr": (I, [P, I, I, P, I, L, I, I, I, L, L, POINTER(GraphOut), P, SZ, P]),
    "ercg_graphify_check_census": (I, [P, I, P, P]),
    "ercg_collate_masks": (I, [P, P, I, L, I, I, P, P, P, P]),
    "ercg_pack_rows": (I, [P, L, L, I, I, P, P, P, L, L, I, P]),
    "ercg_unpack_rows": (I, [P, L, P, P, P, L, L, I, I, L, I, P]),
    "ercg_gemm_nn": (I, [P, L, P, P, L, P, P, L, L, I, I, I, P, L, F, F, U64, P, P]),
    "ercg_gemm_nn_tc_workspace_bytes": (SZ, [I, I]),
    "ercg_gemm_nn_tc_supported": (I, [P, L, P, L, L, I, I]),
    "ercg_gemm_nn_tc": (I, [P, L, P, L, P, P, L, L, I, I, I, P, L, F, F, U64, P, P, P, SZ, P]),
    "ercg_gemm_nn_tc_trace": (I, [P]),
    "ercg_gemm_tn_workspace_bytes": (SZ, [L, I, I]),
    "ercg_gemm_tn": (I, [P, L, P, P, L, P, L, L, I, I, P, SZ, P]),
    "ercg_gemm_tn_tc_workspace_bytes": (SZ, [L, I, I]),
    "ercg_gemm_tn_tc_supported": (I, [P, L, P, L, L, I, I]),
    "ercg_gemm_tn_tc": (I, [P, L, P, L, P, L, L, I, I, P, SZ, P]),
    "ercg_gemm_bf16a_supported": (I, [P, L, L, I]),
    "ercg_gemm_nn_tc_bf16a": (I, [P, L, P, L, P, P, L, L, I, I, P, SZ, P]),
    "ercg_gemm_tn_tc_bf16a": (I, [P, L, P, L, P, L, L, I, I, P, SZ, P]),
    "ercg_cls_tail_bwd_workspace_bytes": (SZ, [I, I]),
    "ercg_cls_tail_bwd": (I, [P, L, P, P, F, P, L, P, P, P, L, I, I, P, SZ, P]),
    "ercg_mask_pos": (I, [P, L, P, L, F, P, L, L, I, P]),
    "ercg_colsum_workspace_bytes": (SZ, [L, I]),
    "ercg_colsum": (I, [P, L, L, I, P, P, SZ, P]),
    "ercg_gather_fwd": (I, [P, L, P, P, P, P, P, I, P, P, L, L, I, P]),
    "ercg_gather_bwd": (I, [P, L, P, L, P, P, P, P, P, P, I, I, P, L, P, L, I, P]),
    "ercg_gather_window_bwd": (I, [P, L, P, P, P, P, P, P, I, I, P, L, L, I, I, I, P]),
    "ercg_attn_fwd": (I, [P, P, P, P, L, P, P, F, P, L, P, P, L, I, P]),
    "ercg_attn_bwd_dst": (I, [P, L, P, P, L, P, P, P, F, P, P, L, P, P, L, I, P]),
    "ercg_attn_bwd_src": (I, [P, L, P, L, P, P, P, P, P, F, P, P, L, L, I, P]),
    "ercg_attn_window_supported": (I, [I, I, I]),
    "ercg_attn_window_fwd": (I, [P, P, P, P, L, P, P, F, P, L, P, L, I, I, I, P]),
    "ercg_attn_window_tiles": (L, [L]),
    "ercg_attn_window_bwd_dst": (I, [P, L, P, P, L, P, P, P, F, P, P, L, P, P, L, I, I, I, P]),
    "ercg_attn_window_bwd_src": (I, [P, L, P, L, P, P, P, P, P, F, P, P, L, P, L, I, I, I, P]),
    "ercg_edgeatt_fwd": (I, [P, L, P, L, P, P, P, P, L, I, P]),
    "ercg_edgeatt_bwd_src": (I, [P, P, P, L, P, P, P, P, P, L, L, I, P]),
    "ercg_edgeatt_bwd_dst": (I, [P, P, L, P, P, P, L, L, I, P]),
    "ercg_lstm_fwd": (I, [P, L, P, P, I, I, P, L, P, P, P, P]),
    "ercg_lstm_bwd": (I, [P, L, P, P, P, P, I, I, P, L, P]),
    "ercg_dropout": (I, [P, P, L, F, U64, P]),
    "ercg_dropout_dev": (I, [P, P, L, F, U64, P, P]),
    "ercg_gru_fwd": (I, [P, L, P, P, P, I, I, P, L, P, P, P]),
    "ercg_gru_bwd": (I, [P, L, P, P, P, P, I, I, P, L, P, L, P]),
    "ercg_bn_workspace_bytes": (SZ, [L, I]),
    "ercg_bn_stats": (I, [P, L, L, I, P, P, P, SZ, P]),
    "ercg_bn_running_update": (I, [P, P, P, P, P, F, F, I, P]),
    "ercg_bn_sync_pack": (I, [P, P, D, I, P, P]),
    "ercg_bn_sync_unpack": (I, [P, I, P, P, P]),
    "ercg_bn_act_fwd": (I, [P, L, P, P, F, P, P, F, P, L, L, I, P]),
    "ercg_bn_act_bwd_reduce": (I, [P, L, P, L, P, P, F, P, P, F, P, L, I, P, SZ, P]),
    "ercg_bn_act_bwd_apply": (I, [P, L, P, L, P, P, F, P, P, F, P, D, I, P, L, L, I, P]),
    "ercg_ce_workspace_bytes": (SZ, [L]),
    "ercg_ce_fwd": (I, [P, L, P, P, P, P, L, L, I, P, SZ, P]),
    "ercg_scale_by_ratio": (I, [P, L, P, P, P]),
    "ercg_sumsq_workspace_bytes": (SZ, [L]),
    "ercg_sumsq": (I, [P, L, P, P, SZ, P]),
    "ercg_adam_step": (I, [P, P, P, P, L, F, F, F, F, F, I, F, P, F, P, P]),
    "ercg_adam_step_guarded": (I, [P, P, P, P, L, F, F, F, F, F, I, F, P, F, P, P, P]),
    # peer-memory all-reduce (csrc/p2p.cu)
    "ercg_p2p_region_bytes": (SZ, [SZ]),
    "ercg_p2p_alloc": (I, [SZ, P, P]),
    "ercg_p2p_open": (I, [P, P]),
    "ercg_p2p_close": (I, [P]),
    "ercg_p2p_free": (I, [P]),
    "ercg_p2p_status": (I, [P, P]),
    "ercg_p2p_status_word": (I, [P, P]),
    "ercg_p2p_allreduce": (I, [P, I, I, P, P, L, I, SZ, P]),
    "ercg_p2p_bn_stats": (I, [P, I, I, P, L, L, I, D, P, P, P, P, P, F, P, SZ, SZ, P]),
    "ercg_p2p_bn_act_bwd_reduce": (I, [P, I, I, P, L, P, L, P, P, F, P, P, F, P, P, L, I, P, SZ, SZ, P]),
    # K7 / K8 (MMGCN)
    "ercg_mmgcn_block_offsets": (I, [P, I, P, P]),
    "ercg_mmgcn_adj_fwd": (I, [P, L, P, P, P, L, L, I, I, P, L, P, P, P, P, P]),
    "ercg_mmgcn_adj_bwd": (I, [P, P, P, P, L, P, P, P, P, L, L, I, I, P, P, L, P]),
    "ercg_mmgcn_spmm": (I, [P, I, P, L, P, L, P, P, P, L, L, I, I, P, L, P, L, P]),
    "ercg_mmgcn_sddmm": (I, [P, L, P, L, P, P, P, L, L, I, I, P, I, P]),
    "ercg_gcnii_layer_fwd": (I, [P, L, P, L, P, L, P, L, L, I, F, F, I, F, U64, P]),
    "ercg_gcnii_layer_fwd_dev": (I, [P, L, P, L, P, L, P, L, L, I, F, F, I, F, U64, P, P]),
    "ercg_gcnii_layer_bwd_input": (I, [P, L, P, L, P, L, L, I, F, F, P]),
    "ercg_node_rows": (I, [P, P, L, I, I, I, P, P]),
    "ercg_speaker_embed_add": (I, [P, L, P, I, P, P, L, P, L, P, P, L, I, P]),
    "ercg_relu_dropout": (I, [P, P, L, F, U64, P]),
    "ercg_relu_dropout_dev": (I, [P, P, L, F, U64, P, P]),
    "ercg_masked_edge_att_fwd": (I, [P, L, P, P, P, P, L, I, I, P, P, L, P]),
    "ercg_masked_edge_att_bwd": (I, [P, L, P, P, P, P, L, I, I, P, P, P, P, L, L, P]),
    # K9 / K10 (DAG-ERC)
    "ercg_dag_build_workspace_bytes": (SZ, [L]),
    "ercg_dag_build": (I, [P, P, P, L, I, P, P, P, P, P, SZ, P]),
    "ercg_dag_dense_masks": (I, [P, I, I, I, P, P, P]),
    "ercg_dag_layer_fwd": (I, [POINTER(DagLayer), P]),
    "ercg_dag_layer_bwd": (I, [POINTER(DagLayer), P]),
    "ercg_dag_gat_fwd": (I, [P, L, P, L, L, P, L, L, P, P, L, P, P, P, P, I, I, I, P]),
    "ercg_dag_gat_bwd": (I, [P, L, L, P, L, P, P, P, P, P, P, P, P, I, I, I, P]),
    # K12 (DialogueRNN)
    "ercg_dialogue_rnn_fwd": (I, [POINTER(DialogueRnnArgs), P]),
    "ercg_dialogue_rnn_bwd": (I, [POINTER(DialogueRnnArgs), P]),
    # K13 (dense masked MatchingAttention), the sequence reversal and log-softmax of the sequence classifiers
    "ercg_match_att_fwd": (I, [P, L, I, I, I, I, P, L, P, I, P, L, P, P, P]),
    "ercg_match_att_bwd": (I, [P, L, I, I, I, I, P, L, P, I, P, P, P, L, P, P, L, P, L, P]),
    "ercg_reverse_seq": (I, [P, L, I, I, I, P, P, L, I, P]),
    "ercg_log_softmax_fwd": (I, [P, L, P, L, L, I, P]),
    "ercg_log_softmax_bwd": (I, [P, L, P, L, P, L, L, I, P]),
}

_lib = None
_timer = None          # active KernelTimer or None


class KernelTimer:
    """Times every libercgraph call with CUDA events on the launching (current) stream.

    Used by bench.py to measure the per-kernel durations behind the roofline numbers live, inside the
    timed region.  ``with KernelTimer() as kt: ...; kt.summary()`` -> {entry point: (calls, total ms)}."""

    def __init__(self, labeler=None):
        self.records = []
        self.labeler = labeler        # optional (entry point, args) -> label, e.g. to split GEMMs by shape

    def __enter__(self):
        global _timer
        _timer = self
        return self

    def __exit__(self, *exc):
        global _timer
        _timer = None

    def summary(self):
        import torch
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self.records:
            c, t = out.get(name, (0, 0.0))
            out[name] = (c + 1, t + e0.elapsed_time(e1))
        return out


class _Timed:
    """Attribute proxy over the CDLL handle that brackets calls with events when a KernelTimer is active."""

    def __init__(self, handle):
        self._h = handle

    def __getattr__(self, name):
        fn = getattr(self._h, name)
        if name.endswith("_bytes") or name.endswith("_supported") or name.endswith("_tiles") or name in ("ercg_strerror", "ercg_version", "ercg_launch_count",
                                               "ercg_graphify_sizes_host", "ercg_p2p_alloc", "ercg_p2p_open", "ercg_p2p_close",
                                               "ercg_p2p_free", "ercg_p2p_status", "ercg_p2p_status_word"):
            setattr(self, name, fn)
            return fn

        def call(*args):
            t = _timer
            if t is None:
                return fn(*args)
            import torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*args)
            e1.record()
            t.records.append((t.labeler(name, args) if t.labeler else name, e0, e1))
            return rc

        setattr(self, name, call)
        return call


def lib():
    """The loaded library; raises ErcgError when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ErcgError(
                "libercgraph.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C %s`; there is no CPU/PyTorch fallback" % (LIB_PATH, os.path.join(_HERE, "csrc")))
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = _Timed(handle)
    return _lib


def check(rc, what):
    if rc != 0:
        raise ErcgError("%s failed: %s (%d)" % (what, lib().ercg_strerror(rc).decode(), rc))


def launch_count():
    return int(lib().ercg_launch_count())
