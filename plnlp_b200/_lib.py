"""ctypes binding of the C-ABI library ``libplnlp_b200.so`` (see include/plnlp_b200.h).

This is the ONLY way the python package reaches the kernels: raw device pointers
(``tensor.data_ptr()``), int64 sizes and the current CUDA stream handle.  There is no
CPU fallback: if the shared library is missing, or a kernel is asked to run on
non-CUDA tensors, a ``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libplnlp_b200.so")

_P, _I, _L, _F, _U = c_void_p, c_int, c_int64, c_float, c_uint64

# name -> (restype, argtypes); mirrors include/plnlp_b200.h declaration by declaration
SIGNATURES = {
    "plnlp_abi_version": (c_int, []),
    "plnlp_check_device": (c_int, []),
    "plnlp_launch_count": (c_int64, []),
    "plnlp_spmm_csr_f32": (c_int, [_P, _P, _P, _L, _P, _P, _P, _P, _P, _P, _I, _F, _U, _P, _L, _L, _P, _L, _L, _P, _P, _P, _L, _P, _L, _F, _P]),
    "plnlp_spmm_csr_bf16": (c_int, [_P, _P, _P, _L, _P, _P, _P, _P, _P, _P, _I, _F, _U, _P, _L, _L, _P, _L, _L, _P, _P, _P, _L, _P, _L, _F, _P]),
    "plnlp_spmm_tune": (c_int, [_I, _I, _I, _I]),
    "plnlp_row_nonzero_index_f32": (c_int, [_P, _L, _L, _L, _P, _P]),
    "plnlp_gemm_f32": (c_int, [_I, _I, _L, _L, _L, _P, _L, _P, _L, _P, _L, _F, _P, _I, _P, _L, _F, _U, _P, _L, _I, _P]),
    "plnlp_gemm_tf32": (c_int, [_I, _I, _I, _L, _L, _L, _P, _L, _P, _L, _P, _L, _F, _P, _I, _P, _L, _F, _U, _P, _L, _I, _P]),
    "plnlp_gemm_tf32_2cta": (c_int, [_I, _I, _I, _L, _L, _L, _P, _L, _P, _L, _P, _L, _F, _P, _I, _P, _L, _F, _U, _P, _L, _I, _P]),
    "plnlp_gemm_tf32_tma_workspace_bytes": (c_int64, [_L, _L]),
    "plnlp_gemm_tf32_tma": (c_int, [_I, _I, _L, _L, _L, _P, _L, _P, _L, _P, _L, _F, _P, _I, _P, _L, _F, _U, _P, _L, _P]),
    "plnlp_gemm_tf32_tma_tn_workspace_bytes": (c_int64, []),
    "plnlp_gemm_tf32_tma_tn": (c_int, [_I, _L, _L, _L, _P, _L, _P, _L, _P, _L, _P, _L, _P]),
    "plnlp_edge_mlp_fwd_tf32": (c_int, [_I, _P, _L, _L, _P, _L, _L, _P, _L, _P, _L, _F, _U, _P, _P, _L, _P, _L, _P]),
    "plnlp_gather_hadamard_f32": (c_int, [_P, _L, _L, _P, _L, _L, _P, _L, _P]),
    "plnlp_segment_softmax_fwd_f32": (c_int, [_P, _L, _P, _F, _P, _P]),
    "plnlp_segment_softmax_bwd_f32": (c_int, [_P, _L, _P, _P, _F, _P, _P]),
    "plnlp_attn_score_csr_f32": (c_int, [_P, _P, _L, _P, _P, _L, _P, _L, _L, _P, _P]),
    "plnlp_gather_rows_f32": (c_int, [_P, _L, _L, _P, _L, _L, _L, _P, _L, _P]),
    "plnlp_row_scatter_sorted_f32": (c_int, [_P, _L, _L, _P, _L, _P, _P, _L, _P]),
    "plnlp_edge_dot_fwd_f32": (c_int, [_P, _L, _L, _P, _L, _L, _P, _P]),
    "plnlp_mlp_out_fwd_f32": (c_int, [_P, _L, _P, _P, _L, _L, _P, _P]),
    "plnlp_mlp_out_bwd_workspace_bytes": (c_int64, [_L, _L]),
    "plnlp_mlp_out_bwd_f32": (c_int, [_P, _L, _P, _P, _L, _L, _I, _F, _P, _L, _P, _P, _P, _P, _L, _P]),
    "plnlp_edge_mlp_bwd_workspace_bytes": (c_int64, [_L, _L, _L, _I]),
    "plnlp_edge_mlp_bwd_tf32": (c_int, [_I, _P, _L, _L, _P, _L, _L, _P, _L, _L, _P, _L, _P, _P, _F, _P, _L, _P, _L, _P, _L, _I, _P]),
    "plnlp_edge_scatter_atomic_f32": (c_int, [_P, _L, _L, _P, _L, _L, _P, _L, _P, _P, _L, _P]),
    "plnlp_edge_scatter_sorted_f32": (c_int, [_P, _L, _L, _P, _L, _L, _P, _L, _P, _P, _P, _L, _P, _P, _L, _P]),
    "plnlp_pair_loss_workspace_bytes": (c_int64, [_L]),
    "plnlp_pair_loss_f32": (c_int, [_I, _P, _P, _P, _L, _I, _P, _P, _P, _P, _L, _P]),
    "plnlp_relu_drop_bwd_f32": (c_int, [_P, _L, _P, _L, _F, _L, _L, _P, _L, _P]),
    "plnlp_colsum_workspace_bytes": (c_int64, [_L, _L]),
    "plnlp_colsum_f32": (c_int, [_P, _L, _L, _L, _F, _P, _P, _L, _P]),
    "plnlp_local_neg_sample": (c_int, [_P, _L, _L, _I, _U, _P, _P]),
    "plnlp_global_neg_candidates": (c_int, [_P, _L, _L, _L, _U, _P, _P, _P, _L, _P]),
    "plnlp_global_neg_keep": (c_int, [_P, _L, _P, _P, _L, _P, _P]),
    "plnlp_kth_largest_f32": (c_int, [_P, _L, _L, _P, _P, _L, _P]),
    "plnlp_count_greater_f32": (c_int, [_P, _L, _P, _P, _P]),
    "plnlp_mrr_counts_f32": (c_int, [_P, _P, _L, _L, _L, _P, _P, _P]),
    "plnlp_score_mask_f32": (c_int, [_P, _L, _L, _L, _P, _P, _P, _I, _P]),
    "plnlp_topk_rows_workspace_bytes": (c_int64, [_L, _L, _L]),
    "plnlp_topk_rows_f32": (c_int, [_P, _L, _L, _L, _L, _P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "plnlp_score_mask_cols_f32": (c_int, [_P, _L, _L, _L, _L, _P, _P, _P, _I, _P]),
    "plnlp_topk_rows_cols_f32": (c_int, [_P, _L, _L, _L, _L, _L, _P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "plnlp_score_mask_cand_f32": (c_int, [_P, _L, _L, _L, _P, _P, _P, _P, _I, _P]),
    "plnlp_topk_rows_cand_f32": (c_int, [_P, _L, _L, _L, _L, _L, _P, _P, _P, _P, _P, _P, _P, _L, _P, _P]),
    "plnlp_topk_merge_f32": (c_int, [_P, _P, _L, _L, _L, _L, _P, _P, _P]),
    "plnlp_graph_make_keys": (c_int, [_P, _P, _L, _L, _I, _I, _P, _P, _P]),
    "plnlp_graph_diag_keys": (c_int, [_L, _L, _P, _P, _L, _P]),
    "plnlp_graph_sort_workspace_bytes": (c_int64, [_L]),
    "plnlp_graph_sort_pairs": (c_int, [_P, _P, _L, _L, _L, _I, _P, _P, _P, _L, _P]),
    "plnlp_graph_unique_workspace_bytes": (c_int64, [_L]),
    "plnlp_graph_unique": (c_int, [_P, _L, _P, _P, _P, _P, _L, _P, _P, _L, _P]),
    "plnlp_graph_keys_to_csr": (c_int, [_P, _L, _L, _L, _P, _P, _P]),
    "plnlp_graph_sym_normalize": (c_int, [_P, _P, _P, _L, _P, _P, _P]),
    "plnlp_subset_plan_count": (c_int, [_P, _P, _L, _I, _P, _P, _P, _P, _P]),
    "plnlp_subset_plan_fill": (c_int, [_P, _P, _L, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "plnlp_random_walk": (c_int, [_P, _P, _P, _L, _I, _P, _U, _P, _P]),
    "plnlp_walk_pairs": (c_int, [_P, _L, _I, _P, _P, _P, _P]),
    "plnlp_link_heuristic_f64": (c_int, [_P, _P, _L, _L, _P, _P, _L, _P, _P]),
    "plnlp_common_neighbour_list": (c_int, [_P, _P, _L, _L, _P, _L, _P, _P, _P]),
    "plnlp_two_hop_mark": (c_int, [_P, _P, _P, _P, _L, _P, _P, _L, _L, _L, _P, _P, _P]),
    "plnlp_two_hop_score_f32": (c_int, [_P, _P, _L, _L, _P, _P, _L, _L, _L, _P, _P, _P, _L, _P]),
    "plnlp_two_hop_score_f64": (c_int, [_P, _P, _L, _L, _P, _P, _L, _L, _L, _P, _P, _P, _L, _P]),
    "plnlp_propagate_f32": (c_int, [_P, _P, _P, _L, _P, _P, _P, _L, _P, _P, _P, _L, _P, _L, _U, _U, _P, _P, _L, _L, _P,
                                    _L, _P]),
}

_ERRORS = {-1: "required pointer is NULL", -2: "bad size", -3: "misaligned pointer / leading dimension",
           -4: "unsupported combination", -5: "workspace too small", -6: "device is not sm_100"}

_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError when it has not been built:
    the product has no other execution path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C plnlp_b200/csrc`). plnlp_b200 has no CPU or eager fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.plnlp_abi_version() != 1:
        raise RuntimeError("libplnlp_b200.so ABI version mismatch")
    apply_spmm_tuning(lib)
    _lib = lib
    return lib


def apply_spmm_tuning(lib=None):
    """SpMM gather knobs (plnlp_spmm_tune): the library's built-in defaults unless the environment overrides them --
    PLNLP_SPMM_PREFETCH (0/1/2), PLNLP_SPMM_STAGED (0..5), PLNLP_SPMM_STAGED_WARPS, PLNLP_L2_FETCH (bytes).  A/B
    tools call plnlp_spmm_tune directly."""
    lib = lib or load()
    env = os.environ.get
    rc = lib.plnlp_spmm_tune(int(env("PLNLP_SPMM_PREFETCH", "-1")), int(env("PLNLP_SPMM_STAGED", "-1")),
                             int(env("PLNLP_SPMM_STAGED_WARPS", "0")), int(env("PLNLP_L2_FETCH", "0")))
    if rc != 0:
        raise RuntimeError(f"plnlp_spmm_tune -> {rc}")


def check(rc, name):
    if rc == 0:
        return
    if rc < 0:
        raise RuntimeError(f"{name}: invalid argument ({_ERRORS.get(rc, rc)})")
    raise RuntimeError(f"{name}: CUDA launch failed with cudaError {rc}")


def stream():
    """raw handle of torch's current CUDA stream (the C call: torch.cuda.current_stream() builds a Stream object and
    resolves the device on every call -- 24 calls per training step were 0.4 ms of host time)"""
    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())


def ptr(t):
    """device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("plnlp_b200 kernels need CUDA tensors; there is no CPU path")
    return t.data_ptr()


def launch_count():
    return int(load().plnlp_launch_count())


class _Workspace:
    """Caller-owned scratch buffers, grown on demand and reused (per device, per tag)."""

    def __init__(self):
        self._bufs = {}

    def get(self, tag, nbytes, device):
        key = (tag, device)
        buf = self._bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
            self._bufs[key] = buf
        return buf


workspace = _Workspace()
