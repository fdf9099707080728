"""ctypes binding of libetpgt_b200.so (the C ABI declared in include/etpgt_b200.h).

The library is the product: there is no Python / CPU fallback.  If the shared object is missing
or a call is made with non-CUDA tensors this module raises immediately.
"""

from __future__ import annotations

import ctypes
from ctypes import c_double, c_float, c_int, c_int64, c_size_t, c_void_p
from pathlib import Path

import torch

_LIB_PATH = Path(__file__).resolve().parent / "libetpgt_b200.so"

P, I, L, F, D, Z = c_void_p, c_int, c_int64, c_float, c_double, c_size_t

# name -> (restype, argtypes); mirrors include/etpgt_b200.h one to one
_PROTOTYPES = {
    "etpgt_version": (I, []),
    "etpgt_last_error": (ctypes.c_char_p, []),
    "etpgt_launch_count": (L, []),
    "etpgt_reset_launch_count": (None, []),
    "etpgt_csr_workspace_bytes": (Z, [L, L]),
    "etpgt_csr_from_coo": (I, [P, P, L, L, P, P, P, P, P, P, P, Z, P]),
    "etpgt_segment_ptr": (I, [P, L, L, P, P]),
    "etpgt_item_graph_workspace_bytes": (Z, [L]),
    "etpgt_item_graph_build": (I, [P, P, L, L, P, P, P, P, Z, P]),
    "etpgt_session_subgraphs_workspace_bytes": (Z, [L, L]),
    "etpgt_session_subgraphs_count": (I, [P, P, P, P, P, L, I, I, I, P, P, P, Z, P]),
    "etpgt_session_subgraphs_fill": (I, [P, P, P, P, P, P, L, I, I, I, P, P, L, P, P, P, P, P, P, Z, P]),
    "etpgt_sample_negatives": (I, [ctypes.c_uint64, ctypes.c_uint32, L, P, P, P, L, I, L, I, P, P]),
    "etpgt_sample_item_pool_workspace_bytes": (Z, [L]),
    "etpgt_sample_item_pool": (I, [P, L, L, ctypes.c_uint64, ctypes.c_uint32, P, P, P, Z, P]),
    "etpgt_in_batch_columns_workspace_bytes": (Z, [L, L]),
    "etpgt_in_batch_columns": (I, [P, L, P, P, L, P, P, L, L, L, D, P, P, P, Z, P]),
    "etpgt_embed_pe_fwd": (I, [P, L, P, L, P, I, P, P, I, I, P, P]),
    "etpgt_embed_pe_fwd_split": (I, [P, L, P, L, P, I, P, P, I, I, P, P, P, P]),
    "etpgt_embed_pe_bwd_workspace_bytes": (Z, [L, I, I]),
    "etpgt_embed_pe_bwd": (I, [P, L, P, L, P, I, I, I, L, P, P, P, P, Z, P]),
    "etpgt_tconv_fwd": (I, [P, L, I, I, P, P, P, L, P, P, P, P, P, P, P, P]),
    "etpgt_tconv_bwd_workspace_bytes": (Z, [L, L, I, I]),
    "etpgt_tconv_bwd": (I, [P, P, L, I, I, P, P, P, P, P, P, L, P, P, P, P, P, P, P, P, P, Z, P]),
    "etpgt_tconv_bwd_split": (I, [P, P, L, I, I, P, P, P, P, P, P, L, P, P, P, P, P, P, P, P, P, P, P, P, Z, P]),
    "etpgt_hub_plan_bytes": (Z, [L]),
    "etpgt_hub_plan_workspace_bytes": (Z, [L]),
    "etpgt_hub_plan": (I, [P, P, L, L, P, P, Z, P]),
    "etpgt_tconv_hub_workspace_bytes": (Z, [L, I]),
    "etpgt_tconv_fwd_hub": (I, [P, L, I, I, P, P, P, L, P, P, P, P, P, P, P, P, P, Z, P]),
    "etpgt_tconv_fwd_bn_workspace_bytes": (Z, [I]),
    "etpgt_tconv_fwd_bn": (I, [P, L, I, I, P, P, P, L, P, P, P, P, P, P, P, P, P, Z, P, P, Z, P]),
    "etpgt_tconv_bwd_split_hub": (I, [P, P, L, I, I, P, P, P, P, P, P, L, P, P, P, P, P, P, P, P, P, P, P, P, Z, P, P, Z,
                                      P]),
    "etpgt_split_bf16_workspace_bytes": (Z, [L, L]),
    "etpgt_split_bf16": (I, [P, L, L, L, P, P, L, P, P, L, P, P, Z, P]),
    "etpgt_gemm_bf16x3_workspace_bytes": (Z, [L, L, L, I]),
    "etpgt_gemm_bf16x3": (I, [P, P, P, P, L, L, L, L, L, P, P, L, I, P, Z, P]),
    "etpgt_gemm_bf16x3_ex": (I, [P, P, P, P, L, L, L, L, L, I, I, P, I, P, L, I, P, Z, P]),
    "etpgt_gemm_bf16x3_gelu": (I, [P, P, P, P, L, L, L, L, L, P, P, L, P, P, L, D, ctypes.c_uint64, P, Z, P]),
    "etpgt_gelu_bwd_split": (I, [P, P, L, L, D, ctypes.c_uint64, P, P, L, P, P, Z, P]),
    "etpgt_lap_sym_block": (I, [P, P, P, L, I, P, P, D, D, D, P, P]),
    "etpgt_gat_fwd": (I, [P, P, P, L, I, I, P, P, P, F, P, P, P, P, P, P]),
    "etpgt_gat_mean_fused_supported": (I, [I, I]),
    "etpgt_gat_fwd_mean": (I, [P, P, P, L, I, I, P, P, P, F, P, P, P, P, P, P, P, P]),
    "etpgt_gat_bwd_mean": (I, [P, P, P, P, P, P, L, I, I, P, P, P, P, P, P, L, F, P, P, P, P, P, P, P, P, P, P, Z, P]),
    "etpgt_gat_input_scores_workspace_bytes": (Z, [L, I, I]),
    "etpgt_gat_input_scores_fwd": (I, [P, P, L, I, I, P, P, P]),
    "etpgt_gat_input_scores_bwd": (I, [P, P, P, P, L, I, I, P, P, P, Z, P]),
    "etpgt_gat_bwd_workspace_bytes": (Z, [L, L, I]),
    "etpgt_gat_bwd": (I, [P, P, P, P, P, L, I, I, P, P, P, P, P, P, L, F, P, P, P, P, P, P, P, P, Z, P]),
    "etpgt_gat_aux_workspace_bytes": (Z, [L, I]),
    "etpgt_gat_scores_fwd": (I, [P, P, P, L, I, I, P, P, P]),
    "etpgt_gat_scores_bwd": (I, [P, P, P, P, P, L, I, I, P, P, P, P, Z, P]),
    "etpgt_head_mean_fwd": (I, [P, P, L, I, I, P, P]),
    "etpgt_head_mean_bwd": (I, [P, L, I, I, P, P, P, Z, P]),
    "etpgt_sage_mean_fwd": (I, [P, L, I, P, P, P, P]),
    "etpgt_sage_mean_bwd": (I, [P, L, I, P, P, P, P, P]),
    "etpgt_sage_mean_bwd_ld": (I, [P, L, P, L, I, P, P, P, P, P]),
    "etpgt_sage_mean_fwd_split": (I, [P, L, I, P, P, P, P, P, L, P]),
    "etpgt_bn_workspace_bytes": (Z, [L, I]),
    "etpgt_bn_stats": (I, [P, L, I, P, P, Z, P]),
    "etpgt_bn_finalize": (I, [P, D, I, F, F, P, P, P, P, P]),
    "etpgt_bn_from_running": (I, [P, P, I, F, P, P, P]),
    "etpgt_bn_apply": (I, [P, L, I, P, P, P, P, P, I, P, P]),
    "etpgt_dropout_mask": (I, [ctypes.c_uint64, D, L, P, P]),
    "etpgt_bn_apply_ex": (I, [P, L, I, P, P, P, P, P, I, D, ctypes.c_uint64, P, P, P, P]),
    "etpgt_bn_bwd_stats_ex": (I, [P, P, P, L, I, P, P, I, D, ctypes.c_uint64, P, P, Z, P]),
    "etpgt_bn_bwd_apply_ex": (I, [P, P, P, L, I, P, P, P, I, I, P, D, P, D, ctypes.c_uint64, P, P, P, P, P]),
    "etpgt_bn_bwd_stats": (I, [P, P, P, L, I, P, P, I, P, P, Z, P]),
    "etpgt_bn_bwd_apply": (I, [P, P, P, L, I, P, P, P, I, I, P, D, P, P, P, P, P]),
    "etpgt_readout_fwd": (I, [P, P, L, I, I, P, P, P, P]),
    "etpgt_readout_bwd": (I, [P, P, P, P, L, L, I, I, P, P, P, P]),
    "etpgt_sampled_loss_workspace_bytes": (Z, [L, I, I]),
    "etpgt_sampled_loss_fwd": (I, [P, P, P, P, L, I, I, I, F, F, D, P, P, P, Z, P]),
    "etpgt_sampled_loss_bwd": (I, [P, P, P, P, L, I, I, I, F, F, D, P, P, L, L, P, P, P, Z, P]),
    "etpgt_full_softmax_workspace_bytes": (Z, [L, L, I]),
    "etpgt_full_softmax_fwd": (I, [P, P, P, L, L, I, F, D, L, P, P, P, Z, P]),
    "etpgt_full_softmax_bwd": (I, [P, P, P, P, P, L, L, I, F, D, L, P, P, P, Z, P]),
    "etpgt_pool_softmax_workspace_bytes": (Z, [L, L, I]),
    "etpgt_pool_softmax_fwd": (I, [P, P, P, P, P, L, L, L, I, F, D, L, P, P, P, P, Z, P]),
    "etpgt_pool_softmax_bwd": (I, [P, P, P, P, P, P, P, P, L, L, L, I, F, D, L, P, P, P, Z, P]),
    "etpgt_full_softmax_fwd_ex": (I, [P, P, P, L, L, I, F, D, L, P, P, P, Z, P, I]),
    "etpgt_full_softmax_bwd_ex": (I, [P, P, P, P, P, L, L, I, F, D, L, P, P, P, Z, P, I]),
    "etpgt_pool_softmax_fwd_ex": (I, [P, P, P, P, P, L, L, L, I, F, D, L, P, P, P, P, Z, P, I]),
    "etpgt_pool_softmax_bwd_ex": (I, [P, P, P, P, P, P, P, P, L, L, L, I, F, D, L, P, P, P, Z, P, I]),
    "etpgt_score_topk_workspace_bytes": (Z, [L, L, I, I]),
    "etpgt_score_topk_f32": (I, [P, P, L, L, I, I, L, P, P, P, Z, P]),
    "etpgt_f32_to_bf16": (I, [P, P, L, P]),
    "etpgt_score_topk_bf16_workspace_bytes": (Z, [L, L, I]),
    "etpgt_score_topk_bf16": (I, [P, P, L, L, I, I, L, P, P, P, Z, P]),
    "etpgt_score_topk_bf16_eval": (I, [P, P, L, L, I, I, L, P, P, P, P, P, Z, P]),
    "etpgt_score_topk_bf16_exclude": (I, [P, P, L, L, I, I, L, P, P, P, P, P, L, P, Z, P]),
    "etpgt_score_topk_f32_exclude": (I, [P, P, L, L, I, I, L, P, P, P, L, P, Z, P]),
    "etpgt_topk_merge": (I, [P, P, L, I, I, P, P, P]),
    "etpgt_topk_metrics": (I, [P, P, L, I, I, P, P]),
    "etpgt_scatter_rows_workspace_bytes": (Z, [L]),
    "etpgt_scatter_rows": (I, [P, P, P, L, I, I, L, L, P, P, Z, P]),
    "etpgt_scatter_plan_workspace_bytes": (Z, [L]),
    "etpgt_scatter_plan": (I, [P, L, L, P, P, P, Z, P]),
    "etpgt_batch_prepare_workspace_bytes": (Z, [L, L, L]),
    "etpgt_batch_prepare": (I, [P, P, L, L, P, P, P, L, I, L, P, P, P, P, P, P, P, P, P, P, P, Z, P]),
    "etpgt_scatter_plan_loss": (I, [P, P, L, I, L, P, P, P, Z, P]),
    "etpgt_scatter_rows_planned": (I, [P, P, P, P, L, I, I, L, P, P]),
    "etpgt_embed_pe_bwd_planned": (I, [P, L, P, L, P, I, I, I, L, P, P, P, P, P, P, Z, P]),
    "etpgt_sampled_loss_bwd_planned": (I, [P, P, P, P, L, I, I, I, F, F, D, P, P, L, L, P, P, P, P, P, Z, P]),
    "etpgt_cooc_graph_workspace_bytes": (Z, [L, I]),
    "etpgt_cooc_graph_build": (I, [P, P, P, L, L, I, L, L, P, P, P, P, P, P, Z, P]),
    "etpgt_gt_step_arena_bytes": (Z, [P]),
    "etpgt_gt_step_num_phases": (I, [P]),
    "etpgt_gt_step_run": (I, [P, I, I, P]),
    "etpgt_graph_create": (I, [P]),
    "etpgt_graph_destroy": (I, [P]),
    "etpgt_graph_rebuilds": (L, [P]),
    "etpgt_gt_step_run_graph": (I, [P, I, I, P, P]),
    "etpgt_adam_step": (I, [P, I, D, D, D, D, D, I, L, I, P]),
    "etpgt_adam_rows": (I, [P, P, P, P, L, I, D, D, D, D, D, I, L, I, P, P]),
    "etpgt_sparse_adam": (I, [P, P, P, L, I, P, P, L, D, D, D, D, I, L, I, P, P]),
    "etpgt_topk_merge_parts": (I, [P, I, Z, Z, L, I, L, L, P, P, P, P, P]),
    "etpgt_hit_metrics": (I, [P, L, I, P, P]),
    "etpgt_ids_check": (I, [P, L, P, L, P, L, L, P, P]),
    "etpgt_comm_control_bytes": (Z, []),
    "etpgt_comm_create": (I, [I, I, Z, P]),
    "etpgt_comm_ipc_handle": (I, [P, P]),
    "etpgt_comm_connect_ipc": (I, [P, P]),
    "etpgt_comm_connect_ptrs": (I, [P, P]),
    "etpgt_comm_region": (P, [P, I]),
    "etpgt_comm_set_timeout": (I, [P, D]),
    "etpgt_comm_destroy": (I, [P]),
    "etpgt_comm_barrier": (I, [P, I, P]),
    "etpgt_comm_allreduce_f64": (I, [P, P, P, I, P]),
    "etpgt_comm_sum_f32": (I, [P, Z, L, P, P]),
    "etpgt_comm_status": (I, [P, P]),
    "etpgt_dp_adam_table": (I, [P, Z, Z, P, P, L, I, L, L, D, D, D, D, D, I, L, P]),
}

_lib = None


def exported_symbols() -> list[str]:
    return sorted(_PROTOTYPES)


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Loads the shared library once and installs the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise ImportError(
            f"{_LIB_PATH} is missing: build it with `python gat-recommendation_b200/build.py` "
            "(etpgt_b200 has no CPU or PyTorch fallback)"
        )
    lib = ctypes.CDLL(str(_LIB_PATH))
    for name, (restype, argtypes) in _PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error() -> str:
    return load().etpgt_last_error().decode()


def ptr(t: torch.Tensor | None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("etpgt_b200 runs on CUDA tensors only (no CPU fallback); got a CPU tensor")
    if not t.is_contiguous():
        raise RuntimeError("etpgt_b200 kernels need contiguous tensors")
    return c_void_p(t.data_ptr())


def stream() -> c_void_p:
    """Raw handle of torch's current stream on the current device.  (`torch.cuda.current_stream()`
    builds a Python Stream object and costs ~15 us per call — a third of the host time of a step.)"""
    return c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def call(name: str, *args):
    """Calls an int-returning entry point and raises with the library's message on failure."""
    rc = getattr(load(), name)(*args)
    if rc != 0:
        msg = last_error()
        if "Unknown" in msg:  # mirrors the reference's ValueError for unknown readout / loss kinds
            raise ValueError(msg)
        raise RuntimeError(f"{name} failed ({rc}): {msg}")


def size(name: str, *args) -> int:
    return int(getattr(load(), name)(*args))


def launch_count() -> int:
    return int(load().etpgt_launch_count())


def reset_launch_count() -> None:
    load().etpgt_reset_launch_count()
