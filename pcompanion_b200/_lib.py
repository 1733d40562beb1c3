"""ctypes binding of the C ABI in include/pcompanion_b200.h.

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no
fallback: if the shared object is missing the import of this package fails, and every wrapper
refuses tensors that are not contiguous CUDA tensors of the expected dtype.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

import torch

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libpcompanion_b200.so")

P = c_void_p  # every pointer crosses the ABI as void*

# name -> (restype, argtypes); mirrors include/pcompanion_b200.h one to one (checked by tests/test_abi.py)
PROTOTYPES = {
    "pc_abi_version": (c_int, []),
    "pc_last_error": (c_char_p, []),
    "pc_device_info": (c_int, [P, P, P]),
    "pc_edge_keys_pack": (c_int, [P, P, c_int64, P, P]),
    "pc_edge_keys_unpack": (c_int, [P, c_int64, P, P, P]),
    "pc_sort_keys_workspace_bytes": (c_size_t, [c_int64]),
    "pc_sort_keys": (c_int, [P, c_int64, c_uint32, P, c_size_t, P]),
    "pc_compact_workspace_bytes": (c_size_t, [c_int64]),
    "pc_unique_sorted_keys": (c_int, [P, c_int64, P, P, P, c_size_t, P]),
    "pc_set_filter_sorted": (c_int, [P, c_int64, P, c_int64, c_int, P, P, P, c_size_t, P]),
    "pc_csr_from_sorted_keys": (c_int, [P, c_int64, c_int64, P, P, P]),
    "pc_csr_transpose_keys": (c_int, [P, P, c_int64, c_int64, P, P]),
    "pc_gat_fwd": (c_int, [P, c_int64, P, P, P, c_int64, c_int, c_float, c_uint64, P, P, P, P]),
    "pc_gat_bwd_dst": (c_int, [P, c_int64, P, P, P, c_int64, c_int, c_float, c_uint64, P, P, P, c_int64, P, P, c_int64, P]),
    "pc_gat_bwd_src": (c_int, [P, c_int64, P, P, P, c_int64, c_int, c_float, c_uint64, P, c_int64, P, P, c_int64, c_int64, P, P]),
    "pc_gat_merge_segments": (c_int, [P, P, P, P, c_int64, c_int, P, P, P]),
    "pc_gat_delta": (c_int, [P, P, c_int64, c_int64, c_int, P, P]),
    "pc_col_reduce_workspace_bytes": (c_size_t, [c_int]),
    "pc_col_stats": (c_int, [P, c_int64, c_int, c_int64, P, P, c_size_t, P]),
    "pc_col_sum_unselected": (c_int, [P, c_int64, c_int, c_int64, P, P, P, c_size_t, P]),
    "pc_bn_bwd_reduce": (c_int, [P, c_int64, P, c_int64, c_int64, c_int, P, P, P, P, c_size_t, P]),
    "pc_scale_shift_tanh": (c_int, [P, c_int64, c_int64, c_int, P, P, c_int, P, c_int64, P]),
    "pc_affine2": (c_int, [P, c_int64, P, c_int64, c_int64, c_int, P, P, P, P, c_int64, P]),
    "pc_mask_split": (c_int, [P, c_int64, c_int, P, P, P, P]),
    "pc_linear_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pc_linear_tf32x3": (c_int, [P, c_int64, c_int, c_int64, P, c_int, P, c_int, P, c_int64, P, P, c_int64, c_int, P, c_int64, P, P, c_size_t, P]),
    "pc_wgrad_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pc_wgrad_tf32x3": (c_int, [P, c_int64, c_int, c_int64, P, c_int, c_int64, P, P, P, c_size_t, P]),
    "pc_type_scores_topk_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "pc_type_scores_topk": (c_int, [P, c_int64, c_int, c_int64, P, c_int, P, c_int64, c_int, P, P, P, c_size_t, P]),
    "pc_mlp2_fwd": (c_int, [P, P, c_int64, c_int, c_int, c_int, P, P, P, P, c_float, c_uint64, P, P, P, P]),
    "pc_mlp2_bwd_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pc_mlp2_bwd": (c_int, [P, P, P, P, c_int64, c_int, c_int, c_int, P, P, c_float, P, P, P, P, P, P, c_size_t, P]),
    "pc_item_combine_fwd": (c_int, [P, P, c_int64, c_int, c_int, P, P]),
    "pc_item_combine_bwd": (c_int, [P, P, P, c_int64, c_int, c_int, P, P, P]),
    "pc_hinge_type_factored_bwd": (c_int, [P, P, P, P, P, P, c_int64, c_int, P, P, P]),
    "pc_hinge_rows_fwd": (c_int, [P, P, P, c_int64, c_int, c_int, c_int, c_float, c_float, P, P, P]),
    "pc_hinge_rows_bwd": (c_int, [P, P, P, c_int64, c_int, c_int, c_int, c_float, c_float, P, P, P, P, P]),
    "pc_hinge_type_fwd": (c_int, [P, P, P, c_int64, c_int64, c_float, P, P, P]),
    "pc_hinge_type_bwd": (c_int, [P, P, P, c_int64, c_int64, c_float, P, P, P]),
    "pc_sample_negatives": (c_int, [P, P, P, c_int64, ctypes.c_int32, c_int, c_uint64, P, P]),
    "pc_triplet_batch_rows": (c_int, [P, c_int64, c_int, P, P, P, c_int64, c_int, P, P, P, c_int64, P, P, P]),
    "pc_topk_groups_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "pc_topk_groups": (c_int, [P, c_int64, c_int, P, P, P, P, P, P, c_int64, c_int, c_int, c_int64, P, P, P, c_size_t, P]),
    "pc_topk_by_type_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "pc_topk_by_type": (c_int, [P, c_int64, c_int, P, P, P, c_int, P, c_int, c_int, c_int64, P, P, P, c_size_t, P]),
    "pc_rank_by_type_workspace_bytes": (c_size_t, [c_int64]),
    "pc_rank_by_type": (c_int, [P, c_int64, c_int, P, P, P, c_int, P, P, P, c_int, c_int64, P, P, c_size_t, P]),
    "pc_topk_by_type_excluding": (c_int, [P, c_int64, c_int, P, P, P, c_int, P, c_int, c_int, c_int64, P, P, c_int64, P, P, P,
                                          P, c_size_t, P]),
    "pc_rank_remove_excluded": (c_int, [P, c_int64, c_int, P, c_int64, P, P, P, P, c_int64, P, P, c_int64, P, P, P]),
    "pc_score_topk_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "pc_score_topk_dense": (c_int, [P, c_int64, c_int, P, c_int64, P, P, c_int, c_int, c_int64, c_float, P, P, P, P, c_size_t, P]),
    "pc_topk_rows_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "pc_topk_rows": (c_int, [P, c_int64, c_int64, c_int, c_int, P, P, P, c_size_t, P]),
    "pc_topk_merge": (c_int, [P, P, c_int64, c_int, c_int, P, P, P]),
    "pc_rows_gather": (c_int, [P, P, c_int64, c_int, P, P]),
    "pc_rows_scatter_add": (c_int, [P, P, c_int64, c_int, P, P]),
    "pc_rows_reduce_peers": (c_int, [P, P, c_int, c_int64, c_int, P, P]),
    "pc_halo_push": (c_int, [P, c_int64, P, c_int, P, P, P, P, c_int64, c_int, P]),
    "pc_rows_index_grad_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "pc_rows_index_grad": (c_int, [P, P, c_int64, c_int64, c_int, P, P, P, c_size_t, P]),
    "pc_triplet_indexed": (c_int, [P, P, c_int64, c_int, c_int, c_float, c_float, P, P, P, P]),
    "pc_rows_segment_sum": (c_int, [P, P, P, c_int64, c_int, P, P]),
}


class NativeLibraryError(RuntimeError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} is missing - build it with `python __graft_entry__.py` (nvcc, sm_100a). "
            "pcompanion_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise NativeLibraryError(f"{LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype = res
        fn.argtypes = args
    if lib.pc_abi_version() != 1:
        raise NativeLibraryError("ABI version mismatch between _lib.py and the shared library; rebuild it")
    return lib


LIB = _load()
LAUNCHES = 0  # number of C-ABI compute entry points invoked (bench.py reports kernels launched)
PROFILE = None  # when a list: (name, start_event, end_event) per native call, for bench.py's per-kernel timing


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError(f"pcompanion_b200 native call failed ({rc}): {LIB.pc_last_error().decode()}")


def call(name: str, *args) -> None:
    global LAUNCHES
    LAUNCHES += 1
    if PROFILE is None:
        check(getattr(LIB, name)(*args))
        return
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    check(getattr(LIB, name)(*args))
    end.record()
    PROFILE.append((name, start, end))


class region:
    """with region("wait:h_block"): ...  - when bench.py's per-call profiling is on, the enclosed stream work (waits on
    other streams / peers) is timed like a native call; otherwise free."""

    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        if PROFILE is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            PROFILE.append((self.name, self.start, end))
        return False


def stream() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def dev(t: torch.Tensor | None, dtype: torch.dtype, what: str) -> c_void_p | None:
    """Device pointer of a contiguous CUDA tensor of `dtype` (None passes through as NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError(f"{what}: expected a CUDA tensor, got device {t.device} - "
                           "pcompanion_b200 runs on the GPU only (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{what}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{what}: tensor must be contiguous")
    return c_void_p(t.data_ptr())


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)


def device_info():
    sm, major, minor = c_int(), c_int(), c_int()
    check(LIB.pc_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)))
    return sm.value, major.value, minor.value
