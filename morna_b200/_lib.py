"""ctypes binding of libmorna_b200.so (the C ABI in include/morna_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, the
caller gets an exception.  Device memory is owned by torch tensors; only raw
pointers and sizes cross the boundary.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libmorna_b200.so")

OK = 0
ERR_INVALID_ARGUMENT = -1
ERR_WORKSPACE_TOO_SMALL = -2
ERR_CUDA = -3
ERR_UNSUPPORTED_DEVICE = -4
ERR_NO_SAMPLES = -5
ERR_CAPACITY = -6

_c_i32, _c_i64, _c_sz, _c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_void_p
ABI_VERSION = 4


class RerankJob(ctypes.Structure):
    """morna_rerank_job (include/morna_b200.h): another batch's re-rank, carried by a scoring call."""
    _fields_ = [("vectors", _c_vp), ("pp", _c_vp), ("n", _c_i64), ("dim", _c_i32), ("ld", _c_i64), ("id_base", _c_i32),
                ("queries", _c_vp), ("nq", _c_i64), ("q_ld", _c_i64), ("k", _c_i32),
                ("overflow", _c_vp), ("workspace", _c_vp), ("workspace_bytes", _c_sz)]


# name -> (restype, argtypes); mirrors include/morna_b200.h
_SIGNATURES = {
    "morna_abi_version": (ctypes.c_int, []),
    "morna_status_string": (ctypes.c_char_p, [ctypes.c_int]),
    "morna_last_cuda_error": (ctypes.c_int, []),
    "morna_kernel_launch_count": (_c_i64, []),
    "morna_note_graph_replay": (ctypes.c_int, [_c_i64]),
    "morna_device_info": (ctypes.c_int, [_c_vp, _c_vp, _c_vp]),
    "morna_hash_junctions": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_vp, _c_vp, _c_vp, _c_vp]),
    "morna_idf_host": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_vp]),
    "morna_assign_internal_ids_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32]),
    "morna_assign_internal_ids": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_vp,
                                                 _c_vp, _c_sz, _c_vp]),
    "morna_tokenize_count": (ctypes.c_int, [_c_vp, _c_sz, _c_i32, _c_vp, _c_vp, _c_vp]),
    "morna_tokenize_fill": (ctypes.c_int, [_c_vp, _c_sz, _c_i32, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]),
    "morna_index_accumulate_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32]),
    "morna_index_accumulate": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_i64,
                                              _c_vp, _c_i32, _c_i32, _c_i32, _c_i32, _c_vp, _c_i64, _c_vp, _c_sz, _c_vp]),
    "morna_junction_table_bytes": (_c_sz, [_c_i64]),
    "morna_junction_table_build": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_sz, _c_vp]),
    "morna_junction_lookup_workspace_bytes": (_c_sz, [_c_i64]),
    "morna_junction_lookup": (ctypes.c_int, [_c_vp, _c_sz, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp,
                                             _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_round_store": (ctypes.c_int, [_c_vp, _c_i64, _c_i32, _c_i32, _c_vp, _c_i64, _c_vp]),
    "morna_row_norms": (ctypes.c_int, [_c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_vp]),
    "morna_angular_distances": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_i64, _c_i64,
                                               _c_vp, _c_i64, _c_vp]),
    "morna_select_topk_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32]),
    "morna_select_topk": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_vp,
                                         _c_vp, _c_sz, _c_vp]),
    "morna_merge_sorted_topk": (ctypes.c_int, [_c_vp, _c_vp, _c_i32, _c_i64, _c_i32, _c_i32, _c_vp, _c_vp, _c_vp]),
    "morna_merge_packed_topk": (ctypes.c_int, [_c_vp, _c_i32, _c_i64, _c_i32, _c_i32, _c_vp, _c_vp, _c_vp]),
    "morna_knn_exact_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32]),
    "morna_knn_exact": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64, _c_i64,
                                       _c_i32, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_knn_exact_excl": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64, _c_i64,
                                            _c_i32, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, _c_vp, _c_vp]),
    "morna_sparse_max_nnz": (_c_i32, []),
    "morna_knn_exact_sparse_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32]),
    "morna_knn_exact_sparse": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i32, _c_i32, _c_vp, _c_i64, _c_i64, _c_i32,
                                              _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_knn_exact_sparse_excl": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_i32, _c_i32, _c_vp, _c_i64, _c_i64,
                                                   _c_i32, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, _c_vp, _c_vp]),
    "morna_knn_single_workspace_bytes": (_c_sz, [_c_i64]),
    "morna_knn_single_workspace_init": (ctypes.c_int, [_c_vp, _c_sz, _c_vp]),
    "morna_knn_single": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i32, _c_vp, _c_vp,
                                        _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_knn_single_stream": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64, _c_i32, _c_i32,
                                               _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_tensor_operand_ld": (_c_i64, [_c_i32]),
    "morna_prepare_tensor_operand": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_i64, _c_vp, _c_vp]),
    "morna_knn_batched_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32, _c_i32]),
    "morna_knn_batched": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32,
                                         _c_vp, _c_i64, _c_i64, _c_i32, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, _c_vp]),
    "morna_knn_batched_score": (ctypes.c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i32, _c_vp, _c_i64, _c_i64, _c_i32,
                                               _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, ctypes.POINTER(RerankJob), _c_vp, _c_vp]),
    "morna_knn_batched_score_excl": (ctypes.c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i32, _c_vp, _c_i64, _c_i64, _c_i32,
                                                    _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, ctypes.POINTER(RerankJob), _c_vp, _c_vp, _c_vp,
                                                    _c_vp]),
    "morna_knn_batched_approx": (ctypes.c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i32, _c_vp, _c_i64, _c_i64, _c_i32,
                                                _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_union_kth_bound": (ctypes.c_int, [_c_vp, _c_i32, _c_i64, _c_i32, _c_vp, _c_vp]),
    "morna_knn_batched_finalize": (ctypes.c_int, [_c_i64, _c_i64, _c_i32, _c_i32, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_knn_batched_rerank": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64, _c_i64, _c_i32,
                                                _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_i32, _c_vp]),
    "morna_range_batched_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32]),
    "morna_range_batched": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64,
                                           _c_i64, ctypes.c_double, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_range_batched_excl": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64,
                                                _c_i64, ctypes.c_double, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, _c_vp, _c_vp]),
    "morna_range_batched_emit": (ctypes.c_int, [_c_i64, _c_i64, _c_i32, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_range_exact_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i64]),
    "morna_range_exact_count": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_i64, _c_i64, ctypes.c_double,
                                               _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_range_exact_count_excl": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_i64, _c_i64, ctypes.c_double,
                                                    _c_vp, _c_vp, _c_sz, _c_vp, _c_vp, _c_vp]),
    "morna_range_exact_fill": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64, _c_i64, ctypes.c_double,
                                              _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_range_exact_fill_excl": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_i64, _c_i64,
                                                   ctypes.c_double, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp, _c_sz, _c_vp, _c_vp, _c_vp]),
    "morna_merge_sorted_csr": (ctypes.c_int, [_c_vp, _c_i32, _c_i64, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_vp, _c_vp]),
    "morna_cap_sorted_lists_workspace_bytes": (_c_sz, [_c_i64, _c_i64]),
    "morna_cap_sorted_lists": (ctypes.c_int, [_c_vp, _c_i64, _c_vp, _c_vp, _c_i64, _c_vp, _c_i32, _c_i64, _c_i32, _c_i64,
                                              _c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_sz, _c_vp]),
    "morna_knn_batched_capped_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_i32, _c_i32]),
    "morna_knn_batched_capped": (ctypes.c_int, [_c_vp, _c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp,
                                                _c_i64, _c_i64, _c_i32, _c_vp, _c_i32, _c_vp, _c_i32, _c_vp, _c_vp, _c_vp, _c_vp,
                                                _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_within_group_workspace_bytes": (_c_sz, [_c_i64]),
    "morna_within_group_topk": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_i32, _c_vp, _c_vp, _c_i64, _c_i64,
                                               _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i32, _c_vp, _c_vp, _c_i32, _c_vp, _c_vp,
                                               _c_vp, _c_sz, _c_vp]),
    "morna_within_group_range_count": (ctypes.c_int, [_c_vp, _c_vp, _c_i64, _c_i32, _c_i64, _c_vp, _c_vp, _c_i64, _c_i64,
                                                      _c_vp, _c_i64, _c_vp, _c_i64, _c_vp, _c_i32, _c_vp, _c_vp,
                                                      ctypes.c_double, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_within_group_range_fill": (ctypes.c_int, [_c_i64, _c_vp, _c_i32, _c_vp, _c_i64, _c_vp, _c_i32, _c_vp, _c_vp,
                                                     _c_vp, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_debug_tensor_scores": (ctypes.c_int, [_c_vp, _c_i64, _c_vp, _c_i64, _c_i32, _c_vp, _c_i64, _c_i64, _c_vp,
                                                 _c_i64, _c_vp, _c_vp, _c_sz, _c_vp]),
    "morna_debug_set_tuning": (ctypes.c_int, [_c_i32, _c_i32]),
    "morna_debug_gemm_counters": (ctypes.c_int, [_c_vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class MornaLibraryError(RuntimeError):
    pass


def load():
    """dlopen the in-tree library and type every entry point.  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise MornaLibraryError(
            "morna_b200: %s is missing -- build it with `python -m morna_b200.build` "
            "(there is no CPU fallback)" % SO_PATH)
    lib = ctypes.CDLL(SO_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)         # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.morna_abi_version() != ABI_VERSION:
        raise MornaLibraryError("morna_b200: ABI version mismatch")
    _lib = lib
    return lib


def check(status, what):
    if status == OK:
        return
    lib = load()
    msg = lib.morna_status_string(status).decode()
    if status == ERR_CUDA:
        msg += " (cudaError %d)" % lib.morna_last_cuda_error()
    if status == ERR_NO_SAMPLES:
        raise ValueError("No internal ids were assigned, indicating that no samples were added "
                         "to the index. Likely caused when no junctions pass the sample threshold.")
    raise MornaLibraryError("%s failed: %s" % (what, msg))


def require_cuda():
    if not torch.cuda.is_available():
        raise MornaLibraryError("morna_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def ptr(t):
    """Raw pointer of a contiguous tensor (0 for None)."""
    if t is None:
        return None
    assert t.is_contiguous(), "tensor must be contiguous"
    return ctypes.c_void_p(t.data_ptr())


def dev_ptr(t, dtype=None):
    if t is None:
        return None
    assert t.is_cuda, "expected a CUDA tensor"
    if dtype is not None:
        assert t.dtype == dtype, "expected %s, got %s" % (dtype, t.dtype)
    return ptr(t)


def stream_ptr(stream=None):
    s = stream if stream is not None else torch.cuda.current_stream()
    return ctypes.c_void_p(s.cuda_stream)


def launch_count():
    return int(load().morna_kernel_launch_count())


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
