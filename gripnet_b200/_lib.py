"""ctypes binding of ``libgripnet_b200.so`` (the C ABI of ``include/gripnet_b200.h``).

There is no CPU fallback: if the shared library is missing or cannot be loaded
the import of any compute module fails loudly (``GripnetLibraryError``).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgripnet_b200.so")


class GripnetLibraryError(RuntimeError):
    pass


class GnCsr(C.Structure):
    """Mirror of ``gn_csr`` (include/gripnet_b200.h)."""
    _fields_ = [
        ("n_rows", C.c_int32), ("n_cols", C.c_int32), ("nnz", C.c_int32), ("chunk_len", C.c_int32),
        ("n_chunks", C.c_int32), ("flags", C.c_int32),
        ("rowptr", C.c_void_p), ("col", C.c_void_p), ("val", C.c_void_p),
        ("chunk_ptr", C.c_void_p), ("chunk_row", C.c_void_p), ("chunk_beg", C.c_void_p),
        ("row_counter", C.c_void_p),
    ]


class GnAdamTensor(C.Structure):
    """Mirror of ``gn_adam_tensor`` (include/gripnet_b200.h)."""
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
                ("n", C.c_int64)]


class GnPeerSegment(C.Structure):
    """Mirror of ``gn_peer_segment``."""
    _fields_ = [("src", C.c_void_p), ("bytes", C.c_int64), ("slot_offset", C.c_int64), ("peer", C.c_int32)]


class GnHaloPeer(C.Structure):
    """Mirror of ``gn_halo_peer``."""
    _fields_ = [("idx", C.c_void_p), ("count", C.c_int64), ("dst_row", C.c_int64)]


class GnSumSegment(C.Structure):
    """Mirror of ``gn_sum_segment``."""
    _fields_ = [("dst", C.c_void_p), ("n", C.c_int64), ("slot_offset", C.c_int64)]


_P, _I32, _I64, _F, _SZ, _INT = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t, C.c_int
_CSR = C.POINTER(GnCsr)

# name -> (restype, argtypes); every symbol declared in include/gripnet_b200.h
SIGNATURES = {
    "gn_version": (_INT, []),
    "gn_error_string": (C.c_char_p, [_INT]),
    "gn_last_cuda_error": (_INT, []),
    "gn_last_cuda_error_string": (C.c_char_p, []),
    "gn_launch_count": (C.c_uint64, []),
    "gn_csr_from_keys_workspace_bytes": (_SZ, [_I64, _I32]),
    "gn_csr_from_keys": (_INT, [_P, _I64, _I32, _P, _P, _P, _SZ, _P]),
    "gn_rowptr_slice": (_INT, [_P, _I32, _I32, _P, _P]),
    "gn_build_chunks_workspace_bytes": (_SZ, [_I32]),
    "gn_build_chunks": (_INT, [_P, _I32, _I32, _P, _P, _P, _I64, _P, _P, _SZ, _P]),
    "gn_gcn_prep_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "gn_gcn_prep": (_INT, [_P, _P, _P, _I64, _I32, _I32, _INT, _F, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                           _P, _P, _P, _P, _SZ, _P]),
    "gn_edge_filter_workspace_bytes": (_SZ, [_I64]),
    "gn_edge_filter": (_INT, [_P, _P, _P, _I64, _INT, _I64, _I64, _P, _P, _P, _P, _I64, _P, _P, _SZ, _P]),
    "gn_gcn_part_workspace_bytes": (_SZ, [_I64, _I32]),
    "gn_gcn_part_structure": (_INT, [_P, _P, _P, _I64, _I32, _I32, _INT, _F, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gn_gcn_part_values": (_INT, [_P, _P, _I32, _I32, _P, _P, _INT, _P, _P]),
    "gn_rgcn_prep_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "gn_rgcn_prep": (_INT, [_P, _P, _I64, _P, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gn_index_prep_workspace_bytes": (_SZ, [_I64, _I32]),
    "gn_index_prep": (_INT, [_P, _I64, _I32, _P, _P, _P, _SZ, _P]),
    "gn_spmm": (_INT, [_CSR, _P, _I64, _I32, _P, _P, _P, _I64, _INT, _P, _I64, _P, _P]),
    "gn_sgemm_workspace_bytes": (_SZ, [_I32, _I32, _I32, _I32, _INT]),
    "gn_sgemm": (_INT, [_INT, _INT, _I32, _I32, _I32, _P, _I64, _P, _I64, _P, _I64, _I32, _I64, _I64, _I64, _INT,
                        _F, _INT, _P, _I64, _P, _I64, _P, _I32, _P, _SZ, _P]),
    "gn_tc_gemm_workspace_bytes": (_SZ, [_I32, _I32, _I32]),
    "gn_tc_gemm": (_INT, [_INT, _I32, _I32, _I32, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _P, _SZ, _P]),
    "gn_tc_gemm_rel_workspace_bytes": (_SZ, [_I32, _I32, _I32, _I32]),
    "gn_tc_gemm_rel": (_INT, [_I32, _I32, _I32, _I32, _P, _I64, _P, _P, _I64, _P, _SZ, _P]),
    "gn_tc_rel_image": (_INT, [_I32, _I32, _I32, _I32, _P, _P, _SZ, _P]),
    "gn_tc_gemm_rel_image": (_INT, [_I32, _I32, _I32, _I32, _P, _I64, _P, _SZ, _P, _I64, _P]),
    "gn_tc_tn_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "gn_tc_tn": (_INT, [_P, _I64, _P, _I64, _I64, _I32, _I32, _P, _I64, _I32, _I64, _P, _SZ, _P]),
    "gn_distmult_fwd": (_INT, [_P, _I64, _I32, _P, _P, _P, _P, _I64, _INT, _P, _P]),
    "gn_distmult_coef": (_INT, [_P, _P, _I64, _INT, _P, _P]),
    "gn_pair_prep_workspace_bytes": (_SZ, [_I64]),
    "gn_pair_prep": (_INT, [_P, _P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _SZ, _P]),
    "gn_distmult_bwd_pairs": (_INT, [_CSR, _P, _P, _P, _P, _I64, _I32, _P, _P, _P]),
    "gn_distmult_grads_workspace_bytes": (_SZ, [_I32, _I32, _I32]),
    "gn_distmult_grads": (_INT, [_P, _P, _I32, _I32, _I32, _P, _I64, _P, _P, _I64, _P, _P, _SZ, _P]),
    "gn_softmax_fwd": (_INT, [_P, _I64, _I32, _P, _P]),
    "gn_softmax_bwd": (_INT, [_P, _P, _I64, _I32, _P, _P]),
    "gn_map2d": (_INT, [_INT, _P, _I64, _P, _I64, _I64, _I32, _P]),
    "gn_relu_bwd": (_INT, [_P, _I64, _P, _I64, _P, _I64, _I64, _I32, _P]),
    "gn_abs_bwd": (_INT, [_P, _I64, _P, _I64, _P, _I64, _I64, _I32, _F, _P]),
    "gn_axpby": (_INT, [_P, _I64, _F, _P, _I64, _F, _P, _I64, _I64, _I32, _P]),
    "gn_zero": (_INT, [_P, _SZ, _P]),
    "gn_mean3": (_INT, [_P, _I64, _P, _I64, _P, _I64, _P, _I64, _I64, _I32, _P]),
    "gn_colsum_workspace_bytes": (_SZ, [_I64, _I32]),
    "gn_colsum": (_INT, [_P, _I64, _I64, _I32, _P, _P, _SZ, _P]),
    "gn_loss_workspace_bytes": (_SZ, [_I64]),
    "gn_lp_loss_fwd": (_INT, [_P, _I64, _P, _I64, _F, _P, _P, _SZ, _P]),
    "gn_lp_loss_bwd": (_INT, [_P, _I64, _P, _I64, _F, _P, _P, _P, _P]),
    "gn_nc_loss_fwd": (_INT, [_P, _I64, _I32, _P, _F, _P, _P, _SZ, _P]),
    "gn_nc_loss_bwd": (_INT, [_P, _I64, _I32, _P, _F, _P, _P, _P]),
    "gn_negsample_table_bytes": (_SZ, [_I64]),
    "gn_negsample_build": (_INT, [_P, _P, _I64, _I64, _P, _I32, _P, _SZ, _P]),
    "gn_negsample_draw": (_INT, [_P, _SZ, _I64, _I64, _P, _I32, C.c_uint64, _P, _P, _P, _P]),
    "gn_adam_max_tensors_per_launch": (_INT, []),
    "gn_adam_step": (_INT, [_P, _I32, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _P, _P]),
    "gn_lp_metrics_workspace_bytes": (_SZ, [_I64, _I64, _I32]),
    "gn_lp_metrics": (_INT, [_P, _I64, _P, _I64, _P, _P, _I32, _P, _P, _SZ, _P]),
    "gn_argmax_rows": (_INT, [_P, _I64, _I64, _I32, _P, _P]),
    "gn_nc_metrics_workspace_bytes": (_SZ, [_I32]),
    "gn_nc_metrics": (_INT, [_P, _P, _I64, _I32, _P, _P, _SZ, _P]),
    "gn_rank_csr_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "gn_rank_csr": (_INT, [_P, _P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gn_rank_query_rows": (_INT, [_P, _I64, _I32, _P, _I32, _P, _P, _P, _I64, _P, _I64, _P]),
    "gn_rank_count": (_INT, [_P, _I64, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "gn_rank_max_hits": (_INT, []),
    "gn_rank_metrics": (_INT, [_P, _P, _P, _I32, _P, _I32, _P, _P]),
    "gn_rank_topk": (_INT, [_P, _I64, _I32, _I32, _P, _P, _I64, _P, _P, _I32, _INT, _P, _P, _P]),
    "gn_rank_pair_csr_workspace_bytes": (_SZ, [_I64]),
    "gn_rank_pair_csr": (_INT, [_P, _P, _P, _I64, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "gn_rank_pair_lookup": (_INT, [_P, _P, _I32, _P, _P, _P, _P, _I64, _P, _P]),
    "gn_rank_pair_rows": (_INT, [_P, _I64, _I32, _P, _P, _P, _P, _I64, _P, _I64, _P]),
    "gn_rank_pair_count": (_INT, [_P, _I64, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gn_rank_pair_topk": (_INT, [_P, _I64, _I32, _I64, _P, _P, _P, _I32, _INT, _P, _P, _P]),
    "gn_rank_rel_pairs_workspace_bytes": (_SZ, [_I64, _I32, _I32]),
    "gn_rank_rel_pairs_select": (_INT, [_P, _I64, _I32, _P, _I32, _I32, _P, _I64, _P, _P, _I32, _P, _SZ, _P]),
    "gn_rank_rel_pairs_merge": (_INT, [_P, _SZ, _I32, _I64, _I32, _INT, _P, _P, _P, _P]),
    "gn_peer_max_world": (_INT, []),
    "gn_peer_allgather": (_INT, [_P, _I32, _I32, _I64, _I64, _I64, _I32, _P, _P, _P, _P]),
    "gn_peer_halo_grid": (_INT, []),
    "gn_peer_halo_push": (_INT, [_P, _I32, _I32, _I64, _I64, _P, _I32, _P, _I64, _I32, _P, _P, _P, _P]),
    "gn_peer_max_segments": (_INT, []),
    "gn_peer_push": (_INT, [_P, _I32, _I32, _I64, _I64, _P, _I32, _I64, _I32, _P, _P, _P, _P]),
    "gn_slot_sum": (_INT, [_P, _I32, _I64, _P, _I32, _P]),
}

GN_ERR_CUDA = -4
EW_COPY, EW_ABS, EW_RELU, EW_ADD = 0, 1, 2, 3
CSR_ROW_IS_CHUNK = 1

_lib = None


def load():
    """Load the shared library (once) and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise GripnetLibraryError(
            f"{LIB_PATH} not found: build it with `python -m gripnet_b200.build` "
            "(nvcc, sm_100a).  gripnet_b200 has no CPU or PyTorch fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise GripnetLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what=""):
    if status != 0:
        msg = load().gn_error_string(status).decode()
        if status == GN_ERR_CUDA and load().gn_last_cuda_error() != 0:
            msg += " [cuda: %s]" % load().gn_last_cuda_error_string().decode()
        raise RuntimeError(f"gripnet_b200: {what or 'call'} failed: {msg} (status {status})")


def launch_count():
    return int(load().gn_launch_count())
