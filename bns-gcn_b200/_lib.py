"""ctypes binding of ``csrc/libbnsgcn.so`` (the C ABI declared in ``include/bnsgcn.h``).

There is deliberately no fallback: if the shared library is missing or does not export a symbol the
header declares, importing this module raises.  Build it with ``python __graft_entry__.py`` (or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libbnsgcn.so")

ABI_VERSION = 3
P2P_HANDLE_BYTES = 64
COMM_ID_BYTES = 128

MAX_PEERS = 16      # BNS_MAX_PEERS


class EpochMaps(Structure):          # bns_epoch_maps
    _fields_ = [("n_seg", c_int32), ("sel_begin", c_int64 * (MAX_PEERS + 1)), ("hop_begin", c_int64 * (MAX_PEERS + 1)),
                ("pos", c_void_p * MAX_PEERS), ("inv", c_void_p * MAX_PEERS), ("selected_cat", c_void_p),
                ("one_hops_cat", c_void_p), ("slot", c_void_p), ("n_in", c_int64)]


class PutAll(Structure):             # bns_put_all
    _fields_ = [("n_seg", c_int32), ("row_begin", c_int64 * (MAX_PEERS + 1)), ("peer", c_int32 * MAX_PEERS),
                ("remote_off", c_uint64 * MAX_PEERS), ("src_begin", c_int64 * MAX_PEERS), ("div", c_float * MAX_PEERS)]


class DeriveEntry(Structure):        # bns_derive_entry
    _fields_ = [("op", c_int32), ("rows", c_int32), ("cols", c_int32), ("ld_a", c_int32), ("ld_dst", c_int32),
                ("pad_", c_int32), ("a", c_void_p), ("b", c_void_p), ("dst", c_void_p)]


# name -> (restype, argtypes); must list every function of include/bnsgcn.h (tests check this)
SIGNATURES = {
    "bns_abi_version": (c_int, []),
    "bns_last_error": (c_char_p, []),
    "bns_launch_count": (c_uint64, []),
    "bns_device_info": (c_int, [c_char_p, c_size_t, POINTER(c_int), POINTER(c_int64), POINTER(c_int), POINTER(c_int)]),
    "bns_graph_create": (c_int, [POINTER(c_void_p), c_int64, c_int64, c_int64, c_void_p, c_void_p, c_int32, c_void_p]),
    "bns_graph_transpose": (c_int, [c_void_p, POINTER(c_void_p), c_void_p]),
    "bns_graph_destroy": (c_int, [c_void_p]),
    "bns_graph_info": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64),
                               POINTER(c_int64)]),
    "bns_graph_copy_csr": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "bns_spmm_workspace_bytes": (c_size_t, [c_void_p, c_int64]),
    "bns_spmm_sum_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_int64, c_int64, c_int32, c_int, c_void_p, c_size_t, c_void_p]),
    "bns_sddmm_dot_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64,
                                  c_void_p, c_int64, c_void_p]),
    "bns_graph_copy_perm": (c_int, [c_void_p, c_void_p, c_void_p]),
    "bns_gather_div_f32": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_float, c_void_p, c_int64, c_void_p]),
    "bns_scatter_add_div_f32": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_float, c_void_p, c_int64,
                                        c_void_p]),
    "bns_copy_rows_f32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "bns_sample_workspace_bytes": (c_size_t, [c_int64]),
    "bns_sample_boundary": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int64, c_int64, c_uint64, c_uint64,
                                    c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "bns_ln_bwd_workspace_bytes": (c_size_t, [c_int64]),
    "bns_ln_relu_dropout_fwd_f32": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_float, c_float,
                                            c_uint64, c_uint64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "bns_ln_relu_dropout_bwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                            c_void_p, c_void_p, c_float, c_float, c_uint64, c_uint64, c_void_p, c_void_p,
                                            c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "bns_dense_tn_3xtf32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                    c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "bns_colsum_workspace_bytes": (c_size_t, [c_int64]),
    "bns_colsum_f32": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "bns_dense_nt_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "bns_dense_nt_3xtf32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                    c_void_p, c_size_t, c_void_p]),
    "bns_fill_i32": (c_int, [c_void_p, c_int64, c_int32, c_void_p]),
    "bns_halo_slot_update": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p]),
    "bns_p2p_create": (c_int, [POINTER(c_void_p), c_int32, c_int32, c_size_t, c_int32]),
    "bns_p2p_destroy": (c_int, [c_void_p]),
    "bns_p2p_local": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_size_t)]),
    "bns_p2p_export": (c_int, [c_void_p, c_void_p]),
    "bns_p2p_import": (c_int, [c_void_p, c_int32, c_void_p, c_size_t]),
    "bns_p2p_set_peer": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_size_t]),
    "bns_p2p_put_rows_f32": (c_int, [c_void_p, c_int32, c_size_t, c_int64, c_void_p, c_int64, c_int64, c_void_p,
                                     c_int64, c_float, c_int32, c_uint64, c_void_p, c_void_p]),
    "bns_p2p_wait_flag": (c_int, [c_void_p, c_int32, c_uint64, c_void_p, c_void_p]),
    # ---- ABI 2 ----
    "bns_epoch_maps_update": (c_int, [POINTER(EpochMaps), c_void_p, c_size_t, c_void_p]),
    "bns_graph_compact_cols": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "bns_gat_colsum_f32": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_void_p]),
    "bns_spmm_weighted_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int,
                                      c_void_p, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "bns_spmm_compact_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p,
                                     c_int64, c_void_p, c_int64, c_int32, c_int, c_void_p, c_size_t, c_void_p]),
    "bns_gat_proj_f32": (c_int, [c_void_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "bns_gat_proj_bwd_f32": (c_int, [c_void_p, c_int64, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_int64,
                                     c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "bns_gat_scores_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p,
                                   c_float, c_float, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "bns_gat_softmax_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p,
                                        c_float, c_float, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p]),
    "bns_p2p_put_all_f32": (c_int, [c_void_p, POINTER(PutAll), c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int32,
                                    c_int32, c_uint64, c_void_p, c_void_p]),
    "bns_p2p_put_ids_i64": (c_int, [c_void_p, c_int32, POINTER(c_int64), POINTER(c_int32), POINTER(c_uint64), c_void_p,
                                    c_int32, c_int32, c_uint64, c_void_p, c_void_p]),
    "bns_p2p_wait_all": (c_int, [c_void_p, c_int32, POINTER(c_int32), c_uint64, c_void_p, c_void_p]),
    "bns_scatter_rows_all_f32": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int32, POINTER(c_void_p), POINTER(c_void_p),
                                         c_int64, POINTER(c_float), c_void_p]),
    "bns_xent_workspace_bytes": (c_size_t, []),
    "bns_xent_f32": (c_int, [c_void_p, c_int64, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_void_p, c_float, c_void_p,
                             c_void_p, c_int64, c_int32, c_void_p, c_size_t, c_void_p]),
    "bns_derive_entry_bytes": (c_size_t, []),
    "bns_adam_step_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float,
                                  c_float, c_void_p, c_void_p]),
    "bns_derive_refresh": (c_int, [c_void_p, c_int32, c_void_p, c_void_p]),
    "bns_bn_workspace_bytes": (c_size_t, [c_int64]),
    "bns_bn_colsums_f32": (c_int, [c_int, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_size_t, c_void_p]),
    "bns_bn_apply_f32": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_float, c_float, c_void_p, c_void_p, c_float,
                                 c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "bns_bn_bwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_float, c_void_p, c_int64, c_void_p]),
    "bns_comm_unique_id": (c_int, [c_void_p]),
    "bns_ctx_create": (c_int, [POINTER(c_void_p), c_int32, c_int32, c_void_p]),
    "bns_ctx_destroy": (c_int, [c_void_p]),
    "bns_allreduce_sum_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "bns_alltoallv_f32": (c_int, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_void_p, POINTER(c_int64),
                                  POINTER(c_int64), c_int64, c_void_p]),
    "bns_alltoallv_i64": (c_int, [c_void_p, c_void_p, POINTER(c_int64), POINTER(c_int64), c_void_p, POINTER(c_int64),
                                  POINTER(c_int64), c_void_p]),
    "bns_alltoallv_bytes": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_int64), POINTER(c_void_p), POINTER(c_int64),
                                    c_void_p]),
    "bns_dropout_f32": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_float, c_uint64, c_uint64, c_void_p, c_void_p,
                                c_int64, c_void_p]),
    "bns_scale_rows_f32": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
}


class BnsError(RuntimeError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. Run `python __graft_entry__.py` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise ImportError(f"{LIB_PATH} does not export {name} (declared in include/bnsgcn.h)") from e
        fn.restype, fn.argtypes = res, args
    if lib.bns_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.bns_abi_version()} != {ABI_VERSION}; rebuild")
    return lib


lib = _load()


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib.bns_last_error()
        raise BnsError(f"{what or 'libbnsgcn'} failed ({rc}): {msg.decode() if msg else ''}")
