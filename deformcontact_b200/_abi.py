"""ctypes binding of ``libdcb200.so`` — the C ABI declared in ``include/dcb200.h``.

This is the only place Python touches native code.  There is **no fallback**: if the shared
library is missing or a call fails, an exception is raised (the product path never routes
through PyTorch eager or the CPU oracle).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdcb200.so")

DC_OK, DC_EINVAL, DC_ENOSUP, DC_ECUDA, DC_EWORKSPACE = 0, -1, -2, -3, -4
GEMM_AUTO, GEMM_FP32, GEMM_TF32X3, GEMM_PREFER_TC = 0, 1, 2, 3


class DcError(RuntimeError):
    pass


class GemmSeg(C.Structure):
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int64), ("B", C.c_void_p), ("ldb", C.c_int64), ("K", C.c_int64)]


class GemmProblem(C.Structure):
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int64), ("B", C.c_void_p), ("ldb", C.c_int64), ("C", C.c_void_p), ("ldc", C.c_int64),
                ("M", C.c_int64), ("N", C.c_int64), ("K", C.c_int64), ("E", C.c_void_p), ("lde", C.c_int64), ("rowv", C.c_void_p)]


class Hop(C.Structure):
    _fields_ = [("inp", C.c_void_p), ("ldin", C.c_int64), ("add", C.c_void_p), ("ldadd", C.c_int64), ("out", C.c_void_p),
                ("ldout", C.c_int64)]


class SddmmPair(C.Structure):
    _fields_ = [("g", C.c_void_p), ("ldg", C.c_int64), ("h", C.c_void_p), ("ldh", C.c_int64)]


MAX_CHAIN = 4
MAX_SEGS = 4      # dc_gemm: K-segments per call (csrc/gemm.cu); ops.gemm chains larger lists

_p, _i64, _i32, _f32, _sz, _int = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_size_t, C.c_int

# name -> (restype, argtypes); mirrors include/dcb200.h one to one
PROTOTYPES = {
    "dc_version": (_int, []),
    "dc_last_error": (C.c_char_p, []),
    "dc_launch_count": (C.c_uint64, []),
    "dc_csr_build_workspace_bytes": (_sz, [_i64, _i64]),
    "dc_csr_build": (_int, [_p, _i64, _i64, _int, _int, _p, _p, _p, _p, _sz, _p]),
    "dc_deg_inv_sqrt": (_int, [_p, _i64, _int, _p, _p]),
    "dc_spmm": (_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _p, _i64, _p, _i64, _i64, _i32, _int, _p, _int, _p]),
    "dc_edge_weights": (_int, [_p, _p, _p, _i64, _p, _p, _p]),
    "dc_spmm_tiled": (_int, [_p, _p, _p, _p, _p, _i64, _p, _i64, _p, _i64, _i64, _i32, _int, _p, _int, _p, _i64, _i32, _int, _p]),
    "dc_pack_edges": (_int, [_p, _p, _i64, _p, _p]),
    "dc_spmm_lean": (_int, [_p, _p, _p, _p, _i64, _p, _i64, _p, _i64, _i64, _i32, _int, _p, _int, _p, _i64, _i32, _p]),
    "dc_spmm_chain": (_int, [_p, _p, _p, C.POINTER(Hop), _i32, _i64, _i32, _int, _p, _i64, _i32, _p]),
    "dc_spmm_stream": (_int, [_p, _p, C.POINTER(Hop), _i32, _i64, _i32, _p, _i64, _i32, _p]),
    "dc_spmm_stage_supported": (_int, [_i64, _i32]),
    "dc_spmm_stage": (_int, [_p, _p, _p, C.POINTER(Hop), _i32, _i64, _i32, _int, _p, _i64, _i32, _i64, _p]),
    "dc_blocks_workspace_bytes": (_sz, [_i64]),
    "dc_blocks_record_capacity": (_i64, [_i64, _i64, _i64]),
    "dc_blocks_build": (_int, [_p, _p, _p, _p, _i64, _i64, _i32, _p, _p, _i64, _p, _p, _p, _sz, _p]),
    "dc_spmm_blocks": (_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _i64, _p, _i64, _p, _i64, _i32, _int, _p, _int, _int, _p]),
    "dc_edge_relu": (_int, [_p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _int, _p]),
    "dc_gemm_workspace_bytes": (_sz, [_i64, _i64, _i64, _int, _int]),
    "dc_gemm": (_int, [C.POINTER(GemmSeg), _int, _int, _int, _i64, _i64, _p, _i64, _p, _int, _int, _int, _p, _sz, _p]),
    "dc_gemm_batched_workspace_bytes": (_sz, [_i32]),
    "dc_gemm_batched": (_int, [C.POINTER(GemmProblem), _i32, _int, _int, _int, _int, _p, _sz, _p, _sz, _p]),
    "dc_colsum_workspace_bytes": (_sz, [_i64, _i64]),
    "dc_colsum": (_int, [_p, _i64, _i64, _i64, _p, _p, _sz, _p]),
    "dc_edge_loss": (_int, [_p, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p]),
    "dc_rowdot": (_int, [_p, _i64, _p, _i64, _i64, _i64, _p, _p]),
    "dc_softmax_rows": (_int, [_p, _i64, _i64, _i64, _p]),
    "dc_softmax_bwd_rows": (_int, [_p, _i64, _p, _i64, _i64, _i64, _p]),
    "dc_relu_bwd": (_int, [_p, _p, _p, _i64, _p]),
    "dc_relu_bwd_colsum": (_int, [_p, _i64, _p, _i64, _p, _i64, _i64, _i64, _p, _p, _sz, _p]),
    "dc_knn": (_int, [_p, _p, _i64, _i64, _i32, _int, _p, _p]),
    "dc_radius": (_int, [_p, _p, _i64, _i64, _f32, _i32, _int, _p, _p, _p]),
    "dc_knn_grid_workspace_bytes": (_sz, [_i64]),
    "dc_knn_grid": (_int, [_p, _i64, _i32, _int, _p, _p, _p, _sz, _p]),
    "dc_knn_grid_batched_workspace_bytes": (_sz, [_i64, _i64]),
    "dc_knn_grid_batched": (_int, [_p, _p, _i64, _i64, _i32, _int, _p, _p, _sz, _p]),
    "dc_radius_grid_batched": (_int, [_p, _p, _i64, _i64, _f32, _i32, _int, _p, _p, _p, _sz, _p]),
    "dc_radius_grid": (_int, [_p, _i64, _f32, _i32, _int, _p, _p, _p, _p, _sz, _p]),
    "dc_cell_order": (_int, [_p, _i64, _p, _p, _sz, _p]),
    "dc_permute_rows": (_int, [_p, _i64, _p, _p, _i64, _i64, _i32, _p]),
    "dc_nbr_to_edge_index_workspace_bytes": (_sz, [_i64]),
    "dc_nbr_to_edge_index": (_int, [_p, _i64, _i32, _p, _i64, _p, _p, _sz, _p]),
    "dc_mesh_edges": (_int, [_p, _i64, _i64, _p, _i64, _i64, _p]),
    "dc_posenc": (_int, [_p, _i64, _p, _i64, _i32, _p]),
    "dc_batch_vector": (_int, [_p, _i64, _i64, _p, _p]),
    "dc_edges_offset": (_int, [_p, _i32, _i64, _p, _p, _i64, _i64, _p, _i64, _p]),
    "dc_mesh_edges_batched": (_int, [_p, _i32, _p, _p, _i64, _i64, _i64, _i64, _p, _i64, _p]),
    "dc_node_features": (_int, [_p, _p, _i32, _p, _i64, _i64, _p, _i64, _p]),
    "dc_instance_points": (_int, [_p, _p, _i64, _i64, _p, _p]),
    "dc_gat_scores": (_int, [_p, _i64, _i64, _i32, _i32, _p, _p, _p, _p, _p]),
    "dc_gat_softmax": (_int, [_p, _p, _p, _p, _p, _f32, _i64, _p, _p, _p]),
    "dc_gat_bwd_edge": (_int, [_p, _p, _p, _p, _p, _f32, _p, _p, _p, _i64, _p, _i64, _i32, _i64, _p, _p, _p, _p]),
    "dc_segment_sum": (_int, [_p, _p, _p, _p, _i64, _p, _p]),
    "dc_gat_aggregate": (_int, [_p, _p, _p, _p, _i64, _p, _p, _f32, _i32, _i32, _i32, _p, _i32, _i64, _p, _i64, _p, _p, _p]),
    "dc_gat_bwd_edge_heads": (_int, [_p, _p, _p, _p, _p, _f32, _p, _p, _p, _i64, _p, _i64, _i64, _f32, _i32, _i32, _i64, _p, _p, _p,
                                     _p]),
    "dc_gat_bwd_edge_heads_ext": (_int, [_p, _p, _p, _p, _p, _f32, _p, _p, _p, _i64, _p, _i64, _i64, _f32, _i32, _i32, _i64, _p, _p,
                                         _p, _p, _p, _p]),
    "dc_gat_scatter_heads": (_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _f32, _i32, _i32, _i64, _p, _i64, _p,
                                    _p]),
    "dc_gat_att_grad_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "dc_gat_att_grad": (_int, [_p, _i64, _p, _p, _i64, _i32, _i32, _p, _p, _p, _sz, _p]),
    "dc_gcn_norm_weighted": (_int, [_p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _f32, _int, _int, _p, _p, _p, _p, _p, _p, _p, _p,
                                    _p]),
    "dc_edge_sddmm": (_int, [_p, _p, _p, C.POINTER(SddmmPair), _i32, _i64, _i32, _int, _p, _p, _p]),
    "dc_gcn_norm_weighted_backward": (_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _p, _p]),
}

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DcError(f"{LIB_PATH} not found - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or `make -C deformcontact_b200/csrc`). There is no fallback path.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the header and the library disagree
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc, what):
    if rc != DC_OK:
        msg = lib().dc_last_error()
        raise DcError(f"{what} failed with status {rc}: {msg.decode() if msg else ''}")


def call(name, *args):
    check(getattr(lib(), name)(*args), name)
