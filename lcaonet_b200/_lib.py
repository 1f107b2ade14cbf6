"""ctypes binding of liblcao_b200.so (the C ABI declared in include/lcao_b200.h).

The product path has NO fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "liblcao_b200.so")

MAX_UNIQUE_ORB, MAX_POLY = 18, 8
CUT = {"polynomial": 0, "envelope": 1, "cosine": 2}
RBF = {"hydrogen": 0, "sphericalbessel": 1}
ACT_NONE, ACT_SILU = 0, 1
# include/lcao_b200.h LCAO_ACT_*: the parameter-free activations fused into the kernels
ACT = {"none": 0, "silu": 1, "shiftedsoftplus": 2, "softplus": 3, "relu": 4, "tanh": 5, "sigmoid": 6, "gelu": 7, "elu": 8,
       "leakyrelu": 9}
GEMM_FP32, GEMM_TF32X3, GEMM_TF32 = 0, 1, 2
CELL_CHUNK = 128  # LCAO_CELL_CHUNK: nodes per partial of lcao_geom_cell_bwd (its scratch is (N // 128 + B) * 18 doubles)


class BasisSpec(C.Structure):
    _fields_ = [("n_unique", C.c_int32), ("n_rep", C.c_int32), ("cutoff_kind", C.c_int32), ("rbf_kind", C.c_int32),
                ("rc", C.c_double), ("a0", C.c_double),
                ("n", C.c_int32 * MAX_UNIQUE_ORB), ("l", C.c_int32 * MAX_UNIQUE_ORB), ("deg", C.c_int32 * MAX_UNIQUE_ORB),
                ("norm", C.c_double * MAX_UNIQUE_ORB), ("poly", (C.c_double * MAX_POLY) * MAX_UNIQUE_ORB)]


class LcaoError(RuntimeError):
    pass


_p, _i32, _i64 = C.c_void_p, C.c_int32, C.c_int64
# name -> argtypes (must mirror include/lcao_b200.h; tests/test_abi.py checks every symbol is exported)
SIGNATURES = {
    "lcao_bucket_sort": [_p, _p, _i64, _i64, _p, _p, _p, _i32, _p],
    "lcao_validate_graph": [_p, _i64, _i64, _p, _i64, _p, _i64, _p, _p],
    "lcao_graph_index_build": [_p, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "lcao_triplet_offsets": [_p, _p, _p, _i64, _p, _p, _p],
    "lcao_triplets_fill": [_p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p],
    "lcao_histogram": [_p, _i64, _i64, _p, _p],
    "lcao_neighbor_count": [_p, _p, _p, _p, _p, _i64, C.c_double, _p, _p],
    "lcao_neighbor_fill": [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, C.c_double, _i32, _p, _p, _p, _p],
    "lcao_geom_basis_fwd": [_p, _p, _p, _p, _p, _p, _i64, C.POINTER(BasisSpec), _p, _p, _p, _p, _p],
    "lcao_geom_basis_bwd": [_p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _p, _p, _p],
    "lcao_geom_cell_bwd": [_p, _p, _p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p, _i64, _p, _p, _p, _p],
    "lcao_coeff_contract_fwd": [_p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p],
    "lcao_coeff_contract_bwd": [_p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p, _p],
    "lcao_pair_contract_fwd": [_p, _p, _p, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p, _p, _p],
    "lcao_pair_contract_bwd": [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _i32, _i32, _i32, _p, _p, _p, _p],
    "lcao_coeff_gram": [_p, _i32, _i64, _i32, _i32, _p, _p],
    "lcao_table_norm_fwd": [_p, _p, _p, _p, _i64, _i32, C.c_float, C.c_float, _i32, _p, _p, _p, _p, _p, _p, _p],
    "lcao_table_norm_bwd": [_p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _p],
    "lcao_pair_outer_fwd": [_p, _p, _p, _i32, _i32, _i32, _p, _p],
    "lcao_pair_outer_bwd": [_p, _p, _p, _p, _i32, _i32, _i32, _p, _p, _p, _p],
    "lcao_sigmoid_rows": [_p, _i64, _p, _i64, _i64, _i32, _p],
    "lcao_threebody_fwd": [_p, _i32, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _i64, _i64, _i32, _i32, _p, _p],
    "lcao_threebody_bwd": [_p, _i32, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _i64, _i64, _i32, _i32, _p, _p, _p, _p, _p,
                           _p, _p],
    "lcao_twobody_fwd": [_p, _i32, _p, _i64, _i32, _i32, _i32, _p, _p],
    "lcao_twobody_bwd": [_p, _i32, _p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p, _p],
    "lcao_edge_pair_fwd": [_p, _i64, _p, _i64, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p],
    "lcao_segment_sum": [_p, _i64, _p, _i64, _p, _p, _i64, _i32, _i32, _p, _i64, _p],
    "lcao_msg_bwd": [_p, _i64, _p, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p],
    "lcao_gather_rows": [_p, _i64, _p, _i32, _p, _i64, _i64, _i32, _p, _i64, _p],
    "lcao_reduce_by_key": [_p, _i64, _p, _p, _i64, _i64, _i32, _p, _p],
    "lcao_linear_fwd": [_p, _i64, _p, _p, _p, _i64, _p, _i64, _i64, _i32, _i32, _i32, _i32, _p],
    "lcao_linear_dgrad": [_p, _i64, _p, _i64, _i32, _p, _p, _i64, _i64, _i32, _i32, _i32, _i32, _p, _p],
    "lcao_linear_dgrad_act": [_p, _i64, _p, _p, _i64, _i32, _p, _i64, _i64, _i32, _i32, _i32, _p],
    "lcao_linear_wgrad": [_p, _i64, _p, _i64, _i32, _p, _i64, _p, _p, _i64, _i32, _i32, _i32, _p, _p],
    "lcao_linear_wgrad_deferred": [_p, _i64, _p, _i64, _p, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _p],
    "lcao_wgrad_reduce_batch": [_p, _i32, _p],
    "lcao_act_bwd": [_p, _i64, _p, _i64, _p, _i64, _i64, _i32, _i32, _p],
    "lcao_act_fwd": [_p, _i64, _p, _i64, _i64, _i32, _i32, _p],
}

_lib = None


def load():
    """Load (once) and return the CDLL; raises LcaoError when the CUDA library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LcaoError(f"{LIB_PATH} not found: build it with `python -m lcaonet_b200.csrc.build` "
                        "(there is no CPU or PyTorch fallback for the LCAO hot path)")
    lib = C.CDLL(LIB_PATH)
    lib.lcao_version.restype = C.c_int
    lib.lcao_last_error.restype = C.c_char_p
    lib.lcao_launch_count.restype = C.c_int64
    lib.lcao_linear_bwd_scratch.restype = C.c_int64
    lib.lcao_linear_bwd_scratch.argtypes = [_p, _i64, _p, _i64, _i32, _p, _p, _i64, _p, _i64, _i64, _i32, _i32, _i32]
    lib.lcao_pair_contract_bwd_scratch.restype = C.c_int64
    lib.lcao_pair_contract_bwd_scratch.argtypes = [_i64, _i64, _i32, _i32, _i32]
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    _lib = lib
    return lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    """raw cudaStream_t of torch's current stream on the current device (the fast C accessor: the
    torch.cuda.current_stream() object path costs ~15 us per call)"""
    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())


def call(name: str, *args):
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise LcaoError(f"{name} failed ({rc}): {lib.lcao_last_error().decode()}")


def launch_count() -> int:
    return int(load().lcao_launch_count())


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise LcaoError("lcaonet_b200 runs on CUDA (sm_100a) tensors only; got a CPU tensor. "
                            "Move the model and the batch to a B200 (`.to('cuda')`): there is no CPU fallback.")
