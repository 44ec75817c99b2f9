"""ctypes binding of libb200lanczos.so — the only way the host layer reaches the GPU.

There is NO CPU fallback: if the library cannot be loaded every entry point raises
`RuntimeError` (the product path must fail loudly when the CUDA extension is missing).
Signatures mirror `include/b200_lanczos.h`.
"""

from __future__ import annotations

import ctypes as C
import os

from experiments_lanczos_adjoints_b200 import build as _build

BL_F32, BL_F64 = 0, 1
BL_OK, BL_EINVAL, BL_EDEPTH, BL_ECUDA, BL_ENOMEM, BL_ECALLBACK = range(6)

ALLREDUCE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p)
MATVEC_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p)
VJP_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p)

_vp, _i64, _i32, _sz, _dbl = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_double
_pvp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); every symbol declared in include/b200_lanczos.h
SIGNATURES = {
    "bl_last_error": (C.c_char_p, []),
    "bl_version": (C.c_char_p, []),
    "bl_device_count": (_i32, [C.POINTER(C.c_int)]),
    "bl_set_device": (_i32, [_i32]),
    "bl_get_device": (_i32, [C.POINTER(C.c_int)]),
    "bl_device_sm_count": (_i32, [C.POINTER(C.c_int)]),
    "bl_malloc": (_i32, [_pvp, _sz]),
    "bl_free": (_i32, [_vp]),
    "bl_host_alloc": (_i32, [_pvp, _sz]),
    "bl_host_free": (_i32, [_vp]),
    "bl_memcpy_h2d": (_i32, [_vp, _vp, _sz, _vp]),
    "bl_memcpy_d2h": (_i32, [_vp, _vp, _sz, _vp]),
    "bl_memcpy_d2d": (_i32, [_vp, _vp, _sz, _vp]),
    "bl_memset": (_i32, [_vp, _i32, _sz, _vp]),
    "bl_stream_create": (_i32, [_pvp]),
    "bl_stream_destroy": (_i32, [_vp]),
    "bl_stream_sync": (_i32, [_vp]),
    "bl_device_sync": (_i32, []),
    "bl_event_create": (_i32, [_pvp]),
    "bl_event_destroy": (_i32, [_vp]),
    "bl_event_record": (_i32, [_vp, _vp]),
    "bl_stream_wait_event": (_i32, [_vp, _vp]),
    "bl_event_sync": (_i32, [_vp]),
    "bl_event_elapsed_ms": (_i32, [_vp, _vp, C.POINTER(C.c_float)]),
    "bl_launch_count": (_i32, [C.POINTER(C.c_uint64)]),
    "bl_set_blocks_per_sm": (_i32, [_i32]),
    "bl_get_blocks_per_sm": (_i32, [C.POINTER(C.c_int)]),
    "bl_profile_begin": (_i32, []),
    "bl_profile_end": (_i32, [C.POINTER(C.c_uint64), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "bl_dist_set_reduce_hook": (_i32, [ALLREDUCE_CB, _vp]),
    "bl_dist_comm_create": (_i32, [_i32, _i32, _pvp]),
    "bl_dist_comm_local": (_i32, [_vp, _pvp, _vp]),
    "bl_dist_comm_connect_ipc": (_i32, [_vp, _vp]),
    "bl_dist_comm_connect_ptrs": (_i32, [_vp, _pvp]),
    "bl_dist_comm_activate": (_i32, [_vp]),
    "bl_dist_comm_window_create": (_i32, [_vp, C.c_size_t, _vp]),
    "bl_dist_comm_window_local": (_i32, [_vp, _pvp]),
    "bl_dist_comm_window_connect_ipc": (_i32, [_vp, _vp]),
    "bl_dist_comm_window_connect_ptrs": (_i32, [_vp, _pvp]),
    "bl_op_sharded_sparse_create": (_i32, [_vp, _vp, _vp, _i64, _i64, _pvp]),
    "bl_dist_comm_error": (_i32, [_vp, C.POINTER(C.c_int)]),
    "bl_dist_comm_destroy": (_i32, [_vp]),
    "bl_op_wave_set_comm": (_i32, [_vp, _vp]),
    "bl_arnoldi_forward_batch": (_i32, [_vp, _i32, _i64, _i64, _i32, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp,
                                        C.c_size_t, _vp]),
    "bl_arnoldi_adjoint_batch": (_i32, [_vp, _i32, _i64, _i64, _i32, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _i64, _vp, _vp, C.c_size_t, _vp]),
    "bl_op_deferred_grad": (_i32, [_vp, _i32, C.POINTER(C.c_int)]),
    "bl_dist_nccl_available": (_i32, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "bl_dist_nccl_unique_id": (_i32, [_vp]),
    "bl_dist_nccl_init": (_i32, [_vp, _i32, _i32, _pvp]),
    "bl_dist_nccl_allreduce": (_i32, [_vp, _vp, _i64, _i32, _i32, _vp]),
    "bl_dist_nccl_allgather": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp]),
    "bl_dist_nccl_sendrecv": (_i32, [_vp, _vp, _i32, _vp, _i32, _i64, _i32, _vp]),
    "bl_dist_nccl_reduce_hook": (_i32, [_vp]),
    "bl_dist_nccl_destroy": (_i32, [_vp]),
    "bl_step_trace_begin": (_i32, []),
    "bl_step_trace_end": (_i32, [_vp, _i64, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "bl_precond_create": (_i32, [_i32, _i64, _i64, _vp, _i64, _vp, _pvp]),
    "bl_precond_set_shift": (_i32, [_vp, C.c_double, _vp]),
    "bl_precond_apply": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "bl_precond_destroy": (_i32, [_vp]),
    "bl_pcg_workspace_bytes": (C.c_size_t, [_i64, _i32]),
    "bl_pcg_solve": (_i32, [_vp, _i32, _i64, _vp, _vp, _i64, _i64, C.c_double, C.c_double, _i32, _vp, _vp,
                            C.POINTER(C.c_int64), _vp, C.c_size_t, _vp]),
    "bl_pcg_batch_workspace_bytes": (C.c_size_t, [_i64, _i64, _i32]),
    "bl_pcg_solve_batch": (_i32, [_vp, _i32, _i64, _i64, _vp, _i64, _vp, _i64, _i64, C.c_double, C.c_double, _i32, _vp,
                                  _vp, C.POINTER(C.c_int64), _vp, C.c_size_t, _vp]),
    "bl_rows_dot_pairs": (_i32, [_i32, _i64, _i64, _vp, _vp, _i64, _vp, _vp]),
    "bl_cholesky_workspace_bytes": (C.c_size_t, [_i64, _i64, _i32]),
    "bl_cholesky_partial": (_i32, [_vp, _i32, _i64, _i64, _i32, _vp, _i64, C.POINTER(C.c_int), C.POINTER(C.c_int64),
                                   _vp, C.c_size_t, _vp]),
    "bl_op_sparse_create": (_i32, [_i64, _i64, _i64, _vp, _vp, _pvp]),
    "bl_op_sparse_clone": (_i32, [_vp, _pvp]),
    "bl_op_sparse_export_csr": (_i32, [_vp, _vp, _vp, _vp]),
    "bl_op_sparse_export_sell": (_i32, [_vp, _i32, _vp, _vp]),
    "bl_op_dense_create": (_i32, [_i64, _i32, _pvp]),
    "bl_op_gram_create": (_i32, [_i64, _i64, _i32, _vp, _pvp]),
    "bl_op_gram_set_path": (_i32, [_vp, _i32]),
    "bl_op_gram_tile_distances": (_i32, [_vp, _i64, _i64, _vp, _vp]),
    "bl_gram_cross_create": (_i32, [_vp, _i64, _vp, _pvp]),
    "bl_gram_cross_destroy": (_i32, [_vp]),
    "bl_gram_cross_matvec": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "bl_gram_cross_columns": (_i32, [_vp, _i32, _i64, _i64, _vp, _i64, _vp]),
    "bl_gram_cross_prior_diag": (_i32, [_vp, _i32, _vp, _vp]),
    "bl_op_wave_create": (_i32, [_i64, _vp, _pvp]),
    "bl_op_wave_slab_create": (_i32, [_i64, _i64, _i32, _i32, _vp, _pvp]),
    "bl_op_wave_halo": (_i32, [_vp, _i32, _pvp]),
    "bl_op_callback_create": (_i32, [_i64, MATVEC_CB, VJP_CB, _vp, _pvp]),
    "bl_op_destroy": (_i32, [_vp]),
    "bl_op_size": (_i32, [_vp, C.POINTER(C.c_int64)]),
    "bl_op_num_params": (_i32, [_vp, C.POINTER(C.c_int)]),
    "bl_op_param_size": (_i32, [_vp, _i32, C.POINTER(C.c_int64)]),
    "bl_op_set_params": (_i32, [_vp, _i32, _pvp, _i32, _vp]),
    "bl_op_matvec": (_i32, [_vp, _i32, _vp, _vp, _vp]),
    "bl_op_vjp": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp]),
    "bl_op_grad_zero": (_i32, [_vp, _i32, _vp]),
    "bl_op_grad_export": (_i32, [_vp, _i32, _pvp, _i32, _vp]),
    "bl_arnoldi_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "bl_arnoldi_forward": (_i32, [_vp, _i32, _i64, _i64, _i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bl_arnoldi_adjoint": (
        _i32,
        [_vp, _i32, _i64, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp],
    ),
    "bl_lanczos3_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "bl_lanczos3_forward": (_i32, [_vp, _i32, _i64, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "bl_lanczos3_adjoint": (
        _i32,
        [_vp, _i32, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp],
    ),
    "bl_vec_dot": (_i32, [_i32, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "bl_vec_axpby": (_i32, [_i32, _i64, _dbl, _vp, _dbl, _vp, _vp, _vp]),
    "bl_transpose": (_i32, [_i32, _i64, _i64, _vp, _i64, _vp, _i64, _vp]),
    "bl_rows_dot": (_i32, [_i32, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "bl_rows_combine": (_i32, [_i32, _i64, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _sz, _vp]),
    "bl_vec_workspace_bytes": (_sz, []),
}

_lib = None
_load_error = None


def library_path() -> str:
    return _build.LIB


def load():
    """Load (building first if the sources changed and nvcc is present) the CUDA library."""
    global _lib, _load_error
    if _lib is not None:
        return _lib
    if _load_error is not None:
        raise RuntimeError(_load_error)
    try:
        path = _build.build()
        lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    except Exception as exc:  # no fallback: surface the failure on every use
        _load_error = (
            f"libb200lanczos.so is not available ({exc}); this package has no CPU fallback. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` on a machine with nvcc."
        )
        raise RuntimeError(_load_error) from exc
    _lib = lib
    return lib


class BLError(RuntimeError):
    pass


def check(rc: int):
    """Translate a BL_E* code into the exception the reference raises for that mistake."""
    if rc == BL_OK:
        return
    msg = load().bl_last_error().decode()
    if rc == BL_EDEPTH:
        raise ValueError(msg)  # arnoldi.py:58-60 -> ValueError mentioning "depth"
    if rc == BL_EINVAL:
        raise ValueError(msg)
    if rc == BL_ENOMEM:
        raise MemoryError(msg)
    raise BLError(f"libb200lanczos error {rc}: {msg}")


def call(name: str, *args):
    check(getattr(load(), name)(*args))
