"""ctypes binding of libmemento_b200.so (the C ABI in include/memento_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, an exception is raised.
Tensors are passed as raw device pointers (``tensor.data_ptr()``); the current torch CUDA stream of
the tensor's device is used for every launch.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmemento_b200.so")

_i32, _i64, _u64, _vp = C.c_int32, C.c_int64, C.c_uint64, C.c_void_p

# name -> argument ctypes after the leading (device, stream); every function returns int status
SIGNATURES = {
    "mm_csr_row_sums": [_vp, _vp, _vp, _i64, _vp, _vp],
    "mm_seg_moments": [_vp, _vp, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _vp],
    "mm_validate_counts": [_vp, _i64, _vp],
    "mm_upload": [_vp, _vp, _i64, _i32],
    "mm_csr_check_sorted": [_vp, _vp, _i64, _vp],
    "mm_relayout_count": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _i64],
    "mm_relayout_fill": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _i64],
    "mm_block_panels": [_vp, _vp, _vp, _i32, _i32, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp],
    "mm_cell_weights": [_vp, _i32, _i64, _u64, C.c_uint32, _vp],
    "mm_seg_weighted_stats": [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "mm_block_boot_update": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _i64],
    "mm_block_boot_finish": [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp],
    "mm_block_gemm": [_vp, _vp, _i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i64],
    "mm_block_scaling": [_vp, _i32, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _vp],
    "mm_block_cross_batch": [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp,
                             _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i64, _i64],
    "mm_pair_products": [_vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp],
    "mm_seg_unique": [_vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp,
                      _vp, _vp, _vp, _vp],
    "mm_bootstrap_1d": [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _u64, _vp, _vp, _vp, _vp,
                        _vp, _vp, _i32, _vp, _vp],
    "mm_poisson_tables": [_i32, _vp, _vp, _vp, _vp, _vp],
    "mm_boot_prepare": [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp, C.c_float],
    "mm_bootstrap_1d_replay": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp],
    "mm_fill_log": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _u64, _vp, _vp, _vp, _vp, _vp],
    "mm_wls_functional": [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp],
    "mm_regress_resampled": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _u64, _vp, _vp,
                             _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32],
    "mm_pair_unique": [_vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                       _vp],
    "mm_pair_prepare": [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _vp],
    "mm_pair_bootstrap": [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _u64, _vp, _vp, _vp, _vp],
    "mm_pair_bootstrap_replay": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp],
    "mm_gev_tail_asl": [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32],
    "mm_regress_asl": [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp,
                       _vp],
}

# host-only helpers (no leading device / stream arguments)
HOST_SIGNATURES = {"mm_poisson_table_size": [_i32, _vp, _vp], "mm_launch_count": [], "mm_reload_tuning": [], "mm_upload_release": []}

_lib = None


class MementoCudaError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MementoCudaError(
            "libmemento_b200.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` or `make -C scrna-parameter-estimation_b200/csrc`; there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.mm_last_error.restype = C.c_char_p
    lib.mm_version.restype = C.c_int
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = [C.c_int, _vp] + args
    for name, args in HOST_SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int64 if name == "mm_launch_count" else C.c_int
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        assert t.is_cuda and t.is_contiguous(), "device-resident contiguous tensor required"
        return t.data_ptr()
    return t


def call(name, device, *args):
    """Invoke ``name`` on ``device`` (torch.device or index) on that device's current stream."""
    lib = load()
    idx = device.index if isinstance(device, torch.device) else int(device)
    stream = torch.cuda.current_stream(idx).cuda_stream
    conv = [_ptr(a) if (a is None or isinstance(a, torch.Tensor)) else a for a in args]
    status = getattr(lib, name)(idx, stream, *conv)
    if status != 0:
        raise MementoCudaError("%s failed (status %d): %s" % (name, status, lib.mm_last_error().decode()))


def launch_count():
    """Kernels launched by the library in this process so far (counted at every launch site in csrc/)."""
    return int(load().mm_launch_count())


def reload_tuning():
    """Re-read the MM_MOMENTS_KERNEL test hook (otherwise read once, at library load; include/memento_b200.h)."""
    load().mm_reload_tuning()


def poisson_table_offsets(n_max):
    """Host helper: (offsets int32[n_max + 1], total) of the universal Poisson inversion tables."""
    import numpy as np
    lib = load()
    off = np.zeros(n_max + 1, dtype=np.int32)
    total = C.c_int64(0)
    status = lib.mm_poisson_table_size(n_max, off.ctypes.data, C.addressof(total))
    if status != 0:
        raise MementoCudaError("mm_poisson_table_size failed: %s" % lib.mm_last_error().decode())
    return off, int(total.value)
