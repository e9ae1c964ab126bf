"""ctypes loader of libswd_b200.so (the C-ABI in include/swd_b200.h).

There is no CPU fallback: if the CUDA library is missing or no GPU is visible the decoders raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SWD_LIB", os.path.join(_HERE, "libswd_b200.so"))


class SwdConfig(C.Structure):
    _fields_ = [("kind", C.c_int), ("device", C.c_int),
                ("max_iter", C.c_int), ("ms_scaling_factor", C.c_double),
                ("max_iter_per_step", C.c_int), ("max_step", C.c_int),
                ("max_tree_depth", C.c_int), ("max_side_depth", C.c_int),
                ("max_tree_branch_step", C.c_int), ("max_side_branch_step", C.c_int),
                ("gdg_factor", C.c_double), ("new_n", C.c_int),
                ("multi_thread", C.c_int), ("low_error_mode", C.c_int),
                ("post_max_iter", C.c_int), ("osd_method", C.c_int), ("osd_order", C.c_int), ("bp_method", C.c_int)]


class SwdCounters(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("shots", "pre_bp_edge_iters", "path_edge_iters", "gdg_shots", "osd_shots",
                                          "kernel_launches", "paths_run", "bp_calls", "path_vn_iters", "path_cn_iters",
                                          "path_slot_iters", "osd_cols_scanned", "osd_pivots")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


KIND_BPGDG, KIND_BPGD, KIND_OSD_WINDOW = 0, 1, 2
KERNEL_CLASSES = ["pre_bp", "sort_reset", "path_main", "path_side", "select", "osd", "path_trunk", "post_bp"]
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOMEM = 0, -1, -2, -3, -4

_vp, _i32p, _u8p, _dp, _f64p = C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.POINTER(C.c_double)
_vpp = C.POINTER(_vp)
_i = C.c_int

# name -> (restype, argtypes) of every exported symbol (argtypes None: left unset)
_SIGNATURES = {
    "swd_create": (_i, [C.POINTER(SwdConfig), _i, _i, _i32p, _i32p, _f64p, _vpp]),
    "swd_destroy": (None, [_vp]),
    "swd_decode_batch_host": (_i, [_vp, _u8p, C.c_int64, _u8p, _u8p, _dp]),
    "swd_decode_batch_device": (_i, [_vp, _u8p, C.c_int64, _u8p, _u8p, _dp, _vp]),
    "swd_decode_batch_host_packed": (_i, [_vp, _vp, C.c_int64, _vp, _u8p, _dp]),
    "swd_decode_batch_device_packed": (_i, [_vp, _vp, C.c_int64, _vp, _u8p, _dp, _vp]),
    "swd_decode_batch_host_llr": (_i, [_vp, _u8p, C.c_int64, _u8p, _u8p, _dp, _dp]),
    "swd_decode_batch_device_llr": (_i, [_vp, _u8p, C.c_int64, _u8p, _u8p, _dp, _dp, _vp]),
    "swd_decode_batch_host_packed_llr": (_i, [_vp, _vp, C.c_int64, _vp, _u8p, _dp, _dp]),
    "swd_decode_batch_device_packed_llr": (_i, [_vp, _vp, C.c_int64, _vp, _u8p, _dp, _dp, _vp]),
    "swd_pack_bits": (_i, [_i, _vp, C.c_int64, _i, _vp, _vp]),
    "swd_unpack_bits": (_i, [_i, _vp, C.c_int64, _i, _vp, _vp]),
    "swd_is_streamed": (_i, [_vp]),
    "swd_pre_bp_layout": (_i, [_i, _i, _i32p, _i32p, _i, _vp, _vp, _vp]),
    "swd_osd_last_outputs": (_i, [_vp, C.c_int64, _u8p, _u8p, _u8p, _dp, _vp]),
    "swd_set_profiling": (_i, [_vp, _i]),
    "swd_get_kernel_times": (_i, [_vp, _f64p, C.POINTER(C.c_uint64)]),
    "swd_get_counters": (_i, [_vp, C.POINTER(SwdCounters)]),
    "swd_reset_counters": (_i, [_vp]),
    "swd_rank": (_i, [_vp]),
    "swd_new_n": (_i, [_vp]),
    "swd_window_create": (_i, [_i, _i, _i, _i32p, _i32p, _i, _i32p, _i32p, _vpp]),
    "swd_window_destroy": (None, [_vp]),
    "swd_window_extract": (_i, [_vp, _u8p, C.c_int64, _i, _i, _u8p, _vp]),
    "swd_window_commit": (_i, [_vp, _u8p, C.c_int64, _i, _i, _i, _u8p, _u8p, _vp]),
    "swd_window_count_failures": (_i, [_vp, _u8p, _u8p, C.c_int64, _vp, _vp]),
    "swd_window_set_priors": (_i, [_vp, _f64p]),
    "swd_window_sample": (_i, [_vp, C.c_uint64, C.c_int64, C.c_int64, _u8p, _u8p, _u8p, _vp]),
    "swd_window_set_pauli_priors": (_i, [_vp, _i] + [_f64p] * 3 + [C.c_double, _f64p]),
    "swd_window_sample_pauli": (_i, [_vp, C.c_uint64, C.c_int64, C.c_int64, _u8p, _u8p, _u8p, _u8p, _dp, _vp]),
    "swd_window_set_circuit_noise": (_i, [_vp, _i, _i32p, _i32p] + [_f64p] * 3),
    "swd_window_sample_circuit": (_i, [_vp, C.c_uint64, C.c_int64, C.c_int64, _u8p, _u8p, _u8p, _u8p, _dp, _vp]),
    "swd_window_set_circuit_readout": (_i, [_vp, _i, _i32p, _i] + [_f64p] * 3),
    "swd_window_sample_circuit_readout": (_i, [_vp, C.c_uint64, C.c_int64, C.c_int64, _u8p, _u8p, _u8p, _u8p, _u8p, _dp, _vp]),
    "swd_bp4_create": (_i, [_i, _i, _i, _i, _i32p, _i32p, _i32p, _i32p] + [_f64p] * 5 + [_i, C.c_double, _i, _i, _vpp]),
    "swd_bp4_destroy": (None, [_vp]),
    "swd_bp4_rank": (_i, [_vp, _i]),
    "swd_bp4_decode_batch_host": (_i, [_vp, _u8p, _u8p, C.c_int64, _u8p, _u8p, _u8p, _u8p, _dp, _vp]),
    "swd_bp4_camel_decode_batch_host": (_i, [_vp, _u8p, _u8p, C.c_int64, _u8p, _u8p, _dp, _dp, _vp]),
    "swd_bp4_decode_batch_device": (_i, [_vp, _vp, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "swd_bp4_camel_decode_batch_device": (_i, [_vp, _vp, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "swd_bp4_decode_batch_host_llr": (_i, [_vp, _u8p, _u8p, C.c_int64, _u8p, _u8p, _u8p, _u8p, _dp, _vp, _dp]),
    "swd_bp4_decode_batch_device_llr": (_i, [_vp, _vp, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _dp, _vp]),
    "swd_bp4_camel_decode_batch_host_llr": (_i, [_vp, _u8p, _u8p, C.c_int64, _u8p, _u8p, _dp, _dp, _vp, _dp]),
    "swd_bp4_camel_decode_batch_device_llr": (_i, [_vp, _vp, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _dp, _vp]),
    "swd_strerror": (C.c_char_p, [_i]),
    "swd_last_error": (C.c_char_p, None),
    "swd_version": (C.c_char_p, None),
}
EXPORTS = list(_SIGNATURES)

_lib = None


def load():
    """Load the shared library (no CUDA call is made here)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(make -C slidingwindowdecoder_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def call(name, args, llr=None, stream=None):
    """Calls entry point `name` with args, or its per-shot-prior twin name + "_llr" with the priors pointer llr appended;
    device entry points take `stream` last.  Raises on an error status."""
    if llr is not None:
        name, args = name + "_llr", (*args, llr)
    if stream is not None:
        args = (*args, stream)
    check(getattr(load(), name)(*args), name)


def current_stream(device):
    """The current torch CUDA stream of `device` as the `void *stream` argument of the C-ABI."""
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Window:
    """Owns one swd_window handle over `chk` (and `obs`, or no observables if None): CSC matrices with sorted indices.  The
    object is passed to the C-ABI as the handle (ctypes reads `_as_parameter_`) and destroys it when collected."""

    def __init__(self, device, chk, obs=None):
        self._lib = load()
        mats = (chk,) if obs is None else (chk, obs)
        self._cp = tuple(np.ascontiguousarray(a, dtype=np.int32) for M in mats for a in (M.indptr, M.indices))
        ptrs = [a.ctypes.data_as(_i32p) for a in self._cp] + [None, None] * (obs is None)
        h = C.c_void_p()
        check(self._lib.swd_window_create(int(device), chk.shape[0], chk.shape[1], ptrs[0], ptrs[1],
                                          0 if obs is None else obs.shape[0], ptrs[2], ptrs[3], C.byref(h)), "swd_window_create")
        self._as_parameter_ = h

    def __del__(self):
        h = getattr(self, "_as_parameter_", None)
        if h is not None and h.value:
            self._lib.swd_window_destroy(h)
            h.value = None


def check(status, what=""):
    if status == OK:
        return
    lib = load()
    msg = f"{what}: {lib.swd_strerror(status).decode()} ({lib.swd_last_error().decode()})"
    if status == ERR_INVALID:
        raise ValueError(msg)
    if status == ERR_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)
