"""ctypes loader of libswd_b200.so (the C-ABI in include/swd_b200.h).

There is no CPU fallback: if the CUDA library is missing or no GPU is visible the decoders raise.
"""
import ctypes as C
import os

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

EXPORTS = ["swd_create", "swd_destroy", "swd_decode_batch_host", "swd_decode_batch_device", "swd_decode_batch_host_packed",
           "swd_decode_batch_device_packed", "swd_decode_batch_host_llr", "swd_decode_batch_device_llr",
           "swd_decode_batch_host_packed_llr", "swd_decode_batch_device_packed_llr", "swd_pack_bits", "swd_unpack_bits", "swd_is_streamed", "swd_pre_bp_layout", "swd_osd_last_outputs",
           "swd_set_profiling", "swd_get_kernel_times", "swd_get_counters", "swd_reset_counters", "swd_rank", "swd_new_n", "swd_window_create", "swd_window_destroy",
           "swd_window_extract", "swd_window_commit", "swd_window_count_failures", "swd_window_set_priors", "swd_window_sample",
           "swd_window_set_pauli_priors", "swd_window_sample_pauli", "swd_window_set_circuit_noise", "swd_window_sample_circuit",
           "swd_window_set_circuit_readout", "swd_window_sample_circuit_readout",
           "swd_bp4_create", "swd_bp4_destroy", "swd_bp4_rank", "swd_bp4_decode_batch_host", "swd_bp4_camel_decode_batch_host", "swd_bp4_decode_batch_device", "swd_bp4_camel_decode_batch_device",
           "swd_bp4_decode_batch_host_llr", "swd_bp4_decode_batch_device_llr", "swd_bp4_camel_decode_batch_host_llr",
           "swd_bp4_camel_decode_batch_device_llr", "swd_strerror", "swd_last_error",
           "swd_version"]

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
    vp, i32p, u8p, dp = C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p
    lib.swd_create.argtypes = [C.POINTER(SwdConfig), C.c_int, C.c_int, i32p, i32p, C.POINTER(C.c_double), C.POINTER(vp)]
    lib.swd_create.restype = C.c_int
    lib.swd_destroy.argtypes = [vp]
    lib.swd_destroy.restype = None
    lib.swd_decode_batch_host.argtypes = [vp, u8p, C.c_int64, u8p, u8p, dp]
    lib.swd_decode_batch_host.restype = C.c_int
    lib.swd_decode_batch_device.argtypes = [vp, u8p, C.c_int64, u8p, u8p, dp, vp]
    lib.swd_decode_batch_device.restype = C.c_int
    lib.swd_decode_batch_host_packed.argtypes = [vp, vp, C.c_int64, vp, u8p, dp]
    lib.swd_decode_batch_host_packed.restype = C.c_int
    lib.swd_decode_batch_device_packed.argtypes = [vp, vp, C.c_int64, vp, u8p, dp, vp]
    lib.swd_decode_batch_device_packed.restype = C.c_int
    lib.swd_decode_batch_host_llr.argtypes = [vp, u8p, C.c_int64, u8p, u8p, dp, dp]
    lib.swd_decode_batch_host_llr.restype = C.c_int
    lib.swd_decode_batch_device_llr.argtypes = [vp, u8p, C.c_int64, u8p, u8p, dp, dp, vp]
    lib.swd_decode_batch_device_llr.restype = C.c_int
    lib.swd_decode_batch_host_packed_llr.argtypes = [vp, vp, C.c_int64, vp, u8p, dp, dp]
    lib.swd_decode_batch_host_packed_llr.restype = C.c_int
    lib.swd_decode_batch_device_packed_llr.argtypes = [vp, vp, C.c_int64, vp, u8p, dp, dp, vp]
    lib.swd_decode_batch_device_packed_llr.restype = C.c_int
    lib.swd_pack_bits.argtypes = [C.c_int, vp, C.c_int64, C.c_int, vp, vp]
    lib.swd_pack_bits.restype = C.c_int
    lib.swd_unpack_bits.argtypes = [C.c_int, vp, C.c_int64, C.c_int, vp, vp]
    lib.swd_unpack_bits.restype = C.c_int
    lib.swd_is_streamed.argtypes = [vp]
    lib.swd_is_streamed.restype = C.c_int
    lib.swd_pre_bp_layout.argtypes = [C.c_int, C.c_int, i32p, i32p, C.c_int, vp, vp, vp]
    lib.swd_pre_bp_layout.restype = C.c_int
    lib.swd_osd_last_outputs.argtypes = [vp, C.c_int64, u8p, u8p, u8p, dp, vp]
    lib.swd_osd_last_outputs.restype = C.c_int
    lib.swd_get_counters.argtypes = [vp, C.POINTER(SwdCounters)]
    lib.swd_get_counters.restype = C.c_int
    lib.swd_set_profiling.argtypes = [vp, C.c_int]
    lib.swd_set_profiling.restype = C.c_int
    lib.swd_get_kernel_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    lib.swd_get_kernel_times.restype = C.c_int
    lib.swd_reset_counters.argtypes = [vp]
    lib.swd_reset_counters.restype = C.c_int
    lib.swd_rank.argtypes = [vp]
    lib.swd_rank.restype = C.c_int
    lib.swd_new_n.argtypes = [vp]
    lib.swd_new_n.restype = C.c_int
    lib.swd_window_create.argtypes = [C.c_int, C.c_int, C.c_int, i32p, i32p, C.c_int, i32p, i32p, C.POINTER(vp)]
    lib.swd_window_create.restype = C.c_int
    lib.swd_window_destroy.argtypes = [vp]
    lib.swd_window_destroy.restype = None
    lib.swd_window_extract.argtypes = [vp, u8p, C.c_int64, C.c_int, C.c_int, u8p, vp]
    lib.swd_window_extract.restype = C.c_int
    lib.swd_window_commit.argtypes = [vp, u8p, C.c_int64, C.c_int, C.c_int, C.c_int, u8p, u8p, vp]
    lib.swd_window_commit.restype = C.c_int
    lib.swd_window_count_failures.argtypes = [vp, u8p, u8p, C.c_int64, vp, vp]
    lib.swd_window_count_failures.restype = C.c_int
    lib.swd_window_set_priors.argtypes = [vp, C.POINTER(C.c_double)]
    lib.swd_window_set_priors.restype = C.c_int
    lib.swd_window_sample.argtypes = [vp, C.c_uint64, C.c_int64, C.c_int64, u8p, u8p, u8p, vp]
    lib.swd_window_sample.restype = C.c_int
    lib.swd_window_set_pauli_priors.argtypes = [vp, C.c_int] + [C.POINTER(C.c_double)] * 3 + [C.c_double, C.POINTER(C.c_double)]
    lib.swd_window_set_pauli_priors.restype = C.c_int
    lib.swd_window_sample_pauli.argtypes = [vp, C.c_uint64, C.c_int64, C.c_int64, u8p, u8p, u8p, u8p, dp, vp]
    lib.swd_window_sample_pauli.restype = C.c_int
    lib.swd_window_set_circuit_noise.argtypes = [vp, C.c_int, i32p, i32p] + [C.POINTER(C.c_double)] * 3
    lib.swd_window_set_circuit_noise.restype = C.c_int
    lib.swd_window_sample_circuit.argtypes = [vp, C.c_uint64, C.c_int64, C.c_int64, u8p, u8p, u8p, u8p, dp, vp]
    lib.swd_window_sample_circuit.restype = C.c_int
    lib.swd_window_set_circuit_readout.argtypes = [vp, C.c_int, i32p, C.c_int] + [C.POINTER(C.c_double)] * 3
    lib.swd_window_set_circuit_readout.restype = C.c_int
    lib.swd_window_sample_circuit_readout.argtypes = [vp, C.c_uint64, C.c_int64, C.c_int64, u8p, u8p, u8p, u8p, u8p, dp, vp]
    lib.swd_window_sample_circuit_readout.restype = C.c_int
    lib.swd_bp4_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, i32p, i32p] + [C.POINTER(C.c_double)] * 5 + \
                                  [C.c_int, C.c_double, C.c_int, C.c_int, C.POINTER(vp)]
    lib.swd_bp4_create.restype = C.c_int
    lib.swd_bp4_destroy.argtypes = [vp]
    lib.swd_bp4_destroy.restype = None
    lib.swd_bp4_rank.argtypes = [vp, C.c_int]
    lib.swd_bp4_rank.restype = C.c_int
    lib.swd_bp4_decode_batch_host.argtypes = [vp, u8p, u8p, C.c_int64, u8p, u8p, u8p, u8p, dp, vp]
    lib.swd_bp4_decode_batch_host.restype = C.c_int
    lib.swd_bp4_camel_decode_batch_host.argtypes = [vp, u8p, u8p, C.c_int64, u8p, u8p, dp, dp, vp]
    lib.swd_bp4_camel_decode_batch_host.restype = C.c_int
    lib.swd_bp4_decode_batch_device.argtypes = [vp, vp, vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp]
    lib.swd_bp4_decode_batch_device.restype = C.c_int
    lib.swd_bp4_camel_decode_batch_device.argtypes = [vp, vp, vp, C.c_int64, vp, vp, vp, vp, vp, vp]
    lib.swd_bp4_camel_decode_batch_device.restype = C.c_int
    lib.swd_bp4_decode_batch_host_llr.argtypes = [vp, u8p, u8p, C.c_int64, u8p, u8p, u8p, u8p, dp, vp, dp]
    lib.swd_bp4_decode_batch_host_llr.restype = C.c_int
    lib.swd_bp4_camel_decode_batch_host_llr.argtypes = [vp, u8p, u8p, C.c_int64, u8p, u8p, dp, dp, vp, dp]
    lib.swd_bp4_camel_decode_batch_host_llr.restype = C.c_int
    lib.swd_bp4_decode_batch_device_llr.argtypes = [vp, vp, vp, C.c_int64, vp, vp, vp, vp, vp, vp, dp, vp]
    lib.swd_bp4_decode_batch_device_llr.restype = C.c_int
    lib.swd_bp4_camel_decode_batch_device_llr.argtypes = [vp, vp, vp, C.c_int64, vp, vp, vp, vp, vp, dp, vp]
    lib.swd_bp4_camel_decode_batch_device_llr.restype = C.c_int
    lib.swd_strerror.argtypes = [C.c_int]
    lib.swd_strerror.restype = C.c_char_p
    lib.swd_last_error.restype = C.c_char_p
    lib.swd_version.restype = C.c_char_p
    _lib = lib
    return lib


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
