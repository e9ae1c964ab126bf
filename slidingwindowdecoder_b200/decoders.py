"""Drop-in decoder classes: the reference's Cython API on top of the B200 C-ABI.

  bpgdg_decoder  <- src/bp_guessing_decoder.pyx:160-469
  bpgd_decoder   <- src/bp_guessing_decoder.pyx:473-570
  osd_window     <- src/osd_window.pyx:6-549

Same constructor kwargs / defaults, `decode(syndrome) -> np.int64[n]`, `.converge`, and the
osd_window read-only properties.  Added: `decode_batch(syndromes[B, m])`, which is what the
sliding-window driver uses (one call per window for ALL shots).  All arithmetic runs in the CUDA
library; there is no CPU path.
"""
import ctypes as C
import math

import numpy as np
from scipy.sparse import spmatrix, csc_matrix

from . import _lib

_OSD_METHODS = {"osd_0": 0, "0": 0, "osd0": 0,
                "osd_e": 1, "1": 1, "osde": 1, "exhaustive": 1, "e": 1,
                "osd_cs": 2, "2": 2, "osdcs": 2, "combination_sweep": 2, "cs": 2}


_BP_METHODS = {"minimum_sum": 0, "ms": 0, "min_sum": 0, "msl": 0, "0": 0,
               "product_sum": 1, "ps": 1, "prod_sum": 1, "psl": 1, "1": 1}


def _libm_llr(channel_probs, n):
    """log((1-p)/p) with libm's log, as bp_guessing_decoder.pyx:46 (numpy's vector log differs by ulps).  The reference only
    fills channel_llr when channel_probs[0] is not None (pyx:19-23, :44-46) - the LLRs then stay 0 - and its cdivision
    arithmetic gives +inf for p = 0 (-inf for p = 1) instead of raising."""
    out = np.zeros(n, dtype=np.float64)
    if channel_probs[0] is None:
        return out
    for v in range(n):
        p = float(channel_probs[v])
        if p <= 0.0:
            out[v] = math.inf
        elif p >= 1.0:
            out[v] = -math.inf
        else:
            out[v] = math.log((1.0 - p) / p)
    return out


def pack_bits(a):
    """[B, k] array of 0/1 -> [B, ceil(k/64)] uint64, bit j of a row = (word[j >> 6] >> (j & 63)) & 1 (the C-ABI's packed layout)."""
    a = np.ascontiguousarray(np.asarray(a), dtype=np.uint8)
    B, k = a.shape
    w = (k + 63) // 64
    out = np.zeros((B, w * 8), dtype=np.uint8)
    pk = np.packbits(a, axis=1, bitorder="little")
    out[:, :pk.shape[1]] = pk
    return out.view(np.uint64)


def unpack_bits(p, k):
    """inverse of pack_bits: [B, ceil(k/64)] uint64 -> [B, k] uint8"""
    p = np.ascontiguousarray(p, dtype=np.uint64)
    return np.unpackbits(p.view(np.uint8), axis=1, bitorder="little")[:, :k]


def _is_torch_cuda(x):
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda") and x.is_cuda


def _check_llr(channel_llr, shape, device=None, allow_inf=True):
    """Per-shot priors of a batched call, checked and contiguous.  device None: a host call, which takes a numpy float64 array
    and rejects NaN (and +-inf unless allow_inf).  Otherwise a device call, which takes a torch CUDA float64 tensor on `device`;
    it is not scanned for NaN or inf, as that would synchronise the stream (such values are undefined behaviour, as at the
    C-ABI)."""
    if device is None:
        if _is_torch_cuda(channel_llr) or not isinstance(channel_llr, np.ndarray):
            raise ValueError("channel_llr must be a numpy float64 array when the syndromes are host arrays "
                             f"(got {type(channel_llr).__name__})")
        if channel_llr.dtype != np.float64:
            raise ValueError(f"channel_llr must be float64, got {channel_llr.dtype}")
    else:
        if not _is_torch_cuda(channel_llr):
            raise ValueError("channel_llr must be a torch CUDA float64 tensor when the syndromes are torch CUDA tensors "
                             f"(got {type(channel_llr).__name__})")
        import torch
        if channel_llr.dtype != torch.float64:
            raise ValueError(f"channel_llr must be float64, got {channel_llr.dtype}")
    if tuple(channel_llr.shape) != shape:
        raise ValueError(f"channel_llr must have shape {list(shape)}, got {list(channel_llr.shape)}")
    if device is not None:
        if channel_llr.device != device:
            raise ValueError(f"channel_llr lives on {channel_llr.device}, syndromes on {device}")
        return channel_llr.contiguous()
    if allow_inf and np.isnan(channel_llr).any():
        raise ValueError("channel_llr contains NaN (allowed: finite values, +-inf; 0.0 marks an erasure)")
    if not allow_inf and not np.isfinite(channel_llr).all():
        raise ValueError("channel_llr contains inf or NaN (allowed: finite values)")
    return np.ascontiguousarray(channel_llr)


class _window_decoder_base:
    """Shared constructor checks (bp_guessing_decoder.pyx:6-46, osd_window.pyx:8-34) and batch plumbing."""

    _kind = None

    def _setup(self, parity_check_matrix, channel_probs, cfg, device):
        if not (isinstance(parity_check_matrix, np.ndarray) or isinstance(parity_check_matrix, spmatrix)):
            raise TypeError("The input matrix is of an invalid type. Please input a np.ndarray or "
                            f"scipy.sparse.spmatrix object, not {type(parity_check_matrix)}")
        self.m, self.n = parity_check_matrix.shape
        if channel_probs is None:
            raise TypeError("channel_probs is required")
        if channel_probs[0] is not None and len(channel_probs) != self.n:
            raise ValueError(f"The length of the channel probability vector must be eqaul to the block length n={self.n}.")
        A = csc_matrix(parity_check_matrix)
        A.eliminate_zeros()
        A.sort_indices()
        self._colptr = np.ascontiguousarray(A.indptr, dtype=np.int32)
        self._rowidx = np.ascontiguousarray(A.indices, dtype=np.int32)
        self.channel_llr = _libm_llr(channel_probs, self.n)
        cfg.kind = self._kind
        cfg.device = int(device)
        cfg.bp_method = _BP_METHODS[str(getattr(self, "_bp_method", "minimum_sum")).lower()]
        self._cfg = cfg
        self._device = int(device)
        self._handle = C.c_void_p()
        lib = _lib.load()
        st = lib.swd_create(C.byref(cfg), self.m, self.n, self._colptr.ctypes.data_as(C.POINTER(C.c_int32)),
                            self._rowidx.ctypes.data_as(C.POINTER(C.c_int32)),
                            self.channel_llr.ctypes.data_as(C.POINTER(C.c_double)), C.byref(self._handle))
        _lib.check(st, "swd_create")
        self._lib = lib
        self.new_n = lib.swd_new_n(self._handle)
        self._converge = 0
        self.min_pm_batch = None

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            self._lib.swd_destroy(h)
            self._handle = C.c_void_p()

    @property
    def converge(self):
        return self._converge

    # ------------------------------------------------------------------ batched entry points
    def decode_batch(self, syndromes, return_pm=False, channel_llr=None):
        """syndromes: [B, m] of 0/1.  numpy in -> numpy out (host copies inside the call);
        torch CUDA uint8 tensor in -> torch CUDA tensors out (asynchronous on the current stream).
        channel_llr: optional per-shot priors [B, n] float64 (numpy with numpy syndromes, a torch CUDA tensor on the
        decoder's device with torch syndromes): row b decodes syndrome b as a decoder built with channel_llr = row b would.
        0.0 marks an erasure (p = 1/2); +inf and negative values are allowed, NaN is not.
        Returns (corrections [B, n] uint8, converge [B] uint8[, min_pm [B] float64])."""
        if _is_torch_cuda(syndromes):
            import torch
            s = (syndromes if syndromes.dtype == torch.uint8 else syndromes.to(torch.uint8)).contiguous()
        else:
            s = np.ascontiguousarray(np.asarray(syndromes), dtype=np.uint8)
        if s.ndim != 2 or s.shape[1] != self.m:
            raise ValueError(f"decode_batch expects syndromes of shape [B, {self.m}], got {tuple(s.shape)}")
        return self._batch(s, False, return_pm, channel_llr)

    def decode_batch_packed(self, synd_packed, return_pm=False, channel_llr=None):
        """Bit-packed twin of decode_batch (swd_decode_batch_host_packed / _device_packed): synd_packed [B, ceil(m/64)] uint64
        (see pack_bits) -> (corrections [B, ceil(n/64)] uint64, converge [B] uint8[, min_pm]).  numpy in -> numpy out with the
        copies inside the call; torch CUDA int64/uint64 tensor in -> torch CUDA tensors out on the current stream.
        channel_llr: optional per-shot priors [B, n] float64, as for decode_batch."""
        wm = (self.m + 63) // 64
        if _is_torch_cuda(synd_packed):
            s = synd_packed.contiguous()
            ok = s.element_size() == 8
        else:
            s, ok = np.ascontiguousarray(synd_packed, dtype=np.uint64), True
        if s.ndim != 2 or s.shape[1] != wm or not ok:
            raise ValueError(f"decode_batch_packed expects 64-bit words of shape [B, {wm}], got {tuple(s.shape)}")
        return self._batch(s, True, return_pm, channel_llr)

    def _batch(self, s, packed, return_pm, channel_llr):
        """Decodes the shape-checked syndromes s ([B, m] bytes, or [B, ceil(m/64)] words if packed): numpy in -> numpy out
        through the host entry point, torch CUDA in -> torch CUDA out on the current stream through the device entry point."""
        B, n_out = s.shape[0], (self.n + 63) // 64 if packed else self.n
        device = _is_torch_cuda(s)
        if device:
            import torch
            dev = s.device
            if dev.index != self._device:
                raise ValueError(f"syndromes live on cuda:{dev.index}, decoder on cuda:{self._device}")
            llr = None if channel_llr is None else _check_llr(channel_llr, (B, self.n), dev)
            out = (torch.empty((B, n_out), dtype=torch.int64 if packed else torch.uint8, device=dev),
                   torch.empty(B, dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.float64, device=dev))
            kind, ptr, stream = "device", torch.Tensor.data_ptr, _lib.current_stream(dev)
        else:
            llr = None if channel_llr is None else _check_llr(channel_llr, (B, self.n))
            out = (np.empty((B, n_out), dtype=np.uint64 if packed else np.uint8), np.empty(B, dtype=np.uint8),
                   np.empty(B, dtype=np.float64))
            kind, ptr, stream = "host", (lambda a: a.ctypes.data), None
        _lib.call("swd_decode_batch_" + kind + "_packed" * packed, (self._handle, ptr(s), B, *map(ptr, out)),
                  None if llr is None else ptr(llr), stream)
        if device:
            self._keepalive = s if llr is None else (s, llr)
        self._last_B = B
        return out if return_pm else out[:2]

    @property
    def streamed_bp(self):
        """True if the full-window BP streams its messages from HBM (the window graph exceeds one SM's shared memory)."""
        return bool(self._lib.swd_is_streamed(self._handle) == 1)

    def _decode_one(self, input_vector):
        input_length = input_vector.shape[0]
        if input_length != self.m:
            raise ValueError(f"The input to the ldpc.bp_decoder.decode must be a syndrome (of length={self.m}). The inputted "
                             f"vector has length={input_length}. Valid formats are `np.ndarray` or `scipy.sparse.spmatrix`.")
        s = np.asarray(input_vector).reshape(1, self.m)
        corr, conv, pm = self.decode_batch(s, return_pm=True)
        self._converge = int(conv[0])
        self._min_pm = float(pm[0])
        return corr[0].astype(np.int64)

    def counters(self):
        c = _lib.SwdCounters()
        _lib.check(self._lib.swd_get_counters(self._handle, C.byref(c)), "swd_get_counters")
        return c.as_dict()

    def set_profiling(self, enable=True):
        _lib.check(self._lib.swd_set_profiling(self._handle, int(bool(enable))), "swd_set_profiling")

    def kernel_times(self):
        """{kernel class: (total ms, launches)} since the last call (needs set_profiling(True))."""
        ms = (C.c_double * 8)()
        ln = (C.c_uint64 * 8)()
        _lib.check(self._lib.swd_get_kernel_times(self._handle, ms, ln), "swd_get_kernel_times")
        return {k: (float(ms[i]), int(ln[i])) for i, k in enumerate(_lib.KERNEL_CLASSES)}

    def reset_counters(self):
        _lib.check(self._lib.swd_reset_counters(self._handle), "swd_reset_counters")


class bpgdg_decoder(_window_decoder_base):
    """BP + Guided Decimation Guessing (bp_guessing_decoder.pyx:160-469)."""
    _kind = _lib.KIND_BPGDG

    def __init__(self, parity_check_matrix, **kwargs):
        cfg = _lib.SwdConfig()
        cfg.max_iter = int(kwargs.get("max_iter", 50))
        cfg.ms_scaling_factor = float(kwargs.get("ms_scaling_factor", 1.0))
        cfg.max_iter_per_step = int(kwargs.get("max_iter_per_step", 6))
        cfg.max_step = int(kwargs.get("max_step", 25))
        cfg.max_tree_depth = int(kwargs.get("max_tree_depth", 3))
        cfg.max_side_depth = int(kwargs.get("max_side_depth", 10))
        cfg.max_tree_branch_step = int(kwargs.get("max_tree_branch_step", 10))
        cfg.max_side_branch_step = int(kwargs.get("max_side_branch_step", 10))
        cfg.gdg_factor = float(kwargs.get("gdg_factor", 1.0))
        new_n = kwargs.get("new_n", None)
        cfg.new_n = 0 if new_n is None else int(new_n)
        cfg.multi_thread = int(bool(kwargs.get("multi_thread", False)))
        cfg.low_error_mode = int(bool(kwargs.get("low_error_mode", False)))
        self.multi_thread = bool(cfg.multi_thread)
        self._setup(parity_check_matrix, kwargs.get("channel_probs"), cfg, kwargs.get("device", 0))

    def decode(self, input_vector):
        return self._decode_one(input_vector)


class bpgd_decoder(_window_decoder_base):
    """BP + guided decimation (bp_guessing_decoder.pyx:473-570)."""
    _kind = _lib.KIND_BPGD

    def __init__(self, parity_check_matrix, **kwargs):
        cfg = _lib.SwdConfig()
        cfg.max_iter = int(kwargs.get("max_iter", 50))
        cfg.ms_scaling_factor = float(kwargs.get("ms_scaling_factor", 1.0))
        cfg.max_iter_per_step = int(kwargs.get("max_iter_per_step", 6))
        cfg.max_step = int(kwargs.get("max_step", 25))
        cfg.gdg_factor = float(kwargs.get("gd_factor", 1.0))
        new_n = kwargs.get("new_n", None)
        cfg.new_n = 0 if new_n is None else int(new_n)
        self._setup(parity_check_matrix, kwargs.get("channel_probs"), cfg, kwargs.get("device", 0))

    def decode(self, input_vector):
        return self._decode_one(input_vector)


class osd_window(_window_decoder_base):
    """BP on the window, shortening, BP on the shortened window, OSD (osd_window.pyx)."""
    _kind = _lib.KIND_OSD_WINDOW

    def __init__(self, parity_check_matrix, **kwargs):
        cfg = _lib.SwdConfig()
        cfg.max_iter = int(kwargs.get("pre_max_iter", 8))
        cfg.post_max_iter = int(kwargs.get("post_max_iter", 100))
        cfg.ms_scaling_factor = float(kwargs.get("ms_scaling_factor", 1.0))
        new_n = kwargs.get("new_n", None)
        cfg.new_n = 0 if new_n is None else int(new_n)
        osd_method = kwargs.get("osd_method", "osd_0")
        osd_order = kwargs.get("osd_order", 0)
        key = str(osd_method).lower()
        if key not in _OSD_METHODS:
            raise ValueError(f"ERROR: OSD method '{osd_method}' invalid. Please choose from the following methods: "
                             "'OSD_0', 'OSD_E' or 'OSD_CS'.")
        cfg.osd_method = _OSD_METHODS[key]
        cfg.osd_order = 0 if cfg.osd_method == 0 else int(osd_order)
        self.osd_method, self.osd_order = cfg.osd_method, cfg.osd_order
        try:
            self._setup(parity_check_matrix, kwargs.get("channel_probs"), cfg, kwargs.get("device", 0))
        except ValueError as e:
            if "osd_order" in str(e):
                raise ValueError("For this code, the OSD order should be set in the range 0<=osd_oder<=new_n-rank.") from e
            raise
        self.rank = self._lib.swd_rank(self._handle)
        self._min_pm = 0.0
        self._last_B = 0

    def decode(self, input_vector):
        return self._decode_one(input_vector)

    def last_outputs(self, B=None):
        """dict of the per-shot read-only properties of the last batch (host numpy arrays)."""
        B = self._last_B if B is None else B
        n = self.n
        bp = np.empty((B, n), dtype=np.uint8)
        o0 = np.empty((B, n), dtype=np.uint8)
        ow = np.empty((B, n), dtype=np.uint8)
        lpr = np.empty((B, n, 4), dtype=np.float64)
        it = np.empty(B, dtype=np.int32)
        st = self._lib.swd_osd_last_outputs(self._handle, B, bp.ctypes.data, o0.ctypes.data, ow.ctypes.data, lpr.ctypes.data,
                                            it.ctypes.data)
        _lib.check(st, "swd_osd_last_outputs")
        return dict(bp_decoding=bp, osd0_decoding=o0, osdw_decoding=ow, log_prob_ratios=lpr, bp_iteration=it)

    @property
    def min_pm(self):
        return self._min_pm

    @property
    def bp_iteration(self):
        return int(self.last_outputs(1)["bp_iteration"][0])

    @property
    def bp_decoding(self):
        return self.last_outputs(1)["bp_decoding"][0].astype(np.int64)

    @property
    def osd0_decoding(self):
        return self.last_outputs(1)["osd0_decoding"][0].astype(np.int64)

    @property
    def osdw_decoding(self):
        return self.last_outputs(1)["osdw_decoding"][0].astype(np.int64)

    @property
    def log_prob_ratios(self):
        return self.last_outputs(1)["log_prob_ratios"][0].copy()


class BpOsdDecoder(osd_window):
    """Facade with the constructor kwargs the reference's drivers pass to `ldpc.BpOsdDecoder`
    (osd.py:142-150, guessing.py:150-158, simulation.py:39-47): min-sum BP for `max_iter` iterations on the whole
    matrix (no shortening: new_n = n, no second BP stage), then OSD.  It runs this repository's `osd_window`
    kernels; `ldpc` itself is a third-party dependency that is not vendored by the reference, so its exact
    tie-breaking (it ranks by the last posterior, this ranks by the 4-iteration history sum) is NOT reproduced:
    parity with `ldpc` is unpinned (DESIGN.md section 4).  `osd0_decoding` / `converge` follow osd_window."""

    def __init__(self, parity_check_matrix, **kwargs):
        method = str(kwargs.get("bp_method", "minimum_sum")).lower()
        if method not in _BP_METHODS:
            raise ValueError(f"bp_method '{method}' invalid: choose 'minimum_sum' or 'product_sum'")
        self._bp_method = method        # product-sum: restated from ldpc's published algorithm, parity unpinned (DESIGN.md section 4)
        n = parity_check_matrix.shape[1]
        super().__init__(parity_check_matrix, channel_probs=kwargs.get("channel_probs"),
                         pre_max_iter=int(kwargs.get("max_iter", 0)) or n, post_max_iter=0,
                         ms_scaling_factor=float(kwargs.get("ms_scaling_factor", 1.0)), new_n=n,
                         osd_method=kwargs.get("osd_method", "osd_0"), osd_order=kwargs.get("osd_order", 0),
                         device=kwargs.get("device", 0))


class bp4_osd:
    """Quaternary BP + OSD for CSS codes under depolarizing noise (src/bp4_osd.pyx): same constructor kwargs
    (`channel_probs_x/y/z`, `max_iter=32`, `ms_scaling_factor=1.0`, `osd_method="osd_0"`, `osd_order=0`),
    `decode(synd_x, synd_z) -> np.int64[2, n]` (row 0: X part, row 1: Z part), `.converge`, `.bp_iteration`, `.min_pm`
    (0.0, as in the reference whose decode never updates it), `.bp_decoding_x/z`, `.osd0_decoding_x/z`,
    `.osdw_decoding_x/z`, `.log_prob_ratios` [n, 3], and `camel_decode(synd_x, synd_z)` (pyx:223-248: four BP runs with the last
    qubit pinned to I / X / Z / Y, best converged path metric; sets `.converge`, `.min_pm`).
    Added: `decode_batch(synd_x[B, mx], synd_z[B, mz], channel_llr=None)`, `camel_decode_batch(...)`, and `.channel_llr`
    [5, n]: the static priors llr_x, llr_y, llr_z, prior_llr_x, prior_llr_z.  Per-shot priors are a [5, B, n] float64 array
    of the same five rows per shot (an erased qubit, px = py = pz = 1/4, is 0.0 in all five)."""

    def __init__(self, Hx, Hz, **kwargs):
        if not (isinstance(Hx, np.ndarray) or isinstance(Hx, spmatrix)):
            raise TypeError("The input matrix is of an invalid type. Please input a np.ndarray or scipy.sparse.spmatrix object.")
        if Hx.shape[1] != Hz.shape[1]:
            raise ValueError("Hx, Hz blocklength does not match!")
        self.mx, self.n = Hx.shape
        self.mz = Hz.shape[0]
        px, py, pz = kwargs.get("channel_probs_x"), kwargs.get("channel_probs_y"), kwargs.get("channel_probs_z")
        if px is None or py is None or pz is None:
            raise TypeError("channel_probs_x, channel_probs_y and channel_probs_z are required")
        if len(px) != self.n or len(py) != self.n or len(pz) != self.n:     # the reference checks px only (bp4_osd.pyx:40-42) and reads past py / pz
            raise ValueError(f"The length of the channel probability vector must be eqaul to the block length n={self.n}.")
        self._device = int(kwargs.get("device", 0))
        osd_method = kwargs.get("osd_method", "osd_0")
        key = str(osd_method).lower()
        if key not in _OSD_METHODS:
            raise ValueError(f"ERROR: OSD method '{osd_method}' invalid. Please choose from the following methods: "
                             "'OSD_0', 'OSD_E' or 'OSD_CS'.")
        meth = _OSD_METHODS[key]
        order = 0 if meth == 0 else int(kwargs.get("osd_order", 0))
        n = self.n
        llr = np.empty((5, n))
        for v in range(n):                                                   # pyx:123-133, libm log
            num = 1.0 - (float(px[v]) + float(py[v]) + float(pz[v]))
            llr[0, v] = math.log(num / float(px[v])); llr[1, v] = math.log(num / float(py[v])); llr[2, v] = math.log(num / float(pz[v]))
            den = float(px[v]) + float(py[v]); llr[3, v] = math.log((1.0 - den) / den)
            den = float(pz[v]) + float(py[v]); llr[4, v] = math.log((1.0 - den) / den)
        self._llr = np.ascontiguousarray(llr)
        self.channel_llr = self._llr.copy()
        A, Bz = csc_matrix(Hx), csc_matrix(Hz)
        for M in (A, Bz):
            M.eliminate_zeros(); M.sort_indices()
        self._hx = (np.ascontiguousarray(A.indptr, dtype=np.int32), np.ascontiguousarray(A.indices, dtype=np.int32))
        self._hz = (np.ascontiguousarray(Bz.indptr, dtype=np.int32), np.ascontiguousarray(Bz.indices, dtype=np.int32))
        lib = _lib.load()
        self._lib = lib
        self._handle = C.c_void_p()
        i32p, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
        st = lib.swd_bp4_create(int(kwargs.get("device", 0)), self.mx, self.mz, n, self._hx[0].ctypes.data_as(i32p),
                                self._hx[1].ctypes.data_as(i32p), self._hz[0].ctypes.data_as(i32p), self._hz[1].ctypes.data_as(i32p),
                                *[self._llr[i].ctypes.data_as(dp) for i in range(5)], int(kwargs.get("max_iter", 32)),
                                float(kwargs.get("ms_scaling_factor", 1.0)), meth, order, C.byref(self._handle))
        try:
            _lib.check(st, "swd_bp4_create")
        except ValueError as e:
            if "osd_order" in str(e):
                raise ValueError("For this code, the OSD order should be set in the range 0<=osd_oder<=n-rank.") from e
            raise
        self.rank_x, self.rank_z = lib.swd_bp4_rank(self._handle, 0), lib.swd_bp4_rank(self._handle, 1)
        self.osd_method, self.osd_order = meth, order
        self.converge, self.bp_iteration, self.min_pm = 0, 0, 0.0
        self._last = None

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h is not None and h.value:
            self._lib.swd_bp4_destroy(h)
            self._handle = C.c_void_p()

    def decode_batch(self, synd_x, synd_z, channel_llr=None):
        """-> dict(dec [B, 2, n] uint8, converge [B], bp_decoding [B, 2, n], osd0 [B, 2, n], log_prob_ratios [B, n, 3],
        bp_iteration [B]).  channel_llr: optional per-shot priors [5, B, n] float64 (numpy with numpy syndromes, a torch CUDA
        tensor on the decoder's device with torch syndromes): row b of the five planes decodes shot b as a bp4_osd built
        with those priors would.  Finite values only; 0.0 in all five planes marks an erased qubit."""
        return self._batch(synd_x, synd_z, channel_llr, camel=False)

    def decode(self, input_vector_x, input_vector_z):
        if input_vector_x.shape[0] != self.mx or input_vector_z.shape[0] != self.mz:
            raise ValueError(f"The input to the bp4_osd.decode must be a syndrome (of length={self.mx}).")
        out = self.decode_batch(np.asarray(input_vector_x).reshape(1, -1), np.asarray(input_vector_z).reshape(1, -1))
        self._last = {k: v[0] for k, v in out.items()}
        self.converge = int(self._last["converge"]); self.bp_iteration = int(self._last["bp_iteration"])
        return self._last["dec"].astype(np.int64)

    def camel_decode_batch(self, synd_x, synd_z, channel_llr=None):
        """-> dict(dec [B, 2, n] uint8, converge [B], min_pm [B], log_prob_ratios [B, n, 3] and bp_iteration [B] of the last run).
        channel_llr: optional per-shot priors [5, B, n], as for decode_batch (planes 0-2 are used)."""
        return self._batch(synd_x, synd_z, channel_llr, camel=True)

    def _batch(self, synd_x, synd_z, channel_llr, camel):
        """numpy syndromes in -> dict of numpy arrays out (host entry points, copies inside the call); torch CUDA tensors in ->
        dict of torch CUDA tensors out, asynchronous on the current stream (device entry points; calls on one decoder must be
        stream-ordered)."""
        device = _is_torch_cuda(synd_x) and _is_torch_cuda(synd_z)
        if device:
            import torch
            sx, sz = synd_x.to(torch.uint8).contiguous(), synd_z.to(torch.uint8).contiguous()
        else:
            sx, sz = (np.ascontiguousarray(np.asarray(a), dtype=np.uint8) for a in (synd_x, synd_z))
        if sx.ndim != 2 or sz.ndim != 2 or sx.shape[1] != self.mx or sz.shape[1] != self.mz or sx.shape[0] != sz.shape[0]:
            raise ValueError(f"{'camel_decode_batch' if camel else 'decode_batch'} expects syndromes of shape [B, {self.mx}] "
                             f"and [B, {self.mz}]")
        B, n = sx.shape[0], self.n
        spec = [("dec", (B, 2, n), "uint8"), ("converge", B, "uint8")]
        spec += [("min_pm", B, "float64")] if camel else [("bp_decoding", (B, 2, n), "uint8"), ("osd0", (B, 2, n), "uint8")]
        spec += [("log_prob_ratios", (B, n, 3), "float64"), ("bp_iteration", B, "int32")]
        if device:
            if sx.device.index != self._device or sz.device.index != self._device:
                raise ValueError(f"syndromes live on cuda:{sx.device.index} / cuda:{sz.device.index}, decoder on cuda:{self._device}")
            llr = None if channel_llr is None else _check_llr(channel_llr, (5, B, n), sx.device, allow_inf=False)
            out = {k: torch.empty(shape, dtype=getattr(torch, dt), device=sx.device) for k, shape, dt in spec}
            kind, ptr, stream = "device", (lambda t: t.data_ptr()), _lib.current_stream(sx.device)
        else:
            llr = None if channel_llr is None else _check_llr(channel_llr, (5, B, n), allow_inf=False)
            out = {k: np.empty(shape, dtype=dt) for k, shape, dt in spec}
            kind, ptr, stream = "host", (lambda a: a.ctypes.data), None
        _lib.call("swd_bp4_" + "camel_" * camel + "decode_batch_" + kind, (self._handle, ptr(sx), ptr(sz), B, *map(ptr, out.values())),
                  None if llr is None else ptr(llr), stream)
        if device:
            self._keepalive = (sx, sz) if llr is None else (sx, sz, llr)
        return out

    def camel_decode(self, input_vector_x, input_vector_z):
        if input_vector_x.shape[0] != self.mx or input_vector_z.shape[0] != self.mz:
            raise ValueError(f"The input to the bp4_osd.decode must be a syndrome (of length={self.mx}).")
        out = self.camel_decode_batch(np.asarray(input_vector_x).reshape(1, -1), np.asarray(input_vector_z).reshape(1, -1))
        last = {k: v[0] for k, v in out.items()}
        # the reference keeps the winning run in osd0_decoding and leaves bp_decoding at the last (Y) run, which is not kept here
        last["osd0"] = last["dec"]; last["bp_decoding"] = last["dec"]
        self._last = last
        self.converge = int(last["converge"]); self.bp_iteration = int(last["bp_iteration"]); self.min_pm = float(last["min_pm"])
        return last["dec"].astype(np.int64)

    bp_decoding_x = property(lambda self: self._last["bp_decoding"][0].astype(np.int64))
    bp_decoding_z = property(lambda self: self._last["bp_decoding"][1].astype(np.int64))
    osd0_decoding_x = property(lambda self: self._last["osd0"][0].astype(np.int64))
    osd0_decoding_z = property(lambda self: self._last["osd0"][1].astype(np.int64))
    osdw_decoding_x = property(lambda self: self._last["dec"][0].astype(np.int64))
    osdw_decoding_z = property(lambda self: self._last["dec"][1].astype(np.int64))
    log_prob_ratios = property(lambda self: self._last["log_prob_ratios"].copy())
