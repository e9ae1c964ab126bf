"""A device allocation the GPU refuses returns SWD_ERR_NOMEM and leaves the handle working: after a batch far too large
for the device, the same handle decodes an earlier batch again with identical outputs.  The oversized call passes the
small host arrays of the first batch; the allocation is refused before any copy, so they are never read."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HUGE_B = 1 << 40        # shots: the first buffer sized by B alone would need tens of terabytes


def _code():
    from slidingwindowdecoder_b200.codes import bb_code
    return bb_code(72)[0]


def _syndromes(H, B, p, rng):
    err = (rng.random((B, H.shape[1])) < p).astype(np.int64)
    return np.ascontiguousarray(err @ H.T % 2, dtype=np.uint8)


def _check_refusal_and_retry(call, B, outs):
    """call(batch) -> status of a decode of the first `batch` shots into outs: OK for B, NOMEM for HUGE_B, then OK for B with
    the same outputs."""
    from slidingwindowdecoder_b200 import _lib
    lib = _lib.load()
    assert call(B) == _lib.OK
    first = [a.copy() for a in outs]
    assert any(a.any() for a in first)
    assert call(HUGE_B) == _lib.ERR_NOMEM
    assert b"cudaMalloc" in lib.swd_last_error()
    for a in outs:
        a.fill(0)
    assert call(B) == _lib.OK, lib.swd_last_error().decode()
    for a, b in zip(outs, first):
        np.testing.assert_array_equal(a, b)


def test_bp4_decoder_survives_refused_allocation():
    from slidingwindowdecoder_b200 import _lib, bp4_osd
    code = _code()
    n = code.N
    p = np.full(n, 0.02)
    dec = bp4_osd(code.hx, code.hz, channel_probs_x=p, channel_probs_y=p, channel_probs_z=p, osd_method="osd_cs", osd_order=4)
    rng = np.random.default_rng(11)
    B = 64
    sx, sz = _syndromes(code.hx, B, 0.03, rng), _syndromes(code.hz, B, 0.03, rng)
    outs = [np.zeros((B, 2, n), np.uint8), np.zeros(B, np.uint8), np.zeros((B, 2, n), np.uint8), np.zeros((B, 2, n), np.uint8),
            np.zeros((B, n, 3)), np.zeros(B, np.int32)]
    lib = _lib.load()

    def call(batch):
        return lib.swd_bp4_decode_batch_host(dec._handle, sx.ctypes.data, sz.ctypes.data, batch, *(a.ctypes.data for a in outs))

    _check_refusal_and_retry(call, B, outs)


def test_window_decoder_survives_refused_allocation():
    from slidingwindowdecoder_b200 import _lib, bpgdg_decoder
    code = _code()
    H, n = code.hx, code.N
    dec = bpgdg_decoder(H, channel_probs=np.full(n, 0.03), max_iter=8, multi_thread=True)
    B = 128
    synd = _syndromes(H, B, 0.04, np.random.default_rng(12))
    outs = [np.zeros((B, n), np.uint8), np.zeros(B, np.uint8), np.zeros(B)]
    lib = _lib.load()

    def call(batch):
        return lib.swd_decode_batch_host(dec._handle, synd.ctypes.data, batch, *(a.ctypes.data for a in outs))

    _check_refusal_and_retry(call, B, outs)
