"""Host-side pieces of code-capacity sampling (no GPU): the statistics of the numpy restatement tests/pauli_oracle.py::sample_pauli
that the device sampler is tested against bit for bit, the C-ABI declarations, and the argument checks that the Python layer
makes before any library call."""
import os

import numpy as np
import pytest

from conftest import ROOT

PAULI_SYMBOLS = ("swd_window_set_pauli_priors", "swd_window_sample_pauli")


def _stacked(code):
    from scipy.sparse import bmat, csc_matrix
    hx, hz, lx, lz = (csc_matrix(M) for M in (code.hx, code.hz, code.lx, code.lz))
    return bmat([[None, hx], [hz, None]], format="csc"), bmat([[lz, None], [None, lx]], format="csc")


def test_sample_pauli_statistics():
    from pauli_oracle import sample_pauli
    from slidingwindowdecoder_b200.codes import bb_code
    code, _, _ = bb_code(72)
    chk, obs = _stacked(code)
    n, shots, rate = code.N, 20000, 0.1
    px, py, pz = np.full(n, 0.05), np.full(n, 0.02), np.full(n, 0.08)
    llr5 = np.arange(5 * n, dtype=np.float64).reshape(5, n) + 1.0
    det, ob, err, erased, L = sample_pauli(chk, obs, px, py, pz, rate, shots, seed=(7 << 32) | 11, shot_offset=3 << 32, llr5=llr5)
    assert det.shape == (shots, code.hx.shape[0] + code.hz.shape[0]) and ob.shape == (shots, 2 * code.K)
    assert err.shape == (shots, 2 * n) and erased.shape == (shots, n) and L.shape == (5, shots, n)
    e = err.astype(np.int64)
    assert np.array_equal(det, (np.asarray(chk.todense()).astype(np.int64) @ e.T % 2).T)
    assert np.array_equal(ob, (np.asarray(obs.todense()).astype(np.int64) @ e.T % 2).T)
    ex, ez = err[:, :n].astype(bool), err[:, n:].astype(bool)
    pauli = np.where(ex & ~ez, 1, np.where(ex & ez, 2, np.where(ez, 3, 0)))
    er = erased.astype(bool)

    def within(count, total, p):
        return abs(count - total * p) <= 5 * np.sqrt(total * p * (1 - p))

    assert within(er.sum(), er.size, rate)
    kept = pauli[~er]
    for k, p in ((1, 0.05), (2, 0.02), (3, 0.08)):
        assert within((kept == k).sum(), kept.size, p), k
    lost = pauli[er]
    for k in range(4):
        assert within((lost == k).sum(), lost.size, 0.25), k
    assert (L[:, er] == 0.0).all() and (L[:, ~er] == np.broadcast_to(llr5[:, None, :], L.shape)[:, ~er]).all()


def test_sample_pauli_draw_layout():
    """Word 2j / 2j + 1 of the call with counter (k, 1, shot) are the erasure / Pauli draws of qubit 2k + j."""
    from oracle.philox import philox4x32_10
    from pauli_oracle import sample_pauli
    from scipy.sparse import csc_matrix
    n, shot, seed = 5, (1 << 32) + 9, (3 << 32) | 5
    chk = csc_matrix(np.eye(2 * n, dtype=np.uint8))
    obs = csc_matrix(np.zeros((1, 2 * n), dtype=np.uint8))
    _, _, err, erased, _ = sample_pauli(chk, obs, np.zeros(n), np.zeros(n), np.zeros(n), 1.0, 1, seed=seed, shot_offset=shot)
    assert erased.all()
    for v in range(n):
        r = philox4x32_10(np.uint32(v // 2), np.uint32(1), np.uint32(shot & 0xFFFFFFFF), np.uint32(shot >> 32), seed & 0xFFFFFFFF, seed >> 32)
        pauli = int(r[2 * (v % 2) + 1]) >> 30
        assert err[0, v] == (pauli in (1, 2)) and err[0, n + v] == (pauli in (2, 3)), v
    # no erasures and px = 1: every qubit is X whatever the draw
    _, _, err, erased, _ = sample_pauli(chk, obs, np.ones(n), np.zeros(n), np.zeros(n), 0.0, 4, seed=seed)
    assert not erased.any() and err[:, :n].all() and not err[:, n:].any()


def test_code_capacity_entry_points_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "swd_b200.h")).read()
    for sym in PAULI_SYMBOLS:
        assert sym + "(" in header, sym
    decl = header[header.index("swd_window_sample_pauli("):]
    decl = decl[:decl.index(";")]
    for arg in ("d_det", "d_obs", "d_err", "d_erased", "double *d_channel_llr", "void *stream"):
        assert arg in decl, arg
    from slidingwindowdecoder_b200 import _lib
    for sym in PAULI_SYMBOLS:
        assert sym in _lib.EXPORTS, sym


@pytest.fixture()
def no_library(monkeypatch):
    """Any call into the native library fails the test: the checks below must fire first."""
    from slidingwindowdecoder_b200 import _lib

    def refuse():
        raise AssertionError("the native library was loaded before the arguments were checked")
    monkeypatch.setattr(_lib, "load", refuse)


def test_python_validation_before_library(no_library):
    from slidingwindowdecoder_b200 import CodeCapacitySampler, depolarizing_noise_decoding
    from slidingwindowdecoder_b200.codes import bb_code
    code, _, _ = bb_code(72)
    n = code.N
    p = np.full(n, 0.01)
    args = (code.hx, code.hz, code.lx, code.lz)
    bad = [
        dict(px=np.full(n - 1, 0.01)),                                   # wrong length
        dict(py=np.full((n, 1), 0.01)),                                  # wrong shape
        dict(pz=np.where(np.arange(n) == 3, -0.01, 0.01)),               # negative
        dict(px=np.where(np.arange(n) == 0, np.nan, 0.01)),              # NaN
        dict(px=np.full(n, 0.5), py=np.full(n, 0.3), pz=np.full(n, 0.3)),  # px + py + pz > 1
        dict(erasure_rate=-0.1), dict(erasure_rate=1.5), dict(erasure_rate=float("nan")),
        dict(channel_llr=np.zeros((5, n - 1))), dict(channel_llr=np.zeros((4, n))),
    ]
    for kw in bad:
        full = dict(px=p, py=p, pz=p)
        full.update(kw)
        with pytest.raises(ValueError):
            CodeCapacitySampler(*args, **full)
    with pytest.raises(ValueError):
        CodeCapacitySampler(code.hx, code.hz[:, :-1], code.lx, code.lz, p, p, p)
    for kw in (dict(p=0.0), dict(p=1.0), dict(p=-0.1), dict(p=0.01, batch=0), dict(p=0.01, num_shots=-1),
               dict(p=0.01, shot_offset=-1)):
        with pytest.raises(ValueError):
            depolarizing_noise_decoding(code, verbose=False, **kw)
