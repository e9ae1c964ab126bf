"""Host-side pieces of circuit-level erasure sampling (no GPU): dem.noise_locations against detector_error_model, the
statistics of the numpy restatement tests/circuit_oracle.py::sample_circuit that the device sampler is tested against bit
for bit, the C-ABI declarations, and the argument checks the Python layer makes before any library call."""
import hashlib
import os

import numpy as np
import pytest

from conftest import ROOT

CIRCUIT_SYMBOLS = ("swd_window_set_circuit_noise", "swd_window_sample_circuit")


def _circuits():
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, shyps_memory_circuit
    out = []
    for N, rounds in ((72, 6), (144, 12)):
        code, A, B = bb_code(N)
        for z in (True, False):
            out.append((f"bb{N}x{rounds}_{'z' if z else 'x'}", bb_memory_circuit(code, A, B, 0.003, rounds, z_basis=z)))
    for z in (True, False):
        out.append((f"shyps3_{'z' if z else 'x'}", shyps_memory_circuit(3, 0.003, 3, z_basis=z)))
    return out


# sha256 (first 16 hex digits) of detector_error_model's output before noise_locations shared its backward pass
DEM_DIGEST = {"bb72x6_z": "383439c98d09168e", "bb72x6_x": "7c48667fe273f68f", "bb144x12_z": "082d23a96f7a85b6",
              "bb144x12_x": "28f78f8ce9f2fab2", "shyps3_z": "fe7ad2c8a7429f55", "shyps3_x": "667093c0a81c68c7"}
SIZES = {"bb72x6": (3924, 41004, 2232), "bb144x12": (15624, 164088, 8784)}


def _digest(dem):
    syms, probs, nd, no = dem
    m = hashlib.sha256()
    for s in syms:
        m.update(s.to_bytes((s.bit_length() + 7) // 8, "little") + b"|")
    m.update(np.asarray(probs, dtype=np.float64).tobytes())
    m.update(f"{nd},{no}".encode())
    return m.hexdigest()[:16]


def _combine_backward(locs, num_col):
    """XOR-combine mech_prob per column in detector_error_model's order: locations last to first, targets of one instruction
    first to last, mechanisms in order."""
    L = locs.num_locations
    order = np.lexsort((np.arange(L), -locs.op.astype(np.int64)))
    pri, seen = np.zeros(num_col), np.zeros(num_col, dtype=bool)
    for loc in order:
        for k in range(locs.mech_ptr[loc], locs.mech_ptr[loc + 1]):
            c, p = locs.mech_col[k], locs.mech_prob[k]
            if c < 0 or p <= 0.0:
                continue
            if seen[c]:
                q = pri[c]
                pri[c] = q * (1.0 - p) + p * (1.0 - q)
            else:
                pri[c], seen[c] = p, True
    return pri


def test_noise_locations_reproduce_dem():
    from slidingwindowdecoder_b200.dem import NOISE_KINDS, dem_to_check_matrices, detector_error_model, noise_locations
    for name, circ in _circuits():
        dem = detector_error_model(circ)
        assert _digest(dem) == DEM_DIGEST[name], name
        _, _, priors = dem_to_check_matrices(dem)
        locs = noise_locations(circ)
        L, M = locs.num_locations, int(locs.mech_ptr[-1])
        assert locs.mech_ptr.dtype == np.int32 and locs.mech_col.dtype == np.int32 and locs.mech_prob.dtype == np.float64
        assert locs.mech_ptr[0] == 0 and len(locs.mech_ptr) == L + 1 and len(locs.mech_col) == M == len(locs.mech_prob)
        cnt = np.diff(locs.mech_ptr)
        for kind, n in zip(NOISE_KINDS, (1, 1, 3, 15)):
            assert (cnt[locs.kind == kind] == n).all(), kind
        assert set(locs.kind) <= set(NOISE_KINDS) and (np.diff(locs.op) >= 0).all()
        assert -1 <= locs.mech_col.min() and locs.mech_col.max() < len(priors)
        assert not locs.mech_unmapped.any()
        assert np.array_equal(_combine_backward(locs, len(priors)), priors), name
        if name[:-2] in SIZES:
            assert (L, M, len(priors)) == SIZES[name[:-2]], name


def _one_gate(z_basis, p):
    """One CNOT with DEPOLARIZE2(p) between reset and measurement; the two detectors read the gate's X frames (z basis) or
    Z frames (x basis) of its two qubits."""
    from slidingwindowdecoder_b200.dem import Ops
    c = Ops()
    c.gate("R" if z_basis else "RX", 0, 1)
    c.gate("CNOT", 0, 1)
    c.noise("DEPOLARIZE2", p, 0, 1)
    c.gate("M" if z_basis else "MX", 0, 1)
    c.detector([-2])
    c.detector([-1])
    return c


@pytest.mark.parametrize("z_basis", (True, False))
def test_oracle_outcome_frequencies(z_basis):
    from scipy.stats import chisquare
    from circuit_oracle import sample_circuit
    from slidingwindowdecoder_b200.dem import _noise_locations, dem_to_check_matrices
    p, shots = 0.3, 20000
    locs, dem = _noise_locations(_one_gate(z_basis, p))
    chk, obs, priors = dem_to_check_matrices(dem)
    assert locs.num_locations == 1 and chk.shape == (2, 3)
    llr = np.log((1 - priors) / priors)
    # of the 15 non-identity two-qubit Paulis, 4 leave (0, 0) in the frames the detectors read, 4 give each other outcome
    for rate, want, seed in ((0.0, np.array([1 - p + 3 * p / 15] + [4 * p / 15] * 3), 5), (1.0, np.full(4, 0.25), 6)):
        det, _, err, erased, L = sample_circuit(chk, obs, locs, rate, llr, shots, seed=seed, shot_offset=1 << 33)
        assert (erased == (rate == 1.0)).all()
        assert np.array_equal(det, (err.astype(np.int64) @ chk.T.toarray() % 2).astype(np.uint8))
        assert np.array_equal(L, np.zeros_like(L) if rate else np.broadcast_to(llr, L.shape))
        k = det[:, 0].astype(np.int64) + 2 * det[:, 1]
        freq = np.bincount(k, minlength=4)
        assert chisquare(freq, want * shots).pvalue > 1e-3, (rate, freq)
        # per column: the DEM prior without erasures, 1/2 with
        col = err.mean(axis=0)
        target = priors if rate == 0 else np.full(3, 0.5)
        assert (np.abs(col - target) < 5 * np.sqrt(target * (1 - target) / shots)).all(), (rate, col)


def test_oracle_draw_layout():
    """Draw t of location l is word t & 3 of the call with counter (l, 2 + (t >> 2), shot): with every location erased,
    mechanism k fires iff draw 1 + k has its top bit clear."""
    from circuit_oracle import sample_circuit
    from oracle.philox import philox4x32_10
    from slidingwindowdecoder_b200.dem import _noise_locations, dem_to_check_matrices
    locs, dem = _noise_locations(_one_gate(True, 0.1))
    chk, obs, priors = dem_to_check_matrices(dem)
    shot, seed = (1 << 32) + 9, (3 << 32) | 5
    _, _, err, erased, _ = sample_circuit(chk, obs, locs, 1.0, np.zeros(3), 1, seed=seed, shot_offset=shot)
    assert erased.all()
    words = np.concatenate([np.array(philox4x32_10(np.uint32(0), np.uint32(2 + c), np.uint32(shot & 0xFFFFFFFF),
                                                   np.uint32(shot >> 32), seed & 0xFFFFFFFF, seed >> 32)).ravel() for c in range(4)])
    fired = words[1:16] < 0x80000000
    want = np.zeros(3, dtype=np.int64)
    for k in range(15):
        if fired[k] and locs.mech_col[k] >= 0:
            want[locs.mech_col[k]] ^= 1
    assert np.array_equal(err[0], want)


def test_circuit_entry_points_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "swd_b200.h")).read()
    for sym in CIRCUIT_SYMBOLS:
        assert sym + "(" in header, sym
    decl = header[header.index("swd_window_sample_circuit("):]
    decl = decl[:decl.index(";")]
    for arg in ("d_det", "d_obs", "d_err", "d_erased", "double *d_channel_llr", "void *stream"):
        assert arg in decl, arg
    decl = header[header.index("swd_window_set_circuit_noise("):]
    decl = decl[:decl.index(";")]
    for arg in ("int num_loc", "const int32_t *mech_ptr", "const int32_t *mech_col", "const double *mech_prob",
                "const double *erasure_rate", "const double *col_llr"):
        assert arg in decl, arg
    from slidingwindowdecoder_b200 import _lib
    for sym in CIRCUIT_SYMBOLS:
        assert sym in _lib.EXPORTS, sym


@pytest.fixture()
def no_library(monkeypatch):
    """Any call into the native library fails the test: the checks below must fire first."""
    from slidingwindowdecoder_b200 import _lib

    def refuse():
        raise AssertionError("the native library was loaded before the arguments were checked")
    monkeypatch.setattr(_lib, "load", refuse)


def test_python_validation_before_library(no_library):
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, circuit_erasure_decoding
    from slidingwindowdecoder_b200.dem import Ops, noise_locations
    circ = _one_gate(True, 0.01)
    L = noise_locations(circ).num_locations
    for rate in (-0.1, 1.5, float("nan"), np.zeros(L + 1), np.zeros((L, 1)), np.full(L, np.nan), np.full(L, 2.0)):
        with pytest.raises(ValueError):
            CircuitNoiseSampler(circ, erasure_rate=rate)
    # an erased location whose mechanism has no DEM column (p = 0 and no other mechanism with its symptom)
    c = Ops()
    c.gate("R", 0, 1)
    c.noise("X_ERROR", 0.01, 0)
    c.noise("DEPOLARIZE2", 0.0, 0, 1)
    c.gate("M", 0, 1)
    c.detector([-2])
    c.detector([-1])
    locs = noise_locations(c)
    assert locs.mech_unmapped.any()
    with pytest.raises(ValueError):
        CircuitNoiseSampler(c, erasure_rate=0.5)
    with pytest.raises(ValueError):
        CircuitNoiseSampler(c, erasure_rate=np.array([0.0, 0.5]))
    empty = Ops()
    empty.gate("R", 0)
    empty.gate("M", 0)
    empty.detector([-1])
    with pytest.raises(ValueError):
        CircuitNoiseSampler(empty)
    for kw in (dict(N=7), dict(p=0.0), dict(p=0.5), dict(p=-0.1), dict(batch=0), dict(num_shots=-1), dict(shot_offset=-1),
               dict(decoder="bp")):
        full = dict(N=72, p=0.001, erasure_rate=0.01)
        full.update(kw)
        with pytest.raises(ValueError):
            circuit_erasure_decoding(**full)
