"""Host-side pieces of soft measurement readout (no GPU): dem.readout_locations, with_readout_error and gaussian_readout, the
per-class LLR table against a direct XOR-combination, the statistics and draw layout of the numpy restatement
tests/readout_oracle.py that the device sampler is tested against bit for bit, the C-ABI declarations, and the argument
checks the Python layer makes before any library call."""
import math
import os

import numpy as np
import pytest

from conftest import ROOT

READOUT_SYMBOLS = ("swd_window_set_circuit_readout", "swd_window_sample_circuit_readout")
# readout locations, and how many of them have a DEM column
COUNTS = {"bb72x6_z": (432, 216), "bb72x6_x": (432, 216), "bb144x12_z": (1728, 864), "shyps3_z": (343, 196)}


def _circuit(name, p=0.003):
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, shyps_memory_circuit
    if name == "shyps3_z":
        return shyps_memory_circuit(3, p, 3)
    N, rounds = (72, 6) if name.startswith("bb72") else (144, 12)
    code, A, B = bb_code(N)
    return bb_memory_circuit(code, A, B, p, rounds, z_basis=name.endswith("_z"))


def _target(locs, l):
    """(op index, target position) of location l."""
    oi = int(locs.op[l])
    return oi, l - int(np.searchsorted(locs.op, oi))


@pytest.mark.parametrize("name", sorted(COUNTS))
def test_readout_locations(name):
    from slidingwindowdecoder_b200.dem import _noise_locations, readout_locations
    circ = _circuit(name)
    locs, dem = _noise_locations(circ)
    ro = readout_locations(circ)
    assert ro.dtype == np.int32 and (np.diff(ro) > 0).all()
    cnt = np.diff(locs.mech_ptr)
    assert (cnt[ro] == 1).all()
    cols = locs.mech_col[locs.mech_ptr[ro]]
    assert (len(ro), int((cols >= 0).sum())) == COUNTS[name]
    assert len(np.unique(cols[cols >= 0])) == int((cols >= 0).sum())          # no two share a DEM column
    basis = {"X_ERROR": ("M", "MR"), "Z_ERROR": ("MX", "MRX")}
    is_ro = np.zeros(locs.num_locations, dtype=bool)
    is_ro[ro] = True
    for l in np.flatnonzero(np.isin(locs.kind, ("X_ERROR", "Z_ERROR"))):
        oi, k = _target(locs, l)
        name_, t, _ = circ.ops[oi]
        q = t[k]
        nxt = next((op for op in circ.ops[oi + 1:] if op[0] not in ("DETECTOR", "OBSERVABLE_INCLUDE", "TICK") and q in op[1]), None)
        assert is_ro[l] == (nxt is not None and nxt[0] in basis[name_]), l


def test_with_readout_error():
    from slidingwindowdecoder_b200.dem import Ops, detector_error_model, noise_locations, readout_locations, with_readout_error
    circ = _circuit("bb72x6_z", p=0.003)
    same = with_readout_error(circ, 0.003)
    assert same.ops == circ.ops and same is not circ
    assert detector_error_model(same) == detector_error_model(circ)
    other = with_readout_error(circ, 0.02)
    ro = readout_locations(circ)
    locs = noise_locations(circ)
    changed = {i for i, (a, b) in enumerate(zip(circ.ops, other.ops)) if a != b}
    assert changed == {int(locs.op[l]) for l in ro}
    assert all(other.ops[i][2] == 0.02 and other.ops[i][:2] == circ.ops[i][:2] for i in changed)
    assert (other.num_measurements, other.num_detectors, other.num_observables) == \
        (circ.num_measurements, circ.num_detectors, circ.num_observables)
    assert np.array_equal(readout_locations(other), ro)
    lo = noise_locations(other)
    assert (lo.mech_prob[lo.mech_ptr[ro]] == 0.02).all()
    for bad in (-0.1, 0.6, float("nan")):
        with pytest.raises(ValueError):
            with_readout_error(circ, bad)
    part = Ops()                                   # X_ERROR on 0 and 1, only qubit 0 measured next
    part.gate("R", 0, 1)
    part.noise("X_ERROR", 0.01, 0, 1)
    part.gate("M", 0)
    part.gate("H", 1)
    part.gate("M", 1)
    part.detector([-2])
    assert readout_locations(part).tolist() == [0]
    with pytest.raises(ValueError):
        with_readout_error(part, 0.02)


@pytest.mark.parametrize("p_meas", (1e-4, 0.003, 0.01, 0.2))
@pytest.mark.parametrize("K", (1, 2, 4, 16, 256))
def test_gaussian_readout(p_meas, K):
    from slidingwindowdecoder_b200.dem import ReadoutModel, gaussian_readout
    m = gaussian_readout(p_meas, K)
    assert isinstance(m, ReadoutModel) and m.num_classes == K
    assert m.weights.dtype == np.float64 and m.flip_prob.dtype == np.float64
    assert abs(math.fsum(m.weights) - 1.0) <= 1e-12 and (m.weights > 0).all()
    assert abs(m.marginal - p_meas) <= 1e-12 * p_meas
    assert (np.diff(m.flip_prob) <= 0).all() and (m.flip_prob >= 0).all() and (m.flip_prob <= 0.5).all()
    if K == 1:
        assert m.flip_prob.tolist() == [p_meas]


def test_gaussian_readout_values():
    """p_meas = 0.003, K = 16: class 0 flips with 4.7e-2, class 15 with about 1.7e-11."""
    from slidingwindowdecoder_b200.dem import gaussian_readout
    q = gaussian_readout(0.003, 16).flip_prob
    assert q[0] == pytest.approx(0.0474, rel=1e-2) and q[15] == pytest.approx(1.66e-11, rel=2e-2)


def _fold_by_column(locs):
    """Per DEM column: its mechanisms in detector_error_model's fold order."""
    order = np.lexsort((np.arange(locs.num_locations), -locs.op.astype(np.int64)))
    out = {}
    for l in order:
        for k in range(locs.mech_ptr[l], locs.mech_ptr[l + 1]):
            if locs.mech_col[k] >= 0:
                out.setdefault(int(locs.mech_col[k]), []).append(k)
    return out


@pytest.mark.parametrize("name", ("bb72x6_z", "bb72x6_x", "shyps3_z"))
def test_class_llr(name):
    from slidingwindowdecoder_b200.decoders import _libm_llr
    from slidingwindowdecoder_b200.dem import _noise_locations, dem_to_check_matrices, gaussian_readout, readout_locations
    from slidingwindowdecoder_b200.simulation import _readout_class_llr
    circ = _circuit(name, p=0.004)
    locs, dem = _noise_locations(circ)
    _, _, priors = dem_to_check_matrices(dem)
    static = _libm_llr(priors, len(priors))
    ro = readout_locations(circ)
    cols = locs.mech_col[locs.mech_ptr[ro]]
    one = _readout_class_llr(locs, ro, [0.004], len(priors))
    assert one.shape == (len(ro), 1)
    assert np.array_equal(one[cols >= 0, 0].view(np.uint64), static[cols[cols >= 0]].view(np.uint64))
    assert (one[cols < 0] == 0.0).all()
    q = gaussian_readout(0.004, 16).flip_prob
    table = _readout_class_llr(locs, ro, q, len(priors))
    by_col = _fold_by_column(locs)
    for r in np.flatnonzero(cols >= 0):
        for k in range(16):
            acc = None
            for m in by_col[int(cols[r])]:
                p = q[k] if m == locs.mech_ptr[ro[r]] else locs.mech_prob[m]
                if p > 0:
                    acc = p if acc is None else acc * (1 - p) + p * (1 - acc)
            want = math.log((1 - acc) / acc)
            assert abs(table[r, k] - want) <= 1e-12 * max(1.0, abs(want)), (r, k)
    assert (np.diff(table[cols >= 0], axis=1) >= 0).all()               # more reliable classes, larger LLR


def _one_readout(p, basis="Z"):
    """One flip before one measurement, read by one detector."""
    from slidingwindowdecoder_b200.dem import Ops
    c = Ops()
    c.gate("R" if basis == "Z" else "RX", 0)
    c.noise("X_ERROR" if basis == "Z" else "Z_ERROR", p, 0)
    c.gate("M" if basis == "Z" else "MX", 0)
    c.detector([-1])
    return c


@pytest.mark.parametrize("basis", ("Z", "X"))
def test_oracle_statistics(basis):
    """Class frequencies against the weights, and the flip frequency per class against q (chi-square); erased flips 1/2."""
    from scipy.stats import chisquare
    from readout_oracle import sample_circuit_readout
    from slidingwindowdecoder_b200.dem import ReadoutModel, _noise_locations, dem_to_check_matrices, readout_locations
    w, q = np.array([0.1, 0.2, 0.3, 0.4]), np.array([0.4, 0.2, 0.1, 0.01])
    model = ReadoutModel(w, q)
    locs, dem = _noise_locations(_one_readout(model.marginal, basis))
    chk, obs, priors = dem_to_check_matrices(dem)
    ro = readout_locations(_one_readout(model.marginal, basis))
    assert ro.tolist() == [0] and chk.shape == (1, 1)
    shots = 40000
    table = np.log((1 - q) / q)[None, :]
    for rate, seed in ((0.0, 3), (1.0, 4)):
        det, _, err, erased, cls, L = sample_circuit_readout(chk, obs, locs, rate, np.log((1 - priors) / priors), ro, w, q, table,
                                                             shots, seed=seed, shot_offset=(1 << 34) + 5)
        assert (erased == rate).all() and np.array_equal(det, err)
        c = cls[:, 0].astype(np.int64)
        freq = np.bincount(c, minlength=4)
        assert chisquare(freq, w * shots).pvalue > 1e-3, freq
        flips = np.bincount(c, weights=det[:, 0], minlength=4)
        want = q if rate == 0 else np.full(4, 0.5)
        stat = ((flips - freq * want) ** 2 / (freq * want * (1 - want))).sum()
        from scipy.stats import chi2
        assert chi2.sf(stat, 4) > 1e-3, (flips / freq, want)
        assert np.array_equal(L[:, 0], np.zeros(shots) if rate else table[0, c])


def test_oracle_draw_layout():
    """Readout location l: words 0, 1, 2 of the call with counter (l, 2, shot) are the erasure, flip and class draws."""
    from oracle.philox import philox4x32_10, thresholds
    from readout_oracle import class_thresholds, sample_circuit_readout
    from slidingwindowdecoder_b200.dem import _noise_locations, dem_to_check_matrices
    w, q = np.full(8, 1 / 8), np.linspace(0.45, 0.0, 8)
    locs, dem = _noise_locations(_one_readout(float(np.dot(w, q))))
    chk, obs, _ = dem_to_check_matrices(dem)
    seed = (7 << 32) | 11
    for shot in (0, (1 << 32) + 9, 12345):
        det, _, _, erased, cls, _ = sample_circuit_readout(chk, obs, locs, 0.3, np.zeros(1), [0], w, q, np.zeros((1, 8)), 1,
                                                           seed=seed, shot_offset=shot)
        r = [int(np.ravel(x)[0]) for x in philox4x32_10(np.uint32(0), np.uint32(2), np.uint32(shot & 0xFFFFFFFF), np.uint32(shot >> 32),
                                              seed & 0xFFFFFFFF, seed >> 32)]
        er = r[0] < int(thresholds(np.array([0.3]))[0])
        k = int((r[2] >= class_thresholds(w)).sum())
        fire = r[1] < (0x80000000 if er else int(thresholds(q)[k]))
        assert (erased[0, 0], cls[0, 0], det[0, 0]) == (er, k, fire), shot


def test_readout_entry_points_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "swd_b200.h")).read()
    decl = header[header.index("swd_window_set_circuit_readout("):]
    decl = decl[:decl.index(";")]
    for arg in ("int num_readout", "const int32_t *readout_loc", "int num_classes", "const double *class_weight",
                "const double *flip_prob", "const double *class_llr"):
        assert arg in decl, arg
    decl = header[header.index("swd_window_sample_circuit_readout("):]
    decl = decl[:decl.index(";")]
    for arg in ("d_det", "d_obs", "d_err", "d_erased", "uint8_t *d_readout", "double *d_channel_llr", "void *stream"):
        assert arg in decl, arg
    from slidingwindowdecoder_b200 import _lib
    import slidingwindowdecoder_b200 as pkg
    for sym in READOUT_SYMBOLS:
        assert sym in _lib.EXPORTS, sym
    for name in ("CircuitNoiseSampler", "circuit_soft_readout_decoding", "gaussian_readout"):
        assert hasattr(pkg, name), name


@pytest.fixture()
def no_library(monkeypatch):
    """Any call into the native library fails the test: the checks below must fire first."""
    from slidingwindowdecoder_b200 import _lib

    def refuse():
        raise AssertionError("the native library was loaded before the arguments were checked")
    monkeypatch.setattr(_lib, "load", refuse)


def test_python_validation_before_library(no_library):
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, circuit_soft_readout_decoding, gaussian_readout
    from slidingwindowdecoder_b200.dem import Ops, ReadoutModel
    for w, q in (([], []), (np.full(257, 1 / 257), np.zeros(257)), ([0.5, 0.5], [0.1]), ([1.5, -0.5], [0.1, 0.1]),
                 ([0.5, 0.6], [0.1, 0.1]), ([np.nan, 1.0], [0.1, 0.1]), ([1.0], [0.6]), ([1.0], [-0.1]), ([1.0], [np.nan])):
        with pytest.raises(ValueError):
            ReadoutModel(w, q)
    for p, K in ((0.0, 4), (0.5, 4), (-0.1, 4), (float("nan"), 4), (0.01, 0), (0.01, 257)):
        with pytest.raises(ValueError):
            gaussian_readout(p, K)
    circ = _one_readout(0.01)
    with pytest.raises(ValueError):
        CircuitNoiseSampler(circ, readout=(np.ones(1), np.full(1, 0.01)))        # not a ReadoutModel
    with pytest.raises(ValueError):
        CircuitNoiseSampler(circ, readout=ReadoutModel([1.0], [0.0101]))          # marginal differs from the circuit's 0.01
    with pytest.raises(ValueError, match="location 0 "):
        CircuitNoiseSampler(circ, readout=gaussian_readout(0.02, 4))
    no_ro = Ops()                                                                 # a flip, but not right before the measurement
    no_ro.gate("R", 0)
    no_ro.noise("X_ERROR", 0.01, 0)
    no_ro.gate("H", 0)
    no_ro.gate("H", 0)
    no_ro.gate("M", 0)
    no_ro.detector([-1])
    with pytest.raises(ValueError):
        CircuitNoiseSampler(no_ro, readout=ReadoutModel([1.0], [0.01]))
    shared = Ops()                                                                # two flips whose symptoms are the same column
    shared.gate("R", 0, 1)
    shared.noise("X_ERROR", 0.01, 0, 1)
    shared.gate("M", 0, 1)
    shared.detector([-1, -2])
    with pytest.raises(ValueError, match="share"):
        CircuitNoiseSampler(shared, readout=ReadoutModel([1.0], [0.01]))
    for kw in (dict(N=7), dict(p=0.0), dict(p=0.5), dict(p_meas=0.0), dict(p_meas=0.5), dict(p_meas=-0.1), dict(num_classes=0),
               dict(num_classes=257), dict(batch=0), dict(num_shots=-1), dict(shot_offset=-1), dict(decoder="bp")):
        full = dict(N=72, p=0.001, p_meas=0.01, num_classes=16)
        full.update(kw)
        with pytest.raises(ValueError):
            circuit_soft_readout_decoding(**full)
