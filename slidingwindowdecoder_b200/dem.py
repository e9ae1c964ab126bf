"""Stim-free circuit-level noise model -> detector error model (host-side setup, numpy).

The reference builds its syndrome-extraction circuits with stim (src/build_circuit.py:6-234) and
turns `circuit.detector_error_model()` into (chk, obs, priors) with dem_to_check_matrices
(src/build_circuit.py:236-299).  stim is not available here, so this module provides

  * `Ops`: a flat instruction list (Clifford gates R/RX/H/CNOT/M/MX/MR/MRX, the Pauli noise
    channels X_ERROR/Z_ERROR/DEPOLARIZE1/DEPOLARIZE2, DETECTOR / OBSERVABLE_INCLUDE),
  * `bb_memory_circuit`: the BB-code memory experiment with exactly the gate schedule and noise
    placement of build_circuit.py (default flags: HZH=False, use_both=False),
  * `detector_error_model`: backward Pauli-sensitivity propagation (which detectors/observables
    would an X or Z fault at this point flip), independent-mechanism probabilities for the
    depolarising channels, and merging of mechanisms with identical symptoms,
  * `dem_to_check_matrices`: same return values as the reference function,
  * `readout_locations`, `with_readout_error`, `gaussian_readout` / `ReadoutModel`: the measurement flips of a circuit and
    the soft-readout model that CircuitNoiseSampler samples them with.

Symptom sets are Python ints used as bit masks: bit d = detector d, bit num_detectors + o =
observable o.
"""
import math
from dataclasses import dataclass

import numpy as np
from scipy.sparse import csc_matrix


class Ops:
    """Flat circuit: list of tuples (name, targets tuple, arg)."""

    def __init__(self):
        self.ops = []
        self.num_measurements = 0
        self.num_detectors = 0
        self.num_observables = 0

    def gate(self, name, *qubits):
        self.ops.append((name, tuple(int(q) for q in qubits), None))
        if name in ("M", "MX", "MR", "MRX"):
            self.num_measurements += len(qubits)

    def noise(self, name, p, *qubits):
        self.ops.append((name, tuple(int(q) for q in qubits), float(p)))

    def detector(self, rec_offsets):
        """rec_offsets: negative look-back indices into the measurement record (stim's rec[-k])."""
        abs_idx = tuple(self.num_measurements + int(k) for k in rec_offsets)
        assert all(0 <= a < self.num_measurements for a in abs_idx)
        self.ops.append(("DETECTOR", abs_idx, self.num_detectors))
        self.num_detectors += 1

    def observable(self, index, rec_offsets):
        abs_idx = tuple(self.num_measurements + int(k) for k in rec_offsets)
        assert all(0 <= a < self.num_measurements for a in abs_idx)
        self.ops.append(("OBSERVABLE_INCLUDE", abs_idx, int(index)))
        self.num_observables = max(self.num_observables, int(index) + 1)


def _perm_targets(M):
    """For a permutation matrix: out[i] = column of the 1 in row i (build_circuit.py:12-14)."""
    M = np.asarray(M)
    r, c = np.nonzero(M)
    out = np.zeros(M.shape[0], dtype=np.int64)
    out[r] = c
    return out


def bb_memory_circuit(code, A_list, B_list, p, num_repeat, z_basis=True):
    """Noisy memory experiment of a bivariate-bicycle code: the circuit of build_circuit.py:6-234.

    Qubit layout: X-check ancillas 0..n/2-1, L data n/2..n-1, R data n..3n/2-1, Z-check ancillas
    3n/2..2n-1.  Each round has 8 layers; depolarising noise after every CNOT and on idling data
    qubits, flips after resets and before measurements, all with the same strength p.
    """
    n = code.N
    h = n // 2
    a1, a2, a3 = [np.asarray(a) for a in A_list]
    b1, b2, b3 = [np.asarray(b) for b in B_list]
    A1, A2, A3 = _perm_targets(a1), _perm_targets(a2), _perm_targets(a3)
    B1, B2, B3 = _perm_targets(b1), _perm_targets(b2), _perm_targets(b3)
    A1t, A2t, A3t = _perm_targets(a1.T), _perm_targets(a2.T), _perm_targets(a3.T)
    B1t, B2t, B3t = _perm_targets(b1.T), _perm_targets(b2.T), _perm_targets(b3.T)
    XC, LD, RD, ZC = 0, h, n, 3 * h

    c = Ops()

    def cnot(ctrl, tgt):
        c.gate("CNOT", ctrl, tgt)
        c.noise("DEPOLARIZE2", p, ctrl, tgt)

    # (x-check target block, x-check target perm, z-check source block, z-check source perm) for layers 2..6
    middle = [(LD, A2, RD, A3t), (RD, B2, LD, B1t), (RD, B1, LD, B2t), (RD, B3, LD, B3t), (LD, A1, RD, A2t)]

    def block(repeat):
        # layer 1
        if repeat:
            for i in range(h):
                c.noise("X_ERROR", p, ZC + i)
                c.noise("Z_ERROR", p, XC + i)
                c.noise("DEPOLARIZE1", p, RD + i)
        else:
            for i in range(h):
                c.gate("H", XC + i)
        for i in range(h):
            cnot(RD + A1t[i], ZC + i)
            c.noise("DEPOLARIZE1", p, LD + i)
        # layers 2..6
        for xt_blk, xt, zs_blk, zs in middle:
            for i in range(h):
                cnot(XC + i, xt_blk + xt[i])
                cnot(zs_blk + zs[i], ZC + i)
        # layer 7
        for i in range(h):
            cnot(XC + i, LD + A3[i])
            c.noise("X_ERROR", p, ZC + i)
            c.gate("MR", ZC + i)
        if z_basis:
            for i in range(h):
                c.detector([-h + i, -n - h + i] if repeat else [-h + i])
        # layer 8
        for i in range(h):
            c.noise("Z_ERROR", p, XC + i)
            c.gate("MRX", XC + i)
        if not z_basis:
            for i in range(h):
                c.detector([-h + i, -n - h + i] if repeat else [-h + i])

    for i in range(h):
        c.gate("R", XC + i)
        c.gate("R", ZC + i)
        c.noise("X_ERROR", p, XC + i)
        c.noise("X_ERROR", p, ZC + i)
    for i in range(n):
        c.gate("R" if z_basis else "RX", LD + i)
        c.noise("X_ERROR" if z_basis else "Z_ERROR", p, LD + i)
    block(False)
    for _ in range(num_repeat - 1):
        block(True)
    for i in range(n):
        c.gate("M" if z_basis else "MX", LD + i)
    pcm = code.hz if z_basis else code.hx
    logical = code.lz if z_basis else code.lx
    for i, row in enumerate(np.asarray(pcm)):
        rec = [-n + int(j) for j in np.nonzero(row)[0]]
        rec.append(-n - n + i if z_basis else -n - h + i)
        c.detector(rec)
    for i, row in enumerate(np.asarray(logical)):
        c.observable(i, [-n + int(j) for j in np.nonzero(row)[0]])
    return c


def _gf2_polydiv(num, den):
    """Quotient and remainder of GF(2) polynomials given as coefficient lists (increasing degree)."""
    num = list(num); den = list(den)
    dn = max(i for i, c in enumerate(den) if c)
    quo = [0] * max(1, len(num) - dn)
    for i in range(len(num) - 1, dn - 1, -1):
        if num[i]:
            quo[i - dn] = 1
            for k in range(dn + 1):
                num[i - dn + k] ^= den[k]
    return quo, num[:dn]


def shyps_code(r):
    """Subsystem hypergraph-product simplex code (build_SHYPS_circuit.py:9-57): gauge / stabiliser / logical matrices."""
    n_r = 2 ** r - 1
    taps = {3: [0, 2, 3], 4: [0, 3, 4], 5: [0, 2, 5]}[r]          # primitive h(x)
    hpoly = [0] * (max(taps) + 1)
    for t in taps:
        hpoly[t] = 1
    first = np.zeros(n_r, dtype=np.int64); first[:len(hpoly)] = hpoly
    H = np.array([np.roll(first, i) for i in range(n_r)])
    xn = [1] + [0] * (n_r - 1) + [1]                                # x^n - 1
    gpoly, rem = _gf2_polydiv(xn, hpoly)
    assert not any(rem)
    gfirst = np.zeros(n_r, dtype=np.int64); gfirst[:len(gpoly)] = gpoly
    G = np.array([np.roll(gfirst, i) for i in range(r)])
    assert not (G @ H % 2).any()
    I = np.identity(n_r, dtype=np.int64)
    from .codes import gf2_row_reduce
    # P with P G^T = I_r: row-reduce G^T (n_r x r); the transform's first r rows invert the pivot block
    R, piv, rk, Tm = gf2_row_reduce(G.T)
    assert rk == r
    P = Tm[:r].astype(np.int64)
    assert np.array_equal(P @ G.T % 2, np.identity(r, dtype=np.int64))
    return dict(r=r, n_r=n_r, N=n_r * n_r, H=H, G=G,
                S_X=np.kron(H.T, G), gauge_X=np.kron(H.T, I), aggregate_X=np.kron(I, G),
                S_Z=np.kron(G, H.T), gauge_Z=np.kron(I, H.T), aggregate_Z=np.kron(G, I),
                L_X=np.kron(P, G), L_Z=np.kron(G, P))


def _edge_colouring_circulant(M):
    """Proper edge colouring of a bipartite graph whose every row and column has the same degree D, by repeated
    perfect matchings (Hall); returns D lists of (row, col).  (The reference uses Hopcroft-Karp matchings,
    utils.py:577-623; any proper colouring is a valid CNOT schedule.)"""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import maximum_bipartite_matching
    M = np.array(M, dtype=np.int64).copy()
    colours = []
    while M.any():
        match = maximum_bipartite_matching(csr_matrix(M), perm_type="column")
        layer = [(u, int(v)) for u, v in enumerate(match) if v >= 0]
        for u, v in layer:
            M[u, v] = 0
        colours.append(layer)
    return colours


def shyps_memory_circuit(r, p, num_repeat, z_basis=True):
    """Memory experiment of the SHYPS code with the gate order and noise placement of build_SHYPS_circuit.py:59-191
    (gauge measurements in 3 + 3 CNOT layers per round, detectors on aggregated gauge outcomes)."""
    cd = shyps_code(r)
    N = cd["N"]
    XG, DQ, ZG = 0, N, 2 * N
    col_Z = _edge_colouring_circulant(cd["gauge_Z"])
    col_X = _edge_colouring_circulant(cd["gauge_X"])
    assert len(col_Z) == 3 and len(col_X) == 3
    agg = cd["aggregate_Z"] if z_basis else cd["aggregate_X"]
    c = Ops()

    def detectors(repeat):
        for row in agg:
            rec = []
            for i in np.nonzero(row)[0]:
                rec.append(-N + int(i))
                if repeat:
                    rec.append(-3 * N + int(i))
            c.detector(rec)

    def block(repeat):
        if repeat:
            for i in range(N):
                c.noise("X_ERROR", p, ZG + i)
                c.noise("Z_ERROR", p, XG + i)
                c.noise("DEPOLARIZE1", p, DQ + i)
        for layer in col_Z:
            for g, dq in layer:
                c.gate("CNOT", DQ + dq, ZG + g)
                c.noise("DEPOLARIZE2", p, DQ + dq, ZG + g)
        for i in range(N):
            c.noise("X_ERROR", p, ZG + i)
            c.gate("M", ZG + i)
        if z_basis:
            detectors(repeat)
        for i in range(N):
            c.gate("RX", XG + i)
            c.noise("Z_ERROR", p, XG + i)
        for layer in col_X:
            for g, dq in layer:
                c.gate("CNOT", XG + g, DQ + dq)
                c.noise("DEPOLARIZE2", p, XG + g, DQ + dq)
        for i in range(N):
            c.noise("Z_ERROR", p, XG + i)
            c.gate("MX", XG + i)
        if not z_basis:
            detectors(repeat)
        for i in range(N):
            c.gate("R", ZG + i)
            c.noise("X_ERROR", p, ZG + i)

    for i in range(N):
        c.gate("RX", XG + i); c.noise("Z_ERROR", p, XG + i)
        c.gate("R", ZG + i); c.noise("X_ERROR", p, ZG + i)
    for i in range(N):
        c.gate("R" if z_basis else "RX", DQ + i)
        c.noise("X_ERROR" if z_basis else "Z_ERROR", p, DQ + i)
    block(False)
    for _ in range(num_repeat - 1):
        block(True)
    for i in range(N):
        c.noise("X_ERROR" if z_basis else "Z_ERROR", p, DQ + i)
        c.gate("M" if z_basis else "MX", DQ + i)
    pcm = cd["S_Z"] if z_basis else cd["S_X"]
    logical = cd["L_Z"] if z_basis else cd["L_X"]
    for ri, row in enumerate(pcm):
        rec = [-N + int(j) for j in np.nonzero(row)[0]]
        rec += [-(3 if z_basis else 2) * N + int(j) for j in np.nonzero(agg[ri])[0]]
        c.detector(rec)
    for i, row in enumerate(logical):
        c.observable(i, [-N + int(j) for j in np.nonzero(row)[0]])
    return c


def _backward_pass(circ, record=None):
    """Backward Pauli-sensitivity propagation over `circ` -> {symptom: merged probability} (mechanisms with an empty symptom
    or p <= 0 are dropped; identical symptoms merge with p <- p1 (1-p2) + p2 (1-p1) in the order the pass meets them).
    record: optional list; one entry (op index, target position, kind, [symptom per mechanism], [probability per mechanism])
    is appended per noise location, in the pass's (backward) order, with the mechanisms in the order they are merged."""
    ND = circ.num_detectors
    # measurement index -> symptom mask
    meas_mask = {}
    for name, targets, arg in circ.ops:
        if name == "DETECTOR":
            for a in targets:
                meas_mask[a] = meas_mask.get(a, 0) ^ (1 << arg)
        elif name == "OBSERVABLE_INCLUDE":
            for a in targets:
                meas_mask[a] = meas_mask.get(a, 0) ^ (1 << (ND + arg))
    xs, zs = {}, {}         # per qubit: symptoms flipped by an X / Z fault at the current point
    merged = {}

    def add(sym, p):
        if sym == 0 or p <= 0.0:
            return
        q = merged.get(sym)
        merged[sym] = p if q is None else q * (1.0 - p) + p * (1.0 - q)

    def location(oi, pos, name, syms, p):
        for s in syms:
            add(s, p)
        if record is not None:
            record.append((oi, pos, name, syms, p))

    mi = circ.num_measurements
    for oi in range(len(circ.ops) - 1, -1, -1):
        name, t, arg = circ.ops[oi]
        if name == "CNOT":
            c_, t_ = t
            xs[c_] = xs.get(c_, 0) ^ xs.get(t_, 0)      # X on control spreads to target
            zs[t_] = zs.get(t_, 0) ^ zs.get(c_, 0)      # Z on target spreads to control
        elif name == "H":
            q = t[0]
            xs[q], zs[q] = zs.get(q, 0), xs.get(q, 0)
        elif name in ("M", "MR"):
            for q in reversed(t):
                mi -= 1
                mk = meas_mask.get(mi, 0)
                if name == "MR":
                    xs[q] = mk; zs[q] = 0
                else:
                    xs[q] = xs.get(q, 0) ^ mk
        elif name in ("MX", "MRX"):
            for q in reversed(t):
                mi -= 1
                mk = meas_mask.get(mi, 0)
                if name == "MRX":
                    zs[q] = mk; xs[q] = 0
                else:
                    zs[q] = zs.get(q, 0) ^ mk
        elif name in ("R", "RX"):
            for q in t:
                xs[q] = 0; zs[q] = 0
        elif name == "X_ERROR":
            for k, q in enumerate(t):
                location(oi, k, name, (xs.get(q, 0),), arg)
        elif name == "Z_ERROR":
            for k, q in enumerate(t):
                location(oi, k, name, (zs.get(q, 0),), arg)
        elif name == "DEPOLARIZE1":
            pc = 0.5 - 0.5 * math.sqrt(1.0 - 4.0 * arg / 3.0)
            for k, q in enumerate(t):
                x, z = xs.get(q, 0), zs.get(q, 0)
                location(oi, k, name, (x, z, x ^ z), pc)
        elif name == "DEPOLARIZE2":
            pc = 0.5 - 0.5 * (1.0 - 16.0 * arg / 15.0) ** 0.125
            a, b = t
            pa = (0, xs.get(a, 0), zs.get(a, 0), xs.get(a, 0) ^ zs.get(a, 0))
            pb = (0, xs.get(b, 0), zs.get(b, 0), xs.get(b, 0) ^ zs.get(b, 0))
            location(oi, 0, name, tuple(pa[i] ^ pb[j] for i in range(4) for j in range(4) if i or j), pc)
        elif name in ("DETECTOR", "OBSERVABLE_INCLUDE", "TICK"):
            pass
        else:
            raise NotImplementedError(name)
    assert mi == 0
    return merged


def _sorted_dem(merged, circ):
    def targets(sym):
        return tuple(i for i in range(sym.bit_length()) if (sym >> i) & 1)

    items = sorted(merged.items(), key=lambda kv: targets(kv[0]))
    return [k for k, _ in items], [v for _, v in items], circ.num_detectors, circ.num_observables


def detector_error_model(circ):
    """-> (symptoms list[int], probs list[float], num_detectors, num_observables).

    One entry per distinct non-empty symptom set; identical symptoms are merged with
    p <- p1 (1-p2) + p2 (1-p1).  Entries are sorted lexicographically by their (detectors...,
    observables...) target lists, detectors before observables.
    """
    return _sorted_dem(_backward_pass(circ), circ)


NOISE_KINDS = ("X_ERROR", "Z_ERROR", "DEPOLARIZE1", "DEPOLARIZE2")


@dataclass
class NoiseLocations:
    """The noise locations of a circuit and their independent mechanisms (see `noise_locations`)."""
    kind: np.ndarray          # [L] str: the instruction of location l (one of NOISE_KINDS)
    op: np.ndarray            # [L] int32: index of that instruction in circ.ops
    mech_ptr: np.ndarray      # [L + 1] int32: the mechanisms of location l are mech_ptr[l] .. mech_ptr[l + 1] - 1
    mech_col: np.ndarray      # [M] int32: DEM column of the mechanism's symptom, -1 if it has none
    mech_prob: np.ndarray     # [M] float64: the mechanism's probability
    mech_unmapped: np.ndarray  # [M] bool: non-empty symptom that is no DEM column (only when every mechanism with it has p = 0)

    @property
    def num_locations(self):
        return len(self.kind)


def _noise_locations(circ):
    """-> (NoiseLocations, detector_error_model(circ)) from one backward pass."""
    rec = []
    dem = _sorted_dem(_backward_pass(circ, rec), circ)
    rec.sort(key=lambda r: (r[0], r[1]))                 # program order
    col = {s: j for j, s in enumerate(dem[0])}
    counts = [len(r[3]) for r in rec]
    mech_ptr = np.zeros(len(rec) + 1, dtype=np.int32)
    mech_ptr[1:] = np.cumsum(counts)
    syms = [s for r in rec for s in r[3]]
    locs = NoiseLocations(kind=np.array([r[2] for r in rec], dtype=object),
                          op=np.array([r[0] for r in rec], dtype=np.int32),
                          mech_ptr=mech_ptr,
                          mech_col=np.array([col.get(s, -1) for s in syms], dtype=np.int32),
                          mech_prob=np.repeat(np.array([r[4] for r in rec], dtype=np.float64), counts),
                          mech_unmapped=np.array([s != 0 and s not in col for s in syms], dtype=bool))
    return locs, dem


def noise_locations(circ):
    """The noise locations of `circ` in program order: one per DEPOLARIZE2 instruction, one per target of an X_ERROR,
    Z_ERROR or DEPOLARIZE1 instruction.  Each carries the independent mechanisms `detector_error_model` adds for it, in
    the same order: X_ERROR / Z_ERROR one (probability p), DEPOLARIZE1 three (x, z, x^z; pc = 1/2 - 1/2 sqrt(1 - 4p/3)),
    DEPOLARIZE2 fifteen ((i, j) != (0, 0) of the products of (I, X, Z, Y) on the two targets in row-major order;
    pc = 1/2 - 1/2 (1 - 16p/15)^(1/8)).  mech_col refers to the column order of
    dem_to_check_matrices(detector_error_model(circ)): XOR-combining mech_prob per column, locations last to first
    (the targets of one instruction first to last), reproduces its priors bit for bit.  -> NoiseLocations."""
    return _noise_locations(circ)[0]


def dem_to_check_matrices(dem):
    """(chk csc [num_det, num_faults], obs csc [num_obs, num_faults], priors) as build_circuit.py:251-299."""
    syms, probs, ND, NO = dem
    rows, cols, orow, ocol = [], [], [], []
    for j, s in enumerate(syms):
        for i in range(s.bit_length()):
            if (s >> i) & 1:
                if i < ND:
                    rows.append(i); cols.append(j)
                else:
                    orow.append(i - ND); ocol.append(j)
    nf = len(syms)
    chk = csc_matrix((np.ones(len(rows), dtype=np.uint8), (rows, cols)), shape=(ND, nf))
    obs = csc_matrix((np.ones(len(orow), dtype=np.uint8), (orow, ocol)), shape=(NO, nf))
    return chk, obs, np.array(probs, dtype=np.float64)


_READOUT_BASIS = {"X_ERROR": ("M", "MR"), "Z_ERROR": ("MX", "MRX")}


def _readout_flips(circ):
    """-> (readout location indices, {op index: number of its targets that are readout flips}) in one forward scan.  The
    location index of an X_ERROR / Z_ERROR target is its position in noise_locations' program order."""
    pending = {}                # qubit -> (location, flip kind, op index) of the last X_ERROR / Z_ERROR on it
    out, per_op, loc = [], {}, 0
    for oi, (name, t, _) in enumerate(circ.ops):
        if name in ("DETECTOR", "OBSERVABLE_INCLUDE", "TICK"):
            continue
        for q in t:
            prev = pending.pop(q, None)
            if prev is not None and name in _READOUT_BASIS[prev[1]]:
                out.append(prev[0])
                per_op[prev[2]] = per_op.get(prev[2], 0) + 1
        if name in _READOUT_BASIS:
            for k, q in enumerate(t):
                pending[q] = (loc + k, name, oi)
        if name in ("X_ERROR", "Z_ERROR", "DEPOLARIZE1"):
            loc += len(t)
        elif name == "DEPOLARIZE2":
            loc += 1
    return np.array(sorted(out), dtype=np.int32), per_op


def readout_locations(circ):
    """The measurement flips of `circ`: every X_ERROR (Z_ERROR) target whose next instruction on that qubit is M or MR (MX
    or MRX), DETECTOR, OBSERVABLE_INCLUDE and TICK skipped.  -> int32 array of indices into noise_locations(circ),
    increasing.  Each is a single-mechanism location, so soft readout information about it changes one DEM column."""
    return _readout_flips(circ)[0]


def with_readout_error(circ, p_meas):
    """A copy of `circ` with the probability of every measurement flip (readout_locations) set to p_meas in [0, 1/2], so that
    readout noise can be set apart from gate noise.  ValueError for an X_ERROR / Z_ERROR instruction whose targets are only
    partly measurement flips (none of the package's circuits has one)."""
    p_meas = float(p_meas)
    if not 0.0 <= p_meas <= 0.5:
        raise ValueError(f"p_meas must lie in [0, 1/2], got {p_meas}")
    _, per_op = _readout_flips(circ)
    out = Ops()
    out.num_measurements, out.num_detectors, out.num_observables = circ.num_measurements, circ.num_detectors, circ.num_observables
    out.ops = list(circ.ops)
    for oi, n in per_op.items():
        name, t, _ = circ.ops[oi]
        if n != len(t):
            raise ValueError(f"instruction {oi} ({name}) has {n} measurement-flip targets out of {len(t)}; split it first")
        out.ops[oi] = (name, t, p_meas)
    return out


@dataclass
class ReadoutModel:
    """Soft measurement readout shared by all readout locations: a location draws reliability class k with probability
    weights[k] and then flips with probability flip_prob[k].  1 <= K <= 256 classes; weights >= 0 summing to 1 (within
    1e-9), flip_prob in [0, 1/2].  Its marginal flip probability sum_k weights[k] flip_prob[k] must equal the readout
    locations' probability in the circuit, so that the DEM and its priors do not change."""
    weights: np.ndarray
    flip_prob: np.ndarray

    def __post_init__(self):
        self.weights = np.array(self.weights, dtype=np.float64).reshape(-1)
        self.flip_prob = np.array(self.flip_prob, dtype=np.float64).reshape(-1)
        K = len(self.weights)
        if not 1 <= K <= 256 or self.flip_prob.shape != (K,):
            raise ValueError(f"need 1 to 256 classes with one weight and one flip probability each, got {K} and {len(self.flip_prob)}")
        if not (self.weights >= 0.0).all() or not abs(math.fsum(self.weights) - 1.0) <= 1e-9:
            raise ValueError("class weights must be non-negative and sum to 1")
        if not ((self.flip_prob >= 0.0) & (self.flip_prob <= 0.5)).all():
            raise ValueError("flip probabilities must lie in [0, 1/2]")

    @property
    def num_classes(self):
        return len(self.weights)

    @property
    def marginal(self):
        """sum_k weights[k] flip_prob[k]: the flip probability of a readout location."""
        return float(np.dot(self.weights, self.flip_prob))


def gaussian_readout(p_meas, num_classes):
    """ReadoutModel of a symmetric Gaussian readout: the signal is x = +-1 + sigma z with Phi(-1/sigma) = p_meas in (0, 1/2),
    binned into num_classes equiprobable bins of |x| (class 0 the least reliable), q[k] = P(wrong sign | |x| in bin k).
    sum w q = p_meas up to rounding; num_classes = 1 gives q = [p_meas]."""
    from scipy.optimize import brentq
    from scipy.stats import norm
    p_meas, K = float(p_meas), int(num_classes)
    if not 0.0 < p_meas < 0.5:
        raise ValueError(f"p_meas must lie in (0, 1/2), got {p_meas}")
    if not 1 <= K <= 256:
        raise ValueError(f"num_classes must lie in 1 .. 256, got {num_classes}")
    if K == 1:
        return ReadoutModel([1.0], [p_meas])
    sigma = -1.0 / norm.ppf(p_meas)

    def mass(a):                            # P(|x| <= a)
        return norm.cdf((a - 1.0) / sigma) - norm.cdf((-a - 1.0) / sigma)

    hi = 1.0 + 40.0 * sigma
    edges = [0.0] + [brentq(lambda a, k=k: mass(a) - k / K, 0.0, hi, xtol=1e-15, rtol=4 * np.finfo(float).eps) for k in range(1, K)]
    wrong_below = np.array([norm.cdf((-a - 1.0) / sigma) for a in edges] + [0.0])   # P(x < -a) for x = +1 + sigma z
    w = np.full(K, 1.0 / K)
    q = np.minimum((wrong_below[:-1] - wrong_below[1:]) * K, 0.5)
    return ReadoutModel(w, q)
