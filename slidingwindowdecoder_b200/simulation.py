"""Code-capacity driver: the GDG part of the reference's src/simulation.py:10-99 with batched decoding.

`data_qubit_noise_decoding(code, p, num_shots)` samples iid X errors, decodes all syndromes of hx with
`bpgdg_decoder` (same kwargs as simulation.py:66-82) in ONE batched call and counts logical errors against
`hz_perp`.  The `ldpc.BpOsdDecoder` legs of the reference function are third-party and not reproduced.

`depolarizing_noise_decoding(code, p, num_shots, erasure_rate)` is the `bp4_osd` counterpart under depolarizing noise with
heralded erasures: `CodeCapacitySampler` draws the errors, erasures and per-shot LLR planes on the device, and the commit /
count kernels of the window driver score the corrections, so no shot data crosses PCIe.

`CircuitNoiseSampler(circ, erasure_rate)` is the circuit-level counterpart: it samples the noise locations of an `Ops` circuit
(dem.noise_locations), with heralded erasures, on the device and returns shots in the DEM's column order together with the
per-shot LLR rows that `SlidingWindowDecoder.decode_device(channel_llr=...)` takes.  With `readout=` a dem.ReadoutModel
it also draws a reliability class per measurement flip (soft readout) and writes the matching rows.
"""
import ctypes as C
import time

import numpy as np

from . import _lib
from .decoders import bpgdg_decoder


def data_qubit_noise_decoding(code, p, num_shots=1000, max_step=40, max_tree_step=30, max_iter_per_step=6, seed=None,
                              extra_decoders=(), device=0, verbose=True):
    rng = np.random.default_rng(seed)
    err = (rng.random((num_shots, code.N)) < p).astype(np.uint8)             # simulation.py:15
    syndrome = (err.astype(np.int64) @ code.hx.T % 2).astype(np.uint8)       # simulation.py:16
    priors = np.ones(code.N) * p
    results = {}
    decoders = list(extra_decoders)
    decoders.append(("GDG", bpgdg_decoder(                                   # simulation.py:66-82
        code.hx, channel_probs=priors, max_iter_per_step=max_iter_per_step, gdg_factor=0.625, max_step=max_step,
        max_tree_depth=4, max_side_depth=20, max_tree_branch_step=max_tree_step, max_side_branch_step=max_step - 20,
        multi_thread=True, low_error_mode=True, max_iter=24, ms_scaling_factor=0.625, new_n=code.N, device=device)))
    for name, dec in decoders:
        t0 = time.perf_counter()
        e_hat, conv = dec.decode_batch(syndrome)
        dt = time.perf_counter() - t0
        e_diff = (e_hat.astype(np.int64) + err) % 2
        logical = ((e_diff @ code.hz_perp.T) % 2).any(axis=1)                 # simulation.py:90-91
        results[name] = dict(num_flagged=int((1 - conv.astype(np.int64)).sum()), num_logical=int(logical.sum()),
                             ler=float(logical.mean()), elapsed=dt)
        if verbose:
            print(f"{name}: num flagged error {results[name]['num_flagged']}")
            print(f"{name}: num logical error {results[name]['num_logical']}/{num_shots}, LER {results[name]['ler']}")
            print("Elapsed time:", dt)
    return results


def _sample_args(B, seed, shot_offset):
    """The checked (B, seed, shot_offset) of a sampler call, as ints."""
    B, seed, shot_offset = int(B), int(seed), int(shot_offset)
    if B < 0 or shot_offset < 0 or not 0 <= seed < 1 << 64:
        raise ValueError(f"need B >= 0, shot_offset >= 0 and 0 <= seed < 2**64 (got {B}, {shot_offset}, {seed})")
    return B, seed, shot_offset


class CodeCapacitySampler:
    """Depolarizing noise with heralded erasures on the data qubits of a CSS code, sampled on the device
    (`swd_window_sample_pauli`).  The experiment is a window plan over 2n columns: column v is the X part of qubit v, column
    n + v its Z part (the [B, 2, n] layout of `bp4_osd`'s `dec`); chk = [[0, Hx], [Hz, 0]] so det = [synd_x | synd_z]
    (synd_x = Hx . e_z, synd_z = Hz . e_x); obs = [[lz, 0], [0, lx]].  `px / py / pz` are per-qubit probabilities; an
    erased qubit carries a uniformly random Pauli.  `channel_llr` is the [5, n] static LLR rows (normally
    `bp4_osd(...).channel_llr`): `sample(..., return_llr=True)` returns them per shot with 0.0 at erased qubits.  Shot s of
    a call depends only on (seed, shot_offset + s)."""

    def __init__(self, Hx, Hz, lx, lz, px, py, pz, erasure_rate=0.0, channel_llr=None, device=0):
        from scipy.sparse import bmat, csc_matrix
        Hx, Hz, lx, lz = (csc_matrix(np.asarray(M.todense() if hasattr(M, "todense") else M) % 2) for M in (Hx, Hz, lx, lz))
        n = Hx.shape[1]
        if Hz.shape[1] != n or lx.shape[1] != n or lz.shape[1] != n:
            raise ValueError(f"Hx, Hz, lx and lz must have the same number of columns (Hx has {n})")
        px, py, pz = (np.ascontiguousarray(a, dtype=np.float64) for a in (px, py, pz))
        if px.shape != (n,) or py.shape != (n,) or pz.shape != (n,):
            raise ValueError(f"px, py and pz must have shape ({n},)")
        if not ((px >= 0).all() and (py >= 0).all() and (pz >= 0).all()):
            raise ValueError("px, py and pz must be non-negative and not NaN")
        if ((px + py) + pz > 1.0).any():
            raise ValueError("px + py + pz exceeds 1 on some qubit")
        erasure_rate = float(erasure_rate)
        if not 0.0 <= erasure_rate <= 1.0:
            raise ValueError(f"erasure_rate must lie in [0, 1], got {erasure_rate}")
        llr5 = None
        if channel_llr is not None:
            llr5 = np.ascontiguousarray(channel_llr, dtype=np.float64)
            if llr5.shape != (5, n):
                raise ValueError(f"channel_llr must have shape (5, {n}), got {llr5.shape}")
        import torch
        self.torch = torch
        self.n, self.mx, self.mz = n, Hx.shape[0], Hz.shape[0]
        self.device = int(device)
        chk = bmat([[None, Hx], [Hz, None]], format="csc", dtype=np.uint8)
        obs = bmat([[lz, None], [None, lx]], format="csc", dtype=np.uint8)
        chk.sort_indices(); obs.sort_indices()
        self.num_det, self.num_obs = chk.shape[0], obs.shape[0]
        self.chk, self.obs = chk, obs
        self.lib = _lib.load()
        dp = C.POINTER(C.c_double)
        self._win = _lib.Window(self.device, chk, obs)
        self._cp = self._win._cp               # int32 CSC arrays of chk and obs: (chk indptr, chk indices, obs indptr, obs indices)
        self.has_llr = llr5 is not None
        _lib.check(self.lib.swd_window_set_pauli_priors(self._win, n, px.ctypes.data_as(dp), py.ctypes.data_as(dp), pz.ctypes.data_as(dp),
                                                        erasure_rate, llr5.ctypes.data_as(dp) if self.has_llr else None),
                   "swd_window_set_pauli_priors")
        self.erasure_rate = erasure_rate

    def sample(self, B, seed=0, shot_offset=0, return_errors=False, return_erasures=False, return_llr=False):
        """-> dict of torch CUDA tensors on the current stream: synd_x [B, mx], synd_z [B, mz] (contiguous copies of det's two
        halves), det [B, mx + mz], obs [B, num_obs] (uint8), and on request err [B, 2, n], erased [B, n] (uint8),
        channel_llr [5, B, n] (float64)."""
        B, seed, shot_offset = _sample_args(B, seed, shot_offset)
        if return_llr and not self.has_llr:
            raise ValueError("return_llr needs the static rows: pass channel_llr to CodeCapacitySampler")
        torch, n = self.torch, self.n
        dev = torch.device("cuda", self.device)
        u8 = dict(dtype=torch.uint8, device=dev)
        out = dict(det=torch.empty((B, self.num_det), **u8), obs=torch.empty((B, self.num_obs), **u8))
        if return_errors:
            out["err"] = torch.empty((B, 2, n), **u8)
        if return_erasures:
            out["erased"] = torch.empty((B, n), **u8)
        if return_llr:
            out["channel_llr"] = torch.empty((5, B, n), dtype=torch.float64, device=dev)
        if B:
            ptr = lambda k: out[k].data_ptr() if k in out and out[k].numel() else None    # noqa: E731
            _lib.check(self.lib.swd_window_sample_pauli(self._win, seed, shot_offset, B, ptr("det"), ptr("obs"), ptr("err"),
                                                        ptr("erased"), ptr("channel_llr"), _lib.current_stream(dev)),
                       "swd_window_sample_pauli")
        out["synd_x"] = out["det"][:, :self.mx].contiguous()
        out["synd_z"] = out["det"][:, self.mx:].contiguous()
        return out

    def count_failures(self, dec, det, obs):
        """Commit the corrections dec [B, 2, n] into det / obs (in place) and count over the batch -> [2] int64 device
        tensor (flagged: the syndrome is not reproduced; failed: flagged, or the residual flips a logical)."""
        torch = self.torch
        B = det.shape[0]
        if tuple(dec.shape) != (B, 2, self.n) or tuple(det.shape) != (B, self.num_det) or tuple(obs.shape) != (B, self.num_obs):
            raise ValueError(f"expected dec [B, 2, {self.n}], det [B, {self.num_det}], obs [B, {self.num_obs}]")
        if not (det.is_contiguous() and obs.is_contiguous()) or det.dtype != torch.uint8 or obs.dtype != torch.uint8:
            raise ValueError("det and obs must be contiguous uint8 tensors (they are updated in place)")
        counts = torch.zeros(2, dtype=torch.int64, device=det.device)
        if B == 0:
            return counts
        dec = dec.to(torch.uint8).contiguous()
        stream = _lib.current_stream(self.device)
        obs_ptr = obs.data_ptr() if self.num_obs else None
        _lib.check(self.lib.swd_window_commit(self._win, dec.data_ptr(), B, 2 * self.n, 0, 2 * self.n, det.data_ptr(), obs_ptr,
                                              stream), "swd_window_commit")
        _lib.check(self.lib.swd_window_count_failures(self._win, det.data_ptr(), obs_ptr, B, counts.data_ptr(), stream),
                   "swd_window_count_failures")
        return counts


def depolarizing_noise_decoding(code, p, num_shots=1000, erasure_rate=0.0, batch=65536, seed=0, shot_offset=0, device=0,
                                verbose=True, **bp4_kwargs):
    """Logical error rate of `bp4_osd` on `code` (hx, hz, lx, lz) under depolarizing noise px = py = pz = p/3, with
    heralded erasures at `erasure_rate`, sampled, decoded and counted on the device.  Shots
    [shot_offset, shot_offset + num_shots) of the seed's stream are decoded in batches of `batch`: the counts do not depend
    on `batch`, and `distributed.shard_range` splits a job.  -> dict with the leg `static` (decoded with the static priors)
    and, when erasure_rate > 0, `erasure_aware` (decoded with the sampled [5, B, n] planes, 0.0 at erased qubits); each
    leg holds num_flagged, num_logical, ler and num_bp_unconverged.  Also erased_fraction and elapsed (seconds)."""
    import torch
    from .decoders import bp4_osd
    p, num_shots, batch = float(p), int(num_shots), int(batch)
    if not 0.0 < p < 1.0:
        raise ValueError(f"p must lie in (0, 1), got {p}")
    if num_shots < 0 or batch <= 0 or int(shot_offset) < 0:
        raise ValueError("need num_shots >= 0, batch > 0 and shot_offset >= 0")
    n = code.hx.shape[1]
    pr = np.full(n, p / 3)
    dec = bp4_osd(code.hx, code.hz, channel_probs_x=pr, channel_probs_y=pr, channel_probs_z=pr, device=device, **bp4_kwargs)
    erase = float(erasure_rate) > 0
    sampler = CodeCapacitySampler(code.hx, code.hz, code.lx, code.lz, pr, pr, pr, erasure_rate=erasure_rate,
                                  channel_llr=dec.channel_llr if erase else None, device=device)
    legs = ("static", "erasure_aware") if erase else ("static",)
    dev = torch.device("cuda", int(device))
    acc = torch.zeros((len(legs), 3), dtype=torch.int64, device=dev)      # flagged, failed, BP not converged
    erased = torch.zeros((), dtype=torch.int64, device=dev)
    t0 = time.perf_counter()
    for start in range(0, num_shots, batch):
        B = min(batch, num_shots - start)
        s = sampler.sample(B, seed=seed, shot_offset=int(shot_offset) + start, return_erasures=erase, return_llr=erase)
        for i, leg in enumerate(legs):
            L = s["channel_llr"] if leg == "erasure_aware" else None
            out = dec.decode_batch(s["synd_x"], s["synd_z"], channel_llr=L)
            last = i == len(legs) - 1
            det, obs = (s["det"], s["obs"]) if last else (s["det"].clone(), s["obs"].clone())
            acc[i, :2] += sampler.count_failures(out["dec"], det, obs)
            acc[i, 2] += (out["converge"] == 0).sum()
        if erase:
            erased += s["erased"].sum()
    counts = acc.cpu().tolist()
    n_erased = int(erased.item())
    elapsed = time.perf_counter() - t0
    results = dict(erased_fraction=n_erased / max(1, num_shots * n), elapsed=elapsed)
    for leg, (flagged, failed, unconv) in zip(legs, counts):
        results[leg] = dict(num_flagged=int(flagged), num_logical=int(failed), ler=failed / max(1, num_shots),
                            num_bp_unconverged=int(unconv))
        if verbose:
            print(f"{leg}: num flagged error {flagged}")
            print(f"{leg}: num logical error {failed}/{num_shots}, LER {results[leg]['ler']}")
    if verbose:
        print("Elapsed time:", elapsed)
    return results


class CircuitNoiseSampler:
    """Circuit-level noise with heralded erasures, sampled per noise location on the device (`swd_window_sample_circuit`).

    The locations are those of `dem.noise_locations(circ)`: one per DEPOLARIZE2 instruction, one per target of X_ERROR,
    Z_ERROR or DEPOLARIZE1.  An erased location carries a uniformly random Pauli (each of its independent mechanisms fires
    with probability 1/2); any other location keeps its Pauli channel, so at erasure rate 0 the shots have the law of the
    DEM sampler.  `erasure_rate`: a scalar applies to every DEPOLARIZE2 location (gate erasure conversion), an array gives
    one rate per location.  `.chk, .obs, .priors` are dem_to_check_matrices(detector_error_model(circ)) and
    `.channel_llr` [num_col] their static LLRs log((1-p)/p); a shot's LLR row is 0.0 at the columns of its erased locations.
    Shot s of a call depends only on (seed, shot_offset + s).

    `readout`: None, or a dem.ReadoutModel for soft measurement readout (`swd_window_sample_circuit_readout`).  Each
    measurement flip (`.readout_locations` = dem.readout_locations(circ)) draws a reliability class k with probability
    weights[k] and flips with probability flip_prob[k]; every flip's probability in the circuit must equal the model's
    marginal (within 1e-9 relative), so the DEM is unchanged.  `.class_llr` [num_readout, K] is the LLR of readout r's DEM
    column when r is in class k (the column's prior XOR-folded as in noise_locations with r's probability replaced by
    flip_prob[k]; 0.0 for a readout without a column), and a shot's LLR row takes class_llr[r, class_r] at that column,
    0.0 at the columns of erased locations overriding it."""

    def __init__(self, circ, erasure_rate=0.0, readout=None, device=0):
        from .decoders import _libm_llr
        from .dem import ReadoutModel, _noise_locations, dem_to_check_matrices, readout_locations
        if readout is not None and not isinstance(readout, ReadoutModel):
            raise ValueError(f"readout must be None or a dem.ReadoutModel, got {type(readout).__name__}")
        locs, dem = _noise_locations(circ)
        L = locs.num_locations
        if L == 0:
            raise ValueError("the circuit has no noise locations")
        if np.ndim(erasure_rate) == 0:
            e = float(erasure_rate)
            if not 0.0 <= e <= 1.0:
                raise ValueError(f"erasure_rate must lie in [0, 1], got {e}")
            rate = np.where(locs.kind == "DEPOLARIZE2", e, 0.0)
        else:
            rate = np.ascontiguousarray(erasure_rate, dtype=np.float64)
            if rate.shape != (L,):
                raise ValueError(f"erasure_rate must be a scalar or have shape ({L},) (one rate per noise location), got {rate.shape}")
            if not ((rate >= 0.0) & (rate <= 1.0)).all():
                raise ValueError("erasure_rate must lie in [0, 1] (and not be NaN) at every location")
        lost = np.add.reduceat(locs.mech_unmapped.astype(np.int64), locs.mech_ptr[:-1]) > 0
        if (lost & (rate > 0)).any():
            raise ValueError(f"location {int(np.flatnonzero(lost & (rate > 0))[0])} has a non-zero erasure rate but a mechanism "
                             "whose symptom is no DEM column (its probability is 0): its erasure cannot be represented")
        chk, obs, priors = dem_to_check_matrices(dem)
        chk.sort_indices(); obs.sort_indices()
        self.readout = readout
        if readout is not None:
            ro = readout_locations(circ)
            if len(ro) == 0:
                raise ValueError("the circuit has no readout locations (X_ERROR / Z_ERROR right before a measurement in its basis)")
            p_ro, m = locs.mech_prob[locs.mech_ptr[ro]], readout.marginal
            bad = np.flatnonzero(np.abs(p_ro - m) > 1e-9 * np.maximum(np.abs(p_ro), abs(m)))
            if len(bad):
                raise ValueError(f"readout location {int(ro[bad[0]])} has probability {p_ro[bad[0]]!r}, but the readout model's "
                                 f"marginal sum(w q) is {m!r} (dem.with_readout_error sets it)")
            cols = locs.mech_col[locs.mech_ptr[ro]]
            u, n = np.unique(cols[cols >= 0], return_counts=True)
            if (n > 1).any():
                raise ValueError(f"two readout locations share DEM column {int(u[n > 1][0])}: their soft information cannot be "
                                 "given per column")
            self.readout_locations = ro
            self.class_llr = _readout_class_llr(locs, ro, readout.flip_prob, len(priors))
        import torch
        self.torch = torch
        self.device = int(device)
        self.chk, self.obs, self.priors = chk, obs, priors
        self.num_det, self.num_col = chk.shape
        self.num_obs = obs.shape[0]
        self.locations, self.num_locations = locs, L
        self.erasure_rate = rate
        self.channel_llr = _libm_llr(priors, self.num_col)
        self.lib = _lib.load()
        i32p, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
        self._win = _lib.Window(self.device, chk, obs)
        self._cp = self._win._cp               # int32 CSC arrays of chk and obs: (chk indptr, chk indices, obs indptr, obs indices)
        _lib.check(self.lib.swd_window_set_circuit_noise(self._win, L, locs.mech_ptr.ctypes.data_as(i32p), locs.mech_col.ctypes.data_as(i32p),
                                                         locs.mech_prob.ctypes.data_as(dp), rate.ctypes.data_as(dp),
                                                         self.channel_llr.ctypes.data_as(dp)),
                   "swd_window_set_circuit_noise")
        if readout is not None:
            _lib.check(self.lib.swd_window_set_circuit_readout(self._win, len(self.readout_locations),
                                                               self.readout_locations.ctypes.data_as(i32p), readout.num_classes,
                                                               readout.weights.ctypes.data_as(dp), readout.flip_prob.ctypes.data_as(dp),
                                                               self.class_llr.ctypes.data_as(dp)),
                       "swd_window_set_circuit_readout")

    def sample(self, B, seed=0, shot_offset=0, return_errors=False, return_erasures=False, return_llr=False, return_readout=False):
        """-> (det [B, num_det], obs [B, num_obs][, err [B, num_col]][, erased [B, num_locations]][, readout [B, num_readout]]
        uint8 [, channel_llr [B, num_col] float64]) as torch CUDA tensors written on the current stream.  Columns are in the
        DEM's order (what build_windows and decode_device(channel_llr=...) take); err is the parity of the fired mechanisms
        per column, so det = chk . err and obs = obs . err; readout holds the classes in readout_locations order (needs a
        readout model)."""
        B, seed, shot_offset = _sample_args(B, seed, shot_offset)
        if return_readout and self.readout is None:
            raise ValueError("return_readout needs a sampler built with a readout model")
        torch = self.torch
        dev = torch.device("cuda", self.device)
        u8 = dict(dtype=torch.uint8, device=dev)
        out = dict(det=torch.empty((B, self.num_det), **u8), obs=torch.empty((B, self.num_obs), **u8))
        if return_errors:
            out["err"] = torch.empty((B, self.num_col), **u8)
        if return_erasures:
            out["erased"] = torch.empty((B, self.num_locations), **u8)
        if return_readout:
            out["readout"] = torch.empty((B, len(self.readout_locations)), **u8)
        if return_llr:
            out["channel_llr"] = torch.empty((B, self.num_col), dtype=torch.float64, device=dev)
        if B:
            ptr = lambda k: out[k].data_ptr() if k in out and out[k].numel() else None    # noqa: E731
            stream = _lib.current_stream(dev)
            if self.readout is None:
                _lib.check(self.lib.swd_window_sample_circuit(self._win, seed, shot_offset, B, ptr("det"), ptr("obs"), ptr("err"),
                                                              ptr("erased"), ptr("channel_llr"), stream),
                           "swd_window_sample_circuit")
            else:
                _lib.check(self.lib.swd_window_sample_circuit_readout(self._win, seed, shot_offset, B, ptr("det"), ptr("obs"),
                                                                      ptr("err"), ptr("erased"), ptr("readout"), ptr("channel_llr"),
                                                                      stream),
                           "swd_window_sample_circuit_readout")
        return tuple(out[k] for k in ("det", "obs", "err", "erased", "readout", "channel_llr") if k in out)


def _readout_class_llr(locs, readout, flip_prob, num_col):
    """class_llr [R, K] of CircuitNoiseSampler: for readout r with DEM column c, the mechanisms of c are XOR-folded in
    detector_error_model's order (locations last to first, the targets of one instruction first to last, mechanisms in
    order; p <= 0 skipped, p <- q (1 - p) + p (1 - q)) with r's probability replaced by flip_prob[k], and the result goes
    through log((1 - p) / p) as decoders._libm_llr.  With flip_prob = [p_r] this is the static LLR of c bit for bit."""
    from .decoders import _libm_llr
    q = np.asarray(flip_prob, dtype=np.float64)
    R, K, L = len(readout), len(q), locs.num_locations
    out = np.zeros((R, K), dtype=np.float64)
    ro_mech = locs.mech_ptr[readout]
    ro_col = locs.mech_col[ro_mech]
    want = np.zeros(num_col, dtype=bool)
    want[ro_col[ro_col >= 0]] = True
    order = np.lexsort((np.arange(L), -locs.op.astype(np.int64)))
    mechs = np.concatenate([np.arange(locs.mech_ptr[l], locs.mech_ptr[l + 1]) for l in order])
    col = locs.mech_col[mechs]
    mechs = mechs[(col >= 0) & want[np.maximum(col, 0)]]
    mechs = mechs[np.argsort(locs.mech_col[mechs], kind="stable")]          # grouped by column, fold order kept
    bounds = np.searchsorted(locs.mech_col[mechs], np.arange(num_col + 1))
    for r in range(R):
        c = int(ro_col[r])
        if c < 0:
            continue
        acc, seen = np.zeros(K), np.zeros(K, dtype=bool)
        for m in mechs[bounds[c]:bounds[c + 1]]:
            p = q if m == ro_mech[r] else np.full(K, locs.mech_prob[m])
            use = p > 0.0
            acc = np.where(use & seen, acc * (1.0 - p) + p * (1.0 - acc), np.where(use, p, acc))
            seen |= use
        # a column with no mechanism of positive probability has prior 0 (LLR +inf, as _libm_llr)
        out[r] = _libm_llr(np.where(seen, acc, 0.0), K)
    return out
