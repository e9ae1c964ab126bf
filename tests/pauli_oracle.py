"""numpy restatement of the device code-capacity sampler (slidingwindowdecoder_b200/csrc/swd_window.cuh:
window_sample_pauli_kernel), bit-identical to swd_window_sample_pauli.  Test infrastructure, built on the Philox4x32-10 and
threshold rule of oracle/philox.py that the DEM sampler is tested with."""
import numpy as np

from oracle.philox import MASK, philox4x32_10, thresholds


def sample_pauli(chk, obs, px, py, pz, erasure_rate, shots, seed=0, shot_offset=0, llr5=None):
    """Code-capacity depolarizing noise with heralded erasures, bit-identical to swd_window_sample_pauli.
    Columns v and n + v of chk / obs are the X and Z part of qubit v.  One Philox call per qubit pair k with counter
    (k, 1, shot): words 2j / 2j + 1 are the erasure and Pauli draws of qubit 2k + j.  An erased qubit (w_e < thr(rate)) takes
    the Pauli w_p >> 30 (0 I, 1 X, 2 Y, 3 Z); any other qubit X if w_p < thr(px), Y if < thr(px + py), Z if < thr(px + py + pz).
    -> (det [shots, num_det], obs [shots, num_obs], err [shots, 2n], erased [shots, n]) uint8 and L [5, shots, n] float64
    (llr5 with 0.0 at erased qubits; None without llr5)."""
    px, py, pz = (np.asarray(a, dtype=np.float64) for a in (px, py, pz))
    n = len(px)
    t_x, t_xy, t_xyz = thresholds(px), thresholds(px + py), thresholds((px + py) + pz)
    t_e = thresholds([erasure_rate])[0]
    k = np.arange((n + 1) // 2, dtype=np.uint64)[None, :]
    shot = (np.arange(shots, dtype=np.uint64) + np.uint64(shot_offset))[:, None]
    r = philox4x32_10(k, np.uint64(1), shot & MASK, shot >> np.uint64(32), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    w_e = np.stack((r[0], r[2]), axis=2).reshape(shots, -1)[:, :n]
    w_p = np.stack((r[1], r[3]), axis=2).reshape(shots, -1)[:, :n]
    erased = w_e < t_e
    pauli = np.where(w_p < t_x, 1, np.where(w_p < t_xy, 2, np.where(w_p < t_xyz, 3, 0)))
    pauli = np.where(erased, (w_p >> np.uint32(30)).astype(np.int64), pauli)
    err = np.concatenate(((pauli == 1) | (pauli == 2), (pauli == 2) | (pauli == 3)), axis=1).astype(np.uint8)
    e = err.astype(np.int64)
    det = (np.asarray(chk @ e.T).T % 2).astype(np.uint8)
    ob = (np.asarray(obs @ e.T).T % 2).astype(np.uint8)
    L = None
    if llr5 is not None:
        L = np.repeat(np.asarray(llr5, dtype=np.float64)[:, None, :], shots, axis=1)
        L[:, erased] = 0.0
    return det, ob, err, erased.astype(np.uint8), L
