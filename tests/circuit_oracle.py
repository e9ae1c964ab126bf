"""numpy restatement of the device circuit-level sampler (slidingwindowdecoder_b200/csrc/swd_window.cuh:
window_sample_circuit_kernel), bit-identical to swd_window_sample_circuit.  Test infrastructure, built on the Philox4x32-10 and
threshold rule of oracle/philox.py that the DEM sampler is tested with."""
import numpy as np
from scipy.sparse import csc_matrix

from oracle.philox import MASK, philox4x32_10, thresholds


def sample_circuit(chk, obs, locs, erasure_rate, col_llr, shots, seed=0, shot_offset=0, chunk=256):
    """Location l (locs = dem.noise_locations) with n_l mechanisms uses draws t = 0 .. n_l: word t & 3 of the Philox call
    with counter (l, 2 + (t >> 2), shot).  Draw 0 erases l iff it is below thr(erasure_rate[l]); draw 1 + k fires mechanism
    k iff it is below 2^31 (erased) or thr(mech_prob[k]).  -> det [shots, num_det], obs [shots, num_obs], err [shots,
    num_col], erased [shots, L] (uint8) and the LLR rows [shots, num_col] (col_llr with 0.0 at the columns of erased
    locations)."""
    L, num_col = locs.num_locations, chk.shape[1]
    ptr = np.asarray(locs.mech_ptr, dtype=np.int64)
    cnt = np.diff(ptr)
    M = int(ptr[-1])
    mloc = np.repeat(np.arange(L), cnt)                       # location of each mechanism
    mt = np.arange(M) - ptr[mloc] + 1                         # its draw index t
    col = np.asarray(locs.mech_col, dtype=np.int64)
    has = col >= 0
    mech_to_col = csc_matrix((np.ones(int(has.sum()), dtype=np.int64), (np.flatnonzero(has), col[has])), shape=(M, num_col))
    loc_to_col = csc_matrix((np.ones(int(has.sum()), dtype=np.int64), (mloc[has], col[has])), shape=(L, num_col))
    t_mech = thresholds(locs.mech_prob)
    t_erase = thresholds(np.broadcast_to(np.asarray(erasure_rate, dtype=np.float64), (L,)))
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    outs = []
    for s0 in range(0, shots, chunk):
        n = min(chunk, shots - s0)
        shot = (np.arange(n, dtype=np.uint64) + np.uint64(shot_offset + s0))[:, None]
        draws = np.zeros((n, L, 16), dtype=np.uint32)
        for call in range(4):
            need = np.flatnonzero(cnt >= 4 * call)
            r = philox4x32_10(need.astype(np.uint64)[None, :], np.uint64(2 + call), shot & MASK, shot >> np.uint64(32), k0, k1)
            draws[:, need, 4 * call:4 * call + 4] = np.stack(r, axis=2)
        erased = draws[:, :, 0] < t_erase[None, :]
        w = draws[:, mloc, mt]
        fired = np.where(erased[:, mloc], w < np.uint32(0x80000000), w < t_mech[None, :])
        err = (np.asarray((mech_to_col.T @ fired.T.astype(np.int64))).T % 2).astype(np.uint8)
        e = err.astype(np.int64)
        det = (np.asarray(chk @ e.T).T % 2).astype(np.uint8)
        ob = (np.asarray(obs @ e.T).T % 2).astype(np.uint8)
        lost = np.asarray(loc_to_col.T @ erased.T.astype(np.int64)).T > 0
        llr = np.where(lost, 0.0, np.asarray(col_llr, dtype=np.float64)[None, :])
        outs.append((det, ob, err, erased.astype(np.uint8), llr))
    return tuple(np.concatenate([o[i] for o in outs], axis=0) for i in range(5))
