"""numpy restatement of the device circuit-level sampler with soft measurement readout (slidingwindowdecoder_b200/csrc/
swd_window.cuh: window_sample_circuit_kernel<true>), bit-identical to swd_window_sample_circuit_readout.  Test
infrastructure, built on the Philox4x32-10 and threshold rule of oracle/philox.py; every location that is not a readout
location draws as tests/circuit_oracle.py::sample_circuit."""
import numpy as np
from scipy.sparse import csc_matrix

from oracle.philox import MASK, philox4x32_10, thresholds


def class_thresholds(weights):
    """thr(w_0 + .. + w_{k-1}) for k = 1 .. K-1, the sums taken left to right in double."""
    return thresholds(np.cumsum(np.asarray(weights, dtype=np.float64))[:-1])


def sample_circuit_readout(chk, obs, locs, erasure_rate, col_llr, readout_loc, weights, flip_prob, class_llr, shots, seed=0,
                           shot_offset=0, chunk=256):
    """Location l (locs = dem.noise_locations) with n_l mechanisms uses draws t = 0 .. n_l: word t & 3 of the Philox call
    with counter (l, 2 + (t >> 2), shot); draw 0 erases l iff it is below thr(erasure_rate[l]).  At a readout location r
    (readout_loc[r], one mechanism) draw 2 is the class (the number of k in 1 .. K-1 with the draw >= thr(w_0 + .. + w_{k-1}))
    and draw 1 fires the flip iff it is below 2^31 (erased) or thr(flip_prob[class]); elsewhere draw 1 + k fires mechanism k
    iff it is below 2^31 (erased) or thr(mech_prob[k]).  -> det [shots, num_det], obs [shots, num_obs], err [shots,
    num_col], erased [shots, L], classes [shots, R] (uint8) and the LLR rows [shots, num_col]: col_llr, class_llr[r, class]
    at readout r's column, 0.0 at the columns of erased locations."""
    L, num_col = locs.num_locations, chk.shape[1]
    ptr = np.asarray(locs.mech_ptr, dtype=np.int64)
    cnt = np.diff(ptr)
    M = int(ptr[-1])
    ro = np.asarray(readout_loc, dtype=np.int64)
    assert (cnt[ro] == 1).all()
    ro_mech = ptr[ro]
    mloc = np.repeat(np.arange(L), cnt)
    mt = np.arange(M) - ptr[mloc] + 1
    col = np.asarray(locs.mech_col, dtype=np.int64)
    has = col >= 0
    mech_to_col = csc_matrix((np.ones(int(has.sum()), dtype=np.int64), (np.flatnonzero(has), col[has])), shape=(M, num_col))
    loc_to_col = csc_matrix((np.ones(int(has.sum()), dtype=np.int64), (mloc[has], col[has])), shape=(L, num_col))
    t_mech = thresholds(locs.mech_prob)
    t_erase = thresholds(np.broadcast_to(np.asarray(erasure_rate, dtype=np.float64), (L,)))
    t_class = class_thresholds(weights)
    t_flip = thresholds(np.asarray(flip_prob, dtype=np.float64))
    ro_col = col[ro_mech]
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
        cls = (draws[:, ro, 2][:, :, None] >= t_class[None, None, :]).sum(axis=2)
        thr = np.broadcast_to(t_mech[None, :], (n, M)).copy()
        thr[:, ro_mech] = t_flip[cls]
        w = draws[:, mloc, mt]
        fired = np.where(erased[:, mloc], w < np.uint32(0x80000000), w < thr)
        err = (np.asarray((mech_to_col.T @ fired.T.astype(np.int64))).T % 2).astype(np.uint8)
        e = err.astype(np.int64)
        det = (np.asarray(chk @ e.T).T % 2).astype(np.uint8)
        ob = (np.asarray(obs @ e.T).T % 2).astype(np.uint8)
        lost = np.asarray(loc_to_col.T @ erased.T.astype(np.int64)).T > 0
        llr = np.broadcast_to(np.asarray(col_llr, dtype=np.float64)[None, :], (n, num_col)).copy()
        with_col = np.flatnonzero(ro_col >= 0)
        llr[:, ro_col[with_col]] = np.asarray(class_llr)[with_col[None, :], cls[:, with_col]]
        llr[lost] = 0.0
        outs.append((det, ob, err, erased.astype(np.uint8), cls.astype(np.uint8), llr))
    # C-contiguous like the device outputs (the transposed matrix products above are not)
    return tuple(np.ascontiguousarray(np.concatenate([o[i] for o in outs], axis=0)) for i in range(6))
