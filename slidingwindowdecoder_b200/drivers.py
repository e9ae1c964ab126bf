"""The reference's two driver scripts as functions with their own signatures, running on one B200.

  sliding_window_decoder      <- guessing.py:18-236  (GDG per window, last window decoded again with BP+OSD-CS10)
  sliding_window_osd_decoder  <- osd.py:15-199       (BP+OSD per window; shorten=True uses osd_window)
  circuit_erasure_decoding    the window decoder under circuit noise with heralded gate erasures, with and without the
                              per-shot erasure information (no reference counterpart)

Same arguments, same printed statistics (per-window flagged counts, overall flagged / logical errors, logical error
per round); the per-shot Python loops are replaced by one batched call per window with the shot data resident on the
device (SlidingWindowDecoder), the stim circuit / DEM / sampler by this package's stim-free builder and Philox sampler.
`plot` is accepted and ignored.  Both return a dict with the numbers they print.
"""
import time

import numpy as np

from .codes import bb_code
from .dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
from .sliding_window import SlidingWindowDecoder
from .windows import build_windows


def _plan(N, p, num_repeat, W, F, z_basis, noisy_prior, method, keep_cols=None):
    try:
        code, A_list, B_list = bb_code(N)
    except KeyError:
        print("unsupported N")                                           # guessing.py:38-40
        return None, None
    chk, obs, priors = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A_list, B_list, p, num_repeat, z_basis=z_basis)))
    return code, build_windows(chk, obs, priors, code.N, W=W, F=F, method=method, noisy_prior=noisy_prior, keep_cols=keep_cols)


def _report(counts, num_shots, num_repeat):
    num_flagged, num_err = int(counts[0]), int(counts[1])
    print(f"Overall Flagged Errors: {num_flagged}/{num_shots}")
    print(f"Logical Errors: {num_err}/{num_shots}")
    p_l = num_err / num_shots
    p_l_per_round = 1 - (1 - p_l) ** (1 / num_repeat)
    print("logical error per round:", p_l_per_round)
    return dict(num_flagged=num_flagged, num_logical=num_err, p_l=p_l, p_l_per_round=p_l_per_round)


def sliding_window_decoder(N, p=0.003, num_repeat=12, num_shots=10000, max_iter=200, W=3, F=1, z_basis=True,
                           noisy_prior=None, method=1, plot=False, low_error_mode=False,
                           max_step=25, max_iter_per_step=6, max_tree_depth=3, max_side_depth=10, max_side_branch_step=10,
                           last_win_gdg_factor=1.0, last_win_bp_factor=1.0, seed=0, device=0, streams=2):
    """guessing.py:18-236.  Note the reference passes max_tree_branch_step=max_side_branch_step (guessing.py:168-169)."""
    code, plan = _plan(N, p, num_repeat, W, F, z_basis, noisy_prior, method)
    if plan is None:
        return None
    kw = dict(max_iter=max_iter, max_iter_per_step=max_iter_per_step, max_step=max_step, max_tree_depth=max_tree_depth,
              max_side_depth=max_side_depth, max_tree_branch_step=max_side_branch_step, max_side_branch_step=max_side_branch_step,
              multi_thread=True, low_error_mode=low_error_mode)
    swd = SlidingWindowDecoder(plan, decoder="gdg", device=device, streams=streams, last_window_osd=True,
                               last_window_kwargs=dict(gdg_factor=last_win_gdg_factor, ms_scaling_factor=last_win_bp_factor), **kw)
    t0 = time.perf_counter()
    det, obs = swd.sample_device(num_shots, seed=seed)
    swd.torch.cuda.synchronize()
    print(f"Stim: noise sampling for {num_shots} shots, elapsed time:", time.perf_counter() - t0)
    t0 = time.perf_counter()
    out = swd.decode_device(det, obs)
    counts = out["counts"].cpu().numpy()
    unconv = out["window_unconverged"].cpu().numpy()
    elapsed = time.perf_counter() - t0
    for i, k in enumerate(unconv):
        print(f"Window {i}, flagged Errors: {int(k)}/{num_shots}")
    print("Elapsed time:", elapsed)
    print("last round osd", False)
    res = dict(gdg=_report(counts, num_shots, num_repeat), window_flagged=[int(k) for k in unconv], elapsed=elapsed)
    print("last round osd", True)
    res["last_window_osd"] = _report(out["counts_last_window_osd"].cpu().numpy(), num_shots, num_repeat)
    return res


def sliding_window_osd_decoder(N, p=0.003, num_repeat=12, num_shots=10000, max_iter=200, W=2, F=1, z_basis=True,
                               noisy_prior=None, method=0, plot=False, shorten=False, seed=0, device=0, streams=2):
    """osd.py:15-199 (`sliding_window_decoder` there).  shorten=False: BpOsdDecoder(max_iter, minimum_sum, OSD_CS 10) per
    window (this package's facade; parity with the third-party ldpc package unpinned); shorten=True:
    osd_window(pre_max_iter=8, post_max_iter=max_iter, osd_cs, osd_order=0) as osd.py:152-161.  The x basis keeps n
    un-merged columns of the next round (osd.py:83,106)."""
    code, plan = _plan(N, p, num_repeat, W, F, z_basis, noisy_prior, method, keep_cols=None)
    if plan is None:
        return None
    if not z_basis and method == 1:
        code, plan = _plan(N, p, num_repeat, W, F, z_basis, noisy_prior, method, keep_cols=code.N)
    if shorten:
        from .decoders import osd_window as cls
        kw = dict(pre_max_iter=8, post_max_iter=max_iter, ms_scaling_factor=1.0, new_n=None, osd_method="osd_cs", osd_order=0)
    else:
        from .decoders import BpOsdDecoder as cls
        kw = dict(max_iter=max_iter, bp_method="minimum_sum", ms_scaling_factor=1.0, osd_method="OSD_CS", osd_order=10)
    swd = SlidingWindowDecoder(plan, decoder=cls, device=device, streams=streams, **kw)
    t0 = time.perf_counter()
    det, obs = swd.sample_device(num_shots, seed=seed)
    swd.torch.cuda.synchronize()
    print(f"Stim: noise sampling for {num_shots} shots, elapsed time:", time.perf_counter() - t0)
    t0 = time.perf_counter()
    out = swd.decode_device(det, obs, window_residuals=True)
    counts = out["counts"].cpu().numpy()
    flagged = out["window_flagged"].cpu().numpy()
    elapsed = time.perf_counter() - t0
    for i, k in enumerate(flagged):
        print(f"Window {i}, flagged Errors: {int(k)}/{num_shots}")       # osd.py:166-176: H e_hat != window syndrome
    print("Elapsed time:", elapsed)
    res = _report(counts, num_shots, num_repeat)
    res.update(window_flagged=[int(k) for k in flagged], elapsed=elapsed)
    return res


_GDG_DEFAULTS = dict(max_iter=200, max_iter_per_step=6, max_step=25, max_tree_depth=3, max_side_depth=10, max_tree_branch_step=10,
                     max_side_branch_step=10, multi_thread=True, low_error_mode=False)          # sliding_window_decoder's
_OSD_DEFAULTS = dict(pre_max_iter=8, post_max_iter=200, osd_method="osd_cs", osd_order=10)


def circuit_erasure_decoding(N, p, erasure_rate, num_repeat=12, num_shots=10000, W=3, F=1, z_basis=True, decoder="gdg",
                             batch=32768, seed=0, shot_offset=0, device=0, streams=2, **decoder_kwargs):
    """Logical error rate of the sliding-window decoder on the BB-code memory experiment `bb_memory_circuit` (noise strength
    p, `num_repeat` rounds) when `erasure_rate` of the two-qubit gates are erased (a heralded, uniformly random two-qubit
    Pauli; an array gives one rate per noise location, see CircuitNoiseSampler).  Shots [shot_offset, shot_offset +
    num_shots) of the seed's stream are sampled on the device (CircuitNoiseSampler) in batches of `batch` and each batch is
    decoded twice by one SlidingWindowDecoder (method 1 windows, W, F; decoder "gdg" with sliding_window_decoder's
    defaults or "osd" with osd_window BP + OSD-CS10, updated by decoder_kwargs):
      static         with the DEM's priors, as if the erasures were not heralded;
      erasure_aware  with the sampled per-shot LLR rows (0.0 at the DEM columns of erased gates).
    Counts do not depend on `batch` or `streams`, and `distributed.shard_range` splits a job by shot_offset.  -> dict with
    per leg num_flagged, num_logical, p_l, p_l_per_round, window_unconverged (list per window), plus erased_fraction (over
    all noise locations of all shots) and elapsed (seconds)."""
    import torch
    from .simulation import CircuitNoiseSampler
    p, num_shots, batch = float(p), int(num_shots), int(batch)
    if not 0.0 < p < 0.5:
        raise ValueError(f"p must lie in (0, 0.5), got {p}")
    if num_shots < 0 or batch <= 0 or int(shot_offset) < 0:
        raise ValueError("need num_shots >= 0, batch > 0 and shot_offset >= 0")
    if decoder not in ("gdg", "osd"):
        raise ValueError(f"decoder must be 'gdg' or 'osd', got {decoder!r}")
    try:
        code, A_list, B_list = bb_code(N)
    except KeyError:
        raise ValueError(f"unsupported N = {N}") from None
    kw = dict(_GDG_DEFAULTS if decoder == "gdg" else _OSD_DEFAULTS)
    kw.update(decoder_kwargs)
    sampler = CircuitNoiseSampler(bb_memory_circuit(code, A_list, B_list, p, num_repeat, z_basis=z_basis), erasure_rate=erasure_rate,
                                  device=device)
    plan = build_windows(sampler.chk, sampler.obs, sampler.priors, code.N, W=W, F=F, method=1)
    swd = SlidingWindowDecoder(plan, decoder=decoder, device=device, streams=streams, **kw)
    legs = ("static", "erasure_aware")
    dev = torch.device("cuda", int(device))
    counts = torch.zeros((2, 2), dtype=torch.int64, device=dev)
    unconv = torch.zeros((2, len(plan.windows)), dtype=torch.int64, device=dev)
    erased = torch.zeros((), dtype=torch.int64, device=dev)
    t0 = time.perf_counter()
    for start in range(0, num_shots, batch):
        B = min(batch, num_shots - start)
        det, obs, er, L = sampler.sample(B, seed=seed, shot_offset=int(shot_offset) + start, return_erasures=True, return_llr=True)
        erased += er.sum(dtype=torch.int64)
        out = swd.decode_device(det.clone(), obs.clone())
        counts[0] += out["counts"]
        unconv[0] += out["window_unconverged"]
        out = swd.decode_device(det, obs, channel_llr=L)
        counts[1] += out["counts"]
        unconv[1] += out["window_unconverged"]
    c, u = counts.cpu().tolist(), unconv.cpu().tolist()
    n_erased = int(erased.item())
    res = dict(erased_fraction=n_erased / max(1, num_shots * sampler.num_locations), elapsed=time.perf_counter() - t0)
    for i, leg in enumerate(legs):
        p_l = c[i][1] / max(1, num_shots)
        res[leg] = dict(num_flagged=int(c[i][0]), num_logical=int(c[i][1]), p_l=p_l, p_l_per_round=1 - (1 - p_l) ** (1 / num_repeat),
                        window_unconverged=[int(k) for k in u[i]])
    return res
