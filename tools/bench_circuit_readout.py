"""Circuit-level sampling with soft measurement readout, and decoding with it, on one GPU.

Workloads: bb_memory_circuit of [[72,12,6]] x 6 rounds and [[144,12,12]] x 12 rounds (z basis, p = 0.003 for gates and
measurements), Gaussian readout with K = 16 classes (dem.gaussian_readout), --shots shots per call.  Three modes per
workload, timed with CUDA events after --warmup calls and alternated call by call in one process:
  (a) readout_sampler   swd_window_sample_circuit_readout with det, obs, classes and the per-shot LLR rows;
  (b) circuit_sampler   swd_window_sample_circuit with det, obs and the LLR rows, on the same window (the readout set-up
                        is ignored there), so (a) / (b) is the cost of the readout path;
  (c) soft_loop         the device loop of circuit_soft_readout_decoding's soft_aware leg: sampler, then
                        SlidingWindowDecoder.decode_device(channel_llr=rows) with bench.py's c3_gdg kwargs (GDG per window,
                        W = 3, F = 1, method 1, two streams); the sampler's share of the loop is (a) over (c).
Then the failure counts of both legs of circuit_soft_readout_decoding at the points of LER_POINTS.  The card's name and
power limit are read in the same run and written on every line.

    python tools/bench_circuit_readout.py [--shots 65536] [--calls 5] [--warmup 2] [--out profiles/circuit_readout.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

P, K = 0.003, 16
C3_GDG = dict(max_iter=8, max_iter_per_step=6, max_step=25, max_tree_depth=3, max_side_depth=10, max_tree_branch_step=10,
              max_side_branch_step=10, multi_thread=True, low_error_mode=False)         # bench.py's c3_gdg kwargs
# (N, p, p_meas, K, rounds, shots, seed): readout noise well above gate noise; the first is the point
# test_soft_information_helps pins
LER_POINTS = ((72, 0.003, 0.04, 16, 6, 4000, 2024), (72, 0.003, 0.04, 16, 6, 20000, 2024), (144, 0.003, 0.04, 16, 12, 20000, 7))


def run(N, rounds, args, info):
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, _lib, gaussian_readout
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from slidingwindowdecoder_b200.windows import build_windows
    code, A, B_ = bb_code(N)
    s = CircuitNoiseSampler(bb_memory_circuit(code, A, B_, P, rounds), readout=gaussian_readout(P, K))
    plan = build_windows(s.chk, s.obs, s.priors, code.N, W=3, F=1, method=1)
    swd = SlidingWindowDecoder(plan, decoder="gdg", streams=2, **C3_GDG)
    B, dev = args.shots, torch.device("cuda", 0)
    R = len(s.readout_locations)
    lib = _lib.load()
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    u8 = dict(dtype=torch.uint8, device=dev)
    det, obs = torch.empty((B, s.num_det), **u8), torch.empty((B, s.num_obs), **u8)
    cls = torch.empty((B, R), **u8)
    L = torch.empty((B, s.num_col), dtype=torch.float64, device=dev)

    def mode_a(i):
        _lib.check(lib.swd_window_sample_circuit_readout(s._win, 7, i * B, B, det.data_ptr(), obs.data_ptr(), None, None,
                                                         cls.data_ptr(), L.data_ptr(), stream), "sample_circuit_readout")

    def mode_b(i):
        _lib.check(lib.swd_window_sample_circuit(s._win, 7, i * B, B, det.data_ptr(), obs.data_ptr(), None, None, L.data_ptr(),
                                                 stream), "sample_circuit")

    def mode_c(i):
        d, o, rows = s.sample(B, seed=11, shot_offset=i * B, return_llr=True)
        return swd.decode_device(d, o, channel_llr=rows)["counts"]

    times = {m: [] for m in "abc"}
    last = None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(args.warmup + args.calls):
        for m, fn in (("a", mode_a), ("b", mode_b), ("c", mode_c)):
            torch.cuda.synchronize()
            e0.record()
            r = fn(i)
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                times[m].append(e0.elapsed_time(e1) / 1e3)
            if m == "c":
                last = r
    base = dict(workload=f"bb{N}x{rounds}_z_p{P}", num_classes=K, num_locations=int(s.num_locations), num_readout=R,
                num_readout_with_column=int((s.locations.mech_col[s.locations.mech_ptr[s.readout_locations]] >= 0).sum()),
                num_col=int(s.num_col), num_det=int(s.num_det), shots=B, calls=args.calls, warmup=args.warmup)
    t = {m: sum(v) / args.calls for m, v in times.items()}
    lines = [dict(base, mode="a_readout_sampler", outputs="det, obs, readout classes, channel_llr", ms_per_call=round(1e3 * t["a"], 3),
                  ms_min=round(1e3 * min(times["a"]), 3), shots_per_s=round(B / t["a"], 1), over_circuit_sampler=round(t["a"] / t["b"], 4)),
             dict(base, mode="b_circuit_sampler", outputs="det, obs, channel_llr", ms_per_call=round(1e3 * t["b"], 3),
                  ms_min=round(1e3 * min(times["b"]), 3), shots_per_s=round(B / t["b"], 1)),
             dict(base, mode="c_soft_loop", decoder="gdg", decoder_kwargs=C3_GDG, ms_per_call=round(1e3 * t["c"], 3),
                  shots_per_s=round(B / t["c"], 1), sampler_share=round(t["a"] / t["c"], 4),
                  flagged=int(last[0]), logical_failures=int(last[1]))]
    for line in lines:
        line.update(info)
    return lines


def ler_point(N, p, p_meas, num_classes, rounds, shots, seed, info):
    from slidingwindowdecoder_b200 import circuit_soft_readout_decoding
    t0 = time.perf_counter()
    res = circuit_soft_readout_decoding(N, p, p_meas=p_meas, num_classes=num_classes, num_repeat=rounds, num_shots=shots, seed=seed,
                                        max_iter=8)
    a, b = res["static"]["num_logical"], res["soft_aware"]["num_logical"]
    line = dict(mode="d_ler", workload=f"bb{N}x{rounds}_z", p=p, p_meas=p_meas, num_classes=num_classes, shots=shots, seed=seed,
                decoder="gdg", decoder_kwargs="sliding_window_decoder defaults, max_iter=8", class_histogram=res["class_histogram"],
                wall_s=round(time.perf_counter() - t0, 2), difference_in_sd=round((a - b) / max(1.0, np.sqrt(a + b)), 2))
    for leg in ("static", "soft_aware"):
        line[leg] = {k: res[leg][k] for k in ("num_flagged", "num_logical", "p_l", "p_l_per_round")}
    line.update(info)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shots", type=int, default=65536)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "circuit_readout.jsonl"), help="append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from bench_per_shot_llr import card_info
    info = card_info()
    with open(args.out, "a") as out:
        def emit(line):
            s = json.dumps(line)
            print(s, flush=True)
            out.write(s + "\n")
        for N, rounds in ((72, 6), (144, 12)):
            for line in run(N, rounds, args, info):
                emit(line)
        for pt in LER_POINTS:
            emit(ler_point(*pt, info))


if __name__ == "__main__":
    main()
