"""Circuit-level erasure sampling and decoding on one GPU.

Workloads: bb_memory_circuit of [[72,12,6]] x 6 rounds and [[144,12,12]] x 12 rounds (z basis, p = 0.003), each at gate
erasure rate 0 and 0.01, --shots shots per call.  Three modes per workload, timed with CUDA events after --warmup calls and
alternated call by call in one process:
  (a) circuit_sampler   swd_window_sample_circuit with det, obs, erased and the per-shot LLR rows (what the driver asks for);
  (b) dem_sampler       swd_window_sample (one Bernoulli per DEM column) on the same DEM, det and obs;
  (c) erasure_loop      the device loop of circuit_erasure_decoding's erasure_aware leg: sampler, then
                        SlidingWindowDecoder.decode_device(channel_llr=rows) with bench.py's c3_gdg kwargs (GDG per window,
                        W = 3, F = 1, method 1, two streams); the sampler's share of the loop is (a) over (c).
Then the LER of both legs of circuit_erasure_decoding at the points of LER_POINTS.  The card's name and power limit are read in
the same run and written on every line.

    python tools/bench_circuit_erasure.py [--shots 65536] [--calls 5] [--warmup 2] [--out profiles/circuit_erasure.jsonl]
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

P = 0.003
RATES = (0.0, 0.01)
C3_GDG = dict(max_iter=8, max_iter_per_step=6, max_step=25, max_tree_depth=3, max_side_depth=10, max_tree_branch_step=10,
              max_side_branch_step=10, multi_thread=True, low_error_mode=False)         # bench.py's c3_gdg kwargs
# (N, p, gate erasure rate, rounds, shots, seed): the first is the point test_erasure_information_helps pins
LER_POINTS = ((72, 0.001, 0.01, 6, 4000, 2024), (144, 0.001, 0.005, 12, 20000, 7))


def run(N, rounds, rate, args, info):
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, _lib
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from slidingwindowdecoder_b200.windows import build_windows
    code, A, B_ = bb_code(N)
    s = CircuitNoiseSampler(bb_memory_circuit(code, A, B_, P, rounds), erasure_rate=rate)
    plan = build_windows(s.chk, s.obs, s.priors, code.N, W=3, F=1, method=1)
    swd = SlidingWindowDecoder(plan, decoder="gdg", streams=2, **C3_GDG)
    B, dev = args.shots, torch.device("cuda", 0)
    lib = _lib.load()
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    u8 = dict(dtype=torch.uint8, device=dev)
    det, obs = torch.empty((B, s.num_det), **u8), torch.empty((B, s.num_obs), **u8)
    erased = torch.empty((B, s.num_locations), **u8)
    L = torch.empty((B, s.num_col), dtype=torch.float64, device=dev)
    pri = np.ascontiguousarray(plan.priors, dtype=np.float64)          # swd._win holds the plan's column order
    _lib.check(lib.swd_window_set_priors(swd._win, pri.ctypes.data_as(C.POINTER(C.c_double))), "set_priors")

    def mode_a(i):
        _lib.check(lib.swd_window_sample_circuit(s._win, 7, i * B, B, det.data_ptr(), obs.data_ptr(), None, erased.data_ptr(),
                                                 L.data_ptr(), stream), "sample_circuit")

    def mode_b(i):
        _lib.check(lib.swd_window_sample(swd._win, 7, i * B, B, det.data_ptr(), obs.data_ptr(), None, stream), "sample")

    def mode_c(i):
        d, o, _, rows = s.sample(B, seed=11, shot_offset=i * B, return_erasures=True, return_llr=True)
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
    locs = s.locations
    philox_calls = int(((locs.mech_ptr[1:] - locs.mech_ptr[:-1]) // 4 + 1).sum())
    base = dict(workload=f"bb{N}x{rounds}_z_p{P}", num_locations=int(s.num_locations), num_mechanisms=int(locs.mech_ptr[-1]),
                num_col=int(s.num_col), num_det=int(s.num_det), gate_erasure_rate=rate, shots=B, calls=args.calls,
                warmup=args.warmup, philox_calls_per_shot=philox_calls, dem_philox_calls_per_shot=(s.num_col + 3) // 4)
    t = {m: sum(v) / args.calls for m, v in times.items()}
    lines = [dict(base, mode="a_circuit_sampler", outputs="det, obs, erased, channel_llr", ms_per_call=round(1e3 * t["a"], 3),
                  shots_per_s=round(B / t["a"], 1)),
             dict(base, mode="b_dem_sampler", outputs="det, obs", ms_per_call=round(1e3 * t["b"], 3), shots_per_s=round(B / t["b"], 1)),
             dict(base, mode="c_erasure_loop", decoder="gdg", decoder_kwargs=C3_GDG, ms_per_call=round(1e3 * t["c"], 3),
                  shots_per_s=round(B / t["c"], 1), sampler_share=round(t["a"] / t["c"], 4),
                  flagged=int(last[0]), logical_failures=int(last[1]))]
    for line in lines:
        line.update(info)
    return lines


def ler_point(N, p, rate, rounds, shots, seed, info):
    from slidingwindowdecoder_b200 import circuit_erasure_decoding
    t0 = time.perf_counter()
    res = circuit_erasure_decoding(N, p, rate, num_repeat=rounds, num_shots=shots, seed=seed, max_iter=8)
    line = dict(mode="d_ler", workload=f"bb{N}x{rounds}_z", p=p, gate_erasure_rate=rate, shots=shots, seed=seed, decoder="gdg",
                decoder_kwargs="sliding_window_decoder defaults, max_iter=8", erased_fraction=res["erased_fraction"],
                wall_s=round(time.perf_counter() - t0, 2))
    for leg in ("static", "erasure_aware"):
        line[leg] = {k: res[leg][k] for k in ("num_flagged", "num_logical", "p_l", "p_l_per_round")}
    line.update(info)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shots", type=int, default=65536)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "circuit_erasure.jsonl"), help="append the JSON lines to this file")
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
            for rate in RATES:
                for line in run(N, rounds, rate, args, info):
                    emit(line)
        for pt in LER_POINTS:
            emit(ler_point(*pt, info))


if __name__ == "__main__":
    main()
