"""Cost of per-shot channel priors on the bench workloads (device-resident shot data, one B200).

For the default C3 workload (bench.py: [[144,12,12]], 12 rounds, W=3 F=1, GDG) the same syndromes are decoded in three modes:
  (a) no channel_llr (the static path);
  (b) channel_llr rows equal to the plan's priors (per-shot kernels, identical results);
  (c) 1 % of the DEM columns of every shot erased (LLR 0).
For g144_osd (un-windowed DEM, HBM-streamed BP) modes (a) and (b).  Modes alternate step by step; the script asserts that (a) and
(b) give identical counts, window_unconverged and corrections, and prints one JSON line per workload and mode with the card's
name and power limit read in the same run.

    python tools/bench_per_shot_llr.py [--batch 32768] [--steps 5] [--warmup 2] [--workloads c3_gdg,g144_osd]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STREAMS = {"c3_gdg": 3, "g144_osd": 1}        # bench.py's settings for these workloads


def card_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        pl, mx = (x.strip() for x in out.split(","))
        return dict(gpu=name, power_limit_w=float(pl), sm_max_mhz=float(mx))
    except Exception as e:        # noqa: BLE001 - report what could not be read rather than fail the measurement
        return dict(gpu=name, power_limit_w=None, sm_max_mhz=None, note=f"nvidia-smi: {e}")


def run_workload(key, args, info):
    import torch
    import bench
    from slidingwindowdecoder_b200.decoders import _libm_llr
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    bench.select_workload(key)
    wl = bench.WL
    plan = bench.build_plan()
    swd = SlidingWindowDecoder(plan, decoder=wl["decoder"], device=0, streams=STREAMS[key], **wl["kw"])
    dev = torch.device("cuda", 0)
    B, K, W = args.batch, args.steps, args.warmup
    det0, obs0 = swd.sample_device(B, seed=4321)
    num_col = swd.num_col
    # mode (b): the plan's priors as LLRs, in the DEM's column order (plan column j is DEM column col_order[j])
    llr_plan = _libm_llr(plan.priors, num_col)
    llr_dem = np.empty(num_col)
    order = plan.col_order if plan.col_order is not None else np.arange(num_col)
    llr_dem[order] = llr_plan
    L_b = torch.from_numpy(llr_dem).to(dev).unsqueeze(0).expand(B, -1).contiguous()
    modes = {"a_static": None, "b_plan_rows": L_b}
    if key == "c3_gdg":
        g = torch.Generator(device=dev); g.manual_seed(7)
        L_c = L_b.clone()
        L_c[torch.rand((B, num_col), generator=g, device=dev) < 0.01] = 0.0
        modes["c_erase_1pct"] = L_c

    def step(L, corrections=False):
        det, obs = det0.clone(), obs0.clone()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = swd.decode_device(det, obs, return_corrections=corrections, channel_llr=L)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    # identical results of (a) and (b), checked once outside the timed steps
    _, oa = step(None, True)
    _, ob = step(L_b, True)
    for k in ("counts", "window_unconverged", "total_e_hat"):
        assert torch.equal(oa[k], ob[k]), f"{key}: mode (a) and (b) differ in {k}"
    del oa, ob
    times = {m: [] for m in modes}
    counts = {}
    for i in range(W + K):
        for m, L in modes.items():
            t, out = step(L)
            if i >= W:
                times[m].append(t)
            counts[m] = out["counts"].cpu().tolist()
    base = B * K / sum(times["a_static"])
    lines = []
    for m in modes:
        rate = B * K / sum(times[m])
        lines.append(dict(workload=key, mode=m, shots_per_s=round(rate, 1), vs_static=round(rate / base, 4),
                          ms_per_step=round(1e3 * sum(times[m]) / K, 3), batch=B, steps=K, warmup=W, streams=STREAMS[key],
                          counts_flagged_failed=counts[m], **info))
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="c3_gdg,g144_osd")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    info = card_info()
    for key in args.workloads.split(","):
        for line in run_workload(key, args, info):
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
