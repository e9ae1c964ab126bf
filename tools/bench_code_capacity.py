"""Code-capacity simulation loop for bp4_osd under depolarizing noise with heralded erasures (one GPU).

Workloads: the [[72,12,6]] pair, per-qubit probabilities and kwargs of the c1_bp4_osd_cs8 fixture, and codes.bb_code(144) at
p = 0.06 (px = py = pz = p/3) with the same kwargs; each at erasure rate 0 and 0.05, --shots shots per call.  Three modes, timed
after --warmup calls and alternated call by call in one process:
  (a) sampler         swd_window_sample_pauli alone with every output (det, obs, err, erased, channel_llr), CUDA events around
                      the launch.  Reports shots/s and the bytes written per shot, 2n + mx + mz + num_obs + n + 40n, over kernel
                      time as a share of the HBM copy roof bench.py uses (MEASURED_PEAKS.json's hbm_gbs when present, else
                      bench.py's fallback; the line names which);
  (b) device_loop     CodeCapacitySampler.sample -> bp4_osd.decode_batch -> count_failures, all on the device, CUDA events;
  (c) host_sampler    the numpy sampler of tools/bench_bp4_per_shot_llr.py, the [5, B, n] planes built on the host, the H2D copies
                      of the syndromes (and planes), the same decode, the D2H copy of the corrections and a numpy failure count;
                      host clock around work that ends in a device synchronise.
(b) and (c) decode once per shot: with the static priors at erasure rate 0, with the sampled planes at 0.05.  The card's name
and power limit are read in the same run and written on every line.

    python tools/bench_code_capacity.py [--shots 65536] [--calls 5] [--warmup 2] [--out profiles/code_capacity.jsonl]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

RATES = (0.0, 0.05)
HBM_FALLBACK_GBS = 6650.0                      # bench.py's value when MEASURED_PEAKS.json is absent


def hbm_roof():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return HBM_FALLBACK_GBS, "fallback (bench.py)"


def workloads():
    """-> [(name, g)] with g = dict(hx, hz csc, lx, lz, px, py, pz, kwargs) in the form bench_bp4_per_shot_llr.sample reads."""
    from scipy.sparse import csc_matrix
    from conftest import load_golden_bp4
    from slidingwindowdecoder_b200.codes import bb_code
    g72 = load_golden_bp4("c1_bp4_osd_cs8")
    c72, _, _ = bb_code(72)
    c144, _, _ = bb_code(144)
    p = np.full(c144.N, 0.06 / 3)
    return [("bb72_c1_bp4_osd_cs8", dict(hx=g72["hx"], hz=g72["hz"], lx=c72.lx, lz=c72.lz, px=g72["px"], py=g72["py"], pz=g72["pz"],
                                         kwargs=g72["kwargs"])),
            ("bb144_p0.06", dict(hx=csc_matrix(c144.hx), hz=csc_matrix(c144.hz), lx=c144.lx, lz=c144.lz, px=p, py=p, pz=p,
                                 kwargs=g72["kwargs"]))]


def host_failures(g, dec, ex, ez):
    """Residual not a stabilizer: the syndrome is not reproduced, or it anticommutes with a logical."""
    hx, hz = (np.asarray(g[k].todense()).astype(np.int64) for k in ("hx", "hz"))
    rx, rz = ex ^ dec[:, 0].astype(np.int64), ez ^ dec[:, 1].astype(np.int64)
    bad = ((rz @ hx.T) % 2).any(axis=1) | ((rx @ hz.T) % 2).any(axis=1)
    bad |= ((rx @ g["lz"].T) % 2).any(axis=1) | ((rz @ g["lx"].T) % 2).any(axis=1)
    return int(bad.sum())


def run(name, g, rate, args, info, roof):
    import torch
    from bench_bp4_per_shot_llr import sample as host_sample
    from slidingwindowdecoder_b200 import CodeCapacitySampler, _lib, bp4_osd
    dec = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **g["kwargs"])
    s = CodeCapacitySampler(g["hx"], g["hz"], g["lx"], g["lz"], g["px"], g["py"], g["pz"], erasure_rate=rate, channel_llr=dec.channel_llr)
    B, n, dev = args.shots, s.n, torch.device("cuda", 0)
    erase = rate > 0
    u8 = dict(dtype=torch.uint8, device=dev)
    bufs = [torch.empty((B, s.num_det), **u8), torch.empty((B, s.num_obs), **u8), torch.empty((B, 2, n), **u8),
            torch.empty((B, n), **u8), torch.empty((5, B, n), dtype=torch.float64, device=dev)]
    bytes_per_shot = 2 * n + s.num_det + s.num_obs + n + 40 * n
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    lib = _lib.load()
    rng = np.random.default_rng(2024)
    L_static = np.repeat(dec.channel_llr[:, None, :], B, axis=1)

    def mode_a(i):
        _lib.check(lib.swd_window_sample_pauli(s._win, 7, i * B, B, *(t.data_ptr() for t in bufs), stream), "sample_pauli")

    def mode_b(i):
        out = s.sample(B, seed=11, shot_offset=i * B, return_llr=erase)
        d = dec.decode_batch(out["synd_x"], out["synd_z"], channel_llr=out["channel_llr"] if erase else None)
        return s.count_failures(d["dec"], out["det"], out["obs"])

    def mode_c(i):
        er, ex, ez, sx, sz = host_sample(g, B, rng, rate)
        L = None
        if erase:
            L = L_static.copy()
            L[:, er] = 0.0
            L = torch.from_numpy(L).to(dev)
        d = dec.decode_batch(torch.from_numpy(sx).to(dev), torch.from_numpy(sz).to(dev), channel_llr=L)["dec"].cpu().numpy()
        return host_failures(g, d, ex, ez)

    times = {m: [] for m in "abc"}
    last = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(args.warmup + args.calls):
        for m, fn in (("a", mode_a), ("b", mode_b)):
            torch.cuda.synchronize()
            e0.record()
            r = fn(i)
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                times[m].append(e0.elapsed_time(e1) / 1e3)
            last[m] = r
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last["c"] = mode_c(i)
        torch.cuda.synchronize()
        if i >= args.warmup:
            times["c"].append(time.perf_counter() - t0)
    base = dict(workload=name, n=int(n), mx=int(s.mx), mz=int(s.mz), num_obs=int(s.num_obs), erasure_rate=rate, kwargs=g["kwargs"],
                shots=B, calls=args.calls, warmup=args.warmup)
    lines = []
    for m, label in (("a", "a_sampler"), ("b", "b_device_loop"), ("c", "c_host_sampler")):
        t = sum(times[m]) / args.calls
        line = dict(base, mode=label, shots_per_s=round(B / t, 1), ms_per_call=round(1e3 * t, 3))
        if m == "a":
            gbs = B * bytes_per_shot / t / 1e9
            line.update(bytes_per_shot=bytes_per_shot, written_gbs=round(gbs, 1), hbm_roof_gbs=roof[0], hbm_roof_source=roof[1],
                        share_of_hbm_roof=round(gbs / roof[0], 4))
        elif m == "b":
            flagged, failed = (int(x) for x in last["b"].tolist())
            line.update(flagged=flagged, logical_failures=failed)
        else:
            line.update(logical_failures=last["c"])
        line.update(info)
        lines.append(line)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shots", type=int, default=65536)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "code_capacity.jsonl"), help="append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from bench_per_shot_llr import card_info
    info = card_info()
    roof = hbm_roof()
    with open(args.out, "a") as out:
        for name, g in workloads():
            for rate in RATES:
                for line in run(name, g, rate, args, info, roof):
                    s = json.dumps(line)
                    print(s, flush=True)
                    out.write(s + "\n")


if __name__ == "__main__":
    main()
