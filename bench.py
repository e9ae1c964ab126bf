#!/usr/bin/env python
"""Benchmark of the hot path: sliding-window GDG decoding throughput (decoded shots / s).

Workload (BASELINE.json configs[2], the configuration the metric is quoted on):
  [[144,12,12]] gross code, circuit-level noise p = 0.003, 12 rounds, sliding window (W, F) = (3, 1)
  -> 11 windows of 216 x (1656 | 1728 | 1656), GDG per window (bpgdg_decoder, max_iter=8, multi_thread tree).
A "step" = one pass of the whole window pipeline over one batch of `--batch` synthetic shots per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]
Under torchrun (N > 1) every rank decodes its own batch (weak scaling); the only collective is the
all-reduce of the failure counters.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

_STDOUT = sys.stdout
import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[2] - the configuration the metric is quoted on (default)
    "c3_gdg": dict(N=144, p=0.003, rounds=12, W=3, F=1, method=1, decoder="gdg",
                   kw=dict(max_iter=8, max_iter_per_step=6, max_step=25, max_tree_depth=3, max_side_depth=10,
                           max_tree_branch_step=10, max_side_branch_step=10, multi_thread=True, low_error_mode=False),
                   name="[[144,12,12]] circuit-level p=0.003, 12 rounds, sliding window W=3 F=1 (11 windows), GDG per window",
                   decoder_name="bpgdg_decoder(max_iter=8, multi_thread=True, defaults)"),
    # configs[1]: BP + OSD-CS10 per window (osd_window, the reference's own BP+OSD)
    "c2_osd": dict(N=72, p=0.003, rounds=6, W=3, F=1, method=1, decoder="osd",
                   kw=dict(pre_max_iter=8, post_max_iter=200, osd_method="osd_cs", osd_order=10),
                   name="[[72,12,6]] circuit-level p=0.003, 6 rounds, sliding window W=3 F=1 (5 windows), BP+OSD-CS10 per window",
                   decoder_name="osd_window(pre_max_iter=8, post_max_iter=200, osd_cs, order 10)"),
    # configs[3]: large windows (576 x 4896), BP + OSD
    "c4_osd": dict(N=288, p=0.003, rounds=18, W=4, F=1, method=1, decoder="osd",
                   kw=dict(pre_max_iter=8, post_max_iter=200, osd_method="osd_cs", osd_order=10),
                   name="[[288,12,18]] circuit-level p=0.003, 18 rounds, sliding window W=4 F=1 (16 windows), BP+OSD-CS10 per window",
                   decoder_name="osd_window(pre_max_iter=8, post_max_iter=200, osd_cs, order 10)"),
    # configs[0]: code capacity, the reference's own CPU-runnable case (src/simulation.py:10-99 with its GDG kwargs :66-82);
    # one "window" = the whole hx, observables = hz_perp (logical check of simulation.py:90-91)
    "c1_gdg": dict(code="capacity", N=72, p=0.05, decoder="gdg",
                   kw=dict(max_iter_per_step=6, gdg_factor=0.625, max_step=40, max_tree_depth=4, max_side_depth=20,
                           max_tree_branch_step=30, max_side_branch_step=20, multi_thread=True, low_error_mode=True,
                           max_iter=24, ms_scaling_factor=0.625, new_n=72),
                   name="[[72,12,6]] BB code, code-capacity data-qubit noise p=0.05, GDG decode via simulation.py",
                   decoder_name="bpgdg_decoder(simulation.py:66-82 kwargs, multi_thread=True)"),
    # configs[4]: SHYPS r=3 memory experiment (SHYPS.ipynb cell 1: windows without merged identity columns), GDG and BP+OSD
    "c5_gdg": dict(code="shyps", r=3, p=0.003, rounds=6, W=3, F=1, method=0, decoder="gdg",
                   kw=dict(max_iter=8, max_iter_per_step=6, max_step=25, max_tree_depth=3, max_side_depth=10,
                           max_tree_branch_step=10, max_side_branch_step=10, multi_thread=True, low_error_mode=False),
                   name="SHYPS r=3 memory experiment p=0.003, 6 rounds, sliding window W=3 F=1, GDG per window",
                   decoder_name="bpgdg_decoder(max_iter=8, multi_thread=True, defaults)"),
    "c5_osd": dict(code="shyps", r=3, p=0.003, rounds=6, W=3, F=1, method=0, decoder="osd",
                   kw=dict(pre_max_iter=8, post_max_iter=100, osd_method="osd_cs", osd_order=10),
                   name="SHYPS r=3 memory experiment p=0.003, 6 rounds, sliding window W=3 F=1, BP+OSD-CS10 per window",
                   decoder_name="osd_window(pre_max_iter=8, post_max_iter=100, osd_cs, order 10)"),
    # the un-windowed [[144,12,12]] DEM of IBM.ipynb cell 2 (936 x 8784, 30672 edges): messages exceed one SM's shared memory, the
    # full-window BP runs HBM-streamed (swd_stream.cuh); decoder kwargs of IBM.ipynb:122-123
    "g144_osd": dict(code="global", N=144, p=0.004, rounds=12, decoder="osd",
                     kw=dict(pre_max_iter=16, post_max_iter=1000, osd_method="osd_cs", osd_order=10),
                     name="[[144,12,12]] circuit-level p=0.004, 12 rounds, un-windowed DEM 936 x 8784 (IBM.ipynb), BP+OSD-CS10 on the whole DEM",
                     decoder_name="osd_window(pre_max_iter=16, post_max_iter=1000, osd_cs, order 10)"),
}
WL = dict(WORKLOADS["c3_gdg"], _key="c3_gdg")
METRIC = {"gdg": "decoded shots/sec (sliding-window GDG)", "osd": "decoded shots/sec (sliding-window BP+OSD)"}


def select_workload(key, p=None):
    global WL
    WL = dict(WORKLOADS[key], _key=key)
    if p is not None:
        WL["name"] = WL["name"].replace(f"p={WL['p']}", f"p={p}")
        WL["p"] = p


def build_plan():
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    if WL.get("code") == "capacity":
        from scipy.sparse import csc_matrix
        from slidingwindowdecoder_b200.windows import WindowPlan, Window
        code, _, _ = bb_code(WL["N"])
        hx, lz = csc_matrix(code.hx), csc_matrix(code.hz_perp)
        pri = np.full(code.N, WL["p"])
        win = Window(0, hx, pri, 0, hx.shape[0], 0, code.N, code.N, True)
        return WindowPlan(hx, lz, pri, [(0, 0), (hx.shape[0], code.N)], [win], code.N // 2, 1, 1)
    if WL.get("code") == "shyps":
        from slidingwindowdecoder_b200.dem import shyps_memory_circuit
        r = WL["r"]
        chk, obs, pri = dem_to_check_matrices(detector_error_model(shyps_memory_circuit(r, WL["p"], WL["rounds"])))
        return build_windows(chk, obs, pri, h=r * (2 ** r - 1), W=WL["W"], F=WL["F"], method=WL["method"])
    code, A, B = bb_code(WL["N"])
    circ = bb_memory_circuit(code, A, B, WL["p"], WL["rounds"], z_basis=True)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(circ))
    if WL.get("code") == "global":          # one "window" = the whole DEM, every column committed
        from scipy.sparse import csc_matrix
        from slidingwindowdecoder_b200.windows import WindowPlan, Window
        chk, obs = csc_matrix(chk), csc_matrix(obs)
        win = Window(0, chk, pri, 0, chk.shape[0], 0, chk.shape[1], chk.shape[1], True)
        return WindowPlan(chk, obs, pri, [(0, 0), chk.shape], [win], code.N // 2, 1, 1)
    return build_windows(chk, obs, pri, code.N, W=WL["W"], F=WL["F"], method=WL["method"])


# ------------------------------------------------------------------------------------------ CPU arm
_CPU = {}


def _cpu_init(plan_blob, use_ref=False, wl_key="c3_gdg", wl_p=None):
    """use_ref: decode with oracle/_ref (the reference's own bpgd.cpp, 15 std::threads per shot) instead of the C port."""
    import ctypes as C
    from oracle.oracle import Oracle, ref_lib, _p
    select_workload(wl_key, wl_p)
    _CPU["plan"] = plan_blob
    _CPU["orc"] = [Oracle(w.mat, w.prior) for w in plan_blob.windows]
    _CPU["chkT"] = plan_blob.chk.T.tocsr()
    _CPU["obsT"] = plan_blob.obs.T.tocsr()
    _CPU["ref"] = None
    if use_ref:
        lib = ref_lib()
        lib.ref_gdg_create.restype = C.c_void_p
        kw = WL["kw"]
        hs = []
        for o in _CPU["orc"]:
            h = lib.ref_gdg_create(o.m, o.n, _p(o.cp, C.c_int), _p(o.cr, C.c_int), _p(o.llr, C.c_double), kw["max_iter"],
                                   C.c_double(1.0), kw["max_iter_per_step"], kw["max_step"], kw["max_tree_depth"],
                                   kw["max_side_depth"], kw["max_tree_branch_step"], kw["max_side_branch_step"],
                                   C.c_double(1.0), 0, 0)
            hs.append(C.c_void_p(h))
        _CPU["ref"] = (lib, hs)


def _decode_window(i, synd):
    import ctypes as C
    from oracle.oracle import _p
    if _CPU["ref"] is None:
        if WL["decoder"] == "osd":
            dec, conv, _, _ = _CPU["orc"][i].osd_window_batch(synd, **WL["kw"])
        else:
            dec, conv, _, _ = _CPU["orc"][i].bpgdg_batch(synd, **WL["kw"])
        return dec
    lib, hs = _CPU["ref"]
    o = _CPU["orc"][i]
    s = np.ascontiguousarray(synd.astype(np.int8))
    dec = np.zeros((s.shape[0], o.n), dtype=np.int8)
    conv = np.zeros(s.shape[0], dtype=np.int8)
    lib.ref_gdg_decode_batch(hs[i], _p(s, C.c_int8), C.c_longlong(s.shape[0]), _p(dec, C.c_int8), _p(conv, C.c_int8))
    return dec


def _cpu_decode_shard(args):
    """The reference's sliding-window loop (guessing.py:141-227) on a shard of shots with the C oracle."""
    det, obs = args
    plan = _CPU["plan"]
    B = det.shape[0]
    new_det = det.copy()
    total = np.zeros((B, plan.chk.shape[1]), dtype=np.uint8)
    for w in plan.windows:
        dec = _decode_window(w.index, new_det[:, w.row0:w.row1])
        total[:, w.col0:w.col0 + w.ncommit] = dec[:, :w.ncommit]
        upd = np.asarray(total[:, w.col0:w.col0 + w.ncommit].astype(np.float32) @ _CPU["chkT"][w.col0:w.col0 + w.ncommit].astype(np.float32)) % 2
        new_det = (new_det + upd.astype(np.uint8)) % 2
    flagged = new_det.any(axis=1)
    logical = ((obs + np.asarray(total.astype(np.float32) @ _CPU["obsT"].astype(np.float32)) % 2).astype(np.uint8) % 2).any(axis=1)
    return int(flagged.sum()), int(np.logical_or(flagged, logical).sum())


def sample_host(plan, shots, seed):
    from slidingwindowdecoder_b200.sliding_window import sample_dem
    det, obs, _ = sample_dem(plan.chk, plan.obs, plan.priors, shots, np.random.default_rng(seed))
    return det, obs


class CpuArm:
    """Oracle port on all host cores (process-level sharding over shots: the 'all-core' CPU figure of BASELINE.md §3)."""

    def __init__(self, plan, use_ref=False, procs=None):
        import multiprocessing as mp
        self.cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        self.procs = procs or self.cores
        self.plan = plan
        self.pool = mp.get_context("fork").Pool(self.procs, initializer=_cpu_init, initargs=(plan, use_ref, WL.get("_key", "c3_gdg"), WL["p"]))

    def run(self, det, obs):
        B = det.shape[0]
        nshard = min(B, self.procs * 4)
        idx = np.array_split(np.arange(B), nshard)
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_decode_shard, [(det[i], obs[i]) for i in idx if len(i)])
        dt = time.perf_counter() - t0
        return dt, sum(r[0] for r in res), sum(r[1] for r in res)

    def close(self):
        self.pool.close()
        self.pool.join()


def _quiet_stderr():
    """the reference prints "Error setting thread affinity" per thread on hosts with < 15 cores"""
    class _Q:
        def __enter__(self):
            self.devnull = os.open(os.devnull, os.O_WRONLY); self.saved = os.dup(2); os.dup2(self.devnull, 2)
        def __exit__(self, *a):
            os.dup2(self.saved, 2); os.close(self.devnull); os.close(self.saved)
    return _Q()


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _rate(arm, plan, shots, seed):
    det, obs = sample_host(plan, shots, seed)
    dt, fl, fa = arm.run(det, obs)
    return shots / max(dt, 1e-9), dt, fa


def cpu_reference_modes(plan, calib_s=3.0):
    """Which way of running the reference's CPU implementation on this host is fastest ("all the host threads it can use"):
      ref xP  : oracle/_ref = the reference's own bpgd.cpp / mod2sparse.c compiled in place (BPGD_main_thread::do_work, 15
                std::threads per decode, as bpgdg_decoder(multi_thread=True) runs it), P processes over disjoint shot shards
      port    : the C restatement (oracle/swd_oracle.c, gcc -O2), one process per core
    -> (modes: {name: shots/s}, best real-reference (procs, rate) or None, port rate)."""
    from oracle.oracle import ref_lib
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    modes, best = {}, None
    if ref_lib() is not None and WL["decoder"] == "gdg":
        with _quiet_stderr():
            for P in sorted({1, max(1, cores // 8), max(1, cores // 4), max(1, cores // 2), cores}):
                arm = CpuArm(plan, use_ref=True, procs=P)
                r0, _, _ = _rate(arm, plan, max(8, 2 * P), 990 + P)                    # warm-up / first estimate
                r, _, _ = _rate(arm, plan, int(max(4 * P, min(4000, r0 * calib_s))), 995 + P)
                arm.close()
                modes[f"ref_x{P}"] = round(r, 2)
                if best is None or r > best[1]:
                    best = (P, r)
    arm = CpuArm(plan)
    r0, _, _ = _rate(arm, plan, arm.cores * 4, 999)
    rp, _, _ = _rate(arm, plan, int(max(arm.cores * 4, min(20000, r0 * calib_s))), 998)
    arm.close()
    modes["port_per_core"] = round(rp, 2)
    return modes, best, rp, cores


def cpu_baseline_block(plan, target_s):
    """cpu_baseline of the contract: the reference's CPU path on this box's host cores, bounded sample (~target_s of work)."""
    modes, best, rp, cores = cpu_reference_modes(plan)
    if best is not None:
        P, r = best
        n = int(max(1000, min(50000, r * target_s)))
        with _quiet_stderr():
            arm = CpuArm(plan, use_ref=True, procs=P)
            rate, dt, fa = _rate(arm, plan, n, 4321)
            arm.close()
        kind = "reference"
        how = (f"{n} shots x {len(plan.windows)} windows through oracle/_ref (the reference's own bpgd.cpp + mod2sparse.c, g++ -O2; "
               f"do_work with 15 std::threads per decode), {P} process(es) = the fastest of {modes}; {dt:.1f} s; failed {fa}/{n}")
    else:
        arm = CpuArm(plan)
        n = int(max(arm.cores * 4, min(50000, rp * target_s)))
        rate, dt, fa = _rate(arm, plan, n, 4321)
        arm.close()
        kind = "port"
        how = (f"{n} shots x {len(plan.windows)} windows through the oracle port (C restatement of the reference, gcc -O2), one process "
               f"per core; {dt:.1f} s; failed {fa}/{n}" + ("" if WL["decoder"] == "gdg" else " (oracle/_ref binds the GDG path only)"))
    return {"value": round(rate, 2), "unit": "shots/s", "cores": cores, "kind": kind, "sample": how, "modes_shots_per_s": modes,
            "port_per_core_shots_per_s": round(rp, 2), "cpu_model": _cpu_model(), "nproc": os.cpu_count(), "compiler_flags": "-O2 (as the reference's setup.py)"}


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ GPU arm
def gpu_sample(swd, shots, seed):
    """Independent Bernoulli per DEM column drawn on the device (what CompiledDemSampler draws, guessing.py:129-130):
    the repository's own Philox sampler kernel (swd_window_sample), bit-identical to oracle/philox.py."""
    return swd.sample_device(shots, seed=seed)


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(dirname, out):
    """Writes what the timed path (SlidingWindowDecoder.decode_device) returned in its last step as DIR/<name>.npy:
    counts (flagged, failed) and window_unconverged whole, as float64; the residual syndromes and observables it leaves in
    det / obs as float32 rows of a fixed seeded sample of the batch's shots (their indices in sampled_shots.npy), as many as
    keep the files within DUMP_BYTES.  Same arguments, same inputs: two builds can be compared file by file."""
    det, obs = out["residual_det"], out["residual_obs"]
    B = det.shape[0]
    rows = min(B, (DUMP_BYTES - (1 << 20)) // (4 * (det.shape[1] + obs.shape[1]) + 8))
    idx = np.sort(np.random.default_rng(0).choice(B, size=rows, replace=False))
    arrays = {"counts": out["counts"].cpu().numpy().astype(np.float64),
              "window_unconverged": out["window_unconverged"].cpu().numpy().astype(np.float64),
              "sampled_shots": idx.astype(np.float64),
              "residual_det": det.cpu().numpy()[idx].astype(np.float32),
              "residual_obs": obs.cpu().numpy()[idx].astype(np.float32)}
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def config_block(args):
    """The workload the metric is quoted on - the same dict in the product arm and in the reference arm."""
    return {"workload": WL["name"], "shots_per_step_per_gpu": args.batch, "decoder": WL["decoder_name"], "streams": args.streams,
            "inputs": "synthetic DEM samples (independent Bernoulli per DEM column), a distinct batch per step; working set > L2, no L2 flush"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    assert torch.cuda.is_available(), "bench.py needs CUDA (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from slidingwindowdecoder_b200.distributed import reduce_counters, max_over_ranks
    plan = build_plan()
    swd = SlidingWindowDecoder(plan, decoder=WL["decoder"], device=local, streams=args.streams, **WL["kw"])
    B, K, W = args.batch, args.steps, args.warmup
    nsteps = K + W
    torch.backends.cuda.matmul.allow_tf32 = False
    if args.total_shots:
        return run_strong(args, swd, plan, rank, world, dev, dist)
    det_all, obs_all = gpu_sample(swd, B * nsteps, 1234 + rank)
    det_all = det_all.view(nsteps, B, -1); obs_all = obs_all.view(nsteps, B, -1)
    h_det = torch.empty(det_all.shape, dtype=torch.uint8, pin_memory=True); h_det.copy_(det_all)
    h_obs = torch.empty(obs_all.shape, dtype=torch.uint8, pin_memory=True); h_obs.copy_(obs_all)
    h_counts = torch.zeros((nsteps, 2), dtype=torch.int64, pin_memory=True)
    decs = swd.unique_decoders()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    last_step = {}

    def step_resident(i):
        det = det_all[i].clone(); obs = obs_all[i].clone()
        out = swd.decode_device(det, obs)
        if i == W + K - 1:              # the last timed step: what --dump-outputs writes
            last_step.update(out, residual_det=det, residual_obs=obs)
        return out["counts"]

    def step_single_stream(i):          # kernels launched back to back on one stream: clean per-kernel event times
        det = det_all[i].clone(); obs = obs_all[i].clone()
        return swd.decode_device(det, obs, streams=1)["counts"]

    def step_e2e(i):
        # the public host-buffer entry: pinned host syndromes in, python ints (flagged, failed) out - H2D, all windows, D2H
        r = swd.decode(h_det[i], h_obs[i])
        return torch.tensor([r["flagged"], r["failed"]], dtype=torch.int64, device=dev)

    from slidingwindowdecoder_b200.decoders import pack_bits
    wc = (swd.num_col + 63) // 64
    h_detp = torch.from_numpy(pack_bits(h_det.view(-1, h_det.shape[2]).numpy()).view(np.int64)).view(nsteps, B, -1).pin_memory()
    h_obsp = torch.from_numpy(pack_bits(h_obs.view(-1, h_obs.shape[2]).numpy()).view(np.int64)).view(nsteps, B, -1).pin_memory()
    h_corrp = torch.empty((B, wc), dtype=torch.int64, pin_memory=True)

    def step_e2e_corr(i):
        # bit-packed host buffers in, bit-packed corrections (total_e_hat) + counts back to the host
        r = swd.decode_packed(h_detp[i], h_obsp[i], return_corrections=True, pinned_out=h_corrp)
        return torch.tensor([r["flagged"], r["failed"]], dtype=torch.int64, device=dev)

    def timed(fn, profile, K=K):
        for i in range(W):
            fn(i)
        for d in decs:
            d.kernel_times() if profile else None
            d.reset_counters()
            d.set_profiling(profile)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        e0.record()
        for i in range(W, W + K):
            counts += fn(i)
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1), dev)                # device time, max over ranks
        counts = reduce_counters(counts, dev)                        # the path's only collective: failure counters
        return ms, np.array(counts)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    def read_counters():
        out = {}
        for d in decs:
            for k, v in d.counters().items():
                out[k] = out.get(k, 0) + v
        return out

    ms_res, counts_res = timed(step_resident, False)
    ctr_timed = read_counters()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_step)
    last_step.clear()
    ms_e2e, counts_e2e = timed(step_e2e, False)
    ms_e2ec, counts_e2ec = timed(step_e2e_corr, False)
    assert np.array_equal(counts_e2e, counts_res) and np.array_equal(counts_e2ec, counts_res), "e2e legs disagree with the resident leg"
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel CUDA-event times + work counters for the roofline: same batches, one stream (with several streams
    # the kernels of different sub-batches overlap and their individual durations are not additive)
    Kp = min(K, 4)
    ms_prof, _ = timed(step_single_stream, True, K=Kp)
    ktimes = {}
    for d in decs:
        for k, (t, ln) in d.kernel_times().items():
            a = ktimes.setdefault(k, [0.0, 0]); a[0] += t; a[1] += ln
        d.set_profiling(False)
    ctr = read_counters()

    # per-window latency (p50) at the throughput batch and at batch 1
    def window_latency(batch, reps):
        lat = []
        for r in range(reps):
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in plan.windows]
            det = det_all[r % nsteps][:batch].clone(); obs = obs_all[r % nsteps][:batch].clone()
            swd.decode_device(det, obs, window_events=ev)
            torch.cuda.synchronize()
            lat += [a.elapsed_time(b) for a, b in ev]
        return float(np.median(lat)), float(np.percentile(lat, 99))
    p50_b, p99_b = window_latency(B, 2)
    p50_1, p99_1 = window_latency(1, 20)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    total_shots = world * B * K
    value = total_shots / (ms_res / 1e3)
    e2e = total_shots / (ms_e2e / 1e3)
    # ---- roofline (VERDICT r1 #2): every message-passing kernel against the roof that binds it, peaks MEASURED on this
    # pool's B200s: HBM copy bandwidth from MEASURED_PEAKS.json (driver-written), shared-memory LDS.64+STS.64 streaming
    # and issue rate from profiles/onchip_peaks.json (tools/onchip_peak.cu at the path kernel's launch shape).
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak = float(json.load(open(peaks_path))["hbm_gbs"]); hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        hbm_peak = 6650.0; hbm_src = "fallback (B200_PROFILING.md)"
    onchip = {}
    op = os.path.join(ROOT, "profiles", "onchip_peaks.json")
    if os.path.exists(op):
        onchip = json.load(open(op))
    shapes = {sh["threads"]: sh for sh in onchip.get("shapes", [])}
    small, large = shapes.get(128, {}), shapes.get(1024, {})
    smem_peak = float(small.get("smem_ld64_st64_gbs", 148 * 128 * 1.965))
    smem_src = "measured (profiles/onchip_peaks.json: conflict-free LDS.64 + STS.64, 128-thread CTAs x 8 per SM)" if small else \
               "datasheet (148 SMs x 128 B/clk x 1.965 GHz) - profiles/onchip_peaks.json missing"
    issue_peak = float(small.get("issue_gwarp_inst_per_s", 148 * 4 * 1.965))
    gdg = WL["decoder"] == "gdg"
    n_win = len(plan.windows)
    streamed = any(d.streamed_bp for d in decs)
    kernel_ms = {k: round(v[0], 3) for k, v in ktimes.items() if v[1]}
    tot_k = sum(kernel_ms.values()) or 1.0

    def kt(*keys):
        return sum(ktimes.get(k, [0, 0])[0] for k in keys), sum(ktimes.get(k, [0, 0])[1] for k in keys)

    def block(name, bound, bytes_, ms, launches, peak, peak_src, extra=None):
        ach = bytes_ / (ms / 1e3) / 1e9 if ms > 0 else 0.0
        out = {"kernel": name, "bound": bound, "achieved": round(ach, 1), "peak": round(peak, 1), "unit": "GB/s",
               "frac": round(ach / peak, 4) if peak else None, "peak_source": peak_src,
               "algorithmic_bytes_per_launch": round(bytes_ / max(1, launches)), "avg_launch_ms": round(ms / max(1, launches), 4),
               "launches": launches, "share_of_kernel_time": round(ms / tot_k, 4)}
        out.update(extra or {})
        return out

    # B_iter = 4 E w + 2 n_a w + (n_a + m_a)/8 with w = 8 (SURVEY.md 8(d)), summed over executed iterations (device counters)
    path_bytes = 32.0 * ctr["path_edge_iters"] + 16.0 * ctr["path_vn_iters"] + (ctr["path_vn_iters"] + ctr["path_cn_iters"]) / 8.0
    path_ms, path_launches = kt("path_main", "path_side", "path_trunk") if gdg else kt("post_bp")
    blocks = {}
    live_slots = ctr["path_edge_iters"] / max(1, ctr.get("path_slot_iters", 0)) if ctr.get("path_slot_iters") else None
    blocks["path" if gdg else "post_bp"] = block(
        "path_kernel (GDG branch paths: shared-prefix nodes + main/tree + side launches)" if gdg else
        "post_bp_kernel (masked min-sum on the shortened graph)", "smem", path_bytes, path_ms, path_launches, smem_peak, smem_src,
        {"hbm_equivalent_frac": round(path_bytes / (path_ms / 1e3) / 1e9 / hbm_peak, 4) if path_ms else None,
         "live_slot_fraction": round(live_slots, 4) if live_slots else None,
         "note": "messages live in shared memory: algorithmic message bytes/s against the measured shared-memory streaming roof; "
                 "hbm_equivalent_frac > 1 would be impossible for an HBM-streaming design; live_slot_fraction = active edges / "
                 "message slots scanned by the check passes (the rest are decided-VN and pad slots)"})
    pre_ms, pre_l = kt("pre_bp")
    n_cols = float(np.mean([w.mat.shape[1] for w in plan.windows])); nnz_w = float(np.mean([w.mat.nnz for w in plan.windows]))
    if streamed:
        pre_bytes = ctr["pre_bp_edge_iters"] * (32.0 + 8.0 * n_cols / nnz_w)       # + one posterior per column and iteration
        blocks["pre_bp"] = block("pre_bp_stream_kernel (HBM-streamed full-window min-sum, one thread per shot)", "hbm", pre_bytes, pre_ms,
                                 pre_l, hbm_peak, hbm_src,
                                 {"note": "32 B x edges x iterations (read + write in both passes) + 8 B x columns x iterations of posterior "
                                          "history: what the kernel moves through HBM by construction"})
    else:
        pre_bytes = 32.0 * ctr["pre_bp_edge_iters"]
        blocks["pre_bp"] = block("pre_bp_kernel (full-window min-sum, messages in shared memory)", "smem", pre_bytes, pre_ms, pre_l, smem_peak, smem_src)
    if not gdg:
        osd_ms, osd_l = kt("osd")
        mrows = float(np.mean([w.mat.shape[0] for w in plan.windows])); w64 = math.ceil(mrows / 64)
        dbar = nnz_w / n_cols
        # GF(2) elimination: every scanned column gathers its <= 6 rows of T (W64 words each); every pivot is folded into
        # all m + 1 columns of T (read + write)
        osd_bytes = 8.0 * w64 * (ctr.get("osd_cols_scanned", 0) * dbar + 2.0 * ctr.get("osd_pivots", 0) * (mrows + 1))
        blocks["osd"] = block("osd_kernel (bit-packed GF(2) Gauss-Jordan + OSD-CS candidates)", "smem", osd_bytes, osd_ms, osd_l,
                              float(large.get("smem_ld64_st64_gbs", smem_peak)), smem_src.replace("128-thread CTAs x 8", "one 1024-thread CTA"))
    dom = max(blocks, key=lambda k: blocks[k]["share_of_kernel_time"])
    traffic, traffic_src, ncu_facts = None, None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath)).get({"path": "path_kernel", "post_bp": "osd_pipeline", "pre_bp": "pre_bp_" + args.workload, "osd": "osd_kernel"}[dom], {})
        if tj.get("batch") == B and tj.get("workload", "c3_gdg") == args.workload:   # the capture was taken on this workload at this batch size
            traffic = int(tj["dram_bytes_per_launch_avg"]); traffic_src = tj.get("source"); ncu_facts = tj.get("ncu")
    roofline = dict(blocks[dom])
    roofline.update({"traffic": traffic, "traffic_source": traffic_src, "ncu": ncu_facts,
                     "issue_peak_gwarp_inst_per_s": round(issue_peak, 1),
                     "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
                     "kernels": {k: v for k, v in blocks.items() if k != dom},
                     "kernel_ms": kernel_ms, "kernel_ms_steps": Kp, "single_stream_ms_per_step": round(ms_prof / Kp, 3)})
    # minimal-I/O figure (SURVEY.md 8(d)): a design that keeps everything else on chip moves (m + n) / 8 + 1 bytes per shot-window
    # (bit-packed syndrome in, correction + converge flag out) through HBM
    mio = float(np.mean([(w.mat.shape[0] + w.mat.shape[1]) / 8.0 + 1.0 for w in plan.windows]))
    roofline["minimal_io"] = {"bytes_per_shot_window": round(mio, 1),
                              "gbs_at_value": round(value / world * n_win * mio / 1e9, 4),
                              "frac_of_hbm_peak": round(value / world * n_win * mio / 1e9 / hbm_peak, 6)}
    # ---- CPU baseline on a bounded sample (rank 0, at every N)
    cpu_baseline = None if args.skip_cpu else cpu_baseline_block(plan, 12.0)
    launches = ctr_timed["kernel_launches"] + K * args.streams * (2 * len(plan.windows) + 1)
    line = {
        "metric": METRIC[WL["decoder"]], "value": round(value, 1), "unit": "shots/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": round(ms_res / K, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_block(args),
        "inputs": "DEM samples drawn on the device (Philox, independent Bernoulli per column); distinct batch per step, "
                  f"{(B * (det_all.shape[2] + obs_all.shape[2]) * nsteps) >> 20} MiB of syndromes in total (> L2), no L2 flush",
        "e2e": {"value": round(e2e, 1), "unit": "shots/s", "h2d_bytes_per_step": int(B * (det_all.shape[2] + obs_all.shape[2])),
                "d2h_bytes_per_step": 16 + 8 * n_win, "ms_per_step": round(ms_e2e / K, 3),
                "api": "SlidingWindowDecoder.decode(pinned host det, obs) -> flagged / failed counts (one byte per bit in)"},
        "e2e_corrections": {"value": round(total_shots / (ms_e2ec / 1e3), 1), "unit": "shots/s",
                            "h2d_bytes_per_step": int(8 * B * (h_detp.shape[2] + h_obsp.shape[2])),
                            "d2h_bytes_per_step": int(8 * B * wc) + 16 + 8 * n_win, "ms_per_step": round(ms_e2ec / K, 3),
                            "api": "SlidingWindowDecoder.decode_packed(bit-packed host det, obs) -> bit-packed total_e_hat + counts"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
        "window_latency_ms": {"p50_at_batch": round(p50_b, 4), "p99_at_batch": round(p99_b, 4), "p50_batch1": round(p50_1, 4), "p99_batch1": round(p99_1, 4)},
        "results": {"shots": int(total_shots), "flagged": int(counts_res[0]), "failed": int(counts_res[1]),
                    "gdg_fraction": round(ctr["gdg_shots"] / max(1, ctr["shots"]), 4)},
        "counters": ctr_timed,
        # the min-sum work counters (edge / VN / CN / slot iterations) only accumulate while profiling is on (counting them costs
        # 1.7 % of the shots/s): these are the ones of the `kernel_ms_steps` profiled single-stream steps the roofline is computed from
        "work_counters_profiled_steps": {k: int(ctr[k]) for k in ("shots", "gdg_shots", "paths_run", "bp_calls", "path_edge_iters", "path_vn_iters",
                                                                   "path_cn_iters", "path_slot_iters", "pre_bp_edge_iters") if k in ctr},
    }
    print(json.dumps(line), file=_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_strong(args, swd, plan, rank, world, dev, dist):
    """BASELINE configs[2] as written: ONE fixed job of --total-shots shots (10^7) sharded over the ranks with shard_range,
    every shot drawn on the device (Philox counter = global shot index: the job's syndromes do not depend on the number of
    GPUs) and decoded through all windows; sampling is inside the clock.  Strong scaling: the line reports wall seconds."""
    import torch
    from slidingwindowdecoder_b200.distributed import shard_range, reduce_counters, max_over_ranks
    total, B = int(args.total_shots), args.batch
    lo, hi = shard_range(total, rank, world)

    def job(limit=None):
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        s0 = lo
        end = hi if limit is None else min(hi, lo + limit)
        while s0 < end:
            nb = min(B, end - s0)
            det, obs = swd.sample_device(nb, seed=20261017, shot_offset=s0)
            counts += swd.decode_device(det, obs)["counts"]
            s0 += nb
        return counts

    job(limit=2 * B)                                        # warm-up: workspaces, lazy module loads
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier(); torch.cuda.synchronize()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", 0)))
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    counts = job()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier(); torch.cuda.synchronize()
    wall = max_over_ranks(time.perf_counter() - t0, dev)
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    counts = reduce_counters(counts, dev)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        line = {"metric": METRIC[WL["decoder"]], "value": round(total / (ms / 1e3), 1), "unit": "shots/s", "n_gpus": world, "steps": 1, "warmup": 1,
                "ms_per_step": round(ms, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": dict(config_block(args), total_shots=total),
                "job": {"total_shots": total, "seconds_device_max_over_ranks": round(ms / 1e3, 3), "seconds_wall_max_over_ranks": round(wall, 3),
                        "includes": "on-device DEM sampling (Philox) + all windows + counter reduction; shots sharded with shard_range, no data-path collective"},
                "results": {"shots": total, "flagged": int(counts[0]), "failed": int(counts[1])}, "clocks": clocks}
        print(json.dumps(line), file=_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    """The reference's own CPU implementation of the path on this box's host cores, same metric / config / steps contract.
    Each step is a bounded sample of the workload (the CPU needs minutes for what the GPU does per step): shots per step are
    sized so that warm-up + steps finish in ~90 s; throughput = shots / time over the timed steps."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    plan = build_plan()
    modes, best, rp, cores = cpu_reference_modes(plan, calib_s=min(3.0, args.ref_seconds / 10.0))
    K, W = max(1, args.steps), max(0, args.warmup)
    use_ref = best is not None
    P, rate0 = (best if use_ref else (None, rp))
    nsample = int(max(4 * (P or cores), min(20000, rate0 * args.ref_seconds / (K + W))))
    times, fails, n = [], 0, 0
    with _quiet_stderr():
        arm = CpuArm(plan, use_ref=use_ref, procs=P)
        for i in range(W + K):
            det, obs = sample_host(plan, nsample, 100 + i)
            dt, fl, fa = arm.run(det, obs)
            if i >= W:
                times.append(dt); fails += fa; n += nsample
        arm.close()
    v = n / sum(times)
    how = (f"{nsample} shots x {len(plan.windows)} windows per step through oracle/_ref (the reference's own bpgd.cpp + mod2sparse.c, "
           f"g++ -O2; do_work with 15 std::threads per decode), {P} process(es) = the fastest of {modes}") if use_ref else \
          (f"{nsample} shots x {len(plan.windows)} windows per step through the oracle port (C restatement, gcc -O2), one process per core"
           + ("" if WL["decoder"] == "gdg" else " (oracle/_ref binds the GDG path only)"))
    line = {"impl": "reference", "metric": METRIC[WL["decoder"]], "value": round(v, 2), "unit": "shots/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": K, "warmup": W, "ms_per_step": round(1e3 * sum(times) / K, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(args), "sample_shots_per_step": nsample,
            "cpu_baseline": {"value": round(v, 2), "unit": "shots/s", "cores": cores, "kind": "reference" if use_ref else "port", "sample": how,
                             "modes_shots_per_s": modes, "port_per_core_shots_per_s": round(rp, 2), "cpu_model": _cpu_model(),
                             "nproc": os.cpu_count(), "compiler_flags": "-O2 (as the reference's setup.py)"},
            "e2e": {"value": round(v, 2), "unit": "shots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "results": {"shots": n, "failed": fails}}
    print(json.dumps(line), file=_STDOUT, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3_gdg", choices=sorted(WORKLOADS), help="default: BASELINE.json configs[2], the metric's configuration")
    ap.add_argument("--streams", type=int, default=3, help="concurrent sub-batches per GPU (fills kernel tails)")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs only: do not time the CPU baseline")
    ap.add_argument("--p", type=float, default=None, help="override the workload's physical error rate (BASELINE configs[4]: p sweep 1e-3 .. 5e-3)")
    ap.add_argument("--total-shots", type=int, default=0, help="strong scaling: decode ONE job of this many shots (configs[2]: 10000000), sharded over the GPUs; "
                                                            "sampling inside the clock; prints wall seconds")
    ap.add_argument("--ref-seconds", type=float, default=90.0, help="--impl reference: CPU seconds spent on warm-up + timed steps together")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.total_shots):
        ap.error("--dump-outputs writes the outputs of the timed steps of --impl ours; it does not apply to --impl reference or --total-shots")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    # the contract is ONE JSON line on stdout: libraries that write to fd 1 themselves (NCCL prints its version banner
    # there) are sent to stderr, the line itself goes to the saved descriptor
    global _STDOUT
    sys.stdout.flush()
    _STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    select_workload(args.workload, args.p)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
