"""Cost and use of per-shot channel priors for bp4_osd (device-resident shot data, one GPU).

Workloads: the [[72,12,6]] pair and kwargs of the c1_bp4_osd_cs8 fixture through decode_batch (BP4 + OSD-CS8 per basis), and the
CAMEL-shaped pair (all-ones last column) of c1_bp4_camel_tied through camel_decode_batch.  Every call decodes --shots torch CUDA
shots through the device-pointer entry points (swd_bp4_*_device[_llr]) and is timed with CUDA events after a warm-up; the
modes alternate call by call in one process:
  (a) a_static       no channel_llr: the static priors (swd_bp4_decode_batch_device / swd_bp4_camel_decode_batch_device);
  (b) b_static_rows  [5, B, n] rows equal to the static priors (the per-shot kernels; asserted to give (a)'s outputs exactly);
  (c) c_erasure_rows 5 % of the qubits of every shot erased - the erased qubit carries a uniformly random Pauli in the sampled
                     error, and all five of its LLRs are 0.0 in the rows;
  (c0) c_static      the syndromes of (c) decoded with the static priors, i.e. without using the erasure information.
For (c) and (c0) the line also gives the logical failures: the residual e + e_hat anticommutes with a logical of
codes.bb_code(72) (lz against the x part, lx against the z part), or does not reproduce the syndrome.  On the CAMEL pair a
residual on the tying column counts as a failure too.  The card's name and power limit are read in the same run.

    python tools/bench_bp4_per_shot_llr.py [--shots 65536] [--calls 5] [--warmup 2] [--out FILE.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

WORKLOADS = (("c1_bp4_osd_cs8", "decode"), ("c1_bp4_camel_tied", "camel_decode"))
ERASE = 0.05


def sample(g, B, rng, erase):
    """Depolarizing errors from the fixture's px / py / pz; qubits in the erasure mask get a uniformly random Pauli instead.
    -> (erased [B, n] bool, ex, ez [B, n] int64, synd_x, synd_z uint8)"""
    n = g["hx"].shape[1]
    px, py, pz = (np.broadcast_to(g[k], (B, n)).copy() for k in ("px", "py", "pz"))
    er = rng.random((B, n)) < erase
    px[er] = py[er] = pz[er] = 0.25
    r = rng.random((B, n))
    isx, isy, isz = r < px, (r >= px) & (r < px + py), (r >= px + py) & (r < px + py + pz)
    ex, ez = (isx | isy).astype(np.int64), (isy | isz).astype(np.int64)
    hx, hz = np.asarray(g["hx"].todense()).astype(np.int64), np.asarray(g["hz"].todense()).astype(np.int64)
    return er, ex, ez, (ez @ hx.T % 2).astype(np.uint8), (ex @ hz.T % 2).astype(np.uint8)


def logical_failures(g, dec, ex, ez, sx, sz):
    """Shots whose residual is not a stabilizer of the [[72,12,6]] code (see the module docstring)."""
    from slidingwindowdecoder_b200.codes import bb_code
    code, _, _ = bb_code(72)
    hx, hz = np.asarray(g["hx"].todense()).astype(np.int64), np.asarray(g["hz"].todense()).astype(np.int64)
    rx, rz = ex ^ dec[:, 0].astype(np.int64), ez ^ dec[:, 1].astype(np.int64)
    bad = ((rz @ hx.T) % 2).any(axis=1) | ((rx @ hz.T) % 2).any(axis=1)
    if rx.shape[1] > code.N:                                                   # the CAMEL pair's tying column
        bad |= (rx[:, code.N:] | rz[:, code.N:]).any(axis=1)
        rx, rz = rx[:, :code.N], rz[:, :code.N]
    bad |= ((rx @ code.lz.T) % 2).any(axis=1) | ((rz @ code.lx.T) % 2).any(axis=1)
    return int(bad.sum())


def run_workload(name, method, args, info):
    import torch
    from conftest import load_golden_bp4
    from slidingwindowdecoder_b200 import bp4_osd
    g = load_golden_bp4(name)
    dec = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **g["kwargs"])
    fn = dec.decode_batch if method == "decode" else dec.camel_decode_batch
    B, n = args.shots, dec.n
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(2024)
    _, ex0, ez0, sx0, sz0 = sample(g, B, rng, 0.0)
    er, ex1, ez1, sx1, sz1 = sample(g, B, rng, ERASE)
    L_static = np.ascontiguousarray(np.repeat(dec.channel_llr[:, None, :], B, axis=1))
    L_erase = L_static.copy()
    L_erase[:, er] = 0.0
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)          # noqa: E731
    tx0, tz0, tx1, tz1, tL_static, tL_erase = (to(a) for a in (sx0, sz0, sx1, sz1, L_static, L_erase))
    modes = {"a_static": (tx0, tz0, None), "b_static_rows": (tx0, tz0, tL_static),
             "c_erasure_rows": (tx1, tz1, tL_erase), "c_static": (tx1, tz1, None)}
    # (a) and (b) give identical outputs, checked outside the timed calls
    oa, ob = fn(tx0, tz0), fn(tx0, tz0, channel_llr=tL_static)
    torch.cuda.synchronize()
    for k in oa:
        assert torch.equal(oa[k], ob[k]), f"{name}: mode (a) and (b) differ in {k}"
    del oa, ob
    times = {m: [] for m in modes}
    last = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(args.warmup + args.calls):
        for m, (tx, tz, L) in modes.items():
            torch.cuda.synchronize()
            e0.record()
            out = fn(tx, tz, channel_llr=L)
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                times[m].append(e0.elapsed_time(e1) / 1e3)
            last[m] = out
    base = B * args.calls / sum(times["a_static"])
    lines = []
    for m in modes:
        rate = B * args.calls / sum(times[m])
        d = last[m]["dec"].cpu().numpy()
        line = dict(workload=name, method=f"bp4_osd.{method}_batch", mode=m, n=int(n), kwargs=g["kwargs"], shots=B,
                    shots_per_s=round(rate, 1), vs_static=round(rate / base, 4), ms_per_call=round(1e3 * sum(times[m]) / args.calls, 3),
                    calls=args.calls, warmup=args.warmup, converged=round(float(last[m]["converge"].float().mean()), 6))
        if m.startswith("c_"):
            line.update(erased_fraction=round(float(er.mean()), 6),
                        logical_failures=logical_failures(g, d, ex1, ez1, sx1, sz1))
        else:
            line.update(logical_failures=logical_failures(g, d, ex0, ez0, sx0, sz0))
        line.update(info)
        lines.append(line)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shots", type=int, default=65536)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    from bench_per_shot_llr import card_info
    info = card_info()
    out = open(args.out, "a") if args.out else None
    for name, method in WORKLOADS:
        for line in run_workload(name, method, args, info):
            s = json.dumps(line)
            print(s, flush=True)
            if out:
                out.write(s + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
