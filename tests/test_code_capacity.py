"""Code-capacity simulation on the device: swd_window_sample_pauli against its numpy restatement (tests/pauli_oracle.py::sample_pauli)
bit for bit, the per-shot LLR planes against bp4_osd.channel_llr, commit + count against numpy, and
depolarizing_noise_decoding against the same pipeline run on the host."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden_bp4

pytestmark = pytest.mark.gpu

CS8 = dict(max_iter=24, ms_scaling_factor=0.9, osd_method="osd_cs", osd_order=8)     # the c1_bp4_osd_cs8 fixture's kwargs


def _bb72():
    from slidingwindowdecoder_b200.codes import bb_code
    return bb_code(72)[0]


def _case(name, rng):
    """-> (Hx, Hz, lx, lz, px, py, pz, llr5 or None): the pairs and channels the sampler is checked on."""
    from slidingwindowdecoder_b200 import bp4_osd
    if name == "bb72_uniform":
        code = _bb72()
        p = np.full(code.N, 0.05 / 3)
        llr5 = bp4_osd(code.hx, code.hz, channel_probs_x=p, channel_probs_y=p, channel_probs_z=p).channel_llr
        return code.hx, code.hz, code.lx, code.lz, p, p, p, llr5
    if name == "bb72_nonuniform":
        code = _bb72()
        n = code.N
        px, py, pz = (rng.uniform(0.0, 0.2, n) for _ in range(3))
        py[rng.random(n) < 0.3] = 0.0
        zero = rng.random(n) < 0.15
        px[zero] = py[zero] = pz[zero] = 0.0
        px[0], py[0], pz[0] = 0.5, 0.25, 0.25                                 # px + py + pz = 1 exactly
        return code.hx, code.hz, code.lx, code.lz, px, py, pz, rng.normal(size=(5, n))
    if name == "camel_tied":                                                   # n = 73; unit rows on the tying column
        g = load_golden_bp4("c1_bp4_camel_tied")
        code = _bb72()
        tie = np.zeros((1, 73), dtype=np.int64); tie[0, 72] = 1
        lx = np.vstack([np.hstack([code.lx, np.zeros((code.K, 1), dtype=np.int64)]), tie])
        lz = np.vstack([np.hstack([code.lz, np.zeros((code.K, 1), dtype=np.int64)]), tie])
        llr5 = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"]).channel_llr
        return g["hx"], g["hz"], lx, lz, g["px"], g["py"], g["pz"], llr5
    assert name == "random_sparse"                                             # mx + mz = 77 > 64 detectors, odd n
    n = 51
    hx, hz = ((rng.random((m, n)) < 0.08).astype(np.int64) for m in (40, 37))
    lx, lz = ((rng.random((k, n)) < 0.2).astype(np.int64) for k in (5, 3))
    p = rng.uniform(0.0, 0.3, (3, n))
    return hx, hz, lx, lz, p[0], p[1], p[2], rng.normal(size=(5, n))


CASES = ("bb72_uniform", "bb72_nonuniform", "camel_tied", "random_sparse")
SEEDS = ((0, 0), ((0xDEADBEEF << 32) | 12345, (1 << 32) + 77))                 # (seed, shot_offset)


def _sampler(case, rate, rng=None):
    from slidingwindowdecoder_b200 import CodeCapacitySampler
    hx, hz, lx, lz, px, py, pz, llr5 = _case(case, rng if rng is not None else np.random.default_rng(5))
    s = CodeCapacitySampler(hx, hz, lx, lz, px, py, pz, erasure_rate=rate, channel_llr=llr5)
    return s, (px, py, pz, llr5)


def _host(t):
    return t.cpu().numpy()


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("rate", (0.0, 0.05, 1.0))
def test_sampler_bit_exact(case, rate):
    import torch
    from pauli_oracle import sample_pauli
    s, (px, py, pz, llr5) = _sampler(case, rate)
    B = 2999
    for seed, off in SEEDS:
        out = s.sample(B, seed=seed, shot_offset=off, return_errors=True, return_erasures=True, return_llr=True)
        det, ob, err, erased, L = sample_pauli(s.chk, s.obs, px, py, pz, rate, B, seed=seed, shot_offset=off, llr5=llr5)
        assert np.array_equal(_host(out["det"]), det) and np.array_equal(_host(out["obs"]), ob)
        assert np.array_equal(_host(out["err"]).reshape(B, -1), err)
        assert np.array_equal(_host(out["erased"]), erased)
        assert np.array_equal(_host(out["channel_llr"]).view(np.uint64), L.view(np.uint64))
        assert np.array_equal(_host(out["synd_x"]), det[:, :s.mx]) and np.array_equal(_host(out["synd_z"]), det[:, s.mx:])
        assert out["synd_x"].is_contiguous() and out["synd_z"].is_contiguous()
        if rate == 1.0:
            assert erased.mean() > 0.999
        # the optional outputs do not change det / obs
        bare = s.sample(B, seed=seed, shot_offset=off)
        assert torch.equal(bare["det"], out["det"]) and torch.equal(bare["obs"], out["obs"])
        # shot b at offset o is shot 0 at offset o + b
        for b in (0, 1, 17, B - 1):
            one = s.sample(1, seed=seed, shot_offset=off + b, return_errors=True)
            assert torch.equal(one["det"][0], out["det"][b]) and torch.equal(one["err"][0], out["err"][b])


def test_sampler_grid_stride_and_empty():
    """More shots than one grid holds (the kernel loops over shots), and B == 0."""
    from pauli_oracle import sample_pauli
    s, (px, py, pz, llr5) = _sampler("bb72_uniform", 0.05)
    B, seed, off = 40001, 99, (5 << 32) + 3
    out = s.sample(B, seed=seed, shot_offset=off, return_errors=True, return_erasures=True, return_llr=True)
    det, ob, err, erased, L = sample_pauli(s.chk, s.obs, px, py, pz, 0.05, B, seed=seed, shot_offset=off, llr5=llr5)
    assert np.array_equal(_host(out["det"]), det) and np.array_equal(_host(out["obs"]), ob)
    assert np.array_equal(_host(out["err"]).reshape(B, -1), err) and np.array_equal(_host(out["erased"]), erased)
    assert np.array_equal(_host(out["channel_llr"]), L)
    empty = s.sample(0, return_errors=True, return_erasures=True, return_llr=True)
    assert empty["det"].shape == (0, s.num_det) and empty["channel_llr"].shape == (5, 0, s.n)


def test_llr_planes_are_bp4_rows():
    from slidingwindowdecoder_b200 import CodeCapacitySampler, bp4_osd
    g = load_golden_bp4("c1_bp4_osd_cs8")
    code = _bb72()
    dec = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **g["kwargs"])
    s = CodeCapacitySampler(g["hx"], g["hz"], code.lx, code.lz, g["px"], g["py"], g["pz"], erasure_rate=0.05,
                            channel_llr=dec.channel_llr)
    out = s.sample(4096, seed=3, return_erasures=True, return_llr=True)
    L, er = _host(out["channel_llr"]), _host(out["erased"]).astype(bool)
    assert 0.03 < er.mean() < 0.07
    rows = np.broadcast_to(dec.channel_llr[:, None, :], L.shape)
    assert np.array_equal(L.view(np.uint64)[:, ~er], rows.view(np.uint64)[:, ~er])
    assert (L.view(np.uint64)[:, er] == 0).all()                             # +0.0 in all five planes


def _numpy_counts(s, err, dec):
    r = err.reshape(err.shape[0], -1).astype(np.int64) ^ dec.reshape(dec.shape[0], -1).astype(np.int64)
    flagged = (np.asarray(s.chk @ r.T).T % 2).any(axis=1)
    failed = flagged | (np.asarray(s.obs @ r.T).T % 2).any(axis=1)
    return int(flagged.sum()), int(failed.sum())


def test_commit_and_count():
    import torch
    from slidingwindowdecoder_b200 import bp4_osd
    s, (px, py, pz, llr5) = _sampler("bb72_uniform", 0.05)
    code = _bb72()
    n = code.N
    dec = bp4_osd(code.hx, code.hz, channel_probs_x=px, channel_probs_y=py, channel_probs_z=pz, **CS8)
    for rate_seed in (1, 2):
        out = s.sample(3000, seed=rate_seed, return_errors=True, return_llr=True)
        for L in (None, out["channel_llr"]):
            d = dec.decode_batch(out["synd_x"], out["synd_z"], channel_llr=L)["dec"]
            det, obs = out["det"].clone(), out["obs"].clone()
            got = s.count_failures(d, det, obs)
            assert got.dtype == torch.int64 and got.shape == (2,)
            assert tuple(got.tolist()) == _numpy_counts(s, _host(out["err"]), _host(d))
            assert 0 < got[1] < 3000
    # crafted residuals: decoded = residual against a zero syndrome
    zero_det = lambda B: torch.zeros((B, s.num_det), dtype=torch.uint8, device="cuda")   # noqa: E731
    zero_obs = lambda B: torch.zeros((B, s.num_obs), dtype=torch.uint8, device="cuda")   # noqa: E731
    stab, logical, single = np.zeros((3, 2, 2, n), dtype=np.uint8)
    stab[0, 0] = code.hx[0]; stab[1, 1] = code.hz[5]                           # X stabilizer in the x part, Z in the z part
    logical[0, 0] = code.lx[0]; logical[1, 1] = code.lz[3]
    single[0, 0, 4] = 1; single[1, 1, 9] = 1
    for res, want in ((stab, (0, 0)), (logical, (0, 2)), (single, (2, 2))):
        got = s.count_failures(torch.from_numpy(res).cuda(), zero_det(2), zero_obs(2))
        assert tuple(got.tolist()) == want, (res, want)
        assert _numpy_counts(s, np.zeros((2, 2 * n), dtype=np.uint8), res) == want


def _host_pipeline(code, p, shots, rate, seed, offset, kwargs):
    from pauli_oracle import sample_pauli
    from slidingwindowdecoder_b200 import CodeCapacitySampler, bp4_osd
    n = code.N
    pr = np.full(n, p / 3)
    dec = bp4_osd(code.hx, code.hz, channel_probs_x=pr, channel_probs_y=pr, channel_probs_z=pr, **kwargs)
    s = CodeCapacitySampler(code.hx, code.hz, code.lx, code.lz, pr, pr, pr, erasure_rate=rate, channel_llr=dec.channel_llr)
    det, _, err, erased, L = sample_pauli(s.chk, s.obs, pr, pr, pr, rate, shots, seed=seed, shot_offset=offset, llr5=dec.channel_llr)
    sx, sz = np.ascontiguousarray(det[:, :s.mx]), np.ascontiguousarray(det[:, s.mx:])
    legs = {}
    for leg, planes in (("static", None), ("erasure_aware", L)):
        out = dec.decode_batch(sx, sz, channel_llr=planes)
        flagged, failed = _numpy_counts(s, err, out["dec"])
        legs[leg] = dict(num_flagged=flagged, num_logical=failed, num_bp_unconverged=int((out["converge"] == 0).sum()))
    return legs, float(erased.mean())


def _counts(res):
    return {k: {f: v[f] for f in ("num_flagged", "num_logical", "num_bp_unconverged")} for k, v in res.items() if isinstance(v, dict)}


def test_driver_matches_host_pipeline():
    from slidingwindowdecoder_b200 import depolarizing_noise_decoding
    code = _bb72()
    res = depolarizing_noise_decoding(code, 0.05, num_shots=5000, erasure_rate=0.05, seed=21, verbose=False, **CS8)
    ref, frac = _host_pipeline(code, 0.05, 5000, 0.05, 21, 0, CS8)
    assert _counts(res) == ref
    assert res["erased_fraction"] == pytest.approx(frac, abs=1e-12)
    for leg in ("static", "erasure_aware"):
        assert res[leg]["ler"] == res[leg]["num_logical"] / 5000
    assert 0 < res["static"]["num_logical"] < 5000
    no_erasure = depolarizing_noise_decoding(code, 0.05, num_shots=500, seed=21, verbose=False, **CS8)
    assert set(no_erasure) == {"static", "erased_fraction", "elapsed"} and no_erasure["erased_fraction"] == 0.0


def test_driver_batch_and_shard_independence():
    from slidingwindowdecoder_b200 import depolarizing_noise_decoding
    from slidingwindowdecoder_b200.distributed import shard_range
    code = _bb72()
    kw = dict(erasure_rate=0.05, seed=(1 << 40) + 3, verbose=False, **CS8)
    runs = [_counts(depolarizing_noise_decoding(code, 0.06, num_shots=5000, batch=b, **kw)) for b in (1000, 4096, 5000)]
    assert runs[0] == runs[1] == runs[2]
    parts = [_counts(depolarizing_noise_decoding(code, 0.06, num_shots=hi - lo, shot_offset=lo, **kw))
             for lo, hi in (shard_range(5000, r, 2) for r in range(2))]
    for leg in runs[0]:
        for f in runs[0][leg]:
            assert parts[0][leg][f] + parts[1][leg][f] == runs[0][leg][f], (leg, f)


def test_erasure_information_helps():
    from slidingwindowdecoder_b200 import depolarizing_noise_decoding
    res = depolarizing_noise_decoding(_bb72(), 0.01, num_shots=4000, erasure_rate=0.1, seed=2024, verbose=False, **CS8)
    assert res["erasure_aware"]["num_logical"] < res["static"]["num_logical"]


def test_argument_errors():
    import torch
    from slidingwindowdecoder_b200 import _lib
    lib = _lib.load()
    s, (px, py, pz, llr5) = _sampler("bb72_uniform", 0.05)
    n, dp, i32p = s.n, C.POINTER(C.c_double), C.POINTER(C.c_int32)

    def window():
        h = C.c_void_p()
        _lib.check(lib.swd_window_create(0, s.num_det, 2 * n, *(a.ctypes.data_as(i32p) for a in s._cp[:2]), s.num_obs,
                                         *(a.ctypes.data_as(i32p) for a in s._cp[2:]), C.byref(h)), "create")
        return h

    def set_priors(h, nn=n, x=px, y=py, z=pz, rate=0.05, llr=None):
        arr = [np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, z)]
        llr = None if llr is None else np.ascontiguousarray(llr)
        return lib.swd_window_set_pauli_priors(h, nn, *(a.ctypes.data_as(dp) for a in arr), rate,
                                               None if llr is None else llr.ctypes.data_as(dp))

    h = window()
    try:
        neg, nan, big = px.copy(), px.copy(), px.copy()
        neg[2] = -1e-3; nan[3] = np.nan; big[4] = 1.0
        for kw in (dict(nn=n + 1), dict(nn=n - 1), dict(x=neg), dict(y=nan), dict(z=big), dict(rate=-0.01), dict(rate=1.01),
                   dict(rate=float("nan"))):
            assert set_priors(h, **{k: v for k, v in kw.items()}) == _lib.ERR_INVALID, kw
        det = torch.empty((8, s.num_det), dtype=torch.uint8, device="cuda")
        obs = torch.empty((8, s.num_obs), dtype=torch.uint8, device="cuda")
        L = torch.empty((5, 8, n), dtype=torch.float64, device="cuda")
        sample = lambda B=8, off=0, d=det.data_ptr(), o=obs.data_ptr(), llr=None: lib.swd_window_sample_pauli(  # noqa: E731
            h, 1, off, B, d, o, None, None, llr, None)
        assert sample() == _lib.ERR_INVALID                                   # no set-up call yet
        assert set_priors(h) == _lib.OK                                       # without llr5
        assert sample(llr=L.data_ptr()) == _lib.ERR_INVALID                   # planes need llr5
        for kw in (dict(d=None), dict(o=None), dict(B=-1), dict(off=-1)):
            assert sample(**kw) == _lib.ERR_INVALID, kw
        assert sample(B=0) == _lib.OK
        assert sample() == _lib.OK
        assert set_priors(h, llr=llr5) == _lib.OK
        assert sample(llr=L.data_ptr()) == _lib.OK
        torch.cuda.synchronize()
    finally:
        lib.swd_window_destroy(h)
    from slidingwindowdecoder_b200 import CodeCapacitySampler
    plain = CodeCapacitySampler(_bb72().hx, _bb72().hz, _bb72().lx, _bb72().lz, px, py, pz)
    for kw in (dict(B=-1), dict(B=4, shot_offset=-1), dict(B=4, seed=-1), dict(B=4, seed=1 << 64)):
        with pytest.raises(ValueError):
            s.sample(**kw)
    with pytest.raises(ValueError):
        plain.sample(4, return_llr=True)
    out = s.sample(4, return_errors=True)
    for d, dt, ob in ((out["err"][:, :, :-1], out["det"], out["obs"]), (out["err"], out["det"][:3], out["obs"]),
                      (out["err"], out["det"], out["obs"][:, :-1]), (out["err"], out["det"].t(), out["obs"])):
        with pytest.raises(ValueError):
            s.count_failures(d, dt, ob)
