"""Soft measurement readout on the device: swd_window_sample_circuit_readout against its numpy restatement
(tests/readout_oracle.py::sample_circuit_readout) bit for bit, its K = 1 case against swd_window_sample_circuit, the
per-shot LLR rows against the classes and erasures, and circuit_soft_readout_decoding against the same pipeline fed from
the host."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEEDS = ((0, 0), ((0xDEADBEEF << 32) | 12345, (1 << 32) + 77))                 # (seed, shot_offset), as test_circuit_erasure
FAST_GDG = dict(max_iter=8)                                                     # bench.py's c3_gdg pre-BP iterations
P = 0.01


def _circuit(name, p=P):
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, shyps_memory_circuit
    if name == "shyps3_z":
        return shyps_memory_circuit(3, p, 3)
    code, A, B = bb_code(72)
    return bb_memory_circuit(code, A, B, p, 6, z_basis=name == "bb72x6_z")


def _rate(locs, rate):
    """'random': one rate per location, readout locations included, some zero."""
    if rate != "random":
        return rate
    rng = np.random.default_rng(23)
    r = rng.uniform(0.0, 0.3, locs.num_locations)
    r[rng.random(len(r)) < 0.3] = 0.0
    return r


def _host(t):
    return t.cpu().numpy()


def _oracle(s, B, seed, off):
    from readout_oracle import sample_circuit_readout
    return sample_circuit_readout(s.chk, s.obs, s.locations, s.erasure_rate, s.channel_llr, s.readout_locations, s.readout.weights,
                                  s.readout.flip_prob, s.class_llr, B, seed=seed, shot_offset=off)


@pytest.mark.parametrize("circ", ("bb72x6_z", "bb72x6_x", "shyps3_z"))
@pytest.mark.parametrize("K", (1, 4, 16, 256))
@pytest.mark.parametrize("rate", (0.0, "random"))
def test_sampler_bit_exact(circ, K, rate):
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, gaussian_readout
    from slidingwindowdecoder_b200.dem import noise_locations
    c = _circuit(circ)
    s = CircuitNoiseSampler(c, erasure_rate=_rate(noise_locations(c), rate), readout=gaussian_readout(P, K))
    B = 999                                                                     # not a multiple of the warps per block
    for seed, off in SEEDS:
        got = s.sample(B, seed=seed, shot_offset=off, return_errors=True, return_erasures=True, return_readout=True, return_llr=True)
        want = _oracle(s, B, seed, off)
        for g, ref, what in zip(got[:5], want[:5], ("det", "obs", "err", "erased", "readout")):
            assert np.array_equal(_host(g), ref), what
        assert np.array_equal(_host(got[5]).view(np.uint64), want[5].view(np.uint64))
        if K > 1:
            assert len(np.unique(want[4])) > 1
        # the optional outputs do not change det / obs
        d2, o2 = s.sample(B, seed=seed, shot_offset=off)
        assert torch.equal(d2, got[0]) and torch.equal(o2, got[1])


@pytest.mark.parametrize("circ", ("bb72x6_z", "shyps3_z"))
@pytest.mark.parametrize("rate", (0.0, 0.05, "random"))
def test_one_class_equals_circuit_sampler(circ, rate):
    """K = 1, q = [p]: the readout entry point reproduces swd_window_sample_circuit bit for bit."""
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler
    from slidingwindowdecoder_b200.dem import ReadoutModel, noise_locations
    c = _circuit(circ)
    e = _rate(noise_locations(c), rate)
    plain = CircuitNoiseSampler(c, erasure_rate=e)
    soft = CircuitNoiseSampler(c, erasure_rate=e, readout=ReadoutModel([1.0], [P]))
    for seed, off in SEEDS:
        a = plain.sample(1000, seed=seed, shot_offset=off, return_errors=True, return_erasures=True, return_llr=True)
        b = soft.sample(1000, seed=seed, shot_offset=off, return_errors=True, return_erasures=True, return_readout=True, return_llr=True)
        for i in range(4):
            assert torch.equal(a[i], b[i]), i
        assert torch.equal(a[4].view(torch.int64), b[5].view(torch.int64))
        assert (b[4] == 0).all()


def test_llr_rows_from_classes_and_erasures():
    """A row is the static row with class_llr[r, class_r] at readout r's column and +0.0 at every column of an erased
    location, the erasure winning."""
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, gaussian_readout
    c = _circuit("bb72x6_z", p=0.003)
    s = CircuitNoiseSampler(c, erasure_rate=0.02, readout=gaussian_readout(0.003, 16))
    _, _, erased, cls, L = s.sample(2048, seed=3, return_erasures=True, return_readout=True, return_llr=True)
    er, cls, L = _host(erased).astype(bool), _host(cls), _host(L)
    locs, ro = s.locations, s.readout_locations
    ro_col = locs.mech_col[locs.mech_ptr[ro]]
    assert er.any() and len(np.unique(cls)) == 16
    hit = 0
    for b in range(0, 2048, 97):
        want = s.channel_llr.copy()
        for r in np.flatnonzero(ro_col >= 0):
            want[ro_col[r]] = s.class_llr[r, cls[b, r]]
        for loc in np.flatnonzero(er[b]):
            mc = locs.mech_col[locs.mech_ptr[loc]:locs.mech_ptr[loc + 1]]
            want[mc[mc >= 0]] = 0.0
            hit += int(np.isin(mc, ro_col[ro_col >= 0]).any())
        assert np.array_equal(L[b].view(np.uint64), want.view(np.uint64)), b
    assert hit > 0                                                   # some erased location shares a column with a readout
    assert (L.view(np.uint64)[L == 0.0] == 0).all()                 # +0.0, not -0.0


def test_batch_and_shard_independence():
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, gaussian_readout
    s = CircuitNoiseSampler(_circuit("bb72x6_x"), erasure_rate=0.05, readout=gaussian_readout(P, 16))
    off = (3 << 32) + 11
    kw = dict(return_errors=True, return_erasures=True, return_readout=True, return_llr=True)
    whole = s.sample(1000, seed=4, shot_offset=off, **kw)
    parts = [s.sample(hi - lo, seed=4, shot_offset=off + lo, **kw) for lo, hi in ((0, 1), (1, 300), (300, 1000))]
    for i, t in enumerate(whole):
        assert torch.equal(t, torch.cat([p[i] for p in parts])), i
    empty = s.sample(0, **kw)
    R = len(s.readout_locations)
    assert [tuple(t.shape) for t in empty] == [(0, s.num_det), (0, s.num_obs), (0, s.num_col), (0, s.num_locations), (0, R),
                                               (0, s.num_col)]
    with pytest.raises(ValueError):
        CircuitNoiseSampler(_circuit("bb72x6_x")).sample(4, return_readout=True)


def _legs(res):
    return {k: (v["num_flagged"], v["num_logical"], tuple(v["window_unconverged"])) for k, v in res.items() if isinstance(v, dict)}


def test_driver_one_class_legs_agree():
    from slidingwindowdecoder_b200 import circuit_soft_readout_decoding
    res = circuit_soft_readout_decoding(72, 0.004, num_classes=1, num_repeat=6, num_shots=3000, seed=5, **FAST_GDG)
    legs = _legs(res)
    assert legs["static"] == legs["soft_aware"]
    assert res["class_histogram"] == [3000 * 432] and 0 < res["static"]["num_logical"] < 3000


def test_driver_matches_host_pipeline_and_is_batch_independent():
    import torch
    from readout_oracle import sample_circuit_readout
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, circuit_soft_readout_decoding, gaussian_readout
    from slidingwindowdecoder_b200.dem import with_readout_error
    from slidingwindowdecoder_b200.distributed import shard_range
    from slidingwindowdecoder_b200.drivers import _GDG_DEFAULTS
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from slidingwindowdecoder_b200.windows import build_windows
    shots, seed = 2000, (1 << 40) + 3
    kw = dict(p_meas=0.04, num_classes=16, num_repeat=6, seed=seed, **FAST_GDG)
    res = circuit_soft_readout_decoding(72, 0.003, num_shots=shots, **kw)
    model = gaussian_readout(0.04, 16)
    s = CircuitNoiseSampler(with_readout_error(_circuit("bb72x6_z", p=0.003), 0.04), readout=model)
    det, obs, _, _, cls, L = sample_circuit_readout(s.chk, s.obs, s.locations, 0.0, s.channel_llr, s.readout_locations,
                                                    model.weights, model.flip_prob, s.class_llr, shots, seed=seed)
    assert res["class_histogram"] == np.bincount(cls.ravel(), minlength=16).tolist()
    plan = build_windows(s.chk, s.obs, s.priors, 72, W=3, F=1, method=1)
    swd = SlidingWindowDecoder(plan, decoder="gdg", streams=2, **dict(_GDG_DEFAULTS, **FAST_GDG))
    dev = torch.device("cuda", 0)
    for leg, rows in (("static", None), ("soft_aware", L)):
        on_dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
        out = swd.decode_device(on_dev(det), on_dev(obs), channel_llr=None if rows is None else on_dev(rows))
        f, n = (int(x) for x in out["counts"].cpu().tolist())
        assert (res[leg]["num_flagged"], res[leg]["num_logical"]) == (f, n), leg
        assert res[leg]["window_unconverged"] == [int(x) for x in out["window_unconverged"].cpu().tolist()], leg
        assert res[leg]["p_l"] == n / shots
    assert _legs(res)["static"] != _legs(res)["soft_aware"]
    for batch, streams in ((700, 1), (2000, 2)):
        again = circuit_soft_readout_decoding(72, 0.003, num_shots=shots, batch=batch, streams=streams, **kw)
        assert _legs(again) == _legs(res) and again["class_histogram"] == res["class_histogram"]
    parts = [circuit_soft_readout_decoding(72, 0.003, num_shots=hi - lo, shot_offset=lo, **kw)
             for lo, hi in (shard_range(shots, r, 2) for r in range(2))]
    assert [a + b for a, b in zip(parts[0]["class_histogram"], parts[1]["class_histogram"])] == res["class_histogram"]
    for leg, (f, n, u) in _legs(res).items():
        pl = [_legs(x)[leg] for x in parts]
        assert (pl[0][0] + pl[1][0], pl[0][1] + pl[1][1]) == (f, n), leg
        assert tuple(a + b for a, b in zip(pl[0][2], pl[1][2])) == u, leg


def test_soft_information_helps():
    """[[72,12,6]] x 6 rounds, p = 0.003, p_meas = 0.04, K = 16, 4000 shots at seed 2024 (the pinned point of
    tools/bench_circuit_readout.py; on one B200: 166 static vs 75 soft-aware failures, 5.9 standard deviations): the decoder
    that knows the readout classes fails fewer shots, by more than four standard deviations of the difference."""
    from slidingwindowdecoder_b200 import circuit_soft_readout_decoding
    res = circuit_soft_readout_decoding(72, 0.003, p_meas=0.04, num_classes=16, num_repeat=6, num_shots=4000, seed=2024, **FAST_GDG)
    a, b = res["static"]["num_logical"], res["soft_aware"]["num_logical"]
    assert a - b > 4 * np.sqrt(a + b), res


def test_argument_errors():
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, _lib, gaussian_readout
    lib = _lib.load()
    model = gaussian_readout(P, 4)
    s = CircuitNoiseSampler(_circuit("shyps3_z"), erasure_rate=0.05, readout=model)
    plain = CircuitNoiseSampler(_circuit("shyps3_z"), erasure_rate=0.05)
    locs, L, ro, R = s.locations, s.num_locations, s.readout_locations, len(s.readout_locations)
    i32p, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    h = C.c_void_p()
    _lib.check(lib.swd_window_create(0, s.num_det, s.num_col, *(a.ctypes.data_as(i32p) for a in s._cp[:2]), s.num_obs,
                                     *(a.ctypes.data_as(i32p) for a in s._cp[2:]), C.byref(h)), "create")

    def set_noise():
        return lib.swd_window_set_circuit_noise(h, L, locs.mech_ptr.ctypes.data_as(i32p), locs.mech_col.ctypes.data_as(i32p),
                                                locs.mech_prob.ctypes.data_as(dp), s.erasure_rate.ctypes.data_as(dp),
                                                s.channel_llr.ctypes.data_as(dp))

    def set_ro(nr=R, loc=ro, K=4, w=model.weights, q=model.flip_prob, llr=s.class_llr, null=()):
        arrs = dict(loc=np.ascontiguousarray(loc, dtype=np.int32), w=np.ascontiguousarray(w, dtype=np.float64),
                    q=np.ascontiguousarray(q, dtype=np.float64), llr=np.ascontiguousarray(llr, dtype=np.float64))
        a = {k: (None if k in null else v.ctypes.data_as(i32p if k == "loc" else dp)) for k, v in arrs.items()}
        return lib.swd_window_set_circuit_readout(h, nr, a["loc"], K, a["w"], a["q"], a["llr"])

    det = torch.empty((8, s.num_det), dtype=torch.uint8, device="cuda")
    obs = torch.empty((8, s.num_obs), dtype=torch.uint8, device="cuda")
    Lr = torch.empty((8, s.num_col), dtype=torch.float64, device="cuda")
    cls = torch.empty((8, R), dtype=torch.uint8, device="cuda")
    sample = lambda B=8, off=0, d=det.data_ptr(), o=obs.data_ptr(), llr=None: lib.swd_window_sample_circuit_readout(  # noqa: E731
        h, 1, off, B, d, o, None, None, cls.data_ptr(), llr, None)
    try:
        assert set_ro() == _lib.ERR_INVALID                                   # before swd_window_set_circuit_noise
        assert sample() == _lib.ERR_INVALID
        assert set_noise() == _lib.OK
        assert sample() == _lib.ERR_INVALID                                   # before swd_window_set_circuit_readout
        dep1 = int(np.flatnonzero(locs.kind == "DEPOLARIZE1")[0])
        bad = [dict(nr=0), dict(nr=-1), dict(null=("loc",)), dict(null=("w",)), dict(null=("q",)), dict(K=0), dict(K=257),
               dict(loc=np.r_[ro[:-1], L]), dict(loc=np.r_[ro[:-1], -1]), dict(loc=np.r_[ro[:-1], ro[0]]),
               dict(loc=np.r_[ro[:-1], dep1]), dict(w=[0.5, 0.5, 0.5, -0.5]), dict(w=[np.nan, 0.5, 0.25, 0.25]),
               dict(w=[0.25, 0.25, 0.25, 0.25 + 2e-9]), dict(q=[0.6, 0.1, 0.0, 0.0]), dict(q=[-0.1, 0.1, 0.0, 0.0]),
               dict(q=[np.nan, 0.1, 0.0, 0.0])]
        for kw in bad:
            assert set_ro(**kw) == _lib.ERR_INVALID, kw
        assert set_ro(w=[0.25, 0.25, 0.25, 0.25 + 5e-10]) == _lib.OK          # within 1e-9 of 1
        assert set_ro(null=("llr",)) == _lib.OK                               # without class_llr
        assert sample(llr=Lr.data_ptr()) == _lib.ERR_INVALID                  # rows need class_llr
        assert sample() == _lib.OK
        assert set_ro() == _lib.OK
        for kw in (dict(d=None), dict(o=None), dict(B=-1), dict(off=-1)):
            assert sample(**kw) == _lib.ERR_INVALID, kw
        assert sample(B=0) == _lib.OK
        assert sample(llr=Lr.data_ptr()) == _lib.OK
        # swd_window_sample_circuit ignores the readout set-up
        d1, o1 = plain.sample(8, seed=1)
        assert lib.swd_window_sample_circuit(h, 1, 0, 8, det.data_ptr(), obs.data_ptr(), None, None, None, None) == _lib.OK
        torch.cuda.synchronize()
        assert torch.equal(det, d1) and torch.equal(obs, o1)
        # a new circuit-noise set-up clears the readout set-up
        assert set_noise() == _lib.OK
        assert sample() == _lib.ERR_INVALID
        torch.cuda.synchronize()
    finally:
        lib.swd_window_destroy(h)

    # two readout locations whose flips land in one DEM column
    from slidingwindowdecoder_b200.dem import Ops, _noise_locations, dem_to_check_matrices
    c2 = Ops()
    c2.gate("R", 0, 1)
    c2.noise("X_ERROR", P, 0, 1)
    c2.gate("M", 0, 1)
    c2.detector([-1, -2])
    l2, dem2 = _noise_locations(c2)
    chk2 = dem_to_check_matrices(dem2)[0]
    cp, ri = np.ascontiguousarray(chk2.indptr, dtype=np.int32), np.ascontiguousarray(chk2.indices, dtype=np.int32)
    h2 = C.c_void_p()
    _lib.check(lib.swd_window_create(0, chk2.shape[0], chk2.shape[1], cp.ctypes.data_as(i32p), ri.ctypes.data_as(i32p), 0, None,
                                     None, C.byref(h2)), "create")
    try:
        zero, one, q = np.zeros(2), np.ones(1), np.full(1, P)
        assert lib.swd_window_set_circuit_noise(h2, 2, l2.mech_ptr.ctypes.data_as(i32p), l2.mech_col.ctypes.data_as(i32p),
                                                l2.mech_prob.ctypes.data_as(dp), zero.ctypes.data_as(dp), None) == _lib.OK
        for locs2, want in (([0, 1], _lib.ERR_INVALID), ([1], _lib.OK)):
            a = np.array(locs2, dtype=np.int32)
            assert lib.swd_window_set_circuit_readout(h2, len(a), a.ctypes.data_as(i32p), 1, one.ctypes.data_as(dp),
                                                      q.ctypes.data_as(dp), None) == want, locs2
    finally:
        lib.swd_window_destroy(h2)
