"""Circuit-level erasure sampling on the device: swd_window_sample_circuit against its numpy restatement
(tests/circuit_oracle.py::sample_circuit) bit for bit, the per-shot LLR rows against the erasures, the law at erasure rate 0
against the DEM sampler, and circuit_erasure_decoding against the same pipeline fed from the host."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEEDS = ((0, 0), ((0xDEADBEEF << 32) | 12345, (1 << 32) + 77))                 # (seed, shot_offset)
FAST_GDG = dict(max_iter=8)                                                     # bench.py's c3_gdg pre-BP iterations


def _circuit(name, p=0.003):
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, shyps_memory_circuit
    if name == "shyps3_z":
        return shyps_memory_circuit(3, p, 3)
    code, A, B = bb_code(72)
    return bb_memory_circuit(code, A, B, p, 6, z_basis=name == "bb72x6_z")


def _rate(s_locs, rate):
    """'random': one rate per location, X_ERROR / Z_ERROR / DEPOLARIZE1 locations included, some zero."""
    if rate != "random":
        return rate
    rng = np.random.default_rng(17)
    r = rng.uniform(0.0, 0.3, s_locs.num_locations)
    r[rng.random(len(r)) < 0.3] = 0.0
    r[0] = 1.0
    assert (r[s_locs.kind == "X_ERROR"] > 0).any()
    return r


def _host(t):
    return t.cpu().numpy()


@pytest.mark.parametrize("circ", ("bb72x6_z", "bb72x6_x", "shyps3_z"))
@pytest.mark.parametrize("rate", (0.0, 0.05, 1.0, "random"))
def test_sampler_bit_exact(circ, rate):
    import torch
    from circuit_oracle import sample_circuit
    from slidingwindowdecoder_b200 import CircuitNoiseSampler
    from slidingwindowdecoder_b200.dem import noise_locations
    c = _circuit(circ, p=0.01)
    e = _rate(noise_locations(c), rate)
    s = CircuitNoiseSampler(c, erasure_rate=e)
    B = 999                                                                     # not a multiple of the warps per block
    for seed, off in SEEDS:
        det, obs, err, erased, L = s.sample(B, seed=seed, shot_offset=off, return_errors=True, return_erasures=True, return_llr=True)
        want = sample_circuit(s.chk, s.obs, s.locations, s.erasure_rate, s.channel_llr, B, seed=seed, shot_offset=off)
        for got, ref, what in zip((det, obs, err, erased), want[:4], ("det", "obs", "err", "erased")):
            assert np.array_equal(_host(got), ref), what
        assert np.array_equal(_host(L).view(np.uint64), want[4].view(np.uint64))
        e_host = _host(err).astype(np.int64)
        assert np.array_equal(_host(det), (np.asarray(s.chk @ e_host.T).T % 2).astype(np.uint8))
        if rate == 1.0:
            assert (_host(erased)[:, s.locations.kind == "DEPOLARIZE2"] == 1).all()
        # the optional outputs do not change det / obs
        d2, o2 = s.sample(B, seed=seed, shot_offset=off)
        assert torch.equal(d2, det) and torch.equal(o2, obs)


def test_llr_rows_from_erasures():
    """A row is the static row with +0.0 exactly at the DEM columns of the shot's erased locations."""
    from slidingwindowdecoder_b200 import CircuitNoiseSampler
    s = CircuitNoiseSampler(_circuit("bb72x6_z"), erasure_rate=0.01)
    _, _, erased, L = s.sample(2048, seed=3, return_erasures=True, return_llr=True)
    er, L = _host(erased).astype(bool), _host(L)
    locs = s.locations
    assert 0 < er.mean() and er[:, locs.kind != "DEPOLARIZE2"].sum() == 0
    for b in (0, 1, 100, 2047):
        cols = set()
        for loc in np.flatnonzero(er[b]):
            mc = locs.mech_col[locs.mech_ptr[loc]:locs.mech_ptr[loc + 1]]
            cols.update(int(c) for c in mc[mc >= 0])
        want = s.channel_llr.copy()
        want[sorted(cols)] = 0.0
        assert np.array_equal(L[b].view(np.uint64), want.view(np.uint64)), b
    assert (L.view(np.uint64)[L == 0.0] == 0).all()                           # +0.0, not -0.0


def test_no_erasure_has_the_dem_law():
    """At e = 0 columns fire independently with the DEM priors: per-column rates against priors, and det / obs rates against
    the DEM sampler swd_window_sample."""
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from slidingwindowdecoder_b200.windows import build_windows
    s = CircuitNoiseSampler(_circuit("bb72x6_z", p=0.01))
    B = 1 << 16
    det, obs, err, L = s.sample(B, seed=9, return_errors=True, return_llr=True)
    assert np.array_equal(_host(L[:7]), np.broadcast_to(s.channel_llr, (7, s.num_col)))
    rate = _host(err.sum(dim=0, dtype=torch.int64)) / B
    sd = np.sqrt(s.priors * (1 - s.priors) / B)
    assert (np.abs(rate - s.priors) <= 5 * sd + 1e-9).all()
    plan = build_windows(s.chk, s.obs, s.priors, 72, W=3, F=1, method=1)
    swd = SlidingWindowDecoder(plan, decoder="gdg", **FAST_GDG)
    det2, obs2 = swd.sample_device(B, seed=10)
    for a, b_ in ((det, det2), (obs, obs2)):
        m1 = _host(a.sum(dim=0, dtype=torch.int64)) / B
        m2 = _host(b_.sum(dim=0, dtype=torch.int64)) / B
        pm = (m1 + m2) / 2
        assert (np.abs(m1 - m2) <= 5 * np.sqrt(2 * pm * (1 - pm) / B) + 1e-9).all()


def test_batch_and_shard_independence():
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler
    s = CircuitNoiseSampler(_circuit("bb72x6_x"), erasure_rate=0.05)
    off = (3 << 32) + 11
    whole = s.sample(1000, seed=4, shot_offset=off, return_errors=True, return_erasures=True, return_llr=True)
    parts = [s.sample(hi - lo, seed=4, shot_offset=off + lo, return_errors=True, return_erasures=True, return_llr=True)
             for lo, hi in ((0, 1), (1, 300), (300, 1000))]
    for i, t in enumerate(whole):
        assert torch.equal(t, torch.cat([p[i] for p in parts])), i
    empty = s.sample(0, return_errors=True, return_erasures=True, return_llr=True)
    assert [tuple(t.shape) for t in empty] == [(0, s.num_det), (0, s.num_obs), (0, s.num_col), (0, s.num_locations), (0, s.num_col)]


def _legs(res):
    return {k: (v["num_flagged"], v["num_logical"], tuple(v["window_unconverged"])) for k, v in res.items() if isinstance(v, dict)}


def test_driver_without_erasures_legs_agree():
    from slidingwindowdecoder_b200 import circuit_erasure_decoding
    res = circuit_erasure_decoding(72, 0.004, 0.0, num_repeat=6, num_shots=3000, seed=5, **FAST_GDG)
    legs = _legs(res)
    assert legs["static"] == legs["erasure_aware"]
    assert res["erased_fraction"] == 0.0 and 0 < res["static"]["num_logical"] < 3000


def test_driver_matches_host_pipeline_and_is_batch_independent():
    from circuit_oracle import sample_circuit
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, circuit_erasure_decoding
    from slidingwindowdecoder_b200.distributed import shard_range
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from slidingwindowdecoder_b200.windows import build_windows
    shots, seed = 2000, (1 << 40) + 3
    res = circuit_erasure_decoding(72, 0.002, 0.02, num_repeat=6, num_shots=shots, seed=seed, **FAST_GDG)
    s = CircuitNoiseSampler(_circuit("bb72x6_z", p=0.002), erasure_rate=0.02)
    det, obs, _, erased, L = sample_circuit(s.chk, s.obs, s.locations, s.erasure_rate, s.channel_llr, shots, seed=seed)
    plan = build_windows(s.chk, s.obs, s.priors, 72, W=3, F=1, method=1)
    from slidingwindowdecoder_b200.drivers import _GDG_DEFAULTS
    swd = SlidingWindowDecoder(plan, decoder="gdg", streams=2, **dict(_GDG_DEFAULTS, **FAST_GDG))
    for leg, rows in (("static", None), ("erasure_aware", L)):
        ref = swd.decode(det, obs, channel_llr=rows)
        assert (res[leg]["num_flagged"], res[leg]["num_logical"]) == (ref["flagged"], ref["failed"]), leg
        assert res[leg]["window_unconverged"] == ref["window_unconverged"], leg
        assert res[leg]["p_l"] == ref["failed"] / shots
    assert res["erased_fraction"] == pytest.approx(erased.mean(), abs=1e-12)
    assert _legs(res)["static"] != _legs(res)["erasure_aware"]
    kw = dict(num_repeat=6, seed=seed, **FAST_GDG)
    for batch, streams in ((700, 1), (2000, 2)):
        assert _legs(circuit_erasure_decoding(72, 0.002, 0.02, num_shots=shots, batch=batch, streams=streams, **kw)) == _legs(res)
    parts = [_legs(circuit_erasure_decoding(72, 0.002, 0.02, num_shots=hi - lo, shot_offset=lo, **kw))
             for lo, hi in (shard_range(shots, r, 2) for r in range(2))]
    for leg, (f, n, u) in _legs(res).items():
        assert (parts[0][leg][0] + parts[1][leg][0], parts[0][leg][1] + parts[1][leg][1]) == (f, n), leg
        assert tuple(a + b for a, b in zip(parts[0][leg][2], parts[1][leg][2])) == u, leg


def test_erasure_information_helps():
    """[[72,12,6]] x 6 rounds, p = 0.001, 1 % of the gates erased, 4000 shots at seed 2024: the decoder that knows the
    erasures fails strictly less often."""
    from slidingwindowdecoder_b200 import circuit_erasure_decoding
    res = circuit_erasure_decoding(72, 0.001, 0.01, num_repeat=6, num_shots=4000, seed=2024, **FAST_GDG)
    assert res["erasure_aware"]["num_logical"] < res["static"]["num_logical"], res


def test_argument_errors():
    import torch
    from slidingwindowdecoder_b200 import CircuitNoiseSampler, _lib
    lib = _lib.load()
    s = CircuitNoiseSampler(_circuit("shyps3_z"), erasure_rate=0.05)
    locs, L = s.locations, s.num_locations
    i32p, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)

    def window():
        h = C.c_void_p()
        _lib.check(lib.swd_window_create(0, s.num_det, s.num_col, *(a.ctypes.data_as(i32p) for a in s._cp[:2]), s.num_obs,
                                         *(a.ctypes.data_as(i32p) for a in s._cp[2:]), C.byref(h)), "create")
        return h

    def set_noise(h, nl=L, ptr=locs.mech_ptr, col=locs.mech_col, prob=locs.mech_prob, rate=s.erasure_rate, llr=None, null=()):
        arrs = dict(ptr=np.ascontiguousarray(ptr, dtype=np.int32), col=np.ascontiguousarray(col, dtype=np.int32),
                    prob=np.ascontiguousarray(prob, dtype=np.float64), rate=np.ascontiguousarray(rate, dtype=np.float64))
        a = {k: (None if k in null else v.ctypes.data_as(i32p if k in ("ptr", "col") else dp)) for k, v in arrs.items()}
        llr = None if llr is None else np.ascontiguousarray(llr)
        return lib.swd_window_set_circuit_noise(h, nl, a["ptr"], a["col"], a["prob"], a["rate"],
                                                None if llr is None else llr.ctypes.data_as(dp))

    h = window()
    try:
        ptr_off = locs.mech_ptr.copy(); ptr_off += 1
        ptr_zero = locs.mech_ptr.copy(); ptr_zero[1] = ptr_zero[0]                # a location without mechanisms
        ptr_16 = locs.mech_ptr.copy(); ptr_16[1] = 16                              # location 0 with 16 mechanisms
        ptr_dec = locs.mech_ptr.copy(); ptr_dec[2] = ptr_dec[1] - 1                # not monotone
        bad = [dict(nl=0), dict(nl=-1), dict(null=("ptr",)), dict(null=("col",)), dict(null=("prob",)), dict(null=("rate",)),
               dict(ptr=ptr_off), dict(ptr=ptr_zero), dict(ptr=ptr_16), dict(ptr=ptr_dec)]
        for k, v in (("col", -2), ("col", s.num_col), ("prob", -0.1), ("prob", 0.6), ("prob", np.nan), ("rate", -0.1),
                     ("rate", 1.1), ("rate", np.nan)):
            a = np.array(dict(col=locs.mech_col, prob=locs.mech_prob, rate=s.erasure_rate)[k], copy=True)
            a[len(a) // 2] = v
            bad.append({k: a})
        for kw in bad:
            assert set_noise(h, **kw) == _lib.ERR_INVALID, kw
        det = torch.empty((8, s.num_det), dtype=torch.uint8, device="cuda")
        obs = torch.empty((8, s.num_obs), dtype=torch.uint8, device="cuda")
        Lr = torch.empty((8, s.num_col), dtype=torch.float64, device="cuda")
        sample = lambda B=8, off=0, d=det.data_ptr(), o=obs.data_ptr(), llr=None: lib.swd_window_sample_circuit(  # noqa: E731
            h, 1, off, B, d, o, None, None, llr, None)
        assert sample() == _lib.ERR_INVALID                                   # before swd_window_set_circuit_noise
        assert set_noise(h) == _lib.OK                                        # without col_llr
        assert sample(llr=Lr.data_ptr()) == _lib.ERR_INVALID                  # rows need col_llr
        for kw in (dict(d=None), dict(o=None), dict(B=-1), dict(off=-1)):
            assert sample(**kw) == _lib.ERR_INVALID, kw
        assert sample(B=0) == _lib.OK
        assert sample() == _lib.OK
        assert set_noise(h, llr=s.channel_llr) == _lib.OK
        assert sample(llr=Lr.data_ptr()) == _lib.OK
        torch.cuda.synchronize()
    finally:
        lib.swd_window_destroy(h)
    for kw in (dict(B=-1), dict(B=4, shot_offset=-1), dict(B=4, seed=-1), dict(B=4, seed=1 << 64)):
        with pytest.raises(ValueError):
            s.sample(**kw)
