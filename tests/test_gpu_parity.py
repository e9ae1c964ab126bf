"""CUDA decoders (through the C-ABI) against the CPU oracle and the reference's golden vectors."""
import numpy as np
import pytest

from conftest import load_golden, GOLDEN_GDG, GOLDEN_OSD

pytestmark = pytest.mark.gpu


def _gdg_cls():
    from slidingwindowdecoder_b200 import bpgdg_decoder
    return bpgdg_decoder


@pytest.mark.parametrize("name", [g for g in GOLDEN_GDG if g.endswith("mt1")])
def test_gdg_multi_thread_matches_oracle_and_golden(name, oracle_mod):
    g = load_golden(name)
    dec = _gdg_cls()(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    corr, conv, pm = dec.decode_batch(g["synd"], return_pm=True)
    orc = oracle_mod.Oracle(g["mat"], g["priors"])
    o_dec, o_conv, o_pm, _ = orc.bpgdg_batch(g["synd"], **g["kwargs"])
    assert np.array_equal(conv, o_conv.astype(np.uint8))
    assert np.array_equal(corr, o_dec.astype(np.uint8))                 # bit-exact vs the oracle (same tie rule)
    gdg = pm < 9999.0
    assert np.array_equal(pm[gdg], o_pm[gdg])                           # identical fp64 path metrics
    # vs the threaded reference: identical except exact-pm ties (resolved by thread timing there)
    assert np.array_equal(conv, g["conv"])
    from test_oracle_golden import check_only_ties
    bad = np.nonzero((corr != g["dec"]).any(axis=1))[0]
    check_only_ties(g, orc, corr, conv, pm, bad, name)


@pytest.mark.parametrize("name", [g for g in GOLDEN_GDG if g.endswith("mt0")] + ["c1_gdg_sim_uniform_mt0"])
def test_gdg_single_thread_matches_golden(name, oracle_mod):
    """multi_thread=False (the constructor default): deterministic schedule, exact vectors vs the reference."""
    g = load_golden(name)
    dec = _gdg_cls()(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    corr, conv = dec.decode_batch(g["synd"])
    assert np.array_equal(conv, g["conv"])
    bad = np.nonzero((corr != g["dec"]).any(axis=1))[0]
    assert len(bad) == 0, f"shots {bad[:10]}"


@pytest.mark.parametrize("name", __import__("conftest").GOLDEN_BPGD)
def test_bpgd_matches_oracle_and_golden(name, oracle_mod):
    from slidingwindowdecoder_b200 import bpgd_decoder
    g = load_golden(name)
    dec = bpgd_decoder(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    corr, conv = dec.decode_batch(g["synd"])
    assert np.array_equal(conv, g["conv"])
    assert np.array_equal(corr, g["dec"])


def test_single_shot_api(oracle_mod):
    g = load_golden("c1_gdg_default_mt1")
    dec = _gdg_cls()(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    for i in range(20):
        e = dec.decode(g["synd"][i])
        assert e.dtype == np.int64 and e.shape == (g["mat"].shape[1],)
        assert dec.converge == g["conv"][i]
    with pytest.raises(ValueError):
        dec.decode(np.zeros(5, dtype=np.uint8))


@pytest.mark.parametrize("name", ["c3_w5_gdg_mt1", "c3_w5_gdg_mt0", "c3_w5_bpgd", "c5_w4_gdg_mt1"])
def test_latency_configuration_equals_throughput_configuration(name):
    """Tiny batches run the branch paths in the latency configuration (one VN per thread: 448 instead of 128 threads per path on a
    [[144,12,12]] window) and one worst-case shared-memory tier: the corrections of shots decoded one, two and three at a time must
    equal those of the same shots decoded in one large batch (and the reference's goldens for the single-thread kinds)."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder
    g = load_golden(name)
    cls = bpgd_decoder if name.endswith("bpgd") else bpgdg_decoder
    dec = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    synd = g["synd"][:240]
    big, bconv, bpm = dec.decode_batch(synd, return_pm=True)
    for step in (1, 2, 3):
        for i in range(0, 60, step):
            c, v, pm = dec.decode_batch(synd[i:i + step], return_pm=True)
            assert np.array_equal(c, big[i:i + step]) and np.array_equal(v, bconv[i:i + step]) and np.array_equal(pm, bpm[i:i + step]), (step, i)
    if not name.endswith("mt1"):
        assert np.array_equal(big, g["dec"][:240])


def test_edge_cases(oracle_mod):
    g = load_golden("c1_gdg_default_mt1")
    dec = _gdg_cls()(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    m, n = g["mat"].shape
    corr, conv = dec.decode_batch(np.zeros((0, m), dtype=np.uint8))            # empty batch
    assert corr.shape == (0, n) and conv.shape == (0,)
    corr, conv = dec.decode_batch(np.zeros((3, m), dtype=np.uint8))            # trivial syndromes
    assert not corr.any() and conv.all()
    # ragged batch sizes give the same per-shot results as one big batch
    big, bigc = dec.decode_batch(g["synd"][:257])
    parts = [dec.decode_batch(g["synd"][a:b]) for a, b in ((0, 1), (1, 130), (130, 257))]
    assert np.array_equal(big, np.concatenate([p[0] for p in parts]))
    assert np.array_equal(bigc, np.concatenate([p[1] for p in parts]))
    # max_iter = 0: no pre-BP iterations, straight to GDG on the identity column order
    kw = dict(g["kwargs"], max_iter=0)
    d0 = _gdg_cls()(g["mat"], channel_probs=g["priors"], **kw)
    c0, v0 = d0.decode_batch(g["synd"][:200])
    orc = oracle_mod.Oracle(g["mat"], g["priors"])
    o_dec, o_conv, _, _ = orc.bpgdg_batch(g["synd"][:200], **kw)
    assert np.array_equal(c0, o_dec.astype(np.uint8)) and np.array_equal(v0, o_conv.astype(np.uint8))


def test_torch_device_path(oracle_mod):
    import torch
    g = load_golden("c2_w1_gdg_mt1")
    dec = _gdg_cls()(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    host, hconv = dec.decode_batch(g["synd"])
    t = torch.from_numpy(g["synd"]).cuda()
    corr, conv = dec.decode_batch(t)
    torch.cuda.synchronize()
    assert np.array_equal(corr.cpu().numpy(), host) and np.array_equal(conv.cpu().numpy(), hconv)


def test_large_batch_properties():
    """BASELINE-size window ([[144,12,12]] (3,1) middle window) at a large batch: every converged correction
    reproduces its syndrome; determinism across two runs; converge rate sane."""
    g = load_golden("c3_w5_gdg_mt1")
    rng = np.random.default_rng(5)
    H = g["mat"]
    B = 20000
    err = (rng.random((B, H.shape[1])) < g["priors"][None, :]).astype(np.uint8)
    synd = np.asarray((H @ err.T.astype(np.int32)).T % 2).astype(np.uint8)
    dec = _gdg_cls()(H, channel_probs=g["priors"], **g["kwargs"])
    corr, conv = dec.decode_batch(synd)
    ok = conv == 1
    resid = np.asarray((H @ corr[ok].T.astype(np.int32)).T % 2).astype(np.uint8)
    assert np.array_equal(resid, synd[ok])
    assert ok.mean() > 0.995
    corr2, conv2 = dec.decode_batch(synd)
    assert np.array_equal(corr, corr2) and np.array_equal(conv, conv2)


def test_sliding_window_driver_matches_reference_loop(oracle_mod):
    """[[72,12,6]] p=0.003, 6 rounds, (3,1): the device window pipeline vs the reference's loop run with the oracle."""
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder, sample_dem
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 6)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    det, ob, _ = sample_dem(plan.chk, plan.obs, plan.priors, 1500, np.random.default_rng(11))
    kw = dict(max_iter=8, multi_thread=True)
    swd = SlidingWindowDecoder(plan, decoder="gdg", **kw)
    res = swd.decode(det, ob, return_corrections=True)
    oracles = {}

    def decode_window(w, synd):
        if w.index not in oracles:
            oracles[w.index] = oracle_mod.Oracle(w.mat, w.prior)
        d, c, _, _ = oracles[w.index].bpgdg_batch(synd, **kw)
        return d, c

    ref = oracle_mod.sliding_window_reference(plan, det, ob, decode_window)
    assert np.array_equal(res["total_e_hat"], ref["total_e_hat"].astype(np.uint8))
    assert res["flagged"] == int(ref["flagged"].sum())
    assert res["failed"] == int(ref["failed"].sum())
    assert res["window_unconverged"] == ref["window_unconverged"]


@pytest.mark.parametrize("name", GOLDEN_OSD)
def test_osd_window_bit_exact(name, oracle_mod):
    """osd_window: BP decisions, OSD-0 / OSD-CS / OSD-E corrections, min_pm, bp_iteration and the posterior
    history, bit-exact against the reference's recorded outputs."""
    from slidingwindowdecoder_b200 import osd_window
    g = load_golden(name)
    dec = osd_window(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    corr, conv, pm = dec.decode_batch(g["synd"], return_pm=True)
    out = dec.last_outputs()
    assert np.array_equal(conv, g["conv"])
    bad = np.nonzero((corr != g["dec"]).any(axis=1))[0]
    assert len(bad) == 0, f"shots {bad[:10]}"
    assert np.array_equal(out["bp_decoding"], g["bp_decoding"])
    assert np.array_equal(out["bp_iteration"], g["bp_iteration"])
    assert np.array_equal(pm, g["min_pm"])
    orc = oracle_mod.Oracle(g["mat"], g["priors"])
    ran_osd = np.array([orc.osd_window(s, **g["kwargs"])["stats"].stage == 2 for s in g["synd"]])
    assert ran_osd.any()
    assert np.array_equal(out["osd0_decoding"][ran_osd], g["osd0"][ran_osd])
    assert dec.counters()["osd_shots"] == int(ran_osd.sum())
    for i in range(min(len(g["lpr_first8"]), len(corr))):
        if g["bp_iteration"][i] >= 4:
            assert np.array_equal(out["log_prob_ratios"][i], g["lpr_first8"][i]), i


def test_osd_window_bp_only_order_minus_one():
    """ADVICE r1: osd_order = -1 ("BP only", osd_window.pyx:86,192; osd.py's "-1 for no osd") is accepted: no OSD stage, shots
    whose post-BP does not converge return bp_decoding with converge = 0 and min_pm = 0.  Bit-exact vs the reference's golden."""
    from slidingwindowdecoder_b200 import osd_window
    g = load_golden("c2_w1_osdw_noosd")
    dec = osd_window(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    corr, conv, pm = dec.decode_batch(g["synd"], return_pm=True)
    out = dec.last_outputs()
    assert np.array_equal(conv, g["conv"]) and np.array_equal(corr, g["dec"])
    assert np.array_equal(out["bp_decoding"], g["bp_decoding"]) and np.array_equal(out["bp_iteration"], g["bp_iteration"])
    assert np.array_equal(pm, g["min_pm"])
    assert dec.counters()["osd_shots"] == 0
    e = dec.decode(g["synd"][0])
    assert np.array_equal(e, g["dec"][0]) and dec.converge == g["conv"][0]


def test_osd_window_single_shot_properties():
    from slidingwindowdecoder_b200 import osd_window
    g = load_golden("c2_w1_osdw_cs10")
    dec = osd_window(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    i = int(np.nonzero(g["conv"] == 0)[0][0])
    e = dec.decode(g["synd"][i])
    assert np.array_equal(e.astype(np.uint8), g["dec"][i])
    assert dec.converge == 0 and dec.min_pm == g["min_pm"][i] and dec.bp_iteration == g["bp_iteration"][i]
    assert np.array_equal(dec.osd0_decoding.astype(np.uint8), g["osd0"][i])
    assert np.array_equal(dec.osdw_decoding.astype(np.uint8), g["dec"][i])
    H = g["mat"].toarray().astype(np.int64)
    assert not ((H @ e + g["synd"][i]) % 2).any()          # OSD always reproduces the syndrome
    with pytest.raises(ValueError):
        osd_window(g["mat"], channel_probs=g["priors"], osd_method="osd_cs", osd_order=10 ** 6)


@pytest.fixture(scope="module")
def c4_window():
    """[[288,12,18]] p=0.003, 6 rounds (same window shapes as 18 rounds), (W,F)=(4,1): middle window 576 x 4896."""
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import sample_dem
    code, A, B = bb_code(288)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 6)))
    plan = build_windows(chk, obs, pri, code.N, W=4, F=1, method=1)
    w = plan.windows[1]
    assert w.mat.shape == (576, 4896) and w.mat.nnz == 16992
    det, _, _ = sample_dem(plan.chk, plan.obs, plan.priors, 400, np.random.default_rng(288))
    s = det[:, w.row0:w.row1]
    return w, s[s.any(axis=1)][:160]


def test_c4_large_window_osd(c4_window, oracle_mod):
    """Config 4: BP + OSD-CS10 on the large [[288,12,18]] window, bit-exact vs the oracle."""
    from slidingwindowdecoder_b200 import osd_window
    w, synd = c4_window
    kw = dict(pre_max_iter=8, post_max_iter=200, ms_scaling_factor=1.0, osd_method="osd_cs", osd_order=10)
    dec = osd_window(w.mat, channel_probs=w.prior, **kw)
    corr, conv, pm = dec.decode_batch(synd, return_pm=True)
    orc = oracle_mod.Oracle(w.mat, w.prior)
    n_osd = 0
    for i in range(len(synd)):
        r = orc.osd_window(synd[i], **kw)
        assert conv[i] == r["converge"], i
        assert np.array_equal(corr[i], r["dec"].astype(np.uint8)), i
        assert pm[i] == r["min_pm"], i
        n_osd += int(r["stats"].stage == 2)
    assert n_osd > 0
    H = w.mat.toarray().astype(np.int64)
    assert not ((corr.astype(np.int64) @ H.T + synd) % 2).any()        # OSD: every output reproduces its syndrome


def test_c4_large_window_gdg(c4_window, oracle_mod):
    from slidingwindowdecoder_b200 import bpgdg_decoder
    w, synd = c4_window
    kw = dict(max_iter=8, max_tree_depth=4, max_side_depth=20, max_step=40, max_tree_branch_step=30, max_side_branch_step=20,
              multi_thread=True, low_error_mode=True)
    dec = bpgdg_decoder(w.mat, channel_probs=w.prior, **kw)
    corr, conv = dec.decode_batch(synd[:64])
    orc = oracle_mod.Oracle(w.mat, w.prior)
    o_dec, o_conv, _, _ = orc.bpgdg_batch(synd[:64], **kw)
    assert np.array_equal(conv, o_conv.astype(np.uint8))
    assert np.array_equal(corr, o_dec.astype(np.uint8))


def _random_pcm(m, n, rng, wmin, wmax):
    """Random sparse PCM with column weights in [wmin, wmax] (SHYPS-like: heavy columns, long rows)."""
    H = np.zeros((m, n), dtype=np.uint8)
    for c in range(n):
        H[rng.choice(m, size=int(rng.integers(wmin, wmax + 1)), replace=False), c] = 1
    return H


@pytest.mark.parametrize("kind", ["gdg_mt", "gdg_st", "bpgd", "osd_cs", "osd_e"])
def test_heavy_columns_long_rows(kind, oracle_mod):
    """Column weight up to 12 (DMAX=16 kernels) and rows longer than 64 (generic check update), as in the SHYPS DEMs
    (r=4: row weight <= 88, column weight <= 12; SHYPS.ipynb:212)."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder, osd_window
    rng = np.random.default_rng(99)
    m, n = 63, 588
    H = _random_pcm(m, n, rng, 2, 12)
    assert H.sum(axis=1).max() > 64
    pri = 0.004 * (1 + rng.random(n))
    err = (rng.random((300, n)) < pri * 1.5).astype(np.int64)
    synd = (err @ H.T % 2).astype(np.uint8)
    orc = oracle_mod.Oracle(H, pri)
    if kind.startswith("gdg"):
        kw = dict(max_iter=8, multi_thread=(kind == "gdg_mt"))
        corr, conv = bpgdg_decoder(H, channel_probs=pri, **kw).decode_batch(synd)
        o_dec, o_conv, _, _ = orc.bpgdg_batch(synd, **kw)
    elif kind == "bpgd":
        kw = dict(max_iter=8, ms_scaling_factor=0.9, max_iter_per_step=6, max_step=25, gd_factor=0.9)
        corr, conv = bpgd_decoder(H, channel_probs=pri, **kw).decode_batch(synd)
        o = [orc.bpgd(s, **kw) for s in synd]
        o_dec = np.array([x[0] for x in o]); o_conv = np.array([x[1] for x in o])
    else:
        kw = dict(pre_max_iter=8, post_max_iter=40, ms_scaling_factor=0.9,
                  osd_method="osd_cs" if kind == "osd_cs" else "osd_e", osd_order=10 if kind == "osd_cs" else 5)
        corr, conv = osd_window(H, channel_probs=pri, **kw).decode_batch(synd)
        o = [orc.osd_window(s, **kw) for s in synd]
        o_dec = np.array([x["dec"] for x in o]); o_conv = np.array([x["converge"] for x in o])
    assert np.array_equal(conv, o_conv.astype(np.uint8))
    bad = np.nonzero((corr != o_dec.astype(np.uint8)).any(axis=1))[0]
    assert len(bad) == 0, f"shots {bad[:10]}"


@pytest.mark.parametrize("seed", list(range(24)))
def test_random_graphs_all_kinds_all_paths(seed, oracle_mod, monkeypatch):
    """Fuzz: random sparse check matrices of ragged shapes (m from 5 to 150, n not a multiple of anything, column weights 1..9, a few
    no empty rows: the reference requires deg > 0, random new_n, scaling factors, tree depths, OSD orders), random syndromes - some of them not in the
    column space of H -, every decoder kind, and on odd seeds the large-graph code paths forced (HBM-streamed BP, big radix select,
    large-T OSD layout).  Bit-exact vs the CPU oracle: corrections, converge flags, path metrics."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder, osd_window
    rng = np.random.default_rng(1000 + seed)
    m = int(rng.integers(5, 150)); n = int(rng.integers(m + 3, 6 * m + 40))
    wmax = int(rng.integers(2, 10))
    H = _random_pcm(m, n, rng, 1, min(wmax, m))
    for r in np.nonzero(H.sum(axis=1) == 0)[0]:          # the reference requires every check to have a column (osd_window.pyx:117)
        H[r, int(rng.integers(0, n))] = 1
    pri = 10 ** rng.uniform(-3, -1.2, size=n)
    B = 96
    err = (rng.random((B, n)) < pri * rng.uniform(0.5, 3.0)).astype(np.int64)
    synd = (err @ H.T % 2).astype(np.uint8)
    synd[::7] ^= (rng.random((len(synd[::7]), m)) < 0.05).astype(np.uint8)          # not necessarily a syndrome of anything
    if seed % 2:
        for k in ("SWD_FORCE_STREAM", "SWD_FORCE_BIG_SORT", "SWD_FORCE_BIG_OSD"):
            monkeypatch.setenv(k, "1")
    orc = oracle_mod.Oracle(H, pri)
    new_n = None if seed % 3 else int(rng.integers(max(2, m // 2), n + 1))
    f = float(rng.choice([1.0, 0.9, 0.625]))
    # multi-thread / single-thread GDG
    for mt in (True, False):
        kw = dict(max_iter=int(rng.integers(0, 12)), ms_scaling_factor=f, gdg_factor=f, max_iter_per_step=int(rng.integers(2, 8)),
                  max_step=int(rng.integers(3, 20)), max_tree_depth=int(rng.integers(1, 4)), max_side_depth=int(rng.integers(4, 9)),
                  max_tree_branch_step=int(rng.integers(2, 8)), max_side_branch_step=int(rng.integers(2, 8)), multi_thread=mt,
                  low_error_mode=bool(seed & 4), new_n=new_n)
        kw["max_step"] = max(kw["max_step"], kw["max_tree_depth"])
        corr, conv, pm = bpgdg_decoder(H, channel_probs=pri, **kw).decode_batch(synd, return_pm=True)
        o_dec, o_conv, o_pm, _ = orc.bpgdg_batch(synd, **kw)
        assert np.array_equal(conv, o_conv.astype(np.uint8)), (seed, mt)
        assert np.array_equal(corr, o_dec.astype(np.uint8)), (seed, mt)
        if mt:
            assert np.array_equal(pm[pm < 9999.0], o_pm[pm < 9999.0])
    # BPGD
    kw = dict(max_iter=int(rng.integers(1, 10)), ms_scaling_factor=f, max_iter_per_step=int(rng.integers(2, 8)), max_step=int(rng.integers(3, 30)),
              gd_factor=f, new_n=new_n)
    corr, conv = bpgd_decoder(H, channel_probs=pri, **kw).decode_batch(synd)
    o = [orc.bpgd(x, **kw) for x in synd]
    assert np.array_equal(conv, np.array([x[1] for x in o]).astype(np.uint8)) and np.array_equal(corr, np.array([x[0] for x in o]).astype(np.uint8)), seed
    # osd_window: OSD-0 / CS / E / BP only
    for meth, order in (("osd_0", 0), ("osd_cs", int(rng.integers(0, 6))), ("osd_e", int(rng.integers(0, 4))), ("osd_cs", -1)):
        kw = dict(pre_max_iter=int(rng.integers(0, 10)), post_max_iter=int(rng.integers(0, 40)), ms_scaling_factor=f, osd_method=meth,
                  osd_order=order, new_n=new_n)
        try:
            dec = osd_window(H, channel_probs=pri, **kw)
        except ValueError as e:                      # osd_order > new_n - rank (the reference raises the same way)
            assert "OSD order" in str(e)
            continue
        corr, conv, pm = dec.decode_batch(synd, return_pm=True)
        o_dec, o_conv, o_pm, _ = orc.osd_window_batch(synd, **kw)
        assert np.array_equal(conv, np.asarray(o_conv).astype(np.uint8)), (seed, meth, order)
        assert np.array_equal(corr, np.asarray(o_dec).astype(np.uint8)), (seed, meth, order)
        assert np.array_equal(pm, o_pm), (seed, meth, order)


def test_chunked_workspace_gives_identical_results(monkeypatch):
    """Batches larger than the workspace capacity are decoded in chunks (SWD_WS_BYTES caps the workspace)."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    g = load_golden("c2_w1_gdg_mt1")
    synd = np.concatenate([g["synd"]] * 3)
    ref, refc = bpgdg_decoder(g["mat"], channel_probs=g["priors"], **g["kwargs"]).decode_batch(synd)
    monkeypatch.setenv("SWD_WS_BYTES", str(40 << 20))
    small = bpgdg_decoder(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    corr, conv = small.decode_batch(synd)
    assert np.array_equal(corr, ref) and np.array_equal(conv, refc)
    go = load_golden("c2_w1_osdw_cs10")
    so = np.concatenate([go["synd"]] * 3)
    d = osd_window(go["mat"], channel_probs=go["priors"], **go["kwargs"])
    corr, conv, pm = d.decode_batch(so, return_pm=True)
    out = d.last_outputs()
    assert np.array_equal(corr, np.concatenate([go["dec"]] * 3))
    assert np.array_equal(pm, np.concatenate([go["min_pm"]] * 3))
    assert np.array_equal(out["bp_iteration"], np.concatenate([go["bp_iteration"]] * 3))


def test_bposd_facade_matches_osd_window_semantics(oracle_mod):
    """`BpOsdDecoder(max_iter, osd_method, osd_order)` == osd_window(pre_max_iter=max_iter, post_max_iter=0, new_n=n)."""
    from slidingwindowdecoder_b200 import BpOsdDecoder
    g = load_golden("c2_w1_osdw_cs10")          # middle window: full row rank, every syndrome has a solution
    dec = BpOsdDecoder(g["mat"], channel_probs=list(g["priors"]), max_iter=30, bp_method="minimum_sum", ms_scaling_factor=1.0,
                       osd_method="OSD_CS", osd_order=10)
    synd = g["synd"][:200]
    corr, conv = dec.decode_batch(synd)
    orc = oracle_mod.Oracle(g["mat"], g["priors"])
    kw = dict(pre_max_iter=30, post_max_iter=0, ms_scaling_factor=1.0, new_n=g["mat"].shape[1], osd_method="osd_cs", osd_order=10)
    for i, s in enumerate(synd):
        r = orc.osd_window(s, **kw)
        assert conv[i] == r["converge"] and np.array_equal(corr[i], r["dec"].astype(np.uint8)), i
    H = g["mat"].toarray().astype(np.int64)
    assert not ((corr.astype(np.int64) @ H.T + synd) % 2).any()


def test_device_dem_sampler_matches_numpy_restatement():
    """swd_window_sample (Philox4x32-10, one Bernoulli per DEM column) against oracle/philox.py: bit-exact errors,
    detectors and observables; the stream is a pure function of (seed, absolute shot index)."""
    import torch
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    from oracle.philox import sample_dem
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 6)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    swd = SlidingWindowDecoder(plan, decoder="gdg", max_iter=8, multi_thread=True)
    det, ob, err = swd.sample_device(700, seed=(7 << 32) + 3, shot_offset=12345, return_errors=True)
    rdet, rob, rerr = sample_dem(plan.chk, plan.obs, plan.priors, 700, seed=(7 << 32) + 3, shot_offset=12345)
    assert np.array_equal(err.cpu().numpy(), rerr)
    assert np.array_equal(det.cpu().numpy(), rdet)
    assert np.array_equal(ob.cpu().numpy(), rob)
    det2, ob2 = swd.sample_device(300, seed=(7 << 32) + 3, shot_offset=12345 + 400)
    assert torch.equal(det2, det[400:]) and torch.equal(ob2, ob[400:])
    det3, _ = swd.sample_device(300, seed=8, shot_offset=12345 + 400)
    assert not torch.equal(det3, det2)
    # the sampled batch decodes like any other input
    res = swd.decode_device(det.clone(), ob.clone())
    assert int(res["counts"][1]) <= 700


def test_last_window_bposd_redecode_matches_reference_loop(oracle_mod):
    """guessing.py:149-158,229-236: after the GDG pass the last window is decoded again with BP(200) + OSD-CS10 on the same
    residual syndrome and a second pair of counts is reported.  Checked against the same loop run with the oracle
    (osd_window semantics with new_n = n and no second BP stage, as the BpOsdDecoder facade defines them)."""
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder, sample_dem
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.004, 6)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    det, ob, _ = sample_dem(plan.chk, plan.obs, plan.priors, 600, np.random.default_rng(21))
    kw = dict(max_iter=8, multi_thread=True)
    for streams in (1, 2):
        swd = SlidingWindowDecoder(plan, decoder="gdg", last_window_osd=True, streams=streams, **kw)
        res = swd.decode(det, ob)
        oracles = {}
        state = {}

        def decode_window(w, synd):
            if w.index not in oracles:
                oracles[w.index] = oracle_mod.Oracle(w.mat, w.prior)
            if w.last:
                state["synd"] = np.array(synd, dtype=np.uint8)
            d, c, _, _ = oracles[w.index].bpgdg_batch(synd, **kw)
            return d, c

        ref = oracle_mod.sliding_window_reference(plan, det, ob, decode_window)
        assert res["flagged"] == int(ref["flagged"].sum()) and res["failed"] == int(ref["failed"].sum())
        w = plan.windows[-1]
        d2, _, _, _ = oracles[w.index].osd_window_batch(state["synd"], pre_max_iter=200, post_max_iter=0, new_n=w.mat.shape[1],
                                                        osd_method="osd_cs", osd_order=10)
        total = ref["total_e_hat"].copy()
        total[:, w.col0:w.col0 + w.ncommit] = d2[:, :w.ncommit]
        chkd = np.asarray(plan.chk.todense()).astype(np.int64); obd = np.asarray(plan.obs.todense()).astype(np.int64)
        flagged = ((det.astype(np.int64) + total @ chkd.T) % 2).any(axis=1)
        logical = ((ob.astype(np.int64) + total @ obd.T) % 2).any(axis=1)
        assert res["flagged_last_window_osd"] == int(flagged.sum())
        assert res["failed_last_window_osd"] == int(np.logical_or(flagged, logical).sum())


def test_full_size_pipeline_properties_and_logical_error_rate(oracle_mod):
    """BASELINE configs[2] at bench size: [[144,12,12]] p=0.003, 12 rounds, (3,1), 65536 device-sampled shots.
    Size-independent properties: (i) the residual syndrome after all commits equals det + chk . total_e_hat, and a shot
    is flagged exactly when that residual is non-zero; (ii) results do not depend on the number of streams nor on the
    workspace chunking; (iii) 4096 of those shots through the reference's window loop with the CPU oracle (one process per
    host core): committed corrections of all 11 windows, per-window non-convergence and failure counts are EQUAL - which
    also puts the logical error rate inside any confidence interval of the reference's (north_star)."""
    import torch
    import bench
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    bench.select_workload("c3_gdg")
    plan = bench.build_plan()
    kw = bench.WL["kw"]
    swd = SlidingWindowDecoder(plan, decoder="gdg", streams=2, **kw)
    shots = 65536
    det, obs = swd.sample_device(shots, seed=2024)
    d1, o1 = det.clone(), obs.clone()
    out = swd.decode_device(d1, o1, return_corrections=True)
    torch.cuda.synchronize()
    counts = out["counts"].cpu().numpy()
    # (i) residuals recomputed densely on the device for a slice
    sl = slice(0, 8192)
    chk = torch.from_numpy(np.asarray(plan.chk.todense(), dtype=np.float32)).cuda()
    tot = out["total_e_hat"][sl].to(torch.float32)
    resid = torch.remainder(det[sl].to(torch.float32) + tot @ chk.T, 2).to(torch.uint8)
    assert torch.equal(resid, d1[sl])
    flagged = (d1 != 0).any(dim=1)
    assert int(flagged.sum()) == int(counts[0])
    logical = (o1 != 0).any(dim=1)
    assert int((flagged | logical).sum()) == int(counts[1])
    # (ii) one stream, same answer
    d2, o2 = det.clone(), obs.clone()
    out2 = swd.decode_device(d2, o2, return_corrections=True, streams=1)
    assert torch.equal(out2["total_e_hat"], out["total_e_hat"]) and torch.equal(out2["counts"], out["counts"])
    # (iii) EXACT whole-pipeline comparison at the headline configuration (VERDICT r1 #5): 4096 of the device-sampled shots go
    # through the reference's window loop (guessing.py:141-227) with the CPU oracle per window, one process per host core;
    # the committed corrections of all 11 windows, the per-window non-convergence counts and the failure counts must be equal
    n_ref = 4096
    hdet, hobs = det[:n_ref].cpu().numpy(), obs[:n_ref].cpu().numpy()
    ref = _reference_pipeline_parallel(plan, hdet, hobs, kw)
    tot_gpu = out["total_e_hat"][:n_ref].cpu().numpy()
    bad = np.nonzero((tot_gpu != ref["total_e_hat"]).any(axis=1))[0]
    assert len(bad) == 0, f"{len(bad)} of {n_ref} shots differ from the reference loop, first {bad[:5]}"
    d3, o3 = det[:n_ref].clone(), obs[:n_ref].clone()
    out3 = swd.decode_device(d3, o3)
    c3 = out3["counts"].cpu().numpy()
    assert int(c3[0]) == int(ref["flagged"].sum()) and int(c3[1]) == int(ref["failed"].sum())
    assert out3["window_unconverged"].cpu().numpy().tolist() == ref["window_unconverged"]
    assert ref["failed"].sum() > 0                         # the sample contains logical failures (p_fail ~ 0.25 %)


_PIPE = {}


def _pipe_init(plan, kw):
    from oracle import oracle as om
    _PIPE["plan"] = plan; _PIPE["kw"] = kw; _PIPE["om"] = om
    _PIPE["orc"] = [om.Oracle(w.mat, w.prior) for w in plan.windows]


def _pipe_run(args):
    det, obs = args
    om, kw = _PIPE["om"], _PIPE["kw"]

    def decode_window(w, synd):
        d, c, _, _ = _PIPE["orc"][w.index].bpgdg_batch(synd, **kw)
        return d, c
    r = om.sliding_window_reference(_PIPE["plan"], det, obs, decode_window)
    return r["flagged"], r["failed"], r["total_e_hat"].astype(np.uint8), r["window_unconverged"]


def _reference_pipeline_parallel(plan, det, obs, kw):
    """oracle.sliding_window_reference over shot shards, one process per host core"""
    import multiprocessing as mp
    import os
    procs = max(1, len(os.sched_getaffinity(0)))
    idx = [i for i in np.array_split(np.arange(det.shape[0]), procs * 4) if len(i)]
    with mp.get_context("fork").Pool(procs, initializer=_pipe_init, initargs=(plan, kw)) as pool:
        parts = pool.map(_pipe_run, [(det[i], obs[i]) for i in idx])
    return dict(flagged=np.concatenate([p[0] for p in parts]), failed=np.concatenate([p[1] for p in parts]),
                total_e_hat=np.concatenate([p[2] for p in parts]),
                window_unconverged=[int(sum(p[3][k] for p in parts)) for k in range(len(plan.windows))])


def test_simulation_data_qubit_noise_decoding_matches_oracle(oracle_mod):
    """simulation.data_qubit_noise_decoding (the reference's src/simulation.py:10-99 GDG leg, BASELINE configs[0]): same
    seeded errors through the oracle with the kwargs of simulation.py:66-82 -> identical flagged / logical counts."""
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.simulation import data_qubit_noise_decoding
    code, _, _ = bb_code(72)
    p, shots, seed = 0.05, 3000, 5
    res = data_qubit_noise_decoding(code, p, num_shots=shots, seed=seed, verbose=False)["GDG"]
    rng = np.random.default_rng(seed)
    err = (rng.random((shots, code.N)) < p).astype(np.uint8)
    synd = (err.astype(np.int64) @ code.hx.T % 2).astype(np.uint8)
    orc = oracle_mod.Oracle(code.hx, np.ones(code.N) * p)
    o_dec, o_conv, _, _ = orc.bpgdg_batch(synd, max_iter_per_step=6, gdg_factor=0.625, max_step=40, max_tree_depth=4, max_side_depth=20,
                                          max_tree_branch_step=30, max_side_branch_step=20, multi_thread=True, low_error_mode=True,
                                          max_iter=24, ms_scaling_factor=0.625, new_n=code.N)
    assert res["num_flagged"] == int((1 - o_conv.astype(np.int64)).sum())
    logical = ((((o_dec.astype(np.int64) + err) % 2) @ code.hz_perp.T) % 2).any(axis=1)
    # uniform priors: exact path-metric ties between different corrections exist (resolved by thread timing in the reference,
    # by branch order here and in the oracle) - the counts are equal because GPU and oracle share the tie rule
    assert res["num_logical"] == int(logical.sum())
    assert 0 < res["num_logical"] < shots // 2


def test_product_sum_bposd_matches_oracle_within_tolerance(oracle_mod):
    """BpOsdDecoder(bp_method="product_sum"): tanh / log come from libdevice on the GPU and from libm in the oracle, so the
    bar is the floating-point one of north_star - posterior LLRs within 1e-6 relative, decisions equal on >= 99.9 % of
    the shots (parity with the third-party ldpc package itself is unpinned)."""
    from slidingwindowdecoder_b200 import BpOsdDecoder
    g = load_golden("c2_w1_osdw_cs10")
    H, pri, synd = g["mat"], g["priors"], g["synd"][:400]
    dec = BpOsdDecoder(H, channel_probs=list(pri), max_iter=30, bp_method="product_sum", osd_method="OSD_CS", osd_order=10)
    corr, conv = dec.decode_batch(synd)
    out = dec.last_outputs(len(synd))
    orc = oracle_mod.Oracle(H, pri)
    oracle_mod.set_bp_method("product_sum")
    try:
        same_bp, same_final, worst = 0, 0, 0.0
        for i in range(len(synd)):
            r = orc.osd_window(synd[i], pre_max_iter=30, post_max_iter=0, new_n=H.shape[1], osd_method="osd_cs", osd_order=10)
            assert int(r["bp_iteration"]) == int(out["bp_iteration"][i]) or abs(int(r["bp_iteration"]) - int(out["bp_iteration"][i])) <= 1
            if int(r["bp_iteration"]) == int(out["bp_iteration"][i]):
                a, b = out["log_prob_ratios"][i], r["log_prob_ratios"]
                worst = max(worst, float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))))
            same_bp += int(np.array_equal(out["bp_decoding"][i], r["bp_decoding"].astype(np.uint8)))
            same_final += int(np.array_equal(corr[i], r["dec"].astype(np.uint8)) and int(conv[i]) == int(r["converge"]))
        assert worst < 1e-6, worst
        assert same_bp >= 0.999 * len(synd) and same_final >= 0.999 * len(synd), (same_bp, same_final)
    finally:
        oracle_mod.set_bp_method("minimum_sum")
    # every OSD output reproduces its syndrome (window matrices have full row rank)
    resid = np.asarray((H @ corr.T.astype(np.int32)).T % 2).astype(np.uint8)
    assert np.array_equal(resid, synd)


@pytest.mark.parametrize("decoder", ["gdg", "osd"])
def test_shyps_sliding_window_driver_matches_reference_loop(decoder, oracle_mod):
    """BASELINE configs[4]: SHYPS r=3 memory experiment, (3,1) windows without merged identity columns (SHYPS.ipynb cell 1),
    GDG and BP+OSD-CS10 per window: device pipeline vs the reference's loop run with the oracle, exact."""
    import bench
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder, sample_dem
    bench.select_workload("c5_gdg" if decoder == "gdg" else "c5_osd")
    try:
        plan = bench.build_plan()
        kw = bench.WL["kw"]
        det, ob, _ = sample_dem(plan.chk, plan.obs, plan.priors, 1200, np.random.default_rng(31))
        swd = SlidingWindowDecoder(plan, decoder=decoder, streams=2, **kw)
        res = swd.decode(det, ob, return_corrections=True)
        oracles = {}

        def decode_window(w, synd):
            if w.index not in oracles:
                oracles[w.index] = oracle_mod.Oracle(w.mat, w.prior)
            if decoder == "gdg":
                d, c, _, _ = oracles[w.index].bpgdg_batch(synd, **kw)
            else:
                d, c, _, _ = oracles[w.index].osd_window_batch(synd, **kw)
            return d, c

        ref = oracle_mod.sliding_window_reference(plan, det, ob, decode_window)
        assert np.array_equal(res["total_e_hat"], ref["total_e_hat"].astype(np.uint8))
        assert res["flagged"] == int(ref["flagged"].sum()) and res["failed"] == int(ref["failed"].sum())
        assert res["window_unconverged"] == ref["window_unconverged"]
    finally:
        bench.select_workload("c3_gdg")


def test_x_basis_osd_windows_match_reference_loop(oracle_mod):
    """osd.py:83,106: x-basis memory experiment, windows keep n (not 3h) un-merged columns of the next round; BP+OSD-CS10
    per window through the device pipeline vs the reference loop with the oracle, exact.  Also covers the
    single-tier launch sequence used for small batches (latency mode): a batch of 8 shots gives identical corrections."""
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder, sample_dem
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 6, z_basis=False)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1, keep_cols=code.N)
    det, ob, _ = sample_dem(plan.chk, plan.obs, plan.priors, 1000, np.random.default_rng(41))
    kw = dict(pre_max_iter=8, post_max_iter=200, osd_method="osd_cs", osd_order=10)
    swd = SlidingWindowDecoder(plan, decoder="osd", **kw)
    res = swd.decode(det, ob, return_corrections=True)
    oracles = {}

    def decode_window(w, synd):
        if w.index not in oracles:
            oracles[w.index] = oracle_mod.Oracle(w.mat, w.prior)
        d, c, _, _ = oracles[w.index].osd_window_batch(synd, **kw)
        return d, c

    ref = oracle_mod.sliding_window_reference(plan, det, ob, decode_window)
    assert np.array_equal(res["total_e_hat"], ref["total_e_hat"].astype(np.uint8))
    assert res["failed"] == int(ref["failed"].sum())
    small = swd.decode(det[:8], ob[:8], return_corrections=True)
    assert np.array_equal(small["total_e_hat"], res["total_e_hat"][:8])
    gdg = SlidingWindowDecoder(plan, decoder="gdg", max_iter=8, multi_thread=True)
    big = gdg.decode(det, ob, return_corrections=True)
    few = gdg.decode(det[:8], ob[:8], return_corrections=True)
    assert np.array_equal(few["total_e_hat"], big["total_e_hat"][:8])


def test_reference_driver_functions(oracle_mod, capsys):
    """guessing.py / osd.py as functions with their own signatures (drivers.py): the printed statistics equal what the
    reference's loops give when run with the oracle on the same (device-sampled) shots."""
    from slidingwindowdecoder_b200.drivers import sliding_window_decoder, sliding_window_osd_decoder, _plan
    from oracle.philox import sample_dem
    shots, seed = 500, 5
    res = sliding_window_decoder(72, p=0.004, num_repeat=5, num_shots=shots, max_iter=8, W=3, F=1, seed=seed)
    text = capsys.readouterr().out
    assert "Window 0, flagged Errors:" in text and "last round osd True" in text and "logical error per round:" in text
    code, plan = _plan(72, 0.004, 5, 3, 1, True, None, 1)
    det, ob, _ = sample_dem(plan.chk, plan.obs, plan.priors, shots, seed=seed)
    kw = dict(max_iter=8, multi_thread=True, max_tree_branch_step=10)
    oracles = {}

    def decode_window(w, synd):
        if w.index not in oracles:
            oracles[w.index] = oracle_mod.Oracle(w.mat, w.prior)
        d, c, _, _ = oracles[w.index].bpgdg_batch(synd, **kw)
        return d, c

    ref = oracle_mod.sliding_window_reference(plan, det, ob, decode_window)
    assert res["gdg"]["num_flagged"] == int(ref["flagged"].sum()) and res["gdg"]["num_logical"] == int(ref["failed"].sum())
    assert res["window_flagged"] == ref["window_unconverged"]
    assert sliding_window_decoder(73) is None                              # "unsupported N"
    # osd.py, shorten=True: osd_window(pre 8, post max_iter, osd_cs, order 0) per window, W=2, method=0
    r2 = sliding_window_osd_decoder(72, p=0.004, num_repeat=5, num_shots=shots, max_iter=50, W=2, F=1, method=0, shorten=True, seed=seed)
    code, plan2 = _plan(72, 0.004, 5, 2, 1, True, None, 0)
    det2, ob2, _ = sample_dem(plan2.chk, plan2.obs, plan2.priors, shots, seed=seed)
    kw2 = dict(pre_max_iter=8, post_max_iter=50, ms_scaling_factor=1.0, osd_method="osd_cs", osd_order=0)
    orc2, flagged = {}, []

    def decode_window2(w, synd):
        if w.index not in orc2:
            orc2[w.index] = oracle_mod.Oracle(w.mat, w.prior)
        d, c, _, _ = orc2[w.index].osd_window_batch(synd, **kw2)
        H = np.asarray(w.mat.todense()).astype(np.int64)
        flagged.append(int((((d.astype(np.int64) @ H.T) + np.asarray(synd).astype(np.int64)) % 2).any(axis=1).sum()))
        return d, c

    ref2 = oracle_mod.sliding_window_reference(plan2, det2, ob2, decode_window2)
    assert r2["num_logical"] == int(ref2["failed"].sum()) and r2["num_flagged"] == int(ref2["flagged"].sum())
    assert r2["window_flagged"] == flagged
    r3 = sliding_window_osd_decoder(72, p=0.004, num_repeat=5, num_shots=shots, max_iter=30, W=2, F=1, method=0, shorten=False, seed=seed)
    assert r3["window_flagged"] == [0] * len(plan2.windows)                   # OSD always reproduces the window syndrome


@pytest.mark.parametrize("name", __import__("conftest").GOLDEN_BP4)
def test_bp4_osd_matches_oracle_and_golden(name, oracle_mod):
    """bp4_osd (quaternary BP over Hx, Hz + OSD per basis): the BP stage uses exp / log1p (libdevice on the GPU, libm in
    the oracle and the reference), so the floating-point bar applies: posterior LLRs within 1e-6 relative, iteration
    counts and converge flags equal, corrections equal on >= 99.9 % of the shots (measured: all); the OSD stage is
    integer work and must reproduce its syndrome exactly."""
    from conftest import load_golden_bp4
    from slidingwindowdecoder_b200 import bp4_osd
    g = load_golden_bp4(name)
    dec = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **g["kwargs"])
    out = dec.decode_batch(g["synd_x"], g["synd_z"])
    B, n = len(g["conv"]), g["hx"].shape[1]
    assert np.array_equal(out["converge"], g["conv"])
    assert np.array_equal(out["bp_iteration"], g["bp_iteration"])
    same = (out["dec"].reshape(B, 2 * n) == g["dec"]).all(axis=1)
    assert same.mean() >= 0.999, same.mean()
    a, b = out["log_prob_ratios"][:16], g["lpr_first16"]
    assert np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))) < 1e-6
    # every returned correction reproduces both syndromes (OSD is exact GF(2) work; Hx, Hz have full row rank here or
    # the syndrome is consistent by construction)
    hx, hz = np.asarray(g["hx"].todense()).astype(np.int64), np.asarray(g["hz"].todense()).astype(np.int64)
    ex, ez = out["dec"][:, 0].astype(np.int64), out["dec"][:, 1].astype(np.int64)
    ok = (out["converge"] == 1) | (dec.osd_order >= 0)
    assert np.array_equal((ez[ok] @ hx.T) % 2, g["synd_x"][ok]) and np.array_equal((ex[ok] @ hz.T) % 2, g["synd_z"][ok])
    # single-shot API and properties
    one = dec.decode(g["synd_x"][3], g["synd_z"][3])
    assert one.shape == (2, n) and np.array_equal(one.reshape(-1).astype(np.uint8), out["dec"][3].reshape(-1))
    assert dec.converge == int(g["conv"][3]) and dec.bp_iteration == int(g["bp_iteration"][3])
    assert dec.log_prob_ratios.shape == (n, 3) and dec.osdw_decoding_x.shape == (n,)


@pytest.mark.parametrize("name", __import__("conftest").GOLDEN_CAMEL)
def test_bp4_camel_decode_matches_golden(name, oracle_mod):
    """bp4_osd.camel_decode on the GPU against the compiled reference's outputs (floating-point bar as for bp4_osd.decode:
    exp / log1p come from libdevice): converge flags and iteration counts equal, corrections equal on >= 99.9 % of the shots,
    path metrics and posteriors within 1e-6 relative.  The tied fixture has an all-ones last column (weight 36 per basis)."""
    from conftest import load_golden_bp4
    from slidingwindowdecoder_b200 import bp4_osd
    g = load_golden_bp4(name)
    dec = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **g["kwargs"])
    out = dec.camel_decode_batch(g["synd_x"], g["synd_z"])
    B, n = len(g["conv"]), g["hx"].shape[1]
    assert np.array_equal(out["converge"], g["conv"])
    assert np.array_equal(out["bp_iteration"], g["bp_iteration"])
    same = (out["dec"].reshape(B, 2 * n) == g["dec"]).all(axis=1)
    assert same.mean() >= 0.999, same.mean()
    assert np.max(np.abs(out["min_pm"] - g["min_pm"]) / np.maximum(1.0, np.abs(g["min_pm"]))) < 1e-6
    a, b = out["log_prob_ratios"][:16], g["lpr_first16"]
    assert np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))) < 1e-6
    hx, hz = np.asarray(g["hx"].todense()).astype(np.int64), np.asarray(g["hz"].todense()).astype(np.int64)
    ex, ez = out["dec"][:, 0].astype(np.int64), out["dec"][:, 1].astype(np.int64)
    ok = out["converge"] == 1
    assert np.array_equal((ez[ok] @ hx.T) % 2, g["synd_x"][ok]) and np.array_equal((ex[ok] @ hz.T) % 2, g["synd_z"][ok])
    assert not out["dec"][~ok].any()
    one = dec.camel_decode(g["synd_x"][5], g["synd_z"][5])
    assert one.shape == (2, n) and np.array_equal(one.reshape(-1).astype(np.uint8), out["dec"][5].reshape(-1))
    assert dec.converge == int(g["conv"][5]) and abs(dec.min_pm - g["min_pm"][5]) < 1e-6 * max(1.0, abs(g["min_pm"][5]))
    # decode() on the tied pair exercises the OSD on a graph with a weight-36 column
    o2 = dec.decode_batch(g["synd_x"][:64], g["synd_z"][:64])
    orc = oracle_mod.Bp4Oracle(g["hx"], g["hz"], g["px"], g["py"], g["pz"])
    agree = 0
    for i in range(64):
        o = orc.decode(g["synd_x"][i], g["synd_z"][i], **g["kwargs"])
        agree += int(np.array_equal(o["dec"].reshape(-1).astype(np.uint8), o2["dec"][i].reshape(-1)) and o["converge"] == int(o2["converge"][i]))
    assert agree >= 63, agree


@pytest.mark.parametrize("big", [False, True])
@pytest.mark.parametrize("kind", ["gdg_mt", "bpgd"])
def test_sort_select_with_many_equal_keys(kind, big, oracle_mod, monkeypatch):
    """sort_reset_kernel on a [[144,12,12]] window (n = 1728, new_n = 432): the GDG kinds radix-select the new_n smallest
    keys and sort only those; with uniform priors many columns have exactly equal posterior sums, so boundary buckets get
    crowded (ties must stay together, the crowded case falls back to the full stable argsort) - the result has to equal
    the reference's std::stable_sort order either way: corrections bit-exact vs the oracle.
    big: the selection used for n > 8192 (keys re-read from HBM, radix descent over all 64 key bits, equal keys ranked by
    index - no full-sort fall-back), forced on this window."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder
    if big:
        monkeypatch.setenv("SWD_FORCE_BIG_SORT", "1")
    g = load_golden("c3_w5_gdg_mt1")
    n = g["mat"].shape[1]
    rng = np.random.default_rng(77)
    for pri in (np.full(n, 0.003), np.where(rng.random(n) < 0.5, 0.002, 0.004)):
        synd = g["synd"][:96]
        if kind == "gdg_mt":
            kw = dict(max_iter=8, multi_thread=True)
            dec = bpgdg_decoder(g["mat"], channel_probs=pri, **kw)
            o_dec, o_conv, _, _ = oracle_mod.Oracle(g["mat"], pri).bpgdg_batch(synd, **kw)
        else:
            kw = dict(max_iter=8, max_step=25)
            dec = bpgd_decoder(g["mat"], channel_probs=pri, **kw)
            orc = oracle_mod.Oracle(g["mat"], pri)
            res = [orc.bpgd(x, **kw) for x in synd]
            o_dec, o_conv = np.array([r[0] for r in res]), np.array([r[1] for r in res])
        corr, conv = dec.decode_batch(synd)
        assert 0 < int(conv.sum())
        assert np.array_equal(conv, np.asarray(o_conv).astype(np.uint8))
        assert np.array_equal(corr, np.asarray(o_dec).astype(np.uint8))


@pytest.mark.parametrize("big", [False, True])
def test_osd_window_reset_failure_on_large_window(big, oracle_mod, monkeypatch):
    """osd_window on a [[144,12,12]] window takes the radix-select path of sort_reset_kernel, which orders only the kept
    columns; when decimating the dropped columns hits a check whose every column is dropped while its syndrome bit is 1
    (osd_window.pyx:178-181) the failure position needs the order of the dropped columns too and the kernel sorts
    everything after all.  Forced here: the columns of one check get a 1e-12 prior, its syndrome bit is set and a small
    scaling factor keeps their posteriors large.  Bit-exact vs the oracle (corrections, flags, BP decisions)."""
    from slidingwindowdecoder_b200 import osd_window
    if big:
        monkeypatch.setenv("SWD_FORCE_BIG_SORT", "1")
    g = load_golden("c3_w5_osdw_cs10")
    H = np.asarray(g["mat"].todense()) if hasattr(g["mat"], "todense") else np.asarray(g["mat"])
    pri = np.array(g["priors"], dtype=np.float64).copy()
    r0 = 17
    pri[H[r0] != 0] = 1e-12
    synd = np.array(g["synd"][:48]).copy()
    synd[::2, r0] = 1
    kw = dict(g["kwargs"]); kw["ms_scaling_factor"] = 0.1
    orc = oracle_mod.Oracle(g["mat"], pri)
    o_dec, o_conv, o_pm, _ = orc.osd_window_batch(synd, **kw)
    dec = osd_window(g["mat"], channel_probs=pri, **kw)
    corr, conv, pm = dec.decode_batch(synd, return_pm=True)
    assert np.array_equal(conv, np.asarray(o_conv).astype(np.uint8))
    assert np.array_equal(corr, np.asarray(o_dec).astype(np.uint8))
    per = [orc.osd_window(x, **kw) for x in synd]
    assert np.array_equal(dec.last_outputs()["bp_decoding"], np.array([r["bp_decoding"] for r in per]).astype(np.uint8))


@pytest.mark.parametrize("force", ["SWD_FORCE_STREAM", "SWD_FORCE_BIG_OSD"])
@pytest.mark.parametrize("name", ["c3_w5_gdg_mt1", "c3_w5_osdw_cs10", "c5_w4_osdw_cs10"])
def test_streamed_bp_equals_shared_memory_bp(name, force, monkeypatch):
    """The HBM-streamed full-window BP (swd_stream.cuh: one thread per shot, shot-interleaved messages; what graphs beyond
    one SM's shared memory run) forced on windows that also fit the shared-memory kernel: corrections, flags, path metrics,
    BP decisions, iteration counts and the posterior history must be bit-identical, and equal to the reference's goldens.
    SWD_FORCE_BIG_OSD: the same for osd_kernel's large-window layout (sort keys alias T, reduced columns / scan array in HBM);
    a GDG decoder has no OSD stage, so there the switch must leave every output unchanged."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    g = load_golden(name)
    cls = osd_window if "osdw" in name else bpgdg_decoder
    a = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    ra = a.decode_batch(g["synd"], return_pm=True)
    oa = a.last_outputs() if cls is osd_window else None
    monkeypatch.setenv(force, "1")
    b = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    rb = b.decode_batch(g["synd"], return_pm=True)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    assert np.array_equal(rb[1], g["conv"])
    if oa is not None:
        ob = b.last_outputs()
        for k in oa:
            assert np.array_equal(oa[k], ob[k]), k
        assert np.array_equal(rb[0], g["dec"])
    assert b.counters()["pre_bp_edge_iters"] == a.counters()["pre_bp_edge_iters"]


@pytest.mark.parametrize("name", ["c1_osdw_osd_cs10", "c3_w5_osdw_cs10", "c5_w4_gdg_mt1", "c4_w7_osdw_cs10"])
def test_pre_bp_static_layout_equals_csr_order(name, monkeypatch):
    """The full-window BP kernel with its host-chosen message layout (padded row starts, permuted slots inside a row, jagged
    edge map; swd_api.cu pre_layout) against the same kernel with the slots in plain CSR order (SWD_PRE_NO_LAYOUT=1): the
    check update does not depend on the order of the slots of a row, so corrections, flags, path metrics, BP decisions,
    iteration counts and the whole posterior history must be bit-identical - and equal to the reference's goldens."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    g = load_golden(name)
    cls = osd_window if "osdw" in name else bpgdg_decoder
    nshot = min(len(g["synd"]), 200)
    a = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    ra = a.decode_batch(g["synd"][:nshot], return_pm=True)
    oa = a.last_outputs() if cls is osd_window else None
    monkeypatch.setenv("SWD_PRE_NO_LAYOUT", "1")
    b = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    rb = b.decode_batch(g["synd"][:nshot], return_pm=True)
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)
    assert np.array_equal(ra[1], g["conv"][:nshot])
    if oa is not None:
        ob = b.last_outputs()
        for k in oa:
            assert np.array_equal(oa[k], ob[k]), k
        assert np.array_equal(ra[0], g["dec"][:nshot])
    assert b.counters()["pre_bp_edge_iters"] == a.counters()["pre_bp_edge_iters"]


def test_unwindowed_144_limits_lifted():
    """ADVICE r1: the un-windowed [[144,12,12]] DEM (936 x 8784, 30672 edges; IBM.ipynb:122-123) used to be rejected with
    SWD_ERR_UNSUPPORTED because its messages exceed one SM's shared memory.  It now constructs for all three kinds and a
    decode of trivial / weight-1 syndromes returns consistent corrections."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder, osd_window
    g = load_golden("g144_osdw_cs10")
    H = g["mat"].tocsc()
    synd = np.zeros((3, H.shape[0]), dtype=np.uint8)
    synd[1] = np.asarray(H[:, 100].todense()).ravel() % 2
    synd[2] = np.asarray((H[:, 7] + H[:, 4000]).todense()).ravel() % 2
    for dec in (osd_window(H, channel_probs=g["priors"], **g["kwargs"]), bpgdg_decoder(H, channel_probs=g["priors"], max_iter=16, multi_thread=True),
                bpgd_decoder(H, channel_probs=g["priors"], max_iter=16)):
        corr, conv = dec.decode_batch(synd)
        assert conv.all()
        assert not ((corr.astype(np.int64) @ H.T.toarray() + synd) % 2).any()


@pytest.mark.parametrize("stream", [False, True])
def test_shyps_r4_dem(stream, oracle_mod, monkeypatch):
    """SHYPS r = 4 memory experiment, 4 rounds: the 300 x 3825 DEM of SHYPS.ipynb:212 (row weight up to 88, column weight up to
    12 - the long-row check update and the 16-wide variable update), decoded as one window by GDG and by BP+OSD-CS10: bit-exact
    vs the oracle.  stream: the same through the HBM-streamed BP kernel (rows longer than its 64-bit sign mask)."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    from slidingwindowdecoder_b200.dem import shyps_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.sliding_window import sample_dem
    chk, obs, pri = dem_to_check_matrices(detector_error_model(shyps_memory_circuit(4, 0.002, 4)))
    assert chk.shape == (300, 3825)
    det, _, _ = sample_dem(chk, obs, pri, 200, np.random.default_rng(44))
    s = det[np.nonzero(det.any(axis=1))[0][:48]]
    if stream:
        monkeypatch.setenv("SWD_FORCE_STREAM", "1")
    orc = oracle_mod.Oracle(chk, pri)
    kw = dict(max_iter=8, multi_thread=True)
    corr, conv = bpgdg_decoder(chk, channel_probs=pri, **kw).decode_batch(s)
    o_dec, o_conv, _, _ = orc.bpgdg_batch(s, **kw)
    assert np.array_equal(conv, o_conv.astype(np.uint8)) and np.array_equal(corr, o_dec.astype(np.uint8))
    kw = dict(pre_max_iter=8, post_max_iter=100, osd_method="osd_cs", osd_order=10)
    corr, conv = osd_window(chk, channel_probs=pri, **kw).decode_batch(s)
    o_dec, o_conv, _, _ = orc.osd_window_batch(s, **kw)
    assert np.array_equal(conv, np.asarray(o_conv).astype(np.uint8)) and np.array_equal(corr, np.asarray(o_dec).astype(np.uint8))


def test_bit_packed_entry_points_equal_byte_entry_points():
    """swd_decode_batch_host_packed / _device_packed (bit-packed syndromes in, bit-packed corrections out, the layout of
    decoders.pack_bits) return exactly what the byte entry points return; SlidingWindowDecoder.decode_packed returns the packed
    image of decode(return_corrections=True)."""
    import torch
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    from slidingwindowdecoder_b200.decoders import pack_bits, unpack_bits
    for name, cls in (("c3_w5_gdg_mt1", bpgdg_decoder), ("c2_w1_osdw_cs10", osd_window), ("c5_w0_gdg_mt1", bpgdg_decoder)):
        g = load_golden(name)
        dec = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
        corr, conv, pm = dec.decode_batch(g["synd"], return_pm=True)
        pc, pconv, ppm = dec.decode_batch_packed(pack_bits(g["synd"]), return_pm=True)
        assert pc.dtype == np.uint64 and pc.shape == (len(corr), (dec.n + 63) // 64)
        assert np.array_equal(unpack_bits(pc, dec.n), corr) and np.array_equal(pconv, conv) and np.array_equal(ppm, pm)
        assert np.array_equal(pc, pack_bits(corr))                       # pad bits are zero
        t = torch.from_numpy(pack_bits(g["synd"]).view(np.int64)).cuda()
        dc, dconv = dec.decode_batch_packed(t)
        torch.cuda.synchronize()
        assert np.array_equal(dc.cpu().numpy().view(np.uint64), pc) and np.array_equal(dconv.cpu().numpy(), conv)
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.004, 5)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    swd = SlidingWindowDecoder(plan, decoder="gdg", streams=2, max_iter=8, multi_thread=True)
    det, ob = swd.sample_device(777, seed=11)
    hdet, hob = det.cpu().numpy(), ob.cpu().numpy()
    a = swd.decode(hdet, hob, return_corrections=True)
    b = swd.decode_packed(pack_bits(hdet), pack_bits(hob))
    assert (a["flagged"], a["failed"], a["window_unconverged"]) == (b["flagged"], b["failed"], b["window_unconverged"])
    assert np.array_equal(b["total_e_hat_packed"], pack_bits(a["total_e_hat"]))


@pytest.mark.parametrize("N", [360, 756])
def test_large_bb_code_windows(N, oracle_mod):
    """ADVICE r1: codes.bb_code / drivers accept N = 360 and N = 756 (guessing.py:35-37).  A (3,1) window of the [[756,16,<=34]]
    code is 1134 x 9072 with 31374 edges - beyond one SM's shared memory: pre-BP runs HBM-streamed, the column selection takes
    the n > 8192 path.  GDG and BP+OSD corrections on sampled window syndromes are bit-exact vs the oracle."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import sample_dem
    code, A, B = bb_code(N)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 4, z_basis=True)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    det, _, _ = sample_dem(plan.chk, plan.obs, plan.priors, 64, np.random.default_rng(N))
    w = plan.windows[1]
    s = det[:, w.row0:w.row1]
    s = s[np.nonzero(s.any(axis=1))[0][:10]]
    orc = oracle_mod.Oracle(w.mat, w.prior)
    kw = dict(max_iter=8, multi_thread=True)
    corr, conv = bpgdg_decoder(w.mat, channel_probs=w.prior, **kw).decode_batch(s)
    o_dec, o_conv, _, _ = orc.bpgdg_batch(s, **kw)
    assert np.array_equal(conv, o_conv.astype(np.uint8)) and np.array_equal(corr, o_dec.astype(np.uint8))
    kw = dict(pre_max_iter=8, post_max_iter=100, osd_method="osd_cs", osd_order=10)
    corr, conv = osd_window(w.mat, channel_probs=w.prior, **kw).decode_batch(s)
    o_dec, o_conv, _, _ = orc.osd_window_batch(s, **kw)
    assert np.array_equal(conv, np.asarray(o_conv).astype(np.uint8)) and np.array_equal(corr, np.asarray(o_dec).astype(np.uint8))


def test_bp4_device_pointer_entry_points_match_host_calls():
    """swd_bp4_decode_batch_device / swd_bp4_camel_decode_batch_device (torch CUDA tensors in and out, caller's stream) return
    exactly what the host-buffer calls return."""
    import torch
    from conftest import load_golden_bp4
    from slidingwindowdecoder_b200 import bp4_osd
    g = load_golden_bp4("c1_bp4_camel_tied")
    kw = dict(g["kwargs"], osd_method="osd_cs", osd_order=6)
    dec = bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **kw)
    sx, sz = g["synd_x"], g["synd_z"]
    tx, tz = torch.from_numpy(sx).cuda(), torch.from_numpy(sz).cuda()
    for host, devc in ((dec.decode_batch(sx, sz), dec.decode_batch(tx, tz)), (dec.camel_decode_batch(sx, sz), dec.camel_decode_batch(tx, tz))):
        torch.cuda.synchronize()
        assert set(host) == set(devc)
        for k in host:
            assert torch.is_tensor(devc[k]) and devc[k].is_cuda
            assert np.array_equal(host[k], devc[k].cpu().numpy()), k
