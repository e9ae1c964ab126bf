"""Per-shot channel priors (decode_batch(..., channel_llr=L) with L [B, n]): row b must decode exactly as a fresh decoder built
with channel_llr = L[b] - corrections, converge, min_pm and the osd_window outputs - on every decoder kind and kernel path."""
import ctypes as C
import zlib

import numpy as np
import pytest

from conftest import load_golden

pytestmark = pytest.mark.gpu

GDG_KW = dict(max_iter=8, multi_thread=True)
BPGD_KW = dict(max_iter=8, ms_scaling_factor=0.9, max_iter_per_step=6, max_step=25, gd_factor=0.9)
OSD_CS_KW = dict(pre_max_iter=8, post_max_iter=60, osd_method="osd_cs", osd_order=10)
OSD_E_KW = dict(pre_max_iter=8, post_max_iter=60, osd_method="osd_e", osd_order=5)


def _random_llr(base, B, rng, erase=0.02):
    """The static priors scaled by a per-shot factor, ~2 % exact zeros (erasures), a few +inf and a few negative values."""
    L = base[None, :] * rng.uniform(0.5, 1.8, size=(B, 1))
    L[rng.random(L.shape) < erase] = 0.0
    L[rng.random(L.shape) < 0.002] = np.inf
    neg = (rng.random(L.shape) < 0.003) & np.isfinite(L)
    L[neg] = -rng.uniform(0.1, 3.0, size=int(neg.sum()))
    return np.ascontiguousarray(L)


def _make(kind, H, pri, **extra):
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder, osd_window, BpOsdDecoder
    if kind == "gdg_mt":
        return bpgdg_decoder(H, channel_probs=pri, **dict(GDG_KW, **extra))
    if kind == "gdg_st":
        return bpgdg_decoder(H, channel_probs=pri, **dict(GDG_KW, multi_thread=False, **extra))
    if kind == "bpgd":
        return bpgd_decoder(H, channel_probs=pri, **dict(BPGD_KW, **extra))
    if kind == "osd_cs":
        return osd_window(H, channel_probs=pri, **dict(OSD_CS_KW, **extra))
    if kind == "osd_e":
        return osd_window(H, channel_probs=pri, **dict(OSD_E_KW, **extra))
    if kind == "facade":
        return BpOsdDecoder(H, channel_probs=list(pri), max_iter=30, osd_method="OSD_CS", osd_order=10, **extra)
    raise KeyError(kind)


def _oracle_rows(orc, kind, synd, L, n):
    """Oracle per shot with orc.llr = L[b] -> (dec [B, n], conv [B], pm [B], list of osd dicts or None)."""
    B = len(synd)
    dec = np.zeros((B, n), dtype=np.uint8); conv = np.zeros(B, dtype=np.uint8); pm = np.zeros(B); outs = []
    for b in range(B):
        orc.llr = np.ascontiguousarray(L[b])
        if kind in ("gdg_mt", "gdg_st"):
            d, c, p, _ = orc.bpgdg_batch(synd[b:b + 1], **dict(GDG_KW, multi_thread=(kind == "gdg_mt")))
            dec[b], conv[b], pm[b] = d[0], c[0], p[0]
        elif kind == "bpgd":
            d, c, p, _ = orc.bpgd(synd[b], **BPGD_KW)
            dec[b], conv[b], pm[b] = d, c, p
        else:
            kw = OSD_CS_KW if kind == "osd_cs" else OSD_E_KW if kind == "osd_e" else \
                dict(pre_max_iter=30, post_max_iter=0, new_n=n, osd_method="osd_cs", osd_order=10)
            r = orc.osd_window(synd[b], **kw)
            dec[b], conv[b], pm[b] = r["dec"], r["converge"], r["min_pm"]
            outs.append(r)
    return dec, conv, pm, (outs or None)


def _check_osd_outputs(out, ref, idx=None):
    for b, r in enumerate(ref):
        i = b if idx is None else idx[b]
        assert np.array_equal(out["bp_decoding"][i], r["bp_decoding"].astype(np.uint8)), b
        assert int(out["bp_iteration"][i]) == int(r["bp_iteration"]), b
        if r["stats"].stage == 2:
            assert np.array_equal(out["osd0_decoding"][i], r["osd0_decoding"].astype(np.uint8)), b
            assert np.array_equal(out["osdw_decoding"][i], r["osdw_decoding"].astype(np.uint8)), b
        if int(r["bp_iteration"]) >= 4:
            assert np.array_equal(out["log_prob_ratios"][i], r["log_prob_ratios"]), b


# ------------------------------------------------------------------------------------------------ 1. constant rows
@pytest.mark.parametrize("name", ["c1_gdg_default_mt1", "c3_w5_gdg_mt1", "c3_w5_gdg_mt0", "c3_w5_bpgd", "c2_w1_osdw_cs10",
                                  "c1_osdw_osd_e6", "c4_w7_osdw_cs10", "g144_osdw_cs10"])
def test_constant_rows_equal_static_path(name):
    """Rows equal to the decoder's own priors: the per-shot kernels (computed first check pass, gathered priors) give the
    static path's outputs bit for bit, including min_pm and last_outputs()."""
    from slidingwindowdecoder_b200 import bpgdg_decoder, bpgd_decoder, osd_window
    g = load_golden(name)
    cls = osd_window if "osdw" in name else bpgd_decoder if "bpgd" in name else bpgdg_decoder
    dec = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    synd = g["synd"][:256]
    c0, v0, p0 = dec.decode_batch(synd, return_pm=True)
    o0 = dec.last_outputs() if cls is osd_window else None
    L = np.ascontiguousarray(np.tile(dec.channel_llr, (len(synd), 1)))
    c1, v1, p1 = dec.decode_batch(synd, return_pm=True, channel_llr=L)
    assert np.array_equal(c0, c1) and np.array_equal(v0, v1) and np.array_equal(p0, p1)
    if o0 is not None:
        o1 = dec.last_outputs()
        for k in o0:
            assert np.array_equal(o0[k], o1[k]), k
    if name == "g144_osdw_cs10":
        assert dec.streamed_bp


# ------------------------------------------------------------------------------------------------ 2. random rows vs oracle
WINDOWS = {"c1": "c1_gdg_default_mt1", "c2": "c2_w1_gdg_mt1", "c3": "c3_w5_gdg_mt1", "c5": "c5_w4_gdg_mt1"}


@pytest.mark.parametrize("kind", ["gdg_mt", "gdg_st", "bpgd", "osd_cs", "osd_e", "facade"])
@pytest.mark.parametrize("win", sorted(WINDOWS))
def test_random_rows_match_oracle(win, kind, oracle_mod):
    g = load_golden(WINDOWS[win])
    H, pri = g["mat"], g["priors"]
    rng = np.random.default_rng(zlib.crc32(f"{win}/{kind}".encode()))
    B = 64 if win in ("c3", "c5") else 128
    synd = g["synd"][:B]
    dec = _make(kind, H, pri)
    L = _random_llr(dec.channel_llr, len(synd), rng)
    corr, conv, pm = dec.decode_batch(synd, return_pm=True, channel_llr=L)
    orc = oracle_mod.Oracle(H, pri)
    o_dec, o_conv, o_pm, o_osd = _oracle_rows(orc, kind, synd, L, H.shape[1])
    assert np.array_equal(conv, o_conv), (win, kind)
    bad = np.nonzero((corr != o_dec).any(axis=1))[0]
    assert len(bad) == 0, (win, kind, bad[:10])
    if kind == "gdg_mt":
        assert np.array_equal(pm[pm < 9999.0], o_pm[pm < 9999.0])
    if o_osd is not None:
        assert np.array_equal(pm, o_pm)
        _check_osd_outputs(dec.last_outputs(), o_osd)


def _random_pcm(m, n, rng, wmin, wmax):
    H = np.zeros((m, n), dtype=np.uint8)
    for c in range(n):
        H[rng.choice(m, size=int(rng.integers(wmin, wmax + 1)), replace=False), c] = 1
    for r in np.nonzero(H.sum(axis=1) == 0)[0]:
        H[r, int(rng.integers(0, n))] = 1
    return H


@pytest.mark.parametrize("seed", list(range(6)))
def test_random_graphs_random_rows(seed, oracle_mod, monkeypatch):
    """Random graphs as in the all-kinds fuzz test; odd seeds force the large-graph paths (streamed BP, big sort, big OSD)."""
    rng = np.random.default_rng(5000 + seed)
    m = int(rng.integers(5, 150)); n = int(rng.integers(m + 3, 6 * m + 40))
    H = _random_pcm(m, n, rng, 1, min(int(rng.integers(2, 10)), m))
    pri = 10 ** rng.uniform(-3, -1.2, size=n)
    err = (rng.random((96, n)) < pri * 2.0).astype(np.int64)
    synd = (err @ H.T % 2).astype(np.uint8)
    if seed % 2:
        for k in ("SWD_FORCE_STREAM", "SWD_FORCE_BIG_SORT", "SWD_FORCE_BIG_OSD"):
            monkeypatch.setenv(k, "1")
    orc = oracle_mod.Oracle(H, pri)
    for kind in ("gdg_mt", "gdg_st", "bpgd", "osd_cs", "osd_e"):
        try:
            dec = _make(kind, H, pri)
        except ValueError as e:            # OSD order beyond new_n - rank on a small graph
            assert "OSD order" in str(e)
            continue
        L = _random_llr(dec.channel_llr, len(synd), rng)
        corr, conv, pm = dec.decode_batch(synd, return_pm=True, channel_llr=L)
        o_dec, o_conv, o_pm, o_osd = _oracle_rows(orc, kind, synd, L, n)
        assert np.array_equal(conv, o_conv), (seed, kind)
        assert np.array_equal(corr, o_dec), (seed, kind)
        if kind == "gdg_mt":
            assert np.array_equal(pm[pm < 9999.0], o_pm[pm < 9999.0])
        if o_osd is not None:
            assert np.array_equal(pm, o_pm)


# ------------------------------------------------------------------------------------------------ 3. fresh decoders
@pytest.mark.parametrize("kind", ["gdg_mt", "osd_cs"])
def test_row_equals_fresh_decoder(kind):
    """Row b of a batched call == a decoder constructed with channel_probs = P[b] (its first check pass comes from the
    constructor's table, the batched call computes it)."""
    from slidingwindowdecoder_b200.decoders import _libm_llr
    g = load_golden("c2_w1_gdg_mt1")
    H, pri = g["mat"], g["priors"]
    n = H.shape[1]
    rng = np.random.default_rng(3)
    S = g["synd"][:8]
    P = pri[None, :] * rng.uniform(0.3, 3.0, size=(8, n))
    L = np.stack([_libm_llr(P[b], n) for b in range(8)])
    dec = _make(kind, H, pri)
    corr, conv, pm = dec.decode_batch(S, return_pm=True, channel_llr=L)
    out = dec.last_outputs() if kind == "osd_cs" else None
    for b in range(8):
        fresh = _make(kind, H, P[b])
        e = fresh.decode(S[b])
        assert np.array_equal(e.astype(np.uint8), corr[b]) and fresh.converge == conv[b], b
        assert fresh._min_pm == pm[b], b
        if out is not None:
            fo = fresh.last_outputs(1)
            for k in fo:
                assert np.array_equal(fo[k][0], out[k][b]), (b, k)


# ------------------------------------------------------------------------------------------------ 4. forced paths
@pytest.mark.parametrize("name", ["c2_w1_gdg_mt1", "c2_w1_osdw_cs10"])
def test_forced_paths_give_default_results(name, monkeypatch):
    from slidingwindowdecoder_b200 import bpgdg_decoder, osd_window
    g = load_golden(name)
    cls = osd_window if "osdw" in name else bpgdg_decoder
    synd = g["synd"][:300]
    rng = np.random.default_rng(17)
    ref_dec = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
    L = _random_llr(ref_dec.channel_llr, len(synd), rng)
    ref = ref_dec.decode_batch(synd, return_pm=True, channel_llr=L)
    ref_out = ref_dec.last_outputs() if cls is osd_window else None
    # B <= 4: the latency configuration
    small = ref_dec.decode_batch(synd[:4], return_pm=True, channel_llr=L[:4])
    for a, b in zip(small, ref):
        assert np.array_equal(a, b[:4])
    for env in ("SWD_FORCE_STREAM", "SWD_FORCE_BIG_SORT", "SWD_FORCE_BIG_OSD", "SWD_WS_BYTES"):
        with monkeypatch.context() as mp:
            mp.setenv(env, str(24 << 20) if env == "SWD_WS_BYTES" else "1")
            d = cls(g["mat"], channel_probs=g["priors"], **g["kwargs"])
            got = d.decode_batch(synd, return_pm=True, channel_llr=L)
            for a, b in zip(got, ref):
                assert np.array_equal(a, b), env
            if ref_out is not None:
                o = d.last_outputs()
                for k in o:
                    assert np.array_equal(o[k], ref_out[k]), (env, k)


def test_product_sum_rows(oracle_mod):
    """BpOsdDecoder(bp_method="product_sum"): constant rows bit-exact; random rows against the oracle with the product-sum
    tolerance of the static path (libdevice vs libm tanh / log)."""
    from slidingwindowdecoder_b200 import BpOsdDecoder
    g = load_golden("c2_w1_osdw_cs10")
    H, pri, synd = g["mat"], g["priors"], g["synd"][:200]
    dec = BpOsdDecoder(H, channel_probs=list(pri), max_iter=30, bp_method="product_sum", osd_method="OSD_CS", osd_order=10)
    c0, v0 = dec.decode_batch(synd)
    o0 = dec.last_outputs()
    c1, v1 = dec.decode_batch(synd, channel_llr=np.ascontiguousarray(np.tile(dec.channel_llr, (len(synd), 1))))
    o1 = dec.last_outputs()
    assert np.array_equal(c0, c1) and np.array_equal(v0, v1)
    for k in o0:
        assert np.array_equal(o0[k], o1[k]), k
    L = _random_llr(dec.channel_llr, len(synd), np.random.default_rng(23), erase=0.0)
    corr, conv = dec.decode_batch(synd, channel_llr=L)
    out = dec.last_outputs(len(synd))
    orc = oracle_mod.Oracle(H, pri)
    oracle_mod.set_bp_method("product_sum")
    try:
        same_bp, same_final, worst = 0, 0, 0.0
        for i in range(len(synd)):
            orc.llr = np.ascontiguousarray(L[i])
            r = orc.osd_window(synd[i], pre_max_iter=30, post_max_iter=0, new_n=H.shape[1], osd_method="osd_cs", osd_order=10)
            assert abs(int(r["bp_iteration"]) - int(out["bp_iteration"][i])) <= 1
            if int(r["bp_iteration"]) == int(out["bp_iteration"][i]):
                a, b = out["log_prob_ratios"][i], r["log_prob_ratios"]
                fin = np.isfinite(b)
                assert np.array_equal(a[~fin], b[~fin])
                worst = max(worst, float(np.max(np.abs(a[fin] - b[fin]) / np.maximum(1.0, np.abs(b[fin])), initial=0.0)))
            same_bp += int(np.array_equal(out["bp_decoding"][i], r["bp_decoding"].astype(np.uint8)))
            same_final += int(np.array_equal(corr[i], r["dec"].astype(np.uint8)) and int(conv[i]) == int(r["converge"]))
        assert worst < 1e-6, worst
        assert same_bp >= 0.999 * len(synd) and same_final >= 0.999 * len(synd), (same_bp, same_final)
    finally:
        oracle_mod.set_bp_method("minimum_sum")


# ------------------------------------------------------------------------------------------------ 5. entry points
@pytest.mark.parametrize("kind", ["gdg_mt", "osd_cs"])
def test_entry_points_agree(kind):
    import torch
    from slidingwindowdecoder_b200.decoders import pack_bits, unpack_bits
    g = load_golden("c2_w1_gdg_mt1")
    H, pri = g["mat"], g["priors"]
    m, n = H.shape
    synd = g["synd"][:300]
    dec = _make(kind, H, pri)
    L = _random_llr(dec.channel_llr, len(synd), np.random.default_rng(8))
    c0, v0, p0 = dec.decode_batch(synd, return_pm=True, channel_llr=L)
    cp, vp, pp = dec.decode_batch_packed(pack_bits(synd), return_pm=True, channel_llr=L)
    assert np.array_equal(unpack_bits(cp, n), c0) and np.array_equal(vp, v0) and np.array_equal(pp, p0)
    dev = torch.device("cuda", 0)
    sd, Ld = torch.from_numpy(synd).to(dev), torch.from_numpy(L).to(dev)
    ct, vt, pt = dec.decode_batch(sd, return_pm=True, channel_llr=Ld)
    assert np.array_equal(ct.cpu().numpy(), c0) and np.array_equal(vt.cpu().numpy(), v0) and np.array_equal(pt.cpu().numpy(), p0)
    sp = torch.from_numpy(pack_bits(synd).view(np.int64)).to(dev)
    cpt, vpt, ppt = dec.decode_batch_packed(sp, return_pm=True, channel_llr=Ld)
    assert np.array_equal(unpack_bits(cpt.cpu().numpy().view(np.uint64), n), c0)
    assert np.array_equal(vpt.cpu().numpy(), v0) and np.array_equal(ppt.cpu().numpy(), p0)
    # without channel_llr the same decoder is unchanged
    c2, v2 = dec.decode_batch(synd)
    c3, v3 = _make(kind, H, pri).decode_batch(synd)
    assert np.array_equal(c2, c3) and np.array_equal(v2, v3)


# ------------------------------------------------------------------------------------------------ 6. sliding-window driver
@pytest.fixture(scope="module")
def c2_plan():
    from slidingwindowdecoder_b200.codes import bb_code
    from slidingwindowdecoder_b200.dem import bb_memory_circuit, detector_error_model, dem_to_check_matrices
    from slidingwindowdecoder_b200.windows import build_windows
    from slidingwindowdecoder_b200.sliding_window import sample_dem
    code, A, B = bb_code(72)
    chk, obs, pri = dem_to_check_matrices(detector_error_model(bb_memory_circuit(code, A, B, 0.003, 6)))
    plan = build_windows(chk, obs, pri, code.N, W=3, F=1, method=1)
    det, ob, _ = sample_dem(plan.chk, plan.obs, plan.priors, 240, np.random.default_rng(41))
    # row-major: decode_device works on the tensors' storage in place, and torch.from_numpy keeps numpy's strides
    return plan, np.asarray(pri), np.ascontiguousarray(det), np.ascontiguousarray(ob)


@pytest.mark.parametrize("decoder", ["gdg", "osd"])
def test_driver_matches_reference_loop(decoder, c2_plan, oracle_mod):
    import torch
    from slidingwindowdecoder_b200.decoders import _libm_llr
    from slidingwindowdecoder_b200.sliding_window import SlidingWindowDecoder
    plan, pri_dem, det, ob = c2_plan
    B, num_col = det.shape[0], len(pri_dem)
    kw = dict(max_iter=8, multi_thread=True) if decoder == "gdg" else dict(OSD_CS_KW)
    osd_kw = dict(max_iter=200, osd_method="OSD_CS", osd_order=10)
    swd = SlidingWindowDecoder(plan, decoder=decoder, streams=2, last_window_osd=osd_kw, **kw)
    L = _random_llr(oracle_mod.libm_llr(pri_dem), B, np.random.default_rng(5))      # DEM column order
    res = swd.decode(det, ob, return_corrections=True, channel_llr=L)
    Lp = L[:, plan.col_order]

    def rows(w):
        tail = _libm_llr(w.prior, w.mat.shape[1])[w.ncols_dem:]
        return np.concatenate([Lp[:, w.col0:w.col0 + w.ncols_dem], np.tile(tail, (B, 1))], axis=1)

    oracles = {}

    def decode_window(w, synd, last_osd=False):
        key = (w.index, last_osd)
        if key not in oracles:
            oracles[key] = oracle_mod.Oracle(w.mat, w.prior)
        orc, R = oracles[key], rows(w)
        n = w.mat.shape[1]
        dec, conv = np.zeros((len(synd), n), dtype=np.int64), np.zeros(len(synd), dtype=np.int64)
        for b in range(len(synd)):
            orc.llr = np.ascontiguousarray(R[b])
            if last_osd:
                r = orc.osd_window(synd[b], pre_max_iter=200, post_max_iter=0, new_n=n, osd_method="osd_cs", osd_order=10)
                dec[b], conv[b] = r["dec"], r["converge"]
            elif decoder == "gdg":
                d, c, _, _ = orc.bpgdg_batch(synd[b:b + 1], **kw)
                dec[b], conv[b] = d[0], c[0]
            else:
                r = orc.osd_window(synd[b], **kw)
                dec[b], conv[b] = r["dec"], r["converge"]
        return dec, conv

    ref = oracle_mod.sliding_window_reference(plan, det, ob, decode_window)
    assert np.array_equal(res["total_e_hat"], ref["total_e_hat"].astype(np.uint8))
    assert res["flagged"] == int(ref["flagged"].sum()) and res["failed"] == int(ref["failed"].sum())
    assert res["window_unconverged"] == ref["window_unconverged"]
    ref_osd = oracle_mod.sliding_window_reference(plan, det, ob, lambda w, s: decode_window(w, s, last_osd=w.last))
    assert res["flagged_last_window_osd"] == int(ref_osd["flagged"].sum())
    assert res["failed_last_window_osd"] == int(ref_osd["failed"].sum())
    # streams = 1 and 2 give identical results
    dev = torch.device("cuda", 0)
    outs = []
    for ns in (1, 2):
        d_det, d_obs = torch.from_numpy(det).to(dev), torch.from_numpy(ob).to(dev)
        o = swd.decode_device(d_det, d_obs, return_corrections=True, streams=ns, channel_llr=torch.from_numpy(L).to(dev))
        outs.append({k: v.cpu().numpy() for k, v in o.items()})
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k
    assert np.array_equal(outs[0]["total_e_hat"], res["total_e_hat"])
    # rows built from the plan's own priors == a call without channel_llr
    L0 = np.ascontiguousarray(np.tile(oracle_mod.libm_llr(pri_dem), (B, 1)))
    a = swd.decode(det, ob, return_corrections=True, channel_llr=L0)
    b = swd.decode(det, ob, return_corrections=True)
    for k in b:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


# ------------------------------------------------------------------------------------------------ 7. argument errors
def test_argument_errors():
    import torch
    from slidingwindowdecoder_b200 import _lib
    g = load_golden("c2_w1_gdg_mt1")
    H, pri = g["mat"], g["priors"]
    n = H.shape[1]
    synd = np.ascontiguousarray(g["synd"][:8])
    dec = _make("gdg_mt", H, pri)
    L = np.ascontiguousarray(np.tile(dec.channel_llr, (8, 1)))
    dev = torch.device("cuda", 0)
    with pytest.raises(ValueError):
        dec.decode_batch(synd, channel_llr=L[:, :-1])                         # wrong shape
    with pytest.raises(ValueError):
        dec.decode_batch(synd, channel_llr=L[:7])
    with pytest.raises(ValueError):
        dec.decode_batch(synd, channel_llr=L.astype(np.float32))              # wrong dtype
    bad = L.copy(); bad[3, 5] = np.nan
    with pytest.raises(ValueError):
        dec.decode_batch(synd, channel_llr=bad)                               # NaN in a host array
    with pytest.raises(ValueError):
        dec.decode_batch_packed(__import__("slidingwindowdecoder_b200.decoders", fromlist=["pack_bits"]).pack_bits(synd), channel_llr=bad)
    with pytest.raises(ValueError):
        dec.decode_batch(synd, channel_llr=torch.from_numpy(L).to(dev))       # host syndromes, device priors
    with pytest.raises(ValueError):
        dec.decode_batch(torch.from_numpy(synd).to(dev), channel_llr=L)       # device syndromes, host priors
    with pytest.raises(ValueError):
        dec.decode_batch(torch.from_numpy(synd).to(dev), channel_llr=torch.from_numpy(L))      # a CPU tensor
    with pytest.raises(ValueError):
        dec.decode_batch(torch.from_numpy(synd).to(dev), channel_llr=torch.from_numpy(L).to(dev).float())
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            dec.decode_batch(torch.from_numpy(synd).to(dev), channel_llr=torch.from_numpy(L).to("cuda:1"))   # wrong device
    # NULL priors at the C-ABI
    lib = _lib.load()
    corr = np.empty((8, n), dtype=np.uint8); conv = np.empty(8, dtype=np.uint8)
    assert lib.swd_decode_batch_host_llr(dec._handle, synd.ctypes.data, 8, corr.ctypes.data, conv.ctypes.data, None, None) == _lib.ERR_INVALID
    assert lib.swd_decode_batch_host_packed_llr(dec._handle, synd.ctypes.data, 8, corr.ctypes.data, conv.ctypes.data, None, None) == _lib.ERR_INVALID
    assert lib.swd_decode_batch_device_llr(dec._handle, synd.ctypes.data, 8, corr.ctypes.data, conv.ctypes.data, None, None,
                                           C.c_void_p(0)) == _lib.ERR_INVALID
    assert lib.swd_decode_batch_device_packed_llr(dec._handle, synd.ctypes.data, 8, corr.ctypes.data, conv.ctypes.data, None, None,
                                                  C.c_void_p(0)) == _lib.ERR_INVALID
