"""Per-shot channel priors for bp4_osd (decode_batch / camel_decode_batch(..., channel_llr=L) with L [5, B, n]): row b of
the five planes (llr_x, llr_y, llr_z, prior_llr_x, prior_llr_z) must decode shot b exactly as a bp4_osd built with those
priors would, in every output."""
import ctypes as C
import math
import zlib

import numpy as np
import pytest

from conftest import GOLDEN_BP4, GOLDEN_CAMEL, load_golden_bp4

pytestmark = pytest.mark.gpu

DECODE_KEYS = ("dec", "converge", "bp_decoding", "osd0", "log_prob_ratios", "bp_iteration")
CAMEL_KEYS = ("dec", "converge", "min_pm", "log_prob_ratios", "bp_iteration")


def _make(g, **kw):
    from slidingwindowdecoder_b200 import bp4_osd
    return bp4_osd(g["hx"], g["hz"], channel_probs_x=g["px"], channel_probs_y=g["py"], channel_probs_z=g["pz"], **dict(g["kwargs"], **kw))


def _llr5(px, py, pz):
    """[5, n] LLRs of one shot with libm's log, in the order and arithmetic of bp4_osd.__init__ / Bp4Oracle.__init__."""
    n = len(px)
    L = np.empty((5, n))
    for v in range(n):
        x, y, z = float(px[v]), float(py[v]), float(pz[v])
        num = 1.0 - (x + y + z)
        L[0, v] = math.log(num / x); L[1, v] = math.log(num / y); L[2, v] = math.log(num / z)
        L[3, v] = math.log((1.0 - (x + y)) / (x + y)); L[4, v] = math.log((1.0 - (z + y)) / (z + y))
    return L


def _random_shots(g, B, rng, erase=0.05):
    """Per-shot depolarizing channels: the fixture's probabilities times a per-shot scale, x and z biased independently per
    shot (px != pz), ~5 % of the qubits erased (px = py = pz = 1/4, all five LLRs exactly 0.0).  Errors and syndromes are
    sampled from the same per-shot probabilities.  -> (probs [3, B, n], L [5, B, n], synd_x, synd_z, e_x, e_z)"""
    n = g["hx"].shape[1]
    scale = rng.uniform(0.4, 2.0, size=(B, 1))
    px = g["px"][None, :] * scale * rng.uniform(0.5, 1.6, size=(B, 1))
    py = g["py"][None, :] * scale
    pz = g["pz"][None, :] * scale * rng.uniform(0.5, 1.6, size=(B, 1))
    er = rng.random((B, n)) < erase
    px[er] = py[er] = pz[er] = 0.25
    L = np.stack([_llr5(px[b], py[b], pz[b]) for b in range(B)], axis=1)
    assert (L[:, er] == 0.0).all()
    r = rng.random((B, n))
    isx, isy, isz = r < px, (r >= px) & (r < px + py), (r >= px + py) & (r < px + py + pz)
    ex, ez = (isx | isy).astype(np.int64), (isy | isz).astype(np.int64)
    hx, hz = np.asarray(g["hx"].todense()).astype(np.int64), np.asarray(g["hz"].todense()).astype(np.int64)
    sx, sz = (ez @ hx.T % 2).astype(np.uint8), (ex @ hz.T % 2).astype(np.uint8)
    return np.stack([px, py, pz]), np.ascontiguousarray(L), sx, sz, ex, ez


def _const_rows(dec, B):
    return np.ascontiguousarray(np.repeat(dec.channel_llr[:, None, :], B, axis=1))


def _assert_bitwise(a, b, keys):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape and np.array_equal(x, y), k


def _to_host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


# ------------------------------------------------------------------------------------------------ 1. constant rows
@pytest.mark.parametrize("name", GOLDEN_BP4)
def test_constant_rows_equal_static_decode(name):
    """Rows equal to the decoder's own priors give the static path's outputs bit for bit (same arithmetic, same order)."""
    g = load_golden_bp4(name)
    dec = _make(g)
    assert dec.channel_llr.shape == (5, dec.n)
    a = dec.decode_batch(g["synd_x"], g["synd_z"])
    b = dec.decode_batch(g["synd_x"], g["synd_z"], channel_llr=_const_rows(dec, len(g["synd_x"])))
    _assert_bitwise(a, b, DECODE_KEYS)


@pytest.mark.parametrize("name", GOLDEN_CAMEL)
def test_constant_rows_equal_static_camel(name):
    g = load_golden_bp4(name)
    dec = _make(g)
    a = dec.camel_decode_batch(g["synd_x"], g["synd_z"])
    b = dec.camel_decode_batch(g["synd_x"], g["synd_z"], channel_llr=_const_rows(dec, len(g["synd_x"])))
    _assert_bitwise(a, b, CAMEL_KEYS)


# ------------------------------------------------------------------------------------------------ 2. random rows vs oracle
def _rel(a, b):
    return np.abs(a - b) / np.maximum(1.0, np.abs(b))


@pytest.mark.parametrize("name,method", [("c1_bp4_osd_cs8", "decode"), ("c1_bp4_osd_e5", "decode"),
                                         ("c1_bp4_camel_tied", "decode"), ("c1_bp4_camel_tied", "camel")])
def test_random_rows_match_oracle(name, method, oracle_mod):
    """Per-shot scale, x / z bias and 5 % erasures against the CPU oracle with its five arrays set to the shot's rows.  The BP
    stage uses exp / log1p (libdevice on the GPU, libm in the oracle), so the project's floating-point bar for bp4 applies:
    converge flags and iteration counts equal, corrections equal on >= 99.9 % of the shots, posteriors (and min_pm) within
    1e-6 relative on those shots; every converged or OSD correction reproduces both syndromes."""
    g = load_golden_bp4(name)
    rng = np.random.default_rng(zlib.crc32(f"{name}/{method}".encode()))
    B = 1200
    _, L, sx, sz, _, _ = _random_shots(g, B, rng)
    dec = _make(g)
    camel = method == "camel"
    out = dec.camel_decode_batch(sx, sz, channel_llr=L) if camel else dec.decode_batch(sx, sz, channel_llr=L)
    orc = oracle_mod.Bp4Oracle(g["hx"], g["hz"], g["px"], g["py"], g["pz"])
    kw = {k: g["kwargs"][k] for k in ("max_iter", "ms_scaling_factor")} if camel else g["kwargs"]
    n = dec.n
    same = np.zeros(B, dtype=bool)
    ref_conv, ref_it = np.zeros(B, dtype=np.uint8), np.zeros(B, dtype=np.int32)
    worst_lpr = worst_pm = 0.0
    for b in range(B):
        orc.llrx, orc.llry, orc.llrz, orc.prior_x, orc.prior_z = (np.ascontiguousarray(L[k, b]) for k in range(5))
        o = orc.camel_decode(sx[b], sz[b], **kw) if camel else orc.decode(sx[b], sz[b], **kw)
        ref_conv[b], ref_it[b] = o["converge"], o["bp_iteration"]
        same[b] = np.array_equal(o["dec"].reshape(-1).astype(np.uint8), out["dec"][b].reshape(-1))
        if not camel:
            same[b] &= np.array_equal(o["bp_decoding"].astype(np.uint8), out["bp_decoding"][b])
        if same[b]:
            worst_lpr = max(worst_lpr, float(_rel(out["log_prob_ratios"][b], o["log_prob_ratios"]).max()))
            if camel:
                worst_pm = max(worst_pm, float(_rel(out["min_pm"][b], o["min_pm"])))
    assert np.array_equal(out["converge"], ref_conv)
    assert np.array_equal(out["bp_iteration"], ref_it)
    assert same.mean() >= 0.999, (same.mean(), np.nonzero(~same)[0][:10])
    assert worst_lpr < 1e-6 and worst_pm < 1e-6, (worst_lpr, worst_pm)
    hx, hz = np.asarray(g["hx"].todense()).astype(np.int64), np.asarray(g["hz"].todense()).astype(np.int64)
    ex, ez = out["dec"][:, 0].astype(np.int64), out["dec"][:, 1].astype(np.int64)
    ok = (out["converge"] == 1) if camel else (out["converge"] == 1) | (dec.osd_order >= 0)
    assert np.array_equal((ez[ok] @ hx.T) % 2, sx[ok]) and np.array_equal((ex[ok] @ hz.T) % 2, sz[ok])
    if camel:
        assert not out["dec"][out["converge"] == 0].any()
    else:
        assert (out["converge"] == 0).any(), "no shot reached the OSD stage"


# ------------------------------------------------------------------------------------------------ 3. a row == a fresh decoder
@pytest.mark.parametrize("name", ["c1_bp4_osd_cs8", "c1_bp4_osd_e5", "c1_bp4_camel_tied"])
def test_row_equals_fresh_decoder(name):
    """For a few shots, a bp4_osd built with that shot's channel_probs_x/y/z decodes it bit for bit as row b of the batch."""
    from slidingwindowdecoder_b200 import bp4_osd
    g = load_golden_bp4(name)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    B = 256
    probs, L, sx, sz, _, _ = _random_shots(g, B, rng)
    dec = _make(g)
    out = dec.decode_batch(sx, sz, channel_llr=L)
    cam = dec.camel_decode_batch(sx, sz, channel_llr=L)
    pick = list(np.nonzero(out["converge"] == 0)[0][:4]) + list(np.nonzero(out["converge"] == 1)[0][:4])
    assert len(pick) == 8
    for b in pick:
        one = bp4_osd(g["hx"], g["hz"], channel_probs_x=probs[0, b], channel_probs_y=probs[1, b], channel_probs_z=probs[2, b],
                      **g["kwargs"])
        assert np.array_equal(one.channel_llr, L[:, b])
        r = one.decode_batch(sx[b:b + 1], sz[b:b + 1])
        _assert_bitwise(r, {k: v[b:b + 1] for k, v in out.items()}, DECODE_KEYS)
        r = one.camel_decode_batch(sx[b:b + 1], sz[b:b + 1])
        _assert_bitwise(r, {k: v[b:b + 1] for k, v in cam.items()}, CAMEL_KEYS)


# ------------------------------------------------------------------------------------------------ 4. chunked OSD
@pytest.mark.parametrize("budget", [1, 256 << 10])
def test_chunked_osd_pass(budget, monkeypatch):
    """A small workspace budget splits each basis' OSD pass into several chunks (one shot per chunk at budget 1): the chunk's
    rows of planes 3 / 4 are addressed chunk-locally, and the outputs equal the one-chunk default bit for bit."""
    name = "c1_bp4_osd_cs8"
    g = load_golden_bp4(name)
    rng = np.random.default_rng(zlib.crc32(f"chunk/{budget}".encode()))
    _, L, sx, sz, _, _ = _random_shots(g, 700, rng)
    ref = _make(g).decode_batch(sx, sz, channel_llr=L)
    with monkeypatch.context() as mp:
        mp.setenv("SWD_WS_BYTES", str(budget))
        dec = _make(g)
        out = dec.decode_batch(sx, sz, channel_llr=L)
    assert (ref["converge"] == 0).sum() > 20
    _assert_bitwise(ref, out, DECODE_KEYS)


# ------------------------------------------------------------------------------------------------ 5. entry points agree
@pytest.mark.parametrize("name", ["c1_bp4_osd_e5", "c1_bp4_camel_tied"])
def test_host_and_device_entry_points_agree(name):
    """swd_bp4_*_host_llr (numpy) and swd_bp4_*_device_llr (torch, current stream) give the same outputs; so do the five
    planes given as a non-contiguous view."""
    import torch
    g = load_golden_bp4(name)
    rng = np.random.default_rng(zlib.crc32(f"entry/{name}".encode()))
    _, L, sx, sz, _, _ = _random_shots(g, 512, rng)
    dec = _make(g)
    dev = torch.device("cuda", 0)
    tx, tz, tL = (torch.from_numpy(a).to(dev) for a in (sx, sz, L))
    L_view = np.ascontiguousarray(L.transpose(1, 0, 2)).transpose(1, 0, 2)          # [B, 5, n] storage seen as [5, B, n]
    assert not L_view.flags.c_contiguous
    tL_view = torch.from_numpy(np.ascontiguousarray(L.transpose(1, 0, 2))).to(dev).transpose(0, 1)
    assert not tL_view.is_contiguous()
    for fn, keys in ((dec.decode_batch, DECODE_KEYS), (dec.camel_decode_batch, CAMEL_KEYS)):
        host = fn(sx, sz, channel_llr=L)
        _assert_bitwise(host, fn(sx, sz, channel_llr=L_view), keys)
        d1 = fn(tx, tz, channel_llr=tL)
        d2 = fn(tx, tz, channel_llr=tL_view)
        torch.cuda.synchronize()
        _assert_bitwise(host, _to_host(d1), keys)
        _assert_bitwise(host, _to_host(d2), keys)


# ------------------------------------------------------------------------------------------------ 6. argument errors
def test_argument_errors():
    import torch
    from slidingwindowdecoder_b200 import _lib
    g = load_golden_bp4("c1_bp4_camel_tied")
    dec = _make(g)
    B, n = 8, dec.n
    sx, sz = np.ascontiguousarray(g["synd_x"][:B]), np.ascontiguousarray(g["synd_z"][:B])
    L = _const_rows(dec, B)
    dev = torch.device("cuda", 0)
    tx, tz = torch.from_numpy(sx).to(dev), torch.from_numpy(sz).to(dev)
    for fn in (dec.decode_batch, dec.camel_decode_batch):
        for bad in (L[:, :-1], L[:4], L[:, :, :-1], np.ascontiguousarray(L.transpose(1, 0, 2)), L.astype(np.float32)):
            with pytest.raises(ValueError):
                fn(sx, sz, channel_llr=bad)                                    # wrong shape or dtype
        for v in (np.nan, np.inf, -np.inf):
            bad = L.copy(); bad[4, 3, 5] = v
            with pytest.raises(ValueError):
                fn(sx, sz, channel_llr=bad)                                    # non-finite value in a host array
        with pytest.raises(ValueError):
            fn(sx, sz, channel_llr=torch.from_numpy(L).to(dev))                # host syndromes, device priors
        with pytest.raises(ValueError):
            fn(tx, tz, channel_llr=L)                                          # device syndromes, host priors
        with pytest.raises(ValueError):
            fn(tx, tz, channel_llr=torch.from_numpy(L))                        # a CPU tensor
        with pytest.raises(ValueError):
            fn(tx, tz, channel_llr=torch.from_numpy(L).to(dev).float())       # wrong dtype
        with pytest.raises(ValueError):
            fn(tx, tz, channel_llr=torch.from_numpy(L[:, :-1]).to(dev))        # wrong shape
        if torch.cuda.device_count() > 1:
            with pytest.raises(ValueError):
                fn(tx, tz, channel_llr=torch.from_numpy(L).to("cuda:1"))       # wrong device
    # NULL priors at the C-ABI
    lib = _lib.load()
    dec8 = np.empty((B, 2, n), dtype=np.uint8); conv = np.empty(B, dtype=np.uint8)
    h = dec._handle
    assert lib.swd_bp4_decode_batch_host_llr(h, sx.ctypes.data, sz.ctypes.data, B, dec8.ctypes.data, conv.ctypes.data,
                                             None, None, None, None, None) == _lib.ERR_INVALID
    assert lib.swd_bp4_camel_decode_batch_host_llr(h, sx.ctypes.data, sz.ctypes.data, B, dec8.ctypes.data, conv.ctypes.data,
                                                   None, None, None, None) == _lib.ERR_INVALID
    td, tc = torch.empty((B, 2, n), dtype=torch.uint8, device=dev), torch.empty(B, dtype=torch.uint8, device=dev)
    assert lib.swd_bp4_decode_batch_device_llr(h, tx.data_ptr(), tz.data_ptr(), B, td.data_ptr(), tc.data_ptr(), None, None, None,
                                               None, None, C.c_void_p(0)) == _lib.ERR_INVALID
    assert lib.swd_bp4_camel_decode_batch_device_llr(h, tx.data_ptr(), tz.data_ptr(), B, td.data_ptr(), tc.data_ptr(), None, None,
                                                     None, None, C.c_void_p(0)) == _lib.ERR_INVALID
    # the decoder still works after the refused calls
    _assert_bitwise(dec.decode_batch(sx, sz), dec.decode_batch(sx, sz, channel_llr=L), DECODE_KEYS)
