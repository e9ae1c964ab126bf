"""Sliding-window driver: the per-window loop of the reference (guessing.py:141-227, osd.py:134-179)
re-hosted for batched decoding on one B200.

For every window: extract the window syndrome of ALL shots, decode them with one batched call,
commit the first F rounds of the correction, update the remaining syndrome with the sparse
equivalent of `new_det = (det + total_e_hat @ chk.T) % 2`, slide.  Shot data stays on the device
between windows; PyTorch is used only to own device buffers and streams.
"""
import ctypes as C

import numpy as np

from . import _lib
from .decoders import bpgdg_decoder, osd_window
from .windows import WindowPlan


def sample_dem(chk, obs, priors, shots, rng):
    """What stim's CompiledDemSampler draws (guessing.py:129-130): independent Bernoulli per DEM column.
    -> (det [shots, num_det] uint8, obs [shots, num_obs] uint8, err [shots, num_col] uint8)"""
    err = (rng.random((shots, len(priors))) < priors[None, :]).astype(np.uint8)
    e = err.astype(np.float32)
    det = (np.asarray(e @ chk.T.astype(np.float32)) % 2).astype(np.uint8)
    ob = (np.asarray(e @ obs.T.astype(np.float32)) % 2).astype(np.uint8)
    return det, ob, err


class SlidingWindowDecoder:
    """Holds one decoder per distinct window matrix (the reference rebuilds one per window,
    guessing.py:160-174) and the device-side window bookkeeping."""

    def __init__(self, plan: WindowPlan, decoder="gdg", device=0, last_window_kwargs=None, streams=1,
                 last_window_osd=None, **decoder_kwargs):
        """streams > 1: every batch is split into that many sub-batches which run the window loop on their own CUDA
        streams with their own decoder workspaces, so that one sub-batch's kernel tails (a few long branch paths
        finishing) are filled by the next sub-batch's work.  Results do not depend on `streams`."""
        import torch
        self.torch = torch
        self.plan = plan
        self.device = int(device)
        self.lib = _lib.load()
        chk = plan.chk.tocsc(); chk.sort_indices()
        obs = plan.obs.tocsc(); obs.sort_indices()
        self.num_det, self.num_col = chk.shape
        self.num_obs = obs.shape[0]
        self._chk_cp = np.ascontiguousarray(chk.indptr, dtype=np.int32)
        self._chk_ri = np.ascontiguousarray(chk.indices, dtype=np.int32)
        self._obs_cp = np.ascontiguousarray(obs.indptr, dtype=np.int32)
        self._obs_ri = np.ascontiguousarray(obs.indices, dtype=np.int32)
        i32p = C.POINTER(C.c_int32)
        self._win = C.c_void_p()
        st = self.lib.swd_window_create(self.device, self.num_det, self.num_col, self._chk_cp.ctypes.data_as(i32p),
                                        self._chk_ri.ctypes.data_as(i32p), self.num_obs, self._obs_cp.ctypes.data_as(i32p),
                                        self._obs_ri.ctypes.data_as(i32p), C.byref(self._win))
        _lib.check(st, "swd_window_create")
        cls = {"gdg": bpgdg_decoder, "osd": osd_window}.get(decoder, decoder)
        self.nstreams = max(1, int(streams))
        self.decoder_sets = []                 # [stream][window] -> decoder (windows with equal matrices share one)
        for _ in range(self.nstreams):
            decs, cache = [], []
            for w in plan.windows:
                kw = dict(decoder_kwargs)
                if w.last and last_window_kwargs:
                    kw.update(last_window_kwargs)
                found = None
                for (m0, p0, kw0, d0) in cache:
                    if kw0 == kw and m0.shape == w.mat.shape and m0.nnz == w.mat.nnz and (m0 != w.mat).nnz == 0 and np.array_equal(p0, w.prior):
                        found = d0
                        break
                if found is None:
                    found = cls(w.mat, channel_probs=w.prior, device=self.device, **kw)
                    cache.append((w.mat, w.prior, kw, found))
                decs.append(found)
            self.decoder_sets.append(decs)
        self.decoders = self.decoder_sets[0]
        self._side_streams = None
        self._llr_cache = {}                   # per-shot priors: plan column order, static noisy-column LLRs per window decoder
        # guessing.py:149-158,229-236: the GDG driver decodes the LAST window a second time with BP + OSD-CS
        # (ldpc.BpOsdDecoder there, this repository's BpOsdDecoder facade here) and reports a second set of counts.
        # last_window_osd = True or a dict of BpOsdDecoder kwargs (defaults: the reference's max_iter=200, OSD_CS 10).
        self.last_osd = None
        if last_window_osd:
            from .decoders import BpOsdDecoder
            kw = dict(max_iter=200, bp_method="minimum_sum", ms_scaling_factor=1.0, osd_method="OSD_CS", osd_order=10)
            if isinstance(last_window_osd, dict):
                kw.update(last_window_osd)
            w = plan.windows[-1]
            self.last_osd = [BpOsdDecoder(w.mat, channel_probs=list(w.prior), device=self.device, **kw) for _ in range(self.nstreams)]

    def __del__(self):
        w = getattr(self, "_win", None)
        if w is not None and w.value:
            self.lib.swd_window_destroy(w)
            self._win = C.c_void_p()
        for h, _, _ in getattr(self, "_res_win", {}).values():
            if h.value:
                self.lib.swd_window_destroy(h)
        self.__dict__["_res_win"] = {}

    def sample_device(self, shots, seed=0, shot_offset=0, return_errors=False):
        """Draw `shots` DEM samples on the device (Philox, one Bernoulli per DEM column; the stand-in for
        `dem.compile_sampler().sample(shots)` of guessing.py:129-130).  -> (det [shots, num_det], obs [shots, num_obs]
        [, err [shots, num_col]]) as torch CUDA uint8 tensors.  Reproducible: shot s of the stream depends only on
        (seed, shot_offset + s)."""
        torch = self.torch
        dev = torch.device("cuda", self.device)
        if not getattr(self, "_priors_set", False):
            pri = np.ascontiguousarray(self.plan.priors, dtype=np.float64)
            _lib.check(self.lib.swd_window_set_priors(self._win, pri.ctypes.data_as(C.POINTER(C.c_double))), "set_priors")
            self._priors_set = True
        det = torch.empty((shots, self.num_det), dtype=torch.uint8, device=dev)
        obs = torch.empty((shots, self.num_obs), dtype=torch.uint8, device=dev)
        err = torch.empty((shots, self.num_col), dtype=torch.uint8, device=dev) if return_errors else None
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(self.lib.swd_window_sample(self._win, int(seed), int(shot_offset), int(shots), det.data_ptr(),
                                              obs.data_ptr() if self.num_obs else None, err.data_ptr() if return_errors else None,
                                              stream), "sample")
        return (det, obs, err) if return_errors else (det, obs)

    def unique_decoders(self):
        seen, out = set(), []
        for decs in self.decoder_sets:
            for d in decs:
                if id(d) not in seen:
                    seen.add(id(d)); out.append(d)
        return out

    def _residual_window(self, w, dec):
        """swd_window handle over one window matrix (cached per decoder): lets the commit / count kernels evaluate
        `(mat @ e_hat + detector_win) % 2` of osd.py:168."""
        cache = self.__dict__.setdefault("_res_win", {})
        if id(dec) not in cache:
            A = w.mat.tocsc(); A.sort_indices()
            cp = np.ascontiguousarray(A.indptr, dtype=np.int32); ri = np.ascontiguousarray(A.indices, dtype=np.int32)
            h = C.c_void_p()
            i32p = C.POINTER(C.c_int32)
            _lib.check(self.lib.swd_window_create(self.device, A.shape[0], A.shape[1], cp.ctypes.data_as(i32p), ri.ctypes.data_as(i32p),
                                                  0, None, None, C.byref(h)), "swd_window_create")
            cache[id(dec)] = (h, cp, ri)
        return cache[id(dec)][0]

    def _plan_llr(self, channel_llr, det):
        """Per-shot priors [B, num_col] in the column order of the DEM given to build_windows (torch CUDA float64 on det's
        device) -> the same rows in the plan's column order."""
        torch = self.torch
        if not (torch.is_tensor(channel_llr) and channel_llr.is_cuda):
            raise ValueError(f"channel_llr must be a torch CUDA float64 tensor here, got {type(channel_llr).__name__}")
        if channel_llr.dtype != torch.float64:
            raise ValueError(f"channel_llr must be float64, got {channel_llr.dtype}")
        if tuple(channel_llr.shape) != (det.shape[0], self.num_col):
            raise ValueError(f"channel_llr must have shape [B, num_col] = [{det.shape[0]}, {self.num_col}], got {tuple(channel_llr.shape)}")
        if channel_llr.device != det.device:
            raise ValueError(f"channel_llr lives on {channel_llr.device}, shot data on {det.device}")
        order = self.plan.col_order
        if order is None:
            return channel_llr.contiguous()
        key = ("order", det.device)
        if key not in self._llr_cache:
            self._llr_cache[key] = torch.as_tensor(np.asarray(order, dtype=np.int64), device=det.device)
        return channel_llr.index_select(1, self._llr_cache[key])

    def _window_llr(self, w, dec, llr):
        """Rows of window w: its DEM columns [col0, col0 + ncols_dem) of the plan-ordered priors, then the decoder's static LLRs
        of the noisy-syndrome identity columns (method 1: the plan's fixed noisy_prior, the same for every shot)."""
        torch = self.torch
        body = llr[:, w.col0:w.col0 + w.ncols_dem]
        if dec.n == w.ncols_dem:
            return body.contiguous()
        key = (id(dec), w.ncols_dem, llr.device)
        if key not in self._llr_cache:
            self._llr_cache[key] = torch.as_tensor(np.ascontiguousarray(dec.channel_llr[w.ncols_dem:]), device=llr.device)
        tail = self._llr_cache[key]
        return torch.cat([body, tail.unsqueeze(0).expand(llr.shape[0], -1)], dim=1)

    def _run_windows(self, det, obs, decs, total, window_events, osd_dec=None, residuals=False, llr=None):
        """The window loop for one (sub-)batch on the current stream; det / obs are updated in place.  llr: per-shot priors
        [B, num_col] in the plan's column order, or None."""
        torch = self.torch
        B = det.shape[0]
        stream = C.c_void_p(torch.cuda.current_stream(det.device).cuda_stream)
        unconv = []
        flagged = []
        counts_osd = None
        for w, dec in zip(self.plan.windows, decs):
            m = w.row1 - w.row0
            synd = torch.empty((B, m), dtype=torch.uint8, device=det.device)
            _lib.check(self.lib.swd_window_extract(self._win, det.data_ptr(), B, w.row0, m, synd.data_ptr(), stream), "extract")
            if w.last and osd_dec is not None:
                # second decode of the last window with BP + OSD on the same residual syndrome (guessing.py:229-236)
                det2, obs2 = det.clone(), obs.clone()
                corr2, _ = osd_dec.decode_batch(synd, channel_llr=None if llr is None else self._window_llr(w, osd_dec, llr))
                _lib.check(self.lib.swd_window_commit(self._win, corr2.data_ptr(), B, corr2.shape[1], w.col0, w.ncommit, det2.data_ptr(),
                                                      obs2.data_ptr() if self.num_obs else None, stream), "commit")
                counts_osd = torch.zeros(2, dtype=torch.int64, device=det.device)
                _lib.check(self.lib.swd_window_count_failures(self._win, det2.data_ptr(), obs2.data_ptr() if self.num_obs else None, B,
                                                              counts_osd.data_ptr(), stream), "count")
            if window_events is not None:
                window_events[w.index][0].record()
            corr, conv = dec.decode_batch(synd, channel_llr=None if llr is None else self._window_llr(w, dec, llr))
            if window_events is not None:
                window_events[w.index][1].record()
            n_win = corr.shape[1]
            if residuals:                       # shots whose correction does not reproduce the window syndrome (osd.py:168)
                rw = self._residual_window(w, dec)
                resid = synd.clone()
                _lib.check(self.lib.swd_window_commit(rw, corr.data_ptr(), B, n_win, 0, n_win, resid.data_ptr(), None, stream), "residual")
                c2 = torch.zeros(2, dtype=torch.int64, device=det.device)
                _lib.check(self.lib.swd_window_count_failures(rw, resid.data_ptr(), None, B, c2.data_ptr(), stream), "residual count")
                flagged.append(c2[0])
            _lib.check(self.lib.swd_window_commit(self._win, corr.data_ptr(), B, n_win, w.col0, w.ncommit, det.data_ptr(),
                                                  obs.data_ptr() if self.num_obs else None, stream), "commit")
            unconv.append((B - conv.sum(dtype=torch.int64)))
            if total is not None:
                total[:, w.col0:w.col0 + w.ncommit] = corr[:, :w.ncommit]
        counts = torch.zeros(2, dtype=torch.int64, device=det.device)
        _lib.check(self.lib.swd_window_count_failures(self._win, det.data_ptr(), obs.data_ptr() if self.num_obs else None, B,
                                                      counts.data_ptr(), stream), "count")
        return counts, torch.stack(unconv), counts_osd, (torch.stack(flagged) if residuals else None)

    def decode_device(self, det, obs, return_corrections=False, window_events=None, streams=None, window_residuals=False,
                      channel_llr=None):
        """det [B, num_det], obs [B, num_obs]: torch CUDA uint8 tensors, MODIFIED IN PLACE into the residual
        syndrome / residual observables.  Returns dict with device tensors:
          counts uint64[2] = (flagged shots, failed shots), window_unconverged int64[num_win].
        streams: use fewer concurrent sub-batches than the decoder was built with (1 = plain sequential launches).
        channel_llr: optional per-shot priors, torch CUDA float64 [B, num_col] in the column order of the DEM given to
        build_windows (log((1-p)/p); 0.0 = erased).  Every window (and the last-window BP + OSD re-decode) decodes shot b with
        row b's LLRs of its DEM columns; the noisy-syndrome columns of method 1 keep their static prior."""
        torch = self.torch
        B = det.shape[0]
        llr = None if channel_llr is None else self._plan_llr(channel_llr, det)
        total = torch.zeros((B, self.num_col), dtype=torch.uint8, device=det.device) if return_corrections else None
        ns = self.nstreams if streams is None else max(1, min(int(streams), self.nstreams))
        if window_events is not None or B < 2 * ns:
            ns = 1
        if ns == 1:
            counts, unconv, counts_osd, wflag = self._run_windows(det, obs, self.decoders, total, window_events,
                                                                  self.last_osd[0] if self.last_osd else None, window_residuals, llr)
        else:
            if self._side_streams is None:
                self._side_streams = [torch.cuda.Stream(device=det.device) for _ in range(self.nstreams)]
            cur = torch.cuda.current_stream(det.device)
            bounds = [(B * i) // ns for i in range(ns + 1)]
            parts = []
            for i in range(ns):
                st = self._side_streams[i]
                st.wait_stream(cur)
                lo, hi = bounds[i], bounds[i + 1]
                with torch.cuda.stream(st):
                    parts.append(self._run_windows(det[lo:hi], obs[lo:hi], self.decoder_sets[i],
                                                   None if total is None else total[lo:hi], None,
                                                   self.last_osd[i] if self.last_osd else None, window_residuals,
                                                   None if llr is None else llr[lo:hi]))
                for t in (det, obs, total, llr):
                    if t is not None:
                        t.record_stream(st)
            for st in self._side_streams[:ns]:
                cur.wait_stream(st)
            counts = sum(p[0] for p in parts)
            unconv = sum(p[1] for p in parts)
            counts_osd = sum(p[2] for p in parts) if self.last_osd else None
            wflag = sum(p[3] for p in parts) if window_residuals else None
        out = dict(counts=counts, window_unconverged=unconv)
        if window_residuals:
            out["window_flagged"] = wflag                   # per window: shots with mat @ e_hat != window syndrome
        if counts_osd is not None:
            out["counts_last_window_osd"] = counts_osd      # (flagged, failed) when the last window is decoded by BP + OSD
        if return_corrections:
            out["total_e_hat"] = total
        return out

    def _host_llr_to_device(self, channel_llr, B, dev):
        """numpy (or torch CPU) float64 [B, num_col] per-shot priors -> torch CUDA tensor; NaN is rejected here."""
        torch = self.torch
        if torch.is_tensor(channel_llr):
            if channel_llr.is_cuda:
                raise ValueError("channel_llr is a CUDA tensor but the shot data are host arrays (use decode_device)")
            channel_llr = channel_llr.numpy()
        if not isinstance(channel_llr, np.ndarray) or channel_llr.dtype != np.float64:
            raise ValueError(f"channel_llr must be a float64 array, got {getattr(channel_llr, 'dtype', type(channel_llr).__name__)}")
        if channel_llr.shape != (B, self.num_col):
            raise ValueError(f"channel_llr must have shape [B, num_col] = [{B}, {self.num_col}], got {channel_llr.shape}")
        if np.isnan(channel_llr).any():
            raise ValueError("channel_llr contains NaN (allowed: finite values, +-inf; 0.0 marks an erasure)")
        return torch.from_numpy(np.ascontiguousarray(channel_llr)).to(dev)

    def decode_packed(self, det_packed, obs_packed, return_corrections=True, pinned_out=None, channel_llr=None):
        """Host entry point with bit-packed shot data (decoders.pack_bits layout): det_packed [B, ceil(num_det/64)] and
        obs_packed [B, ceil(num_obs/64)] uint64 (numpy or pinned torch CPU tensors) -> dict(flagged, failed,
        window_unconverged, total_e_hat_packed [B, ceil(num_col/64)] uint64).  8x fewer bytes cross PCIe than with one byte
        per bit (configs[2]: 82 MB instead of 658 MB of corrections per 32768 shots).  pinned_out: optional pinned torch
        int64 CPU tensor [B, ceil(num_col/64)] that receives the packed corrections.  channel_llr: optional per-shot priors,
        numpy float64 [B, num_col] (see decode_device)."""
        torch = self.torch
        dev = torch.device("cuda", self.device)

        def to_dev(x):
            t = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x).view(np.int64))
            return t.to(dev, non_blocking=True)
        dp, op = to_dev(det_packed), to_dev(obs_packed)
        B = dp.shape[0]
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        det = torch.empty((B, self.num_det), dtype=torch.uint8, device=dev)
        obs = torch.empty((B, self.num_obs), dtype=torch.uint8, device=dev)
        llr = None if channel_llr is None else self._host_llr_to_device(channel_llr, B, dev)
        _lib.check(self.lib.swd_unpack_bits(self.device, dp.data_ptr(), B, self.num_det, det.data_ptr(), stream), "unpack det")
        if self.num_obs:
            _lib.check(self.lib.swd_unpack_bits(self.device, op.data_ptr(), B, self.num_obs, obs.data_ptr(), stream), "unpack obs")
        out = self.decode_device(det, obs, return_corrections, channel_llr=llr)
        res = {}
        if return_corrections:
            wn = (self.num_col + 63) // 64
            packed = torch.empty((B, wn), dtype=torch.int64, device=dev)
            _lib.check(self.lib.swd_pack_bits(self.device, out["total_e_hat"].data_ptr(), B, self.num_col, packed.data_ptr(), stream), "pack e_hat")
            if pinned_out is not None:
                pinned_out.copy_(packed, non_blocking=True)
                host = pinned_out
            else:
                host = packed.cpu()
            res["total_e_hat_packed"] = host
        counts = out["counts"].cpu().numpy()          # synchronises the stream: the packed corrections have landed as well
        res.update(shots=int(B), flagged=int(counts[0]), failed=int(counts[1]),
                   window_unconverged=out["window_unconverged"].cpu().numpy().tolist())
        if return_corrections and not torch.is_tensor(det_packed):
            res["total_e_hat_packed"] = res["total_e_hat_packed"].numpy().view(np.uint64)
        return res

    def decode(self, det_data, obs_data, return_corrections=False, channel_llr=None):
        """Host entry point (numpy uint8 - or torch CPU tensors, e.g. pinned - in, python ints out): H2D copy, all windows,
        D2H of the counters (and of the corrections, one byte per bit, if asked for; decode_packed moves 8x less).
        channel_llr: optional per-shot priors, numpy float64 [B, num_col] (see decode_device)."""
        torch = self.torch
        dev = torch.device("cuda", self.device)

        def to_dev(x):
            t = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.uint8))
            return t.to(dev, non_blocking=True)
        det, obs = to_dev(det_data), to_dev(obs_data)
        llr = None if channel_llr is None else self._host_llr_to_device(channel_llr, det.shape[0], dev)
        out = self.decode_device(det, obs, return_corrections, channel_llr=llr)
        counts = out["counts"].cpu().numpy()
        res = dict(shots=int(det.shape[0]), flagged=int(counts[0]), failed=int(counts[1]),
                   window_unconverged=out["window_unconverged"].cpu().numpy().tolist())
        if "counts_last_window_osd" in out:
            c2 = out["counts_last_window_osd"].cpu().numpy()
            res["flagged_last_window_osd"], res["failed_last_window_osd"] = int(c2[0]), int(c2[1])
        if return_corrections:
            res["total_e_hat"] = out["total_e_hat"].cpu().numpy()
        return res
