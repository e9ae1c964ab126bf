"""Sliding-window geometry on a detector error model (host-side setup, numpy/scipy).

Restates the window construction of the reference drivers (guessing.py:49-126, osd.py:49-118):
columns are regrouped by the detector rounds they touch, anchors mark the first column of every
round, window i covers W rounds of detectors and all faults starting in them; with method=1 the
faults that reach beyond the window are replaced by one "noisy syndrome" identity column per check
of the last round (prior = summed prior of the merged columns), keeping 3h columns of the next
round un-merged.  After decoding window i the first F rounds of columns are committed.
"""
import math
from dataclasses import dataclass

import numpy as np
from scipy.sparse import csc_matrix, hstack as sp_hstack, identity as sp_identity, vstack as sp_vstack


@dataclass
class Window:
    index: int
    mat: csc_matrix          # window PCM  (rows a0:b0)
    prior: np.ndarray        # per-column error probability
    row0: int                # a[0]
    row1: int                # b[0]
    col0: int                # a[1]  first DEM column of the window
    ncommit: int             # columns committed after decoding (c[1]-a[1]; whole window for the last one)
    ncols_dem: int           # number of leading window columns that are genuine DEM columns
    last: bool


@dataclass
class WindowPlan:
    chk: csc_matrix          # reshuffled detector matrix  [num_det, num_col]
    obs: csc_matrix          # reshuffled observable matrix
    priors: np.ndarray
    anchors: list
    windows: list
    n_half: int
    W: int
    F: int
    noisy_prior: np.ndarray = None
    col_order: np.ndarray = None   # column j of chk / obs / priors is column col_order[j] of the DEM given to build_windows


def reshuffle_by_round(chk, obs, priors, n=None, h=None):
    """guessing.py:49-84 (h = n/2 detectors per round) / SHYPS.ipynb cell 1 (h = r(2^r-1)): regroup the columns by
    (first, last) detector round; compute anchors."""
    return _reshuffle(chk, obs, priors, n, h)[:4]


def _reshuffle(chk, obs, priors, n=None, h=None):
    """reshuffle_by_round plus the column order it applied (-> chk, obs, priors, anchors, order)."""
    chk = csc_matrix(chk)
    obs = csc_matrix(obs)
    num_row, num_col = chk.shape
    if h is None:
        h = n // 2
    regions = []
    i = 0
    while i < num_row:
        regions.append((i, i + h))
        if i + 2 * h > num_row:
            break
        regions.append((i, i + 2 * h))
        i += h
    region_id = {r: k for k, r in enumerate(regions)}
    buckets = [[] for _ in regions]
    indptr, indices = chk.indptr, chk.indices
    for c in range(num_col):
        rows = indices[indptr[c]:indptr[c + 1]]
        lo = int(rows.min()) // h * h
        hi = (int(rows.max()) // h + 1) * h
        buckets[region_id[(lo, hi)]].append(c)
    order = np.array([c for b in buckets for c in b], dtype=np.int64)
    chk = chk[:, order].tocsc()
    obs = obs[:, order].tocsc()
    priors = np.asarray(priors)[order]
    chk.sort_indices()
    anchors = []
    j = 0
    indptr, indices = chk.indptr, chk.indices
    for c in range(num_col):
        if int(indices[indptr[c]:indptr[c + 1]].min()) >= j:
            anchors.append((j, c))
            j += h
    anchors.append((num_row, num_col))
    return chk, obs, priors, anchors, order


def build_windows(chk, obs, priors, n=None, W=3, F=1, method=1, noisy_prior=None, h=None, keep_cols=None):
    """-> WindowPlan.  chk/obs/priors as returned by dem_to_check_matrices (any column order).
    n: number of data qubits of a BB code (h = n/2 detectors per round); or pass h directly (SHYPS: method=0).
    keep_cols: un-merged columns of the round after the window for method=1 (default 3h as guessing.py:90,112;
    osd.py:83,106 uses n for the x basis)."""
    if h is None:
        h = n // 2
    if keep_cols is None:
        keep_cols = 3 * h
    chk, obs, priors, anchors, order = _reshuffle(chk, obs, priors, h=h)
    if noisy_prior is None and method != 0:
        b = anchors[W]
        c = anchors[W - 1]
        if method == 1:
            c = (c[0], c[1] + keep_cols)
        sub = chk[c[0]:b[0], c[1]:b[1]]
        noisy_prior = np.asarray(sub.multiply(priors[c[1]:b[1]][None, :]).sum(axis=1)).ravel()
    noisy = None if method == 0 else np.ones(h) * noisy_prior
    num_win = math.ceil((len(anchors) - W + F - 1) / F)
    windows = []
    top_left = 0
    for i in range(num_win):
        a = anchors[top_left]
        b = anchors[min(top_left + W, len(anchors) - 1)]
        last = (i == num_win - 1)
        if not last and method != 0:
            c = anchors[top_left + W - 1]
            if method == 1:
                c = (c[0], c[1] + keep_cols)
            body = chk[a[0]:b[0], a[1]:c[1]]
            ident = sp_vstack([csc_matrix((h * (W - 1), h), dtype=np.uint8), sp_identity(h, dtype=np.uint8, format="csc")])
            mat = sp_hstack([body, ident]).tocsc()
            prior = np.concatenate([priors[a[1]:c[1]], noisy])
            ncols_dem = c[1] - a[1]
        else:
            mat = chk[a[0]:b[0], a[1]:b[1]].tocsc()
            prior = priors[a[1]:b[1]].copy()
            ncols_dem = b[1] - a[1]
        mat.sort_indices()
        commit_end = b[1] if last else anchors[top_left + F][1]
        windows.append(Window(i, mat, prior, a[0], b[0], a[1], commit_end - a[1], ncols_dem, last))
        top_left += F
    return WindowPlan(chk, obs, priors, anchors, windows, h, W, F, None if method == 0 else np.asarray(noisy_prior), order)
