"""Host stage between the two device stages: the "rate-change fit".

BASELINE.json's north star keeps this part in Python on the host and outside the timed
window: the continuity filter, the per-feature gain fit, the 70->1 compression of the
pass-1 path, the L1 linear programme and the grouping of its solution into line clusters
(reference describealign.py:702-893), plus the node list built from the final path
(describealign.py:995-1027).  The corridor planning with its sub-frame offset refinement
(describealign.py:895-932) runs on the device (csrc/refine.cuh).

The arithmetic goes through the same numpy / scipy entry points the reference calls
(np.convolve, np.linalg.lstsq, np.std, scipy.optimize.linprog with HiGHS) on operands of
the same dtype and order, because the LP has degenerate optima and anything else would not
reproduce the reference's segments.  Written from the functional description in
SURVEY.md appendix A.6/A.7, not from the reference's source text.

Native host stage (SURVEY.md 8f N1): the continuity error, the path compression, the assembly
of the LP and the grouping of its solution into line clusters run in C++ inside the library
(csrc/host_stage.cpp, `dab_host_*`), restating numpy's pairwise sums, OpenBLAS' ddot order and
numpy's scalar rounding; `continuity_error`, `compress_path`, `_lp_problem` and `line_clusters`
below call them.  The numpy versions stay as `*_numpy`: they are
what the native code is tested against, bit for bit (tests/test_host_native.py), next to the
reference's own intermediate values in tests/golden/.  `np.std`, `np.linalg.lstsq` (LAPACK) and
`scipy.optimize.linprog` (HiGHS) stay library calls.
"""
from __future__ import annotations

from collections import OrderedDict
from dataclasses import dataclass

import numpy as np
import scipy.optimize
import scipy.signal
import scipy.sparse

FRAMES_PER_SECOND = 210
SPN = FRAMES_PER_SECOND // 10          # frames per node (describealign.py:596)
CORRIDOR_RADIUS = FRAMES_PER_SECOND * 30   # +/- 30 s (describealign.py:863)

FAILED_MSG = "Alignment failed, are the input files mismatched?"
LP_FAILED_MSG = "Smooth Alignment L1-Min Optimization Failed!"


def hann41() -> np.ndarray:
    """41-tap f64 Hann window, normalised (describealign.py:597-598)."""
    w = scipy.signal.windows.hann(2 * SPN + 1)[1:-1]
    return w / np.sum(w)


def local_mean(arr, window=None):
    """describealign.py:599 (`get_mean`)."""
    window = hann41() if window is None else window
    return np.convolve(window, arr, mode="same")[:len(arr)]


def min_path_length(n_video_energy: int, n_audio_energy: int) -> float:
    """Shortest acceptable path (describealign.py:698, 991)."""
    return max(min(n_video_energy, n_audio_energy) / 500.0, 5 * FRAMES_PER_SECOND)


def _native():
    from . import _cabi
    return _cabi.load()


def _ptr(a):
    return a.ctypes.data


def continuity_error(x, y, deriv=False, window=None):
    """Distance of every path point from a line extrapolated from its smoothed future or
    past neighbours, whichever is closer (describealign.py:706-724).  Native (dab_host_continuity_error)."""
    x, y = np.asarray(x), np.asarray(y)
    n = len(x)
    if window is not None or n < 51 or len(y) != n:
        return continuity_error_numpy(x, y, deriv, window)
    err = np.empty(n - (1 if deriv else 0), dtype=np.float64)
    lib = _native()
    if np.issubdtype(x.dtype, np.integer) and np.issubdtype(y.dtype, np.integer):
        xi, yi = np.ascontiguousarray(x, dtype=np.int64), np.ascontiguousarray(y, dtype=np.int64)
        rc = lib.dab_host_continuity_error(_ptr(xi), _ptr(yi), n, int(bool(deriv)), _ptr(err))
    else:
        xf, yf = np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(y, dtype=np.float64)
        rc = lib.dab_host_continuity_error_f64(_ptr(xf), _ptr(yf), None, None, n, int(bool(deriv)), _ptr(err))
    if rc != 0:
        raise RuntimeError(f"dab_host_continuity_error failed ({rc})")
    return err


def continuity_error_numpy(x, y, deriv=False, window=None):
    """The numpy statement of continuity_error (describealign.py:706-724): checker of the native code."""
    window = hann41() if window is None else window
    head = window[:SPN - 1]
    head = head / np.sum(head)
    half = SPN // 2
    delay = SPN + half - 2

    def lines(kernel):
        xs = np.convolve(x, kernel, mode="valid")
        ys = np.convolve(y, kernel, mode="valid")
        slope = (ys[half:] - ys[:-half]) / (xs[half:] - xs[:-half])
        return xs, ys, slope

    xs, ys, slope_f = lines(head)
    off_f = ys[:-half] - xs[:-half] * slope_f
    xs, ys, slope_p = lines(head[::-1])
    off_p = ys[half:] - xs[half:] * slope_p
    shift = 1 if deriv else 0
    err = np.full(len(x) - shift, np.inf)
    k = delay - shift
    err[:-k] = np.abs(slope_f * x[:-delay] + off_f - y[:-delay])
    err[k:] = np.minimum(err[k:], np.abs(slope_p * x[delay:] + off_p - y[delay:]))
    return err


def scale_features(video_features, audio_features, x, y):
    """Least-squares gain per feature, keep the first three, stack as (len, 3) float32
    (describealign.py:733-741).  x = audio indices, y = video indices of the kept path."""
    a_cols, v_cols = [], []
    for v_feat, a_feat in list(zip(video_features, audio_features))[:3]:
        a_std = np.std(a_feat)
        gain = np.linalg.lstsq(v_feat[y][:, None], a_feat[x], rcond=None)[0]
        a_cols.append(a_feat / a_std)
        v_cols.append(v_feat * gain / a_std)
    na = min(len(c) for c in a_cols)
    nv = min(len(c) for c in v_cols)
    audio_scaled = np.stack([c[:na] for c in a_cols], axis=1)
    video_scaled = np.stack([c[:nv] for c in v_cols], axis=1)
    return np.ascontiguousarray(audio_scaled), np.ascontiguousarray(video_scaled)


def feature_gains(video_features, audio_features, x, y):
    """The six scalars the scaled feature arrays are made from (describealign.py:733-741): per feature
    the least-squares gain and the audio standard deviation, plus the lengths of the stacked arrays.
    Returns (gains f32[3], audio_stds f32[3], n_audio, n_video); the arrays themselves are rebuilt on
    the device (dab_pair_stage_b_clusters, dab_engine_submit_b).  Raises TypeError unless the first three
    features are float32: the device cannot redo numpy's arithmetic on other types from float32 scalars."""
    gains, stds = [], []
    for v_feat, a_feat in list(zip(video_features, audio_features))[:3]:
        if np.asarray(v_feat).dtype != np.float32 or np.asarray(a_feat).dtype != np.float32:
            raise TypeError("the first three features must be float32 (as get_energy / get_zero_crossings / get_freq_bands return them)")
        stds.append(np.std(a_feat))
        gains.append(np.linalg.lstsq(v_feat[y][:, None], a_feat[x], rcond=None)[0][0])
    na = min(len(f) for f in list(audio_features)[:3])
    nv = min(len(f) for f in list(video_features)[:3])
    return np.array(gains, np.float32), np.array(stds, np.float32), na, nv


def compress_path(x, y, window=None):
    """Replace well-behaved runs of 70 path points by their mean point and merge entries
    that share an audio index (describealign.py:743-767), quirks included.  Native (dab_host_compress_path)."""
    x, y = np.asarray(x), np.asarray(y)
    n = len(x)
    if window is not None or n < 41 or not (np.issubdtype(x.dtype, np.integer) and np.issubdtype(y.dtype, np.integer)):
        return compress_path_numpy(x, y, window)
    if n - 80 <= 10:
        raise RuntimeError(FAILED_MSG)
    import ctypes
    xi, yi = np.ascontiguousarray(x, dtype=np.int64), np.ascontiguousarray(y, dtype=np.int64)
    ox, oy = np.empty(n, dtype=np.float64), np.empty(n, dtype=np.float64)
    cnt = ctypes.c_int64(0)
    rc = _native().dab_host_compress_path(_ptr(xi), _ptr(yi), n, _ptr(ox), _ptr(oy), ctypes.byref(cnt))
    if rc != 0:
        raise RuntimeError(f"dab_host_compress_path failed ({rc})")
    return ox[:cnt.value].copy(), oy[:cnt.value].copy()


def compress_path_numpy(x, y, window=None):
    """The numpy statement of compress_path (describealign.py:743-767): checker of the native code."""
    sx = local_mean(x, window)
    sy = local_mean(y, window)
    slope = np.diff(sy) / np.diff(sx)
    offset = sy[:-1] - sx[:-1] * slope
    err_y = slope * x[:-1] + offset - y[:-1]
    cx, cy = list(x[0:10]), list(y[0:10])
    start = None
    for start in range(10, len(x) - 80, 70):
        if np.all(np.abs(err_y[start:start + 70]) < 3):
            cx.append(np.mean(x[start:start + 70]))
            cy.append(np.mean(y[start:start + 70]))
        else:
            cx.extend(x[start:start + 70])
            cy.extend(y[start:start + 70])
    if start is None:
        raise RuntimeError(FAILED_MSG)
    # one further fixed slice is kept raw; points after it are dropped (reference quirk)
    cx.extend(x[start + 70:start + 140])
    cy.extend(y[start + 70:start + 140])
    groups = OrderedDict()
    for xi, yi in zip(cx, cy):
        groups.setdefault(xi, []).append(yi)
    ux = np.array(list(groups.keys()))
    uy = np.array([np.mean(groups[k]) for k in ux])
    return ux, uy


@dataclass
class RateFit:
    x: np.ndarray           # fit points, audio frames
    y: np.ndarray           # fit points, video frames
    fit_err: np.ndarray
    slopes: np.ndarray      # per interval, len n-1
    median_slope: float


def _lp_problem(x, y, window=None):
    """Objective, equality constraints (CSC), right-hand side and bounds of the rate-change LP
    (describealign.py:769-836).  Native assembly (dab_host_lp_assemble)."""
    n = len(x)
    if window is not None or n < 51:
        return _lp_problem_numpy(x, y, window)
    import ctypes
    xf, yf = np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(y, dtype=np.float64)
    cost = np.empty(12 * n - 9, dtype=np.float64)
    indptr = np.empty(12 * n - 8, dtype=np.int32)
    indices = np.empty(24 * n, dtype=np.int32)
    data = np.empty(24 * n, dtype=np.float64)
    b_eq = np.empty(3 * n - 4, dtype=np.float64)
    nnz = ctypes.c_int64(0)
    rc = _native().dab_host_lp_assemble(_ptr(xf), _ptr(yf), n, _ptr(cost), _ptr(indptr), _ptr(indices), _ptr(data),
                                        _ptr(b_eq), ctypes.byref(nnz))
    if rc != 0:
        raise RuntimeError(f"dab_host_lp_assemble failed ({rc})")
    k = nnz.value
    a_eq = scipy.sparse.csc_matrix((data[:k].copy(), indices[:k].copy(), indptr), shape=(3 * n - 4, 12 * n - 9))
    bounds = [[0, None]] * (4 * n - 2) + [[0, 2.0]] * (2 * n) + [[0, None]] * (6 * n - 8) + [[None, None]]
    return cost, a_eq, b_eq, bounds


def _lp_problem_numpy(x, y, window=None):
    """The numpy / scipy.sparse statement of _lp_problem: checker of the native assembly."""
    n = len(x)
    dx = np.diff(x)
    dy = np.diff(y)
    inv = 1.0 / dx
    jump_cost = np.full(n - 1, 10.0)
    jump_cost /= np.maximum(1, np.sqrt(continuity_error_numpy(x, y, deriv=True, window=window) / 3.0))
    cost = np.hstack([np.ones(2 * n), jump_cost, jump_cost,
                      np.full(n, .01), np.full(n, .01),
                      np.full(n - 1, 3), np.full(n - 1, 3),
                      np.full(n - 1, .001), np.full(n - 1, .001),
                      np.full(n - 2, 10.0 * 4000), np.full(n - 2, 10.0 * 4000), [0, ]])
    # column offsets of the variable groups
    c_fe_p, c_fe_m = 0, n
    c_j_p, c_j_m = 2 * n, 3 * n - 1
    c_sn_p, c_sn_m = 4 * n - 2, 5 * n - 2
    c_snj_p, c_snj_m = 6 * n - 2, 7 * n - 3
    c_rcj_p, c_rcj_m = 8 * n - 4, 9 * n - 5
    c_rc_p, c_rc_m = 10 * n - 6, 11 * n - 8
    c_med = 12 * n - 10
    rows, cols, vals = [], [], []

    def put(r, c, v):
        rows.append(np.asarray(r, dtype=np.int64))
        cols.append(np.asarray(c, dtype=np.int64))
        vals.append(np.broadcast_to(np.asarray(v, dtype=np.float64), np.shape(r)).copy())

    r1 = np.arange(n - 1)
    # block 1: local slope of the fitted path = median slope + jumps  (n-1 rows)
    for base, sign in ((c_fe_p, 1.0), (c_fe_m, -1.0)):
        put(r1, base + r1, sign * -inv)
        put(r1, base + r1 + 1, sign * inv)
    for base, sign in ((c_j_p, 1.0), (c_j_m, -1.0), (c_snj_p, 1.0), (c_snj_m, -1.0),
                       (c_rcj_p, 1.0), (c_rcj_m, -1.0)):
        put(r1, base + r1, sign * inv)
    put(r1, np.full(n - 1, c_med), 1.0)
    # block 2: shot-noise jumps are the differences of the shot-noise terms  (n-1 rows)
    r2 = (n - 1) + r1
    put(r2, c_sn_p + r1, -1.0)
    put(r2, c_sn_p + r1 + 1, 1.0)
    put(r2, c_sn_m + r1, 1.0)
    put(r2, c_sn_m + r1 + 1, -1.0)
    put(r2, c_snj_p + r1, -1.0)
    put(r2, c_snj_m + r1, 1.0)
    # block 3: rate changes are the differences of consecutive rate-change jumps  (n-2 rows)
    r3i = np.arange(n - 2)
    r3 = 2 * (n - 1) + r3i
    for base, sign in ((c_rcj_p, 1.0), (c_rcj_m, -1.0)):
        put(r3, base + r3i, sign * -inv[:-1])
        put(r3, base + r3i + 1, sign * inv[1:])
    put(r3, c_rc_p + r3i, -1.0)
    put(r3, c_rc_m + r3i, 1.0)
    a_eq = scipy.sparse.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))),
                                   shape=(3 * n - 4, 12 * n - 9)).tocsc()
    b_eq = np.hstack((dy / dx, np.zeros(2 * n - 3)))
    bounds = [[0, None]] * (4 * n - 2) + [[0, 2.0]] * (2 * n) + [[0, None]] * (6 * n - 8) + [[None, None]]
    return cost, a_eq, b_eq, bounds


def rate_change_fit(x, y, window=None, linprog=None) -> RateFit:
    """L1 fit of a piece-wise linear path with few rate changes (describealign.py:769-858)."""
    linprog = scipy.optimize.linprog if linprog is None else linprog
    n = len(x)
    cost, a_eq, b_eq, bounds = _lp_problem(x, y, window)
    fit = linprog(cost, A_eq=a_eq, b_eq=b_eq, bounds=bounds, method="highs-ds")
    if not fit.success and fit.status == 4:
        fit = linprog(cost, A_eq=a_eq, b_eq=b_eq, bounds=bounds, method="highs-ipm")
    if not fit.success:
        print(fit)
        raise RuntimeError(LP_FAILED_MSG)
    sol = fit.x
    fit_err = sol[:n] - sol[n:2 * n]
    slope_jumps = sol[8 * n - 4:9 * n - 5] - sol[9 * n - 5:10 * n - 6]
    median_slope = sol[-1]
    slopes = median_slope + slope_jumps / np.diff(x)
    return RateFit(x=x, y=y, fit_err=fit_err, slopes=slopes, median_slope=median_slope)


def line_clusters(fit: RateFit):
    """Group the smooth path's points into co-linear clusters and fit a line to each
    (describealign.py:861-893).  Returns a list of (x array, offset, slope).  The grouping is native
    (dab_host_line_clusters); the line fit per cluster is the reference's np.linalg.lstsq call."""
    import ctypes
    n = len(fit.x)
    x = np.ascontiguousarray(fit.x, dtype=np.float64)
    y = np.ascontiguousarray(fit.y - fit.fit_err, dtype=np.float64)
    slopes = np.ascontiguousarray(np.hstack((fit.slopes[:1], fit.slopes, fit.slopes[-1:])), dtype=np.float64)
    if n < 1 or len(slopes) != n + 1 or not np.all(np.isfinite(slopes)):
        return line_clusters_numpy(fit)
    ox, oy = np.empty(2 * n, dtype=np.float64), np.empty(2 * n, dtype=np.float64)
    start = np.empty(2 * n + 1, dtype=np.int64)
    count = ctypes.c_int64(0)
    rc = _native().dab_host_line_clusters(_ptr(x), _ptr(y), _ptr(slopes), n, _ptr(ox), _ptr(oy), _ptr(start), ctypes.byref(count))
    if rc != 0:
        return line_clusters_numpy(fit)
    out = []
    for c in range(count.value):
        cx, cy = ox[start[c]:start[c + 1]].copy(), oy[start[c]:start[c + 1]].copy()
        sol = np.linalg.lstsq(np.hstack((np.ones((len(cx), 1)), cx[:, None])), cy, rcond=None)[0]
        out.append((cx, sol[0], sol[1]))
    return out


def line_clusters_numpy(fit: RateFit):
    """The Python statement of line_clusters (describealign.py:861-893): checker of the native grouping."""
    smooth = list(zip(fit.x, fit.y - fit.fit_err))
    slopes = np.hstack((fit.slopes[:1], fit.slopes, fit.slopes[-1:]))
    groups = {}
    for k, (px, py) in enumerate(smooth):
        for slope in slopes[k:k + 2]:
            if slope < .1 or slope > 10:
                continue
            key = (round(slope, 6), int(round(py - slope * px, 0)))
            groups.setdefault(key, []).append((px, py))
    clusters = []
    taken = set()
    for key, members in sorted(groups.items(), key=lambda kv: -len(kv[1])):
        if key in taken:
            continue
        slope, offset = key
        cluster = members
        taken.add(key)
        del groups[key]
        for key2, members2 in list(groups.items()):
            first, last = members2[0], members2[-1]
            if abs(first[1] - (first[0] * slope + offset)) < 3 and abs(last[1] - (last[0] * slope + offset)) < 3:
                cluster.extend(members2)
                taken.add(key2)
                del groups[key2]
        clusters.append(cluster)
    clusters = [sorted(c) for c in clusters]
    clusters = [c for c in clusters if abs(c[0][0] - c[-1][0]) > 10 and len(c) > 5]
    out = []
    for c in clusters:
        cx, cy = np.array(c).T
        sol = np.linalg.lstsq(np.hstack((np.ones((len(cx), 1)), cx[:, None])), cy, rcond=None)[0]
        out.append((cx, sol[0], sol[1]))
    return out


# ------------------------------------------------------------------------------------------
# Stage-B host helpers
# ------------------------------------------------------------------------------------------

def cluster_lines(clusters):
    """What stage B needs of the line clusters: (cluster index, first x, last x, offset, slope) per
    cluster.  The corridor planning itself (row limits, sub-frame offset refinement, +-30 s extension,
    describealign.py:895-932) runs on the device (csrc/refine.cuh)."""
    return [(idx, float(cx[0]), float(cx[-1]), float(offset), float(slope)) for idx, (cx, offset, slope) in enumerate(clusters)]


def build_nodes(path, n_audio_energy: int, n_video_energy: int, n_audio_scaled: int, n_video_scaled: int):
    """Similarity percentage and break-point nodes from the final path rows
    (j, i, cluster, qual, cum) (describealign.py:993-1026).  Scales path[:, :2] in place."""
    y, x, cluster, quals, _ = path.T
    keep = (quals == 0) | (quals > .3)
    sim_x = float(len(np.unique(x[keep]))) / n_audio_scaled       # len(set(...)) of the reference
    sim_y = float(len(np.unique(y[keep]))) / n_video_scaled
    similarity = 100 * max(sim_x, sim_y)
    # break-points where the cluster changes, in path order: (point k - .1, point k+1 + .1) per change
    ch = np.flatnonzero(cluster[:-1] != cluster[1:])
    px = np.empty(2 * len(ch)); py = np.empty(2 * len(ch))
    px[0::2], px[1::2] = x[ch] - .1, x[ch + 1] + .1
    py[0::2], py[1::2] = y[ch] - .1, y[ch + 1] + .1
    nodes = []
    if cluster[0] == cluster[1]:
        nodes.append((x[0], y[0]))
    nodes.extend(zip(px, py))
    if cluster[-2] == cluster[-1]:
        nodes.append((x[-1], y[-1]))
    nx, ny = np.array(nodes).T / 210.
    if (nx[1] - nx[0]) > 2:
        s = (ny[1] - ny[0]) / (nx[1] - nx[0])
        nx[0] = 0
        ny[0] = ny[1] - (nx[1] * s)
        if ny[0] < 0:
            nx[0] = nx[1] - (ny[1] / s)
            ny[0] = 0
    if (nx[-1] - nx[-2]) > 2:
        s = (ny[-1] - ny[-2]) / (nx[-1] - nx[-2])
        nx[-1] = ((n_audio_energy - 1) / 210.)
        ny[-1] = ny[-2] + ((nx[-1] - nx[-2]) * s)
        if ny[-1] > ((n_video_energy - 1) / 210.):
            ny[-1] = ((n_video_energy - 1) / 210.)
            nx[-1] = nx[-2] + ((ny[-1] - ny[-2]) / s)
    path[:, :2] /= 210.
    return nx, ny, similarity
