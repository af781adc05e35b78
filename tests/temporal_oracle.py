"""NumPy / Python restatement of the temporal depth filter (include/vsc_b200.h, vsc_stage_temporal_depth).

Output frame t is a pure function of the depth maps D_lo .. D_hi around it:
  * exact integer sums S_j = sum D_j, Q_j = sum D_j^2, P_tj = sum D_t D_j (Python ints);
  * cov = n P_tj - S_t S_j, var_j = n Q_j - S_j^2, var_t likewise, each converted to double with float(int);
  * neighbour j is cut when var_j <= 0, var_t <= 0, cov <= 0, 2 cov^2 < var_j var_t or a = cov / var_j > 16, and a cut
    also excludes every neighbour farther out on that side;
  * E_j = clamp((A D_j + B + 32768) >> 16, 0, M) with A = rint(a 65536), B = rint(b 65536),
    b = (S_t - a S_j) / n, all in IEEE double;
  * w[m][d] = float32(exp(-0.5 m^2 / k^2 - 0.5 d^2 / sigma^2)), d = |E_j - D_t| (>> 8 for uint16), at most 255;
  * out = (sum_j w E_j) / (sum_j w) over j ascending, in float32.
"""
from __future__ import annotations

import math

import numpy as np

MIN_R2 = 0.5           # a neighbour whose squared correlation with D_t is below this is a scene cut
MAX_SLOPE = 16.0       # ... and so is one that needs a larger alignment slope
MAX_RADIUS = 8
MAX_SIGMA = 64.0


def max_value(dtype) -> int:
    dt = np.dtype(dtype)
    if dt == np.uint8:
        return 255
    if dt == np.uint16:
        return 65535
    raise TypeError(f'temporal filtering takes uint8 or uint16 depth, not {dt}')


def weight_table(radius: int, sigma: float) -> np.ndarray:
    """float32 [radius + 1, 256]: w[m][d] = exp(-0.5 m^2 / k^2 - 0.5 d^2 / sigma^2), computed in double."""
    w = np.empty((radius + 1, 256), np.float32)
    for m in range(radius + 1):
        tm = 0.0 if m == 0 else 0.5 * (m * m) / (radius * radius)
        for d in range(256):
            w[m, d] = np.float32(math.exp(-tm - 0.5 * (d * d) / (sigma * sigma)))
    return w


def plane_sums(d: np.ndarray):
    """(S, Q) of one plane as Python ints."""
    x = d.astype(np.uint64).ravel()
    return int(x.sum()), int((x * x).sum())


def cross_sum(a: np.ndarray, b: np.ndarray) -> int:
    return int((a.astype(np.uint64).ravel() * b.astype(np.uint64).ravel()).sum())


def align(n: int, s_t: int, q_t: int, s_j: int, q_j: int, p_tj: int):
    """(A, B) of neighbour j, or None when the cut rule cuts it."""
    cov = n * p_tj - s_t * s_j
    var_j = n * q_j - s_j * s_j
    var_t = n * q_t - s_t * s_t
    if var_j <= 0 or var_t <= 0 or cov <= 0:
        return None
    c, vj, vt = float(cov), float(var_j), float(var_t)
    if 2.0 * c * c < vj * vt:
        return None
    a = c / vj
    if a > MAX_SLOPE:
        return None
    b = (float(s_t) - a * float(s_j)) / float(n)
    return int(round(a * 65536.0)), int(round(b * 65536.0))


def check_args(radius: int, sigma: float) -> None:
    if not (isinstance(radius, (int, np.integer)) and 0 <= radius <= MAX_RADIUS):
        raise ValueError(f'radius must be an integer in [0, {MAX_RADIUS}]')
    if not (0.0 < float(sigma) <= MAX_SIGMA):
        raise ValueError(f'sigma must be in (0, {MAX_SIGMA}]')


def temporal_depth(depths, t: int, radius: int, sigma: float = 6.0):
    """(out float32 [H, W], lo, hi): frame t of the consecutive planes `depths`, filtered over the window lo..hi
    (indices into `depths`) that survives the cut rule."""
    check_args(radius, sigma)
    d_t = depths[t]
    mx = max_value(d_t.dtype)
    n = d_t.size
    s_t, q_t = plane_sums(d_t)
    win = {t: None}
    for side in (-1, 1):
        for m in range(1, radius + 1):
            j = t + side * m
            if j < 0 or j >= len(depths):
                break
            d_j = depths[j]
            ab = align(n, s_t, q_t, *plane_sums(d_j), cross_sum(d_t, d_j))
            if ab is None:
                break
            win[j] = ab
    lo, hi = min(win), max(win)
    w = weight_table(radius, sigma)
    dt = d_t.astype(np.int64)
    num = np.zeros(d_t.shape, np.float32)
    den = np.zeros(d_t.shape, np.float32)
    for j in range(lo, hi + 1):
        if j == t:
            e = dt
        else:
            a, b = win[j]
            e = np.clip((a * depths[j].astype(np.int64) + b + 32768) >> 16, 0, mx)
        delta = np.abs(e - dt)
        if mx == 65535:
            delta >>= 8
        wt = w[abs(j - t)][np.minimum(delta, 255)]
        num = num + wt * e.astype(np.float32)
        den = den + wt
    return (num / den).astype(np.float32), lo, hi


def group_windows(n_depth: int, first: int, n: int, radius: int):
    """(lo, hi) plane range that frame i of a window submission sees before the cut rule, for i in 0..n-1."""
    return [(max(0, first + i - radius), min(n_depth - 1, first + i + radius)) for i in range(n)]


def filter_group(depths, first: int, n: int, radius: int, sigma: float = 6.0):
    """The f32 planes vsc_submit_window feeds the pipeline for frames depths[first .. first + n)."""
    out = []
    for i, (lo, hi) in enumerate(group_windows(len(depths), first, n, radius)):
        o, _, _ = temporal_depth(depths[lo:hi + 1], first + i - lo, radius, sigma)
        out.append(o)
    return out
