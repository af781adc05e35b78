"""Torch CPU restatement of the three module-level helpers of the reference's `helper/stereo_core.py` (`:71-190`):
`normalize_depth`, `apply_depth_gamma` and `forward_warp_stereo`, for the helper tests.

Each function states the reference's algorithm literally, in the same torch operations on the CPU and in the input's
float32, so it accepts any float32 input the reference accepts: negative or unnormalised depth, ±0.0, ±inf and NaN.
The tests compare the library's helpers with these functions bit for bit.
"""
from __future__ import annotations

import numpy as np
import torch


def normalize_depth(depth: torch.Tensor) -> torch.Tensor:
    """Global min / max; zeros if max - min < 1e-6, else (d - min) / (max - min) (SURVEY a6).  torch's min() and max()
    propagate NaN, so a NaN anywhere gives an all-NaN result.  The range test is the float32 tensor comparison."""
    mn, mx = depth.min(), depth.max()
    if mx - mn < 1e-6:
        return torch.zeros_like(depth)
    return (depth - mn) / (mx - mn)


def apply_depth_gamma(depth: torch.Tensor, gamma: float) -> torch.Tensor:
    """clamp(d, 0.001, 1) ** gamma, with torch's pow stated exactly: the float64 power rounded to float32, except ATen's
    float products for gamma = 2 and 3 (pow_tensor_scalar_optimized_kernel).  clamp propagates NaN, and x ** 0 is 1 for
    every x, NaN included.  torch.pow itself is within 1 ulp of this (Sleef)."""
    x = torch.clamp(depth, 0.001, 1.0)
    g = float(np.float32(gamma))          # ATen casts the scalar exponent to the tensor's float32
    if g == 2.0:
        return x * x
    if g == 3.0:
        return x * x * x
    return torch.from_numpy(np.power(x.numpy().astype(np.float64), g).astype(np.float32))


def warp_literal(image: np.ndarray, depth: np.ndarray, md: float, sign: int):
    """forward_warp_stereo's algorithm for one direction (sign +1: left view, -1: right view), stated literally:
    ascending-depth argsort, floor scatters, then ceil scatters of the frac > 0.3 subset, last writer wins.

    image [C, H, W] f32, depth [H, W] f32 -> (warped [C, H, W] f32, mask [H, W] u8 = weight > 0.1).  A source whose
    target is NaN, ±inf or outside int64 writes nothing: torch's floor().long() gives INT64_MIN for it on the CPU
    (test_floor_long_of_non_finite_is_negative pins that)."""
    c, h, w = image.shape
    d = torch.from_numpy(depth).flatten()
    order = torch.argsort(d)
    ys = (torch.arange(h * w) // w)[order]
    xs = (torch.arange(h * w) % w).float()[order]
    tx = xs + sign * (d * md)[order]
    fl = tx.floor().long()
    frac = tx - fl.float()
    img = torch.from_numpy(image).reshape(c, -1)
    out = torch.zeros(c, h * w)
    wgt = torch.zeros(h * w)
    ok = (fl >= 0) & (fl < w)
    idx = (ys * w + fl)[ok]
    for ch in range(c):
        out[ch].scatter_(0, idx, img[ch, order[ok]])
    wgt.scatter_(0, idx, (1.0 - frac)[ok])
    ce = fl + 1
    ok = (ce >= 0) & (ce < w) & (frac > 0.3)
    idx = (ys * w + ce)[ok]
    for ch in range(c):
        out[ch].scatter_(0, idx, img[ch, order[ok]])
    wgt.scatter_(0, idx, frac[ok])
    return out.reshape(c, h, w).numpy(), (wgt > 0.1).reshape(h, w).numpy().astype(np.uint8)


def forward_warp_stereo(image: torch.Tensor, depth: torch.Tensor, max_disparity: float):
    """image [1, C, H, W], depth [1, 1, H, W] -> (left, left_mask, right, right_mask) float32 tensors of the reference's
    shapes [1, C, H, W] / [1, 1, H, W]; the masks hold 0 / 1."""
    _, c, h, w = image.shape
    img = np.ascontiguousarray(image[0].numpy())
    dep = np.ascontiguousarray(depth.reshape(h, w).numpy())
    res = []
    for sign in (+1, -1):
        v, m = warp_literal(img, dep, max_disparity, sign)
        res += [torch.from_numpy(v)[None], torch.from_numpy(m.astype(np.float32))[None, None]]
    return tuple(res)
