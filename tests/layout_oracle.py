"""NumPy restatement of the output layouts (include/vsc_b200.h VSC_LAYOUT_*), for the layout tests.

Every layout is a fixed function of the full side-by-side frame that oracle.process_frame computes, so the tests
compare the library's layout outputs with pack_layout(sbs, layout) bit for bit.
"""
from __future__ import annotations

import numpy as np

# ---- output layouts (include/vsc_b200.h VSC_LAYOUT_*) --------------------------------------------
LAYOUTS = ('sbs', 'half-sbs', 'tb', 'half-tb', 'anaglyph')
ANAGLYPH_ML = np.array([[0.437, 0.449, 0.164], [-0.062, -0.062, -0.024], [-0.048, -0.050, -0.017]], np.float32)
ANAGLYPH_MR = np.array([[-0.011, -0.032, -0.007], [0.377, 0.761, 0.009], [-0.026, -0.093, 1.234]], np.float32)


def _avg2_rhe(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """(a + b) / 2 of u8 arrays, rounded half to even: (s >> 1) + (s & (s >> 1) & 1) on the integer sum."""
    s = a.astype(np.uint16) + b.astype(np.uint16)
    return ((s >> 1) + (s & (s >> 1) & 1)).astype(np.uint8)


def anaglyph(left: np.ndarray, right: np.ndarray) -> np.ndarray:
    """Dubois least-squares red-cyan of two u8 [H, W, 3] eyes: float32, every product and sum rounded in the order
    ((((ML0*l0 + ML1*l1) + ML2*l2) + MR0*r0) + MR1*r1) + MR2*r2, then clamp to [0, 255] and round half to even."""
    l, r = left.astype(np.float32), right.astype(np.float32)
    out = np.empty(left.shape, np.uint8)
    for c in range(3):
        s = ANAGLYPH_ML[c, 0] * l[..., 0] + ANAGLYPH_ML[c, 1] * l[..., 1]
        s = s + ANAGLYPH_ML[c, 2] * l[..., 2]
        s = s + ANAGLYPH_MR[c, 0] * r[..., 0]
        s = s + ANAGLYPH_MR[c, 1] * r[..., 1]
        s = s + ANAGLYPH_MR[c, 2] * r[..., 2]
        out[..., c] = np.rint(np.clip(s, np.float32(0), np.float32(255))).astype(np.uint8)
    return out


def pack_layout(sbs: np.ndarray, layout: str) -> np.ndarray:
    """The frame `layout` makes of a full side-by-side frame u8 [H, 2W, 3] (left | right)."""
    h, w2, _ = sbs.shape
    w = w2 // 2
    left, right = sbs[:, :w], sbs[:, w:]
    if layout == 'sbs':
        return sbs.copy()
    if layout == 'tb':
        return np.ascontiguousarray(np.vstack([left, right]))
    if layout == 'half-sbs':
        if w % 2:
            raise ValueError('half-sbs needs an even width')
        return np.ascontiguousarray(np.hstack([_avg2_rhe(e[:, 0::2], e[:, 1::2]) for e in (left, right)]))
    if layout == 'half-tb':
        if h % 2:
            raise ValueError('half-tb needs an even height')
        return np.ascontiguousarray(np.vstack([_avg2_rhe(e[0::2], e[1::2]) for e in (left, right)]))
    if layout == 'anaglyph':
        return anaglyph(left, right)
    raise ValueError(f'unknown layout {layout!r}')
