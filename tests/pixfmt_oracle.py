"""NumPy restatement of the output pixel formats (include/vsc_b200.h VSC_PIXFMT_*, VSC_MATRIX_*), for the pixel-format
tests.

Every pixel format is a fixed integer function of the final u8 RGB frame of the chosen layout, so the tests compare the
library's outputs with pack_pixfmt(pack_layout(sbs, layout), pixfmt, matrix) bit for bit.
"""
from __future__ import annotations

import numpy as np

PIXFMTS = ('rgb24', 'yuv420p', 'yuv420p10le')
MATRICES = ('bt709', 'bt601')
# rows cy, cu, cv in Q20 (limited range folded in: 219/255 for luma, 224/255 for chroma)
MATRIX = {
    'bt709': np.array([[191455, 644068, 65019], [-105533, -355018, 460551], [460551, -418321, -42230]], np.int64),
    'bt601': np.array([[269484, 528482, 102760], [-155188, -305135, 460324], [460324, -385875, -74448]], np.int64),
}


def bt709_table() -> np.ndarray:
    """The bt709 rows recomputed from Kr = 0.2126 and Kb = 0.0722 (every chroma row sums to 0)."""
    kr, kb, q = 0.2126, 0.0722, float(1 << 20)
    cy_r, cy_b = round(kr * 219 / 255 * q), round(kb * 219 / 255 * q)
    cy_g = round(219 / 255 * q) - cy_r - cy_b
    half = round(0.5 * 224 / 255 * q)
    cu_r = round(-kr / (2 * (1 - kb)) * 224 / 255 * q)
    cv_b = round(-kb / (2 * (1 - kr)) * 224 / 255 * q)
    return np.array([[cy_r, cy_g, cy_b], [cu_r, -half - cu_r, half], [half, -half - cv_b, cv_b]], np.int64)


def pack_pixfmt(rgb: np.ndarray, pixfmt: str, matrix: str = 'bt709') -> np.ndarray:
    """The frame `pixfmt` makes of a u8 RGB frame [oh, ow, 3]: rgb24 is the frame itself; the YUV formats are the I420
    planes Y [oh][ow], U [oh/2][ow/2], V [oh/2][ow/2] as one [oh * 3 // 2, ow] array (uint8, or uint16 holding 10 bits)."""
    if pixfmt == 'rgb24':
        return rgb.copy()
    if pixfmt not in PIXFMTS:
        raise ValueError(f'unknown pixel format {pixfmt!r}')
    m = MATRIX[matrix]
    oh, ow, _ = rgb.shape
    if oh % 2 or ow % 2:
        raise ValueError('yuv420 needs an even frame size')
    x = rgb.astype(np.int64)
    y = x @ m[0] + (16 << 20)
    s = x[0::2, 0::2] + x[0::2, 1::2] + x[1::2, 0::2] + x[1::2, 1::2]          # 2x2 block sums, centre-sited chroma
    cb, cr = s @ m[1] + (128 << 22), s @ m[2] + (128 << 22)
    assert y.min() >= 0 and y.max() < 2 ** 31 and min(cb.min(), cr.min()) >= 0 and max(cb.max(), cr.max()) < 2 ** 31
    if pixfmt == 'yuv420p':
        planes = [(y + (1 << 19)) >> 20, (cb + (1 << 21)) >> 22, (cr + (1 << 21)) >> 22]
        dt = np.uint8
    else:
        planes = [(y + (1 << 17)) >> 18, (cb + (1 << 19)) >> 20, (cr + (1 << 19)) >> 20]
        dt = np.uint16
    flat = np.concatenate([p.reshape(-1) for p in planes]).astype(dt)
    return flat.reshape(oh * 3 // 2, ow)


def split_planes(frame: np.ndarray):
    """(Y, U, V) views of a [oh * 3 // 2, ow] I420 frame."""
    oh, ow = frame.shape[0] * 2 // 3, frame.shape[1]
    flat = frame.reshape(-1)
    n = oh * ow
    return (flat[:n].reshape(oh, ow), flat[n:n + n // 4].reshape(oh // 2, ow // 2),
            flat[n + n // 4:].reshape(oh // 2, ow // 2))
