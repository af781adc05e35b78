"""Coverage manifest of the CUDA kernel variants: a restatement of the host dispatch in vsc_api.cu.

Every GPU parity case is mapped to the cells it reaches: a kernel instantiation together with the device-side branch
or tile edge that the host's choice of geometry puts it on.  REQUIRED lists the cells the suite must reach, each group
with the dispatch line that creates it.  test_variant_matrix.py checks, on the CPU, that the cases of the GPU test
files reach every required cell, that this restatement agrees with the library's own geometry and that the
instantiation lists of vsc_api.cu are the ones listed here.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

# ---- instantiations (the template arguments vsc_api.cu launches) ------------------------------------------------
BILATERAL_RADII = (2, 3, 4, 5, 6, 7)          # run_bilateral: switch (a.taps.radius)
BACKEND_K = (0, 2, 3, 4)                      # run_backend: switch (K), set_smem_attrs: backend_attrs<K>
MARCH_WARPS = (16, 32)                        # run_telea: telea_march_kernel<32> (one slot) / <16>
DEPTH_FRONT_TAPS = (0, 31)                    # run_depth_front: depth_front_kernel<31> / <0> (run-time tap count)
LAYOUTS = ('sbs', 'half-sbs', 'tb', 'half-tb', 'anaglyph')
PIXFMTS = ('rgb24', 'yuv420p', 'yuv420p10le')

BE_OX, BE_OY = 32, 8                          # vsc_kernels.cuh: back-end output tile
DF_T = 64                                     # vsc_kernels.cuh: depth front-end output tile
WARP_SEG = 1024                               # run_warp: nseg = (ss_w + 1023) / 1024
MARCH_SMEM_COUNTERS = 32768                   # vsc_march.cuh: counters of larger clusters live in global memory
LANCZOS_ES = {'rgb': 3, 'u8': 1, 'u16': 2, 'f32': 4}


def params(**kw):
    """The stereo parameters with the library's defaults (vsc_default_params)."""
    p = dict(max_disparity=50.0, convergence=-10.0, super_sampling=3.0, edge_softness=20.0, artifact_smoothing=1.0,
             depth_gamma=0.2, sharpen=14.0)
    p.update(kw)
    return SimpleNamespace(**p)


def blur_k(edge_softness: float) -> int:
    """Depth blur taps (vsc_geometry; 0 = no blur, depth_point_kernel)."""
    if edge_softness <= 0:
        return 0
    return max(min(int(edge_softness * 6) | 1, 31), 5)


def bilateral_d(smoothing: float) -> int:
    """Bilateral window (vsc_geometry, run_bilateral; 0 = no filter)."""
    return max(min(int(smoothing * 4), 15), 5) if smoothing > 0 else 0


def backend_k(hs: int, cw: int, h: int, w: int) -> int:
    """run_backend: compile-time tile geometry for integer super-sampling 2..4, else 0 (1x included)."""
    k = 0
    for c in (2, 3, 4):
        if hs == c * h and cw == c * w:
            k = c
    return k


def geometry(h: int, w: int, p) -> dict:
    """vsc_geometry in Python: the frame geometry, and `refused` = the reason the library refuses the frame (or None)."""
    total = 2.0 * p.max_disparity + abs(p.convergence)
    sw = int(w * (1.0 + total / w))
    ss = p.super_sampling > 1.0
    hs, ws = (int(h * p.super_sampling), int(sw * p.super_sampling)) if ss else (h, sw)
    base = (sw - w) // 2
    cs = round(p.convergence)
    lo, ro = base + cs, base - cs
    if ss:
        r = ws / sw
        lc, rc, cw = int(lo * r), int(ro * r), int(w * r)
    else:
        lc, rc, cw = lo, ro, w
    g = dict(h=h, w=w, sw=sw, hs=hs, ws=ws, lc=lc, rc=rc, cw=cw, ss=ss, blur_k=blur_k(p.edge_softness),
             bilateral_d=bilateral_d(p.artifact_smoothing), K=backend_k(hs, cw, h, w), refused=None)
    if h < 8 or w < 8:
        g['refused'] = 'smaller than 8x8'
    elif lo < 0 or ro < 0:
        g['refused'] = 'crop left of the stretched view'
    elif cw < 3 or hs < 3:
        g['refused'] = 'crop too small'
    elif g['blur_k'] // 2 >= hs or g['blur_k'] // 2 >= ws:
        g['refused'] = 'depth blur does not fit (reflect pad)'
    return g


def tile_class(h: int, w: int) -> str:
    """Back-end tiles of an h x w output: all FULL, or partial along x (W % 32), y (H % 8) or both."""
    px, py = w % BE_OX != 0, h % BE_OY != 0
    return {(False, False): 'full', (True, False): 'partial-x', (False, True): 'partial-y', (True, True): 'partial-xy'}[(px, py)]


def _edge64(n: int) -> str:
    if n < DF_T:
        return '<64'
    return {DF_T - 1: '64k-1', 0: '64k', 1: '64k+1'}.get(n % DF_T, 'mid')


def _gamma_class(g: float) -> str:
    return {1.0: '1', 2.0: '2', 3.0: '3'}.get(float(g), 'frac')


# ---- cells of one stage call -------------------------------------------------------------------------------------
def lanczos_cells(h: int, w: int, dw: int):
    """vsc_stage_lanczos for rgb, u8, u16 and f32 rows of h x w (test_lanczos_all_dtypes).  Rows 0..h-2 are staged by
    TMA from `g & ~15` (start residue y * w * es mod 16); the last row (the only one at h = 1) goes through LSU loads."""
    cells = set()
    for dt, es in LANCZOS_ES.items():
        cells.add(('lanczos', dt, 'len', (w * es) % 16, 'H1' if h == 1 else 'H2+'))
        for y in range(min(h - 1, 16)):
            cells.add(('lanczos', dt, 'tma-start', (y * w * es) % 16))
    return cells


def depth_cells(h: int, sw: int, kw: dict):
    """vsc_stage_depth (test_depth_front): run_depth_front picks depth_front_kernel<31>, <0> (k taps) or
    depth_point_kernel; tiles of 64 x 64 outputs for the blur kernels."""
    p = params(**kw)
    up = p.super_sampling > 1.0
    hs, ws = (int(h * p.super_sampling), int(sw * p.super_sampling)) if up else (h, sw)
    k = blur_k(p.edge_softness)
    kern = 'point' if k == 0 else k
    cells = {('depth', kern, 'up' if up else '1x'),
             ('depth-gamma', 'point' if k == 0 else 'front', _gamma_class(p.depth_gamma))}
    if k:
        cells |= {('depth-edge', 'w', _edge64(ws)), ('depth-edge', 'h', _edge64(hs))}
    return cells


def warp_cells(h: int, sw: int, s: float, md: float, kind: str = '', scale255: bool = False):
    """vsc_stage_warp (test_warp_bit_exact; scale255 adds the MODE 2 re-run): segments of 1024 targets, halo R."""
    hs, ws = (int(h * s), int(sw * s)) if s > 1.0 else (h, sw)
    nseg = (ws + WARP_SEG - 1) // WARP_SEG
    ts = -(-((ws + nseg - 1) // nseg) // 32) * 32
    halo = math.ceil(md) + 1
    cells = {('warp-mode', 0)}
    if ws == nseg * WARP_SEG:
        cells.add(('warp-seg', nseg, 'exact'))
    elif ws == (nseg - 1) * WARP_SEG + 1:
        cells.add(('warp-seg', nseg, 'plus1'))
    cells.add(('warp-md', 'zero' if md == 0 else 'halo>TS' if halo > ts else 'frac' if md != int(md) else 'int'))
    if scale255:
        cells.add(('warp-mode', 2))
    return cells


def bilateral_cells(h: int, w: int, s: float):
    """vsc_stage_bilateral: bilateral_kernel<R>; interior 32 x 32 tiles stage pixel pairs, aligned when Ws and R are
    even, else with odd-start rows (all rows for odd R and even Ws, every other row for odd Ws); border tiles reflect."""
    r = bilateral_d(s) // 2
    cells = {('bilateral', r, 'reflect')}
    interior = h >= 64 + r and w >= 64 + r
    if interior:
        cells.add(('bilateral', r, 'odd-alternate' if w % 2 else 'odd-all' if r % 2 else 'aligned'))
    return cells


def backend_stage_cells(hs, ws, h, w, lc, rc, cw, sharp):
    """vsc_stage_backend (test_backend_bit_exact): K with the tile class of the h x w output, sharpen on or off
    (1x super-sampling is K = 0 through its own branch), and crop windows at the edges of the views."""
    k = backend_k(hs, cw, h, w)
    kc = '1x' if (hs, cw) == (h, w) else k
    cells = {('backend-stage', kc, tile_class(h, w), 'sharpen' if sharp > 0 else 'no-sharpen')}
    if 0 in (lc, rc):
        cells.add(('backend-crop', 'left-edge'))
    if ws in (lc + cw, rc + cw):
        cells.add(('backend-crop', 'right-edge'))
    return cells


def layout_frame_cells(h: int, w: int, kw: dict):
    """One frame through StereoGenerator in every layout and pixel format (BT.709, and BT.601 for the YUV formats):
    backend_kernel<K, L, P> on the frame's tiles (run_backend -> launch_backend)."""
    g = geometry(h, w, params(**kw))
    cells = set()
    for lay in LAYOUTS:
        for pf in PIXFMTS:
            cells.add(('backend', g['K'], tile_class(h, w), lay, pf))
    cells |= {('yuv-matrix', pf, 'bt601') for pf in PIXFMTS[1:]}
    return cells


def march_cells(rect_h: int, rect_w: int, n_slots: int):
    """One rectangular cluster whose dilated mask is rect_h x rect_w through vsc_stage_inpaint: its tasks are the hole
    pixels of the dilated mask; the march counts in shared memory up to MARCH_SMEM_COUNTERS tasks, in global memory
    above; a one-slot context runs the 32-warp march."""
    ntask = rect_h * rect_w
    nw = 32 if n_slots == 1 else 16
    cells = {('march', nw, 'smem' if ntask <= MARCH_SMEM_COUNTERS else 'global')}
    if ntask in (MARCH_SMEM_COUNTERS, MARCH_SMEM_COUNTERS + 1):
        cells.add(('march-ntask', ntask))
    return cells


def min_frame_cells(h: int, w: int, name: str):
    return {('min-frame', h, w, name)}


def device_offset_cells(offset: int, depth_dtype: str):
    """vsc_submit_device with rgb and depth pointers `offset` bytes past a 16-byte boundary: the Lanczos kernels'
    TMA staging starts at `g & ~15`."""
    return {('submit-device', 'rgb', offset), ('submit-device', depth_dtype, offset)}


# ---- what the suite must reach -----------------------------------------------------------------------------------
def _required():
    req = set()
    # run_lanczos_rgb / run_lanczos_depth: every row-length residue at H = 1 (LSU only) and H >= 2, and every TMA row
    # start residue an element size allows (cp.async.bulk from g & ~15, vsc_common.cuh)
    for dt, es in LANCZOS_ES.items():
        res = sorted({(i * es) % 16 for i in range(16)})
        req |= {('lanczos', dt, 'len', r, hh) for r in res for hh in ('H1', 'H2+')}
        req |= {('lanczos', dt, 'tma-start', r) for r in res}
    # run_depth_front: depth_front_kernel<31> for k = 31, depth_front_kernel<0> for every other odd k, and
    # depth_point_kernel for edge_softness 0, each with and without the bilinear upsample (g.super_sampled)
    for kern in [k for k in range(5, 32, 2)] + ['point']:
        req |= {('depth', kern, 'up'), ('depth', kern, '1x')}
    # grid ((ss_w + 63) / 64, (ss_h + 63) / 64): both sides at a tile edge and below one tile
    req |= {('depth-edge', ax, e) for ax in 'wh' for e in ('<64', '64k-1', '64k', '64k+1')}
    # det_powf (vsc_common.cuh): gamma 1 skips it (apply_gamma), 2 and 3 are exact products, anything else the tables
    req |= {('depth-gamma', kern, g) for kern in ('front', 'point') for g in ('1', '2', '3', 'frac')}
    # run_warp: nseg = (ss_w + 1023) / 1024, one segment exactly full and the first target of a new segment
    req |= {('warp-seg', 1, 'exact'), ('warp-seg', 2, 'plus1'), ('warp-seg', 2, 'exact'), ('warp-seg', 3, 'plus1'),
            ('warp-seg', 4, 'plus1')}
    # run_warp: a.R = ceil(md) + 1 against the segment width TS
    req |= {('warp-md', m) for m in ('zero', 'frac', 'int', 'halo>TS')}
    # warp_kernel<0>; <1> in enqueue_group (smoothing on) re-runs the views whose max is <= 1; <2> in vsc_stage_warp
    req |= {('warp-mode', 0), ('warp-mode', 2), ('warp-mode', 1, 'one-eye'), ('warp-mode', 1, 'both')}
    # run_bilateral: bilateral_kernel<R>, R = 2..7, staging branches of vsc_kernels.cuh (((Ws | R) & 1) == 0)
    for r in BILATERAL_RADII:
        req |= {('bilateral', r, 'reflect'), ('bilateral', r, 'odd-alternate'),
                ('bilateral', r, 'odd-all' if r % 2 else 'aligned')}
    # run_backend via vsc_stage_backend: K in {0, 1x, 2, 3, 4}, FULL and partial tiles (backend_kernel's
    # blockIdx test), sharpen on and off (a.do_sharpen)
    for kc in (0, '1x', 2, 3, 4):
        req |= {('backend-stage', kc, t, s) for t in ('full', 'partial-x', 'partial-y', 'partial-xy')
                for s in ('sharpen', 'no-sharpen')}
    req |= {('backend-crop', 'left-edge'), ('backend-crop', 'right-edge')}
    # launch_backend<K>(layout, pixfmt): every backend_kernel<K, L, P> on a partial-tile frame and on an all-FULL one
    req |= {('backend', k, t, lay, pf) for k in BACKEND_K for t in ('full', 'partial-xy') for lay in LAYOUTS
            for pf in PIXFMTS}
    req |= {('yuv-matrix', pf, 'bt601') for pf in PIXFMTS[1:]}               # kYuvMatrix[VSC_MATRIX_BT601]
    # run_telea: telea_march_kernel<32> / <16>; march_colour: `small = ntask <= MARCH_SMEM_COUNTERS`
    req |= {('march', nw, c) for nw in MARCH_WARPS for c in ('smem', 'global')}
    req |= {('march-ntask', MARCH_SMEM_COUNTERS), ('march-ntask', MARCH_SMEM_COUNTERS + 1)}
    req.add(('march-views', 8))                                                # TELEA_MAX_VIEWS: 4 frames x 2 eyes
    # vsc_geometry accepts frames from 8 x 8
    for hw in ((8, 8), (8, 9), (9, 8), (10, 33)):
        req |= {('min-frame', *hw, name) for name in ('default', 'ss1-noblur', 'ss2', 'ss4')}
    # vsc_submit_device: any element-aligned input pointer
    req |= {('submit-device', 'rgb', o) for o in range(1, 16)}
    req |= {('submit-device', 'u8', o) for o in range(1, 16, 2)} | {('submit-device', 'u16', o) for o in range(2, 16, 2)}
    return req


REQUIRED = frozenset(_required())
