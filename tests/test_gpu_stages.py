"""Stage-wise parity of the CUDA kernels (through the C ABI) against the CPU oracle.

Integer / index / mask stages must be bit-exact.  The float stages are bit-exact too, because the
kernels follow the oracle's operation order (DESIGN.md "Float order"); the tolerance that applies
between the oracle and the reference itself is pinned in test_oracle_golden.py.
"""
import ctypes as C

import numpy as np
import pytest

import oracle as O
from vsc_b200 import _lib
from vsc_b200.synthetic import make_depth, make_pair, make_rgb

pytestmark = pytest.mark.gpu


def _params(**kw):
    p = O.Params(**kw)
    return p, _lib.make_params(p)


# Rows of 100..115 pixels: every row-length residue mod 16 bytes, at H = 1 (the last row of a buffer is read with LSU
# loads) and at H = 17 (rows 0..15 are staged by TMA from g & ~15; an odd width puts their starts on every residue).
# Widths 100 and 112 at H >= 2 have the residues of the cases above.
LANCZOS_CASES = [(37, 160, 270), (24, 1920, 2030), (9, 3840, 3949), (11, 100, 137), (8, 64, 64)]
LANCZOS_EDGE_CASES = [(h, w, w + 37) for h in (1, 17) for w in range(100, 116) if h == 1 or w not in (100, 112)]


@pytest.mark.parametrize('h,w,dw', LANCZOS_CASES + LANCZOS_EDGE_CASES)
def test_lanczos_all_dtypes(ctx, h, w, dw):
    rng = np.random.default_rng(h * w)
    lib = _lib.load()
    rgb = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    out = np.empty((h, dw, 3), np.uint8)
    _lib.check(lib.vsc_stage_lanczos(ctx.handle, _lib.ptr(rgb), _lib.DEPTH_U8, 3, h, w, dw, _lib.ptr(out)))
    assert np.array_equal(out, O.lanczos4_h(rgb, dw))
    for dt, code, hi in ((np.uint8, _lib.DEPTH_U8, 256), (np.uint16, _lib.DEPTH_U16, 65536)):
        d = rng.integers(0, hi, (h, w)).astype(dt)
        o = np.empty((h, dw), dt)
        _lib.check(lib.vsc_stage_lanczos(ctx.handle, _lib.ptr(d), code, 1, h, w, dw, _lib.ptr(o)))
        assert np.array_equal(o, O.lanczos4_h(d, dw)), dt
    d = (rng.random((h, w), dtype=np.float32) * 3 - 1).astype(np.float32)
    o = np.empty((h, dw), np.float32)
    _lib.check(lib.vsc_stage_lanczos(ctx.handle, _lib.ptr(d), _lib.DEPTH_F32, 1, h, w, dw, _lib.ptr(o)))
    assert np.array_equal(o, O.lanczos4_h(d, dw))


def _oracle_depth(depth_st, hs, ws, p):
    d = O.normalize_depth(depth_st)
    if p.super_sampling > 1.0:
        d = O.bilinear_up(d, hs, ws)
    if p.edge_softness > 0:
        d = O.gauss_blur(d, O.soft_kernel_size(p.edge_softness), p.edge_softness)
    if p.depth_gamma != 1.0:
        d = O.apply_gamma(d, p.depth_gamma)
    return d


DEPTH_CASES = [
    (120, 270, {}),
    (90, 200, dict(super_sampling=2.5, edge_softness=3.0, depth_gamma=0.5)),
    (100, 180, dict(super_sampling=1.0, edge_softness=0.0, depth_gamma=1.0)),
    (70, 130, dict(super_sampling=1.0, edge_softness=7.5, depth_gamma=2.0)),
    (64, 150, dict(super_sampling=4.0, edge_softness=0.0, depth_gamma=0.1)),
    (200, 333, dict(super_sampling=1.7, edge_softness=30.0, depth_gamma=1.3)),
    (81, 111, {}),                                                                   # odd super-sampled width (333): scalar stores, last column unpaired
    (75, 131, dict(super_sampling=1.0, edge_softness=10.0, depth_gamma=0.7)),        # odd width, generic tap count
]
# Every generic tap count k = 5..29 with and without the upsample, depth_point_kernel at gamma 2 and 3, and 1x grids
# at the 64-pixel tile edges (64k - 1, 64k, 64k + 1) and below one tile.  Their depth maps have flat areas at the
# minimum and the maximum, so gamma meets the clamp at 0.001 and x = 1.
DEPTH_EDGE_CASES = [
    (63, 127, dict(super_sampling=1.0, edge_softness=5 / 6, depth_gamma=2.0)),
    (64, 128, dict(super_sampling=1.0, edge_softness=7 / 6, depth_gamma=3.0)),
    (65, 129, dict(super_sampling=1.0, edge_softness=9 / 6, depth_gamma=1.0)),
    (127, 63, dict(super_sampling=1.0, edge_softness=11 / 6, depth_gamma=0.5)),
    (128, 65, dict(super_sampling=1.0, edge_softness=13 / 6, depth_gamma=0.37)),
    (129, 64, dict(super_sampling=1.0, edge_softness=15 / 6, depth_gamma=3.0)),
    (20, 50, dict(super_sampling=1.0, edge_softness=17 / 6, depth_gamma=2.0)),
    (40, 191, dict(super_sampling=1.0, edge_softness=19 / 6, depth_gamma=0.2)),
    (45, 70, dict(super_sampling=1.0, edge_softness=21 / 6, depth_gamma=1.0)),
    (50, 100, dict(super_sampling=1.0, edge_softness=23 / 6, depth_gamma=0.8)),
    (33, 65, dict(super_sampling=1.0, edge_softness=25 / 6, depth_gamma=1.6)),
    (60, 130, dict(super_sampling=1.0, edge_softness=27 / 6, depth_gamma=2.0)),
    (31, 129, dict(super_sampling=1.0, edge_softness=29 / 6, depth_gamma=3.0)),
    (30, 60, dict(super_sampling=2.0, edge_softness=5 / 6, depth_gamma=3.0)),
    (25, 51, dict(super_sampling=2.5, edge_softness=7 / 6, depth_gamma=2.0)),
    (32, 64, dict(super_sampling=1.5, edge_softness=9 / 6, depth_gamma=1.0)),
    (21, 43, dict(super_sampling=3.0, edge_softness=11 / 6, depth_gamma=0.6)),
    (40, 80, dict(super_sampling=1.6, edge_softness=13 / 6, depth_gamma=3.0)),
    (22, 40, dict(super_sampling=2.9, edge_softness=15 / 6, depth_gamma=0.25)),
    (35, 71, dict(super_sampling=2.0, edge_softness=17 / 6, depth_gamma=2.0)),
    (18, 45, dict(super_sampling=4.0, edge_softness=21 / 6, depth_gamma=1.0)),
    (27, 60, dict(super_sampling=2.2, edge_softness=23 / 6, depth_gamma=0.4)),
    (29, 66, dict(super_sampling=1.9, edge_softness=25 / 6, depth_gamma=3.0)),
    (31, 70, dict(super_sampling=2.0, edge_softness=27 / 6, depth_gamma=1.3)),
    (33, 65, dict(super_sampling=2.0, edge_softness=29 / 6, depth_gamma=2.0)),
    (50, 90, dict(super_sampling=1.0, edge_softness=0.0, depth_gamma=2.0)),
    (26, 70, dict(super_sampling=2.0, edge_softness=0.0, depth_gamma=3.0)),
]


@pytest.mark.parametrize('h,sw,kw', DEPTH_CASES + DEPTH_EDGE_CASES)
def test_depth_front(ctx, h, sw, kw):
    p, cp = _params(**kw)
    depth_st = make_depth(h, sw, seed=h, dtype=np.uint16).astype(np.float32)
    if (h, sw, kw) in DEPTH_EDGE_CASES:
        depth_st[:h // 4] = 0
        depth_st[-h // 4:, :sw // 3] = 65535
    ss = p.super_sampling > 1.0
    hs, ws = (int(h * p.super_sampling), int(sw * p.super_sampling)) if ss else (h, sw)
    out = np.empty((hs, ws), np.float32)
    _lib.check(_lib.load().vsc_stage_depth(ctx.handle, _lib.ptr(depth_st), h, sw, hs, ws, C.byref(cp), _lib.ptr(out)))
    ref = _oracle_depth(depth_st, hs, ws, p)
    assert np.array_equal(out, ref), f'{(out != ref).sum()} of {out.size} differ, max {np.abs(out - ref).max()}'


def test_depth_flat_is_uniform(ctx):
    """Flat depth: range < 1e-6 -> zeros -> clamp(0.001)^gamma everywhere (SURVEY 7.3-5)."""
    p, cp = _params()
    d = np.full((64, 96), 1234.0, np.float32)
    out = np.empty((192, 288), np.float32)
    _lib.check(_lib.load().vsc_stage_depth(ctx.handle, _lib.ptr(d), 64, 96, 192, 288, C.byref(cp), _lib.ptr(out)))
    assert np.array_equal(out, _oracle_depth(d, 192, 288, p))
    assert np.unique(out).size == 1


def _oracle_warp_u8(rgb_st, depth_ss, hs, ws, md, ss, scale255=False):
    rgb_t = np.ascontiguousarray(rgb_st.astype(np.float32).transpose(2, 0, 1))
    if ss:
        rgb_t = O.bilinear_up(rgb_t, hs, ws)
    res = []
    for sign in (+1, -1):
        w, m = O.warp(rgb_t, depth_ss, md, sign)
        hwc = w.transpose(1, 2, 0)
        img = (hwc * 255).astype(np.uint8) if scale255 else hwc.astype(np.uint8)
        res += [np.ascontiguousarray(img), m, float(w.max())]
    return res


WARP_CASES = [
    (60, 200, 3.0, 50.0, 'random'), (45, 333, 1.0, 17.5, 'ties'), (30, 500, 2.0, 100.0, 'ramp'),
    (40, 1500, 1.0, 100.0, 'random'), (33, 410, 2.5, 5.0, 'discs'), (20, 2300, 1.0, 63.5, 'discs'),
]
# ss_w on the 1024-target segment edges (1024, 1025, 2048, 2049, 3073), md = 0, and a halo ceil(md) + 1 = 101 wider
# than the 96-target segment of a 90-pixel row
WARP_EDGE_CASES = [
    (4, 1024, 1.0, 30.0, 'random'), (3, 1025, 1.0, 0.0, 'random'), (3, 2048, 1.0, 12.25, 'ties'),
    (2, 2049, 1.0, 100.0, 'ramp'), (2, 3073, 1.0, 40.0, 'discs'), (12, 90, 1.0, 100.0, 'random'),
]
WARP_SCALE255_CASE = (24, 120, 3.0, 20.0)


@pytest.mark.parametrize('h,sw,s,md,kind', WARP_CASES + WARP_EDGE_CASES)
def test_warp_bit_exact(ctx, h, sw, s, md, kind):
    rng = np.random.default_rng(int(md * 10) + h)
    ss = s > 1.0
    hs, ws = (int(h * s), int(sw * s)) if ss else (h, sw)
    rgb_st = make_rgb(h, sw, seed=h)
    if kind == 'random':
        depth = rng.random((hs, ws), dtype=np.float32)
    elif kind == 'ties':
        depth = (np.rint(rng.random((hs, ws)) * 255) / 255).astype(np.float32)
    elif kind == 'ramp':
        depth = np.tile(np.linspace(0, 1, ws, dtype=np.float32)[None] ** 3, (hs, 1))
    else:
        depth = make_depth(hs, ws, seed=3, dtype=np.float32)
    depth = np.ascontiguousarray(depth)
    outs = [np.empty((hs, ws, 3), np.uint8), np.empty((hs, ws), np.uint8), np.empty((hs, ws, 3), np.uint8),
            np.empty((hs, ws), np.uint8)]
    vmax = np.zeros(2, np.float32)
    _lib.check(_lib.load().vsc_stage_warp(ctx.handle, _lib.ptr(rgb_st), _lib.ptr(depth), h, sw, hs, ws, md, 0,
                                          *[_lib.ptr(o) for o in outs], _lib.ptr(vmax)))
    l, lm, lmax, r, rm, rmax = _oracle_warp_u8(rgb_st, depth, hs, ws, md, ss)
    assert np.array_equal(outs[1], lm) and np.array_equal(outs[3], rm), 'hole masks differ'
    assert np.array_equal(outs[0], l) and np.array_equal(outs[2], r), 'warped colours differ'
    assert vmax[0] == np.float32(lmax) and vmax[1] == np.float32(rmax)


def test_warp_scale255_branch(ctx):
    """stereo_core.py:404-407: a view whose float max is <= 1.0 is multiplied by 255 before the uint8 cast."""
    h, sw, s, md = WARP_SCALE255_CASE
    hs, ws = int(h * s), int(sw * s)
    rng = np.random.default_rng(5)
    rgb_st = rng.integers(0, 2, (h, sw, 3), dtype=np.uint8)
    depth = rng.random((hs, ws), dtype=np.float32)
    outs = [np.empty((hs, ws, 3), np.uint8), np.empty((hs, ws), np.uint8), np.empty((hs, ws, 3), np.uint8),
            np.empty((hs, ws), np.uint8)]
    _lib.check(_lib.load().vsc_stage_warp(ctx.handle, _lib.ptr(rgb_st), _lib.ptr(depth), h, sw, hs, ws, md, 1,
                                          *[_lib.ptr(o) for o in outs], None))
    l, lm, _, r, rm, _ = _oracle_warp_u8(rgb_st, depth, hs, ws, md, True, scale255=True)
    assert np.array_equal(outs[0], l) and np.array_equal(outs[2], r)
    assert np.array_equal(outs[1], lm) and np.array_equal(outs[3], rm)
    assert outs[0].max() > 1


@pytest.mark.parametrize('s', [0.3, 1.0, 2.0, 3.3, 5.0])
def test_bilateral_bit_exact(ctx, s):
    rng = np.random.default_rng(int(s * 10))
    img = make_rgb(97, 131, seed=4)
    img[20:40, 30:60] = 0                      # black hole band participates in the filter
    img[rng.random((97, 131)) < 0.02] = 0
    out = np.empty_like(img)
    _lib.check(_lib.load().vsc_stage_bilateral(ctx.handle, _lib.ptr(img), 97, 131, s, _lib.ptr(out)))
    d, sc, ss = O.bilateral_params(s)
    assert np.array_equal(out, O.bilateral(img, d, sc, ss, use_fma=True))


def _inpaint_case(ctx, img, valid, keep=None):
    h, w = valid.shape
    out = img.copy()
    k0, kw = keep if keep else (0, w)
    _lib.check(_lib.load().vsc_stage_inpaint(ctx.handle, _lib.ptr(out), _lib.ptr(valid), h, w, k0, kw))
    mask = ((1 - valid.astype(np.float32)) * 255).astype(np.uint8)
    ref = img.copy()
    if mask.any():
        ref = O.telea(img, O.dilate3(mask), 3)
    return out, ref


def _masks(h, w):
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:h, 0:w]
    m = {}
    m['none'] = np.zeros((h, w), bool)
    m['1px'] = rng.random((h, w)) < 0.004
    v = np.zeros((h, w), bool); v[:, w // 3] = True; m['vcrack'] = v
    v = np.zeros((h, w), bool); v[30:50, 40:47] = True; v[60:64, 80:120] = True; m['blobs'] = v
    v = np.zeros((h, w), bool); v[:, :25] = True; m['left_band'] = v
    v = np.zeros((h, w), bool); v[:, -30:] = True; v[0:10, :] = True; m['right_band_top'] = v
    v = np.zeros((h, w), bool); v[0, 0] = v[h - 1, w - 1] = v[0, w - 1] = v[h - 1, 0] = True; v[0, 50:60] = True; v[40:50, 0] = True
    m['corners'] = v
    m['disc'] = (yy - h // 2) ** 2 + (xx - w // 2) ** 2 <= (h // 3) ** 2
    m['dense'] = rng.random((h, w)) < 0.08
    v = np.ones((h, w), bool); v[50:70, 60:90] = False; m['mostly_hole'] = v
    m['diag'] = np.abs(yy - xx * h // w) < 2
    return m


@pytest.mark.parametrize('name', ['none', '1px', 'vcrack', 'blobs', 'left_band', 'right_band_top', 'corners', 'disc',
                                  'dense', 'mostly_hole', 'diag'])
def test_inpaint_bit_exact(ctx, name):
    h, w = 120, 170
    img = make_rgb(h, w, seed=2)
    hole = _masks(h, w)[name]
    valid = (~hole).astype(np.uint8)
    img[hole] = 0
    out, ref = _inpaint_case(ctx, img, valid)
    assert np.array_equal(out, ref), f'{(out != ref).any(axis=2).sum()} px differ'


def _march_state(ctx, h, w):
    """arrival times, state bytes and order words of the last vsc_stage_inpaint call"""
    tt = np.empty((h, w), np.float32); st = np.empty((h, w), np.uint8); od = np.empty((h, w), np.uint32)
    _lib.check(_lib.load().vsc_debug_telea_state(ctx.handle, 0, _lib.ptr(tt), _lib.ptr(st), _lib.ptr(od), h * w))
    return tt, st, od


@pytest.mark.parametrize('name', ['1px', 'vcrack', 'blobs', 'left_band', 'corners', 'disc', 'dense', 'diag'])
def test_march_times_and_order_match_the_sequential_march(ctx, name):
    """Stage A of the march on its own: every arrival time T (holes, band, outer ring) equals the one-pop-at-a-time
    oracle bit for bit, and inside every cluster the hole pixels are computed in the oracle's order."""
    from scipy import ndimage
    h, w = 120, 170
    img = make_rgb(h, w, seed=2)
    hole = _masks(h, w)[name]
    valid = (~hole).astype(np.uint8)
    img[hole] = 0
    _inpaint_case(ctx, img, valid)
    tt, st, od = _march_state(ctx, h, w)
    mask = O.dilate3(((1 - valid.astype(np.float32)) * 255).astype(np.uint8))
    t_ref, ord_ref, _ = O.march_model(mask)
    _, t_seq = O.telea(img, mask, 3, return_t=True)
    assert np.array_equal(t_ref.view(np.uint32), t_seq.view(np.uint32))       # the model is the sequential march
    near = st != 0                                                             # hole, band or ring
    assert np.array_equal(near & (mask > 0), mask > 0)
    bad_t = near & (tt.view(np.uint32) != t_ref[1:-1, 1:-1].view(np.uint32))
    assert not bad_t.any(), f'{bad_t.sum()} arrival times differ, first at {np.argwhere(bad_t)[0]}'
    # clusters as the library forms them: 8x8 tiles that hold a hole / band / ring pixel, 8-connected
    th, tw = (h + 7) // 8, (w + 7) // 8
    occ = np.zeros((th * 8, tw * 8), bool); occ[:h, :w] = near
    lab, ncl = ndimage.label(occ.reshape(th, 8, tw, 8).any(axis=(1, 3)), structure=np.ones((3, 3)))
    lab_px = np.repeat(np.repeat(lab, 8, 0), 8, 1)[:h, :w]
    for c in range(1, ncl + 1):
        sel = (lab_px == c) & (mask > 0)
        if not sel.any():
            continue
        got, ref = od[sel].astype(np.int64), ord_ref[sel].astype(np.int64)
        assert len(np.unique(got)) == len(got)
        assert np.array_equal(np.argsort(got), np.argsort(ref)), f'cluster {c}: computation order differs'


def test_inpaint_const_image(ctx):
    """Constant image: the ill-conditioned unit-gradient term makes every ulp count (SURVEY A.3 item 7)."""
    img = np.full((20, 20, 3), 101, np.uint8)
    valid = np.ones((20, 20), np.uint8)
    valid[10, 10] = 0
    out, ref = _inpaint_case(ctx, img, valid)
    assert np.array_equal(out, ref)
    assert set(np.unique(out[9:12, 9:12])) <= {100, 101, 102}


def test_inpaint_crop_culling_keeps_window_exact(ctx):
    """Clusters that do not reach the kept columns are skipped; the kept columns must still be exact."""
    h, w = 160, 400
    img = make_rgb(h, w, seed=9)
    rng = np.random.default_rng(3)
    hole = np.zeros((h, w), bool)
    hole[:, 100:300] = rng.random((h, 200)) < 0.003
    hole[:, :30] = True
    hole[:, -18:] = True
    valid = (~hole).astype(np.uint8)
    img[hole] = 0
    k0, kw = 60, 280
    out, ref = _inpaint_case(ctx, img, valid, keep=(k0, kw))
    assert np.array_equal(out[:, k0:k0 + kw], ref[:, k0:k0 + kw])
    assert not np.array_equal(out[:, :20], ref[:, :20])      # the far band was really skipped
    assert (out[:, :20] == 0).all()


def test_inpaint_band_connected_to_window_stops_early(ctx):
    """A border band linked to an in-window crack is one cluster.  The march may stop once every in-window
    hole pixel is filled (later pops cannot influence earlier pixels): the window must be exact, and the deep
    part of the band, which the back end never reads, is left untouched."""
    h, w = 200, 300
    img = make_rgb(h, w, seed=12)
    hole = np.zeros((h, w), bool)
    hole[:, 240:] = True                 # wide band touching the right border
    hole[20:180, 232] = True             # crack 8 px left of the band: same cluster, inside the kept window
    hole[60:64, 150:170] = True          # separate small blob inside the window
    valid = (~hole).astype(np.uint8)
    img[hole] = 0
    k0, kw = 10, 228                     # kept columns [10, 238): crack yes, band no
    out, ref = _inpaint_case(ctx, img, valid, keep=(k0, kw))
    assert np.array_equal(out[:, k0:k0 + kw], ref[:, k0:k0 + kw])
    assert (out[:, 280:] == 0).all() and (ref[:, 280:] != 0).any()     # the deep band was not marched
    full, ref2 = _inpaint_case(ctx, img, valid)
    assert np.array_equal(full, ref2)


def test_inpaint_real_warp_masks(ctx):
    """Masks as the warp produces them at sharp depth edges (edge_softness=0)."""
    rgb, depth = make_pair(150, 260, seed=3)
    taps = {}
    O.process_frame(rgb, depth, O.Params(edge_softness=0.0, depth_gamma=1.0, super_sampling=2.0), taps)
    for side in ('left', 'right'):
        img, valid = taps['smooth_' + side], taps['mask_' + side]
        out, ref = _inpaint_case(ctx, img, valid)
        assert np.array_equal(ref, taps['inpaint_' + side])
        assert np.array_equal(out, ref), f'{side}: {(out != ref).any(axis=2).sum()} px differ'


BACKEND_CASES = [
    (360, 810, 120, 160, 135, 195, 480, 14.0), (225, 540, 90, 150, 40, 70, 375, 6.5), (100, 245, 100, 180, 37, 27, 180, 14.0),
    (360, 810, 120, 160, 135, 195, 480, 0.0), (130, 300, 100, 211, 3, 9, 274, 16.0), (256, 700, 64, 150, 50, 38, 600, 1.0),
]


def _backend_edge_cases():
    """K = 0 (2.5x), 1x, 2, 3 and 4, each on outputs of all-FULL tiles, partial tiles along x (W % 32 != 0), along y
    (H % 8 != 0) and both, with and without sharpening; the sharpened crops touch both edges of the views.  The
    combinations BACKEND_CASES already has are left out."""
    have = {(2.5, 20, 70, True), (1, 20, 70, True), (3, 16, 64, True), (3, 16, 64, False), (4, 16, 70, True)}
    cases = []
    for s in (2.5, 1, 2, 3, 4):
        for h, w in ((16, 64), (16, 70), (20, 64), (20, 70)):
            hs, cw = int(h * s), int(w * s)
            if (s, h, w, True) not in have:
                cases.append((hs, cw + 40, h, w, 0, 40, cw, 3.5 + s))
            if (s, h, w, False) not in have:
                cases.append((hs, cw + 40, h, w, 17, 23, cw, 0.0))
    return cases


BACKEND_EDGE_CASES = _backend_edge_cases()


@pytest.mark.parametrize('hs,ws,h,w,lc,rc,cw,sharp', BACKEND_CASES + BACKEND_EDGE_CASES)
def test_backend_bit_exact(ctx, hs, ws, h, w, lc, rc, cw, sharp):
    rng = np.random.default_rng(hs + w)
    left = make_rgb(hs, ws, seed=1)
    right = make_rgb(hs, ws, seed=2)
    out = np.empty((h, 2 * w, 3), np.uint8)
    _lib.check(_lib.load().vsc_stage_backend(ctx.handle, _lib.ptr(left), _lib.ptr(right), hs, ws, lc, rc, cw, h, w, sharp,
                                             _lib.ptr(out)))
    halves = []
    for img, off in ((left, lc), (right, rc)):
        v = np.ascontiguousarray(img.astype(np.float32).transpose(2, 0, 1)[:, :, off:off + cw])
        if sharp > 0:
            v = O.sharpen(v, sharp)
        if (hs, cw) != (h, w):
            v = O.area_pool(v, h, w)
        halves.append(O.to_u8_trunc(v.transpose(1, 2, 0)))
    ref = np.hstack(halves)
    assert np.array_equal(out, ref), f'{(out != ref).sum()} values differ, max {np.abs(out.astype(int) - ref).max()}'


@pytest.mark.parametrize('h,w,H,W,bits', [(153, 153, 108, 192, 16), (96, 128, 270, 480, 8), (384, 384, 1080, 1920, 16), (77, 131, 50, 60, 8)])
def test_depth_post_bit_exact(ctx, h, w, H, W, bits):
    """Producer-side depth post-processing (SURVEY 8(f) rank 3) through the C ABI: identical to the oracle."""
    from vsc_b200 import StereoGenerator
    rng = np.random.default_rng(h + bits)
    import cv2
    src = cv2.GaussianBlur(rng.random((h, w), dtype=np.float32) * 20 - 3, (0, 0), 3)
    out = np.empty((H, W), np.uint16 if bits == 16 else np.uint8)
    ok = C.c_int(0)
    _lib.check(_lib.load().vsc_stage_depth_post(ctx.handle, _lib.ptr(src), h, w, H, W, bits, _lib.ptr(out), C.byref(ok)))
    assert ok.value == 1 and np.array_equal(out, O.depth_post(src, (W, H), bits))
    flat = np.full((h, w), 1.25, np.float32)
    _lib.check(_lib.load().vsc_stage_depth_post(ctx.handle, _lib.ptr(flat), h, w, H, W, bits, _lib.ptr(out), C.byref(ok)))
    ref = O.depth_post(flat, (W, H), bits)      # a flat input may come out of the float resize not quite flat: follow the oracle
    assert bool(ok.value) == (ref is not None) and (ref is None or np.array_equal(out, ref))


def test_depth_post_feeds_the_frame_on_the_device():
    """Depth map post-processed on the slot's stream and consumed by vsc_submit_device without leaving the GPU: same
    SBS frame as quantising on the host first."""
    import torch
    from vsc_b200 import StereoGenerator, StereoParams
    rgb, _ = make_pair(108, 192, seed=4)
    rng = np.random.default_rng(9)
    import cv2
    raw = cv2.GaussianBlur(rng.random((96, 96), dtype=np.float32) * 7, (0, 0), 5)
    gen = StereoGenerator('cuda', n_slots=1)
    try:
        d_raw, d_rgb = torch.from_numpy(raw).cuda(), torch.from_numpy(rgb).cuda()
        d_q = torch.empty((108, 192), dtype=torch.uint16, device='cuda')
        d_out = torch.empty((108, 384, 3), dtype=torch.uint8, device='cuda')
        torch.cuda.synchronize()
        gen.depth_post_device(0, d_raw.data_ptr(), 96, 96, (192, 108), 16, d_q.data_ptr())
        gen.submit_device(0, d_rgb.data_ptr(), d_q.data_ptr(), np.uint16, 108, 192, d_out.data_ptr(), StereoParams())
        gen.wait(0)
        q = O.depth_post(raw, (192, 108), 16)
        assert np.array_equal(d_q.cpu().numpy().view(np.uint16), q)
        assert np.array_equal(d_out.cpu().numpy(), O.process_frame(rgb, q, O.Params()))
    finally:
        gen.close()


@pytest.mark.parametrize('which', [0, 1])
def test_arithmetic_identities_on_the_device(ctx, which):
    """The bilateral filter's reciprocal (MUFU.RCP + one Newton step, no range check) and the back end's division
    by 3 (multiply + two FMAs, scalar and packed) replace correctly rounded library operations; the device compares
    them with those operations for EVERY float of their range ([1, 256) and [0, 2295])."""
    bad = C.c_ulonglong(123)
    _lib.check(_lib.load().vsc_debug_selftest(ctx.handle, which, C.byref(bad)))
    assert bad.value == 0
