"""Kernel variants at their edges, each bit-exact against the oracle: bilateral radii and staging branches, the back end's
layouts and pixel formats on partial and FULL tiles, the warp's per-eye re-run, the march's counter stores and warp
counts, the smallest frames and unaligned device inputs.  The module-level case lists are what variant_matrix.py maps
to kernel cells; test_variant_matrix.py checks on the CPU that they reach every required cell."""
import numpy as np
import pytest

import layout_oracle as LO
import oracle as O
import pixfmt_oracle as PO
from vsc_b200 import StereoGenerator, StereoParams, _lib
from vsc_b200.synthetic import make_pair, make_rgb

pytestmark = pytest.mark.gpu

# (Hs, Ws, smoothing): R = 2..7 at an even and an odd width, interior tiles, Hs not a multiple of 4 or 32
BILATERAL_CASES = [(101, 130, 0.3), (101, 131, 0.3), (101, 130, 1.5), (101, 131, 1.5), (101, 130, 2.0), (101, 131, 2.0),
                   (101, 130, 2.5), (101, 131, 2.5), (101, 130, 3.0), (101, 131, 3.0), (101, 130, 3.5), (101, 131, 5.0)]

# (H, W, params): K = 0 (2.5x), 2, 3 and 4 on a frame with partial tiles along x and y (W % 32, H % 8 != 0) and on an
# all-FULL frame; both sides divisible by 4 so that every layout takes every pixel format
_LP = dict(max_disparity=12.0, convergence=-3.0, edge_softness=2.0, artifact_smoothing=1.0, depth_gamma=0.5, sharpen=6.0)
LAYOUT_FRAMES = [(h, w, dict(_LP, super_sampling=s)) for s in (2.5, 2.0, 3.0, 4.0) for h, w in ((52, 100), (48, 96))]

# warp_kernel<1>: the views whose float max is <= 1.0 are warped again and scaled by 255 (smoothing on)
WARP_MODE1_FRAMES = ['one-eye', 'both']

# (rows, cols of the dilated hole rectangle, slots of the context): 32 768 tasks count in shared memory, 32 769 in
# global memory; one slot runs telea_march_kernel<32>, two slots <16>
MARCH_CASES = [(128, 256, 1), (128, 256, 2), (99, 331, 1), (99, 331, 2)]

# the smallest frames vsc_geometry accepts, at default parameters, 1x without the depth blur, 2x and 4x
MIN_PARAMS = {'default': {}, 'ss1-noblur': dict(super_sampling=1.0, edge_softness=0.0), 'ss2': dict(super_sampling=2.0),
              'ss4': dict(super_sampling=4.0)}
MIN_FRAMES = [(h, w, name) for h, w in ((8, 8), (8, 9), (9, 8), (10, 33)) for name in MIN_PARAMS]

# (byte offset of the rgb and depth pointers past a 16-byte boundary, depth dtype): element-aligned offsets 1..15
DEVICE_OFFSETS = [(o, 'u16' if o % 2 == 0 else 'u8') for o in range(1, 16)]
_DT = {'u8': np.uint8, 'u16': np.uint16}


@pytest.fixture(scope='module')
def ctx1():
    c = _lib.Context(0, 1)
    yield c
    c.close()


@pytest.fixture(scope='module')
def ctx2():
    c = _lib.Context(0, 2)
    yield c
    c.close()


@pytest.fixture(scope='module')
def gen():
    g = StereoGenerator('cuda', n_slots=2)
    yield g
    g.close()


@pytest.mark.parametrize('h,w,s', BILATERAL_CASES)
def test_bilateral_radius_and_staging(ctx2, h, w, s):
    img = make_rgb(h, w, seed=w)
    img[40:60, 50:90] = 0
    img[np.random.default_rng(h + w).random((h, w)) < 0.02] = 0
    out = np.empty_like(img)
    _lib.check(_lib.load().vsc_stage_bilateral(ctx2.handle, _lib.ptr(img), h, w, s, _lib.ptr(out)))
    d, sc, ss = O.bilateral_params(s)
    ref = O.bilateral(img, d, sc, ss, use_fma=True)
    assert np.array_equal(out, ref), f'{(out != ref).any(axis=2).sum()} px differ, first at {np.argwhere((out != ref).any(axis=2))[0]}'


_sbs_cache = {}


def _layout_frame(i):
    """The frame of LAYOUT_FRAMES[i] and its oracle SBS frame (computed once)."""
    if i not in _sbs_cache:
        h, w, kw = LAYOUT_FRAMES[i]
        rgb, depth = make_pair(h, w, seed=i, depth_dtype=np.uint16)
        _sbs_cache[i] = rgb, depth, O.process_frame(rgb, depth, O.Params(**kw))
    return _sbs_cache[i]


@pytest.mark.parametrize('i', range(len(LAYOUT_FRAMES)), ids=[f'{h}x{w}-ss{kw["super_sampling"]}' for h, w, kw in LAYOUT_FRAMES])
def test_every_layout_and_pixfmt_on_the_tile_edges(gen, i):
    h, w, kw = LAYOUT_FRAMES[i]
    rgb, depth, sbs = _layout_frame(i)
    p = StereoParams(**kw)
    combos = [(lay, pf, 'bt709') for lay in LO.LAYOUTS for pf in PO.PIXFMTS] + [('sbs', pf, 'bt601') for pf in PO.PIXFMTS[1:]]
    try:
        for lay, pf, mx in combos:
            gen.set_layout(lay)
            gen.set_pixfmt(pf, mx)
            out = gen.process_frame(rgb, depth, p)
            ref = PO.pack_pixfmt(LO.pack_layout(sbs, lay), pf, mx)
            assert out.shape == ref.shape and np.array_equal(out, ref), (lay, pf, mx, int((out != ref).sum()))
    finally:
        gen.set_layout('sbs')
        gen.set_pixfmt('rgb24')


def mode1_frame(which):
    """A frame whose warped views have float max <= 1.0 in both eyes ('both': rgb in {0, 1}) or in the right eye only
    ('one-eye': a bright strip at the left border on the nearest depth, which the right eye's shift pushes out of the
    view)."""
    h, w = 40, 120
    rng = np.random.default_rng(7)
    rgb = rng.integers(0, 2, (h, w, 3), dtype=np.uint8)
    depth = np.zeros((h, w), np.uint8)
    depth[:, :24] = 255
    if which == 'one-eye':
        rgb[:, :4] = 200
    kw = dict(max_disparity=40.0, convergence=0.0, super_sampling=2.0, edge_softness=0.0, artifact_smoothing=1.5,
              depth_gamma=1.0, sharpen=4.0)
    return rgb, depth, kw


@pytest.mark.parametrize('which', WARP_MODE1_FRAMES)
def test_warp_rerun_per_eye(gen, which):
    rgb, depth, kw = mode1_frame(which)
    taps = {}
    ref = O.process_frame(rgb, depth, O.Params(**kw), taps)
    scaled = (taps['warp_left'].max() <= 1.0, taps['warp_right'].max() <= 1.0)
    assert scaled == {'one-eye': (False, True), 'both': (True, True)}[which]
    assert np.array_equal(gen.process_frame(rgb, depth, StereoParams(**kw)), ref)


def march_image(rect_h, rect_w):
    """An image with one hole rectangle whose 3x3 dilation is rect_h x rect_w (the cluster's hole pixels)."""
    h, w = rect_h + 37, rect_w + 45
    img = make_rgb(h, w, seed=rect_w)
    hole = np.zeros((h, w), bool)
    hole[21:21 + rect_h - 2, 17:17 + rect_w - 2] = True
    img[hole] = 0
    return img, (~hole).astype(np.uint8)


@pytest.mark.parametrize('rect_h,rect_w,n_slots', MARCH_CASES)
def test_march_counter_store_and_warp_count(ctx1, ctx2, rect_h, rect_w, n_slots):
    c = ctx1 if n_slots == 1 else ctx2
    img, valid = march_image(rect_h, rect_w)
    h, w = valid.shape
    out = img.copy()
    _lib.check(_lib.load().vsc_stage_inpaint(c.handle, _lib.ptr(out), _lib.ptr(valid), h, w, 0, w))
    mask = O.dilate3(((1 - valid.astype(np.float32)) * 255).astype(np.uint8))
    assert (mask > 0).sum() == rect_h * rect_w
    ref, t_seq = O.telea(img, mask, 3, return_t=True)
    assert np.array_equal(out, ref), f'{(out != ref).any(axis=2).sum()} px differ'
    tt = np.empty((h, w), np.float32); st = np.empty((h, w), np.uint8); od = np.empty((h, w), np.uint32)
    _lib.check(_lib.load().vsc_debug_telea_state(c.handle, 0, _lib.ptr(tt), _lib.ptr(st), _lib.ptr(od), h * w))
    t_ref, ord_ref, _ = O.march_model(mask)
    assert np.array_equal(t_ref.view(np.uint32), t_seq.view(np.uint32))
    near = st != 0
    bad_t = near & (tt.view(np.uint32) != t_ref[1:-1, 1:-1].view(np.uint32))
    assert not bad_t.any(), f'{bad_t.sum()} arrival times differ'
    sel = mask > 0
    assert np.array_equal(np.argsort(od[sel].astype(np.int64)), np.argsort(ord_ref[sel].astype(np.int64)))


def group_frames():
    """Four frames of one size: frame 0 has a sharp depth step whose disocclusion is one cluster of more than 32 768
    hole pixels; the others have small clusters."""
    frames = [make_pair(128, 256, seed=s, depth_dtype=np.uint8) for s in range(4)]
    rgb0 = frames[0][0]
    d0 = np.zeros((128, 256), np.uint8)
    d0[:, 128:] = 255
    frames[0] = (rgb0, d0)
    kw = dict(max_disparity=100.0, convergence=0.0, super_sampling=3.0, edge_softness=0.0, depth_gamma=1.0)
    return frames, kw


def test_grouped_march_with_one_big_cluster():
    from scipy import ndimage
    frames, kw = group_frames()
    refs, big = [], 0
    for rgb, depth in frames:
        taps = {}
        refs.append(O.process_frame(rgb, depth, O.Params(**kw), taps))
        for side in ('left', 'right'):
            m = O.dilate3(taps['inpaint_mask_' + side]) > 0
            lab, n = ndimage.label(m, structure=np.ones((3, 3)))
            big = max([big] + [int((lab == c).sum()) for c in range(1, n + 1)])
    assert big > 32768
    g = StereoGenerator('cuda', n_slots=1, group_size=4)
    try:
        outs = g.process_batch(frames, StereoParams(**kw))
    finally:
        g.close()
    for i, (o, r) in enumerate(zip(outs, refs)):
        assert np.array_equal(o, r), f'frame {i}: {(o != r).sum()} values differ'


@pytest.mark.parametrize('h,w,name', MIN_FRAMES)
def test_smallest_frames(gen, h, w, name):
    kw = MIN_PARAMS[name]
    rgb, depth = make_pair(h, w, seed=h * w, depth_dtype=np.uint16)
    ref = O.process_frame(rgb, depth, O.Params(**kw))
    assert np.array_equal(gen.process_frame(rgb, depth, StereoParams(**kw)), ref)


_aligned_cache = {}


@pytest.mark.parametrize('offset,dt', DEVICE_OFFSETS)
def test_submit_device_unaligned_inputs(gen, offset, dt):
    import torch
    h, w = 24, 70
    rgb, depth = make_pair(h, w, seed=5, depth_dtype=_DT[dt])
    p = StereoParams(max_disparity=20.0, convergence=-4.0)
    shape = gen.output_shape(h, w)

    def run(off):
        rb, db = rgb.tobytes(), depth.tobytes()
        buf_r = torch.zeros(len(rb) + 64, dtype=torch.uint8, device='cuda')
        buf_d = torch.zeros(len(db) + 64, dtype=torch.uint8, device='cuda')
        buf_r[off:off + len(rb)] = torch.frombuffer(bytearray(rb), dtype=torch.uint8).cuda()
        buf_d[off:off + len(db)] = torch.frombuffer(bytearray(db), dtype=torch.uint8).cuda()
        out = torch.empty(shape, dtype=torch.uint8, device='cuda')
        torch.cuda.synchronize()
        assert buf_r.data_ptr() % 256 == 0 and buf_d.data_ptr() % 256 == 0
        gen.submit_device(0, buf_r.data_ptr() + off, buf_d.data_ptr() + off, _DT[dt], h, w, out.data_ptr(), p)
        gen.wait(0)
        return out.cpu().numpy()

    if dt not in _aligned_cache:
        aligned = run(0)
        assert np.array_equal(aligned, O.process_frame(rgb, depth, O.Params(max_disparity=20.0, convergence=-4.0)))
        _aligned_cache[dt] = aligned
    assert np.array_equal(run(offset), _aligned_cache[dt])
