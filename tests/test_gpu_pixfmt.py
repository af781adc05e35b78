"""Output pixel formats on the GPU: every YUV frame of every path equals
pixfmt_oracle.pack_pixfmt(layout_oracle.pack_layout(SBS frame)), bit for bit.  The generators and contexts here are this
file's own, so that no format leaks into the shared session context."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import layout_oracle as LO
import oracle as O
import pixfmt_oracle as PO
from conftest import ROOT
from vsc_b200 import StereoGenerator, StereoParams, _lib
from vsc_b200.stereo_core import LAYOUTS, MATRICES, layout_code, matrix_code, output_dtype, output_shape, pixfmt_code
from vsc_b200.synthetic import make_pair

pytestmark = pytest.mark.gpu

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')
YUV = ('yuv420p', 'yuv420p10le')

# every back-end instantiation: K = 3 (default), 2, 4 and the generic K = 0 (2.5 and 1.0); partial edge tiles
CASES = [
    ((120, 160), np.uint8, {}),
    ((92, 172), np.uint16, {}),                                          # partial tiles the half layouts take
    ((90, 166), np.uint16, dict(super_sampling=2.5, edge_softness=3.0, depth_gamma=0.5, max_disparity=20.0, convergence=-7.0,
                                artifact_smoothing=0.0, sharpen=0.0)),   # partial tiles; half-sbs / half-tb refuse it
    ((96, 200), np.float32, dict(super_sampling=2.0, edge_softness=0.0, depth_gamma=1.0, max_disparity=100.0, convergence=-50.0,
                                 artifact_smoothing=5.0)),
    ((64, 256), np.uint8, dict(super_sampling=4.0, edge_softness=30.0, depth_gamma=2.0, max_disparity=100.0, convergence=50.0,
                               artifact_smoothing=2.5, sharpen=16.0)),
    ((100, 180), np.uint8, dict(super_sampling=1.0, edge_softness=0.0, depth_gamma=1.0, max_disparity=30.0, convergence=5.0,
                                artifact_smoothing=5.0)),
]


def _takes(layout, h, w, pixfmt):
    try:
        output_shape(layout, h, w, pixfmt)
        return True
    except ValueError:
        return False


def _want(sbs, layout, pixfmt, matrix='bt709'):
    return PO.pack_pixfmt(LO.pack_layout(sbs, layout), pixfmt, matrix)


@pytest.fixture(scope='module')
def gen():
    g = StereoGenerator('cuda', n_slots=2)
    yield g
    g.close()


def _use(g, layout, pixfmt, matrix='bt709'):
    g.set_layout(layout)
    g.set_pixfmt(pixfmt, matrix)
    return g


_oracle_cache = {}


def _oracle_sbs(i):
    if i not in _oracle_cache:
        shape, dt, kw = CASES[i]
        rgb, depth = make_pair(shape[0], shape[1], seed=7, depth_dtype=dt)
        _oracle_cache[i] = (rgb, depth, O.process_frame(rgb, depth, O.Params(**kw)))
    return _oracle_cache[i]


@pytest.mark.parametrize('matrix', MATRICES)
@pytest.mark.parametrize('pixfmt', YUV)
@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('case', range(len(CASES)))
def test_process_frame_matches_packed_oracle(gen, case, layout, pixfmt, matrix):
    shape, dt, kw = CASES[case]
    rgb, depth, sbs = _oracle_sbs(case)
    g = _use(gen, layout, pixfmt, matrix)
    if not _takes(layout, *shape, pixfmt):
        with pytest.raises(ValueError, match='divisible by 4'):
            g.process_frame(rgb, depth, StereoParams(**kw))
        # the library refuses it too, without the Python-side shape check in front
        import torch
        d_rgb = torch.from_numpy(rgb).cuda()
        d_depth = torch.from_numpy(np.ascontiguousarray(depth)).cuda()
        d_out = torch.empty(shape[0] * shape[1] * 6, dtype=torch.uint8, device='cuda')
        with pytest.raises(_lib.VscError) as e:
            g.submit_device(0, d_rgb.data_ptr(), d_depth.data_ptr(), depth.dtype, shape[0], shape[1], d_out.data_ptr(),
                            StereoParams(**kw))
        assert e.value.code == _lib.VSC_E_INVALID
        return
    out = g.process_frame(rgb, depth, StereoParams(**kw))
    want = _want(sbs, layout, pixfmt, matrix)
    assert out.shape == want.shape == output_shape(layout, *shape, pixfmt) and out.dtype == want.dtype == output_dtype(pixfmt)
    assert np.array_equal(out, want), f'{int((out != want).sum())} values differ'


@pytest.mark.parametrize('h,w,dt', [(1080, 1920, np.uint8), (2160, 3840, np.uint16)])
def test_full_frames_per_layout_and_format(gen, h, w, dt):
    rgb, depth = make_pair(h, w, seed=0, depth_dtype=dt)
    sbs = _use(gen, 'sbs', 'rgb24').process_frame(rgb, depth)
    launches = gen.last_frame_launches(0)
    for layout in LAYOUTS:
        for pixfmt in YUV:
            for matrix in (MATRICES if layout == 'sbs' else ('bt709',)):
                out = _use(gen, layout, pixfmt, matrix).process_frame(rgb, depth)
                assert np.array_equal(out, _want(sbs, layout, pixfmt, matrix)), (layout, pixfmt, matrix)
                assert gen.last_frame_launches(0) == launches, (layout, pixfmt)  # the format is an epilogue, not a launch


def test_launch_count_does_not_depend_on_format(gen):
    rgb, depth = make_pair(90, 160, seed=3)
    counts = {}
    for pixfmt in ('rgb24',) + YUV:
        _use(gen, 'sbs', pixfmt).process_frame(rgb, depth)
        counts[pixfmt] = gen.last_frame_launches(0)
    assert len(set(counts.values())) == 1 and counts['rgb24'] > 0, counts


def _frames(n, h=92, w=160):
    return [make_pair(h, w, seed=50 + s, depth_dtype=np.uint16) for s in range(n)]


@pytest.fixture(scope='module')
def sbs_refs(gen):
    frames = _frames(4)
    g = _use(gen, 'sbs', 'rgb24')
    return frames, [g.process_frame(r, d) for r, d in frames]


@pytest.mark.parametrize('pixfmt', YUV)
@pytest.mark.parametrize('layout', ['sbs', 'half-tb', 'anaglyph'])
def test_submit_host_group_of_four(sbs_refs, layout, pixfmt):
    frames, refs = sbs_refs
    g = StereoGenerator('cuda', n_slots=2, group_size=4, layout=layout, pixfmt=pixfmt, matrix='bt601')
    try:
        g.submit_host(1, frames)
        outs = g.collect(1)
        assert len(outs) == 4
        for o, r in zip(outs, refs):
            assert o.dtype == output_dtype(pixfmt) and np.array_equal(o, _want(r, layout, pixfmt, 'bt601'))
        batch = g.process_batch(frames + frames[:3])
        assert all(np.array_equal(o, _want(r, layout, pixfmt, 'bt601')) for o, r in zip(batch, refs + refs[:3]))
        g.submit_host(0, frames[:1])
        with pytest.raises(RuntimeError, match='collect'):
            g.set_pixfmt('rgb24')
        g.collect(0)
        g.set_pixfmt('rgb24')                                          # back to the reference's frames
        assert np.array_equal(g.process_frame(*frames[0]), LO.pack_layout(refs[0], layout))
    finally:
        g.close()


@pytest.mark.parametrize('pixfmt', YUV)
@pytest.mark.parametrize('layout', ['tb', 'half-sbs'])
def test_submit_device_group_into_torch(sbs_refs, layout, pixfmt):
    import torch
    frames, refs = sbs_refs
    h, w = frames[0][0].shape[:2]
    g = StereoGenerator('cuda', n_slots=1, group_size=4, layout=layout, pixfmt=pixfmt)
    try:
        tdt = torch.int16 if g.output_dtype == np.uint16 else torch.uint8          # the same bytes as uint16
        d_in = [(torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda()) for r, d in frames]
        d_out = [torch.full(g.output_shape(h, w), 7, dtype=tdt, device='cuda') for _ in frames]
        torch.cuda.synchronize()
        g.submit_device_group(0, [(a.data_ptr(), b.data_ptr(), o.data_ptr()) for (a, b), o in zip(d_in, d_out)], np.uint16, h, w)
        g.wait(0)
        for o, r in zip(d_out, refs):
            assert np.array_equal(o.cpu().numpy().view(g.output_dtype), _want(r, layout, pixfmt))
    finally:
        g.close()


def test_slots_in_flight_keep_their_own_format(sbs_refs):
    """vsc_set_pixfmt (and vsc_set_layout) between submissions: each slot comes back in the format it was submitted with."""
    frames, refs = sbs_refs
    (r0, d0), (r1, d1) = frames[0], frames[1]
    h, w = r0.shape[:2]
    lib = _lib.load()
    ctx = _lib.Context(0, 4)
    try:
        p = _lib.make_params(StereoParams())
        plan = [('sbs', 'yuv420p10le', 'bt709', r0, d0, refs[0]), ('half-sbs', 'yuv420p', 'bt601', r1, d1, refs[1]),
                ('sbs', 'rgb24', 'bt709', r0, d0, refs[0]), ('anaglyph', 'yuv420p10le', 'bt601', r1, d1, refs[1])]
        outs = []
        for slot, (layout, pixfmt, matrix, r, d, _) in enumerate(plan):
            _lib.check(lib.vsc_set_layout(ctx.handle, layout_code(layout)))
            _lib.check(lib.vsc_set_pixfmt(ctx.handle, pixfmt_code(pixfmt), matrix_code(matrix)))
            out = np.full(output_shape(layout, h, w, pixfmt), 7, output_dtype(pixfmt))
            n = C.c_size_t()
            _lib.check(lib.vsc_output_size(layout_code(layout), pixfmt_code(pixfmt), h, w, C.byref(n)))
            assert n.value == out.nbytes
            outs.append(out)
            _lib.check(lib.vsc_submit(ctx.handle, slot, _lib.ptr(r), _lib.ptr(d), _lib.DEPTH_U16, h, w, C.byref(p), _lib.ptr(out)))
        for slot in (3, 1, 0, 2):
            _lib.check(lib.vsc_wait(ctx.handle, slot))
        for out, (layout, pixfmt, matrix, _, _, ref) in zip(outs, plan):
            assert np.array_equal(out, _want(ref, layout, pixfmt, matrix)), (layout, pixfmt, matrix)
        assert len({lib.vsc_slot_launches(ctx.handle, s) for s in range(4)}) == 1
        # a frame size the current format cannot take is refused at submission
        _lib.check(lib.vsc_set_layout(ctx.handle, layout_code('sbs')))
        _lib.check(lib.vsc_set_pixfmt(ctx.handle, pixfmt_code('yuv420p'), 0))
        odd_r, odd_d = make_pair(91, 160, seed=1)
        big = np.empty((91, 320, 3), np.uint8)
        assert lib.vsc_submit(ctx.handle, 0, _lib.ptr(odd_r), _lib.ptr(odd_d), _lib.DEPTH_U8, 91, 160, C.byref(p), _lib.ptr(big)) \
            == _lib.VSC_E_INVALID
        assert lib.vsc_set_pixfmt(ctx.handle, 3, 0) == _lib.VSC_E_INVALID
        assert lib.vsc_set_pixfmt(ctx.handle, 1, 2) == _lib.VSC_E_INVALID
    finally:
        ctx.close()


def test_default_generator_is_rgb24():
    rgb, depth = make_pair(100, 180, seed=9, depth_dtype=np.uint16)
    g = StereoGenerator('cuda')
    try:
        assert (g.pixfmt, g.matrix, g.output_dtype) == ('rgb24', 'bt709', np.uint8)
        out = g.process_frame(rgb, depth)
        assert np.array_equal(out, O.process_frame(rgb, depth, O.Params()))
    finally:
        g.close()


# ---- drivers ------------------------------------------------------------------------------------
def _workflow(root, n=3, h=72, w=128):
    import cv2
    wf = root / 'wf'
    for d in ('frames', 'depth_maps', 'sbs'):
        (wf / d).mkdir(parents=True)
    cfg = {'input_video': 'in.mkv', 'output_video': 'out.mkv',
           'directories': {'frames': 'frames', 'depth_maps': 'depth_maps', 'sbs': 'sbs', 'chunks': 'chunks'},
           'stereo': {'max_disparity': 50.0, 'convergence': -10.0, 'super_sampling': 3.0, 'edge_softness': 20.0,
                      'artifact_smoothing': 1.0, 'depth_gamma': 0.2, 'sharpen': 14.0},
           'free_space': {'sbs_generator': 'none', 'chunk_generator': 'none'}}
    (wf / 'config.json').write_text(json.dumps(cfg))
    for i in range(n):
        rgb, depth = make_pair(h, w, seed=i, depth_dtype=np.uint16)
        cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(rgb, cv2.COLOR_RGB2BGR))
        cv2.imwrite(str(wf / 'depth_maps' / f'depth_frame_{i:06d}.tif'), depth)
    return wf


def _expected(wf, n):
    from vsc_b200 import load_image_pair
    g = StereoGenerator('cuda')
    try:
        return [g.process_frame(*load_image_pair(wf / 'frames' / f'frame_{i:06d}.png', wf / 'depth_maps' / f'depth_frame_{i:06d}.tif'))
                for i in range(n)]
    finally:
        g.close()


def test_sbs_generator_raw_sink_yuv420p10le(tmp_path):
    n = 3
    wf = _workflow(tmp_path, n)
    want = [PO.pack_pixfmt(s, 'yuv420p10le', 'bt709') for s in _expected(wf, n)]
    raw = tmp_path / 'clip.yuv'
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive', '--gpus', '1',
                        '--slots', '2', '--group', '2', '--raw-sink', str(raw), '--pixfmt', 'yuv420p10le'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    meta = json.loads((tmp_path / 'clip.yuv.json').read_text())
    assert (meta['pix_fmt'], meta['matrix'], meta['height'], meta['width']) == ('yuv420p10le', 'bt709', 72, 256)
    assert meta['bytes_per_frame'] == 72 * 256 * 3 and os.path.getsize(raw) == n * meta['bytes_per_frame']
    frames = np.fromfile(raw, '<u2').reshape(n, 72 * 3 // 2, 256)
    for i in range(n):
        assert np.array_equal(frames[i], want[i]), i
    assert not list((wf / 'sbs').glob('sbs_*.png'))
