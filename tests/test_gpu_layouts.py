"""Output layouts on the GPU: every layout of every path equals layout_oracle.pack_layout of the SBS frame, bit for bit.
The generators and contexts here are this file's own, so that no layout leaks into the shared session context."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import layout_oracle as LO
import oracle as O
from conftest import ROOT
from vsc_b200 import StereoGenerator, StereoParams, _lib
from vsc_b200.stereo_core import LAYOUTS, layout_code, output_shape
from vsc_b200.synthetic import make_pair

pytestmark = pytest.mark.gpu

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')

# the shapes, depth dtypes and parameters of test_gpu_e2e.py::CASES
CASES = [
    ((120, 160), np.uint8, {}),
    ((135, 240), np.uint16, {}),
    ((100, 180), np.uint8, dict(super_sampling=1.0, edge_softness=0.0, depth_gamma=1.0, max_disparity=30.0, convergence=5.0,
                                artifact_smoothing=5.0)),
    ((90, 150), np.uint16, dict(super_sampling=2.5, edge_softness=3.0, depth_gamma=0.5, max_disparity=20.0, convergence=-7.0,
                                artifact_smoothing=0.0, sharpen=0.0)),
    ((96, 200), np.float32, dict(super_sampling=2.0, edge_softness=0.0, depth_gamma=1.0, max_disparity=100.0, convergence=-50.0,
                                 artifact_smoothing=5.0)),
    ((64, 256), np.uint8, dict(super_sampling=4.0, edge_softness=30.0, depth_gamma=2.0, max_disparity=100.0, convergence=50.0,
                               artifact_smoothing=2.5, sharpen=16.0)),
    ((80, 120), np.uint16, dict(super_sampling=1.3, edge_softness=0.5, depth_gamma=0.1, max_disparity=5.0, convergence=0.0,
                                artifact_smoothing=0.1, sharpen=0.5)),
]


def _takes(layout, h, w):
    try:
        output_shape(layout, h, w)
        return True
    except ValueError:
        return False


@pytest.fixture(scope='module')
def gens():
    g = {name: StereoGenerator('cuda', n_slots=2, layout=name) for name in LAYOUTS}
    yield g
    for x in g.values():
        x.close()


_oracle_cache = {}


def _oracle_sbs(i):
    if i not in _oracle_cache:
        shape, dt, kw = CASES[i]
        rgb, depth = make_pair(shape[0], shape[1], seed=7, depth_dtype=dt)
        _oracle_cache[i] = (rgb, depth, O.process_frame(rgb, depth, O.Params(**kw)))
    return _oracle_cache[i]


@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('case', range(len(CASES)))
def test_process_frame_matches_packed_oracle(gens, layout, case):
    shape, dt, kw = CASES[case]
    rgb, depth, sbs = _oracle_sbs(case)
    gen = gens[layout]
    if not _takes(layout, *shape):
        with pytest.raises(ValueError, match='odd'):
            gen.process_frame(rgb, depth, StereoParams(**kw))
        # the library refuses it too, without the Python-side shape check in front
        import torch
        d_rgb = torch.from_numpy(rgb).cuda()
        d_depth = torch.from_numpy(np.ascontiguousarray(depth)).cuda()
        d_out = torch.empty(shape[0] * shape[1] * 6, dtype=torch.uint8, device='cuda')
        with pytest.raises(_lib.VscError) as e:
            gen.submit_device(0, d_rgb.data_ptr(), d_depth.data_ptr(), depth.dtype, shape[0], shape[1], d_out.data_ptr(),
                              StereoParams(**kw))
        assert e.value.code == _lib.VSC_E_INVALID
        return
    out = gen.process_frame(rgb, depth, StereoParams(**kw))
    want = LO.pack_layout(sbs, layout)
    assert out.shape == want.shape == output_shape(layout, *shape) and out.dtype == np.uint8
    assert np.array_equal(out, want), f'{int((out != want).sum())} values differ'


@pytest.mark.parametrize('h,w,dt', [(1080, 1920, np.uint8), (2160, 3840, np.uint16)])
def test_full_frames_per_layout(gens, h, w, dt):
    rgb, depth = make_pair(h, w, seed=0, depth_dtype=dt)
    sbs = gens['sbs'].process_frame(rgb, depth)
    launches = gens['sbs'].last_frame_launches(0)
    for layout in LAYOUTS[1:]:
        out = gens[layout].process_frame(rgb, depth)
        assert np.array_equal(out, LO.pack_layout(sbs, layout)), layout
        assert gens[layout].last_frame_launches(0) == launches, layout      # the layout is an epilogue, not a launch


def test_launch_count_does_not_depend_on_layout(gens):
    rgb, depth = make_pair(90, 160, seed=3)
    counts = {}
    for layout in LAYOUTS:
        gens[layout].process_frame(rgb, depth)
        counts[layout] = gens[layout].last_frame_launches(0)
    assert len(set(counts.values())) == 1 and counts['sbs'] > 0, counts


def _frames(n, h=90, w=160):
    return [make_pair(h, w, seed=50 + s, depth_dtype=np.uint16) for s in range(n)]


@pytest.fixture(scope='module')
def sbs_refs(gens):
    frames = _frames(4)
    return frames, [gens['sbs'].process_frame(r, d) for r, d in frames]


@pytest.mark.parametrize('layout', LAYOUTS)
def test_submit_host_group_of_four(sbs_refs, layout):
    frames, refs = sbs_refs
    g = StereoGenerator('cuda', n_slots=2, group_size=4, layout=layout)
    try:
        g.submit_host(1, frames)
        outs = g.collect(1)
        assert len(outs) == 4
        for o, r in zip(outs, refs):
            assert np.array_equal(o, LO.pack_layout(r, layout))
        batch = g.process_batch(frames + frames[:3])
        assert all(np.array_equal(o, LO.pack_layout(r, layout)) for o, r in zip(batch, refs + refs[:3]))
    finally:
        g.close()


@pytest.mark.parametrize('layout', LAYOUTS)
def test_submit_device_group_into_torch(sbs_refs, layout):
    import torch
    frames, refs = sbs_refs
    h, w = frames[0][0].shape[:2]
    g = StereoGenerator('cuda', n_slots=1, group_size=4, layout=layout)
    try:
        d_in = [(torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda()) for r, d in frames]
        d_out = [torch.full(output_shape(layout, h, w), 7, dtype=torch.uint8, device='cuda') for _ in frames]
        torch.cuda.synchronize()
        g.submit_device_group(0, [(a.data_ptr(), b.data_ptr(), o.data_ptr()) for (a, b), o in zip(d_in, d_out)], np.uint16, h, w)
        g.wait(0)
        for o, r in zip(d_out, refs):
            assert np.array_equal(o.cpu().numpy(), LO.pack_layout(r, layout))
    finally:
        g.close()


def test_slots_in_flight_keep_their_own_layout(sbs_refs):
    """vsc_set_layout between two submissions: each slot comes back in the layout it was submitted with."""
    frames, refs = sbs_refs
    (r0, d0), (r1, d1) = frames[0], frames[1]
    h, w = r0.shape[:2]
    lib = _lib.load()
    ctx = _lib.Context(0, 3)
    try:
        p = _lib.make_params(StereoParams())
        plan = [('half-sbs', r0, d0, refs[0]), ('tb', r1, d1, refs[1]), ('anaglyph', r0, d0, refs[0])]
        outs = []
        for slot, (layout, r, d, _) in enumerate(plan):
            _lib.check(lib.vsc_set_layout(ctx.handle, layout_code(layout)))
            out = np.full(output_shape(layout, h, w), 7, np.uint8)
            outs.append(out)
            _lib.check(lib.vsc_submit(ctx.handle, slot, _lib.ptr(r), _lib.ptr(d), _lib.DEPTH_U16, h, w, C.byref(p), _lib.ptr(out)))
        for slot in (2, 0, 1):
            _lib.check(lib.vsc_wait(ctx.handle, slot))
        for out, (layout, _, _, ref) in zip(outs, plan):
            assert np.array_equal(out, LO.pack_layout(ref, layout)), layout
        assert len({lib.vsc_slot_launches(ctx.handle, s) for s in range(3)}) == 1
        # a frame size the current layout cannot take is refused at submission
        _lib.check(lib.vsc_set_layout(ctx.handle, layout_code('half-tb')))
        odd_r, odd_d = make_pair(91, 160, seed=1)
        big = np.empty((91, 320, 3), np.uint8)
        assert lib.vsc_submit(ctx.handle, 0, _lib.ptr(odd_r), _lib.ptr(odd_d), _lib.DEPTH_U8, 91, 160, C.byref(p), _lib.ptr(big)) \
            == _lib.VSC_E_INVALID
        assert lib.vsc_set_layout(ctx.handle, 5) == _lib.VSC_E_INVALID
    finally:
        ctx.close()


def test_default_context_equals_explicit_sbs():
    rgb, depth = make_pair(100, 180, seed=9, depth_dtype=np.uint16)
    h, w = rgb.shape[:2]
    lib = _lib.load()
    ctx = _lib.Context(0, 1)
    try:
        plain = np.empty((h, 2 * w, 3), np.uint8)
        p = _lib.make_params(StereoParams())
        _lib.check(lib.vsc_process_frame(ctx.handle, _lib.ptr(rgb), _lib.ptr(depth), _lib.DEPTH_U16, h, w, C.byref(p), _lib.ptr(plain)))
    finally:
        ctx.close()
    g = StereoGenerator('cuda', layout='sbs')
    try:
        assert np.array_equal(plain, g.process_frame(rgb, depth))
        assert np.array_equal(plain, O.process_frame(rgb, depth, O.Params()))
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


def test_sbs_generator_half_sbs_pngs_and_raw_sink(tmp_path):
    import cv2
    n = 3
    wf = _workflow(tmp_path, n)
    want = [LO.pack_layout(s, 'half-sbs') for s in _expected(wf, n)]
    run = lambda *a: subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive',  # noqa: E731
                                     '--gpus', '1', '--slots', '2', '--group', '2', '--layout', 'half-sbs', *a],
                                    capture_output=True, text=True, timeout=600)
    r = run()
    assert r.returncode == 0, r.stdout + r.stderr
    for i in range(n):
        got = cv2.cvtColor(cv2.imread(str(wf / 'sbs' / f'sbs_{i:06d}.png'), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
        assert np.array_equal(got, want[i]), i
    raw = tmp_path / 'clip.rgb'
    r = run('--raw-sink', str(raw))
    assert r.returncode == 0, r.stdout + r.stderr
    meta = json.loads((tmp_path / 'clip.rgb.json').read_text())
    assert (meta['height'], meta['width']) == (72, 128)
    frames = np.fromfile(raw, np.uint8).reshape(n, 72, 128, 3)
    for i in range(n):
        assert np.array_equal(frames[i], want[i]), i
    # resuming the PNG outputs in another layout is refused
    (wf / 'sbs' / 'sbs_000002.png').unlink()
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive'], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 2 and 'ERROR:' in r.stdout


def test_sweep_writes_its_layout(tmp_path):
    wf = _workflow(tmp_path, 1)
    out = tmp_path / 'sweep'
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_sweep.py'), str(wf), '--layout', 'anaglyph', '--out', str(out),
                        '--param', 'max_disparity=20,40'], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    meta = json.loads((out / 'sweep.json').read_text())
    assert meta['layout'] == 'anaglyph' and all(x['refused'] is None for x in meta['results'])
    import cv2
    assert cv2.imread(str(out / 'sweep_0000.png')).shape == (72, 128, 3)
