"""Temporal depth stabilisation on the GPU: vsc_stage_temporal_depth is bit-exact against tests/temporal_oracle.py
(output and surviving window), the device's 128-bit to double conversion rounds like Python's float(int), and a window
submission equals a plain submission of the oracle's f32 planes byte for byte, in every output form."""
import ctypes as C
import random

import numpy as np
import pytest

import temporal_oracle as TO
from vsc_b200 import StereoGenerator, StereoParams, _lib
from vsc_b200.stereo_core import temporal_depth
from vsc_b200.synthetic import make_depth, make_rgb

pytestmark = pytest.mark.gpu

P = StereoParams(max_disparity=8.0, convergence=-2.0, super_sampling=2.0, edge_softness=2.0, artifact_smoothing=1.0,
                 depth_gamma=0.5, sharpen=4.0)


def _clip(n, h, w, dtype=np.uint8, seed=0, cut_at=None):
    """n maps of one scene with per-frame noise and restretch; from cut_at on, another scene."""
    rng = np.random.default_rng(seed)
    base = make_depth(h, w, seed, np.float64, discs=6)
    other = make_depth(h, w, seed + 50, np.float64, discs=6)[::-1].copy()
    mx = TO.max_value(dtype)
    out = []
    for t in range(n):
        d = (other if cut_at is not None and t >= cut_at else base) + rng.normal(0, 0.01, (h, w))
        d = (d - d.min()) / max(d.max() - d.min(), 1e-9)
        out.append(np.rint(d * mx).astype(dtype))
    return out


# ---- the filter alone -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16])
@pytest.mark.parametrize('k', [1, 4, 8])
@pytest.mark.parametrize('case', ['middle', 'start', 'end', 'cut'])
def test_stage_parity(dtype, k, case):
    maps = _clip(13, 45, 67, dtype, seed=k, cut_at=8 if case == 'cut' else None)
    t = {'middle': 6, 'start': 1, 'end': 12, 'cut': 6}[case]
    out, lo, hi = temporal_depth(maps, t, k, 6.0)
    ref, rlo, rhi = TO.temporal_depth(maps, t, k, 6.0)
    assert (lo, hi) == (rlo, rhi)
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    if case == 'cut':
        assert hi == min(7, t + k)


@pytest.mark.parametrize('h,w,dtype', [(1079, 1917, np.uint16), (1079, 1917, np.uint8), (1, 1, np.uint8), (1, 1, np.uint16),
                                       (3, 5, np.uint8), (7, 1, np.uint16)])
def test_stage_parity_sizes(h, w, dtype):
    rng = np.random.default_rng(h * w)
    mx = TO.max_value(dtype)
    if h * w > 64:
        maps = _clip(9, h, w, dtype, seed=3)
    else:               # tiny planes: random values (flat ones are cut)
        maps = [rng.integers(0, mx + 1, (h, w)).astype(dtype) for _ in range(9)]
    for t, k, sigma in ((4, 4, 6.0), (0, 8, 0.5), (8, 2, 64.0)):
        out, lo, hi = temporal_depth(maps, t, k, sigma)
        ref, rlo, rhi = TO.temporal_depth(maps, t, k, sigma)
        assert (lo, hi) == (rlo, rhi) and np.array_equal(out.view(np.uint32), ref.view(np.uint32))


def test_stage_radius_zero_and_refusals():
    maps = _clip(3, 16, 16)
    out, lo, hi = temporal_depth(maps, 1, 0)
    assert (lo, hi) == (1, 1) and np.array_equal(out, maps[1].astype(np.float32))
    lib = _lib.load()
    ctx = _lib.Context(0, 1)
    try:
        vp = (C.c_void_p * 3)(*[m.ctypes.data for m in maps])
        o = np.empty((16, 16), np.float32)
        for args in ((3, 1, _lib.DEPTH_F32, 2, 6.0), (3, 1, _lib.DEPTH_U8, 9, 6.0), (3, 1, _lib.DEPTH_U8, 2, 0.0),
                     (3, 1, _lib.DEPTH_U8, 2, 65.0), (3, 3, _lib.DEPTH_U8, 2, 6.0), (0, 0, _lib.DEPTH_U8, 2, 6.0)):
            n, t, dt, k, s = args
            assert lib.vsc_stage_temporal_depth(ctx.handle, vp, n, t, dt, 16, 16, k, s, _lib.ptr(o), None, None) == _lib.VSC_E_INVALID
    finally:
        ctx.close()


def test_i128_to_double_rounds_like_python():
    vals = [0, 1, -1, 2 ** 53 + 1, 2 ** 53 + 3, -(2 ** 53 + 1), 2 ** 63, 2 ** 64 - 1, 2 ** 64, 2 ** 64 + 1, 2 ** 82 - 1,
            -(2 ** 82 - 1), 2 ** 82 + 2 ** 29, 2 ** 82 + 2 ** 29 + 1, 2 ** 82 + 3 * 2 ** 29, 2 ** 117 + 2 ** 64, 2 ** 127 - 1,
            -(2 ** 127), -(2 ** 127) + 1, (2 ** 53 - 1) << 60, ((2 ** 53 - 1) << 60) + (1 << 59), ((2 ** 53) + 1) << 11]
    rng = random.Random(5)
    for bits in range(1, 127):
        for _ in range(6):
            v = rng.getrandbits(bits)
            vals += [v, -v]
    words = np.array([w for v in vals for w in (v & (2 ** 64 - 1), (v >> 64) & (2 ** 64 - 1))], np.uint64)
    out = np.empty(len(vals), np.float64)
    ctx = _lib.Context(0, 1)
    try:
        _lib.check(_lib.load().vsc_debug_i128_to_double(ctx.handle, _lib.ptr(words), len(vals), _lib.ptr(out)))
    finally:
        ctx.close()
    bad = [(v, float(v), o) for v, o in zip(vals, out.tolist()) if float(v) != o]
    assert not bad, bad[:5]


# ---- window submissions ---------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def gen4():
    g = StereoGenerator('cuda:0', n_slots=2, group_size=4)
    yield g
    g.close()


def _plain(gen, frames, depths):
    """Plain submission of (rgb, f32 depth) frames as one group."""
    gen.submit_frames(0, list(zip(frames, depths)), P)
    r = gen.collect(0)
    return r if isinstance(r, list) else [r]


def _window(gen, frames, maps, first, k, sigma=6.0):
    gen.submit_window(0, frames, maps, first, P, radius=k, sigma=sigma)
    r = gen.collect(0)
    return r if isinstance(r, list) else [r]


@pytest.mark.parametrize('n', [1, 2, 3, 4])
@pytest.mark.parametrize('dtype', [np.uint8, np.uint16])
def test_window_equals_plain_submission_of_the_oracle(gen4, n, dtype):
    h, w = 54, 96
    maps = _clip(n + 6, h, w, dtype, seed=n, cut_at=n + 4)
    first = 2
    frames = [make_rgb(h, w, seed=i) for i in range(n)]
    ref = _plain(gen4, frames, TO.filter_group(maps, first, n, 3))
    got = _window(gen4, frames, maps, first, 3)
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))


@pytest.mark.parametrize('layout,pixfmt,encode', [('half-tb', 'rgb24', None), ('sbs', 'yuv420p10le', None),
                                                  ('sbs', 'rgb24', 'png'), ('anaglyph', 'rgb24', None)])
def test_window_in_every_output_form(layout, pixfmt, encode):
    h, w = 54, 96
    maps = _clip(7, h, w, np.uint16, seed=9)
    frames = [make_rgb(h, w, seed=20 + i) for i in range(3)]
    g = StereoGenerator('cuda:0', n_slots=1, group_size=4, layout=layout, pixfmt=pixfmt, encode=encode)
    try:
        ref = _plain(g, frames, TO.filter_group(maps, 0, 3, 4))
        got = _window(g, frames, maps, 0, 4)
        assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    finally:
        g.close()


def test_device_window_equals_host_window(gen4):
    import torch
    h, w = 54, 96
    maps = _clip(8, h, w, np.uint8, seed=4)
    frames = [make_rgb(h, w, seed=i) for i in range(2)]
    ref = _window(gen4, frames, maps, 3, 4)
    d_rgb = [torch.from_numpy(f).cuda() for f in frames]
    d_maps = [torch.from_numpy(m).cuda() for m in maps]
    shape = gen4.output_shape(h, w)
    d_out = [torch.empty(shape, dtype=torch.uint8, device='cuda') for _ in frames]
    torch.cuda.synchronize()
    gen4.submit_device_window(1, [(r.data_ptr(), o.data_ptr()) for r, o in zip(d_rgb, d_out)], [m.data_ptr() for m in d_maps],
                              3, np.uint8, h, w, P, radius=4)
    gen4.wait(1)
    assert all(np.array_equal(o.cpu().numpy(), r) for o, r in zip(d_out, ref))


@pytest.mark.parametrize('dtype', [np.uint8, np.uint16])
def test_radius_zero_window_is_submit_group(gen4, dtype):
    h, w = 54, 96
    maps = _clip(5, h, w, dtype, seed=2)
    frames = [make_rgb(h, w, seed=i) for i in range(3)]
    gen4.submit_frames(0, list(zip(frames, maps[1:4])), P)
    ref = gen4.collect(0)
    got = _window(gen4, frames, maps, 1, 0)
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))


def test_window_refusals(gen4):
    h, w = 32, 32
    lib = _lib.load()
    maps = [np.zeros((h, w), np.float32) + i for i in range(3)]
    rgb = make_rgb(h, w)
    out = np.empty(gen4.output_shape(h, w), np.uint8)
    vp1 = (C.c_void_p * 1)
    dp = (C.c_void_p * 3)(*[m.ctypes.data for m in maps])
    prm = C.byref(_lib.make_params(P))
    call = lambda n_depth, first, dt, k, s: lib.vsc_submit_window(gen4._ctx.handle, 0, 1, vp1(rgb.ctypes.data), n_depth, dp, first, dt,
                                                                 h, w, k, s, prm, vp1(out.ctypes.data))
    assert call(3, 1, _lib.DEPTH_F32, 2, 6.0) == _lib.VSC_E_INVALID          # f32 depth with k > 0
    assert call(3, 3, _lib.DEPTH_U8, 2, 6.0) == _lib.VSC_E_INVALID           # frame beyond the planes
    assert call(3, -1, _lib.DEPTH_U8, 2, 6.0) == _lib.VSC_E_INVALID
    assert call(3, 1, _lib.DEPTH_U8, 9, 6.0) == _lib.VSC_E_INVALID
    assert call(3, 1, _lib.DEPTH_U8, 2, float('nan')) == _lib.VSC_E_INVALID
    assert call(3, 1, _lib.DEPTH_F32, 0, 6.0) == _lib.VSC_OK                 # k = 0 is the plain path, f32 included
    _lib.check(lib.vsc_wait(gen4._ctx.handle, 0))


def test_process_batch_temporal_equals_the_oracle():
    h, w, n, k = 54, 96, 11, 3
    maps = _clip(n, h, w, np.uint8, seed=11, cut_at=6)
    frames = [make_rgb(h, w, seed=i) for i in range(n)]
    ref_depth = [TO.temporal_depth(maps, t, k, 6.0)[0] for t in range(n)]
    g = StereoGenerator('cuda:0', n_slots=3, group_size=4)
    try:
        got = g.process_batch(list(zip(frames, maps)), P, temporal=(k, 6.0))
        ref = g.process_batch(list(zip(frames, ref_depth)), P)
        assert all(np.array_equal(a, b) for a, b in zip(got, ref))
        assert all(np.array_equal(a, b) for a, b in zip(g.process_batch(list(zip(frames, maps)), P, temporal=(0, 6.0)),
                                                         g.process_batch(list(zip(frames, maps)), P)))
    finally:
        g.close()


def test_temporal_kernels_are_profiled(gen4):
    h, w = 54, 96
    maps = _clip(6, h, w, np.uint8)
    gen4.set_profiling(True)
    try:
        _window(gen4, [make_rgb(h, w)] * 2, maps, 2, 2)
        names = [nm for nm, ms in gen4.kernel_times(0)]
    finally:
        gen4.set_profiling(False)
    assert names[:2] == ['temporal_sums_kernel', 'temporal_filter_kernel']


# ---- driver -----------------------------------------------------------------------------------------------------------
def _temporal_workflow(tmp_path, n=21, h=36, w=64, extra=None):
    import json
    import cv2
    wf = tmp_path / 'wf'
    for d in ('frames', 'depth_maps', 'sbs'):
        (wf / d).mkdir(parents=True)
    cfg = {'input_video': 'in.mkv', 'output_video': 'out.mkv',
           'directories': {'frames': 'frames', 'depth_maps': 'depth_maps', 'sbs': 'sbs', 'chunks': 'chunks'},
           'stereo': {'max_disparity': 5.0, 'convergence': 0.0, 'super_sampling': 2.0, 'edge_softness': 1.0,
                      'artifact_smoothing': 1.0, 'depth_gamma': 0.5, 'sharpen': 2.0},
           'free_space': {'sbs_generator': 'none', 'chunk_generator': 'none'}, 'sbs_temporal_radius': 4}
    cfg.update(extra or {})
    (wf / 'config.json').write_text(json.dumps(cfg))
    maps = _clip(n, h, w, np.uint8, seed=7, cut_at=13)
    for i in range(n):
        if i == 9:
            continue                                            # a gap in the clip
        cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(make_rgb(h, w, seed=i), cv2.COLOR_RGB2BGR))
        cv2.imwrite(str(wf / 'depth_maps' / f'depth_frame_{i:06d}.png'), maps[i])
    return wf, maps


def _drive(wf, *args):
    import subprocess
    import sys
    from conftest import ROOT
    r = subprocess.run([sys.executable, f'{ROOT}/video-stereo-converter_b200/sbs_generator.py', str(wf), '--no-interactive',
                        '--slots', '3', *map(str, args)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout, r.stderr)
    return {p.name: p.read_bytes() for p in sorted((wf / 'sbs').glob('sbs_*.png'))}


def _fresh(wf):
    for p in (wf / 'sbs').iterdir():
        p.unlink()


def test_driver_gives_identical_files_however_it_runs(tmp_path):
    import cv2
    import torch
    wf, maps = _temporal_workflow(tmp_path)
    ref = _drive(wf, '--gpus', '1')
    assert len(ref) == 20
    _fresh(wf)
    assert _drive(wf, '--gpus', '1', '--group', '3') == ref
    _fresh(wf)
    assert _drive(wf, '--gpus', '1', '--group', '1', '--temporal-radius', '4') == ref
    if torch.cuda.device_count() >= 2:
        _fresh(wf)
        assert _drive(wf, '--gpus', '2', '--group', '3') == ref
    for name in ('sbs_000004.png', 'sbs_000005.png', 'sbs_000006.png', 'sbs_000014.png', 'sbs_000020.png'):
        (wf / 'sbs' / name).unlink()                            # an interrupted run: resume redoes these only
    assert _drive(wf, '--gpus', '1') == ref
    # process_batch(temporal=...) over each run of consecutive frames gives the same frames
    from vsc_b200 import StereoGenerator, StereoParams
    sp = StereoParams(max_disparity=5.0, convergence=0.0, super_sampling=2.0, edge_softness=1.0, artifact_smoothing=1.0,
                      depth_gamma=0.5, sharpen=2.0)
    g = StereoGenerator('cuda:0', n_slots=2, group_size=4)
    try:
        for run in (range(0, 9), range(10, 21)):
            outs = g.process_batch([(make_rgb(36, 64, seed=i), maps[i]) for i in run], sp, temporal=(4, 6.0))
            for i, o in zip(run, outs):
                png = cv2.cvtColor(cv2.imread(str(wf / 'sbs' / f'sbs_{i:06d}.png')), cv2.COLOR_BGR2RGB)
                assert np.array_equal(png, o), i
    finally:
        g.close()
    # and the filter is on: radius 0 gives other files (the clip's maps are noisy)
    _fresh(wf)
    plain = _drive(wf, '--gpus', '1', '--temporal-radius', '0')
    assert plain.keys() == ref.keys() and plain != ref


def test_driver_free_space_keeps_the_maps_a_resume_needs(tmp_path):
    fs = {'free_space': {'sbs_generator': 'depth', 'chunk_generator': 'none'}}
    ref = _drive(_temporal_workflow(tmp_path / 'ref')[0], '--gpus', '1')
    # a complete run that deletes maps: the same files, and every map goes once every frame is done
    wf, _ = _temporal_workflow(tmp_path / 'full', extra=fs)
    assert _drive(wf, '--gpus', '1') == ref and not list((wf / 'depth_maps').iterdir())
    # an interrupted one: frames 0..7 were published, and with radius 4 only the maps of 0..3 were deleted; the resumed
    # run reads the maps of 4..7 for the windows of frames 8..11 and writes the same files
    wf, _ = _temporal_workflow(tmp_path / 'resumed', extra=fs)
    for i in range(8):
        (wf / 'sbs' / f'sbs_{i:06d}.png').write_bytes(ref[f'sbs_{i:06d}.png'])
    for i in range(4):
        (wf / 'depth_maps' / f'depth_frame_{i:06d}.png').unlink()
    assert _drive(wf, '--gpus', '1') == ref
    assert sorted(p.name for p in (wf / 'depth_maps').iterdir()) == [f'depth_frame_{i:06d}.png' for i in range(4, 8)]
