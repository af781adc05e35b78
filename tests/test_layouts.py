"""Output layouts without a GPU: the NumPy restatement (layout_oracle.pack_layout) against OpenCV and float64, the library's
host-only shape rules (vsc_layout_shape), and the drivers' layout choice, resume check and raw-sink geometry."""
import ctypes as C
import json
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest

import layout_oracle as LO
from conftest import ROOT
from vsc_b200 import _lib
from vsc_b200.stereo_core import LAYOUTS, output_shape
from vsc_b200.synthetic import make_pair
from vsc_b200.workflow import ConfigError, LayoutError, config_layout, load_config

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')
sys.path.insert(0, PKG)
import sbs_generator  # noqa: E402


def _sbs(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, 2 * w, 3), dtype=np.uint8)


# ---- pack_layout --------------------------------------------------------------------------------
@pytest.mark.parametrize('ipp', [True, False])
@pytest.mark.parametrize('h,w', [(8, 8), (30, 46), (136, 240), (1080, 1920)])
def test_half_layouts_equal_cv2_inter_area(ipp, h, w):
    sbs = _sbs(h, w, seed=h + w)
    left, right = sbs[:, :w], sbs[:, w:]
    was = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(ipp)
    try:
        hs = [cv2.resize(e, (w // 2, h), interpolation=cv2.INTER_AREA) for e in (left, right)]
        tb = [cv2.resize(e, (w, h // 2), interpolation=cv2.INTER_AREA) for e in (left, right)]
    finally:
        cv2.ipp.setUseIPP(was)
    assert np.array_equal(LO.pack_layout(sbs, 'half-sbs'), np.hstack(hs))
    assert np.array_equal(LO.pack_layout(sbs, 'half-tb'), np.vstack(tb))


def test_rounding_is_half_to_even_not_half_up():
    """Plain (s + 1) >> 1 differs from INTER_AREA on about a quarter of the pairs."""
    a = np.arange(256, dtype=np.uint8).repeat(256)
    b = np.tile(np.arange(256, dtype=np.uint8), 256)
    sbs = np.stack([a, b], 1).reshape(1, -1, 1).repeat(3, 2)          # [1, 2 * 65536, 3]: left | right halves
    s = a.astype(int) + b.astype(int)
    got = LO._avg2_rhe(a, b).astype(int)
    assert np.array_equal(got, np.round(s / 2).astype(int))            # numpy rounds half to even
    assert ((s + 1) >> 1 != got).mean() > 0.2
    assert LO.pack_layout(sbs, 'half-sbs').shape == (1, 65536, 3)


def test_full_layouts_are_rearrangements():
    sbs = _sbs(9, 13, seed=3)
    left, right = sbs[:, :13], sbs[:, 13:]
    assert np.array_equal(LO.pack_layout(sbs, 'sbs'), sbs)
    tb = LO.pack_layout(sbs, 'tb')
    assert tb.shape == (18, 13, 3) and np.array_equal(tb[:9], left) and np.array_equal(tb[9:], right)
    with pytest.raises(ValueError):
        LO.pack_layout(sbs, 'half-sbs')                                 # odd width
    with pytest.raises(ValueError):
        LO.pack_layout(sbs, 'half-tb')                                  # odd height
    with pytest.raises(ValueError):
        LO.pack_layout(sbs, 'side-by-side')


@pytest.mark.parametrize('l,r,want', [
    ((255, 255, 255), (255, 255, 255), (255, 255, 255)),
    ((128, 128, 128), (128, 128, 128), (128, 128, 128)),
    ((255, 0, 0), (0, 0, 0), (111, 0, 0)),
    ((0, 0, 0), (0, 255, 255), (0, 196, 255)),
    ((200, 30, 60), (10, 220, 90), (103, 156, 78)),
])
def test_anaglyph_known_answers(l, r, want):
    sbs = np.array([[l, r]], np.uint8)
    assert tuple(int(v) for v in LO.pack_layout(sbs, 'anaglyph')[0, 0]) == want


def test_anaglyph_random_pixels_within_one_of_float64():
    h, w = 64, 512
    sbs = _sbs(h, w, seed=11)
    got = LO.pack_layout(sbs, 'anaglyph').astype(int)
    ml = np.array([[0.437, 0.449, 0.164], [-0.062, -0.062, -0.024], [-0.048, -0.050, -0.017]])
    mr = np.array([[-0.011, -0.032, -0.007], [0.377, 0.761, 0.009], [-0.026, -0.093, 1.234]])
    l, r = sbs[:, :w].astype(np.float64), sbs[:, w:].astype(np.float64)
    ref = np.clip(l @ ml.T + r @ mr.T, 0, 255)
    assert np.abs(got - ref).max() <= 1.0
    assert got.shape == (h, w, 3)


# ---- vsc_layout_shape (host only) ----------------------------------------------------------------
def _shape(layout, h, w):
    oh, ow = C.c_int(-1), C.c_int(-1)
    rc = _lib.load().vsc_layout_shape(layout, h, w, C.byref(oh), C.byref(ow))
    return rc, (oh.value, ow.value)


def test_layout_shape_known_answers():
    assert [_shape(k, 1080, 1920) for k in range(5)] == [
        (0, (1080, 3840)), (0, (1080, 1920)), (0, (2160, 1920)), (0, (1080, 1920)), (0, (1080, 1920))]
    assert (_lib.LAYOUT_SBS, _lib.LAYOUT_HALF_SBS, _lib.LAYOUT_TB, _lib.LAYOUT_HALF_TB, _lib.LAYOUT_ANAGLYPH) == (0, 1, 2, 3, 4)
    for name in LAYOUTS:
        assert output_shape(name, 10, 12) == LO.pack_layout(_sbs(10, 12, 0), name).shape


def test_layout_shape_refusals():
    lib = _lib.load()
    assert _shape(_lib.LAYOUT_HALF_SBS, 100, 201)[0] == _lib.VSC_E_INVALID and b'odd' in lib.vsc_last_error()
    assert _shape(_lib.LAYOUT_HALF_TB, 101, 200)[0] == _lib.VSC_E_INVALID and b'odd' in lib.vsc_last_error()
    assert _shape(_lib.LAYOUT_HALF_SBS, 101, 200)[0] == 0 and _shape(_lib.LAYOUT_HALF_TB, 100, 201)[0] == 0
    for k in (0, 2, 4):
        assert _shape(k, 101, 201)[0] == 0                             # the full-size layouts take any size
    for bad in (-1, 5, 99):
        assert _shape(bad, 100, 200)[0] == _lib.VSC_E_INVALID and b'unknown' in lib.vsc_last_error()
    assert lib.vsc_layout_shape(0, 10, 10, None, None) == _lib.VSC_E_INVALID
    assert lib.vsc_set_layout(None, 0) == _lib.VSC_E_INVALID
    with pytest.raises(ValueError, match='odd'):
        output_shape('half-sbs', 10, 11)
    with pytest.raises(ValueError, match='unknown'):
        output_shape('HSBS', 10, 10)


def test_generator_refuses_unknown_layout_before_touching_a_device():
    from vsc_b200 import StereoGenerator
    with pytest.raises(ValueError, match='unknown output layout'):
        StereoGenerator('cuda', layout='side-by-side')


# ---- drivers ------------------------------------------------------------------------------------
def _workflow(tmp_path, n=2, h=32, w=48, layout=None):
    wf = tmp_path / 'wf'
    for d in ('frames', 'depth_maps', 'sbs'):
        (wf / d).mkdir(parents=True)
    cfg = {'input_video': 'in.mkv', 'output_video': 'out.mkv',
           'directories': {'frames': 'frames', 'depth_maps': 'depth_maps', 'sbs': 'sbs', 'chunks': 'chunks'},
           'stereo': {'max_disparity': 5.0, 'convergence': 0.0, 'super_sampling': 1.0, 'edge_softness': 0.0,
                      'artifact_smoothing': 0.0, 'depth_gamma': 1.0, 'sharpen': 0.0},
           'free_space': {'sbs_generator': 'none', 'chunk_generator': 'none'}}
    if layout is not None:
        cfg['sbs_layout'] = layout
    (wf / 'config.json').write_text(json.dumps(cfg))
    for i in range(n):
        rgb, depth = make_pair(h, w, seed=i)
        cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(rgb, cv2.COLOR_RGB2BGR))
        cv2.imwrite(str(wf / 'depth_maps' / f'depth_frame_{i:06d}.png'), depth)
    return wf


def _run(script, *args):
    return subprocess.run([sys.executable, os.path.join(PKG, script), *map(str, args)], capture_output=True, text=True,
                          timeout=300)


def test_config_layout_key(tmp_path):
    wf = _workflow(tmp_path, n=0)
    assert config_layout(load_config(wf)) == 'sbs'
    for name in LAYOUTS:
        wf2 = _workflow(tmp_path / name, n=0, layout=name)
        assert config_layout(load_config(wf2)) == name
    for i, bad in enumerate(('HSBS', 3, '', ['sbs'])):
        wf3 = _workflow(tmp_path / f'bad{i}', n=0, layout=bad)
        with pytest.raises(LayoutError):
            load_config(wf3)
        assert issubclass(LayoutError, ConfigError)


def test_cli_layout_flag_parsing():
    p = sbs_generator.build_parser()
    assert p.parse_args(['wf']).layout is None
    for name in LAYOUTS:
        assert p.parse_args(['wf', '--layout', name]).layout == name


def test_cli_refuses_bad_layouts_with_exit_2(tmp_path):
    wf = _workflow(tmp_path)
    r = _run('sbs_generator.py', wf, '--layout', 'hsbs')
    assert r.returncode == 2 and 'invalid choice' in r.stderr
    cfg = json.loads((wf / 'config.json').read_text())
    cfg['sbs_layout'] = 'over-under'
    (wf / 'config.json').write_text(json.dumps(cfg))
    r = _run('sbs_generator.py', wf, '--no-interactive')
    assert r.returncode == 2 and r.stdout.startswith('ERROR:') and 'sbs_layout' in r.stdout
    r = _run('sbs_sweep.py', wf)
    assert r.returncode == 2 and 'sbs_layout' in r.stdout


def test_cli_refuses_an_odd_side_for_a_half_layout(tmp_path):
    wf = _workflow(tmp_path, h=32, w=47)
    r = _run('sbs_generator.py', wf, '--no-interactive', '--layout', 'half-sbs')
    assert r.returncode == 2 and 'ERROR:' in r.stdout and 'odd' in r.stdout


def test_png_size_reads_the_ihdr(tmp_path):
    f = tmp_path / 'x.png'
    cv2.imwrite(str(f), np.zeros((17, 29, 3), np.uint8))
    assert sbs_generator.png_size(f) == (17, 29)
    (tmp_path / 'y.png').write_bytes(b'not a png at all, but long enough')
    assert sbs_generator.png_size(tmp_path / 'y.png') is None
    assert sbs_generator.png_size(tmp_path / 'missing.png') is None


def test_resume_refuses_outputs_of_another_layout(tmp_path):
    """Frame 0 was written in the default layout (32 x 96); continuing frame 1 as half-sbs (32 x 48) would mix sizes."""
    wf = _workflow(tmp_path, n=2, h=32, w=48)
    cv2.imwrite(str(wf / 'sbs' / 'sbs_000000.png'), np.zeros((32, 96, 3), np.uint8))
    r = _run('sbs_generator.py', wf, '--no-interactive', '--layout', 'half-sbs')
    assert r.returncode == 2 and 'ERROR:' in r.stdout and 'sbs_000000.png is 96x32' in r.stdout
    cfg = json.loads((wf / 'config.json').read_text())
    cfg['sbs_layout'] = 'tb'
    (wf / 'config.json').write_text(json.dumps(cfg))
    r = _run('sbs_generator.py', wf, '--no-interactive')
    assert r.returncode == 2 and "layout 'tb' makes 48x64" in r.stdout
    # the flag wins over the config key, and the matching layout passes the check (then needs a GPU, or runs on it)
    assert sbs_generator.layout_refusal(wf / 'sbs', wf / 'frames' / 'frame_000001.png', 'sbs') is None
    assert sbs_generator.layout_refusal(wf / 'sbs', wf / 'frames' / 'frame_000001.png', 'anaglyph') is not None
    r = _run('sbs_generator.py', wf, '--no-interactive', '--layout', 'sbs')
    assert 'sbs_000000.png is' not in r.stdout and r.returncode in (0, 100), r.stdout
    # nothing written yet: no check
    empty = _workflow(tmp_path / 'e', n=2)
    assert sbs_generator.layout_refusal(empty / 'sbs', empty / 'frames' / 'frame_000000.png', 'half-tb') is None


@pytest.mark.parametrize('layout', LAYOUTS)
def test_raw_sink_geometry_follows_the_layout(tmp_path, layout):
    wf = _workflow(tmp_path, n=3, h=32, w=48)
    from vsc_b200.workflow import find_frame_pairs
    pairs = find_frame_pairs(wf / 'frames', wf / 'depth_maps')[0]
    path = str(tmp_path / 'out.rgb')
    sink = sbs_generator.open_raw_sink(path, pairs, layout)
    oh, ow, _ = output_shape(layout, 32, 48)
    if layout != 'sbs':
        with pytest.raises(ValueError):
            sink.put(0, np.zeros((32, 96, 3), np.uint8))              # an SBS frame does not fit another layout's stream
    for i in range(3):
        sink.put(i, np.full((oh, ow, 3), i, np.uint8))
    assert sink.close()
    meta = json.loads(open(path + '.json').read())
    assert (meta['height'], meta['width'], meta['bytes_per_frame'], meta['frames']) == (oh, ow, oh * ow * 3, 3)
    assert f'-s {ow}x{oh}' in meta['ffmpeg_input']
    assert os.path.getsize(path) == 3 * oh * ow * 3
