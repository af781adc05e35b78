"""Output pixel formats without a GPU: the NumPy restatement (pixfmt_oracle.pack_pixfmt) against its recipe and OpenCV,
the library's host-only size rules (vsc_output_size, output_shape), the raw sink's YUV frames and side-car, and the
driver's pixel-format choice."""
import ctypes as C
import json
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest

import layout_oracle as LO
import pixfmt_oracle as PO
from conftest import ROOT
from vsc_b200 import _lib
from vsc_b200.sharder import RawFrameSink
from vsc_b200.stereo_core import LAYOUTS, MATRICES, PIXFMTS, output_dtype, output_shape
from vsc_b200.synthetic import make_pair
from vsc_b200.workflow import LayoutError, config_pixfmt, load_config

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')
sys.path.insert(0, PKG)
import sbs_generator  # noqa: E402

YUV = ('yuv420p', 'yuv420p10le')


def _rgb(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


# ---- pack_pixfmt --------------------------------------------------------------------------------
def test_bt709_table_follows_from_kr_kb():
    assert np.array_equal(PO.bt709_table(), PO.MATRIX['bt709'])
    m = PO.MATRIX['bt709']
    assert m[1].sum() == 0 and m[2].sum() == 0                        # grey has no chroma
    # OpenCV's bt601 rows are rounded one by one: each sums to +1, too little to move grey off 128 / 512
    assert PO.MATRIX['bt601'][1].sum() == 1 and PO.MATRIX['bt601'][2].sum() == 1
    for m in PO.MATRIX.values():
        assert m[1, 2] == m[2, 0]                                      # cu_b == cv_r


@pytest.mark.parametrize('matrix', MATRICES)
@pytest.mark.parametrize('value,y8,y10', [(0, 16, 64), (255, 235, 940), (128, None, None), (77, None, None)])
def test_black_white_grey(matrix, value, y8, y10):
    frame = np.full((4, 6, 3), value, np.uint8)
    for fmt, y_want, c_want in (('yuv420p', y8, 128), ('yuv420p10le', y10, 512)):
        out = PO.pack_pixfmt(frame, fmt, matrix)
        assert out.shape == (6, 6) and out.dtype == output_dtype(fmt)
        y, u, v = PO.split_planes(out)
        assert (u == c_want).all() and (v == c_want).all()
        if y_want is not None:
            assert (y == y_want).all()
        assert len(np.unique(y)) == 1


@pytest.mark.parametrize('h,w', [(2, 2), (30, 46), (136, 240), (1080, 1920)])
def test_bt601_equals_cv2_i420(h, w):
    """OpenCV's RGB2YUV_I420 is the 8-bit bt601 formula: luma on any image; chroma samples the top-left pixel of each
    2x2 block, which equals the centre-sited box on images that are constant over 2x2 blocks (S = 4p)."""
    rgb = _rgb(h, w, seed=h + w)
    ref, got = cv2.cvtColor(rgb, cv2.COLOR_RGB2YUV_I420), PO.pack_pixfmt(rgb, 'yuv420p', 'bt601')
    assert ref.shape == got.shape == output_shape('anaglyph', h, w, 'yuv420p')
    assert np.array_equal(PO.split_planes(got)[0], PO.split_planes(ref)[0])
    blocky = np.repeat(np.repeat(rgb[::2, ::2], 2, 0), 2, 1)
    assert np.array_equal(PO.pack_pixfmt(blocky, 'yuv420p', 'bt601'), cv2.cvtColor(blocky, cv2.COLOR_RGB2YUV_I420))


@pytest.mark.parametrize('matrix', MATRICES)
def test_ranges_and_10_bit_agree_with_8_bit(matrix):
    rgb = _rgb(64, 128, seed=5)
    y8, u8, v8 = (p.astype(int) for p in PO.split_planes(PO.pack_pixfmt(rgb, 'yuv420p', matrix)))
    y10, u10, v10 = (p.astype(int) for p in PO.split_planes(PO.pack_pixfmt(rgb, 'yuv420p10le', matrix)))
    assert 16 <= y8.min() and y8.max() <= 235 and 64 <= y10.min() and y10.max() <= 940
    for c8, c10 in ((u8, u10), (v8, v10)):
        assert 16 <= c8.min() and c8.max() <= 240 and 64 <= c10.min() and c10.max() <= 960
        assert np.abs(c10 - 4 * c8).max() <= 2
    assert np.abs(y10 - 4 * y8).max() <= 2
    # float reference: the rounded Q20 integers stay within one 10-bit step of the real-valued matrix
    kr, kb = (0.2126, 0.0722) if matrix == 'bt709' else (0.299, 0.114)
    x = rgb.astype(np.float64) / 255
    yf = kr * x[..., 0] + (1 - kr - kb) * x[..., 1] + kb * x[..., 2]
    assert np.abs(y10 - (64 + 876 * yf)).max() <= 1.0


def test_rgb24_is_the_frame_itself():
    rgb = _rgb(5, 7, seed=1)
    assert np.array_equal(PO.pack_pixfmt(rgb, 'rgb24'), rgb)
    with pytest.raises(ValueError):
        PO.pack_pixfmt(rgb, 'yuv420p')                                  # odd size
    with pytest.raises(ValueError):
        PO.pack_pixfmt(rgb[:4, :6], 'nv12')


# ---- vsc_output_size / output_shape (host only) --------------------------------------------------
def _size(layout, pixfmt, h, w):
    n = C.c_size_t(0)
    rc = _lib.load().vsc_output_size(layout, pixfmt, h, w, C.byref(n))
    return rc, n.value


@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('pixfmt', PIXFMTS)
def test_output_size_every_layout_and_format(layout, pixfmt):
    h, w = 36, 44
    oh, ow, _ = output_shape(layout, h, w)
    shape = output_shape(layout, h, w, pixfmt)
    want = (oh, ow, 3) if pixfmt == 'rgb24' else (oh * 3 // 2, ow)
    assert shape == want
    frame = PO.pack_pixfmt(LO.pack_layout(_rgb(h, 2 * w, 0), layout), pixfmt)
    assert frame.shape == shape and frame.dtype == output_dtype(pixfmt)
    rc, n = _size(LAYOUTS.index(layout), PIXFMTS.index(pixfmt), h, w)
    assert rc == 0 and n == frame.nbytes


def test_output_size_known_answers():
    assert (_lib.PIXFMT_RGB24, _lib.PIXFMT_YUV420P, _lib.PIXFMT_YUV420P10LE) == (0, 1, 2)
    assert (_lib.MATRIX_BT709, _lib.MATRIX_BT601) == (0, 1)
    # 1080p side-by-side: 12.4 MB rgb24, half of it as yuv420p, the same bytes as yuv420p10le
    assert [_size(0, f, 1080, 1920)[1] for f in range(3)] == [12441600, 6220800, 12441600]
    assert [_size(1, f, 2160, 3840)[1] for f in range(3)] == [24883200, 12441600, 24883200]


@pytest.mark.parametrize('pixfmt', YUV)
def test_output_size_refusals(pixfmt):
    lib, f = _lib.load(), PIXFMTS.index(pixfmt)
    for layout in range(5):
        for h, w in ((101, 200), (100, 201)):                         # odd sides: no whole 2x2 blocks
            assert _size(layout, f, h, w)[0] == _lib.VSC_E_INVALID
            with pytest.raises(ValueError):
                output_shape(LAYOUTS[layout], h, w, pixfmt)
    # half-sbs needs W % 4 == 0 and half-tb H % 4 == 0 (each eye starts on an even coordinate)
    assert _size(_lib.LAYOUT_HALF_SBS, f, 100, 202)[0] == _lib.VSC_E_INVALID and b'divisible by 4' in lib.vsc_last_error()
    assert _size(_lib.LAYOUT_HALF_TB, f, 102, 200)[0] == _lib.VSC_E_INVALID and b'divisible by 4' in lib.vsc_last_error()
    assert _size(_lib.LAYOUT_HALF_SBS, f, 102, 200)[0] == 0 and _size(_lib.LAYOUT_HALF_TB, f, 100, 202)[0] == 0
    for layout in (0, 2, 4):
        assert _size(layout, f, 102, 202)[0] == 0
    assert _size(_lib.LAYOUT_HALF_SBS, 0, 100, 202)[0] == 0            # rgb24 keeps the layout's own rule
    with pytest.raises(ValueError, match='divisible by 4'):
        output_shape('half-tb', 102, 200, pixfmt)


def test_output_size_and_set_pixfmt_reject_unknown_values():
    lib = _lib.load()
    for bad in (-1, 3, 99):
        assert _size(0, bad, 100, 200)[0] == _lib.VSC_E_INVALID and b'unknown pixel format' in lib.vsc_last_error()
    assert _size(5, 1, 100, 200)[0] == _lib.VSC_E_INVALID
    assert lib.vsc_output_size(0, 0, 10, 10, None) == _lib.VSC_E_INVALID
    assert lib.vsc_set_pixfmt(None, 0, 0) == _lib.VSC_E_INVALID
    with pytest.raises(ValueError, match='unknown pixel format'):
        output_shape('sbs', 10, 10, 'nv12')
    with pytest.raises(ValueError, match='unknown pixel format'):
        output_dtype('p010')


def test_generator_refuses_unknown_format_before_touching_a_device():
    from vsc_b200 import StereoGenerator
    with pytest.raises(ValueError, match='unknown pixel format'):
        StereoGenerator('cuda', pixfmt='yuv444p')
    with pytest.raises(ValueError, match='unknown yuv matrix'):
        StereoGenerator('cuda', pixfmt='yuv420p', matrix='bt2020')


# ---- raw sink -------------------------------------------------------------------------------------
@pytest.mark.parametrize('matrix', MATRICES)
@pytest.mark.parametrize('pixfmt', YUV)
def test_raw_sink_yuv_bytes_and_side_car(tmp_path, pixfmt, matrix):
    h, w, n = 6, 10, 4
    path = str(tmp_path / 'out.yuv')
    sink = RawFrameSink(path, n, h, w, max_ahead=4, frame_numbers=range(7, 7 + n), pixfmt=pixfmt, matrix=matrix)
    frames = [PO.pack_pixfmt(_rgb(h, w, i), pixfmt, matrix) for i in range(n)]
    with pytest.raises(ValueError):
        sink.put(0, np.zeros((h, w, 3), np.uint8))                    # an rgb24 frame does not fit a YUV stream
    with pytest.raises(ValueError):
        sink.put(0, frames[0].astype(np.uint32))
    for i in (3, 0, 2):
        sink.put(i, frames[i])
    sink.skip(1)
    assert sink.close()
    data = open(path, 'rb').read()
    bpf = frames[0].nbytes
    assert len(data) == n * bpf == n * h * w * (3 if pixfmt == 'yuv420p10le' else 1.5)
    black = np.frombuffer(data[bpf:2 * bpf], '<u2' if pixfmt == 'yuv420p10le' else 'u1').reshape(frames[0].shape)
    y, u, v = PO.split_planes(black)
    assert (y == (64 if pixfmt == 'yuv420p10le' else 16)).all() and (u == v).all()
    assert (u == (512 if pixfmt == 'yuv420p10le' else 128)).all()
    for i in (0, 2, 3):
        got = np.frombuffer(data[i * bpf:(i + 1) * bpf], '<u2' if pixfmt == 'yuv420p10le' else 'u1').reshape(frames[0].shape)
        assert np.array_equal(got, frames[i])
    # the black frame is what pack_pixfmt makes of black rgb
    assert np.array_equal(black, PO.pack_pixfmt(np.zeros((h, w, 3), np.uint8), pixfmt, matrix))
    meta = json.loads(open(path + '.json').read())
    colour = {'bt709': 'bt709', 'bt601': 'smpte170m'}[matrix]
    assert meta['pix_fmt'] == pixfmt and meta['matrix'] == matrix and meta['range'] == 'tv'
    assert meta['chroma_location'] == 'center' and meta['bytes_per_frame'] == bpf
    assert (meta['width'], meta['height'], meta['frames'], meta['frame_numbers']) == (w, h, n, list(range(7, 7 + n)))
    assert meta['ffmpeg_input'] == (f'-f rawvideo -pix_fmt {pixfmt} -s {w}x{h} -color_range tv -colorspace {colour} '
                                    f'-color_primaries {colour} -color_trc {colour} -i {path}')


def test_raw_sink_rgb24_side_car_unchanged(tmp_path):
    path = str(tmp_path / 'out.rgb')
    sink = RawFrameSink(path, 1, 4, 6)
    sink.put(0, np.zeros((4, 6, 3), np.uint8))
    assert sink.close()
    meta = json.loads(open(path + '.json').read())
    assert list(meta) == ['pix_fmt', 'width', 'height', 'frames', 'bytes_per_frame', 'frame_numbers', 'ffmpeg_input']
    assert meta['ffmpeg_input'] == f'-f rawvideo -pix_fmt rgb24 -s 6x4 -i {path}'


def test_raw_sink_refuses_bad_formats(tmp_path):
    with pytest.raises(ValueError):
        RawFrameSink(str(tmp_path / 'a'), 1, 4, 6, pixfmt='nv12')
    with pytest.raises(ValueError):
        RawFrameSink(str(tmp_path / 'b'), 1, 4, 6, pixfmt='yuv420p', matrix='bt2020')
    with pytest.raises(ValueError):
        RawFrameSink(str(tmp_path / 'c'), 1, 5, 6, pixfmt='yuv420p')


# ---- drivers ------------------------------------------------------------------------------------
def _workflow(tmp_path, n=2, h=32, w=48, extra=None):
    wf = tmp_path / 'wf'
    for d in ('frames', 'depth_maps', 'sbs'):
        (wf / d).mkdir(parents=True)
    cfg = {'input_video': 'in.mkv', 'output_video': 'out.mkv',
           'directories': {'frames': 'frames', 'depth_maps': 'depth_maps', 'sbs': 'sbs', 'chunks': 'chunks'},
           'stereo': {'max_disparity': 5.0, 'convergence': 0.0, 'super_sampling': 1.0, 'edge_softness': 0.0,
                      'artifact_smoothing': 0.0, 'depth_gamma': 1.0, 'sharpen': 0.0},
           'free_space': {'sbs_generator': 'none', 'chunk_generator': 'none'}}
    cfg.update(extra or {})
    (wf / 'config.json').write_text(json.dumps(cfg))
    for i in range(n):
        rgb, depth = make_pair(h, w, seed=i)
        cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(rgb, cv2.COLOR_RGB2BGR))
        cv2.imwrite(str(wf / 'depth_maps' / f'depth_frame_{i:06d}.png'), depth)
    return wf


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), *map(str, args)], capture_output=True,
                          text=True, timeout=300)


def test_config_pixfmt_keys(tmp_path):
    assert config_pixfmt(load_config(_workflow(tmp_path, n=0))) == ('rgb24', 'bt709')
    wf = _workflow(tmp_path / 'y', n=0, extra={'sbs_pixfmt': 'yuv420p10le', 'sbs_matrix': 'bt601'})
    assert config_pixfmt(load_config(wf)) == ('yuv420p10le', 'bt601')
    for i, extra in enumerate(({'sbs_pixfmt': 'nv12'}, {'sbs_pixfmt': 1}, {'sbs_matrix': 'bt2020'}, {'sbs_matrix': None})):
        with pytest.raises(LayoutError):
            load_config(_workflow(tmp_path / f'bad{i}', n=0, extra=extra))


def test_cli_pixfmt_flag_parsing():
    p = sbs_generator.build_parser()
    a = p.parse_args(['wf'])
    assert a.pixfmt is None and a.matrix is None
    for f in PIXFMTS:
        for m in MATRICES:
            a = p.parse_args(['wf', '--pixfmt', f, '--matrix', m])
            assert (a.pixfmt, a.matrix) == (f, m)


def test_cli_refuses_bad_pixfmt_with_exit_2(tmp_path):
    wf = _workflow(tmp_path)
    r = _run(wf, '--pixfmt', 'nv12', '--raw-sink', tmp_path / 'o.yuv')
    assert r.returncode == 2 and 'invalid choice' in r.stderr
    r = _run(wf, '--pixfmt', 'yuv420p', '--matrix', 'bt2020', '--raw-sink', tmp_path / 'o.yuv')
    assert r.returncode == 2 and 'invalid choice' in r.stderr
    bad = _workflow(tmp_path / 'cfg', extra={'sbs_pixfmt': 'p010'})
    r = _run(bad, '--no-interactive')
    assert r.returncode == 2 and r.stdout.startswith('ERROR:') and 'sbs_pixfmt' in r.stdout


@pytest.mark.parametrize('pixfmt', YUV)
def test_cli_refuses_yuv_without_raw_sink(tmp_path, pixfmt):
    wf = _workflow(tmp_path)
    r = _run(wf, '--no-interactive', '--pixfmt', pixfmt)
    assert r.returncode == 2 and 'ERROR:' in r.stdout and '--raw-sink' in r.stdout
    assert not list((wf / 'sbs').iterdir())
    cfg = _workflow(tmp_path / 'cfg', extra={'sbs_pixfmt': pixfmt})
    r = _run(cfg, '--no-interactive')
    assert r.returncode == 2 and '--raw-sink' in r.stdout


def test_cli_refuses_a_size_the_format_cannot_take(tmp_path):
    wf = _workflow(tmp_path, h=32, w=46)
    r = _run(wf, '--no-interactive', '--pixfmt', 'yuv420p', '--layout', 'half-sbs', '--raw-sink', tmp_path / 'o.yuv')
    assert r.returncode == 2 and 'ERROR:' in r.stdout and 'divisible by 4' in r.stdout


@pytest.mark.parametrize('pixfmt', YUV)
def test_open_raw_sink_follows_layout_and_format(tmp_path, pixfmt):
    wf = _workflow(tmp_path, n=2, h=32, w=48)
    from vsc_b200.workflow import find_frame_pairs
    pairs = find_frame_pairs(wf / 'frames', wf / 'depth_maps')[0]
    path = str(tmp_path / 'o.yuv')
    sink = sbs_generator.open_raw_sink(path, pairs, 'tb', pixfmt, 'bt601')
    assert (sink.h, sink.w, sink.shape) == (64, 48, output_shape('tb', 32, 48, pixfmt))
    assert sink.dtype == output_dtype(pixfmt)
    for i in range(2):
        sink.skip(i)
    assert sink.close()
    meta = json.loads(open(path + '.json').read())
    assert meta['pix_fmt'] == pixfmt and meta['matrix'] == 'bt601' and '-s 48x64' in meta['ffmpeg_input']
