"""PNG output without a GPU: the NumPy oracle (png_oracle) against itself and OpenCV, the library's host-only capacity
rule and argument refusals, and the driver's choice of PNG encoder."""
import ctypes as C
import json
import os
import subprocess
import sys
import zlib

import cv2
import numpy as np
import pytest

import png_oracle as PN
from conftest import ROOT
from vsc_b200 import _lib
from vsc_b200.stereo_core import ENCODINGS, LAYOUTS, encode_code, encoded_capacity, layout_code, output_shape
from vsc_b200.synthetic import make_pair
from vsc_b200.workflow import LayoutError, config_png_encoder, load_config

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')
sys.path.insert(0, PKG)
import sbs_generator  # noqa: E402


def _frames():
    rng = np.random.default_rng(3)
    yield rng.integers(0, 256, (7, 5, 3), dtype=np.uint8)                       # noise
    yield np.zeros((4, 9, 3), np.uint8)
    yield np.full((3, 3, 3), 200, np.uint8)
    g = np.linspace(0, 255, 40 * 33 * 3).astype(np.uint8).reshape(40, 33, 3)     # gradients: sub / up / avg / paeth
    yield g
    yield np.ascontiguousarray(g.transpose(1, 0, 2))
    yield make_pair(24, 30, seed=1)[0]
    yield rng.integers(0, 256, (1, 1, 3), dtype=np.uint8)


def _filter_row_scalar(cur, prev):
    """One row of the heuristic restated byte by byte."""
    best = None
    for t in range(5):
        out = []
        for i, x in enumerate(cur):
            a = cur[i - 3] if i >= 3 else 0
            b = prev[i]
            c = prev[i - 3] if i >= 3 else 0
            if t == 0:
                pred = 0
            elif t == 1:
                pred = a
            elif t == 2:
                pred = b
            elif t == 3:
                pred = (a + b) // 2
            else:
                p = a + b - c
                pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
                pred = a if pa <= pb and pa <= pc else (b if pb <= pc else c)
            out.append((x - pred) & 255)
        cost = sum(min(v, 256 - v) for v in out)
        if best is None or cost < best[0]:
            best = (cost, bytes([t] + out))
    return best[1]


# ---- oracle ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('i', range(7))
def test_filter_then_unfilter_is_the_identity(i):
    frame = list(_frames())[i]
    h, w, _ = frame.shape
    f = PN.filter_rows(frame)
    assert len(f) == h * (1 + 3 * w)
    assert np.array_equal(PN.unfilter(f, h, w), frame)


def test_filter_rows_equals_the_scalar_restatement():
    for frame in _frames():
        if frame.shape[0] * frame.shape[1] > 400:
            frame = frame[:12, :11]
        frame = np.ascontiguousarray(frame)
        h, w, _ = frame.shape
        rows = frame.reshape(h, 3 * w).astype(int).tolist()
        want, prev = b'', [0] * (3 * w)
        for r in rows:
            want += _filter_row_scalar(r, prev)
            prev = r
        assert PN.filter_rows(frame) == want


def test_filter_rows_uses_every_type_and_breaks_ties_low():
    types = set()
    for frame in _frames():
        h, w, _ = frame.shape
        types |= set(PN.filter_rows(frame)[::1 + 3 * w])
    assert types == {0, 1, 2, 3, 4}
    # a constant row: types 0 and 2 cost the same on row 0 (zero row above); 1 and 4 cost less
    assert PN.filter_rows(np.zeros((2, 4, 3), np.uint8))[::13] == b'\x00\x00'


@pytest.mark.parametrize('i', range(7))
def test_oracle_assembled_png_decodes_in_cv2(i):
    frame = list(_frames())[i]
    data = PN.assemble(frame)
    img = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_UNCHANGED)
    assert np.array_equal(img[..., ::-1], frame)
    assert [t for t, _ in PN.chunks(data)] == [b'IHDR', b'IDAT', b'IEND']


def test_check_png_rejects_a_wrong_file():
    frame = list(_frames())[3]
    with pytest.raises(AssertionError):            # one IDAT of a zlib.compress stream: not this format's framing
        PN.check_png(PN.assemble(frame), frame)
    data = bytearray(PN.assemble(frame))
    data[40] ^= 1
    with pytest.raises(AssertionError):
        PN.chunks(bytes(data))


def test_model_size_counts_segments():
    f = np.zeros((100, 200, 3), np.uint8)
    n = len(PN.filter_rows(f))
    assert n > PN.SEG
    assert PN.model_size(f) < n // 50
    z = zlib.decompressobj(-15)
    c = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_RLE)
    assert z.decompress(c.compress(PN.filter_rows(f)[:PN.SEG]) + c.flush(zlib.Z_SYNC_FLUSH)) == PN.filter_rows(f)[:PN.SEG]


# ---- host-only library rules -----------------------------------------------------------------------
def _cap(layout, encode, h, w):
    n = C.c_size_t()
    rc = _lib.load().vsc_encoded_capacity(layout, encode, h, w, C.byref(n))
    return rc, n.value


@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('h,w', [(1, 1), (1, 10922), (2, 10923), (37, 91), (1080, 1920), (2160, 3840)])
def test_capacity_formula(layout, h, w):
    try:
        oh, ow, _ = output_shape(layout, h, w)
    except ValueError:
        assert _cap(layout_code(layout), _lib.ENCODE_PNG, h, w)[0] == _lib.VSC_E_INVALID
        with pytest.raises(ValueError):
            encoded_capacity(layout, h, w)
        return
    n = oh * (1 + 3 * ow)
    nseg = -(-n // PN.SEG)
    want = 53 + n + 22 * nseg
    assert _cap(layout_code(layout), _lib.ENCODE_PNG, h, w) == (0, want)
    assert encoded_capacity(layout, h, w) == want
    assert _cap(layout_code(layout), _lib.ENCODE_NONE, h, w) == (0, oh * ow * 3)


def test_capacity_covers_the_stored_worst_case():
    # every segment stored: 5 + n + 5 bytes of deflate; framing 8 + 25 + 12 per IDAT + 2 + 2 + 4 + 12
    for oh, ow in [(1, 1), (3, 5000), (1080, 3840)]:
        n = oh * (1 + 3 * ow)
        segs = [min(PN.SEG, n - o) for o in range(0, n, PN.SEG)]
        worst = 8 + 25 + sum(12 + s + 10 for s in segs) + 2 + 2 + 4 + 12
        assert encoded_capacity('anaglyph', oh, ow) == worst


def test_capacity_refusals():
    assert _cap(0, 2, 8, 8)[0] == _lib.VSC_E_INVALID
    assert _cap(0, -1, 8, 8)[0] == _lib.VSC_E_INVALID
    assert _cap(7, _lib.ENCODE_PNG, 8, 8)[0] == _lib.VSC_E_INVALID
    assert _cap(0, _lib.ENCODE_PNG, 0, 8)[0] == _lib.VSC_E_INVALID
    assert _cap(layout_code('half-sbs'), _lib.ENCODE_PNG, 8, 7)[0] == _lib.VSC_E_INVALID
    assert _lib.load().vsc_encoded_capacity(0, _lib.ENCODE_PNG, 8, 8, None) == _lib.VSC_E_INVALID


def test_encode_entry_points_refuse_without_a_context():
    lib = _lib.load()
    n = C.c_size_t()
    assert lib.vsc_set_encode(None, _lib.ENCODE_PNG) == _lib.VSC_E_INVALID
    assert lib.vsc_encoded_bytes(None, 0, 0, C.byref(n)) == _lib.VSC_E_INVALID
    assert lib.vsc_stage_png(None, None, 1, 1, None, 0, C.byref(n)) == _lib.VSC_E_INVALID
    assert lib.vsc_debug_png_stats(None, None) == _lib.VSC_E_INVALID


def test_encoding_names():
    assert ENCODINGS == ('png',)
    assert encode_code(None) == _lib.ENCODE_NONE and encode_code('png') == _lib.ENCODE_PNG
    for bad in ('PNG', 'jpeg', '', 1):
        with pytest.raises(ValueError):
            encode_code(bad)


# ---- driver -----------------------------------------------------------------------------------------
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


def test_config_png_encoder_key(tmp_path):
    assert config_png_encoder(load_config(_workflow(tmp_path, n=0))) == 'cv2'
    assert config_png_encoder(load_config(_workflow(tmp_path / 'g', n=0, extra={'sbs_png_encoder': 'gpu'}))) == 'gpu'
    for i, bad in enumerate(('GPU', 'nvjpeg', 1, None)):
        with pytest.raises(LayoutError):
            load_config(_workflow(tmp_path / f'bad{i}', n=0, extra={'sbs_png_encoder': bad}))


def test_cli_png_encoder_flag_parsing():
    p = sbs_generator.build_parser()
    assert p.parse_args(['wf']).png_encoder is None
    for e in ('cv2', 'gpu'):
        assert p.parse_args(['wf', '--png-encoder', e]).png_encoder == e


def test_cli_refuses_bad_png_encoder_with_exit_2(tmp_path):
    wf = _workflow(tmp_path)
    r = _run(wf, '--png-encoder', 'nvenc')
    assert r.returncode == 2 and 'invalid choice' in r.stderr
    bad = _workflow(tmp_path / 'cfg', extra={'sbs_png_encoder': 'fast'})
    r = _run(bad, '--no-interactive')
    assert r.returncode == 2 and r.stdout.startswith('ERROR:') and 'sbs_png_encoder' in r.stdout


def test_cli_refuses_gpu_png_with_raw_sink_or_yuv(tmp_path):
    wf = _workflow(tmp_path)
    r = _run(wf, '--no-interactive', '--png-encoder', 'gpu', '--raw-sink', tmp_path / 'o.rgb')
    assert r.returncode == 2 and 'ERROR:' in r.stdout and 'raw sink' in r.stdout
    for pixfmt in ('yuv420p', 'yuv420p10le'):
        r = _run(wf, '--no-interactive', '--png-encoder', 'gpu', '--pixfmt', pixfmt)
        assert r.returncode == 2 and 'ERROR:' in r.stdout and 'rgb24' in r.stdout
    cfg = _workflow(tmp_path / 'cfg', extra={'sbs_png_encoder': 'gpu'})
    r = _run(cfg, '--no-interactive', '--raw-sink', tmp_path / 'o2.rgb')
    assert r.returncode == 2 and 'raw sink' in r.stdout
    assert not list((wf / 'sbs').iterdir()) and not list((cfg / 'sbs').iterdir())


@pytest.mark.parametrize('flag,cfg,want', [(None, None, 'cv2'), ('gpu', None, 'gpu'), (None, 'gpu', 'gpu'), ('cv2', 'gpu', 'cv2')])
def test_torchrun_branch_passes_the_png_encoder(tmp_path, monkeypatch, flag, cfg, want):
    """Under torchrun (WORLD_SIZE > 1) main() calls process_shard with its own argument list: the encoder must reach it."""
    import torch
    import torch.distributed as dist
    from vsc_b200 import sharder
    wf = _workflow(tmp_path, extra={'sbs_png_encoder': cfg} if cfg else None)
    calls = []

    def fake_shard(*a, **kw):
        calls.append(kw)
        return 0
    monkeypatch.setenv('WORLD_SIZE', '2')
    monkeypatch.setenv('RANK', '1')
    monkeypatch.setenv('LOCAL_RANK', '1')
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: True)
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: 2)
    monkeypatch.setattr(dist, 'init_process_group', lambda *a, **k: None)
    monkeypatch.setattr(dist, 'destroy_process_group', lambda *a, **k: None)
    monkeypatch.setattr(sharder, 'barrier', lambda: None)
    monkeypatch.setattr(sbs_generator, 'process_shard', fake_shard)
    argv = [str(wf), '--no-interactive'] + (['--png-encoder', flag] if flag else [])
    assert sbs_generator.main(argv) == 0
    assert len(calls) == 1 and calls[0]['png_encoder'] == want and calls[0]['layout'] == 'sbs'
