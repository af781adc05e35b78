"""PNG output on the GPU: every file the library writes passes png_oracle.check_png against the rgb24 frame it encodes
(chunk CRCs, zlib header, one IDAT per segment, an inflate that equals the oracle's filtered stream byte for byte, the
Adler-32 and a cv2 decode), through vsc_stage_png on crafted frames and through every submit path of the pipeline."""
import ctypes as C
import json
import os
import subprocess
import sys
import threading

import cv2
import numpy as np
import pytest

import png_oracle as PN
from conftest import ROOT
from vsc_b200 import StereoGenerator, StereoParams, _lib
from vsc_b200.stereo_core import LAYOUTS, encoded_capacity, layout_code, output_shape
from vsc_b200.synthetic import make_pair

pytestmark = pytest.mark.gpu

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')


@pytest.fixture(scope='module')
def pctx():
    c = _lib.Context(0, 1)
    yield c
    c.close()


def _stage(ctx, frame):
    """(file bytes, debug counters) of vsc_stage_png on an rgb24 frame."""
    frame = np.ascontiguousarray(frame, np.uint8)
    h, w, _ = frame.shape
    cap = encoded_capacity('anaglyph', h, w)
    out = np.empty(cap, np.uint8)
    n = C.c_size_t()
    lib = _lib.load()
    _lib.check(lib.vsc_stage_png(ctx.handle, _lib.ptr(frame), h, w, _lib.ptr(out), cap, C.byref(n)))
    st = (C.c_ulonglong * 3)()
    _lib.check(lib.vsc_debug_png_stats(ctx.handle, st))
    assert 0 < n.value <= cap
    return out[:n.value].tobytes(), list(st)


def _rng(seed):
    return np.random.default_rng(seed)


# ---- crafted frames through vsc_stage_png ------------------------------------------------------------
@pytest.mark.parametrize('h,w', [(1, 1), (1, 2), (1, 7), (7, 1), (64, 1), (5, 3), (13, 17), (31, 33), (2, 10923),
                                 (1, 20000), (20, 1365), (40, 1000), (200, 301)])
@pytest.mark.parametrize('kind', ['blocky', 'noise'])
def test_sizes(pctx, h, w, kind):
    rng = _rng(h * 7919 + w)
    if kind == 'noise':
        frame = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    else:
        small = rng.integers(0, 4, ((h + 7) // 8, (w + 7) // 8, 3), dtype=np.uint8) * 60
        frame = np.repeat(np.repeat(small, 8, 0), 8, 1)[:h, :w]
    data, st = _stage(pctx, frame)
    PN.check_png(data, frame)


def test_segment_edges_on_and_off_rows(pctx):
    # rows of 1 + 3 * 1365 = 4096 bytes: every segment edge falls exactly on a row; 3001-byte rows: mid-row
    for h, w in ((20, 1365), (40, 1000)):
        frame = make_pair(h, w, seed=4)[0]
        n = h * (1 + 3 * w)
        assert n > 2 * PN.SEG and (w != 1365 or PN.SEG % (1 + 3 * w) == 0)
        data, _ = _stage(pctx, frame)
        PN.check_png(data, frame)


@pytest.mark.parametrize('kind', ['black', 'constant', 'letterbox', 'white_rows', 'gradient'])
def test_flat_frames(pctx, kind):
    h, w = 270, 480
    if kind == 'black':
        frame = np.zeros((h, w, 3), np.uint8)
    elif kind == 'constant':
        frame = np.full((h, w, 3), (17, 200, 99), np.uint8)
    elif kind == 'letterbox':
        frame = np.zeros((h, w, 3), np.uint8)
        frame[40:-40] = cv2.GaussianBlur(make_pair(h - 80, w, seed=2)[0], (9, 9), 3)
    elif kind == 'white_rows':
        frame = np.zeros((h, w, 3), np.uint8)
        frame[::3] = 255
    else:
        frame = np.broadcast_to(np.arange(w, dtype=np.uint8)[None, :, None], (h, w, 3)).copy()
    data, st = _stage(pctx, frame)
    PN.check_png(data, frame)
    assert st[2] == 0                                    # nothing here needs a stored block
    assert len(data) <= 1.05 * PN.model_size(frame)


def _marker_frame(L, d):
    """A black 250 x 100 frame whose filtered stream (every row filter 0: isolated 1s cost least unfiltered) holds a run
    of exactly L zero bytes with d of them before the first segment edge, and a second such run across the second."""
    w, h = 100, 250
    R = 1 + 3 * w
    frame = np.zeros((h, w, 3), np.uint8)
    flat = frame.reshape(h, 3 * w)
    for edge in (PN.SEG, 2 * PN.SEG):
        for s in (edge - d - 1, edge - d + L):
            assert s % R != 0
            flat[s // R, s % R - 1] = 1
    return frame


@pytest.mark.parametrize('L', [258, 259, 260, 261, 516, 517])
@pytest.mark.parametrize('d', [0, 1, 2, 3, 100, 257])
def test_runs_across_segment_edges(pctx, L, d):
    frame = _marker_frame(L, d)
    f = PN.filter_rows(frame)
    s = PN.SEG - d - 1
    assert f[s] == 1 and f[s + L + 1] == 1 and f[s + 1:s + L + 1] == bytes(L)
    data, _ = _stage(pctx, frame)
    PN.check_png(data, frame)


def test_noise_falls_back_to_stored_blocks(pctx):
    frame = _rng(5).integers(0, 256, (300, 400, 3), dtype=np.uint8)
    data, st = _stage(pctx, frame)
    PN.check_png(data, frame)
    nseg = -(-300 * 1201 // PN.SEG)
    assert st[2] == nseg
    assert len(data) <= encoded_capacity('anaglyph', 300, 400)


def _fibonacci_frame():
    """One row: pixels (v, v, v) for v = 1..17, F(v) of each (Fibonacci), each followed by a black pixel.  Filter 0 wins
    (sub and paeth cost twice as much, up ties and average costs more); no run reaches 4, so the segment is all literals
    with Fibonacci-like frequencies: an unlimited Huffman code needs 17+ bits."""
    fib = [1, 1]
    while len(fib) < 17:
        fib.append(fib[-1] + fib[-2])
    px = []
    for v, n in zip(range(1, 18), fib):
        px += [(v, v, v), (0, 0, 0)] * n
    return np.array(px, np.uint8)[None]


def _huffman_depth(freq):
    import heapq
    heap = [(f, i, 0) for i, f in enumerate(freq) if f]
    depth = {}
    nodes = {i: [i] for _, i, _ in heap}
    nxt = len(freq)
    while len(heap) > 1:
        f1, i1, _ = heapq.heappop(heap)
        f2, i2, _ = heapq.heappop(heap)
        for leaf in nodes[i1] + nodes[i2]:
            depth[leaf] = depth.get(leaf, 0) + 1
        nodes[nxt] = nodes.pop(i1) + nodes.pop(i2)
        heapq.heappush(heap, (f1 + f2, nxt, 0))
        nxt += 1
    return max(depth.values())


def test_length_limit_path(pctx):
    frame = _fibonacci_frame()
    f = PN.filter_rows(frame)
    assert f[0] == 0 and len(f) <= PN.SEG
    freq = np.bincount(np.frombuffer(f, np.uint8), minlength=256).tolist() + [1]    # + end of block
    assert _huffman_depth(freq) > 15
    data, st = _stage(pctx, frame)
    PN.check_png(data, frame)
    assert st[0] == 1 and st[2] == 0


def test_stage_refusals(pctx):
    lib = _lib.load()
    frame = np.zeros((4, 4, 3), np.uint8)
    cap = encoded_capacity('anaglyph', 4, 4)
    out = np.empty(cap, np.uint8)
    n = C.c_size_t()
    assert lib.vsc_stage_png(pctx.handle, _lib.ptr(frame), 4, 4, _lib.ptr(out), cap - 1, C.byref(n)) == _lib.VSC_E_INVALID
    assert lib.vsc_stage_png(pctx.handle, _lib.ptr(frame), 0, 4, _lib.ptr(out), cap, C.byref(n)) == _lib.VSC_E_INVALID
    assert lib.vsc_stage_png(pctx.handle, None, 4, 4, _lib.ptr(out), cap, C.byref(n)) == _lib.VSC_E_INVALID


# ---- the pipeline --------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def gen():
    g = StereoGenerator('cuda', n_slots=2)
    yield g
    g.close()


_pairs = {}


def _pair(h, w):
    if (h, w) not in _pairs:
        _pairs[(h, w)] = make_pair(h, w, seed=11, depth_dtype=np.uint16 if h > 1080 else np.uint8)
    return _pairs[(h, w)]


@pytest.mark.parametrize('layout', LAYOUTS)
@pytest.mark.parametrize('h,w', [(1080, 1920), (2160, 3840)])
def test_pipeline_png_decodes_to_the_raw_frame(gen, layout, h, w):
    rgb, depth = _pair(h, w)
    gen.set_encode(None)
    gen.set_layout(layout)
    raw = gen.process_frame(rgb, depth)
    gen.set_encode('png')
    data = gen.process_frame(rgb, depth)
    gen.set_encode(None)
    assert data.dtype == np.uint8 and data.ndim == 1 and data.size <= encoded_capacity(layout, h, w)
    assert raw.shape == output_shape(layout, h, w)
    PN.check_png(data, raw)
    if h == 1080:
        ok, ref = cv2.imencode('.png', cv2.cvtColor(raw, cv2.COLOR_RGB2BGR))
        assert data.size <= ref.size
        assert data.size <= 1.05 * PN.model_size(raw)


def test_grouped_and_pinned_submissions(gen):
    frames = [make_pair(136, 240, seed=s) for s in range(5)]
    gen.set_layout('sbs')
    raw = gen.process_batch(frames)
    g = StereoGenerator('cuda', n_slots=2, group_size=3, layout='sbs', encode='png')
    try:
        files = g.process_batch(frames)
        assert len(files) == 5
        for d, r in zip(files, raw):
            PN.check_png(d, r)
        g.submit_frames(0, frames[:3])
        outs = g.collect(0, copy=False)
        assert [g.encoded_bytes(0, i) for i in range(3)] == [o.size for o in outs]
        for d, r in zip(outs, raw[:3]):
            PN.check_png(d, r)
    finally:
        g.close()


def test_device_resident_submissions():
    import torch
    frames = [make_pair(136, 240, seed=s, depth_dtype=np.uint16) for s in range(3)]
    ref = StereoGenerator('cuda', n_slots=1, layout='tb')
    raw = [ref.process_frame(r, d) for r, d in frames]
    ref.close()
    g = StereoGenerator('cuda', n_slots=2, group_size=2, layout='tb', encode='png')
    try:
        cap = encoded_capacity('tb', 136, 240)
        d_in = [(torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda()) for r, d in frames]
        d_out = [torch.zeros(cap, dtype=torch.uint8, device='cuda') for _ in frames]
        torch.cuda.synchronize()
        g.submit_device(0, d_in[0][0].data_ptr(), d_in[0][1].data_ptr(), np.uint16, 136, 240, d_out[0].data_ptr())
        g.submit_device_group(1, [(d_in[i][0].data_ptr(), d_in[i][1].data_ptr(), d_out[i].data_ptr()) for i in (1, 2)],
                              np.uint16, 136, 240)
        g.wait(0)
        g.wait(1)
        sizes = [g.encoded_bytes(0), g.encoded_bytes(1, 0), g.encoded_bytes(1, 1)]
        for i in range(3):
            PN.check_png(d_out[i][:sizes[i]].cpu().numpy(), raw[i])
    finally:
        g.close()


def test_switching_encodings_with_frames_in_flight():
    lib = _lib.load()
    ctx = _lib.Context(0, 2)
    try:
        rgb, depth = make_pair(120, 160, seed=3)
        p = C.byref(_lib.make_params(StereoParams()))
        raw = _lib.PinnedBuffer((120, 320, 3), np.uint8)
        cap = encoded_capacity('sbs', 120, 160)
        png = _lib.PinnedBuffer((cap,), np.uint8)
        _lib.check(lib.vsc_submit(ctx.handle, 0, _lib.ptr(rgb), _lib.ptr(depth), _lib.DEPTH_U8, 120, 160, p, _lib.ptr(raw.array)))
        _lib.check(lib.vsc_set_encode(ctx.handle, _lib.ENCODE_PNG))
        _lib.check(lib.vsc_submit(ctx.handle, 1, _lib.ptr(rgb), _lib.ptr(depth), _lib.DEPTH_U8, 120, 160, p, _lib.ptr(png.array)))
        _lib.check(lib.vsc_set_encode(ctx.handle, _lib.ENCODE_NONE))
        n = C.c_size_t()
        assert lib.vsc_encoded_bytes(ctx.handle, 1, 0, C.byref(n)) == _lib.VSC_E_STATE     # still in flight
        _lib.check(lib.vsc_wait(ctx.handle, 0))
        _lib.check(lib.vsc_wait(ctx.handle, 1))
        assert lib.vsc_encoded_bytes(ctx.handle, 0, 0, C.byref(n)) == _lib.VSC_E_STATE     # a raw submission
        _lib.check(lib.vsc_encoded_bytes(ctx.handle, 1, 0, C.byref(n)))
        PN.check_png(png.array[:n.value], raw.array)
        assert lib.vsc_encoded_bytes(ctx.handle, 1, 1, C.byref(n)) == _lib.VSC_E_INVALID
        raw.free()
        png.free()
    finally:
        ctx.close()


def test_png_and_yuv_refuse_each_other():
    lib = _lib.load()
    ctx = _lib.Context(0, 1)
    try:
        _lib.check(lib.vsc_set_pixfmt(ctx.handle, _lib.PIXFMT_YUV420P, _lib.MATRIX_BT709))
        assert lib.vsc_set_encode(ctx.handle, _lib.ENCODE_PNG) == _lib.VSC_E_INVALID
        _lib.check(lib.vsc_set_pixfmt(ctx.handle, _lib.PIXFMT_RGB24, _lib.MATRIX_BT709))
        _lib.check(lib.vsc_set_encode(ctx.handle, _lib.ENCODE_PNG))
        assert lib.vsc_set_pixfmt(ctx.handle, _lib.PIXFMT_YUV420P10LE, _lib.MATRIX_BT709) == _lib.VSC_E_INVALID
        assert lib.vsc_set_encode(ctx.handle, 2) == _lib.VSC_E_INVALID
    finally:
        ctx.close()
    with pytest.raises(_lib.VscError):
        StereoGenerator('cuda', pixfmt='yuv420p', encode='png')
    g = StereoGenerator('cuda', n_slots=1)
    try:
        g.submit(0, *make_pair(64, 64, seed=1))
        with pytest.raises(RuntimeError):
            g.set_encode('png')
        g.collect(0)
        g.set_encode('png')
        assert g.encode == 'png'
    finally:
        g.close()


def test_eight_threads_encoding_at_once():
    frames = [make_pair(96, 128 + 8 * i, seed=i) for i in range(8)]
    ref = StereoGenerator('cuda', n_slots=1)
    raw = [ref.process_frame(r, d) for r, d in frames]
    ref.close()
    errors, results = [], [None] * 8

    def work(i):
        try:
            g = StereoGenerator('cuda', n_slots=1, encode='png')
            try:
                results[i] = [g.process_frame(*frames[i]) for _ in range(3)]
            finally:
                g.close()
        except BaseException as e:   # noqa: BLE001
            errors.append(e)
    ths = [threading.Thread(target=work, args=(i,)) for i in range(8)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert not errors
    for i in range(8):
        assert all(np.array_equal(x, results[i][0]) for x in results[i])
        PN.check_png(results[i][0], raw[i])


# ---- the driver -------------------------------------------------------------------------------------------
def _workflow(root, n, h=64, w=96, extra=None):
    wf = root / 'wf'
    for d in ('frames', 'depth_maps', 'sbs'):
        (wf / d).mkdir(parents=True)
    cfg = {'input_video': 'in.mkv', 'output_video': 'out.mkv',
           'directories': {'frames': 'frames', 'depth_maps': 'depth_maps', 'sbs': 'sbs', 'chunks': 'chunks'},
           'stereo': {'max_disparity': 10.0, 'convergence': -2.0, 'super_sampling': 2.0, 'edge_softness': 5.0,
                      'artifact_smoothing': 1.0, 'depth_gamma': 0.5, 'sharpen': 4.0},
           'free_space': {'sbs_generator': 'none', 'chunk_generator': 'none'}}
    cfg.update(extra or {})
    (wf / 'config.json').write_text(json.dumps(cfg))
    for i in range(n):
        rgb, depth = make_pair(h, w, seed=i)
        cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(rgb, cv2.COLOR_RGB2BGR))
        cv2.imwrite(str(wf / 'depth_maps' / f'depth_frame_{i:06d}.png'), depth)
    return wf


def _run(*args):
    env = dict(os.environ, VSC_FAST_RETRY='1')
    return subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), *map(str, args)], capture_output=True,
                          text=True, timeout=600, env=env)


def _decode(p):
    return cv2.imread(str(p), cv2.IMREAD_UNCHANGED)


def test_driver_gpu_encoder_matches_cv2_and_resumes(tmp_path):
    n = 10
    a = _workflow(tmp_path / 'cv2', n)
    b = _workflow(tmp_path / 'gpu', n, extra={'free_space': {'sbs_generator': 'all', 'chunk_generator': 'none'}})
    r = _run(a, '--no-interactive', '--gpus', '1', '--slots', '2', '--group', '2')
    assert r.returncode == 0, r.stdout + r.stderr
    r = _run(b, '--no-interactive', '--gpus', '1', '--slots', '2', '--group', '2', '--png-encoder', 'gpu')
    assert r.returncode == 0, r.stdout + r.stderr
    names = sorted(p.name for p in (a / 'sbs').iterdir())
    assert names == sorted(p.name for p in (b / 'sbs').iterdir()) and len(names) == n
    for name in names:
        pa, pb = _decode(a / 'sbs' / name), _decode(b / 'sbs' / name)
        assert np.array_equal(pa, pb)
        PN.check_png((b / 'sbs' / name).read_bytes(), pa[..., ::-1])
    # free_space 'all': every input is gone, and only once its output exists
    assert not list((b / 'frames').iterdir()) and not list((b / 'depth_maps').iterdir())
    # resume: outputs that exist are kept, the missing ones are made again
    c = _workflow(tmp_path / 'resume', n, extra={'sbs_png_encoder': 'gpu'})
    r = _run(c, '--no-interactive', '--gpus', '1')
    assert r.returncode == 0, r.stdout + r.stderr
    (c / 'sbs' / names[3]).unlink()
    (c / 'sbs' / names[7]).unlink()
    before = {p.name: p.stat().st_mtime_ns for p in (c / 'sbs').iterdir()}
    r = _run(c, '--no-interactive', '--gpus', '1')
    assert r.returncode == 0 and '2 to process' in r.stdout, r.stdout
    assert all((c / 'sbs' / k).stat().st_mtime_ns == v for k, v in before.items())
    for name in names:
        assert np.array_equal(_decode(c / 'sbs' / name), _decode(a / 'sbs' / name))
    # the layout-size check reads IHDR of the library's files too
    r = _run(c, '--no-interactive', '--gpus', '1', '--layout', 'tb')
    assert r.returncode == 0 and 'All frames already processed' in r.stdout
    (c / 'sbs' / names[0]).unlink()
    r = _run(c, '--no-interactive', '--gpus', '1', '--layout', 'tb')
    assert r.returncode == 2 and 'layout' in r.stdout
