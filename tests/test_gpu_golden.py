"""CUDA path against the golden vectors of the UNMODIFIED reference (tests/golden), and the drop-in driver."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from conftest import ROOT
from test_oracle_golden import (GOLDEN, GOLDEN_BIG, big_inputs, check_sbs_against_reference, fixture_name, load,
                                rebuild_reference, sha)
from vsc_b200 import StereoGenerator, StereoParams, _lib
from vsc_b200.synthetic import make_pair

pytestmark = pytest.mark.gpu
PKG = os.path.join(ROOT, 'video-stereo-converter_b200')


@pytest.fixture(scope='module')
def gen():
    g = StereoGenerator('cuda', n_slots=2)
    yield g
    g.close()


@pytest.mark.parametrize('path', GOLDEN_BIG, ids=[fixture_name(p) for p in GOLDEN_BIG])
def test_cuda_matches_reference_full_size(gen, path):
    """Full 1080p frame / 3840-wide band against the reference's own output (rebuilt from the fixture's patches and
    proven by its digest): the pinned distance, with and without IPP."""
    z, kw = load(path)
    rgb, depth = big_inputs(z)
    out = gen.process_frame(rgb, depth, StereoParams(**kw))
    name = fixture_name(path)
    check_sbs_against_reference(out, rebuild_reference(z, out), name, 'ipp')
    check_sbs_against_reference(out, rebuild_reference(z, out, '_noipp'), name, 'noipp')


@pytest.mark.parametrize('path', GOLDEN, ids=[fixture_name(p) for p in GOLDEN])
def test_cuda_matches_reference_golden(gen, path):
    z, kw = load(path)
    out = gen.process_frame(z['rgb'], z['depth'], StereoParams(**kw))
    check_sbs_against_reference(out, z['sbs'], fixture_name(path), 'ipp')
    check_sbs_against_reference(out, z['sbs_noipp'], fixture_name(path), 'noipp')
    # hole masks / shift indices as the reference produced them: bit-exact (stage-wise, through the C ABI)
    lib = _lib.load()
    h, w = z['rgb'].shape[:2]
    g = _lib.geometry(h, w, StereoParams(**kw))
    taps = {}
    O.process_frame(z['rgb'], z['depth'], O.Params(**kw), taps)
    outs = [np.empty((g.ss_h, g.ss_w, 3), np.uint8), np.empty((g.ss_h, g.ss_w), np.uint8), np.empty((g.ss_h, g.ss_w, 3), np.uint8),
            np.empty((g.ss_h, g.ss_w), np.uint8)]
    depth_ss = np.ascontiguousarray(taps['depth_ss'])
    _lib.check(lib.vsc_stage_warp(gen._ctx.handle, _lib.ptr(taps['rgb_stretched']), _lib.ptr(depth_ss), h, g.stretched_w, g.ss_h, g.ss_w,
                                  float(kw.get('max_disparity', 50.0)), 0, *[_lib.ptr(o) for o in outs], None))
    shape = tuple(z['mask_shape'])
    for k, side in ((1, 'left'), (3, 'right')):
        ref_mask = np.unpackbits(z['mask_' + side])[:shape[0] * shape[1]].reshape(shape)
        assert np.array_equal(outs[k], ref_mask), side


def _make_workflow(tmp_path, n, h=72, w=128):
    import cv2
    wf = tmp_path / 'wf'
    for d in ('frames', 'depth_maps', 'sbs'):
        (wf / d).mkdir(parents=True)
    cfg = {'input_video': 'in.mkv', 'output_video': 'out.mkv',
           'directories': {'frames': 'frames', 'depth_maps': 'depth_maps', 'sbs': 'sbs', 'chunks': 'chunks'},
           'stereo': {'max_disparity': 50.0, 'convergence': -10.0, 'super_sampling': 3.0, 'edge_softness': 20.0,
                      'artifact_smoothing': 1.0, 'depth_gamma': 0.2, 'sharpen': 14.0},
           'depth': {'save_16bit': True}, 'encoding': {'crf': 19, 'preset': 'slow'},
           'free_space': {'sbs_generator': 'none', 'chunk_generator': 'none'}}
    (wf / 'config.json').write_text(json.dumps(cfg))
    frames = []
    for i in range(n):
        rgb, depth = make_pair(h, w, seed=i, depth_dtype=np.uint16 if i % 2 else np.uint8)
        cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(rgb, cv2.COLOR_RGB2BGR))
        cv2.imwrite(str(wf / 'depth_maps' / (f'depth_frame_{i:06d}.tif' if i % 2 else f'depth_frame_{i:06d}.png')), depth)
        frames.append((rgb, depth))
    return wf, frames


def test_sbs_generator_cli_end_to_end(tmp_path):
    import cv2
    n = 9
    wf, frames = _make_workflow(tmp_path, n)
    # frame 3 is already done: must be skipped, not rewritten (resume rule, sbs_generator.py:178-185)
    (wf / 'sbs' / 'sbs_000003.png').write_bytes(b'sentinel')
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive', '--gpus', '1', '--slots', '3'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert f'Found: {n} frame pairs, 1 already processed, {n - 1} to process' in r.stdout
    assert (wf / 'sbs' / 'sbs_000003.png').read_bytes() == b'sentinel'
    assert sorted(p.name for p in (wf / 'sbs').iterdir()) == [f'sbs_{i:06d}.png' for i in range(n)]
    for i, (rgb, depth) in enumerate(frames):
        if i == 3:
            continue
        got = cv2.cvtColor(cv2.imread(str(wf / 'sbs' / f'sbs_{i:06d}.png'), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
        assert np.array_equal(got, O.process_frame(rgb, depth, O.Params())), i
    # second run: nothing left
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive'], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and 'All frames already processed.' in r.stdout


def test_sbs_generator_survives_an_unreadable_frame(tmp_path):
    """One corrupt frame: it is reported and skipped, every other frame is written and visible, the run ends with exit
    code 0 and a second run has nothing but that frame left (reference: sbs_generator.py:229-230)."""
    n = 10
    wf, frames = _make_workflow(tmp_path, n)
    (wf / 'frames' / 'frame_000004.png').write_bytes(b'not a png')
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive', '--gpus', '1', '--slots', '2'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert 'Error loading 000004' in r.stdout and 'Skipped 1 frame' in r.stdout
    assert sorted(p.name for p in (wf / 'sbs').iterdir()) == [f'sbs_{i:06d}.png' for i in range(n) if i != 4]


def test_sbs_generator_raw_sink_and_free_space(tmp_path):
    """--raw-sink: the frames arrive as raw rgb24 in clip order and equal the oracle's; free_space deletes inputs only
    in PNG mode after publication (checked in a second run with free_space = all)."""
    import cv2
    n = 6
    wf, frames = _make_workflow(tmp_path, n, h=64, w=96)
    sink = tmp_path / 'out.rgb'
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive', '--gpus', '1', '--raw-sink', str(sink)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    raw = np.fromfile(sink, np.uint8).reshape(n, 64, 192, 3)
    for i, (rgb, depth) in enumerate(frames):
        assert np.array_equal(raw[i], O.process_frame(rgb, depth, O.Params())), i
    cfg = json.loads((wf / 'config.json').read_text())
    cfg['free_space']['sbs_generator'] = 'all'
    (wf / 'config.json').write_text(json.dumps(cfg))
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_generator.py'), str(wf), '--no-interactive', '--gpus', '1'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert len(list((wf / 'sbs').glob('sbs_*.png'))) == n
    assert not list((wf / 'frames').iterdir()) and not list((wf / 'depth_maps').iterdir())
    got = cv2.cvtColor(cv2.imread(str(wf / 'sbs' / 'sbs_000002.png'), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
    assert np.array_equal(got, raw[2])


def test_sbs_sweep_cli(tmp_path):
    """sbs_sweep.py end to end: a 2 x 2 grid plus an invalid corner, images equal the oracle's, refusal recorded."""
    import cv2
    wf, frames = _make_workflow(tmp_path, 2, h=64, w=96)
    out = tmp_path / 'sweep'
    r = subprocess.run([sys.executable, os.path.join(PKG, 'sbs_sweep.py'), str(wf), '--frame', '0', '--out', str(out),
                        '--param', 'max_disparity=5,40', '--param', 'convergence=-50,0'], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads((out / 'sweep.json').read_text())['results']
    assert len(res) == 4
    for e in res:
        p = O.Params(**e['params'])
        if e['params']['max_disparity'] == 5.0 and e['params']['convergence'] == -50.0:
            assert e['refused'] and not (out / f"sweep_{e['index']:04d}.png").exists()     # crop window left of the view
            continue
        assert e['refused'] is None and e['ms'] > 0
        img = cv2.cvtColor(cv2.imread(str(out / f"sweep_{e['index']:04d}.png"), cv2.IMREAD_COLOR), cv2.COLOR_BGR2RGB)
        assert np.array_equal(img, O.process_frame(frames[0][0], frames[0][1], p))


def test_bench_line_contract(tmp_path):
    """bench.py on a small configuration: one JSON line with the contract's keys (value, e2e with copy bytes, roofline
    with measured kernel time, workloads, cpu_baseline of the staged reference or the port), and the launch count; and the
    --dump-outputs sample of the last timed step, whose values are the oracle's for the same frames."""
    dump = tmp_path / 'dump'
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1', '--warmup', '3', '--batch', '16', '--slots', '2',
                        '--batch-4k', '4', '--slots-4k', '1', '--no-8k', '--no-driver', '--cpu-frames', '1', '--dump-outputs', str(dump)],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, VSC_BENCH_NO_CLOCKS='1'))
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['unit'] == 'frames/s' and d['n_gpus'] == 1 and d['steps'] == 1 and d['higher_is_better'] is True and d['scaling'] == 'weak'
    assert d['value'] > 0 and d['e2e']['value'] > 0 and d['vs_baseline'] is None
    assert d['e2e']['h2d_bytes_per_step'] == 16 * (1080 * 1920 * 4) and d['e2e']['d2h_bytes_per_step'] == 16 * 1080 * 3840 * 3
    rf = d['roofline']
    assert rf['bound'] == 'hbm' and rf['kernel'].startswith('telea_') and 0 < rf['frac'] < 1 and rf['kernel_ms_per_launch'] > 0
    assert rf['algorithmic_bytes_per_launch'] == 20736000 * rf['frames_per_launch']
    assert d['gpu_launches'] > 0 and d['launches_per_frame'] < 16
    w = d['workloads']['4k']
    assert w['value'] > 0 and w['e2e']['value'] > 0 and w['roofline']['algorithmic_bytes_per_launch'] % 91238400 == 0
    assert d['cpu_baseline']['kind'] in ('reference', 'port') and d['cpu_baseline']['value'] > 0
    files = {p.name: np.load(p) for p in dump.iterdir()}
    assert sorted(files) == sorted(f'{k}_{n}.npy' for k in ('1080p', '4k') for n in ('sbs_sample', 'frames', 'sample_index'))
    assert all(a.dtype in (np.float32, np.float64) for a in files.values()) and sum(a.nbytes for a in files.values()) <= 64 << 20
    for key, (fh, fw, dt, n_distinct) in {'1080p': (1080, 1920, np.uint8, 16), '4k': (2160, 3840, np.uint16, 4)}.items():
        sample, frames, idx = (files[f'{key}_{n}.npy'] for n in ('sbs_sample', 'frames', 'sample_index'))
        assert 0 < len(frames) <= n_distinct and set(frames) <= set(range(n_distinct))
        assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < fh * 2 * fw * 3 and sample.shape == (len(frames), len(idx))
        if key == '1080p':        # one frame of the timed path against the oracle
            rgb, depth = make_pair(fh, fw, seed=int(frames[-1]), depth_dtype=dt)
            ref = O.process_frame(rgb, depth, O.Params()).reshape(-1)[idx.astype(np.int64)]
            assert np.array_equal(sample[-1], ref.astype(np.float32))
