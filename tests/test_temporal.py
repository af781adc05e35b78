"""Temporal depth stabilisation without a GPU: properties of the oracle (tests/temporal_oracle.py), the stabilisation it
gives on a synthetic clip, the Python argument checks, and the driver's window, chunking and free-space logic."""
import math

import numpy as np
import pytest

import temporal_oracle as TO
from vsc_b200.stereo_core import check_temporal
from vsc_b200.synthetic import make_depth


def _clip(n=12, h=64, w=96, seed=0, dtype=np.uint8, disc=True):
    """A static scene whose per-frame maps are min/max restretched after per-frame noise and an outlier, plus one moving
    disc.  Returns (maps, disc masks)."""
    rng = np.random.default_rng(seed)
    base = make_depth(h, w, seed, np.float64, discs=6)
    y, x = np.mgrid[0:h, 0:w]
    maps, masks = [], []
    mx = TO.max_value(dtype)
    for t in range(n):
        d = base + rng.normal(0.0, 0.02, (h, w))
        oy, ox = rng.integers(0, h - 2), rng.integers(0, w - 2)
        d[oy:oy + 2, ox:ox + 2] = rng.uniform(1.0, 1.1)                    # outlier: moves the per-frame max
        m = np.zeros((h, w), bool)
        if disc:
            m = (y - h / 2) ** 2 + (x - (8 + 3 * t)) ** 2 <= 16
            d = np.where(m, 0.95, d)
        d = (d - d.min()) / (d.max() - d.min())
        maps.append(np.rint(d * mx).astype(dtype))
        masks.append(m)
    return maps, masks


def test_weight_table():
    w = TO.weight_table(4, 6.0)
    assert w.dtype == np.float32 and w.shape == (5, 256)
    assert w[0, 0] == 1.0
    assert w[4, 0] == np.float32(math.exp(-0.5))
    assert np.all(np.diff(w, axis=1) <= 0) and np.all(np.diff(w, axis=0) <= 0)
    assert TO.weight_table(0, 6.0).shape == (1, 256)


@pytest.mark.parametrize('dtype', [np.uint8, np.uint16])
def test_lone_frame_or_radius_zero_gives_the_map(dtype):
    maps, _ = _clip(5, dtype=dtype)
    out, lo, hi = TO.temporal_depth(maps[2:3], 0, 4)
    assert (lo, hi) == (0, 0) and out.dtype == np.float32 and np.array_equal(out, maps[2].astype(np.float32))
    out, lo, hi = TO.temporal_depth(maps, 2, 0)
    assert (lo, hi) == (2, 2) and np.array_equal(out, maps[2].astype(np.float32))


def test_window_is_clipped_at_the_clip_ends():
    maps, _ = _clip(6, disc=False)
    assert TO.temporal_depth(maps, 0, 4)[1:] == (0, 4)
    assert TO.temporal_depth(maps, 5, 2)[1:] == (3, 5)
    assert TO.temporal_depth(maps, 2, 8)[1:] == (0, 5)


@pytest.mark.parametrize('kind', ['inverted', 'flat', 'unrelated'])
def test_a_cut_gives_the_truncated_window(kind):
    maps, _ = _clip(9, disc=False)
    other = {'inverted': 255 - maps[6], 'flat': np.full_like(maps[6], 77),
             'unrelated': make_depth(*maps[0].shape, seed=99, dtype=np.uint8)}[kind]
    cut = maps[:6] + [other] + maps[7:]
    out, lo, hi = TO.temporal_depth(cut, 4, 4)
    assert (lo, hi) == (0, 5)                     # frame 6 is cut, and frames 7, 8 beyond it go with it
    ref, rlo, rhi = TO.temporal_depth(maps[:6], 4, 4)
    assert (rlo, rhi) == (0, 5) and np.array_equal(out, ref)
    out2, lo2, hi2 = TO.temporal_depth(cut, 7, 4)
    assert lo2 == 7 and hi2 == 8                  # seen from the other side of the cut


def test_slope_limit_cuts():
    base = np.zeros((16, 16), np.uint8)
    base[:, 8:] = 1                                       # a faint map: aligning it to a strong one needs a > 16
    strong = (base * 200).astype(np.uint8)
    assert TO.align(base.size, *TO.plane_sums(strong), *TO.plane_sums(base), TO.cross_sum(strong, base)) is None
    assert TO.align(base.size, *TO.plane_sums(base), *TO.plane_sums(strong), TO.cross_sum(base, strong)) is not None


def test_u8_and_u16_copies_of_a_clip_give_the_same_windows():
    maps, _ = _clip(10)
    maps[7] = 255 - maps[7]
    for t in range(10):
        a = TO.temporal_depth(maps, t, 3)
        b = TO.temporal_depth([m.astype(np.uint16) * 257 for m in maps], t, 3)
        assert a[1:] == b[1:]


def _normalise(d):
    d = d.astype(np.float64)
    return (d - d.min()) / (d.max() - d.min())


def test_stabilisation_of_a_synthetic_clip():
    """After the per-frame min/max normalisation the pipeline applies, the per-pixel std over frames of the static scene
    drops below that of the raw maps, and on the disc's trail the output stays at D_t (no ghosting)."""
    maps, masks = _clip(12)
    ts = range(2, 10)
    outs = [TO.temporal_depth(maps, t, 4)[0] for t in ts]
    trail = np.any(np.stack(masks), axis=0)
    static = ~trail
    raw = np.stack([_normalise(maps[t]) for t in ts]).std(axis=0)[static].mean()
    stab = np.stack([_normalise(o) for o in outs]).std(axis=0)[static].mean()
    ratio = stab / raw
    assert ratio < 0.8, ratio
    assert ratio == pytest.approx(0.7216, abs=0.01)
    ghost = max(float(np.abs(o - maps[t].astype(np.float32))[trail].max()) for o, t in zip(outs, ts))
    assert ghost <= 6.0, ghost


def test_check_temporal():
    assert check_temporal(0, 6) == (0, 6.0) and check_temporal(8, 64.0) == (8, 64.0)
    assert check_temporal(np.int64(3), np.float32(0.5)) == (3, 0.5)
    for r, s in ((-1, 6.0), (9, 6.0), (2.0, 6.0), (True, 6.0), ('2', 6.0), (2, 0.0), (2, -1.0), (2, 64.5),
                 (2, float('nan')), (2, float('inf')), (2, None), (2, '6')):
        with pytest.raises(ValueError):
            check_temporal(r, s)


# ---- driver -----------------------------------------------------------------------------------------------------------
import json  # noqa: E402
import os  # noqa: E402
import subprocess  # noqa: E402
import sys  # noqa: E402

import cv2  # noqa: E402

from conftest import ROOT  # noqa: E402
from vsc_b200.sharder import DelayedFree, consecutive_chunks, shard_items  # noqa: E402
from vsc_b200.workflow import LayoutError, config_temporal, load_config  # noqa: E402

PKG = os.path.join(ROOT, 'video-stereo-converter_b200')
sys.path.insert(0, PKG)
import sbs_generator  # noqa: E402


def _pairs(nums):
    return [(f'f{n}', f'd{n}', f'{n:06d}') for n in nums]


def test_chunks_hold_consecutive_frames_only():
    items = _pairs(range(40))
    assert [len(c) for c in consecutive_chunks(items, 4)] == [4] * 10
    for rank in range(2):                   # --group 3 with blocks of 16: a chunk never straddles a block
        mine = shard_items(items, 2, rank)
        chunks = consecutive_chunks(mine, 3)
        assert [it for c in chunks for it in c] == mine
        for c in chunks:
            nums = [int(it[2]) for it in c]
            assert len(c) <= 3 and nums == list(range(nums[0], nums[0] + len(c)))
            assert len({n // 16 for n in nums}) == 1
    gappy = _pairs([0, 1, 2, 5, 6, 9, 10, 11, 12, 13])      # resume or missing maps leave gaps
    assert [[int(i[2]) for i in c] for c in consecutive_chunks(gappy, 4)] == [[0, 1, 2], [5, 6], [9, 10, 11, 12], [13]]
    assert consecutive_chunks([], 4) == []


class _FakeCache:
    def __init__(self, maps):
        self.maps, self.calls = maps, []

    def get(self, path, size):
        self.calls.append(path)
        return self.maps.get(path)


def test_windows_end_at_clip_ends_gaps_and_unreadable_maps():
    clip = {int(p[2]): p for p in _pairs([0, 1, 2, 3, 4, 5, 6, 8, 9, 10])}
    maps = {f'd{n}': np.full((4, 4), n, np.uint8) for n in range(11)}
    maps['d9'] = None                                         # fails to decode
    maps['d1'] = np.zeros((4, 4), np.uint16)                  # another dtype
    cache = _FakeCache(maps)
    own = lambda nums: [maps[f'd{n}'] for n in nums]          # noqa: E731
    got, first = sbs_generator.window_maps(_pairs([3, 4]), own([3, 4]), clip, 3, cache)
    assert [int(m[0, 0]) for m in got] == [2, 3, 4, 5, 6] and first == 1      # d1 ends the left side, the gap at 7 the right
    got, first = sbs_generator.window_maps(_pairs([8]), own([8]), clip, 2, cache)
    assert [int(m[0, 0]) for m in got] == [8] and first == 0                  # 7 missing, 9 unreadable
    got, first = sbs_generator.window_maps(_pairs([10]), own([10]), clip, 8, cache)
    assert [int(m[0, 0]) for m in got] == [10] and first == 0
    got, first = sbs_generator.window_maps(_pairs([0]), own([0]), {0: clip[0]}, 4, cache)
    assert len(got) == 1 and first == 0
    # resumed frames still give their maps: the window comes from the whole clip, not from the frames to do
    assert [p[2] for p in sbs_generator.neighbours(clip, 5, 4, -1)] == ['000004', '000003', '000002', '000001']


def test_depth_cache_decodes_each_map_once(tmp_path):
    import threading
    p = tmp_path / 'd.png'
    cv2.imwrite(str(p), np.arange(48, dtype=np.uint8).reshape(6, 8))
    cache = sbs_generator.DepthCache(4)
    outs = []
    ths = [threading.Thread(target=lambda: outs.append(cache.get(p, (6, 8)))) for _ in range(8)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    assert cache.decodes == 1 and all(np.array_equal(o, outs[0]) for o in outs)
    assert cache.get(tmp_path / 'missing.png', (6, 8)) is None
    assert cache.get(p, (12, 16)).shape == (12, 16)           # resized to the frame, as the loaders do


def test_delayed_free_space_deletion():
    freed = []
    gate = DelayedFree(range(10), [], 2, freed.append)
    for n in range(10):
        gate.published(n)
        assert all(g <= n - 2 or (n == 9 and g <= 9) for g in freed)
    assert freed == list(range(10))
    # resume: 0..3 done before (their inputs already gone or kept), frame 5 skipped in this run
    freed = []
    gate = DelayedFree(range(10), [0, 1, 2, 3], 2, freed.append)
    for n in (4, 6, 7, 8, 9):
        gate.published(n)
    assert freed == [8, 9]                                   # a re-run of frame 5 needs the maps of 3..7
    freed = []
    gate = DelayedFree(range(5), [], 0, freed.append)
    for n in range(5):
        gate.published(n)
        assert freed[-1] == n                                 # radius 0: at once, as without the filter


def _workflow(tmp_path, n=2, h=32, w=48, extra=None):
    from vsc_b200.synthetic import make_pair
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


def test_config_temporal_keys(tmp_path):
    assert config_temporal(load_config(_workflow(tmp_path, n=0))) == (0, 6.0)
    cfg = load_config(_workflow(tmp_path / 'g', n=0, extra={'sbs_temporal_radius': 4, 'sbs_temporal_sigma': 3}))
    assert config_temporal(cfg) == (4, 3.0)
    for i, bad in enumerate(({'sbs_temporal_radius': 9}, {'sbs_temporal_radius': -1}, {'sbs_temporal_radius': 2.5},
                             {'sbs_temporal_radius': '4'}, {'sbs_temporal_radius': True}, {'sbs_temporal_sigma': 0},
                             {'sbs_temporal_sigma': 65}, {'sbs_temporal_sigma': None})):
        with pytest.raises(LayoutError):
            load_config(_workflow(tmp_path / f'bad{i}', n=0, extra=bad))


def test_cli_temporal_flags():
    p = sbs_generator.build_parser()
    a = p.parse_args(['wf'])
    assert a.temporal_radius is None and a.temporal_sigma is None
    a = p.parse_args(['wf', '--temporal-radius', '4', '--temporal-sigma', '2.5'])
    assert (a.temporal_radius, a.temporal_sigma) == (4, 2.5)


@pytest.mark.parametrize('args,extra,word', [(['--temporal-radius', '9'], None, 'radius'),
                                             (['--temporal-radius', '-1'], None, 'radius'),
                                             (['--temporal-sigma', '0'], None, 'sigma'),
                                             (['--temporal-sigma', '100'], None, 'sigma'),
                                             ([], {'sbs_temporal_radius': 12}, 'sbs_temporal_radius'),
                                             ([], {'sbs_temporal_sigma': -2}, 'sbs_temporal_sigma')])
def test_cli_refuses_bad_temporal_values_with_exit_2(tmp_path, args, extra, word):
    wf = _workflow(tmp_path, extra=extra)
    r = _run(wf, '--no-interactive', *args)
    assert r.returncode == 2 and r.stdout.startswith('ERROR:') and word in r.stdout, (r.stdout, r.stderr)
    assert not list((wf / 'sbs').iterdir())
    r = _run(wf, '--temporal-radius', 'two')
    assert r.returncode == 2 and 'invalid int' in r.stderr


@pytest.mark.parametrize('flag,cfg,want', [(None, None, (0, 6.0)), ('3', None, (3, 6.0)), (None, 5, (5, 6.0)), ('2', 5, (2, 6.0))])
def test_torchrun_branch_passes_the_temporal_filter(tmp_path, monkeypatch, flag, cfg, want):
    import torch
    import torch.distributed as dist
    from vsc_b200 import sharder
    wf = _workflow(tmp_path, extra={'sbs_temporal_radius': cfg} if cfg else None)
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
    argv = [str(wf), '--no-interactive'] + (['--temporal-radius', flag] if flag else [])
    assert sbs_generator.main(argv) == 0
    assert calls and calls[0]['temporal'] == want and len(calls[0]['clip']) == 2
