#!/usr/bin/env python
"""Frames/s and file sizes of the GPU PNG encoding (StereoGenerator(..., encode='png')) against raw rgb24, on one GPU.

    python tools/bench_png.py [--steps 3] [--rounds 3] [--out profiles/bench_png_b200.json]

Pipeline legs, layout sbs, default stereo parameters: 1080p uint8 depth (300 frames per step, 16 slots x 4 frames) and
4K uint16 depth (64 frames per step, 10 slots x 4).  Per encoding two legs as bench.py measures them: device-resident
(inputs and outputs in HBM, submit_device_group) and end to end (pinned host inputs; raw: H2D + kernels + D2H of the
frame; PNG: the device writes the file straight into the pinned output).  Raw and PNG alternate for `--rounds` rounds on
one generator (set_encode between runs).
Driver leg: sbs_generator.process_shard writing sbs_*.png for the 192 real 1080p PNG pairs of bench.py's driver leg,
with the cv2 encoder and with the GPU encoder, alternated, each on a generator that has seen the clip's first 24 frames.
Sizes: the GPU files of 16 distinct 1080p SBS frames against cv2.imencode at its defaults and against the zlib Z_RLE
model (tests/png_oracle.model_size).  The GPU's name and power limit go into the output.
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time
from pathlib import Path

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'video-stereo-converter_b200'), os.path.join(ROOT, 'tests')]

import numpy as np  # noqa: E402

from bench import make_frames  # noqa: E402
from bench_pixfmt import WORKLOADS, gpu_info  # noqa: E402

ENCODINGS = (None, 'png')


def run_workload(key, steps, warmup, rounds):
    import torch
    from vsc_b200 import StereoGenerator, StereoParams, _lib
    from vsc_b200.stereo_core import encoded_capacity
    wl = WORKLOADS[key]
    H, W, DT, batch, slots, group = wl['h'], wl['w'], wl['dtype'], wl['batch'], wl['slots'], wl['group']
    params = StereoParams()
    gen = StereoGenerator('cuda:0', n_slots=slots, group_size=group)
    frames = make_frames(wl['distinct'], H, W, DT)
    n = len(frames)
    d_rgb = [torch.from_numpy(r).cuda() for r, _ in frames]
    d_dep = [torch.from_numpy(d).cuda() for _, d in frames]
    pin_rgb = [_lib.PinnedBuffer((H, W, 3), np.uint8) for _ in range(n)]
    pin_dep = [_lib.PinnedBuffer((H, W), DT) for _ in range(n)]
    for i, (r, d) in enumerate(frames):
        np.copyto(pin_rgb[i].array, r)
        np.copyto(pin_dep[i].array, d)
    cap = encoded_capacity('sbs', H, W)
    d_out = [[torch.empty(cap, dtype=torch.uint8, device='cuda') for _ in range(group)] for _ in range(slots)]
    sizes = {}

    def device_run(nsteps, step0=0):
        free, busy = list(range(slots)), []
        for step in range(step0, step0 + nsteps):
            for i0 in range(0, batch, group):
                if not free:
                    s = gen.wait_any(busy)
                    gen.wait(s)
                    busy.remove(s)
                    free.append(s)
                s = free.pop(0)
                tri = [(d_rgb[f].data_ptr(), d_dep[f].data_ptr(), d_out[s][k].data_ptr())
                       for k, f in enumerate((step * batch + i0 + k) % n for k in range(min(group, batch - i0)))]
                gen.submit_device_group(s, tri, DT, H, W, params)
                busy.append(s)
        for s in busy:
            gen.wait(s)

    def e2e_run(nsteps, step0=0):
        free, busy = list(range(slots)), []

        def harvest(s):
            outs = gen.collect(s, copy=False)
            if gen.encode:
                for o in (outs if isinstance(outs, list) else [outs]):
                    sizes.setdefault(key, []).append(int(o.size))
        for step in range(step0, step0 + nsteps):
            for i0 in range(0, batch, group):
                if not free:
                    s = gen.wait_any(busy)
                    harvest(s)
                    busy.remove(s)
                    free.append(s)
                s = free.pop(0)
                idx = [(step * batch + i0 + k) % n for k in range(min(group, batch - i0))]
                gen.submit_host(s, [(pin_rgb[f].array, pin_dep[f].array) for f in idx], params)
                busy.append(s)
        for s in busy:
            harvest(s)

    def timed(fn):
        torch.cuda.synchronize()
        gen.timer_begin()
        t0 = time.perf_counter()
        fn(steps, warmup)
        ms = gen.timer_end()
        return ms, (time.perf_counter() - t0) * 1e3

    runs = []
    for _ in range(rounds):
        for enc in ENCODINGS:
            gen.set_encode(enc)
            for s_ in range(slots):
                for k_ in range(group):
                    gen.pinned_inputs(s_, H, W, DT, k_)
            device_run(warmup)
            ms_dev, wall_dev = timed(device_run)
            e2e_run(max(1, warmup))
            sizes.pop(key, None)
            ms_e2e, wall_e2e = timed(e2e_run)
            nf = steps * batch
            r = {'encode': enc or 'raw', 'frames': nf, 'device_fps': round(nf / (wall_dev / 1e3), 2),
                 'device_ms': round(ms_dev, 2), 'e2e_fps': round(nf / (wall_e2e / 1e3), 2),
                 'launches_per_frame': gen.last_frame_launches(0) / group}
            if enc:
                r['mean_file_bytes'] = float(np.mean(sizes[key]))
            runs.append(r)
            print(f'  {key} {enc or "raw":4s} device {r["device_fps"]:8.1f} fps   e2e {r["e2e_fps"]:8.1f} fps',
                  file=sys.stderr, flush=True)
    gen.close()
    summary = {}
    for enc in ENCODINGS:
        mine = [r for r in runs if r['encode'] == (enc or 'raw')]
        summary[enc or 'raw'] = {'device_fps_median': float(np.median([r['device_fps'] for r in mine])),
                                 'device_fps_runs': [r['device_fps'] for r in mine],
                                 'e2e_fps_median': float(np.median([r['e2e_fps'] for r in mine])),
                                 'e2e_fps_runs': [r['e2e_fps'] for r in mine],
                                 'launches_per_frame': mine[0]['launches_per_frame']}
    for k in ('device', 'e2e'):
        summary['png'][f'{k}_vs_raw'] = round(summary['png'][f'{k}_fps_median'] / summary['raw'][f'{k}_fps_median'], 4)
    summary['png']['mean_file_bytes'] = float(np.mean([r['mean_file_bytes'] for r in runs if r['encode'] == 'png']))
    summary['raw']['frame_bytes'] = H * 2 * W * 3
    return {'workload': {k: (str(np.dtype(v)) if k == 'dtype' else v) for k, v in wl.items()}, 'steps': steps,
            'warmup_steps': warmup, 'rounds': rounds, 'summary': summary, 'runs': runs}


def driver_leg(rounds, n_frames=192):
    """sbs_*.png files through process_shard with the cv2 and the GPU encoder (bench.py's driver workflow)."""
    from concurrent.futures import ThreadPoolExecutor
    import cv2
    import sbs_generator
    from vsc_b200 import StereoGenerator, StereoParams
    from vsc_b200.sharder import InOrderPublisher
    wl = WORKLOADS['1080p']
    H, W = wl['h'], wl['w']
    base = '/dev/shm' if os.path.isdir('/dev/shm') and shutil.disk_usage('/dev/shm').free > (6 << 30) else None
    wf = Path(tempfile.mkdtemp(prefix='vsc_bench_png_', dir=base))
    try:
        for d in ('frames', 'depth_maps', 'sbs'):
            (wf / d).mkdir()
        distinct = make_frames(16, H, W, wl['dtype'], seed0=500)
        cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)

        def write(i):
            rgb, depth = distinct[i % len(distinct)]
            cv2.imwrite(str(wf / 'frames' / f'frame_{i:06d}.png'), cv2.cvtColor(rgb, cv2.COLOR_RGB2BGR), [cv2.IMWRITE_PNG_COMPRESSION, 1])
            cv2.imwrite(str(wf / 'depth_maps' / f'depth_frame_{i:06d}.png'), depth, [cv2.IMWRITE_PNG_COMPRESSION, 1])
        with ThreadPoolExecutor(max_workers=cores) as ex:
            list(ex.map(write, range(n_frames)))
        pairs = [(wf / 'frames' / f'frame_{i:06d}.png', wf / 'depth_maps' / f'depth_frame_{i:06d}.png', f'{i:06d}') for i in range(n_frames)]
        io_threads = max(2, cores - 2)
        gens = {e: StereoGenerator('cuda:0', n_slots=6, group_size=4, encode='png' if e == 'gpu' else None) for e in ('cv2', 'gpu')}
        out = {'workload': f'{n_frames} files {W}x{H} PNG + 8-bit PNG depth (16 distinct synthetic frames), default params',
               'io_threads': io_threads, 'slots': 6, 'frames_per_slot': 4, 'runs': []}
        try:
            for e, g in gens.items():
                sbs_generator.process_shard(pairs[:24], wf / 'sbs', StereoParams(), 0, 6, io_threads, 'none', True, gen=g,
                                            png_encoder=e)
                for p in (wf / 'sbs').iterdir():
                    p.unlink()
            for _ in range(rounds):
                for e, g in gens.items():
                    pub = InOrderPublisher([str(wf / 'sbs' / f'sbs_{p[2]}.png') for p in pairs])
                    t0 = time.perf_counter()
                    n = sbs_generator.process_shard(pairs, wf / 'sbs', StereoParams(), 0, 6, io_threads, 'none', True, gen=g,
                                                    png_encoder=e)
                    ok = pub.run(timeout_s=60)
                    dt = time.perf_counter() - t0
                    nbytes = sum(p.stat().st_size for p in (wf / 'sbs').iterdir())
                    out['runs'].append({'encoder': e, 'fps': round(n / dt, 2), 'frames': n, 'complete': bool(ok),
                                        'seconds': round(dt, 3), 'mean_file_bytes': nbytes / max(n, 1)})
                    print(f'  driver {e:4s} {n / dt:8.1f} fps', file=sys.stderr, flush=True)
                    shutil.rmtree(wf / 'sbs')
                    (wf / 'sbs').mkdir()
        finally:
            for g in gens.values():
                g.close()
        for e in ('cv2', 'gpu'):
            out[e] = {'fps_median': float(np.median([r['fps'] for r in out['runs'] if r['encoder'] == e])),
                      'mean_file_bytes': float(np.mean([r['mean_file_bytes'] for r in out['runs'] if r['encoder'] == e]))}
        return out
    finally:
        shutil.rmtree(wf, ignore_errors=True)


def sizes_leg():
    """GPU file bytes of 16 distinct 1080p SBS frames against cv2.imencode (defaults) and the zlib model."""
    import cv2
    import png_oracle as PN
    from vsc_b200 import StereoGenerator
    wl = WORKLOADS['1080p']
    frames = make_frames(16, wl['h'], wl['w'], wl['dtype'], seed0=500)
    g = StereoGenerator('cuda:0', n_slots=4)
    try:
        raw = g.process_batch(frames)
        g.set_encode('png')
        files = g.process_batch(frames)
    finally:
        g.close()
    rows = []
    for r, f in zip(raw, files):
        PN.check_png(f, r)
        t0 = time.perf_counter()
        ok, ref = cv2.imencode('.png', cv2.cvtColor(r, cv2.COLOR_RGB2BGR))
        t_cv2 = time.perf_counter() - t0
        rows.append({'gpu_bytes': int(f.size), 'cv2_bytes': int(ref.size), 'model_bytes': PN.model_size(r),
                     'cv2_encode_ms_one_core': round(t_cv2 * 1e3, 1)})
    return {'frames': len(rows), 'gpu_vs_cv2_mean': float(np.mean([x['gpu_bytes'] / x['cv2_bytes'] for x in rows])),
            'gpu_vs_model_mean': float(np.mean([x['gpu_bytes'] / x['model_bytes'] for x in rows])),
            'gpu_vs_cv2_max': float(np.max([x['gpu_bytes'] / x['cv2_bytes'] for x in rows])),
            'gpu_vs_model_max': float(np.max([x['gpu_bytes'] / x['model_bytes'] for x in rows])), 'per_frame': rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=3, help='timed steps per run')
    ap.add_argument('--warmup', type=int, default=1, help='warm-up steps per run')
    ap.add_argument('--rounds', type=int, default=3, help='rounds of (raw, png)')
    ap.add_argument('--workloads', default='1080p,4k')
    ap.add_argument('--no-driver', action='store_true')
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print('bench_png: no CUDA device', file=sys.stderr)
        return 1
    res = {'tool': 'tools/bench_png.py', 'device': gpu_info(), 'torch_device_name': torch.cuda.get_device_name(0),
           'gpus_visible': torch.cuda.device_count(), 'workloads': {}}
    for key in args.workloads.split(','):
        res['workloads'][key] = run_workload(key, args.steps, args.warmup, args.rounds)
    res['sizes_1080p_sbs'] = sizes_leg()
    if not args.no_driver:
        res['driver_png_files'] = driver_leg(args.rounds)
    res['device_after'] = gpu_info()
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')
    print(text)
    return 0


if __name__ == '__main__':
    sys.exit(main())
