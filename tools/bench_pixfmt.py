#!/usr/bin/env python
"""Frames/s of the output pixel formats (rgb24, yuv420p, yuv420p10le) against each other, on one GPU.

    python tools/bench_pixfmt.py [--steps 3] [--rounds 3] [--out profiles/bench_pixfmt_b200.json]

Workloads: 1080p uint8 depth (300 frames per step, 16 slots x 4 frames) and 4K uint16 depth (64 frames per step,
10 slots x 4), default stereo parameters, in the layouts sbs and half-sbs.  Per (layout, format) two legs, as bench.py
measures them: device-resident (inputs and outputs in HBM, submit_device_group) and end to end (pinned host inputs,
H2D + kernels + D2H, submit_host / collect), where the smaller yuv420p frame halves the device-to-host bytes.
One generator per workload; layout and format are switched between runs (set_layout, set_pixfmt), and the formats
alternate (rgb24, yuv420p, yuv420p10le, rgb24, ...) for `--rounds` rounds.  Bytes per frame: rgb in + depth in + the
output frame.  The GPU's name and power limit go into the output.  The 4K end-to-end figure over eight GPUs is not
measured by this tool.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'video-stereo-converter_b200')]

import numpy as np  # noqa: E402

from bench import make_frames  # noqa: E402

WORKLOADS = {
    '1080p': dict(h=1080, w=1920, dtype=np.uint8, batch=300, slots=16, group=4, distinct=48),
    '4k': dict(h=2160, w=3840, dtype=np.uint16, batch=64, slots=10, group=4, distinct=16),
}


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=10).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in out.split(',')]
        return {'gpu': name, 'power_limit': power, 'sm_max_clock': clk}
    except Exception as e:          # noqa: BLE001
        return {'gpu': None, 'error': str(e)}


LAYOUTS = ('sbs', 'half-sbs')


def out_bytes(layout, pixfmt, h, w):
    from vsc_b200.stereo_core import output_dtype, output_shape
    return int(np.prod(output_shape(layout, h, w, pixfmt))) * output_dtype(pixfmt).itemsize


def frame_bytes(layout, pixfmt, h, w, depth_itemsize):
    return h * w * 3 + h * w * depth_itemsize + out_bytes(layout, pixfmt, h, w)


def run_workload(key, steps, warmup, rounds):
    import torch
    from vsc_b200 import StereoGenerator, StereoParams, _lib
    from vsc_b200.stereo_core import PIXFMTS, output_shape
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
    d_out_max = [[torch.empty(H * W * 6, dtype=torch.uint8, device='cuda') for _ in range(group)] for _ in range(slots)]

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
                tri = [(d_rgb[f].data_ptr(), d_dep[f].data_ptr(), d_out_max[s][k].data_ptr())
                       for k, f in enumerate((step * batch + i0 + k) % n for k in range(min(group, batch - i0)))]
                gen.submit_device_group(s, tri, DT, H, W, params)
                busy.append(s)
        for s in busy:
            gen.wait(s)

    def e2e_run(nsteps, step0=0):
        free, busy, last = list(range(slots)), [], None
        for step in range(step0, step0 + nsteps):
            for i0 in range(0, batch, group):
                if not free:
                    s = gen.wait_any(busy)
                    last = gen.collect(s, copy=False)
                    busy.remove(s)
                    free.append(s)
                s = free.pop(0)
                idx = [(step * batch + i0 + k) % n for k in range(min(group, batch - i0))]
                gen.submit_host(s, [(pin_rgb[f].array, pin_dep[f].array) for f in idx], params)
                busy.append(s)
        for s in busy:
            last = gen.collect(s, copy=False)
        return last

    def timed(fn):
        torch.cuda.synchronize()
        gen.timer_begin()
        t0 = time.perf_counter()
        fn(steps, warmup)
        ms = gen.timer_end()
        wall = (time.perf_counter() - t0) * 1e3
        return ms, wall

    runs = []

    def one(layout, pixfmt):
        gen.set_layout(layout)
        gen.set_pixfmt(pixfmt)
        for s_ in range(slots):                 # pinned outputs of this layout and format, outside the timed region
            for k_ in range(group):
                gen.pinned_inputs(s_, H, W, DT, k_)
        device_run(warmup)
        ms_dev, wall_dev = timed(device_run)
        e2e_run(max(1, warmup))
        ms_e2e, wall_e2e = timed(e2e_run)
        nf = steps * batch
        r = {'layout': layout, 'pixfmt': pixfmt, 'out_shape': list(output_shape(layout, H, W, pixfmt)), 'frames': nf,
             'device_fps': round(nf / (wall_dev / 1e3), 2), 'device_ms': round(ms_dev, 2), 'device_wall_ms': round(wall_dev, 2),
             'e2e_fps': round(nf / (wall_e2e / 1e3), 2), 'e2e_wall_ms': round(wall_e2e, 2),
             'launches_per_frame': gen.last_frame_launches(0) / group,
             'bytes_per_frame': frame_bytes(layout, pixfmt, H, W, np.dtype(DT).itemsize),
             'd2h_bytes_per_frame': out_bytes(layout, pixfmt, H, W)}
        r['device_GBps'] = round(r['device_fps'] * r['bytes_per_frame'] / 1e9, 2)
        runs.append(r)
        print(f'  {key} {layout:9s} {pixfmt:12s} device {r["device_fps"]:8.1f} fps   e2e {r["e2e_fps"]:8.1f} fps',
              file=sys.stderr, flush=True)

    for _ in range(rounds):
        for layout in LAYOUTS:
            for pixfmt in PIXFMTS:
                one(layout, pixfmt)
    gen.close()
    summary = {}
    for layout in LAYOUTS:
        for pixfmt in PIXFMTS:
            mine = [r for r in runs if r['layout'] == layout and r['pixfmt'] == pixfmt]
            summary[f'{layout}/{pixfmt}'] = {
                'device_fps_median': float(np.median([r['device_fps'] for r in mine])),
                'device_fps_runs': [r['device_fps'] for r in mine],
                'e2e_fps_median': float(np.median([r['e2e_fps'] for r in mine])),
                'e2e_fps_runs': [r['e2e_fps'] for r in mine],
                'bytes_per_frame': mine[0]['bytes_per_frame'], 'd2h_bytes_per_frame': mine[0]['d2h_bytes_per_frame'],
                'launches_per_frame': mine[0]['launches_per_frame']}
        base = summary[f'{layout}/rgb24']
        for pixfmt in PIXFMTS:
            x = summary[f'{layout}/{pixfmt}']
            x['device_vs_rgb24'] = round(x['device_fps_median'] / base['device_fps_median'], 4)
            x['e2e_vs_rgb24'] = round(x['e2e_fps_median'] / base['e2e_fps_median'], 4)
    return {'workload': {k: (str(np.dtype(v)) if k == 'dtype' else v) for k, v in wl.items()}, 'steps': steps,
            'warmup_steps': warmup, 'rounds': rounds, 'summary': summary, 'runs': runs}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--steps', type=int, default=3, help='timed steps per run')
    ap.add_argument('--warmup', type=int, default=1, help='warm-up steps per run')
    ap.add_argument('--rounds', type=int, default=3, help='rounds of (rgb24, yuv420p, yuv420p10le) per layout')
    ap.add_argument('--workloads', default='1080p,4k')
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        print('bench_pixfmt: no CUDA device', file=sys.stderr)
        return 1
    res = {'tool': 'tools/bench_pixfmt.py', 'device': gpu_info(), 'torch_device_name': torch.cuda.get_device_name(0),
           'gpus_visible': torch.cuda.device_count(), 'workloads': {},
           '4k_n8_e2e': 'not measured (this tool runs one GPU)'}
    for key in args.workloads.split(','):
        res['workloads'][key] = run_workload(key, args.steps, args.warmup, args.rounds)
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
