#!/usr/bin/env python
"""Cost of the temporal depth filter (StereoGenerator.submit_window) on one GPU.

    python tools/bench_temporal.py [--steps 3] [--rounds 3] [--out profiles/bench_temporal_b200.json]

Device-resident frames/s through vsc_submit_device_window at 1080p (uint8 depth; 240 frames per step, 16 slots x 4) and
4K (uint16 depth; 64 frames per step, 10 slots x 4), default stereo and filter parameters, radius k in {0, 2, 4, 8}
(k = 0 is vsc_submit_group), the radii alternated for `--rounds` rounds on one generator.  Every submission is 4
consecutive frames mid-clip, so each frame has its full window of 2k neighbours; the depth maps are one scene shifted by
a pixel per frame, so no neighbour is cut.  A separate run with per-kernel events gives the temporal kernels' own device
time per frame (vsc_slot_kernel_times).  Also recorded: the GPU's name and power limit, and the host-to-device bytes a
host submission copies per frame beyond vsc_submit_group (2k / 4 extra depth maps).
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'video-stereo-converter_b200'), os.path.join(ROOT, 'tools')]

import numpy as np  # noqa: E402

from bench_pixfmt import gpu_info  # noqa: E402

WORKLOADS = {
    '1080p': dict(h=1080, w=1920, dtype=np.uint8, batch=240, slots=16, group=4, distinct=16),
    '4k': dict(h=2160, w=3840, dtype=np.uint16, batch=64, slots=10, group=4, distinct=8),
}
RADII = (0, 2, 4, 8)
MAPS = 40           # depth maps of the synthetic clip (>= 4 + 2 * 8)


def run_workload(key, steps, warmup, rounds):
    import torch
    from vsc_b200 import StereoGenerator, StereoParams
    from vsc_b200.synthetic import make_depth, make_rgb
    wl = WORKLOADS[key]
    H, W, DT, batch, slots, group = wl['h'], wl['w'], wl['dtype'], wl['batch'], wl['slots'], wl['group']
    params = StereoParams()
    gen = StereoGenerator('cuda:0', n_slots=slots, group_size=group)
    d_rgb = [torch.from_numpy(make_rgb(H, W, seed=i)).cuda() for i in range(wl['distinct'])]
    base = make_depth(H, W, seed=1, dtype=DT)
    d_dep = [torch.from_numpy(np.ascontiguousarray(np.roll(base, j, axis=1))).cuda() for j in range(MAPS)]
    shape = gen.output_shape(H, W)
    d_out = [[torch.empty(shape, dtype=torch.uint8, device='cuda') for _ in range(group)] for _ in range(slots)]
    torch.cuda.synchronize()

    def run(k, nsteps):
        free, busy = list(range(slots)), []
        f = 0
        for _ in range(nsteps):
            for i0 in range(0, batch, group):
                if not free:
                    s = gen.wait_any(busy)
                    gen.wait(s)
                    busy.remove(s)
                    free.append(s)
                s = free.pop(0)
                a = f % (MAPS - group - 2 * k)            # window maps a .. a + group + 2k - 1, frames from a + k
                maps = [d_dep[j].data_ptr() for j in range(a, a + group + 2 * k)]
                trip = [(d_rgb[(f + i) % len(d_rgb)].data_ptr(), d_out[s][i].data_ptr()) for i in range(group)]
                gen.submit_device_window(s, trip, maps, k, DT, H, W, params, radius=k)
                busy.append(s)
                f += group
        for s in busy:
            gen.wait(s)

    fps = {k: [] for k in RADII}
    for k in RADII:
        run(k, warmup)
    for _ in range(rounds):
        for k in RADII:
            gen.timer_begin()
            run(k, steps)
            ms = gen.timer_end()
            fps[k].append(steps * batch / (ms / 1e3))
    # the temporal kernels' own time: one submission in flight at a time, per-kernel events
    kern = {}
    gen.set_profiling(True)
    for k in RADII[1:]:
        tot, n = {}, 0
        for rep in range(8):
            maps = [d_dep[j].data_ptr() for j in range(rep, rep + group + 2 * k)]
            trip = [(d_rgb[i].data_ptr(), d_out[0][i].data_ptr()) for i in range(group)]
            gen.submit_device_window(0, trip, maps, k, DT, H, W, params, radius=k)
            gen.wait(0)
            if rep < 2:
                continue
            for name, ms in gen.kernel_times(0):
                if name.startswith('temporal_'):
                    tot[name] = tot.get(name, 0.0) + ms
            n += group
        kern[k] = {name: v / n for name, v in tot.items()}
    gen.set_profiling(False)
    gen.close()
    plane = H * W * np.dtype(DT).itemsize
    med = {k: float(np.median(v)) for k, v in fps.items()}
    out = {'h': H, 'w': W, 'depth_dtype': np.dtype(DT).name, 'slots': slots, 'group': group, 'frames_per_step': batch,
           'steps': steps, 'rounds': rounds, 'fps_rounds': {str(k): v for k, v in fps.items()},
           'fps_median': {str(k): v for k, v in med.items()},
           'frame_time_share_vs_k0': {str(k): 1.0 - med[k] / med[0] for k in RADII[1:]},
           'temporal_kernel_ms_per_frame': {str(k): v for k, v in kern.items()},
           'temporal_kernel_share_of_k0_frame_time': {str(k): sum(v.values()) / (1e3 / med[0]) for k, v in kern.items()},
           'h2d_extra_bytes_per_frame': {str(k): plane * 2 * k // group for k in RADII}}
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None, help='JSON file to write (default: print only)')
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_temporal.py measures on a CUDA device; none is available')
    res = {'gpu_info': gpu_info(), 'workloads': {}}
    for key in WORKLOADS:
        res['workloads'][key] = run_workload(key, args.steps, args.warmup, args.rounds)
        print(key, json.dumps(res['workloads'][key]['fps_median']), json.dumps(res['workloads'][key]['temporal_kernel_ms_per_frame']),
              flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_info']))


if __name__ == '__main__':
    main()
