#!/usr/bin/env python
"""bench.py — SBS frames/s of the B200 hot path (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[1]): a 1080p synthetic clip, uint8 depth, default config.json stereo
parameters; a "step" is one pass of the hot path over one batch of `--batch` frames.  Frames are independent, so with
N GPUs every rank processes its own frame range (no collective; "scaling": "weak") and the value is total frames /
max-over-ranks device time.  The K timed steps are K consecutive batches of ONE continuous clip: they overlap in the
slot pipeline the way consecutive seconds of a video do, and the timed region is bracketed by a barrier + full drain
+ synchronize on both sides (pipeline fill and drain are inside it).

  value  frames/s with the inputs already resident in HBM (vsc_submit_device_group), timed with CUDA events across all
         slot streams (vsc_timer_begin/end)
  e2e    frames/s through the public StereoGenerator submit / collect API with HOST buffers: every frame's H2D copy
         (from pinned host memory, where a decoder would leave it) and every SBS frame's D2H copy are inside the timed
         region; the host sleeps in vsc_wait_any between submissions
  roofline      dominant kernel: algorithmic bytes per frame (SURVEY.md 8(d)) / its mean device time (CUDA events on
                its stream), against MEASURED_PEAKS.json hbm_gbs; `in_load_ms_per_launch` is the same kernel's
                duration with the pipeline full
  workloads     the same measurements for BASELINE.json configs[2] / [3]: the 4K (3840x2160, 16-bit depth) clip,
                frame-sharded over the N GPUs like the headline; and for one corner of configs[4]: 8K VR frames with
                maximum disparity and aggressive hole filling (16 frames per step)
  driver        frames/s of the drop-in frame loop on a synthetic workflow directory of real PNG files (rank 0, N = 1)
  cpu_baseline  the reference's CPU path timed on this box's host cores, bounded sample (rank 0, N = 1 only)
--impl reference times the reference's own CPU implementation alone: the UNMODIFIED helper/stereo_core.py staged
under oracle/_ref by oracle/make_ref.py (cpu_baseline.kind "reference"; every timed step one full 1080p frame), or,
where that copy is absent, the oracle's C port of it (kind "port").

--dump-outputs DIR writes, after the timed steps, what the device-resident leg of every workload returned in its last
timed step (rank 0): `<workload>_sbs_sample.npy` (float32 [frames, DUMP_SAMPLES], the SBS uint8 values at fixed seeded
positions of each distinct frame of that step), `<workload>_frames.npy` (the rows' distinct synthetic frames, i.e. their
make_pair seeds) and `<workload>_sample_index.npy` (the positions, flat indices into the [H, 2W, 3] frame).  Inputs and
positions depend on the arguments only, so two builds run with the same arguments can be compared value for value.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')   # one hardware queue per frame slot (before CUDA init)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(ROOT, 'video-stereo-converter_b200')]

import numpy as np  # noqa: E402

WORKLOADS = {
    # distinct frames are cycled; together they exceed the 126 MB L2 (48 x 8.3 MB, 16 x 41 MB of inputs)
    '1080p': dict(h=1080, w=1920, dtype=np.uint8, distinct=48,
                  metric='SBS frames/sec (1080p, default stereo params)',
                  name='1080p (1920x1080) synthetic clip, uint8 depth, default config.json stereo params'),
    '4k': dict(h=2160, w=3840, dtype=np.uint16, distinct=16,
               metric='SBS frames/sec (4K, 16-bit depth, default stereo params)',
               name='4K (3840x2160) synthetic clip, uint16 depth, full-width SBS, default config.json stereo params'),
    # BASELINE.json configs[4]: one corner of the sbs_tester sweep (sbs_tester.py:356-362) on 8K VR frames - maximum
    # disparity, convergence at its limit, no edge softening (sharp depth edges: wide disocclusions) and the largest
    # artifact smoothing (15x15 bilateral window); super_sampling 1, the setting the CPU side can still check
    '8k': dict(h=3840, w=7680, dtype=np.uint16, distinct=6,
               metric='SBS frames/sec (8K VR 7680x3840, max disparity, aggressive hole filling)',
               name='8K VR (7680x3840) synthetic frames, uint16 depth, max_disparity=100 convergence=-50 super_sampling=1 '
                    'edge_softness=0 artifact_smoothing=5 depth_gamma=1 sharpen=14 (sbs_tester sweep corner)',
               params=dict(max_disparity=100.0, convergence=-50.0, super_sampling=1.0, edge_softness=0.0, artifact_smoothing=5.0,
                           depth_gamma=1.0, sharpen=14.0)),
}


def algorithmic_bytes(h, w, depth_itemsize):
    """SURVEY.md 8(d): rgb in + depth in + SBS out, per frame."""
    return h * w * 3 + h * w * depth_itemsize + h * 2 * w * 3


def hbm_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.index, self.samples, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        if os.environ.get('VSC_BENCH_NO_CLOCKS'):
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace('.', '').isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i].lower() == 'active'})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(self.samples)}


def make_frames(n, h, w, dtype, seed0=0):
    from vsc_b200.synthetic import make_pair
    return [make_pair(h, w, seed0 + i, dtype) for i in range(n)]


# 1 % of a 1080p SBS frame; at most 48 + 16 + 6 distinct frames of the three workloads: 37 MB of float32 samples plus
# 3 MB of positions, inside the 64 MB a dump may take
DUMP_SAMPLES = 1 << 17
DUMP_SEED = 20240


def dump_outputs(dump_dir, key, outs):
    """Write a fixed, seeded sample of the SBS frames `outs` ({frame index: uint8 [H, 2W, 3] CUDA tensor})."""
    import torch
    frames = sorted(outs)
    n = outs[frames[0]].numel()
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_SAMPLES), replace=False))
    d_idx = torch.from_numpy(idx).to(outs[frames[0]].device)
    sample = torch.stack([outs[f].reshape(-1)[d_idx] for f in frames]).float().cpu().numpy()
    os.makedirs(dump_dir, exist_ok=True)
    np.save(os.path.join(dump_dir, f'{key}_sbs_sample.npy'), sample)
    np.save(os.path.join(dump_dir, f'{key}_frames.npy'), np.array(frames, np.float64))
    np.save(os.path.join(dump_dir, f'{key}_sample_index.npy'), idx.astype(np.float64))


# ------------------------------------------------------------------------------------------------
def run_workload(key, batch, slots, group, steps, warmup, rank, world, local_rank, dist, profile, dump_dir=None):
    """Device-resident leg, end-to-end leg and (rank 0) the per-kernel profile of one workload."""
    import torch
    from vsc_b200 import StereoGenerator, StereoParams, _lib
    wl = WORKLOADS[key]
    H, W, DT = wl['h'], wl['w'], wl['dtype']
    params = StereoParams(**wl.get('params', {}))
    gen = StereoGenerator(f'cuda:{local_rank}', n_slots=slots, group_size=group)
    n_distinct = min(wl['distinct'], max(batch, slots))
    frames = make_frames(n_distinct, H, W, DT, seed0=rank * 1000)          # this rank's frame range of the synthetic clip
    d_rgb = [torch.from_numpy(r).cuda() for r, _ in frames]
    d_dep = [torch.from_numpy(d).cuda() for _, d in frames]
    d_out = [[torch.empty((H, 2 * W, 3), dtype=torch.uint8, device='cuda') for _ in range(group)] for _ in range(slots)]
    # the e2e leg's inputs live in pinned host memory, where a decoder / the extractor hand-off would leave them
    pin_rgb = [_lib.PinnedBuffer((H, W, 3), np.uint8) for _ in range(n_distinct)]
    pin_dep = [_lib.PinnedBuffer((H, W), DT) for _ in range(n_distinct)]
    for i, (r, d) in enumerate(frames):
        np.copyto(pin_rgb[i].array, r)
        np.copyto(pin_dep[i].array, d)
    for s_ in range(slots):          # pinned output buffers of every slot, allocated outside the timed region
        for k_ in range(group):
            gen.pinned_inputs(s_, H, W, DT, k_)
    torch.cuda.synchronize()

    class Pipe:
        def __init__(self):
            self.free, self.busy, self.last = list(range(slots)), [], None

    written = {}        # (slot, k) -> (step, frame) last submitted into d_out[slot][k]

    def device_step(step, pipe):
        """one batch, inputs resident in HBM; a finished slot is reused at once (no head-of-line blocking);
        every submission carries `group` frames that share the slot's stream and one hole-filling launch"""
        for i0 in range(0, batch, group):
            if not pipe.free:
                s = gen.wait_any(pipe.busy)
                gen.wait(s)
                pipe.busy.remove(s)
                pipe.free.append(s)
            s = pipe.free.pop(0)
            tri = []
            for k in range(min(group, batch - i0)):
                f = (step * batch + i0 + k) % n_distinct
                tri.append((d_rgb[f].data_ptr(), d_dep[f].data_ptr(), d_out[s][k].data_ptr()))
                written[(s, k)] = (step, f)
            gen.submit_device_group(s, tri, DT, H, W, params)
            pipe.busy.append(s)

    def device_drain(pipe):
        for s in pipe.busy:
            gen.wait(s)
        pipe.free += pipe.busy
        pipe.busy = []

    e2e_reads = []

    def e2e_step(step, pipe):
        for i0 in range(0, batch, group):
            if not pipe.free:
                s = gen.wait_any(pipe.busy)
                pipe.last = gen.collect(s, copy=False)
                pipe.busy.remove(s)
                pipe.free.append(s)
            s = pipe.free.pop(0)
            idx = [(step * batch + i0 + k) % n_distinct for k in range(min(group, batch - i0))]
            gen.submit_host(s, [(pin_rgb[f].array, pin_dep[f].array) for f in idx], params)
            pipe.busy.append(s)
        if pipe.last is not None:        # host read of the newest finished SBS frame (pinned, already transferred)
            last = pipe.last[-1] if isinstance(pipe.last, list) else pipe.last
            e2e_reads.append(int(last[0, 0, 0]))

    def e2e_drain(pipe):
        for s in pipe.busy:
            pipe.last = gen.collect(s, copy=False)
        pipe.free += pipe.busy
        pipe.busy = []
        last = pipe.last[-1] if isinstance(pipe.last, list) else pipe.last
        e2e_reads.append(int(last[0, 0, 0]))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, drain, nsteps):
        pipe = Pipe()
        barrier()
        gen.timer_begin()
        t0 = time.perf_counter()
        for k in range(nsteps):
            fn(k, pipe)
        drain(pipe)
        ms = gen.timer_end()
        wall = (time.perf_counter() - t0) * 1e3
        barrier()
        if dist is not None:
            t = torch.tensor([ms, wall], device='cuda', dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1])
        return ms, wall

    wp = Pipe()
    for k in range(warmup):
        device_step(k, wp)
    device_drain(wp)
    launches_per_frame = gen.last_frame_launches(0) / group
    written.clear()
    with ClockSampler(local_rank) as clk:
        ms_dev, wall_dev = timed(device_step, device_drain, steps)
    if dump_dir is not None and rank == 0:
        # d_out is reused within a step: the last step's frames whose buffers still hold them (with the default
        # arguments, every distinct frame)
        dump_outputs(dump_dir, key, {f: d_out[s][k] for (s, k), (st, f) in written.items() if st == steps - 1})
    wp = Pipe()
    for k in range(max(1, warmup // 2)):
        e2e_step(k, wp)
    e2e_drain(wp)
    ms_e2e, wall_e2e = timed(e2e_step, e2e_drain, steps)

    # per-kernel times for the roofline (separate, untimed passes with event pairs around every launch): first one slot
    # submission in flight at a time ("solo"), then with every slot busy ("in load", the regime `value` is measured in)
    kt, kt_load = {}, {}
    if rank == 0 and profile:
        gen.set_profiling(True)

        def tri_for(i, s):
            return [(d_rgb[(i * group + k) % n_distinct].data_ptr(), d_dep[(i * group + k) % n_distinct].data_ptr(),
                     d_out[s][k].data_ptr()) for k in range(group)]

        def harvest(dst, s):
            per = {}
            for name, t in gen.kernel_times(s):
                per[name] = per.get(name, 0.0) + t / group
            for name, t in per.items():
                dst.setdefault(name, []).append(t)
        for i in range(6):
            gen.submit_device_group(0, tri_for(i, 0), DT, H, W, params)
            gen.wait(0)
            if i >= 2:
                harvest(kt, 0)
        for rnd in range(3):
            for s in range(slots):
                gen.submit_device_group(s, tri_for(rnd * slots + s, s), DT, H, W, params)
            for s in range(slots):
                gen.wait(s)
                if rnd >= 1:
                    harvest(kt_load, s)
        gen.set_profiling(False)
    frames_total = batch * steps * world
    bytes_frame = algorithmic_bytes(H, W, np.dtype(DT).itemsize)
    in_bytes = H * W * 3 + H * W * np.dtype(DT).itemsize
    out_bytes = H * 2 * W * 3
    res = None
    if rank == 0:
        peak, peak_src = hbm_peak()
        fps, fps_e2e = frames_total / (ms_dev * 1e-3), frames_total / (ms_e2e * 1e-3)
        res = {
            'metric': wl['metric'], 'value': fps, 'unit': 'frames/s', 'ms_per_step': ms_dev / steps,
            'config': {'workload': wl['name'], 'frames_per_step_per_gpu': batch, 'slots_in_flight': slots, 'frames_per_slot': group,
                       'distinct_frames': n_distinct, 'l2_policy': 'inputs larger than L2 (%d distinct frames cycled)' % n_distinct,
                       'sharding': 'frame-range, no collective'},
            'e2e': {'value': fps_e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': batch * in_bytes, 'd2h_bytes_per_step': batch * out_bytes,
                    'ms_per_step': ms_e2e / steps, 'h2d_gbs_per_rank': fps_e2e / world * in_bytes / 1e9,
                    'd2h_gbs_per_rank': fps_e2e / world * out_bytes / 1e9,
                    'host_side': 'inputs pre-staged in pinned host memory, no per-frame host copy; the submitting thread sleeps in vsc_wait_any'},
            'gpu_launches': int(round(launches_per_frame * batch * steps)), 'launches_per_frame': launches_per_frame,
            'clocks': clk.summary(), 'wall_ms': {'device_leg': wall_dev, 'e2e_leg': wall_e2e},
            'whole_path': {'achieved': fps / world * bytes_frame / 1e9, 'frac': fps / world * bytes_frame / 1e9 / peak, 'unit': 'GB/s'},
        }
        if kt:
            per_kernel = {k: float(np.mean(v)) for k, v in kt.items()}   # device ms per frame, one slot submission in flight
            per_load = {k: float(np.mean(v)) for k, v in kt_load.items()}
            grp = lambda k: group if k.startswith('telea_') else 1       # hole-filling kernels: one launch per slot submission
            frame_serial = float(sum(per_kernel.values()))
            dom = max(per_kernel, key=per_kernel.get)
            achieved = bytes_frame / (per_kernel[dom] * 1e-3) / 1e9
            traffic = None
            try:
                with open(os.path.join(ROOT, 'profiles', 'dominant_kernel_traffic.json')) as f:
                    tj = json.load(f)
                    if tj.get('kernel') == dom and tj.get('workload', '1080p') == key:
                        traffic = tj.get('dram_bytes_per_launch')
            except Exception:
                pass
            res['roofline'] = {'bound': 'hbm', 'kernel': dom, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                               'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                               'algorithmic_bytes_per_launch': bytes_frame * grp(dom), 'frames_per_launch': grp(dom),
                               'kernel_ms_per_launch': per_kernel[dom] * grp(dom), 'kernel_ms_per_frame': per_kernel[dom],
                               'in_load_ms_per_launch': per_load.get(dom, 0.0) * grp(dom) or None,
                               'share_of_serial_frame': per_kernel[dom] / frame_serial if frame_serial else None,
                               'whole_path': res['whole_path']}
            res['kernel_ms_per_frame'] = {k: round(v, 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1])}
            res['kernel_ms_per_frame_in_load'] = {k: round(v, 4) for k, v in sorted(per_load.items(), key=lambda kv: -kv[1])}
    gen.close()
    for b in pin_rgb + pin_dep:
        b.free()
    del d_rgb, d_dep, d_out
    torch.cuda.empty_cache()
    return res


def run_ours(args, rank, world, local_rank):
    import torch
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dump = args.dump_outputs
    head = run_workload('1080p', args.batch, args.slots, args.group, args.steps, args.warmup, rank, world, local_rank, dist, True, dump)
    extra = None
    if not args.no_4k:
        extra = run_workload('4k', args.batch_4k, args.slots_4k, args.group, args.steps, args.warmup, rank, world, local_rank, dist, True,
                             dump)
    sweep = None
    if not args.no_8k:
        sweep = run_workload('8k', 16, 4, 2, args.steps, args.warmup, rank, world, local_rank, dist, True, dump)
    out = None
    if rank == 0:
        out = {'metric': head['metric'], 'value': head['value'], 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
               'warmup': args.warmup, 'ms_per_step': head['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
               'vs_baseline': None, 'dtype': 'u8/f32', 'data': 'synthetic'}
        out.update({k: v for k, v in head.items() if k not in ('metric', 'value', 'unit', 'ms_per_step', 'whole_path')})
        if extra is not None:
            out['workloads'] = {'4k': extra}
        if sweep is not None:
            out.setdefault('workloads', {})['8k'] = sweep
        if world == 1 and not args.no_driver:
            try:
                out['driver'] = driver_fps()
            except Exception as e:       # the kernels' numbers must not depend on the file-I/O demonstration
                out['driver'] = {'error': f'{type(e).__name__}: {e}'}
        if world == 1 and not args.no_cpu_baseline:
            out['cpu_baseline'] = cpu_baseline(sample_frames=args.cpu_frames)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return out


def driver_fps(n_frames=192, n_png=48):
    """The drop-in frame loop (video-stereo-converter_b200/sbs_generator.py: process_shard) on a synthetic workflow
    directory of real files, rank 0 / N = 1 only: PNG decode of frames and depth maps by the loader pool, grouped
    pinned submissions, and either the raw rgb24 hand-off to an encoder (--raw-sink) or sbs_*.png files.  Wall clock
    around process_shard with a generator that has already seen the clip's first 24 frames (steady state of a long clip)."""
    import shutil
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    from pathlib import Path
    import cv2
    sys.path.insert(0, os.path.join(ROOT, 'video-stereo-converter_b200'))
    import sbs_generator
    from vsc_b200 import StereoParams
    from vsc_b200.sharder import InOrderPublisher, RawFrameSink
    wl = WORKLOADS['1080p']
    H, W = wl['h'], wl['w']
    base = '/dev/shm' if os.path.isdir('/dev/shm') and shutil.disk_usage('/dev/shm').free > (6 << 30) else None
    wf = Path(tempfile.mkdtemp(prefix='vsc_bench_wf_', dir=base))
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
        out = {'workload': f'{n_frames} files {W}x{H} PNG + 8-bit PNG depth (16 distinct synthetic frames), default params',
               'io_threads': io_threads, 'slots': 6, 'frames_per_slot': 4}
        from vsc_b200 import StereoGenerator
        gen = StereoGenerator('cuda:0', n_slots=6, group_size=4)      # one generator for the whole clip, as in the CLI
        try:
            warm = pairs[:24]          # first frames of a clip: context, buffers and page-locked staging come into being
            ws = RawFrameSink(str(wf / 'warm.rgb'), len(warm), H, 2 * W)
            sbs_generator.process_shard(warm, wf / 'sbs', StereoParams(), 0, 6, io_threads, 'none', True, None, ws,
                                        {p[2]: i for i, p in enumerate(warm)}, 4, gen)
            ws.close()
            os.remove(wf / 'warm.rgb')
            sink = RawFrameSink(str(wf / 'sbs.rgb'), n_frames, H, 2 * W)
            t0 = time.perf_counter()
            n = sbs_generator.process_shard(pairs, wf / 'sbs', StereoParams(), 0, 6, io_threads, 'none', True, None, sink,
                                            {p[2]: i for i, p in enumerate(pairs)}, 4, gen)
            complete = sink.close()
            dt = time.perf_counter() - t0
            out['raw_sink'] = {'value': n / dt, 'unit': 'frames/s', 'frames': n, 'complete': bool(complete), 'seconds': dt}
            os.remove(wf / 'sbs.rgb')
            sub = pairs[:n_png]
            pub = InOrderPublisher([str(wf / 'sbs' / f'sbs_{p[2]}.png') for p in sub])
            t0 = time.perf_counter()
            n = sbs_generator.process_shard(sub, wf / 'sbs', StereoParams(), 0, 6, io_threads, 'none', True, gen=gen)
            ok = pub.run(timeout_s=30)
            dt = time.perf_counter() - t0
            out['png_files'] = {'value': n / dt, 'unit': 'frames/s', 'frames': n, 'complete': bool(ok), 'seconds': dt}
        finally:
            gen.close()
        return out
    finally:
        shutil.rmtree(wf, ignore_errors=True)


def _use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU baseline is meant to use every host core."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    os.environ['OMP_NUM_THREADS'] = str(n)
    return n


def _reference_generator():
    """The unmodified reference module (oracle/_ref or /root/reference), or None."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    try:
        import ref_runner
        if not ref_runner.reference_available():
            return None, ''
        n = _use_all_host_threads()
        import cv2
        import torch
        torch.set_num_threads(n)
        cv2.setNumThreads(n)
        sc = ref_runner.import_reference()
        return sc, ref_runner.reference_origin()
    except Exception as e:       # pragma: no cover - reported in the JSON line
        return None, f'unavailable: {e}'


def cpu_baseline(sample_frames=1):
    """The reference's CPU path on this box's host cores, bounded sample of the headline workload: the unmodified
    reference when it is staged here (one 1080p frame after a warm-up band), else the oracle's C port."""
    wl = WORKLOADS['1080p']
    H, W = wl['h'], wl['w']
    sc, origin = _reference_generator()
    if sc is not None:
        import torch
        frames = make_frames(2, H, W, wl['dtype'], seed0=0)
        g = sc.StereoGenerator('cpu')
        g.process_frame(frames[0][0][:136], frames[0][1][:136], sc.StereoParams())      # warm-up band
        t0 = time.perf_counter()
        n = max(1, min(2, sample_frames))
        for r, d in frames[:n]:
            g.process_frame(r, d, sc.StereoParams())
        dt = time.perf_counter() - t0
        return {'value': n / dt, 'unit': 'frames/s', 'cores': torch.get_num_threads(), 'kind': 'reference',
                'sample': f'{n} synthetic {W}x{H} frame(s), default params, unmodified helper/stereo_core.py '
                          f'StereoGenerator("cpu").process_frame ({origin}), torch {torch.get_num_threads()} threads; {dt:.1f} s',
                'host_cpus': os.cpu_count()}
    _use_all_host_threads()
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import oracle as O
    O.build()
    frames = make_frames(sample_frames, H, W, wl['dtype'], seed0=0)
    t0 = time.perf_counter()
    for r, d in frames:
        O.process_frame(r, d, O.Params())
    dt = time.perf_counter() - t0
    return {'value': sample_frames / dt, 'unit': 'frames/s', 'cores': O.num_threads(), 'kind': 'port',
            'sample': f'{sample_frames} synthetic {W}x{H} frame(s), default params, oracle/ C+numpy port of '
                      f'helper/stereo_core.py with OpenMP ({O.num_threads()} threads); {dt:.1f} s (reference not staged: {origin or "oracle/_ref absent"})',
            'host_cpus': os.cpu_count()}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation on the host cores, rank 0 only."""
    if rank != 0:
        return None
    wl = WORKLOADS['1080p']
    H, W = wl['h'], wl['w']
    tiny = bool(os.environ.get('VSC_BENCH_TINY'))     # unit tests only: keep the CPU suite fast
    rows = 64 if tiny else H
    frames = make_frames(2, rows, W, wl['dtype'], seed0=0)
    sc, origin = (None, 'VSC_BENCH_FORCE_PORT') if os.environ.get('VSC_BENCH_FORCE_PORT') else _reference_generator()
    if sc is not None:
        import torch
        g, p = sc.StereoGenerator('cpu'), sc.StereoParams()
        step = lambda k: g.process_frame(frames[k % 2][0], frames[k % 2][1], p)
        warm = lambda k: g.process_frame(frames[k % 2][0][:min(rows, 272)], frames[k % 2][1][:min(rows, 272)], p)
        kind, cores = 'reference', torch.get_num_threads()
        what = f'unmodified helper/stereo_core.py StereoGenerator("cpu").process_frame ({origin})'
    else:
        _use_all_host_threads()
        sys.path.insert(0, os.path.join(ROOT, 'oracle'))
        import oracle as O
        O.build()
        step = lambda k: O.process_frame(frames[k % 2][0], frames[k % 2][1], O.Params())
        warm = lambda k: O.process_frame(frames[k % 2][0][:min(rows, 272)], frames[k % 2][1][:min(rows, 272)], O.Params())
        kind, cores = 'port', O.num_threads()
        what = f'oracle/ C+numpy port of helper/stereo_core.py (reference not staged: {origin or "oracle/_ref absent"})'
    for k in range(args.warmup):
        warm(k)
    t0 = time.perf_counter()
    for k in range(args.steps):
        step(k)
    dt = time.perf_counter() - t0
    value = args.steps * (rows / H) / dt
    base = {'value': value, 'unit': 'frames/s', 'cores': cores, 'kind': kind,
            'sample': f'each timed step = one full synthetic {W}x{rows} frame, default params, {what}; warm-up steps use a {min(rows, 272)}-row band'}
    return {'impl': 'reference', 'metric': wl['metric'], 'value': value, 'unit': 'frames/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8/f32', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'note': what},
            'cpu_baseline': base, 'e2e': {'value': value, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=300, help='1080p frames per step per GPU (BASELINE.json configs[1]: a 300-frame clip)')
    ap.add_argument('--slots', type=int, default=16, help='slots (CUDA streams) per GPU, 1080p')
    ap.add_argument('--group', type=int, default=4, help='frames per slot submission (share a stream and one hole-filling launch)')
    ap.add_argument('--batch-4k', type=int, default=64, help='4K frames per step per GPU')
    ap.add_argument('--slots-4k', type=int, default=10, help='slots per GPU at 4K (2.75 GB per frame in flight)')
    ap.add_argument('--no-4k', action='store_true', help='skip the 4K workload')
    ap.add_argument('--no-8k', action='store_true', help='skip the 8K sweep-corner workload')
    ap.add_argument('--cpu-frames', type=int, default=2, help='frames of the bounded CPU-baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-driver', action='store_true', help='skip the file-based frame-loop measurement (driver)')
    ap.add_argument('--dump-outputs', metavar='DIR', help="write a seeded sample of each workload's last timed step's SBS "
                                                          'frames to DIR/*.npy (rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        out = run_reference(args, rank, world)
    else:
        if world == 1 and args.gpus > 1:
            # launched without torchrun: spawn one rank per GPU ourselves
            cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={args.gpus}',
                   '--master-addr', '127.0.0.1', '--master-port', '29531', os.path.abspath(__file__)] + sys.argv[1:]
            sys.exit(subprocess.call(cmd))
        out = run_ours(args, rank, world, local_rank)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
