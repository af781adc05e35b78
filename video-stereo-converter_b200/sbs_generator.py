#!/usr/bin/env python
"""Stereo 3D Generator on B200 — drop-in for the reference's sbs_generator.py.

Same command line, files and exit codes as /root/reference/sbs_generator.py
(`python sbs_generator.py <workflow_dir> [--cpu] [--no-interactive]`, :131-133; resume by skipping
existing sbs_<n>.png :178-185; exit code 100 on a GPU failure :41,317; free-space deletion :279-290;
a carriage-return progress line on stdout that the orchestrator scrapes), but the frame loop
(:304-328) is a batched, pinned-host, multi-stream pipeline:

    loader pool --(decode straight into the slot's pinned buffers)--> submit a group of frames (H2D | kernels |
    D2H on the slot's CUDA stream) --> vsc_wait_any --> collect --> saver pool (PNG encode) --> in-order publish

and a frame-range sharder spreads one clip over the GPUs of the box (`--gpus N`, or launch under
torchrun with one process per GPU).  Frames are independent, so there is no collective.
There is no CPU path: `--cpu` is refused.

`--layout` (or the top-level config.json key "sbs_layout") picks the output frame layout: the reference's full-width
side-by-side (default), half side-by-side, top-bottom, half top-bottom or a red-cyan anaglyph (INTEGRATION.md).
`--pixfmt` / `--matrix` (or the top-level keys "sbs_pixfmt" / "sbs_matrix") hand the raw sink encoder-ready YUV 4:2:0
(yuv420p, yuv420p10le; BT.709 or BT.601, limited range) instead of rgb24; a YUV format needs `--raw-sink`.
`--png-encoder gpu` (or the top-level key "sbs_png_encoder") has the GPU encode sbs_*.png and the savers write its bytes
verbatim; the default `cv2` encodes on the saver threads with cv2.imencode.
`--temporal-radius K` / `--temporal-sigma S` (or the top-level keys "sbs_temporal_radius" / "sbs_temporal_sigma") filter
every depth map over its neighbours up to K frames away in the clip before the frame is converted; the default K = 0 is
the per-frame behaviour.
"""
from __future__ import annotations

import os
import struct
import sys
import threading
import time
from argparse import ArgumentParser, RawDescriptionHelpFormatter
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from vsc_b200.stereo_core import LAYOUTS, MATRICES, PIXFMTS  # noqa: E402
from vsc_b200.workflow import PNG_ENCODERS  # noqa: E402

GPU_ERROR_EXIT_CODE = 100      # reference: sbs_generator.py:41


def _load_config_api():
    """Prefer the reference's own config_manager when this file sits in the reference tree."""
    try:
        from helper.config_manager import ConfigError, get_path, load_config  # type: ignore
        return ConfigError, get_path, load_config
    except Exception:
        from vsc_b200.workflow import ConfigError, get_path, load_config
        return ConfigError, get_path, load_config


def build_parser() -> ArgumentParser:
    p = ArgumentParser(formatter_class=RawDescriptionHelpFormatter,
                       description='Stereo 3D Generator - Create side-by-side stereo images (B200 CUDA path)',
                       epilog='Example:\n  python sbs_generator.py "D:/Video-Processing/workflow"\n')
    p.add_argument('workflow_path', type=Path, help='Path to workflow directory containing config.json')
    p.add_argument('--cpu', action='store_true', help='(reference flag) refused: this implementation has no CPU path')
    p.add_argument('--no-interactive', action='store_true', help='Exit on error instead of waiting for user input (for orchestrator)')
    p.add_argument('--gpus', type=int, default=0, help='number of GPUs to shard the clip over (0 = all visible, or the torchrun world)')
    p.add_argument('--slots', type=int, default=6, help='frame slots (CUDA streams) per GPU')
    p.add_argument('--group', type=int, default=4, help='frames per slot submission (they share one hole-filling launch)')
    p.add_argument('--io-threads', type=int, default=8, help='loader and saver threads per GPU')
    p.add_argument('--raw-sink', default=None, metavar='PATH',
                   help="hand the SBS frames to an encoder instead of writing sbs_*.png: raw --pixfmt frames, in clip order, into PATH "
                        "(a file or FIFO; '-' = stdout); geometry in PATH.json.  Processes every frame pair (no resume)")
    p.add_argument('--layout', choices=LAYOUTS, default=None,
                   help="output frame layout (default: config.json \"sbs_layout\", else sbs): sbs [H,2W], half-sbs [H,W], "
                        "tb [2H,W], half-tb [H,W], anaglyph [H,W] (red-cyan)")
    p.add_argument('--pixfmt', choices=PIXFMTS, default=None,
                   help='pixel format of the frames (default: config.json "sbs_pixfmt", else rgb24); yuv420p and '
                        'yuv420p10le (I420, limited range) need --raw-sink')
    p.add_argument('--matrix', choices=MATRICES, default=None,
                   help='YUV matrix of the yuv420 formats (default: config.json "sbs_matrix", else bt709)')
    p.add_argument('--png-encoder', choices=PNG_ENCODERS, default=None,
                   help='who encodes sbs_*.png (default: config.json "sbs_png_encoder", else cv2): cv2 on the CPU saver '
                        'threads, or gpu (rgb24 only, not with --raw-sink)')
    p.add_argument('--temporal-radius', type=int, default=None, metavar='K',
                   help='filter every depth map over its neighbours up to K frames away, aligned to it and cut at scene '
                        'changes, against frame-to-frame depth flicker (default: config.json "sbs_temporal_radius", else 0 = '
                        'off; at most 8)')
    p.add_argument('--temporal-sigma', type=float, default=None, metavar='S',
                   help='depth difference, in 8-bit depth units, at which a neighbour\'s weight falls to exp(-1/2) (default: '
                        'config.json "sbs_temporal_sigma", else 6; in (0, 64])')
    return p


def png_size(path):
    """(height, width) from a PNG's IHDR chunk (bytes 16-24) without decoding it; None if the file is no PNG."""
    try:
        with open(path, 'rb') as f:
            head = f.read(24)
    except OSError:
        return None
    if len(head) < 24 or head[:8] != b'\x89PNG\r\n\x1a\n' or head[12:16] != b'IHDR':
        return None
    w, h = struct.unpack('>II', head[16:24])
    return h, w


def layout_refusal(output_dir: Path, frame_path, layout: str):
    """Why `layout` cannot continue this clip, or None.  The layout must take the frame size, and on a resume the
    outputs already written must have the size this layout gives (one clip with mixed frame sizes breaks the encode)."""
    from vsc_b200.stereo_core import output_shape
    size = png_size(frame_path)
    if size is None:
        return None
    try:
        want = output_shape(layout, *size)[:2]
    except ValueError as e:
        return str(e)
    existing = sorted(output_dir.glob('sbs_*.png'))
    have = png_size(existing[0]) if existing else None
    if have is not None and have != want:
        return (f"{existing[0].name} is {have[1]}x{have[0]}, but layout '{layout}' makes {want[1]}x{want[0]} frames of this "
                f"clip: continue with the layout the existing outputs were written in, or move them away")
    return None


def format_refusal(frame_path, layout: str, pixfmt: str):
    """Why `pixfmt` cannot take this clip's frames in `layout` (a YUV format needs whole 2x2 blocks), or None."""
    from vsc_b200.stereo_core import output_shape
    size = png_size(frame_path)
    if size is None:
        return None
    try:
        output_shape(layout, *size, pixfmt)
    except ValueError as e:
        return str(e)
    return None


def _read_depth(path, size):
    """A depth map as the loaders use it: grey, resized to size = (height, width) of its frame; None if unreadable."""
    import cv2
    from vsc_b200.stereo_core import _resize_depth_to
    depth = cv2.imread(str(path), cv2.IMREAD_UNCHANGED)
    if depth is None:
        return None
    if depth.ndim == 3:
        depth = cv2.cvtColor(depth, cv2.COLOR_BGR2GRAY)
    if depth.shape[:2] != tuple(size):
        depth = _resize_depth_to(depth, size[1], size[0])
    return depth


def _decode_into(item, gen, slot, index, expected, cache=None):
    """Loader job: decode one (frame, depth) pair.  When the pair has the clip's geometry and depth dtype the colour
    conversion writes straight into the slot's pinned input buffers (no staging copy); otherwise the arrays are
    returned for the single-frame path.  Returns ('pinned', None) | ('odd', (rgb, depth)) | ('error', message).
    With a DepthCache (temporal filter) the depth map comes from the cache and 'pinned' returns it instead of copying it
    into the slot: the window submission reads it, and its neighbours', from there."""
    import cv2
    import numpy as np
    try:
        bgr = cv2.imread(str(item[0]), cv2.IMREAD_COLOR)
        if bgr is None:
            raise ValueError(f'Could not load RGB: {item[0]}')
        depth = cache.get(item[1], bgr.shape[:2]) if cache is not None else _read_depth(item[1], bgr.shape[:2])
        if depth is None:
            raise ValueError(f'Could not load depth: {item[1]}')
        if expected is not None and (bgr.shape[0], bgr.shape[1], depth.dtype.str) == expected:
            prgb, pdepth = gen.pinned_inputs(slot, expected[0], expected[1], np.dtype(expected[2]), index)
            cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB, dst=prgb)
            if cache is not None:
                return 'pinned', depth
            np.copyto(pdepth, depth)
            return 'pinned', None
        return 'odd', (cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB), depth)
    except Exception as e:          # reference: the loader logs and skips (sbs_generator.py:229-230)
        return 'error', str(e)


class DepthCache:
    """Depth maps decoded once for the windows of the temporal filter: keyed by (path, frame size), the map as
    _read_depth gives it (grey, resized to the frame size), or None when it cannot be read.  A map decoded by one
    loader thread is not decoded again by another that asks for it meanwhile.  Keeps the `capacity` latest maps."""

    def __init__(self, capacity: int):
        from collections import OrderedDict
        self._maps = OrderedDict()
        self._capacity = int(capacity)
        self._lock = threading.Lock()
        self.decodes = 0

    def get(self, path, size):
        from concurrent.futures import Future
        key = (str(path), tuple(size))
        with self._lock:
            f = self._maps.get(key)
            if f is None:
                f = self._maps[key] = Future()
                mine = True
                while len(self._maps) > self._capacity:
                    self._maps.popitem(last=False)
            else:
                self._maps.move_to_end(key)
                mine = False
        if mine:
            f.set_result(self._decode(path, size))
        return f.result()

    def _decode(self, path, size):
        self.decodes += 1
        try:
            return _read_depth(path, size)
        except Exception:       # noqa: BLE001  (an unreadable neighbour ends the window)
            return None


def neighbours(clip, num: int, radius: int, step: int):
    """Pairs of the frames num + step, num + 2 step, ... within `radius` that the clip has, up to the first gap."""
    out = []
    for m in range(1, radius + 1):
        p = clip.get(num + step * m)
        if p is None:
            break
        out.append(p)
    return out


def window_maps(items, own, clip, radius: int, cache: DepthCache):
    """(maps, first) of a window submission of the consecutive clip frames `items` with their depth maps `own`: the maps
    of up to `radius` neighbours on each side, each side ending at the first frame that is missing, fails to decode or
    does not match the frames' size and dtype."""
    shape, dt = own[0].shape, own[0].dtype

    def side(step, num):
        maps = []
        for p in neighbours(clip, num, radius, step):
            d = cache.get(p[1], shape)
            if d is None or d.shape != shape or d.dtype != dt:
                break
            maps.append(d)
        return maps
    left, right = side(-1, int(items[0][2])), side(1, int(items[-1][2]))
    return left[::-1] + list(own) + right, len(left)


def open_raw_sink(path: str, pairs, layout: str, pixfmt: str = 'rgb24', matrix: str = 'bt709'):
    """RawFrameSink for `pairs` in clip order; frame geometry (and the JSON side-car) from the first frame, the layout
    and the pixel format.  OSError when the first frame cannot be read, ValueError when the layout or pixel format
    cannot take its size."""
    import cv2
    from vsc_b200.sharder import RawFrameSink
    from vsc_b200.stereo_core import output_shape
    probe = cv2.imread(str(pairs[0][0]), cv2.IMREAD_COLOR)
    if probe is None:
        raise OSError(f'cannot read {pairs[0][0]}')
    oh, ow, _ = output_shape(layout, probe.shape[0], probe.shape[1])
    output_shape(layout, probe.shape[0], probe.shape[1], pixfmt)       # refuses a size the pixel format cannot take
    return RawFrameSink(path, len(pairs), oh, ow, frame_numbers=[p[2] for p in pairs], pixfmt=pixfmt, matrix=matrix)


def process_shard(pairs, output_dir: Path, params, device_index: int, slots: int, io_threads: int, free_space_mode: str,
                  no_interactive: bool, progress=None, sink=None, sink_index=None, group: int = 4, gen=None,
                  layout: str = 'sbs', pixfmt: str = 'rgb24', matrix: str = 'bt709', png_encoder: str = 'cv2',
                  temporal=(0, 6.0), clip=None) -> int:
    """Run `pairs` [(frame_path, depth_path, frame_num)] through one GPU.  Returns frames written.

    The pipeline the benchmark times: `slots` frame slots of `group` frames each.  A slot is filled by the loader
    pool (decode straight into its pinned input buffers), submitted as ONE group (H2D | kernels | D2H on the slot's
    stream, one hole-filling launch for the group) and harvested with vsc_wait_any; finished frames go to the saver
    pool (bounded backlog) and become visible in frame order through the InOrderPublisher.
    With `sink` (a RawFrameSink shared by all GPUs of the process) frames go to it at position
    `sink_index[frame_num]` instead of into sbs_<n>.png.  `layout`, `pixfmt` and `matrix` set the output of a generator
    made here (a YUV pixfmt only with a sink).  png_encoder='gpu' has that generator encode the PNG files (a caller's
    generator must then have encode='png'), and the savers write its bytes as they are.
    temporal=(radius, sigma) with radius > 0 filters every depth map over its neighbours in `clip` (every pair of the
    clip, resumed ones included; default `pairs`): submissions then hold consecutive clip frames only, and each depth map
    is decoded once, through a DepthCache."""
    import cv2
    import numpy as np
    from vsc_b200 import StereoGenerator
    from vsc_b200.sharder import InOrderPublisher, consecutive_chunks
    radius, sigma = temporal
    clip_map = {int(p[2]): p for p in (clip if clip is not None else pairs)} if radius else None
    cache = DepthCache(2 * group * max(2, slots // 2) + 2 * radius + 8) if radius else None

    own_gen = gen is None         # a caller may pass a warm generator (n_slots >= slots, group_size >= group) and keep it
    if own_gen:
        gen = StereoGenerator(f'cuda:{device_index}', n_slots=slots, group_size=group, layout=layout, pixfmt=pixfmt,
                              matrix=matrix, encode='png' if png_encoder == 'gpu' else None)
    loaders = ThreadPoolExecutor(max_workers=io_threads, thread_name_prefix='load')
    savers = ThreadPoolExecutor(max_workers=io_threads, thread_name_prefix='save')
    backlog = threading.BoundedSemaphore(max(2 * io_threads, group))     # frames waiting for / inside the savers
    save_failed = threading.Event()
    written = [0]
    lock = threading.Lock()

    def final_of(item):
        return str(output_dir / f'sbs_{item[2]}.png')

    def skip(item, why):
        print(f'  Error loading {item[2]}: {why}')
        if sink is not None:
            sink.skip(sink_index[item[2]])                  # keep the stream gap-free
        else:
            InOrderPublisher.mark_skipped(final_of(item))   # the frames after it must not wait for this one

    def save(sbs, item):
        try:
            if sink is not None:
                try:
                    sink.put(sink_index[item[2]], sbs)
                except Exception as e:
                    print(f'\nRaw sink failed at SBS frame #{item[2]}: {e}')
                    save_failed.set()
                    return
            else:
                final = final_of(item)
                staged = InOrderPublisher.staged_path(final)
                for attempt in range(3):        # reference: 3 retries, 60 s apart (sbs_generator.py:241-262)
                    try:
                        if gen.encode == 'png':
                            buf = sbs                       # already the PNG file
                        else:
                            ok, buf = cv2.imencode('.png', cv2.cvtColor(sbs, cv2.COLOR_RGB2BGR))
                            if not ok:
                                raise IOError(f'PNG encode failed for {final}')
                        with open(staged, 'wb') as f:
                            f.write(buf.tobytes())
                        InOrderPublisher.mark_ready(final)
                        break
                    except Exception as e:
                        print(f'\nSave failed for SBS frame #{item[2]} ({attempt + 1}/3): {e}')
                        if attempt == 2:
                            InOrderPublisher.mark_skipped(final)
                            save_failed.set()
                            return
                        time.sleep(60 if not os.environ.get('VSC_FAST_RETRY') else 0.01)
            with lock:
                written[0] += 1
            if progress:
                progress(item)
        finally:
            backlog.release()

    def hand_over(frames, items):
        for sbs, item in zip(frames, items):
            backlog.acquire()                               # blocks the frame loop while the savers are behind
            savers.submit(save, sbs, item)

    # geometry / depth dtype of the clip: from the first readable pair
    expected = None
    for item in pairs[:8]:
        kind, payload = _decode_into(item, gen, 0, 0, None)
        if kind == 'odd':
            expected = (payload[0].shape[0], payload[0].shape[1], payload[1].dtype.str)
            break
    if expected is not None:        # page-locked staging for every frame of every slot, before the loaders start
        for s_ in range(slots):
            for k_ in range(group):
                gen.pinned_inputs(s_, expected[0], expected[1], np.dtype(expected[2]), k_)
    chunks = consecutive_chunks(pairs, group) if radius else [pairs[i:i + group] for i in range(0, len(pairs), group)]
    free_slots = list(range(slots))
    loading = []            # (slot, items, futures), in clip order
    inflight = {}           # slot -> items in the submission
    odd = []                # (item, rgb, depth): frames that do not have the clip's geometry
    nxt = 0

    def harvest(s):
        items = inflight.pop(s)
        res = gen.collect(s)                                # fresh arrays: the slot is reused while the savers still encode
        hand_over(res if isinstance(res, list) else [res], items)
        free_slots.append(s)

    def start_loading():
        nonlocal nxt
        while nxt < len(chunks) and free_slots and len(loading) < max(2, slots // 2):
            s = free_slots.pop(0)
            items = chunks[nxt]
            nxt += 1
            if radius:          # the frames and their depth maps, and the neighbours' maps the window will read
                futs = [loaders.submit(_decode_into, it, gen, s, k, expected, cache) for k, it in enumerate(items)]
                if expected is not None:
                    halo = neighbours(clip_map, int(items[0][2]), radius, -1) + neighbours(clip_map, int(items[-1][2]), radius, 1)
                    futs += [loaders.submit(cache.get, p[1], expected[:2]) for p in halo]
            else:
                futs = [loaders.submit(_decode_into, it, gen, s, k, expected) for k, it in enumerate(items)]
            loading.append((s, items, futs))

    def submit_temporal(s, items, results):
        """Submit a loaded chunk as one window submission, or hand its frames to the single-frame path."""
        own = [payload for kind, payload in results]
        if all(kind == 'pinned' for kind, _ in results) and own[0].dtype in (np.uint8, np.uint16):
            maps, first = window_maps(items, own, clip_map, radius, cache)
            rgbs = [gen.pinned_inputs(s, expected[0], expected[1], np.dtype(expected[2]), k)[0] for k in range(len(items))]
            gen.submit_window(s, rgbs, maps, first, params, radius, sigma)
            inflight[s] = items
            return
        for k, (it, (kind, payload)) in enumerate(zip(items, results)):
            if kind == 'error':
                skip(it, payload)
            elif kind == 'pinned':
                odd.append((it, gen.pinned_inputs(s, expected[0], expected[1], np.dtype(expected[2]), k)[0].copy(), payload))
            else:
                odd.append((it, payload[0], payload[1]))
        free_slots.append(s)

    try:
        start_loading()
        while (loading or inflight or odd) and not save_failed.is_set():
            if loading and all(f.done() for f in loading[0][2]):
                s, items, futs = loading.pop(0)
                if radius:
                    submit_temporal(s, items, [f.result() for f in futs[:len(items)]])
                    start_loading()
                    continue
                ok_idx, ok_items = [], []
                for k, (it, f) in enumerate(zip(items, futs)):
                    kind, payload = f.result()
                    if kind == 'pinned':
                        ok_idx.append(k)
                        ok_items.append(it)
                    elif kind == 'odd':
                        odd.append((it, payload[0], payload[1]))
                    else:
                        skip(it, payload)
                if ok_idx:
                    gen.submit_host(s, [gen.pinned_inputs(s, expected[0], expected[1], np.dtype(expected[2]), k) for k in ok_idx], params)
                    inflight[s] = ok_items
                else:
                    free_slots.append(s)
            elif odd and free_slots:
                it, rgb, depth = odd.pop(0)
                s = free_slots.pop(0)
                if radius and depth.dtype in (np.uint8, np.uint16):
                    maps, first = window_maps([it], [depth], clip_map, radius, cache)
                    gen.submit_window(s, [rgb], maps, first, params, radius, sigma)
                else:
                    gen.submit_frames(s, [(rgb, depth)], params)
                inflight[s] = [it]
            elif inflight:
                ready = [s for s in inflight if gen.ready(s)]
                if ready:
                    harvest(ready[0])
                elif loading and not free_slots:
                    harvest(gen.wait_any(list(inflight)))
                elif loading or (odd and not free_slots):
                    time.sleep(0.0005)                      # decoders are the bottleneck: let them work
                else:
                    harvest(gen.wait_any(list(inflight)))
            else:
                time.sleep(0.0005)
            start_loading()
        for s in list(inflight):
            harvest(s)
    finally:
        loaders.shutdown(wait=False, cancel_futures=True)
        savers.shutdown(wait=True)
        if own_gen:
            gen.close()
    if save_failed.is_set():
        print('\nERROR: Failed to write output file.' + (' Exiting (non-interactive mode).' if no_interactive else ''))
    return written[0]


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    if args.raw_sink == '-':
        sys.stdout = sys.stderr          # stdout carries the frames
    if not args.workflow_path.is_dir():
        print(f'ERROR: Workflow directory not found: {args.workflow_path}')
        return 0
    ConfigError, get_path, load_config = _load_config_api()
    from vsc_b200.workflow import LayoutError, config_layout, config_pixfmt, config_png_encoder, config_temporal
    try:
        config = load_config(args.workflow_path)
    except ConfigError as e:
        print(f'ERROR: {e}')
        return 2 if isinstance(e, LayoutError) else 0
    frames_dir = get_path(args.workflow_path, config, 'frames')
    depth_dir = get_path(args.workflow_path, config, 'depth_maps')
    output_dir = get_path(args.workflow_path, config, 'sbs')
    if not frames_dir.exists():
        print(f'ERROR: Frames directory not found: {frames_dir}')
        return 0
    if not depth_dir.exists():
        print(f'ERROR: Depth directory not found: {depth_dir}')
        return 0
    output_dir.mkdir(parents=True, exist_ok=True)
    if args.cpu:
        print('ERROR: --cpu is not supported: the B200 SBS path has no CPU fallback (use the reference implementation).')
        return 2
    try:
        layout = args.layout or config_layout(config)
        cfg_pixfmt, cfg_matrix = config_pixfmt(config)
        png_encoder = args.png_encoder or config_png_encoder(config)
        cfg_radius, cfg_sigma = config_temporal(config)
    except LayoutError as e:
        print(f'ERROR: {e}')
        return 2
    from vsc_b200.stereo_core import check_temporal
    try:
        temporal = check_temporal(cfg_radius if args.temporal_radius is None else args.temporal_radius,
                                  cfg_sigma if args.temporal_sigma is None else args.temporal_sigma)
    except ValueError as e:
        print(f'ERROR: {e}')
        return 2
    pixfmt, matrix = args.pixfmt or cfg_pixfmt, args.matrix or cfg_matrix
    if png_encoder == 'gpu' and args.raw_sink:
        print('ERROR: --png-encoder gpu encodes sbs_*.png files; the raw sink takes raw frames (drop one of the two)')
        return 2
    if png_encoder == 'gpu' and pixfmt != 'rgb24':
        print(f'ERROR: --png-encoder gpu writes rgb24 PNG files, not pixel format {pixfmt}')
        return 2
    if pixfmt != 'rgb24' and not args.raw_sink:
        print(f'ERROR: pixel format {pixfmt} is for the raw sink only (--raw-sink); sbs_*.png files are rgb24')
        return 2

    from vsc_b200 import StereoParams
    from vsc_b200._lib import VscCudaError
    from vsc_b200.sharder import InOrderPublisher, barrier, dist_env, shard_items
    from vsc_b200.workflow import find_frame_pairs
    sc = config['stereo']
    params = StereoParams(**{k: sc[k] for k in ('max_disparity', 'convergence', 'super_sampling', 'edge_softness',
                                                'artifact_smoothing', 'depth_gamma', 'sharpen')})
    rank, world, local_rank = dist_env()
    if rank == 0:
        print('Scanning for frame pairs...')
    all_pairs, missing, first, last = find_frame_pairs(frames_dir, depth_dir)
    if missing and rank == 0:
        print(f'Missing depth maps: {missing} of {missing + len(all_pairs)} frames in range of frame_{first} to frame_{last}')
    pairs = [p for p in all_pairs if args.raw_sink or not (output_dir / f'sbs_{p[2]}.png').exists()]
    skipped = len(all_pairs) - len(pairs)
    if rank == 0:
        print(f'Found: {len(all_pairs)} frame pairs, {skipped} already processed, {len(pairs)} to process')
    if not pairs:
        if rank == 0:
            print('All frames already processed.')
        return 0
    why = layout_refusal(output_dir, pairs[0][0], layout) if not args.raw_sink else format_refusal(pairs[0][0], layout, pixfmt)
    if why:
        print(f'ERROR: {why}')
        return 2

    import torch
    if not torch.cuda.is_available():
        print('ERROR: no CUDA device available and this implementation has no CPU path')
        return GPU_ERROR_EXIT_CODE
    ngpu = torch.cuda.device_count()
    free_space_mode = config.get('free_space', {}).get('sbs_generator', 'none')
    if rank == 0:
        print(f'Using GPU: {torch.cuda.get_device_name(0)} x{world if world > 1 else (args.gpus or ngpu)}')
        print(f'Parameters: disparity={params.max_disparity}, convergence={params.convergence}, '
              f'super_sampling={params.super_sampling}, edge_softness={params.edge_softness}, '
              f'smoothing={params.artifact_smoothing}, gamma={params.depth_gamma}, sharpen={params.sharpen}, layout={layout}'
              + (f', pixfmt={pixfmt}, matrix={matrix}' if pixfmt != 'rgb24' else '')
              + (', png_encoder=gpu' if png_encoder == 'gpu' else '')
              + (f', temporal_radius={temporal[0]}, temporal_sigma={temporal[1]:g}' if temporal[0] else ''))

    finals = [str(output_dir / f'sbs_{p[2]}.png') for p in pairs]

    def free_pair(p):
        if free_space_mode in ('frame', 'all'):
            Path(p[0]).unlink(missing_ok=True)
        if free_space_mode in ('depth', 'all'):
            Path(p[1]).unlink(missing_ok=True)

    def free_inputs(i):         # free_space (sbs_generator.py:279-290): only once sbs_<n>.png exists under its final name
        free_pair(pairs[i])
    if temporal[0] and free_space_mode != 'none' and not args.raw_sink:
        # neighbours read a frame's depth map: its inputs go once every frame within the radius has its output
        from vsc_b200.sharder import DelayedFree
        by_num = {int(p[2]): p for p in all_pairs}
        todo = {p[2] for p in pairs}
        gate = DelayedFree(by_num, [int(p[2]) for p in all_pairs if p[2] not in todo], temporal[0], lambda g: free_pair(by_num[g]))

        def free_inputs(i):     # noqa: F811
            gate.published(int(pairs[i][2]))
    sink = sink_index = None
    if args.raw_sink:
        if world > 1:
            print('ERROR: --raw-sink needs all GPUs in one process (use --gpus N, not torchrun)')
            return 2
        try:
            sink = open_raw_sink(args.raw_sink, pairs, layout, pixfmt, matrix)
        except OSError as e:
            print(f'ERROR: {e}')
            return 0
        except ValueError as e:         # the layout or pixel format cannot take the frame size
            print(f'ERROR: {e}')
            return 2
        sink_index = {p[2]: i for i, p in enumerate(pairs)}
    t0 = time.time()
    done = [0]
    published_all = True

    def progress(_item):
        done[0] += 1
        if rank == 0:
            el = time.time() - t0
            sys.stdout.write(f'\r{skipped + done[0] * max(1, world)}/{len(all_pairs)} [{el:.0f}s, {done[0] * max(1, world) / max(el, 1e-6):.2f}img/s]')
            sys.stdout.flush()

    try:
        if world > 1:
            # torchrun: this process is one rank = one GPU
            import torch.distributed as dist
            dist.init_process_group('nccl' if torch.cuda.is_available() else 'gloo')
            mine = shard_items(pairs, world, rank)
            pub = InOrderPublisher(finals, on_published=free_inputs)
            t = threading.Thread(target=pub.run, daemon=True) if rank == 0 else None
            if t:
                t.start()
            n = process_shard(mine, output_dir, params, local_rank, args.slots, args.io_threads, free_space_mode, args.no_interactive, progress,
                              group=args.group, layout=layout, png_encoder=png_encoder, temporal=temporal, clip=all_pairs)
            barrier()
            if t:
                pub.stop()
                t.join()
                published_all = pub.run(timeout_s=60, final=True)
            dist.destroy_process_group()
        else:
            g = args.gpus or ngpu
            g = max(1, min(g, ngpu, len(pairs)))
            pub = InOrderPublisher([] if sink is not None else finals, on_published=free_inputs)
            t = threading.Thread(target=pub.run, daemon=True)
            t.start()
            if g == 1:
                n = process_shard(pairs, output_dir, params, 0, args.slots, args.io_threads, free_space_mode, args.no_interactive, progress,
                                  sink, sink_index, args.group, layout=layout, pixfmt=pixfmt, matrix=matrix, png_encoder=png_encoder,
                                  temporal=temporal, clip=all_pairs)
            else:
                # one worker thread per GPU; each owns a StereoGenerator (its own CUDA context state, streams, pinned ring)
                results = [0] * g
                errors = []

                def work(k):
                    try:
                        results[k] = process_shard(shard_items(pairs, g, k), output_dir, params, k, args.slots, args.io_threads,
                                                   free_space_mode, args.no_interactive, progress, sink, sink_index, args.group,
                                                   layout=layout, pixfmt=pixfmt, matrix=matrix, png_encoder=png_encoder,
                                                   temporal=temporal, clip=all_pairs)
                    except BaseException as e:   # noqa: BLE001
                        errors.append(e)
                ths = [threading.Thread(target=work, args=(k,)) for k in range(g)]
                for th in ths:
                    th.start()
                for th in ths:
                    th.join()
                if errors:
                    raise errors[0]
                n = sum(results)
            pub.stop()
            t.join()
            published_all = pub.run(timeout_s=60, final=True)
            if sink is not None and not sink.close():
                print(f'\nWARNING: raw sink holds {sink.written} of {len(pairs)} frames (stream ends at the first missing frame)')
    except VscCudaError as e:
        print(f'\nERROR: GPU failure - {e}')
        return GPU_ERROR_EXIT_CODE
    if rank == 0:
        if pub.skipped:
            print(f'\nSkipped {len(pub.skipped)} frame(s) that could not be read or written: '
                  + ', '.join(os.path.basename(f) for f in pub.skipped[:8]) + (' ...' if len(pub.skipped) > 8 else ''))
        if not published_all:
            print(f'\nERROR: only {pub.published} of {len(pairs)} outputs became visible (a worker did not finish its frames).')
            return 1
        print(f'\nDone! Processed {n if world == 1 else len(pairs) - len(pub.skipped)} of {len(pairs)} frames.')
    return 0


if __name__ == '__main__':
    sys.exit(main())
