#!/usr/bin/env python
"""Headless parameter sweep — the `sbs_tester.py` workflow without the Tk window (SURVEY.md 8(f) rank 4).

The reference's tester (sbs_tester.py:652-707) renders ONE frame with the slider values and shows it; tuning
means moving a slider, waiting for the CPU, and looking.  At GPU speed the same question — "what do these
parameters do to this frame?" — is answered for a whole grid at once:

    python sbs_sweep.py <workflow_dir> --frame 120 --param max_disparity=20:60:10 --param depth_gamma=0.2,0.3,0.5

renders the cartesian product of the given values (every other parameter from config.json `stereo`), writes
`sweep_<i>.png` plus `sweep.json` (parameters, milliseconds, refusals) into `--out`, through the same
`StereoGenerator` the batch driver uses.  Parameter names, ranges and step sizes are the tester's sliders
(sbs_tester.py:356-362); a combination whose convergence crop is invalid is recorded as refused, like the
tester's red status line.  `--layout anaglyph` renders red-cyan previews, which show the depth effect of
`max_disparity` and `convergence` on any screen with a pair of red-cyan glasses.
"""
from __future__ import annotations

import itertools
import json
import os
import sys
import time
from argparse import ArgumentParser
from pathlib import Path

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from vsc_b200.stereo_core import LAYOUTS  # noqa: E402

# slider ranges of the reference's tester: name -> (from, to, step)   (sbs_tester.py:356-362)
SLIDERS = {
    'max_disparity': (5.0, 100.0, 0.5), 'convergence': (-50.0, 50.0, 1.0), 'super_sampling': (1.0, 4.0, 0.1),
    'edge_softness': (0.0, 30.0, 0.5), 'artifact_smoothing': (0.0, 5.0, 0.1), 'depth_gamma': (0.1, 2.0, 0.05),
    'sharpen': (0.0, 16.0, 0.5),
}


def parse_param(spec: str):
    """'name=a,b,c' or 'name=lo:hi:step' (inclusive) -> (name, [values]); values must lie in the slider's range."""
    if '=' not in spec:
        raise ValueError(f"expected name=values, got '{spec}'")
    name, rhs = spec.split('=', 1)
    name = name.strip()
    if name not in SLIDERS:
        raise ValueError(f"unknown parameter '{name}' (one of {', '.join(SLIDERS)})")
    lo, hi, _ = SLIDERS[name]
    if ':' in rhs:
        parts = [float(x) for x in rhs.split(':')]
        if len(parts) != 3 or parts[2] <= 0 or parts[1] < parts[0]:
            raise ValueError(f"range must be lo:hi:step with step > 0, got '{rhs}'")
        n = int((parts[1] - parts[0]) / parts[2] + 1e-9) + 1
        values = [round(parts[0] + i * parts[2], 6) for i in range(n)]
    else:
        values = [float(x) for x in rhs.split(',') if x.strip()]
    if not values:
        raise ValueError(f"no values for '{name}'")
    for v in values:
        if not (lo <= v <= hi):
            raise ValueError(f"{name}={v} is outside the tester's slider range [{lo}, {hi}]")
    return name, values


def grid(base: dict, specs):
    """Cartesian product of the swept parameters over the base parameter set (list of dicts, deterministic order)."""
    names, lists = [], []
    for spec in specs:
        n, v = parse_param(spec)
        if n in names:
            raise ValueError(f"parameter '{n}' given twice")
        names.append(n)
        lists.append(v)
    out = []
    for combo in itertools.product(*lists) if lists else [()]:
        p = dict(base)
        p.update(dict(zip(names, combo)))
        out.append(p)
    return out


def main(argv=None) -> int:
    ap = ArgumentParser(description='Headless stereo parameter sweep (B200 CUDA path)')
    ap.add_argument('workflow_path', type=Path, help='workflow directory containing config.json, frames and depth maps')
    ap.add_argument('--frame', type=int, default=None, help='frame number (default: the first frame pair)')
    ap.add_argument('--param', action='append', default=[], metavar='NAME=VALUES', help='a,b,c or lo:hi:step; repeatable')
    ap.add_argument('--out', type=Path, default=None, help='output directory (default: <workflow>/sweep)')
    ap.add_argument('--slots', type=int, default=4, help='frames in flight')
    ap.add_argument('--no-images', action='store_true', help='only write sweep.json (timings, refusals)')
    ap.add_argument('--layout', choices=LAYOUTS, default=None,
                    help='output layout of the previews (default: config.json "sbs_layout", else sbs)')
    args = ap.parse_args(argv)

    from vsc_b200.workflow import ConfigError, config_layout, find_frame_pairs, get_path, load_config
    try:
        config = load_config(args.workflow_path)
        layout = args.layout or config_layout(config)
    except ConfigError as e:
        print(f'ERROR: {e}')
        return 2
    keys = list(SLIDERS)
    base = {k: float(config['stereo'][k]) for k in keys}
    try:
        combos = grid(base, args.param)
    except ValueError as e:
        print(f'ERROR: {e}')
        return 2
    pairs, _, _, _ = find_frame_pairs(get_path(args.workflow_path, config, 'frames'), get_path(args.workflow_path, config, 'depth_maps'))
    if args.frame is not None:
        pairs = [p for p in pairs if int(p[2]) == args.frame]
    if not pairs:
        print('ERROR: no matching frame pair')
        return 2
    frame_path, depth_path, frame_num = pairs[0]

    import cv2
    from vsc_b200 import StereoGenerator, StereoParams, load_image_pair
    rgb, depth = load_image_pair(frame_path, depth_path)
    out_dir = args.out or (args.workflow_path / 'sweep')
    out_dir.mkdir(parents=True, exist_ok=True)
    gen = StereoGenerator('cuda:0', n_slots=max(1, args.slots), layout=layout)
    results = [None] * len(combos)
    t0 = time.time()
    inflight, free = [], list(range(gen.n_slots))

    def finish(slot, i, t_sub):
        try:
            sbs = gen.collect(slot)
            results[i] = {'index': i, 'params': combos[i], 'ms': round(gen.last_frame_ms(slot), 3), 'refused': None}
            if not args.no_images:
                cv2.imwrite(str(out_dir / f'sweep_{i:04d}.png'), cv2.cvtColor(sbs, cv2.COLOR_RGB2BGR))
        except RuntimeError as e:          # the tester shows 'Error: ...' in red (sbs_tester.py:699-700)
            results[i] = {'index': i, 'params': combos[i], 'ms': None, 'refused': str(e)}
        free.append(slot)

    for i, p in enumerate(combos):
        if not free:
            s, j, ts = inflight.pop(0)
            finish(s, j, ts)
        s = free.pop(0)
        try:
            gen.submit(s, rgb, depth, StereoParams(**p))
            inflight.append((s, i, time.time()))
        except RuntimeError as e:          # invalid crop window: refused at submission
            results[i] = {'index': i, 'params': p, 'ms': None, 'refused': str(e)}
            free.append(s)
    for s, j, ts in inflight:
        finish(s, j, ts)
    gen.close()
    dt = time.time() - t0
    ok = [r for r in results if r['refused'] is None]
    with open(out_dir / 'sweep.json', 'w') as f:
        json.dump({'frame': int(frame_num), 'shape': list(rgb.shape), 'layout': layout, 'swept': args.param, 'seconds': round(dt, 3),
                   'results': results}, f, indent=1)
    print(f'{len(ok)} of {len(combos)} parameter sets rendered in {dt:.2f} s ({len(ok) / max(dt, 1e-9):.1f} previews/s), '
          f'{len(combos) - len(ok)} refused; results in {out_dir}')
    return 0


if __name__ == '__main__':
    sys.exit(main())
