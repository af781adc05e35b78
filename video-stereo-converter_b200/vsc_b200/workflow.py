"""Minimal reader for a workflow directory's config.json (the parts the SBS stage uses).

The reference's helper/config_manager.py (load_config :267, get_path :342, the `stereo` schema
:43-54) stays the owner of the format; this module reads the same file with the same rules for the
keys this stage needs, so that sbs_generator.py runs both inside the reference tree (where
`helper.config_manager` is importable and preferred) and standalone.

One key is this implementation's own: the optional top-level "sbs_layout" (output layout of the SBS stage, one of
stereo_core.LAYOUTS, default "sbs").  It sits at the top level because the reference's validator accepts extra
top-level keys while the reference builds StereoParams from the whole `stereo` block.  So do the optional
"sbs_pixfmt" (pixel format of the frames, one of stereo_core.PIXFMTS, default "rgb24") and "sbs_matrix" (YUV matrix, one
of stereo_core.MATRICES, default "bt709"), and "sbs_png_encoder" (who encodes sbs_*.png, one of PNG_ENCODERS, default
"cv2"), and "sbs_temporal_radius" / "sbs_temporal_sigma" (temporal depth filter, radius 0..8 frames, default 0 = off;
sigma in (0, 64], default 6).
"""
from __future__ import annotations

import json
from pathlib import Path
from typing import Dict

STEREO_KEYS = ('max_disparity', 'convergence', 'super_sampling', 'edge_softness', 'artifact_smoothing', 'depth_gamma', 'sharpen')
DIR_KEYS = ('frames', 'depth_maps', 'sbs')
LAYOUT_KEY = 'sbs_layout'
PIXFMT_KEY, MATRIX_KEY = 'sbs_pixfmt', 'sbs_matrix'
PNG_ENCODER_KEY = 'sbs_png_encoder'
# who encodes sbs_*.png: 'cv2' (cv2.imencode on the saver threads) or 'gpu' (the library's PNG encoding, written verbatim)
PNG_ENCODERS = ('cv2', 'gpu')
TEMPORAL_RADIUS_KEY, TEMPORAL_SIGMA_KEY = 'sbs_temporal_radius', 'sbs_temporal_sigma'


class ConfigError(Exception):
    """Raised when config.json is missing or fails validation (reference: config_manager.py:78)."""


class LayoutError(ConfigError):
    """One of the optional output keys ("sbs_layout", "sbs_pixfmt", "sbs_matrix", "sbs_png_encoder") holds something
    other than a name it takes."""


def config_layout(cfg: Dict) -> str:
    """The output layout a config asks for: top-level "sbs_layout", default 'sbs'."""
    from .stereo_core import LAYOUTS
    v = cfg.get(LAYOUT_KEY, 'sbs')
    if v not in LAYOUTS:
        raise LayoutError(f"Invalid '{LAYOUT_KEY}' {v!r} (expected one of {', '.join(LAYOUTS)})")
    return v


def config_pixfmt(cfg: Dict):
    """(pixel format, yuv matrix) a config asks for: top-level "sbs_pixfmt" and "sbs_matrix", default ('rgb24', 'bt709')."""
    from .stereo_core import MATRICES, PIXFMTS
    out = []
    for key, names, default in ((PIXFMT_KEY, PIXFMTS, 'rgb24'), (MATRIX_KEY, MATRICES, 'bt709')):
        v = cfg.get(key, default)
        if v not in names:
            raise LayoutError(f"Invalid '{key}' {v!r} (expected one of {', '.join(names)})")
        out.append(v)
    return tuple(out)


def config_png_encoder(cfg: Dict) -> str:
    """The PNG encoder a config asks for: top-level "sbs_png_encoder", default 'cv2'."""
    v = cfg.get(PNG_ENCODER_KEY, 'cv2')
    if v not in PNG_ENCODERS:
        raise LayoutError(f"Invalid '{PNG_ENCODER_KEY}' {v!r} (expected one of {', '.join(PNG_ENCODERS)})")
    return v


def config_temporal(cfg: Dict):
    """(radius, sigma) of the temporal depth filter a config asks for: top-level "sbs_temporal_radius" (an integer in
    0..8, default 0 = off) and "sbs_temporal_sigma" (a number in (0, 64], default 6)."""
    from .stereo_core import TEMPORAL_SIGMA, check_temporal
    r, s = cfg.get(TEMPORAL_RADIUS_KEY, 0), cfg.get(TEMPORAL_SIGMA_KEY, TEMPORAL_SIGMA)
    try:
        return check_temporal(r, s)
    except ValueError as e:
        raise LayoutError(f"Invalid '{TEMPORAL_RADIUS_KEY}' {r!r} / '{TEMPORAL_SIGMA_KEY}' {s!r}: {e}")


def load_config(workflow_path) -> Dict:
    f = Path(workflow_path) / 'config.json'
    if not f.exists():
        raise ConfigError(f'Config file not found: {f}')
    try:
        cfg = json.loads(f.read_text(encoding='utf-8'))
    except json.JSONDecodeError as e:
        raise ConfigError(f'Invalid JSON in config file: {e}')
    if not isinstance(cfg.get('directories'), dict):
        raise ConfigError("Missing required key: 'directories'")
    for k in DIR_KEYS:
        if not isinstance(cfg['directories'].get(k), str):
            raise ConfigError(f"Missing or invalid 'directories.{k}' (expected str)")
    if not isinstance(cfg.get('stereo'), dict):
        raise ConfigError("Missing required key: 'stereo'")
    for k in STEREO_KEYS:
        v = cfg['stereo'].get(k)
        # ints are accepted for floats (config_manager.py:114); bools are not numbers here
        if isinstance(v, bool) or not isinstance(v, (int, float)):
            raise ConfigError(f"Missing or invalid 'stereo.{k}' (expected float)")
    config_layout(cfg)
    config_pixfmt(cfg)
    config_png_encoder(cfg)
    config_temporal(cfg)
    return cfg


def get_path(workflow_path, config: Dict, key: str) -> Path:
    if key not in config['directories']:
        raise KeyError(f'Unknown directory key: {key}')
    return Path(workflow_path) / config['directories'][key]


def find_frame_pairs(frames_dir: Path, depth_dir: Path):
    """Matching (frame_path, depth_path, frame_num) triples; .tif depth preferred over .png
    (reference: sbs_generator.py:71-116).  Returns (pairs, missing_count, first_missing, last_missing)."""
    pairs, missing, first, last = [], 0, None, None
    for frame_path in sorted(Path(frames_dir).glob('frame_*.png')):
        num = frame_path.stem.replace('frame_', '')
        dp = Path(depth_dir) / f'depth_frame_{num}.tif'
        if not dp.exists():
            dp = Path(depth_dir) / f'depth_frame_{num}.png'
            if not dp.exists():
                first = first if first is not None else num
                last = num
                missing += 1
                continue
        pairs.append((frame_path, dp, num))
    return pairs, missing, first, last
