"""Drop-in for the reference's `helper/stereo_core.py` on top of libvsc_b200.so.

Same `__all__`, same signatures, same defaults and the same error behaviour for the hot call as
/root/reference/helper/stereo_core.py:22-29, :193-311 — the arithmetic runs in hand-written
sm_100a CUDA kernels behind the C ABI of include/vsc_b200.h.  There is no CPU path:
`StereoGenerator('cpu')` raises, and a missing CUDA library raises on import of `_lib`.

Additions that the reference does not have (used by the frame loop in sbs_generator.py):
`StereoGenerator.submit/collect` (asynchronous, pinned, multi-slot) and `process_batch`, and output layouts
(`StereoGenerator(..., layout='half-sbs')`, `LAYOUTS`, `output_shape`): every output path then returns frames of
`output_shape(layout, h, w)` instead of the side-by-side [h, 2w, 3].  Output pixel formats
(`StereoGenerator(..., pixfmt='yuv420p10le', matrix='bt709')`, `PIXFMTS`, `MATRICES`, `output_dtype`): the YUV formats
return the I420 planes of that frame as one [rows * 3 // 2, cols] array, the shape cv2's COLOR_RGB2YUV_I420 uses.
PNG output (`StereoGenerator(..., encode='png')`, `ENCODINGS`, `encoded_capacity`): every output path returns the PNG file
of the rgb24 frame, encoded on the GPU, as a 1-D uint8 array of exactly the file's bytes.
Temporal depth stabilisation (`StereoGenerator.submit_window`, `process_batch(..., temporal=(radius, sigma))`,
`temporal_depth`): each frame's depth map is filtered over its neighbours within `radius` frames, aligned to it and cut at
scene boundaries, before the frame is converted (include/vsc_b200.h has the exact filter).
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass
from pathlib import Path
from typing import Iterable, List, Optional, Tuple

import numpy as np

from . import _lib

__all__ = [
    'load_image_pair',
    'normalize_depth',
    'apply_depth_gamma',
    'forward_warp_stereo',
    'StereoParams',
    'StereoGenerator',
]


@dataclass
class StereoParams:
    """Parameters for stereo image generation (reference: stereo_core.py:193-202; config.json
    `stereo` block, helper/config_manager.py:43-54)."""
    max_disparity: float = 50.0
    convergence: float = -10.0
    super_sampling: float = 3.0
    edge_softness: float = 20.0
    artifact_smoothing: float = 1.0
    depth_gamma: float = 0.2
    sharpen: float = 14.0


# output layouts (include/vsc_b200.h VSC_LAYOUT_*): name -> C enum.  'sbs' is the reference's output.
LAYOUTS = ('sbs', 'half-sbs', 'tb', 'half-tb', 'anaglyph')


def layout_code(layout: str) -> int:
    """C enum of a layout name; ValueError for anything else."""
    if layout not in LAYOUTS:
        raise ValueError(f'unknown output layout {layout!r} (one of {", ".join(LAYOUTS)})')
    return LAYOUTS.index(layout)


# output pixel formats (include/vsc_b200.h VSC_PIXFMT_*) and the matrices of the YUV formats (VSC_MATRIX_*):
# name -> C enum, named as ffmpeg names them.  'rgb24' is the reference's output.
PIXFMTS = ('rgb24', 'yuv420p', 'yuv420p10le')
MATRICES = ('bt709', 'bt601')


def pixfmt_code(pixfmt: str) -> int:
    """C enum of a pixel format name; ValueError for anything else."""
    if pixfmt not in PIXFMTS:
        raise ValueError(f'unknown pixel format {pixfmt!r} (one of {", ".join(PIXFMTS)})')
    return PIXFMTS.index(pixfmt)


def matrix_code(matrix: str) -> int:
    """C enum of a YUV matrix name; ValueError for anything else."""
    if matrix not in MATRICES:
        raise ValueError(f'unknown yuv matrix {matrix!r} (one of {", ".join(MATRICES)})')
    return MATRICES.index(matrix)


def output_dtype(pixfmt: str) -> np.dtype:
    """Element type of the frames of a pixel format: uint16 (value in the low 10 bits) for yuv420p10le, else uint8."""
    return np.dtype(np.uint16 if pixfmt_code(pixfmt) == _lib.PIXFMT_YUV420P10LE else np.uint8)


# encoded outputs (include/vsc_b200.h VSC_ENCODE_*): name -> C enum; None (raw frames) is VSC_ENCODE_NONE
ENCODINGS = ('png',)


def encode_code(encode: Optional[str]) -> int:
    """C enum of an encoding name (None: raw frames); ValueError for anything else."""
    if encode is None:
        return _lib.ENCODE_NONE
    if encode not in ENCODINGS:
        raise ValueError(f'unknown encoding {encode!r} (None or one of {", ".join(ENCODINGS)})')
    return ENCODINGS.index(encode) + 1


def encoded_capacity(layout: str, h: int, w: int) -> int:
    """Worst-case bytes of the PNG file of the frame `layout` makes of an h x w input (the size an output buffer of an
    encoding generator must have).  ValueError for an unknown layout or a size it cannot take."""
    n = C.c_size_t()
    rc = _lib.load().vsc_encoded_capacity(layout_code(layout), _lib.ENCODE_PNG, int(h), int(w), C.byref(n))
    if rc != _lib.VSC_OK:
        raise ValueError((_lib.load().vsc_last_error() or b'').decode('utf-8', 'replace'))
    return int(n.value)


def output_shape(layout: str, h: int, w: int, pixfmt: str = 'rgb24') -> Tuple[int, ...]:
    """Shape (rows, cols, 3) of the frame `layout` makes of an h x w input (the library's vsc_layout_shape).  For a YUV
    pixel format: (rows * 3 // 2, cols), the I420 planes Y [rows][cols], U and V [rows/2][cols/2] one after the other.
    ValueError for an unknown layout or format, or a size they cannot take (an odd side that a half layout halves; for
    YUV an odd side, or a width (half-sbs) or height (half-tb) not divisible by 4)."""
    code = layout_code(layout)
    oh, ow = C.c_int(), C.c_int()
    rc = _lib.load().vsc_layout_shape(code, int(h), int(w), C.byref(oh), C.byref(ow))
    if rc != _lib.VSC_OK:
        raise ValueError((_lib.load().vsc_last_error() or b'').decode('utf-8', 'replace'))
    if pixfmt_code(pixfmt) == _lib.PIXFMT_RGB24:
        return oh.value, ow.value, 3
    n = C.c_size_t()
    rc = _lib.load().vsc_output_size(code, pixfmt_code(pixfmt), int(h), int(w), C.byref(n))
    if rc != _lib.VSC_OK:
        raise ValueError((_lib.load().vsc_last_error() or b'').decode('utf-8', 'replace'))
    return oh.value * 3 // 2, ow.value


# ------------------------------------------------------------------------------------------------
# file loading (reference: stereo_core.py:32-68) — plain OpenCV I/O, not part of the GPU path
# ------------------------------------------------------------------------------------------------
def load_image_pair(rgb_path: Path, depth_path: Path) -> Tuple[np.ndarray, np.ndarray]:
    """Load an RGB frame and its depth map; raises ValueError when a file cannot be read."""
    import cv2
    rgb = cv2.imread(str(rgb_path), cv2.IMREAD_COLOR)
    depth = cv2.imread(str(depth_path), cv2.IMREAD_UNCHANGED)
    if rgb is None:
        raise ValueError(f'Could not load RGB: {rgb_path}')
    if depth is None:
        raise ValueError(f'Could not load depth: {depth_path}')
    if depth.ndim == 3:
        depth = cv2.cvtColor(depth, cv2.COLOR_BGR2GRAY)
    if rgb.shape[:2] != depth.shape[:2]:
        depth = _resize_depth_to(depth, rgb.shape[1], rgb.shape[0])
    return cv2.cvtColor(rgb, cv2.COLOR_BGR2RGB), depth


def _resize_depth_to(depth: np.ndarray, w: int, h: int) -> np.ndarray:
    """Size-mismatch branch of load_image_pair (stereo_core.py:64-65): LANCZOS4 to the frame size."""
    import cv2
    return cv2.resize(depth, (w, h), interpolation=cv2.INTER_LANCZOS4)


# ------------------------------------------------------------------------------------------------
# shared default context for the module-level helpers
# ------------------------------------------------------------------------------------------------
_default_ctx: Optional[_lib.Context] = None
# The helpers share _default_ctx, i.e. one stream and one set of device scalars (its slot 0), and ctypes releases the
# GIL during a call: every use of that context holds this lock, so concurrent helper calls run one after the other.
_helper_lock = threading.Lock()


def _ctx() -> _lib.Context:
    """The helpers' shared context; call with _helper_lock held."""
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = _lib.Context(_current_device(), 1)
    return _default_ctx


def _current_device() -> int:
    try:
        import torch
        if torch.cuda.is_available():
            return int(torch.cuda.current_device())
    except Exception:
        pass
    return 0


def _as_f32(t):
    """torch tensor -> contiguous float32 numpy on host (+ a function to map results back).  The helpers compute in
    float32 whatever the input's dtype, and cast the results back to it."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError('expected a torch.Tensor')
    dev, dt = t.device, t.dtype
    a = np.ascontiguousarray(t.detach().to('cpu', torch.float32).numpy())

    def back(x: np.ndarray):
        return torch.from_numpy(x).to(device=dev, dtype=dt)
    return a, back


def normalize_depth(depth):
    """Normalize depth to [0, 1] (reference: stereo_core.py:71-88); zeros if the range is < 1e-6."""
    a, back = _as_f32(depth)
    out = np.empty_like(a)
    with _helper_lock:
        _lib.check(_lib.load().vsc_stage_normalize_f32(_ctx().handle, _lib.ptr(a), a.size, _lib.ptr(out)))
    return back(out)


def apply_depth_gamma(depth, gamma: float):
    """pow(clamp(depth, 0.001, 1), gamma) (reference: stereo_core.py:91-107)."""
    a, back = _as_f32(depth)
    out = np.empty_like(a)
    with _helper_lock:
        _lib.check(_lib.load().vsc_stage_gamma_f32(_ctx().handle, _lib.ptr(a), a.size, float(gamma), _lib.ptr(out)))
    return back(out)


def forward_warp_stereo(image, depth, max_disparity: float):
    """Left/right forward warp with occlusion ordering (reference: stereo_core.py:110-190).

    image [1, C, H, W], depth [1, 1, H, W] -> (left, left_mask, right, right_mask) with the
    reference's shapes [1, C, H, W] / [1, 1, H, W].  B must be 1, as in the reference (:146).
    """
    if image.dim() != 4 or image.shape[0] != 1:
        raise RuntimeError('forward_warp_stereo requires a [1, C, H, W] image (the reference views it as [C, -1])')
    img, back = _as_f32(image)
    dep, _ = _as_f32(depth)
    _, c, h, w = img.shape
    if dep.size != h * w:
        raise RuntimeError('depth must have H*W elements')
    left, right = np.empty((1, c, h, w), np.float32), np.empty((1, c, h, w), np.float32)
    lm, rm = np.empty((1, 1, h, w), np.float32), np.empty((1, 1, h, w), np.float32)
    with _helper_lock:
        _lib.check(_lib.load().vsc_stage_warp_f32(_ctx().handle, _lib.ptr(img), _lib.ptr(dep), c, h, w, float(max_disparity),
                                                  _lib.ptr(left), _lib.ptr(lm), _lib.ptr(right), _lib.ptr(rm)))
    return back(left), back(lm), back(right), back(rm)


TEMPORAL_SIGMA = 6.0       # default sigma of the temporal filter's depth-difference weight, in 8-bit depth units


def check_temporal(radius, sigma) -> Tuple[int, float]:
    """(radius, sigma) of the temporal filter as (int, float); ValueError unless radius is an integer in 0..8 and sigma a
    number in (0, 64]."""
    if isinstance(radius, bool) or not isinstance(radius, (int, np.integer)) or not 0 <= radius <= _lib.TEMPORAL_MAX_RADIUS:
        raise ValueError(f'temporal radius must be an integer in [0, {_lib.TEMPORAL_MAX_RADIUS}], got {radius!r}')
    if isinstance(sigma, bool) or not isinstance(sigma, (int, float, np.integer, np.floating)) \
            or not 0.0 < float(sigma) <= _lib.TEMPORAL_MAX_SIGMA:
        raise ValueError(f'temporal sigma must be a number in (0, {_lib.TEMPORAL_MAX_SIGMA:g}], got {sigma!r}')
    return int(radius), float(sigma)


def _depth_planes(depths):
    """Contiguous uint8 / uint16 planes of one size, and their C enum."""
    planes = [np.ascontiguousarray(d) for d in depths]
    if not planes:
        raise ValueError('no depth maps')
    shape, dt = planes[0].shape, planes[0].dtype
    if len(shape) != 2 or any(d.shape != shape or d.dtype != dt for d in planes):
        raise ValueError('the depth maps of a window must be [H, W] arrays of one size and dtype')
    if dt not in (np.uint8, np.uint16):
        raise ValueError(f'temporal filtering takes uint8 or uint16 depth maps, not {dt}')
    return planes, _lib.depth_code(dt)


def temporal_depth(depths, t: int, radius: int, sigma: float = TEMPORAL_SIGMA):
    """The temporal filter alone: depth map t of the consecutive maps `depths`, filtered over its window.  Returns
    (float32 [H, W] in depth units, lo, hi), where lo..hi (indices into `depths`) is the window that survived the cut
    rule."""
    radius, sigma = check_temporal(radius, sigma)
    planes, code = _depth_planes(depths)
    if not 0 <= t < len(planes):
        raise ValueError(f'frame {t} is not one of the {len(planes)} depth maps')
    h, w = planes[0].shape
    out = np.empty((h, w), np.float32)
    lo, hi = C.c_int(), C.c_int()
    vp = C.c_void_p * len(planes)
    with _helper_lock:
        _lib.check(_lib.load().vsc_stage_temporal_depth(_ctx().handle, vp(*[d.ctypes.data for d in planes]), len(planes), int(t),
                                                        code, h, w, radius, sigma, _lib.ptr(out), C.byref(lo), C.byref(hi)))
    return out, lo.value, hi.value


# ------------------------------------------------------------------------------------------------
# the generator
# ------------------------------------------------------------------------------------------------
def _parse_device(device: str) -> int:
    dev = str(device)
    if dev == 'cuda':
        return _current_device()
    if dev.startswith('cuda:'):
        return int(dev.split(':', 1)[1])
    raise RuntimeError(
        f"StereoGenerator(device={device!r}): the B200 SBS path runs on CUDA only and has no CPU fallback; "
        "use the reference implementation for CPU processing")


class StereoGenerator:
    """Batch processor for stereo SBS image generation (reference: stereo_core.py:205-311).

    `process_frame(rgb, depth, params)` keeps the reference's numpy-in / numpy-out contract.
    `n_slots` frames can be in flight through `submit` / `collect` for the driver loop.
    `layout` (one of LAYOUTS, default the reference's 'sbs') sets the shape of every frame this generator returns, and
    `pixfmt` (one of PIXFMTS, default 'rgb24') with `matrix` (one of MATRICES, for the YUV formats) its pixel format.
    `encode='png'` (rgb24 only) makes every output path return the frame's PNG file as a 1-D uint8 array instead.
    """
    _DEFAULT_PARAMS = StereoParams()

    def __init__(self, device: str, n_slots: int = 1, group_size: int = 1, layout: str = 'sbs', pixfmt: str = 'rgb24',
                 matrix: str = 'bt709', encode: Optional[str] = None) -> None:
        self.device = device
        code, fcode, mcode, ecode = layout_code(layout), pixfmt_code(pixfmt), matrix_code(matrix), encode_code(encode)
        self._ctx = _lib.Context(_parse_device(device), n_slots, group_size)
        self._lib = _lib.load()
        _lib.check(self._lib.vsc_set_layout(self._ctx.handle, code))
        _lib.check(self._lib.vsc_set_pixfmt(self._ctx.handle, fcode, mcode))
        _lib.check(self._lib.vsc_set_encode(self._ctx.handle, ecode))
        self.layout, self.pixfmt, self.matrix, self.encode = layout, pixfmt, matrix, encode
        self.n_slots, self.group_size = n_slots, group_size
        self._pending = [None] * n_slots        # per slot: number of frames in flight
        # pinned staging per (slot, frame index within the slot's group): (key, rgb, depth, out) PinnedBuffers
        self._pinned = [[None] * group_size for _ in range(n_slots)]

    # -- reference API ---------------------------------------------------------------------------
    def process_frame(self, rgb: np.ndarray, depth: np.ndarray, params: StereoParams | None = None) -> np.ndarray:
        """Process a single frame to a side-by-side stereo image (left | right), uint8 [H, 2W, 3]
        (with another layout or pixel format: output_shape(layout, H, W, pixfmt) of output_dtype(pixfmt); with
        encode='png': the PNG file's bytes)."""
        p = params or self._DEFAULT_PARAMS
        rgb_c, depth_c, code = self._check_inputs(rgb, depth)
        h, w = rgb_c.shape[:2]
        out = np.empty(*self._out_spec(h, w))
        _lib.check(self._lib.vsc_process_frame(self._ctx.handle, _lib.ptr(rgb_c), _lib.ptr(depth_c), code, h, w,
                                               C.byref(_lib.make_params(p)), _lib.ptr(out)))
        return out[:self.encoded_bytes(0)].copy() if self.encode else out

    # -- asynchronous pipeline ---------------------------------------------------------------------
    def pinned_inputs(self, slot: int, h: int, w: int, depth_dtype=np.uint8, index: int = 0):
        """Page-locked (rgb[h,w,3], depth[h,w]) arrays of frame `index` of `slot` for a loader to decode into."""
        key = (int(h), int(w), np.dtype(depth_dtype).str)
        self.output_shape(h, w)             # a size the layout or format cannot take is refused before any buffer changes
        pin = self._pinned[slot][index]
        if pin is None or pin[0] != key:
            if self._pending[slot] is not None:
                raise RuntimeError(f'slot {slot} has an uncollected frame')
            if pin is not None:
                for b in pin[1:]:
                    b.free()
            pin = (key, _lib.PinnedBuffer((h, w, 3), np.uint8), _lib.PinnedBuffer((h, w), depth_dtype),
                   _lib.PinnedBuffer(*self._out_spec(h, w)))
            self._pinned[slot][index] = pin
        return pin[1].array, pin[2].array

    def submit_pinned(self, slot: int, params: StereoParams | None = None, n: int = 1) -> None:
        """Enqueue H2D + kernels + D2H for the n frames currently in the slot's pinned input arrays."""
        p = params or self._DEFAULT_PARAMS
        pins = self._pinned[slot][:n]
        if any(x is None for x in pins):
            raise RuntimeError('call pinned_inputs(slot, h, w, dtype, index) for every frame first')
        if self._pending[slot] is not None:
            raise RuntimeError(f'slot {slot} has an uncollected frame')
        if len({x[0] for x in pins}) != 1:
            raise ValueError('the frames of one submission must share size and depth dtype')
        h, w, _ = pins[0][0]
        vp = C.c_void_p * n
        _lib.check(self._lib.vsc_submit_group(
            self._ctx.handle, slot, n, vp(*[x[1].array.ctypes.data for x in pins]), vp(*[x[2].array.ctypes.data for x in pins]),
            _lib.depth_code(pins[0][2].array.dtype), h, w, C.byref(_lib.make_params(p)), vp(*[x[3].array.ctypes.data for x in pins])))
        self._pending[slot] = n

    def submit_host(self, slot: int, frames, params: StereoParams | None = None) -> None:
        """Enqueue H2D + kernels + D2H for up to `group_size` caller-owned (rgb, depth) arrays WITHOUT staging copies:
        the arrays are read by the copy engine directly (page-locked memory, e.g. _lib.PinnedBuffer, makes that copy
        asynchronous) and must stay untouched until the slot is collected.  Results land in the slot's pinned outputs."""
        p = params or self._DEFAULT_PARAMS
        frames = list(frames)
        n = len(frames)
        if not 1 <= n <= self.group_size:
            raise ValueError(f'a slot takes 1..{self.group_size} frames per submission')
        if self._pending[slot] is not None:
            raise RuntimeError(f'slot {slot} has an uncollected frame')
        h, w = frames[0][0].shape[:2]
        dt = frames[0][1].dtype
        for rgb, depth in frames:
            if (rgb.dtype != np.uint8 or rgb.shape != (h, w, 3) or depth.shape != (h, w) or depth.dtype != dt
                    or not rgb.flags.c_contiguous or not depth.flags.c_contiguous):
                raise ValueError('submit_host needs C-contiguous uint8 [H,W,3] frames and [H,W] depth maps of one size and dtype')
        outs = []
        for i in range(n):
            self.pinned_inputs(slot, h, w, dt, i)
            outs.append(self._pinned[slot][i][3].array.ctypes.data)
        vp = C.c_void_p * n
        _lib.check(self._lib.vsc_submit_group(
            self._ctx.handle, slot, n, vp(*[f[0].ctypes.data for f in frames]), vp(*[f[1].ctypes.data for f in frames]),
            _lib.depth_code(dt), h, w, C.byref(_lib.make_params(p)), vp(*outs)))
        self._pending[slot] = n
        self._held = getattr(self, '_held', {})
        self._held[slot] = frames            # keep the arrays alive until collect()

    def submit(self, slot: int, rgb: np.ndarray, depth: np.ndarray, params: StereoParams | None = None) -> None:
        """Copy one frame into the slot's pinned staging buffers and enqueue H2D + kernels + D2H."""
        self.submit_frames(slot, [(rgb, depth)], params)

    def submit_frames(self, slot: int, frames, params: StereoParams | None = None) -> None:
        """Same for up to `group_size` frames of identical size (they share the slot's stream and one
        hole-filling launch)."""
        frames = list(frames)
        if not 1 <= len(frames) <= self.group_size:
            raise ValueError(f'a slot takes 1..{self.group_size} frames per submission')
        for i, (rgb, depth) in enumerate(frames):
            rgb_c, depth_c, _ = self._check_inputs(rgb, depth)
            h, w = rgb_c.shape[:2]
            prgb, pdepth = self.pinned_inputs(slot, h, w, depth_c.dtype, i)
            np.copyto(prgb, rgb_c)
            np.copyto(pdepth, depth_c)
        self.submit_pinned(slot, params, len(frames))

    def submit_window(self, slot: int, frames, depths, first: int, params: StereoParams | None = None,
                      radius: int = 4, sigma: float = TEMPORAL_SIGMA) -> None:
        """Enqueue up to `group_size` consecutive clip frames with temporally filtered depth.  `frames` are their rgb
        arrays, `depths` the consecutive depth maps around them: frame i's own map is depths[first + i], and its window is
        every map within `radius` of it in `depths` (pass fewer at a clip end or a gap).  The rgb is staged in the slot's
        pinned buffers; the depth arrays are read in place and must stay untouched until the slot is collected.
        radius 0 is submit_frames."""
        radius, sigma = check_temporal(radius, sigma)
        p = params or self._DEFAULT_PARAMS
        frames = list(frames)
        n = len(frames)
        if not 1 <= n <= self.group_size:
            raise ValueError(f'a slot takes 1..{self.group_size} frames per submission')
        if self._pending[slot] is not None:
            raise RuntimeError(f'slot {slot} has an uncollected frame')
        planes, code = _depth_planes(depths)
        if not (0 <= first and first + n <= len(planes)):
            raise ValueError(f'frames {first}..{first + n - 1} are not all among the {len(planes)} depth maps')
        h, w = planes[0].shape
        for i, rgb in enumerate(frames):
            rgb_c, _, _ = self._check_inputs(rgb, planes[first + i])
            prgb, _ = self.pinned_inputs(slot, h, w, planes[0].dtype, i)
            np.copyto(prgb, rgb_c)
        pins = self._pinned[slot][:n]
        vp = C.c_void_p * n
        _lib.check(self._lib.vsc_submit_window(
            self._ctx.handle, slot, n, vp(*[x[1].array.ctypes.data for x in pins]), len(planes),
            (C.c_void_p * len(planes))(*[d.ctypes.data for d in planes]), int(first), code, h, w, radius, sigma,
            C.byref(_lib.make_params(p)), vp(*[x[3].array.ctypes.data for x in pins])))
        self._pending[slot] = n
        self._held = getattr(self, '_held', {})
        self._held[slot] = planes            # keep the maps alive until collect()

    def submit_device_window(self, slot: int, triples, d_depths, first: int, depth_dtype, h: int, w: int,
                             params: StereoParams | None = None, radius: int = 4, sigma: float = TEMPORAL_SIGMA) -> None:
        """Device-resident submit_window: `triples` = [(d_rgb, d_out)] raw device pointers (<= group_size), `d_depths` the
        window's depth maps (raw device pointers), frame i's own map d_depths[first + i]."""
        radius, sigma = check_temporal(radius, sigma)
        p = params or self._DEFAULT_PARAMS
        triples, d_depths = list(triples), list(d_depths)
        n = len(triples)
        vp = C.c_void_p * n
        _lib.check(self._lib.vsc_submit_device_window(
            self._ctx.handle, slot, n, vp(*[t[0] for t in triples]), len(d_depths), (C.c_void_p * len(d_depths))(*d_depths),
            int(first), _lib.depth_code(depth_dtype), h, w, radius, sigma, C.byref(_lib.make_params(p)),
            vp(*[t[1] for t in triples])))

    def collect(self, slot: int, copy: bool = True):
        """Wait for the slot's submission.  Returns the output frame (a list of frames if more than one was
        submitted).  copy=True returns fresh arrays the caller owns (the reference hands its result to another
        thread, sbs_generator.py:325, so it must not alias a reused buffer); copy=False returns the pinned
        outputs, valid until the slot is submitted again."""
        n = self._pending[slot]
        if n is None:
            raise RuntimeError(f'slot {slot} has no frame in flight')
        try:
            _lib.check(self._lib.vsc_wait(self._ctx.handle, slot))
        finally:
            self._pending[slot] = None
            getattr(self, '_held', {}).pop(slot, None)
        outs = [self._pinned[slot][i][3].array for i in range(n)]
        if self.encode:
            outs = [o[:self.encoded_bytes(slot, i)] for i, o in enumerate(outs)]
        if copy:
            outs = [o.copy() for o in outs]
        return outs[0] if n == 1 else outs

    def submit_device(self, slot: int, d_rgb: int, d_depth: int, depth_dtype, h: int, w: int, d_out: int,
                      params: StereoParams | None = None) -> None:
        """Device-resident variant: raw device pointers (e.g. torch tensor .data_ptr()), no copies.  d_out must hold
        output_shape(h, w) of output_dtype (self.output_shape, self.output_dtype); with encode='png', encoded_capacity
        bytes, of which encoded_bytes(slot) are the file once the slot has been waited for."""
        p = params or self._DEFAULT_PARAMS
        _lib.check(self._lib.vsc_submit_device(self._ctx.handle, slot, C.c_void_p(d_rgb), C.c_void_p(d_depth),
                                               _lib.depth_code(depth_dtype), h, w, C.byref(_lib.make_params(p)),
                                               C.c_void_p(d_out)))

    def submit_device_group(self, slot: int, triples, depth_dtype, h: int, w: int, params: StereoParams | None = None) -> None:
        """Device-resident group submission: `triples` = [(d_rgb, d_depth, d_out) raw device pointers] (<= group_size)."""
        p = params or self._DEFAULT_PARAMS
        triples = list(triples)
        n = len(triples)
        vp = C.c_void_p * n
        _lib.check(self._lib.vsc_submit_device_group(
            self._ctx.handle, slot, n, vp(*[t[0] for t in triples]), vp(*[t[1] for t in triples]), _lib.depth_code(depth_dtype),
            h, w, C.byref(_lib.make_params(p)), vp(*[t[2] for t in triples])))

    def encoded_bytes(self, slot: int, index: int = 0) -> int:
        """Bytes of the PNG file of frame `index` of the slot's last completed submission (encode='png')."""
        n = C.c_size_t()
        _lib.check(self._lib.vsc_encoded_bytes(self._ctx.handle, slot, index, C.byref(n)))
        return int(n.value)

    def wait(self, slot: int) -> None:
        _lib.check(self._lib.vsc_wait(self._ctx.handle, slot))

    def ready(self, slot: int) -> bool:
        """True once the slot's frame has finished on the device (wait/collect will not block)."""
        r = self._lib.vsc_query(self._ctx.handle, slot)
        if r < 0:
            _lib.check(r)
        return r == 1

    def wait_any(self, slots) -> int:
        """Sleep until one of the given in-flight slots has finished; returns that slot (not yet collected).
        The wait happens inside the library on a condition variable (no polling, the GIL is released)."""
        slots = list(slots)
        arr = (C.c_int * len(slots))(*slots)
        which = C.c_int(-1)
        while which.value < 0:
            _lib.check(self._lib.vsc_wait_any(self._ctx.handle, arr, len(slots), 2000, C.byref(which)))
            if which.value < 0:          # timed out: a faulted stream never runs its completion callback - surface the error
                for s in slots:
                    if self.ready(s):
                        return s
        return int(which.value)

    # -- producer-side depth post-processing (depth_map_generator.py:217-236) ------------------------
    def depth_post(self, depth: np.ndarray, size, bits: int = 16) -> Optional[np.ndarray]:
        """Bilinear resize of a float depth map to size = (width, height), min/max normalisation and quantisation to
        uint8 / uint16, as the reference's depth stage does before writing the file.  None if the map is flat."""
        d = np.ascontiguousarray(depth, np.float32)
        w, h = int(size[0]), int(size[1])
        out = np.empty((h, w), np.uint16 if bits == 16 else np.uint8)
        ok = C.c_int(0)
        _lib.check(self._lib.vsc_stage_depth_post(self._ctx.handle, _lib.ptr(d), d.shape[0], d.shape[1], h, w, int(bits), _lib.ptr(out), C.byref(ok)))
        return out if ok.value else None

    def depth_post_device(self, slot: int, d_depth: int, h: int, w: int, size, bits: int, d_out: int) -> None:
        """Device-resident variant on `slot`'s stream (raw device pointers): follow it with submit_device on the same
        slot and the quantised depth map never leaves the GPU."""
        _lib.check(self._lib.vsc_depth_post_device(self._ctx.handle, slot, C.c_void_p(d_depth), h, w, int(size[1]), int(size[0]), int(bits),
                                                   C.c_void_p(d_out)))

    # -- measurement -------------------------------------------------------------------------------
    def timer_begin(self) -> None:
        _lib.check(self._lib.vsc_timer_begin(self._ctx.handle))

    def timer_end(self) -> float:
        ms = C.c_float()
        _lib.check(self._lib.vsc_timer_end(self._ctx.handle, C.byref(ms)))
        return float(ms.value)

    def set_profiling(self, on: bool) -> None:
        _lib.check(self._lib.vsc_set_profiling(self._ctx.handle, int(on)))

    def kernel_times(self, slot: int = 0):
        names = (C.c_char_p * 64)()
        ms = (C.c_float * 64)()
        n = self._lib.vsc_slot_kernel_times(self._ctx.handle, slot, 64, names, ms)
        if n < 0:
            _lib.check(n)
        return [(names[i].decode(), float(ms[i])) for i in range(n)]

    def process_batch(self, frames: Iterable[Tuple[np.ndarray, np.ndarray]],
                      params: StereoParams | None = None, temporal: Optional[Tuple[int, float]] = None) -> List[np.ndarray]:
        """Run an iterable of (rgb, depth) through all slots, keeping `n_slots * group_size` frames in flight.
        Results are returned in input order.  With temporal=(radius, sigma) the frames are consecutive frames of one clip
        (one size, uint8 or uint16 depth) and every depth map is filtered over its neighbours (submit_window)."""
        frames = list(frames)
        if temporal is not None:
            return self._process_batch_temporal(frames, params, *check_temporal(*temporal))
        out: List[Optional[np.ndarray]] = [None] * len(frames)
        g = self.group_size
        chunks = [list(range(i, min(i + g, len(frames)))) for i in range(0, len(frames), g)]
        inflight: List[Tuple[int, List[int]]] = []
        free = list(range(self.n_slots))

        def harvest(slot, idxs):
            res = self.collect(slot)
            res = res if isinstance(res, list) else [res]
            for i, r in zip(idxs, res):
                out[i] = r
            free.append(slot)

        for idxs in chunks:
            # frames of one submission must share size / dtype: fall back to singles otherwise
            keys = {(frames[i][0].shape, frames[i][1].shape, frames[i][1].dtype.str) for i in idxs}
            parts = [idxs] if len(keys) == 1 else [[i] for i in idxs]
            for part in parts:
                if not free:
                    slot = self.wait_any([s for s, _ in inflight])
                    ids = next(x for s, x in inflight if s == slot)
                    inflight.remove((slot, ids))
                    harvest(slot, ids)
                slot = free.pop(0)
                self.submit_frames(slot, [frames[i] for i in part], params)
                inflight.append((slot, part))
        for slot, ids in inflight:
            harvest(slot, ids)
        return out  # type: ignore[return-value]

    def _process_batch_temporal(self, frames, params, radius: int, sigma: float) -> List[np.ndarray]:
        depths, _ = _depth_planes([f[1] for f in frames]) if frames else ([], None)
        out: List[Optional[np.ndarray]] = [None] * len(frames)
        inflight: List[Tuple[int, range]] = []
        free = list(range(self.n_slots))
        for a in range(0, len(frames), self.group_size):
            idxs = range(a, min(a + self.group_size, len(frames)))
            if not free:
                slot = self.wait_any([s for s, _ in inflight])
                ids = next(x for s, x in inflight if s == slot)
                inflight.remove((slot, ids))
                res = self.collect(slot)
                for i, r in zip(ids, res if isinstance(res, list) else [res]):
                    out[i] = r
                free.append(slot)
            slot = free.pop(0)
            lo, hi = max(0, idxs[0] - radius), min(len(frames) - 1, idxs[-1] + radius)
            self.submit_window(slot, [frames[i][0] for i in idxs], depths[lo:hi + 1], idxs[0] - lo, params, radius, sigma)
            inflight.append((slot, idxs))
        for slot, ids in inflight:
            res = self.collect(slot)
            for i, r in zip(ids, res if isinstance(res, list) else [res]):
                out[i] = r
        return out  # type: ignore[return-value]

    def last_frame_ms(self, slot: int = 0) -> float:
        ms = C.c_float()
        _lib.check(self._lib.vsc_slot_elapsed_ms(self._ctx.handle, slot, C.byref(ms)))
        return float(ms.value)

    def last_frame_launches(self, slot: int = 0) -> int:
        return int(self._lib.vsc_slot_launches(self._ctx.handle, slot))

    def close(self) -> None:
        for row in self._pinned:
            for pin in row:
                if pin is not None:
                    for b in pin[1:]:
                        b.free()
        self._pinned = [[None] * self.group_size for _ in range(self.n_slots)]
        self._ctx.close()

    def set_layout(self, layout: str) -> None:
        """Switch the output layout of frames submitted from now on.  Every slot must be collected: the pinned output
        buffers of the old shape are released (pinned_inputs allocates them again)."""
        code = layout_code(layout)
        if any(x is not None for x in self._pending):
            raise RuntimeError('collect every slot before changing the layout')
        _lib.check(self._lib.vsc_set_layout(self._ctx.handle, code))
        self.layout = layout
        self._release_pinned()

    def set_pixfmt(self, pixfmt: str, matrix: str = 'bt709') -> None:
        """Switch the pixel format (and YUV matrix) of frames submitted from now on.  Every slot must be collected, as for
        set_layout."""
        fcode, mcode = pixfmt_code(pixfmt), matrix_code(matrix)
        if any(x is not None for x in self._pending):
            raise RuntimeError('collect every slot before changing the pixel format')
        _lib.check(self._lib.vsc_set_pixfmt(self._ctx.handle, fcode, mcode))
        self.pixfmt, self.matrix = pixfmt, matrix
        self._release_pinned()

    def set_encode(self, encode: Optional[str]) -> None:
        """Switch the encoding of frames submitted from now on (None: raw frames, 'png').  Every slot must be collected,
        as for set_layout."""
        ecode = encode_code(encode)
        if any(x is not None for x in self._pending):
            raise RuntimeError('collect every slot before changing the encoding')
        _lib.check(self._lib.vsc_set_encode(self._ctx.handle, ecode))
        self.encode = encode
        self._release_pinned()

    # -- helpers -----------------------------------------------------------------------------------
    def _out_spec(self, h: int, w: int):
        """(shape, dtype) of the output buffer of one frame: the frame, or with an encoding its worst-case file."""
        if self.encode:
            return (encoded_capacity(self.layout, h, w),), np.dtype(np.uint8)
        return self.output_shape(h, w), self.output_dtype

    def output_shape(self, h: int, w: int) -> Tuple[int, ...]:
        """Shape of the frames this generator returns for h x w inputs."""
        return output_shape(self.layout, h, w, self.pixfmt)

    @property
    def output_dtype(self) -> np.dtype:
        """Element type of the frames this generator returns."""
        return output_dtype(self.pixfmt)

    def _release_pinned(self) -> None:
        """Free the pinned buffers of every slot (pinned_inputs allocates them again in the current output shape)."""
        for row in self._pinned:
            for i, pin in enumerate(row):
                if pin is not None:
                    for b in pin[1:]:
                        b.free()
                    row[i] = None

    @staticmethod
    def _check_inputs(rgb: np.ndarray, depth: np.ndarray):
        if rgb.ndim != 3 or rgb.shape[2] != 3:
            raise ValueError(f'rgb must be [H, W, 3], got {rgb.shape}')
        if rgb.dtype != np.uint8:
            rgb = rgb.astype(np.uint8)
        if depth.ndim != 2:
            raise ValueError(f'depth must be [H, W], got {depth.shape}')
        if depth.shape != rgb.shape[:2]:
            raise ValueError(f'depth {depth.shape} does not match frame {rgb.shape[:2]}')
        if depth.dtype not in (np.uint8, np.uint16, np.float32):
            # the reference casts any numeric dtype to float32 after cv2.resize (stereo_core.py:328)
            depth = depth.astype(np.float32)
        return np.ascontiguousarray(rgb), np.ascontiguousarray(depth), _lib.depth_code(depth.dtype)
