"""ctypes binding of libvsc_b200.so (include/vsc_b200.h).  No torch types cross this boundary."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

# Frames in flight live on separate CUDA streams; with the default of 8 hardware work queues, streams beyond
# the 8th alias onto the same queue and serialise.  Must be set before the CUDA context is created.
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('VSC_B200_LIB', os.path.normpath(os.path.join(_HERE, '..', 'lib', 'libvsc_b200.so')))

VSC_OK, VSC_E_INVALID, VSC_E_PARAMS, VSC_E_CUDA, VSC_E_NOMEM, VSC_E_STATE = 0, -1, -2, -3, -4, -5
DEPTH_U8, DEPTH_U16, DEPTH_F32 = 0, 1, 2
LAYOUT_SBS, LAYOUT_HALF_SBS, LAYOUT_TB, LAYOUT_HALF_TB, LAYOUT_ANAGLYPH = 0, 1, 2, 3, 4
PIXFMT_RGB24, PIXFMT_YUV420P, PIXFMT_YUV420P10LE = 0, 1, 2
MATRIX_BT709, MATRIX_BT601 = 0, 1
ENCODE_NONE, ENCODE_PNG = 0, 1
GPU_ERROR_EXIT_CODE = 100      # sbs_generator.py:41

EXPORTS = [
    'vsc_abi_version', 'vsc_last_error', 'vsc_default_params', 'vsc_create', 'vsc_create_grouped', 'vsc_group_size',
    'vsc_submit_group', 'vsc_submit_device_group', 'vsc_destroy', 'vsc_device',
    'vsc_num_slots', 'vsc_geometry', 'vsc_process_frame', 'vsc_host_alloc', 'vsc_host_free', 'vsc_submit',
    'vsc_wait', 'vsc_query', 'vsc_wait_any', 'vsc_submit_device', 'vsc_sync', 'vsc_slot_stream', 'vsc_slot_elapsed_ms', 'vsc_slot_launches',
    'vsc_stage_lanczos', 'vsc_stage_depth', 'vsc_stage_warp', 'vsc_stage_bilateral', 'vsc_stage_inpaint',
    'vsc_stage_backend', 'vsc_stage_depth_post', 'vsc_depth_post_device', 'vsc_stage_warp_f32', 'vsc_stage_normalize_f32', 'vsc_stage_gamma_f32',
    'vsc_set_profiling', 'vsc_slot_kernel_times', 'vsc_timer_begin', 'vsc_timer_end', 'vsc_debug_fetch',
    'vsc_debug_telea_state', 'vsc_debug_telea_stats', 'vsc_debug_set_telea_capacity', 'vsc_debug_selftest',
    'vsc_layout_shape', 'vsc_set_layout', 'vsc_output_size', 'vsc_set_pixfmt',
    'vsc_set_encode', 'vsc_encoded_capacity', 'vsc_encoded_bytes', 'vsc_stage_png', 'vsc_debug_png_stats',
]


class VscParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in ('max_disparity', 'convergence', 'super_sampling', 'edge_softness',
                                          'artifact_smoothing', 'depth_gamma', 'sharpen')]


class VscGeom(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('height', 'width', 'stretched_w', 'ss_h', 'ss_w', 'left_crop', 'right_crop',
                                         'crop_w', 'blur_k', 'bilateral_d', 'super_sampled')]


class VscError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f'libvsc_b200: {msg} (code {code})')
        self.code = code


class VscCudaError(VscError):
    """CUDA failure: drivers of the frame loop exit with GPU_ERROR_EXIT_CODE (sbs_generator.py:317)."""


_lib = None


def load():
    """Load the CUDA library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} not found: build it with video-stereo-converter_b200/csrc/build.sh '
            '(or __graft_entry__.build()).  The B200 SBS path has no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    vp, i, d = C.c_void_p, C.c_int, C.c_double
    lib.vsc_abi_version.restype = i
    lib.vsc_last_error.restype = C.c_char_p
    lib.vsc_default_params.argtypes = [C.POINTER(VscParams)]
    lib.vsc_default_params.restype = None
    lib.vsc_create.argtypes = [i, i, C.POINTER(vp)]
    lib.vsc_create_grouped.argtypes = [i, i, i, C.POINTER(vp)]
    lib.vsc_group_size.argtypes = [vp]
    lib.vsc_submit_group.argtypes = [vp, i, i, C.POINTER(vp), C.POINTER(vp), i, i, i, C.POINTER(VscParams), C.POINTER(vp)]
    lib.vsc_submit_device_group.argtypes = [vp, i, i, C.POINTER(vp), C.POINTER(vp), i, i, i, C.POINTER(VscParams), C.POINTER(vp)]
    lib.vsc_destroy.argtypes = [vp]
    lib.vsc_destroy.restype = None
    lib.vsc_device.argtypes = [vp]
    lib.vsc_num_slots.argtypes = [vp]
    lib.vsc_geometry.argtypes = [i, i, C.POINTER(VscParams), C.POINTER(VscGeom)]
    lib.vsc_stage_depth_post.argtypes = [vp, vp, i, i, i, i, i, vp, C.POINTER(C.c_int)]
    lib.vsc_depth_post_device.argtypes = [vp, i, vp, i, i, i, i, i, vp]
    lib.vsc_wait_any.argtypes = [vp, C.POINTER(C.c_int), i, i, C.POINTER(C.c_int)]
    lib.vsc_process_frame.argtypes = [vp, vp, vp, i, i, i, C.POINTER(VscParams), vp]
    lib.vsc_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    lib.vsc_host_free.argtypes = [vp]
    lib.vsc_submit.argtypes = [vp, i, vp, vp, i, i, i, C.POINTER(VscParams), vp]
    lib.vsc_submit_device.argtypes = [vp, i, vp, vp, i, i, i, C.POINTER(VscParams), vp]
    lib.vsc_wait.argtypes = [vp, i]
    lib.vsc_query.argtypes = [vp, i]
    lib.vsc_sync.argtypes = [vp]
    lib.vsc_slot_stream.argtypes = [vp, i]
    lib.vsc_slot_stream.restype = vp
    lib.vsc_slot_elapsed_ms.argtypes = [vp, i, C.POINTER(C.c_float)]
    lib.vsc_slot_launches.argtypes = [vp, i]
    lib.vsc_stage_lanczos.argtypes = [vp, vp, i, i, i, i, i, vp]
    lib.vsc_stage_depth.argtypes = [vp, vp, i, i, i, i, C.POINTER(VscParams), vp]
    lib.vsc_stage_warp.argtypes = [vp, vp, vp, i, i, i, i, d, i, vp, vp, vp, vp, vp]
    lib.vsc_stage_bilateral.argtypes = [vp, vp, i, i, d, vp]
    lib.vsc_stage_inpaint.argtypes = [vp, vp, vp, i, i, i, i]
    lib.vsc_stage_backend.argtypes = [vp, vp, vp, i, i, i, i, i, i, i, d, vp]
    lib.vsc_stage_warp_f32.argtypes = [vp, vp, vp, i, i, i, d, vp, vp, vp, vp]
    lib.vsc_stage_normalize_f32.argtypes = [vp, vp, C.c_size_t, vp]
    lib.vsc_stage_gamma_f32.argtypes = [vp, vp, C.c_size_t, d, vp]
    lib.vsc_set_profiling.argtypes = [vp, i]
    lib.vsc_slot_kernel_times.argtypes = [vp, i, i, C.POINTER(C.c_char_p), C.POINTER(C.c_float)]
    lib.vsc_timer_begin.argtypes = [vp]
    lib.vsc_timer_end.argtypes = [vp, C.POINTER(C.c_float)]
    lib.vsc_debug_fetch.argtypes = [vp, i, vp, C.c_size_t]
    lib.vsc_debug_telea_state.argtypes = [vp, i, vp, vp, vp, C.c_size_t]
    lib.vsc_debug_telea_stats.argtypes = [vp, vp]
    lib.vsc_debug_set_telea_capacity.argtypes = [vp, C.c_size_t]
    lib.vsc_debug_selftest.argtypes = [vp, i, C.POINTER(C.c_ulonglong)]
    lib.vsc_layout_shape.argtypes = [i, i, i, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.vsc_set_layout.argtypes = [vp, i]
    lib.vsc_output_size.argtypes = [i, i, i, i, C.POINTER(C.c_size_t)]
    lib.vsc_set_pixfmt.argtypes = [vp, i, i]
    lib.vsc_set_encode.argtypes = [vp, i]
    lib.vsc_encoded_capacity.argtypes = [i, i, i, i, C.POINTER(C.c_size_t)]
    lib.vsc_encoded_bytes.argtypes = [vp, i, i, C.POINTER(C.c_size_t)]
    lib.vsc_stage_png.argtypes = [vp, vp, i, i, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.vsc_debug_png_stats.argtypes = [vp, C.POINTER(C.c_ulonglong)]
    if lib.vsc_abi_version() != 1:
        raise ImportError('libvsc_b200.so ABI version mismatch')
    _lib = lib
    return lib


def check(rc: int):
    if rc == VSC_OK:
        return
    msg = (load().vsc_last_error() or b'').decode('utf-8', 'replace')
    if rc == VSC_E_CUDA:
        raise VscCudaError(rc, msg)
    raise VscError(rc, msg)


def ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


def make_params(p) -> VscParams:
    return VscParams(float(p.max_disparity), float(p.convergence), float(p.super_sampling), float(p.edge_softness),
                     float(p.artifact_smoothing), float(p.depth_gamma), float(p.sharpen))


def depth_code(dtype) -> int:
    dt = np.dtype(dtype)
    if dt == np.uint8:
        return DEPTH_U8
    if dt == np.uint16:
        return DEPTH_U16
    if dt == np.float32:
        return DEPTH_F32
    raise TypeError(f'depth dtype {dt} not supported (uint8, uint16, float32)')


def geometry(h: int, w: int, p) -> VscGeom:
    g = VscGeom()
    check(load().vsc_geometry(int(h), int(w), C.byref(make_params(p)), C.byref(g)))
    return g


class PinnedBuffer:
    """Page-locked host array for the double-buffered frame pipeline."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(load().vsc_host_alloc(max(nbytes, 1), C.byref(p)))
        self._p = p
        buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._p is not None:
            self.array = None
            load().vsc_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """Owns a vsc_ctx (one CUDA device, n_slots frames in flight)."""

    def __init__(self, device: int = 0, n_slots: int = 1, group_size: int = 1):
        self._lib = load()
        h = C.c_void_p()
        check(self._lib.vsc_create_grouped(int(device), int(n_slots), int(group_size), C.byref(h)))
        self._h = h
        self.device, self.n_slots, self.group_size = int(device), int(n_slots), int(group_size)

    def close(self):
        if getattr(self, '_h', None):
            self._lib.vsc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h
