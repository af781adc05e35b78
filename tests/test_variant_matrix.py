"""The coverage manifest (variant_matrix.py) against the GPU test files' case lists and the library's source and
geometry.  No GPU needed."""
import os
import re

import numpy as np
import pytest

import test_gpu_stages as S
import test_gpu_variants as GV
import variant_matrix as VM
from conftest import ROOT

API = os.path.join(ROOT, 'video-stereo-converter_b200', 'csrc', 'vsc_api.cu')


def _case_cells():
    """(case name, cells) of every GPU case the manifest knows about; `new` marks the edge cases of this manifest."""
    out = []
    for c in S.LANCZOS_CASES:
        out.append((f'lanczos{c}', VM.lanczos_cells(*c), False))
    for c in S.LANCZOS_EDGE_CASES:
        out.append((f'lanczos{c}', VM.lanczos_cells(*c), True))
    for c in S.DEPTH_CASES:
        out.append((f'depth{c[:2]}', VM.depth_cells(*c), False))
    for c in S.DEPTH_EDGE_CASES:
        out.append((f'depth{c[:2]}', VM.depth_cells(*c), True))
    for c in S.WARP_CASES:
        out.append((f'warp{c}', VM.warp_cells(*c), False))
    for c in S.WARP_EDGE_CASES:
        out.append((f'warp{c}', VM.warp_cells(*c), True))
    out.append(('warp_scale255', VM.warp_cells(*S.WARP_SCALE255_CASE, scale255=True), False))
    for c in S.BACKEND_CASES:
        out.append((f'backend{c}', VM.backend_stage_cells(*c), False))
    for c in S.BACKEND_EDGE_CASES:
        out.append((f'backend{c}', VM.backend_stage_cells(*c), True))
    for c in GV.BILATERAL_CASES:
        out.append((f'bilateral{c}', VM.bilateral_cells(*c), True))
    for h, w, kw in GV.LAYOUT_FRAMES:
        out.append((f'layouts{(h, w, kw["super_sampling"])}', VM.layout_frame_cells(h, w, kw), True))
    for which in GV.WARP_MODE1_FRAMES:
        out.append((f'warp_mode1_{which}', {('warp-mode', 1, which)}, True))
    for c in GV.MARCH_CASES:
        out.append((f'march{c}', VM.march_cells(*c), True))
    out.append(('grouped_march', {('march-views', 8)}, True))
    for c in GV.MIN_FRAMES:
        out.append((f'min_frame{c}', VM.min_frame_cells(*c), True))
    for c in GV.DEVICE_OFFSETS:
        out.append((f'submit_device{c}', VM.device_offset_cells(*c), True))
    return out


def test_the_gpu_cases_reach_every_required_cell():
    reached = set().union(*(c for _, c, _ in _case_cells()))
    missing = sorted(VM.REQUIRED - reached, key=repr)
    assert not missing, f'{len(missing)} required cells no GPU case reaches: {missing[:20]}'


def test_every_edge_case_is_the_only_one_to_reach_some_cell():
    """Each edge case earns its place: removing it leaves a required cell unreached."""
    cases = _case_cells()
    count = {}
    for _, cells, _ in cases:
        for c in cells & VM.REQUIRED:
            count[c] = count.get(c, 0) + 1
    spare = [name for name, cells, new in cases if new and not any(count[c] == 1 for c in cells & VM.REQUIRED)]
    assert not spare, f'cases that reach no required cell of their own: {spare}'


def _instantiated(pattern):
    src = open(API).read()
    return sorted({int(x) for x in re.findall(pattern, src)})


def test_instantiation_lists_match_the_manifest():
    assert _instantiated(r'bilateral_kernel<(\d+)>') == sorted(VM.BILATERAL_RADII)
    assert _instantiated(r'launch_backend<(\d+)>\(layout') == sorted(VM.BACKEND_K)
    assert _instantiated(r'backend_attrs<(\d+)>\(big\)') == sorted(VM.BACKEND_K)
    assert _instantiated(r'telea_march_kernel<(\d+)>') == sorted(VM.MARCH_WARPS)
    assert _instantiated(r'depth_front_kernel<(\d+)>') == sorted(VM.DEPTH_FRONT_TAPS)
    src = open(API).read()
    layouts = set(re.findall(r'backend_kernel<K, (VSC_LAYOUT_\w+), P>', src))
    pixfmts = set(re.findall(r'backend_kernel<K, L, (VSC_PIXFMT_\w+)>', src))
    assert len(layouts) == len(VM.LAYOUTS) and len(pixfmts) == len(VM.PIXFMTS)


def _frame_cases():
    cases = [(h, w, kw) for h, w, kw in GV.LAYOUT_FRAMES]
    cases += [(h, w, GV.MIN_PARAMS[n]) for h, w, n in GV.MIN_FRAMES]
    cases += [GV.mode1_frame(x)[0].shape[:2] + (GV.mode1_frame(x)[2],) for x in GV.WARP_MODE1_FRAMES]
    frames, kw = GV.group_frames()
    cases.append(frames[0][0].shape[:2] + (kw,))
    cases.append((24, 70, dict(max_disparity=20.0, convergence=-4.0)))
    return cases


def test_restated_geometry_agrees_with_the_library():
    from vsc_b200 import _lib
    try:
        _lib.load()
    except OSError:
        pytest.skip('libvsc_b200.so is not built')
    import oracle as O
    for h, w, kw in _frame_cases():
        g = VM.geometry(h, w, VM.params(**kw))
        assert g['refused'] is None, (h, w, kw)
        lg = _lib.geometry(h, w, O.Params(**kw))
        assert (g['hs'], g['ws'], g['blur_k'], g['bilateral_d']) == (lg.ss_h, lg.ss_w, lg.blur_k, lg.bilateral_d), (h, w, kw)
        assert (g['lc'], g['rc'], g['cw']) == (lg.left_crop, lg.right_crop, lg.crop_w)
        assert g['K'] == VM.backend_k(lg.ss_h, lg.crop_w, h, w)
    for h, sw, kw in S.DEPTH_CASES + S.DEPTH_EDGE_CASES:
        assert VM.blur_k(kw.get('edge_softness', 20.0)) == O.soft_kernel_size(kw.get('edge_softness', 20.0)) or \
            kw.get('edge_softness') == 0.0


def test_march_cases_hold_the_task_counts_they_name():
    """A cluster's tasks are its hole pixels (march_order's return value); the sequential march model computes exactly
    rect_h * rect_w of them for each rectangle."""
    import oracle as O
    for rect_h, rect_w, _ in GV.MARCH_CASES:
        _, valid = GV.march_image(rect_h, rect_w)
        mask = O.dilate3(((1 - valid.astype(np.float32)) * 255).astype(np.uint8))
        _, order, _ = O.march_model(mask)
        assert order[mask > 0].max() + 1 == (mask > 0).sum() == rect_h * rect_w


@pytest.mark.parametrize('k', range(5, 32, 2))
@pytest.mark.parametrize('axis', ['h', 'w'])
def test_geometry_refuses_where_the_reflect_pad_raises(k, axis):
    """The depth blur pads by r = k // 2 with torch's reflect mode, which raises when r >= the side: vsc_geometry refuses
    exactly then (side r vs r + 1, at 1x so the side is the frame's own)."""
    import torch
    import oracle as O
    from vsc_b200 import _lib
    try:
        _lib.load()
    except OSError:
        pytest.skip('libvsc_b200.so is not built')
    r = k // 2
    es = k / 6
    assert VM.blur_k(es) == k
    for side in (r, r + 1):
        if side < 8:
            continue        # below the 8 x 8 minimum: refused for that reason
        h, w = (side, 64) if axis == 'h' else (64, side)
        p = dict(super_sampling=1.0, edge_softness=es, max_disparity=0.0, convergence=0.0)
        g = VM.geometry(h, w, VM.params(**p))
        hs, ws = g['hs'], g['ws']
        try:
            torch.nn.functional.pad(torch.zeros(1, 1, hs, ws), (r, r, r, r), mode='reflect')
            raises = False
        except RuntimeError:
            raises = True
        try:
            _lib.geometry(h, w, O.Params(**p))
            refused = False
        except _lib.VscError:
            refused = True
        assert refused == raises == (g['refused'] is not None), (k, axis, side)
