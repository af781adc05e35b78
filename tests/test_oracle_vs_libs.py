"""The oracle's restatements of third-party arithmetic against the libraries themselves (OpenCV and
PyTorch are part of the image; the reference calls exactly these functions, SURVEY.md Appendix A)."""
import numpy as np
import pytest

import oracle as O
from vsc_b200.synthetic import make_depth, make_rgb

cv2 = pytest.importorskip('cv2')
torch = pytest.importorskip('torch')
F = torch.nn.functional

from helper_reference import warp_literal  # noqa: E402  (needs torch)


@pytest.mark.parametrize('h,w,dw', [(37, 160, 270), (12, 1920, 2030), (6, 3840, 3949), (11, 100, 137)])
def test_lanczos4_bit_exact_vs_cv2(h, w, dw):
    rng = np.random.default_rng(h)
    for a in (rng.integers(0, 256, (h, w, 3), dtype=np.uint8), rng.integers(0, 256, (h, w), dtype=np.uint8),
              rng.integers(0, 65536, (h, w)).astype(np.uint16), rng.random((h, w), dtype=np.float32)):
        ref = cv2.resize(a, (dw, h), interpolation=cv2.INTER_LANCZOS4)
        assert np.array_equal(O.lanczos4_h(a, dw), ref), a.dtype


@pytest.mark.parametrize('h,w,s', [(120, 270, 3.0), (108, 203, 2.5), (64, 99, 1.3)])
def test_bilinear_bit_exact_vs_torch(h, w, s):
    rng = np.random.default_rng(w)
    x = rng.integers(0, 256, (3, h, w)).astype(np.float32)
    oh, ow = int(h * s), int(w * s)
    ref = F.interpolate(torch.from_numpy(x)[None], size=(oh, ow), mode='bilinear', align_corners=False)[0].numpy()
    assert np.array_equal(O.bilinear_up(x, oh, ow), ref)


def _kornia_blur(x, k, sigma):
    n = torch.arange(k, dtype=torch.float32) - (k // 2)
    g = torch.exp(-(n * n) / (2.0 * float(sigma) ** 2))
    g = g / g.sum()
    c = x.shape[1]
    x = F.conv2d(F.pad(x, (k // 2, k // 2, 0, 0), mode='reflect'), g.view(1, 1, 1, k).expand(c, 1, 1, k), groups=c)
    x = F.conv2d(F.pad(x, (0, 0, k // 2, k // 2), mode='reflect'), g.view(1, 1, k, 1).expand(c, 1, k, 1), groups=c)
    return x, g.numpy()


@pytest.mark.parametrize('k,sigma,c', [(31, 20.0, 1), (5, 1.0, 3), (13, 2.2, 1)])
def test_gaussian_blur_vs_torch_conv(k, sigma, c):
    rng = np.random.default_rng(k)
    x = rng.random((c, 90, 130), dtype=np.float32) * 255
    ref, taps = _kornia_blur(torch.from_numpy(x)[None], k, sigma)
    assert np.array_equal(O.gauss_taps(k, sigma), taps)
    # conv2d's summation order is backend- and shape-dependent (A.4): a couple of ulp, never more
    mine = O.gauss_blur(x, k, sigma)
    r = ref[0].numpy()
    assert np.abs(mine - r).max() <= 1e-6 * np.abs(r).max() * 4


def test_gauss_taps_match_torch_for_most_slider_values():
    bad = 0
    for es in np.arange(0.5, 30.5, 0.5):
        k = O.soft_kernel_size(float(es))
        n = torch.arange(k, dtype=torch.float32) - (k // 2)
        g = torch.exp(-(n * n) / (2.0 * float(es) ** 2))
        bad += not np.array_equal((g / g.sum()).numpy(), O.gauss_taps(k, float(es)))
    assert bad <= 6      # torch's vectorised expf differs from the correctly rounded exp for a few sigmas (<= 1 ulp)


def test_sharpen_and_area_pool_bit_exact_vs_torch():
    rng = np.random.default_rng(3)
    x = rng.integers(0, 256, (3, 120, 150)).astype(np.float32)
    xt = torch.from_numpy(x)[None]
    blur, _ = _kornia_blur(xt, 5, 1.0)
    ref = (xt + 14.0 * (xt - blur)).clamp(0, 255)
    mine = O.sharpen(x, 14.0)
    assert np.abs(mine - ref[0].numpy()).max() <= 2e-3      # 15x amplification of the blur's last ulp
    refn = np.ascontiguousarray(ref[0].numpy())
    for oh, ow in ((40, 50), (48, 60), (100, 111)):
        r = F.interpolate(ref, size=(oh, ow), mode='area')[0].numpy()
        assert np.array_equal(O.area_pool(refn, oh, ow), r)


@pytest.mark.parametrize('g', [0.1, 0.2, 0.55, 1.5, 2.0])
def test_gamma_within_one_ulp_of_torch(g):
    rng = np.random.default_rng(0)
    d = rng.random(200000, dtype=np.float32)
    ref = torch.pow(torch.from_numpy(d).clamp(0.001, 1.0), g).numpy()
    mine = O.apply_gamma(d, g)
    assert np.abs(ref.view(np.int32) - mine.view(np.int32)).max() <= 1
    exact = np.power(np.clip(d, np.float32(0.001), 1).astype(np.float64), float(np.float32(g))).astype(np.float32)
    assert (mine != exact).mean() < 1e-3          # the oracle's pow is correctly rounded almost everywhere


def test_pow_specification_tables_and_accuracy():
    """The deterministic pow (DESIGN.md, float order): its tables are what the specification says and the result is the
    correctly rounded power for every sampled input (the CUDA path is compared with this oracle bit for bit)."""
    import ctypes as C
    invc, log2c, exp2t = (C.c_double * 128)(), (C.c_double * 128)(), (C.c_double * 64)()
    O.lib().orc_pow_tables(invc, log2c, exp2t)
    c = 1.0 + (np.arange(128) + 0.5) / 128.0
    assert np.array_equal(np.array(invc), 1.0 / c)                               # IEEE division: exact agreement
    assert np.abs(np.array(log2c) - np.log2(c)).max() < 4e-16
    assert np.abs(np.array(exp2t) - np.exp2(np.arange(64) / 64.0)).max() < 4e-16 and exp2t[0] == 1.0
    rng = np.random.default_rng(7)
    x = np.clip(rng.random(400000, dtype=np.float32), np.float32(0.001), 1)
    x[:4] = [0.001, 1.0, 0.5, np.nextafter(np.float32(1), np.float32(0))]
    for g in (0.1, 0.2, 0.35, 0.9, 1.7, 2.5):
        exact = np.power(x.astype(np.float64), float(np.float32(g))).astype(np.float32)
        assert np.array_equal(O.apply_gamma(x, g), exact), g
    # ATen's special cases are float products (pow_tensor_scalar_optimized_kernel), not correctly rounded powers
    assert np.array_equal(O.apply_gamma(x, 2.0), x * x) and np.array_equal(O.apply_gamma(x, 3.0), (x * x) * x)


@pytest.mark.parametrize('kind', ['random', 'ties', 'ramp'])
def test_sort_free_warp_equals_literal_argsort_scatter(kind):
    rng = np.random.default_rng(5)
    h, w, md = 40, 300, 37.5
    img = rng.integers(0, 256, (3, h, w)).astype(np.float32)
    if kind == 'random':
        dep = rng.random((h, w), dtype=np.float32)
    elif kind == 'ties':
        dep = (np.rint(rng.random((h, w)) * 255) / 255).astype(np.float32)
    else:
        dep = np.tile(np.linspace(0, 1, w, dtype=np.float32)[None] ** 3, (h, 1))
    for sign in (+1, -1):
        ref_img, ref_mask = warp_literal(img, dep, md, sign)
        mine_img, mine_mask = O.warp(img, dep, md, sign)
        assert np.array_equal(mine_mask, ref_mask) and np.array_equal(mine_img, ref_img)


@pytest.mark.parametrize('s', [1.0, 2.0, 5.0])
def test_bilateral_vs_cv2(s):
    img = make_rgb(150, 210, seed=1)
    img[40:60, 50:90] = 0
    d, sc, ss = O.bilateral_params(s)
    mine = O.bilateral(img, d, sc, ss)
    ref = cv2.bilateralFilter(img, d=d, sigmaColor=30, sigmaSpace=s * 25)
    diff = np.abs(mine.astype(int) - ref.astype(int))
    assert diff.max() <= 1 and (diff > 0).mean() < 1e-4


def _telea_masks(h, w):
    rng = np.random.default_rng(5)
    yy, xx = np.mgrid[0:h, 0:w]
    m = [rng.random((h, w)) < 0.01]
    v = np.zeros((h, w), bool); v[:, 50] = True; m.append(v)
    v = np.zeros((h, w), bool); v[:, :25] = True; v[0:10, :] = True; m.append(v)
    v = np.zeros((h, w), bool); v[0, 0] = v[h - 1, w - 1] = v[0, w - 1] = v[h - 1, 0] = True; v[0, 50:60] = True; m.append(v)
    m.append((yy - 60) ** 2 + (xx - 80) ** 2 <= 35 ** 2)
    m.append(cv2.dilate((rng.random((h, w)) < 0.15).astype(np.uint8), np.ones((3, 3), np.uint8)) > 0)
    return m


def test_telea_bit_exact_vs_cv2():
    h, w = 120, 170
    img = make_rgb(h, w, seed=3)
    for hole in _telea_masks(h, w):
        mask = hole.astype(np.uint8) * 255
        ref = cv2.inpaint(img, mask, 3, cv2.INPAINT_TELEA)
        assert np.array_equal(O.telea(img, mask, 3), ref)
        assert np.array_equal(O.dilate3(mask), cv2.dilate(mask, np.ones((3, 3), np.uint8)))


def test_telea_order_then_colour_decomposition():
    """Arrival times and the computation order of hole pixels depend on the mask alone; computing the colours
    afterwards in that order ('still unknown' = later in the order) reproduces the one-pass algorithm exactly.
    This is the property the next step of the GPU march relies on (DESIGN.md section 6)."""
    rng = np.random.default_rng(21)
    for h, w, kind in [(60, 90, 'speckle'), (80, 70, 'dense'), (50, 120, 'cracks'), (64, 64, 'blob'), (40, 40, 'full-rows')]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        if kind == 'speckle':
            m = rng.random((h, w)) < 0.03
        elif kind == 'dense':
            m = rng.random((h, w)) < 0.35
        elif kind == 'cracks':
            m = np.zeros((h, w), bool); m[:, 20] = True; m[25, :] = True; m[5:45, 60:63] = True
        elif kind == 'blob':
            yy, xx = np.mgrid[:h, :w]; m = (yy - 30) ** 2 + (xx - 34) ** 2 < 15 ** 2
        else:
            m = np.zeros((h, w), bool); m[10:14] = True; m[:, :2] = True
        mask = m.astype(np.uint8) * 255
        one = O.telea(img, mask, 3)
        two = O.telea_two_pass(img, mask, 3)
        assert np.array_equal(one, two), kind
        assert np.array_equal(one, cv2.inpaint(img, mask, 3, cv2.INPAINT_TELEA)), kind


def test_march_model_equals_the_sequential_march():
    """The GPU march's schedule (T buckets of 0.7, stable sort by T, first-popped-neighbour ownership, prefix-sum task
    order, distances by fixed-point sweeps; march_model.c) gives the arrival times and the computation order of the
    one-pop-at-a-time algorithm, bit for bit, and needs few sweeps."""
    rng = np.random.default_rng(5)
    masks = []
    m = np.zeros((150, 200), np.uint8)
    for _ in range(20):
        cv2.circle(m, (int(rng.integers(0, 200)), int(rng.integers(0, 150))), int(rng.integers(1, 22)), 255, -1)
    masks.append(m)
    masks.append(cv2.dilate((rng.random((90, 120)) < 0.08).astype(np.uint8) * 255, np.ones((3, 3), np.uint8)))
    m = np.zeros((200, 150), np.uint8); m[:, 50:53] = 255; m[10:180, 90:130] = 255; m[100:103, :] = 255; m[:, :9] = 255
    masks.append(m)
    m = np.zeros((160, 160), np.uint8)
    cv2.line(m, (5, 5), (150, 110), 255, 3); cv2.line(m, (5, 155), (155, 20), 255, 7); cv2.ellipse(m, (80, 80), (60, 30), 30, 0, 360, 255, 5)
    masks.append(m)
    for mask in masks:
        img = rng.integers(0, 256, mask.shape + (3,), dtype=np.uint8)
        _, t = O.telea(img, mask, 3, return_t=True)
        _, order = O.telea_two_pass(img, mask, 3, return_order=True)
        t2, order2, stats = O.march_model(mask)
        assert np.array_equal(t.view(np.uint32), t2.view(np.uint32))
        assert np.array_equal(order, order2)
        assert stats['generations'] > 0 and stats['max_sweeps'] <= 8, stats
        assert stats['tasks'] >= int((mask > 0).sum())          # hole pixels + ring pixels


@pytest.mark.parametrize('h,w,H,W', [(153, 153, 108, 192), (96, 128, 270, 480), (77, 131, 50, 60)])
def test_depth_post_vs_cv2(h, w, H, W):
    """Producer-side depth post-processing (depth_map_generator.py:217-236): bilinear resize + min/max + quantise.
    Against OpenCV's own code (IPP off) the quantised maps agree except for <= 1 LSB at 16 bit on a few values of the
    clamped first / last rows; against the IPP build that ships: <= 1 LSB."""
    rng = np.random.default_rng(h)
    src = cv2.GaussianBlur(rng.random((h, w), dtype=np.float32) * 20 - 3, (0, 0), 3)
    try:
        for ipp in (False, True):
            cv2.ipp.setUseIPP(ipp)
            r = cv2.resize(src, (W, H), interpolation=cv2.INTER_LINEAR)
            for bits, q in ((8, 255), (16, 65535)):
                ref = (((r - r.min()) / (r.max() - r.min())) * q).round().astype(np.uint16 if bits == 16 else np.uint8)
                d = np.abs(O.depth_post(src, (W, H), bits).astype(int) - ref.astype(int))
                assert d.max() <= 1
                if not ipp:
                    assert (d > 0).sum() <= (0 if bits == 8 else 8)
    finally:
        cv2.ipp.setUseIPP(True)
    assert O.depth_post(np.full((9, 9), 2.5, np.float32), (20, 12), 16) is None        # flat map: no depth file


@pytest.mark.parametrize('seed', range(6))
def test_march_model_random_masks(seed):
    """Random mixtures of speckle, lines, blobs and border-touching bands: the generation schedule reproduces the
    sequential march's arrival times and order on every one of them."""
    rng = np.random.default_rng(100 + seed)
    h, w = int(rng.integers(40, 110)), int(rng.integers(40, 140))
    m = (rng.random((h, w)) < rng.choice([0.0, 0.01, 0.05])).astype(np.uint8) * 255
    for _ in range(int(rng.integers(0, 6))):
        p0 = (int(rng.integers(0, w)), int(rng.integers(0, h))); p1 = (int(rng.integers(0, w)), int(rng.integers(0, h)))
        cv2.line(m, p0, p1, 255, int(rng.integers(1, 6)))
    for _ in range(int(rng.integers(0, 4))):
        cv2.circle(m, (int(rng.integers(0, w)), int(rng.integers(0, h))), int(rng.integers(2, 18)), 255, -1)
    if seed % 2:
        m[:, :int(rng.integers(1, 30))] = 255
    if seed % 3 == 0:
        m[-int(rng.integers(1, 12)):, :] = 255
    if not m.any():
        m[h // 2, w // 2] = 255
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    _, t = O.telea(img, m, 3, return_t=True)
    _, order = O.telea_two_pass(img, m, 3, return_order=True)
    t2, order2, stats = O.march_model(m)
    assert np.array_equal(t.view(np.uint32), t2.view(np.uint32)) and np.array_equal(order, order2)
    assert stats['max_sweeps'] <= 10


def test_telea_known_answers():
    """const-101 image with a 1-px hole inpaints to 102 (+0.5 and round both apply), const-100 to 100 (SURVEY 8c-v)."""
    for val, want in ((101, 102), (100, 100)):
        img = np.full((20, 20, 3), val, np.uint8)
        mask = np.zeros((20, 20), np.uint8)
        mask[10, 10] = 255
        out = O.telea(img, mask, 3)
        assert out[10, 10, 0] == want == cv2.inpaint(img, mask, 3, cv2.INPAINT_TELEA)[10, 10, 0]


def test_truncation_not_rounding():
    assert O.to_u8_trunc(np.array([254.999, 0.6, 300.0, -3.0], np.float32)).tolist() == [254, 0, 255, 0]
