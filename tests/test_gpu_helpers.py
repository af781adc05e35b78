"""The module-level helpers normalize_depth, apply_depth_gamma and forward_warp_stereo over their whole input domain.

The reference's helpers are plain torch and take any float tensor, so each helper is compared bit for bit (NaN positions
included) with the torch CPU restatement in helper_reference.py: negative, signed-zero, unnormalised, huge and
non-finite depth, rows wider than one warp segment (1024 targets), and more.  apply_depth_gamma is also held within
1 ulp of torch.pow itself.  The tests without the gpu mark pin the CPU oracle against the same restatement where the
oracle restates these operations, and check the helpers' argument errors.
"""
import threading

import numpy as np
import pytest

import oracle as O

torch = pytest.importorskip('torch')

import helper_reference as HR  # noqa: E402  (needs torch)
from vsc_b200 import apply_depth_gamma, forward_warp_stereo, normalize_depth  # noqa: E402

gpu = pytest.mark.gpu


def same(a, b) -> bool:
    """Bit-exact equality of two float arrays or tensors, NaN positions included (NaN payloads are not compared)."""
    a = a.numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint8), b[~nb].view(np.uint8)))


def ulp_diff(a: np.ndarray, b: np.ndarray) -> int:
    """Largest distance in float32 units in the last place between two arrays of non-negative floats."""
    return int(np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)).max())


# ---- inputs --------------------------------------------------------------------------------------------------------
NORM_KINDS = ('random', 'negative', 'mixed_zero', 'below_1e-6', 'above_1e-6', 'constant', 'float_max', 'pos_inf', 'neg_inf',
              'nan')
NORM_SHAPES = ((1,), (31,), (32,), (33,), (2 ** 20 + 7,), (1, 1), (32, 33), (1, 1, 31, 33), (1, 1, 1, 1))


def norm_input(kind: str, shape, seed: int = 0) -> torch.Tensor:
    """A float32 tensor of `shape` for normalize_depth.  Where both signed zeros occur the minimum is negative: the
    reference's result for -0.0 - min depends on which zero torch's min() returns when the minimum is a zero."""
    rng = np.random.default_rng(seed)
    n = int(np.prod(shape))
    f32 = np.float32
    if kind == 'random':
        a = rng.random(n, dtype=f32) * 7 + 3
    elif kind == 'negative':
        a = -(rng.random(n, dtype=f32) * 5 + f32(0.5))
    elif kind == 'mixed_zero':
        a = rng.random(n, dtype=f32) * 2 - 1
        a[0::5], a[2::5] = 0.0, -0.0
        a[-1] = -0.75
    elif kind in ('below_1e-6', 'above_1e-6'):
        top = np.nextafter(f32(1e-6), f32(0 if kind == 'below_1e-6' else 1))   # unambiguous in float32 and float64
        a = rng.random(n, dtype=f32) * top
        a[0], a[-1] = 0.0, top
    elif kind == 'constant':
        a = np.full(n, 3.5, f32)
    elif kind == 'float_max':        # every value above 3.4e38: the minimum must not start from a finite sentinel
        a = np.full(n, np.finfo(f32).max, f32)
        a[1::2] = np.nextafter(np.finfo(f32).max, f32(0))
    else:
        a = rng.random(n, dtype=f32) * 2 - 0.5
        a[n // 2] = {'pos_inf': np.inf, 'neg_inf': -np.inf, 'nan': np.nan}[kind]
    return torch.from_numpy(a.reshape(shape))


GAMMAS = (0.01, 0.1, 0.2, 1.0, 2.0, 3.0, 7.5, 13.0, 20.0, 0.0, -1.5)


def gamma_input(with_nan: bool = True) -> np.ndarray:
    rng = np.random.default_rng(11)
    f32 = np.float32
    special = [0.0, -0.0, 1e-4, 5e-4, 0.001, np.nextafter(f32(0.001), f32(0)), np.nextafter(f32(0.001), f32(1)),
               0.5, np.nextafter(f32(1), f32(0)), 1.0, 1.5, 2.0, -0.3, -5.0, 1e-40, 3e38, np.inf, -np.inf]
    if with_nan:
        special += [np.nan, -np.nan]
    return np.concatenate([np.array(special, f32), rng.random(65536, dtype=f32) * 1.2 - 0.1,
                           rng.random(4096, dtype=f32) * 0.002])


WARP_KINDS = ('random', 'ties', 'ramp', 'negative', 'mixed_zero', 'unnormalised', 'huge', 'nonfinite')
WARP_WIDTHS = (1, 31, 1023, 1024, 1025, 2049, 3000)
WARP_MDS = (0.0, 0.5, 33.0, -33.0, 250.0)


def warp_depth(kind: str, h: int, w: int, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    f32 = np.float32
    u = rng.random((h, w), dtype=f32)
    if kind == 'random':
        return u
    if kind == 'ties':             # u8-quantised, as a depth map decoded from an 8-bit file
        return (np.rint(u * 255) / f32(255)).astype(f32)
    if kind == 'ramp':
        return np.tile(np.linspace(0, 1, w, dtype=f32)[None] ** 3, (h, 1)).astype(f32)
    if kind == 'negative':
        return -(u + f32(0.001))
    if kind == 'mixed_zero':
        d = u * 2 - 1
        d[rng.random((h, w)) < 0.15] = 0.0
        d[rng.random((h, w)) < 0.15] = -0.0
        return d
    if kind == 'unnormalised':     # |d * md| well beyond one 1024-target segment's old halo
        return u * 8
    if kind == 'huge':             # |d * md| > 2^31 for most sources; the rest move normally
        d = u.copy()
        pick = rng.random((h, w)) < 0.6
        d[pick] = (np.sign(u[pick] - 0.3) * 10.0 ** (8 + 2 * u[pick])).astype(f32)
        return d
    if kind == 'nonfinite':
        d = u.copy()
        r = rng.random((h, w))
        d[r < 0.04], d[(r >= 0.04) & (r < 0.07)], d[(r >= 0.07) & (r < 0.1)] = np.nan, np.inf, -np.inf
        return d
    raise ValueError(kind)


def unique_image(c: int, h: int, w: int, seed: int = 0) -> np.ndarray:
    """Distinct value per pixel and channel: a wrong source shows up in the colours as well as in the masks."""
    return (np.random.default_rng(seed).permutation(c * h * w) + 1).astype(np.float32).reshape(c, h, w)


def check_warp(img: np.ndarray, dep: np.ndarray, md: float) -> None:
    c, h, w = img.shape
    got = forward_warp_stereo(torch.from_numpy(img)[None], torch.from_numpy(dep)[None, None], md)
    ref = HR.forward_warp_stereo(torch.from_numpy(img)[None], torch.from_numpy(dep)[None, None], md)
    for name, g, r in zip(('left', 'left_mask', 'right', 'right_mask'), got, ref):
        assert g.shape == r.shape and g.dtype == torch.float32, name
        if not same(g, r):
            bad = np.argwhere(g.numpy() != r.numpy())
            raise AssertionError(f'{name}: {len(bad)} values differ (C={c}, W={w}, md={md}), first at {bad[0].tolist()}')


# ---- CPU: the restatement's assumptions, the oracle against it, argument errors -------------------------------------
def test_floor_long_of_non_finite_is_negative():
    """warp_literal drops a source whose target is NaN, ±inf or outside int64 because torch's floor().long() gives
    INT64_MIN for it on the CPU; were that not so here, the restatement would not be the reference's behaviour."""
    t = torch.tensor([np.nan, np.inf, -np.inf, 1e20, -1e20, 3.5e9], dtype=torch.float32)
    assert (t.floor().long()[:5] < 0).all() and int(t.floor().long()[5]) == 3500000000


def test_gamma_restatement_within_one_ulp_of_torch_pow():
    x = torch.from_numpy(gamma_input())
    for g in GAMMAS:
        ref, tp = HR.apply_depth_gamma(x, g).numpy(), torch.pow(torch.clamp(x, 0.001, 1.0), g).numpy()
        nan = np.isnan(ref)
        assert np.array_equal(nan, np.isnan(tp)) and ulp_diff(ref[~nan], tp[~nan]) <= 1, g


@pytest.mark.parametrize('kind', [k for k in NORM_KINDS if k != 'nan'])
def test_oracle_normalize_equals_restatement(kind):
    """The oracle restates the pipeline's normalisation, which is not specified for NaN depth; every other kind must agree."""
    for shape in NORM_SHAPES:
        d = norm_input(kind, shape)
        assert same(O.normalize_depth(d.numpy().ravel()), HR.normalize_depth(d).numpy().ravel()), shape


def test_oracle_gamma_equals_restatement():
    x = gamma_input(with_nan=False)
    for g in GAMMAS:
        assert same(O.apply_gamma(x, g), HR.apply_depth_gamma(torch.from_numpy(x), g)), g


@pytest.mark.parametrize('kind', WARP_KINDS)
def test_oracle_warp_equals_restatement(kind):
    for i, w in enumerate((31, 1025, 3000)):
        dep = warp_depth(kind, 3, w, seed=i)
        img = unique_image((1, 3, 4)[i], 3, w, seed=i)
        for md in WARP_MDS:
            for sign in (+1, -1):
                ref_img, ref_mask = HR.warp_literal(img, dep, md, sign)
                o_img, o_mask = O.warp(img, dep, md, sign)
                assert np.array_equal(o_mask, ref_mask) and same(o_img, ref_img), (w, md, sign)


def test_warp_argument_errors():
    img = torch.zeros(2, 3, 4, 5)
    with pytest.raises(RuntimeError):
        forward_warp_stereo(img, torch.zeros(2, 1, 4, 5), 10.0)          # B != 1
    with pytest.raises(RuntimeError):
        forward_warp_stereo(torch.zeros(3, 4, 5), torch.zeros(1, 1, 4, 5), 10.0)
    with pytest.raises(RuntimeError):
        forward_warp_stereo(img[:1], torch.zeros(1, 1, 4, 6), 10.0)       # depth is not H x W


# ---- GPU: the helpers against the restatement -----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize('kind', NORM_KINDS)
def test_normalize_depth(kind):
    for shape in NORM_SHAPES:
        d = norm_input(kind, shape)
        got = normalize_depth(d)
        assert got.shape == d.shape and got.dtype == torch.float32
        assert same(got, HR.normalize_depth(d)), shape


@gpu
@pytest.mark.parametrize('g', GAMMAS)
def test_apply_depth_gamma(g):
    x = torch.from_numpy(gamma_input())
    got = apply_depth_gamma(x, g)
    assert same(got, HR.apply_depth_gamma(x, g))
    tp = torch.pow(torch.clamp(x, 0.001, 1.0), g).numpy()
    nan = np.isnan(tp)
    assert np.array_equal(np.isnan(got.numpy()), nan) and ulp_diff(got.numpy()[~nan], tp[~nan]) <= 1


@gpu
@pytest.mark.parametrize('w', WARP_WIDTHS)
@pytest.mark.parametrize('kind', WARP_KINDS)
def test_forward_warp_stereo(kind, w):
    h = 3
    dep = warp_depth(kind, h, w, seed=w)
    for i, md in enumerate(WARP_MDS):
        check_warp(unique_image((1, 3, 4)[(i + w) % 3], h, w, seed=i), dep, md)


@gpu
def test_cuda_inputs_come_back_on_their_device():
    rng = np.random.default_rng(3)
    d = torch.from_numpy(rng.random((1, 1, 20, 1100), dtype=np.float32) * 4 - 1)
    img = torch.from_numpy(unique_image(3, 20, 1100))[None]
    dc, ic = d.cuda(), img.cuda()
    n = normalize_depth(dc)
    assert n.device == dc.device and n.dtype == torch.float32 and same(n.cpu(), HR.normalize_depth(d))
    g = apply_depth_gamma(dc, 0.2)
    assert g.device == dc.device and same(g.cpu(), HR.apply_depth_gamma(d, 0.2))
    got = forward_warp_stereo(ic, dc, 40.0)
    for a, b in zip(got, HR.forward_warp_stereo(img, d, 40.0)):
        assert a.device == dc.device and a.dtype == torch.float32 and same(a.cpu(), b)


@gpu
def test_non_contiguous_inputs():
    rng = np.random.default_rng(4)
    base = torch.from_numpy(rng.random((1, 1, 40, 2100), dtype=np.float32) * 3)
    d = base[..., ::2]                                    # [1, 1, 40, 1050], strided
    img = torch.from_numpy(unique_image(3, 1050, 40)).permute(0, 2, 1)[None]     # [1, 3, 40, 1050], transposed
    assert not d.is_contiguous() and not img.is_contiguous()
    assert same(normalize_depth(d), HR.normalize_depth(d.contiguous()))
    assert same(apply_depth_gamma(d, 0.35), HR.apply_depth_gamma(d.contiguous(), 0.35))
    for a, b in zip(forward_warp_stereo(img, d, 90.0), HR.forward_warp_stereo(img.contiguous(), d.contiguous(), 90.0)):
        assert same(a, b)


@gpu
@pytest.mark.parametrize('dtype', [torch.float64, torch.float16])
def test_other_dtypes_compute_in_float32(dtype):
    """The helpers compute in float32 and cast the results back to the input's dtype (INTEGRATION.md)."""
    rng = np.random.default_rng(5)
    d = torch.from_numpy(rng.random((1, 1, 12, 1500)) * 6 - 2).to(dtype)
    img = torch.from_numpy(unique_image(3, 12, 1500) / 64).to(dtype)[None]
    n = normalize_depth(d)
    assert n.dtype == dtype and same(n, HR.normalize_depth(d.float()).to(dtype))
    g = apply_depth_gamma(d, 0.2)
    assert g.dtype == dtype and same(g, HR.apply_depth_gamma(d.float(), 0.2).to(dtype))
    for a, b in zip(forward_warp_stereo(img, d, 30.0), HR.forward_warp_stereo(img.float(), d.float(), 30.0)):
        assert a.dtype == dtype and same(a, b.to(dtype))


@gpu
def test_concurrent_calls_equal_calls_made_alone():
    """Eight threads call the helpers at once; every result equals the same call made alone."""
    rng = np.random.default_rng(6)
    calls = []
    for k in range(8):
        d = torch.from_numpy((rng.random((1, 1, 64, 1500), dtype=np.float32) * (k + 1) - k / 3).astype(np.float32))
        if k % 3 == 0:
            calls.append((normalize_depth, (d,)))
        elif k % 3 == 1:
            calls.append((apply_depth_gamma, (d, 0.1 * k)))
        else:
            calls.append((forward_warp_stereo, (torch.from_numpy(unique_image(3, 64, 1500, seed=k))[None], d, 20.0 * k)))

    def flat(r):
        return r if isinstance(r, tuple) else (r,)

    alone = [flat(f(*a)) for f, a in calls]
    results = [[] for _ in calls]
    errors = []
    start = threading.Barrier(len(calls))

    def run(i):
        try:
            f, a = calls[i]
            start.wait()
            for _ in range(12):
                results[i].append(flat(f(*a)))
        except Exception as e:      # surfaced by the assertion below
            errors.append(e)

    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(calls))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i, rs in enumerate(results):
        assert len(rs) == 12
        for r in rs:
            assert all(same(a, b) for a, b in zip(r, alone[i])), f'call {i} ({calls[i][0].__name__}) differs'
