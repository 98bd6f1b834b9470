"""cv::fastNlMeansDenoising (8-bit BGR, NORM_L2), the --denoise step of the reference's run() (src/poppy.cpp:172, 269-311):
integer arithmetic after a host-built weight table, so BIT-EXACT. The numpy restatement (oracle/denoise.py) is pinned to the
committed fixture and to cv2 where it imports; poppy_cuda_denoise is compared with all three byte for byte."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from oracle import denoise as nlm

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "conditioning", "denoise.npz")
ERR_NO_DEVICE, ERR_INVALID = -1, -2


def _golden():
    g = np.load(GOLDEN)
    for i in range(int(g["n"])):
        h, tw, sw = g[f"params{i}"]
        yield g[f"src{i}"], float(h), int(tw), int(sw), g[f"dst{i}"]


def _noisy(rows, cols, seed, amp=20):
    """A smooth base with noise of +-amp: content on which denoising moves most pixels."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:rows, 0:cols]
    base = np.stack([96 + 60 * np.sin(xx / 9.0 + c) * np.cos(yy / 13.0 - c) for c in range(3)], -1)
    return np.clip(base + rng.integers(-amp, amp + 1, base.shape), 0, 255).astype(np.uint8)


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


def _gpu_visible():
    try:
        import torch
        return torch.cuda.is_available()
    except ImportError:
        return False


# ---- the restatement (no GPU) -------------------------------------------------------------------------------------------

def test_restatement_matches_golden():
    for i, (src, h, tw, sw, want) in enumerate(_golden()):
        assert (nlm.denoise(src, h, tw, sw) == want).all(), i


def test_golden_cases_change_most_pixels():
    """The fixture is content on which the call does something (a low h on strong noise would leave it unchanged)."""
    moved = [float((want != src).mean()) for src, h, _, _, want in _golden() if h > 0 and src.size > 3]
    assert min(moved) > 0.5, moved


def test_restatement_matches_cv2_on_random_cases():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(77)
    for k in range(12):
        rows, cols = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        h = float(rng.choice([0.0, 2.5, 5.0, 10.0, 17.5, 30.0, -8.0]))
        tw, sw = int(rng.integers(1, 12)), int(rng.integers(1, 30))
        src = _noisy(rows, cols, 100 + k, amp=int(rng.integers(8, 26)))
        assert (nlm.denoise(src, h, tw, sw) == cv2.fastNlMeansDenoising(src, None, h, tw, sw)).all(), (rows, cols, h, tw, sw)


@pytest.mark.parametrize("h,tw,sw", [(3.0, 7, 21), (10.0, 7, 21), (25.0, 7, 21), (10.0, 5, 15), (12.0, 3, 35), (7.5, 8, 20),
                                     (60.0, 15, 45)])
def test_weight_table_prefix_matches_formula(h, tw, sw):
    """lut[a] = cvRound(mult * exp(-a m / den)) is 0 once it falls below 0.001 * mult, i.e. once
    mult * exp(-a m / den) < ceil(0.001 mult) - 1/2: the first zero is floor(den / m * ln(mult / (ceil(0.001 mult) - 1/2))) + 1,
    about 3 ln(1000) h^2 / m = 20.7 h^2 / m entries."""
    lut, shift = nlm.weight_table(h, tw, sw)
    th, sh = nlm.windows(tw, sw)
    tw, sw = 2 * th + 1, 2 * sh + 1
    mult = (2 ** 31 - 1) // (sw * sw * 255)
    m = (1 << shift) / (tw * tw)
    den = float(np.float32(np.float32(h) * np.float32(h)) * np.float32(3))
    n = nlm.nonzero_prefix(lut)
    assert n == math.floor(den / m * math.log(mult / (math.ceil(0.001 * mult) - 0.5))) + 1
    assert abs(n - 3 * math.log(1000) * h * h / m) < 0.02 * n      # the rounding of a small mult moves it by ~1 %
    assert lut[0] == mult and (np.diff(lut[:n + 1]) <= 0).all() and lut[n] == 0
    if (h, tw, sw) == (10.0, 7, 21):
        assert (shift, mult, len(lut), n) == (6, 19096, 149355, 1582)


def test_denoise_without_gpu_returns_no_device(native_lib):
    if _gpu_visible() or native_lib.poppy_cuda_device_count() > 0:
        pytest.skip("a GPU is visible")
    src = np.zeros((8, 9, 3), np.uint8)
    dst = np.empty_like(src)
    rc = native_lib.poppy_cuda_denoise(0, src.ctypes.data_as(C.c_void_p), 27, 9, 8, 3.0, 7, 21, dst.ctypes.data_as(C.c_void_p), 27)
    assert rc == ERR_NO_DEVICE
    assert b"no such CUDA device" in native_lib.poppy_cuda_blur_margin_last_error()


# ---- the GPU ------------------------------------------------------------------------------------------------------------

def _check(src, h=3.0, tw=7, sw=21, oracle=True):
    """api.denoise against the restatement and cv2 (where it imports); returns the GPU output."""
    from poppy_b200 import api
    got = api.denoise(src, h, tw, sw)
    assert got.shape == src.shape and got.dtype == np.uint8
    if oracle:
        want = nlm.denoise(src, h, tw, sw)
        assert int((got != want).sum()) == 0, "differs from the restatement"
    cv2 = _cv2()
    if cv2 is not None:
        assert int((got != cv2.fastNlMeansDenoising(np.ascontiguousarray(src), None, h, tw, sw)).sum()) == 0, "differs from cv2"
    return got


@pytest.mark.gpu
def test_cuda_denoise_matches_golden(native_lib):
    from poppy_b200 import api
    for i, (src, h, tw, sw, want) in enumerate(_golden()):
        assert int((api.denoise(src, h, tw, sw) != want).sum()) == 0, i
        _check(src, h, tw, sw)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1), (5, 3), (13, 9), (3, 200), (200, 3), (1, 57)])
def test_cuda_denoise_images_smaller_than_the_border(native_lib, shape):
    _check(_noisy(*shape, seed=shape[0] * 1000 + shape[1]), 10.0)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(63, 31), (64, 32), (65, 33), (127, 95), (128, 96), (129, 97), (63, 97), (129, 31)])
def test_cuda_denoise_tile_edges(native_lib, shape):
    """The kernel's tile is 32 columns x 64 rows: sizes one below, at and one above its multiples."""
    _check(_noisy(*shape, seed=shape[0] + 7 * shape[1]), 10.0)


@pytest.mark.gpu
@pytest.mark.parametrize("h,tw,sw", [(0.0, 7, 21), (-10.0, 7, 21), (10.0, 8, 20), (25.0, 6, 14), (10.0, 5, 15),
                                     (25.0, 3, 35), (10.0, 1, 21), (10.0, 7, 1), (12.0, 15, 45), (12.0, 15, 63), (1e30, 7, 21)])
def test_cuda_denoise_parameters(native_lib, h, tw, sw):
    """h = 0 (only the pixel itself weighs), negative h (h^2 counts), even sizes, the smallest and largest windows, h
    whose square overflows float (every weight equal)."""
    _check(_noisy(41, 70, seed=int(abs(h)) % 1000 + tw + sw), h, tw, sw)


@pytest.mark.gpu
def test_cuda_denoise_weight_table_in_l1(native_lib):
    """h = 80: the table's non-zero prefix (~100 k entries) does not fit in shared memory and is read through L1."""
    lut, _ = nlm.weight_table(80.0)
    assert nlm.nonzero_prefix(lut) * 4 > 228 * 1024
    _check(_noisy(70, 45, seed=80, amp=25), 80.0)


@pytest.mark.gpu
def test_cuda_denoise_flat_image(native_lib):
    src = np.full((50, 70, 3), (17, 200, 93), np.uint8)
    assert (_check(src, 10.0) == src).all()


@pytest.mark.gpu
def test_cuda_denoise_saturated_pixels(native_lib):
    src = _noisy(90, 80, seed=3, amp=25)
    src[:30, :40] = 0
    src[60:, 40:] = 255
    src[45, :, 1] = 255
    _check(src, 25.0)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(360, 640), (1080, 1920)])
def test_cuda_denoise_large(native_lib, shape):
    _check(_noisy(*shape, seed=shape[1]), 10.0)


@pytest.mark.gpu
def test_cuda_denoise_4k_against_cv2(native_lib):
    pytest.importorskip("cv2")
    _check(_noisy(2160, 3840, seed=4), 10.0, oracle=False)


@pytest.mark.gpu
def test_cuda_denoise_strided_rows_and_in_place(native_lib):
    from poppy_b200 import api
    src = _noisy(45, 61, seed=11)
    want = nlm.denoise(src, 10.0)
    wide = np.zeros((45, 70, 3), np.uint8)
    wide[:, 5:66] = src
    roi = wide[:, 5:66]
    assert roi.strides[0] == 70 * 3
    assert (api.denoise(roi, 10.0) == want).all()
    # dst == src through the C ABI, on a strided ROI
    rc = native_lib.poppy_cuda_denoise(0, roi.ctypes.data_as(C.c_void_p), roi.strides[0], 61, 45, 10.0, 7, 21,
                                       roi.ctypes.data_as(C.c_void_p), roi.strides[0])
    assert rc == 0
    assert (wide[:, 5:66] == want).all()
    assert (wide[:, :5] == 0).all() and (wide[:, 66:] == 0).all()


@pytest.mark.gpu
def test_cuda_denoise_is_deterministic(native_lib):
    from poppy_b200 import api
    src = _noisy(300, 410, seed=9)
    a, b = api.denoise(src, 10.0), api.denoise(src, 10.0)
    assert (a == b).all() and (a != src).mean() > 0.5


@pytest.mark.gpu
def test_cuda_denoise_rejects_invalid_arguments(native_lib):
    src = _noisy(20, 30, seed=5)
    dst = np.empty_like(src)
    sp, dp = src.ctypes.data_as(C.c_void_p), dst.ctypes.data_as(C.c_void_p)

    def call(s=sp, s_step=90, cols=30, rows=20, h=3.0, tw=7, sw=21, d=dp, d_step=90):
        return native_lib.poppy_cuda_denoise(0, s, s_step, cols, rows, h, tw, sw, d, d_step)

    bad = [dict(s=None), dict(d=None), dict(cols=0), dict(rows=0), dict(cols=-3), dict(s_step=89), dict(d_step=60),
           dict(tw=0), dict(sw=0), dict(tw=-7), dict(h=float("nan")), dict(h=float("inf")), dict(h=float("-inf")),
           dict(tw=16), dict(tw=17), dict(sw=64), dict(sw=65)]
    for kw in bad:
        assert call(**kw) == ERR_INVALID, kw
        assert native_lib.poppy_cuda_blur_margin_last_error().startswith(b"denoise:"), kw
    assert call(tw=15, sw=63) == 0                   # the largest supported windows (16 and 64 round up past them)
    assert call() == 0
    assert (dst == nlm.denoise(src)).all()
    from poppy_b200 import api
    with pytest.raises(ValueError):
        api.denoise(src.astype(np.float32))
    with pytest.raises(RuntimeError, match="denoise"):
        api.denoise(src, template_window_size=17)
