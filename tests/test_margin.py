"""SURVEY.md 8(f-3), the input conditioning ahead of the path.
blur_margin (reference src/util.cpp:574-602): integer arithmetic, BIT-EXACT - the numpy restatement (oracle/margin.py) is
pinned against the reference library and the committed fixture; poppy_cuda_blur_margin is compared with both.
gabor_filter (src/util.cpp:40-60): floating point with a TOLERANCE - the reference evaluates the 16 correlations by a
double-precision DFT, the restatement and the CUDA kernel sum them directly in double; the float results may differ by one
ulp where the exact value sits on a rounding boundary, and where the exact response is 0 (black margins) the DFT leaves
round-off of ~1e-15 that the direct sum does not have. Tolerance: |diff| <= GABOR_ATOL everywhere; on textured images at
most GABOR_PPM values per million differ by more than GABOR_NOISE (flat synthetic regions share one value and flip
together, so the count is only asserted on texture)."""
import os

import numpy as np
import pytest

from oracle import margin, ref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "conditioning", "blur_margin.npz")
# (rows, cols, union_h, union_w): both axes padded, one axis, none (1-pixel margins), tall/wide, margins wider than the padding
CASES = [(100, 150, 120, 180), (100, 150, 100, 150), (200, 100, 200, 160), (90, 90, 150, 90), (333, 211, 400, 300),
         (64, 48, 70, 300), (500, 500, 512, 512)]


GABOR_ATOL = 1.2e-7          # one float ulp below 1.0 is 6e-8; the mean of 16 clamped planes moves by at most ulp / 16 * k
GABOR_PPM = 20
GABOR_NOISE = 1e-12          # DFT round-off of the reference around exact zeros is ~1e-15


def _gabor_close(a, b, textured=True):
    d = np.abs(a - b)
    differ = int((d > GABOR_NOISE).sum())
    few = differ <= max(2, GABOR_PPM * a.size // 1_000_000) if textured else True
    return float(d.max()) <= GABOR_ATOL and few, (float(d.max()), differ)


def _img(rng, h, w):
    return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


def test_fixed_point_kernel_of_blur_margin():
    k = margin.gaussian_kernel_fixed(127, 6.0)
    assert sum(k) == 256 and k[63] == 18 and k == k[::-1]
    assert [i for i, v in enumerate(k) if v][0] == 46 and k[46:50] == [1, 0, 1, 1]       # error diffusion leaves a gap


@pytest.mark.skipif(not ref.available(), reason="reference library not built")
def test_kernel_matches_reference_impulse_response():
    # a 1-row image shrinks the vertical kernel to [1]; 255 * tap / 256 rounds back to the tap for taps < 128
    img = np.zeros((1, 301, 3), np.uint8)
    img[0, 150] = 255
    out = ref.gaussian_blur_u8(img, 127, 6.0)
    assert out[0, 150 - 63:150 + 64, 1].astype(int).tolist() == margin.gaussian_kernel_fixed(127, 6.0)


@pytest.mark.skipif(not ref.available(), reason="reference library not built")
@pytest.mark.parametrize("shape", [(40, 70), (1, 50), (50, 1), (3, 3), (130, 20), (20, 200), (2, 2), (127, 127), (300, 190)])
def test_oracle_gaussian_blur_u8_matches_reference(shape):
    img = _img(np.random.default_rng(shape[0] * 1000 + shape[1]), *shape)
    assert (ref.gaussian_blur_u8(img, 127, 6.0) == margin.gaussian_blur_u8(img, 127, 6.0)).all()


@pytest.mark.skipif(not ref.available(), reason="reference library not built")
@pytest.mark.parametrize("case", CASES)
def test_oracle_blur_margin_matches_reference(case):
    h, w, uh, uw = case
    img = _img(np.random.default_rng(h + 7 * w), h, w)
    assert (ref.blur_margin(img, (uw, uh)) == margin.blur_margin(img, (uw, uh))).all()


def test_oracle_blur_margin_matches_golden():
    g = np.load(GOLDEN)
    for i in range(int(g["n"])):
        got = margin.blur_margin(g[f"src{i}"], tuple(g[f"union{i}"]))
        assert (got == g[f"dst{i}"]).all(), i


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES + [(1080, 1920, 1200, 2100)])
def test_cuda_blur_margin_matches_oracle_and_reference(native_lib, case):
    from poppy_b200 import api
    h, w, uh, uw = case
    img = _img(np.random.default_rng(h + 7 * w), h, w)
    got = api.blur_margin(img, (uw, uh))
    want = ref.blur_margin(img, (uw, uh)) if ref.available() else margin.blur_margin(img, (uw, uh))
    assert got.shape == want.shape and (got == want).all()
    # strided input rows (a cv::Mat ROI of a wider image)
    wide = np.zeros((h, w + 9, 3), np.uint8)
    wide[:, :w] = img
    assert (api.blur_margin(wide[:, :w], (uw, uh)) == want).all()


@pytest.mark.gpu
def test_cuda_blur_margin_matches_golden_and_rejects_bad_geometry(native_lib):
    from poppy_b200 import api
    g = np.load(GOLDEN)
    for i in range(int(g["n"])):
        assert (api.blur_margin(g[f"src{i}"], tuple(g[f"union{i}"])) == g[f"dst{i}"]).all(), i
    with pytest.raises(RuntimeError):          # the source is larger than the union: cv::Mat ROI assertion in the reference
        api.blur_margin(np.zeros((50, 80, 3), np.uint8), (60, 50))


@pytest.mark.skipif(not ref.available(), reason="reference library not built")
def test_gabor_kernels_are_bit_equal_to_getGaborKernel():
    thetas = margin.gabor_thetas()
    assert thetas[:3] == [0.0, 11.0, 22.0] and len(thetas) == 16           # float step = 180 / 16 in integers
    for th in thetas:
        a = ref.gabor_kernel(13, 5.0, th, 10.0, 0.04, np.pi / 4)
        b = margin.gabor_kernel(13, 5.0, th, 10.0, 0.04, np.pi / 4)
        assert (a.view(np.uint32) == b.view(np.uint32)).all(), th


@pytest.mark.skipif(not ref.available(), reason="reference library not built")
@pytest.mark.parametrize("shape", [(60, 80), (7, 9), (1, 40), (300, 260)])
def test_oracle_gabor_filter_matches_reference_within_tolerance(shape):
    src = np.random.default_rng(shape[1]).random((*shape, 3), dtype=np.float32)
    ok, detail = _gabor_close(ref.gabor_filter(src), margin.gabor_filter(src))
    assert ok, detail


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(60, 80), (7, 9), (1, 40), (300, 260), (512, 512), (1080, 1920)])
def test_cuda_gabor_filter_matches_reference_within_tolerance(native_lib, shape):
    from poppy_b200 import api, synth
    h, w = shape
    src = (synth.noise_image(w, h, 5).astype(np.float32) / np.float32(255)) if h >= 300 else \
        np.random.default_rng(w).random((h, w, 3), dtype=np.float32)
    got = api.gabor_filter(src)
    want = ref.gabor_filter(src) if ref.available() else margin.gabor_filter(src)
    ok, detail = _gabor_close(got, want)
    assert ok, detail


@pytest.mark.gpu
def test_frames_from_cuda_conditioning_equal_the_reference_chain(native_lib):
    """blur_margin -> gabor_filter -> morph_images entirely on the GPU against the same three calls of the reference (or
    of the restatements pinned to it where the reference library is not built)."""
    from poppy_b200 import api, synth
    from tests.util import reference
    cond = ref if ref.available() else margin
    inp = synth.block_inputs(200, 160, 40, seed=9)
    small = inp.bgr2[10:150, 20:180].copy()
    c2_gpu, c2_ref = api.blur_margin(small, (200, 160)), cond.blur_margin(small, (200, 160))
    assert (c2_gpu == c2_ref).all()
    g_gpu = api.gabor_filter(c2_gpu.astype(np.float32) / np.float32(255))
    g_ref = cond.gabor_filter(c2_ref.astype(np.float32) / np.float32(255))
    assert _gabor_close(g_gpu, g_ref, textured=False)[0]          # flat blocks and black margins
    api.Settings.instance().pyramid_levels = 5
    dst, _ = api.morph_images(inp.bgr1, c2_gpu, inp.bgr1, c2_gpu, g_gpu, inp.pts1, inp.pts2, 0.4, 0.4)
    want, _ = reference().morph_images(inp.bgr1, c2_ref, g_ref, inp.pts1, inp.pts2, 0.4, 0.4, 5)
    api.release()
    assert (dst == want).all()
