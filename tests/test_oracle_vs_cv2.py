"""Pins the CPU restatement (oracle/poppy_oracle.cpp, oracle/margin.py) to cv2 (tests/cv2_ref.py) at every row-tail residue.

The restatement selects its association per element position the way the OpenCV loops it restates do (pyrDown's
width0, h1_end, (dw * cn) & ~3; the Gaussian's (w * cn) % 8 tail), and the CUDA kernels copy those selections. The
committed fixtures fix them at about a dozen frame sizes; cv2 is independent code, so sweeping it over every width and
height residue checks the positions the fixtures miss. Bit-exact everywhere except the two known differences between
OpenCV 4.6.0 and cv2 4.13 that tests/cv2_ref.py names; the tests below fail if cv2 differs anywhere else."""
import numpy as np
import pytest

from oracle import margin, port
from tests import cv2_ref
from tests.test_margin import CASES as MARGIN_CASES, _gabor_close
from tests.util import bits_differ, random_triangles, remap_map_families

cv2 = cv2_ref.cv2


def _rand(h, w, cn, seed):
    rng = np.random.default_rng(seed)
    return rng.random((h, w, cn) if cn == 3 else (h, w), dtype=np.float32)


PYR_SIZES = sorted({(h, w) for h in (1, 2, 3, 5, 16) for w in range(1, 261)} |
                   {(h, w) for w in (1, 7, 130) for h in range(1, 71)})


@pytest.mark.parametrize("cn", [1, 3])
def test_pyramid_primitives_at_every_residue(cn):
    bad = []
    for h, w in PYR_SIZES:
        img = _rand(h, w, cn, w * 1000 + h * 10 + cn)
        down = cv2_ref.pyr_down(img)
        if bits_differ(down, port.pyr_down(img)):
            bad.append(("pyrDown", w, h))
        if bits_differ(cv2_ref.pyr_up(down, (w, h)), port.pyr_up(down, (w, h))):
            bad.append(("pyrUp", w, h))
    assert not bad, bad[:20]


@pytest.mark.parametrize("cn", [1, 3])
def test_pyramid_primitives_with_odd_dstsize(cn):
    """pyrDown to the other admissible size of an odd axis ((n - 1) / 2), pyrUp to an odd size (2n - 1 and 2n + 1).
    Not from one column to three: OpenCV's one-column branch of pyrUp leaves the third column of its row buffer unwritten,
    and cv2 returns whatever that buffer held. The path never asks for it (lap_blend's pyrUp targets at most 2n)."""
    bad = []
    for h, w in [(1, 1), (3, 5), (7, 1), (5, 9), (9, 17), (16, 31), (33, 129), (17, 257), (2, 131)]:
        img = _rand(h, w, cn, w * 77 + h + cn)
        for dsize in {(w // 2 or 1, h // 2 or 1), ((w + 1) // 2, h // 2 or 1), (w // 2 or 1, (h + 1) // 2)}:
            if bits_differ(cv2_ref.pyr_down(img, dsize), port.pyr_down(img, dsize)):
                bad.append(("pyrDown", w, h, dsize))
        for dsize in {(2 * w - 1, 2 * h - 1), (2 * w + 1, 2 * h + 1), (2 * w - 1, 2 * h + 1), (2 * w + 1, 2 * h)}:
            if w == 1 and dsize[0] == 3:
                continue
            if bits_differ(cv2_ref.pyr_up(img, dsize), port.pyr_up(img, dsize)):
                bad.append(("pyrUp", w, h, dsize))
    assert not bad, bad


# sizes whose pyramids reach 1 x 1 within a few levels and then repeat it
LAP_SIZES = [(1, 1), (1, 5), (7, 1), (2, 3), (3, 2), (5, 9), (37, 53), (31, 200), (17, 129), (64, 33), (9, 130)]


@pytest.mark.parametrize("h,w", LAP_SIZES)
def test_lap_blend_through_one_pixel_levels(h, w):
    rng = np.random.default_rng(w * 31 + h)
    l, r = rng.random((h, w, 3), dtype=np.float32), rng.random((h, w, 3), dtype=np.float32)
    m = rng.random((h, w), dtype=np.float32)
    for levels in (*range(1, 9), 20, 64):
        assert bits_differ(cv2_ref.lap_blend(l, r, m, levels), port.lap_blend(l, r, m, levels)) == 0, levels


def test_tail_positions():
    assert cv2_ref.tail_positions(8, 3).tolist() == []                  # 24 elements: no tail
    assert cv2_ref.tail_positions(2, 3).tolist() == [0, 1, 2, 3]        # 6: all tail
    assert cv2_ref.tail_positions(7, 3).tolist() == [16, 17, 18, 19]    # 21: 5-element tail
    assert cv2_ref.tail_positions(3, 3).tolist() == []                  # 9: 1-element tail
    assert cv2_ref.tail_positions(12, 1).tolist() == [8, 9, 10, 11]
    assert cv2_ref.tail_positions(1, 3).tolist() == []                  # one column: the kernel shrinks to [1]


@pytest.mark.parametrize("cn", [1, 3])
def test_gaussian9_bit_exact_outside_the_known_tail(cn):
    """Bit-exact outside tail_positions. Differences inside them are 4.13's extra vector step; any difference outside
    them fails, so a cv2 whose Gaussian changes more does not pass unnoticed."""
    outside = []
    for h in (1, 2, 3, 5, 16):
        for w in (*range(1, 70), 127, 128, 129, 130, 255, 256, 257, 301):
            img = _rand(h, w, cn, w * 1000 + h * 10 + cn)
            a = cv2_ref.gaussian9(img).reshape(h, w * cn)
            b = port.gaussian9(img).reshape(h, w * cn)
            cols = np.nonzero((a.view(np.uint32) != b.view(np.uint32)).any(0))[0]
            tail = cv2_ref.tail_positions(w, cn)
            extra = np.setdiff1d(cols, tail)
            if extra.size:
                outside.append((w, h, extra.tolist()))
    assert not outside, outside[:10]


# w % 8 in {0, 1, 3, 6}: (3 w) % 8 < 4, no element of the blur where 4.13 may differ
UNSHARP_WIDTHS = [w for w in range(1, 70) if w % 8 in (0, 1, 3, 6)] + [128, 129, 131, 134, 256, 257, 259, 262]


@pytest.mark.parametrize("h", [1, 2, 3, 9, 20])
def test_unsharp_at_widths_clear_of_the_tail(h):
    bad = []
    for w in UNSHARP_WIDTHS:
        assert cv2_ref.tail_positions(w, 3).size == 0
        rng = np.random.default_rng(w * 100 + h)
        blocks = (rng.integers(0, 2, (h, w, 3)) * 1.0).astype(np.float32)       # drives the threshold branch
        smooth = rng.random((h, w, 3), dtype=np.float32) * np.float32(0.2)
        for img in (blocks, smooth):
            for amount in (1.0, 0.31, 0.0):
                if bits_differ(cv2_ref.unsharp(img, amount), port.unsharp(img, amount, 0.3)):
                    bad.append((w, amount))
        if h * w >= 100:
            assert (cv2_ref.unsharp(blocks, 1.0) != blocks).any(), ("threshold branch not exercised", w)
    assert not bad, bad


@pytest.mark.parametrize("cn", [1, 3])
def test_median3(cn):
    bad = []
    for h in (1, 2, 3, 5, 16):
        for w in (*range(1, 40), 127, 128, 129, 257):
            img = _rand(h, w, cn, w * 13 + h + cn)
            img[..., ::3] = np.float32(0.5)           # ties
            if bits_differ(cv2_ref.median3(img), port.median3(img)):
                bad.append((w, h))
    assert not bad, bad


@pytest.mark.parametrize("h,w", [(57, 83), (1, 1), (3, 130), (40, 7)])
def test_remap_borders_ties_and_saturation(h, w):
    src = np.random.default_rng(8 + w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    for name, (mx, my) in remap_map_families(w, h).items():
        assert (cv2_ref.remap_u8c3(src, mx, my) == port.remap_u8c3(src, mx, my)).all(), name


def test_fill_triangles_random_and_degenerate():
    w, h = 97, 71
    tris = random_triangles(w, h, 4000)
    # one triangle at a time (coverage of each) and all together (later index wins)
    for i in range(4000):
        assert (cv2_ref.paint_triangles(w, h, tris[i:i + 1]) == port.fill_triangles(w, h, tris[i:i + 1])).all(), tris[i]
    assert (cv2_ref.paint_triangles(w, h, tris) == port.fill_triangles(w, h, tris)).all()


@pytest.mark.parametrize("shape", [(40, 70), (1, 50), (50, 1), (3, 3), (130, 20), (20, 200), (2, 2), (127, 127), (300, 190)])
def test_margin_gaussian_blur_u8(shape):
    img = np.random.default_rng(shape[0] * 1000 + shape[1]).integers(0, 256, (*shape, 3), dtype=np.uint8)
    assert (cv2.GaussianBlur(img, (127, 127), 6.0) == margin.gaussian_blur_u8(img, 127, 6.0)).all()


@pytest.mark.parametrize("case", MARGIN_CASES)
def test_margin_blur_margin(case):
    h, w, uh, uw = case
    img = np.random.default_rng(h + 7 * w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    assert (cv2_ref.blur_margin(img, (uw, uh)) == margin.blur_margin(img, (uw, uh))).all()


def test_gabor_kernels_are_bit_equal_to_getGaborKernel():
    for th in margin.gabor_thetas():
        a = cv2.getGaborKernel((13, 13), 5.0, th, 10.0, 0.04, np.pi / 4, ktype=cv2.CV_32F)
        b = margin.gabor_kernel(13, 5.0, th, 10.0, 0.04, np.pi / 4)
        assert (a.view(np.uint32) == b.view(np.uint32)).all(), th


GABOR_SIZES = [(h, w) for h in range(1, 8) for w in range(1, 8)] + \
              [(h, w) for h in (3, 4, 5) for w in (31, 32, 33)] + [(60, 80), (300, 260)]


def test_margin_gabor_filter_small_and_block_edge_sizes():
    worst = []
    for h, w in GABOR_SIZES:
        src = np.random.default_rng(w * 100 + h).random((h, w, 3), dtype=np.float32)
        ok, detail = _gabor_close(cv2_ref.gabor_filter(src), margin.gabor_filter(src))
        assert ok, ((h, w), detail)
        worst.append(detail[0])
    assert max(worst) == 0.0, max(worst)      # both evaluate the correlations in double; none has differed yet


def _fma32(a, b, c):
    """float32 fma(a, b, c) for float32 a, c and a float32 scalar b: a * b is exact in double, so rounding the double sum
    to float rounds the exact value the same way unless the sum landed on a float midpoint, which the helper rejects."""
    s = a.astype(np.float64) * np.float64(b) + c.astype(np.float64)
    r = s.astype(np.float32)
    nb = np.nextafter(r, np.where(s > r, np.float32(np.inf), np.float32(-np.inf))).astype(np.float64)
    assert not ((r.astype(np.float64) + nb) / 2 == s).any()
    return r


def test_cv2_gray_is_the_scalar_association_on_every_column():
    """Why the blend mask is not pinned to cv2: cv2 4.13's BGR2GRAY of 32F data is fma(r, .299, fma(b, .114, g * .587))
    on every column, which the reference's 4.6.0 evaluates only on its scalar tail (x >= w & ~7); the restatement's body
    columns stay pinned by the committed fixtures alone."""
    rng = np.random.default_rng(5)
    img = rng.random((23, 61, 3), dtype=np.float32)
    b, g, r = img[..., 0], img[..., 1], img[..., 2]
    scalar = _fma32(r, np.float32(0.299), _fma32(b, np.float32(0.114), g * np.float32(0.587)))
    assert bits_differ(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), scalar) == 0
    body = _fma32(r, np.float32(0.299), _fma32(g, np.float32(0.587), b * np.float32(0.114)))
    assert bits_differ(body, scalar) > 0           # the two associations are distinguishable on this input
