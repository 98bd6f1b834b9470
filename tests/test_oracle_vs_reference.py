"""Pins the CPU restatement (oracle/poppy_oracle.cpp) against the real reference: the library built from the
unmodified reference sources + vendored OpenCV 4.6.0 (oracle/_ref). Bit-exact at every stage boundary.
Skipped where the reference library is not present (it travels to the GPU box; tests/test_golden.py pins the
restatement from committed fixtures everywhere)."""
import numpy as np
import pytest

from oracle import port, ref
from poppy_b200 import synth
from tests.util import bits_differ, random_triangles, remap_map_families

needs_ref = pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libpoppy_ref.so not built")

CASES = [
    (160, 120, 80, 0.37, 6, "noise"), (203, 157, 60, 0.5, 64, "noise"), (257, 131, 100, 0.9, 4, "noise"),
    (100, 75, 20, 0.0, 6, "noise"), (100, 75, 20, 1.0, 6, "noise"), (333, 222, 50, 0.123, 3, "noise"),
    (120, 100, 30, 0.3, 64, "shapes"), (90, 70, 24, 0.1, 3, "blocks"), (33, 17, 5, 0.6, 8, "noise"),
]


def _inputs(kind, w, h, n):
    if kind == "shapes":
        return synth.shape_inputs(w, h, n, seed=5)
    if kind == "blocks":
        return synth.block_inputs(w, h, n, seed=6)
    return synth.make_inputs(w, h, n, 8.0, seed=7)


@needs_ref
@pytest.mark.parametrize("w,h,n,s,levels,kind", CASES)
def test_every_stage_bit_exact(w, h, n, s, levels, kind):
    inp = _inputs(kind, w, h, n)
    a = ref.stages(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, s, s, levels)
    b = port.morph_frame(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, a.tri_idx, s, s, levels)
    for k in a.__dataclass_fields__:
        assert bits_differ(getattr(a, k), getattr(b, k)) == 0, k


@needs_ref
def test_stage_decomposition_equals_morph_images():
    inp = synth.make_inputs(150, 110, 50, 8.0, seed=9)
    dst, mp = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, 0.4, 0.6, 5)
    st = ref.stages(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, 0.4, 0.6, 5)
    assert (dst == st.dst).all() and bits_differ(mp, st.morphed_points) == 0


@needs_ref
def test_fill_convex_poly_random_and_degenerate():
    w, h = 97, 71
    tris = random_triangles(w, h, 4000)
    # one triangle at a time (coverage of each) and all together (later index wins)
    for i in range(0, 4000, 7):
        assert (ref.fill_triangles(w, h, tris[i:i + 1]) == port.fill_triangles(w, h, tris[i:i + 1])).all(), tris[i]
    assert (ref.fill_triangles(w, h, tris) == port.fill_triangles(w, h, tris)).all()


@needs_ref
@pytest.mark.parametrize("size", [(135, 240), (68, 120), (34, 60), (17, 30), (9, 15), (5, 8), (3, 4), (2, 2), (1, 1),
                                  (1, 5), (7, 1), (2, 3), (21, 13), (64, 33)])
@pytest.mark.parametrize("cn", [1, 3])
def test_pyramid_primitives(size, cn):
    h, w = size
    rng = np.random.default_rng(w * 1000 + h + cn)
    img = rng.random((h, w, cn), dtype=np.float32) if cn == 3 else rng.random((h, w), dtype=np.float32)
    d_ref, d_port = ref.pyr_down(img), port.pyr_down(img)
    assert bits_differ(d_ref, d_port) == 0
    assert bits_differ(ref.pyr_up(d_ref, (w, h)), port.pyr_up(d_ref, (w, h))) == 0


@needs_ref
@pytest.mark.parametrize("size", [(40, 57), (9, 9), (4, 30), (30, 3), (1, 12), (12, 1), (2, 2), (1, 1)])
def test_gaussian_median_unsharp_primitives(size):
    h, w = size
    rng = np.random.default_rng(w * 77 + h)
    img = rng.random((h, w, 3), dtype=np.float32)
    assert bits_differ(ref.gaussian_blur(img, 1.0), port.gaussian9(img)) == 0
    assert bits_differ(ref.median3(img), port.median3(img)) == 0
    blocks = (rng.integers(0, 2, (h, w, 3)) * 1.0).astype(np.float32)      # drives the threshold branch
    for amount in (1.0, 0.31, 0.0):
        a, b = ref.unsharp(blocks, 1.0, amount, 0.3), port.unsharp(blocks, amount, 0.3)
        assert bits_differ(a, b) == 0
    if h * w >= 100:
        assert (ref.unsharp(blocks, 1.0, 1.0, 0.3) != blocks).any(), "threshold branch not exercised"


@needs_ref
def test_remap_borders_ties_and_saturation():
    rng = np.random.default_rng(8)
    h, w = 57, 83
    src = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    for name, (mx, my) in remap_map_families(w, h).items():
        assert (ref.remap_u8c3(src, mx, my) == port.remap_u8c3(src, mx, my)).all(), name


@needs_ref
@pytest.mark.parametrize("w", [8, 9, 15, 17, 100, 203, 257])
def test_mask_tail_columns(w):
    g = synth.smooth_field(w, 40, seed=w)
    for mr in (0.0, 0.37, 0.5, 1.0):
        assert bits_differ(ref.mask(g, mr), port.mask(g, mr)) == 0


@needs_ref
def test_lap_blend_levels_beyond_one_pixel():
    rng = np.random.default_rng(2)
    l, r = rng.random((37, 53, 3), dtype=np.float32), rng.random((37, 53, 3), dtype=np.float32)
    m = rng.random((37, 53), dtype=np.float32)
    for levels in (1, 2, 6, 7, 20, 64):
        assert bits_differ(ref.lap_blend(l, r, m, levels), port.lap_blend(l, r, m, levels)) == 0
