"""The CUDA stages against cv2 (tests/cv2_ref.py) at every row-tail residue, each stage fed the GPU's own inputs for it, so
a failure names the stage whose kernel is wrong rather than the first frame byte it moved.

Sweep: every width 1..260 at height 37, every height 1..100 at widths 61 and 130, and 1279 x 719, 2049 x 33 and 3840 x 216
(a 4K row of one 216-row band of the unsharp strip kernel), each at three pyramid depths: the deepest that reaches 1 x 1,
one level and 64 levels. For each size and depth, frame FRAME of a BATCH-frame sequence, rendered alone with its stages
kept:
  * TRI_MAP equals cv2.fillConvexPoly of the GPU's morphed points, truncated, in painter's order;
  * WARPED1 / WARPED2 equal cv2.remap of the sources through the restatement's maps (oracle/port.morph_frame), and MASK
    the restatement's mask (its gray is not cv2's, tests/cv2_ref.py);
  * LAP_BLEND equals the cv2 composition of the Laplacian blend of the two warps and the GPU's MASK, bit for bit;
  * the frame equals unsharp + convertTo composed from cv2 on the GPU's LAP_BLEND where w % 8 is 0, 1, 3 or 6, and the
    restatement's unsharp elsewhere (cv2 4.13's Gaussian may differ from 4.6.0's at those tails, tests/cv2_ref.py);
  * the same frame rendered in the whole BATCH-frame batch without stage dumps, on the calm and on the dense unsharp
    route, is byte-identical: this carries the sweep through the batched pyramid, the TMA collapse and the calm route.
Conditioning: gabor_filter and blur_margin against their cv2 compositions, and the mask basis derived on the GPU
(gabor2=None) at every width 1..40: its MASK equals the restatement's mask of cv2's gabor filter of corrected2."""
import math

import numpy as np
import pytest

from oracle import port
from poppy_b200 import host
from tests import cv2_ref
from tests.test_margin import CASES as MARGIN_CASES, _gabor_close
from tests.util import any_size_inputs, bits_differ, flat_tri

pytestmark = pytest.mark.gpu

BATCH = 32
FRAME = 11


def deepest_levels(w, h):
    """Pyramid levels until the top level is 1 x 1 (at least one)."""
    levels = 0
    while w > 1 or h > 1:
        w, h, levels = (w + 1) // 2, (h + 1) // 2, levels + 1
    return max(levels, 1)


SIZES = [(w, 37) for w in range(1, 261)] + [(61, h) for h in range(1, 101)] + [(130, h) for h in range(1, 101)]
SIZES += [(1279, 719), (2049, 33), (3840, 216)]
SWEEP = [(w, h, L) for w, h in SIZES for L in sorted({deepest_levels(w, h), 1, 64})]


def _stages(w, h, levels, bgr1, bgr2, gab, p1, p2, s, m, tri):
    from poppy_b200 import renderer as R
    with R.MorphRenderer(w, h, levels, len(p1), max(len(tri), 1), 1, keep_stages=True) as r:
        r.set_pair(bgr1, bgr2, gab)
        r.set_points(p1, p2)
        r.render([s], [m], *flat_tri([tri]))
        frame = r.download(0, 1)[0]
        return frame, {k: r.read_stage(getattr(R, "STAGE_" + k), 0) for k in
                       ("MORPHED_POINTS", "TRI_MAP", "WARPED1", "WARPED2", "MASK", "LAP_BLEND")}


def _batch(w, h, levels, bgr1, bgr2, gab, p1, p2, shapes, masks, plan, mode):
    from poppy_b200.renderer import MorphRenderer
    with MorphRenderer(w, h, levels, len(p1), max(plan.max_triangles, 1), BATCH, chunk_frames=BATCH) as r:
        r.set_unsharp_mode(mode)
        r.set_pair(bgr1, bgr2, gab)
        r.set_points(p1, p2)
        r.render(shapes, masks, plan.tri_idx, plan.tri_offsets)
        return r.download(FRAME, 1)[0]


@pytest.mark.parametrize("w,h,levels", SWEEP, ids=[f"{w}x{h}_L{L}" for w, h, L in SWEEP])
def test_stages_against_cv2(native_lib, w, h, levels):
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h)
    shapes = np.linspace(0.0, 1.0, BATCH, dtype=np.float32)
    masks = np.random.Generator(np.random.PCG64(w * 1000 + h)).permutation(np.linspace(0.0, 1.0, BATCH))
    s, m = shapes[FRAME], float(masks[FRAME])
    plan = host.SequencePlan(p1, p2, w, h, shapes)
    try:
        tri = plan.triangles(FRAME)
        frame, st = _stages(w, h, levels, bgr1, bgr2, gab, p1, p2, s, m, tri)
        batched = {mode: _batch(w, h, levels, bgr1, bgr2, gab, p1, p2, shapes, masks, plan, mode) for mode in (2, 1)}
    finally:
        plan.close()
    bad = []
    xy = np.trunc(st["MORPHED_POINTS"][tri]).astype(np.int32).reshape(-1, 6)
    if bits_differ(st["TRI_MAP"], cv2_ref.paint_triangles(w, h, xy)):
        bad.append("TRI_MAP")
    maps = port.morph_frame(bgr1, bgr2, gab, p1, p2, tri, float(s), m, levels)
    if bits_differ(st["WARPED1"], cv2_ref.remap_u8c3(bgr1, maps.mapx1, maps.mapy1)):
        bad.append("WARPED1")
    if bits_differ(st["WARPED2"], cv2_ref.remap_u8c3(bgr2, maps.mapx2, maps.mapy2)):
        bad.append("WARPED2")
    if bits_differ(st["MASK"], maps.mask):
        bad.append("MASK")
    lap = cv2_ref.lap_blend(cv2_ref.u8_to_f32(st["WARPED1"]), cv2_ref.u8_to_f32(st["WARPED2"]), st["MASK"], levels)
    if bits_differ(st["LAP_BLEND"], lap):
        bad.append("LAP_BLEND")
    amount = float(np.float32(1.0 - math.sin(m * math.pi)))
    sharp = cv2_ref.unsharp(st["LAP_BLEND"], amount) if w % 8 in (0, 1, 3, 6) else port.unsharp(st["LAP_BLEND"], amount, 0.3)
    if bits_differ(frame, cv2_ref.to_u8(sharp)):
        bad.append("unsharp + convertTo")
    for mode, name in ((2, "calm"), (1, "dense")):
        if bits_differ(batched[mode], frame):
            bad.append(f"{BATCH}-frame batch, {name} route")
    assert not bad, bad


# Where the unsharp blur's scalar tail starts only moves the blur by about one ulp, which the 8-bit frame almost never
# shows: on random content about one byte in several million tail elements. These inputs were found by rendering
# any_size_inputs(w, h, seed) with the restatement twice, once with the tail starting 8 elements early and once 8
# elements late, and keeping the first frame where the 8-bit result changed. They are 5-column frames because each row
# then has 8 elements before the tail and 7 in it: (w, h, seed, shape, mask ratio, levels, which shift the frame shows).
TAIL_CASES = [(5, 20000, 20, 0.3, 0.0, 4, "8 early"), (5, 20000, 15, 0.6, 1.0, 4, "8 late")]


@pytest.mark.parametrize("w,h,seed,s,m,levels,shift", TAIL_CASES, ids=[c[-1].replace(" ", "_") for c in TAIL_CASES])
def test_unsharp_tail_start_shows_in_the_frame(native_lib, w, h, seed, s, m, levels, shift):
    """The frame equals the restatement's unsharp of the GPU's LAP_BLEND on inputs where a shifted tail start changes a byte.
    LAP_BLEND must also equal the restatement's: the case only keeps its sensitivity with the blend it was found on."""
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=seed)
    want = port.stages(bgr1, bgr2, gab, p1, p2, s, m, levels)
    frame, st = _stages(w, h, levels, bgr1, bgr2, gab, p1, p2, np.float32(s), m, want.tri_idx)
    assert bits_differ(st["LAP_BLEND"], want.lap_blend) == 0
    amount = float(np.float32(1.0 - math.sin(m * math.pi)))
    assert bits_differ(frame, cv2_ref.to_u8(port.unsharp(st["LAP_BLEND"], amount, 0.3))) == 0, shift


GABOR_SIZES = [(h, w) for h in range(1, 8) for w in range(1, 8)] + \
              [(h, w) for h in (3, 4, 5) for w in (31, 32, 33)] + [(1080, 1920), (2160, 3840)]


# max |GPU - cv2| measured on a B200: 0 everywhere but 4K, where it is 2^-29, one float ulp of a value in [1/64, 1/32):
# cv2's DFT evaluation and the direct double sum round a value on a rounding boundary apart (tests/test_margin.py).
# A larger difference fails even where _gabor_close would allow it.
GABOR_MAX_DIFF = {(2160, 3840): 2.0 ** -29}


@pytest.mark.parametrize("h,w", GABOR_SIZES, ids=[f"{w}x{h}" for h, w in GABOR_SIZES])
def test_gabor_filter_against_cv2(native_lib, h, w):
    from poppy_b200 import api, synth
    src = (synth.noise_image(w, h, 5).astype(np.float32) / np.float32(255)) if h >= 300 else \
        np.random.default_rng(w * 100 + h).random((h, w, 3), dtype=np.float32)
    ok, (max_diff, differ) = _gabor_close(api.gabor_filter(src), cv2_ref.gabor_filter(src))
    assert ok and max_diff <= GABOR_MAX_DIFF.get((h, w), 0.0), (max_diff, differ)


# (rows, cols, union_h, union_w): the margin cases of tests/test_margin.py, 1-pixel margins (no padding on an axis), 1080p
BLUR_MARGIN_CASES = MARGIN_CASES + [(1, 1, 1, 1), (2, 3, 2, 3), (1, 40, 1, 40), (40, 1, 40, 1), (7, 9, 7, 9), (30, 40, 30, 45),
                                    (30, 40, 33, 40), (1080, 1920, 1080, 1920), (1080, 1920, 1200, 2100)]


@pytest.mark.parametrize("case", BLUR_MARGIN_CASES)
def test_blur_margin_against_cv2(native_lib, case):
    from poppy_b200 import api
    h, w, uh, uw = case
    img = np.random.default_rng(h + 7 * w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    got = api.blur_margin(img, (uw, uh))
    want = cv2_ref.blur_margin(img, (uw, uh))
    assert got.shape == want.shape and (got == want).all()


@pytest.mark.parametrize("w", range(1, 41))
def test_derived_mask_against_cv2_gabor(native_lib, w):
    """gabor2=None: the basis is filtered on the GPU from corrected2. cv2 pins the filter, the restatement the gray and the
    addWeighted, on both sides of the gray's w & ~7 body."""
    from poppy_b200.renderer import STAGE_MASK, MorphRenderer
    h, mask_ratio = 9, 0.37
    rng = np.random.default_rng(w)
    c1, c2 = (rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(2))
    with MorphRenderer(w, h, 3, 8, 8, 1, keep_stages=True) as r:
        r.set_pair(c1, c2, None)
        r.set_points(np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32))
        r.render([0.4], [mask_ratio], np.zeros((0, 3), np.int32), [0, 0])
        got = r.read_stage(STAGE_MASK, 0)
    want = port.mask(cv2_ref.gabor_filter(cv2_ref.u8_to_f32(c2)), mask_ratio)
    assert bits_differ(got, want) == 0
