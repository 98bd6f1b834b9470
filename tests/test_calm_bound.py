"""The bound behind the calm route of the unsharp stage (DESIGN.md §5.1), checked on the CPU.

The calm route skips the blur and the median wherever the second differences of the emitted bytes say that
unsharp_mask cannot fire (kernels_unsharp.cu, k_calm_scan / k_calm_blocks / k_calm_chunks). These tests derive the
constants of that argument from the CPU restatement of the blur (oracle.port), feed the restatement of unsharp_mask
adversarial and ordinary frames and require every pixel it changes to lie in a block the model (tests/calm_model.py)
flags, and measure how tight the bound is."""
import re

import numpy as np
import pytest

from oracle import port
from poppy_b200 import synth
from tests import calm_model as cm

# Smallest neighbourhood max hx + max hy at which unsharp_mask changes an output byte, over the patterns of
# _tight_patterns(): a valley whose floor is the first column, q = (4, 50, 186, 255, ...) along x and constant along y.
# The blur reflects the image at the border (BORDER_REFLECT_101) while the median replicates it, so column 0 fills six
# of the nine median taps. (With the floor at 0 the median fires at the same value, but the sharpened value clamps back
# to byte 0.) Away from the border the least value found is INTERIOR_TIGHT, a valley with a two-pixel floor
# (4, 4) and walls rising by about 2 h + 1 per column. Paraboloid bowls clipped to the byte range change bytes only
# from about 84.
TIGHT = 46
INTERIOR_TIGHT = 50
FLOOR = 4


def _x(img: np.ndarray) -> np.ndarray:
    """Grey 8-bit content as lapBlend of an identical pair: u8 * float32(1/255) in all three channels."""
    x = img.astype(np.float32) * np.float32(1.0 / 255.0)
    if x.ndim == 2:
        x = np.repeat(x[..., None], 3, -1)
    return np.ascontiguousarray(x)


def _fire_nbhd(x: np.ndarray):
    """(neighbourhood values of the pixels whose output byte unsharp_mask changes, analysis)."""
    an = cm.analyse(x)
    f = (cm.emit(port.unsharp(x, 1.0, np.float32(cm.NORM_T)))[0] != an.q).any(-1)
    return an.pixel_nbhd()[f], an


def gauss_taps() -> np.ndarray:
    """The 9 taps of GaussianBlur(sigma 1) as the impulse response of the restatement (a one-row image: no column pass)."""
    imp = np.zeros((1, 17, 1), np.float32)
    imp[0, 8, 0] = 1.0
    return port.gaussian9(imp)[0, 4:13, 0]


def test_blur_taps_and_second_moment():
    g = gauss_taps().astype(np.float64)
    assert np.array_equal(g, g[::-1]) and (g > 0).all()
    # the kernel's taps (gk() in kernels_unsharp.cu) are the ones the restatement uses
    bits = [int(b, 16) for b in re.findall(r"0x([0-9a-f]{8})u", re.search(r"gk\(int j\)(.*?)\n}", cm._UNSHARP, re.S).group(1))]
    assert np.array_equal(np.array(bits, np.uint32).view(np.float32).astype(np.float64), g[4:])
    # |(I - B) x| <= sum_{a>0} a^2 g_a max|d2 x|: the constant of DESIGN.md §5.1 (0.4999640, so 0.49997 bounds it and
    # the 0.49996 the bound once used did not)
    s = sum(a * a * g[4 + a] for a in range(1, 5))
    assert 0.49996 < s <= 0.49997, s
    assert abs(g.sum() - 1.0) < 1e-6


def test_static_assert_inequality_holds_for_the_source_constant():
    src = cm._UNSHARP
    m = re.search(r"static_assert\(\(2 \* CALM_SUM \+ 2 \* ([0-9.]+)\) / 255\.0 \* ([0-9.]+) < ([0-9.]+), \"calm bound\"\);", src)
    assert m, "the calm-bound static_assert is gone"
    slack, moment, limit = (float(v) for v in m.groups())
    g = gauss_taps().astype(np.float64)
    assert moment >= sum(a * a * g[4 + a] for a in range(1, 5))
    # |q[-1] + q[+1] - 2 q| <= 2 h + 1 and |255 x - q| <= 0.5 per pixel: 2 h + 3, plus fp32 rounding
    assert slack >= 3.0
    assert (2 * cm.CALM_SUM + 2 * slack) / 255.0 * moment < limit
    assert 3 * limit ** 2 < cm.NORM_T ** 2 and limit < np.float32(cm.NORM_T) / np.sqrt(3.0)
    assert cm.CALM_SUM < TIGHT


def _tight_patterns(width=24, rows=16):
    """Grey profiles along x (constant along y): valleys against the left border, (f, f + a, f + b, 255, ...), and
    interior valleys with a one- and a two-pixel floor. Yields (kind, image)."""
    for a in range(20, 120):
        for b in range(a, 256 - FLOOR, 2):
            p = np.full(width, 255.0)
            p[:3] = 0, a, b
            p[:3] += FLOOR
            yield "border", np.tile(p, (rows, 1))
            p = np.full(width, 255.0)
            p[8:10] = 0
            p[7], p[10], p[6], p[11] = a, a, b, b
            p[6:12] += FLOOR
            yield "interior", np.tile(p, (rows, 1))
            p = np.full(width, 255.0)
            p[8] = 0
            p[7], p[9], p[6], p[10] = a, a, b, b
            p[6:11] += FLOOR
            yield "interior", np.tile(p, (rows, 1))


def _profile_nbhd(img) -> int:
    dx, dy = cm.second_dev(img.astype(np.uint8)[..., None])
    return int(max(dx.max(), 0) + dy.max())


def test_tightness_of_the_bound():
    """The least neighbourhood hx + hy at which unsharp_mask fires, over valley profiles (in all four orientations, so
    each image border is tried). Candidates are tried in order of their second-difference maximum, and the search stops
    after the first level at which something fires."""
    best = {}
    cands = sorted(((_profile_nbhd(img), kind, img) for kind, img in _tight_patterns()), key=lambda t: t[0])
    for v, kind, img in cands:
        if kind in best and v > best[kind]:
            if len(best) == 2:
                break
            continue
        for im in (img, img[:, ::-1], img.T, img.T[::-1]):
            nb, _ = _fire_nbhd(_x(np.ascontiguousarray(im)))
            if nb.size:
                best[kind] = min(best.get(kind, 999), int(nb.min()))
    assert best == {"border": TIGHT, "interior": INTERIOR_TIGHT}, best
    assert cm.CALM_SUM < min(best.values())


def tight_valley(n_rows: int, h: int) -> np.ndarray:
    """The border valley of TIGHT scaled to neighbourhood value h: columns f + (0, h, 4 h - 2, 6 h - 6), 255, ...,
    clipped to 255 (h = TIGHT: (4, 50, 186, 255, ...)). Its neighbourhood value is h for h in 38 .. 63."""
    p = np.full(24, 255.0)
    p[:4] = np.minimum(np.array((0, h, 4 * h - 2, 6 * h - 6)) + FLOOR, 255)
    return np.tile(p, (n_rows, 1))


def test_tight_valley_fires_at_tight_and_not_below():
    nb, an = _fire_nbhd(_x(tight_valley(16, TIGHT)))
    assert nb.size and nb.min() == TIGHT
    for h in range(TIGHT - 6, TIGHT):
        nb, an = _fire_nbhd(_x(tight_valley(16, h)))
        assert nb.size == 0 and an.nbhd.max() == h


def _adversarial():
    rng = np.random.Generator(np.random.PCG64(7))
    yy, xx = np.mgrid[0:40, 0:48]
    for k in np.arange(1.0, 40.0, 1.5):                       # paraboloid bowls and domes, clipped to the byte range
        for c in ((20.0, 16.0), (20.5, 16.5), (0.0, 0.0), (47.0, 39.0)):
            bowl = k * ((xx - c[0]) ** 2 + (yy - c[1]) ** 2)
            yield _x(np.clip(np.rint(bowl), 0, 255))
            yield _x(np.clip(np.rint(255 - bowl), 0, 255))
    for s in range(4, 90, 3):                                  # steep ramps into each border
        for img in (np.clip(255 - s * xx, 0, 255), np.clip(s * (47 - xx), 0, 255), np.clip(255 - s * yy, 0, 255),
                    np.clip(s * (39 - yy), 0, 255)):
            yield _x(img)
    for h in range(30, 60):                                    # the tight valleys, rotated
        v = tight_valley(40, h)[:, :40]
        for im in (v, v[:, ::-1], v.T, v.T[::-1]):
            yield _x(np.ascontiguousarray(im))
    for sigma in (0.7, 1.0, 1.5, 2.5, 4.0):                    # random smooth fields, also overshooting [0, 1] slightly
        f = synth.smooth_field(64, 48, int(rng.integers(1 << 30)), sigma=sigma)
        yield np.ascontiguousarray(f)
        yield np.ascontiguousarray((f * np.float32(1.002) - np.float32(0.001)).astype(np.float32))
        yield np.ascontiguousarray((f * np.float32(1.3) - np.float32(0.15)).astype(np.float32))


def test_bound_is_sound_on_adversarial_frames():
    n_fired = 0
    for x in _adversarial():
        an = cm.analyse(x)
        f = cm.fired(x, port.unsharp(x, 1.0, np.float32(cm.NORM_T)))
        assert not (f & ~an.pixel_block_flags()).any(), np.argwhere(f & ~an.pixel_block_flags())[:4]
        n_fired += int(f.sum())
    assert n_fired > 1000


@pytest.mark.parametrize("kind", ["noise", "shapes", "blocks"])
def test_bound_is_sound_on_lap_blend_frames(native_lib, kind):
    """lapBlend of the synthetic inputs (the restatement's stages): every byte unsharp_mask changes lies in a flagged
    strip chunk, every pixel it moves in a flagged block. The restatement triangulates with the product's host stage,
    so the native library is built (no GPU needed)."""
    w, h, levels = 124, 75, 5
    inp = {"noise": lambda: synth.make_inputs(w, h, 24, 8.0, seed=61), "shapes": lambda: synth.shape_inputs(w, h, 24, seed=62),
           "blocks": lambda: synth.block_inputs(w, h, 24, seed=63)}[kind]()
    flagged = []
    for s in (0.0, 0.3, 0.5, 1.0):
        st = port.stages(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, s, s, levels)
        x = st.lap_blend
        an = cm.analyse(x)
        amount = np.float32(1.0 - np.sin(s * np.pi))
        f = cm.fired(x, port.unsharp(x, amount, np.float32(cm.NORM_T)))
        assert not (f & ~an.pixel_block_flags()).any()
        changed = (st.dst != an.q).any(-1)
        assert not (changed & ~an.pixel_chunk_flags()).any()
        flagged.append(an.block_flags.mean())
    assert max(flagged) > 0 and (kind != "noise" or min(flagged) < 1)


def test_model_flags_and_force_all():
    """Hand-checked cases of the model: the neighbourhood reaches 2 block columns and 1 block row, the chunk and tile
    margins follow k_calm_chunks, and widths the byte scan cannot take flag everything."""
    assert cm.force_all(333, 64) and cm.force_all(4, 64) and cm.force_all(64, 1) and not cm.force_all(8, 2)
    x = np.full((64, 256, 3), 0.5, np.float32)
    x[20, 130] = 0.9                                           # one bright pixel: block (2, 32)
    an = cm.analyse(x)
    ys, xs = np.nonzero(an.block_flags)
    assert (ys.min(), ys.max(), xs.min(), xs.max()) == (1, 3, 30, 34)
    # blocks 30..34 = columns 120..139 (strip 1 only), block rows 1..3 = rows 8..31 (chunk rows 0 and 1)
    assert an.chunk_flags.tolist() == [[False, True, False], [False, True, False], [False, False, False]]
    # strip 1 stages columns 112..247 (tiles 0 and 1); chunk row 1 stages rows 19..52 (tile rows 0 and 1)
    assert an.tile_flags.tolist() == [[True, True], [True, True]]
    x[20, 130] = 1.01                                          # clamp excess beyond the tolerance: the block says nothing
    an = cm.analyse(x)
    assert an.excess[2, 32].all() and an.hx[2, 32] == 255
