"""The calm route of the unsharp stage (DESIGN.md §5.1) at its bound, its lane, word, block, strip, chunk and tile
edges, and on lane scratch that still holds earlier content.

Most frames come from an identical pair (pts1 == pts2 == the four corners, bgr1 == bgr2), so lapBlend is the image over
255 and the content can be placed pixel by pixel. Each such frame holds one feature on a calm base: a kink that the
byte scan sees only through one neighbour (at every residue mod 8, on lane, CTA, strip, chunk and tile edges and on the
border), the border valleys of tests/test_calm_bound.py at and just below the least neighbourhood value at which
unsharp_mask changes a byte, border ramps, or valleys next to collapse-tile edges over stale lane scratch. The tests
derive from keep_stages renders what the content exercised and assert it, compare the calm route (mode 2), the dense
route (mode 1) and the adaptive router (mode 0) with each other and with the reference, and check the calm route's
flagged-chunk counts against the model (tests/calm_model.py) and against the geometry of the block neighbourhood."""
import numpy as np
import pytest

from poppy_b200 import host, synth
from poppy_b200.renderer import STAGE_LAP_BLEND, STAGE_WARPED1, MorphRenderer
from tests import calm_model as cm
from tests.test_calm_bound import TIGHT, tight_valley
from tests.util import bits_differ, frame_checksum, reference

pytestmark = pytest.mark.gpu

LEVELS = 5


def corners(w, h):
    return np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float32)


def kink_profile(n, x0, d, side, base=60):
    """A grey profile of length n whose only second difference with a floor-average deviation above 15 sits at x0 and
    equals d: flat `base` on one side of x0, and on the other (`side`, "left" or "right") a ramp whose increments start
    at 2 d (d at an image border, which the scan reflects) and fall by 30 per pixel. The scan sees the kink only through
    the neighbour of x0 on the ramp side: on a lane, word or CTA edge that neighbour comes from another lane or load."""
    q = np.full(n, float(base))
    step = d if (x0 == 0 and side == "right") or (x0 == n - 1 and side == "left") else 2 * d
    k, v = x0, float(base)
    while step > 0:
        k += 1 if side == "right" else -1
        if not 0 <= k < n:
            break
        v += step
        q[k] = v
        step -= 30
    if side == "right":
        q[k + 1:] = v
    else:
        q[:max(k, 0)] = v
    return q


def kink_positions(n, edges):
    """(x0, side) pairs at the given positions whose kink profile is the sole deviation above CALM_SUM."""
    out = []
    for x0 in sorted({e for e in edges if 0 <= e < n}):
        for side in ("left", "right"):
            q = kink_profile(n, x0, cm.CALM_SUM + 1, side)
            dev, _ = cm.second_dev(np.tile(q.astype(np.uint8)[None, :, None], (2, 1, 1)))
            if np.flatnonzero(dev[0, :, 0] > cm.CALM_SUM).tolist() == [x0] and dev[0, :, 0].max() == cm.CALM_SUM + 1:
                out.append((x0, side))
    return out


def kink_frames(w, h):
    """Frames of kinks across x (constant along y) at residues 0..7 mod 8, lane / word edges (4k), CTA edges of the scan
    (128k) and strip edges (120k), and the border columns; and across y at rows 8k (blocks), 16k / 64k (scan threads and
    CTAs), 24k (chunks), 32k (tiles) and the border rows. Each at d = CALM_SUM + 1 (flags its neighbourhood) and
    d = CALM_SUM (flags nothing; every third kink). Yields (axis, position, d, image)."""
    xe = list(range(9)) + [119, 120, 123, 124, 127, 128, 131, 132, 239, 240, 243, 244] + [w - k for k in range(1, 5)]
    ye = list(range(9)) + [15, 16, 23, 24, 31, 32, 47, 48, 63, 64] + [h - k for k in range(1, 4)]
    for axis, n, edges in ((1, w, xe), (0, h, ye)):
        for i, (x0, side) in enumerate(kink_positions(n, edges)):
            for d in (cm.CALM_SUM + 1, cm.CALM_SUM) if i % 3 == 0 else (cm.CALM_SUM + 1,):
                q = np.clip(kink_profile(n, x0, d, side), 0, 255).astype(np.uint8)
                g = np.broadcast_to(q[None, :] if axis == 1 else q[:, None], (h, w))
                yield axis, x0, d, np.ascontiguousarray(np.repeat(g[..., None], 3, -1))


def reach(pos, n, block, unit, radius):
    """Strips (unit = 120 columns) or chunk rows (unit = 24 rows) holding a block within `radius` blocks of pos."""
    nb = cm.div_up(n, block)
    b = pos // block
    return {min(c, n - 1) // unit for k in range(max(b - radius, 0), min(b + radius, nb - 1) + 1)
            for c in (k * block, k * block + block - 1)}


def render_frames(w, h, pair, pts, shapes, masks, mode, keep=False, chunk=None, per_call=True, r=None):
    """Render the frames one per call (or all in one call); returns (frames, per-call unsharp_stats, lapBlend planes)."""
    bgr1, bgr2, gab = pair
    pts1, pts2 = pts
    shapes = np.asarray(shapes, np.float32)
    masks = np.asarray(masks, np.float64)
    plan = host.SequencePlan(pts1, pts2, w, h, shapes)
    own = r is None
    if own:
        r = MorphRenderer(w, h, LEVELS, len(pts1), max(plan.max_triangles, 1), len(shapes), keep_stages=keep,
                          chunk_frames=chunk)
    try:
        r.set_unsharp_mode(mode)
        r.set_pair(bgr1, bgr2, gab)
        r.set_points(pts1, pts2)
        r.unsharp_stats()
        stats, laps = [], []
        calls = [(i, i + 1) for i in range(len(shapes))] if per_call else [(0, len(shapes))]
        for a, b in calls:
            off = plan.tri_offsets[a:b + 1]
            r.render(shapes[a:b], masks[a:b], plan.tri_idx[off[0]:off[-1]], off - off[0], first_slot=a)
            stats.append(r.unsharp_stats())
            if keep:
                laps.append(r.read_stage(STAGE_LAP_BLEND, b - 1))
                if a == 0 and bgr1 is bgr2 and len(pts1) == 4:
                    assert bits_differ(r.read_stage(STAGE_WARPED1, b - 1), bgr1) == 0     # the identity warp
        return r.download(0, len(shapes)), stats, laps
    finally:
        if own:
            r.close()


def check_frames(w, h, imgs, gab):
    """Identical-pair frames (one image each, corner points, mask ratio 0) rendered one per call by the dense route
    (keep_stages) and the calm route: equal to each other and to the reference, and the calm route's flagged-chunk
    count of every frame equal to the model's. Returns (analyses, dense frames)."""
    cpts = corners(w, h)
    plan = host.SequencePlan(cpts, cpts, w, h, np.zeros(1, np.float32))
    ref = reference()
    ans, out = [], []
    with MorphRenderer(w, h, LEVELS, 4, plan.max_triangles, 1, keep_stages=True) as rd, \
            MorphRenderer(w, h, LEVELS, 4, plan.max_triangles, 1) as rc:
        rc.set_unsharp_mode(2)
        rd.set_points(cpts, cpts)
        rc.set_points(cpts, cpts)
        for img in imgs:
            frames = []
            for r in (rd, rc):
                r.set_pair(img, img, gab)
                r.unsharp_stats()
                r.render(np.zeros(1, np.float32), np.zeros(1), plan.tri_idx, plan.tri_offsets)
                frames.append(r.download(0, 1)[0])
            exact, total = rc.unsharp_stats()
            assert bits_differ(rd.read_stage(STAGE_WARPED1, 0), img) == 0        # the identity warp
            an = cm.analyse(rd.read_stage(STAGE_LAP_BLEND, 0))
            assert bits_differ(frames[1], frames[0]) == 0
            assert (exact, total) == (an.flagged_chunks, an.chunk_flags.size)
            want, _ = ref.morph_images(img, img, gab, cpts, cpts, 0.0, 0.0, LEVELS)
            assert bits_differ(frames[0], want) == 0
            ans.append(an)
            out.append(frames[0])
    return ans, out


def check_routes(w, h, pair, pts, shapes, masks, ref_frames=None):
    """Mode 2 (one frame per call) against the dense route and the reference; the flagged-chunk count of every call
    against the model. Returns the analyses of the frames."""
    dense, _, laps = render_frames(w, h, pair, pts, shapes, masks, 1, keep=True)
    calm, stats, _ = render_frames(w, h, pair, pts, shapes, masks, 2)
    assert bits_differ(calm, dense) == 0
    ans = [cm.analyse(x) for x in laps]
    for k, (an, (exact, total)) in enumerate(zip(ans, stats)):
        assert total == an.chunk_flags.size and exact == an.flagged_chunks, (k, exact, an.flagged_chunks)
    ref = reference()
    for k in range(len(shapes)) if ref_frames is None else ref_frames:
        want, _ = ref.morph_images(pair[0], pair[1], pair[2], pts[0], pts[1], float(shapes[k]), float(masks[k]), LEVELS)
        assert bits_differ(dense[k], want) == 0, k
    return ans, dense, laps


WIDTHS = (8, 12, 124, 128, 132, 244, 248)
HEIGHTS = (2, 3, 7, 8, 9, 23, 25, 65)


@pytest.mark.parametrize("w", WIDTHS)
def test_kinks_at_lane_word_block_strip_and_border_edges(native_lib, w):
    """Each frame holds one kink (kink_frames) on a calm base. At d = CALM_SUM + 1 the calm route must flag exactly the
    strip chunks whose blocks lie within 2 block columns / 1 block row of it, read the same count as the model, and skip
    the rest; at d = CALM_SUM it must flag nothing. Either way the frame equals the dense route and the reference."""
    residues = {0: set(), 1: set()}
    partial = 0
    for h in HEIGHTS:
        gab = synth.smooth_field(w, h, seed=h)
        frames = list(kink_frames(w, h))
        imgs = [f[3] for f in frames]
        ans, dense = check_frames(w, h, imgs, gab)
        strips, chunks_y = cm.div_up(w, cm.STRIP_W), cm.div_up(h, cm.CHUNK_ROWS)
        for (axis, pos, d, _), an in zip(frames, ans):
            assert not an.forced
            dx, dy = cm.second_dev(an.q)
            dev = (dx if axis == 1 else dy).max(axis=(1 - axis, 2))         # per column (axis 1) / row (axis 0)
            if d > cm.CALM_SUM:
                # the rendered content carries its kink and nothing else above the bound: the sole flag source
                assert np.flatnonzero(dev > cm.CALM_SUM).tolist() == [pos] and (dx if axis == 0 else dy).max() == 0
                residues[axis].add(pos % 8)
                if axis == 1:
                    want = len(reach(pos, w, cm.BLOCK_W, cm.STRIP_W, 2)) * chunks_y
                else:
                    want = len(reach(pos, h, cm.BLOCK_H, cm.CHUNK_ROWS, 1)) * strips
                assert an.flagged_chunks == want, (axis, pos, an.flagged_chunks, want)
                partial += 0 < want < an.chunk_flags.size
            else:
                assert an.flagged_chunks == 0 and an.nbhd.max() == cm.CALM_SUM
    assert residues[1] == set(range(8)) and residues[0] == set(range(8)), residues
    assert partial > 0


def test_tight_valleys_fire_at_the_tightness_value_only(native_lib):
    """The border valleys at (left, bottom) and just below (right, top) the tightness value on a 248 x 65
    frame: the exact path moves pixels of the first two only."""
    w, h = 248, 65
    gab = synth.smooth_field(w, h, seed=6)
    cols = np.full((h, w), 255.0)
    cols[:, :24] = tight_valley(1, TIGHT)[0]
    cols[:, w - 24:] = tight_valley(1, TIGHT - 1)[0, ::-1]
    rows = np.full((h, w), 255.0)
    rows[:24] = tight_valley(1, TIGHT - 1)[0][:, None]
    rows[h - 24:] = tight_valley(1, TIGHT)[0][::-1, None]
    for g, fires, calm in ((cols, np.s_[:, :4], np.s_[:, w - 4:]), (rows, np.s_[h - 4:], np.s_[:4])):
        img = np.ascontiguousarray(np.repeat(g.astype(np.uint8)[..., None], 3, -1))
        ans, dense, _ = check_routes(w, h, (img, img, gab), (corners(w, h), corners(w, h)), [0.0], [0.0])
        an, changed = ans[0], (dense[0] != ans[0].q).any(-1)
        assert changed[fires].any() and not changed[calm].any()
        assert an.pixel_nbhd()[fires].max() == TIGHT and an.pixel_nbhd()[calm].max() == TIGHT - 1
        assert an.pixel_chunk_flags()[fires].all()


def test_border_ramps(native_lib):
    """Ramps of slope 62 into each border, q = 50, 112, 174, 236, 255, ...: the blur reflects them into a kink of second
    difference 124 (neighbourhood value 62) that interior second differences do not show, and the median fires there."""
    w, h = 132, 65
    gab = synth.smooth_field(w, h, seed=7)
    for axis in (0, 1):
        n = (h, w)[axis]
        q = np.minimum(50 + 62 * np.arange(n), 255).astype(np.uint8)
        for flip in (False, True):
            prof = q[::-1] if flip else q
            g = np.broadcast_to(prof[:, None] if axis == 0 else prof[None, :], (h, w))
            img = np.ascontiguousarray(np.repeat(g[..., None], 3, -1))
            ans, dense, _ = check_routes(w, h, (img, img, gab), (corners(w, h), corners(w, h)), [0.0], [0.0])
            an, changed = ans[0], (dense[0] != ans[0].q).any(-1)
            edge = np.s_[-1:] if flip else np.s_[:1]
            border = changed[edge] if axis == 0 else changed[:, edge]
            assert border.all() and an.nbhd.max() == 62, (axis, flip)


def _excess_classes(x):
    """(blocks that leave [0, 1] by at most EMIT_EXCESS_TOL in 255ths, blocks that leave it by more)."""
    _, ex = cm.emit(x)
    blk = np.stack([cm._block_max(ex[..., c]) for c in range(3)], -1).max(-1)
    return int(((blk > 0) & (blk <= cm.EMIT_EXCESS_TOL)).sum()), int((blk > cm.EMIT_EXCESS_TOL).sum())


def test_clamp_excess_classes(native_lib):
    """Two different pictures through a mask transition: lapBlend leaves [0, 1] by less than the tolerance in some
    blocks and by more in others; the calm route equals the dense route and the reference on every frame."""
    w, h = 640, 360
    inp = synth.block_inputs(w, h, 40, seed=71)
    masks = [0.2, 0.45, 0.6, 0.85]
    _, _, laps = check_routes(w, h, (inp.bgr1, inp.bgr2, inp.gabor2), (inp.pts1, inp.pts2), masks, masks)
    small, big = np.sum([_excess_classes(x) for x in laps], 0)
    assert small > 0 and big > 0, (small, big)


VALLEY = np.array([255, 255, 210, 85, 4, 4, 85, 210, 255, 255], np.float64)     # |x - blur| = 0.145 on the floor


def stale_content(w, h):
    """Sparse content on a white base, and the mask of the pixels the busy content before it keeps white.

    A calm valley (VALLEY: neighbourhood value CALM_SUM, median of |x - blur| just under the threshold) with its
    two-pixel floor next to a collapse-tile edge, and a line a little further away that flags the strip chunks on the
    valley's side only. The tile on the other side of the edge is then read only through a margin of k_calm_chunks:
    if it is not recomputed it still holds the busy content, which is white there, pushes the floor's median over the
    threshold and turns its byte 4 into 0.
    640 x 360, the row margins: rows 91..95 of tile row 2 are read only by chunk row 4 (Y0 = 96, through Y0 - 5), rows
    192..196 of tile row 6 only by chunk row 7 (Y1 = 192, through Y1 + 5).
    3840 x 2160, the column margins: in the top half, columns 1912..1919 of tile 14 are read only by strip 16
    (x0 = 1920, through x0 - 8); in the bottom half, columns 1920..1927 of tile 15 only by strip 15 (x0 = 1800,
    through x0 + 128)."""
    g = np.full((h, w), 255.0)
    white = np.zeros((h, w), bool)
    if w <= 1920:
        g[92:102] = VALLEY[:, None]               # floor rows 96, 97
        g[110] = 60                               # block rows 12..14 = chunk row 4
        g[186:196] = VALLEY[:, None]              # floor rows 190, 191
        g[180] = 60                               # block rows 21..23 = chunk row 7
        white[84:100] = white[188:204] = True
    else:
        top, bot = slice(0, h // 2), slice(h // 2, h)
        g[top, 1916:1926] = VALLEY                # floor columns 1920, 1921
        g[top, 1960] = 60                         # strip 16 only
        g[bot, 1914:1924] = VALLEY                # floor columns 1918, 1919
        g[bot, 1840] = 60                         # strip 15 only
        white[:, 1872:1968] = True
    img = np.ascontiguousarray(np.repeat(g.astype(np.uint8)[..., None], 3, -1))
    return img, white


def stale_then_sparse(w, h, chunk, frames):
    """Busy content through every lane, then the sparse content on the same renderer in mode 2. Returns the frames'
    checksums, the reference frame and the analysis of the sparse frame."""
    busy = synth.block_inputs(w, h, 30, seed=81)
    img, white = stale_content(w, h)
    busy.bgr1[white] = 255
    busy.bgr2[white] = 255
    gab = synth.smooth_field(w, h, seed=82)
    cpts = corners(w, h)
    shapes = np.linspace(0, 1, frames, dtype=np.float32)
    masks = np.zeros(frames)
    plan_busy = host.SequencePlan(busy.pts1, busy.pts2, w, h, shapes)
    plan = host.SequencePlan(cpts, cpts, w, h, shapes)
    with MorphRenderer(w, h, LEVELS, len(busy.pts1), max(plan_busy.max_triangles, plan.max_triangles), frames,
                       chunk_frames=chunk) as r:
        r.set_unsharp_mode(1)
        r.set_pair(busy.bgr1, busy.bgr2, busy.gabor2)
        r.set_points(busy.pts1, busy.pts2)
        r.render(shapes, shapes.astype(np.float64), plan_busy.tri_idx, plan_busy.tri_offsets)
        r.sync()
        r.set_unsharp_mode(2)
        r.set_pair(img, img, gab)
        r.set_points(cpts, cpts)
        r.unsharp_stats()
        r.render(shapes, masks, plan.tri_idx, plan.tri_offsets)
        exact, total = r.unsharp_stats()
        sums = [r.checksum(i, 1) for i in range(frames)]
    want, _ = reference().morph_images(img, img, gab, cpts, cpts, 0.0, 0.0, LEVELS)
    with MorphRenderer(w, h, LEVELS, 4, plan.max_triangles, 1, keep_stages=True) as r:
        r.set_pair(img, img, gab)
        r.set_points(cpts, cpts)
        r.render(shapes[:1], masks[:1], plan.tri_idx[:plan.tri_offsets[1]], plan.tri_offsets[:2])
        an = cm.analyse(r.read_stage(STAGE_LAP_BLEND, 0))
    assert exact == frames * an.flagged_chunks and total == frames * an.chunk_flags.size
    return sums, want, an


def margin_tiles(an, w, h, **margins):
    """Tiles flagged with the margins of k_calm_chunks but not with the given ones."""
    _, tiles = cm.chunk_and_tile_flags(an.block_flags, w, h, False, **margins)
    return an.tile_flags & ~tiles


@pytest.mark.parametrize("w,h,chunk,frames", [(640, 360, 2, 8), (3840, 2160, 32, 128)])
def test_stale_lane_scratch(native_lib, w, h, chunk, frames):
    """Level-0 float tiles the calm route does not recompute still hold the previous content (stale_content): every
    frame must equal the reference, which needs each margin of the tile range k_calm_chunks flags."""
    sums, want, an = stale_then_sparse(w, h, chunk, frames)
    ref_sum = frame_checksum(want)
    assert all(s == ref_sum for s in sums), [i for i, s in enumerate(sums) if s != ref_sum]
    # coverage: the valleys are calm, and each margin is what makes the calm route recompute some tile
    assert 0 < an.flagged_chunks < an.chunk_flags.size
    assert an.nbhd.max() > cm.CALM_SUM
    if w <= 1920:
        assert an.chunk_flags[:, 0].tolist() == [k in (4, 7) for k in range(an.chunk_flags.shape[0])]
        assert margin_tiles(an, w, h, row_margin=(0, 5))[2].all()
        assert margin_tiles(an, w, h, row_margin=(5, 0))[6].all()
    else:
        top, bot = slice(0, 40), slice(50, 90)     # chunk rows clear of the seam between the halves
        assert an.chunk_flags[top, 16].all() and not an.chunk_flags[top, 14:16].any()
        assert an.chunk_flags[bot, 15].all() and not an.chunk_flags[bot, 16:18].any() and not an.chunk_flags[bot, 14].any()
        assert margin_tiles(an, w, h, col_margin=(0, 128))[:30, 14].all()
        assert margin_tiles(an, w, h, col_margin=(8, 120))[36:, 15].all()


def test_mixed_flags_in_one_32_frame_chunk(native_lib):
    """A calm / busy pair with mask ratios alternating 0 and 1 in one 32-frame chunk: some frames flag many chunks and
    some none; the calm route equals the dense route and the reference frame by frame, and the flagged-chunk total
    matches the model."""
    w, h = 256, 96
    busy = synth.block_inputs(w, h, 8, seed=91)
    calm = np.ascontiguousarray(np.repeat(np.full((h, w), 120, np.uint8)[..., None], 3, -1))
    gab = np.zeros((h, w, 3), np.float32)
    cpts = corners(w, h)
    n = 32
    shapes = np.zeros(n, np.float32)
    masks = np.array([k % 2 for k in range(n)], np.float64)
    pair = (calm, busy.bgr1, gab)
    dense, _, laps = render_frames(w, h, pair, (cpts, cpts), shapes[:2], masks[:2], 1, keep=True)
    ans = [cm.analyse(x) for x in laps]
    counts = [a.flagged_chunks for a in ans]
    assert counts[0] != counts[1] and min(counts) < ans[0].chunk_flags.size // 4, counts
    frames2, stats2, _ = render_frames(w, h, pair, (cpts, cpts), shapes, masks, 2, chunk=32, per_call=False)
    frames1, _, _ = render_frames(w, h, pair, (cpts, cpts), shapes, masks, 1, chunk=32, per_call=False)
    assert bits_differ(frames2, frames1) == 0
    assert bits_differ(frames1[:2], dense) == 0
    ref = reference()
    for m in (0.0, 1.0):
        want, _ = ref.morph_images(calm, busy.bgr1, gab, cpts, cpts, 0.0, m, LEVELS)
        for k in range(int(m), n, 2):                      # frames of one mask ratio are the same frame
            assert bits_differ(frames2[k], want) == 0, k
    assert stats2[0] == (n // 2 * sum(counts), n * ans[0].chunk_flags.size)


def test_router_switches_routes_and_stays_exact(native_lib):
    """Mode 0 over calm, then busy, then calm content, one frame per chunk: the router takes both routes and every
    frame equals the dense route."""
    w, h = 128, 64
    ramp = np.repeat(np.tile(np.arange(w, dtype=np.uint8), (h, 1))[..., None], 3, -1)
    calm_img = np.ascontiguousarray(ramp)             # no second differences: no chunk flagged
    busy = synth.block_inputs(w, h, 8, seed=92)
    gab = synth.smooth_field(w, h, seed=93)
    cpts = corners(w, h)
    # the router starts dense and probes every 8th chunk; its running share halves per calm probe, so the calm route
    # starts within about 32 chunks (64 after busy content has stretched the probe interval)
    phases = [("calm", 48), ("busy", 6), ("calm", 100)]
    total = sum(n for _, n in phases)
    plan = host.SequencePlan(cpts, cpts, w, h, np.zeros(1, np.float32))
    routes, frames = {}, {}
    for mode in (0, 1):
        with MorphRenderer(w, h, LEVELS, 4, plan.max_triangles, total, chunk_frames=1) as r:
            r.set_unsharp_mode(mode)
            r.set_points(cpts, cpts)
            slot, seen = 0, []
            for kind, n in phases:
                img = calm_img if kind == "calm" else busy.bgr1
                r.set_pair(img, img if kind == "calm" else busy.bgr2, gab)
                r.unsharp_stats()
                for _ in range(n):
                    r.render(np.zeros(1, np.float32), np.zeros(1), plan.tri_idx, plan.tri_offsets, first_slot=slot)
                    exact, tot = r.unsharp_stats()
                    seen.append((kind, "calm" if exact < tot else "dense"))
                    slot += 1
            frames[mode] = r.download(0, total)
            routes[mode] = seen
    assert bits_differ(frames[0], frames[1]) == 0
    r0 = routes[0]
    assert r0[0] == ("calm", "dense")                              # the router starts on the dense route
    assert ("calm", "calm") in r0[:48]                             # ... and takes the calm route on calm content
    assert ("calm", "calm") in r0[54:]                             # ... and again after the busy stretch
    assert all(route == "dense" for _, route in routes[1])
