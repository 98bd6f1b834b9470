"""Triangle lists made by the caller, not by the Delaunay stage: poppy_cuda_render accepts any list with valid indices, and
even Delaunay lists overlap once their vertices are truncated to integers. The rasteriser's painting order ("later
triangle wins", atomicMax on the colour), its inclusive tile bounding boxes, the Bresenham outline pieces across tile
edges, the list-overflow path and the zero matrices of degenerate triangles (at shape 1 the inverse warp of image 1
is the zero matrix, whose z = 0 takes the division fallback of map_eval) must give the triangle map, the warps and
the frame of the CPU restatement (oracle/port.py, whose fill is pinned to cv::fillConvexPoly by
tests/test_oracle_vs_reference.py) bit for bit.

pts1 == pts2 and shape 0.5 or 1: the morphed points are the clipped points exactly, so a list names its integer
vertices."""
import numpy as np
import pytest

from tests.route_model import TILE_H as TH, TILE_W as TW, tile_list_entries
from tests.util import any_size_inputs, bits_differ

pytestmark = pytest.mark.gpu

MASK, LEVELS = 0.3, 4


def below(v):
    """The float just below v: truncates to v - 1."""
    return np.nextafter(np.float32(v), np.float32(-np.inf))


def random_overlapping(w, h, n_pts, n_tri, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    pts = (rng.uniform(0, 1, (n_pts, 2)) * [w - 1, h - 1]).astype(np.float32)
    return pts, rng.integers(0, n_pts, (n_tri, 3)).astype(np.int32)


def degenerate(w, h):
    """Zero-area triangles (collinear vertices, a repeated index, three equal indices, horizontal and vertical segments)
    over and under ordinary ones."""
    pts = np.array([[10, 10], [50, 30], [90, 50], [130, 70], [20, 90], [250, 5], [250, 95], [5, 60], [290, 60],
                    [70.5, 40.25], [180, 20], [200, 80], [33.7, 33.7]], np.float32)
    tri = [[0, 1, 2], [0, 4, 5], [1, 3, 2], [3, 3, 4], [9, 9, 9], [5, 6, 6], [7, 8, 7], [4, 10, 11], [0, 2, 3],
           [12, 12, 12], [5, 6, 5], [7, 8, 1], [10, 11, 10]]
    return pts, np.array(tri, np.int32)


def tile_slivers(w, h):
    """Thin triangles whose bounding boxes end exactly on the last column / row of a tile or on the first of the next."""
    pts, tri = [], []
    for k in (1, 2, 3):
        for x1 in (TW * k - 1, TW * k):
            i = len(pts)
            pts += [[x1 - 40, 3 + 2 * k], [x1, 5 + 2 * k], [x1 - 20, 6 + 2 * k]]
            tri.append([i, i + 1, i + 2])
        for y1 in (TH * k - 1, TH * k):
            if y1 >= h:
                continue
            i = len(pts)
            pts += [[20 * k + 3, y1 - 25], [20 * k + 5, y1], [20 * k + 4, y1 - 12]]
            tri.append([i, i + 1, i + 2])
    # one that ends on both at once, and a sliver along a tile's top row
    i = len(pts)
    pts += [[100, 40], [TW * 2, TH * 2], [110, TH * 2 - 1], [10, TH], [200, TH], [100, TH + 1]]
    tri += [[i, i + 1, i + 2], [i + 3, i + 4, i + 5]]
    return np.array(pts, np.float32), np.array(tri, np.int32)


def borders(w, h):
    """Vertices on rows and columns 0 and w - 1 / h - 1 and just past them (clip_points keeps w - 1 < x <= w), and
    triangles covering the whole frame."""
    pts = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1], [w, h], [w, 0.5], [0.5, h], [w - 0.5, h - 0.5],
                    [w // 2, 0], [0, h // 2], [w - 1, h // 2], [w // 2, h - 1], [-5, -5], [w + 9, h + 9]], np.float32)
    tri = [[0, 1, 2], [1, 3, 2], [8, 9, 11], [4, 5, 6], [10, 11, 7], [0, 8, 9], [12, 13, 1], [3, 4, 7], [0, 3, 1],
           [2, 10, 8]]
    return pts, np.array(tri, np.int32)


def long_thin(w, h):
    """On a 7000 x 3 frame: triangles across the whole width, one to three rows tall (Bresenham pieces in 110 tiles)."""
    pts = np.array([[0, 0], [w - 1, 1], [w - 1, 2], [0, 2], [w // 2, 0], [w - 1, 0], [0, 1], [4321, 2], [17, 0],
                    [6990, 2]], np.float32)
    tri = [[0, 1, 2], [3, 4, 5], [6, 7, 5], [8, 9, 2], [0, 5, 3], [1, 8, 7]]
    return pts, np.array(tri, np.int32)


def just_below_integers(w, h):
    """Vertices a float below integers (truncation toward zero takes them one lower) next to the integers themselves."""
    ints = np.array([[64, 32], [128, 10], [100, 64], [1, 1], [200, 90], [30, 96], [150, 50]], np.float32)
    pts = np.concatenate([ints, below(ints)])
    n = len(ints)
    tri = [[0, 1, 2], [n, n + 1, n + 2], [3, 4, 5], [n + 3, n + 4, n + 5], [0, n + 6, 4], [n, 6, n + 4]]
    return pts, np.array(tri, np.int32)


W, H = 300, 100
LISTS = {       # name: (w, h, list, shape ratio)
    "random_overlapping": (W, H, lambda: random_overlapping(W, H, 60, 300, seed=5), 0.5),
    "random_overlapping_reversed": (W, H, lambda: (lambda p, t: (p, t[::-1].copy()))(*random_overlapping(W, H, 60, 300, seed=5)),
                                    0.5),
    "degenerate": (W, H, lambda: degenerate(W, H), 0.5),
    "degenerate_shape1": (W, H, lambda: degenerate(W, H), 1.0),
    "tile_edge_slivers": (W, H, lambda: tile_slivers(W, H), 0.5),
    "borders_and_whole_frame": (W, H, lambda: borders(W, H), 0.5),
    "long_thin_7000x3": (7000, 3, lambda: long_thin(7000, 3), 0.5),
    "just_below_integers": (W, H, lambda: just_below_integers(W, H), 0.5),
    "empty": (W, H, lambda: (np.array([[1, 1], [W - 2, H - 2], [5, H - 3]], np.float32), np.zeros((0, 3), np.int32)), 0.5),
    "max_triangles": (W, H, lambda: random_overlapping(W, H, 200, 2048, seed=6), 0.5),
}


def render_list(w, h, pts, tri, shape, list_capacity=None):
    from poppy_b200 import renderer as R
    bgr1, bgr2, gab, _, _ = any_size_inputs(w, h, seed=3)
    with R.MorphRenderer(w, h, LEVELS, len(pts), max(len(tri), 1), 1, keep_stages=True) as r:
        if list_capacity:
            r.set_tile_list_capacity(list_capacity)
        r.set_pair(bgr1, bgr2, gab)
        r.set_points(pts, pts)
        r.render([shape], [MASK], tri, [0, len(tri)])
        got = {"dst": r.download(0, 1)[0], "morphed_points": r.read_stage(R.STAGE_MORPHED_POINTS, 0),
               "tri_map": r.read_stage(R.STAGE_TRI_MAP, 0), "warped1": r.read_stage(R.STAGE_WARPED1, 0),
               "warped2": r.read_stage(R.STAGE_WARPED2, 0)}
        if len(tri):
            got["inv_m1"] = r.read_stage(R.STAGE_INV_M1, 0, len(tri))
            got["inv_m2"] = r.read_stage(R.STAGE_INV_M2, 0, len(tri))
    return got, (bgr1, bgr2, gab)


@pytest.mark.parametrize("list_capacity", [None, 1], ids=["binned", "overflow"])
@pytest.mark.parametrize("name", list(LISTS))
def test_caller_triangle_list(native_lib, name, list_capacity):
    from oracle import port
    w, h, make, shape = LISTS[name]
    pts, tri = make()
    got, (bgr1, bgr2, gab) = render_list(w, h, pts, tri, shape, list_capacity)
    want = port.morph_frame(bgr1, bgr2, gab, pts, pts, tri, shape, MASK, LEVELS)
    clipped = port.morph_points(pts, pts, 0.0, w, h)
    assert bits_differ(want.morphed_points, clipped) == 0           # the list names its vertices exactly
    assert bits_differ(got["morphed_points"], want.morphed_points) == 0
    assert bits_differ(got["tri_map"], want.tri_map) == 0, "triangle-ID map"
    if list_capacity:           # every non-empty list overflows a one-entry capacity: every tile tests every triangle
        assert (tile_list_entries(w, h, np.trunc(clipped[tri])) > list_capacity) == (len(tri) > 0)
    if len(tri):
        v = np.trunc(clipped[tri]).astype(np.int32).reshape(-1, 6)
        _, _, _, im1, im2 = port.triangle_matrices(v, v, np.float32(shape))
        assert bits_differ(got["inv_m1"], im1) == 0
        assert bits_differ(got["inv_m2"], im2) == 0
        if name == "degenerate_shape1":              # zero-area triangles: image 1's inverse warp is the zero matrix
            a = v.reshape(-1, 3, 2).astype(np.int64)
            area2 = (a[:, 1, 0] - a[:, 0, 0]) * (a[:, 2, 1] - a[:, 0, 1]) - (a[:, 1, 1] - a[:, 0, 1]) * (a[:, 2, 0] - a[:, 0, 0])
            assert (area2 == 0).sum() >= 6 and not im1[area2 == 0].any()
    assert bits_differ(got["warped1"], want.warped1) == 0, "remap of image 1"
    assert bits_differ(got["warped2"], want.warped2) == 0, "remap of image 2"
    assert bits_differ(got["dst"], want.dst) == 0, "final 8-bit frame"
    # what the list exercises
    ids = want.tri_map
    if name == "random_overlapping_reversed":             # the triangles overlap: their order decides the map
        _, fwd = LISTS["random_overlapping"][2]()
        same_ids = np.where(ids > 0, len(tri) + 1 - ids, 0)
        assert bits_differ(port.morph_frame(bgr1, bgr2, gab, pts, pts, fwd, shape, MASK, LEVELS).tri_map, same_ids) > 1000
    if name == "empty":
        assert not ids.any()
