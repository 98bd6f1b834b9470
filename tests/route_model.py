"""Which code route the frame path takes at a given frame size, pyramid depth and batch size.

The frame path is bit-identical at every legal size, but the kernels that produce the bytes are chosen from the level
sizes and from the number of frames in a kernel batch (a lane's chunk). This module restates those choices from
poppy_b200/csrc/poppy_cuda.cu (render_chunk, ensure_chunk, poppy_cuda_create) and device/kernels_pyramid.cu (the launch
wrappers and k_pyramid_tail), so that a test can name the routes a case exercises and check that a case list reaches all
of them. tests/test_route_model.py pins the thresholds below to the source text.

Labels:
  tail / blend_coarsest          the levels from the first one no larger than TAIL_MAX x TAIL_MAX on run in one CTA per
                                 frame (k_pyramid_tail), else the coarsest level is blended by k_blend_coarsest
  tail_k0_1 / tail_k0_last       the tail starts at level 1 / at level L - 1
  tail_down_warp / _block        a pyrDown step of the tail ends with a warp-only sync (one job per plane) / a block barrier
  tail_up_warp / _block          the same for a collapse step of the tail (one job per channel)
  pyramid_L1                     a one-level pyramid: no pyrDown launch after level 0 -> 1, no collapse above level 0
  pyr_down_R4 / _R16             k_pyr_down_roll<4> / <16> for a level below the tail
  collapse_tma_R4 / _R16         k_collapse_tma for a level k >= 1 below the tail, 4 or 16 coarse rows per warp
  collapse_roll_R4 / _R16        k_collapse_roll for such a level (too narrow or too flat for the 128 x 2 / 72 x 1 boxes)
  collapse0_tma / collapse0_roll the level-0 collapse with or without tensor maps
  collapse0_tma_h1               the level-0 tensor maps of a one-row frame (their 128 x 2 box is taller than the tensor)
  unsharp_dense                  level-0 collapse to float planes + the exact unsharp pass on every pixel
  calm_emit_tma / calm_emit_roll the calm route at a size where the calm analysis runs: the fused level-0 collapse
                                 (k_collapse_*<true,true>) stores the frame and only flagged strip chunks are recomputed
  calm_forced                    the calm route at a size where the analysis flags every chunk (tests/calm_model.py
                                 force_all: w % 4 != 0, w < 8 or h < 2): the exact pass rewrites every byte of the emit

The unsharp mode is set by the caller; routes() reports both routes, as the route tests render every case on both. Whether
a calm-route frame keeps any emitted byte depends on its content as well: the route tests assert it from the flagged-chunk
counts. The tile-list choice (binned lists or, when a frame's lists exceed the capacity, every triangle in every tile)
depends on the triangle list only: tile_list_entries() counts what a list needs."""
from __future__ import annotations

import itertools

import numpy as np

from tests.calm_model import force_all

SMS = 148                 # CTAs below SMS * CTAS_PER_SM: the 16-row walks are cut into 4-row walks
CTAS_PER_SM = 12
TAIL_MAX = 32             # the tail starts at the first level k >= 1 with w, h <= TAIL_MAX
DN_R = 16                 # output rows per warp of k_pyr_down_roll<DN_R>
CL_R = 16                 # coarse rows per warp of the collapse kernels
FINE_MIN_PITCH = 128      # fine level of a TMA collapse: pitch >= 128 and h >= 2 (the 128 x 2 box)
FINE_MIN_H = 2
COARSE_MIN_PITCH = 72     # coarse level of a TMA collapse: pitch >= 72 (the 72 x 1 box)


def div_up(a, b):
    return -(-a // b)


def levels(w, h, L):
    """[(w, h, pitch)] of levels 0..L: (n + 1) / 2 per level, pitch rounded up to 32 floats."""
    out = []
    for _ in range(L + 1):
        out.append((w, h, (w + 31) & ~31))
        w, h = (w + 1) // 2, (h + 1) // 2
    return out


def tail_k0(w, h, L):
    """First level k in 1 .. L - 1 no larger than TAIL_MAX x TAIL_MAX, or 0 (no tail)."""
    lv = levels(w, h, L)
    for k in range(1, L):
        if lv[k][0] <= TAIL_MAX and lv[k][1] <= TAIL_MAX:
            return k
    return 0


def has_collapse_maps(lv, k):
    """Whether ensure_chunk builds tensor maps for the collapse of level k (fine) from level k + 1 (coarse)."""
    fw, fh, fp = lv[k]
    cp = lv[k + 1][2]
    if k > 0 and (fp < FINE_MIN_PITCH or fh < FINE_MIN_H):
        return False
    return cp >= COARSE_MIN_PITCH


def pyr_down_rows(dw, dh, frames):
    """Output rows per warp of launch_pyr_down for a destination level dw x dh."""
    return 4 if div_up(dw, 128) * div_up(dh, 4 * DN_R) * frames * 7 < SMS * CTAS_PER_SM else DN_R


def collapse_rows(fw, fh, frames):
    """Coarse rows per warp of launch_collapse for a fine level fw x fh."""
    return 4 if div_up(fw, 128) * div_up(fh, 2 * CL_R) * frames < SMS * CTAS_PER_SM else CL_R


def routes(w, h, L, frames_per_chunk):
    """The route labels (module docstring) of one render of w x h frames, L pyramid levels, frames_per_chunk frames per
    kernel batch."""
    lv = levels(w, h, L)
    k0 = tail_k0(w, h, L)
    top = k0 if k0 else L
    out = {"unsharp_dense"}
    if L == 1:
        out.add("pyramid_L1")
    for k in range(1, top):                                 # per-level pyrDown launches: level k -> k + 1
        out.add(f"pyr_down_R{pyr_down_rows(lv[k + 1][0], lv[k + 1][1], frames_per_chunk)}")
    if k0:
        out.add("tail")
        if k0 == 1:
            out.add("tail_k0_1")
        if k0 == L - 1:
            out.add("tail_k0_last")
        for k in range(k0, L):
            dw, dh = lv[k + 1][:2]
            jobs = 7 * div_up(dw, 64) * div_up(dh, 4)
            out.add("tail_down_warp" if jobs == 7 and k + 1 < L else "tail_down_block")
        for k in range(L - 1, k0 - 1, -1):
            jobs = 3 * div_up(lv[k][0], 128) * div_up(lv[k][1], 8)
            nxt = 3 * div_up(lv[k - 1][0], 128) * div_up(lv[k - 1][1], 8) if k > k0 else 0
            out.add("tail_up_warp" if jobs == 3 and nxt == 3 else "tail_up_block")
    else:
        out.add("blend_coarsest")
    for k in range(top - 1, 0, -1):                          # per-level collapses below the tail
        kind = "tma" if has_collapse_maps(lv, k) else "roll"
        out.add(f"collapse_{kind}_R{collapse_rows(lv[k][0], lv[k][1], frames_per_chunk)}")
    level0 = "tma" if has_collapse_maps(lv, 0) else "roll"
    out.add(f"collapse0_{level0}")
    if level0 == "tma" and h == 1:
        out.add("collapse0_tma_h1")
    out.add("calm_forced" if force_all(w, h) else f"calm_emit_{level0}")
    return out


TILE_W, TILE_H = 64, 32      # screen tiles of the rasteriser (RW_TW x RW_TH)


def tile_list_entries(w, h, verts):
    """Entries the binned tile lists of one frame need (k_tri_geometry / tile_bbox): per triangle, the tiles its bounding
    box touches once clamped to the frame. verts: T x 3 x 2 integer (truncated) vertices. With a capacity below this
    count the frame takes the overflow path."""
    v = np.asarray(verts, np.int64).reshape(-1, 3, 2)
    x0, x1 = np.maximum(v[..., 0].min(1), 0), np.minimum(v[..., 0].max(1), w - 1)
    y0, y1 = np.maximum(v[..., 1].min(1), 0), np.minimum(v[..., 1].max(1), h - 1)
    inside = (x0 <= x1) & (y0 <= y1)
    return int(((x1 // TILE_W - x0 // TILE_W + 1) * (y1 // TILE_H - y0 // TILE_H + 1))[inside].sum())


def launches(w, h, L):
    """Launches per kernel class (poppy_cuda_stage_times names) of a one-chunk render on the dense route."""
    k0 = tail_k0(w, h, L)
    top = k0 if k0 else L
    # pyrDown: level 0 -> 1, then one launch per level below the tail (the tail counts as a collapse launch)
    # collapse: the tail or k_blend_coarsest, one collapse per level top - 1 .. 1, the level-0 collapse
    return {"pyr_down": 1 + (top - 1), "blend_collapse": 1 + (top - 1) + 1}


GRID_SIZES = (1, 2, 3, 5, 7, 8, 9, 31, 32, 33, 63, 64, 65, 127, 128, 129, 130, 255, 256, 300, 1000, 2000, 2048, 4000)
GRID_LEVELS = (1, 2, 3, 4, 6, 64)
GRID_FRAMES = (1, 8, 32, 64, 128)


def enumerate_routes():
    """Every label routes() gives over a grid of sizes, pyramid depths and batch sizes wide enough to reach all of them."""
    out = set()
    for w, h, L, f in itertools.product(GRID_SIZES, GRID_SIZES, GRID_LEVELS, GRID_FRAMES):
        out |= routes(w, h, L, f)
    return out
