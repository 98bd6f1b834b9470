"""The route model (tests/route_model.py) against the source it restates: if a threshold it mirrors moves, these tests
fail instead of the route tests silently dropping coverage."""
import os
import re

from tests import route_model as m

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "poppy_b200", "csrc")


def _source(rel):
    with open(os.path.join(CSRC, rel)) as f:
        return re.sub(r"\s+", " ", f.read())


def test_model_thresholds_appear_in_the_source():
    host = _source("poppy_cuda.cu")
    pyr = _source(os.path.join("device", "kernels_pyramid.cu"))
    # level geometry and the tail's first level (poppy_cuda_create)
    assert "d.pitch = (lw + 31) & ~31" in host
    assert "lw = (lw + 1) / 2; lh = (lh + 1) / 2;" in host
    assert f"for (int k = 1; k < pyramid_levels; ++k) if (c->lv[k].w <= {m.TAIL_MAX} && c->lv[k].h <= {m.TAIL_MAX})" in host
    # the collapse tensor maps (ensure_chunk)
    assert f"if (fl.pitch < {m.FINE_MIN_PITCH} || fl.h < {m.FINE_MIN_H}) continue;" in host
    assert f"if (ok && cl.pitch < {m.COARSE_MIN_PITCH}) {{ m = CollapseMaps(); continue; }}" in host
    # the per-level launches and the tail (render_chunk)
    assert "for (int k = 1; k < (k0 ? k0 : L); ++k)" in host
    assert "for (int k = (k0 ? k0 : L) - 1; k >= 1; --k)" in host
    # 4- or 16-row walks (launch_pyr_down, launch_collapse)
    assert f"constexpr int DN_R = {m.DN_R};" in pyr and f"constexpr int CL_R = {m.CL_R};" in pyr
    assert pyr.count(f"< {m.SMS} * {m.CTAS_PER_SM}") == 2
    assert "ctas16 = (long long)div_up(dl.w, 128) * div_up(dl.h, 4 * DN_R) * frames * 7;" in pyr
    assert "ctas16 = (long long)div_up(fl.w, 128) * div_up(fl.h, 2 * CL_R) * frames;" in pyr
    # the level-0 collapse always walks CL_R coarse rows
    assert pyr.count("const dim3 grid(div_up(w, 128), div_up(h, 2 * CL_R), frames);") == 2
    # the tail's syncs (k_pyramid_tail)
    assert "jobs = 7 * ncol * nrow;" in pyr and "const int ncol = div_up(D.w, 64), nrow = div_up(D.h, 4)" in pyr
    assert "if (jobs == 7 && k + 1 < L) __syncwarp(); else __syncthreads();" in pyr
    assert "const int ncol = div_up(F.w, 128), nrow = div_up(F.h, 8), jobs = 3 * ncol * nrow;" in pyr
    assert "const int next_jobs = k > k0 ? 3 * div_up(lv[k - 1].w, 128) * div_up(lv[k - 1].h, 8) : 0;" in pyr
    assert "if (jobs == 3 && next_jobs == 3) __syncwarp(); else __syncthreads();" in pyr
    # the calm analysis flags every chunk of frames it cannot scan (launch_calm_analysis)
    assert "if ((w & 3) != 0 || w < 8 || h < 2 ||" in _source(os.path.join("device", "kernels_unsharp.cu"))
    # tile lists: inclusive bounding boxes clamped to the frame, 64 x 32 tiles; overflow above the capacity
    geo = _source(os.path.join("device", "kernels_geometry.cu"))
    assert ("const int x0 = max(min(min(r.vx[0], r.vx[1]), r.vx[2]), 0), x1 = min(max(max(r.vx[0], r.vx[1]), r.vx[2]), w - 1);"
            in geo)
    assert ("const int y0 = max(min(min(r.vy[0], r.vy[1]), r.vy[2]), 0), y1 = min(max(max(r.vy[0], r.vy[1]), r.vy[2]), h - 1);"
            in geo)
    assert "tx0 = x0 / RW_TW; tx1 = x1 / RW_TW; ty0 = y0 / RW_TH; ty1 = y1 / RW_TH;" in geo
    assert "overflow[f] = carry_s > cap ? 1 : 0;" in geo
    assert f"constexpr int RW_TW = {m.TILE_W}, RW_TH = {m.TILE_H};" in _source(os.path.join("device", "common.cuh"))


def test_enumerate_routes_reaches_every_label():
    labels = m.enumerate_routes()
    want = {"tail", "blend_coarsest", "tail_k0_1", "tail_k0_last", "tail_down_warp", "tail_down_block", "tail_up_warp",
            "tail_up_block", "pyramid_L1", "pyr_down_R4", "pyr_down_R16", "collapse_tma_R4", "collapse_tma_R16",
            "collapse_roll_R4", "collapse_roll_R16", "collapse0_tma", "collapse0_roll", "collapse0_tma_h1",
            "unsharp_dense", "calm_emit_tma", "calm_emit_roll", "calm_forced"}
    assert labels == want, labels ^ want


def test_model_examples():
    # R depends on the frames per batch: 2048 x 64 keeps its 16-row pyrDown walks only with a full 128-frame batch
    assert "pyr_down_R16" in m.routes(2048, 64, 6, 128) and "pyr_down_R4" in m.routes(2048, 64, 6, 128)
    assert not any(r.endswith("R16") for r in m.routes(2048, 64, 6, 32))
    assert "collapse_roll_R16" in m.routes(1, 2000, 2, 64)
    assert "collapse_tma_R16" in m.routes(4000, 3, 2, 128)
    # the level-0 maps of a one-row frame from w = 129 on
    assert "collapse0_tma_h1" in m.routes(129, 1, 6, 1) and "collapse0_roll" in m.routes(128, 1, 6, 1)
    # 1 x 1 frames: levels repeat at 1 x 1, the tail from level 1 on
    assert m.levels(1, 1, 3) == [(1, 1, 32)] * 4 and m.tail_k0(1, 1, 3) == 1 and m.tail_k0(1, 1, 1) == 0
    assert m.launches(1, 1, 1) == {"pyr_down": 1, "blend_collapse": 2}
    assert m.launches(2048, 64, 6) == {"pyr_down": 6, "blend_collapse": 7}
    # the calm analysis runs at 8 x 9 and 124 x 33; at 7 x 9, 130 x 33 and 4000 x 1 it flags everything
    assert "calm_emit_roll" in m.routes(8, 9, 6, 8) and "calm_emit_roll" in m.routes(124, 33, 4, 8)
    assert all("calm_forced" in m.routes(w, h, 4, 8) for w, h in ((7, 9), (130, 33), (4000, 1)))
    # tile-list entries: a triangle in one tile, one across a tile corner, one clamped to the frame, one outside it
    tris = [[[1, 1], [5, 1], [1, 5]], [[60, 30], [70, 30], [60, 40]], [[-9, -9], [300, 0], [0, 200]], [[400, 5], [410, 5], [400, 9]]]
    assert m.tile_list_entries(300, 100, tris) == 1 + 4 + 5 * 4
