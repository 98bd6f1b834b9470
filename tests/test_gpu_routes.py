"""Every route of the frame path (tests/route_model.py) against the reference, bit for bit: degenerate frames (w or h of
1, w < 8), one-level pyramids, one-row frames on the level-0 tensor maps, and batches large enough for the 16-row walks.

For each case (w, h, L, chunk):
  * stages: a keep_stages render (one frame per chunk, dense route) equals the reference stage by stage, launches the
    pyrDown and collapse kernels the model predicts, and gives the same triangle map, warps and frame with a one-entry
    tile list (every tile tests every triangle);
  * batch: `chunk` frames of distinct shape and mask ratios in one kernel batch equal the reference and the same frames
    rendered one per chunk, on the dense and on the calm route. The content is smooth, so that where the calm analysis
    runs some strip chunks keep the bytes the fused level-0 collapse stored; each route renders on its own renderer;
  * chain: a 6-frame chain (api.morph_sequence) equals the reference's frame loop."""
import numpy as np
import pytest

from poppy_b200 import host
from tests import calm_model as cm
from tests import route_model as model
from tests.util import any_size_inputs, bits_differ, flat_tri, reference

CASES = [
    # w, h, levels, frames per chunk
    (1, 1, 1, 1),
    (1, 1, 3, 8),
    (1, 2, 2, 8),
    (1, 3, 64, 8),
    (1, 40, 4, 8),
    (1, 40, 1, 8),
    (1, 65, 3, 8),
    (40, 1, 4, 8),
    (2, 2, 3, 8),
    (3, 5, 64, 8),
    (7, 9, 6, 8),
    (8, 9, 6, 8),               # the narrowest frame the calm analysis scans
    (124, 33, 4, 8),            # ... and one without level-0 tensor maps
    (129, 1, 6, 8),             # level-0 tensor maps of a one-row frame
    (300, 1, 3, 8),
    (4000, 2, 12, 8),
    (200, 150, 1, 8),           # one-level pyramid with level-0 tensor maps
    (256, 200, 4, 8),           # the tail starts at level L - 1
    (1, 300, 2, 128),           # 16-row pyrDown walks at modest sizes: the batch is full
    (1, 2000, 2, 64),           # ... k_collapse_roll with 16-row walks
    (4000, 3, 2, 128),          # ... k_collapse_tma with 16-row walks
    (2048, 64, 6, 128),         # 4- and 16-row pyrDown walks in one render
    (2048, 64, 6, 32),          # the same frame size with 4-row walks only
]


# the stage and chain checks do not depend on the batch size
FRAME_CASES = sorted({c[:3] for c in CASES})


def case_id(c):
    return "{}x{}_L{}".format(*c[:3]) + ("_c{}".format(c[3]) if len(c) > 3 else "")


def test_cases_cover_every_route():
    covered = set().union(*(model.routes(*c) for c in CASES))
    assert covered == model.enumerate_routes(), model.enumerate_routes() - covered
    # the batch decides the walk length: at 32 frames per chunk 2048 x 64 keeps to 4-row walks
    for c in ((1, 300, 2, 128), (1, 2000, 2, 64), (4000, 3, 2, 128), (2048, 64, 6, 128)):
        assert any(r.endswith("_R16") for r in model.routes(*c)), c
    assert not any(r.endswith("_R16") for r in model.routes(2048, 64, 6, 32))


@pytest.mark.parametrize("w,h,L", FRAME_CASES, ids=[case_id(c) for c in FRAME_CASES])
def test_reference_runs_at_case_size(w, h, L):
    """The reference takes every case size with these inputs (synth.make_inputs does not go below about 8 x 8)."""
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h)
    st = reference().stages(bgr1, bgr2, gab, p1, p2, 0.4, 0.6, L)
    assert st.dst.shape == (h, w, 3) and st.morphed_points.shape == p1.shape
    assert (st.tri_idx >= 0).all() and (st.tri_idx < len(p1)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,L", FRAME_CASES, ids=[case_id(c) for c in FRAME_CASES])
def test_stages_and_launches(native_lib, w, h, L):
    from oracle import port
    from poppy_b200 import renderer as R
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h)
    s, m = 0.37, 0.61
    want = reference().stages(bgr1, bgr2, gab, p1, p2, s, m, L)
    tri = want.tri_idx
    cat, offs = flat_tri([tri])
    with R.MorphRenderer(w, h, L, len(p1), max(len(tri), 1), 1, keep_stages=True, stage_timing=True) as r:
        r.set_pair(bgr1, bgr2, gab)
        r.set_points(p1, p2)
        r.render([s], [m], cat, offs)
        got = r.download(0, 1)[0]
        counts = {k: v["launches"] for k, v in r.stage_times().items() if k in ("pyr_down", "blend_collapse")}
        assert counts == model.launches(w, h, L), (counts, model.tail_k0(w, h, L))
        assert bits_differ(r.read_stage(R.STAGE_MORPHED_POINTS, 0), want.morphed_points) == 0
        tri_map = r.read_stage(R.STAGE_TRI_MAP, 0)
        assert bits_differ(tri_map, want.tri_map) == 0, "triangle-ID map"
        if len(tri):
            c1 = port.morph_points(p1, p1, 0.0, w, h)
            c2 = port.morph_points(p2, p2, 0.0, w, h)
            t1 = np.trunc(c1[tri]).astype(np.int32).reshape(-1, 6)
            t2 = np.trunc(c2[tri]).astype(np.int32).reshape(-1, 6)
            _, _, _, im1, im2 = port.triangle_matrices(t1, t2, np.float32(s))
            assert bits_differ(r.read_stage(R.STAGE_INV_M1, 0, len(tri)), im1) == 0
            assert bits_differ(r.read_stage(R.STAGE_INV_M2, 0, len(tri)), im2) == 0
        warped = [r.read_stage(R.STAGE_WARPED1, 0), r.read_stage(R.STAGE_WARPED2, 0)]
        assert bits_differ(warped[0], want.warped1) == 0, "remap of image 1"
        assert bits_differ(warped[1], want.warped2) == 0, "remap of image 2"
        assert bits_differ(r.read_stage(R.STAGE_MASK, 0), want.mask) == 0, "blend mask"
        assert bits_differ(r.read_stage(R.STAGE_LAP_BLEND, 0), want.lap_blend) == 0, "Laplacian blend"
        assert bits_differ(got, want.dst) == 0, "final 8-bit frame"
        # the same frame without tile lists
        r.set_tile_list_capacity(1)
        r.render([s], [m], cat, offs)
        assert bits_differ(r.download(0, 1)[0], got) == 0
        assert bits_differ(r.read_stage(R.STAGE_TRI_MAP, 0), tri_map) == 0
        assert bits_differ(r.read_stage(R.STAGE_WARPED1, 0), warped[0]) == 0
        assert bits_differ(r.read_stage(R.STAGE_WARPED2, 0), warped[1]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,L,chunk", CASES, ids=[case_id(c) for c in CASES])
def test_batch_dense_and_calm(native_lib, w, h, L, chunk):
    from poppy_b200.renderer import MorphRenderer
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=1, smooth=True)
    rng = np.random.Generator(np.random.PCG64(chunk))
    shapes = np.linspace(0.0, 1.0, chunk, dtype=np.float32)
    masks = rng.permutation(np.linspace(0.0, 1.0, chunk))
    plan = host.SequencePlan(p1, p2, w, h, shapes)
    tri_max = max(plan.max_triangles, 1)

    def render(mode, chunk_frames):
        """A fresh renderer: no earlier result sits in its ring or lane scratch. Returns (frames, unsharp_stats)."""
        with MorphRenderer(w, h, L, len(p1), tri_max, chunk, chunk_frames=chunk_frames) as r:
            r.set_unsharp_mode(mode)
            r.set_pair(bgr1, bgr2, gab)
            r.set_points(p1, p2)
            r.unsharp_stats()
            r.render(shapes, masks, plan.tri_idx, plan.tri_offsets)
            stats = r.unsharp_stats()
            return r.download(0, chunk), stats

    calm, (exact, total) = render(2, chunk)         # one lane, one batch of `chunk`
    dense, _ = render(1, chunk)
    single, _ = render(1, 1)
    plan.close()
    ref = reference()
    flagged = chunks = 0
    for k in range(chunk):
        want = ref.stages(bgr1, bgr2, gab, p1, p2, float(shapes[k]), float(masks[k]), L)
        assert bits_differ(dense[k], want.dst) == 0, ("dense route", k)
        assert bits_differ(calm[k], want.dst) == 0, ("calm route", k)
        assert bits_differ(single[k], want.dst) == 0, ("one frame per chunk", k)
        an = cm.analyse(want.lap_blend)
        flagged += an.flagged_chunks
        chunks += an.chunk_flags.size
    # the calm route recomputed exactly the chunks its analysis flags; where the analysis runs, the other chunks keep
    # the bytes of the fused level-0 collapse
    assert (exact, total) == (flagged, chunks)
    if not cm.force_all(w, h):
        assert exact < total


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,L", FRAME_CASES, ids=[case_id(c) for c in FRAME_CASES])
def test_chain(native_lib, w, h, L):
    from poppy_b200 import api
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=2)
    settings = api.Settings.instance()
    old = settings.pyramid_levels
    settings.pyramid_levels = L
    try:
        got = api.morph_sequence(bgr1, bgr2, gab, p1, p2, number_of_frames=6)
    finally:
        settings.pyramid_levels = old
        api.release()
    want, _ = reference().chain(bgr1, bgr2, gab, p1, p2, 6, L)
    for k in range(6):
        assert bits_differ(got[k], want[k]) == 0, k
