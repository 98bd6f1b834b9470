"""GPU parity through the public API (Python mirror of the reference interface -> C ABI -> CUDA kernels):
single frames, the chain recurrence, batched independent phases, the golden fixtures and error behaviour. Without the
reference library the parity cases compare with the CPU restatement, whose triangle lists come from the product's host
stage (see tests.util.reference); the golden fixtures below carry the reference's own triangle lists."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

from poppy_b200 import api, host, synth
from tests.util import assert_frame_parity, bits_differ, flat_tri, reference as _ref

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(autouse=True)
def _fresh_api(native_lib):
    yield
    api.release()


@pytest.mark.parametrize("kind,w,h,n,s,m,levels", [
    ("noise", 320, 240, 150, 0.3, 0.3, 6), ("noise", 501, 333, 90, 0.75, 0.2, 64), ("shapes", 256, 256, 48, 0.5, 0.5, 64),
    ("blocks", 640, 480, 120, 0.1, 0.1, 6), ("blocks", 203, 157, 40, 0.9, 0.95, 3), ("noise", 31, 23, 6, 0.5, 0.5, 8),
])
def test_morph_images_matches_reference(kind, w, h, n, s, m, levels):
    ref = _ref()
    inp = {"noise": lambda: synth.make_inputs(w, h, n, 8.0, seed=3), "shapes": lambda: synth.shape_inputs(w, h, n, seed=4),
           "blocks": lambda: synth.block_inputs(w, h, n, seed=5)}[kind]()
    api.Settings.instance().pyramid_levels = levels
    dst, mp = api.morph_images(inp.bgr1, inp.bgr2, inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, s, m)
    want, want_pts = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, s, m, levels)
    assert bits_differ(mp, want_pts) == 0
    assert_frame_parity(dst, want, (kind, w, h))            # the north-star tolerance ...
    assert bits_differ(dst, want) == 0                      # ... and in fact bit-identical


def test_c_flavour_morph_images(native_lib):
    ref = _ref()
    w, h, levels = 200, 160, 5
    inp = synth.make_inputs(w, h, 70, 6.0, seed=8)
    from poppy_b200.renderer import MorphRenderer
    with MorphRenderer(w, h, levels, 128, 512, 1) as r:
        dst = np.zeros((h, w + 7, 3), np.uint8)             # padded destination rows
        mp = np.zeros((len(inp.pts1), 2), np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = native_lib.poppy_morph_images(r._ctx, p(inp.bgr1), w * 3, p(inp.bgr2), w * 3, p(inp.gabor2), w * 12,
                                           p(inp.pts1), p(inp.pts2), len(inp.pts1), 0.6, 0.4, p(dst), (w + 7) * 3, p(mp))
        assert rc == 0, native_lib.poppy_host_last_error()
    want, want_pts = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, 0.6, 0.4, levels)
    assert bits_differ(dst[:, :w], want) == 0 and bits_differ(mp, want_pts) == 0


def test_chain_sequence_matches_golden():
    g = np.load(os.path.join(GOLDEN, "chain_shapes_80x64_N12_L64.npz"))
    api.Settings.instance().pyramid_levels = int(g["levels"])
    frames = api.morph_sequence(g["bgr1"], g["bgr2"], g["gabor2"], g["pts1"], g["pts2"], number_of_frames=int(g["n_frames"]))
    for j in range(len(frames)):
        assert bits_differ(frames[j], g["frames"][j]) == 0, f"chain frame {j}"


def test_chain_sequence_matches_reference_live():
    ref = _ref()
    w, h, n_frames, levels = 240, 180, 20, 6
    inp = synth.shape_inputs(w, h, 40, seed=12)
    api.Settings.instance().pyramid_levels = levels

    class Sink:
        def __init__(self):
            self.n = 0

        def write(self, frame):
            self.n += 1

    sink = Sink()
    frames = api.morph_sequence(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, writer=sink, number_of_frames=n_frames)
    want, _ = ref.chain(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, n_frames, levels)
    assert sink.n == n_frames
    for j in range(n_frames):
        assert_frame_parity(frames[j], want[j], f"chain frame {j}")
        assert bits_differ(frames[j], want[j]) == 0, f"chain frame {j}"


@pytest.mark.parametrize("chunk", [1, 3, 16])
def test_batched_phases_match_reference_for_any_chunking(chunk):
    ref = _ref()
    from poppy_b200.renderer import MorphRenderer
    w, h, levels = 330, 250, 6
    inp = synth.make_inputs(w, h, 120, 8.0, seed=15)
    phases = np.linspace(0, 1, 11).astype(np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    with MorphRenderer(w, h, levels, len(inp.pts1), plan.max_triangles, len(phases), chunk_frames=chunk) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
        frames = r.download(0, len(phases))
        for k, s in enumerate(phases):
            want, pts = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, float(s), float(s), levels)
            assert bits_differ(frames[k], want) == 0, (chunk, k)
            assert bits_differ(r.morphed_points(k), pts) == 0


def test_tile_list_overflow_path_is_exact():
    """A frame whose binned triangle lists do not fit the list capacity is rasterised by testing every triangle in
    every tile; the frames must not change."""
    ref = _ref()
    from poppy_b200.renderer import MorphRenderer
    w, h, levels = 400, 300, 5
    inp = synth.make_inputs(w, h, 300, 8.0, seed=21)
    phases = np.array([0.2, 0.8], np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    with MorphRenderer(w, h, levels, len(inp.pts1), plan.max_triangles, len(phases)) as r:
        r.set_tile_list_capacity(7)            # far fewer than the ~600 triangles of a frame
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
        frames = r.download(0, len(phases))
        for k, s in enumerate(phases):
            want, _ = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, float(s), float(s), levels)
            assert bits_differ(frames[k], want) == 0, k


FRAME_FILES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "*.npz"))
                     if not os.path.basename(f).startswith(("chain_", "topology")))


@pytest.mark.parametrize("path", FRAME_FILES, ids=[os.path.basename(f)[:-4] for f in FRAME_FILES])
def test_golden_fixtures_on_gpu(path):
    from poppy_b200 import renderer as R
    g = np.load(path)
    h, w = g["bgr1"].shape[:2]
    s, m, levels = float(g["shape"]), float(g["mask_ratio"]), int(g["levels"])
    tri = host.triangulate(host.morph_points(g["pts1"], g["pts2"], s, w, h), w, h)
    assert (tri == g["tri_idx"]).all()
    with R.MorphRenderer(w, h, levels, len(g["pts1"]), len(tri), 1, keep_stages=True) as r:
        r.set_pair(g["bgr1"], g["bgr2"], g["gabor2"])
        r.set_points(g["pts1"], g["pts2"])
        cat, offs = flat_tri([tri])
        r.render([s], [m], cat, offs)
        assert bits_differ(r.download(0, 1)[0], g["dst"]) == 0
        for stage, key in ((R.STAGE_MORPHED_POINTS, "morphed_points"), (R.STAGE_TRI_MAP, "tri_map"),
                           (R.STAGE_WARPED1, "warped1"), (R.STAGE_WARPED2, "warped2"), (R.STAGE_MASK, "mask"),
                           (R.STAGE_LAP_BLEND, "lap_blend")):
            assert bits_differ(r.read_stage(stage, 0), g[key]) == 0, key


def test_error_behaviour(native_lib):
    from poppy_b200._lib import PoppyCudaError
    from poppy_b200.renderer import MorphRenderer
    w, h = 64, 48
    inp = synth.make_inputs(w, h, 10, 3.0, seed=2)
    tri = host.triangulate(host.morph_points(inp.pts1, inp.pts2, 0.5, w, h), w, h)
    cat, offs = flat_tri([tri])
    with MorphRenderer(w, h, 3, 32, 4, 2) as r:                      # room for 4 triangles only
        with pytest.raises(PoppyCudaError) as e:
            r.render([0.5], [0.5], cat, offs)                        # before set_pair / set_points
        assert e.value.code == -4
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        with pytest.raises(PoppyCudaError) as e:
            r.render([0.5], [0.5], cat, offs)
        assert e.value.code == -3                                    # capacity
        with pytest.raises(PoppyCudaError) as e:
            r.render([0.5] * 3, [0.5] * 3, np.zeros((0, 3), np.int32), [0, 0, 0, 0])
        assert e.value.code == -3                                    # more frames than the ring holds
    with MorphRenderer(w, h, 3, 32, 64, 1) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        bad = cat.copy()
        bad[0, 0] = 10_000
        with pytest.raises(PoppyCudaError) as e:
            r.render([0.5], [0.5], bad, offs)
        assert e.value.code == -2                                    # vertex index out of range
        with pytest.raises(PoppyCudaError):
            r.set_points(np.zeros((100, 2), np.float32), np.zeros((100, 2), np.float32))   # > max_points
    with pytest.raises(PoppyCudaError):
        MorphRenderer(40000, 10, 3, 32, 64, 1)                       # cv::remap size limit


def test_render_range_streams_slices_through_the_ring(native_lib):
    """poppy_cuda_render_range: a sequence rendered slice by slice into consecutive ring slots, with the download of
    each slice overlapping the next render (copy stream), equals the one-call render; re-rendering slots whose download
    is still pending waits for it."""
    from poppy_b200.renderer import MorphRenderer
    w, h, levels, F = 320, 200, 5, 12
    inp = synth.make_inputs(w, h, 90, 6.0, seed=21)
    phases = np.linspace(0.0, 1.0, F).astype(np.float32)
    masks = phases.astype(np.float64)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    with MorphRenderer(w, h, levels, len(inp.pts1), plan.max_triangles, F, chunk_frames=2) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        r.render(phases, masks, plan.tri_idx, plan.tri_offsets)
        want = r.download(0, F)
        want_pts = [r.morphed_points(k) for k in range(F)]
        got = np.zeros_like(want)
        for a in range(0, F, 5):                                   # ragged slices: 5, 5, 2
            b = min(a + 5, F)
            p = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases[a:b])
            r.render(phases[a:b], masks[a:b], p.tri_idx, p.tri_offsets, first_slot=a)
            r.download_async(a, b - a, got[a:].ctypes.data, w * 3, w * h * 3)
        r.sync()
        assert bits_differ(got, want) == 0
        for k in range(F):
            assert bits_differ(r.morphed_points(k), want_pts[k]) == 0
        # overwrite slots 0..4 with other phases while their download is pending, then read them back
        r.download_async(0, 5, got.ctypes.data, w * 3, w * h * 3)
        p = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases[5:10])
        r.render(phases[5:10], masks[5:10], p.tri_idx, p.tri_offsets, first_slot=0)
        r.sync()
        assert bits_differ(got[:5], want[:5]) == 0                 # the pending download saw the old frames
        assert bits_differ(r.download(0, 5), want[5:10]) == 0
        with pytest.raises(Exception):
            r.render(phases[:5], masks[:5], plan.tri_idx[:plan.tri_offsets[5]], plan.tri_offsets[:6], first_slot=F - 2)


# ---- the C++ shim (poppy::morph_images / poppy::morph_sequence) through its C entry points --------------------------
_WRITE = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_size_t)


def test_cpp_shim_morph_images_matches_reference(native_lib):
    ref = _ref()
    w, h, levels = 230, 170, 7
    inp = synth.block_inputs(w, h, 50, seed=61)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    dst = np.zeros((h, w, 3), np.uint8)
    mp = np.zeros((len(inp.pts1), 2), np.float32)
    try:
        rc = native_lib.poppy_shim_morph_images(w, h, levels, p(inp.bgr1), w * 3, p(inp.bgr2), w * 3, p(inp.gabor2), w * 12, p(inp.pts1),
                                                p(inp.pts2), len(inp.pts1), 0.3, 0.7, p(dst), w * 3, p(mp))
        assert rc == 0, native_lib.poppy_host_last_error()
    finally:
        native_lib.poppy_shim_release()
    want, want_pts = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, 0.3, 0.7, levels)
    assert bits_differ(dst, want) == 0 and bits_differ(mp, want_pts) == 0


def test_cpp_shim_morph_sequence_writes_the_golden_chain_in_order(native_lib):
    """poppy::morph_sequence: the chain rendered slice by slice (frame j-1 resident across the calls) with every slice handed
    to the writer ring; the frames reach `write` in order and equal the reference frame loop's."""
    g = np.load(os.path.join(GOLDEN, "chain_shapes_80x64_N12_L64.npz"))
    bgr1, bgr2, gab = (np.ascontiguousarray(g[k]) for k in ("bgr1", "bgr2", "gabor2"))
    pts1, pts2 = np.ascontiguousarray(g["pts1"], np.float32), np.ascontiguousarray(g["pts2"], np.float32)
    h, w = bgr1.shape[:2]
    N = int(g["n_frames"])
    got = []

    def write(user, idx, bgr, fw, fh, step):
        got.append((idx, np.ctypeslib.as_array(bgr, shape=(fh * step,)).reshape(fh, step)[:, :fw * 3].reshape(fh, fw, 3).copy()))

    p = lambda a: a.ctypes.data_as(C.c_void_p)
    cb = _WRITE(write)
    try:
        rc = native_lib.poppy_shim_morph_sequence(w, h, int(g["levels"]), p(bgr1), w * 3, p(bgr2), w * 3, p(gab), w * 12, p(pts1), p(pts2),
                                                  len(pts1), N, cb, None)
        assert rc == 0, native_lib.poppy_host_last_error()
    finally:
        native_lib.poppy_shim_release()
    assert [i for i, _ in got] == list(range(N))
    for j, (_, f) in enumerate(got):
        assert bits_differ(f, g["frames"][j]) == 0, f"chain frame {j}"


@pytest.mark.parametrize("n", [2, 0])
def test_fewer_than_three_points_render_like_the_reference(n):
    """No triangle can be formed: the reference blends the unwarped pair (an empty Delaunay mesh); so does the renderer."""
    ref = _ref()
    w, h, levels = 96, 72, 5
    inp = synth.make_inputs(w, h, 10, 4.0, seed=71)
    p1, p2 = inp.pts1[:n].copy(), inp.pts2[:n].copy()
    api.Settings.instance().pyramid_levels = levels
    dst, mp = api.morph_images(inp.bgr1, inp.bgr2, inp.bgr1, inp.bgr2, inp.gabor2, p1, p2, 0.4, 0.4)
    want, want_pts = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, p1, p2, 0.4, 0.4, levels)
    assert bits_differ(dst, want) == 0 and mp.shape == want_pts.shape and (n == 0 or bits_differ(mp, want_pts) == 0)


def test_sliced_chain_continues_across_render_calls(native_lib):
    """A chain rendered in slices (chain = 1, first_slot > 0 continues the previous call) equals the one-call chain."""
    from poppy_b200.renderer import MorphRenderer
    g = np.load(os.path.join(GOLDEN, "chain_shapes_80x64_N12_L64.npz"))
    h, w = g["bgr1"].shape[:2]
    N = int(g["n_frames"])
    ratio = np.array([host.chain_ratio(j, N) for j in range(N)], np.float64)
    plan = host.SequencePlan(g["pts1"], g["pts2"], w, h, ratio.astype(np.float32), chain=True)
    offs = plan.tri_offsets
    with MorphRenderer(w, h, int(g["levels"]), len(g["pts1"]), plan.max_triangles, N) as r:
        r.set_pair(np.ascontiguousarray(g["bgr1"]), np.ascontiguousarray(g["bgr2"]), np.ascontiguousarray(g["gabor2"]))
        r.set_points(g["pts1"], g["pts2"])
        for a in range(0, N, 5):
            b = min(a + 5, N)
            r.render(ratio[a:b].astype(np.float32), ratio[a:b], plan.tri_idx[offs[a]:offs[b]], offs[a:b + 1] - offs[a], chain=True,
                     first_slot=a)
        frames = r.download(0, N)
        with pytest.raises(Exception):          # a chain cannot continue anywhere but after its last frame
            r.render(ratio[:2].astype(np.float32), ratio[:2], plan.tri_idx[offs[0]:offs[2]], offs[0:3] - offs[0], chain=True, first_slot=3)
    plan.close()
    for j in range(N):
        assert bits_differ(frames[j], g["frames"][j]) == 0, f"chain frame {j}"


def test_two_contexts_on_two_devices_in_one_process(native_lib):
    """The > 48 KB dynamic shared memory opt-in is per device (ADVICE round 1): a context on device 1 after one on device 0
    must render the same frame. Skipped on a single-GPU box."""
    import ctypes as C
    n = C.c_int(0)
    try:
        C.CDLL("libcudart.so").cudaGetDeviceCount(C.byref(n))
    except OSError:
        import torch
        n.value = torch.cuda.device_count()
    if n.value < 2:
        pytest.skip("needs two GPUs")
    from poppy_b200 import api, synth
    inp = synth.block_inputs(320, 200, 60, seed=21)
    frames = []
    for dev in (0, 1, 0):
        s = api.Settings.instance()
        s.cuda_device, s.pyramid_levels = dev, 5
        dst, _ = api.morph_images(inp.bgr1, inp.bgr2, inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, 0.35, 0.6)
        frames.append(dst)
        api.release()
        assert (api.blur_margin(inp.bgr1[:150, :300], (320, 200)) == api.blur_margin(inp.bgr1[:150, :300], (320, 200))).all()
    api.Settings.instance().cuda_device = 0
    assert (frames[0] == frames[1]).all() and (frames[0] == frames[2]).all()


def test_resident_plan_renders_the_same_frames(native_lib):
    """poppy_cuda_set_plan + render_planned (triangle lists validated and uploaded once) against render with host lists,
    whole and in slices with a plan offset; a bad index is rejected at set_plan."""
    from poppy_b200.renderer import MorphRenderer
    w, h, L = 256, 160, 5
    inp = synth.make_inputs(w, h, 120, 5.0, seed=77)
    phases = np.linspace(0.05, 0.95, 11).astype(np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    with MorphRenderer(w, h, L, len(inp.pts1), plan.max_triangles, len(phases), chunk_frames=3) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
        want = [r.checksum(k, 1) for k in range(len(phases))]
        r.set_plan(plan.tri_idx, plan.tri_offsets)
        r.render_planned(phases, phases.astype(np.float64))
        assert [r.checksum(k, 1) for k in range(len(phases))] == want
        r.render_planned(phases[4:9], phases[4:9].astype(np.float64), plan_first=4, first_slot=2)      # a slice into other slots
        assert [r.checksum(2 + k, 1) for k in range(5)] == want[4:9]
        with pytest.raises(RuntimeError):
            r.render_planned(phases, phases.astype(np.float64), plan_first=3)                           # runs past the plan
        bad = plan.tri_idx.copy()
        bad[5, 1] = len(inp.pts1)
        with pytest.raises(RuntimeError):
            r.set_plan(bad, plan.tri_offsets)
