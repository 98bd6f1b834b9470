"""Segments of a multi-image sequence rendered together (poppy_cuda_render_segments, api.morph_segments).

The reference's run() (src/poppy.cpp:266-328) morphs each consecutive pair of an image list as one chain of number_of_frames
frames. The segments are independent, so the renderer puts step j of a group of them into one kernel batch. Every test
here holds a batched segment to the same segment rendered alone (or to the reference pipeline's recorded frames): batching
must not change a single byte or a single point."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.util import bits_differ, frame_checksum

HERE = os.path.dirname(os.path.abspath(__file__))
FULL = os.path.join(HERE, "golden", "full")
LEVELS = 64
_WRITE = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_size_t)


def _golden(config):
    return np.load(os.path.join(FULL, f"c{config}.npz"))


def _segments(K, config=1, seed=0):
    """K segments of the golden pair's size: the recorded segment itself, the reversed pair, one with only the 4 corners,
    one with n = 2 (no triangles), then pairs with seeded point jitter; explicit and derived gabor2 mixed."""
    g = _golden(config)
    c1, c2, g2 = g["corrected1"], g["corrected2"], g["gabor2"]
    p1, p2 = g["pts1"].astype(np.float32), g["pts2"].astype(np.float32)
    h, w = c1.shape[:2]
    corners = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float32)
    rng = np.random.default_rng(seed)
    out = []
    for i in range(K):
        kind = i % 6
        if kind == 0:
            out.append((c1, c2, g2, p1, p2))
        elif kind == 1:
            out.append((c2, c1, None, p2, p1))
        elif kind == 2:
            out.append((c1, c2, g2, corners, corners + np.float32([[6, 4], [-5, 7], [3, -6], [-4, -3]])))
        elif kind == 3:
            out.append((c2, c1, None, p2[:2], p1[:2]))
        else:
            j1 = (p1 + rng.normal(0, 2.0, p1.shape)).astype(np.float32)
            j2 = (p2 + rng.normal(0, 2.0, p2.shape)).astype(np.float32)
            out.append((c1, c2, g2 if kind == 4 else None, j1, j2))
    return out


def _alone(seg, n_frames):
    """One segment through api.morph_sequence: its frames and every step's morphed points."""
    from poppy_b200 import api
    c1, c2, g2, p1, p2 = seg
    frames = api.morph_sequence(c1, c2, g2, p1, p2, number_of_frames=n_frames)
    r = next(iter(api._cache.values()))
    pts = [r.morphed_points(j) for j in range(n_frames)]
    return frames, pts


def _renderer(segs, n_frames, window=None, ring=None, chunk=None, unsharp_mode=None):
    from poppy_b200.renderer import MorphRenderer
    h, w = segs[0][0].shape[:2]
    n_max = max(len(s[3]) for s in segs)
    K, W = len(segs), window or n_frames
    r = MorphRenderer(w, h, LEVELS, max(n_max, 4), 2 * n_max + 16, ring or K * W, chunk_frames=chunk)
    if unsharp_mode is not None:
        r.set_unsharp_mode(unsharp_mode)
    r.set_segments(K, W)
    for s, (c1, c2, g2, p1, p2) in enumerate(segs):
        r.set_segment(s, c1, c2, g2, p1, p2)
    return r


def _plans(segs, n_frames):
    from poppy_b200 import host
    h, w = segs[0][0].shape[:2]
    ratio = np.array([host.chain_ratio(j, n_frames) for j in range(n_frames)], np.float64)
    plans = [host.SequencePlan(p1, p2, w, h, ratio.astype(np.float32), chain=True) for _, _, _, p1, p2 in segs]
    return ratio, plans


def _render_batched(segs, n_frames, slice_steps=None, window=None, **kw):
    """All segments batched: frames (K, N, H, W, 3) and points [s][j]; with slice_steps, slices of that many steps with a
    download after each."""
    from poppy_b200 import api
    K = len(segs)
    h, w = segs[0][0].shape[:2]
    ratio, plans = _plans(segs, n_frames)
    r = _renderer(segs, n_frames, window=window, **kw)
    frames = np.empty((K, n_frames, h, w, 3), np.uint8)
    pts = [[None] * n_frames for _ in range(K)]
    step = slice_steps or n_frames
    try:
        for a in range(0, n_frames, step):
            b = min(n_frames, a + step)
            sub = [_SlicedPlan(p, a, b) for p in plans]
            tri, offs = api.interleave_segment_plans(sub, b - a)
            r.render_segments(a, ratio[a:b].astype(np.float32), ratio[a:b], tri, offs)
            for s in range(K):
                for j in range(a, b):
                    frames[s, j] = r.download(r.segment_slot(s, j), 1)[0]
                    pts[s][j] = r.segment_points(s, j)
        return frames, pts, r
    finally:
        for p in plans:
            p.close()


class _SlicedPlan:
    """Steps [a, b) of a plan, as interleave_segment_plans takes them."""

    def __init__(self, plan, a, b):
        self.plan, self.a = plan, a
        self.tri_offsets = plan.tri_offsets[a:b + 1]

    def triangles(self, j):
        return self.plan.triangles(self.a + j)


@pytest.fixture
def levels64():
    from poppy_b200 import api
    old = api.Settings.instance().pyramid_levels
    api.Settings.instance().pyramid_levels = LEVELS
    yield
    api.Settings.instance().pyramid_levels = old
    api.release()


# ---- 1. equal to one segment at a time ---------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 3, 7])
def test_batched_segments_equal_each_segment_rendered_alone(native_lib, levels64, K):
    N = 60
    segs = _segments(K, seed=K)
    frames, pts, r = _render_batched(segs, N)
    r.close()
    for s, seg in enumerate(segs):
        want, want_pts = _alone(seg, N)
        bad = [j for j in range(N) if bits_differ(frames[s, j], want[j])]
        assert not bad, f"K={K} segment {s}: frames {bad[:8]} differ from the segment rendered alone"
        for j in range(N):
            assert pts[s][j].shape == want_pts[j].shape and pts[s][j].tobytes() == want_pts[j].tobytes(), (K, s, j)


# ---- 2. equal to the reference pipeline ---------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("config", [1, 2])
def test_golden_segment_inside_a_batch_reproduces_the_reference(native_lib, levels64, config):
    from poppy_b200 import api
    g = _golden(config)
    segs = _segments(5, config=config, seed=10 + config)
    segs = segs[1:3] + [segs[0]] + segs[3:]          # the recorded segment in the middle of the batch
    got = api.morph_segments(segs, number_of_frames=int(g["n_frames"]))
    assert got.shape == (5, int(g["n_frames"])) + g["corrected1"].shape
    frames = got[2]
    bad = [j for j in range(len(g["hashes"])) if frame_checksum(frames[j]) != int(g["hashes"][j])]
    assert not bad, f"config {config}: frames {bad[:8]} differ from the reference pipeline"
    for j, want in zip(g["kept"], g["kept_frames"]):
        assert bits_differ(frames[j], want) == 0, (config, int(j))


# ---- 3. grouping and lanes ----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_groups_on_several_lanes_equal_one_group_and_chunk_one(native_lib):
    N, K = 8, 10
    segs = _segments(K, seed=3)
    ref, ref_pts, r = _render_batched(segs, N)                 # default chunk: one group of 10
    r.close()
    for chunk in (4, 1):                                       # 3 groups on 3 lanes; 10 groups round-robin over 4 lanes
        got, got_pts, r = _render_batched(segs, N, chunk=chunk)
        r.close()
        assert bits_differ(got, ref) == 0, chunk
        assert all(got_pts[s][j].tobytes() == ref_pts[s][j].tobytes() for s in range(K) for j in range(N)), chunk


# ---- 4. sliced rendering ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_slices_through_a_small_window_equal_one_call(native_lib):
    N, K = 20, 4
    segs = _segments(K, seed=4)
    ref, ref_pts, r = _render_batched(segs, N)
    r.close()
    got, got_pts, r = _render_batched(segs, N, slice_steps=4, window=8)
    r.close()
    assert bits_differ(got, ref) == 0
    assert all(got_pts[s][j].tobytes() == ref_pts[s][j].tobytes() for s in range(K) for j in range(N))


# ---- 5. unsharp routes --------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_unsharp_routes_give_identical_batched_frames(native_lib):
    N, K = 12, 6
    segs = _segments(K, seed=5)
    outs = []
    for mode in (0, 1, 2):
        got, _, r = _render_batched(segs, N, unsharp_mode=mode)
        r.close()
        outs.append(got)
    assert bits_differ(outs[0], outs[1]) == 0
    assert bits_differ(outs[0], outs[2]) == 0


# ---- 6. launches per step do not grow with K ---------------------------------------------------------------------------

@pytest.mark.gpu
def test_launches_per_step_do_not_grow_with_the_number_of_segments(native_lib):
    from poppy_b200 import api
    N = 6
    per_step = {}
    for K in (1, 8):
        segs = _segments(K, seed=6)
        ratio, plans = _plans(segs, N)
        tri, offs = api.interleave_segment_plans(plans, N)
        r = _renderer(segs, N, unsharp_mode=1)
        before = r.launch_count()
        r.render_segments(0, ratio.astype(np.float32), ratio, tri, offs)
        r.sync()
        per_step[K] = (r.launch_count() - before) / N
        r.close()
        for p in plans:
            p.close()
    assert per_step[8] == per_step[1], per_step


# ---- 7. errors and coexistence ------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_segment_errors_return_the_documented_status(native_lib):
    from poppy_b200 import api
    from poppy_b200._lib import PoppyCudaError
    from poppy_b200.renderer import MorphRenderer
    INVALID, CAPACITY, STATE = -2, -3, -4
    N = 4
    segs = _segments(2, seed=7)
    ratio, plans = _plans(segs, N)
    tri, offs = api.interleave_segment_plans(plans, N)
    c1, c2, g2, p1, p2 = segs[0]
    h, w = c1.shape[:2]

    def code(fn, *a):
        with pytest.raises(PoppyCudaError) as e:
            fn(*a)
        return e.value.code

    with MorphRenderer(w, h, LEVELS, 256, 2 * 256 + 16, 8) as r:
        shape32, offs32 = ratio.astype(np.float32), offs.astype(np.int32)
        rc = native_lib.poppy_cuda_render_segments(r._ctx, 0, N, shape32.ctypes.data, ratio.ctypes.data, tri.ctypes.data,
                                                   offs32.ctypes.data)
        assert rc == STATE                                                                       # no set_segments
        assert code(r.set_segments, 2, 1) == INVALID                                             # W < 2
        assert code(r.set_segments, 3, 3) == CAPACITY                                            # K * W > ring
        r.set_segments(2, N)
        assert code(r.set_segment, 2, c1, c2, g2, p1, p2) == INVALID                             # bad s
        assert code(r.set_segment, -1, c1, c2, g2, p1, p2) == INVALID
        with pytest.raises(ValueError):
            r.set_segment(0, c1[:, :-1], c2, g2, p1, p2)                                         # wrong image size
        rc = native_lib.poppy_cuda_set_segment(r._ctx, 0, c1.ctypes.data, w * 3 - 1, c2.ctypes.data, w * 3, None, 0,
                                               p1.ctypes.data, p2.ctypes.data, len(p1))
        assert rc == INVALID                                                                     # rows shorter than the frame
        r.set_segment(0, c1, c2, g2, p1, p2)
        assert code(r.render_segments, 0, ratio.astype(np.float32), ratio, tri, offs) == STATE     # segment 1 not set
        r.set_segment(1, *segs[1])
        bad = tri.copy()
        bad[offs[1]] = len(segs[1][3])                 # segment 1's list of step 0 names a point it does not have
        assert code(r.render_segments, 0, ratio.astype(np.float32), ratio, bad, offs) == INVALID
        r.render_segments(0, ratio[:2].astype(np.float32), ratio[:2], tri[:offs[4]], offs[:5])
        sub_off = offs[4:] - offs[4]
        assert code(r.render_segments, 3, ratio[3:].astype(np.float32), ratio[3:], tri[offs[6]:], offs[6:] - offs[6]) == STATE
        r.render_segments(2, ratio[2:].astype(np.float32), ratio[2:], tri[offs[4]:], sub_off)
        assert code(r.segment_points, 0, N) == INVALID
    for p in plans:
        p.close()
    with MorphRenderer(w, h, LEVELS, 256, 528, 8, keep_stages=True) as r:
        r.set_segments(1, 2)
        r.set_segment(0, c1, c2, g2, p1, p2)
        assert code(r.render_segments, 0, [0.0], [0.0], np.zeros((0, 3), np.int32), [0, 0]) == STATE


@pytest.mark.gpu
def test_pair_render_after_segments_still_matches_morph_sequence(native_lib, levels64):
    from poppy_b200 import host
    N = 10
    segs = _segments(3, seed=8)
    batched, _, r = _render_batched(segs, N)
    c1, c2, g2, p1, p2 = segs[1]
    h, w = c1.shape[:2]
    ratio = np.array([host.chain_ratio(j, N) for j in range(N)], np.float64)
    plan = host.SequencePlan(p1, p2, w, h, ratio.astype(np.float32), chain=True)
    r.set_pair(c1, c2, g2)
    r.set_points(p1, p2)
    r.render(ratio.astype(np.float32), ratio, plan.tri_idx, plan.tri_offsets, chain=True)
    got = r.download(0, N)
    plan.close()
    r.close()
    want, _ = _alone(segs[1], N)
    assert bits_differ(got, want) == 0
    assert bits_differ(batched[1], want) == 0


# ---- 8. the C shim ------------------------------------------------------------------------------------------------------

class _Seg(C.Structure):
    _fields_ = [("corrected1", C.c_void_p), ("step1", C.c_size_t), ("corrected2", C.c_void_p), ("step2", C.c_size_t),
                ("gabor2", C.c_void_p), ("gstep", C.c_size_t), ("pts1_xy", C.c_void_p), ("pts2_xy", C.c_void_p), ("n", C.c_int)]


@pytest.mark.gpu
def test_shim_morph_segments_delivers_the_reference_order(native_lib):
    N, K = 12, 3
    segs = [tuple(np.ascontiguousarray(a) if a is not None else None for a in s) for s in _segments(K, seed=9)]
    h, w = segs[0][0].shape[:2]
    p = lambda a: a.ctypes.data if a is not None else None

    def collect():
        got = []

        def write(user, idx, bgr, fw, fh, step):
            f = np.ctypeslib.as_array(bgr, shape=(fh * step,)).reshape(fh, step)[:, :fw * 3].reshape(fh, fw, 3)
            got.append((idx, f.copy()))
        return got, _WRITE(write)

    try:
        want = []
        for c1, c2, g2, p1, p2 in segs:
            got, cb = collect()
            rc = native_lib.poppy_shim_morph_sequence(w, h, LEVELS, p(c1), w * 3, p(c2), w * 3, p(g2), w * 12, p(p1), p(p2), len(p1),
                                                      N, cb, None)
            assert rc == 0, native_lib.poppy_host_last_error()
            want += [f for _, f in got]
        arr = (_Seg * K)(*[_Seg(p(c1), w * 3, p(c2), w * 3, p(g2), w * 12, p(p1), p(p2), len(p1)) for c1, c2, g2, p1, p2 in segs])
        got, cb = collect()
        rc = native_lib.poppy_shim_morph_segments(w, h, LEVELS, C.cast(arr, C.c_void_p), K, N, cb, None)
        assert rc == 0, native_lib.poppy_host_last_error()
    finally:
        native_lib.poppy_shim_release()
    assert [i for i, _ in got] == list(range(K * N))
    bad = [i for i, f in got if bits_differ(f, want[i])]
    assert not bad, f"frames {bad[:8]} of {K * N} differ from {K} calls of poppy_shim_morph_sequence"
