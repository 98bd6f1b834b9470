"""Rendered frames downloaded as I420 (YUV 4:2:0), converted on the GPU: poppy_cuda_download_i420, the I420 writer ring,
MorphRenderer.download_i420 and pixel_format="i420" of api.morph_sequence / render_phases / morph_segments.

The contract is cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420) byte for byte. oracle/yuv.py restates it; the CPU tests pin the
restatement to cv2 (a stored fixture, and cv2 itself where it imports), and the GPU tests hold every I420 frame to the
restatement of the same slot's BGR download."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from oracle import yuv
from tests.util import any_size_inputs

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "output", "i420.npz")
_WRITE = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_size_t)
INVALID = -2


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


# ---- CPU: the restatement -------------------------------------------------------------------------------------------
def test_restatement_equals_the_cv2_fixture():
    g = np.load(GOLDEN)
    for i in range(int(g["n"])):
        bgr, want = g[f"bgr{i}"], g[f"i420_{i}"]
        got = yuv.restate(bgr)
        assert got.shape == want.shape == (bgr.shape[0] * 3 // 2, bgr.shape[1]) and got.dtype == np.uint8
        assert (got == want).all(), f"case {i} {bgr.shape}"


def test_restatement_equals_cv2_on_seeded_sizes():
    cv2 = _cv2()
    if cv2 is None:
        pytest.skip("cv2 not importable")
    rng = np.random.default_rng(7)
    for _ in range(40):
        h, w = 2 * int(rng.integers(1, 60)), 2 * int(rng.integers(1, 60))
        bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        assert (yuv.restate(bgr) == cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)).all(), (w, h)
    stack = rng.integers(0, 256, (3, 6, 10, 3), dtype=np.uint8)
    assert (yuv.restate(stack) == np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in stack])).all()


@pytest.mark.parametrize("h,w", [(3, 4), (4, 3), (1, 2), (2, 1)])
def test_restatement_rejects_odd_sizes(h, w):
    with pytest.raises(ValueError):
        yuv.restate(np.zeros((h, w, 3), np.uint8))


# ---- CPU: argument checks that need no GPU ---------------------------------------------------------------------------
def test_c_abi_rejects_missing_context_and_ticket(native_lib):
    buf = np.zeros(64, np.uint8)
    t = C.c_uint64(0)
    p = buf.ctypes.data_as(C.c_void_p)
    assert native_lib.poppy_cuda_download_i420(None, 0, 1, p, 6) == INVALID
    assert native_lib.poppy_cuda_download_i420_async(None, 0, 1, p, 6, C.byref(t)) == INVALID
    out = C.c_void_p()
    assert native_lib.poppy_host_writer_create_i420(C.byref(out), None, 4, _WRITE(lambda *a: None), None, 0, None) == INVALID
    assert not out.value


def _inputs(w, h):
    bgr1, bgr2, _, p1, p2 = any_size_inputs(w, h)
    return bgr1, bgr2, p1, p2


@pytest.mark.parametrize("w,h", [(33, 18), (34, 17), (1, 1)])
def test_api_rejects_i420_at_odd_sizes_before_rendering(native_lib, w, h):
    from poppy_b200 import api
    bgr1, bgr2, p1, p2 = _inputs(w, h)
    with pytest.raises(ValueError, match="even frame size"):
        api.morph_sequence(bgr1, bgr2, None, p1, p2, number_of_frames=3, pixel_format="i420")
    with pytest.raises(ValueError, match="even frame size"):
        api.render_phases(bgr1, bgr2, None, p1, p2, [0.5], pixel_format="i420")
    with pytest.raises(ValueError, match="even frame size"):
        api.morph_segments([(bgr1, bgr2, None, p1, p2)], number_of_frames=3, pixel_format="i420")
    with pytest.raises(ValueError, match="even frame size"):
        api.morph_segments([(bgr1, bgr2, None, p1, p2)] * 2, number_of_frames=3, devices=[0, 1], pixel_format="i420")


@pytest.mark.parametrize("fmt", ["yuv420p", "I420", "nv12", None, "rgb"])
def test_api_rejects_unknown_pixel_formats_before_rendering(native_lib, fmt):
    from poppy_b200 import api
    bgr1, bgr2, p1, p2 = _inputs(34, 18)
    with pytest.raises(ValueError, match="pixel_format"):
        api.morph_sequence(bgr1, bgr2, None, p1, p2, number_of_frames=3, pixel_format=fmt)
    with pytest.raises(ValueError, match="pixel_format"):
        api.render_phases(bgr1, bgr2, None, p1, p2, [0.5], pixel_format=fmt)
    with pytest.raises(ValueError, match="pixel_format"):
        api.morph_segments([(bgr1, bgr2, None, p1, p2)], number_of_frames=3, pixel_format=fmt)
    with pytest.raises(ValueError, match="pixel_format"):
        api.morph_segments([(bgr1, bgr2, None, p1, p2)] * 2, number_of_frames=3, devices=[0, 1], pixel_format=fmt)


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _renderer(w, h, ring, seed=0):
    """A renderer with a ring of `ring` slots, every slot rendered from seeded content."""
    from poppy_b200.renderer import MorphRenderer
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=seed)
    r = MorphRenderer(w, h, 6, len(p1), 2 * len(p1) + 16, ring)
    r.set_pair(bgr1, bgr2, gab)
    r.set_points(p1, p2)
    r.render(*_plan(r, p1, p2, ring))
    return r, (p1, p2)


def _plan(r, p1, p2, n, phases=None):
    """Direct-mode render of n phases: (shape ratios, mask ratios, triangle lists, offsets)."""
    from poppy_b200 import host
    phases = np.linspace(0.05, 0.95, n, dtype=np.float32) if phases is None else np.asarray(phases, np.float32)
    plan = host.SequencePlan(p1, p2, r.width, r.height, phases)
    try:
        return phases, phases[::-1].astype(np.float64), plan.tri_idx, plan.tri_offsets
    finally:
        plan.close()


def _check(got, bgr, what=""):
    """got == restatement of bgr, and == cv2 where it imports; a stack of frames."""
    want = yuv.restate(bgr)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert (got == want).all(), (what, int((got != want).sum()))
    cv2 = _cv2()
    if cv2 is not None:
        for k in range(min(len(bgr), 2)):
            assert (got[k] == cv2.cvtColor(bgr[k], cv2.COLOR_BGR2YUV_I420)).all(), (what, "cv2", k)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(2, 2), (2, 640), (480, 2), (34, 18), (18, 4), (1920, 1080), (3840, 2160)])
def test_download_i420_equals_the_restatement(native_lib, w, h):
    r, _ = _renderer(w, h, 3)
    with r:
        bgr = r.download(0, 3)
        assert len(np.unique(bgr)) > 16          # real content, not a blank ring
        got = r.download_i420(0, 3)
        _check(got, bgr, f"{w}x{h}")


@pytest.mark.gpu
def test_pieces_first_slot_and_launch_count(native_lib):
    """20 frames from slot 3 go through the 8-frame staging in 3 pieces: one conversion launch each."""
    r, _ = _renderer(640, 360, 24)
    with r:
        bgr = r.download(0, 24)
        before = r.launch_count()
        got = r.download_i420(3, 20)
        assert r.launch_count() - before == 3
        _check(got, bgr[3:23], "pieces")
        _check(r.download_i420(23, 1), bgr[23:], "last slot")


@pytest.mark.gpu
def test_slots_past_2gib(native_lib):
    """At 4K (24.9 MB a frame) slot 87 starts beyond 2^31 bytes of the ring."""
    w, h, ring = 3840, 2160, 90
    assert 87 * w * h * 3 > 2 ** 31
    r, _ = _renderer(w, h, ring, seed=3)
    with r:
        got = r.download_i420(84, 6)
        _check(got, r.download(84, 6), "slots 84-89")


@pytest.mark.gpu
def test_frame_stride_keeps_the_padding(native_lib):
    w, h, n, pad = 34, 18, 11, 37
    r, _ = _renderer(w, h, n)
    with r:
        bgr = r.download(0, n)
        fb = w * h * 3 // 2
        buf = np.full(n * (fb + pad), 0xA5, np.uint8)
        rc = native_lib.poppy_cuda_download_i420(r._ctx, 0, n, buf.ctypes.data_as(C.c_void_p), fb + pad)
        assert rc == 0
        r.sync()
        frames = buf.reshape(n, fb + pad)
        assert (frames[:, fb:] == 0xA5).all()
        _check(frames[:, :fb].reshape(n, h * 3 // 2, w), bgr, "strided")


@pytest.mark.gpu
def test_c_abi_argument_checks(native_lib):
    from poppy_b200.renderer import MorphRenderer
    from poppy_b200._lib import PoppyCudaError
    buf = np.zeros(1 << 16, np.uint8)
    p = buf.ctypes.data_as(C.c_void_p)
    with MorphRenderer(3, 4, 2, 8, 32, 2) as r:
        assert native_lib.poppy_cuda_download_i420(r._ctx, 0, 1, p, 64) == INVALID
        assert b"even" in native_lib.poppy_cuda_last_error(r._ctx)
        with pytest.raises(PoppyCudaError):
            r.download_i420(0, 1, out=np.zeros((1, 6, 3), np.uint8))
        out = C.c_void_p()
        assert native_lib.poppy_host_writer_create_i420(C.byref(out), r._ctx, 4, _WRITE(lambda *a: None), None, 0, None) == INVALID
    r, _ = _renderer(34, 18, 4)
    with r:
        fb = 34 * 18 * 3 // 2
        for first, count, dst, stride in [(0, 1, None, fb), (-1, 1, p, fb), (0, 0, p, fb), (3, 2, p, fb), (0, 1, p, fb - 1)]:
            assert native_lib.poppy_cuda_download_i420(r._ctx, first, count, dst, stride) == INVALID, (first, count, stride)
            assert native_lib.poppy_cuda_last_error(r._ctx)
        assert native_lib.poppy_cuda_download_i420(r._ctx, 0, 4, p, fb) == 0
        r.sync()


def _pinned(lib, nbytes):
    ptr = C.c_void_p()
    assert lib.poppy_cuda_alloc_pinned(nbytes, C.byref(ptr)) == 0
    return ptr, np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr.value))


@pytest.mark.gpu
def test_async_tickets_interleaved_with_bgr(native_lib):
    w, h, n = 640, 480, 12
    r, _ = _renderer(w, h, n, seed=5)
    with r:
        want = r.download(0, n)
        fb, bb = w * h * 3 // 2, w * h * 3
        (pb, bgr), (py, i420) = _pinned(native_lib, n * bb), _pinned(native_lib, n * fb)
        try:
            tickets = []
            for first in (0, 6):
                for kind in ("bgr", "i420", "bgr"):
                    t = C.c_uint64(0)
                    if kind == "bgr":
                        rc = native_lib.poppy_cuda_download_async(r._ctx, first, 6, C.c_void_p(pb.value + first * bb), w * 3, bb, C.byref(t))
                    else:
                        rc = native_lib.poppy_cuda_download_i420_async(r._ctx, first, 6, C.c_void_p(py.value + first * fb), fb, C.byref(t))
                    assert rc == 0
                    tickets.append(t.value)
            assert tickets == sorted(tickets) and len(set(tickets)) == len(tickets)
            for t in tickets:
                assert native_lib.poppy_cuda_download_wait(r._ctx, t) == 0
            assert (bgr.reshape(n, h, w, 3) == want).all()
            _check(i420.reshape(n, h * 3 // 2, w).copy(), want, "async")
        finally:
            native_lib.poppy_cuda_free_pinned(pb)
            native_lib.poppy_cuda_free_pinned(py)


@pytest.mark.gpu
def test_render_after_download_waits_for_the_conversion(native_lib):
    """An I420 download of slots, then at once a render into those slots: the download delivers the earlier frames."""
    w, h, n = 1920, 1080, 16
    r, (p1, p2) = _renderer(w, h, n, seed=7)
    with r:
        before = r.download(0, n)
        fb = w * h * 3 // 2
        ptr, buf = _pinned(native_lib, n * fb)
        later = _plan(r, p1, p2, n, phases=np.linspace(0.9, 0.1, n))
        try:
            assert native_lib.poppy_cuda_download_i420(r._ctx, 0, n, ptr, fb) == 0
            r.render(*later)
            r.sync()
            after = r.download(0, n)
            assert (after != before).any()
            _check(buf.reshape(n, h * 3 // 2, w).copy(), before, "pre-render frames")
        finally:
            native_lib.poppy_cuda_free_pinned(ptr)


@pytest.mark.gpu
@pytest.mark.parametrize("workers", [0, 3])
def test_i420_writer_ring(native_lib, workers):
    w, h, n = 322, 180, 20
    r, _ = _renderer(w, h, n, seed=9)
    with r:
        want = yuv.restate(r.download(0, n))
        got, converted, lock = [], [], threading.Lock()

        def write(user, idx, y, fw, fh, step):        # an exception here would not reach the test: record, check below
            got.append((idx, (fw, fh, step), np.ctypeslib.as_array(y, shape=(fh * 3 // 2 * fw,)).reshape(fh * 3 // 2, fw).copy()))

        def convert(user, idx, y, fw, fh, step):
            with lock:
                converted.append(idx)

        cw, cc = _WRITE(write), _WRITE(convert)
        wr = C.c_void_p()
        assert native_lib.poppy_host_writer_create_i420(C.byref(wr), r._ctx, 4, cw, cc if workers else None, workers, None) == 0
        try:
            assert native_lib.poppy_host_writer_submit(wr, 0, 12, 0) == 0
            assert native_lib.poppy_host_writer_submit(wr, 12, 8, 12) == 0
            assert native_lib.poppy_host_writer_flush(wr) == 0
        finally:
            native_lib.poppy_host_writer_destroy_cuda(wr)
        assert [i for i, _, _ in got] == list(range(n))
        assert all(geometry == (w, h, w) for _, geometry, _ in got)
        assert sorted(converted) == (list(range(n)) if workers else [])
        for i, _, f in got:
            assert (f == want[i]).all(), i


class _Writer:
    def __init__(self):
        self.frames = []

    def write(self, f):
        self.frames.append(np.array(f, copy=True))


def _segment(w, h, seed):
    """(corrected1, corrected2, None, pts1, pts2): gabor2 derived on the GPU."""
    bgr1, bgr2, _, p1, p2 = any_size_inputs(w, h, seed=seed)
    return bgr1, bgr2, None, p1, p2


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(160, 96), (34, 18)])
def test_api_i420_equals_the_restated_bgr(native_lib, w, h):
    from poppy_b200 import api
    bgr1, bgr2, _, p1, p2 = _segment(w, h, 11)
    try:
        wb, wy = _Writer(), _Writer()
        bgr = api.morph_sequence(bgr1, bgr2, None, p1, p2, writer=wb, number_of_frames=7)
        got = api.morph_sequence(bgr1, bgr2, None, p1, p2, writer=wy, number_of_frames=7, pixel_format="i420")
        assert bgr.shape == (7, h, w, 3) and got.shape == (7, h * 3 // 2, w)
        _check(got, bgr, "morph_sequence")
        assert len(wy.frames) == 7 and all((a == b).all() for a, b in zip(wy.frames, got))
        assert all((a == b).all() for a, b in zip(wb.frames, bgr))

        phases = [0.2, 0.5, 0.8, 0.35]
        bgr = api.render_phases(bgr1, bgr2, None, p1, p2, phases)
        _check(api.render_phases(bgr1, bgr2, None, p1, p2, phases, pixel_format="i420"), bgr, "render_phases")

        segs = [(bgr1, bgr2, None, p1, p2), (bgr2, bgr1, None, p2, p1), _segment(w, h, 12)]
        wb, wy = _Writer(), _Writer()
        bgr = api.morph_segments(segs, number_of_frames=5, writer=wb)
        got = api.morph_segments(segs, number_of_frames=5, writer=wy, pixel_format="i420")
        assert got.shape == (3, 5, h * 3 // 2, w)
        _check(got.reshape(-1, h * 3 // 2, w), bgr.reshape(-1, h, w, 3), "morph_segments")
        assert len(wy.frames) == 15 and all((a == b).all() for a, b in zip(wy.frames, got.reshape(-1, h * 3 // 2, w)))
        assert all((a == b).all() for a, b in zip(wb.frames, bgr.reshape(-1, h, w, 3)))
    finally:
        api.release()


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0], [0, 1]])
def test_api_i420_segments_on_devices(native_lib, devices):
    from poppy_b200 import api
    from poppy_b200.renderer import device_count
    if device_count() < len(devices):
        pytest.skip(f"needs {len(devices)} GPUs")
    w, h = 96, 64
    segs = [_segment(w, h, s) for s in range(3)]
    try:
        bgr = api.morph_segments(segs, number_of_frames=4)
        wy = _Writer()
        got = api.morph_segments(segs, number_of_frames=4, writer=wy, devices=devices, pixel_format="i420")
        assert got.shape == (3, 4, h * 3 // 2, w)
        _check(got.reshape(-1, h * 3 // 2, w), bgr.reshape(-1, h, w, 3), f"devices {devices}")
        assert len(wy.frames) == 12 and all((a == b).all() for a, b in zip(wy.frames, got.reshape(-1, h * 3 // 2, w)))
    finally:
        api.release()
