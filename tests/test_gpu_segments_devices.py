"""Segments of a multi-image sequence sharded over several GPUs of one box (api.morph_segments(devices=...),
poppy::morph_segments(..., devices), poppy_shim_morph_segments_devices).

Device devices[g] renders the contiguous segment range shard.phase_range(g, G, K), G = min(len(devices), K). Every test
on the GPU holds the sharded call to the same call on one device: the same frames, byte for byte, in the same order. The
GPU tests need two devices and skip on a one-GPU box."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from tests.util import bits_differ

HERE = os.path.dirname(os.path.abspath(__file__))
LEVELS = 64
INVALID, NO_DEVICE = -2, -1
_WRITE = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_size_t)


class _Seg(C.Structure):
    _fields_ = [("corrected1", C.c_void_p), ("step1", C.c_size_t), ("corrected2", C.c_void_p), ("step2", C.c_size_t),
                ("gabor2", C.c_void_p), ("gstep", C.c_size_t), ("pts1_xy", C.c_void_p), ("pts2_xy", C.c_void_p), ("n", C.c_int)]


def _segments(K, seed=0):
    """K segments of the golden 512 x 512 pair: the recorded segment, the reversed pair, the 4 corners only, n = 2, then
    seeded point jitter; explicit and derived gabor2 mixed."""
    g = np.load(os.path.join(HERE, "golden", "full", "c1.npz"))
    c1, c2, g2 = (np.ascontiguousarray(g[k]) for k in ("corrected1", "corrected2", "gabor2"))
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
            out.append((c2, c1, None, np.ascontiguousarray(p2[:2]), np.ascontiguousarray(p1[:2])))
        else:
            j1 = (p1 + rng.normal(0, 2.0, p1.shape)).astype(np.float32)
            j2 = (p2 + rng.normal(0, 2.0, p2.shape)).astype(np.float32)
            out.append((c1, c2, g2 if kind == 4 else None, j1, j2))
    return out


def _shim_segments(segs):
    h, w = segs[0][0].shape[:2]
    p = lambda a: a.ctypes.data if a is not None else None
    return (_Seg * len(segs))(*[_Seg(p(c1), w * 3, p(c2), w * 3, p(g2), w * 12, p(p1), p(p2), len(p1))
                                for c1, c2, g2, p1, p2 in segs])


def _shim_call(lib, segs, n_frames, devices, on_frame):
    """poppy_shim_morph_segments (devices=None) or poppy_shim_morph_segments_devices; on_frame(index, frame view)."""
    h, w = segs[0][0].shape[:2]

    def write(user, idx, bgr, fw, fh, step):
        on_frame(idx, np.ctypeslib.as_array(bgr, shape=(fh * step,)).reshape(fh, step)[:, :fw * 3].reshape(fh, fw, 3))
    cb = _WRITE(write)
    arr = _shim_segments(segs)
    if devices is None:
        rc = lib.poppy_shim_morph_segments(w, h, LEVELS, C.cast(arr, C.c_void_p), len(segs), n_frames, cb, None)
    else:
        dev = (C.c_int * len(devices))(*devices)
        rc = lib.poppy_shim_morph_segments_devices(dev, len(devices), w, h, LEVELS, C.cast(arr, C.c_void_p), len(segs), n_frames,
                                                   cb, None)
    assert rc == 0, lib.poppy_host_last_error()


def _gpus(lib):
    return lib.poppy_cuda_device_count()


@pytest.fixture
def two_gpus(native_lib):
    n = _gpus(native_lib)
    if n < 2:
        pytest.skip("needs two GPUs")
    return n


@pytest.fixture
def levels64():
    from poppy_b200 import api
    old = api.Settings.instance().pyramid_levels
    api.Settings.instance().pyramid_levels = LEVELS
    yield
    api.Settings.instance().pyramid_levels = old
    api.release()


# ---- CPU: the partition and the argument checks ------------------------------------------------------------------------

def test_partition_is_contiguous_ordered_disjoint_and_covering():
    from poppy_b200 import shard
    for K in range(1, 21):
        for G in range(1, 9):
            used = min(G, K)
            ranges = [shard.phase_range(g, used, K) for g in range(used)]
            assert ranges[0][0] == 0 and ranges[-1][1] == K, (K, G, ranges)
            assert all(lo < hi for lo, hi in ranges), (K, G, ranges)                  # no used device is idle
            assert all(ranges[g][1] == ranges[g + 1][0] for g in range(used - 1)), (K, G, ranges)
            assert sorted(s for lo, hi in ranges for s in range(lo, hi)) == list(range(K))
            assert max(hi - lo for lo, hi in ranges) - min(hi - lo for lo, hi in ranges) <= 1


@pytest.mark.parametrize("devices", [[], [0, 0], [1, 0, 1], [-1], [0, -2]])
def test_api_rejects_a_malformed_device_list(native_lib, devices):
    from poppy_b200 import api
    segs = [(np.zeros((8, 8, 3), np.uint8), np.zeros((8, 8, 3), np.uint8), None, np.zeros((4, 2), np.float32),
             np.zeros((4, 2), np.float32))]
    with pytest.raises(ValueError, match="device"):
        api.morph_segments(segs, number_of_frames=2, devices=devices)
    assert not api._device_cache


def test_api_without_a_gpu_raises_runtime_error(native_lib):
    if _gpus(native_lib) > 0:
        pytest.skip("a GPU is present")
    from poppy_b200 import api
    segs = [(np.zeros((8, 8, 3), np.uint8), np.zeros((8, 8, 3), np.uint8), None, np.zeros((4, 2), np.float32),
             np.zeros((4, 2), np.float32))]
    with pytest.raises(RuntimeError, match="no CUDA device"):
        api.morph_segments(segs, number_of_frames=2, devices=[0, 1])


def _tiny_shim_args():
    c = np.zeros((8, 8, 3), np.uint8)
    pts = np.zeros((4, 2), np.float32)
    arr = (_Seg * 1)(_Seg(c.ctypes.data, 24, c.ctypes.data, 24, None, 0, pts.ctypes.data, pts.ctypes.data, 4))
    return (c, pts, arr), _WRITE(lambda *a: None)


@pytest.mark.parametrize("devices", [[0, 0], [2, 1, 2], [-1], [1, -3]])
def test_shim_rejects_a_malformed_device_list(native_lib, devices):
    keep, cb = _tiny_shim_args()
    dev = (C.c_int * len(devices))(*devices)
    rc = native_lib.poppy_shim_morph_segments_devices(dev, len(devices), 8, 8, 4, C.cast(keep[2], C.c_void_p), 1, 2, cb, None)
    assert rc == INVALID
    assert b"device" in native_lib.poppy_host_last_error()


def test_shim_rejects_null_and_empty_arguments(native_lib):
    keep, cb = _tiny_shim_args()
    segs = C.cast(keep[2], C.c_void_p)
    dev = (C.c_int * 2)(0, 1)
    f = native_lib.poppy_shim_morph_segments_devices
    assert f(dev, 0, 8, 8, 4, segs, 1, 2, cb, None) == INVALID                   # n_devices < 1
    assert f(dev, -1, 8, 8, 4, segs, 1, 2, cb, None) == INVALID
    assert f(None, 2, 8, 8, 4, segs, 1, 2, cb, None) == INVALID                  # no list
    assert f(dev, 2, 8, 8, 4, None, 1, 2, cb, None) == INVALID                   # no segments
    assert f(dev, 2, 8, 8, 4, segs, 0, 2, cb, None) == INVALID
    assert f(dev, 2, 8, 8, 4, segs, 1, 2, None, None) == INVALID                 # no writer
    bad = (_Seg * 1)(_Seg(None, 24, None, 24, None, 0, None, None, 4))
    assert f(dev, 2, 8, 8, 4, C.cast(bad, C.c_void_p), 1, 2, cb, None) == INVALID


def test_shim_without_a_gpu_returns_no_device(native_lib):
    if _gpus(native_lib) > 0:
        pytest.skip("a GPU is present")
    keep, cb = _tiny_shim_args()
    dev = (C.c_int * 2)(0, 1)
    rc = native_lib.poppy_shim_morph_segments_devices(dev, 2, 8, 8, 4, C.cast(keep[2], C.c_void_p), 1, 2, cb, None)
    assert rc == NO_DEVICE
    assert b"no CUDA device" in native_lib.poppy_host_last_error()


# ---- GPU: an index past the device count --------------------------------------------------------------------------------

@pytest.mark.gpu
def test_an_index_past_the_device_count_is_invalid(native_lib):
    from poppy_b200 import api
    n = _gpus(native_lib)
    segs = _segments(2)
    with pytest.raises(ValueError, match="out of"):
        api.morph_segments(segs, number_of_frames=2, devices=[0, n])
    keep, cb = _tiny_shim_args()
    dev = (C.c_int * 2)(n, 0)
    rc = native_lib.poppy_shim_morph_segments_devices(dev, 2, 8, 8, 4, C.cast(keep[2], C.c_void_p), 1, 2, cb, None)
    assert rc == INVALID and b"not in" in native_lib.poppy_host_last_error()


# ---- GPU: the sharded call equals the single-device call ---------------------------------------------------------------

class _Writer:
    def __init__(self):
        self.frames = []

    def write(self, f):
        self.frames.append(f.copy())


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 2, 3, 7])
def test_two_devices_equal_one_device(two_gpus, levels64, K):
    from poppy_b200 import api
    N = 12
    segs = _segments(K, seed=K)
    want = api.morph_segments(segs, number_of_frames=N)
    wr = _Writer()
    got = api.morph_segments(segs, number_of_frames=N, writer=wr, devices=[0, 1])
    assert got.shape == want.shape == (K, N, 512, 512, 3)
    bad = [(s, j) for s in range(K) for j in range(N) if bits_differ(got[s, j], want[s, j])]
    assert not bad, f"K={K}: frames {bad[:8]} differ from the single-device call"
    assert len(wr.frames) == K * N
    assert all(bits_differ(wr.frames[s * N + j], got[s, j]) == 0 for s in range(K) for j in range(N))
    assert (1 in api._device_cache) == (K > 1)          # K = 1 leaves device 1 idle: no context there


@pytest.mark.gpu
def test_sixteen_segments_over_every_device(two_gpus, levels64):
    from poppy_b200 import api
    N = 8
    segs = _segments(16, seed=16)
    want = api.morph_segments(segs, number_of_frames=N)
    got = api.morph_segments(segs, number_of_frames=N, devices=list(range(two_gpus)))
    assert bits_differ(got, want) == 0
    assert sorted(api._device_cache) == list(range(1, min(two_gpus, 16)))


@pytest.mark.gpu
def test_output_order_is_the_segment_order_not_the_device_order(two_gpus, levels64):
    from poppy_b200 import api
    N, K = 10, 5
    segs = _segments(K, seed=21)
    want = api.morph_segments(segs, number_of_frames=N)
    wr = _Writer()
    got = api.morph_segments(segs, number_of_frames=N, writer=wr, devices=[1, 0])
    assert bits_differ(got, want) == 0
    assert all(bits_differ(wr.frames[s * N + j], want[s, j]) == 0 for s in range(K) for j in range(N))


@pytest.mark.gpu
def test_several_batches_per_device(two_gpus, levels64, monkeypatch):
    from poppy_b200 import api
    N, K = 10, 7
    segs = _segments(K, seed=22)
    want = api.morph_segments(segs, number_of_frames=N)
    monkeypatch.setattr(api, "_SEGMENT_RING_BYTES", 2 * N * 512 * 512 * 3)     # 2 segments per batch: 3 + 4 -> 2 batches each
    wr = _Writer()
    got = api.morph_segments(segs, number_of_frames=N, writer=wr, devices=[0, 1])
    assert bits_differ(got, want) == 0
    assert all(bits_differ(wr.frames[s * N + j], want[s, j]) == 0 for s in range(K) for j in range(N))
    assert api._device_cache[1].max_batch_frames == 2 * N


# ---- GPU: the C shim ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_shim_on_two_devices_equals_one_device(native_lib, two_gpus):
    N, K = 12, 5
    segs = _segments(K, seed=31)
    try:
        want, got = [], []
        _shim_call(native_lib, segs, N, None, lambda i, f: want.append((i, f.copy())))
        _shim_call(native_lib, segs, N, [0, 1], lambda i, f: got.append((i, f.copy())))
    finally:
        native_lib.poppy_shim_release()
    assert [i for i, _ in got] == list(range(K * N)) == [i for i, _ in want]
    bad = [i for (i, f), (_, g) in zip(got, want) if bits_differ(f, g)]
    assert not bad, f"frames {bad[:8]} of {K * N} differ from the single-device call"


def _inputs_4k():
    from poppy_b200 import synth
    a = synth.make_inputs(3840, 2160, 300, seed=41)
    rng = np.random.default_rng(41)
    segs = []
    for i in range(12):
        j1 = (a.pts1 + rng.normal(0, 3.0, a.pts1.shape)).astype(np.float32)
        j2 = (a.pts2 + rng.normal(0, 3.0, a.pts2.shape)).astype(np.float32)
        segs.append((a.bgr1, a.bgr2, None, j1, j2) if i % 2 == 0 else (a.bgr2, a.bgr1, None, j2, j1))
    return segs


@pytest.mark.gpu
def test_shim_4k_several_batches_per_device(native_lib, two_gpus):
    """3840 x 2160, N = 60, K = 12 on 2 devices: 6 segments each against the 5 that fit the 8 GB ring of one device."""
    N = 60
    segs = _inputs_4k()
    digests = {}
    try:
        for devices in (None, [0, 1]):
            d = []

            def on_frame(i, f):
                d.append((i, hashlib.sha1(np.ascontiguousarray(f)).hexdigest()))
            _shim_call(native_lib, segs, N, devices, on_frame)
            digests[str(devices)] = d
    finally:
        native_lib.poppy_shim_release()
    one, two = digests["None"], digests["[0, 1]"]
    assert [i for i, _ in two] == list(range(12 * N))
    bad = [i for (i, a), (_, b) in zip(two, one) if a != b]
    assert not bad, f"frames {bad[:8]} differ from the single-device call"


# ---- GPU: cached contexts ----------------------------------------------------------------------------------------------

def _free_bytes(device):
    import torch
    return torch.cuda.mem_get_info(device)[0]


@pytest.mark.gpu
def test_shim_reuses_its_contexts_and_release_frees_them(native_lib, two_gpus):
    N, K = 60, 4
    segs = _segments(K, seed=51)
    ring = 2 * N * 512 * 512 * 3                   # device 1's share: 2 segments of N frames
    seq = segs[0]
    h, w = seq[0].shape[:2]
    p = lambda a: a.ctypes.data if a is not None else None

    def sequence():
        frames = []
        cb = _WRITE(lambda u, i, bgr, fw, fh, step: frames.append(
            np.ctypeslib.as_array(bgr, shape=(fh * step,)).reshape(fh, step)[:, :fw * 3].copy()))
        c1, c2, g2, p1, p2 = seq
        rc = native_lib.poppy_shim_morph_sequence(w, h, LEVELS, p(c1), w * 3, p(c2), w * 3, p(g2), w * 12, p(p1), p(p2), len(p1),
                                                  N, cb, None)
        assert rc == 0, native_lib.poppy_host_last_error()
        return np.stack(frames)

    try:
        before_seq = sequence()
        native_lib.poppy_shim_release()
        free0 = _free_bytes(1)
        first = []
        _shim_call(native_lib, segs, N, [0, 1], lambda i, f: first.append(f.copy()))
        free1 = _free_bytes(1)
        again = []
        _shim_call(native_lib, segs, N, [0, 1], lambda i, f: again.append(f.copy()))
        free2 = _free_bytes(1)
        assert free0 - free1 >= ring, "no context on device 1"
        assert abs(free2 - free1) < ring // 2, "the second call did not reuse device 1's context"
        assert all(bits_differ(a, b) == 0 for a, b in zip(first, again))
        after_seq = sequence()                                     # device 0's context, after the sharded calls
        assert bits_differ(after_seq, before_seq) == 0
        native_lib.poppy_shim_release()
        assert _free_bytes(1) - free2 >= ring, "poppy_shim_release left device 1's context"
    finally:
        native_lib.poppy_shim_release()


@pytest.mark.gpu
def test_api_reuses_its_renderers_and_release_frees_them(two_gpus, levels64):
    from poppy_b200 import api
    N, K = 10, 4
    segs = _segments(K, seed=52)
    c1, c2, g2, p1, p2 = segs[0]
    before = api.morph_sequence(c1, c2, g2, p1, p2, number_of_frames=N)
    got = api.morph_segments(segs, number_of_frames=N, devices=[0, 1])
    r1 = api._device_cache[1]
    again = api.morph_segments(segs, number_of_frames=N, devices=[0, 1])
    assert api._device_cache[1] is r1 and bits_differ(got, again) == 0
    assert len(api._cache) == 1 and all(k[3] == 0 for k in api._cache)           # device 1 never enters _cache
    after = api.morph_sequence(c1, c2, g2, p1, p2, number_of_frames=N)
    assert bits_differ(after, before) == 0
    api.release()
    assert not api._cache and not api._device_cache and not r1._ctx
