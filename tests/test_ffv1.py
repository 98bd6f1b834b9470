"""Rendered frames as lossless FFV1 packets encoded on the GPU (poppy_cuda_download_ffv1, the FFV1 writer ring,
MorphRenderer.download_ffv1, pixel_format="ffv1") and the Matroska writer (poppy_host_mkv_*, api.MatroskaWriter).

oracle/ffv1.py restates the encoder and a decoder. The CPU tests pin the restatement to libavcodec: its range decoder reads
the configuration record and slice headers cv2 wrote (a stored fixture), and cv2 decodes the restated encoder's streams,
muxed by the C++ writer, to the exact frames. The GPU tests hold every packet to the restated encoder, byte for byte."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import ffv1
from tests.util import any_size_inputs

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "output", "ffv1")
INVALID = -2
_PACKET = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_size_t)


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


def _content(kind, w, h, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "flat":
        return np.full((h, w, 3), (17, 200, 93), np.uint8)
    if kind == "saturated":
        return (rng.integers(0, 2, (h, w, 3)) * 255).astype(np.uint8)
    if kind == "gradient":
        y, x = np.mgrid[0:h, 0:w]
        return np.stack([(x * 255 // max(w - 1, 1)), (y * 255 // max(h - 1, 1)), ((x + y) % 256)], -1).astype(np.uint8)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "morph":      # the renderer's own inputs: smooth photographic-like content
        return any_size_inputs(w, h, seed=seed, smooth=True)[0]
    raise ValueError(kind)


def _record(lib, w, h):
    buf, n = (C.c_uint8 * 256)(), C.c_size_t()
    assert lib.poppy_host_ffv1_config(w, h, buf, 256, C.byref(n)) == 0
    return bytes(buf[:n.value])


def _mux(lib, path, w, h, packets):
    m = C.c_void_p()
    assert lib.poppy_host_mkv_open(C.byref(m), os.fsencode(path), w, h, 30, 1) == 0
    for p in packets:
        assert lib.poppy_host_mkv_write(m, p, len(p)) == 0
    assert lib.poppy_host_mkv_close(m) == 0


def _play(path):
    cv2 = _cv2()
    cap = cv2.VideoCapture(path)
    out = []
    while True:
        ok, f = cap.read()
        if not ok:
            return out
        out.append(f)


# ---- CPU: the restatement against libavcodec -------------------------------------------------------------------------
def test_range_decoder_reads_libavcodec_record_and_slice_headers():
    mkv = ffv1.read_mkv(os.path.join(FIXTURE, "cv2_64x48.mkv"))
    assert mkv["codec_id"] == "V_FFV1" and (mkv["width"], mkv["height"]) == (64, 48)
    c = ffv1.parse_config(mkv["codec_private"])          # CRC checked inside
    assert (c["version"], c["micro_version"], c["coder_type"], c["colorspace_type"]) == (3, 4, 0, 1)
    assert (c["bits_per_raw_sample"], c["chroma_planes"], c["transparency"], c["ec"]) == (8, 1, 1, 1)
    # libavcodec's 8-bit default set is set 0 of its record: the tables this encoder writes
    assert len(c["quant_tables"]) == 2 and c["context_count"][0] == ffv1.CONTEXT_COUNT
    for k, scale in enumerate((1, 11, 121, 0, 0)):
        assert (c["quant_tables"][0][k] == scale * ffv1.QUANT11).all()
    nh, nv = c["num_h_slices"], c["num_v_slices"]
    assert len(mkv["packets"]) == 2
    for k, packet in enumerate(mkv["packets"]):
        slices = ffv1.split_slices(packet, trailer=8)
        assert len(slices) == nh * nv
        seen = set()
        for s, (start, size) in enumerate(slices):
            assert ffv1.crc32_msb(packet[start:start + size + 8]) == 0       # slice CRC (ec 1)
            rd = ffv1.RangeDecoder(packet[start:start + size])
            if s == 0:
                assert rd.bit([128], 0) == (k == 0)                          # keyframe: cv2's first frame only
            hdr, st = ffv1.read_slice_header(rd)
            assert [rd.symbol(st, False) for _ in range(3)] == [0, 0, 0]    # quant-table index of 3 context planes
            assert [rd.symbol(st, False) for _ in range(3)] == [3, 0, 1]    # progressive, aspect ratio 0:1
            seen.add((hdr["slice_x"], hdr["slice_y"]))
        assert seen == {(i, j) for i in range(nh) for j in range(nv)}


def test_state_tables_stay_in_8_to_248():
    """The capacity proof (DESIGN §9.1) needs every reachable state in [8, 248]."""
    reach, todo = set(), [128, 129]
    while todo:
        s = todo.pop()
        if s not in reach:
            reach.add(s)
            todo += [ffv1.ZERO_STATE[s], ffv1.ONE_STATE[s]]
    assert min(reach) == 8 and max(reach) == 248


def test_slice_grid():
    assert ffv1.slice_grid(1, 1) == (1, 1)
    assert ffv1.slice_grid(7, 5) == (1, 1)
    assert ffv1.slice_grid(640, 360) == (5, 4)
    assert ffv1.slice_grid(1920, 1080) == (15, 11)
    assert ffv1.slice_grid(3840, 2160) == (30, 23)
    assert ffv1.slice_grid(10000, 10000) == (32, 32)
    assert ffv1.slice_grid(3, 100000) == (1, 32)
    for w, h in [(640, 360), (1920, 1080), (3840, 2160)]:
        px = [(x1 - x0) * (y1 - y0) for x0, y0, x1, y1 in ffv1.slice_rects(w, h)]
        assert 8000 <= min(px) and max(px) <= 16384 and sum(px) == w * h


def test_largest_grid_cv2_decodes(native_lib, tmp_path):
    """1024 slices decode, 1056 do not: 32 x 32 is the grid's cap."""
    if _cv2() is None:
        pytest.skip("cv2 not importable")
    w = h = 70
    f = _content("morph", w, h, 3)

    def el(eid, payload):                    # an EBML element with an 8-byte size
        return eid + b"\x01" + len(payload).to_bytes(7, "big") + payload

    def u(v):
        return v.to_bytes(max(1, (v.bit_length() + 7) // 8), "big")

    def decodes(grid):
        # the C++ writer always stores the record of slice_grid(w, h): this file carries the probed grid's record instead
        track = el(b"\xd7", u(1)) + el(b"\x73\xc5", u(1)) + el(b"\x86", b"V_FFV1") + el(b"\x83", u(1)) + \
            el(b"\xe0", el(b"\xb0", u(w)) + el(b"\xba", u(h))) + el(b"\x63\xa2", ffv1.config_record(w, h, grid))
        block = el(b"\xa3", b"\x81\x00\x00\x80" + ffv1.encode_frame(f, grid))
        data = el(b"\x1a\x45\xdf\xa3", el(b"\x42\x82", b"matroska")) + el(b"\x18\x53\x80\x67", el(
            b"\x15\x49\xa9\x66", el(b"\x2a\xd7\xb1", u(1000000))) + el(b"\x16\x54\xae\x6b", el(b"\xae", track)) +
            el(b"\x1f\x43\xb6\x75", el(b"\xe7", u(0)) + block))
        path = str(tmp_path / f"g{grid[0]}x{grid[1]}.mkv")
        open(path, "wb").write(data)
        got = _play(path)
        return len(got) == 1 and (got[0] == f).all()

    assert decodes((32, 32)) and decodes((64, 16))
    assert not decodes((33, 32))


def test_host_record_equals_the_restatement(native_lib):
    for w, h in [(1, 1), (2, 3), (64, 48), (640, 360), (1920, 1080), (3840, 2160), (70000, 3)]:
        assert _record(native_lib, w, h) == ffv1.config_record(w, h), (w, h)
    n = C.c_size_t()
    assert native_lib.poppy_host_ffv1_config(64, 48, None, 0, C.byref(n)) == INVALID and n.value > 0
    assert native_lib.poppy_host_ffv1_config(0, 48, None, 0, C.byref(n)) == INVALID


@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (7, 5), (64, 48), (200, 100), (640, 360)])
def test_restated_stream_plays_back_in_cv2(native_lib, tmp_path, w, h):
    kinds = ["flat", "saturated", "gradient", "noise", "morph"]
    frames = [_content(k, w, h, i) for i, k in enumerate(kinds)]
    packets = [ffv1.encode_frame(f) for f in frames]
    rec = _record(native_lib, w, h)
    if w * h <= 20000:                       # the restated decoder is slow; cv2 decodes every size below
        for f, p in zip(frames, packets):
            assert (ffv1.decode_frame(p, w, h, ffv1.parse_config(rec)) == f).all()
    path = str(tmp_path / "x.mkv")
    _mux(native_lib, path, w, h, packets)
    mkv = ffv1.read_mkv(path)
    assert mkv["packets"] == packets and mkv["codec_private"] == rec and mkv["timestamps"] == [0, 33, 67, 100, 133]
    if _cv2() is None:
        pytest.skip("cv2 not importable")
    got = _play(path)
    assert len(got) == len(frames)
    for k, (a, b) in enumerate(zip(got, frames)):
        assert (a == b).all(), kinds[k]


def test_restated_stream_plays_back_in_cv2_at_1080p(native_lib, tmp_path):
    w, h = 1920, 1080
    frames = [_content("flat", w, h), _content("gradient", w, h)]
    path = str(tmp_path / "x.mkv")
    _mux(native_lib, path, w, h, [ffv1.encode_frame(f) for f in frames])
    if _cv2() is None:
        pytest.skip("cv2 not importable")
    got = _play(path)
    assert len(got) == 2 and all((a == b).all() for a, b in zip(got, frames))


def test_mkv_writer_argument_checks(native_lib, tmp_path):
    m = C.c_void_p()
    assert native_lib.poppy_host_mkv_open(C.byref(m), os.fsencode(str(tmp_path / "a.mkv")), 0, 4, 30, 1) == INVALID
    assert native_lib.poppy_host_mkv_open(C.byref(m), os.fsencode(str(tmp_path / "no" / "a.mkv")), 4, 4, 30, 1) == INVALID
    assert native_lib.poppy_host_mkv_open(C.byref(m), os.fsencode(str(tmp_path / "a.mkv")), 4, 4, 30, 1) == 0
    assert native_lib.poppy_host_mkv_write(m, None, 0) == INVALID
    assert native_lib.poppy_host_mkv_close(m) == 0


def test_api_rejects_unknown_pixel_format(native_lib):
    from poppy_b200 import api
    bgr1, bgr2, _, p1, p2 = any_size_inputs(16, 8, seed=1)
    with pytest.raises(ValueError, match="pixel_format"):
        api.morph_segments([(bgr1, bgr2, None, p1, p2)], number_of_frames=3, pixel_format="FFV1")


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _renderer(w, h, ring, seed=0, phases=None):
    from poppy_b200 import host
    from poppy_b200.renderer import MorphRenderer
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=seed)
    r = MorphRenderer(w, h, 6, len(p1), 2 * len(p1) + 16, ring)
    r.set_pair(bgr1, bgr2, gab)
    r.set_points(p1, p2)
    phases = np.linspace(0.05, 0.95, ring, dtype=np.float32) if phases is None else np.asarray(phases, np.float32)
    plan = host.SequencePlan(p1, p2, w, h, phases)
    try:
        r.render(phases, phases[::-1].astype(np.float64), plan.tri_idx, plan.tri_offsets)
    finally:
        plan.close()
    return r


def _upload(r, frames):
    """Overwrite ring slots 0.. with given BGR frames (device pointers of the ring)."""
    import ctypes
    lib = r._lib
    libcudart = ctypes.CDLL("libcudart.so")
    for i, f in enumerate(frames):
        p, step = C.c_void_p(), C.c_size_t()
        assert lib.poppy_cuda_frame_device_ptr(r._ctx, i, C.byref(p), C.byref(step)) == 0
        f = np.ascontiguousarray(f)
        assert libcudart.cudaMemcpy(p, f.ctypes.data_as(C.c_void_p), C.c_size_t(f.nbytes), 1) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (7, 5), (64, 48), (200, 100), (640, 360)])
def test_packets_equal_the_restated_encoder(native_lib, w, h):
    r = _renderer(w, h, 3)
    with r:
        bgr = r.download(0, 3)
        got = r.download_ffv1(0, 3)
        assert [bytes(p) for p in got] == [ffv1.encode_frame(f) for f in bgr]
        # the same frames in another batch shape and from another slot
        assert r.download_ffv1(1, 1) == got[1:2] and r.download_ffv1(2, 1) == got[2:]


@pytest.mark.gpu
def test_noise_overflows_and_still_decodes(native_lib, tmp_path):
    """Uniform noise has RCT residuals above 8 bits per sample: its slices overflow the raw-size slots and are coded again."""
    w, h = 200, 100
    r = _renderer(w, h, 3)
    with r:
        frames = [_content("noise", w, h, 5), _content("morph", w, h, 6), _content("noise", w, h, 7)]
        _upload(r, frames)
        before = np.zeros(1, np.uint64)
        assert native_lib.poppy_cuda_launch_count(r._ctx, before.ctypes.data_as(C.POINTER(C.c_uint64))) == 0
        got = r.download_ffv1(0, 3)
        after = np.zeros(1, np.uint64)
        assert native_lib.poppy_cuda_launch_count(r._ctx, after.ctypes.data_as(C.POINTER(C.c_uint64))) == 0
        assert len(got[0]) > w * h * 3                              # larger than the raw frame
        # symbols, code, re-code of the flagged slices, scan, pack
        assert int(after[0] - before[0]) == 5
        assert got == [ffv1.encode_frame(f) for f in frames]
        rec = ffv1.parse_config(ffv1.config_record(w, h))
        assert all((ffv1.decode_frame(p, w, h, rec) == f).all() for p, f in zip(got, frames))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160)])
def test_packets_decode_in_cv2_at_full_size(native_lib, tmp_path, w, h):
    cv2 = _cv2()
    if cv2 is None:
        pytest.skip("cv2 not importable")
    n = 4
    r = _renderer(w, h, n)
    with r:
        bgr = r.download(0, n)
        got = r.download_ffv1(0, n)
        path = str(tmp_path / "x.mkv")
        _mux(native_lib, path, w, h, got)
        frames = _play(path)
        assert len(frames) == n and all((a == b).all() for a, b in zip(frames, bgr))


@pytest.mark.gpu
def test_c_abi_argument_checks(native_lib):
    r = _renderer(64, 48, 3)
    with r:
        sizes = (C.c_uint32 * 3)()
        buf = (C.c_uint8 * 100000)()
        f = native_lib.poppy_cuda_download_ffv1
        assert f(None, 0, 1, buf, len(buf), sizes) == INVALID
        assert f(r._ctx, 0, 1, None, len(buf), sizes) == INVALID
        assert f(r._ctx, 0, 1, buf, len(buf), None) == INVALID
        assert f(r._ctx, -1, 1, buf, len(buf), sizes) == INVALID
        assert f(r._ctx, 2, 2, buf, len(buf), sizes) == INVALID
        assert f(r._ctx, 0, 0, buf, len(buf), sizes) == INVALID
        assert f(r._ctx, 0, 3, buf, len(buf), sizes) == 0
        need = sum(sizes)
        sizes2 = (C.c_uint32 * 3)()
        assert f(r._ctx, 0, 3, buf, need - 1, sizes2) == INVALID       # too small: sizes still say how much is needed
        assert list(sizes2) == list(sizes)
        assert f(r._ctx, 0, 3, buf, need, sizes2) == 0


@pytest.mark.gpu
def test_render_after_download_waits_for_it(native_lib):
    w, h, n = 1920, 1080, 12
    r = _renderer(w, h, n, seed=7)
    with r:
        before = r.download(0, n)
        want = [ffv1.encode_frame(f) for f in before[:1]]
        got = r.download_ffv1(0, n)
        from poppy_b200 import host
        bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=7)
        phases = np.linspace(0.9, 0.1, n, dtype=np.float32)
        plan = host.SequencePlan(p1, p2, w, h, phases)
        try:
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
        finally:
            plan.close()
        r.sync()
        assert (r.download(0, n) != before).any()
        assert got[:1] == want


@pytest.mark.gpu
@pytest.mark.parametrize("ring", [3, 40])
def test_ffv1_writer_ring(native_lib, ring):
    w, h, n = 322, 180, 20
    r = _renderer(w, h, n, seed=9)
    with r:
        want = r.download_ffv1(0, n)
        got = []

        def packet(user, idx, data, size):
            got.append((idx, C.string_at(data, size)))

        cb = _PACKET(packet)
        wr = C.c_void_p()
        assert native_lib.poppy_host_writer_create_ffv1(C.byref(wr), r._ctx, ring, cb, None) == 0
        try:
            assert native_lib.poppy_host_writer_submit(wr, 0, 12, 0) == 0
            assert native_lib.poppy_host_writer_submit(wr, 12, 8, 12) == 0
            assert native_lib.poppy_host_writer_flush(wr) == 0
        finally:
            native_lib.poppy_host_writer_destroy_cuda(wr)
        assert [i for i, _ in got] == list(range(n))
        assert [p for _, p in got] == want


class _Writer:
    def __init__(self):
        self.frames = []

    def write(self, f):
        self.frames.append(f)


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [None, [0, 1]])
def test_api_routes_write_mkv_equal_to_bgr(native_lib, tmp_path, devices):
    from poppy_b200 import api
    if devices and api.device_count() < 2:
        pytest.skip("needs two GPUs")
    cv2 = _cv2()
    w, h = 160, 96
    bgr1, bgr2, _, p1, p2 = any_size_inputs(w, h, seed=11)
    try:
        if devices is None:
            bgr = api.morph_sequence(bgr1, bgr2, None, p1, p2, number_of_frames=7)
            wr = _Writer()
            got = api.morph_sequence(bgr1, bgr2, None, p1, p2, writer=wr, number_of_frames=7, pixel_format="ffv1")
            assert got == [ffv1.encode_frame(f) for f in bgr] and wr.frames == got
            phases = [0.2, 0.5, 0.8]
            bgr = api.render_phases(bgr1, bgr2, None, p1, p2, phases)
            got = api.render_phases(bgr1, bgr2, None, p1, p2, phases, pixel_format="ffv1")
            assert got == [ffv1.encode_frame(f) for f in bgr]
        segs = [(bgr1, bgr2, None, p1, p2), (bgr2, bgr1, None, p2, p1), (bgr1, bgr2, None, p2, p1)]
        bgr = api.morph_segments(segs, number_of_frames=5, devices=devices)
        path = str(tmp_path / "out.mkv")
        with api.MatroskaWriter(path, w, h) as mw:
            got = api.morph_segments(segs, number_of_frames=5, writer=mw, devices=devices, pixel_format="ffv1")
        assert len(got) == 3 and all(len(s) == 5 for s in got)
        assert ffv1.read_mkv(path)["packets"] == [p for s in got for p in s]
        if cv2 is not None:
            frames = _play(path)
            assert len(frames) == 15 and all((a == b).all() for a, b in zip(frames, bgr.reshape(-1, h, w, 3)))
    finally:
        api.release()
