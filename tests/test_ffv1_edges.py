"""The FFV1 encoder (poppy_cuda_download_ffv1) on the paths real use takes, held to the restated encoder (oracle/ffv1.py):

- natural frames, whose slices fit the raw-size slots of the first pass and are packed straight from them;
- packets that mix slices packed from slots with slices coded again into worst-case scratch;
- slices within a few bytes of the slot's stop point and of its capacity (fixture golden/output/ffv1/slot_boundary.json);
- slice grids whose columns or rows differ in size, up to 4K and the 32-slice column and row caps;
- downloads longer than one staging piece (the host loop), the 4096-frame piece bound and the library route over them;
- the FFV1 writer's heap fallback for a packet larger than its ring buffer;
- residuals at the fold edges (-256, +255, exponent 8) under both signs of the context in both context planes.

Each GPU test asserts on the CPU the regime it names (slice sizes against the slot, an uneven grid, a download longer than a
piece, a packet larger than the writer's buffer), so it cannot pass on another path. Packets up to about 1 Mpx are compared
whole; above that a fixed sample of slices is compared, every slice size is checked from the packet and cv2 decodes it."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from oracle import ffv1
from tests.test_ffv1 import _PACKET, _cv2, _mux, _play
from tests.util import any_size_inputs

BOUNDARY = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "output", "ffv1", "slot_boundary.json")
STAGE_PIXELS = 8 * 3840 * 2160      # kFfv1StagePixels (poppy_cuda.cu): pixels encoded per piece
PIECE_FRAMES = 4096                 # and at most this many frames (the symbol kernel's grid z)
FULL_PX = 1 << 20                   # packets up to this many pixels are compared whole with the restated encoder


# ---- restatements of the host side of poppy_cuda_download_ffv1 ------------------------------------------------------
def piece_frames(w, h, ring):
    """Frames per piece: ffv1_stage's f.frames."""
    return max(1, min(ring, STAGE_PIXELS // (w * h), PIECE_FRAMES))


def slot_cap(w, h):
    """(cap, limit) of ffv1_stage and k_ffv1_code: the first pass codes each slice into `cap` bytes, the raw bytes of the
    largest slice + 64 rounded up to 16, and stops a slice when its committed bytes exceed `limit` before a symbol. A slice
    whose restated size is <= limit is never coded again; one whose size is > cap - 3 always is."""
    nh, nv = ffv1.slice_grid(w, h)
    px = -(-w // nh) * -(-h // nv)
    cap = (px * 3 + 64 + 15) // 16 * 16
    return cap, cap - 22 - 3


def writer_buffer(w, h):
    """Bytes of one FFV1 writer ring buffer (poppy_host_writer_create_ffv1)."""
    return w * h * 3 + 65536


def restated_slices(bgr, which):
    """{s: bytes} of the selected slices of a frame, as encode_frame writes them (slice 0 starts with the keyframe bit)."""
    h, w = bgr.shape[:2]
    nh, _ = ffv1.slice_grid(w, h)
    rects = ffv1.slice_rects(w, h)
    out = {}
    for s in which:
        x0, y0, x1, y1 = rects[s]
        rc = None
        if s == 0:
            rc = ffv1.RangeEncoder()
            rc.bit([128], 0, 1)
        out[s] = ffv1.encode_slice(bgr[y0:y1, x0:x1], s % nh, s // nh, rc)
    return out


def packet_slices(packet):
    return [bytes(packet[a:a + n]) for a, n in ffv1.split_slices(packet)]


def slice_sizes(w, h):
    """(column widths, row heights) of the slice grid."""
    nh, nv = ffv1.slice_grid(w, h)
    return [w * (i + 1) // nh - w * i // nh for i in range(nh)], [h * (j + 1) // nv - h * j // nv for j in range(nv)]


def sample_slices(w, h, seed=0, extra=3):
    """The four corner slices, the first and last slice of every column and row whose size differs from a neighbour's, and
    `extra` seeded random slices."""
    nh, nv = ffv1.slice_grid(w, h)
    cols, rows = slice_sizes(w, h)

    def differs(sz, k):
        return (k > 0 and sz[k] != sz[k - 1]) or (k + 1 < len(sz) and sz[k] != sz[k + 1])

    pick = {0, nh - 1, nh * (nv - 1), nh * nv - 1}
    pick |= {s for i in range(nh) if differs(cols, i) for s in (i, (nv - 1) * nh + i)}
    pick |= {s for j in range(nv) if differs(rows, j) for s in (j * nh, j * nh + nh - 1)}
    rng = np.random.default_rng(seed)
    pick |= set(rng.choice(nh * nv, min(extra, nh * nv), replace=False).tolist())
    return sorted(pick)


def check_packet(packet, bgr, seed=0):
    """packet against the restated encoder: whole up to FULL_PX, else the sampled slices, the slice count and every slice
    size. Returns {slice: restated size} of the slices compared."""
    h, w = bgr.shape[:2]
    nh, nv = ffv1.slice_grid(w, h)
    if w * h <= FULL_PX:
        want = ffv1.encode_frame(bgr)
        assert bytes(packet) == want
        return {s: len(b) for s, b in enumerate(packet_slices(want))}
    got = packet_slices(packet)
    assert len(got) == nh * nv
    cap, _ = slot_cap(w, h)
    scratch_cap = (-(-w // nh) * -(-h // nv) * 38 + 128 + 15) // 16 * 16
    assert all(0 < len(s) <= scratch_cap for s in got) and sum(len(s) + 3 for s in got) == len(packet)
    want = restated_slices(bgr, sample_slices(w, h, seed))
    for s, b in want.items():
        assert got[s] == b, f"slice {s} of {nh} x {nv}"
    return {s: len(b) for s, b in want.items()}


def cv2_decodes(lib, tmp_path, w, h, packets, frames):
    """cv2 plays the packets, muxed into Matroska, back to exactly `frames`."""
    if _cv2() is None:
        return
    path = str(tmp_path / "edges.mkv")
    _mux(lib, path, w, h, packets)
    got = _play(path)
    assert len(got) == len(frames)
    for k, (a, b) in enumerate(zip(got, frames)):
        assert (a == b).all(), k


# ---- content --------------------------------------------------------------------------------------------------------
def smooth(w, h, seed=0):
    """Slow sinusoids in 70..190 (any_size_inputs(..., smooth=True)'s images for seed 0 and 1): slices far below their slot."""
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    return np.stack([130 + 60 * np.sin(x / (17.0 + 4 * c + seed) + y / (23.0 + 3 * c) + c + 2 * seed) for c in range(3)],
                    -1).round().astype(np.uint8)


def noise(w, h, seed=0):
    """Uniform random bytes: RCT residuals above 8 bits per sample, slices above their slot."""
    return np.random.default_rng(1000 + seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def mix(w, h, noisy, seed=0):
    """Smooth content with noise over the rectangles of the slices in `noisy`."""
    f, n = smooth(w, h, seed), noise(w, h, seed)
    for s, (x0, y0, x1, y1) in enumerate(ffv1.slice_rects(w, h)):
        if s in noisy:
            f[y0:y1, x0:x1] = n[y0:y1, x0:x1]
    return f


def boundary_slice(w, h, n, seed):
    """A w x h slice whose first n pixels in raster order are noise and the rest smooth: its restated size grows with n by
    about 3.6 bytes per pixel (make_slot_boundary.py picks n)."""
    f = smooth(w, h).reshape(-1, 3)
    f[:n] = noise(w, h, seed).reshape(-1, 3)[:n]
    return f.reshape(h, w, 3)


PALETTE = np.array([0, 1, 2, 127, 128, 253, 254, 255], np.uint8)


def fold_edges(w, h, seed=1):
    """Extreme palette values: a white first pixel gives G' residual +255 and B', R' residuals 256 (folded to -256,
    exponent 8) against the zero neighbours above a slice; the rest reach both signs of the context in both planes."""
    f = PALETTE[np.random.default_rng(seed).integers(0, len(PALETTE), (h, w, 3))]
    f[0, 0] = 255
    return f


def fold_coverage(bgr):
    """Which fold and context edges a slice's symbols reach (raw contexts before the sign fold, per context plane)."""
    _, res = ffv1.slice_symbols(bgr)
    raw = [ffv1._context_and_pred(p)[0] for p in ffv1._rct_planes(bgr)]
    planes = [raw[0], np.stack(raw[1:])]
    return {"-256": bool((res == -256).any()), "+255": bool((res == 255).any()),
            "ctx0<0": bool((planes[0] < 0).any()), "ctx0>0": bool((planes[0] > 0).any()),
            "ctx1<0": bool((planes[1] < 0).any()), "ctx1>0": bool((planes[1] > 0).any())}


# ---- GPU helpers ----------------------------------------------------------------------------------------------------
def ring(w, h, frames):
    """A renderer whose ring slots are filled by upload() alone."""
    from poppy_b200.renderer import MorphRenderer
    _, _, _, p1, _ = any_size_inputs(w, h)
    return MorphRenderer(w, h, 6, len(p1), 2 * len(p1) + 16, frames)


def rendered(w, h, frames, seed=0):
    """A ring of `frames` slots rendered from smooth inputs: natural frames."""
    from poppy_b200 import host
    bgr1, bgr2, gab, p1, p2 = any_size_inputs(w, h, seed=seed, smooth=True)
    r = ring(w, h, frames)
    r.set_pair(bgr1, bgr2, gab)
    r.set_points(p1, p2)
    phases = np.linspace(0.05, 0.95, frames, dtype=np.float32)
    plan = host.SequencePlan(p1, p2, w, h, phases)
    try:
        r.render(phases, phases[::-1].astype(np.float64), plan.tri_idx, plan.tri_offsets)
    finally:
        plan.close()
    r.sync()
    return r


_cudart = None


def upload(r, frames, first=0):
    """Write BGR frames into ring slots first, first + 1, ... (device pointers of the ring)."""
    global _cudart
    if _cudart is None:
        _cudart = C.CDLL("libcudart.so")
    for i, f in enumerate(frames):
        p, step = C.c_void_p(), C.c_size_t()
        assert r._lib.poppy_cuda_frame_device_ptr(r._ctx, first + i, C.byref(p), C.byref(step)) == 0
        f = np.ascontiguousarray(f)
        assert f.shape == (r.height, r.width, 3) and step.value == f.nbytes
        assert _cudart.cudaMemcpy(p, f.ctypes.data_as(C.c_void_p), C.c_size_t(f.nbytes), 1) == 0


def launches(r, fn):
    """(fn(), kernel launches it made on r's context)."""
    def count():
        v = np.zeros(1, np.uint64)
        assert r._lib.poppy_cuda_launch_count(r._ctx, v.ctypes.data_as(C.POINTER(C.c_uint64))) == 0
        return int(v[0])
    before = count()
    out = fn()
    return out, count() - before


# one piece: symbols, code, scan, pack; a piece with a slice that did not fit its slot also codes the listed slices again
def piece_launches(overflow):
    return 5 if overflow else 4


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_slot_cap_restates_the_stage():
    assert slot_cap(128, 96) == (36928, 36903)
    assert slot_cap(256, 96) == (36928, 36903)
    cap = (128 * 99 * 3 + 64 + 15) // 16 * 16                   # 1080p: the largest slice is 128 x 99
    assert slot_cap(1920, 1080) == (cap, cap - 25)
    assert piece_frames(1920, 1080, 70) == 32 and piece_frames(3840, 2160, 20) == 8
    assert piece_frames(16, 16, 4100) == PIECE_FRAMES < STAGE_PIXELS // 256


@pytest.mark.parametrize("w,h", [(64, 48), (322, 180), (640, 360)])
def test_content_regimes(w, h):
    """smooth slices stay within the first pass's limit, noise slices pass the slot's capacity."""
    cap, limit = slot_cap(w, h)
    sm = [len(b) for b in restated_slices(smooth(w, h, 1), range(ffv1.slice_grid(w, h)[0])).values()]
    no = [len(b) for b in restated_slices(noise(w, h, 1), [0]).values()]
    assert max(sm) <= limit and min(no) > cap - 3, (sm, no, cap)


def test_slot_boundary_fixture_sizes():
    fx = json.load(open(BOUNDARY))
    w, h = fx["w"], fx["h"]
    cap, limit = slot_cap(w, h)
    assert (fx["cap"], fx["limit"]) == (cap, limit) and ffv1.slice_grid(w, h) == (1, 1)
    for p in fx["points"]:
        size = len(ffv1.encode_frame(boundary_slice(w, h, p["n"], fx["seed"]))) - 3
        assert size == p["size"], p
        lo, hi = p["window"]
        assert lo <= size <= hi, p


@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (7, 5), (64, 48), (130, 97)])
def test_fold_edge_content_reaches_the_edges(w, h):
    assert ffv1.slice_grid(w, h) == (1, 1)
    got = fold_coverage(fold_edges(w, h))
    if (w, h) == (1, 1):        # a single sample: no neighbours, context 0
        assert got["-256"] and got["+255"]
    else:
        assert all(got.values()), got


def test_grids_are_uneven():
    for w, h in [(322, 180), (1001, 601), (4200, 64), (64, 4001), (1920, 1080), (3840, 2160)]:
        cols, rows = slice_sizes(w, h)
        assert len(set(cols)) > 1 or len(set(rows)) > 1, (w, h)
    assert ffv1.slice_grid(4200, 64) == (32, 1) and ffv1.slice_grid(64, 4001) == (1, 32)
    assert ffv1.slice_grid(191, 143) == (1, 1) and ffv1.slice_grid(192, 144) == (2, 2)


# ---- GPU: natural frames --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(64, 48), (129, 97), (322, 180), (640, 360), (1001, 601)])
def test_natural_frames_take_the_first_pass_only(native_lib, w, h):
    cap, limit = slot_cap(w, h)
    with rendered(w, h, 2) as r:
        bgr = r.download(0, 2)
        got, n = launches(r, lambda: r.download_ffv1(0, 2))
        for p, f in zip(got, bgr):
            sizes = check_packet(p, f)
            assert len(sizes) == np.prod(ffv1.slice_grid(w, h)) and max(sizes.values()) <= limit, (sizes, limit)
        assert n == piece_launches(False)


# ---- GPU: packets mixing slot and scratch slices --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(322, 180), (640, 360)])
def test_mixed_packets(native_lib, tmp_path, w, h):
    nh, nv = ffv1.slice_grid(w, h)
    cap, limit = slot_cap(w, h)
    last = nh * nv - 1
    kinds = [{s for s in range(nh * nv) if (s % nh + s // nh) % 2 == 0}, {0}, {last}]
    frames = [mix(w, h, noisy, k) for k, noisy in enumerate(kinds)]
    with ring(w, h, len(frames)) as r:
        upload(r, frames)
        got, n = launches(r, lambda: r.download_ffv1(0, len(frames)))
        for p, f, noisy in zip(got, frames, kinds):
            sizes = check_packet(p, f)
            assert all(sizes[s] > cap - 3 for s in noisy) and all(sizes[s] <= limit for s in sizes if s not in noisy)
        assert n == piece_launches(True)
        cv2_decodes(native_lib, tmp_path, w, h, got, frames)


# ---- GPU: the slot boundary -----------------------------------------------------------------------------------------
def _expect_launches(sizes, cap, limit):
    if max(sizes) > cap - 3:
        return {5}
    return {4} if max(sizes) <= limit else {4, 5}


@pytest.mark.gpu
def test_slot_boundary(native_lib):
    fx = json.load(open(BOUNDARY))
    w, h, seed = fx["w"], fx["h"], fx["seed"]
    cap, limit = slot_cap(w, h)
    by = {p["target"]: p for p in fx["points"]}
    one = [boundary_slice(w, h, p["n"], seed) for p in fx["points"]]
    # two slices side by side: one near the stop point or the capacity, its neighbour past the capacity, both ways round
    pairs = [("cap-3", "cap"), ("cap", "cap-3"), ("limit", "cap+16"), ("cap+16", "limit"), ("limit", "limit"),
             ("cap-2", "cap-2"), ("limit-19", "limit+1")]
    two = [np.concatenate([boundary_slice(w, h, by[a]["n"], seed), boundary_slice(w, h, by[b]["n"], seed)], 1)
           for a, b in pairs]
    for frames in (one, two):
        fw = frames[0].shape[1]
        assert slot_cap(fw, h) == (cap, limit)
        with ring(fw, h, len(frames)) as r:
            upload(r, frames)
            for k, f in enumerate(frames):
                (p,), n = launches(r, lambda: r.download_ffv1(k, 1))
                want = ffv1.encode_frame(f)
                sizes = [len(s) for s in packet_slices(want)]
                assert bytes(p) == want, (k, sizes)
                assert n in _expect_launches(sizes, cap, limit), (k, sizes, n)
            # all at once: one piece, the slots and scratch of different frames side by side
            assert r.download_ffv1(0, len(frames)) == [ffv1.encode_frame(f) for f in frames]
    # the pairs put a slice that fits beside one that does not
    sz = [[len(s) for s in packet_slices(ffv1.encode_frame(f))] for f in two]
    assert any(a <= limit and b > cap - 3 for a, b in sz) and any(b <= limit and a > cap - 3 for a, b in sz)


# ---- GPU: uneven slice grids ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(322, 180), (1001, 601), (4200, 64), (64, 4001), (191, 143), (192, 144), (1920, 1080),
                                 (3840, 2160)])
def test_uneven_grids(native_lib, tmp_path, w, h):
    frames = [smooth(w, h, 2), noise(w, h, 3)]
    with ring(w, h, 2) as r:
        upload(r, frames)
        got = r.download_ffv1(0, 2)
        for k, (p, f) in enumerate(zip(got, frames)):
            check_packet(p, f, seed=k)
        cv2_decodes(native_lib, tmp_path, w, h, got, frames)


# ---- GPU: downloads longer than one piece ---------------------------------------------------------------------------
def _pieces_check(lib, tmp_path, r, w, h, count, noisy, check_frames, ranges):
    per = piece_frames(w, h, count)
    assert count > per
    cap, limit = slot_cap(w, h)
    for k, s in enumerate(noisy):
        upload(r, [noise(w, h, 10 + k)], s)
    bgr = r.download(0, count)
    got, n = launches(r, lambda: r.download_ffv1(0, count))
    assert len(got) == count
    # per piece: 4 launches, 5 with a noise frame in it
    assert n == sum(piece_launches(any(p <= s < p + per for s in noisy)) for p in range(0, count, per))
    assert [r.download_ffv1(k, 1)[0] for k in range(count)] == got
    for a, c in ranges:
        assert r.download_ffv1(a, c) == got[a:a + c], (a, c)
    for k in check_frames:
        sizes = check_packet(got[k], bgr[k], seed=k)
        assert min(sizes.values()) > cap - 3 if k in noisy else max(sizes.values()) <= limit, k
    cv2_decodes(lib, tmp_path, w, h, got, bgr)
    return got


@pytest.mark.gpu
def test_pieces_1080p(native_lib, tmp_path):
    w, h = 1920, 1080
    with rendered(w, h, 70) as r:
        # pieces of 32, 32 and 6 frames; pieces 1 and 2 list 165 and 330 slices, so scratch grows between them
        _pieces_check(native_lib, tmp_path, r, w, h, 70, [31, 32, 63, 64], [0, 31, 32, 63, 64, 69],
                      [(5, 60), (30, 4), (33, 37), (60, 10)])


@pytest.mark.gpu
def test_pieces_4k(native_lib, tmp_path):
    w, h = 3840, 2160
    R = writer_buffer(w, h)
    with rendered(w, h, 20) as r:
        # pieces of 8, 8 and 4 frames
        _pieces_check(native_lib, tmp_path, r, w, h, 20, [7, 8, 16], [0, 7, 8, 16, 19], [(5, 12), (9, 11)])
        # nine noise frames in one call: their packets pass MorphRenderer.download_ffv1's first buffer (count x
        # (W * H * 3 + 65536) bytes), so it encodes both pieces again at the size the refused call reported
        frames = [noise(w, h, 20 + k) for k in range(9)]
        upload(r, frames, 2)
        got, n = launches(r, lambda: r.download_ffv1(2, 9))
        assert sum(len(p) for p in got) > 9 * R
        assert n == 2 * 2 * piece_launches(True)
        assert [r.download_ffv1(2 + k, 1)[0] for k in range(9)] == got
        for k in (0, 8):
            check_packet(got[k], frames[k], seed=k)


@pytest.mark.gpu
def test_piece_frame_cap(native_lib):
    """4100 frames of 16 x 16: pieces of 4096 and 4 frames, the frame bound in force rather than the pixel bound. Frames
    repeat with period 13 (4096 = 1 mod 13), so a piece offset by whole frames shows; frame 3 of the period is noise, so
    both pieces code slices again."""
    w, h, count, period, noisy = 16, 16, 4100, 13, 3
    base = [noise(w, h, 4) if k == noisy else smooth(w, h, k) for k in range(period)]
    want = [ffv1.encode_frame(f) for f in base]
    cap, limit = slot_cap(w, h)
    assert all(len(p) - 3 > cap - 3 if k == noisy else len(p) - 3 <= limit for k, p in enumerate(want))
    with ring(w, h, count) as r:
        upload(r, [base[k % period] for k in range(count)])
        assert piece_frames(w, h, count) == PIECE_FRAMES
        got, n = launches(r, lambda: r.download_ffv1(0, count))
        assert any(k % period == noisy for k in range(PIECE_FRAMES, count)) and n == 2 * piece_launches(True)
        assert got == [want[k % period] for k in range(count)]
        assert r.download_ffv1(4090, 10) == [want[k % period] for k in range(4090, 4100)]


@pytest.mark.gpu
def test_library_route_over_two_pieces(native_lib, tmp_path, monkeypatch):
    from poppy_b200 import api
    from poppy_b200.renderer import MorphRenderer
    w, h, N = 1920, 1080, 24
    a1, a2, _, p1, p2 = any_size_inputs(w, h, seed=1, smooth=True)
    segs = [(a1, a2, None, p1, p2), (a2, a1, None, p2, p1)]
    calls = []
    download_ffv1 = MorphRenderer.download_ffv1

    def spy(self, first, count):
        calls.append((first, count))
        return download_ffv1(self, first, count)

    monkeypatch.setattr(MorphRenderer, "download_ffv1", spy)
    try:
        bgr = api.morph_segments(segs, number_of_frames=N).reshape(-1, h, w, 3)
        path = str(tmp_path / "out.mkv")
        with api.MatroskaWriter(path, w, h) as mw:
            got = api.morph_segments(segs, number_of_frames=N, writer=mw, pixel_format="ffv1")
    finally:
        api.release()
    # one batch: one download of 48 frames, two pieces
    assert calls == [(0, 2 * N)] and 2 * N > piece_frames(w, h, 2 * N)
    flat = [p for s in got for p in s]
    assert ffv1.read_mkv(path)["packets"] == flat
    if _cv2() is not None:
        frames = _play(path)
        assert len(frames) == 2 * N and all((a == b).all() for a, b in zip(frames, bgr))
    _, limit = slot_cap(w, h)
    for k in (0, 31, 32, 47):
        assert max(check_packet(flat[k], bgr[k], seed=k).values()) <= limit


# ---- GPU: the writer's large-packet fallback ------------------------------------------------------------------------
@pytest.mark.gpu
def test_writer_large_packet_fallback(native_lib):
    w, h = 640, 360
    frames = [smooth(w, h, 0), noise(w, h, 1), noise(w, h, 2), smooth(w, h, 3), noise(w, h, 4), smooth(w, h, 5)]
    big = ffv1.encode_frame(frames[1])
    assert len(big) > writer_buffer(w, h)
    with ring(w, h, len(frames)) as r:
        upload(r, frames)
        want = r.download_ffv1(0, len(frames))
        assert want[1] == big
        got = []

        def packet(user, idx, data, size):
            got.append((idx, C.string_at(data, size)))

        cb = _PACKET(packet)
        wr = C.c_void_p()
        assert native_lib.poppy_host_writer_create_ffv1(C.byref(wr), r._ctx, 3, cb, None) == 0
        try:
            assert native_lib.poppy_host_writer_submit(wr, 0, 4, 0) == 0
            assert native_lib.poppy_host_writer_submit(wr, 4, 2, 4) == 0
            assert native_lib.poppy_host_writer_flush(wr) == 0
        finally:
            native_lib.poppy_host_writer_destroy_cuda(wr)
        assert [i for i, _ in got] == list(range(len(frames)))
        assert [p for _, p in got] == want
        assert sum(len(p) > writer_buffer(w, h) for p in want) == 3


# ---- GPU: fold and exponent edges -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (7, 5), (64, 48), (130, 97)])
def test_fold_edges(native_lib, w, h):
    frames = [fold_edges(w, h), fold_edges(w, h)[::-1, ::-1], 255 - fold_edges(w, h)]
    with ring(w, h, len(frames)) as r:
        upload(r, frames)
        assert r.download_ffv1(0, len(frames)) == [ffv1.encode_frame(f) for f in frames]
