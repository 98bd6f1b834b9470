"""Python mirror of the reference interface for the morph path.

  Settings                the fields of poppy::Settings (reference src/settings.hpp:14-27); the path reads
                          pyramid_levels (src/algo.cpp:261)
  init(...)               poppy::init (reference src/poppy.hpp:30-44), same argument order
  morph_images(...)       poppy::morph_images (reference src/algo.hpp:26, src/algo.cpp:178-273): one frame, host
                          arrays in, (dst, morphedPoints) out
  morph_sequence(...)     the frame loop of poppy::morph<Twriter>() (reference src/poppy.hpp:177-243, phase < 0):
                          the chain recurrence kept resident on the GPU, frames handed to writer.write() in order
  render_phases(...)      direct mode: N independent phases of one pair ("-f 1 -p s", src/poppy.hpp:186-200)
  morph_segments(...)     the segments of a multi-image sequence (reference run(), src/poppy.cpp:266-328): one chain per
                          consecutive pair, rendered together (step j of every segment in one kernel batch); with
                          devices=[...] sharded by segment over several GPUs of one box

morph_sequence and render_phases take gabor2=None: the GPU then derives it from corrected2 exactly as poppy::morph()
does before its frame loop (gabor_filter(corrected2 * 1/255), src/poppy.hpp:119-122), and the float image never exists.

morph_sequence, render_phases and morph_segments take pixel_format="bgr" (H x W x 3 frames) or "i420": each frame is then
converted on the GPU to what cv2.cvtColor(frame, cv2.COLOR_BGR2YUV_I420) returns, an (H * 3 // 2) x W plane stack (Y, then U
and V at half resolution) that an encoder fed yuv420p takes as it is, and half the bytes cross PCIe. I420 needs an even
frame size. "ffv1" returns lossless FFV1 packets (bytes) encoded on the GPU, the reference's default output format; a
MatroskaWriter(path, w, h) as the writer gives the .mkv that cv::VideoWriter with fourcc FFV1 writes.

Host stages (clip / uniq / Delaunay / index lookup) run in the C++ part of libpoppy_cuda.so, everything else in its
CUDA kernels. Nothing in this module computes pixels; without the native library or a GPU every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from fractions import Fraction

import operator
import threading

import numpy as np

from . import _lib, host, shard
from .renderer import MorphRenderer, device_count


@dataclass
class _Settings:
    show_gui: bool = False
    enable_wait: bool = False
    number_of_frames: float = 60
    frame_rate: float = 30
    match_tolerance: float = 1
    max_keypoints: int = 300
    pyramid_levels: int = 64
    enable_auto_align: bool = False
    enable_radial_mask: bool = False
    enable_face_detection: bool = False
    enable_denoise: bool = False
    enable_src_scaling: bool = False
    face_neighbors: int = 8
    fourcc: str = "FFV1"
    cuda_device: int = 0          # addition: the GPU the renderer runs on


class Settings:
    """Process-wide singleton, as poppy::Settings::instance()."""
    _instance = None

    @classmethod
    def instance(cls) -> _Settings:
        if cls._instance is None:
            cls._instance = _Settings()
        return cls._instance


def init(show_gui, number_of_frames, match_tolerance, auto_align, radial_mask, face_detect, denoise, src_scaling,
         frame_rate, pyramid_levels, fourcc, enable_wait, face_neighbors):
    s = Settings.instance()
    s.show_gui, s.enable_wait, s.number_of_frames, s.frame_rate = show_gui, enable_wait, number_of_frames, frame_rate
    s.match_tolerance, s.enable_auto_align, s.enable_radial_mask = match_tolerance, auto_align, radial_mask
    s.enable_denoise, s.enable_src_scaling, s.enable_face_detection = denoise, src_scaling, face_detect
    s.pyramid_levels, s.fourcc, s.face_neighbors = pyramid_levels, fourcc, face_neighbors


_cache: dict = {}


def _renderer(w, h, n_points, n_tri, n_frames) -> MorphRenderer:
    s = Settings.instance()
    key = (w, h, int(s.pyramid_levels), s.cuda_device)
    r = _cache.get(key)
    if r is None or r.max_points < n_points or r.max_triangles < n_tri or r.max_batch_frames < n_frames:
        if r is not None:
            r.close()
        r = MorphRenderer(w, h, int(s.pyramid_levels), max(n_points, 64), max(n_tri, 2 * n_points + 16), n_frames,
                          device=s.cuda_device)
        _cache.clear()
        _cache[key] = r
    return r


# renderers of morph_segments(devices=...) on the listed GPUs other than Settings.cuda_device, one per device: they neither evict
# nor replace the renderer in _cache, which the single-device entry points share
_device_cache: dict = {}


def _device_renderer(device, w, h, n_points, n_tri, n_frames) -> MorphRenderer:
    levels = int(Settings.instance().pyramid_levels)
    r = _device_cache.get(device)
    if r is None or (r.width, r.height, r.levels) != (w, h, levels) or r.max_points < n_points or r.max_triangles < n_tri \
            or r.max_batch_frames < n_frames:
        if r is not None:
            r.close()
            del _device_cache[device]
        r = MorphRenderer(w, h, levels, max(n_points, 64), max(n_tri, 2 * n_points + 16), n_frames, device=device)
        _device_cache[device] = r
    return r


def release():
    for r in list(_cache.values()) + list(_device_cache.values()):
        r.close()
    _cache.clear()
    _device_cache.clear()


def morph_images(img1, img2, corrected1, corrected2, gabor2, src_points1, src_points2, shape_ratio, mask_ratio,
                 linear=0.0):
    """One frame. img1 supplies only the frame size; img2 and linear are unused, as in the reference.
    Returns (dst HxWx3 uint8, morphedPoints Nx2 float32)."""
    h, w = img1.shape[:2]
    p1 = np.ascontiguousarray(src_points1, np.float32)
    p2 = np.ascontiguousarray(src_points2, np.float32)
    if p1.shape != p2.shape:
        raise ValueError("point sets differ in size")          # assert at src/algo.cpp:51
    morphed = host.morph_points(p1, p2, shape_ratio, w, h)     # host copy, needed for the topology
    r = _renderer(w, h, len(p1), 2 * len(p1) + 16, 1)          # sized for the most triangles these points can give
    # the pair travels to the device (150 MB at 4K) while this thread triangulates; both are C calls that release the GIL
    failure = []

    def upload():
        try:
            r.set_pair(np.ascontiguousarray(corrected1), np.ascontiguousarray(corrected2), np.ascontiguousarray(gabor2))
            r.set_points(p1, p2)
        except Exception as e:      # re-raised on the calling thread
            failure.append(e)
    t = threading.Thread(target=upload)
    t.start()
    try:
        tri = host.triangulate(morphed, w, h, sequential=True)
    finally:
        t.join()
    if failure:
        raise failure[0]
    r.render([shape_ratio], [mask_ratio], tri, [0, len(tri)])
    dst = r.download(0, 1)[0]
    return dst, r.morphed_points(0)


def blur_margin(src, union_size):
    """poppy::blur_margin (reference src/util.cpp:574-602) on the GPU: `src` (H x W x 3 uint8) centred on a black canvas of
    union_size = (width, height) with its four margins Gaussian-blurred. Returns the canvas."""
    from . import _lib
    import ctypes as C
    src = np.ascontiguousarray(src, np.uint8)
    if src.ndim != 3 or src.shape[2] != 3:
        raise ValueError("blur_margin: expected an H x W x 3 uint8 image")
    uw, uh = int(union_size[0]), int(union_size[1])
    dst = np.empty((max(uh, 0), max(uw, 0), 3), np.uint8)
    lib = _lib.load()
    rc = lib.poppy_cuda_blur_margin(Settings.instance().cuda_device, src.ctypes.data_as(C.c_void_p), src.strides[0], src.shape[1],
                                    src.shape[0], uw, uh, dst.ctypes.data_as(C.c_void_p), dst.strides[0] if dst.size else 0)
    if rc != 0:
        raise RuntimeError(f"poppy_cuda_blur_margin failed ({rc}): {lib.poppy_cuda_blur_margin_last_error().decode()}")
    return dst


def gabor_filter(src):
    """poppy::gabor_filter(src, dst) with the reference's defaults (src/util.cpp:40-60) on the GPU; src: H x W x 3 float32.
    Agrees with the reference to float rounding (see include/poppy_cuda.h).
    The reference passes corrected2.convertTo(CV_32F, 1/255), i.e. corrected2.astype(np.float32) * np.float32(1 / 255.0):
    a multiplication, not a division by 255 (the two round 126 of the 256 byte values differently). With the multiplication
    the filter reproduces the gabor2 that reference pipeline recorded for tests/golden/full/c2.npz bit for bit (c1.npz: to
    the DFT's round-off near 0). To feed a pair's renderer, pass gabor2=None to morph_sequence / render_phases /
    MorphRenderer.set_pair instead: the same filter then runs on the device without this round trip."""
    from . import _lib
    import ctypes as C
    src = np.ascontiguousarray(src, np.float32)
    if src.ndim != 3 or src.shape[2] != 3:
        raise ValueError("gabor_filter: expected an H x W x 3 float32 image")
    dst = np.empty_like(src)
    lib = _lib.load()
    rc = lib.poppy_cuda_gabor_filter(Settings.instance().cuda_device, src.ctypes.data_as(C.c_void_p), src.strides[0], src.shape[1],
                                     src.shape[0], dst.ctypes.data_as(C.c_void_p), dst.strides[0])
    if rc != 0:
        raise RuntimeError(f"poppy_cuda_gabor_filter failed ({rc}): {lib.poppy_cuda_blur_margin_last_error().decode()}")
    return dst


def denoise(src, h=3.0, template_window_size=7, search_window_size=21):
    """cv::fastNlMeansDenoising(src, dst, h, template_window_size, search_window_size) on the GPU, bit for bit, with the same
    defaults: the --denoise step the reference's run() applies to every input image (src/poppy.cpp:172, 269-311).
    src: H x W x 3 uint8 (rows may be strided, as in a ROI). Returns a new H x W x 3 uint8 array."""
    from . import _lib
    import ctypes as C
    src = np.asarray(src)
    if src.dtype != np.uint8 or src.ndim != 3 or src.shape[2] != 3:
        raise ValueError("denoise: expected an H x W x 3 uint8 image")
    if src.strides[1:] != (3, 1) or src.strides[0] < 0:
        src = np.ascontiguousarray(src)
    dst = np.empty(src.shape, np.uint8)
    lib = _lib.load()
    rc = lib.poppy_cuda_denoise(Settings.instance().cuda_device, src.ctypes.data_as(C.c_void_p), src.strides[0], src.shape[1],
                                src.shape[0], float(h), int(template_window_size), int(search_window_size),
                                dst.ctypes.data_as(C.c_void_p), dst.strides[0])
    if rc != 0:
        raise RuntimeError(f"poppy_cuda_denoise failed ({rc}): {lib.poppy_cuda_blur_margin_last_error().decode()}")
    return dst


def _optional(gabor2):
    return None if gabor2 is None else np.ascontiguousarray(gabor2)


def _pixel_format(pixel_format, w, h, fn):
    """pixel_format checked before anything is planned or rendered: "bgr", "i420" or "ffv1"; ValueError for any other
    format, or for I420 at an odd frame size (cv::cvtColor throws there too)."""
    if pixel_format not in ("bgr", "i420", "ffv1"):
        raise ValueError(f"{fn}: pixel_format must be 'bgr', 'i420' or 'ffv1', not {pixel_format!r}")
    if pixel_format == "i420" and (w % 2 or h % 2):
        raise ValueError(f"{fn}: I420 needs an even frame size, got {w}x{h}")
    return pixel_format


def _download(r, fmt, count):
    """Ring slots [0, count) of renderer r in pixel format fmt."""
    return {"bgr": r.download, "i420": r.download_i420, "ffv1": r.download_ffv1}[fmt](0, count)


class MatroskaWriter:
    """FFV1 packets (pixel_format="ffv1") into a Matroska file, the reference's default output (cv::VideoWriter with fourcc
    FFV1): write(packet) appends one frame, close() finishes the file. cv2.VideoCapture plays it back."""

    def __init__(self, path, width, height, fps=30):
        self._lib = _lib.load()
        fps = Fraction(fps).limit_denominator(1001000)
        self._m = C.c_void_p()
        if self._lib.poppy_host_mkv_open(C.byref(self._m), os.fsencode(path), int(width), int(height), fps.numerator,
                                         fps.denominator) != 0:
            raise OSError(f"cannot write a {width}x{height} Matroska file at {path!r}")

    def write(self, packet):
        if not self._m:
            raise ValueError("MatroskaWriter is closed")
        if self._lib.poppy_host_mkv_write(self._m, bytes(packet), len(packet)) != 0:
            raise OSError("MatroskaWriter: write failed")

    def close(self):
        if self._m:
            m, self._m = self._m, C.c_void_p()
            if self._lib.poppy_host_mkv_close(m) != 0:
                raise OSError("MatroskaWriter: close failed")

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def morph_sequence(corrected1, corrected2, gabor2, src_points1, src_points2, writer=None, number_of_frames=None,
                   threads=0, pixel_format="bgr"):
    """Chain mode: frame j = morph_images(previous frame, previous morphed points, shape = color = 1/(N-j)).
    Returns the frames (N x H x W x 3, N x 3H/2 x W with pixel_format="i420", or a list of N FFV1 packets with
    pixel_format="ffv1") and calls writer.write(frame) per frame
    if a writer is given. gabor2=None: derived on the GPU from corrected2."""
    n_frames = int(number_of_frames if number_of_frames is not None else Settings.instance().number_of_frames)
    h, w = corrected1.shape[:2]
    fmt = _pixel_format(pixel_format, w, h, "morph_sequence")
    ratio = np.array([host.chain_ratio(j, n_frames) for j in range(n_frames)], np.float64)
    plan = host.SequencePlan(src_points1, src_points2, w, h, ratio.astype(np.float32), chain=True, threads=threads)
    try:
        r = _renderer(w, h, plan.n, plan.max_triangles, n_frames)
        r.set_pair(np.ascontiguousarray(corrected1), np.ascontiguousarray(corrected2), _optional(gabor2))
        r.set_points(src_points1, src_points2)
        r.render(ratio.astype(np.float32), ratio, plan.tri_idx, plan.tri_offsets, chain=True)
        frames = _download(r, fmt, n_frames)
    finally:
        plan.close()
    if writer is not None:
        for f in frames:
            writer.write(f)
    return frames


def render_phases(corrected1, corrected2, gabor2, src_points1, src_points2, phases, mask_ratios=None, threads=0,
                  pixel_format="bgr"):
    """Direct mode: independent phases s_k of one pair, shape = s_k and mask = mask_ratios[k] (default s_k).
    Returns N x H x W x 3 frames, N x 3H/2 x W with pixel_format="i420", or a list of N FFV1 packets with
    pixel_format="ffv1". gabor2=None: derived on the GPU from corrected2."""
    h, w = corrected1.shape[:2]
    fmt = _pixel_format(pixel_format, w, h, "render_phases")
    phases = np.ascontiguousarray(phases, np.float32)
    masks = np.ascontiguousarray(mask_ratios if mask_ratios is not None else phases.astype(np.float64), np.float64)
    plan = host.SequencePlan(src_points1, src_points2, w, h, phases, chain=False, threads=threads)
    try:
        r = _renderer(w, h, plan.n, plan.max_triangles, len(phases))
        r.set_pair(np.ascontiguousarray(corrected1), np.ascontiguousarray(corrected2), _optional(gabor2))
        r.set_points(src_points1, src_points2)
        r.render(phases, masks, plan.tri_idx, plan.tri_offsets, chain=False)
        return _download(r, fmt, len(phases))
    finally:
        plan.close()


def interleave_segment_plans(plans, n_steps):
    """Triangle lists of chain plans in the step-major order of MorphRenderer.render_segments: entry j * K + s is step j of
    segment s. Returns (tri_idx, tri_offsets)."""
    K = len(plans)
    counts = np.array([[p.tri_offsets[j + 1] - p.tri_offsets[j] for p in plans] for j in range(n_steps)], np.int64).reshape(-1)
    offsets = np.zeros(n_steps * K + 1, np.int32)
    np.cumsum(counts, out=offsets[1:])
    parts = [plans[s].triangles(j) for j in range(n_steps) for s in range(K)]
    tri = np.concatenate(parts).astype(np.int32, copy=False) if parts else np.zeros((0, 3), np.int32)
    return tri.reshape(-1, 3), offsets


# ring memory one morph_segments batch may take: segments that do not fit are rendered in further batches
_SEGMENT_RING_BYTES = 8 << 30


def _check_devices(devices):
    """The device list of morph_segments, checked before anything is planned or rendered."""
    devices = [operator.index(d) for d in devices]
    if not devices:
        raise ValueError("morph_segments: the device list is empty")
    if any(d < 0 for d in devices):
        raise ValueError(f"morph_segments: negative device index in {devices}")
    if len(set(devices)) != len(devices):
        raise ValueError(f"morph_segments: a device is listed twice in {devices}")
    n = device_count()
    if n <= 0:
        raise RuntimeError("morph_segments: no CUDA device: the morph renderer has no CPU fallback")
    if any(d >= n for d in devices):
        raise ValueError(f"morph_segments: device index out of [0, {n}) in {devices}")
    return devices


def _render_segment_range(r, segments, plans, lo, hi, per_batch, shape, ratio, frames, fmt, stop=None):
    """Segments [lo, hi) on renderer r, per_batch at a time, downloaded (as BGR, I420 or FFV1 packets) into frames[lo:hi]."""
    n_frames = len(shape)
    for b0 in range(lo, hi, per_batch):
        if stop is not None and stop.is_set():
            return
        batch = range(b0, min(hi, b0 + per_batch))
        r.set_segments(len(batch), n_frames)
        for i, s in enumerate(batch):
            c1, c2, g2, p1, p2 = segments[s]
            r.set_segment(i, np.ascontiguousarray(c1), np.ascontiguousarray(c2), _optional(g2), np.reshape(p1, (-1, 2)),
                          np.reshape(p2, (-1, 2)))
        tri, offs = interleave_segment_plans([plans[s] for s in batch], n_frames)
        r.render_segments(0, shape, ratio, tri, offs)
        if fmt == "ffv1":
            packets = r.download_ffv1(0, len(batch) * n_frames)
            for i in range(len(batch)):
                frames[b0 + i] = packets[i * n_frames:(i + 1) * n_frames]
        else:
            download = r.download_i420 if fmt == "i420" else r.download
            download(0, len(batch) * n_frames, out=frames[b0:b0 + len(batch)].reshape((-1,) + frames.shape[2:]))


def morph_segments(segments, number_of_frames=None, writer=None, threads=0, devices=None, pixel_format="bgr"):
    """The segments of a multi-image sequence: segments[i] = (corrected1, corrected2, gabor2 or None, pts1, pts2) of one
    consecutive pair, all of one frame size. Each is the chain morph_sequence renders, and they are rendered together.
    Returns the frames as a (K, N, H, W, 3) array, (K, N, 3H/2, W) with pixel_format="i420", or K lists of N packets (bytes)
    with pixel_format="ffv1", and calls writer.write(frame)
    in the reference's order: the N frames of segment 0, then those of segment 1, and so on (one video, as run() writes it).

    devices=None renders on Settings.cuda_device. devices=[d0, d1, ...] shards the K segments over the first
    G = min(len(devices), K) of those GPUs: devices[g] renders the contiguous range shard.phase_range(g, G, K) on its own
    renderer and Python thread, each as the single-device call does with its own ring budget. The result and the writer
    calls are the same as with one device. An empty list, a duplicate, a negative index or an index >= device_count()
    raises ValueError, and RuntimeError is raised without a GPU, before anything is planned or rendered."""
    n_frames = int(number_of_frames if number_of_frames is not None else Settings.instance().number_of_frames)
    K = len(segments)
    h, w = segments[0][0].shape[:2] if K else (0, 0)
    fmt = _pixel_format(pixel_format, w, h, "morph_segments")
    if devices is not None:
        devices = _check_devices(devices)
    if K == 0:
        raise ValueError("morph_segments: no segments")
    for c1, c2, _, p1, p2 in segments:
        if c1.shape[:2] != (h, w) or c2.shape[:2] != (h, w):
            raise ValueError("morph_segments: all segments must have the same frame size")
        if np.shape(p1) != np.shape(p2):
            raise ValueError("morph_segments: point sets differ in size")
    ratio = np.array([host.chain_ratio(j, n_frames) for j in range(n_frames)], np.float64)
    shape = ratio.astype(np.float32)
    plans = [host.SequencePlan(np.reshape(p1, (-1, 2)), np.reshape(p2, (-1, 2)), w, h, shape, chain=True, threads=threads)
             for _, _, _, p1, p2 in segments]
    if fmt == "ffv1":
        frames = [None] * K
    else:
        frames = np.empty((K, n_frames, h * 3 // 2, w) if fmt == "i420" else (K, n_frames, h, w, 3), np.uint8)
    n_max, tri_max = max(p.n for p in plans), max(p.max_triangles for p in plans)

    def per_batch(count):
        return max(1, min(count, _SEGMENT_RING_BYTES // (n_frames * w * h * 3)))

    try:
        if devices is None:
            r = _renderer(w, h, n_max, tri_max, per_batch(K) * n_frames)
            _render_segment_range(r, segments, plans, 0, K, per_batch(K), shape, ratio, frames, fmt)
        else:
            G = min(len(devices), K)
            stop, errors = threading.Event(), []

            def run(g):
                try:
                    lo, hi = shard.phase_range(g, G, K)
                    d, b = devices[g], per_batch(hi - lo)
                    r = _renderer(w, h, n_max, tri_max, b * n_frames) if d == Settings.instance().cuda_device \
                        else _device_renderer(d, w, h, n_max, tri_max, b * n_frames)
                    _render_segment_range(r, segments, plans, lo, hi, b, shape, ratio, frames, fmt, stop)
                except BaseException as e:      # the other devices stop before their next batch; re-raised below
                    errors.append(e)
                    stop.set()
            workers = [threading.Thread(target=run, args=(g,)) for g in range(G)]
            for t in workers:
                t.start()
            for t in workers:
                t.join()
            if errors:
                raise errors[0]
    finally:
        for p in plans:
            p.close()
    if writer is not None:
        for seg in frames:
            for f in seg:
                writer.write(f)
    return frames
