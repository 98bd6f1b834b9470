"""Python mirror of the device boundary (include/poppy_cuda.h): a thin, allocation-free-per-call wrapper used by
the tests, bench.py and the batch driver. All arithmetic happens in libpoppy_cuda.so on the GPU."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import PoppyCudaError

STAGE_MORPHED_POINTS, STAGE_TRI_MAP, STAGE_INV_M1, STAGE_INV_M2 = 0, 1, 2, 3
STAGE_WARPED1, STAGE_WARPED2, STAGE_MASK, STAGE_LAP_BLEND = 4, 5, 6, 7
STAGE_MASK_BASIS = 8          # of the current pair: m2 = 1 - gray(gabor2), whatever `frame` says


def device_count() -> int:
    return int(_lib.load().poppy_cuda_device_count())


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class MorphRenderer:
    """One context per GPU (poppy_cuda_create). Holds the image pair, the point sets and the HBM frame ring."""

    def __init__(self, width, height, pyramid_levels, max_points, max_triangles, max_batch_frames, device=0,
                 keep_stages=False, chunk_frames=None, stage_timing=False):
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        rc = self._lib.poppy_cuda_create(C.byref(self._ctx), device, width, height, pyramid_levels, max_points,
                                         max_triangles, max_batch_frames)
        if rc != 0:
            raise PoppyCudaError(rc, self._lib.poppy_cuda_last_error(None).decode())
        self.width, self.height, self.levels = width, height, pyramid_levels
        self.max_points, self.max_triangles, self.max_batch_frames = max_points, max_triangles, max_batch_frames
        self.n_points = 0
        self.n_segments, self.segment_window, self._segment_n = 0, 0, []
        if keep_stages:
            self._check(self._lib.poppy_cuda_set_keep_stages(self._ctx, 1))
        if chunk_frames:
            self._check(self._lib.poppy_cuda_set_chunk_frames(self._ctx, int(chunk_frames)))
        if stage_timing:
            self._check(self._lib.poppy_cuda_set_stage_timing(self._ctx, 1))

    def set_unsharp_mode(self, mode: int):
        """0: adaptive; 1: dense (exact blur + median on every pixel); 2: calm route (exact path only on flagged chunks)."""
        self._check(self._lib.poppy_cuda_set_unsharp_mode(self._ctx, int(mode)))

    def unsharp_stats(self) -> tuple:
        """(strip chunks that took the exact unsharp path, all strip chunks) since the last call."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._check(self._lib.poppy_cuda_unsharp_stats(self._ctx, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def set_tile_list_capacity(self, entries_per_frame: int):
        self._check(self._lib.poppy_cuda_set_tile_list_capacity(self._ctx, int(entries_per_frame)))

    # -- plumbing ------------------------------------------------------------------------------------------------
    def _check(self, rc):
        if rc < 0:
            raise PoppyCudaError(rc, self._lib.poppy_cuda_last_error(self._ctx).decode())
        return rc

    def close(self):
        if self._ctx:
            self._lib.poppy_cuda_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- inputs --------------------------------------------------------------------------------------------------
    def set_pair(self, bgr1: np.ndarray, bgr2: np.ndarray, gabor2: np.ndarray | None = None):
        """corrected1, corrected2 (HxWx3 uint8) and gabor2 (HxWx3 float32) of morph_images (algo.cpp:178).
        gabor2=None: derived on the GPU from corrected2 as poppy::morph() derives it (src/poppy.hpp:119-122), so only the
        two 8-bit images are uploaded."""
        images = ((bgr1, np.uint8), (bgr2, np.uint8)) + (() if gabor2 is None else ((gabor2, np.float32),))
        for a, dt in images:
            if a.dtype != dt or a.shape[:2] != (self.height, self.width) or a.shape[2] != 3 or a.strides[2] != a.itemsize \
                    or a.strides[1] != 3 * a.itemsize:
                raise ValueError("images must be HxWx3, pixel-contiguous, uint8 (bgr) / float32 (gabor2)")
        gab, gstep = (None, 0) if gabor2 is None else (_ptr(gabor2), gabor2.strides[0])
        self._check(self._lib.poppy_cuda_set_pair(self._ctx, _ptr(bgr1), bgr1.strides[0], _ptr(bgr2), bgr2.strides[0],
                                                  gab, gstep))

    def set_points(self, pts1: np.ndarray, pts2: np.ndarray):
        pts1 = np.ascontiguousarray(pts1, np.float32)
        pts2 = np.ascontiguousarray(pts2, np.float32)
        if pts1.shape != pts2.shape or pts1.ndim != 2 or pts1.shape[1] != 2:
            raise ValueError("point sets must both be N x 2")
        self._check(self._lib.poppy_cuda_set_points(self._ctx, _ptr(pts1), _ptr(pts2), pts1.shape[0]))
        self.n_points = pts1.shape[0]

    # -- render --------------------------------------------------------------------------------------------------
    def render(self, shape_ratio, mask_ratio, tri_idx, tri_offsets, chain=False, first_slot=0):
        """Render len(shape_ratio) frames into ring slots first_slot.. . tri_idx: (sum T_f) x 3 int32, tri_offsets: F+1."""
        shape_ratio = np.ascontiguousarray(shape_ratio, np.float32)
        mask_ratio = np.ascontiguousarray(mask_ratio, np.float64)
        tri_idx = np.ascontiguousarray(tri_idx, np.int32).reshape(-1, 3)
        tri_offsets = np.ascontiguousarray(tri_offsets, np.int32)
        n = shape_ratio.shape[0]
        if mask_ratio.shape[0] != n or tri_offsets.shape[0] != n + 1 or tri_offsets[-1] != tri_idx.shape[0]:
            raise ValueError("inconsistent frame / triangle-offset arrays")
        self._check(self._lib.poppy_cuda_render_range(self._ctx, int(first_slot), n, _ptr(shape_ratio), _ptr(mask_ratio),
                                                      _ptr(tri_idx), _ptr(tri_offsets), 1 if chain else 0))
        return n

    def set_plan(self, tri_idx, tri_offsets):
        """Keep the triangle lists of a whole sequence resident in HBM (validated once); see render_planned."""
        tri_idx = np.ascontiguousarray(tri_idx, np.int32).reshape(-1, 3)
        tri_offsets = np.ascontiguousarray(tri_offsets, np.int32)
        if tri_offsets[-1] - tri_offsets[0] > tri_idx.shape[0] - tri_offsets[0]:
            raise ValueError("inconsistent triangle-offset array")
        self._check(self._lib.poppy_cuda_set_plan(self._ctx, _ptr(tri_idx), _ptr(tri_offsets), tri_offsets.shape[0] - 1))

    def render_planned(self, shape_ratio, mask_ratio, plan_first=0, chain=False, first_slot=0):
        """Render len(shape_ratio) frames whose triangle lists are frames plan_first.. of the resident plan."""
        shape_ratio = np.ascontiguousarray(shape_ratio, np.float32)
        mask_ratio = np.ascontiguousarray(mask_ratio, np.float64)
        n = shape_ratio.shape[0]
        if mask_ratio.shape[0] != n:
            raise ValueError("inconsistent frame arrays")
        self._check(self._lib.poppy_cuda_render_planned(self._ctx, int(first_slot), int(plan_first), n, _ptr(shape_ratio),
                                                        _ptr(mask_ratio), 1 if chain else 0))
        return n

    # -- segments of a multi-image sequence (poppy_cuda_set_segments) -------------------------------------------------
    def set_segments(self, n_segments: int, window: int):
        """Room for n_segments independent chains; step j of segment s lands in ring slot s * window + j % window."""
        self._check(self._lib.poppy_cuda_set_segments(self._ctx, int(n_segments), int(window)))
        self.n_segments, self.segment_window = int(n_segments), int(window)
        self._segment_n = [0] * self.n_segments

    def set_segment(self, s: int, bgr1: np.ndarray, bgr2: np.ndarray, gabor2: np.ndarray | None, pts1, pts2):
        """corrected1, corrected2, gabor2 (None: derived on the GPU) and the point sets of segment s."""
        images = ((bgr1, np.uint8), (bgr2, np.uint8)) + (() if gabor2 is None else ((gabor2, np.float32),))
        for a, dt in images:
            if a.dtype != dt or a.shape[:2] != (self.height, self.width) or a.ndim != 3 or a.shape[2] != 3 \
                    or a.strides[2] != a.itemsize or a.strides[1] != 3 * a.itemsize:
                raise ValueError("images must be HxWx3, pixel-contiguous, uint8 (bgr) / float32 (gabor2)")
        pts1 = np.ascontiguousarray(pts1, np.float32).reshape(-1, 2)
        pts2 = np.ascontiguousarray(pts2, np.float32).reshape(-1, 2)
        if pts1.shape != pts2.shape:
            raise ValueError("point sets must both be N x 2")
        gab, gstep = (None, 0) if gabor2 is None else (_ptr(gabor2), gabor2.strides[0])
        self._check(self._lib.poppy_cuda_set_segment(self._ctx, int(s), _ptr(bgr1), bgr1.strides[0], _ptr(bgr2), bgr2.strides[0],
                                                     gab, gstep, _ptr(pts1), _ptr(pts2), pts1.shape[0]))
        self._segment_n[s] = pts1.shape[0]

    def render_segments(self, first_step, shape_ratio, mask_ratio, tri_idx, tri_offsets):
        """Steps first_step .. first_step + len(shape_ratio) - 1 of every segment. tri_offsets: n_steps * K + 1 entries, the
        list of step first_step + r of segment s being entry r * K + s."""
        shape_ratio = np.ascontiguousarray(shape_ratio, np.float32)
        mask_ratio = np.ascontiguousarray(mask_ratio, np.float64)
        tri_idx = np.ascontiguousarray(tri_idx, np.int32).reshape(-1, 3)
        tri_offsets = np.ascontiguousarray(tri_offsets, np.int32)
        n = shape_ratio.shape[0]
        if mask_ratio.shape[0] != n or tri_offsets.shape[0] != n * self.n_segments + 1 or tri_offsets[-1] > tri_idx.shape[0]:
            raise ValueError("inconsistent step / triangle-offset arrays")
        self._check(self._lib.poppy_cuda_render_segments(self._ctx, int(first_step), n, _ptr(shape_ratio), _ptr(mask_ratio),
                                                         _ptr(tri_idx), _ptr(tri_offsets)))
        return n

    def segment_slot(self, s: int, step: int) -> int:
        """Ring slot of step `step` of segment s."""
        return int(s) * self.segment_window + int(step) % self.segment_window

    def segment_points(self, s: int, step: int) -> np.ndarray:
        """morphedPoints of step `step` of segment s (its own n x 2), while the step is in the segment's window."""
        out = np.empty((self._segment_n[s] if 0 <= s < len(self._segment_n) else 0, 2), np.float32)
        self._check(self._lib.poppy_cuda_get_segment_points(self._ctx, int(s), int(step), _ptr(out)))
        return out

    def download(self, first, count, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty((count, self.height, self.width, 3), np.uint8)
        if out.dtype != np.uint8 or out.shape != (count, self.height, self.width, 3) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous (count, H, W, 3) uint8 array")
        self._check(self._lib.poppy_cuda_download(self._ctx, first, count, _ptr(out), out.strides[1], out.strides[0]))
        self.sync()
        return out

    def download_i420(self, first, count, out: np.ndarray | None = None) -> np.ndarray:
        """Frames [first, first + count) as I420, converted on the GPU: (count, H * 3 // 2, W) uint8, per frame what
        cv2.cvtColor(frame, cv2.COLOR_BGR2YUV_I420) returns for the BGR frame (Y rows, then the U and V planes). Needs an even
        frame size."""
        shape = (count, self.height * 3 // 2, self.width)
        if out is None:
            out = np.empty(shape, np.uint8)
        if out.dtype != np.uint8 or out.shape != shape or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous (count, H * 3 // 2, W) uint8 array")
        self._check(self._lib.poppy_cuda_download_i420(self._ctx, first, count, _ptr(out), out.strides[0]))
        self.sync()
        return out

    def download_ffv1(self, first, count) -> list[bytes]:
        """Frames [first, first + count) as lossless FFV1 packets encoded on the GPU, one bytes object per frame; a
        MatroskaWriter of this frame size (api.py) stores them as the .mkv cv::VideoWriter with fourcc FFV1 writes."""
        sizes = np.zeros(count, np.uint32)
        cap = count * (self.width * self.height * 3 + 65536)
        while True:
            out = np.empty(cap, np.uint8)
            rc = self._lib.poppy_cuda_download_ffv1(self._ctx, first, count, _ptr(out), cap,
                                                    sizes.ctypes.data_as(C.POINTER(C.c_uint32)))
            need = int(sizes.sum(dtype=np.uint64))
            if rc == 0 or not (rc == -2 and need > cap):
                break
            cap = need                            # packets larger than their raw frames (noise): encode again at their size
        self._check(rc)
        ends = np.cumsum(sizes, dtype=np.int64)
        data = out[:need].tobytes()
        return [data[e - n:e] for e, n in zip(ends.tolist(), sizes.tolist())]

    def download_async(self, first, count, host_ptr, step, frame_stride):
        """Raw-pointer download into caller-owned (pinned) memory; poppy_cuda_sync() before reading."""
        self._check(self._lib.poppy_cuda_download(self._ctx, first, count, C.c_void_p(host_ptr), step, frame_stride))

    def morphed_points(self, frame) -> np.ndarray:
        out = np.empty((self.n_points, 2), np.float32)
        self._check(self._lib.poppy_cuda_get_morphed_points(self._ctx, frame, _ptr(out)))
        return out

    def checksum(self, first, count) -> int:
        v = C.c_uint64(0)
        self._check(self._lib.poppy_cuda_checksum(self._ctx, first, count, C.byref(v)))
        return int(v.value)

    def sync(self):
        self._check(self._lib.poppy_cuda_sync(self._ctx))

    def stream(self) -> int:
        s = C.c_void_p()
        self._check(self._lib.poppy_cuda_get_stream(self._ctx, C.byref(s)))
        return int(s.value or 0)

    def last_render_ms(self) -> float:
        ms = C.c_float(0)
        self._check(self._lib.poppy_cuda_last_render_ms(self._ctx, C.byref(ms)))
        return float(ms.value)

    def launch_count(self) -> int:
        v = C.c_uint64(0)
        self._check(self._lib.poppy_cuda_launch_count(self._ctx, C.byref(v)))
        return int(v.value)

    def stage_times(self) -> dict:
        cap = 16
        names = (C.c_char_p * cap)()
        ms = (C.c_float * cap)()
        cnt = (C.c_uint64 * cap)()
        n = self._check(self._lib.poppy_cuda_stage_times(self._ctx, names, ms, cnt, cap))
        return {names[i].decode(): {"ms": float(ms[i]), "launches": int(cnt[i])} for i in range(min(n, cap))}

    def frame_device_ptr(self, frame):
        p, b = C.c_void_p(), C.c_size_t()
        self._check(self._lib.poppy_cuda_frame_device_ptr(self._ctx, frame, C.byref(p), C.byref(b)))
        return int(p.value), int(b.value)

    # -- stage dumps (keep_stages contexts) ------------------------------------------------------------------------
    def read_stage(self, stage, frame, n_tri=None) -> np.ndarray:
        h, w = self.height, self.width
        if stage == STAGE_MORPHED_POINTS:
            out = np.empty((self.n_points, 2), np.float32)
        elif stage == STAGE_TRI_MAP:
            out = np.empty((h, w), np.int32)
        elif stage in (STAGE_INV_M1, STAGE_INV_M2):
            out = np.empty((n_tri, 3, 3), np.float32)
        elif stage in (STAGE_WARPED1, STAGE_WARPED2):
            out = np.empty((h, w, 3), np.uint8)
        elif stage in (STAGE_MASK, STAGE_MASK_BASIS):
            out = np.empty((h, w), np.float32)
        elif stage == STAGE_LAP_BLEND:
            out = np.empty((h, w, 3), np.float32)
        else:
            raise ValueError("unknown stage")
        self._check(self._lib.poppy_cuda_debug_read(self._ctx, stage, frame, _ptr(out), out.nbytes))
        return out
