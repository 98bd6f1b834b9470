"""TEST INFRASTRUCTURE ONLY — ctypes binding of oracle/liboracle.so, the CPU restatement of the morph path
(oracle/poppy_oracle.cpp). Same stage-dump layout as oracle/ref.py so the two can be compared field by field.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this module."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from .ref import Stages, _StageDump, _f32, _p, _u8, _cn

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liboracle.so")
_lib = None


def build(force: bool = False):
    src = os.path.join(_HERE, "poppy_oracle.cpp")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(LIB_PATH)
    return _lib


def morph_points(pts1, pts2, s, w, h):
    pts1, pts2 = _f32(pts1), _f32(pts2)
    out = np.empty_like(pts1)
    lib().poppy_oracle_morph_points(_p(pts1), _p(pts2), pts1.shape[0], C.c_float(s), w, h, _p(out))
    return out


def fill_triangles(w, h, tri_xy):
    tri_xy = np.ascontiguousarray(tri_xy, dtype=np.int32).reshape(-1, 6)
    img = np.zeros((h, w), np.int32)
    lib().poppy_oracle_fill_triangles(_p(img), w, h, _p(tri_xy), tri_xy.shape[0])
    return img


def triangle_matrices(tri1_xy, tri2_xy, r):
    a = np.ascontiguousarray(tri1_xy, dtype=np.int32).reshape(-1, 6)
    b = np.ascontiguousarray(tri2_xy, dtype=np.int32).reshape(-1, 6)
    t = a.shape[0]
    outs = [np.empty((t, 3, 3), np.float32) for _ in range(5)]
    lib().poppy_oracle_triangle_matrices(_p(a), _p(b), t, C.c_float(r), *[_p(o) for o in outs])
    return outs  # H, M1, M2, inv(M1), inv(M2)


def remap_u8c3(src, mapx, mapy):
    src, mapx, mapy = _u8(src), _f32(mapx), _f32(mapy)
    h, w = src.shape[:2]
    dh, dw = mapx.shape
    dst = np.empty((dh, dw, 3), np.uint8)
    lib().poppy_oracle_remap(_p(src), w, h, _p(mapx), _p(mapy), dw, dh, _p(dst))
    return dst


def mask(gabor2, mask_ratio):
    gabor2 = _f32(gabor2)
    h, w = gabor2.shape[:2]
    out = np.empty((h, w), np.float32)
    lib().poppy_oracle_mask(_p(gabor2), w, h, C.c_double(mask_ratio), _p(out))
    return out


def pyr_down(src, dsize=None):
    src = _f32(src)
    h, w = src.shape[:2]
    dw, dh = dsize if dsize else ((w + 1) // 2, (h + 1) // 2)
    dst = np.empty((dh, dw) + src.shape[2:], np.float32)
    lib().poppy_oracle_pyr_down(_p(src), w, h, _cn(src), _p(dst), dw, dh)
    return dst


def pyr_up(src, dsize):
    src = _f32(src)
    h, w = src.shape[:2]
    dw, dh = dsize
    dst = np.empty((dh, dw) + src.shape[2:], np.float32)
    lib().poppy_oracle_pyr_up(_p(src), w, h, _cn(src), _p(dst), dw, dh)
    return dst


def lap_blend(l, r, m, levels):
    l, r, m = _f32(l), _f32(r), _f32(m)
    h, w = m.shape
    out = np.empty((h, w, 3), np.float32)
    lib().poppy_oracle_lap_blend(_p(l), _p(r), _p(m), w, h, int(levels), _p(out))
    return out


def gaussian9(src):
    src = _f32(src)
    h, w = src.shape[:2]
    out = np.empty_like(src)
    lib().poppy_oracle_gaussian9(_p(src), w, h, _cn(src), _p(out))
    return out


def median3(src):
    src = _f32(src)
    h, w = src.shape[:2]
    out = np.empty_like(src)
    lib().poppy_oracle_median3(_p(src), w, h, _cn(src), _p(out))
    return out


def unsharp(src, amount, threshold):
    src = _f32(src)
    h, w = src.shape[:2]
    out = np.empty_like(src)
    lib().poppy_oracle_unsharp(_p(src), w, h, C.c_float(amount), C.c_float(threshold), _p(out))
    return out


def morph_frame(bgr1, bgr2, gabor2, pts1, pts2, tri_idx, shape, mask_ratio, levels) -> Stages:
    """One frame of the path (reference src/algo.cpp:178-265) for a given triangle index list."""
    bgr1, bgr2, gabor2, pts1, pts2 = _u8(bgr1), _u8(bgr2), _f32(gabor2), _f32(pts1), _f32(pts2)
    tri_idx = np.ascontiguousarray(tri_idx, dtype=np.int32).reshape(-1, 3)
    h, w = bgr1.shape[:2]
    n, t = pts1.shape[0], tri_idx.shape[0]
    f = np.float32
    out = dict(
        morphed_points=np.empty((n, 2), f), tri_idx=np.empty((t, 3), np.int32), tri_map=np.empty((h, w), np.int32),
        hom=np.empty((t, 3, 3), f), m1=np.empty((t, 3, 3), f), m2=np.empty((t, 3, 3), f),
        mapx1=np.empty((h, w), f), mapy1=np.empty((h, w), f), mapx2=np.empty((h, w), f), mapy2=np.empty((h, w), f),
        warped1=np.empty((h, w, 3), np.uint8), warped2=np.empty((h, w, 3), np.uint8), mask=np.empty((h, w), f),
        lap_blend=np.empty((h, w, 3), f), dst=np.empty((h, w, 3), np.uint8))
    d = _StageDump()
    for k, v in out.items():
        setattr(d, k, v.ctypes.data)
    d.max_tri = t
    lib().poppy_oracle_morph_frame(w, h, _p(bgr1), _p(bgr2), _p(gabor2), _p(pts1), _p(pts2), n, _p(tri_idx), t,
                                   C.c_double(shape), C.c_double(mask_ratio), int(levels), C.byref(d))
    return Stages(**out)


# The entry points of oracle/ref.py with the same signatures: the frame path above around the host topology stage
# (poppy_b200.host, pinned to cv::Subdiv2D by tests/golden/topology.npz). Tests compare against these where the
# reference library is not built.
def stages(bgr1, bgr2, gabor2, pts1, pts2, shape, mask, levels) -> Stages:
    from poppy_b200 import host
    h, w = np.shape(bgr1)[:2]
    tri = host.triangulate(host.morph_points(pts1, pts2, shape, w, h), w, h)
    return morph_frame(bgr1, bgr2, gabor2, pts1, pts2, tri, shape, mask, levels)


def morph_images(bgr1, bgr2, gabor2, pts1, pts2, shape, mask, levels):
    st = stages(bgr1, bgr2, gabor2, pts1, pts2, shape, mask, levels)
    return st.dst, st.morphed_points


def chain(bgr1, bgr2, gabor2, pts1, pts2, n_frames, levels):
    """The frame-loop recurrence of reference src/poppy.hpp:177-243: frame j morphs frame j-1 and its points."""
    from poppy_b200 import host
    frames, points = [], []
    cur_img, cur_pts = bgr1, pts1
    for j in range(n_frames):
        s = host.chain_ratio(j, n_frames)
        cur_img, cur_pts = morph_images(cur_img, bgr2, gabor2, cur_pts, pts2, s, s, levels)
        frames.append(cur_img)
        points.append(cur_pts)
    return np.stack(frames), np.stack(points)
