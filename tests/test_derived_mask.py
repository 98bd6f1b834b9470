"""The mask basis derived on the GPU from corrected2 (set_pair without gabor2, set_image selector 3).

poppy::morph() computes gabor2 = gabor_filter(corrected2 converted with convertTo(CV_32F, 1/255)) before its frame loop
(reference src/poppy.hpp:119-122), and the renderer only ever uses m2 = 1 - gray(gabor2) (src/algo.cpp:250-252).
k_gabor_mask_basis fuses the two: the tests below hold it bit for bit to the two-step route (poppy_cuda_gabor_filter, then
set_pair with its output), and hold the whole chains of the reference pipeline's configs 1 and 2 to their recorded frames
with no gabor2 passed at all. The CPU tests pin the conversion itself: a multiplication by float(1/255), not a division."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import margin
from tests.util import bits_differ, frame_checksum

HERE = os.path.dirname(os.path.abspath(__file__))
FULL = os.path.join(HERE, "golden", "full")
INV255 = np.float32(1 / 255.0)
_WRITE = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_size_t)


def _golden(config):
    return np.load(os.path.join(FULL, f"c{config}.npz"))


def _unit(u8):
    """convertTo(CV_32F, 1/255): float(v) * float(1/255.0), one rounding."""
    return u8.astype(np.float32) * INV255


# ---- CPU: which conversion the reference pipeline applied ---------------------------------------------------------------

def test_gabor2_of_the_reference_pipeline_is_the_filter_of_corrected2_times_one_255th():
    g = _golden(2)
    assert bits_differ(margin.gabor_filter(_unit(g["corrected2"])), g["gabor2"]) == 0
    g = _golden(1)
    # the reference's DFT leaves ~1e-14 of round-off where the exact response is 0; the direct sum does not
    assert float(np.abs(margin.gabor_filter(_unit(g["corrected2"])) - g["gabor2"]).max()) <= 1e-13


def test_dividing_by_255_does_not_give_the_recorded_gabor2():
    """Why the kernel multiplies: u8 / 255 rounds 126 of the 256 byte values differently, and the filter of that input
    misses the recorded gabor2 of config 2 in tens of thousands of values."""
    v = np.arange(256, dtype=np.float32)
    assert int((v * INV255 != v / np.float32(255)).sum()) == 126
    g = _golden(2)
    assert bits_differ(margin.gabor_filter(g["corrected2"].astype(np.float32) / np.float32(255)), g["gabor2"]) > 1000


def test_stage_enum_matches_the_header():
    from poppy_b200 import renderer
    text = open(os.path.join(os.path.dirname(HERE), "include", "poppy_cuda.h")).read()
    assert "POPPY_STAGE_MASK_BASIS = 8" in text and renderer.STAGE_MASK_BASIS == 8


# ---- GPU ----------------------------------------------------------------------------------------------------------------

def _image(kind, w, h, seed):
    from poppy_b200 import synth
    if kind == "random":
        return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "noise":
        return synth.noise_image(w, h, seed)
    return synth.block_inputs(w, h, 8, seed=seed).bgr2


def _explicit_gabor2(c2):
    from poppy_b200 import api
    return api.gabor_filter(_unit(c2))


def _render_basis(c1, c2, gabor2, levels=4):
    """One frame (no points: the blend of the unwarped pair) in a fresh keep_stages context; returns (basis, frame)."""
    from poppy_b200.renderer import STAGE_MASK_BASIS, MorphRenderer
    h, w = c1.shape[:2]
    with MorphRenderer(w, h, levels, 8, 8, 1, keep_stages=True) as r:
        r.set_pair(c1, c2, gabor2)
        r.set_points(np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32))
        r.render([0.4], [0.4], np.zeros((0, 3), np.int32), [0, 0])
        return r.read_stage(STAGE_MASK_BASIS, 0), r.download(0, 1)[0]


BASIS_CASES = [(1, 40, "random"), (40, 1, "random"), (7, 9, "random"), (13, 13, "random"), (61, 45, "random"),
               (61, 45, "noise"), (61, 45, "blocks"), (512, 512, "noise"), (512, 512, "blocks"), (1920, 1080, "noise"),
               (1920, 1080, "blocks"), (3840, 2160, "noise")]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,kind", BASIS_CASES)
def test_derived_basis_is_bit_identical_to_the_filter_then_upload_route(native_lib, w, h, kind):
    c1, c2 = _image(kind, w, h, 2 * w + h), _image(kind, w, h, 3 * w + h + 1)
    want_basis, want_frame = _render_basis(c1, c2, _explicit_gabor2(c2))
    got_basis, got_frame = _render_basis(c1, c2, None)
    assert bits_differ(got_basis, want_basis) == 0
    assert bits_differ(got_frame, want_frame) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("config", [1, 2])
def test_reference_chain_without_gabor2(native_lib, config):
    """The reference pipeline's whole 60-frame chain at 64 levels with gabor2 derived on the device."""
    from poppy_b200 import api
    g = _golden(config)
    api.Settings.instance().pyramid_levels = int(g["levels"])
    try:
        frames = api.morph_sequence(g["corrected1"], g["corrected2"], None, g["pts1"], g["pts2"], number_of_frames=int(g["n_frames"]))
    finally:
        api.release()
    bad = [j for j in range(len(g["hashes"])) if frame_checksum(frames[j]) != int(g["hashes"][j])]
    assert not bad, f"config {config}: frames {bad[:8]} differ from the reference pipeline ({len(bad)} of {len(g['hashes'])})"
    for j, want in zip(g["kept"], g["kept_frames"]):
        assert bits_differ(frames[j], want) == 0, (config, int(j))


@pytest.mark.gpu
def test_cpp_shim_morph_sequence_derives_gabor2_when_given_null(native_lib):
    g = _golden(1)
    c1, c2 = np.ascontiguousarray(g["corrected1"]), np.ascontiguousarray(g["corrected2"])
    pts1, pts2 = np.ascontiguousarray(g["pts1"], np.float32), np.ascontiguousarray(g["pts2"], np.float32)
    h, w = c1.shape[:2]
    N = int(g["n_frames"])
    got = []

    def write(user, idx, bgr, fw, fh, step):
        f = np.ctypeslib.as_array(bgr, shape=(fh * step,)).reshape(fh, step)[:, :fw * 3].reshape(fh, fw, 3)
        got.append((idx, frame_checksum(f), f.copy() if idx in g["kept"] else None))

    p = lambda a: a.ctypes.data_as(C.c_void_p)
    cb = _WRITE(write)
    try:
        rc = native_lib.poppy_shim_morph_sequence(w, h, int(g["levels"]), p(c1), w * 3, p(c2), w * 3, None, 0, p(pts1), p(pts2),
                                                  len(pts1), N, cb, None)
        assert rc == 0, native_lib.poppy_host_last_error()
    finally:
        native_lib.poppy_shim_release()
    assert [i for i, _, _ in got] == list(range(N))
    assert [s for _, s, _ in got] == [int(v) for v in g["hashes"]]
    kept = {i: f for i, _, f in got if f is not None}
    for j, want in zip(g["kept"], g["kept_frames"]):
        assert bits_differ(kept[int(j)], want) == 0, int(j)


@pytest.mark.gpu
@pytest.mark.parametrize("unsharp_mode", [1, 2])
def test_direct_mode_frames_equal_with_derived_and_explicit_gabor2(native_lib, unsharp_mode):
    from poppy_b200 import api
    g = _golden(1)
    c1, c2, pts1, pts2 = g["corrected1"], g["corrected2"], g["pts1"], g["pts2"]
    h, w = c1.shape[:2]
    phases = np.array([0.0, 0.3, 0.5, 0.8, 1.0], np.float32)
    masks = np.array([0.0, 0.5, 1.0, 0.5, 0.0], np.float64)
    api.Settings.instance().pyramid_levels = 64
    try:
        out = []
        for gabor2 in (_explicit_gabor2(c2), None):
            # render_phases reuses the cached context when it is large enough: make it so, with the route under test
            r = api._renderer(w, h, len(pts1), 4 * len(pts1) + 64, len(phases))
            r.set_unsharp_mode(unsharp_mode)
            out.append(api.render_phases(c1, c2, gabor2, pts1, pts2, phases, masks))
            assert api._renderer(w, h, len(pts1), 4 * len(pts1) + 64, len(phases)) is r
    finally:
        api.release()
    assert bits_differ(out[1], out[0]) == 0


def _renderer_with(c1, c2, gabor2, inp, levels=5):
    from poppy_b200.renderer import MorphRenderer
    h, w = c1.shape[:2]
    r = MorphRenderer(w, h, levels, len(inp.pts1), 4 * len(inp.pts1) + 64, 2, keep_stages=True)
    r.set_pair(c1, c2, gabor2)
    r.set_points(inp.pts1, inp.pts2)
    return r


def _render_one(r, tri):
    from poppy_b200.renderer import STAGE_MASK_BASIS
    r.render([0.45], [0.6], tri, [0, len(tri)])
    return r.read_stage(STAGE_MASK_BASIS, 0), r.download(0, 1)[0]


@pytest.mark.gpu
def test_switching_between_explicit_and_derived_on_one_context(native_lib):
    from poppy_b200 import host, synth
    w, h = 230, 170
    inp = synth.make_inputs(w, h, 60, 6.0, seed=17)
    c1, c2 = inp.bgr1, inp.bgr2
    tri = host.triangulate(host.morph_points(inp.pts1, inp.pts2, 0.45, w, h), w, h, sequential=True)
    explicit = _explicit_gabor2(c2)
    fresh = {}
    for name, gab in (("explicit", explicit), ("derived", None), ("unrelated", inp.gabor2)):
        r = _renderer_with(c1, c2, gab, inp)
        fresh[name] = _render_one(r, tri)
        r.close()
    # equal routes, equal bits; the unrelated gabor2 really gives another basis
    assert bits_differ(fresh["explicit"][0], fresh["derived"][0]) == 0
    assert bits_differ(fresh["unrelated"][0], fresh["derived"][0]) > 0
    r = _renderer_with(c1, c2, explicit, inp)
    try:
        for name, gab in (("explicit", explicit), ("derived", None), ("unrelated", inp.gabor2), ("derived", None)):
            r.set_pair(c1, c2, gab)
            basis, frame = _render_one(r, tri)
            assert bits_differ(basis, fresh[name][0]) == 0 and bits_differ(frame, fresh[name][1]) == 0, name
        # set_image(1) leaves the basis alone; set_image(3) replaces it with the derived one
        r.set_pair(c1, c2, inp.gabor2)
        p = c2.ctypes.data_as(C.c_void_p)
        r._check(r._lib.poppy_cuda_set_image(r._ctx, 1, p, w * 3))
        assert bits_differ(_render_one(r, tri)[0], fresh["unrelated"][0]) == 0
        r._check(r._lib.poppy_cuda_set_image(r._ctx, 3, p, w * 3))
        basis, frame = _render_one(r, tri)
        assert bits_differ(basis, fresh["derived"][0]) == 0 and bits_differ(frame, fresh["derived"][1]) == 0
    finally:
        r.close()


@pytest.mark.gpu
def test_set_image_rejects_bad_selectors_pointers_and_strides(native_lib):
    from poppy_b200.renderer import STAGE_MASK_BASIS, MorphRenderer
    w, h = 40, 30
    img = np.zeros((h, w, 3), np.uint8)
    p = img.ctypes.data_as(C.c_void_p)
    with MorphRenderer(w, h, 3, 8, 8, 1, keep_stages=True) as r:
        lib, ctx = r._lib, r._ctx
        assert lib.poppy_cuda_debug_read(ctx, STAGE_MASK_BASIS, 0, np.empty((h, w), np.float32).ctypes.data_as(C.c_void_p),
                                         w * h * 4) == -4      # no basis yet
        for which in (4, -1):
            assert lib.poppy_cuda_set_image(ctx, which, p, w * 3) == -2
        for which in (0, 1, 2, 3):
            assert lib.poppy_cuda_set_image(ctx, which, None, w * 12) == -2
        assert lib.poppy_cuda_set_image(ctx, 3, p, w * 3 - 1) == -2
        assert lib.poppy_cuda_set_pair(ctx, None, w * 3, p, w * 3, None, 0) == -2
        assert lib.poppy_cuda_set_pair(ctx, p, w * 3, None, w * 3, None, 0) == -2
        assert lib.poppy_cuda_set_image(ctx, 3, p, w * 3) == 0
        basis = r.read_stage(STAGE_MASK_BASIS, 0)
        assert (basis == np.float32(1)).all()           # black corrected2: Gabor response 0, grey 0
