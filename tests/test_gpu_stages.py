"""GPU parity, stage by stage: every stage boundary of the CUDA path (through the C ABI) must equal the
reference's (oracle/_ref, the unmodified reference code, or the CPU restatement pinned to it) bit for bit on
seeded inputs."""
import numpy as np
import pytest

from poppy_b200 import synth
from tests.util import bits_differ, flat_tri, reference

pytestmark = pytest.mark.gpu

CASES = [
    # w, h, points, shape/mask ratio, levels
    (320, 240, 200, 0.37, 6),
    (203, 157, 60, 0.5, 64),
    (257, 131, 100, 0.9, 4),
    (641, 479, 300, 0.37, 6),
    (100, 75, 20, 0.0, 6),
    (100, 75, 20, 1.0, 6),
    (333, 222, 50, 0.123, 3),
    (64, 48, 12, 0.5, 2),
    # sizes that exercise the vectorised tile interiors (several tiles / strips / row chunks) and their edges
    (1024, 600, 500, 0.3, 6),
    (508, 436, 200, 0.6, 5),
    (1280, 720, 800, 0.71, 64),
    (250, 1100, 150, 0.45, 7),
]


@pytest.mark.parametrize("w,h,n,s,levels", CASES)
def test_stage_parity_vs_reference(native_lib, w, h, n, s, levels):
    from oracle import port
    from poppy_b200 import renderer as R
    inp = synth.make_inputs(w, h, n, 8.0, seed=7)
    want = reference().stages(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, s, s, levels)
    tri = want.tri_idx
    with R.MorphRenderer(w, h, levels, len(inp.pts1), max(len(tri), 1), 1, keep_stages=True) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        cat, offs = flat_tri([tri])
        r.render([s], [s], cat, offs)
        got_dst = r.download(0, 1)[0]
        assert bits_differ(r.read_stage(R.STAGE_MORPHED_POINTS, 0), want.morphed_points) == 0
        assert bits_differ(r.morphed_points(0), want.morphed_points) == 0
        assert bits_differ(r.read_stage(R.STAGE_TRI_MAP, 0), want.tri_map) == 0, "triangle-ID map"
        # inverse matrices: the reference does not expose them; the pinned CPU restatement does
        p1 = inp.pts1.copy(); p2 = inp.pts2.copy()
        c1 = port.morph_points(p1, p1, 0.0, w, h)  # clip only
        c2 = port.morph_points(p2, p2, 0.0, w, h)
        t1 = np.trunc(c1[tri]).astype(np.int32).reshape(-1, 6)
        t2 = np.trunc(c2[tri]).astype(np.int32).reshape(-1, 6)
        _, _, _, im1, im2 = port.triangle_matrices(t1, t2, np.float32(s))
        assert bits_differ(r.read_stage(R.STAGE_INV_M1, 0, len(tri)), im1) == 0
        assert bits_differ(r.read_stage(R.STAGE_INV_M2, 0, len(tri)), im2) == 0
        assert bits_differ(r.read_stage(R.STAGE_WARPED1, 0), want.warped1) == 0, "remap of image 1"
        assert bits_differ(r.read_stage(R.STAGE_WARPED2, 0), want.warped2) == 0, "remap of image 2"
        assert bits_differ(r.read_stage(R.STAGE_MASK, 0), want.mask) == 0, "blend mask"
        assert bits_differ(r.read_stage(R.STAGE_LAP_BLEND, 0), want.lap_blend) == 0, "Laplacian blend"
        assert bits_differ(got_dst, want.dst) == 0, "final 8-bit frame"
