"""The routes through the unsharp stage (reference src/util.cpp:113-148) give the same bytes: the fused level-0
collapse + calm analysis (exact blur/median only on the strip chunks that can reach the threshold), the exact path
on every pixel, and the adaptive choice between the two; all equal the reference library."""
import numpy as np
import pytest

from poppy_b200 import host, synth
from poppy_b200.renderer import MorphRenderer
from tests.util import bits_differ, reference as _ref

pytestmark = pytest.mark.gpu


CASES = [
    # kind, w, h, points, levels: smooth noise (calm almost everywhere), hard edges (threshold fires), odd sizes
    ("noise", 640, 360, 200, 6), ("blocks", 640, 360, 200, 6), ("shapes", 512, 512, 96, 64), ("blocks", 333, 251, 60, 4),
    ("noise", 130, 75, 20, 6), ("blocks", 37, 29, 8, 3), ("shapes", 1000, 90, 64, 5),
]


@pytest.mark.parametrize("kind,w,h,n,levels", CASES)
def test_calm_route_equals_exact_route_and_reference(native_lib, kind, w, h, n, levels):
    ref = _ref()
    inp = {"noise": lambda: synth.make_inputs(w, h, n, 8.0, seed=31), "shapes": lambda: synth.shape_inputs(w, h, n, seed=32),
           "blocks": lambda: synth.block_inputs(w, h, n, seed=33)}[kind]()
    phases = np.array([0.0, 0.35, 0.5, 1.0], np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    frames, stats = {}, {}
    for mode in (2, 1, 0):
        with MorphRenderer(w, h, levels, len(inp.pts1), plan.max_triangles, len(phases)) as r:
            r.set_unsharp_mode(mode)
            r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
            r.set_points(inp.pts1, inp.pts2)
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
            frames[mode] = r.download(0, len(phases))
            stats[mode] = r.unsharp_stats()
    assert bits_differ(frames[2], frames[1]) == 0 and bits_differ(frames[0], frames[1]) == 0
    assert stats[1][0] == stats[1][1] > 0                      # dense route: every chunk
    assert 0 <= stats[2][0] <= stats[2][1] == stats[1][1]
    for k, s in enumerate(phases):
        want, _ = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, float(s), float(s), levels)
        assert bits_differ(frames[0][k], want) == 0, (kind, k)


def test_calm_analysis_separates_content(native_lib):
    """Smooth content takes the fused route almost everywhere, hard edges force the exact route where they are."""
    w, h, levels = 960, 540, 6
    phases = np.array([0.0], np.float32)
    share = {}
    for kind in ("noise", "blocks"):
        inp = synth.make_inputs(w, h, 300, 8.0, seed=41) if kind == "noise" else synth.block_inputs(w, h, 300, seed=42)
        plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
        with MorphRenderer(w, h, levels, len(inp.pts1), plan.max_triangles, 1) as r:
            r.set_unsharp_mode(2)
            r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
            r.set_points(inp.pts1, inp.pts2)
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
            exact, total = r.unsharp_stats()
            share[kind] = exact / total
    assert share["noise"] < 0.35 and share["blocks"] > 0.9, share
