"""Full-size (BASELINE.json config 4: 3840x2160, 20k points, 6 levels) checks: two frames against the reference
library, and size-independent properties — determinism, chunk-size independence through a device-side checksum,
and the mask-zero property (maskRatio = 0 => the frame ignores the pixels of image 2). Where the reference library is
not built the frames are compared with the CPU restatement, which uses the product's triangulation: the triangle lists of
these 20k- and 50k-point meshes are then not checked against cv::Subdiv2D (see tests.util.reference)."""
import numpy as np
import pytest

from poppy_b200 import host, synth
from tests.util import assert_frame_parity, bits_differ, reference

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def workload(native_lib):
    c = synth.WORKLOADS["4k"]
    inp = synth.make_inputs(c["w"], c["h"], c["n_points"], c["jitter"], c["seed"])
    return c, inp


def test_4k_frames_match_reference(workload):
    ref = reference()
    from poppy_b200.renderer import MorphRenderer
    c, inp = workload
    w, h, L = c["w"], c["h"], c["levels"]
    phases = np.array([0.25, 0.8], np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    assert 39000 < plan.max_triangles < 41000
    with MorphRenderer(w, h, L, len(inp.pts1), plan.max_triangles, 2) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
        frames = r.download(0, 2)
    for k, s in enumerate(phases):
        want, _ = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, float(s), float(s), L)
        rep = assert_frame_parity(frames[k], want, f"4K phase {s}")
        assert rep["differing_bytes"] == 0, rep


def test_4k_determinism_and_chunk_independence(workload):
    from poppy_b200.renderer import MorphRenderer
    c, inp = workload
    w, h, L = c["w"], c["h"], c["levels"]
    phases = np.linspace(0.05, 0.95, 6).astype(np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    sums = []
    for chunk in (1, 6, 4):
        with MorphRenderer(w, h, L, len(inp.pts1), plan.max_triangles, len(phases), chunk_frames=chunk) as r:
            r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
            r.set_points(inp.pts1, inp.pts2)
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
            a = r.checksum(0, len(phases))
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
            assert r.checksum(0, len(phases)) == a, "render is not deterministic"
            sums.append(a)
            per_frame = [r.checksum(k, 1) for k in range(len(phases))]
            assert len(set(per_frame)) == len(phases), "distinct phases must give distinct frames"
    assert sums[0] == sums[1] == sums[2], "frames depend on the chunk size"


def test_mask_zero_ignores_image2_full_size(workload):
    """maskRatio = 0 makes lbmask exactly 1 at every pyramid level (pyrDown of a constant 1 is exactly 1), so the
    right-hand pyramid is multiplied by exactly 0 everywhere: the frame must not depend on the pixels of image 2
    (it still depends on the second point set through the mesh)."""
    from poppy_b200.renderer import MorphRenderer
    c, inp = workload
    w, h, L = c["w"], c["h"], c["levels"]
    shapes = np.array([0.35, 0.8], np.float32)
    masks = np.zeros(2, np.float64)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, shapes)
    sums = []
    with MorphRenderer(w, h, L, len(inp.pts1), plan.max_triangles, 2) as r:
        r.set_points(inp.pts1, inp.pts2)
        for img2 in (inp.bgr2, np.ascontiguousarray(inp.bgr1[::-1])):
            r.set_pair(inp.bgr1, img2, inp.gabor2)
            r.render(shapes, masks, plan.tri_idx, plan.tri_offsets)
            sums.append([r.checksum(k, 1) for k in range(2)])
    assert sums[0] == sums[1]
    assert sums[0][0] != sums[0][1]


def test_4k_overlapping_lanes_are_deterministic(workload):
    """64 phases = 4 chunks alternating between the two render lanes (streams that overlap on the GPU): repeated renders
    must give identical frames. This is the configuration in which a missing generic->async proxy fence in the TMA ring
    of the level 0->1 kernel showed up as rare +-1 LSB differences (tools/stress_determinism.py)."""
    from poppy_b200.renderer import MorphRenderer
    c, inp = workload
    w, h, L = c["w"], c["h"], c["levels"]
    phases = np.linspace(0.0, 1.0, 64).astype(np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    with MorphRenderer(w, h, L, len(inp.pts1), plan.max_triangles, len(phases)) as r:
        r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
        r.set_points(inp.pts1, inp.pts2)
        ref_sums = None
        for run in range(12):
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
            sums = [r.checksum(k, 1) for k in range(len(phases))]
            if ref_sums is None:
                ref_sums = sums
            assert sums == ref_sums, f"run {run}: frames {[k for k in range(64) if sums[k] != ref_sums[k]]} changed"


def test_8k_frame_matches_reference(native_lib):
    """BASELINE.json configs[4] shape: 7680x4320, 50,004 points, 6 levels - one frame against the reference library (which
    needs ~10 s for it) and the chunk-size independence of a 3-frame render through the device checksum."""
    ref = reference()
    from poppy_b200.renderer import MorphRenderer
    c = synth.WORKLOADS["8k"]
    inp = synth.make_inputs(c["w"], c["h"], c["n_points"], c["jitter"], c["seed"])
    w, h, L = c["w"], c["h"], c["levels"]
    phases = np.array([0.37, 0.5, 0.93], np.float32)
    plan = host.SequencePlan(inp.pts1, inp.pts2, w, h, phases)
    sums = []
    for chunk in (3, 1):
        with MorphRenderer(w, h, L, len(inp.pts1), plan.max_triangles, 3, chunk_frames=chunk) as r:
            r.set_pair(inp.bgr1, inp.bgr2, inp.gabor2)
            r.set_points(inp.pts1, inp.pts2)
            r.render(phases, phases.astype(np.float64), plan.tri_idx, plan.tri_offsets)
            sums.append(r.checksum(0, 3))
            if chunk == 3:
                frame = r.download(0, 1)[0]
    assert sums[0] == sums[1], "8K frames depend on the chunk size"
    want, _ = ref.morph_images(inp.bgr1, inp.bgr2, inp.gabor2, inp.pts1, inp.pts2, float(phases[0]), float(phases[0]), L)
    rep = assert_frame_parity(frame, want, "8K phase 0.37")
    assert rep["differing_bytes"] == 0, rep
