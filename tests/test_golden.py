"""The CPU restatement against the committed golden vectors (tests/golden/*.npz, generated from the reference
library by tests/golden/make_golden.py). Runs everywhere, needs neither the reference tree nor a GPU."""
import glob
import os

import numpy as np
import pytest

from oracle import port
from tests.util import bits_differ

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FRAME_FILES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "*.npz"))
                     if not os.path.basename(f).startswith(("chain_", "topology")))
STAGE_KEYS = ["morphed_points", "tri_map", "hom", "m1", "m2", "mapx1", "mapy1", "mapx2", "mapy2", "warped1", "warped2",
              "mask", "lap_blend", "dst"]


def test_fixtures_present():
    assert len(FRAME_FILES) >= 8
    assert os.path.exists(os.path.join(GOLDEN, "chain_shapes_80x64_N12_L64.npz"))
    assert os.path.exists(os.path.join(GOLDEN, "topology.npz"))


@pytest.mark.parametrize("path", FRAME_FILES, ids=[os.path.basename(f)[:-4] for f in FRAME_FILES])
def test_port_reproduces_golden_stages(path):
    g = np.load(path)
    got = port.morph_frame(g["bgr1"], g["bgr2"], g["gabor2"], g["pts1"], g["pts2"], g["tri_idx"], float(g["shape"]),
                           float(g["mask_ratio"]), int(g["levels"]))
    for k in STAGE_KEYS:
        assert bits_differ(getattr(got, k), g[k]) == 0, k


def test_port_reproduces_golden_chain():
    """Frame-loop recurrence (reference src/poppy.hpp:177-243) restated around the port + the host topology."""
    g = np.load(os.path.join(GOLDEN, "chain_shapes_80x64_N12_L64.npz"))
    frames, points = port.chain(g["bgr1"], g["bgr2"], g["gabor2"], g["pts1"], g["pts2"], int(g["n_frames"]), int(g["levels"]))
    for j in range(int(g["n_frames"])):
        assert bits_differ(points[j], g["points"][j]) == 0, j
        assert (frames[j] == g["frames"][j]).all(), j


@pytest.mark.parametrize("path", FRAME_FILES, ids=[os.path.basename(f)[:-4] for f in FRAME_FILES])
def test_port_entry_points_reproduce_golden_frames(path):
    """port.stages / port.morph_images, the stand-ins of the reference library in the GPU parity tests, with their own
    triangulation: the same triangle lists, stages and frames as the reference."""
    g = np.load(path)
    args = (g["bgr1"], g["bgr2"], g["gabor2"], g["pts1"], g["pts2"], float(g["shape"]), float(g["mask_ratio"]), int(g["levels"]))
    st = port.stages(*args)
    assert (st.tri_idx == g["tri_idx"]).all()
    for k in STAGE_KEYS:
        assert bits_differ(getattr(st, k), g[k]) == 0, k
    dst, mp = port.morph_images(*args)
    assert (dst == g["dst"]).all() and bits_differ(mp, g["morphed_points"]) == 0


def test_fixtures_come_from_the_avx2_fma_dispatch_of_the_reference():
    """Bit parity is defined against the reference's AVX2/FMA-dispatched OpenCV build (DESIGN.md 6): the whole-pipeline
    fixtures record the CPU features the reference ran with when they were made."""
    import os
    import numpy as np
    full = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full")
    for c in (1, 2, 3):
        feats = str(np.load(os.path.join(full, f"c{c}.npz"))["cpu_features"])
        assert "AVX2" in feats and "FP16" in feats, feats
