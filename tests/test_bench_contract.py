"""bench.py bookkeeping that needs no GPU: the SURVEY.md section 8(d) byte model and the roofline objects."""
import importlib.util
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_algorithmic_bytes_match_the_survey_table():
    b = _bench()
    assert b.algorithmic_bytes_per_frame(1920, 1080, 6) == 138_905_040
    assert b.algorithmic_bytes_per_frame(3840, 2160, 6) == 555_588_480
    assert b.algorithmic_bytes_per_frame(7680, 4320, 6) == 2_222_322_240


def test_dominant_kernel_roofline_fields():
    b = _bench()
    kern = [{"kernel": "blend_collapse", "ms_per_step": 57.2, "share": 0.30, "launches_per_step": 133, "us_per_launch": 430.0},
            {"kernel": "raster_warp", "ms_per_step": 50.2, "share": 0.26, "launches_per_step": 19, "us_per_launch": 2642.0}]
    traffic = {"source": "test", "bytes_per_frame": {"blend_collapse": 4.2e8, "raster_warp": 7.6e7}}
    d = b.dominant_kernel_roofline(kern, 3840, 2160, 600, 32, 6532.2, traffic, 6)
    assert d["kernel"] == "blend_collapse" and d["unit"] == "GB/s"
    assert 0 < d["frac"] < 1 and abs(d["achieved"] / d["peak"] - d["frac"]) < 1e-12
    # the 7 launches of a 32-frame chunk are rated together; traffic and algorithmic bytes cover the same 32 frames
    assert d["launches_per_chunk"] == 7 and abs(d["us_per_launch"] - 7 * 430.0) < 1e-9
    assert abs(d["traffic"] - 4.2e8 * 32) < 1e3
    assert d["algorithmic_bytes_per_launch"] > 0.8 * d["traffic"]
    d2 = b.dominant_kernel_roofline(kern[1:], 3840, 2160, 600, 32, 6532.2, traffic, 6)
    assert d2["kernel"] == "raster_warp" and d2["algorithmic_bytes_per_launch"] == int((8 * 3840 * 2160 + 8 * 3840 * 2160 / 32) * 32)
    # achieved = the class's algorithmic bytes of the step / its device time
    assert abs(d2["achieved"] - (8 * 3840 * 2160 + 8 * 3840 * 2160 / 32) * 600 / 50.2e-3 / 1e9) < 1e-6


def test_job_configs_are_identical_for_both_arms():
    """The reference arm and the CUDA arm print the same `config` object (the driver compares them)."""
    import argparse
    b = _bench()
    a = argparse.Namespace(mode="chain", workload="4k", total_frames=0, frames=0, ring=0)
    j0, j1 = b.Job(a, 0, 1), b.Job(a, 0, 1)
    assert j0.config() == j1.config() and j0.F == 60 and j0.L == 64 and (j0.W, j0.H) == (512, 512)
    assert j0.phases[0] == 0 and abs(j0.masks[-1] - 1.0) < 1e-12


def test_dump_outputs_writes_a_fixed_float32_sample_under_64_mb(tmp_path):
    """--dump-outputs at the 4K workload: frames sampled from the ring slots of the last slice, the same sample every
    run, float32 files of at most 64 MB in all."""
    import argparse
    import numpy as np
    b = _bench()

    class Ring:                                  # stands in for MorphRenderer: slot k holds frame k of the slice
        def download(self, first, count):
            return np.full((count, 2160, 3840, 3), first % 256, np.uint8) + np.arange(3, dtype=np.uint8)

        def morphed_points(self, k):
            return np.full((20004, 2), k, np.float32)

    a = argparse.Namespace(mode="direct", workload="4k", content="synthetic", total_frames=0, frames=600, ring=0)
    job = b.Job(a, 0, 1)
    sizes = []
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), Ring(), job)
        files = sorted(p.name for p in (tmp_path / run).iterdir())
        assert files == ["frames.npy", "morphed_points.npy"]
        sizes.append(sum((tmp_path / run / f).stat().st_size for f in files))
    assert sizes[0] <= 64 * 2 ** 20
    for f in files:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype == np.float32 and (x == y).all()
    frames = np.load(tmp_path / "a" / "frames.npy")
    assert frames.shape == (b.DUMP_FRAMES, b.DUMP_PIXELS, 3)
    assert frames[0, 0, 0] == 0 and frames[-1, 0, 2] == 599 % 256 + 2   # first and last frame of the 600-frame slice


def test_committed_traffic_file_is_well_formed():
    t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    assert set(t["bytes_per_frame"]) >= {"raster_warp", "pyr_down", "blend_collapse", "unsharp_store"}
    total = sum(t["bytes_per_frame"].values())
    assert 555_588_480 < total < 2 * 555_588_480          # above the algorithmic model, well under 2x


def test_issue_roofline_object():
    b = _bench()
    t = b.ncu_traffic()
    r = b.issue_roofline(t, 3000.0, {"sm_mhz": 1965.0})
    assert r["warp_instructions_per_frame"] == sum(t["warp_instructions_per_frame"].values())
    assert abs(r["roofline_frames_per_s"] * r["frac"] - 3000.0) < 1e-6
    assert 0.3 < r["frac"] < 1.0
