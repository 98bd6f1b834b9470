"""Writes slot_boundary.json here: 128 x 96 frames (one slice) whose restated FFV1 slice lands within a few bytes of the
points where the GPU encoder's first pass changes behaviour. The slot holds cap = 36,928 bytes and the first pass stops a
slice whose committed bytes pass limit = cap - 25 before a symbol (tests/test_ffv1_edges.py, slot_cap). A frame's first n
pixels in raster order are noise and the rest smooth (boundary_slice); n is found by bisection on the restated size, then
the n nearest the target inside its window is kept. tests/test_ffv1_edges.py re-checks every size.

    python tests/golden/output/ffv1/make_slot_boundary.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(HERE)))))

from oracle import ffv1  # noqa: E402
from tests.test_ffv1_edges import boundary_slice, slot_cap  # noqa: E402

W, H, SEED = 128, 96, 0


def size(n):
    return len(ffv1.encode_frame(boundary_slice(W, H, n, SEED))) - 3       # the slice without its 24-bit size


def main():
    cap, limit = slot_cap(W, H)
    # targets at or below a threshold are approached from below, the others from above
    targets = {"limit-19": (limit - 19, -1), "limit": (limit, -1), "limit+1": (limit + 1, 1), "cap-3": (cap - 3, -1),
               "cap-2": (cap - 2, 1), "cap": (cap, 1), "cap+16": (cap + 16, 1)}
    points = []
    for name, (t, side) in targets.items():
        lo, hi = 0, W * H
        while lo < hi:                                  # smallest n with size(n) >= t
            mid = (lo + hi) // 2
            if size(mid) >= t:
                hi = mid
            else:
                lo = mid + 1
        window = [t - 4, t] if side < 0 else [t, t + 4]
        near = [(abs(s - t), n, s) for n in range(max(0, lo - 8), min(W * H, lo + 8) + 1)
                for s in [size(n)] if window[0] <= s <= window[1]]
        _, n, s = min(near)
        points.append({"target": name, "n": n, "size": s, "window": window})
        print(name, t, n, s)
    with open(os.path.join(HERE, "slot_boundary.json"), "w") as f:
        json.dump({"w": W, "h": H, "seed": SEED, "cap": cap, "limit": limit, "points": points}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
