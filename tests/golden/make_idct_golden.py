"""Generates tests/golden/idct_golden.npz: a plane of 8x8 sample blocks (seeded random bytes plus the corner cases all-0, all-255,
alternating 0/255 -- the reference's own known-answer block, c_components/tests/test_idct_scaling.rs:4-18 -- and ramps), a plane of
33 x 5 random blocks (an odd block count), and what the REFERENCE ITSELF (oracle/_ref/libidct_ref.so =
c_components/lib/codecs_jpeg_idct_fast.c compiled unmodified) makes of each with its 14 block scalers.  Needs oracle/_ref, which
__graft_entry__.build() makes only where the reference tree is readable:  python tests/golden/make_idct_golden.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402


def plane():
    rng = np.random.default_rng(20260923)
    p = rng.integers(0, 256, (64, 96), dtype=np.uint8)          # 8 x 12 blocks
    p[0:8, 0:8] = 0
    p[0:8, 8:16] = 255
    p[0:8, 16:24] = np.tile(np.array([0, 255], np.uint8), 32).reshape(8, 8)          # the reference's KAT block
    p[0:8, 24:32] = np.arange(64, dtype=np.uint8).reshape(8, 8) * 4
    p[0:8, 32:40] = (255 - np.arange(64) * 4).astype(np.uint8).reshape(8, 8)
    p[8:16, 0:8] = rng.integers(250, 256, (8, 8), dtype=np.uint8)                    # saturation
    p[8:16, 8:16] = rng.integers(0, 6, (8, 8), dtype=np.uint8)
    return p


if __name__ == "__main__":
    assert oracle.idct_ref_available(), "needs oracle/_ref/libidct_ref.so (built by __graft_entry__.build() next to the reference tree)"
    p = plane()
    r = np.random.default_rng(9).integers(0, 256, (40, 264), dtype=np.uint8)
    out = {"plane": p, "random_plane": r}
    for srgb in (0, 1):
        for n in range(1, 8):
            out[f"out_{srgb}_{n}"] = oracle.flow_scale_spatial_ref(p, n, bool(srgb))
            out[f"random_{srgb}_{n}"] = oracle.flow_scale_spatial_ref(r, n, bool(srgb))
    assert out["out_1_1"][0, 2] == 188                                               # test_idct_scaling.rs:17
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "idct_golden.npz"), **out)
    print("wrote idct_golden.npz", {k: v.shape for k, v in out.items() if k != "plane"})
