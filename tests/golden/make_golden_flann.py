"""Regenerates tests/golden/golden_flann.npz: exact 5-NN answers of REAL FLANN (KDTreeSingleIndex, the index pcl::KdTreeFLANN wraps, through
OpenCV's bundled copy cv2.flann: leaf_max_size 15, exact, sorted) for 4000 jittered queries on each cloud of a map-like scene, plus the squared
distances of FLANN's LINEAR index (brute force) for 200 of them.  The clouds and queries come from the seeded synthetic generator and are not
stored; their checksum is, so that a change of the generator is told apart from a change of the search.  Run: python tests/golden/make_golden_flann.py"""
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from loam_livox_b200 import synthetic as S  # noqa: E402


def inputs():
    """(surface cloud, its queries), (corner cloud, its queries); the linear-index check uses the surface cloud with the first 200 corner queries."""
    mc, ms = S.make_map(5000, 45000)
    rng = np.random.default_rng(1)
    out = []
    for cloud in (ms, mc):
        q = cloud[rng.integers(0, cloud.shape[0], 4000)].copy()
        q[:, :3] += rng.normal(0, 0.05, (4000, 3)).astype(np.float32)
        out.append((cloud, q))
    return out


def crc(arrays):
    return np.array([zlib.crc32(np.ascontiguousarray(a).tobytes()) for a in arrays], dtype=np.uint32)


def build():
    import cv2
    (ms, qs), (mc, qc) = inputs()
    out = {"input_crc": crc([ms, qs, mc, qc])}
    for name, cloud, q in (("surf", ms, qs), ("corner", mc, qc)):
        index = cv2.flann_Index(np.ascontiguousarray(cloud[:, :3]), dict(algorithm=4, leaf_max_size=15))
        fi, fd = index.knnSearch(np.ascontiguousarray(q[:, :3]), 5, params=dict(checks=-1, eps=0.0, sorted=True))
        assert cloud.shape[0] <= np.iinfo(np.uint16).max
        out[f"idx_{name}"], out[f"d2_{name}"] = fi.astype(np.uint16), fd.astype(np.float32)
    lin = cv2.flann_Index(np.ascontiguousarray(ms[:, :3]), dict(algorithm=0))
    _, ld = lin.knnSearch(np.ascontiguousarray(qc[:200, :3]), 5, params=dict(checks=-1, eps=0.0, sorted=True))
    out["linear_d2"] = ld.astype(np.float32)
    return out


if __name__ == "__main__":
    np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_flann.npz"), **build())
    print("written")
