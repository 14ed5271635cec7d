#!/usr/bin/env python
"""Generates tests/golden/flann_knn5.npz: FLANN's exact 5-NN answers on the queries of tests/test_oracle_pins.py.

WHAT THIS FIXTURE IS: the indices and float squared distances that OpenCV's bundled FLANN (cv2.flann_Index, the FLANN
code base behind pcl::KdTreeFLANN, which the reference searches with) returns, for KDTREE_SINGLE (leaf_max_size 15, exact
search) and LINEAR (brute force).  Per case it stores the SHA-256 of the inputs and of the complete answers, plus a fixed,
seeded sample of answer rows, so the oracle is compared with every FLANN answer bit for bit without OpenCV at test time.

Run from the repo root, with OpenCV's Python package installed:  python tests/golden/make_flann_golden.py
"""
import hashlib
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from glio_b200 import synth  # noqa: E402
from oracle import pyoracle as oracle  # noqa: E402

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "flann_knn5.npz")
FLANN_INDEX_LINEAR, FLANN_INDEX_KDTREE_SINGLE = 0, 4
ALGORITHMS = dict(kdtree_single=FLANN_INDEX_KDTREE_SINGLE, linear=FLANN_INDEX_LINEAR)
SAMPLE_ROWS = 256


def digest(*arrays):
    """SHA-256 over dtype, shape and bytes of each array."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode()); h.update(a.tobytes())
    return h.hexdigest()


def small_problem():
    """Small, dense cloud with many near neighbours: map (40k) and scan 0 (3k) in the map frame."""
    P = synth.window_problem(W=2, Q=3000, M=40000, seed=31)
    t2, q2 = synth.lidar_pose_in_world(P["poses_init"][0, :3], P["poses_init"][0, 3:])
    return P["map_xyz"], oracle.transform_points(P["scans"][0], t2, q2)


FULL_SCANS = (3, 17)


def full_problem():
    """The cfg-2 map (M = 1M) and the first 20k points of two scans in the map frame."""
    P = synth.window_problem(W=20, Q=100_000, M=1_000_000, seed=synth.SEED0 + 2)
    qry = {}
    for k in FULL_SCANS:
        t2, q2 = synth.lidar_pose_in_world(P["poses_init"][k, :3], P["poses_init"][k, 3:])
        qry[k] = oracle.transform_points(P["scans"][k][:20000], t2, q2)
    return P["map_xyz"], qry


def assoc_problem():
    """Map (60k), scan 1 (5k) and its lidar pose in the map frame, for the oracle's association."""
    P = synth.window_problem(W=3, Q=5000, M=60000, seed=77)
    t2, q2 = synth.lidar_pose_in_world(P["poses_init"][1, :3], P["poses_init"][1, 3:])
    return P["map_xyz"], P["scans"][1], t2, q2


def record(out, name, map_xyz, qry, idx, sqd):
    rows = np.sort(np.random.default_rng(zlib.crc32(name.encode())).choice(len(qry), SAMPLE_ROWS, replace=False))
    out[name + "_input_sha256"] = np.array(digest(map_xyz, qry))
    out[name + "_idx_sha256"] = np.array(digest(idx)); out[name + "_sqd_sha256"] = np.array(digest(sqd))
    out[name + "_rows"] = rows.astype(np.int32); out[name + "_idx"] = idx[rows]; out[name + "_sqd"] = sqd[rows]


def main():
    import cv2
    params = dict(checks=-1, eps=0.0, sorted=True)

    def flann(map_xyz, qry, algorithm):
        prm = dict(algorithm=algorithm, leaf_max_size=15) if algorithm == FLANN_INDEX_KDTREE_SINGLE else dict(algorithm=algorithm)
        idx, sqd = cv2.flann_Index(np.ascontiguousarray(map_xyz, np.float32), prm).knnSearch(np.ascontiguousarray(qry, np.float32), 5, params=params)
        return idx.astype(np.int32), sqd.astype(np.float32)

    oracle.build()
    out = dict(opencv_version=np.array(cv2.__version__))
    m, q = small_problem()
    for a, algo in ALGORITHMS.items():
        record(out, "small_" + a, m, q, *flann(m, q, algo))
    m, qs = full_problem()
    for k, q in qs.items():
        record(out, f"full_scan{k}", m, q, *flann(m, q, FLANN_INDEX_KDTREE_SINGLE))
    m, scan, t2, q2 = assoc_problem()
    q = oracle.assoc_scan_to_map(m, scan, t2, q2)["pm"]
    record(out, "assoc", m, q, *flann(m, q, FLANN_INDEX_KDTREE_SINGLE))
    np.savez_compressed(PATH, **out)
    print("wrote", PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()
