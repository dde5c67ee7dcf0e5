#!/usr/bin/env python
"""A small stand-in for the reference's demo clouds (demo_data/cloud_bin_{0,1}.ply, 3 MB each), so that the PLY reader and the
demo's registration are tested on the real scene without the reference installed.

    python tests/golden/make_demo_clouds_golden.py <reference checkout>

Every cloud is shrunk to one vertex per occupied 5 cm voxel (the 3DMatch snapshot's `downsample`), chosen at random with a fixed
seed, except that the vertices holding the per-axis minima are always kept: the voxel grid's origin (min - voxel / 2) and hence
the set of occupied voxels, i.e. the demo's key points, stay those of the full cloud.  Output: demo_clouds_sample.npz with, per
cloud i, `header_i` (the file's PLY header, bytes) and `points_i` (the kept vertices [m, 3] float32, in file order)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import fpfh_oracle as F  # noqa: E402

VOXEL = 0.05


def header_of(path):
    with open(path, "rb") as f:
        data = f.read(4096)
    end = data.index(b"end_header\n") + len(b"end_header\n")
    return data[:end]


def one_per_voxel(points, seed):
    p = points.astype(np.float64)
    idx = np.floor((p - (p.min(0) - VOXEL * 0.5)) / VOXEL).astype(np.int64)
    _, group = np.unique(idx, axis=0, return_inverse=True)
    group = group.reshape(-1)
    order = np.random.default_rng(seed).permutation(len(points))
    keep = np.full(group.max() + 1, -1, np.int64)
    keep[group[order]] = order                       # the last write wins: one random vertex per voxel
    keep[group[p.argmin(0)]] = p.argmin(0)           # the minima keep the grid's origin
    return np.sort(keep)


def main():
    ref = sys.argv[1]
    out = {}
    for i in (0, 1):
        path = os.path.join(ref, "demo_data", f"cloud_bin_{i}.ply")
        pts = F.read_ply(path)
        keep = one_per_voxel(pts, i)
        out[f"header_{i}"] = np.frombuffer(header_of(path), np.uint8)
        out[f"points_{i}"] = pts[keep]
        print(f"cloud_bin_{i}.ply: {len(pts)} vertices -> {len(keep)}")
    dst = os.path.join(HERE, "demo_clouds_sample.npz")
    np.savez_compressed(dst, **out)
    print(f"{os.path.basename(dst)}: {os.path.getsize(dst) / 1e3:.0f} KB")


if __name__ == "__main__":
    main()
