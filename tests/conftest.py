import glob
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
GOLDEN = os.path.join(REPO, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_snapshot(dataset):
    """Released state dict (key for key) from tests/golden/snapshot_<dataset>.npz."""
    z = np.load(os.path.join(GOLDEN, f"snapshot_{dataset}.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def golden_cases(dataset=None, detail=None, n_max=None):
    out = []
    for path in sorted(glob.glob(os.path.join(GOLDEN, "case_*.npz"))):
        meta = json.loads(str(np.load(path)["meta"]))
        if dataset and meta["dataset"] != dataset:
            continue
        if detail and meta["detail"] not in detail:
            continue
        if n_max and meta["n"] > n_max:
            continue
        out.append(path)
    return out


def load_case(path):
    z = np.load(path)
    case = {k: z[k] for k in z.files if k != "meta"}
    case["meta"] = json.loads(str(z["meta"]))
    return case


def demo_clouds(directory):
    """The reference's demo clouds shrunk to one vertex per 5 cm voxel (tests/golden/make_demo_clouds_golden.py), written under
    `directory` as cloud_bin_{0,1}.ply behind the files' own headers.  Returns (paths, vertex counts of the full clouds, the
    vertices written)."""
    z = np.load(os.path.join(GOLDEN, "demo_clouds_sample.npz"))
    paths, counts, points = [], [], []
    for i in (0, 1):
        head, pts = bytes(z[f"header_{i}"]).decode("ascii"), z[f"points_{i}"]
        full = re.search(r"^element vertex (\d+)$", head, re.M)
        counts.append(int(full.group(1)))
        paths.append(os.path.join(str(directory), f"cloud_bin_{i}.ply"))
        with open(paths[-1], "wb") as f:
            f.write((head[:full.start(1)] + str(len(pts)) + head[full.end(1):]).encode("ascii"))
            f.write(pts.astype("<f4").tobytes())
        points.append(pts)
    return paths, counts, points


def registration_ok(case):
    """Oracle/reference registration succeeded (SURVEY.md §7 trap 8: failures are chaotic)."""
    scale = 1.0 if case["meta"]["dataset"] == "3dmatch" else 10.0
    return float(np.abs(case["final_trans"] - case["gt_trans"]).max()) < 0.05 * scale


@pytest.fixture(scope="session")
def snapshots():
    return {d: load_snapshot(d) for d in ("3dmatch", "kitti")}
