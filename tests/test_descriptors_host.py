"""CPU-side checks of row f2 (SURVEY.md section 8): the descriptor oracle's own invariants and the host PLY reader of the C ABI.
The oracle is unpinned against open3d (absent from this image); these tests pin what CAN be pinned without it: analytic
normals, histogram mass, rigid-motion invariance, and the reader against the oracle's independent parser."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

from oracle import fpfh_oracle as F
from pointdsc_b200 import _capi
from pointdsc_b200.synth_scene import rigid, scene


def _write_ply(path, pts, binary, double=False, extra=False):
    typ = "double" if double else "float"
    with open(path, "wb") as f:
        head = ["ply", "format " + ("binary_little_endian" if binary else "ascii") + " 1.0", "comment test",
                f"element vertex {len(pts)}"]
        if extra:
            head.append("property uchar red")
        head += [f"property {typ} x", f"property {typ} y"]
        if extra:
            head.append("property float nx")
        head += [f"property {typ} z", "element face 0", "property list uchar int vertex_indices", "end_header"]
        f.write(("\n".join(head) + "\n").encode())
        code = "<d" if double else "<f"
        for p in pts:
            if binary:
                row = b""
                if extra:
                    row += struct.pack("<B", 7)
                row += struct.pack(code, p[0]) + struct.pack(code, p[1])
                if extra:
                    row += struct.pack("<f", 0.25)
                row += struct.pack(code, p[2])
                f.write(row)
            else:
                vals = ([7] if extra else []) + [repr(float(p[0])), repr(float(p[1]))] + ([0.25] if extra else []) + [repr(float(p[2]))]
                f.write((" ".join(str(v) for v in vals) + "\n").encode())


@pytest.mark.parametrize("binary,double,extra", [(False, False, False), (True, False, False), (True, True, True), (False, True, True)])
def test_ply_reader_matches_the_oracle_parser(tmp_path, binary, double, extra):
    pts = scene(5000, seed=3)[:4500]
    path = str(tmp_path / "cloud.ply")
    _write_ply(path, pts, binary, double, extra)
    from pointdsc_b200.descriptors import read_ply
    got = read_ply(path)
    assert got.dtype == np.float32 and got.shape == (4500, 3)
    assert np.array_equal(got, F.read_ply(path))
    assert np.array_equal(got, pts)


def test_ply_reader_errors_are_loud(tmp_path):
    lib = _capi.load()
    n = C.c_int64(0)
    assert lib.pdsc_read_ply(str(tmp_path / "missing.ply").encode(), None, 0, C.byref(n)) != 0
    bad = tmp_path / "bad.ply"
    bad.write_bytes(b"ply\nformat binary_big_endian 1.0\nelement vertex 1\nproperty float x\nend_header\n")
    assert lib.pdsc_read_ply(str(bad).encode(), None, 0, C.byref(n)) != 0
    path = str(tmp_path / "ok.ply")
    _write_ply(path, scene(100, seed=1)[:50], True)
    buf = np.empty((10, 3), np.float32)
    assert lib.pdsc_read_ply(path.encode(), buf.ctypes.data_as(C.c_void_p), 10, C.byref(n)) != 0   # capacity too small
    assert n.value == 50


def test_oracle_voxel_means_and_order():
    rng = np.random.default_rng(0)
    pts = rng.uniform(-1, 1, (4000, 3)).astype(np.float32)
    means, keys = F.voxel_down_sample(pts, 0.25)
    assert (np.diff(keys[:, 0] * 10000 + keys[:, 1] * 100 + keys[:, 2]) > 0).all()          # ascending, distinct
    origin = pts.astype(np.float64).min(0) - 0.125
    assert np.array_equal(np.floor((means - origin) / 0.25).astype(np.int64), keys)          # a mean stays inside its voxel
    counts = np.zeros(len(means))
    idx = np.floor((pts.astype(np.float64) - origin) / 0.25).astype(np.int64)
    lut = {tuple(k): i for i, k in enumerate(keys)}
    acc = np.zeros_like(means)
    for p, k in zip(pts.astype(np.float64), idx):
        acc[lut[tuple(k)]] += p
        counts[lut[tuple(k)]] += 1
    assert np.allclose(acc / counts[:, None], means, rtol=0, atol=1e-12)


def test_oracle_normals_on_analytic_surfaces():
    rng = np.random.default_rng(1)
    plane = np.c_[rng.uniform(0, 1, (400, 2)), np.zeros(400)].astype(np.float32)
    n = F.estimate_normals(plane, 0.2, 30)
    assert np.allclose(n, [0, 0, 1], atol=1e-9)
    v = rng.normal(size=(3000, 3))
    sphere = (2.0 * v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)
    n = F.estimate_normals(sphere, 0.3, 30)
    radial = sphere / 2.0
    assert (np.abs((n * radial).sum(1)) > 0.995).all()
    assert (n[np.arange(len(n)), np.abs(n).argmax(1)] > 0).all()                              # the sign convention
    lonely = np.array([[0, 0, 0], [10, 0, 0], [10.05, 0, 0]], np.float32)
    assert np.array_equal(F.estimate_normals(lonely, 0.2, 30), np.tile([0.0, 0.0, 1.0], (3, 1)))


def test_oracle_fpfh_mass_and_rigid_invariance():
    pts = scene(2500, seed=2)
    kp, _ = F.voxel_down_sample(pts, 0.2)
    kp = kp.astype(np.float32)
    nrm = F.estimate_normals(kp, 0.4, 30)
    f = F.fpfh(kp, nrm, 1.0, 100)
    nb = F.hybrid_neighbours(kp, 1.0, 100)
    has = np.array([len(i) > 1 for i, _ in nb])
    assert has.all()
    assert np.allclose(f.reshape(-1, 3, 11).sum(2), 200.0, atol=1e-9)                         # SPFH 100 + weighted part 100, per feature
    # a rigid motion of the points AND the normals leaves the pair features alone (up to the float32 rounding of the moved points)
    R, t = rigid(3)
    kp2 = (kp.astype(np.float64) @ R.T + t).astype(np.float32)
    f2 = F.fpfh(kp2, nrm @ R.T, 1.0, 100)
    diff = np.abs(f - f2).max(1)
    # rounding moves a few neighbours across the radius / rank / bin boundaries; every such flip touches the ~70 descriptors around it
    assert np.median(diff) < 1e-4 and (diff < 2.0).mean() > 0.9, (np.median(diff), (diff < 2.0).mean())


def test_ply_reader_on_the_reference_demo_clouds(tmp_path):
    """BASELINE.json configs[0] reads demo_data/cloud_bin_{0,1}.ply (binary little-endian float xyz, 258 342 / 268 977 vertices,
    CloudCompare's header): read here behind those same headers, with one vertex per 5 cm voxel of each cloud."""
    from conftest import demo_clouds
    paths, counts, points = demo_clouds(tmp_path)
    assert counts == [258342, 268977]
    from pointdsc_b200.descriptors import read_ply
    for path, want in zip(paths, points):
        n = len(want)
        pts = read_ply(path)
        assert pts.shape == (n, 3) and pts.dtype == np.float32 and np.isfinite(pts).all()
        raw = np.fromfile(path, dtype="<f4", offset=os.path.getsize(path) - 12 * n).reshape(n, 3)   # the payload behind the header
        assert np.array_equal(pts, raw) and np.array_equal(pts, want)
