"""GPU parity of row f2 (SURVEY.md section 8): voxel down-sampling, normals and FPFH kernels against oracle/fpfh_oracle.py
(the CPU restatement of open3d 0.9's algorithms; parity unpinned — open3d is not in this image), then the whole chain
PLY -> FPFH -> match -> PointDSC on a synthetic pair with a known motion."""
import numpy as np
import pytest
import torch

from conftest import load_snapshot
from oracle import fpfh_oracle as F
from pointdsc_b200.synth_scene import rigid, scene

pytestmark = pytest.mark.gpu


def _dev(x, dtype=torch.float32):
    return torch.as_tensor(x, dtype=dtype, device="cuda")


@pytest.mark.parametrize("n,voxel,offset", [(20000, 0.05, 0.0), (6000, 0.1, 0.0), (5000, 0.3, -40.0), (1, 0.05, 0.0), (300000, 0.025, 3.0)])
def test_voxel_down_sample_vs_oracle(n, voxel, offset):
    from pointdsc_b200.descriptors import voxel_down_sample
    pts = scene(max(n, 40), seed=n)[:n] + np.float32(offset)
    got = voxel_down_sample(_dev(pts), voxel).cpu().numpy()
    want, keys = F.voxel_down_sample(pts, voxel)
    assert got.shape == want.shape                        # same occupied voxels (the index arithmetic is bit-exact fp64)
    # means: fp64 sum / count on the CPU, 2^-40-voxel fixed point on the device, both rounded to float32 at the end
    assert np.abs(got.astype(np.float64) - want).max() <= 1.0 * np.spacing(np.float32(np.abs(want).max()))
    again = voxel_down_sample(_dev(pts[::-1].copy()), voxel).cpu().numpy()
    assert np.array_equal(got, again)                     # the result does not depend on the input order (integer accumulation)


def test_voxel_status_is_loud():
    from pointdsc_b200 import PdscError
    from pointdsc_b200.descriptors import voxel_down_sample
    pts = scene(1000, seed=0)
    pts[17, 1] = np.nan
    with pytest.raises(PdscError):
        voxel_down_sample(_dev(pts), 0.05)
    with pytest.raises(PdscError):
        voxel_down_sample(_dev(scene(1000, seed=0)), 1e-7)          # > 2^21 voxels along an axis
    with pytest.raises(PdscError):
        voxel_down_sample(torch.zeros(10, 3), 0.05)                 # CPU tensor: no fallback


def _keypoints(n, voxel, seed):
    from pointdsc_b200.descriptors import voxel_down_sample
    return voxel_down_sample(_dev(scene(n, seed=seed)), voxel)


@pytest.mark.parametrize("n,voxel,max_nn", [(6000, 0.1, 30), (20000, 0.05, 30), (3000, 0.2, 7), (6000, 0.1, 100)])
def test_normals_vs_oracle(n, voxel, max_nn):
    from pointdsc_b200.descriptors import estimate_normals
    kp = _keypoints(n, voxel, 11)
    got = estimate_normals(kp, 2 * voxel, max_nn).cpu().numpy()
    kp_h = kp.cpu().numpy()
    want = F.estimate_normals(kp_h, 2 * voxel, max_nn)
    assert np.allclose(np.linalg.norm(got, axis=1), 1.0, atol=1e-12)
    # the eigenvector of a nearly degenerate covariance is ill-conditioned in ANY solver: compare where the gap is healthy
    gap_ok = np.ones(len(kp_h), bool)
    for i, (idx, _) in enumerate(F.hybrid_neighbours(kp_h, 2 * voxel, max_nn)):
        if len(idx) >= 3:
            w = np.linalg.eigvalsh(np.cov(kp_h[idx].astype(np.float64).T, bias=True))
            gap_ok[i] = (w[1] - w[0]) > 1e-3 * w[2]
    assert gap_ok.mean() > 0.8
    assert np.abs(got - want)[gap_ok].max() < 1e-9
    flipped = np.minimum(np.abs(got - want).max(1), np.abs(got + want).max(1))
    assert (flipped[~gap_ok] < 1e-4).all()


def test_normals_below_three_neighbours():
    from pointdsc_b200.descriptors import estimate_normals
    pts = np.array([[0, 0, 0], [10, 0, 0], [10.05, 0, 0], [20, 0, 0], [20.05, 0, 0], [20, 0.05, 0.01]], np.float32)
    got = estimate_normals(_dev(pts), 0.2, 30).cpu().numpy()
    want = F.estimate_normals(pts, 0.2, 30)
    assert np.array_equal(got[:3], np.tile([0.0, 0.0, 1.0], (3, 1)))
    assert np.allclose(got, want, atol=1e-9)


@pytest.mark.parametrize("n,voxel,max_nn,normalise", [(2500, 0.2, 100, False), (2500, 0.2, 100, True), (4000, 0.15, 20, False),
                                                      (1500, 0.3, 100, False)])
def test_fpfh_vs_oracle(n, voxel, max_nn, normalise):
    from pointdsc_b200.descriptors import compute_fpfh, estimate_normals
    kp = _keypoints(n, voxel, 5)
    nrm = estimate_normals(kp, 2 * voxel, 30)
    got = compute_fpfh(kp, nrm, 5 * voxel, max_nn, normalise=normalise).cpu().numpy()
    want = F.fpfh(kp.cpu().numpy(), nrm.cpu().numpy(), 5 * voxel, max_nn)          # the oracle on the SAME key points and normals
    if normalise:
        want = want / (np.linalg.norm(want, axis=1, keepdims=True) + 1e-6)
    assert got.shape == want.shape == (kp.shape[0], 33)
    assert np.abs(got - want).max() < 1e-8 * (1.0 if normalise else 100.0)
    again = compute_fpfh(kp, nrm, 5 * voxel, max_nn, normalise=normalise).cpu().numpy()
    assert np.array_equal(got, again)


def test_fpfh_isolated_points_and_duplicates():
    from pointdsc_b200.descriptors import compute_fpfh, estimate_normals
    rng = np.random.default_rng(0)
    pts = np.concatenate([rng.uniform(0, 1, (300, 3)), [[50, 50, 50]], rng.uniform(0, 1, (5, 3)) + 100]).astype(np.float32)
    pts[10] = pts[11]                                            # a duplicate: distance 0, skipped by the weighted sum
    kp = _dev(pts)
    nrm = estimate_normals(kp, 0.3, 30)
    got = compute_fpfh(kp, nrm, 0.6, 100).cpu().numpy()
    want = F.fpfh(pts, nrm.cpu().numpy(), 0.6, 100)
    assert np.array_equal(got[300], np.zeros(33))                # no neighbour: all-zero row, as open3d leaves it
    assert np.abs(got - want).max() < 1e-6


def test_neighbourhood_overflow_is_loud():
    from pointdsc_b200 import PdscError
    from pointdsc_b200.descriptors import estimate_normals
    pts = np.random.default_rng(0).uniform(0, 0.1, (6000, 3)).astype(np.float32)
    with pytest.raises(PdscError):
        estimate_normals(_dev(pts), 1.0, 30)                      # 6000 points inside every radius > 4096


def test_descriptor_chain_registers_a_synthetic_pair(tmp_path):
    """demo_registration.py with --descriptor fpfh, end to end on the device: PLY -> voxel -> normals -> FPFH -> mutual matching ->
    PointDSC.  Two independent samplings of one scene, the second moved by a known rigid motion."""
    import struct
    from pointdsc_b200 import PointDSC
    from pointdsc_b200.descriptors import fpfh_descriptors, read_ply
    from pointdsc_b200.frontend import match
    R, t = rigid(5)
    src = scene(60000, seed=1)
    tgt = (scene(60000, seed=2).astype(np.float64) @ R.T + t).astype(np.float32)
    clouds = []
    for name, pts in (("src", src), ("tgt", tgt)):
        path = tmp_path / f"{name}.ply"
        with open(path, "wb") as f:
            f.write(f"ply\nformat binary_little_endian 1.0\nelement vertex {len(pts)}\nproperty float x\nproperty float y\nproperty float z\nend_header\n".encode())
            f.write(pts.astype("<f4").tobytes())
        clouds.append(torch.from_numpy(read_ply(str(path))).cuda())
    voxel = 0.08
    (skp, sf), (tkp, tf) = fpfh_descriptors(clouds[0], voxel), fpfh_descriptors(clouds[1], voxel)
    assert sf.dtype == torch.float64 and sf.shape[1] == 33 and 2000 < skp.shape[0] < 20000
    data = match(sf, tf, skp, tkp, use_mutual=False)
    model = PointDSC(in_dim=6, num_layers=12, num_channels=128, num_iterations=10, ratio=0.1, inlier_threshold=0.10, sigma_d=0.10,
                     k=40, nms_radius=0.10).cuda().eval()
    model.load_state_dict(load_snapshot("3dmatch"), strict=False)
    data["testing"] = True
    res = model(data)
    T = res["final_trans"][0].double().cpu().numpy()
    re = np.degrees(np.arccos(np.clip((np.trace(T[:3, :3].T @ R) - 1) / 2, -1, 1)))
    te = np.linalg.norm(T[:3, 3] - t)
    assert re < 2.0 and te < 0.05, (re, te)


def test_demo_registers_the_reference_clouds(tmp_path):
    """BASELINE.json configs[0]: demo_registration.py --descriptor fpfh on the reference's own demo clouds, on the device
    (demo.py).  The clouds are shrunk to one vertex per 5 cm voxel (conftest.demo_clouds), which keeps the full clouds' key
    points.  No ground truth ships with the clouds: the check is what the reference shows in its open3d window — after the
    estimated motion the source lies on the target (coverage 0.13 -> 0.87 on the full clouds, 0.14 -> 0.87 with the CPU checker
    on the shrunk ones) — plus reproducibility."""
    import sys
    from conftest import REPO, demo_clouds
    paths, _, points = demo_clouds(tmp_path)
    sys.path.insert(0, REPO)
    import demo
    a = demo.register(paths[0], paths[1], verbose=False, return_data=True)
    b = demo.register(paths[0], paths[1], verbose=False)
    assert a["missing_keys"] == [] and a["vertices"] == [len(p) for p in points]
    assert a["key_points"] == [5333, 5131] and a["correspondences"] == a["key_points"][0]     # those of the full clouds
    assert a["inliers"] > 500
    assert a["coverage_before"] < 0.3 and a["coverage_after"] > 0.8
    R = a["final_trans"][:3, :3]
    assert np.allclose(R @ R.T, np.eye(3), atol=1e-5) and np.linalg.det(R) > 0
    assert np.array_equal(a["final_trans"], b["final_trans"]) and a["inliers"] == b["inliers"]
    # the hot path on REAL correspondences (N = 5 333, ~20 % inliers) against the CPU checker: the 1e-4 bar on R / t
    from oracle import pointdsc_oracle as O
    sd = load_snapshot("3dmatch")
    d = {k: v[0].float().cpu() for k, v in a["data"].items()}
    want = O.forward_testing(sd, O.default_config("3dmatch"), d["corr_pos"], d["src_keypts"], d["tgt_keypts"])
    assert np.abs(a["final_trans"] - want["final_trans"].numpy()).max() <= 1e-4
    assert int((a["final_labels"][0].cpu() != want["final_labels"]).sum()) <= 2


@pytest.mark.parametrize("precision", ["fp16x3", "fp32"])
def test_reference_fixture_of_the_demo_pair(precision):
    """Real data, reference-generated: tests/golden/demo_pair_3dmatch.npz holds the 5 333 correspondences of the reference's demo
    pair and what the UNMODIFIED reference module returned for them on CPU (tests/golden/make_demo_golden.py).

    On this pair the reference's argmax over the hypotheses' inlier counts is razor thin — 1061 for its winner, 1060 for SEVEN
    others, 1059 / 1058 behind them — so WHICH of these near-identical hypotheses wins is decided by rounding-level differences of
    the features (profiles/r02_demo_pair_diag.txt).  The exact-arithmetic mode (fp32) reproduces the reference's choice and meets
    the 1e-4 bar; the default fp16x3 mode picks another member of the tied group (seed 96: 1060 in the reference, 1063 here), and
    the refinement then settles 6e-4 away.  The test pins exactly that: fp32 to the bar, fp16x3 to "a hypothesis the reference
    itself scores within 2 of its maximum, the same registration to 2e-3"."""
    import os
    from conftest import GOLDEN
    from pointdsc_b200 import PointDSC
    z = np.load(os.path.join(GOLDEN, "demo_pair_3dmatch.npz"))
    n = len(z["final_labels"])
    model = PointDSC(in_dim=6, num_layers=12, num_channels=128, num_iterations=10, ratio=0.1, inlier_threshold=0.10, sigma_d=0.10,
                     k=40, nms_radius=0.10, precision=precision).cuda().eval()
    model.load_state_dict(load_snapshot("3dmatch"), strict=False)
    d = [_dev(z[k])[None] for k in ("corr_pos", "src_keypts", "tgt_keypts")]
    for batch in (1, 3):                      # bs = 1 (key-split attention) and a small batch (unsplit)
        out = model.run(*[x.repeat(batch, 1, 1) for x in d], taps=["best", "seeds"])
        dT = np.abs(out["final_trans"][batch - 1].cpu().numpy() - z["final_trans"]).max()
        flips = int((out["final_labels"][batch - 1].cpu().numpy() != z["final_labels"]).sum())
        best = int(out["best"][batch - 1])
        ref_counts = np.round(z["fitness"] * n)
        assert ref_counts[best] >= ref_counts.max() - 2, (best, ref_counts[best], ref_counts.max())
        assert np.array_equal(out["seeds"][batch - 1].cpu().numpy()[:100], z["seeds"][:100])     # the untied head of the seed list
        if precision == "fp32":
            assert best == int(z["best"]) and dT <= 1e-4 and flips <= 2, (dT, flips, best)
        else:
            assert dT <= 2e-3 and flips <= n // 100, (dT, flips, best)
