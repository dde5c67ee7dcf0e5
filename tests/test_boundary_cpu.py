"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every declared symbol,
the nn.Module mirrors the reference's state dict, and nothing computes without a GPU."""
import ctypes
import os
import re

import pytest
import torch

from conftest import REPO, load_snapshot


def _header_symbols():
    text = open(os.path.join(REPO, "include", "pointdsc_b200.h")).read()
    return sorted(set(re.findall(r"\b(pdsc_[a-z_]+)\s*\(", text)))


def test_library_builds_and_exports_every_header_symbol():
    import __graft_entry__ as g
    g.build()
    from pointdsc_b200 import _capi
    lib = ctypes.CDLL(_capi.LIB_PATH)
    declared = _header_symbols()
    assert len(declared) >= 13
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/pointdsc_b200.h but not exported"
    assert sorted(_capi.SYMBOLS) == declared          # the ctypes binding covers the header, no more, no less
    assert b"sm_100a" in _capi.load().pdsc_version()


def test_struct_layouts_match_the_header():
    from pointdsc_b200 import _capi
    assert ctypes.sizeof(_capi.Config) == 11 * 4
    # 5 injection + 14 tap pointers, int32 layer_tap (+4 pad), 3 pointers
    assert ctypes.sizeof(_capi.StageIO) == 19 * 8 + 8 + 24
    assert _capi.StageIO.layer_tap.offset == 19 * 8
    assert _capi.StageIO.out_layer_features.offset == 19 * 8 + 8


@pytest.mark.parametrize("dataset", ["3dmatch", "kitti"])
def test_released_snapshot_loads_unchanged(dataset):
    from pointdsc_b200 import PointDSC
    m = PointDSC(in_dim=6, num_layers=12, num_channels=128, num_iterations=10, ratio=0.1, k=40)
    sd = load_snapshot(dataset)
    res = m.load_state_dict(sd, strict=False)
    assert res.missing_keys == [] and res.unexpected_keys == ["gamma"]     # as the reference reports
    own = m.state_dict()
    assert len(own) == 358
    assert sum(p.numel() for p in m.parameters()) == 1053667       # SURVEY.md §8 a14
    for k, v in own.items():
        assert torch.equal(v, sd[k]), k
    assert m.sigma.requires_grad and not m.sigma_spat.requires_grad


def test_constructor_defaults_match_the_reference():
    import inspect

    from pointdsc_b200 import PointDSC
    sig = inspect.signature(PointDSC.__init__)
    want = dict(in_dim=6, num_layers=6, num_channels=128, num_iterations=10, ratio=0.1, inlier_threshold=0.10,
                sigma_d=0.10, k=40, nms_radius=0.10)
    got = {k: v.default for k, v in sig.parameters.items() if k in want}
    assert got == want
    assert list(sig.parameters)[1:10] == list(want)    # positional order as in models/PointDSC.py:81-91


def test_no_cpu_fallback():
    from pointdsc_b200 import PdscError, PointDSC
    m = PointDSC(num_layers=2)
    data = {"corr_pos": torch.zeros(1, 16, 6), "src_keypts": torch.zeros(1, 16, 3), "tgt_keypts": torch.zeros(1, 16, 3),
            "testing": True}
    with pytest.raises(PdscError):
        m(data)
    with pytest.raises(NotImplementedError):
        m({k: v for k, v in data.items() if k != "testing"})


def test_descriptor_entry_points_reject_bad_arguments_without_a_device():
    """Row f2's C-ABI entries validate before they touch CUDA; the Python wrappers refuse CPU tensors (no fallback)."""
    from pointdsc_b200 import PdscError, _capi, descriptors
    lib = _capi.load()
    assert lib.pdsc_voxel_down_sample(None, 10, None, 0.05, None, None, None, None, 0, None) != 0
    assert b"null engine" in lib.pdsc_last_error()
    assert lib.pdsc_estimate_normals(None, 10, None, 0.1, 30, None, None, None, 0, None) != 0
    assert lib.pdsc_compute_fpfh(None, 10, None, None, 0.25, 100, 0, None, None, None, 0, None) != 0
    assert lib.pdsc_voxel_down_sample_scratch_bytes(0) == 0 and lib.pdsc_fpfh_scratch_bytes(0, 100) == 0
    n = 100000
    slots = 262144                      # the next power of two >= 2 n
    assert lib.pdsc_voxel_down_sample_scratch_bytes(n) == 32 + slots * 36 + n * 12
    assert lib.pdsc_fpfh_scratch_bytes(5000, 100) == 5000 * 100 * 4 + 5000 * 4 + 16 + 5000 * 33 * 8
    for fn in (lambda: descriptors.voxel_down_sample(torch.zeros(8, 3), 0.05), lambda: descriptors.estimate_normals(torch.zeros(8, 3), 0.1),
               lambda: descriptors.compute_fpfh(torch.zeros(8, 3), torch.zeros(8, 3), 0.25)):
        with pytest.raises(PdscError):
            fn()


def test_engine_creation_fails_without_a_device():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pointdsc_b200 import _capi
    lib = _capi.load()
    cfg = _capi.Config(6, 12, 128, 10, 0.1, 0.1, 0.1, 40, 0.1, 0, 0)
    h = ctypes.c_void_p()
    assert lib.pdsc_create(ctypes.byref(cfg), ctypes.byref(h)) != 0
    assert b"no CUDA device" in lib.pdsc_last_error()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(REPO, "pointdsc_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(root, f)).read()
                assert "oracle" not in text.replace("oracle/", "").replace("CPU oracle", "") or f == "synth.py", f


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the engine) prints ONE JSON line with the contract's
    keys; a reduced configuration keeps it to a few seconds here."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--n", "160", "--batch", "2"], capture_output=True, text=True, timeout=300, check=True).stdout
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "sets/s" and d["higher_is_better"] is True
    assert d["metric"] == "correspondence-sets/sec (PointDSC.forward, N=160, B=2)"   # not the headline label
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["value"] > 0 and d["gpu_launches"] == 0
    # "reference": the unmodified module from baseline/_ref (installed by __graft_entry__.build() where /root/reference exists);
    # "port": the oracle restatement, when that install is absent
    assert d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_bench_dump_outputs_names_and_size_cap(tmp_path):
    """`bench.py --dump-outputs`: one float32 .npy per returned array; above 64 MB a seeded sample of the sets, the same one
    every run, with its indices."""
    import numpy as np

    import bench
    out = {"final_trans": torch.randn(5, 4, 4), "final_labels": torch.rand(5, 7)}
    bench.dump_outputs(str(tmp_path / "all"), out, 0, 1)
    assert sorted(os.listdir(tmp_path / "all")) == ["final_labels.npy", "final_trans.npy"]
    for k, v in out.items():
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.numpy())
    B, N = 3000, 6000                                   # 72 MB of outputs
    big = {"final_trans": torch.arange(B * 16, dtype=torch.float32).reshape(B, 4, 4), "final_labels": torch.zeros(B, N)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big, 0, 1)
    sets = np.load(tmp_path / "a" / "sets.npy")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    assert len(sets) > 2700 and np.array_equal(sets, np.load(tmp_path / "b" / "sets.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "final_trans.npy"), big["final_trans"].numpy()[sets.astype(np.int64)])


@pytest.mark.gpu
def test_bench_dumps_what_the_timed_steps_returned(tmp_path):
    """The arrays `bench.py --dump-outputs` writes are what the module returns for the benchmark's seeded inputs."""
    import subprocess
    import sys

    import numpy as np

    import bench
    from pointdsc_b200 import PointDSC
    subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "2", "--warmup", "1", "--n", "160", "--batch", "3",
                    "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                   timeout=600, check=True)
    model = PointDSC(in_dim=6, num_layers=12, num_channels=128, num_iterations=10, ratio=0.1, k=40, **bench.CTOR["3dmatch"])
    model.load_state_dict(load_snapshot("3dmatch"), strict=False)
    model = model.cuda().eval()
    x = bench.make_inputs(160, 3, "3dmatch", 0)
    want = model.run(*(x[k].cuda() for k in ("corr_pos", "src_keypts", "tgt_keypts")))
    assert sorted(os.listdir(tmp_path)) == ["final_labels.npy", "final_trans.npy"]
    for k in ("final_trans", "final_labels"):
        assert np.array_equal(np.load(tmp_path / f"{k}.npy"), want[k].cpu().numpy()), k
