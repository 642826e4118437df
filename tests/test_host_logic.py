"""CPU tests of the host-side mirror (parameter mapping, factories, error behaviour) and of bench.py's helpers; one -m gpu run
of bench.py's output dump."""
import os
import sys

import numpy as np
import pytest

from open3d_slam_b200 import _lib as L
from open3d_slam_b200 import dist
from open3d_slam_b200 import engine as E
from open3d_slam_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_parameter_mapping():
    p = E.MapperParameters(seed=9)
    p.icp.maxNumIter = 17; p.icp.maxCorrespondenceDistance = 0.45; p.icp.knn = 7; p.icp.maxDistanceKnn = 1.25
    p.scanProcessing.voxelSize = 0.3; p.scanProcessing.downSamplingRatio = 0.25
    p.scanProcessing.cropper = E.ScanCroppingParameters("Cylinder", 1.0, 40.0, -3.0, 5.0)
    p.mapBuilder.mapVoxelSize = 0.2
    cfg = p.to_config()
    assert (cfg.icp.max_iter, cfg.icp.max_corr_dist, cfg.icp.knn, cfg.icp.knn_radius) == (17, 0.45, 7, 1.25)
    assert cfg.scan.voxel_size == 0.3 and cfg.scan.downsampling_ratio == 0.25 and cfg.scan.seed == 9 and cfg.map_voxel_size == 0.2
    c = cfg.scan.scan_matcher_cropper
    assert (c.kind, c.rmin, c.rmax, c.zmin, c.zmax) == (L.CROP_CYLINDER, 1.0, 40.0, -3.0, 5.0)
    assert cfg.scan.map_builder_cropper.kind == L.CROP_MINMAX_RADIUS


def test_factories_mirror_the_reference_errors():
    p = E.MapperParameters()
    p.scanToMapRegType = "NoSuchIcp"
    with pytest.raises(L.B2SError) as ei:
        p.to_config()
    assert ei.value.code == L.E_UNSUPPORTED
    p.scanToMapRegType = "GeneralizedIcp"
    assert p.to_config().icp.reg_type == L.REG_GENERALIZED
    with pytest.raises(RuntimeError):
        E.cloudRegistrationFactory(None, E.CloudRegistrationParameters(regType="NoSuchIcp"))
    p.scanToMapRegType = "PointToPointIcp"
    assert p.to_config().icp.reg_type == L.REG_POINT_TO_POINT


def test_synthetic_data_is_deterministic_and_sane():
    scene = synth.Scene(); poses = synth.loop_trajectory(5)
    a = synth.lidar_scan(scene, poses[1], seed=3); b = synth.lidar_scan(scene, poses[1], seed=3)
    assert a.dtype == np.float32 and np.array_equal(a, b) and 40000 < len(a) <= 65536
    r = np.linalg.norm(a, axis=1)
    assert r.min() > 0.5 and r.max() < 60.0
    c = synth.lidar_from_cast(synth.lidar_cast(scene, poses[1]), 0.02, seed=3)
    assert c.shape == a.shape and np.abs(c - a).max() < 1e-4
    assert abs(np.linalg.norm(poses[1][:3, 3] - poses[0][:3, 3]) - 0.5) < 0.01
    src, tgt, nrm, T = synth.planar_cloud_config1()
    assert src.shape == (2000, 3) and np.allclose(np.linalg.norm(nrm, axis=1), 1.0)


def test_shard_range_is_a_partition():
    for n in (0, 1, 7, 512, 513):
        for world in (1, 2, 3, 8):
            parts = [dist.shard_range(n, world, r) for r in range(world)]
            flat = [i for p in parts for i in p]
            assert flat == list(range(n))
            sizes = [len(p) for p in parts]
            assert max(sizes) - min(sizes) <= 1


def test_bench_reference_arm_smoke():
    """bench.py --impl reference runs the oracle-only arm (tiny sizes) and prints one JSON line with the contract keys."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3", "--chains", "2"],
                         capture_output=True, text=True, timeout=600, env={**os.environ, "OMP_NUM_THREADS": "4"})
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "config", "cpu_baseline", "e2e"):
        assert k in line
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    # both arms describe the workload with the SAME function of the SAME flags (the driver compares the two `config` objects)
    import argparse
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"config": make_config(args)') == 2          # one per arm, nothing arm-specific inside
    ns = argparse.Namespace(chains=2, scans_per_step=64, ratio=0.3)
    cfg = bench.make_config(ns)
    assert cfg == line["config"] or {k: v for k, v in cfg.items() if k != "chains_per_gpu"} == {k: v for k, v in line["config"].items() if k != "chains_per_gpu"}
    assert set(cfg) == set(line["config"])


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs (small run): the last timed step's results of every chain and scan, poses, map sizes and a map
    sample, float64, within 64 MB, and consistent with what the JSON line reports about the same step."""
    import json
    import subprocess
    chains, steps, spp = 2, 2, 4
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--chains", str(chains), "--steps", str(steps), "--warmup", "3",
                          "--scans-per-step", str(spp), "--no-extras", "--no-sweep", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    d = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
    assert all(a.dtype == np.float64 for a in d.values())
    assert d["transformation"].shape == (chains, spp, 4, 4) and d["pose"].shape == (chains, 4, 4)
    for k in ("fitness", "inlier_rmse", "n_corr", "iters"):
        assert d[k].shape == (chains, spp)
    assert d["map_xyz_sample"].shape == d["map_normals_sample"].shape and d["map_xyz_sample"].shape[:2] == (chains, 16384)
    obs = line["observed"]
    assert d["fitness"][:, -1].min() == obs["min_fitness_last_scan"] and int(d["map_size"].mean()) == obs["map_points"]
    acc = d["fitness"][:, -1] >= 0.7                    # fitness gate passed: the chain's pose is that scan's result
    assert acc.any() and np.array_equal(d["transformation"][acc, -1], d["pose"][acc])


def test_reference_side_shim_type_checks():
    """shim/b2s_open3d_slam.cpp (the C++ subclasses of CloudRegistration / ScanToMapRegistration) compiles against the
    C header and stand-in Open3D/Eigen declarations."""
    import subprocess
    out = subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "shim"), "check"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
