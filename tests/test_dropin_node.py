"""The drop-in boundary (SURVEY.md §8(b)): the reference's OWN node sources — src/liodom_node.cc and
src/liodom_mapping_node.cc — compiled unmodified against this repo's facade headers (include/liodom/*.h in
-DLIODOM_FACADE_USE_PCL mode: real pcl / Eigen / ros / tf type names, here provided by the API shim oracle/refshim/)
and linked with the facade + CUDA library.  `make -C oracle dropin` is the recipe; only `main` is renamed.

CPU part: the libraries build and export the node mains.  GPU part: the reference's main() drives the CUDA path and
its published odometry / maps equal what the C ABI gives directly."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle
from oracle import ref
from conftest import get_sequence, pose_err

pytestmark = pytest.mark.skipif(not ref.dropin_available(), reason="needs the upstream liodom sources (LIODOM_REFERENCE_ROOT) or a prebuilt oracle/_ref")


def _pose_from_odom(row):
    from scipy.spatial.transform import Rotation
    T = np.eye(4)
    T[:3, :3] = Rotation.from_quat(row[:4]).as_matrix()
    T[:3, 3] = row[4:7]
    return T


def test_dropin_libraries_build_and_export_the_reference_mains():
    paths = ref.build_dropin()
    assert paths is not None
    for path, sym in zip(paths, ("liodom_node_main", "liodom_mapping_node_main")):
        out = subprocess.run(["nm", "-D", "--defined-only", "-C", path], capture_output=True, text=True).stdout
        assert sym + "(int, char**)" in out, "%s does not define the reference's main (%s)" % (path, sym)
        # the facade classes the node instantiates come from this repo's facade, not from the reference's library
        assert "liodom::FeatureExtractor::operator()(std::atomic<bool>&)" in out or "mapping" in path
        assert "liodom::Map::updateMap" in out or "mapping" not in path
        ctypes.CDLL(path)   # loads (and with it libliodom_b200.so)


@pytest.mark.gpu
def test_reference_liodom_node_main_over_the_cuda_facade(cuda_lib):
    """src/liodom_node.cc main(): params -> FeatureExtractor / LaserOdometer worker threads -> lidarClb -> published
    nav_msgs/Odometry, all through this repo's facade; poses equal the C ABI's and the oracle's."""
    from liodom_b200 import api
    scans, _ = get_sequence("hdl64_small", 1000, 8)
    odom, ne, produced = ref.dropin_node_run(scans, prev_frames=15, save_results="false")
    assert produced == len(scans)
    ctx = api.Context(prev_frames=15, max_points=32768)
    op = oracle.make_params(prev_frames=15)
    oposes, _, _ = oracle.run_sequence(op, scans)
    for f, s in enumerate(scans):
        ctx.scan_batch([s])
        p, n = ctx.results()
        assert ne[f] == n[0]
        T = _pose_from_odom(odom[f])
        dt, dr = pose_err(T, p[0])
        assert dt < 1e-9 and dr < 1e-9, (f, dt, dr)          # same kernels behind both entry points
        dt, dr = pose_err(T, oposes[f])
        assert dt < 1e-4 and dr < 1e-5, (f, dt, dr)
        if f > 0:   # twist = delta pose / dt (src/laser_odometry.cc:412-432)
            assert np.all(np.isfinite(odom[f][7:13]))
    ctx.close()


@pytest.mark.gpu
def test_reference_mapping_node_main_over_the_cuda_map(cuda_lib):
    """src/liodom_mapping_node.cc main(): lidarClb -> TF lookup -> Map::updateMap -> getMap / getLocalMap -> published
    clouds, through this repo's Map facade; equal to the C ABI Map fed the same clouds and poses."""
    from liodom_b200 import api
    op = oracle.make_params()
    scans, gt = get_sequence("hdl64_small", 1000, 12)
    clouds = [oracle.extract_scan(op, s)[0] for s in scans]
    poses = [np.linalg.inv(gt[0]) @ g for g in gt]
    sizes, last_local, last_map = ref.dropin_mapping_run(clouds, poses)     # node defaults: 40 / 50 / 0.4, cells 2 / 1
    gm = api.Map(40.0, 50.0, 0.4, max_points=1 << 19)
    for f, (c, T) in enumerate(zip(clouds, poses)):
        # the node converts the pose to a tf quaternion and back (tf::transformTFToEigen): feed the Map the same matrix
        from scipy.spatial.transform import Rotation
        gm.update(c, T)
        assert abs(len(gm.get_local_map(T, 2, 1)) - sizes[f]) <= max(2, sizes[f] // 500), f
    assert last_map is not None and abs(len(last_map) - gm.size()[0]) <= max(2, gm.size()[0] // 500)
    gm.close()
