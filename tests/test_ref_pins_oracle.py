"""Pins the restated oracle (oracle/liodom_oracle.cc) against the REFERENCE'S OWN object code:
oracle/_ref/libliodom_ref.so = /root/reference/src/{feature_extractor,laser_odometry,map,params,
shared_data,stats}.cc compiled unmodified (make -C oracle ref) against the API shim oracle/refshim/.

What this pins, per SURVEY.md §8(a) row:
  A1-A4  isValidPoint / splitPointCloud / extractFeatures / extractFeaturesFromRegion: the reference's own
         arithmetic and control flow -> ring clouds and edge lists BIT-EXACT.
  A5     LocalMapManager (incl. the `if`-not-`while` eviction).
  A7-A11 LaserOdometer::operator(): the reference's control flow, prediction algebra, association loop,
         Ceres problem set-up and its Point2LineFactor functor (differentiated by Jets), over shim
         restatements of the third-party calls (PCL transform / kNN / VoxelGrid, Eigen, Ceres LM, tf).
  A12-A13 Map::updateMap / getMap / getLocalMap / getMapEntropy: key arithmetic, creation order, loops.
  (f)4   Stats::writeResults file formats, publishOdom arithmetic.
Still unpinned (third-party source absent, restated on both sides): FLANN's tie order among equal
distances, VoxelGrid's in-voxel order under an unstable sort, Eigen's eigen-solver to the last ulp,
Ceres' trust-region loop.
"""
import os

import numpy as np
import pytest

import oracle
from oracle import ref
from conftest import get_sequence, pose_err

pytestmark = pytest.mark.skipif(not ref.available(), reason="needs the upstream liodom sources (LIODOM_REFERENCE_ROOT) or a prebuilt oracle/_ref")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _setup(**kw):
    """Same parameters on both sides: ROS names for the reference, oracle.Params for the oracle."""
    ref.set_params(**kw)
    okw = {k: (int(v) if isinstance(v, bool) else v) for k, v in kw.items() if k not in ("use_imu", "save_results", "publish_tf")}
    return oracle.make_params(**okw)


# ---------------------------------------------------------------------------------------------------
def test_params_defaults_and_launch_overrides():
    """src/params.cc:40-108 defaults; launch/liodom.launch:17-31 overrides."""
    ref.set_params()
    p = ref.get_params()
    op = oracle.make_params()
    assert (p["min_range"], p["max_range"]) == (op.min_range, op.max_range) == (3.0, 75.0)
    assert (p["lidar_type"], p["scan_lines"], p["scan_regions"], p["edges_per_region"]) == (0, 64, 8, 10)
    assert p["local_map_size"] == op.prev_frames == 5
    assert p["min_points_per_scan"] == 8 * 10 + 10
    assert (p["use_imu"], p["filter_local_map"], p["mapping"], p["publish_tf"], p["save_results"]) == (0, 0, 0, 1, 0)
    ref.set_params(prev_frames=15, scan_regions=16, edges_per_region=20, mapping=True)
    p = ref.get_params()
    assert p["local_map_size"] == 15 and p["min_points_per_scan"] == 330 and p["mapping"] == 1


def test_is_valid_point_boundaries():
    """isValidPoint (src/feature_extractor.cc:84-102): XY range, inclusive bounds, non-finite inputs."""
    op = _setup()
    fe = ref.FeatureExtractor()
    pts = []
    for d in (2.9999999, 3.0, 3.0000001, 74.9999999, 75.0, 75.0000001):
        pts.append([d, 0.0, 0.5, 0.0])
        pts.append([0.0, -d, 40.0, 0.0])          # z does not count
    pts += [[np.nan, 5, 0, 0], [5, np.inf, 0, 0], [5, 5, -np.inf, 0], [0, 0, 0, 0]]
    pts = np.array(pts, np.float32)
    o = oracle.split(op, pts)
    for i, p in enumerate(pts):
        ok, dist = fe.is_valid_point(float(p[0]), float(p[1]), float(p[2]))
        if ok:
            assert dist == np.sqrt(float(p[0]) ** 2 + float(p[1]) ** 2)
        else:
            assert o["ring_of_point"][i] == -1   # invalid for the reference -> dropped by the oracle
    # and the split as a whole agrees
    r = fe.split(pts)
    assert np.array_equal(r["offsets"], o["offsets"]) and np.array_equal(_bits(r["rings"]), _bits(o["rings"]))


@pytest.mark.parametrize("sensor", ["hdl64", "hdl64_firing", "hdl64_small"])
def test_split_and_extract_hdl64_bit_exact(sensor):
    op = _setup(prev_frames=15)
    fe = ref.FeatureExtractor()
    for s in get_sequence(sensor, 1001, 2)[0]:
        r, o = fe.split(s), oracle.split(op, s)
        assert np.array_equal(r["offsets"], o["offsets"])
        assert np.array_equal(_bits(r["rings"]), _bits(o["rings"]))
        for mode in (0, 1):   # literal std::sort and the total order the GPU implements
            oe = oracle.extract(op, o["rings"], o["offsets"], sort_mode=mode)["edges"]
            re_ = fe.extract(r["rings"], r["offsets"])
            assert len(re_) > 1000 and np.array_equal(_bits(re_), _bits(oe))
        assert np.array_equal(_bits(fe.process(s)), _bits(oe))   # through the worker functor + SharedData queues


@pytest.mark.parametrize("lines", [16, 32])
def test_split_vlp16_hdl32_bit_exact(lines):
    """Ring formulas for scan_lines 16 / 32 (src/feature_extractor.cc:139-148) on random rays."""
    rng = np.random.default_rng(lines)
    n = 20000
    az = rng.uniform(-np.pi, np.pi, n)
    el = np.deg2rad(rng.uniform(-35, 20, n))
    rr = rng.uniform(1, 90, n)
    pts = np.stack([rr * np.cos(el) * np.cos(az), rr * np.cos(el) * np.sin(az), rr * np.sin(el), rng.uniform(0, 1, n)], 1).astype(np.float32)
    op = _setup(scan_lines=lines)
    fe = ref.FeatureExtractor()
    r, o = fe.split(pts), oracle.split(op, pts)
    assert np.array_equal(r["offsets"], o["offsets"]) and np.array_equal(_bits(r["rings"]), _bits(o["rings"]))
    assert np.array_equal(_bits(fe.extract(r["rings"], r["offsets"])), _bits(oracle.extract(op, o["rings"], o["offsets"])["edges"]))


def test_points_near_ring_bin_boundaries():
    """Rays 1e-7 .. 1e-2 degrees either side of every HDL-64 bin edge: same ring in both."""
    op = _setup()
    fe = ref.FeatureExtractor()
    edges_deg = [2 - (k - 0.5) / 3 for k in range(0, 33)] + [-8.83 - (k - 0.5) / 2 for k in range(0, 33)] + [2.0, -24.33, -8.83]
    pts = []
    for e in edges_deg:
        for eps in (1e-7, 1e-5, 1e-3, 1e-2):
            for sgn in (-1, 1):
                el = np.deg2rad(e + sgn * eps)
                pts.append([20 * np.cos(el), 0.0, 20 * np.sin(el), 0.0])
    pts = np.array(pts, np.float32)
    r, o = fe.split(pts), oracle.split(op, pts)
    assert np.array_equal(r["offsets"], o["offsets"]) and np.array_equal(_bits(r["rings"]), _bits(o["rings"]))


def test_ouster_c2_bit_exact():
    from liodom_b200 import synth
    w, h = synth.sensor_shape("os1_128")
    op = _setup(lidar_type=1, scan_lines=128, prev_frames=15)
    fe = ref.FeatureExtractor()
    s = get_sequence("os1_128", 1000, 1)[0][0]
    r, o = fe.split(s, w, h), oracle.split(op, s, w, h)
    assert np.array_equal(r["offsets"], o["offsets"]) and np.array_equal(_bits(r["rings"]), _bits(o["rings"]))
    re_ = fe.extract(r["rings"], r["offsets"])
    assert len(re_) > 3000 and np.array_equal(_bits(re_), _bits(oracle.extract(op, o["rings"], o["offsets"])["edges"]))


def test_extract_stress_c3_and_edge_cases():
    op = _setup(scan_regions=16, edges_per_region=20, prev_frames=20)
    fe = ref.FeatureExtractor()
    s = get_sequence("hdl64", 1003, 1)[0][0]
    o = oracle.split(op, s)
    assert np.array_equal(_bits(fe.extract(o["rings"], o["offsets"])), _bits(oracle.extract(op, o["rings"], o["offsets"])["edges"]))
    # short / threshold / ragged rings (min_points_per_scan_ = 90 with the defaults)
    op = _setup()
    fe = ref.FeatureExtractor()
    s = get_sequence("hdl64_small", 1000, 1)[0][0]
    sp = oracle.split(op, s)
    for take in (lambda r: 89, lambda r: 90, lambda r: 90 + 3 * r, lambda r: 91 if r % 2 else 0):
        keep = np.concatenate([sp["src_index"][sp["offsets"][r]:sp["offsets"][r + 1]][:take(r)] for r in range(64)])
        sub = s[np.sort(keep)]
        r, o = fe.split(sub), oracle.split(op, sub)
        assert np.array_equal(r["offsets"], o["offsets"])
        assert np.array_equal(_bits(fe.extract(r["rings"], r["offsets"])), _bits(oracle.extract(op, o["rings"], o["offsets"])["edges"]))
    assert len(fe.process(np.zeros((0, 4), np.float32))) == 0   # empty scan


def test_local_map_manager():
    """LocalMapManager::addPointCloud / getLocalMap / setMaxFrames (src/laser_odometry.cc:24-69)."""
    ref.set_params()
    rng = np.random.default_rng(1)
    rm, om = ref.LocalMapManager(5), oracle.LocalMapManager(5)
    for f in range(12):
        n = int(rng.integers(0, 400)) if f != 3 else 0
        pts = rng.normal(size=(n, 4)).astype(np.float32)
        rm.add(pts); om.add(pts)
        (r, rf), (o, of) = rm.get(), om.get()
        assert rf == of == min(f + 1, 5) and np.array_equal(_bits(r), _bits(o))
    rm.set_max_frames(3); om.set_max_frames(3)   # ONE frame dropped per add (`if`, not `while`)
    for f in range(4):
        pts = rng.normal(size=(50, 4)).astype(np.float32)
        rm.add(pts); om.add(pts)
        (r, rf), (o, of) = rm.get(), om.get()
        assert rf == of and np.array_equal(_bits(r), _bits(o))


def test_point2line_factor_autodiff_of_the_reference_functor():
    """Point2LineFactor::operator() (include/liodom/factors.hpp:71-105) evaluated by the reference's own
    template code, with T = double and T = Jet, vs the oracle's restatement: residuals and the 3x6
    tangent Jacobian, including the negative-weight regime beyond ~75.7 m."""
    rng = np.random.default_rng(0)
    worst_r = worst_j = 0.0
    for k in range(400):
        c = rng.normal(size=3) * [25, 25, 2]
        q = rng.normal(size=4) * [0.05, 0.05, 0.3, 1.0]
        q /= np.linalg.norm(q)
        if k % 7 == 0:
            q = -q                      # w < 0: the slerp branch that flips the sign
        t = rng.normal(size=3) * ([200, 200, 1] if k % 3 == 0 else [5, 5, 0.2])
        a = c + rng.normal(size=3) * 0.3
        b = a + rng.normal(size=3) * 0.5
        r, Jq, Jt, Jl = ref.factor(c, a, b, q, t)
        ro, Jo = oracle.factor(c, a, b, q, t)
        # T = double vs the value part of T = Jet: Jet division multiplies by the reciprocal (as ceres/jet.h does)
        assert np.allclose(ref.factor_residual(c, a, b, q, t), r, rtol=1e-12, atol=1e-11)
        worst_r = max(worst_r, np.abs(r - ro).max() / max(1.0, np.abs(ro).max()))
        worst_j = max(worst_j, np.abs(Jl - Jo).max() / max(1.0, np.abs(Jo).max()))
    assert worst_r < 1e-14 and worst_j < 1e-13, (worst_r, worst_j)


def _free_run(sensor, seed, nframes, width=0, height=0, tol=(1e-9, 1e-10), **kw):
    op = _setup(**kw)
    scans, _ = get_sequence(sensor, seed, nframes)
    rposes, rne = ref.run_sequence(scans, width, height)
    oposes, _, _ = oracle.run_sequence(op, scans, width, height)
    one = [len(oracle.extract_scan(op, s, width, height)[0]) for s in scans]
    assert list(rne) == one
    worst = (0.0, 0.0)
    for f in range(nframes):
        dt, dr = pose_err(rposes[f], oposes[f])
        assert dt < tol[0] and dr < tol[1], "frame %d: %g m %g rad" % (f, dt, dr)
        worst = (max(worst[0], dt), max(worst[1], dr))
    return worst


def test_node_pipeline_free_running_c1():
    """lidarClb -> FeatureExtractor worker -> SharedData -> LaserOdometer worker (src/liodom_node.cc:40-91) on the
    C1 workload with launch/liodom.launch params, vs oracle.run_sequence."""
    w = _free_run("hdl64", 1000, 8, prev_frames=15)
    print("reference object code vs oracle, C1 free run: %.3g m %.3g rad" % w)


def test_node_pipeline_free_running_small_window_eviction():
    """prev_frames = 5 over 14 frames: the window fills and evicts (src/laser_odometry.cc:41-59)."""
    w = _free_run("hdl64_small", 1002, 14, prev_frames=5)
    print("reference object code vs oracle, small free run: %.3g m %.3g rad" % w)


def test_node_pipeline_filter_local_map():
    """filter_local_map = true: VoxelGrid(0.4) of the full window (src/laser_odometry.cc:286-292)."""
    _free_run("hdl64_small", 1001, 9, prev_frames=5, filter_local_map=True, tol=(1e-6, 1e-7))


def test_odometer_teacher_forced_with_received_map():
    """mapping = true: SharedData::setLocalMap feeds local_map_rec, merged into the kNN target and the window
    filter bypassed (src/laser_odometry.cc:276-278, :286, :312-314)."""
    op = _setup(prev_frames=5, mapping=True)
    scans, gt = get_sequence("hdl64_small", 1000, 8)
    edges = [oracle.extract_scan(op, s)[0] for s in scans]
    rod, ood = ref.Odometer(), oracle.Odometer(op)
    for f, e in enumerate(edges):
        if f >= 2:   # a "global map" made of the GT-posed edges of frames 0..f-2
            rec = np.concatenate([oracle.transform(edges[k], np.linalg.inv(gt[0]) @ gt[k]) for k in range(f - 1)])
            ref.set_received_map(rec)
            ood.set_received_map(rec)
        rp = rod.process(e)
        opose, od = ood.process(e)
        if f >= 2:
            assert od.n_map[0] > ood.window()[0].shape[0]   # the received map really took part
        dt, dr = pose_err(rp, opose)
        assert dt < 1e-9 and dr < 1e-10, (f, dt, dr)
    ref.set_received_map(np.zeros((0, 4), np.float32))


def test_odometer_use_imu_and_publish_odom():
    """use_imu roll/pitch override (src/laser_odometry.cc:152-183) with a non-identity base->laser transform, and
    the nav_msgs/Odometry that publishOdom fills (:395-446)."""
    from scipy.spatial.transform import Rotation
    op = _setup(prev_frames=5, use_imu=True)
    l2b_q = Rotation.from_euler("xyz", [0.01, -0.02, 0.3]).as_quat()
    l2b_t = [0.5, 0.1, -1.2]
    ref.set_static_tf("velo_link", "base_link", l2b_t, l2b_q)
    L2B = np.eye(4)
    L2B[:3, :3] = Rotation.from_quat(l2b_q).as_matrix()
    L2B[:3, 3] = l2b_t
    scans, _ = get_sequence("hdl64_small", 1003, 6)
    rod, ood = ref.Odometer(), oracle.Odometer(op)
    seq0 = max(rod.last_odom_msg()[1], 0)   # the shim's bus counts messages per topic over the whole process
    for f, s in enumerate(scans):
        imu_q = Rotation.from_euler("xyz", [0.002 * f, -0.003 * f, 1.0]).as_quat()
        ref.set_imu(imu_q)
        ood.set_imu(1, imu_q, L2B)
        e = oracle.extract_scan(op, s)[0]
        _, o_prev_before = ood.get_pose()
        rp = rod.process(e, dt=0.1)
        opose, _ = ood.process(e)
        dt, dr = pose_err(rp, opose)
        assert dt < 1e-9 and dr < 1e-10, (f, dt, dr)
        msg, seq = rod.last_odom_msg()
        assert seq == seq0 + f + 1
        if f > 0:
            o_odom, o_prev = ood.get_pose()
            expect = oracle.publish_odom(o_odom, o_prev, L2B, 0.1)
            assert np.allclose(msg, expect, rtol=0, atol=1e-8), (f, np.abs(msg - expect).max())


@pytest.mark.parametrize("xy,z,cxy,cz", [(40.0, 50.0, 2, 1), (30.0, 35.0, 3, 2), (20.0, 25.0, 2, 1)])
def test_map_matches_reference(xy, z, cxy, cz):
    """Map::updateMap / getMap / getLocalMap (src/map.cc:90-189) for the three shipped (xy, z, cells) settings."""
    from scipy.spatial.transform import Rotation
    ref.set_params()
    rng = np.random.default_rng(int(xy))
    rm, om = ref.Map(xy, z, 0.4), oracle.Map(xy, z, 0.4)
    T = np.eye(4)
    for f in range(12):
        n = int(rng.integers(1, 3000))
        pts = (rng.normal(size=(n, 4)) * [30, 30, 2, 1]).astype(np.float32)
        T[:3, :3] = Rotation.from_rotvec([0.01 * f, -0.02, 0.1 * f]).as_matrix()
        T[:3, 3] = [4.0 * f - 7.3, -1.5 * f, 0.05 * f]
        rm.update(pts, T); om.update(pts, T)
        (rk, rc), (ok, oc) = rm.cells(), om.cells()
        assert np.array_equal(rk, ok), "cell keys / creation order differ"
        assert np.array_equal(rc, oc), "per-cell counts differ"
        r, o = rm.get_map(), om.get_map()
        assert r.shape == o.shape
        # in-voxel accumulation order follows an unstable sort in PCL: centroids agree to a few ulps x count
        assert np.allclose(r, o, rtol=0, atol=2e-5)
        rl, ol = rm.get_local_map(T, cxy, cz), om.get_local_map(T, cxy, cz)
        assert rl.shape == ol.shape and np.allclose(rl, ol, rtol=0, atol=2e-5)
    assert len(rm.get_map()) > 1000


def test_map_replay_edge_clouds_c4_style():
    """C4-style replay (src/liodom_mapping_node.cc:45-90): edge clouds + GT poses -> updateMap -> getLocalMap."""
    op = _setup()
    scans, gt = get_sequence("hdl64_small", 1000, 25)
    rm, om = ref.Map(20.0, 25.0, 0.4), oracle.Map(20.0, 25.0, 0.4)   # launch/liodom_mapping.launch:15-19
    nexact = 0
    for f, s in enumerate(scans):
        edges = oracle.extract_scan(op, s)[0]
        T = np.linalg.inv(gt[0]) @ gt[f]
        rm.update(edges, T); om.update(edges, T)
        rl, ol = rm.get_local_map(T, 2, 1), om.get_local_map(T, 2, 1)
        assert rl.shape == ol.shape and np.allclose(rl, ol, rtol=0, atol=2e-5), f
        nexact += int(np.array_equal(_bits(rl), _bits(ol)))
    (rk, rc), (ok, oc) = rm.cells(), om.cells()
    assert np.array_equal(rk, ok) and np.array_equal(rc, oc) and len(rk) >= 9
    print("getLocalMap bitwise equal on %d of %d frames" % (nexact, len(scans)))


def test_stats_write_results_files(tmp_path):
    """Stats::writeResults (src/stats.cc:73-132): the five text files, default ostream precision, vs the façade."""
    from liodom_b200 import host_api
    if not os.path.exists(host_api.HOST_SO):
        pytest.skip("facade library not built")
    import ctypes
    lib = host_api.load()
    if not hasattr(lib, "liodom_host_stats_write"):
        pytest.skip("facade has no stats test hook")
    rng = np.random.default_rng(3)
    poses = []
    for k in range(7):
        T = np.eye(4)
        T[:3, :] = rng.normal(size=(3, 4)) * [1, 1, 1, 123.456]
        poses.append(T)
    nfeats = [5630, 0, 12, 99999, 3, 4, 5]
    times = [(3.0, 41.0), (0.0, 7.0), (12.0, 130.0), (1.0, 1.0), (2.0, 2.0), (5.0, 9.0), (7.0, 11.0)]
    d_ref, d_fac = tmp_path / "ref", tmp_path / "fac"
    d_ref.mkdir(); d_fac.mkdir()
    ref.stats_write(poses, nfeats, times, str(d_ref))
    P = np.ascontiguousarray(np.stack(poses).reshape(-1, 16))
    N = np.array(nfeats, np.int64)
    Tm = np.ascontiguousarray(np.array(times, np.float64))
    lib.liodom_host_stats_write(P.ctypes.data_as(ctypes.c_void_p), N.ctypes.data_as(ctypes.c_void_p), Tm.ctypes.data_as(ctypes.c_void_p),
                                len(poses), (str(d_fac) + "/").encode())
    for name in ("poses.txt", "feat_ext_times.txt", "laser_odom_times.txt", "nfeats.txt", "frame_times.txt"):
        a, b = (d_ref / name).read_text(), (d_fac / name).read_text()
        assert a == b, name
        assert len(a.splitlines()) == 7
