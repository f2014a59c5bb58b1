"""GPU parity: LaserOdometer path (window, voxel-hash 5-NN, line gate, LM solve) through the
C ABI against the oracle.  kNN sets / float distances / gates are bit-exact on teacher-forced
inputs; poses agree within 1e-4 m / 1e-5 rad (BASELINE.json north_star)."""
import numpy as np
import pytest

import oracle
from liodom_b200 import api
from conftest import get_sequence, pose_err

pytestmark = pytest.mark.gpu

TOL_T = 1e-4   # metres
TOL_R = 1e-5   # radians


def _edges_of(op, scans):
    out = []
    for s in scans:
        sp = oracle.split(op, s)
        out.append(oracle.extract(op, sp["rings"], sp["offsets"])["edges"])
    return out


def test_local_map_manager(cuda_lib):
    """LocalMapManager::addPointCloud / getLocalMap / setMaxFrames (src/laser_odometry.cc:24-69)."""
    rng = np.random.default_rng(1)
    ctx = api.Context(prev_frames=5, max_points=2048)
    om = oracle.LocalMapManager(5)
    for f in range(12):
        n = int(rng.integers(0, 400)) if f != 3 else 0   # an empty frame too
        pts = rng.normal(size=(n, 4)).astype(np.float32)
        ctx.lmap_add(pts)
        om.add(pts)
        g, gf = ctx.lmap_get()
        o, of = om.get()
        assert gf == of and gf == min(f + 1, 5)
        assert np.array_equal(g.view(np.uint32), o.view(np.uint32))
    # shrinking max_frames drops ONE frame per add (the reference's `if`, not `while`)
    ctx.lmap_set_max_frames(3)
    om.set_max_frames(3)
    for f in range(4):
        pts = rng.normal(size=(50, 4)).astype(np.float32)
        ctx.lmap_add(pts)
        om.add(pts)
        g, gf = ctx.lmap_get()
        o, of = om.get()
        assert gf == of
        assert np.array_equal(g.view(np.uint32), o.view(np.uint32))
    ctx.close()


def _teacher_forced_associate(ctx, edges_seq, gt, K):
    """Window = GT-posed edges of the previous frames; query = next frame at a perturbed pose."""
    nchecked = 0
    for f in range(1, len(edges_seq)):
        ctx.lmap_clear()
        frames = [oracle.transform(edges_seq[k], np.linalg.inv(gt[0]) @ gt[k]) for k in range(max(0, f - K), f)]
        for w in frames:
            ctx.lmap_add(w)
        window = np.concatenate(frames)
        T = np.linalg.inv(gt[0]) @ gt[f]
        T = T.copy()
        T[:3, 3] += [0.05, -0.03, 0.01]
        o = oracle.associate(edges_seq[f], T, window, knn_method=0)
        o_kd = oracle.associate(edges_seq[f], T, window, knn_method=1)
        g = ctx.associate(edges_seq[f], T)
        assert g["n_map"] == len(window)
        assert np.array_equal(g["q_world"].view(np.uint32), o["q_world"].view(np.uint32))
        assert np.array_equal(o["gate"], o_kd["gate"])
        ok = o["tie"] == 0
        assert np.array_equal(g["gate"][ok], o["gate"][ok])
        sel = ok & ((o["gate"] & 1) == 1)
        assert sel.sum() > 100
        assert np.array_equal(g["knn_idx"][sel], o["knn_idx"][sel])
        assert np.array_equal(o_kd["knn_idx"][sel], o["knn_idx"][sel])
        assert np.array_equal(g["knn_d2"][sel].view(np.uint32), o["knn_d2"][sel].view(np.uint32))
        sel2 = sel & ((o["gate"] & 2) == 2)
        assert np.array_equal(g["eig"][sel].view(np.uint64), o["eig"][sel].view(np.uint64))
        nchecked += int(sel2.sum())
    return nchecked


@pytest.mark.parametrize("group", ["1", "4", "8", "16", "pool", "thread"])
def test_associate_teacher_forced_c1(cuda_lib, group, monkeypatch):
    """Every kernel variant (1, 4, 8 or 16 threads per edge; picked by the number of edges in flight) and the warp-pooled
    form of the one-thread-per-edge search (LIODOM_ASSOC_POOL=1 / 0)."""
    monkeypatch.delenv("LIODOM_ASSOC_POOL", raising=False)
    if group in ("pool", "thread"):
        monkeypatch.setenv("LIODOM_ASSOC_POOL", "1" if group == "pool" else "0")
        group = "1"
    monkeypatch.setenv("LIODOM_ASSOC_GROUP", group)
    scans, gt = get_sequence("hdl64", 1000, 5)
    op = oracle.make_params(prev_frames=15)
    edges_seq = _edges_of(op, scans)
    ctx = api.Context(prev_frames=15, max_points=131072)
    assert _teacher_forced_associate(ctx, edges_seq, gt, 15) > 500
    ctx.close()


def test_associate_empty_and_tiny_maps(cuda_lib):
    ctx = api.Context(prev_frames=5, max_points=2048)
    rng = np.random.default_rng(3)
    q = rng.normal(size=(64, 4)).astype(np.float32)
    g = ctx.associate(q, np.eye(4))            # empty window: nothing passes the gate
    assert (g["gate"] == 0).all() and g["n_map"] == 0
    ctx.lmap_add(q[:4])                          # 4 points: the reference reads sq_dist[4] OOB (UB); gate fails here
    g = ctx.associate(q, np.eye(4))
    assert (g["gate"] == 0).all()
    ctx.lmap_add(np.zeros((0, 4), np.float32))
    ctx.lmap_add(q[4:40] * 0.1)
    o = oracle.associate(q, np.eye(4), np.concatenate([q[:4], q[4:40] * 0.1]))
    g = ctx.associate(q, np.eye(4))
    ok = o["tie"] == 0
    assert np.array_equal(g["gate"][ok], o["gate"][ok])
    sel = ok & ((o["gate"] & 1) == 1)
    assert np.array_equal(g["knn_idx"][sel], o["knn_idx"][sel])
    ctx.close()


def test_associate_nonfinite_map_points_skipped(cuda_lib):
    """PCL's kd-tree build skips non-finite points; indices still refer to the full cloud."""
    rng = np.random.default_rng(4)
    m = (rng.normal(size=(500, 4)) * 0.5).astype(np.float32)
    m[::7, 1] = np.nan
    q = (rng.normal(size=(100, 4)) * 0.5).astype(np.float32)
    ctx = api.Context(prev_frames=5, max_points=2048)
    ctx.lmap_add(m)
    o = oracle.associate(q, np.eye(4), m)
    g = ctx.associate(q, np.eye(4))
    sel = (o["tie"] == 0) & ((o["gate"] & 1) == 1)
    assert sel.sum() > 10
    assert np.array_equal(g["knn_idx"][sel], o["knn_idx"][sel])
    assert not np.isin(g["knn_idx"][sel], np.arange(0, 500, 7)).any()
    ctx.close()


def _blocks_from(o, edges, window):
    sel = (o["gate"] & 2) == 2
    idx = o["knn_idx"][sel]
    return np.concatenate([edges[sel][:, :3], window[idx[:, 0]][:, :3], window[idx[:, 1]][:, :3]], 1).astype(np.float64)


def test_solve_matches_oracle(cuda_lib):
    """One ceres::Solve restated on both sides (same residual blocks, same start)."""
    scans, gt = get_sequence("hdl64", 1000, 4)
    op = oracle.make_params(prev_frames=15)
    edges_seq = _edges_of(op, scans)
    ctx = api.Context(prev_frames=15, max_points=131072)
    window = np.concatenate([oracle.transform(edges_seq[k], np.linalg.inv(gt[0]) @ gt[k]) for k in range(3)])
    Tgt = np.linalg.inv(gt[0]) @ gt[3]
    for shift in ([0.0, 0.0, 0.0], [0.2, -0.1, 0.02], [0.5, 0.3, -0.05]):
        T = Tgt.copy()
        T[:3, 3] += shift
        o = oracle.associate(edges_seq[3], T, window)
        cab = _blocks_from(o, edges_seq[3], window)
        assert len(cab) > 200
        # start from the (x,y,z,w) quaternion of T
        q0, t0, _ = oracle.solve(np.zeros((0, 9)), [0, 0, 0, 1], T[:3, 3])
        from scipy.spatial.transform import Rotation
        q0 = Rotation.from_matrix(T[:3, :3]).as_quat()
        if q0[3] < 0:
            q0 = -q0
        oq, ot, osum = oracle.solve(cab, q0, T[:3, 3], linear_solver=0)
        gq, gt_, gsum = ctx.solve(cab, q0, T[:3, 3])
        assert gsum.num_residual_blocks == len(cab)
        assert (gsum.iterations, gsum.successful_steps, gsum.termination) == (osum.iterations, osum.successful_steps, osum.termination)
        assert np.abs(gt_ - ot).max() < 1e-7
        assert np.abs(gq - oq).max() < 1e-8
        assert abs(gsum.initial_cost - osum.initial_cost) <= 1e-9 * max(1.0, osum.initial_cost)
        assert abs(gsum.final_cost - osum.final_cost) <= 1e-7 * max(1.0, osum.final_cost)
    # no residual blocks: parameters untouched
    gq, gt_, gsum = ctx.solve(np.zeros((0, 9)), [0, 0, 0, 1], [1, 2, 3])
    assert gsum.termination == 4 and np.array_equal(gt_, [1, 2, 3])
    ctx.close()


def _run_teacher_forced(sensor, seed, nframes, okw, gkw, max_points, traj=0, width=0, height=0, world_shift=None):
    """Per frame: load the oracle's pre-frame state (odom_, prev_odom_, window) into the GPU
    lane, run one frame on both, compare the poses."""
    scans, gt = get_sequence(sensor, seed, nframes, traj=traj)
    op = oracle.make_params(**okw)
    ctx = api.Context(max_points=max_points, **gkw)
    odo = oracle.Odometer(op)
    K = op.prev_frames
    sizes = []
    worst = (0.0, 0.0)
    for f, s in enumerate(scans):
        sp = oracle.split(op, s, width, height)
        edges = oracle.extract(op, sp["rings"], sp["offsets"])["edges"]
        if f == 1 and world_shift is not None:
            # move the whole world (window + poses) away from the origin on the oracle side;
            # the GPU lane then receives that state like any other teacher-forced frame
            S = np.eye(4)
            S[:3, 3] = world_shift
            w, nf = odo.window()
            odo.set_window(oracle.transform(w, S), sizes)
            o_odom, o_prev = odo.get_pose()
            odo.set_pose(S @ o_odom, S @ o_prev)
        if f > 0:
            w, nf = odo.window()
            assert nf == len(sizes)
            ctx.lmap_clear()
            pos = 0
            for n in sizes:
                ctx.lmap_add(w[pos:pos + n])
                pos += n
            o_odom, o_prev = odo.get_pose()
            ctx.set_pose(o_odom, o_prev)
        opose, od = odo.process(edges)
        gpose, gd = ctx.register(edges)
        if f > 0:
            assert np.abs(np.array(gd.pred_pose).reshape(4, 4) - np.array(od.pred_pose).reshape(4, 4)).max() == 0.0
            for it in range(2):
                assert gd.n_map[it] == od.n_map[it]
                assert gd.n_matches[it] == od.n_matches[it] or it == 1, (f, it, gd.n_matches[it], od.n_matches[it])
                if gd.n_matches[it] != od.n_matches[it]:
                    continue   # outer iteration 1 may see other matches when the first solves differ in the last bits
                g, o = gd.solve[it], od.solve[it]
                gi = (g.iterations, g.successful_steps, g.termination, g.num_residual_blocks, g.cost_evals, g.jac_evals)
                oi = (o.iterations, o.successful_steps, o.termination, o.num_residual_blocks, o.cost_evals, o.jac_evals)
                assert gi == oi and g.num_residual_blocks == gd.n_matches[it], (f, it, gi, oi)
                assert abs(g.initial_cost - o.initial_cost) <= 1e-9 * max(1.0, o.initial_cost), (f, it)
                assert abs(g.final_cost - o.final_cost) <= 1e-7 * max(1.0, o.final_cost), (f, it)
        dt, dr = pose_err(gpose, opose)
        assert dt < TOL_T and dr < TOL_R, "frame %d: %g m, %g rad" % (f, dt, dr)
        worst = (max(worst[0], dt), max(worst[1], dr))
        sizes.append(len(edges))
        if len(sizes) > K:
            sizes.pop(0)
    ctx.close()
    return worst


@pytest.mark.parametrize("group", ["1", "4", "16"])
def test_register_teacher_forced_c1(cuda_lib, group, monkeypatch):
    monkeypatch.setenv("LIODOM_ASSOC_GROUP", group)
    w = _run_teacher_forced("hdl64", 1000, 20, dict(prev_frames=15), dict(prev_frames=15), 131072)
    print("worst teacher-forced pose error C1: %.3g m %.3g rad" % w)


def test_register_teacher_forced_far_from_origin(cuda_lib):
    """World shifted ~190 m from the origin: the range weight of factors.hpp:89-98 (sensor-frame
    point minus world translation) goes negative beyond ~75.7 m."""
    _run_teacher_forced("hdl64_small", 1004, 10, dict(prev_frames=5), dict(prev_frames=5), 32768,
                        world_shift=[150.0, 120.0, 0.0])


def test_register_teacher_forced_c3_stress(cuda_lib):
    kw = dict(scan_regions=16, edges_per_region=20, prev_frames=20)
    _run_teacher_forced("hdl64", 1003, 6, kw, kw, 131072)


def test_register_teacher_forced_c2_ouster(cuda_lib):
    """C2: organised OS1-128-shaped clouds (launch/liodom_ouster.launch params with scan_lines=128)."""
    from liodom_b200 import synth
    w, h = synth.sensor_shape("os1_128")
    kw = dict(lidar_type=1, scan_lines=128, prev_frames=15)
    worst = _run_teacher_forced("os1_128", 1000, 5, kw, kw, 262144, width=w, height=h)
    print("worst teacher-forced pose error C2: %.3g m %.3g rad" % worst)


def test_whole_path_1m_point_scan(cuda_lib):
    """C5: 1M-point scans (64 x 15,625) with scan_regions=64 through the whole path, free-running."""
    scans, _ = get_sequence("hdl64_1m", 1000, 3)
    op = oracle.make_params(prev_frames=15, scan_regions=64)
    oposes, _, _ = oracle.run_sequence(op, scans)
    ctx = api.Context(prev_frames=15, scan_regions=64, max_points=1 << 20)
    for f, s in enumerate(scans):
        ctx.scan_batch([s])
        p, ne = ctx.results()
        assert ne[0] > 30000
        dt, dr = pose_err(p[0], oposes[f])
        assert dt < 1e-4 and dr < 1e-5, (f, dt, dr)
    ctx.close()


def test_free_running_ate_c1(cuda_lib):
    """Free-running whole path (host scans -> poses) vs the oracle's free run over the full 100-frame C1
    sequence (BASELINE.json configs[0]): ATE within 1%."""
    scans, gt = get_sequence("hdl64", 1000, 100)
    op = oracle.make_params(prev_frames=15)
    oposes, _, _ = oracle.run_sequence(op, scans)
    ctx = api.Context(prev_frames=15, max_points=131072)
    gposes = []
    for s in scans:
        ctx.scan_batch([s])
        p, _ = ctx.results()
        gposes.append(p[0].copy())
    gposes = np.stack(gposes)
    rel = np.stack([np.linalg.inv(gt[0]) @ g for g in gt])
    ate_o = np.sqrt(np.mean(np.sum((oposes[:, :3, 3] - rel[:, :3, 3]) ** 2, 1)))
    ate_g = np.sqrt(np.mean(np.sum((gposes[:, :3, 3] - rel[:, :3, 3]) ** 2, 1)))
    assert abs(ate_g - ate_o) <= 0.01 * ate_o, (ate_g, ate_o)
    # and the two trajectories themselves stay together
    assert np.abs(gposes[:, :3, 3] - oposes[:, :3, 3]).max() < 1e-3
    ctx.close()


def test_batched_lanes_match_single_lane(cuda_lib):
    """B independent sequences in one context give the poses each gives alone (no cross-talk),
    and the pipelined (2 scans in flight) enqueue gives the same as the synchronous one."""
    seqs = [get_sequence("hdl64_small", 1000 + k, 6)[0] for k in range(3)]
    single = []
    for sq in seqs:
        ctx = api.Context(prev_frames=5, max_points=32768)
        ps = []
        for s in sq:
            ctx.scan_batch([s])
            ps.append(ctx.results()[0][0].copy())
        single.append(np.stack(ps))
        ctx.close()
    ctx = api.Context(prev_frames=5, max_points=32768, batch=3)
    for f in range(6):
        ctx.scan_batch([seqs[k][f] for k in range(3)])
        poses, ne = ctx.results()
        for k in range(3):
            assert np.array_equal(poses[k], single[k][f]), (f, k)
    ctx.close()


# ---- filter_local_map: VoxelGrid(0.4) of the full window as the kNN target (src/laser_odometry.cc:286-292)
def _check_assoc(g, o, min_sel):
    ok = o["tie"] == 0
    assert np.array_equal(g["gate"][ok], o["gate"][ok])
    sel = ok & ((o["gate"] & 1) == 1)
    assert sel.sum() >= min_sel
    assert np.array_equal(g["knn_idx"][sel], o["knn_idx"][sel])
    assert np.array_equal(g["knn_d2"][sel].view(np.uint32), o["knn_d2"][sel].view(np.uint32))
    assert np.array_equal(g["eig"][sel].view(np.uint64), o["eig"][sel].view(np.uint64))


def test_window_filter_teacher_forced(cuda_lib):
    """The filter applies only once the window holds prev_frames frames; then the kNN target is
    pcl::VoxelGrid(0.4) of the window: same centroids (bit patterns), same order, same 5-NN."""
    K = 6
    scans, gt = get_sequence("hdl64", 1000, K + 3)
    op = oracle.make_params(prev_frames=K, filter_local_map=1)
    edges_seq = _edges_of(op, scans)
    ctx = api.Context(prev_frames=K, filter_local_map=1, max_points=131072)
    frames = []
    for f in range(K + 2):
        w = oracle.transform(edges_seq[f], np.linalg.inv(gt[0]) @ gt[f])
        ctx.lmap_add(w)
        frames = (frames + [w])[-K:]
        window = np.concatenate(frames)
        target = oracle.voxelgrid(window, 0.4) if len(frames) == K else window
        if len(frames) == K:
            assert 0 < len(target) < len(window)
        T = np.linalg.inv(gt[0]) @ gt[f + 1]
        T = T.copy()
        T[:3, 3] += [0.04, -0.02, 0.01]
        o = oracle.associate(edges_seq[f + 1], T, target, knn_method=0)
        g = ctx.associate(edges_seq[f + 1], T)
        assert g["n_map"] == len(target), (f, g["n_map"], len(target), len(window))
        _check_assoc(g, o, 100)
        # LocalMapManager::getLocalMap keeps returning the unfiltered window
        lw, nf = ctx.lmap_get()
        assert nf == len(frames) and np.array_equal(lw.view(np.uint32), window.view(np.uint32))
    ctx.close()


def test_window_filter_random_clouds(cuda_lib):
    """Dense random clouds (many points per voxel, negative coordinates, non-finite points, an empty
    frame): voxel order and the input-order float centroids must match the restated VoxelGrid."""
    rng = np.random.default_rng(11)
    K = 3
    ctx = api.Context(prev_frames=K, filter_local_map=1, scan_lines=16, scan_regions=8, edges_per_region=40, max_points=4096)
    frames = []
    for f in range(7):
        n = [5000, 0, 3000, 5248, 17, 4000, 2500][f]
        w = (rng.normal(size=(n, 4)) * [3.0, 2.0, 0.7, 1.0]).astype(np.float32)
        if f == 3:
            w[::97, 2] = np.nan
            w[5::211, 0] = np.inf
        ctx.lmap_add(w)
        frames = (frames + [w])[-K:]
        window = np.concatenate(frames)
        target = oracle.voxelgrid(window, 0.4) if len(frames) == K else window
        q = (rng.normal(size=(600, 4)) * [2.0, 1.5, 0.5, 1.0]).astype(np.float32)
        o = oracle.associate(q, np.eye(4), target, knn_method=0)
        g = ctx.associate(q, np.eye(4))
        assert g["n_map"] == len(target), (f, g["n_map"], len(target))
        _check_assoc(g, o, 50)
    ctx.close()


def test_register_teacher_forced_window_filter(cuda_lib):
    kw = dict(prev_frames=5, filter_local_map=1)
    _run_teacher_forced("hdl64", 1002, 10, kw, kw, 131072)


def test_batched_window_filter_free_running(cuda_lib):
    """filter_local_map through the batched whole path: lanes at different window fill levels."""
    seqs = [get_sequence("hdl64_small", 1000 + k, 8)[0] for k in range(2)]
    op = oracle.make_params(prev_frames=4, filter_local_map=1)
    refs = [oracle.run_sequence(op, sq)[0] for sq in seqs]
    ctx = api.Context(prev_frames=4, filter_local_map=1, max_points=32768, batch=2)
    for f in range(8):
        ctx.scan_batch([seqs[0][f], seqs[1][f]])
        poses, _ = ctx.results()
        for k in range(2):
            dt, dr = pose_err(poses[k], refs[k][f])
            assert dt < 1e-3 and dr < 1e-4, (f, k, dt, dr)
    ctx.close()


def test_hash_generation_wrap(cuda_lib):
    """The voxel hash tags entries with a 12-bit generation instead of being cleared per build; the
    tables are cleared and every lane rebuilt before the tag can wrap.  Association must stay exact
    across that point (4000 builds)."""
    rng = np.random.default_rng(21)
    ctx = api.Context(prev_frames=3, max_points=2048, scan_lines=16)
    frames = []
    checked = 0
    for f in range(4110):
        w = (rng.normal(size=(48, 4)) * [1.5, 1.5, 0.5, 1.0]).astype(np.float32)
        ctx.lmap_add(w)
        frames = (frames + [w])[-3:]
        if f in (10, 3990, 3998, 3999, 4000, 4001, 4002, 4095, 4096, 4097, 4109):
            window = np.concatenate(frames)
            q = (rng.normal(size=(200, 4)) * [1.0, 1.0, 0.4, 1.0]).astype(np.float32)
            o = oracle.associate(q, np.eye(4), window)
            g = ctx.associate(q, np.eye(4))
            assert g["n_map"] == len(window)
            _check_assoc(g, o, 20)
            checked += 1
    assert checked == 11
    ctx.close()


def test_incremental_hash_every_frame(cuda_lib):
    """The voxel hash follows the window incrementally (evict the oldest frame from the heads of its buckets, append the
    new frame at the tails; full rebuilds only when pool / table headroom runs out).  A drifting cloud over 400 frames:
    cells empty out and come back, buckets move to larger regions, frames of different sizes (one empty, some with
    non-finite points); the association is checked against the oracle on EVERY frame."""
    rng = np.random.default_rng(33)
    ctx = api.Context(prev_frames=6, max_points=2048, scan_lines=16)
    frames = []
    for f in range(400):
        n = 0 if f == 17 else int(rng.integers(20, 300))
        centre = np.array([0.02 * f, 0.5 * np.sin(0.05 * f), 0.0, 0.0])
        w = (rng.normal(size=(n, 4)) * [1.2, 1.2, 0.4, 1.0] + centre).astype(np.float32)
        if f % 23 == 5 and n > 3:
            w[1, 0] = np.nan
            w[2, 2] = np.inf
        ctx.lmap_add(w)
        frames = (frames + [w])[-6:]
        window = np.concatenate(frames)
        q = (rng.normal(size=(150, 4)) * [1.0, 1.0, 0.4, 1.0] + centre).astype(np.float32)
        o = oracle.associate(q, np.eye(4), window)
        g = ctx.associate(q, np.eye(4))
        assert g["n_map"] == len(window), f
        ok = o["tie"] == 0
        assert np.array_equal(g["gate"][ok], o["gate"][ok]), f
        sel = ok & ((o["gate"] & 1) == 1)
        assert np.array_equal(g["knn_idx"][sel], o["knn_idx"][sel]), f
        assert np.array_equal(g["knn_d2"][sel].view(np.uint32), o["knn_d2"][sel].view(np.uint32)), f
    ctx.close()
