"""GPU parity of the BENCHMARKED configuration: liodom_scan_batch with 16 / 64 / 128 lanes per context
(the k_solve<., 2> build, the lane-group multi-stream schedule and the packed single-copy staging of
cabi.cu) against the oracle's free run of the same sequences (src/laser_odometry.cc:198-235).

Every lane is checked, every frame: edge counts exactly, poses within 1e-4 m / 1e-5 rad
(BASELINE.json north_star).  8 distinct C1 seeds x 22 frames, so the 15-frame window fills and the
steady-state code path (eviction) runs for 7 frames.  Once with host pointers (packed staging when the
scans are back to back, per-lane copies when they are not), once with device pointers; lane groups
forced to 1, 2 and 4."""
import numpy as np
import pytest

import oracle
from liodom_b200 import api
from conftest import get_sequence, pose_err

pytestmark = pytest.mark.gpu

TOL_T = 1e-4   # metres
TOL_R = 1e-5   # radians
N_SEEDS = 8
N_FRAMES = 22
PREV = 15

_ORACLE = {}


def _oracle_run(seed):
    """Free-running oracle poses and per-frame edge counts of one C1 sequence."""
    if seed not in _ORACLE:
        scans, _ = get_sequence("hdl64", seed, N_FRAMES)
        op = oracle.make_params(prev_frames=PREV)
        poses, _, _ = oracle.run_sequence(op, scans)
        ne = np.array([len(oracle.extract_scan(op, s)[0]) for s in scans])
        _ORACLE[seed] = (poses, ne)
    return _ORACLE[seed]


def _run_batch(batch, mode, trace=None):
    """mode: 'host_packed' (one buffer, scans back to back), 'host_lanes' (separate arrays), 'device'.  `trace`, when
    given, receives every frame's poses of all lanes."""
    seqs = [get_sequence("hdl64", 1000 + k, N_FRAMES)[0] for k in range(N_SEEDS)]
    ctx = api.Context(prev_frames=PREV, max_points=131072, batch=batch)
    worst = [0.0, 0.0]
    keep = None
    if mode == "device":
        import torch
        dev = [[torch.from_numpy(seqs[k][f]).cuda() for f in range(N_FRAMES)] for k in range(N_SEEDS)]
    for f in range(N_FRAMES):
        cnts = [len(seqs[l % N_SEEDS][f]) for l in range(batch)]
        if mode == "host_packed":
            keep = np.ascontiguousarray(np.concatenate([seqs[l % N_SEEDS][f] for l in range(batch)]))
            offs = np.concatenate([[0], np.cumsum(cnts)[:-1]])
            ptrs = [keep.ctypes.data + int(o) * 16 for o in offs]
            ctx.scan_batch_ptrs(ptrs, cnts, 16, on_device=False)
        elif mode == "host_lanes":
            # odd lanes get their own copy: the pointers are NOT back to back, so the per-lane copy path runs
            keep = [seqs[l % N_SEEDS][f] if l % 2 == 0 else seqs[l % N_SEEDS][f].copy() for l in range(batch)]
            ctx.scan_batch_ptrs([a.ctypes.data for a in keep], cnts, 16, on_device=False)
        else:
            # every lane must read its own addresses only when timing matters; for parity, sharing is fine
            ctx.scan_batch_ptrs([dev[l % N_SEEDS][f].data_ptr() for l in range(batch)], cnts, 16, on_device=True)
        poses, ne = ctx.results()
        if trace is not None:
            trace.append(np.array(poses, copy=True))
        for l in range(batch):
            oposes, one = _oracle_run(1000 + l % N_SEEDS)
            assert ne[l] == one[f], "lane %d frame %d: %d edges, oracle %d" % (l, f, ne[l], one[f])
            dt, dr = pose_err(poses[l], oposes[f])
            assert dt < TOL_T and dr < TOL_R, "lane %d frame %d: %g m, %g rad" % (l, f, dt, dr)
            worst = [max(worst[0], dt), max(worst[1], dr)]
    d = ctx.scan_diag(batch - 1)
    assert d.n_map[0] > 60000, "window did not reach steady state (%d map points)" % d.n_map[0]
    ctx.close()
    return worst


@pytest.mark.parametrize("batch,mode", [(128, "host_packed"), (128, "device"), (64, "host_packed"), (64, "device"),
                                        (16, "host_lanes"), (16, "device")])
def test_batch_free_running_vs_oracle(cuda_lib, batch, mode, monkeypatch):
    monkeypatch.delenv("LIODOM_LANE_GROUPS", raising=False)
    w = _run_batch(batch, mode)
    print("batch %d %s: worst pose error %.3g m %.3g rad over %d lanes x %d frames" % (batch, mode, w[0], w[1], batch, N_FRAMES))


@pytest.mark.parametrize("groups", ["1", "2", "4"])
def test_batch128_lane_groups(cuda_lib, groups, monkeypatch):
    """The lane-group schedule (cabi.cu: groups of lanes on their own streams) must not change any lane's result."""
    monkeypatch.setenv("LIODOM_LANE_GROUPS", groups)
    w = _run_batch(128, "device")
    print("batch 128, %s lane groups: worst pose error %.3g m %.3g rad" % (groups, w[0], w[1]))


_POOL_POSES = {}


@pytest.mark.parametrize("pool", ["0", "1"])
def test_batch128_warp_pooled_association(cuda_lib, pool, monkeypatch):
    """LIODOM_ASSOC_POOL=0 / 1: the thread-per-edge kernel in both outer iterations / the warp-pooled one in both (the
    default is thread-per-edge first, pooled and seeded second: every other test of this file).  Same poses, bit for
    bit: both kernels claim the same five neighbours in the same order, and the gate and the solve are shared."""
    monkeypatch.setenv("LIODOM_ASSOC_POOL", pool)
    trace = []
    w = _run_batch(128, "device", trace)
    _POOL_POSES[pool] = np.stack(trace)
    print("batch 128, LIODOM_ASSOC_POOL=%s: worst pose error %.3g m %.3g rad" % (pool, w[0], w[1]))
    other = _POOL_POSES.get("1" if pool == "0" else "0")
    if other is not None:
        assert np.array_equal(_POOL_POSES[pool].view(np.uint64), other.view(np.uint64))


@pytest.mark.parametrize("name", ["c2_ouster", "c3_stress"])
def test_batch_other_baseline_shapes(cuda_lib, name):
    """The other BASELINE.json shapes through the batched path with a full window (the incremental voxel hash with
    21-frame / 128-ring windows): C2 = OS1-128 organised clouds, C3 = scan_regions / edges_per_region doubled and
    prev_frames = 20.  12 lanes (4 seeds), every lane and frame against the oracle's free run."""
    from liodom_b200 import synth
    if name == "c2_ouster":
        sensor, nfr = "os1_128", 18
        w, h = synth.sensor_shape(sensor)
        kw = dict(lidar_type=1, scan_lines=128, prev_frames=15)
        maxp = 262144
    else:
        sensor, nfr, w, h = "hdl64", 24, 0, 0
        kw = dict(scan_regions=16, edges_per_region=20, prev_frames=20)
        maxp = 131072
    seeds = [1000, 1001, 1002, 1003]
    seqs = [get_sequence(sensor, sd, nfr)[0] for sd in seeds]
    op = oracle.make_params(**kw)
    oruns = [oracle.run_sequence(op, sq, w, h)[0] for sq in seqs]
    nl = 12   # enough edges in flight for the one-thread-per-edge kernels (k_associate<1> + k_associate_pool) at both shapes
    ctx = api.Context(batch=nl, max_points=maxp, **kw)
    for f in range(nfr):
        ctx.scan_batch([seqs[l % 4][f] for l in range(nl)], width=w, height=h)
        poses, ne = ctx.results()
        for l in range(nl):
            dt, dr = pose_err(poses[l], oruns[l % 4][f])
            assert dt < TOL_T and dr < TOL_R, "%s lane %d frame %d: %g m, %g rad" % (name, l, f, dt, dr)
    ctx.close()
