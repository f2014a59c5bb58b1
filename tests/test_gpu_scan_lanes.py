"""Partial steps (liodom_scan_lanes): a step moves only the listed lanes and leaves every other lane as it was.

- the identity list (in order and reversed) is bitwise liodom_scan_batch;
- a staggered schedule (periods 1, 2 and 3, late joiners, a lane that stops early; steps of 1 and of every lane) is
  checked lane by lane against the oracle's free run of each lane's own sequence, and every lane left out of a step
  must report n_edges == -1 and keep its pose and window bit for bit;
- the same with host packed / host per-lane / device inputs, lane groups, both association kernels, the window
  filter and use_imu; two partial steps in flight; a lane restarted while the others step; raw PointCloud2 blobs;
  rejected lane lists."""
import ctypes

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
E_INVALID = -1

_ORACLE = {}


def _seq(seed):
    return get_sequence("hdl64", seed, N_FRAMES)


def _imu_q(seed, f):
    """IMU orientation fed at frame f of a sequence: the ground-truth rotation relative to frame 0."""
    from scipy.spatial.transform import Rotation
    gt = _seq(seed)[1]
    return Rotation.from_matrix((np.linalg.inv(gt[0]) @ gt[f])[:3, :3]).as_quat()


def _oracle_run(seed, kind="plain"):
    """Free-running oracle poses and per-frame edge counts of one C1 sequence (cached per seed and kind)."""
    key = (seed, kind)
    if key not in _ORACLE:
        scans = _seq(seed)[0]
        op = oracle.make_params(prev_frames=PREV, filter_local_map=1 if kind == "filter" else 0)
        ne = np.array([len(oracle.extract_scan(op, s)[0]) for s in scans])
        if kind == "imu":
            odo = oracle.Odometer(op)
            poses = []
            for f, s in enumerate(scans):
                odo.set_imu(1, _imu_q(seed, f), np.eye(4))
                poses.append(odo.process(oracle.extract_scan(op, s)[0])[0])
            poses = np.stack(poses)
        else:
            poses, _, _ = oracle.run_sequence(op, scans)
        _ORACLE[key] = (poses, ne)
    return _ORACLE[key]


def _schedule(B):
    """List of steps, each a list of (lane, frame).  Lane l has period 1 + l % 3; lanes l % 8 == 5 join at step 6;
    lane 1 stops after its frame 10; lane B - 1 joins at step 6 with period 3 and is the only lane left at the end."""
    period = [1 + l % 3 for l in range(B)]
    start = [6 if l % 8 == 5 else 0 for l in range(B)]
    for l in range(B):
        if start[l] == 6 and period[l] == 3:
            period[l] = 2
    start[B - 1], period[B - 1] = 6, 3
    last = [N_FRAMES - 1] * B
    last[1] = 10
    steps, t = [], 0
    while True:
        step = [(l, (t - start[l]) // period[l]) for l in range(B)
                if t >= start[l] and (t - start[l]) % period[l] == 0 and (t - start[l]) // period[l] <= last[l]]
        if not step and all(t - start[l] > period[l] * last[l] for l in range(B)):
            break
        if step:
            steps.append(step)
        t += 1
    return steps, last


def _order(step, t):
    """The step's lanes in a seeded shuffled order (lists need not be sorted)."""
    rng = np.random.default_rng(t)
    return [step[i] for i in rng.permutation(len(step))]


class _Feeder:
    """Enqueues a partial step with host packed / host per-lane / device inputs."""

    def __init__(self, ctx, mode, seeds):
        self.ctx, self.mode, self.keep = ctx, mode, []
        if mode == "device":
            import torch
            self.dev = {sd: [torch.from_numpy(s).cuda() for s in _seq(sd)[0]] for sd in set(seeds)}

    def step(self, lanes, scans, dev_keys=None):
        cnts = [len(s) for s in scans]
        if self.mode == "host_packed":
            buf = np.ascontiguousarray(np.concatenate(scans)) if scans else np.zeros((0, 4), np.float32)
            offs = np.concatenate([[0], np.cumsum(cnts)[:-1]]) if scans else []
            self.keep.append(buf)
            self.ctx.scan_lanes_ptrs(lanes, [buf.ctypes.data + int(o) * 16 for o in offs], cnts, 16, on_device=False)
        elif self.mode == "host_lanes":
            arrs = [s if i % 2 == 0 else s.copy() for i, s in enumerate(scans)]   # not back to back: per-lane copies
            self.keep.append(arrs)
            self.ctx.scan_lanes_ptrs(lanes, [a.ctypes.data for a in arrs], cnts, 16, on_device=False)
        else:
            self.ctx.scan_lanes_ptrs(lanes, [self.dev[sd][f].data_ptr() for sd, f in dev_keys], cnts, 16, on_device=True)
        self.keep = self.keep[-2:]   # host inputs live until their step's results are collected


def _lane_state(ctx, l):
    pose, prev = ctx.get_pose(l)
    win, nf = ctx.lmap_get(l)
    return pose.copy(), prev.copy(), win, nf


def _same_state(a, b):
    return (np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[3] == b[3] and
            np.array_equal(a[2].view(np.uint32), b[2].view(np.uint32)))


def _run_staggered(B, mode, kind="plain"):
    """The staggered schedule on a B-lane context; every stepped lane against the oracle, every other lane unchanged."""
    seeds = [1000 + l % N_SEEDS for l in range(B)]
    steps, last = _schedule(B)
    sizes = {len(s) for s in steps}
    assert 1 in sizes and B in sizes
    kw = dict(filter_local_map=1) if kind == "filter" else (dict(use_imu=1) if kind == "imu" else {})
    ctx = api.Context(prev_frames=PREV, max_points=131072, batch=B, **kw)
    feed = _Feeder(ctx, mode, seeds)
    last_pose = np.zeros((B, 4, 4))
    state = [_lane_state(ctx, l) for l in range(B)]
    worst = [0.0, 0.0]
    for t, step in enumerate(steps):
        step = _order(step, t)
        lanes = [l for l, _ in step]
        if kind == "imu":
            for l, f in step:
                ctx.set_imu(_imu_q(seeds[l], f), lane=l)
        feed.step(lanes, [_seq(seeds[l])[0][f] for l, f in step], [(seeds[l], f) for l, f in step])
        poses, ne = ctx.results()
        stepped = dict(step)
        for l in range(B):
            if l in stepped:
                f = stepped[l]
                oposes, one = _oracle_run(seeds[l], kind)
                assert ne[l] == one[f], "step %d lane %d frame %d: %d edges, oracle %d" % (t, l, f, ne[l], one[f])
                dt, dr = pose_err(poses[l], oposes[f])
                assert dt < TOL_T and dr < TOL_R, "step %d lane %d frame %d: %g m, %g rad" % (t, l, f, dt, dr)
                worst = [max(worst[0], dt), max(worst[1], dr)]
                last_pose[l] = poses[l]
            else:
                assert ne[l] == -1, "step %d: lane %d was not stepped but reports %d edges" % (t, l, ne[l])
                assert np.array_equal(poses[l], last_pose[l]), "step %d: pose row of idle lane %d changed" % (t, l)
            now = _lane_state(ctx, l)
            if l not in stepped:
                assert _same_state(now, state[l]), "step %d: idle lane %d's pose or window changed" % (t, l)
            state[l] = now
    for l in range(B):
        if last[l] == N_FRAMES - 1:   # the filtered target is smaller than the window: count its frames instead
            full = ctx.lmap_get(l)[1] == PREV if kind == "filter" else ctx.scan_diag(l).n_map[0] > 60000
            assert full, "lane %d: window did not fill" % l
    ctx.close()
    return worst, len(steps)


@pytest.mark.parametrize("mode", ["host_packed", "host_lanes", "device"])
def test_staggered_vs_oracle(cuda_lib, mode, monkeypatch):
    monkeypatch.delenv("LIODOM_LANE_GROUPS", raising=False)
    w, n = _run_staggered(32, mode)
    print("32 lanes %s: %d steps, worst pose error %.3g m %.3g rad" % (mode, n, w[0], w[1]))


@pytest.mark.parametrize("env", [("LIODOM_LANE_GROUPS", "1"), ("LIODOM_LANE_GROUPS", "2"), ("LIODOM_LANE_GROUPS", "4"),
                                 ("LIODOM_ASSOC_POOL", "0"), ("LIODOM_ASSOC_POOL", "1")])
def test_staggered_128_lanes(cuda_lib, env, monkeypatch):
    """128 lanes: the lane-group schedule of partial lists (1, 2 and 4 groups of positions), and both association
    kernels; idle lanes' poses and windows are compared bit for bit under each."""
    monkeypatch.delenv("LIODOM_LANE_GROUPS", raising=False)
    monkeypatch.setenv(*env)
    w, n = _run_staggered(128, "device")
    print("128 lanes %s=%s: %d steps, worst pose error %.3g m %.3g rad" % (env[0], env[1], n, w[0], w[1]))


@pytest.mark.parametrize("kind", ["filter", "imu"])
def test_staggered_other_paths(cuda_lib, kind, monkeypatch):
    """filter_local_map = 1 (the k_vg_* kernels and the wholesale hash build) and use_imu = 1."""
    monkeypatch.delenv("LIODOM_LANE_GROUPS", raising=False)
    w, n = _run_staggered(16, "device", kind)
    print("16 lanes %s: %d steps, worst pose error %.3g m %.3g rad" % (kind, n, w[0], w[1]))


@pytest.mark.parametrize("B", [16, 128])
def test_identity_list_is_scan_batch(cuda_lib, B, monkeypatch):
    """lanes = range(B), then reversed: every frame bitwise the poses and edge counts of liodom_scan_batch."""
    import torch
    monkeypatch.delenv("LIODOM_LANE_GROUPS", raising=False)
    dev = {sd: [torch.from_numpy(s).cuda() for s in _seq(sd)[0]] for sd in range(1000, 1000 + N_SEEDS)}
    for order in (list(range(B)), list(range(B))[::-1]):
        ref = api.Context(prev_frames=PREV, max_points=131072, batch=B)
        ctx = api.Context(prev_frames=PREV, max_points=131072, batch=B)
        for f in range(N_FRAMES):
            ptr = [dev[1000 + l % N_SEEDS][f].data_ptr() for l in range(B)]
            cnt = [len(_seq(1000 + l % N_SEEDS)[0][f]) for l in range(B)]
            ref.scan_batch_ptrs(ptr, cnt, 16)
            ctx.scan_lanes_ptrs(order, [ptr[l] for l in order], [cnt[l] for l in order], 16)
            rp, rn = ref.results()
            gp, gn = ctx.results()
            assert np.array_equal(rn, gn), "frame %d: edge counts differ" % f
            assert np.array_equal(rp.view(np.uint64), gp.view(np.uint64)), "frame %d: poses differ" % f
        ref.close()
        ctx.close()


def test_two_partial_steps_in_flight(cuda_lib):
    """Step A (lanes 0..11) and step B (lanes 4..15) enqueued back to back from host memory, then collected with
    results(age=1) and results(age=0): lanes 4..11 take two frames, the others one."""
    B = 16
    seeds = [1000 + l % N_SEEDS for l in range(B)]
    ctx = api.Context(prev_frames=PREV, max_points=131072, batch=B)
    frame = [0] * B
    keep = []
    for rnd in range(N_FRAMES // 2):
        sets = [list(range(0, 12)), list(range(4, 16))[::-1]]
        expect = []
        for lanes in sets:
            scans = [_seq(seeds[l])[0][frame[l]] for l in lanes]
            buf = np.ascontiguousarray(np.concatenate(scans))
            keep = (keep + [buf])[-2:]
            offs = np.concatenate([[0], np.cumsum([len(s) for s in scans])[:-1]])
            ctx.scan_lanes_ptrs(lanes, [buf.ctypes.data + int(o) * 16 for o in offs], [len(s) for s in scans], 16, on_device=False)
            expect.append({l: frame[l] for l in lanes})
            for l in lanes:
                frame[l] += 1
        for age, exp in ((1, expect[0]), (0, expect[1])):
            poses, ne = ctx.results(age)
            for l in range(B):
                if l not in exp:
                    assert ne[l] == -1, (rnd, age, l)
                    continue
                oposes, one = _oracle_run(seeds[l])
                f = exp[l]
                assert ne[l] == one[f], (rnd, age, l, f)
                dt, dr = pose_err(poses[l], oposes[f])
                assert dt < TOL_T and dr < TOL_R, "round %d age %d lane %d frame %d: %g m, %g rad" % (rnd, age, l, f, dt, dr)
    ctx.close()


def test_restart_one_lane(cuda_lib):
    """Lane 3 is reset (reset + lmap_clear) after its frame 11 while the others keep stepping; it then restarts
    another sequence from frame 0 and follows the oracle's run of that sequence."""
    B = 8
    seeds = [1000 + l for l in range(B)]
    ctx = api.Context(prev_frames=PREV, max_points=131072, batch=B)
    frame = [0] * B
    for t in range(N_FRAMES + 14):
        if t == 12:
            ctx.reset(lane=3)
            ctx.lmap_clear(lane=3)
            seeds[3], frame[3] = 1000 + B, 0   # a sequence no other lane runs
        lanes = [l for l in range(B) if frame[l] < N_FRAMES and not (l == 3 and t in (12, 13))]
        if not lanes:
            break
        ctx.scan_lanes(lanes, [_seq(seeds[l])[0][frame[l]] for l in lanes])
        poses, ne = ctx.results()
        for l in lanes:
            oposes, one = _oracle_run(seeds[l])
            assert ne[l] == one[frame[l]], (t, l)
            dt, dr = pose_err(poses[l], oposes[frame[l]])
            assert dt < TOL_T and dr < TOL_R, "step %d lane %d frame %d: %g m, %g rad" % (t, l, frame[l], dt, dr)
            frame[l] += 1
    assert frame[3] == N_FRAMES
    ctx.close()


def test_layout_lanes_match_decoded(cuda_lib):
    """liodom_scan_lanes_layout on raw 22-byte PointXYZIRT blobs: bitwise the poses of the decoded clouds through
    liodom_scan_lanes, on the same partial schedule."""
    dt = np.dtype({"names": ["x", "y", "z", "intensity", "ring", "time"], "formats": ["<f4", "<f4", "<f4", "<f4", "<u2", "<f4"],
                   "offsets": [0, 4, 8, 12, 16, 18], "itemsize": 22})
    lay = api.CloudLayout(22, 0, 0, 4, 8, 12, 0)
    B = 8
    seeds = [1000 + l for l in range(B)]
    a = api.Context(prev_frames=PREV, max_points=131072, batch=B)
    b = api.Context(prev_frames=PREV, max_points=131072, batch=B)
    steps, _ = _schedule(B)
    for t, step in enumerate(steps[:30]):
        step = _order(step, t)
        lanes = [l for l, _ in step]
        scans = [_seq(seeds[l])[0][f] for l, f in step]
        blobs = []
        for s in scans:
            rec = np.zeros(len(s), dt)
            rec["x"], rec["y"], rec["z"], rec["intensity"] = s[:, 0], s[:, 1], s[:, 2], s[:, 3]
            rec["ring"], rec["time"] = 7, 0.5
            blobs.append(rec.view(np.uint8))
        a.scan_lanes_layout(lanes, blobs, [len(s) for s in scans], lay)
        b.scan_lanes(lanes, scans)
        pa, na = a.results()
        pb, nb = b.results()
        assert np.array_equal(na, nb) and np.array_equal(pa.view(np.uint64), pb.view(np.uint64)), "step %d" % t
    a.close()
    b.close()


def test_rejected_lists(cuda_lib):
    """Bad lists return LIODOM_E_INVALID and enqueue nothing; the next valid step matches the oracle.  n_lanes = 0
    enqueues nothing and returns 0."""
    B = 4
    ctx = api.Context(prev_frames=PREV, max_points=131072, batch=B)
    lib = ctx.lib
    scans = [_seq(1000 + l)[0][0] for l in range(B)]
    vp = ctypes.c_void_p

    def call(lanes, k=None, pts=True, n=True):
        k = len(lanes) if k is None else k
        m = max(k, len(lanes or []), 1)
        la = (ctypes.c_int32 * m)(*lanes) if lanes is not None else None
        pa = (vp * m)(*([scans[0].ctypes.data] * m)) if pts else None
        na = (ctypes.c_int * m)(*([len(scans[0])] * m)) if n else None
        return lib.liodom_scan_lanes(ctx.h, la, k, pa, na, 16, 0, 0, 0)

    before = ctx.launch_count
    bad = {"duplicate": dict(lanes=[1, 2, 1]), "negative lane": dict(lanes=[0, -1]), "lane == batch": dict(lanes=[B]),
           "n_lanes < 0": dict(lanes=[0], k=-1), "n_lanes > batch": dict(lanes=[0, 1, 2, 3, 0], k=B + 1),
           "NULL lanes": dict(lanes=None, k=2), "NULL pts": dict(lanes=[0, 1], pts=False), "NULL n": dict(lanes=[0, 1], n=False)}
    for name, kw in bad.items():
        assert call(**kw) == E_INVALID, name
        assert ctx.launch_count == before, name
    assert call([], k=0) == 0 and lib.liodom_scan_lanes(ctx.h, None, 0, None, None, 16, 0, 0, 0) == 0
    assert ctx.launch_count == before
    for f in range(3):
        lanes = [2, 0]
        ctx.scan_lanes(lanes, [_seq(1000 + l)[0][f] for l in lanes])
        poses, ne = ctx.results()
        assert ne[1] == -1 and ne[3] == -1
        for l in lanes:
            oposes, one = _oracle_run(1000 + l)
            assert ne[l] == one[f]
            dt, dr = pose_err(poses[l], oposes[f])
            assert dt < TOL_T and dr < TOL_R, (f, l, dt, dr)
    assert ctx.launch_count > before
    ctx.close()


def test_point_sharded_context_rejects_lists(cuda_lib):
    """A point-sharded context (liodom_shard_init, world 2) refuses liodom_scan_lanes and then steps as before
    (tests/run_sharded_lanes_check.py under torchrun).  Skipped on single-GPU boxes."""
    import json
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29534", os.path.join(root, "tests", "run_sharded_lanes_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    res = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert res["status"] == "ok" and res["rejected"], res
