"""GPU association at its edges: every constructed case of assoc_cases.py through every search build, each edge compared
with the oracle's brute force, ties, partial lists and failed gates included; then the seeded second-iteration search
through the production path (teacher-forced ctx.register), where all builds must give bit-identical results.

The contract is the one register.cu documents: the five best in (d2, logical index) order under float32 L2_Simple,
cut at the 1 m gate d2[4] < 1.0 (src/laser_odometry.cc:324)."""
import numpy as np
import pytest

import oracle
from liodom_b200 import api
from conftest import get_sequence, pose_err
from assoc_cases import cases, by_name, cut_list, _stationary_cloud

pytestmark = pytest.mark.gpu

TOL_T = 1e-4   # metres
TOL_R = 1e-5   # radians

# LIODOM_ASSOC_GROUP / LIODOM_ASSOC_POOL of each search build (None: unset)
BUILDS = {"thread": ("1", "0"), "pool": ("1", "1"), "group4": ("4", None), "group8": ("8", None), "group16": ("16", None)}
NAMES = [c.name for c in cases()]


def _use(monkeypatch, group, pool):
    monkeypatch.setenv("LIODOM_ASSOC_GROUP", group)
    if pool is None:
        monkeypatch.delenv("LIODOM_ASSOC_POOL", raising=False)
    else:
        monkeypatch.setenv("LIODOM_ASSOC_POOL", pool)


def compare_with_oracle(g, o):
    """Every edge: the full five-list, gate and eigenvalues where the oracle's 5th is within 1 m; elsewhere the list cut
    at d2 < 1.0 and a zero gate.  Returns (edges with five, edges with a partial list)."""
    assert np.array_equal(g["q_world"].view(np.uint32), o["q_world"].view(np.uint32))
    assert not (g["gate"] & 4).any(), "closed-form screen and Jacobi disagree"
    full = (o["gate"] & 1) == 1
    assert np.array_equal(full, (o["knn_idx"][:, 4] >= 0) & (o["knn_d2"][:, 4] < np.float32(1.0)))
    bad = np.nonzero((g["knn_idx"][full] != o["knn_idx"][full]).any(1))[0]
    assert len(bad) == 0, "edge %d: gpu %s oracle %s" % (np.nonzero(full)[0][bad[0]], g["knn_idx"][full][bad[0]], o["knn_idx"][full][bad[0]])
    assert np.array_equal(g["knn_d2"][full].view(np.uint32), o["knn_d2"][full].view(np.uint32))
    assert np.array_equal(g["gate"][full], o["gate"][full])
    assert np.array_equal(g["eig"][full].view(np.uint64), o["eig"][full].view(np.uint64))
    idx, d2 = cut_list(o)
    rest = ~full
    bad = np.nonzero((g["knn_idx"][rest] != idx[rest]).any(1))[0]
    assert len(bad) == 0, "edge %d: gpu %s oracle cut %s" % (np.nonzero(rest)[0][bad[0]], g["knn_idx"][rest][bad[0]], idx[rest][bad[0]])
    assert np.array_equal(g["knn_d2"][rest].view(np.uint32), d2[rest].view(np.uint32))
    assert (g["gate"][rest] == 0).all()
    return int(full.sum()), int(((idx >= 0).any(1) & rest).sum())


_ORACLE = {}


def _oracle_of(c):
    if c.name not in _ORACLE:
        _ORACLE[c.name] = oracle.associate(c.edges, c.pose, c.target(), knn_method=0)
    return _ORACLE[c.name]


def _load(ctx, c):
    ctx.lmap_clear()
    for f in c.frames:
        ctx.lmap_add(f)
    if c.received is not None:
        ctx.set_received_map(c.received)


@pytest.mark.parametrize("build", list(BUILDS))
@pytest.mark.parametrize("name", NAMES)
def test_associate_edge_cases(cuda_lib, name, build, monkeypatch):
    c = by_name()[name]
    r = c.check()
    _use(monkeypatch, *BUILDS[build])
    ctx = api.Context(**c.context_kw())
    _load(ctx, c)
    g = ctx.associate(c.edges, c.pose)
    ctx.close()
    assert g["n_map"] == len(c.target())
    nfull, npart = compare_with_oracle(g, _oracle_of(c))
    print("%s %s: %d edges, %d tied, %d partial lists, %d through the fallback, %d with five"
          % (name, build, len(c.edges), int(r["tie"].sum()), npart, int(r["fallback"].sum()), nfull))


# ---- the seeded search through the production path ---------------------------------------------------------------
# GROUP=1 with POOL unset is the production schedule at large batches: thread-per-edge search in the first outer
# iteration, the warp-pooled search seeded with the first iteration's neighbours in the second.
SETTINGS = [("1", None), ("1", "0"), ("1", "1"), ("4", None), ("8", None), ("16", None)]


def _diag_tuple(d):
    s = [(x.iterations, x.successful_steps, x.termination, x.num_residual_blocks, x.cost_evals, x.jac_evals,
          np.float64(x.initial_cost).view(np.uint64), np.float64(x.final_cost).view(np.uint64)) for x in d.solve]
    return (tuple(d.n_map), tuple(d.n_matches), tuple(s), tuple(d.pred_pose))


def _register_everywhere(monkeypatch, frames, odom, prev, edges, K):
    """One teacher-forced frame: the oracle, then the GPU lane loaded with the same window and poses under every
    setting.  All settings must agree bit for bit; the oracle within its tolerances."""
    op = oracle.make_params(prev_frames=K)
    odo = oracle.Odometer(op)
    odo.set_window(np.concatenate(frames), [len(f) for f in frames])
    odo.set_pose(odom, prev)
    opose, od = odo.process(edges)
    ctx = api.Context(prev_frames=K, max_points=131072)
    runs = []
    for group, pool in SETTINGS:
        _use(monkeypatch, group, pool)
        ctx.lmap_clear()
        for f in frames:
            ctx.lmap_add(f)
        ctx.set_pose(odom, prev)
        runs.append(ctx.register(edges))
    ctx.close()
    p0, d0 = runs[0]
    for (group, pool), (p, d) in zip(SETTINGS[1:], runs[1:]):
        assert np.array_equal(p.view(np.uint64), p0.view(np.uint64)), (group, pool)
        assert _diag_tuple(d) == _diag_tuple(d0), (group, pool, _diag_tuple(d), _diag_tuple(d0))
    assert np.array_equal(np.array(d0.pred_pose), np.array(od.pred_pose))
    assert d0.n_map[0] == od.n_map[0] == sum(len(f) for f in frames)
    assert d0.n_matches[0] == od.n_matches[0]
    for it in range(2):
        if d0.n_matches[it] != od.n_matches[it]:
            assert it == 1
            continue
        g, o = d0.solve[it], od.solve[it]
        gi = (g.iterations, g.successful_steps, g.termination, g.num_residual_blocks, g.cost_evals, g.jac_evals)
        oi = (o.iterations, o.successful_steps, o.termination, o.num_residual_blocks, o.cost_evals, o.jac_evals)
        assert gi == oi, (it, gi, oi)
        if np.isfinite(o.initial_cost):
            assert abs(g.initial_cost - o.initial_cost) <= 1e-9 * max(1.0, o.initial_cost)
            assert abs(g.final_cost - o.final_cost) <= 1e-7 * max(1.0, o.final_cost)
    dt, dr = pose_err(p0, opose)
    assert dt < TOL_T and dr < TOL_R, (dt, dr)
    return d0


def test_seeded_stationary_window(cuda_lib, monkeypatch):
    """A stalled sensor: three copies of one cloud in the window, the same cloud as the frame's edges.  Every edge ties
    and the duplicate neighbours stall the solve (termination 1 after 0 iterations) on both sides."""
    cloud = _stationary_cloud()
    d = _register_everywhere(monkeypatch, [cloud] * 3, np.eye(4), np.eye(4), cloud, 3)
    assert d.n_matches[0] > 1000


def _c1_frame(shift=0.3, n_edges=None):
    """Window: four GT-posed C1 frames and mirror pairs (equal float d2, distinct points) around 600 of the frame's
    predicted edge positions.  The prediction is moved by `shift` metres, so some first-iteration neighbours lie beyond
    1 m (a seed >= 1.0) and some edges have none."""
    scans, gt = get_sequence("hdl64", 1000, 5)
    op = oracle.make_params(prev_frames=15)
    T = [np.linalg.inv(gt[0]) @ gt[k] for k in range(5)]
    frames = []
    for k in range(4):
        sp = oracle.split(op, scans[k])
        frames.append(oracle.transform(oracle.extract(op, sp["rings"], sp["offsets"])["edges"], T[k]))
    sp = oracle.split(op, scans[4])
    edges = oracle.extract(op, sp["rings"], sp["offsets"])["edges"]
    if n_edges is not None:
        assert len(edges) >= n_edges
        edges = edges[:n_edges]
    odom = T[4].copy()
    odom[:3, 3] += [shift, 0.0, 0.0]
    rng = np.random.default_rng(5)
    q = oracle.transform(edges, odom)[rng.choice(len(edges), 600, replace=False)]
    v = np.round(rng.uniform(-0.3, 0.3, (600, 3)) * 64) / 64
    mirror = np.concatenate([np.concatenate([q[:, :3] + v, q[:, 3:]], 1), np.concatenate([q[:, :3] - v, q[:, 3:]], 1)])
    frames.append(mirror.astype(np.float32))
    return frames, odom, edges


@pytest.mark.parametrize("n_edges", [None, 2047, 2048, 2049])
def test_seeded_c1_moved_prediction(cuda_lib, monkeypatch, n_edges):
    frames, odom, edges = _c1_frame(0.3, n_edges)
    d = _register_everywhere(monkeypatch, frames, odom, odom, edges, 15)
    assert d.n_matches[0] > 0.3 * len(edges)


def test_free_running_stationary_sequence(cuda_lib, monkeypatch):
    """The same scan six times through the whole path (scan_batch), against the oracle's free run."""
    monkeypatch.delenv("LIODOM_ASSOC_GROUP", raising=False)
    monkeypatch.delenv("LIODOM_ASSOC_POOL", raising=False)
    scans, _ = get_sequence("hdl64", 1000, 1)
    seq = [scans[0]] * 6
    op = oracle.make_params(prev_frames=15)
    oposes, _, _ = oracle.run_sequence(op, seq)
    ctx = api.Context(prev_frames=15, max_points=131072)
    for f, s in enumerate(seq):
        ctx.scan_batch([s])
        p, _ = ctx.results()
        dt, dr = pose_err(p[0], oposes[f])
        assert dt < TOL_T and dr < TOL_R, (f, dt, dr)
    ctx.close()
