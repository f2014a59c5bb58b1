"""GPU: the LM solve (`liodom_b200/csrc/solve.cu`) at its edges against the oracle.

a. `liodom_solve` (k_solve<false, *>) on every case of solve_cases.py.
b. The fixed-order reduction at the CTA / cluster boundaries, against a 40-digit cost.
c. The production solve (k_solve<true, OCC>: float blocks from the line gate, per-CTA compaction, cluster reduction) at
   every (OCC, cluster size) the launch picks, including the uncompacted loop, with teacher-forced lanes.
d. A frame whose window holds a point twice, so that one residual block is NaN: the solve stalls at its start."""
import numpy as np
import pytest

import np_ref
import oracle
import solve_cases
from liodom_b200 import api
from conftest import get_sequence, pose_err

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
INTS = ("iterations", "successful_steps", "termination", "num_residual_blocks", "cost_evals", "jac_evals")
CASES = solve_cases.cases()


def _ints(s):
    return tuple(int(getattr(s, k)) for k in INTS)


def _costs_match(g, o):
    """The contract of test_gpu_register.test_solve_matches_oracle; non-finite costs must be non-finite on both sides."""
    for a, b, tol in ((g.initial_cost, o.initial_cost, 1e-9), (g.final_cost, o.final_cost, 1e-7)):
        if not np.isfinite(b):
            if np.isfinite(a):
                return False
        elif abs(a - b) > tol * max(1.0, abs(b)):
            return False
    return True


def test_liodom_solve_edge_cases(cuda_lib):
    """Below solve_cases.COND_MAX: identical summary integers, t within 1e-7, q within 1e-8, costs as in
    test_solve_matches_oracle, against the oracle's QR.  Above it: the same contract against the oracle's Cholesky
    (the GPU's linear solver), and QR within 0.5 eps * cond (about 4x the spread measured between two QR codes)."""
    ctx = api.Context(prev_frames=15, max_points=131072)
    bad = []
    for c in CASES:
        cab, q0, t0 = c["cab"], c["q"], c["t"]
        gq, gt, gs = ctx.solve(cab, q0, t0)
        oq, ot, os_ = oracle.solve(cab, q0, t0, linear_solver=0)
        _, _, ns = np_ref.lm_solve(cab, q0, t0)
        cond = ns.cond_first
        ill = np.isfinite(cond) and cond >= solve_cases.COND_MAX
        ref = oracle.solve(cab, q0, t0, linear_solver=1) if ill else (oq, ot, os_)
        rq, rt, rs = ref
        dq, dt = np.abs(gq - rq).max(), np.abs(gt - rt).max()
        dqr = max(np.abs(gq - oq).max(), np.abs(gt - ot).max())
        ok = (_ints(gs) == _ints(rs) and dt <= 1e-7 and dq <= 1e-8 and _costs_match(gs, rs)
              and (not ill or dqr <= 0.5 * EPS * cond))
        print("%-34s n=%4d cond=%-9.3g vs %s: ints %s %s |dq|=%.2g |dt|=%.2g |d QR|=%.2g %s"
              % (c["name"], len(cab), cond, "chol" if ill else "QR", _ints(gs), "==" if _ints(gs) == _ints(rs) else
                 "!= %s" % (_ints(rs),), dq, dt, dqr, "ok" if ok else "FAIL"))
        if c["exit"] is not None and gs.termination != c["exit"]:
            ok = False
        if c["name"] == "nan_block" and not (np.array_equal(gq, q0) and np.array_equal(gt, t0)):
            ok = False
        if not ok:
            bad.append(c["name"])
    ctx.close()
    assert not bad, bad


def _marker_scene(n, seed=5):
    """n blocks at the identity pose; the blocks at the first and last index of every 256-thread stride and of the list
    carry distinct quadratic-branch costs (~1e-3 each), every other block ~1e-9: dropping or double-counting any block
    moves the cost by far more than 1e-12 of it."""
    rng = np.random.default_rng(seed)
    idx = np.arange(n)
    marker = (idx % 256 == 0) | (idx % 256 == 255) | (idx == n - 1)
    off = np.where(marker, 0.03 + 0.0005 * (np.cumsum(marker) % 97), 1e-4 * (1 + rng.random(n)))
    I = np.array([0.0, 0.0, 0.0, 1.0])
    return solve_cases.scene(seed, n, I, np.zeros(3), offsets=off), int(marker.sum())


@pytest.mark.parametrize("n", [1, 2, 7, 255, 256, 257, 2047, 2048, 2049, "Ecap"])
def test_solve_reduction_boundaries(cuda_lib, n):
    """liodom_solve strides the blocks over 8 CTAs x 256 threads (2048 per round): every count around those
    boundaries and the capacity.  The block count is exact and the initial cost within 1e-12 of the sum of its
    (positive) terms of np_ref.exact_cost."""
    ctx = api.Context(prev_frames=15, max_points=131072)
    n = ctx.max_edges if n == "Ecap" else n
    cab, nmark = _marker_scene(n)
    I = np.array([0.0, 0.0, 0.0, 1.0])
    gq, gt, gs = ctx.solve(cab, I, np.zeros(3))
    ctx.close()
    ex = np_ref.exact_cost(cab, I, np.zeros(3))
    assert gs.num_residual_blocks == n
    err = abs(float(gs.initial_cost - ex))
    print("n=%d markers=%d initial_cost=%.17g exact=%s err=%.3g" % (n, nmark, gs.initial_cost, float(ex), err))
    assert err <= 1e-12 * float(ex)
    _, _, os_ = oracle.solve(cab, I, np.zeros(3))
    assert _ints(gs) == _ints(os_)


# ---- c. the production solve at every (OCC, C)
LANES = 152
SIZES = [1, 16, 40, 80, 152]
SEEDS = [1000, 1001, 1002, 1003]
KW = dict(lidar_type=1, scan_lines=128, scan_regions=16, edges_per_region=20, prev_frames=3)


def _shape(nl):
    """(OCC, C) the launch picks for a list of nl lanes (solve.cu: launch_solve_kernel, solve_cluster_size)."""
    occ = 2 if nl >= 16 else 1
    c = 8
    while c > 1 and nl * c > 148 * occ:
        c >>= 1
    return occ, c


def _load(ctx, lane, st):
    window, sizes, odom, prev = st
    ctx.lmap_clear(lane)
    pos = 0
    for k in sizes:
        ctx.lmap_add(window[pos:pos + k], lane)
        pos += k
    ctx.set_pose(odom, prev, lane)


def test_production_solve_every_cluster_shape(cuda_lib, monkeypatch):
    """OS1-128 scans with 16 regions x 20 edges (25-27 k edges, so that ceil(n / C) > 8192 at C = 2 and C = 1) in one
    152-lane context with one lane group.  Per frame, lists of 1, 16, 40, 80 and 152 lanes are loaded with the oracle's
    pre-frame state and stepped once: (OCC, C) = (1, 8), (2, 8), (2, 4), (2, 2) uncompacted, (2, 1) uncompacted."""
    from liodom_b200 import synth
    monkeypatch.setenv("LIODOM_LANE_GROUPS", "1")
    w, h = synth.sensor_shape("os1_128")
    nfr = 3
    seqs = [get_sequence("os1_128", s, nfr)[0] for s in SEEDS]
    op = oracle.make_params(**KW)
    odos = [oracle.Odometer(op) for _ in SEEDS]
    sizes = [[] for _ in SEEDS]
    ctx = api.Context(batch=LANES, max_points=262144, **KW)
    ctx.scan_lanes(list(range(LANES)), [seqs[l % 4][0] for l in range(LANES)], w, h)
    ctx.results()
    edges0 = []
    for k, o in enumerate(odos):
        sp = oracle.split(op, seqs[k][0], w, h)
        e = oracle.extract(op, sp["rings"], sp["offsets"])["edges"]
        o.process(e)
        sizes[k].append(len(e))
    rng = np.random.default_rng(9)
    seen = set()
    for f in range(1, nfr):
        states, odiag, opose, edges = [], [], [], []
        for k, o in enumerate(odos):
            win, nf = o.window()
            assert nf == len(sizes[k])
            states.append((win, list(sizes[k]), *o.get_pose()))
            sp = oracle.split(op, seqs[k][f], w, h)
            e = oracle.extract(op, sp["rings"], sp["offsets"])["edges"]
            edges.append(e)
            p, d = o.process(e)
            opose.append(p)
            odiag.append(d)
            sizes[k] = (sizes[k] + [len(e)])[-op.prev_frames:]
        if f == 1:   # the teacher-forcing itself: loaded state + scan_lanes == loaded state + liodom_register
            _load(ctx, 0, states[0])
            preg, _ = ctx.register(edges[0], lane=0)
            _load(ctx, 0, states[0])
            ctx.scan_lanes([0], [seqs[0][f]], w, h)
            assert np.array_equal(ctx.results()[0][0], preg)
        for nl in SIZES:
            lanes = [int(x) for x in rng.permutation(LANES)[:nl]]
            for l in lanes:
                _load(ctx, l, states[l % 4])
            ctx.scan_lanes(lanes, [seqs[l % 4][f] for l in lanes], w, h)
            poses, ne = ctx.results()
            occ, C = _shape(nl)
            first = {}
            for l in lanes:
                k = l % 4
                gd, od = ctx.scan_diag(l), odiag[k]
                assert ne[l] == od.n_edges == len(edges[k]), (nl, l, ne[l], od.n_edges)
                for it in range(2):
                    if it == 1 and gd.n_matches[1] != od.n_matches[1]:
                        continue
                    g, o = gd.solve[it], od.solve[it]
                    assert gd.n_matches[it] == od.n_matches[it] == g.num_residual_blocks, (nl, l, it)
                    assert _ints(g) == _ints(o), (nl, l, it, _ints(g), _ints(o))
                    assert _costs_match(g, o), (nl, l, it, g.initial_cost, o.initial_cost, g.final_cost, o.final_cost)
                dt, dr = pose_err(poses[l], opose[k])
                assert dt < 1e-4 and dr < 1e-5, (nl, l, dt, dr)
                if k in first:   # same input, same step: bit for bit
                    l0 = first[k]
                    assert np.array_equal(poses[l], poses[l0])
                    assert bytes(gd) == bytes(ctx.scan_diag(l0)), (l, l0)
                else:
                    first[k] = l
            compact = all((ne[l] + C - 1) // C <= 8192 for l in lanes)
            if C == 2:
                assert all(ne[l] > 16384 for l in lanes)
            if C == 1:
                assert all(ne[l] > 8192 for l in lanes)
            seen.add((occ, C, compact))
            print("frame %d: %3d lanes -> OCC %d, C %d, %s; edges %d..%d, matches %d..%d"
                  % (f, nl, occ, C, "compacted" if compact else "uncompacted loop", min(ne[l] for l in lanes),
                     max(ne[l] for l in lanes), min(odiag[k].n_matches[0] for k in range(4)),
                     max(odiag[k].n_matches[0] for k in range(4))))
    ctx.close()
    assert seen == {(1, 8, True), (2, 8, True), (2, 4, True), (2, 2, False), (2, 1, False)}, seen


def test_stalled_frame_duplicate_window_point(cuda_lib):
    """A window holding one point twice: an edge whose first two neighbours are the two copies gets a == b, so its
    residual, and with it the cost, gradient and normal equations, are NaN (non-finite on the GPU, where FMA may leave
    inf instead).  The oracle's gradient test then sees ||x - Plus(x, -g)||_inf = 0 (std::max drops NaN; fmax does
    the same on the GPU): termination 1 after 0 iterations, in both outer iterations, and the pose stays at the
    prediction.  The GPU must report the same summaries."""
    scans, _ = get_sequence("hdl64_small", 1004, 3)
    op = oracle.make_params(prev_frames=5)
    odo = oracle.Odometer(op)
    edges = []
    for s in scans:
        sp = oracle.split(op, s)
        edges.append(oracle.extract(op, sp["rings"], sp["offsets"])["edges"])
    sizes = []
    for e in edges[:2]:
        odo.process(e)
        sizes.append(len(e))
    win, _ = odo.window()
    odom, prev = odo.get_pose()
    pred = odom @ np.linalg.inv(prev) @ odom
    a = oracle.associate(edges[2], pred, win)
    found = None
    for i in np.nonzero((a["gate"] & 2) == 2)[0]:
        j = a["knn_idx"][i, 0]
        w2 = np.concatenate([win, win[j:j + 1]])
        b = oracle.associate(edges[2][i:i + 1], pred, w2)
        if b["gate"][0] & 2 and np.array_equal(w2[b["knn_idx"][0, 0], :3], w2[b["knn_idx"][0, 1], :3]):
            found = w2
            break
    assert found is not None
    sizes2 = sizes[:-1] + [sizes[-1] + 1]
    odo.set_window(found, sizes2)
    opose, od = odo.process(edges[2])
    ctx = api.Context(prev_frames=5, max_points=32768)
    _load(ctx, 0, (found, sizes2, odom, prev))
    gpose, gd = ctx.register(edges[2])
    ctx.close()
    for it in range(2):
        g, o = gd.solve[it], od.solve[it]
        print("outer %d: GPU %s cost %r, oracle %s cost %r" % (it, _ints(g), g.initial_cost, _ints(o), o.initial_cost))
        assert gd.n_matches[it] == od.n_matches[it]
        assert _ints(g) == _ints(o)
        assert (o.iterations, o.termination) == (0, 1)
        assert not np.isfinite(g.initial_cost) and not np.isfinite(o.initial_cost)
    assert np.abs(opose - pred).max() < 1e-12 and np.abs(gpose - pred).max() < 1e-12
