"""CPU: the oracle's restated ceres::Solve (`oracle.solve`, DENSE_QR) against `np_ref.lm_solve`, a vectorised NumPy
restatement written from SURVEY.md App. A.5, on the shared edge cases of solve_cases.py: every controller exit, rejected
steps, Huber residuals on both sides of the threshold, negative range weights, a translation at 1e4 m, unnormalised and
w < 0 start quaternions, rotations up to 170 degrees, one to three blocks, parallel and nearly parallel lines and a NaN
block."""
import numpy as np
import pytest

import np_ref
import oracle
import solve_cases
from conftest import get_sequence

EPS = np.finfo(float).eps
CASES = {c["name"]: c for c in solve_cases.cases()}
INTS = ("iterations", "successful_steps", "termination", "num_residual_blocks", "cost_evals", "jac_evals")


def _ints(s):
    return tuple(int(getattr(s, k)) for k in INTS)


def _cost_close(a, b, n):
    """1e-12 relative; for costs near zero the residuals themselves carry ~eps * |lp| of cancellation, so an absolute
    1e-15 per block is the floor."""
    if not (np.isfinite(a) and np.isfinite(b)):
        return np.isnan(a) == np.isnan(b) and (np.isnan(a) or a == b)
    return abs(a - b) <= 1e-12 * max(abs(a), abs(b)) + 1e-15 * n


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_solve_matches_restatement(name):
    """Identical summary integers, costs within 1e-12, parameters within 1e-10, or within eps * cond(J_s'J_s + D^2) for
    the ill-conditioned cases (the two QR factorisations round differently; measured <= 0.11 eps * cond)."""
    c = CASES[name]
    oq, ot, os_ = oracle.solve(c["cab"], c["q"], c["t"], linear_solver=0)
    nq, nt, ns = np_ref.lm_solve(c["cab"], c["q"], c["t"])
    assert _ints(os_) == _ints(ns), (name, _ints(os_), _ints(ns))
    n = len(c["cab"])
    assert _cost_close(os_.initial_cost, ns.initial_cost, n), (os_.initial_cost, ns.initial_cost)
    assert _cost_close(os_.final_cost, ns.final_cost, n), (os_.final_cost, ns.final_cost)
    cond = ns.cond_first
    tol = max(1e-10, EPS * cond) if np.isfinite(cond) else 1e-10
    dp = max(np.abs(oq - nq).max(), np.abs(ot - nt).max())
    print("%-34s n=%4d exit=%d it=%d ok=%d rejected=%d cond=%.3g |dx|=%.3g (tol %.3g)"
          % (name, n, os_.termination, os_.iterations, os_.successful_steps, ns.rejected_steps, cond, dp, tol))
    assert dp <= tol, (name, dp, tol)
    if c["exit"] is not None:
        assert os_.termination == c["exit"], (name, os_.termination, c["exit"])


def test_every_exit_and_a_rejected_step_are_reached():
    """Codes 0 (max iterations), 1 (gradient), 2 (parameter), 3 (function) and 4 (no residual blocks) are each reached by
    the case built for it, and a case takes rejected steps (radius shrink).

    Code 5 cannot occur with max_num_iterations = 4: it needs either 5 consecutive invalid steps, but each one counts as
    an iteration, so the fourth ends the solve with code 0; or a radius below 1e-32, but from 1e4 the radius shrinks by
    at most a factor 2^4 per rejected step (decrease_factor doubles: 2, 4, 8, 16) or 2 per invalid step, so four
    iterations reach no lower than 1e4 / 1024 = 9.8."""
    seen = {}
    rejected = []
    for name, c in CASES.items():
        _, _, s = np_ref.lm_solve(c["cab"], c["q"], c["t"])
        _, _, o = oracle.solve(c["cab"], c["q"], c["t"])
        assert o.termination != 5 and s.termination != 5, name
        seen.setdefault(o.termination, []).append(name)
        if c["exit"] is not None:
            assert o.termination == c["exit"], name
        if s.rejected_steps:
            assert o.iterations - o.successful_steps >= s.rejected_steps   # rejected iterations are not successful
            rejected.append(name)
    assert set(seen) >= {0, 1, 2, 3, 4}, seen
    assert rejected, "no case takes a rejected step"


def test_nan_block_stalls_at_the_start():
    """A block with a == b has an undefined line: residual NaN, so cost, gradient and normal equations are NaN.  The
    gradient norm ||x - Plus(x, -g)||_inf drops the NaN components (std::max / fmax keep the other operand), which
    leaves 0: the gradient test ends the solve at iteration 0 with termination 1 and the parameters untouched.  (Real
    Ceres reports FAILURE at iteration 0 here and also leaves the parameters unchanged.)"""
    c = CASES["nan_block"]
    q, t, s = oracle.solve(c["cab"], c["q"], c["t"])
    assert (s.iterations, s.termination, s.cost_evals, s.jac_evals) == (0, 1, 0, 1)
    assert np.isnan(s.initial_cost) and np.isnan(s.final_cost)
    assert np.array_equal(q, c["q"]) and np.array_equal(t, c["t"])


def test_restated_jacobian_against_central_differences():
    """np_ref's analytic tangent Jacobian (with the lever arm q c q* for a non-unit q) against central differences of
    the residual through EigenQuaternionParameterization::Plus (translations up to 100 m: at 1e4 m the differences lose
    their digits to cancellation), and against the oracle's autodiff (all translations)."""
    rng = np.random.default_rng(7)
    from scipy.spatial.transform import Rotation
    for trial in range(12):
        c = rng.normal(size=3) * 20
        a = c + rng.normal(size=3) * 0.3
        b = a + rng.normal(size=3)
        q = Rotation.from_rotvec(rng.normal(size=3) * (0.2 if trial % 3 else 2.8)).as_quat()
        q *= (1.0, 1 + 1e-6, 1 - 1e-6, 1 + 1e-3)[trial % 4]
        if trial % 5 == 0:
            q = -q
        t = rng.normal(size=3) * (1.0, 100.0, 1e4)[trial % 3]
        x = np.concatenate([q, t])
        cab = np.concatenate([c, a, b])[None]
        _, J, _ = np_ref._blocks_eval(cab, x, 3.0, 75.0, True)
        r = np_ref.point2line_residual(c, a, b, q, t)
        s = float(r @ r)
        sc = 1.0 if s <= 0.04 else np.sqrt(0.2 / np.sqrt(s))
        h = 1e-6
        Jn = np.zeros((3, 6))
        for k in range(6):
            d = np.zeros(6)
            d[k] = h
            rp = np_ref.point2line_residual(c, a, b, np_ref.quat_plus(q, d[:3]), t + d[3:])
            rm = np_ref.point2line_residual(c, a, b, np_ref.quat_plus(q, -d[:3]), t - d[3:])
            Jn[:, k] = (rp - rm) / (2 * h)
        scale = np.abs(Jn).max()
        if trial % 3 != 2:
            assert np.abs(J / sc - Jn).max() <= 1e-6 * scale, (trial, np.abs(J / sc - Jn).max(), scale)
        _, Jo = oracle.factor(c, a, b, q, t)
        assert np.abs(J / sc - Jo).max() <= 1e-10 * np.abs(Jo).max(), trial   # 3e-12 seen at 1e4 m (cancellation)


@pytest.mark.parametrize("name", ["large_offset", "huber_both_sides", "negative_weights", "translation_1e4",
                                  "rotation_170deg", "n1"])
def test_exact_cost_pins_both_costs(name):
    """np_ref.exact_cost (40 digits) against the oracle's initial cost and np_ref's vectorised one."""
    c = CASES[name]
    _, _, o = oracle.solve(c["cab"], c["q"], c["t"])
    ex = float(np_ref.exact_cost(c["cab"], c["q"], c["t"]))
    assert abs(o.initial_cost - ex) <= 1e-12 * ex
    assert abs(np_ref._blocks_eval(c["cab"], np.concatenate([c["q"], c["t"]]), 3.0, 75.0, False)[2] - ex) <= 1e-12 * ex


def _pose_of(q, t):
    """odom_ rebuilt from param_q / param_t without renormalising (src/laser_odometry.cc:222-227)."""
    x, y, z, w = q
    T = np.eye(4)
    T[:3, :3] = [[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                 [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                 [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]]
    T[:3, 3] = t
    return T


def _quat_of(T):
    from scipy.spatial.transform import Rotation
    return Rotation.from_matrix(T[:3, :3]).as_quat()


@pytest.mark.parametrize("shape", ["c1", "c2", "c3"])
def test_real_solves_are_well_conditioned(shape):
    """cond(J_s'J_s + D^2) at the first step of every solve (both outer iterations) of teacher-forced C1 (HDL-64), C2
    (OS1-128) and C3 (HDL-64, 16 regions x 20 edges) frames, from the oracle's own windows, predictions and residual
    blocks.  The pipeline stays far below solve_cases.COND_MAX, the bound under which the GPU's normal-equation
    Cholesky must agree with QR at the 1e-7 / 1e-8 contract."""
    from liodom_b200 import synth
    w = h = 0
    if shape == "c1":
        sensor, kw = "hdl64", dict(prev_frames=15)
    elif shape == "c2":
        sensor, kw = "os1_128", dict(lidar_type=1, scan_lines=128, prev_frames=15)
        w, h = synth.sensor_shape(sensor)
    else:
        sensor, kw = "hdl64", dict(scan_regions=16, edges_per_region=20, prev_frames=20)
    scans, _ = get_sequence(sensor, 1000, 6)
    op = oracle.make_params(**kw)
    odo = oracle.Odometer(op)
    conds = []
    for f, s in enumerate(scans):
        sp = oracle.split(op, s, w, h)
        edges = oracle.extract(op, sp["rings"], sp["offsets"])["edges"]
        if f > 0:
            window, _ = odo.window()
            T = np.array(odo.process(edges)[1].pred_pose).reshape(4, 4)
            q, t = _quat_of(T), T[:3, 3].copy()
            if q[3] < 0:
                q = -q
            for it in range(2):
                a = oracle.associate(edges, T, window)
                sel = (a["gate"] & 2) == 2
                idx = a["knn_idx"][sel]
                cab = np.concatenate([edges[sel][:, :3], window[idx[:, 0]][:, :3], window[idx[:, 1]][:, :3]], 1).astype(float)
                q, t, sm = np_ref.lm_solve(cab, q, t)
                conds.append(sm.cond_first)
                T = _pose_of(q, t)
        else:
            odo.process(edges)
    conds = np.array(conds)
    print("%s: %d solves, cond(J_s'J_s + D^2) min %.3g median %.3g max %.3g (threshold %.3g)"
          % (shape, len(conds), conds.min(), np.median(conds), conds.max(), solve_cases.COND_MAX))
    assert len(conds) == 10 and (conds < solve_cases.COND_MAX / 1e3).all()
