"""Shared edge cases of one LM solve (`oracle.solve`, `np_ref.lm_solve`, `liodom_solve`): every controller exit, the
geometry where the residual, its weight or the linear system degenerate.  Imported by test_oracle_solve_edges.py and
test_gpu_solve_edges.py."""
import numpy as np

# The GPU solves the 6x6 normal equations (J_s'J_s + D^2) y = J_s'r by Cholesky; the reference uses Householder QR on
# [J_s; D].  The two steps differ by about eps * cond(J_s'J_s + D^2) relative to the step (measured on the cases below:
# at most 0.11 eps * cond, steps of at most ~1 in tangent units).  Below COND_MAX that is under the 1e-8 quaternion /
# 1e-7 translation contract of the GPU parity tests; above it the GPU is held to the oracle's Cholesky instead.
COND_MAX = 1e-8 / np.finfo(float).eps


def _rot(axis, angle):
    """(x, y, z, w) quaternion of a rotation by `angle` about `axis`."""
    axis = np.asarray(axis, float)
    axis = axis / np.linalg.norm(axis)
    return np.concatenate([np.sin(angle / 2) * axis, [np.cos(angle / 2)]])


def _apply(q, v):
    qv, w = q[:3], q[3]
    uv = 2.0 * np.cross(qv, v)
    return v + w * uv + np.cross(qv, uv)


def scene(seed, n, q_true, t_true, dirs=None, offsets=None, spread=20.0, centre=(0.0, 0.0, 0.0)):
    """n edges c (sensor frame) and lines through their true world positions R c + t along `dirs`, shifted sideways by
    `offsets` metres (the residual left at the optimum).  -> cab [n, 9]."""
    rng = np.random.default_rng(seed)
    c = rng.normal(size=(n, 3)) * [spread, spread, spread / 8] + centre
    lp = np.array([_apply(np.asarray(q_true, float), ci) for ci in c]).reshape(-1, 3) + t_true
    d = rng.normal(size=(n, 3)) if dirs is None else np.broadcast_to(np.asarray(dirs, float), (n, 3)).copy()
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-300)
    side = np.cross(d, rng.normal(size=(n, 3)))
    side /= np.maximum(np.linalg.norm(side, axis=1, keepdims=True), 1e-300)
    off = np.zeros(n) if offsets is None else np.broadcast_to(np.asarray(offsets, float), (n,))
    base = lp + side * off[:, None]
    s1 = rng.uniform(-1.0, -0.2, size=(n, 1))
    s2 = rng.uniform(0.2, 1.0, size=(n, 1))
    return np.concatenate([c, base + s1 * d, base + s2 * d], 1)


def _perturb(q, t, rotvec, dt):
    from scipy.spatial.transform import Rotation
    qn = (Rotation.from_rotvec(rotvec) * Rotation.from_quat(q)).as_quat()
    if np.dot(qn, q) < 0:
        qn = -qn
    return qn, np.asarray(t, float) + dt


def _mixed(seed, n):
    """Sideways offsets on both sides of the Huber threshold (|r| = 0.2 at unit weight)."""
    rng = np.random.default_rng(seed + 77)
    return np.where(rng.random(n) < 0.5, rng.uniform(0.0, 0.15, n), rng.uniform(0.3, 1.5, n))


def cases():
    """-> list of dict(name, cab, q, t, exit) where `exit` is the termination the case is built to reach (None: any).

    Termination codes: 0 max iterations, 1 gradient, 2 parameter, 3 function, 4 no residual blocks, 5 failure."""
    I = np.array([0.0, 0.0, 0.0, 1.0])
    qa = _rot([0.3, -0.2, 1.0], 0.4)
    ta = np.array([2.0, -1.0, 0.3])
    out = []

    def add(name, cab, q, t, exit=None):
        out.append(dict(name=name, cab=np.ascontiguousarray(cab, float).reshape(-1, 9), q=np.array(q, float),
                        t=np.array(t, float), exit=exit))

    # --- exits
    add("no_blocks", np.zeros((0, 9)), I, [1.0, 2.0, 3.0], exit=4)
    exact = scene(1, 400, qa, ta, dirs=[0.0, 0.0, 1.0])
    add("zero_residual_at_start", exact, qa, ta, exit=1)
    mixed = scene(2, 600, qa, ta, offsets=_mixed(2, 600))
    q, t = _perturb(qa, ta, [0.25, -0.1, 0.3], [1.0, -0.8, 0.4])
    add("large_offset", mixed, q, t, exit=0)
    add("near_optimum_parameter_tolerance", exact, *_optimum(exact, qa, ta, 1e-9), exit=2)
    add("near_optimum_function_tolerance", mixed, *_optimum(mixed, qa, ta, 2e-5), exit=3)
    # six blocks 70 m out, started 1.6 rad and 7 m off: the Gauss-Newton model is poor, so steps are rejected (the
    # radius shrinks) between accepted ones
    t70 = np.array([70.0, 10.0, 0.0])
    cab = scene(741, 6, qa, t70, offsets=_mixed(741, 6))
    add("rejected_steps", cab, *_perturb(qa, t70, [-1.136, 0.421, -1.055], [3.07, -5.984, -1.612]))

    # --- geometry
    add("huber_both_sides", mixed, *_perturb(qa, ta, [0.02, 0.01, -0.03], [0.2, 0.1, -0.05]))
    far_t = np.array([150.0, 120.0, 0.0])        # (c - t)_xy beyond ~75.7 m: negative range weights
    cab = scene(3, 500, qa, far_t, offsets=_mixed(3, 500))
    add("negative_weights", cab, *_perturb(qa, far_t, [0.01, 0.0, 0.02], [0.3, -0.2, 0.1]))
    huge_t = np.array([1e4, -1e4, 25.0])
    cab = scene(4, 500, qa, huge_t, offsets=_mixed(4, 500))
    add("translation_1e4", cab, *_perturb(qa, huge_t, [0.0, 0.005, 0.01], [0.2, 0.1, 0.0]))
    q, t = _perturb(qa, ta, [0.03, -0.02, 0.05], [0.3, 0.2, -0.1])
    add("start_w_negative", mixed, -q, t)
    add("start_norm_plus_1e-6", mixed, q * (1 + 1e-6), t)
    add("start_norm_minus_1e-6", mixed, q * (1 - 1e-6), t)
    q170 = _rot([0.2, 0.1, 1.0], np.deg2rad(170.0))
    cab = scene(5, 500, q170, ta, offsets=_mixed(5, 500))
    add("rotation_170deg", cab, *_perturb(q170, ta, [0.05, 0.02, -0.08], [0.2, -0.3, 0.05]))
    add("rotation_170deg_from_identity", cab, I, [0.0, 0.0, 0.0])
    for n in (1, 2, 3):
        cab = scene(10 + n, n, qa, ta, offsets=[0.1])
        add("n%d" % n, cab, *_perturb(qa, ta, [0.01, -0.02, 0.01], [0.1, 0.05, -0.02]))
    cab = scene(20, 300, qa, ta, dirs=[0.0, 0.0, 1.0], offsets=_mixed(20, 300))
    add("parallel_vertical", cab, *_perturb(qa, ta, [0.0, 0.0, 0.02], [0.2, -0.1, 0.3]))
    for k, tilt in enumerate((1e-3, 1e-4, 1e-5, 1e-6)):
        rng = np.random.default_rng(30 + k)
        ang = rng.uniform(0, 2 * np.pi, 300)
        dirs = np.stack([tilt * np.cos(ang), tilt * np.sin(ang), np.ones(300)], 1)
        cab = scene(30 + k, 300, I, ta, dirs=None, offsets=_mixed(30 + k, 300))
        # rebuild the lines with the nearly vertical directions (scene() draws one direction per block)
        c = cab[:, :3]
        lp = c + ta
        side = np.cross(dirs, rng.normal(size=(300, 3)))
        side /= np.linalg.norm(side, axis=1, keepdims=True)
        base = lp + side * _mixed(30 + k, 300)[:, None]
        dn = dirs / np.linalg.norm(dirs, axis=1, keepdims=True)
        cab = np.concatenate([c, base - 0.5 * dn, base + 0.7 * dn], 1)
        add("nearly_parallel_%g" % tilt, cab, *_perturb(I, ta, [0.0, 0.0, 0.01], [0.1, -0.1, 0.2]))
    nan_cab = mixed[:200].copy()
    nan_cab[57, 6:9] = nan_cab[57, 3:6]           # a == b: the line is undefined, the residual NaN
    add("nan_block", nan_cab, *_perturb(qa, ta, [0.01, 0.0, 0.0], [0.1, 0.0, 0.0]), exit=1)
    return out


def _optimum(cab, q_true, t_true, eps):
    """A point `eps` (tangent units) away from the stationary point of `cab`'s cost nearest the true pose: Gauss-Newton
    on the Huber-corrected system (the model Ceres minimises), run to convergence, then a fixed nudge."""
    import np_ref
    x = np.concatenate([q_true, t_true]).astype(float)
    for _ in range(30):
        r, J, _ = np_ref._blocks_eval(cab, x, 3.0, 75.0, True)
        d = np.linalg.lstsq(J, -r, rcond=None)[0]
        x = np.concatenate([np_ref.quat_plus(x[:4], d[:3]), x[4:] + d[3:]])
    d = np.array([0.6, -0.3, 0.5, 0.4, -0.7, 0.2]) * eps
    return np_ref.quat_plus(x[:4], d[:3]), x[4:] + d[3:]
