"""Independent NumPy / pure-Python restatement of the reference arithmetic, used only to
cross-check the C++ oracle (two restatements written separately must agree).

Citations are to /root/reference (emiliofidalgo/liodom)."""
import numpy as np


def ring_hdl64(x, y, z, min_range=3.0, max_range=75.0):
    """isValidPoint + HDL-64 ring formula (src/feature_extractor.cc:84-102, :126-138)."""
    x, y, z = np.float64(x), np.float64(y), np.float64(z)
    if not (np.isfinite(x) and np.isfinite(y) and np.isfinite(z)):
        return -1
    d = np.sqrt(x * x + y * y)
    if d > max_range or d < min_range:
        return -1
    ang = np.arctan(z / d) * 180 / np.pi
    if ang >= -8.83:
        sid = int((2 - ang) * 3.0 + 0.5)
    else:
        sid = 32 + int((-8.83 - ang) * 2.0 + 0.5)
    if ang > 2 or ang < -24.33 or sid > 63 or sid < 0:
        return -1
    return sid


def curvature(ring):
    """11-tap smoothness of one ring, float32 left-to-right sums then float64 squares
    (src/feature_extractor.cc:196-229). Returns float64 [n] with NaN outside [5, n-5)."""
    p = np.asarray(ring, np.float32)[:, :3]
    n = len(p)
    key = np.full(n, np.nan)
    if n < 11:
        return key
    j = np.arange(5, n - 5)
    acc = p[j - 5] + p[j - 4]
    acc = acc + p[j - 3]
    acc = acc + p[j - 2]
    acc = acc + p[j - 1]
    acc = acc - np.float32(10) * p[j]
    for o in (1, 2, 3, 4, 5):
        acc = acc + p[j + o]
    assert acc.dtype == np.float32
    d = acc.astype(np.float64)
    key[j] = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]
    return key


def select_ring(ring, scan_regions=8, edges_per_region=10):
    """extractFeatures region split + extractFeaturesFromRegion (src/feature_extractor.cc:238-313)
    for one ring; ties sorted by index. Returns the picked ring indices in emission order."""
    p = np.asarray(ring, np.float32)
    n = len(p)
    if n < scan_regions * edges_per_region + 10:
        return []
    key = curvature(p)
    picked = np.zeros(n + 16, bool)
    total = n - 10
    sector = total // scan_regions
    out = []

    def gap(a, b):
        d = (p[a, :3] - p[b, :3]).astype(np.float64)   # float32 difference, widened
        return d[0] * d[0] + d[1] * d[1] + d[2] * d[2]

    for r in range(scan_regions):
        lo = sector * r
        hi = total if r == scan_regions - 1 else sector * (r + 1)
        idx = np.arange(lo, hi) + 5
        order = sorted(idx, key=lambda i: (-key[i], i))
        npick = 0
        for i in order:
            if picked[i]:
                continue
            if key[i] < 0.1 or npick > edges_per_region:
                break
            out.append(int(i))
            npick += 1
            picked[i] = True
            for l in range(1, 6):
                if gap(i + l, i + l - 1) > 0.05:
                    break
                picked[i + l] = True
            for l in range(1, 6):
                if gap(i - l, i - l + 1) > 0.05:
                    break
                picked[i - l] = True
    return out


def transform(pts, T):
    """pcl::transformPointCloud with a double matrix: double math, float store (App. A.1)."""
    p = np.asarray(pts, np.float32)
    x, y, z = (p[:, k].astype(np.float64) for k in range(3))
    T = np.asarray(T, np.float64)
    out = p.copy()
    for r in range(3):
        out[:, r] = (T[r, 0] * x + T[r, 1] * y + T[r, 2] * z + T[r, 3]).astype(np.float32)
    return out


def knn5_bruteforce(map_pts, q):
    """Exact 5-NN under float32 ((dx*dx + dy*dy) + dz*dz), order (d2, idx)."""
    m = np.asarray(map_pts, np.float32)[:, :3]
    q = np.asarray(q, np.float32)[:, :3]
    idx = np.empty((len(q), 5), np.int32)
    d2o = np.empty((len(q), 5), np.float32)
    for i in range(len(q)):
        d = q[i] - m
        d2 = d[:, 0] * d[:, 0]
        d2 = d2 + d[:, 1] * d[:, 1]
        d2 = d2 + d[:, 2] * d[:, 2]
        o = np.lexsort((np.arange(len(m)), d2))[:5]
        idx[i], d2o[i] = o, d2[o]
    return idx, d2o


def cell_of(v):
    """Voxel-hash cell of a coordinate: floor(v / 0.5), saturated to int32 like a float -> int conversion on the GPU."""
    c = np.floor(np.asarray(v, np.float32) * np.float32(2.0)).astype(np.float64)
    return np.clip(np.nan_to_num(c, nan=0.0), -2.0 ** 31, 2.0 ** 31 - 1).astype(np.int64)


def knn5_gate(window, edges, pose, gate_margin=1e-9):
    """src/laser_odometry.cc:300-344 restated: the edges transformed (double math, float store), the exact 5-NN over the
    kNN target `window` under float32 L2_Simple ((dx*dx + dy*dy) + dz*dz, no FMA) in (d2, logical index) order, and the
    line gate d2[4] < 1.0 and lambda2 > 3 lambda1.  Non-finite map points are skipped; a non-finite query has no
    neighbours.

    -> dict with
      q_world [E,4]      the transformed edges;
      knn_idx, knn_d2    the five best cut at d2 < 1.0 (-1 / +inf after the cut);
      idx6, d2_6 [E,6]   the six best, uncut (-1 / +inf where the target has fewer finite points);
      gate [E] uint8     bit 0: d2[4] < 1.0; bit 1: the line test, where decided;
      decided [E] bool   the line test is decided: bit 0 clear, or |lambda2 - 3 lambda1| > gate_margin lambda2
                         (eigenvalues of the double scatter, np.linalg.eigvalsh);
      eig [E,3]          those eigenvalues (0 where bit 0 is clear);
      tie [E] bool       equal d2 between neighbours 1..6 (inside the five, or between the 5th and the 6th);
      fallback [E] bool  the 27-cell cube around the query's 0.5 m cell does not prove the list: fewer than five
                         candidates there, or the 5th of them has d2 >= 0.25 (the search then walks the 5^3 cube)."""
    w = np.asarray(window, np.float32).reshape(-1, 4)
    with np.errstate(invalid="ignore"):
        q = transform(np.asarray(edges, np.float32).reshape(-1, 4), pose)
    E, M = len(q), len(w)
    okm = np.isfinite(w[:, :3]).all(1)
    okq = np.isfinite(q[:, :3]).all(1)
    wc = np.stack([cell_of(w[:, a]) for a in range(3)], 1)
    qc = np.stack([cell_of(q[:, a]) for a in range(3)], 1)
    none = np.uint64(0xFFFFFFFFFFFFFFFF)
    keys6 = np.full((E, 6), none, np.uint64)
    cube5 = np.full(E, none, np.uint64)
    rows = max(1, (1 << 22) // max(M, 1))
    ids = np.arange(M, dtype=np.uint64)
    for a in range(0, E, rows):
        b = min(E, a + rows)
        if M == 0:
            break
        with np.errstate(invalid="ignore", over="ignore"):
            d = q[a:b, None, :3] - w[None, :, :3]
            d2 = d[..., 0] * d[..., 0]
            d2 = d2 + d[..., 1] * d[..., 1]
            d2 = d2 + d[..., 2] * d[..., 2]
        assert d2.dtype == np.float32
        key = (d2.view(np.uint32).astype(np.uint64) << np.uint64(32)) | ids[None, :]
        key[:, ~okm] = none
        key[~okq[a:b]] = none
        k = min(6, M)
        part = np.partition(key, k - 1, axis=1)[:, :k] if M > k else key
        keys6[a:b, :k] = np.sort(part, axis=1)[:, :k]
        incube = (np.abs(qc[a:b, None, :] - wc[None, :, :]) <= 1).all(2)
        ck = np.where(incube, key, none)
        if M >= 5:
            cube5[a:b] = np.partition(ck, 4, axis=1)[:, 4] if M > 5 else np.sort(ck, axis=1)[:, 4]
    have = keys6 != none
    idx6 = np.where(have, (keys6 & np.uint64(0xFFFFFFFF)).astype(np.int64), -1).astype(np.int32)
    d2_6 = np.where(have, (keys6 >> np.uint64(32)).astype(np.uint32), np.uint32(0x7F800000)).view(np.float32)
    d2_6 = d2_6.reshape(E, 6)
    keep = have[:, :5] & (d2_6[:, :5] < np.float32(1.0))
    knn_idx = np.where(keep, idx6[:, :5], -1).astype(np.int32)
    knn_d2 = np.where(keep, d2_6[:, :5], np.float32(np.inf)).astype(np.float32)
    tie = (have[:, 1:] & (d2_6[:, 1:] == d2_6[:, :-1])).any(1)
    cube_d2 = np.where(cube5 != none, (cube5 >> np.uint64(32)).astype(np.uint32), np.uint32(0x7F800000)).view(np.float32)
    fallback = okq & (cube_d2 >= np.float32(0.25))

    gate = np.zeros(E, np.uint8)
    decided = np.ones(E, bool)
    eig = np.zeros((E, 3))
    sel = np.nonzero(keep[:, 4])[0]
    gate[sel] = 1
    if len(sel):
        nn = w[idx6[sel, :5], :3].astype(np.float64)              # [n,5,3], neighbour order
        m = nn[:, 0]
        for r in range(1, 5):
            m = m + nn[:, r]
        m = m / 5.0
        C = np.zeros((len(sel), 3, 3))
        for r in range(5):
            dv = nn[:, r] - m
            C = C + dv[:, :, None] * dv[:, None, :]
        ev = np.linalg.eigvalsh(C)
        eig[sel] = ev
        dd = ev[:, 2] - 3.0 * ev[:, 1]
        decided[sel] = np.abs(dd) > gate_margin * ev[:, 2]
        gate[sel] |= np.where(decided[sel] & (dd > 0), 2, 0).astype(np.uint8)
    return dict(q_world=q, knn_idx=knn_idx, knn_d2=knn_d2, idx6=idx6, d2_6=d2_6, gate=gate, decided=decided, eig=eig,
                tie=tie, fallback=fallback)


def quat_rotate(q, v):
    """Eigen unit-quaternion * vector, q = (x,y,z,w)."""
    qv, w = np.asarray(q[:3], float), float(q[3])
    uv = 2.0 * np.cross(qv, v)
    return v + w * uv + np.cross(qv, uv)


def point2line_residual(c, a, b, q, t, min_range=3.0, max_range=75.0):
    """Point2LineFactor::operator() (include/liodom/factors.hpp:71-105), plain doubles."""
    c, a, b, t = (np.asarray(v, float) for v in (c, a, b, t))
    lp = quat_rotate(q, c) + t
    nu = np.cross(lp - a, lp - b)
    de = a - b
    cpl = c - t
    d = (np.sqrt(cpl[0] ** 2 + cpl[1] ** 2) - min_range) / (max_range - min_range)
    w = 1.01 - d
    return w * nu / np.linalg.norm(de)


def quat_plus(q, delta):
    """EigenQuaternionParameterization::Plus, storage (x,y,z,w): dq (x) q (App. A.5)."""
    delta = np.asarray(delta, float)
    n = np.linalg.norm(delta)
    if n == 0.0:
        return np.array(q, float)
    s = np.sin(n) / n
    dq = np.array([s * delta[0], s * delta[1], s * delta[2], np.cos(n)])
    ax, ay, az, aw = dq
    bx, by, bz, bw = q
    return np.array([aw * bx + ax * bw + ay * bz - az * by,
                     aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx,
                     aw * bw - ax * bx - ay * by - az * bz])


def huber_cost(cab, q, t, a=0.2, min_range=3.0, max_range=75.0):
    """Sum of 0.5 * rho(||r||^2) with ceres::HuberLoss(a)."""
    cost = 0.0
    for row in np.asarray(cab, float).reshape(-1, 9):
        r = point2line_residual(row[0:3], row[3:6], row[6:9], q, t, min_range, max_range)
        s = float(r @ r)
        cost += 0.5 * (s if s <= a * a else 2 * a * np.sqrt(s) - a * a)
    return cost


def _blocks_eval(cab, x, min_range, max_range, jac):
    """All residual blocks at x = (qx, qy, qz, qw, tx, ty, tz), vectorised: Huber-corrected residuals [3n], Jacobian
    [3n, 6] in the tangent space (A.4, A.5) and the cost.  The rows of a block are scaled by sqrt(rho') (the Corrector
    with rho'' <= 0).  q is used as given, unit or not."""
    cab = np.asarray(cab, float).reshape(-1, 9)
    c, a, b = cab[:, 0:3], cab[:, 3:6], cab[:, 6:9]
    qv, qw, t = np.asarray(x[:3], float), float(x[3]), np.asarray(x[4:7], float)
    uv = 2.0 * np.cross(qv, c)
    u = c + qw * uv + np.cross(qv, uv)               # Eigen q * c
    lp = u + t
    nu = np.cross(lp - a, lp - b)
    de = a - b
    with np.errstate(divide="ignore", invalid="ignore"):
        inv_den = 1.0 / np.sqrt(np.sum(de * de, 1))
        pxy = c[:, :2] - t[:2]
        rho = np.sqrt(np.sum(pxy * pxy, 1))
        w = 1.01 - (rho - min_range) / (max_range - min_range)
        r = (w * inv_den)[:, None] * nu
        s = np.sum(r * r, 1)
        big = s > 0.04                                   # HuberLoss(0.2); NaN takes the quadratic branch, as in Ceres
        sq = np.sqrt(np.where(big, s, 0.0))
        rho0 = np.where(big, 0.4 * sq - 0.04, s)
        rho1 = np.where(big, np.maximum(np.finfo(float).tiny, 0.2 / np.where(big, sq, 1.0)), 1.0)
        sc = np.sqrt(rho1)
        cost = 0.5 * float(np.sum(rho0))
        rs = (sc[:, None] * r).reshape(-1)
        if not jac:
            return rs, None, cost
        # d lp / d delta: q+ = dq (x) q with |dq| = 1, and Eigen's q * c equals the sandwich q c q* + (1 - |q|^2) c, so
        # the tangent derivative is 2 e_k x S with S = q c q* = u - (1 - |q|^2) c (for unit q, S = u = R c).
        S = u - (1.0 - float(qv @ qv + qw * qw)) * c
        n = len(cab)
        J = np.empty((n, 3, 6))
        wd = (w * inv_den * sc)[:, None]
        for k in range(3):
            e = np.zeros(3)
            e[k] = 1.0
            dlp = 2.0 * np.cross(e, S)
            J[:, :, k] = wd * np.cross(-de, dlp)                        # d nu / d lp = [b - a]x
            J[:, :, 3 + k] = wd * np.cross(-de, np.broadcast_to(e, de.shape))
        dw = np.zeros((n, 3))
        dw[:, :2] = pxy / (rho[:, None] * (max_range - min_range))     # d w / d t
        nd = (inv_den * sc)[:, None] * nu
        J[:, :, 3:] += nd[:, :, None] * dw[:, None, :]
    return rs, J.reshape(-1, 6), cost


def _state_plus(x, d6):
    return np.concatenate([quat_plus(x[:4], d6[:3]), np.asarray(x[4:7], float) + d6[3:]])


def lm_solve(cab, q, t, min_range=3.0, max_range=75.0, max_iterations=4):
    """ceres::Solve as the reference configures it (SURVEY.md App. A.5): trust-region Levenberg-Marquardt, Jacobi
    scaling computed once, LM diagonal clamped to [1e-6, 1e32], the augmented system [J_s; D] solved by Householder QR,
    model cost change from J, the rho test, the radius update and the three tolerances.

    -> (q, t, summary); summary has the fields of oracle.SolveSummary plus `rejected_steps`, `invalid_steps` and
    `cond_first` = cond(J_s'J_s + D^2) of the first trust-region step (NaN when none was computed)."""
    from types import SimpleNamespace
    cab = np.asarray(cab, float).reshape(-1, 9)
    n = len(cab)
    S = SimpleNamespace(iterations=0, successful_steps=0, termination=0, initial_cost=0.0, final_cost=0.0,
                        num_residual_blocks=n, cost_evals=0, jac_evals=0, rejected_steps=0, invalid_steps=0,
                        cond_first=float("nan"))
    x = np.concatenate([np.asarray(q, float), np.asarray(t, float)])
    if n == 0:
        S.termination = 4
        return x[:4].copy(), x[4:].copy(), S

    def grad_max_norm(x, g):
        # ||x - Plus(x, -g)||_inf; a NaN component is dropped (std::max / fmax keep the other operand)
        d = np.abs(_state_plus(x, -g) - x)
        d = d[~np.isnan(d)]
        return float(d.max(initial=0.0))

    r, J, cost = _blocks_eval(cab, x, min_range, max_range, True)
    S.jac_evals += 1
    S.initial_cost = cost
    scale = 1.0 / (1.0 + np.sqrt(np.sum(J * J, 0)))
    g = J.T @ r
    gmax = grad_max_norm(x, g)
    radius, decrease = 1e4, 2.0
    reuse, success, invalid = False, True, 0
    diagonal = None
    while True:
        if S.iterations >= max_iterations:
            S.termination = 0
            break
        if success and gmax <= 1e-10:
            S.termination = 1
            break
        if radius < 1e-32:
            S.termination = 5
            break
        S.iterations += 1
        Js = J * scale
        if not reuse:
            diagonal = np.minimum(np.maximum(np.sum(Js * Js, 0), 1e-6), 1e32)
        D = np.sqrt(diagonal / radius)
        if np.isnan(S.cond_first):
            S.cond_first = float(np.linalg.cond(Js.T @ Js + np.diag(D * D)))
        reuse = True
        A = np.vstack([Js, np.diag(D)])
        rhs = np.concatenate([r, np.zeros(6)])
        mcc = -np.inf
        if np.isfinite(A).all() and np.isfinite(rhs).all():
            Q, R = np.linalg.qr(A)
            y = np.linalg.solve(R, Q.T @ rhs)
            if np.isfinite(y).all():
                step = -y
                m = Js @ step
                mcc = -float(m @ (r + m / 2.0))
        if not mcc > 0.0:                                   # invalid step
            S.invalid_steps += 1
            invalid += 1
            if invalid >= 5:
                S.termination = 5
                break
            radius *= 0.5
            success = False
            continue
        invalid = 0
        xc = _state_plus(x, step * scale)
        _, _, cc = _blocks_eval(cab, xc, min_range, max_range, False)
        S.cost_evals += 1
        if not np.isfinite(cc):
            cc = cost
        if np.linalg.norm(x - xc) <= 1e-8 * (np.linalg.norm(x) + 1e-8):
            S.termination = 2
            break
        change = cost - cc
        if abs(change) <= 1e-6 * cost:
            S.termination = 3
            break
        rel = change / mcc
        if rel > 1e-3:                                      # accept
            x = xc
            r, J, cost = _blocks_eval(cab, x, min_range, max_range, True)
            S.jac_evals += 1
            g = J.T @ r
            gmax = grad_max_norm(x, g)
            S.successful_steps += 1
            radius = min(1e16, radius / max(1.0 / 3.0, 1.0 - (2.0 * rel - 1.0) ** 3))
            decrease, reuse, success = 2.0, False, True
        else:                                               # reject
            S.rejected_steps += 1
            success = False
            radius /= decrease
            decrease *= 2.0
    S.final_cost = cost
    return x[:4].copy(), x[4:].copy(), S


def exact_cost(cab, q, t, min_range=3.0, max_range=75.0):
    """The Huber cost at one point, every block in 40-digit arithmetic from the double inputs (mpmath)."""
    import mpmath
    old = mpmath.mp.dps
    mpmath.mp.dps = 40
    try:
        F = mpmath.mpf
        qx, qy, qz, qw = (F(float(v)) for v in q)
        tx, ty, tz = (F(float(v)) for v in t)
        lo, span = F(float(min_range)), F(float(max_range)) - F(float(min_range))
        total = F(0)
        for row in np.asarray(cab, float).reshape(-1, 9):
            cx, cy, cz, ax, ay, az, bx, by, bz = (F(float(v)) for v in row)
            ux, uy, uz = 2 * (qy * cz - qz * cy), 2 * (qz * cx - qx * cz), 2 * (qx * cy - qy * cx)
            lx = cx + qw * ux + (qy * uz - qz * uy) + tx
            ly = cy + qw * uy + (qz * ux - qx * uz) + ty
            lz = cz + qw * uz + (qx * uy - qy * ux) + tz
            pax, pay, paz, pbx, pby, pbz = lx - ax, ly - ay, lz - az, lx - bx, ly - by, lz - bz
            nx, ny, nz = pay * pbz - paz * pby, paz * pbx - pax * pbz, pax * pby - pay * pbx
            den2 = (ax - bx) ** 2 + (ay - by) ** 2 + (az - bz) ** 2
            w = F(1.01) - (mpmath.sqrt((cx - tx) ** 2 + (cy - ty) ** 2) - lo) / span
            s = w * w * (nx * nx + ny * ny + nz * nz) / den2
            total += s / 2 if s <= F(0.04) else (F(0.4) * mpmath.sqrt(s) - F(0.04)) / 2   # the double constants
        return total
    finally:
        mpmath.mp.dps = old


def voxelgrid(pts, leaf):
    """pcl::VoxelGrid<PointXYZI> centroids per voxel, output in ascending voxel index
    (App. A.3); in-voxel accumulation in input order (float32).  Non-finite points are skipped; when
    PCL's (max - min) * inv + 1 product exceeds INT32_MAX the input is returned unchanged."""
    p = np.asarray(pts, np.float32)
    p = p[np.isfinite(p[:, :3]).all(1)] if len(p) else p
    if len(p) == 0:
        return p.copy()
    inv = np.float32(1.0) / np.float32(leaf)
    mn, mx = p[:, :3].min(0), p[:, :3].max(0)
    dd = [int(np.float32((mx[a] - mn[a]) * inv)) + 1 for a in range(3)]
    if dd[0] * dd[1] * dd[2] > 2147483647:
        return np.asarray(pts, np.float32).copy()
    minb = np.floor(mn * inv).astype(np.int64)
    maxb = np.floor(mx * inv).astype(np.int64)
    div = maxb - minb + 1
    ijk = (np.floor(p[:, :3] * inv) - minb.astype(np.float32)).astype(np.int64)
    idx = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * div[0] * div[1]
    out = []
    for v in np.unique(idx):
        sel = np.nonzero(idx == v)[0]
        acc = np.zeros(4, np.float32)
        for i in sel:
            acc = acc + p[i]
        out.append(acc / np.float32(len(sel)))
    return np.array(out, np.float32)


def map_cell_key(p, xy=40.0, z=50.0):
    """Map cell key (src/map.cc:103-105)."""
    inv_xy, inv_z = 1.0 / xy, 1.0 / z
    return (int(np.floor(p[0] * inv_xy) * xy + xy / 2.0), int(np.floor(p[1] * inv_xy) * xy + xy / 2.0),
            int(np.floor(p[2] * inv_z) * z + z / 2.0))


class Map:
    """Map::updateMap / getMap (src/map.cc:90-139): a dict keyed by the int key triple in creation order;
    every touched cell is re-filtered by `voxelgrid` over its old centroids followed by its new points."""

    def __init__(self, xy, z, resolution):
        self.xy, self.z, self.leaf = xy, z, np.float32(resolution)
        self.cells = {}

    def update(self, pts, T):
        p = transform(pts, T)
        touched = {}
        for row in p:
            k = map_cell_key(row.astype(np.float64), self.xy, self.z)
            self.cells.setdefault(k, np.zeros((0, 4), np.float32))
            touched.setdefault(k, []).append(row)
        for k, rows in touched.items():
            self.cells[k] = voxelgrid(np.concatenate([self.cells[k], np.array(rows, np.float32)]), self.leaf)

    def keys(self):
        return np.array(list(self.cells), np.int32).reshape(-1, 3)

    def counts(self):
        return np.array([len(v) for v in self.cells.values()], np.int32)

    def get_map(self):
        return np.concatenate(list(self.cells.values())) if self.cells else np.zeros((0, 4), np.float32)
