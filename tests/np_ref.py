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
