"""Constructed inputs of the association stage (window, kNN target, queries, pose), shared by the oracle test and the GPU
test.  Each case is built for one regime of the exact 5-NN search or the line gate (register.cu:704-866) and checks,
through np_ref.knn5_gate, that it reaches that regime, so that an edit cannot quietly turn it into an easy case.

Coordinates are chosen so that the float32 distances come out exactly where they are needed: dyadic offsets, and the
rounding of 0.5 + 2^-30 to 0.5, which puts a point two 0.5 m cells away from the query at a float d2 of exactly 0.25."""
import numpy as np

import np_ref

F = np.float32
INF = F(np.inf)
TINY = F(2.0 ** -30)       # 0.5 + TINY rounds to 0.5 in float32
ECAP = 64 * 8 * 11         # edge capacity of the default parameters (scan_lines x scan_regions x (edges_per_region + 1))


class Case:
    """frames: window frames (oldest first); received: the received map (mapping = 1) or None; edges: the queries before
    the pose; prev_frames: the window length (filter_local_map applies when the window is full)."""

    def __init__(self, name, frames, edges, pose=None, received=None, filter_local_map=False, prev_frames=None, check=None):
        self.name = name
        self.frames = [np.asarray(f, np.float32).reshape(-1, 4) for f in frames]
        self.edges = np.asarray(edges, np.float32).reshape(-1, 4)
        self.pose = np.eye(4) if pose is None else np.asarray(pose, np.float64)
        self.received = None if received is None else np.asarray(received, np.float32).reshape(-1, 4)
        self.filter_local_map = filter_local_map
        self.prev_frames = prev_frames or max(1, len(self.frames))
        self._check = check
        self._ref = None

    def window(self):
        return np.concatenate(self.frames) if self.frames else np.zeros((0, 4), np.float32)

    def target(self):
        """The kNN target in logical order: the window (VoxelGrid(0.4) of it once full, with filter_local_map), then the
        received map (src/laser_odometry.cc:286-314)."""
        w = self.window()
        if self.filter_local_map and self.received is None and len(self.frames) == self.prev_frames:
            w = np_ref.voxelgrid(w, 0.4)
        if self.received is not None:
            w = np.concatenate([w, self.received])
        return w

    def context_kw(self):
        kw = dict(prev_frames=self.prev_frames, filter_local_map=int(self.filter_local_map), max_points=8192)
        if self.received is not None:
            kw.update(mapping=1, max_received_map=max(1024, len(self.received)))
        return kw

    def ref(self):
        if self._ref is None:
            self._ref = np_ref.knn5_gate(self.target(), self.edges, self.pose)
        return self._ref

    def check(self):
        """Asserts the regime the case is named for; returns the restatement's result."""
        r = self.ref()
        if self._check is not None:
            self._check(self, r)
        return r


def cut_list(o):
    """An oracle.associate five-list cut at d2 < 1.0 (-1 / +inf after the cut), as the GPU reports it."""
    keep = (o["knn_idx"] >= 0) & (o["knn_d2"] < np.float32(1.0))
    return np.where(keep, o["knn_idx"], -1), np.where(keep, o["knn_d2"], np.float32(np.inf)).astype(np.float32)


# ---- helpers ------------------------------------------------------------------------------------------------------
def P(*xyz):
    return np.array([xyz[0], xyz[1], xyz[2], 0.0], np.float32)


def d2f(q, p):
    d = np.asarray(q, F)[:3] - np.asarray(p, F)[:3]
    return (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]


def at_d2(q, p0, axis, target, span=1 << 16):
    """p0 with coordinate `axis` moved by at most `span` float steps so that d2f(q, p) == target exactly."""
    p0 = np.asarray(p0, F)
    b = np.int64(np.array([p0[axis]], F).view(np.int32)[0])
    cand = np.arange(b - span, b + span, dtype=np.int64)
    v = cand.astype(np.int32).view(np.float32)
    v = v[np.isfinite(v) & (np.sign(v) == np.sign(p0[axis]))]
    P_ = np.repeat(p0[None], len(v), 0)
    P_[:, axis] = v
    d = np.asarray(q, F)[None, :3] - P_[:, :3]
    dd = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    hit = np.nonzero(dd == F(target))[0]
    assert len(hit), "no float point at d2 = %r" % target
    return P_[hit[len(hit) // 2]]


def cells(p):
    return np.array([np_ref.cell_of(np.float32(p[a])) for a in range(3)])


def nn_cells_apart(q, p):
    return int(np.max(np.abs(cells(p) - cells(q))))


def lowest(frames_lo, frames_hi):
    """Two frames: the first holds the points that must win ties (lower logical indices)."""
    return [np.array(frames_lo, np.float32).reshape(-1, 4), np.array(frames_hi, np.float32).reshape(-1, 4)]


def _index_of(frames, p):
    w = np.concatenate(frames)
    hit = np.nonzero((w[:, :3] == p[:3]).all(1))[0]
    assert len(hit) == 1
    return int(hit[0])


# ---- cases --------------------------------------------------------------------------------------------------------
def _cell_faces():
    """Map points on a 0.5 m lattice (every coordinate k/2 or one ulp either side, zeros of both signs, negative cells)
    and queries on the same values: floorf on the faces and the axis_gap box bounds."""
    rng = np.random.default_rng(101)
    ks = (np.arange(-6, 7) * 0.5).astype(F)
    X, Y, Z = np.meshgrid(ks, ks, ks, indexing="ij")
    p = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)
    nudge = rng.integers(-1, 2, size=p.shape)
    p = np.where(nudge < 0, np.nextafter(p, -INF), np.where(nudge > 0, np.nextafter(p, INF), p)).astype(F)
    p[(p == 0) & (rng.random(p.shape) < 0.5)] = F(-0.0)
    p = p[rng.permutation(len(p))]
    pts = np.concatenate([p, np.zeros((len(p), 1), F)], 1)
    S = []
    for k in range(-5, 6):
        v = F(k * 0.5)
        S += [v, np.nextafter(v, -INF), np.nextafter(v, INF), F(k * 0.5 + 0.25)]
    S += [F(-0.0)]
    S = np.array(S, F)
    q = S[rng.integers(0, len(S), size=(700, 3))]
    q[:30] = F(-0.0)
    q[30:60, 0] = F(-0.0)
    edges = np.concatenate([q, np.ones((len(q), 1), F)], 1)

    def check(c, r):
        qw = r["q_world"][:, :3]
        on_face = (qw * 2 == np.floor(qw * 2)).any(1)
        assert on_face.sum() > 300
        assert (np.signbit(qw) & (qw == 0)).any() and (qw < -1).any()
        assert r["tie"].sum() > 50 and r["fallback"].sum() > 50 and (~r["fallback"]).sum() > 20
    pose = np.eye(4)
    pose[:3, 3] = -0.0                   # x + (-0.0) keeps the sign of a zero coordinate
    return Case("cell_faces", [pts[:1100], pts[1100:]], edges, pose=pose, check=check)


def _slot(g):
    """(y, z) of group g, 3 m from every other group; |y| < 4 keeps the float steps of y fine enough for at_d2."""
    return [-2.75, 0.25, 3.25][g % 3], 0.25 + 3.0 * (g // 3)


def _close4(q):
    """Four points at d2 = 1/64 from q (inside its own cell)."""
    return [P(q[0], q[1], q[2] + 0.125), P(q[0], q[1], q[2] - 0.125), P(q[0], q[1] + 0.125, q[2]), P(q[0], q[1] - 0.125, q[2])]


def _proven_radius():
    """The 5th neighbour at d2 exactly 0.25 (the kProvenD2 hand-off to the fallback) and one ulp either side.  q.x = 0.5
    (cell 1), so a point at x = -2^-30 (cell -1, outside the 27-cell cube) is at a float d2 of exactly 0.25."""
    lo, hi, edges, expect = [], [], [], []
    below, above = np.nextafter(F(0.25), F(0)), np.nextafter(F(0.25), F(1))
    for g in range(12):
        q = P(0.5, *_slot(g))
        y, z = q[1], q[2]
        hi += _close4(q)
        kind = g % 4
        if kind == 0:     # tie at exactly 0.25: outside the cube at the lower index, inside at the higher one
            a, b = P(-TINY, y, z), P(1.0, y, z)
            lo.append(a); hi.append(b); expect.append((0.25, a, 2))
        elif kind == 1:   # 5th one ulp below 0.25 inside the cube; a lower-index point outside at 0.25 must not enter
            c = at_d2(q, P(0.5 - 0.4999, y + 0.01, z), 1, below)
            lo.append(P(-TINY, y, z)); hi.append(c); expect.append((below, c, 1))
        elif kind == 2:   # 5th one ulp above 0.25, outside the cube; a lower-index point inside one ulp further
            c = at_d2(q, P(-TINY, y + 1.7e-4, z), 1, above)
            e = at_d2(q, P(1.0, y + 2.5e-4, z), 1, np.nextafter(above, F(1)))
            lo.append(e); hi.append(c); expect.append((above, c, 2))
        else:             # exactly 0.25 on both sides of the cube along y and z too: five-way tie for the 5th
            pts = [P(-TINY, y, z), P(1.0, y, z), P(0.5, y + 0.5, z), P(0.5, y - 0.5, z), P(0.5, y, z + 0.5)]
            lo.append(pts[0]); hi += pts[1:]; expect.append((0.25, pts[0], 2))
        edges.append(q)
    frames = lowest(lo, hi)

    def check(c, r):
        for i, (d2, p, apart) in enumerate(expect):
            assert r["d2_6"][i, 4] == F(d2), (i, r["d2_6"][i])
            assert r["idx6"][i, 4] == _index_of(c.frames, p), i
            assert nn_cells_apart(r["q_world"][i], p) == apart, i
            assert r["fallback"][i] == (F(d2) >= F(0.25)), i
    return Case("proven_radius", frames, edges, check=check)


def _gate_radius():
    """The 1 m gate: the 5th at d2 exactly 1.0 (fails) and one ulp below (passes); fewer than five within 1 m (partial
    lists: the GPU returns the neighbours within 1 m, -1 for the rest)."""
    lo, hi, edges, kinds = [], [], [], []
    rng = np.random.default_rng(7)
    for g in range(10):
        q = P(0.5, *_slot(g))
        y, z = q[1], q[2]
        kind = g % 5
        if kind == 0:
            hi += _close4(q); hi.append(P(-0.5, y, z))
        elif kind == 1:
            hi += _close4(q); hi.append(at_d2(q, P(0.5 - 0.9999, y + 0.01414, z), 1, np.nextafter(F(1), F(0))))
        elif kind == 2:   # three within 1 m, the rest just beyond
            hi += _close4(q)[:3]
            hi += [P(0.5, y + 1.0, z), P(0.5, y, z - 1.0), P(-0.5, y, z), at_d2(q, P(1.5, y + 0.001, z), 1, np.nextafter(F(1), F(2)))]
        elif kind == 3:   # two between 0.5 m and 1 m only: found by the fallback alone
            hi += [P(0.5, y + 0.75, z), P(0.5, y, z - 0.875), P(0.5 + 1.25, y, z)]
        else:             # nothing within 1 m; several exactly at 1 m
            hi += [P(0.5, y + 1.0, z), P(0.5, y - 1.0, z), P(1.5, y, z), P(-0.5, y, z), P(0.5, y, z + 1.0)]
        kinds.append(kind)
        edges.append(q)
    hi = [hi[i] for i in rng.permutation(len(hi))]
    frames = lowest(np.zeros((0, 4)), hi)

    def check(c, r):
        n = (r["knn_idx"] >= 0).sum(1)
        for i, kind in enumerate(kinds):
            assert n[i] == [4, 5, 3, 2, 0][kind], (i, n[i])
        assert (r["d2_6"][np.array(kinds) == 0, 4] == F(1)).all()
        assert (r["d2_6"][np.array(kinds) == 1, 4] == np.nextafter(F(1), F(0))).all()
    return Case("gate_radius", frames, edges, check=check)


def _fallback_only():
    """The 27-cell cube around the query is empty; all five neighbours lie in the 5^3 ring (0.75 - 0.99 m away)."""
    rng = np.random.default_rng(17)
    pts, edges = [], []
    for g in range(40):
        q = np.array([4.0 * (g % 8) + rng.uniform(0, 0.5), 4.0 * (g // 8) + rng.uniform(0, 0.5), rng.uniform(-1, 1)], F)
        n = 0
        while n < 7:
            u = rng.normal(size=3)
            p = (q + u / np.linalg.norm(u) * rng.uniform(0.75, 0.99)).astype(F)
            if nn_cells_apart(q, p) == 2:
                pts.append(P(*p)); n += 1
        edges.append(P(*q))
    pts = np.array(pts)[rng.permutation(len(pts))]

    def check(c, r):
        assert r["fallback"].all() and (r["gate"] & 1).all()
        w = c.target()
        for i in range(len(c.edges)):
            assert all(nn_cells_apart(r["q_world"][i], w[j]) == 2 for j in r["idx6"][i, :5])
    return Case("fallback_only", [pts[:150], pts[150:]], edges, check=check)


def _ties():
    """Equal float d2 at every tie-break site: duplicates across frames, mirror pairs, six equidistant points straddling
    positions 5 / 6, equal d2 in cells of different group lanes and fallback rows, and a point on the nearest face of a
    neighbour cell whose d2 equals the current 5th at a lower index (the strict > of the cell and row pruning)."""
    rng = np.random.default_rng(23)
    f0, f1, f2, edges, faces = [], [], [], [], []
    # duplicates across frames
    cloud = np.round(rng.normal(size=(200, 3)) * 0.6 * 64) / 64
    for f in (f0, f1, f2):
        f += [P(*p) for p in cloud]
    edges += [P(*p) for p in np.round(rng.normal(size=(100, 3)) * 0.6 * 128) / 128]
    # mirror pairs q +- v (dyadic: q +- v exact, equal d2)
    for g in range(40):
        q = np.array([10.0 + 3.0 * (g % 8), 3.0 * (g // 8), 0.0]) + np.round(rng.uniform(0, 0.5, 3) * 64) / 64
        for _ in range(4):
            v = np.round(rng.uniform(-0.6, 0.6, 3) * 64) / 64
            (f0 if rng.random() < 0.5 else f1).append(P(*(q + v)))
            (f1 if rng.random() < 0.5 else f2).append(P(*(q - v)))
        edges.append(P(*q))
    # six points at equal d2 on the axes, indices in random frames: positions 5 and 6 tie
    for g, a in enumerate([0.375, 0.5, 0.625, 0.875] * 4):
        q = np.array([40.0 + 3.0 * (g % 4), 3.0 * (g // 4), 0.0]) + 0.25
        six = [q + s * a * e for e in np.eye(3) for s in (1.0, -1.0)]
        order = rng.permutation(6)
        for k, j in enumerate(order):
            [f0, f1, f2][k % 3].append(P(*six[j]))
        edges.append(P(*q))
    # a point on the nearest face of a neighbour cell (lowest index) at the d2 of the own cell's five
    for g in range(12):
        axis = g % 3
        base = np.array([60.0 + 3.0 * g, -6.0 + 3.0 * (g % 2), -3.0]) + 0.25
        q = base.copy(); q[axis] += 0.0625                 # 0.1875 from the face at +0.25 of the cell centre
        face = q.copy(); face[axis] = base[axis] + 0.25
        own = []
        for e in range(3):
            for s in ((-1.0, 1.0) if e != axis else (-1.0,)):
                p = q.copy(); p[e] += s * 0.1875; own.append(p)
        f0.append(P(*face))
        for p in own:
            f2.append(P(*p))
        faces.append((len(edges), face))
        edges.append(P(*q))

    def check(c, r):
        assert r["tie"].mean() > 0.6
        n = len(edges) - len(faces)
        # the face point ties with the own cell's five and has the lowest index
        for i, face in faces:
            assert r["d2_6"][i, 5] == r["d2_6"][i, 0] == F(0.1875 ** 2), i
            assert r["idx6"][i, 0] == _index_of(c.frames, P(*face)), i
        assert (r["d2_6"][n - 16:n, 4] == r["d2_6"][n - 16:n, 5]).all()
    return Case("ties", [f0, f1, f2], edges, check=check)


def _stationary_cloud(n=3000, seed=31):
    rng = np.random.default_rng(seed)
    c = rng.normal(size=(n, 4)) * [4.0, 4.0, 1.0, 0.0]
    return c.astype(np.float32)


def _stationary():
    """A stalled sensor: K = 3 bit-identical copies of one cloud; every query is one of its points, so every edge ties."""
    cloud = _stationary_cloud()
    rng = np.random.default_rng(37)
    edges = cloud[rng.choice(len(cloud), 500, replace=False)]

    def check(c, r):
        assert r["tie"].all()
        assert (r["gate"] & 1).mean() > 0.9
    return Case("stationary", [cloud, cloud, cloud], edges, check=check)


def _pool_overflow():
    """32 queries at one point of cell (0, 0, 0) — one warp of a one-thread-per-edge kernel — whose own cell holds five
    points at d2 = 0.125, and 18 neighbour cells that hold 10 copies each of points at the same d2 and lower indices:
    7680 candidates pass their owners' bound (> kPoolSurv = 224) and every query lists 18 buckets (> kPoolSegs = 8)."""
    rng = np.random.default_rng(41)
    side = [F(0.5), F(0.0), -TINY]       # |0.25 - v| rounds to 0.25 for all three; cells +1, 0, -1
    own, nb = [], []
    for a, b in ((0, 1), (0, 2), (1, 2)):
        for va in side:
            for vb in side:
                p = np.full(3, 0.25, F); p[a] = va; p[b] = vb
                (own if (va == 0 and vb == 0) else nb).append(P(*p))
    own = own + own[:2]
    nb = [p for p in nb for _ in range(10)]
    nb = [nb[i] for i in rng.permutation(len(nb))]
    q = P(0.25, 0.25, 0.25)
    edges = [q] * 32 + [P(*(np.array([0.25, 0.25, 0.25]) + rng.uniform(-0.2, 0.2, 3))) for _ in range(32)]

    def check(c, r):
        w = c.target()
        d2 = np.array([d2f(q, p) for p in w])
        same = d2 == r["d2_6"][0, 4]
        assert r["d2_6"][0, 4] == F(0.125) and 32 * same.sum() > 224
        occ = {tuple(cells(p)) for p in w[same]} - {(0, 0, 0)}
        assert len(occ) >= 9
        assert (r["idx6"][:32, :5] < len(nb)).all()
    return Case("pool_overflow", [nb, own], edges, check=check)


def _dense_cell():
    """5000 points on a 1/64 m grid in one 0.5 m cell (the strided own-cell scan of G = 4 / 8 / 16 and the tail of
    knn_scan_bucket), duplicates and equal-d2 ties included."""
    rng = np.random.default_rng(43)
    lo = np.array([1.0, 0.5, 0.0])
    p = lo + np.floor(rng.uniform(0, 0.5, (5000, 3)) * 64) / 64
    pts = np.concatenate([p, np.zeros((len(p), 1))], 1).astype(F)
    side = lo + rng.uniform(-0.5, 1.0, (300, 3))
    spts = np.concatenate([side, np.zeros((300, 1))], 1).astype(F)
    q = np.concatenate([lo + np.floor(rng.uniform(0, 0.5, (200, 3)) * 128) / 128, lo + rng.uniform(-0.5, 1.0, (100, 3))])
    edges = np.concatenate([q, np.ones((len(q), 1))], 1)

    def check(c, r):
        qc = np.stack([np_ref.cell_of(r["q_world"][:200, a]) for a in range(3)], 1)
        assert (qc == [2, 1, 0]).all()
        assert r["tie"][:200].mean() > 0.5
    return Case("dense_cell", [pts[:3000], np.concatenate([pts[3000:], spts])], edges, check=check)


FILTER_CX = (-34, -33, -32, -31, -2, -1, 0, 1, 30, 31, 32, 33)


def _filter_word():
    """Query cells whose 5-cell fallback row (cx - 2 .. cx + 2) or 3-cell cube row crosses a 32-cell occupancy word,
    negative cells included; sparse points so that most queries walk the fallback rows."""
    rng = np.random.default_rng(47)
    pts, edges = [], []
    for g, cx in enumerate(FILTER_CX * 3):
        q = np.array([cx * 0.5 + rng.uniform(0, 0.5), 3.0 * g, rng.uniform(-0.5, 0.5)])
        for _ in range(9):
            u = rng.normal(size=3)
            pts.append(P(*(q + u / np.linalg.norm(u) * rng.uniform(0.3, 1.0))))
        edges.append(P(*q))
    pts = [pts[i] for i in rng.permutation(len(pts))]

    def check(c, r):
        cx = np_ref.cell_of(r["q_world"][:, 0])
        assert set(FILTER_CX) <= set(cx.tolist())
        assert (((cx - 2) & 31) >= 28).sum() >= 24 and r["fallback"].mean() > 0.5
    return Case("filter_word", [pts[:200], pts[200:]], edges, check=check)


def _far_aliased():
    """A window around x = +-16384 m (cells +-32768: the same 16-bit packed key), clusters 32768 m apart (same key), and
    finite points beyond 2^30 m, where the float -> int cell conversion saturates."""
    rng = np.random.default_rng(53)
    pts, q = [], []
    centres = [(16384.3, 0.3, 0.3), (-16383.7, 0.3, 0.3), (0.3, 5.3, 0.3), (32768.3, 5.3, 0.3)]
    for cen in centres:
        pts.append(np.asarray(cen) + rng.normal(size=(300, 3)) * 0.5)
        q.append(np.asarray(cen) + rng.normal(size=(60, 3)) * 0.5)
    for x in (F(1.5 * 2 ** 31), F(-1.5 * 2 ** 31), F(2.0 ** 30)):
        yz = rng.normal(size=(200, 2)) * 0.5
        pts.append(np.concatenate([np.full((200, 1), x), yz], 1))
        q.append(np.concatenate([np.full((40, 1), x), rng.normal(size=(40, 2)) * 0.5], 1))
    pts = np.concatenate(pts)
    pts = np.concatenate([pts, np.zeros((len(pts), 1))], 1).astype(F)
    pts = pts[rng.permutation(len(pts))]
    q = np.concatenate(q)
    edges = np.concatenate([q, np.ones((len(q), 1))], 1).astype(F)

    def check(c, r):
        cx = np_ref.cell_of(r["q_world"][:, 0]) & 0xFFFF   # the x field of the packed cell key
        assert len(set(cx[:60]) & set(cx[60:120])) >= 3 and len(set(cx[120:180]) & set(cx[180:240])) >= 3
        cx = np_ref.cell_of(r["q_world"][:, 0])
        assert (np.abs(cx) >= 2 ** 31 - 1).sum() == 120
        assert (r["gate"] & 1).mean() > 0.8
    return Case("far_aliased", [pts[:1000], pts[1000:]], edges, check=check)


def _nonfinite():
    """NaN and +-inf map points (skipped) and queries (no neighbours)."""
    rng = np.random.default_rng(59)
    pts = (rng.normal(size=(1200, 4)) * [1.0, 1.0, 0.4, 1.0]).astype(F)
    bad = rng.choice(1200, 80, replace=False)
    pts[bad, rng.integers(0, 3, 80)] = rng.choice([np.nan, np.inf, -np.inf], 80)
    q = (rng.normal(size=(300, 4)) * [1.0, 1.0, 0.4, 1.0]).astype(F)
    qbad = rng.choice(300, 30, replace=False)
    q[qbad, rng.integers(0, 3, 30)] = rng.choice([np.nan, np.inf, -np.inf], 30)
    q[:10] = pts[bad[:10]]                # queries on the non-finite map points themselves

    def check(c, r):
        fin = np.isfinite(r["q_world"][:, :3]).all(1)
        assert (~fin).sum() >= 30 and (r["knn_idx"][~fin] == -1).all()
        assert not np.isin(r["idx6"], bad).any()
        assert (r["gate"][fin] & 1).mean() > 0.8
    return Case("nonfinite", [pts[:600], pts[600:]], q, check=check)


def _line_gate_margin():
    """Five neighbours whose scatter has lambda2 / lambda1 within 1e-7 of 3, randomly rotated: the closed-form screen
    (margin 1e-5 lambda2) defers and the Jacobi sweeps decide.  Degenerate scatters: five identical points (all
    eigenvalues 0), collinear points, four identical points and one more."""
    rng = np.random.default_rng(61)
    pts, edges, near = [], [], 0
    g = 0
    while near < 40:
        b = rng.uniform(0.1, 0.3)
        eps = rng.uniform(-8e-8, 8e-8)
        a = b * np.sqrt(3.0 * (1.0 + eps))
        R = np.linalg.qr(rng.normal(size=(3, 3)))[0]
        cen = np.array([3.0 * (g % 10), 3.0 * (g // 10), 0.0]) + rng.uniform(0, 0.5, 3)
        five = cen + np.array([[a, 0, 0], [-a, 0, 0], [0, b, 0], [0, -b, 0], [0, 0, 0]]) @ R.T
        five = five.astype(F)
        ev = np_ref.knn5_gate(np.concatenate([five, np.zeros((5, 1), F)], 1), P(*cen), np.eye(4))["eig"][0]
        m = abs(ev[2] - 3 * ev[1]) / ev[2]
        if not (1e-9 < m < 1e-7):
            continue
        pts += [P(*p) for p in five]
        edges.append(P(*(cen + rng.uniform(-0.01, 0.01, 3))))
        near += 1
        g += 1
    degenerate = [np.zeros((5, 3)), np.outer(np.arange(5) * 0.1, [1.0, 0.5, 0.25]), np.array([[0, 0, 0]] * 4 + [[0.1, 0, 0]])]
    for k, d in enumerate(degenerate):
        cen = np.array([3.0 * k, -6.0, 0.0]) + 0.1
        pts += [P(*p) for p in cen + d]
        edges.append(P(*(cen + 0.05)))

    def check(c, r):
        ev = r["eig"][:40]
        m = np.abs(ev[:, 2] - 3 * ev[:, 1]) / ev[:, 2]
        assert (m < 1e-7).all() and r["decided"][:40].all() and (r["gate"][:40] & 1).all()
        assert 0 < ((r["gate"][:40] & 2) > 0).sum() < 40
        assert (r["eig"][40] == 0).all() and not r["decided"][40]
        assert r["gate"][41] == 3 and r["gate"][42] == 3
    return Case("line_gate_margin", [pts], edges, check=check)


def _received_map():
    """mapping = 1: the received map follows the window in logical order (liodom_oracle.cc:1183-1184); exact copies of
    window points in it tie with them, and the window's copy wins."""
    rng = np.random.default_rng(67)
    f0 = (np.round(rng.normal(size=(400, 4)) * [1.0, 1.0, 0.4, 0] * 64) / 64).astype(F)
    f1 = (np.round(rng.normal(size=(400, 4)) * [1.0, 1.0, 0.4, 0] * 64) / 64).astype(F)
    rec = np.concatenate([f1[:150], f0[:150], (rng.normal(size=(200, 4)) * [1.0, 1.0, 0.4, 0]).astype(F)])
    rec = rec[rng.permutation(len(rec))]
    q = (np.round(rng.normal(size=(400, 4)) * [1.0, 1.0, 0.4, 1] * 128) / 128).astype(F)
    q[:100] = f0[:100] + [0, 0, 0, 1]

    def check(c, r):
        nw = len(c.window())
        mixed = ((r["idx6"][:, :5] >= nw).any(1) & (r["idx6"][:, :5] < nw).any(1))
        assert mixed.sum() > 50 and r["tie"][:100].all()
    return Case("received_map", [f0, f1], q, received=rec, prev_frames=2, check=check)


def _window_filter():
    """filter_local_map = 1, window full: the kNN target is VoxelGrid(0.4) of the window.  Voxels whose centroids
    coincide (three copies of the last float below a voxel face average to the first float above it, the centroid of
    the next voxel's single point) and mirror-symmetric centroids."""
    rng = np.random.default_rng(71)
    frames = [[], [], []]
    edges, dup = [], 0
    k = 4
    while dup < 24:
        k += 1
        xa = F(k * 0.4)                    # the last float of voxel k - 1 (voxel index floor(x * 2.5))
        while np.floor(xa * F(2.5)) >= k:
            xa = np.nextafter(xa, F(0))
        while np.floor(np.nextafter(xa, INF) * F(2.5)) < k:
            xa = np.nextafter(xa, INF)
        xb = np.nextafter(xa, INF)         # the first float of voxel k
        y, z = F(0.25 + (k % 2)), F(0.25)   # dyadic: their averages are exact; neighbouring faces in different rows
        for n in (3, 5, 6, 7, 9, 11):
            s = F(0)
            for _ in range(n):
                s = s + xa
            if s / F(n) == xb:             # n copies of xa average to xb: two voxels with one centroid
                for j in range(n):
                    frames[j % 3].append(P(xa, y, z))
                frames[2].append(P(xb, y, z))
                edges.append(P(xb, y + 0.05, z + 0.05))
                dup += 1
                break
    for g in range(30):
        q = np.array([0.2 + 0.4 * g, 5.0, 0.2])
        for v in (np.array([0.4, 0, 0]), np.array([0, 0.4, 0]), np.array([0, 0, 0.4])):
            frames[g % 3].append(P(*(q + v)))
            frames[(g + 1) % 3].append(P(*(q - v)))
        edges.append(P(*q))
    frames = [np.array(f, np.float32).reshape(-1, 4) for f in frames]

    def check(c, r):
        t = c.target()
        assert 0 < len(t) < len(c.window())
        u, cnt = np.unique(t[:, :3], axis=0, return_counts=True)
        assert (cnt > 1).sum() >= 20, (cnt > 1).sum()
        assert r["tie"].sum() >= 40
    return Case("window_filter", frames, edges, filter_local_map=True, prev_frames=3, check=check)


SIZES = (0, 1, 31, 32, 33, 63, 65, 2047, 2048, 2049, ECAP)


def _sizes():
    """Edge counts around warp and CTA sizes and the 2048-edge k_edge_order chunks, up to the edge capacity."""
    rng = np.random.default_rng(73)
    pts = (np.round(rng.normal(size=(5000, 4)) * [2.0, 2.0, 0.5, 0] * 32) / 32).astype(F)
    pts[2500:3500] = pts[:1000]
    out = []
    for n in SIZES:
        q = (rng.normal(size=(n, 4)) * [2.0, 2.0, 0.5, 1]).astype(F)
        q[: n // 4] = pts[rng.integers(0, len(pts), n // 4)]

        def check(c, r, n=n):
            assert len(c.edges) == n and len(r["gate"]) == n
            if n >= 32:
                assert (r["gate"] & 1).mean() > 0.5 and r["tie"].any()
        pose = np.eye(4)
        pose[:3, 3] = [1 / 64, -1 / 32, 1 / 128]
        out.append(Case("sizes_%d" % n, [pts[:2500], pts[2500:]], q, pose=pose, check=check))
    return out


_CASES = None


def cases():
    global _CASES
    if _CASES is None:
        _CASES = [_cell_faces(), _proven_radius(), _gate_radius(), _fallback_only(), _ties(), _stationary(),
                  _pool_overflow(), _dense_cell(), _filter_word(), _far_aliased(), _nonfinite(), _line_gate_margin(),
                  _received_map(), _window_filter()] + _sizes()
    return _CASES


def by_name():
    return {c.name: c for c in cases()}
