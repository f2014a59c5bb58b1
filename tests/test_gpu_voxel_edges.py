"""Edge cases of the two VoxelGrid restatements on the GPU, against the oracle.

Map (map.cu): cell sizes whose half is not an integer and sizes in [1, 2) (the reference's int key
truncates toward zero, so a key's cell is not centred on it and, below 2 m, cells -1 and 0 share key
0), fine resolutions up to the 10-bit lattice, sort keys of 2 to 6 radix passes, the per-update and
per-map capacities, the pinned-window fallback of getLocalMap and its query-cell limit.

Window filter (voxelgrid.cu, filter_local_map): 1 to 4 radix passes, PCL's int32 overflow rule (the
window itself becomes the kNN target) and its end when the outlier frame leaves the window,
degenerate windows, and lanes of one context in different regimes."""
import math

import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import oracle
from liodom_b200 import api

pytestmark = pytest.mark.gpu

E_INVALID, E_CAPACITY = -1, -3
INT32_MAX = 2147483647


def _same(gm, om, T=None, cells=(2, 1)):
    gk, gc = gm.cells()
    ok, oc = om.cells()
    assert np.array_equal(gk, ok), "cell keys / creation order differ"
    assert np.array_equal(gc, oc), "per-cell counts differ"
    g, o = gm.get_map(), om.get_map()
    assert g.shape == o.shape
    assert np.array_equal(g.view(np.uint32), o.view(np.uint32)), "centroids differ bitwise"
    if T is not None:
        gl, ol = gm.get_local_map(T, *cells), om.get_local_map(T, *cells)
        assert gl.shape == ol.shape
        assert np.array_equal(gl.view(np.uint32), ol.view(np.uint32)), "local map differs"


def _raises(code, fn, *a):
    with pytest.raises(api.LiodomError) as e:
        fn(*a)
    assert "error %d:" % code in str(e.value), str(e.value)


def _pose(rotvec, t):
    T = np.eye(4)
    T[:3, :3] = Rotation.from_rotvec(rotvec).as_matrix()
    T[:3, 3] = t
    return T


# ---- Map ---------------------------------------------------------------------------------------------
def _lat_bits(xy, z, res):
    """Bits per lattice axis of k_map_update's sort key, restated from liodom_map_create."""
    extent = lambda s: 2.0 * s if s < 2.0 else s                       # below 2 m key 0 holds cells -1 and 0
    slack = lambda s: 0.0 if s / 2.0 == math.floor(s / 2.0) else 1.0   # int truncation of the key
    inv = float(np.float32(1.0) / np.float32(res))
    margin = 2 + int(inv / 16.0)
    span = math.ceil(max(extent(xy) + slack(xy), extent(z) + slack(z)) * inv) + 2 * margin + 2
    return max(1, math.ceil(math.log2(span)))


def _map_passes(xy, z, res, n_touched):
    return math.ceil((3 * _lat_bits(xy, z, res) + math.ceil(math.log2(n_touched))) / 8)


def _face_cloud(rng, xy, z, res, n_random=3000):
    """Points straddling the origin and negative cells: cell faces k*size and voxel faces m*res as float,
    one ulp either side of each, -0.0, and random points over +-3 cells."""
    f32 = np.float32
    vals = []
    for s in (xy, z):
        for k in range(-3, 4):
            vals.append(f32(k * s))
    for m in range(-40, 41):
        vals.append(f32(m * res))
    vals = np.array(vals, np.float32)
    vals = np.concatenate([vals, np.nextafter(vals, f32(-np.inf)), np.nextafter(vals, f32(np.inf)), [f32(-0.0)]])
    n = len(vals)
    pts = np.empty((3 * n, 4), np.float32)
    # every face value on every axis, the other two axes drawn from the same set
    for a in range(3):
        blk = pts[a * n:(a + 1) * n]
        blk[:, :3] = rng.choice(vals, size=(n, 3))
        blk[:, a] = vals
    pts[:, 3] = rng.random(len(pts))
    span = np.array([3 * xy, 3 * xy, 3 * z], np.float32)
    rnd = np.concatenate([rng.uniform(-span, span, size=(n_random, 3)), rng.random((n_random, 1))], 1).astype(np.float32)
    return np.concatenate([pts, rnd])


CONFIGS = [(40.0, 50.0, 0.4), (20.0, 25.0, 0.1), (25.0, 25.0, 0.1), (35.0, 35.0, 0.2), (1.0, 1.0, 0.4), (1.0, 1.0, 0.1),
           (1.5, 1.5, 0.1), (1.9, 1.9, 0.05), (40.0, 40.0, 0.04), (2.5, 7.5, 0.3)]
POSES = [np.eye(4), _pose([0.0, 0.0, 0.3], [-3.7, -0.4, -1.2]), _pose([0.02, -0.01, -1.1], [12.25, -7.5, 0.999]),
         _pose([0.3, 0.2, 2.0], [-0.5, 0.5, -0.0])]


@pytest.mark.parametrize("xy,z,res", CONFIGS)
def test_map_sizes_and_resolutions(cuda_lib, xy, z, res):
    rng = np.random.default_rng(int(xy * 100 + res * 1000))
    gm, om = api.Map(xy, z, res, max_points=1 << 20), oracle.Map(xy, z, res)
    for T in POSES:
        pts = _face_cloud(rng, xy, z, res)
        gm.update(pts, T)
        om.update(pts, T)
        _same(gm, om, T, (2, 1))
    for T in POSES:                       # truncated / negative / fractional translations of getLocalMap
        for cells in ((1, 1), (3, 2)):
            gl, ol = gm.get_local_map(T, *cells), om.get_local_map(T, *cells)
            assert np.array_equal(gl.view(np.uint32), ol.view(np.uint32)), cells
    gm.close()


def _cell_centres(xy, z, n, rng):
    """One point near the centre of n cells with distinct keys (a square grid of non-negative cells in x, y: below
    2 m the cells -1 and 0 would share key 0)."""
    side = int(math.ceil(math.sqrt(n)))
    ij = np.stack(np.meshgrid(np.arange(side), np.arange(side), indexing="ij"), -1).reshape(-1, 2)[:n]
    pts = np.zeros((n, 4), np.float32)
    pts[:, :2] = (ij + 0.5) * xy
    pts[:, 2] = 0.5 * z
    pts[:, :3] += rng.uniform(-0.2, 0.2, size=(n, 3)) * min(xy, z)
    pts[:, 3] = rng.random(n)
    return pts


RADIX_CASES = [(c, n) for c in [(1.0, 1.0, 0.4), (1.9, 1.9, 0.05), (20.0, 25.0, 0.1), (40.0, 40.0, 0.04)]
               for n in (1, 2, 256, 257, 3000)]


def test_map_radix_cases_cover_2_to_6_passes():
    assert {_map_passes(*c, n) for c, n in RADIX_CASES} == {2, 3, 4, 5, 6}


@pytest.mark.parametrize("cfg,n_touched", RADIX_CASES)
def test_map_radix_depth(cuda_lib, cfg, n_touched):
    xy, z, res = cfg
    rng = np.random.default_rng(n_touched)
    gm, om = api.Map(xy, z, res, max_points=1 << 18), oracle.Map(xy, z, res)
    base = _cell_centres(xy, z, n_touched, rng)
    for rep in range(3):                  # first creates the cells, then re-averages them with new points
        pts = np.repeat(base, 2, 0) + np.float32(0.01 * rep)
        gm.update(pts, np.eye(4))
        om.update(pts, np.eye(4))
        assert gm.size()[1] == n_touched
        _same(gm, om, np.eye(4))
    gm.close()


def test_map_full_update_and_local_map_beyond_pinned_window(cuda_lib):
    """Updates of exactly 65536 points fill one cell region with distinct voxels until getLocalMap returns more
    than the 2^19-point pinned window and takes the device gather."""
    xy, z, res = 20.0, 25.0, 0.1
    rng = np.random.default_rng(5)
    gm, om = api.Map(xy, z, res, max_points=1 << 20), oracle.Map(xy, z, res)
    nx, ny, nz = 200, 200, 250            # voxels of the cell [0, 20) x [0, 20) x [0, 25)
    vox = rng.choice(nx * ny * nz, size=9 * 65536, replace=False)
    ijk = np.stack([vox % nx, (vox // nx) % ny, vox // (nx * ny)], 1)
    pts = np.concatenate([(ijk + 0.5) * res, rng.random((len(vox), 1))], 1).astype(np.float32)
    for k in range(9):
        gm.update(pts[k * 65536:(k + 1) * 65536], np.eye(4))
        om.update(pts[k * 65536:(k + 1) * 65536], np.eye(4))
    T = _pose([0, 0, 0], [5.0, 5.0, 5.0])
    _same(gm, om, T, (2, 1))
    assert len(om.get_local_map(T, 2, 1)) > 1 << 19
    gm.close()


def _query_cells(xy, zs, cells_xy, cells_z):
    """Cells getLocalMap looks up at the origin: (2 cells_xy + 1)^2 plus the z column, whose bounds use the xy size."""
    vz = int(math.floor(0.0) * zs + zs / 2.0)
    init_z, end_z = int(vz - cells_z * xy), int(vz + cells_z * xy)
    nz, i = 0, init_z
    while i <= end_z:
        nz, i = nz + 1, int(i + zs)
    return (2 * cells_xy + 1) ** 2 + nz


def test_map_query_cell_limit(cuda_lib):
    """getLocalMap serves up to 4095 query cells; 4096 is a capacity error."""
    xy, z = 30.0, 35.0
    assert _query_cells(xy, z, 31, 73) == 4095 and _query_cells(xy, z, 31, 74) == 4096
    gm, om = api.Map(xy, z, 0.4, max_points=1 << 18), oracle.Map(xy, z, 0.4)
    rng = np.random.default_rng(7)
    pts = (rng.uniform(-2500, 2500, size=(20000, 4)) * [0.4, 0.4, 1, 0]).astype(np.float32)
    gm.update(pts, np.eye(4))
    om.update(pts, np.eye(4))
    gl, ol = gm.get_local_map(np.eye(4), 31, 73), om.get_local_map(np.eye(4), 31, 73)
    assert len(gl) > 0 and np.array_equal(gl.view(np.uint32), ol.view(np.uint32))
    _raises(E_CAPACITY, gm.get_local_map, np.eye(4), 31, 74)
    gm.close()


@pytest.mark.parametrize("xy,z,res", [(1.0, 1.0, 0.1), (1.5, 1.5, 0.1), (20.0, 25.0, 0.1)])
def test_map_local_map_key_loops(cuda_lib, xy, z, res):
    """getLocalMap's `int` translation truncation and `int += double` loops (advancing by 1 below 2 m)."""
    rng = np.random.default_rng(9)
    gm, om = api.Map(xy, z, res, max_points=1 << 18), oracle.Map(xy, z, res)
    pts = np.concatenate([rng.uniform(-8 * xy, 8 * xy, size=(20000, 3)), rng.random((20000, 1))], 1).astype(np.float32)
    gm.update(pts, np.eye(4))
    om.update(pts, np.eye(4))
    for t in ([-0.5, -0.5, -0.5], [-1.0, 0.99, -1.01], [-2.7, 3.3, -4.9], [0.49, -0.49, 0.0], [-xy, -xy, -z],
              [-1.5 * xy, 2.5 * xy, -0.5 * z]):
        T = _pose([0, 0, 0.4], t)
        for cells in ((1, 1), (2, 1), (4, 3)):
            gl, ol = gm.get_local_map(T, *cells), om.get_local_map(T, *cells)
            assert np.array_equal(gl.view(np.uint32), ol.view(np.uint32)), (t, cells)
    gm.close()


def test_map_non_finite_points_dropped(cuda_lib):
    """Non-finite points are dropped (the reference has undefined behaviour there): same as the oracle fed
    the cloud without them."""
    rng = np.random.default_rng(13)
    gm, om = api.Map(20.0, 25.0, 0.1, max_points=1 << 18), oracle.Map(20.0, 25.0, 0.1)
    for f in range(4):
        pts = (rng.normal(size=(4000, 4)) * [15, 15, 3, 1]).astype(np.float32)
        pts[f::37, 0] = np.nan
        pts[5 + f::53, 1] = np.inf
        pts[9::101, 2] = -np.inf
        T = _pose([0, 0, 0.2 * f], [-2.5 * f, 1.5, -0.3])
        gm.update(pts, T)
        om.update(pts[np.isfinite(pts[:, :3]).all(1)], T)
        _same(gm, om, T)
    gm.close()


def test_map_error_codes(cuda_lib):
    """Error codes only: the state after an error is unspecified."""
    gm = api.Map(40.0, 50.0, 0.4, max_points=1 << 18)
    _raises(E_INVALID, gm.update, np.array([[2.0 ** 21, 0, 0, 1]], np.float32), np.eye(4))
    gm.close()
    gm = api.Map(40.0, 50.0, 0.4, max_points=1 << 18)
    _raises(E_CAPACITY, gm.update, np.zeros((65537, 4), np.float32), np.eye(4))
    gm.update(_cell_centres(40.0, 50.0, 65536, np.random.default_rng(0)), np.eye(4))
    assert gm.size()[1] == 65536
    _raises(E_CAPACITY, gm.update, np.array([[0.0, 0.0, -100.0, 1.0]], np.float32), np.eye(4))   # the 65537th cell
    gm.close()


def test_map_rejects_key_extents_beyond_the_lattice(cuda_lib):
    api.Map(1.0, 1.0, 0.002).close()                      # key 0 spans 2 m: 1000 voxels
    with pytest.raises(api.LiodomError):
        api.Map(1.0, 1.0, 0.001)                          # 2000 voxels


@pytest.mark.parametrize("xy,z,res", [(20.0, 25.0, 0.1), (1.5, 1.5, 0.1)])
def test_map_long_drifting_run(cuda_lib, xy, z, res):
    """200 updates of random size and pose drifting across negative cells; bit-exact after every update."""
    rng = np.random.default_rng(int(xy * 10))
    gm, om = api.Map(xy, z, res, max_points=1 << 20), oracle.Map(xy, z, res)
    scale = np.array([3 * xy, 3 * xy, z, 1.0])
    for f in range(200):
        n = 0 if f == 50 else int(rng.integers(1, 1500))
        pts = (rng.normal(size=(n, 4)) * scale * rng.uniform(0.1, 1.0)).astype(np.float32)
        T = _pose(rng.normal(size=3) * [0.05, 0.05, 0.5], [(f - 100) * 0.37 * xy / 20, -0.13 * f * xy / 20, rng.normal() * z * 0.3])
        gm.update(pts, T)
        om.update(pts, T)
        _same(gm, om, T if f % 10 == 0 else None)
    gm.close()


# ---- window filter -----------------------------------------------------------------------------------
K = 3
CTX = dict(prev_frames=K, filter_local_map=1, scan_lines=16, scan_regions=8, edges_per_region=40, max_points=4096)
INV = np.float32(1.0) / np.float32(0.4)


def _vg_plan(window):
    """k_vg_plan restated in float32: None when the filter is off (PCL's overflow rule, or a voxel index space
    beyond int32), else the number of radix passes."""
    p = np.asarray(window, np.float32)[:, :3]
    p = p[np.isfinite(p).all(1)]
    if len(p) == 0:
        return 0
    mn, mx = p.min(0), p.max(0)
    dd = [int(np.float32((mx[a] - mn[a]) * INV)) + 1 for a in range(3)]
    div = [int(np.floor(mx[a] * INV)) - int(np.floor(mn[a] * INV)) + 1 for a in range(3)]
    if dd[0] * dd[1] * dd[2] > INT32_MAX:
        return None
    cells = div[0] * div[1] * div[2]
    if cells > INT32_MAX - 1:
        return None
    bits = 1
    while (1 << bits) <= cells:
        bits += 1
    return (bits + 7) // 8


def _cluster(rng, n, centre=(0.0, 0.0, 0.0)):
    return (rng.normal(size=(n, 4)) * [3.0, 2.0, 0.7, 1.0] + [*centre, 0.0]).astype(np.float32)


def _check_assoc(g, o, min_sel):
    ok = o["tie"] == 0
    assert np.array_equal(g["gate"][ok], o["gate"][ok])
    sel = ok & ((o["gate"] & 1) == 1)
    assert sel.sum() >= min_sel
    assert np.array_equal(g["knn_idx"][sel], o["knn_idx"][sel])
    assert np.array_equal(g["knn_d2"][sel].view(np.uint32), o["knn_d2"][sel].view(np.uint32))
    assert np.array_equal(g["eig"][sel].view(np.uint64), o["eig"][sel].view(np.uint64))


def _assoc(ctx, window, filtered, rng, lane=0, min_sel=30, centre=(0.0, 0.0, 0.0)):
    """The lane's kNN target: VoxelGrid(0.4) of the window, or the window itself when the filter is off."""
    target = oracle.voxelgrid(window, 0.4) if filtered else window
    q = (rng.normal(size=(400, 4)) * [2.0, 1.5, 0.5, 1.0] + [*centre, 0.0]).astype(np.float32)
    o = oracle.associate(q, np.eye(4), target, knn_method=0)
    g = ctx.associate(q, np.eye(4), lane=lane)
    assert g["n_map"] == len(target), (g["n_map"], len(target), len(window))
    _check_assoc(g, o, min_sel)


def _fill(ctx, frames, lane=0):
    for w in frames:
        ctx.lmap_add(w, lane=lane)
    return np.concatenate(frames)


def _window_of_passes(rng, passes):
    """K frames around a dense cluster whose bounding box (set by a few far points) needs `passes` radix passes."""
    reach = np.float32({1: (0.5, 0.5, 0.5), 2: (4.0, 4.0, 1.0), 3: (60.0, 60.0, 4.0), 4: (400.0, 400.0, 8.0)}[passes])
    frames = [_cluster(rng, 1500) for _ in range(K)]
    for fr in frames:
        fr[:, :3] = np.clip(fr[:, :3] * (0.05 if passes == 1 else 1.0), -reach, reach)
    frames[1][:2, :3] = [-reach, reach]
    return frames


@pytest.mark.parametrize("passes", [1, 2, 3, 4])
def test_window_filter_radix_passes(cuda_lib, passes):
    rng = np.random.default_rng(passes)
    frames = _window_of_passes(rng, passes)
    window = np.concatenate(frames)
    assert _vg_plan(window) == passes
    ctx = api.Context(**CTX)
    _fill(ctx, frames)
    _assoc(ctx, window, True, rng, min_sel=0 if passes == 1 else 30)
    ctx.close()


def test_window_filter_overflow_rule_and_resume(cuda_lib):
    """An outlier frame makes PCL's dx*dy*dz exceed INT32_MAX: the window itself is the target until the frame
    leaves the window, then the filter resumes."""
    rng = np.random.default_rng(17)
    ctx = api.Context(**CTX)
    frames = []
    for f in range(8):
        w = _cluster(rng, 1200)
        if f == 2:
            w[7, :3] = [900.0, -900.0, 700.0]
        ctx.lmap_add(w)
        frames = (frames + [w])[-K:]
        window = np.concatenate(frames)
        full = len(frames) == K
        outlier = 2 <= f < 2 + K
        assert (_vg_plan(window) is None) == outlier
        _assoc(ctx, window, full and not outlier, rng)
    ctx.close()


BOX_CENTRE = (8.0, 8.0, 8.0)


def _box_window(rng, lo, hi):
    """A dense cluster at BOX_CENTRE plus two points fixing the bounding box to [lo, hi]."""
    frames = [_cluster(rng, 1000, BOX_CENTRE) for _ in range(K)]
    for fr in frames:
        fr[:, :3] = np.clip(fr[:, :3], lo, hi)
    frames[0][0, :3] = lo
    frames[0][1, :3] = hi
    return frames


@pytest.mark.parametrize("zr,filtered", [(858.5, True), (858.9, False)])
def test_window_filter_overflow_boundary(cuda_lib, zr, filtered):
    """dx = dy = 1000 and dz = 2147 (product 2.147e9, just below INT32_MAX: filter on, 4 passes) or 2148 (just
    above: filter off); the box starts on a voxel face, so PCL's div_b equals dx, dy, dz."""
    rng = np.random.default_rng(19)
    lo, hi = np.float32([0.0, 0.0, 0.0]), np.float32([399.7, 399.7, zr])
    frames = _box_window(rng, lo, hi)
    window = np.concatenate(frames)
    dd = [int(np.float32((hi[a] - lo[a]) * INV)) + 1 for a in range(3)]
    assert dd[:2] == [1000, 1000] and dd[2] == (2147 if filtered else 2148)
    assert _vg_plan(window) == (4 if filtered else None)
    ctx = api.Context(**CTX)
    _fill(ctx, frames)
    _assoc(ctx, window, filtered, rng, centre=BOX_CENTRE)
    ctx.close()


def test_window_filter_div_b_overflow_is_unfiltered(cuda_lib):
    """PCL's own check passes (dx*dy*dz <= INT32_MAX) but its voxel index space div_b does not fit an int, where
    PCL's index arithmetic overflows: the filter is off, the window itself is the target."""
    rng = np.random.default_rng(23)
    lo = np.float32([0.3, 0.3, 0.3])
    hi = lo + np.float32([399.7, 399.7, 858.5])
    frames = _box_window(rng, lo, hi)
    window = np.concatenate(frames)
    p = window[:, :3]
    dd = [int(np.float32((p[:, a].max() - p[:, a].min()) * INV)) + 1 for a in range(3)]
    div = [int(np.floor(p[:, a].max() * INV)) - int(np.floor(p[:, a].min() * INV)) + 1 for a in range(3)]
    assert dd[0] * dd[1] * dd[2] <= INT32_MAX < div[0] * div[1] * div[2]
    assert _vg_plan(window) is None
    ctx = api.Context(**CTX)
    _fill(ctx, frames)
    _assoc(ctx, window, False, rng, centre=BOX_CENTRE)
    ctx.close()


def test_window_filter_degenerate_windows(cuda_lib):
    rng = np.random.default_rng(29)
    nan = np.full((50, 4), np.nan, np.float32)
    # every point non-finite: empty target, every gate fails
    ctx = api.Context(**CTX)
    window = _fill(ctx, [nan, nan.copy(), nan.copy()])
    g = ctx.associate(_cluster(rng, 100), np.eye(4))
    assert g["n_map"] == 0 and len(oracle.voxelgrid(window, 0.4)) == 0
    assert not (g["gate"] & 1).any()
    ctx.close()
    # one finite point
    ctx = api.Context(**CTX)
    one = nan.copy()
    one[17] = [0.3, -0.2, 0.1, 0.5]
    window = _fill(ctx, [nan, one, nan.copy()])
    assert _vg_plan(window) == 1
    _assoc(ctx, window, True, rng, min_sel=0)
    ctx.close()
    # the bounding box's lower edge at -0.0 (a +0.0 in another frame)
    ctx = api.Context(**CTX)
    frames = [np.abs(_cluster(rng, 800)) for _ in range(K)]
    frames[1][0, :3] = [-0.0, -0.0, -0.0]
    frames[2][0, :3] = [0.0, 0.0, 0.0]
    window = _fill(ctx, frames)
    _assoc(ctx, window, True, rng, centre=(2.0, 2.0, 0.5))
    ctx.close()
    # points exactly on voxel faces, and one ulp either side
    ctx = api.Context(**CTX)
    faces = (np.arange(-10, 11) * np.float32(0.4)).astype(np.float32)
    faces = np.concatenate([faces, np.nextafter(faces, np.float32(-1)), np.nextafter(faces, np.float32(1))])
    frames = []
    for _ in range(K):
        w = rng.choice(faces, size=(3 * len(faces), 4)).astype(np.float32)
        w[:, 3] = rng.random(len(w))
        frames.append(np.concatenate([w, _cluster(rng, 300)]))
    window = _fill(ctx, frames)
    _assoc(ctx, window, True, rng)
    ctx.close()


def test_window_filter_lanes_in_different_regimes(cuda_lib):
    """One context, four lanes: overflowed (unfiltered), 1-pass, 4-pass and 2-pass windows.  Each lane must match
    its own oracle window, so no per-lane plan state may bleed between lanes."""
    rng = np.random.default_rng(31)
    over = [_cluster(rng, 1200) for _ in range(K)]
    over[1][3, :3] = [-1200.0, 800.0, 600.0]
    windows = [over, _window_of_passes(rng, 1), _window_of_passes(rng, 4), _window_of_passes(rng, 2)]
    assert [_vg_plan(np.concatenate(w)) for w in windows] == [None, 1, 4, 2]
    ctx = api.Context(batch=len(windows), **CTX)
    for k, w in enumerate(windows):
        _fill(ctx, w, lane=k)
    for k, w in enumerate(windows):
        _assoc(ctx, np.concatenate(w), k != 0, rng, lane=k, min_sel=0 if k == 1 else 30)
    ctx.close()
