"""The oracle's VoxelGrid and Map against the NumPy restatements in np_ref, at the edges the GPU tests
in test_gpu_voxel_edges.py rely on: non-finite points, PCL's int32 overflow rule, points on voxel and
cell faces, cell sizes whose half is not an integer, sizes in [1, 2) and fine resolutions."""
import numpy as np
import pytest

import np_ref
import oracle


def _faces(rng, sizes, res, n_random, reach):
    """Cell faces k*size and voxel faces m*res as float, one ulp either side, -0.0, plus random points."""
    vals = [np.float32(k * s) for s in sizes for k in range(-2, 3)] + [np.float32(m * res) for m in range(-12, 13)]
    vals = np.array(vals, np.float32)
    vals = np.concatenate([vals, np.nextafter(vals, np.float32(-np.inf)), np.nextafter(vals, np.float32(np.inf)),
                           [np.float32(-0.0)]])
    face = rng.choice(vals, size=(3 * len(vals), 3))
    rnd = rng.uniform(-reach, reach, size=(n_random, 3))
    xyz = np.concatenate([face, rnd]).astype(np.float32)
    return np.concatenate([xyz, rng.random((len(xyz), 1), np.float32)], 1)


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("leaf", [0.4, 0.1, 0.3, 0.05])
def test_voxelgrid_faces_and_non_finite(leaf):
    rng = np.random.default_rng(int(leaf * 100))
    pts = _faces(rng, (1.0, 2.5), leaf, 1500, 3.0)
    pts[::41, 0] = np.nan
    pts[7::53, 2] = np.inf
    pts[11::67, 1] = -np.inf
    o, n = oracle.voxelgrid(pts, leaf), np_ref.voxelgrid(pts, leaf)
    assert 0 < len(o) < len(pts)
    assert _bits_equal(o, n)


def test_voxelgrid_degenerate_inputs():
    nan = np.full((20, 4), np.nan, np.float32)
    assert len(oracle.voxelgrid(nan, 0.4)) == 0 and len(np_ref.voxelgrid(nan, 0.4)) == 0
    one = nan.copy()
    one[5] = [0.3, -0.2, 0.1, 0.5]
    assert _bits_equal(oracle.voxelgrid(one, 0.4), one[5:6]) and _bits_equal(np_ref.voxelgrid(one, 0.4), one[5:6])
    zero = np.array([[-0.0, -0.0, -0.0, 1.0], [0.0, 0.0, 0.0, 3.0], [0.39, 0.0, 0.0, 1.0], [0.4, 0.4, 0.4, 1.0]], np.float32)
    assert _bits_equal(oracle.voxelgrid(zero, 0.4), np_ref.voxelgrid(zero, 0.4))


@pytest.mark.parametrize("zr,overflow", [(858.5, False), (858.9, True)])
def test_voxelgrid_int32_overflow_rule(zr, overflow):
    """dx = dy = 1000 and dz = 2147 (below INT32_MAX) or 2148 (above: the input is returned unchanged, non-finite
    points included)."""
    rng = np.random.default_rng(3)
    pts = (rng.normal(size=(400, 4)) * [2, 2, 2, 1] + [8, 8, 8, 0]).astype(np.float32)
    pts[:, :3] = np.clip(pts[:, :3], 0.0, 300.0)
    pts[0, :3] = 0.0
    pts[1, :3] = [399.7, 399.7, zr]
    pts[2, 0] = np.nan
    o, n = oracle.voxelgrid(pts, 0.4), np_ref.voxelgrid(pts, 0.4)
    assert _bits_equal(o, n)
    assert (len(o) == len(pts)) == overflow
    if overflow:
        assert _bits_equal(o, pts)


def _same_map(om, nm):
    ok, oc = om.cells()
    assert np.array_equal(ok, nm.keys()), "cell keys / creation order differ"
    assert np.array_equal(oc, nm.counts())
    assert _bits_equal(om.get_map(), nm.get_map())


@pytest.mark.parametrize("xy,z,res", [(20.0, 25.0, 0.1), (25.0, 25.0, 0.4), (35.0, 35.0, 0.2), (1.0, 1.0, 0.1),
                                      (1.5, 1.5, 0.1), (1.9, 1.9, 0.05), (2.5, 7.5, 0.3)])
def test_map_matches_numpy(xy, z, res):
    rng = np.random.default_rng(int(xy * 10 + res * 100))
    om, nm = oracle.Map(xy, z, res), np_ref.Map(xy, z, res)
    poses = [np.eye(4), np.array([[0.0, -1, 0, -0.5], [1, 0, 0, -3.25], [0, 0, 1, -0.75], [0, 0, 0, 1]])]
    for T in poses * 2:
        pts = _faces(rng, (xy, z), res, 300, 2.5 * max(xy, z))
        om.update(pts, T)
        nm.update(pts, T)
        _same_map(om, nm)


def test_map_key_zero_spans_two_cells():
    """Below 2 m the cells -1 and 0 both truncate to key 0: a cloud in +-3 m at 1 m gives 5 keys per axis."""
    g = (np.arange(-3.0, 3.0, 0.5) + 0.25).astype(np.float32)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    pts = np.concatenate([xyz, np.ones((len(xyz), 1), np.float32)], 1)
    om, nm = oracle.Map(1.0, 1.0, 0.1), np_ref.Map(1.0, 1.0, 0.1)
    om.update(pts, np.eye(4))
    nm.update(pts, np.eye(4))
    keys, _ = om.cells()
    assert len(keys) == 125 and sorted(set(keys[:, 0])) == [-2, -1, 0, 1, 2]
    _same_map(om, nm)
