"""GPU parity against the REFERENCE'S OWN object code (oracle/_ref/libliodom_ref.so: the reference's sources
compiled unmodified against oracle/refshim/; on the GPU box the prebuilt library travels with the repo).
Edges bit-exact; poses within 1e-4 m / 1e-5 rad; Map cell keys / creation order / counts exact."""
import numpy as np
import pytest

from oracle import ref
from liodom_b200 import api
from conftest import get_sequence, pose_err

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not ref.available(), reason="needs the upstream liodom sources (LIODOM_REFERENCE_ROOT) or a prebuilt oracle/_ref")]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("name,sensor,rkw,gkw", [
    ("c1", "hdl64", dict(prev_frames=15), dict(prev_frames=15, max_points=131072)),
    ("c1_firing", "hdl64_firing", dict(prev_frames=15), dict(prev_frames=15, max_points=131072)),
    ("c3", "hdl64", dict(scan_regions=16, edges_per_region=20, prev_frames=20), dict(scan_regions=16, edges_per_region=20, prev_frames=20, max_points=131072)),
    ("c2", "os1_128", dict(lidar_type=1, scan_lines=128, prev_frames=15), dict(lidar_type=1, scan_lines=128, prev_frames=15, max_points=262144)),
])
def test_extract_vs_reference_object_code(cuda_lib, name, sensor, rkw, gkw):
    """FeatureExtractor::operator() of the reference (src/feature_extractor.cc:42-82) vs liodom_extract."""
    from liodom_b200 import synth
    w, h = synth.sensor_shape(sensor) if sensor == "os1_128" else (0, 0)
    ref.set_params(**rkw)
    fe = ref.FeatureExtractor()
    ctx = api.Context(**gkw)
    for s in get_sequence(sensor, 1002, 2)[0]:
        r = fe.process(s, w, h)
        g = ctx.extract(s, width=w, height=h)
        assert len(r) > 3000 and np.array_equal(_bits(g), _bits(r)), name
    ctx.close()


@pytest.mark.parametrize("sensor,nframes,prev", [("hdl64", 8, 15), ("hdl64_small", 16, 5)])
def test_whole_path_vs_reference_node_pipeline(cuda_lib, sensor, nframes, prev):
    """lidarClb -> FeatureExtractor -> LaserOdometer of the reference (src/liodom_node.cc:40-91) vs liodom_scan_batch."""
    scans, _ = get_sequence(sensor, 1000, nframes)
    ref.set_params(prev_frames=prev)
    rposes, rne = ref.run_sequence(scans)
    ctx = api.Context(prev_frames=prev, max_points=131072)
    for f, s in enumerate(scans):
        ctx.scan_batch([s])
        p, ne = ctx.results()
        assert ne[0] == rne[f]
        dt, dr = pose_err(p[0], rposes[f])
        assert dt < 1e-4 and dr < 1e-5, (f, dt, dr)
    ctx.close()


def test_map_vs_reference_object_code(cuda_lib):
    """Map::updateMap / getLocalMap of the reference (src/map.cc:90-189) vs liodom_map_*: C4-style replay."""
    import oracle
    op = oracle.make_params()
    ref.set_params()
    scans, gt = get_sequence("hdl64_small", 1000, 20)
    gm, rm = api.Map(20.0, 25.0, 0.4, max_points=1 << 19), ref.Map(20.0, 25.0, 0.4)
    for f, s in enumerate(scans):
        edges = oracle.extract_scan(op, s)[0]
        T = np.linalg.inv(gt[0]) @ gt[f]
        gm.update(edges, T)
        rm.update(edges, T)
        gl, rl = gm.get_local_map(T, 2, 1), rm.get_local_map(T, 2, 1)
        # in-voxel accumulation order: PCL sorts unstably, the GPU (like the oracle) accumulates in input order
        assert gl.shape == rl.shape and np.allclose(gl, rl, rtol=0, atol=2e-5), f
    (gk, gc), (rk, rc) = gm.cells(), rm.cells()
    assert np.array_equal(gk, rk) and np.array_equal(gc, rc)
    gm.close()
