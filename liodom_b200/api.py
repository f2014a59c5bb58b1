"""ctypes binding of the liodom_b200 C ABI (include/liodom_b200.h).

Thin plumbing used by tests and bench.py; the product is the CUDA library behind it.
Loading fails loudly when libliodom_b200.so has not been built — there is no fallback.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libliodom_b200.so")
_vp = ctypes.c_void_p


class Params(ctypes.Structure):
    """liodom_params: numeric liodom::Params fields (reference defaults) + capacities."""
    _fields_ = [("min_range", ctypes.c_double), ("max_range", ctypes.c_double), ("lidar_type", ctypes.c_int),
                ("scan_lines", ctypes.c_int), ("scan_regions", ctypes.c_int), ("edges_per_region", ctypes.c_int),
                ("prev_frames", ctypes.c_int), ("filter_local_map", ctypes.c_int), ("mapping", ctypes.c_int),
                ("max_points", ctypes.c_int), ("max_received_map", ctypes.c_int), ("use_imu", ctypes.c_int)]


class CloudLayout(ctypes.Structure):
    """liodom_cloud_layout: where x, y, z, intensity (FLOAT32) sit in a sensor_msgs/PointCloud2 point."""
    _fields_ = [("point_step", ctypes.c_int), ("row_step", ctypes.c_int), ("off_x", ctypes.c_int), ("off_y", ctypes.c_int),
                ("off_z", ctypes.c_int), ("off_intensity", ctypes.c_int), ("is_bigendian", ctypes.c_int)]


class SolveSummary(ctypes.Structure):
    _fields_ = [("iterations", ctypes.c_int), ("successful_steps", ctypes.c_int), ("termination", ctypes.c_int),
                ("num_residual_blocks", ctypes.c_int), ("cost_evals", ctypes.c_int), ("jac_evals", ctypes.c_int),
                ("initial_cost", ctypes.c_double), ("final_cost", ctypes.c_double)]


class FrameDiag(ctypes.Structure):
    _fields_ = [("n_edges", ctypes.c_int), ("n_map", ctypes.c_int * 2), ("n_matches", ctypes.c_int * 2),
                ("solve", SolveSummary * 2), ("pred_pose", ctypes.c_double * 16)]


NUM_STAGES = 7
STAGE_NAMES = ("split", "extract", "associate0", "solve0", "associate1", "solve1", "window+hash")


class LiodomError(RuntimeError):
    pass


_lib = None


def load():
    """Load the CUDA library; raises if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise LiodomError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(liodom_b200 has no CPU fallback)" % SO_PATH)
        L = ctypes.CDLL(SO_PATH)
        L.liodom_last_error.restype = ctypes.c_char_p
        L.liodom_last_error.argtypes = [_vp]
        L.liodom_stream.restype = _vp
        L.liodom_launch_count.restype = ctypes.c_longlong
        L.liodom_launch_count.argtypes = [_vp]
        L.liodom_stream.argtypes = [_vp]
        if hasattr(L, "liodom_map_create"):
            L.liodom_map_last_error.restype = ctypes.c_char_p
            L.liodom_map_last_error.argtypes = [_vp]
            L.liodom_map_create.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int,
                                            ctypes.c_int, ctypes.POINTER(_vp)]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def shard_unique_id():
    """128-byte NCCL unique id for the point-sharded mode (call on one rank, broadcast to the others)."""
    buf = ctypes.create_string_buffer(128)
    rc = load().liodom_shard_unique_id(buf)
    if rc != 0:
        raise LiodomError("liodom_shard_unique_id failed (%d): %s" % (rc, load().liodom_last_error(None).decode()))
    return buf.raw


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] >= 3
    return a


def _f4(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] == 4
    return a


def make_params(**kw):
    p = Params()
    load().liodom_default_params(ctypes.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


class Context:
    """One liodom_ctx: `batch` independent sequences on one device/stream."""

    def __init__(self, params=None, batch=1, device=0, **kw):
        self.lib = load()
        self.params = params if params is not None else make_params(**kw)
        self.batch = batch
        h = _vp()
        rc = self.lib.liodom_ctx_create(ctypes.byref(self.params), batch, device, ctypes.byref(h))
        if rc != 0:
            raise LiodomError("liodom_ctx_create failed (%d): %s" % (rc, self.lib.liodom_last_error(None).decode()))
        self.h = h
        self.max_edges = self.lib.liodom_max_edges(self.h)

    def close(self):
        if getattr(self, "h", None):
            self.lib.liodom_ctx_destroy(self.h)
            self.h = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise LiodomError("liodom error %d: %s" % (rc, self.lib.liodom_last_error(self.h).decode()))

    # ---- FeatureExtractor --------------------------------------------------------------
    def split(self, pts, lane=0, width=0, height=0):
        pts = _pts(pts)
        n = len(pts)
        L = self.params.scan_lines
        ring = np.empty(n, np.int32)
        rings = np.empty((n, 4), np.float32)
        off = np.empty(L + 1, np.int32)
        src = np.empty(n, np.int32)
        nv = ctypes.c_int()
        na = ctypes.c_int()
        self._ck(self.lib.liodom_split(self.h, lane, _p(pts), n, pts.shape[1] * 4, width, height, _p(ring), _p(rings),
                                       _p(off), _p(src), ctypes.byref(nv), ctypes.byref(na)))
        return dict(ring_of_point=ring, rings=rings[:nv.value].copy(), offsets=off, src_index=src[:nv.value].copy(),
                    n_valid=nv.value, n_ambiguous=na.value)

    def extract(self, pts, lane=0, width=0, height=0, debug=False):
        pts = _pts(pts)
        n = len(pts)
        edges = np.empty((self.max_edges, 4), np.float32)
        ne = ctypes.c_int()
        er = ei = keys = None
        if debug:
            er = np.empty(self.max_edges, np.int32)
            ei = np.empty(self.max_edges, np.int32)
            keys = np.full(max(n, 1), np.nan, np.float64)
        self._ck(self.lib.liodom_extract(self.h, lane, _p(pts), n, pts.shape[1] * 4, width, height, _p(edges),
                                         ctypes.byref(ne), _p(er), _p(ei), _p(keys)))
        e = ne.value
        if not debug:
            return edges[:e].copy()
        return dict(edges=edges[:e].copy(), ring=er[:e].copy(), idx=ei[:e].copy(), keys=keys)

    def extract_layout(self, data, n, layout, lane=0, width=0, height=0):
        """liodom_extract on a raw PointCloud2 blob (uint8 array); -> dict(edges, ring, idx)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        edges = np.empty((self.max_edges, 4), np.float32)
        er = np.empty(self.max_edges, np.int32)
        ei = np.empty(self.max_edges, np.int32)
        ne = ctypes.c_int()
        self._ck(self.lib.liodom_extract_layout(self.h, lane, _p(data), n, ctypes.byref(layout), width, height, _p(edges),
                                                ctypes.byref(ne), _p(er), _p(ei)))
        e = ne.value
        return dict(edges=edges[:e].copy(), ring=er[:e].copy(), idx=ei[:e].copy())

    def scan_batch_layout(self, blobs, counts, layout, width=0, height=0):
        """blobs: list of `batch` uint8 host arrays holding raw PointCloud2 data."""
        assert len(blobs) == self.batch
        arrs = [np.ascontiguousarray(b, dtype=np.uint8) for b in blobs]
        ptrs = (_vp * self.batch)(*[a.ctypes.data for a in arrs])
        ns = (ctypes.c_int * self.batch)(*counts)
        self._keep = arrs
        self._ck(self.lib.liodom_scan_batch_layout(self.h, ptrs, ns, ctypes.byref(layout), width, height, 0))

    # ---- LocalMapManager -----------------------------------------------------------------
    def lmap_add(self, pts, lane=0):
        pts = _f4(pts)
        self._ck(self.lib.liodom_lmap_add(self.h, lane, _p(pts), len(pts)))

    def lmap_get(self, lane=0):
        n = ctypes.c_int()
        f = ctypes.c_int()
        self._ck(self.lib.liodom_lmap_get(self.h, lane, None, 0, ctypes.byref(n), ctypes.byref(f)))
        out = np.empty((n.value, 4), np.float32)
        if n.value:
            self._ck(self.lib.liodom_lmap_get(self.h, lane, _p(out), n.value, ctypes.byref(n), ctypes.byref(f)))
        return out, f.value

    def lmap_set_max_frames(self, k, lane=0):
        self._ck(self.lib.liodom_lmap_set_max_frames(self.h, lane, int(k)))

    def lmap_clear(self, lane=0):
        self._ck(self.lib.liodom_lmap_clear(self.h, lane))

    def set_received_map(self, pts, lane=0):
        pts = _f4(pts)
        self._ck(self.lib.liodom_set_received_map(self.h, lane, _p(pts), len(pts)))

    def set_received_map_from(self, gmap, pose, cells_xy=2, cells_z=1, lane=0):
        """Map::getLocalMap -> SharedData::setLocalMap entirely on the device."""
        buf = _vp()
        cap = ctypes.c_int()
        self._ck(self.lib.liodom_received_map_buffer(self.h, lane, ctypes.byref(buf), ctypes.byref(cap)))
        T = np.ascontiguousarray(pose, dtype=np.float64).reshape(16)
        n = ctypes.c_int()
        gmap._ck(self.lib.liodom_map_get_local_device(gmap.h, _p(T), cells_xy, cells_z, buf, cap.value, ctypes.byref(n)))
        self._ck(self.lib.liodom_commit_received_map(self.h, lane, n.value))
        return n.value

    # ---- LaserOdometer --------------------------------------------------------------------
    def reset(self, lane=0):
        self._ck(self.lib.liodom_odom_reset(self.h, lane))

    def set_pose(self, odom, prev_odom, lane=0):
        o = np.ascontiguousarray(odom, dtype=np.float64).reshape(16)
        q = np.ascontiguousarray(prev_odom, dtype=np.float64).reshape(16)
        self._ck(self.lib.liodom_odom_set_pose(self.h, lane, _p(o), _p(q)))

    def set_imu(self, q_xyzw, lane=0):
        q = np.ascontiguousarray(q_xyzw, dtype=np.float64)
        self._ck(self.lib.liodom_odom_set_imu(self.h, lane, _p(q)))

    def set_laser_to_base(self, T, lane=0):
        T = np.ascontiguousarray(T, dtype=np.float64)
        self._ck(self.lib.liodom_odom_set_laser_to_base(self.h, lane, _p(T)))

    def get_pose(self, lane=0):
        o = np.empty(16)
        q = np.empty(16)
        self._ck(self.lib.liodom_odom_get_pose(self.h, lane, _p(o), _p(q)))
        return o.reshape(4, 4), q.reshape(4, 4)

    def associate(self, edges, pose, lane=0):
        edges = _f4(edges)
        E = len(edges)
        T = np.ascontiguousarray(pose, dtype=np.float64).reshape(16)
        out = dict(knn_idx=np.empty((E, 5), np.int32), knn_d2=np.empty((E, 5), np.float32), gate=np.empty(E, np.uint8),
                   eig=np.empty((E, 3), np.float64), q_world=np.empty((E, 4), np.float32))
        nm = ctypes.c_int()
        self._ck(self.lib.liodom_associate(self.h, lane, _p(edges), E, _p(T), _p(out["knn_idx"]), _p(out["knn_d2"]),
                                           _p(out["gate"]), _p(out["eig"]), _p(out["q_world"]), ctypes.byref(nm)))
        out["n_map"] = nm.value
        return out

    def solve(self, cab, q, t, lane=0):
        cab = np.ascontiguousarray(cab, dtype=np.float64).reshape(-1, 9)
        q = np.array(q, dtype=np.float64)
        t = np.array(t, dtype=np.float64)
        s = SolveSummary()
        self._ck(self.lib.liodom_solve(self.h, lane, _p(cab), len(cab), _p(q), _p(t), ctypes.byref(s)))
        return q, t, s

    def register(self, edges, lane=0):
        edges = _f4(edges)
        pose = np.empty(16)
        d = FrameDiag()
        self._ck(self.lib.liodom_register(self.h, lane, _p(edges), len(edges), _p(pose), ctypes.byref(d)))
        return pose.reshape(4, 4), d

    # ---- batched whole path ---------------------------------------------------------------
    def scan_batch(self, scans, width=0, height=0):
        """scans: list of `batch` float32 host arrays [n,4] (or [n,8] PCL layout)."""
        assert len(scans) == self.batch
        arrs = [_pts(s) for s in scans]
        stride = arrs[0].shape[1] * 4
        ptrs = (_vp * self.batch)(*[a.ctypes.data for a in arrs])
        ns = (ctypes.c_int * self.batch)(*[len(a) for a in arrs])
        self._keep = arrs  # keep alive until results()
        self._ck(self.lib.liodom_scan_batch(self.h, ptrs, ns, stride, width, height, 0))

    def scan_batch_ptrs(self, ptrs, counts, stride_bytes, width=0, height=0, on_device=True):
        """ptrs: integer addresses (device when on_device, else pinned/pageable host)."""
        p = (_vp * self.batch)(*ptrs)
        ns = (ctypes.c_int * self.batch)(*counts)
        self._ck(self.lib.liodom_scan_batch(self.h, p, ns, stride_bytes, width, height, 1 if on_device else 0))

    def scan_batch_layout_ptrs(self, ptrs, counts, layout, width=0, height=0, on_device=False):
        """liodom_scan_batch_layout with integer addresses (pinned host or device memory)."""
        p = (_vp * self.batch)(*ptrs)
        ns = (ctypes.c_int * self.batch)(*counts)
        self._ck(self.lib.liodom_scan_batch_layout(self.h, p, ns, ctypes.byref(layout), width, height, 1 if on_device else 0))

    def scan_lanes(self, lanes, scans, width=0, height=0):
        """Step only lanes[i] with the host scan scans[i] (float32 [n,4] or [n,8]); every other lane stays as it was."""
        assert len(lanes) == len(scans)
        arrs = [_pts(s) for s in scans]
        stride = arrs[0].shape[1] * 4 if arrs else 16
        self._keep = arrs  # keep alive until results()
        self._scan_lanes(lanes, [a.ctypes.data for a in arrs], [len(a) for a in arrs], stride, width, height, False)

    def scan_lanes_ptrs(self, lanes, ptrs, counts, stride_bytes, width=0, height=0, on_device=True):
        """scan_lanes with integer addresses (device when on_device, else pinned/pageable host)."""
        self._scan_lanes(lanes, ptrs, counts, stride_bytes, width, height, on_device)

    def scan_lanes_layout(self, lanes, blobs, counts, layout, width=0, height=0):
        """liodom_scan_lanes_layout: blobs[i] is a uint8 host array of raw PointCloud2 data for lanes[i]."""
        assert len(lanes) == len(blobs) == len(counts)
        arrs = [np.ascontiguousarray(b, dtype=np.uint8) for b in blobs]
        k = len(arrs)
        self._keep = arrs
        self._ck(self.lib.liodom_scan_lanes_layout(self.h, (ctypes.c_int32 * k)(*lanes), k, (_vp * k)(*[a.ctypes.data for a in arrs]),
                                                   (ctypes.c_int * k)(*counts), ctypes.byref(layout), width, height, 0))

    def _scan_lanes(self, lanes, ptrs, counts, stride_bytes, width, height, on_device):
        k = len(lanes)
        assert len(ptrs) == k and len(counts) == k
        self._ck(self.lib.liodom_scan_lanes(self.h, (ctypes.c_int32 * k)(*lanes), k, (_vp * k)(*ptrs), (ctypes.c_int * k)(*counts),
                                            stride_bytes, width, height, 1 if on_device else 0))

    def results(self, age=0):
        """Poses [batch,4,4] and edge counts of the last enqueued scan (age 0) or the one before (age 1).

        After a partial step (scan_lanes) a lane that was not stepped has n_edges == -1; its pose row is its last
        reported pose (zeros if it was never stepped)."""
        poses = np.empty((self.batch, 16))
        ne = np.empty(self.batch, np.int32)
        self._ck(self.lib.liodom_scan_results_of(self.h, age, _p(poses), _p(ne)))
        if age == 0:
            self._keep = None
        return poses.reshape(-1, 4, 4), ne

    def scan_diag(self, lane=0):
        d = FrameDiag()
        self._ck(self.lib.liodom_scan_diag(self.h, lane, ctypes.byref(d)))
        return d

    def scan_edges(self, lane=0):
        out = np.empty((self.max_edges, 4), np.float32)
        n = ctypes.c_int()
        self._ck(self.lib.liodom_scan_edges(self.h, lane, _p(out), self.max_edges, ctypes.byref(n)))
        return out[:n.value].copy()

    def sync(self):
        self._ck(self.lib.liodom_sync(self.h))

    def shard_init(self, rank, world, unique_id):
        """Join the point-sharded group (batch-1 contexts, one per GPU); unique_id: 128 bytes."""
        buf = ctypes.create_string_buffer(bytes(unique_id), 128)
        self._ck(self.lib.liodom_shard_init(self.h, int(rank), int(world), buf))

    @property
    def stream(self):
        """cudaStream_t (integer address) the context enqueues on."""
        return self.lib.liodom_stream(self.h)

    def stage_timing(self, enable=True):
        self._ck(self.lib.liodom_stage_timing(self.h, 1 if enable else 0))

    def stage_times(self):
        """-> (ms per stage summed over the timed scan_batch calls [NUM_STAGES], number of calls)."""
        ms = np.zeros(NUM_STAGES)
        n = ctypes.c_int()
        self._ck(self.lib.liodom_stage_times(self.h, _p(ms), ctypes.byref(n)))
        return ms, n.value

    @property
    def launch_count(self):
        return self.lib.liodom_launch_count(self.h)


class Map:
    """liodom::Map on the GPU (src/map.cc, include/liodom/map.h:94-116)."""

    def __init__(self, voxel_xysize=40.0, voxel_zsize=50.0, resolution=0.4, device=0, max_points=1 << 22):
        self.lib = load()
        h = _vp()
        rc = self.lib.liodom_map_create(voxel_xysize, voxel_zsize, resolution, device, max_points, ctypes.byref(h))
        if rc != 0:
            raise LiodomError("liodom_map_create failed (%d): %s" % (rc, self.lib.liodom_map_last_error(None).decode()))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.liodom_map_destroy(self.h)
            self.h = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise LiodomError("liodom map error %d: %s" % (rc, self.lib.liodom_map_last_error(self.h).decode()))

    def update(self, pts, pose):
        pts = _f4(pts)
        T = np.ascontiguousarray(pose, dtype=np.float64).reshape(16)
        self._ck(self.lib.liodom_map_update(self.h, _p(pts), len(pts), _p(T)))

    def size(self):
        n = ctypes.c_int()
        c = ctypes.c_int()
        self._ck(self.lib.liodom_map_size(self.h, ctypes.byref(n), ctypes.byref(c)))
        return n.value, c.value

    def get_map(self):
        n, _ = self.size()
        out = np.empty((n, 4), np.float32)
        m = ctypes.c_int()
        self._ck(self.lib.liodom_map_get(self.h, _p(out), n, ctypes.byref(m)))
        return out[:m.value]

    def get_local_map(self, pose, cells_xy=2, cells_z=1):
        T = np.ascontiguousarray(pose, dtype=np.float64).reshape(16)
        n = ctypes.c_int()
        self._ck(self.lib.liodom_map_get_local(self.h, _p(T), cells_xy, cells_z, None, 0, ctypes.byref(n)))
        out = np.empty((n.value, 4), np.float32)
        if n.value:
            self._ck(self.lib.liodom_map_get_local(self.h, _p(T), cells_xy, cells_z, _p(out), n.value, ctypes.byref(n)))
        return out

    def cells(self):
        _, nc = self.size()
        keys = np.empty((nc, 3), np.int32)
        counts = np.empty(nc, np.int32)
        m = ctypes.c_int()
        self._ck(self.lib.liodom_map_cells(self.h, _p(keys), _p(counts), nc, ctypes.byref(m)))
        return keys[:m.value], counts[:m.value]
