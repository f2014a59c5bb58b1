"""Step orchestration: the kernel launches each entry point reports, and stage-timed steps against untimed ones.

Launch counts on the C1 shape (64 lines x 8 regions x 11 = 5632 edge slots, incremental hash, no window filter):
split 3, extract 2, predict 2, solve 1, window update 1 + hash build 4, and association 1 or 2.  Association runs
16 threads per edge up to 5632 edges in flight per lane group, 8 up to 11264 and 4 up to 67584, each one kernel that
gates in place; above that one thread per edge, the search kernel followed by k_line_gate."""
import numpy as np
import pytest

from liodom_b200 import api
from conftest import get_sequence, pose_err

pytestmark = pytest.mark.gpu

TOL_T = 1e-4   # metres
TOL_R = 1e-5   # radians
N_SEEDS = 8
N_FRAMES = 10
PREV = 15


@pytest.fixture(autouse=True)
def _default_variants(monkeypatch):
    for v in ("LIODOM_LANE_GROUPS", "LIODOM_ASSOC_GROUP", "LIODOM_ASSOC_POOL"):
        monkeypatch.delenv(v, raising=False)


def _scans(B, f):
    return [get_sequence("hdl64", 1000 + l % N_SEEDS, N_FRAMES)[0][f] for l in range(B)]


def _ctx(B):
    return api.Context(prev_frames=PREV, max_points=131072, batch=B)


def _launches(ctx, call):
    before = ctx.launch_count
    call()
    return ctx.launch_count - before


@pytest.mark.parametrize("B,expect", [(1, 16), (64, 36)])
def test_scan_batch_launches(cuda_lib, B, expect):
    """1 lane: one group, 16 threads per edge.  64 lanes: two groups of 32, one thread per edge (2 x 18)."""
    ctx = _ctx(B)
    for f in range(3):
        scans = _scans(B, f)
        assert _launches(ctx, lambda: ctx.scan_batch(scans)) == expect, f
        ctx.results()
    ctx.close()


def test_scan_lanes_launches_match_batch_k(cuda_lib):
    """k lanes of a 128-lane context report the launches of a batch-k context's step."""
    ctx = _ctx(128)
    for k, expect in ((1, 16), (8, 16), (16, 18), (64, 36)):
        scans = _scans(k, 0)
        ref = _ctx(k)
        assert _launches(ref, lambda: ref.scan_batch(scans)) == expect, k
        ref.results()
        ref.close()
        lanes = list(range(128 - k, 128))[::-1]
        assert _launches(ctx, lambda: ctx.scan_lanes(lanes, scans)) == expect, k
        ctx.results()
    ctx.close()


def test_single_lane_entry_point_launches(cuda_lib):
    """liodom_split 3, liodom_extract 5 (with and without the smoothness keys), liodom_register 11."""
    ctx = _ctx(1)
    seq = get_sequence("hdl64", 1000, N_FRAMES)[0]
    assert _launches(ctx, lambda: ctx.split(seq[0])) == 3
    assert _launches(ctx, lambda: ctx.extract(seq[0], debug=True)) == 5
    for f in range(3):
        edges = ctx.extract(seq[f])
        assert _launches(ctx, lambda: ctx.extract(seq[f])) == 5, f
        assert _launches(ctx, lambda: ctx.register(edges)) == 11, f
    ctx.close()


@pytest.mark.parametrize("B", [32, 64])
def test_timed_steps_match_untimed(cuda_lib, B):
    """Stage timing enqueues the lanes as one group.  At 32 lanes so does the untimed step: bitwise the same poses and
    edge counts.  At 64 lanes the untimed step runs two groups, and k_solve's cluster size (with it the summation order)
    follows the group's lane count: poses within 1e-4 m / 1e-5 rad.  stage_times then holds one call per timed step."""
    timed, plain = _ctx(B), _ctx(B)
    timed.stage_timing(True)
    for f in range(N_FRAMES):
        scans = _scans(B, f)
        timed.scan_batch(scans)
        plain.scan_batch(scans)
        tp, tn = timed.results()
        pp, pn = plain.results()
        assert np.array_equal(tn, pn), "frame %d: edge counts differ" % f
        if B == 32:
            assert np.array_equal(tp.view(np.uint64), pp.view(np.uint64)), "frame %d: poses differ" % f
        else:
            for l in range(B):
                dt, dr = pose_err(tp[l], pp[l])
                assert dt < TOL_T and dr < TOL_R, "frame %d lane %d: %g m, %g rad" % (f, l, dt, dr)
    ms, calls = timed.stage_times()
    assert calls == N_FRAMES
    assert len(ms) == api.NUM_STAGES and np.all(ms > 0), ms
    timed.close()
    plain.close()


def test_single_lane_calls_add_no_stage_events(cuda_lib):
    """liodom_split / liodom_extract / liodom_register between two timed liodom_scan_batch calls time nothing."""
    ctx = _ctx(2)
    ctx.stage_timing(True)
    ctx.scan_batch(_scans(2, 0))
    ctx.results()
    assert ctx.stage_times()[1] == 1
    seq = get_sequence("hdl64", 1001, N_FRAMES)[0]
    ctx.split(seq[1], lane=1)
    ctx.register(ctx.extract(seq[1], lane=1), lane=1)
    assert ctx.stage_times()[1] == 1
    ctx.scan_batch(_scans(2, 2))
    ctx.results()
    ms, calls = ctx.stage_times()
    assert calls == 2 and np.all(ms > 0), (ms, calls)
    ctx.close()
