"""The oracle's association (src/laser_odometry.cc:300-344; brute force and kd-tree) against the NumPy restatement
np_ref.knn5_gate on the constructed cases of assoc_cases.py, ties included: the reference the GPU association test
relies on."""
import numpy as np
import pytest

import np_ref
import oracle
from assoc_cases import cases, by_name, cut_list

NAMES = [c.name for c in cases()]


@pytest.mark.parametrize("name", NAMES)
def test_case_reaches_its_regime(name):
    by_name()[name].check()


@pytest.mark.parametrize("knn_method", [0, 1])
@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_restatement(name, knn_method):
    c = by_name()[name]
    r = c.ref()
    target = c.target()
    if c.filter_local_map:
        assert np.array_equal(oracle.voxelgrid(c.window(), 0.4).view(np.uint32), target.view(np.uint32))
    o = oracle.associate(c.edges, c.pose, target, knn_method=knn_method)
    assert np.array_equal(o["q_world"].view(np.uint32), r["q_world"].view(np.uint32))
    idx, d2 = cut_list(o)
    assert np.array_equal(idx, r["knn_idx"])
    assert np.array_equal(d2.view(np.uint32), r["knn_d2"].view(np.uint32))
    assert np.array_equal(o["gate"] & 1, r["gate"] & 1)
    dec = r["decided"]
    assert np.array_equal(o["gate"][dec] & 2, r["gate"][dec] & 2)
    # A query with an infinite coordinate is at d2 = inf from every map point: the oracle keeps such entries (and flags
    # their equal d2 as a tie), the restatement and the GPU report no neighbours.  Both fail the gate.
    fin = np.isfinite(r["q_world"][:, :3]).all(1)
    assert np.array_equal(o["tie"][fin] == 1, r["tie"][fin])
    assert (o["gate"][~fin] == 0).all()


def test_restatement_matches_bruteforce_lists():
    """knn5_gate's uncut lists equal knn5_bruteforce where every map point and query is finite."""
    c = by_name()["stationary"]
    r = c.ref()
    idx, d2 = np_ref.knn5_bruteforce(c.target(), r["q_world"])
    assert np.array_equal(idx, r["idx6"][:, :5]) and np.array_equal(d2.view(np.uint32), r["d2_6"][:, :5].view(np.uint32))
