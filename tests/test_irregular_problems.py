"""The generators of tests/irregular_problems.py give the shapes they promise (each asserts its own on construction): closure
blocks present in S, no cut where the closure spans the sequence, wrapping tracks, a forest, ragged counts.  CPU only."""
import numpy as np
import pytest

import irregular_problems as ip

syn = ip.syn


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_closure_problems(case):
    p = ip.closure_problem(case)
    assert p.n_cam == 120 and p.depth is not None and np.all(np.diff(p.cam_idx) >= 0)
    assert ip.n_components(p) == 1
    again = ip.closure_problem(case)  # seeded: the same problem twice
    assert np.array_equal(p.cam_idx, again.cam_idx) and np.array_equal(p.uv2, again.uv2)


def test_closed_street_wraps():
    p = ip.closed_street()
    assert p.n_cam == 360 and p.depth is None
    seen_first = set(p.pt_idx[p.cam_idx == 0].tolist())
    assert seen_first & set(p.pt_idx[p.cam_idx == p.n_cam - 1].tolist())


def test_two_maps_is_a_forest():
    a, b = ip.tum_window(12, 5), ip.tum_window(10, 6)
    q = ip.two_maps(a, b)
    assert q.n_cam == a.n_cam + b.n_cam and q.n_pt == a.n_pt + b.n_pt and q.n_obs == a.n_obs + b.n_obs


def test_ragged_inputs():
    p = ip.tum_window(12, 5)
    q = ip.ragged(p, empty_cam=3, one_obs_cam=7, once=20, unobserved=5, duplicates=10)
    per_cam = np.bincount(q.cam_idx, minlength=q.n_cam)
    assert per_cam[3] == 0 and per_cam[7] == 1
    bi, bj = ip.covisibility_blocks(q.cam_idx, q.pt_idx, q.n_cam, q.fixed_cam)
    assert 3 not in bi and 3 not in bj  # no diagonal block of S for the camera without observations
    sym = ip.gpu_symbolic(q)
    assert int(np.sum(sym.node[:, 4] < 0)) >= 3  # the fixed camera and the unobserved one are roots of their own
