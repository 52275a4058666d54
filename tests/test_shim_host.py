"""Host-side (CPU) part of the C++ drop-in shim: K^-1 normalisation, the seeded 8-point hypotheses and the pose
recovery tail of find_E_ransac (host/two_view_host.hpp) must be BIT-IDENTICAL to the compiled reference, so
that the GPU scores the "same seeded hypotheses".  Checked against the CPU checker (conftest.py: the compiled
reference, or the port pinned to it).  No GPU needed."""
import numpy as np
import pytest

import shimlib
from conftest import TEMPLE_K, two_view_scene


@pytest.fixture(scope="module")
def shim():
    return shimlib.load()


@pytest.mark.parametrize("n,iters", [(8, 5), (50, 40), (400, 120), (2200, 60)])
def test_hypotheses_bit_identical(shim, checker, n, iters):
    pi, pj = two_view_scene(n, seed=100 + n)
    K = np.ascontiguousarray(TEMPLE_K.reshape(9))
    xi, xj = np.zeros_like(pi), np.zeros_like(pj)
    assert shim.shim_host_norm_points(K, pi, n, xi) == 0 and shim.shim_host_norm_points(K, pj, n, xj) == 0
    assert np.array_equal(xi, checker.norm_points(TEMPLE_K, pi)) and np.array_equal(xj, checker.norm_points(TEMPLE_K, pj))
    E = np.zeros((iters, 9))
    shim.shim_host_hypotheses(xi, xj, n, iters, E)
    want, _ = checker.ransac_hypotheses(xi, xj, iters)
    assert np.array_equal(E.view(np.uint64), want.view(np.uint64))


@pytest.mark.parametrize("n,iters,thr", [(400, 120, 1e-3), (300, 60, 2e-3), (60, 40, 1e-3)])
def test_pose_recovery_bit_identical(shim, checker, n, iters, thr):
    pi, pj = two_view_scene(n, seed=7 + n)
    want = checker.find_E_ransac(TEMPLE_K, pi, pj, iters, thr, 8)
    assert want is not None
    xi, xj = checker.norm_points(TEMPLE_K, pi), checker.norm_points(TEMPLE_K, pj)
    E, _ = checker.ransac_hypotheses(xi, xj, iters)
    counts, bh, inl = checker.ransac_score(xi, xj, E, thr)
    assert np.array_equal(inl, want[2])
    R, t = np.zeros(9), np.zeros(3)
    shim.shim_host_recover_pose(np.ascontiguousarray(E[bh]), xi, xj, np.ascontiguousarray(inl, np.int32), len(inl), R, t)
    assert np.array_equal(R.reshape(3, 3), want[0]) and np.array_equal(t, want[1])


def test_singular_K_is_reported(shim):
    assert shim.shim_host_norm_points(np.zeros(9), np.zeros((1, 2)), 1, np.zeros((1, 2))) == -1


def test_host_triangulation_bit_identical(shim, checker):
    """host/two_view_host.hpp: triangulate_dlt (:1477-1516) == the CPU checker's, bit for bit (the port's triangulate_dlt
    is pinned by tests/test_oracle_vs_ref.py::test_triangulate_dlt)."""
    from conftest import triangulation_scene
    poses, ia, ib, ui, uj, _ = triangulation_scene(300, seed=11)
    X = np.zeros((300, 3))
    shim.shim_host_triangulate(np.ascontiguousarray(TEMPLE_K.reshape(9)), poses, ia, ib, ui, uj, 300, X)
    assert np.array_equal(X, checker.triangulate_dlt(TEMPLE_K, poses, ia, ib, ui, uj))
