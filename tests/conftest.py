import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def port():
    import oracle
    return oracle.port()


@pytest.fixture(scope="session")
def ref():
    import oracle
    r = oracle.ref()
    if r is None:
        pytest.skip("compiled reference (oracle/_ref/libsfmref.so) not available on this machine")
    return r


@pytest.fixture
def checker():
    """The CPU checker: the compiled reference when oracle/_ref/libsfmref.so is built, else the port
    (oracle/sfm_oracle.cpp).  Stored vectors pin the port everywhere: tests/test_golden.py against outputs of the
    compiled reference (pyramid, corners, KLT, tracker, one RANSAC case, pair front end), tests/test_oracle_vs_ref.py
    against its recorded outputs for every case it compares with the reference (see that module), and live against
    the reference where it is built."""
    import oracle
    return oracle.best()[0]


@pytest.fixture(scope="session")
def ctx():
    import sfmgpu
    c = sfmgpu.Context(0)  # raises when the library or the GPU is missing: no CPU fallback
    yield c
    c.close()


TEMPLE_K = np.array([1520.4, 0, 302.32, 0, 1525.9, 246.87, 0, 0, 1.0]).reshape(3, 3)


def two_view_scene(n, seed=777, outlier_frac=0.3, sigma=0.3):
    """SURVEY.md §8d C4: synthetic two-view correspondences in pixels (numpy PCG64, deterministic)."""
    rng = np.random.default_rng(seed)
    X = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-0.4, 0.4, n), rng.uniform(1.5, 2.5, n)], 1)
    w = np.array([0.02, -0.15, 0.01])
    th = np.linalg.norm(w)
    k = w / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    R = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx
    t = np.array([0.2, 0.01, 0.03])
    X2 = X @ R.T + t
    pi = (X / X[:, 2:3]) @ TEMPLE_K.T
    pj = (X2 / X2[:, 2:3]) @ TEMPLE_K.T
    pi, pj = pi[:, :2] + rng.normal(0, sigma, (n, 2)), pj[:, :2] + rng.normal(0, sigma, (n, 2))
    out = rng.random(n) < outlier_frac
    pj[out] = np.stack([rng.uniform(0, 640, out.sum()), rng.uniform(0, 480, out.sum())], 1)
    return np.ascontiguousarray(pi), np.ascontiguousarray(pj)


def triangulation_scene(n, P=5, seed=3):
    """P camera-to-world poses looking at a cloud of n points; every track is seen from two different poses."""
    rng = np.random.default_rng(seed)
    poses = np.zeros((P, 12))
    Rs, Cs = [], []
    for p in range(P):
        w = rng.normal(0, 0.08, 3)
        th = np.linalg.norm(w)
        k = w / th
        Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        R = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx  # camera -> world
        Cc = rng.normal(0, 0.15, 3)
        poses[p, :9], poses[p, 9:] = R.reshape(9), Cc
        Rs.append(R)
        Cs.append(Cc)
    X = np.c_[rng.uniform(-0.5, 0.5, n), rng.uniform(-0.4, 0.4, n), rng.uniform(1.5, 2.5, n)]
    ia = rng.integers(0, P, n).astype(np.int32)
    ib = ((ia + rng.integers(1, P, n)) % P).astype(np.int32)

    def proj(idx):
        out = np.zeros((n, 2))
        for t in range(n):
            xc = Rs[idx[t]].T @ (X[t] - Cs[idx[t]])
            u = TEMPLE_K @ (xc / xc[2])
            out[t] = u[:2]
        return out + rng.normal(0, 0.3, (n, 2))

    return poses, ia, ib, proj(ia), proj(ib), X
