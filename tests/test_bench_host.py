"""CPU tests of bench.py's host-side logic: the wire format of the N > 1 gather (one packed byte block per rank, li and
inlier indices as int16), the shard partition, and the reference arm's line (runs the compiled reference on a tiny
workload)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_wire_layout_roundtrip():
    rng = np.random.default_rng(1)
    cap, P, world = 37, 23, 4
    shards = [bench.shard_range(P, world, r) for r in range(world)]
    assert shards[0][0] == 0 and shards[-1][1] == P and all(a[1] == b[0] for a, b in zip(shards, shards[1:]))
    full = {"li": rng.integers(0, 4000, (P, cap, 2)).astype(np.int16), "lj": rng.normal(0, 1000, (P, cap, 2)),
            "nk": rng.integers(0, cap, P).astype(np.int32), "nc": rng.integers(0, cap, P).astype(np.int32),
            "status": rng.integers(0, 3, P).astype(np.int32), "best": rng.integers(-1, 4000, (P, 2)).astype(np.int32),
            "inliers": rng.integers(0, cap, (P, cap)).astype(np.int16), "R": rng.normal(size=(P, 9)), "t": rng.normal(size=(P, 3))}

    class _T:  # stands in for a pinned torch tensor: .numpy() gives the byte block
        def __init__(self, a):
            self.a = a

        def numpy(self):
            return self.a

    host = {}
    for r, (a, b) in enumerate(shards):
        lay, total = bench.wire_layout(b - a, cap)
        assert total % 8 == 0 and [k for k, *_ in lay] == [k for k, *_ in bench.WIRE]
        block = np.zeros(max(total, 8), np.uint8)
        for key, dt, shape, off in lay:
            src = np.ascontiguousarray(full[key][a:b]).view(np.uint8).reshape(-1)
            assert src.dtype == np.uint8 and full[key].dtype == dt and full[key][a:b].shape == shape
            block[off:off + src.size] = src
        host[r] = _T(block)
    got = bench.decode_gathered({"host": host}, shards, P, cap)
    for key in full:
        assert np.array_equal(got[key], full[key]), key


def test_dump_outputs(tmp_path):
    """--dump-outputs: float64 arrays of the resident step's results, entries the library leaves undefined masked, the
    same seeded pair sample every run (CPU tensors stand in for the device views)."""
    import torch
    rng = np.random.default_rng(2)
    P, cap = 300, 40
    nk = rng.integers(0, cap + 1, P).astype(np.int32)
    st = rng.integers(0, 3, P).astype(np.int32)
    best = np.stack([rng.integers(-1, 4000, P), rng.integers(0, cap + 1, P)], 1).astype(np.int32)
    dev = [rng.normal(0, 100, (P, cap, 2)), rng.normal(0, 100, (P, cap, 2)), nk, rng.integers(0, 999, P).astype(np.int32),
           st, best, rng.integers(0, cap, (P, cap)).astype(np.int32), rng.normal(size=(P, 9)), rng.normal(size=(P, 3))]

    class _Pairs:
        def torch_views(self, n):
            return [torch.from_numpy(a) for a in dev[:4]]

        def ransac_torch_views(self, n):
            return [torch.from_numpy(a) for a in dev[4:]]

    class _Ctx:
        def sync(self):
            pass

    class _Unit:
        npairs, pairs, ctx = P, _Pairs(), _Ctx()
    _Unit.cap = cap
    for d in ("a", "b"):
        bench.dump_outputs(_Unit, torch, str(tmp_path / d))
    got = {f[:-4]: np.load(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))}
    assert all(np.array_equal(got[k], np.load(str(tmp_path / "b" / f"{k}.npy"))) for k in got)
    assert all(a.dtype == np.float64 for a in got.values())
    s = got["pairs"].astype(int)
    assert len(s) == bench.DUMP_PAIRS and np.all(np.diff(s) > 0) and s[-1] < P
    assert np.array_equal(got["n_kept"], nk) and np.array_equal(got["status"], st) and np.array_equal(got["best_n"], best[:, 1])
    ok = st == 2
    assert np.array_equal(got["R"][ok], dev[7][ok]) and not got["R"][~ok].any() and not got["t"][~ok].any()
    for k, p in enumerate(s):
        n, m = nk[p], best[p, 1] if st[p] == 2 else 0
        assert np.array_equal(got["li"][k, :n], dev[0][p, :n]) and not got["li"][k, n:].any() and not got["lj"][k, n:].any()
        assert np.array_equal(got["inliers"][k, :m], dev[6][p, :m]) and np.all(got["inliers"][k, m:] == -1)


def test_reference_arm_line_tiny():
    """`bench.py --impl reference` prints ONE JSON line with the contract's keys (tiny frames so that it runs in seconds)."""
    env = dict(os.environ)
    code = ("import sys, bench; bench.WORKLOADS['c2'].update(W=160, H=120, corners=60); "
            "sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'c2', '--steps', '1', '--warmup', '0']; bench.main()")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "feature-tracks/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["scaling"] == "strong" and line["higher_is_better"] is True
