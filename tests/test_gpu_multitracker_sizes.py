"""The lock-step tracker over sequences of different image sizes and cameras (sfmgpu_multitracker_create_sized,
sfmgpu_multitracker_set_ransac_cameras).

Sequence s of a mixed tracker runs through the same per-feature arithmetic as a one-sequence tracker of its own size: the KLT
chain reads its images through a per-list geometry table, everything else works on the [S][ROWS] lists as before.  So, with
both pinned to one kernel family, every output is byte-identical.  The sizes include odd ones and one (97 x 61) whose upper
pyramid levels are a few windows wide, so border windows reach the masked lane kernel and the warp-per-feature kernel."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ring_dataset
import sfmgpu
from conftest import TEMPLE_K
from sfmgpu import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200", "host")
E_ARG = -1
OK = 2  # SFMGPU_TV_OK
KW = dict(max_tracks=150, min_tracks=140)  # replenishment within a few frames
SIZES = [(640, 480), (640, 480), (1280, 720), (641, 479), (97, 61), (640, 480)]  # classes: 640x480 twice adjacent, once apart
T = 7
KLT_TOL = 1e-3  # px, the parity budget
CXX = ["g++", "-std=c++20", "-O3", "-DNDEBUG", "-fPIC", "-shared", "-pthread", "-ffp-contract=off"]


def _seq(s, w, h):
    """Value noise; sequence 3 starts with three flat frames (no corners: its list stays empty and it is reset on every frame
    until the first textured one)."""
    return [np.full((h, w), 90, np.uint8) if s == 3 and t < 3 else synth.frame(3100 + s, t, w, h) for t in range(T)]


@pytest.fixture(scope="module")
def seqs():
    return [_seq(s, w, h) for s, (w, h) in enumerate(SIZES)]


def _run(mt, seqs, steps=T):
    """Per step: survivors (prev, cur, ids) per sequence and the track lists per sequence."""
    out = []
    for t in range(steps):
        surv = mt.step([sq[t] for sq in seqs])
        out.append((surv, [mt.tracks(s) for s in range(len(seqs))]))
    return out


def _equal(a, b, where):
    for x, y in zip(a, b):
        assert np.array_equal(x, y), where


def _same_results(a, b, where):
    """Two ransac_results() byte for byte; R and t are written for poses only."""
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), where
    for x, y in zip(a[2], b[2]):
        assert np.array_equal(x, y), where
    ok = a[0] == OK
    assert np.array_equal(a[3][ok], b[3][ok]) and np.array_equal(a[4][ok], b[4][ok]), where


@pytest.mark.parametrize("mode", [1, 2])
def test_mixed_equals_one_sequence_trackers(ctx, seqs, mode):
    """Every step's survivors, ids, track lists and the totals of a mixed tracker equal, byte for byte, those of an S = 1
    tracker per sequence, both pinned to one KLT family (1: warp-per-feature, 2: the lane chain)."""
    ctx.klt_set_mode(mode)
    try:
        mt = ctx.multitracker(len(SIZES), [w for w, _ in SIZES], [h for _, h in SIZES], **KW)
        got = _run(mt, seqs)
        singles = []
        for s, (w, h) in enumerate(SIZES):
            one = ctx.multitracker(1, w, h, **KW)
            singles.append((_run(one, [seqs[s]]), one.totals()))
            one.close()
        resets = 0
        for t in range(T):
            for s in range(len(SIZES)):
                want_surv, want_tracks = singles[s][0][t][0][0], singles[s][0][t][1][0]
                _equal(got[t][0][s], want_surv, (t, s))
                _equal(got[t][1][s], want_tracks, (t, s))
                resets += t > 0 and len(want_surv[2]) == 0 and len(want_tracks[1]) > 0
        assert resets >= 1  # sequence 3 entered a step without tracks and was reset on its textured frame
        tot = mt.totals()
        assert tot[0] == sum(x[1][0] for x in singles) and tot[1] == sum(x[1][1] for x in singles)
        mt.close()
    finally:
        ctx.klt_set_mode(0)


def test_mixed_auto_matches_checker(ctx, checker, seqs):
    """Auto mode against the checker's KLTTracker on two sequences: ids exact, positions within the parity budget."""
    mt = ctx.multitracker(len(SIZES), [w for w, _ in SIZES], [h for _, h in SIZES], **KW)
    refs = {s: checker.tracker(**KW) for s in (2, 4)}
    for t in range(T):
        got = mt.step([sq[t] for sq in seqs])
        for s, ref in refs.items():
            r = ref.step(seqs[s][t])
            assert np.array_equal(got[s][2], r[2]), (t, s)
            for a, b in ((got[s][0], r[0]), (got[s][1], r[1])):
                assert a.shape == b.shape and np.nanmax(np.abs(a - b), initial=0.0) <= KLT_TOL, (t, s)
    mt.close()


def test_sized_with_equal_sizes_equals_create(ctx):
    """create_sized with S equal sizes is create: the same outputs byte for byte and the same launches per step."""
    S, w, h = 4, 320, 240
    frames = [np.stack([synth.frame(3200 + s, t, w, h) for s in range(S)]) for t in range(T)]
    res = []
    for sized in (False, True):
        mt = ctx.multitracker(S, [w] * S, [h] * S, **KW) if sized else ctx.multitracker(S, w, h, **KW)
        mt.set_ransac(TEMPLE_K, 500, 1e-3, 30, 1)
        steps, launches = [], []
        for t in range(T):
            n0 = ctx.launches()
            surv = mt.step(frames[t])
            launches.append(ctx.launches() - n0)
            steps.append((surv, [mt.tracks(s) for s in range(S)], mt.ransac_results()))
        res.append((steps, launches, mt.totals()))
        mt.close()
    (a, la, ta), (b, lb, tb) = res
    assert la == lb and ta == tb
    for t in range(T):
        for s in range(S):
            _equal(a[t][0][s], b[t][0][s], (t, s))
            _equal(a[t][1][s], b[t][1][s], (t, s))
        _same_results(a[t][2], b[t][2], t)


def test_mixed_pipelined_equals_plain(ctx, seqs):
    """Prefetched steps of a mixed tracker (frames staged page-locked by the binding, and frames in device memory) equal plain
    steps."""
    torch = pytest.importorskip("torch")
    S = len(SIZES)
    ws, hs = [w for w, _ in SIZES], [h for _, h in SIZES]
    plain = ctx.multitracker(S, ws, hs, **KW)
    want = [plain.step([sq[t] for sq in seqs]) for t in range(T)]
    plain.close()
    pipe = ctx.multitracker(S, ws, hs, **KW)
    pipe.prefetch([sq[0] for sq in seqs])
    for t in range(T):
        got = pipe.step(None, next_imgs=[sq[t + 1] for sq in seqs] if t + 1 < T else None)
        for s in range(S):
            _equal(got[s], want[t][s], (t, s))
    pipe.close()
    # device memory: the frames of a step back to back in sequence order
    dev = [torch.from_numpy(np.concatenate([sq[t].reshape(-1) for sq in seqs])).to("cuda:0") for t in range(T)]
    torch.cuda.synchronize()
    mt = ctx.multitracker(S, ws, hs, **KW)
    for t in range(T):
        got = mt.step_ptr(dev[t].data_ptr(), dev[t + 1].data_ptr() if t + 1 < T else None, fetch=True) if t == 0 else \
            mt.step_ptr(None, dev[t + 1].data_ptr() if t + 1 < T else None, fetch=True)
        for s in range(S):
            _equal(got[s], want[t][s], (t, s))
    mt.close()


# ---- one camera per sequence ---------------------------------------------------------------------------------------------
ITERS, THR, MIN_INL = 2500, 1e-3, 60  # :1739
KW_TV = dict(max_tracks=400, min_tracks=380)  # tests/test_gpu_multitracker_two_view.py's configuration
CAM_SIZES = [(640, 480), (1280, 720), (641, 479), (800, 600)]


def _K(w, h, s=0):
    """TEMPLE_K scaled to a w x h image, a little different for every sequence s."""
    a, b = w / 640.0, h / 480.0
    return np.array([[1520.4 * a * (1 + 0.01 * s), 0, 302.32 * a + 2 * s], [0, 1525.9 * a * (1 + 0.01 * s), 246.87 * b - s], [0, 0, 1.0]])


@pytest.fixture(scope="module")
def ring():
    """Ray-cast ring sequences, one camera per sequence (its own size and K)."""
    return [[ring_dataset.render(np.deg2rad(2.0 * s + 0.25 * t), w, h, K=_K(w, h, s)) for t in range(5)]
            for s, (w, h) in enumerate(CAM_SIZES)]


def _pairs_stage(ctx, K, prev, cur, cap):
    p = ctx.pairs(1, cap)
    p.set_matches([prev], [cur])
    p.ransac(K, ITERS, THR, MIN_INL, 1)
    st, bn = np.zeros(1, np.int32), np.zeros(1, np.int32)
    inl, R, tt = np.zeros((1, cap), np.int32), np.zeros((1, 9)), np.zeros((1, 3))
    p.ransac_download_all(st, bn, inl, R, tt)
    return st[0], bn[0], inl[0, :bn[0]], R.reshape(3, 3), tt[0]


@pytest.mark.parametrize("mixed", [True, False])
def test_cameras_equal_pairs_stage_and_checker(ctx, checker, ring, mixed):
    """Sequence s's stage results equal pairs_ransac with K_s on the same survivors (status, best_n, inliers, R, t byte for
    byte); the first and the last sequence equal the checker's find_E_ransac.  mixed = False: four cameras at one size."""
    sizes = CAM_SIZES if mixed else [CAM_SIZES[0]] * len(CAM_SIZES)
    Ks = np.stack([_K(*sizes[s], s) for s in range(len(sizes))])
    frames = ring if mixed else [[ring_dataset.render(np.deg2rad(2.0 * s + 0.25 * t), 640, 480, K=Ks[s]) for t in range(5)]
                                 for s in range(len(sizes))]
    S = len(sizes)
    mt = ctx.multitracker(S, [w for w, _ in sizes], [h for _, h in sizes], **KW_TV) if mixed else \
        ctx.multitracker(S, sizes[0][0], sizes[0][1], **KW_TV)
    mt.set_ransac(Ks, ITERS, THR, MIN_INL, 1)
    poses = 0
    for t in range(5):
        surv = mt.step([f[t] for f in frames])
        st, bn, inl, R, tt = mt.ransac_results()
        for s, (prev, cur, _) in enumerate(surv):
            if len(prev) == 0:
                assert st[s] == 0 and bn[s] == 0, (t, s)
                continue
            w = _pairs_stage(ctx, Ks[s], prev, cur, mt.cap)
            assert st[s] == w[0] and bn[s] == w[1] and np.array_equal(inl[s], w[2]), (t, s)
            if st[s] == OK:
                poses += 1
                assert np.array_equal(R[s], w[3]) and np.array_equal(tt[s], w[4]), (t, s)
            if s in (0, S - 1):
                r = checker.find_E_ransac(Ks[s], prev, cur, ITERS, THR, MIN_INL)
                assert (r is None) == (st[s] != OK), (t, s)
                if r is not None:
                    assert np.array_equal(inl[s], r[2]), (t, s)
                    assert np.abs(R[s] - r[0]).max() < 1e-6 and np.abs(tt[s] - r[1]).max() < 1e-6, (t, s)
    assert poses >= S
    mt.close()


def test_uniform_cameras_equal_set_ransac_and_singular_refusal(ctx, ring):
    """set_ransac_cameras with S copies of K equals set_ransac(K) byte for byte.  A singular K_s is refused, names s, and
    leaves the previous configuration and the last step's results in force."""
    S = len(CAM_SIZES)
    ws, hs = [w for w, _ in CAM_SIZES], [h for _, h in CAM_SIZES]
    res = []
    for per_seq in (False, True):
        mt = ctx.multitracker(S, ws, hs, **KW_TV)
        mt.set_ransac(np.stack([TEMPLE_K] * S) if per_seq else TEMPLE_K, ITERS, THR, MIN_INL, 1)
        res.append([(mt.step([f[t] for f in ring]), mt.ransac_results()) for t in range(4)])
        if per_seq:
            before = mt.ransac_results()
            Ks = np.stack([_K(w, h, s) for s, (w, h) in enumerate(CAM_SIZES)])
            Ks[2] = 0.0
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                mt.set_ransac(Ks, ITERS, THR, MIN_INL, 1)
            assert e.value.code == E_ARG and "Singular K" in str(e.value) and "sequence 2" in str(e.value)
            _same_results(before, mt.ransac_results(), "refused")
            # the previous configuration (S copies of TEMPLE_K) is still the one the next step runs
            surv = mt.step([f[4] for f in ring])
            nxt = mt.ransac_results()
            ref = ctx.multitracker(S, ws, hs, **KW_TV)
            ref.set_ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)
            for t in range(5):
                rs = ref.step([f[t] for f in ring])
            _same_results(nxt, ref.ransac_results(), "after the refusal")
            for s in range(S):
                _equal(surv[s], rs[s], s)
            ref.close()
        mt.close()
    for (sa, ra), (sb, rb) in zip(*res):
        for s in range(S):
            _equal(sa[s], sb[s], s)
        _same_results(ra, rb, "uniform")


# ---- refusals -------------------------------------------------------------------------------------------------------------
def test_refusals(ctx, seqs):
    lib, cfg = ctx.lib, sfmgpu.lkcfg(**KW)

    def create(S, w, h):
        p = C.c_void_p()
        rc = lib.sfmgpu_multitracker_create_sized(ctx.h, C.byref(cfg), S, w, h, C.byref(p))
        if rc == 0:
            lib.sfmgpu_multitracker_destroy(ctx.h, p)
        return rc

    arr = lambda v: np.ascontiguousarray(v, np.int32).ctypes.data_as(C.c_void_p)  # noqa: E731
    for S, w, h in ((2, [640, 0], [480, 480]), (2, [640, 32768], [480, 480]), (2, [640, 640], [-1, 480]), (1, [640], [32768])):
        assert create(S, arr(w), arr(h)) == E_ARG, (w, h)
    assert create(0, arr([640]), arr([480])) == E_ARG and create(513, arr([640] * 513), arr([480] * 513)) == E_ARG
    assert create(2, None, arr([480, 480])) == E_ARG and create(2, arr([640, 640]), None) == E_ARG
    assert create(2, arr([32767, 1]), arr([1, 32767])) == 0

    S = len(SIZES)
    mt = ctx.multitracker(S, [w for w, _ in SIZES], [h for _, h in SIZES], **KW)
    mt.step([sq[0] for sq in seqs])
    before = [mt.tracks(s) for s in range(S)]
    f = ctx.frames(640, 480, S, 3)
    for call in (lambda: mt.step_frames(f, np.zeros(S, np.int32)),
                 lambda: mt.step_packed(np.zeros(64, np.uint8), np.zeros(S, np.int32)),
                 lambda: mt.prefetch_packed(np.zeros(64, np.uint8), np.zeros(S, np.int32))):
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            call()
        assert e.value.code == E_ARG and "different image sizes" in str(e.value)
    for s in range(S):  # nothing was queued
        _equal(mt.tracks(s), before[s], s)
    got = mt.step([sq[1] for sq in seqs])
    assert sum(len(g[2]) for g in got) > 0
    mt.close()


# ---- the C++ drop-in ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mszshim(tmp_path_factory):
    """MultiKLTTracker(cfg, sizes) + set_two_view(vector<Mat33>), and KLTTracker + find_E_ransac (tests/cpp/multitracker_sizes_shim.cpp)."""
    sfmgpu.load_library()
    libdir = os.path.dirname(sfmgpu.LIB_PATH)
    so = str(tmp_path_factory.mktemp("mszshim") / "libmszshim.so")
    subprocess.run(CXX + ["-I" + HOST, os.path.join(ROOT, "tests", "cpp", "multitracker_sizes_shim.cpp"), "-o", so, "-L" + libdir,
                          "-lsfmgpu", "-Wl,-rpath," + libdir], check=True)
    lib = C.CDLL(so)
    vp = C.c_void_p
    lib.msz_last_error.restype = C.c_char_p
    lib.msz_create.restype = vp
    lib.msz_create.argtypes = [C.c_int, vp, vp, C.c_int, C.c_int]
    lib.msz_destroy.argtypes = [vp]
    lib.msz_set_two_view.argtypes = [vp, C.c_int, vp, C.c_int, C.c_double, C.c_int]
    lib.msz_step.argtypes = [vp, C.c_int, vp, vp, vp] + [vp] * 4 + [C.c_int] + [vp] * 5
    lib.msz_single_create.restype = vp
    lib.msz_single_create.argtypes = [C.c_int, C.c_int]
    lib.msz_single_destroy.argtypes = [vp]
    lib.msz_single_step.argtypes = [vp, vp, C.c_int, C.c_int, vp, C.c_int, C.c_double, C.c_int] + [vp] * 4 + [C.c_int] + [vp] * 5
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_shim_sized_multitracker_equals_klttracker_and_find_E(mszshim, ring):
    """A sized MultiKLTTracker with one camera per sequence equals a KLTTracker plus find_E_ransac per sequence: survivors and
    ids byte for byte (both take the warp-per-feature family: S x ROWS < 6000), status and inliers exactly, R and t within
    1e-6."""
    lib = mszshim
    S = len(CAM_SIZES)
    ws, hs = np.array([w for w, _ in CAM_SIZES], np.int32), np.array([h for _, h in CAM_SIZES], np.int32)
    Ks = np.ascontiguousarray(np.stack([_K(w, h, s) for s, (w, h) in enumerate(CAM_SIZES)]))
    cap = max(KW_TV["max_tracks"], KW_TV["min_tracks"], 1) + 1
    mt = lib.msz_create(S, _p(ws), _p(hs), KW_TV["max_tracks"], KW_TV["min_tracks"])
    assert mt, lib.msz_last_error().decode()
    singles = [lib.msz_single_create(KW_TV["max_tracks"], KW_TV["min_tracks"]) for _ in range(S)]
    try:
        assert lib.msz_set_two_view(mt, S, _p(Ks), ITERS, THR, MIN_INL) == 0, lib.msz_last_error().decode()
        poses = 0
        for t in range(5):
            imgs = [np.ascontiguousarray(ring[s][t]) for s in range(S)]
            ptrs = (C.c_void_p * S)(*[im.ctypes.data for im in imgs])
            ids, n = np.zeros((S, cap), np.int32), np.zeros(S, np.int32)
            prev, cur = np.zeros((S, cap, 2)), np.zeros((S, cap, 2))
            has, R, tt = np.zeros(S, np.int32), np.zeros((S, 9)), np.zeros((S, 3))
            inl, ninl = np.zeros((S, cap), np.int32), np.zeros(S, np.int32)
            rc = lib.msz_step(mt, S, C.cast(ptrs, C.c_void_p), _p(ws), _p(hs), _p(ids), _p(prev), _p(cur), _p(n), cap, _p(has), _p(R),
                              _p(tt), _p(inl), _p(ninl))
            assert rc == 0, lib.msz_last_error().decode()
            for s in range(S):
                ids1, n1 = np.zeros(cap, np.int32), np.zeros(1, np.int32)
                prev1, cur1 = np.zeros((cap, 2)), np.zeros((cap, 2))
                has1, R1, t1 = np.zeros(1, np.int32), np.zeros(9), np.zeros(3)
                inl1, ninl1 = np.zeros(cap, np.int32), np.zeros(1, np.int32)
                K = np.ascontiguousarray(Ks[s])
                rc = lib.msz_single_step(singles[s], _p(imgs[s]), int(ws[s]), int(hs[s]), _p(K), ITERS, THR, MIN_INL, _p(ids1), _p(prev1),
                                         _p(cur1), _p(n1), cap, _p(has1), _p(R1), _p(t1), _p(inl1), _p(ninl1))
                assert rc == 0, lib.msz_last_error().decode()
                k = n[s]
                assert k == n1[0] and np.array_equal(ids[s, :k], ids1[:k]), (t, s)
                assert np.array_equal(prev[s, :k], prev1[:k]) and np.array_equal(cur[s, :k], cur1[:k]), (t, s)
                assert has[s] == has1[0], (t, s)
                if has[s]:
                    poses += 1
                    assert ninl[s] == ninl1[0] and np.array_equal(inl[s, :ninl[s]], inl1[:ninl1[0]]), (t, s)
                    assert np.abs(R[s] - R1).max() < 1e-6 and np.abs(tt[s] - t1).max() < 1e-6, (t, s)
        assert poses >= S
    finally:
        lib.msz_destroy(mt)
        for o in singles:
            lib.msz_single_destroy(o)
