"""GPU tests of the RANSAC stage inside the lock-step tracker: find_E_ransac(K, step.prev_pts, step.cur_pts, 2500, 1e-3, 60)
(cpp/src/templering_sfm.cpp:1739) on every sequence's survivors, skipped where a sequence has none (:1715), computed inside
sfmgpu_multitracker's step with no extra host round trip.

The sequences mix real two-view geometry (the ray-cast ring scene of tests/ring_dataset.py seen from cameras moving along
the ring) with the planar value-noise frames of sfmgpu.synth, one quantised sequence (many identical corner scores) and one
sparse sequence (a small textured window on a flat background: fewer survivors than min_inliers, so no pose)."""
import ctypes as C
import os

import numpy as np
import pytest

import ring_dataset
import sfmgpu
from conftest import TEMPLE_K
from sfmgpu import synth

pytestmark = pytest.mark.gpu

W, H, T = 640, 480, 6
KW = dict(max_tracks=400, min_tracks=380)  # replenishment in most steps
OK = 2  # SFMGPU_TV_OK
ITERS, THR, MIN_INL = 2500, 1e-3, 60  # :1739
RING_STARTS_DEG = (0.0, 3.0, 6.0)
RING_STEP_DEG = 0.25  # ~2 px of parallax between the sphere and the wall per frame


def _sparse(t):
    img = np.full((H, W), 100, np.uint8)
    img[200:240, 300:340] = synth.frame(20261103, t, W, H)[200:240, 300:340]
    return img


@pytest.fixture(scope="module")
def frames():
    """[T, S, H, W]: three ring sequences, a value-noise one, a quantised one, a sparse one."""
    seqs = [[ring_dataset.render(np.deg2rad(a + RING_STEP_DEG * t), W, H) for t in range(T)] for a in RING_STARTS_DEG]
    seqs.append([synth.frame(20261101, t, W, H) for t in range(T)])
    seqs.append([synth.frame(20261102, t, W, H) >> 3 << 3 for t in range(T)])
    seqs.append([_sparse(t) for t in range(T)])
    return np.ascontiguousarray(np.stack([np.stack([s[t] for s in seqs]) for t in range(T)]))


def _run(ctx, frames, ransac=(ITERS, THR, MIN_INL, 1), cfg=None, steps=T):
    """Step a fresh tracker through `frames`; per step (survivors, track lists, stage results or None)."""
    S = frames.shape[1]
    mt = ctx.multitracker(S, W, H, **(cfg or KW))
    if ransac is not None:
        mt.set_ransac(TEMPLE_K, *ransac)
    out = []
    for t in range(steps):
        surv = mt.step(frames[t])
        out.append((surv, [mt.tracks(s) for s in range(S)], mt.ransac_results() if ransac is not None else None))
    mt.close()
    return out


def _same_results(a, b):
    st, bn, inl, R, t = a
    st2, bn2, inl2, R2, t2 = b
    assert np.array_equal(st, st2) and np.array_equal(bn, bn2)
    for s in range(len(st)):
        assert np.array_equal(inl[s], inl2[s]), s
    ok = st == OK
    assert np.array_equal(R[ok], R2[ok]) and np.array_equal(t[ok], t2[ok])  # R, t are written for poses only


@pytest.mark.parametrize("solver_mode", [1, 3, 0])
@pytest.mark.parametrize("thr", [THR, 1e-6])
def test_stage_equals_find_E_ransac(ctx, checker, frames, thr, solver_mode):
    """Every sequence and step against find_E_ransac on the survivors the step returned: status, best_n and inlier list
    exactly, R and t within 1e-6.  thr 1e-6: no early hypothesis explains every survivor, every hypothesis is scored.
    The one exception to the R, t bound is a winning octet with a repeated index (sampling is with replacement): its design
    matrix has a two-dimensional null space, and which member the reference's Jacobi iteration returns is not reproduced
    bit for bit by the device solver (DESIGN.md §4) - the same inlier list, another E of that null space, another pose."""
    ctx.solver_set_mode(solver_mode)
    try:
        res = _run(ctx, frames, (ITERS, thr, MIN_INL, 1))
    finally:
        ctx.solver_set_mode(1)
    seen, repeated = [], 0
    for t, (surv, _, (st, bn, inl, R, tt)) in enumerate(res):
        for s, (prev, cur, _) in enumerate(surv):
            seen.append(int(st[s]))
            if len(prev) == 0:  # the first step, or no survivors: find_E_ransac is not called (:1715)
                assert st[s] == 0 and bn[s] == 0, (t, s)
                continue
            r = checker.find_E_ransac(TEMPLE_K, prev, cur, ITERS, thr, MIN_INL)
            if r is None:
                assert st[s] == 1, (t, s, st[s])
                continue
            wR, wt, winl = r
            assert st[s] == OK and bn[s] == len(winl) and np.array_equal(inl[s], winl), (t, s, st[s], bn[s], len(winl))
            if np.abs(R[s] - wR).max() >= 1e-6 or np.abs(tt[s] - wt).max() >= 1e-6:
                xi, xj = checker.norm_points(TEMPLE_K, prev), checker.norm_points(TEMPLE_K, cur)
                E, idx = checker.ransac_hypotheses(xi, xj, ITERS)
                wbh = checker.ransac_score(xi, xj, E, thr)[1]
                assert len(set(idx[wbh])) < 8, (t, s, np.abs(R[s] - wR).max())
                repeated += 1
    print(f"thr {thr} mode {solver_mode}: {repeated} of {seen.count(OK)} poses from a repeated-index winning octet")
    assert repeated <= seen.count(OK) // 4
    assert all(st == 0 for st in res[0][2][0])
    assert seen.count(0) >= frames.shape[1] and seen.count(1) >= 1 and seen.count(2) >= 5, seen


def test_stage_equals_pairs_stage(ctx, frames):
    """The same survivors through sfmgpu_pairs (set_matches + ransac, the same S, capacity and configuration): every output
    bit for bit - one stage serves both."""
    S = frames.shape[1]
    mt = ctx.multitracker(S, W, H, **KW)
    mt.set_ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)
    pairs = ctx.pairs(S, mt.cap)
    for t in range(T):
        surv = mt.step(frames[t])
        got = mt.ransac_results()
        pairs.set_matches([o[0] for o in surv], [o[1] for o in surv])
        pairs.ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)
        st, bn = np.zeros(S, np.int32), np.zeros(S, np.int32)
        inl, R, tt = np.zeros((S, mt.cap), np.int32), np.zeros((S, 9)), np.zeros((S, 3))
        pairs.ransac_download_all(st, bn, inl, R, tt)
        _same_results(got, (st, bn, [inl[s, :bn[s]] for s in range(S)], R.reshape(S, 3, 3), tt))
        assert t == 0 or (st == OK).sum() >= 2, t


def test_early_stop_is_exact(ctx, frames):
    """Stop on against stop off in tracker mode: identical results, and sets do stop early at the reference's threshold."""
    res, stopped = {}, {}
    try:
        for early in (1, 0):
            ctx.ransac_set_early_stop(early)
            S = frames.shape[1]
            mt = ctx.multitracker(S, W, H, **KW)
            mt.set_ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)
            mt.ransac_early()
            res[early] = []
            for t in range(T):
                mt.step(frames[t])
                res[early].append(mt.ransac_results())
            stopped[early] = mt.ransac_early()
    finally:
        ctx.ransac_set_early_stop(1)
    assert stopped[0] == 0 and stopped[1] > 0, stopped
    for a, b in zip(res[1], res[0]):
        _same_results(a, b)


@pytest.mark.parametrize("cfg", [KW, dict(max_tracks=120, min_tracks=100, fb_thresh=-1.0)], ids=["replenish", "total_loss"])
def test_stage_changes_nothing_else(ctx, frames, cfg):
    """Survivors, ids and track lists (replenishment included) equal those of a tracker without the stage, step by step.
    fb_thresh = -1 drops every track in every step: every set is SKIPPED."""
    on, off = _run(ctx, frames, cfg=cfg), _run(ctx, frames, ransac=None, cfg=cfg)
    for t, (a, b) in enumerate(zip(on, off)):
        for s in range(frames.shape[1]):
            for x, y in zip(a[0][s], b[0][s]):
                assert np.array_equal(x, y), (t, s)
            for x, y in zip(a[1][s], b[1][s]):
                assert np.array_equal(x, y), (t, s)
        if cfg.get("fb_thresh") == -1.0:
            assert (a[2][0] == 0).all() and (a[2][1] == 0).all(), t
    # replenishment happened: a track list longer than the step's survivors
    assert any(len(on[t][1][s][1]) > len(on[t][0][s][2]) for t in range(1, T) for s in range(frames.shape[1]))


def test_pipelined_step_equals_plain(ctx, frames):
    S = frames.shape[1]
    stack = ctx.pinned_empty(frames.shape, np.uint8)
    stack[:] = frames
    plain, piped = ctx.multitracker(S, W, H, **KW), ctx.multitracker(S, W, H, **KW)
    for mt in (plain, piped):
        mt.set_ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)
    piped.prefetch(stack[0])
    for t in range(T):
        want = plain.step(stack[t])
        got = piped.step(None, next_imgs=stack[t + 1] if t + 1 < T else None)
        for s in range(S):
            for a, b in zip(got[s], want[s]):
                assert np.array_equal(a, b), (t, s)
        _same_results(piped.ransac_results(), plain.ransac_results())


def test_no_stale_results(ctx, frames):
    """After reset() and after a step with the stage off the download refuses; the first step after reset() is all SKIPPED."""
    S = frames.shape[1]
    mt = ctx.multitracker(S, W, H, **KW)
    mt.set_ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)
    for t in range(3):
        mt.step(frames[t])
    assert (mt.ransac_results()[0] == OK).sum() >= 2
    mt.reset()
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        mt.ransac_results()
    assert e.value.code == -4
    mt.step(frames[0])
    st, bn, inl, _, _ = mt.ransac_results()
    assert (st == 0).all() and (bn == 0).all() and all(len(x) == 0 for x in inl)
    mt.step(frames[1])
    assert (mt.ransac_results()[0] == OK).sum() >= 2
    mt.set_ransac(TEMPLE_K, ITERS, THR, MIN_INL, 1)  # a new configuration: nothing to download until the next step
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        mt.ransac_results()
    assert e.value.code == -4
    mt.set_ransac(None)
    mt.step(frames[2])
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        mt.ransac_results()
    assert e.value.code == -4


def test_errors(ctx, frames):
    S = frames.shape[1]
    mt = ctx.multitracker(S, W, H, **KW)
    with pytest.raises(sfmgpu.SfmGpuError, match="Singular K"):
        mt.set_ransac(np.zeros((3, 3)))
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        mt.set_ransac(TEMPLE_K, iters=-1)
    assert e.value.code == -1
    mt.set_ransac(TEMPLE_K)
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        mt.ransac_results()  # no step yet
    assert e.value.code == -4


def _shim_tv():
    """libsfmshim_tv.so (tests/shim_two_view_capi.cpp): MultiKLTTracker with set_two_view behind flat C wrappers."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libsfmshim_tv.so")
    if not os.path.exists(path):
        sfmgpu.build_library()
    lib = C.CDLL(path)
    f8, i4 = np.ctypeslib.ndpointer(np.float64, flags="C"), np.ctypeslib.ndpointer(np.int32, flags="C")
    lib.shim_tv_last_error.restype = C.c_char_p
    lib.shim_tv_create.restype = C.c_void_p
    lib.shim_tv_create.argtypes = [C.c_int] * 5
    lib.shim_tv_destroy.argtypes = [C.c_void_p]
    lib.shim_tv_set_two_view.argtypes = [C.c_void_p, f8, C.c_int, C.c_double, C.c_int]
    lib.shim_tv_step.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.uint8, flags="C"), C.c_int, C.c_int, C.c_int, i4, i4, C.c_int, i4,
                                 f8, f8, i4, i4]
    return lib


def test_shim_multitracker_two_view(ctx, frames):
    """MultiKLTTracker::set_two_view: per sequence the same std::optional<RelPose> as the C ABI's results."""
    shim = _shim_tv()

    def ck(rc):
        if rc != 0:
            raise RuntimeError(shim.shim_tv_last_error().decode())

    S = frames.shape[1]
    cap = KW["max_tracks"] + 1
    h = shim.shim_tv_create(S, W, H, KW["max_tracks"], KW["min_tracks"])
    assert h, shim.shim_tv_last_error().decode()
    try:
        ck(shim.shim_tv_set_two_view(h, np.ascontiguousarray(TEMPLE_K.reshape(9)), ITERS, THR, MIN_INL))
        want = _run(ctx, frames)
        for t in range(T):
            ids, n = np.zeros((S, cap), np.int32), np.zeros(S, np.int32)
            has, n_inl = np.zeros(S, np.int32), np.zeros(S, np.int32)
            R, tt, inl = np.zeros((S, 9)), np.zeros((S, 3)), np.zeros((S, cap), np.int32)
            ck(shim.shim_tv_step(h, frames[t], S, W, H, ids, n, cap, has, R, tt, inl, n_inl))
            st, bn, winl, wR, wt = want[t][2]
            for s in range(S):
                assert np.array_equal(ids[s, :n[s]], want[t][0][s][2]), (t, s)
                assert has[s] == (st[s] == OK), (t, s)
                if has[s]:
                    assert np.array_equal(inl[s, :n_inl[s]], winl[s]), (t, s)
                    assert np.array_equal(R[s], wR[s].reshape(9)) and np.array_equal(tt[s], wt[s]), (t, s)
    finally:
        shim.shim_tv_destroy(h)
