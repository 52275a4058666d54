"""Segment mode (SURVEY.md §8e): contiguous segments of ONE resident sequence, each a fresh KLTTracker, run as lock-step tracker
slots that read their frames from an sfmgpu_frames batch (sfmgpu_multitracker_step_frames), with find_E_ransac(K, prev, cur,
2500, 1e-3, 60) (cpp/src/templering_sfm.cpp:1739) on every step's survivors, into the rows of a pairs object
(sfmgpu_pair_frontend_segments) with the track ids, and gathered by the scheduler.

Byte-for-byte comparisons between runs of different batch sizes pin the KLT kernel family (the lane and warp kernels agree to
~1e-13 px, and the automatic choice depends on the batch size) and the RANSAC solver mode (the screening solver is chosen by the
size of a launch set)."""
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
HERE = os.path.dirname(os.path.abspath(__file__))

W, H = 640, 480
KW = dict(max_tracks=400, min_tracks=380)  # replenishment in most steps
RANSAC = (2500, 1e-3, 60, 1)  # :1739, min_points 1 = the `prev_pts.empty()` guard (:1715)
OK = 2
ROWS = 401  # max(max_tracks, min_tracks, 1) + 1
E_ARG, E_STATE = -1, -4


@pytest.fixture(scope="module")
def ring():
    """Nine frames of the ray-cast ring scene from a camera moving along the ring (real two-view geometry)."""
    return np.stack([ring_dataset.render(np.deg2rad(2.0 + 0.25 * t), W, H) for t in range(9)])


@pytest.fixture(scope="module")
def noise():
    return np.stack([synth.frame(20261121, t, W, H) for t in range(9)])


@pytest.fixture
def pinned(ctx):
    """KLT lane kernel and Jacobi solver for every launch: results independent of batch sizes."""
    ctx.klt_set_mode(2)
    ctx.solver_set_mode(0)
    yield
    ctx.klt_set_mode(0)
    ctx.solver_set_mode(1)


def resident(ctx, imgs):
    f = ctx.frames(imgs.shape[2], imgs.shape[1], len(imgs), 3)
    f.upload(0, imgs)
    f.build_pyramid()
    return f


def run_segments(ctx, f, seg_first, steps, cfg, ransac=RANSAC, pairs=None):
    """Rows of a segment call: (nk, nc, li, lj, ids, stage results or None), li / lj / ids cut to n_kept per row."""
    P = len(seg_first) * steps
    p = pairs or ctx.pairs(max(P, 1), ROWS)
    if ransac is not None:
        p.set_ransac(TEMPLE_K, *ransac)
    p.run_segments(f, seg_first, steps, cfg)
    li, lj = np.zeros((P, p.cap, 2)), np.zeros((P, p.cap, 2))
    nk, nc = np.zeros(P, np.int32), np.zeros(P, np.int32)
    p.download_all(li, lj, nk, nc)
    ids = p.ids_download_all(P)
    tv = None
    if ransac is not None:
        st, bn, inl = np.zeros(P, np.int32), np.zeros(P, np.int32), np.zeros((P, p.cap), np.int32)
        R, t = np.zeros((P, 9)), np.zeros((P, 3))
        p.ransac_download_all(st, bn, inl, R, t)
        tv = (st, bn, [inl[r, :bn[r]] for r in range(P)], R, t)
    rows = [(li[r, :nk[r]], lj[r, :nk[r]], ids[r, :nk[r]]) for r in range(P)]
    return nk, nc, rows, tv


def separate_run(ctx, imgs, first, steps, cfg, ransac=RANSAC):
    """One segment through a host-fed one-sequence lock-step tracker: per step (n_corners, (prev, cur, ids), stage results)."""
    h, w = imgs.shape[1:]
    mt = ctx.multitracker(1, w, h, **cfg)
    if ransac is not None:
        mt.set_ransac(TEMPLE_K, *ransac)
    out = []
    for k in range(steps + 1):
        n_in = len(mt.tracks(0)[1])
        surv = mt.step(imgs[first + k][None])[0]
        if k:
            out.append((n_in, surv, mt.ransac_results() if ransac is not None else None))
    mt.close()
    return out


def assert_rows_equal(got, imgs, ctx, seg_first, steps, cfg, ransac=RANSAC, cache=None):
    nk, nc, rows, tv = got
    cache = {} if cache is None else cache
    for j, s0 in enumerate(seg_first):
        if s0 not in cache:
            cache[s0] = separate_run(ctx, imgs, s0, steps, cfg, ransac)
        for k, (n_in, surv, res) in enumerate(cache[s0]):
            r = j * steps + k
            assert nc[r] == n_in and nk[r] == len(surv[0]), (j, k, nc[r], n_in, nk[r], len(surv[0]))
            for a, b in zip(rows[r], surv):
                assert np.array_equal(a, b), (j, k)
            if ransac is not None:
                st, bn, inl, R, t = tv
                assert st[r] == res[0][0] and bn[r] == res[1][0] and np.array_equal(inl[r], res[2][0]), (j, k)
                if st[r] == OK:
                    assert np.array_equal(R[r], res[3][0].reshape(9)) and np.array_equal(t[r], res[4][0]), (j, k)


# ---- 1. step_frames equals step ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [KW, dict(max_tracks=120, min_tracks=100, fb_thresh=-1.0)], ids=["replenish", "total_loss"])
def test_step_frames_equals_step(ctx, ring, noise, cfg):
    """Three sequences over arbitrary (repeated, backwards) indices of a resident batch against host-fed steps of the same
    images: survivors, ids, track lists and stage results byte for byte.  fb_thresh = -1 loses every track in every step
    (replenishment refills the lists): every set is SKIPPED."""
    imgs = np.concatenate([ring, noise])
    f = resident(ctx, imgs)
    order = np.array([[0, 1, 2, 3, 4, 5, 6, 7], [17, 16, 15, 14, 13, 12, 11, 10], [2, 3, 3, 4, 9, 10, 4, 5]], np.int32)
    S, T = order.shape
    a, b = ctx.multitracker(S, W, H, **cfg), ctx.multitracker(S, W, H, **cfg)
    for mt in (a, b):
        mt.set_ransac(TEMPLE_K, *RANSAC)
    seen = []
    for t in range(T):
        got = a.step_frames(f, order[:, t])
        want = b.step(imgs[order[:, t]])
        for s in range(S):
            for x, y in zip(got[s], want[s]):
                assert np.array_equal(x, y), (t, s)
            for x, y in zip(a.tracks(s), b.tracks(s)):
                assert np.array_equal(x, y), (t, s)
        ra, rb = a.ransac_results(), b.ransac_results()
        assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[1], rb[1]), t
        for s in range(S):
            assert np.array_equal(ra[2][s], rb[2][s]), (t, s)
        ok = ra[0] == OK
        assert np.array_equal(ra[3][ok], rb[3][ok]) and np.array_equal(ra[4][ok], rb[4][ok]), t
        seen += list(ra[0])
    if cfg.get("fb_thresh") == -1.0:
        assert set(seen) == {0}
    else:
        assert seen.count(OK) >= 6, seen
        assert any(len(a.tracks(s)[1]) > len(got[s][2]) for s in range(S))  # the last step replenished


def test_step_frames_refusals(ctx, ring):
    """Refused before any work: the tracker then goes on exactly like one that never saw the bad calls."""
    f = resident(ctx, ring)
    small = ctx.frames(320, 240, 2, 3)
    two = ctx.frames(W, H, 2, 2)
    a, b = ctx.multitracker(2, W, H, **KW), ctx.multitracker(2, W, H, **KW)
    a.step_frames(f, [0, 1])
    b.step_frames(f, [0, 1])
    for bad in ([0, 9], [-1, 0]):
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            a.step_frames(f, bad)
        assert e.value.code == E_ARG
    for other in (small, two):
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            a.step_frames(other, [0, 1])
        assert e.value.code == E_ARG
    n = np.zeros(2, np.int32)
    assert ctx.lib.sfmgpu_multitracker_step_frames(ctx.h, a.h_, f.h_, None, None, None, None, n.ctypes.data_as(C.c_void_p)) == E_ARG
    a.prefetch(ring[[5, 6]])
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        a.step_frames(f, [1, 2])
    assert e.value.code == E_STATE
    got = a.step(None)  # consumes the prefetched frames 5, 6
    want = b.step_frames(f, [5, 6])
    for s in range(2):
        for x, y in zip(got[s], want[s]):
            assert np.array_equal(x, y), s
    got, want = a.step_frames(f, [6, 7]), b.step_frames(f, [6, 7])
    for s in range(2):
        for x, y in zip(got[s], want[s]):
            assert np.array_equal(x, y), s


# ---- 2. segments equal separate runs -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("seg_first,steps", [([0, 3, 3, 1, 4], 4), ([0, 7, 5, 7, 0], 1), ([2], 6)],
                         ids=["overlap_repeat_last", "one_step", "one_segment"])
def test_segments_equal_separate_runs(ctx, ring, pinned, seg_first, steps):
    """Overlapping and repeated segments, a segment ending on the last frame, steps = 1: every row equals the matching step
    of a separate tracker run of that segment, stage results included."""
    f = resident(ctx, ring)
    got = run_segments(ctx, f, seg_first, steps, sfmgpu.lkcfg(**KW))
    assert_rows_equal(got, ring, ctx, seg_first, steps, KW)
    st = got[3][0]
    assert (st == OK).sum() >= len(seg_first) * steps // 2, st


def test_segments_total_loss(ctx, noise, pinned):
    """fb_thresh = -1 loses every track in every step (replenishment refills the list): no survivors, every row SKIPPED by
    min_points = 1, as in separate runs."""
    cfg = dict(max_tracks=120, min_tracks=100, fb_thresh=-1.0)
    f = resident(ctx, noise)
    got = run_segments(ctx, f, [0, 2], 4, sfmgpu.lkcfg(**cfg), pairs=ctx.pairs(8, 121))
    nk, nc, _, tv = got
    assert (nk == 0).all() and (nc == 120).all() and (tv[0] == 0).all(), (nk, nc, tv[0])
    assert_rows_equal(got, noise, ctx, [0, 2], 4, cfg)


def test_segments_more_than_one_lock_step(ctx, pinned):
    """601 segments at 160 x 120: more than the 512 slots of one lock step, so two chunks of 301 slots, the last one with a
    spare slot.  Segments repeat (nine distinct starts), so one separate run per start is the reference for every row."""
    w, h, N, steps = 160, 120, 12, 3
    imgs = np.stack([synth.frame(20261122, t, w, h) for t in range(N)])
    f = resident(ctx, imgs)
    seg_first = [(5 * j) % 7 + (j % 3) for j in range(601)]
    cfg = dict(max_tracks=150, min_tracks=140)
    p = ctx.pairs(601 * steps, 151)
    p.set_ransac(TEMPLE_K, *RANSAC)
    p.run_segments(f, seg_first, steps, sfmgpu.lkcfg(**cfg))
    P = 601 * steps
    li, lj = np.zeros((P, 151, 2)), np.zeros((P, 151, 2))
    nk, nc = np.zeros(P, np.int32), np.zeros(P, np.int32)
    p.download_all(li, lj, nk, nc)
    ids = p.ids_download_all(P)
    st, bn = np.zeros(P, np.int32), np.zeros(P, np.int32)
    p.ransac_download_all(st, bn)
    ref = {s0: separate_run(ctx, imgs, s0, steps, cfg) for s0 in sorted(set(seg_first))}
    for j, s0 in enumerate(seg_first):
        for k, (n_in, surv, res) in enumerate(ref[s0]):
            r = j * steps + k
            assert nc[r] == n_in and nk[r] == len(surv[0]), (j, k)
            assert np.array_equal(li[r, :nk[r]], surv[0]) and np.array_equal(lj[r, :nk[r]], surv[1]), (j, k)
            assert np.array_equal(ids[r, :nk[r]], surv[2]), (j, k)
            assert st[r] == res[0][0] and bn[r] == res[1][0], (j, k)


# ---- 3. segments against the checker ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene", ["ring", "noise"])
def test_segments_against_checker(ctx, checker, ring, noise, scene):
    """Per segment a fresh checker KLTTracker and find_E_ransac on every step's survivors: ids and counts exact, positions
    within 1e-3 px, status / best_n / inlier list exact, R and t within 1e-6 except for a winning octet with a repeated index
    (see tests/test_gpu_multitracker_two_view.py: another member of a two-dimensional null space)."""
    imgs = ring if scene == "ring" else noise
    seg_first, steps = [0, 2, 4], 4
    f = resident(ctx, imgs)
    nk, nc, rows, (st, bn, inl, R, t) = run_segments(ctx, f, seg_first, steps, sfmgpu.lkcfg(**KW))
    iters, thr, min_inl, _ = RANSAC
    oks = repeated = 0
    for j, s0 in enumerate(seg_first):
        tr = checker.tracker(**KW)
        tr.step(imgs[s0])
        for k in range(steps):
            r = j * steps + k
            n_in = len(tr.tracks()[1])
            prev, cur, ids = tr.step(imgs[s0 + k + 1])
            assert nc[r] == n_in and nk[r] == len(ids) and np.array_equal(rows[r][2], ids), (j, k)
            assert np.abs(rows[r][0] - prev).max(initial=0) <= 1e-3 and np.abs(rows[r][1] - cur).max(initial=0) <= 1e-3, (j, k)
            if len(prev) == 0:
                assert st[r] == 0 and bn[r] == 0, (j, k)
                continue
            res = checker.find_E_ransac(TEMPLE_K, prev, cur, iters, thr, min_inl)
            if res is None:
                assert st[r] == 1, (j, k, st[r])
                continue
            wR, wt, winl = res
            assert st[r] == OK and bn[r] == len(winl) and np.array_equal(inl[r], winl), (j, k)
            oks += 1
            if np.abs(R[r] - wR.reshape(9)).max() >= 1e-6 or np.abs(t[r] - wt).max() >= 1e-6:
                xi, xj = checker.norm_points(TEMPLE_K, prev), checker.norm_points(TEMPLE_K, cur)
                E, idx = checker.ransac_hypotheses(xi, xj, iters)
                assert len(set(idx[checker.ransac_score(xi, xj, E, thr)[1]])) < 8, (j, k)
                repeated += 1
    assert oks >= 6 and repeated <= oks // 4, (oks, repeated)


# ---- 4. readers and refusals ------------------------------------------------------------------------------------------------
def test_readers_and_gather(ctx, ring, pinned):
    f = resident(ctx, ring)
    seg_first, steps = [0, 4, 1], 4
    P = len(seg_first) * steps
    p = ctx.pairs(P, ROWS)
    nk, nc, rows, (st, bn, inl, R, t) = run_segments(ctx, f, seg_first, steps, sfmgpu.lkcfg(**KW), pairs=p)
    corners, kept, iters = p.totals()
    assert corners == nc.sum() and kept == nk.sum() and iters >= kept
    for r in range(P):
        li, lj, n_corn = p.download(r)
        assert n_corn == nc[r] and np.array_equal(li, rows[r][0]) and np.array_equal(lj, rows[r][1])
        s1, _, inl1, _, R1, t1 = p.ransac_download(r)
        assert s1 == st[r] and np.array_equal(inl1, inl[r])
        if s1 == OK:
            assert np.array_equal(R1.reshape(9), R[r]) and np.array_equal(t1, t[r])
    # world = 1: the gathers are local copies of the same rows
    lib, vp = ctx.lib, (lambda x: x.ctypes.data_as(C.c_void_p))
    s = C.c_void_p()
    ctx._ck(lib.sfmgpu_sched_create(ctx.h, 1, 0, None, None, C.byref(s)))
    try:
        gli, glj = np.zeros((P, ROWS, 2)), np.zeros((P, ROWS, 2))
        gnk, gnc, gst, gbn = (np.zeros(P, np.int32) for _ in range(4))
        ginl, gR, gt = np.zeros((P, ROWS), np.int32), np.zeros((P, 9)), np.zeros((P, 3))
        gids = np.zeros((P, ROWS), np.int32)
        ctx._ck(lib.sfmgpu_sched_gather_pairs(ctx.h, s, p.h_, P, 0, 1, vp(gli), vp(glj), vp(gnk), vp(gnc), vp(gst), vp(gbn), vp(ginl),
                                              vp(gR), vp(gt)))
        ctx._ck(lib.sfmgpu_sched_gather_pair_ids(ctx.h, s, p.h_, P, 0, vp(gids)))
        assert np.array_equal(gnk, nk) and np.array_equal(gnc, nc) and np.array_equal(gst, st) and np.array_equal(gbn, bn)
        for r in range(P):
            n = nk[r]
            assert np.array_equal(gli[r, :n], rows[r][0]) and np.array_equal(glj[r, :n], rows[r][1])
            assert np.array_equal(gids[r, :n], rows[r][2]) and np.array_equal(ginl[r, :bn[r]], inl[r])
        ok = st == OK
        assert np.array_equal(gR[ok], R[ok]) and np.array_equal(gt[ok], t[ok])
        assert lib.sfmgpu_sched_gather_pair_ids(ctx.h, s, p.h_, P + 1, 0, vp(gids)) == E_ARG  # block size mismatch
        # ids belong to segment calls only
        ptr = C.c_void_p()
        assert lib.sfmgpu_pairs_ids_device_ptr(p.h_, C.byref(ptr)) == 0 and ptr.value
        p.set_ransac(None)
        p.run(f, 0, 3, sfmgpu.lkcfg(max_tracks=ROWS))
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            p.ids_download_all(3)
        assert e.value.code == E_STATE
        assert lib.sfmgpu_pairs_ids_device_ptr(p.h_, C.byref(ptr)) == E_STATE
        assert lib.sfmgpu_sched_gather_pair_ids(ctx.h, s, p.h_, 3, 0, vp(gids)) == E_STATE
    finally:
        lib.sfmgpu_sched_destroy(ctx.h, s)


def test_segment_refusals(ctx, ring):
    """Every E_ARG case is reported before any work: the previous batch (rows, ids) is still what the readers return."""
    f = resident(ctx, ring)
    cfg = sfmgpu.lkcfg(**KW)
    p = ctx.pairs(8, ROWS)
    p.run_segments(f, [0, 2], 3, cfg)
    nk0, ids0 = np.zeros(6, np.int32), p.ids_download_all(6).copy()
    p.download_all(None, None, nk0, None)
    bad = [([0, 6], 3, cfg, p),  # 6 + 3 >= 9 frames
           ([0, -1], 3, cfg, p),
           ([0, 1, 2], 3, cfg, p),  # 9 rows > max_pairs 8
           ([0], 0, cfg, p),  # steps < 1
           ([0], 3, sfmgpu.lkcfg(pyr_levels=2, **KW), p),  # cfg does not match f
           ([0], 3, cfg, ctx.pairs(8, ROWS - 1))]  # rows narrower than a track list
    for seg_first, steps, c, q in bad:
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            q.run_segments(f, seg_first, steps, c)
        assert e.value.code == E_ARG, (seg_first, steps)
    assert ctx.lib.sfmgpu_pair_frontend_segments(ctx.h, f.h_, None, 2, 3, C.byref(cfg), p.h_) == E_ARG
    nk1 = np.zeros(6, np.int32)
    p.download_all(None, None, nk1, None)
    assert np.array_equal(nk1, nk0) and np.array_equal(p.ids_download_all(6), ids0)
    # the segment's last frame may be the batch's last
    p.run_segments(f, [5], 3, cfg)


# ---- multi-rank ---------------------------------------------------------------------------------------------------------------
def test_segments_cpp_program():
    """tests/segments_test: one host thread per GPU runs its block of segments, rank 0 gathers rows, ids and stage results over
    NCCL and compares them byte for byte with a one-GPU run of all segments (one rank on a one-GPU machine)."""
    exe = os.path.join(HERE, "segments_test")
    assert os.path.exists(exe), "tests/segments_test is missing: run __graft_entry__.build()"
    r = subprocess.run([exe, "2", "40", "8"], capture_output=True, text=True, timeout=900)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "OK" in r.stdout
