"""GPU parity tests: the CUDA path (through the C ABI) against the CPU checker (compiled reference when
oracle/_ref is present, else the port) and against the committed golden vectors.

Bars (BASELINE.json north_star): pyramid bytes, corner candidates, corners, NMS survivors, std::sort permutation,
inlier counts / winner / mask: BIT-EXACT.  KLT positions: within 1e-3 px (KLT_TOL); measured deviation is ~1e-11.
"""
import os

import numpy as np
import pytest

from conftest import TEMPLE_K, two_view_scene, triangulation_scene
from sfmgpu import synth
import sfmgpu

pytestmark = pytest.mark.gpu
KLT_TOL = 1e-3  # px, the tolerance north_star states
W, H, SEED = 320, 240, 20261018


def _images():
    rng = np.random.default_rng(3)
    return {
        "kat": synth.kat_image(320, 200),
        "synth": synth.frame(11, 0, 320, 240),
        "ties": (synth.frame(12, 0, 200, 160) >> 4 << 4),
        "noise_odd": rng.integers(0, 256, (97, 131), dtype=np.uint8),
        "flat": np.full((24, 40), 77, np.uint8),
        "tiny": rng.integers(0, 256, (4, 9), dtype=np.uint8),
        "one_bright": np.pad(np.full((1, 1), 255, np.uint8), 20),
        "wide": synth.frame(13, 5, 700, 90),
    }


def _frames(ctx, imgs, levels=3):
    imgs = [np.ascontiguousarray(i) for i in imgs]
    f = ctx.frames(imgs[0].shape[1], imgs[0].shape[0], len(imgs), levels)
    f.upload(0, np.stack(imgs))
    f.build_pyramid()
    return f


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "frontend_golden.npz"))


# ---- synthetic generator ----------------------------------------------------------------------------------
def test_device_generator_matches_numpy(ctx):
    for (w, h) in [(320, 240), (333, 77)]:
        f = ctx.frames(w, h, 4, 1)
        f.synth(0, 4, 77, 62)  # covers the triangle-wave turn at t = 64
        for k in range(4):
            assert np.array_equal(f.download(k, 0), synth.frame(77, 62 + k, w, h))


# ---- pyramid -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(_images()))
@pytest.mark.parametrize("levels", [1, 2, 3, 4, 5])
def test_pyramid(ctx, checker, name, levels):
    img = _images()[name]
    f = _frames(ctx, [img, img[::-1].copy()], levels)
    for k, im in enumerate([img, img[::-1].copy()]):
        want = checker.build_pyr(im, levels)
        for l in range(levels):
            got = f.download(k, l)
            assert got.shape == want[l].shape and np.array_equal(got, want[l]), (name, k, l)


def test_pyramid_golden(ctx, g):
    f = _frames(ctx, [synth.frame(SEED, 0, W, H)])
    assert np.array_equal(f.download(0, 1), g["pyr_l1"]) and np.array_equal(f.download(0, 2), g["pyr_l2"])


# ---- corners -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(_images()))
def test_candidates_bit_exact(ctx, port, name):
    img = _images()[name]
    f = _frames(ctx, [img], 1)
    for q in (0.01, 0.3, 0.0, 1.0):
        xy, s, mx = f.candidates(0, q)
        wxy, ws, wmx = port.candidates(img, q)
        assert mx == wmx, (name, q)
        assert np.array_equal(xy, wxy) and np.array_equal(s.view(np.uint64), ws.view(np.uint64)), (name, q)


@pytest.mark.parametrize("n,distinct", [(0, 1), (1, 1), (16, 2), (17, 2), (33, 1), (1000, 3), (2049, 5), (5000, 40), (70000, 200),
                                        (70000, 10**6), (300000, 1000)])
def test_device_std_sort_permutation(ctx, port, n, distinct):
    rng = np.random.default_rng(n + distinct)
    for variant in range(3):
        keys = rng.integers(0, distinct, n).astype(np.float64)
        if variant == 1:
            keys = np.sort(keys)[::-1].copy()
        if variant == 2:
            keys = np.sort(keys).copy()
        assert np.array_equal(ctx.sort_perm_desc(keys), port.sort_perm_desc(keys)), (n, distinct, variant)


@pytest.mark.parametrize("name", list(_images()))
@pytest.mark.parametrize("mc,q,d", [(2200, 0.01, 8), (50, 0.2, 3), (0, 0.01, 8), (300, 0.0, 1), (100, 0.01, 0), (4000, 0.001, 2),
                                    (500, 0.01, 25)])
@pytest.mark.parametrize("select_mode", [0, 1, 14, 20, 1064, 1300])
def test_corners_bit_exact(ctx, checker, name, mc, q, d, select_mode):
    """select_mode 0: bucket selection + exact introsort fallback on observable score ties; 1: introsort emulation;
    14 / 20: bucket selection with 14- / 20-bit order codes (equal codes everywhere: the exact-score path orders them;
    with 14 bits a bucket is a few codes wide); 1064 / 1300: gathers of 64 / 300 words (every bucket is oversized: walked
    in runs of its sub-buckets, or handed to the exact emulation where a sub-bucket alone is too large)."""
    img = _images()[name]
    f = _frames(ctx, [img], 1)
    ctx.select_set_mode(select_mode)
    try:
        got = f.corners(0, mc, q, d)
    finally:
        ctx.select_set_mode(0)
    want = checker.shi_tomasi(img, mc, q, d)
    assert got.shape == want.shape and np.array_equal(got, want), (name, mc, q, d, len(got), len(want))


@pytest.mark.parametrize("period,mc,d", [(32, 3000, 8), (48, 500, 3), (17, 20000, 0), (64, 8000, 12)])
def test_corners_periodic_image_ties(ctx, checker, period, mc, d):
    """A periodic image: every score occurs dozens of times, so std::sort's tie order decides the corners from the first
    candidate on (the bucket selection must hand every such frame to the exact emulation), next to tie-free frames in one
    batch."""
    rng = np.random.default_rng(period)
    cell = rng.integers(0, 256, (period, period), dtype=np.uint8)
    w, h = 1280, 720
    img = np.tile(cell, (h // period + 1, w // period + 1))[:h, :w]
    mixed = img.copy()
    mixed[:, w // 2:] = synth.frame(3, 1, w, h)[:, w // 2:]  # ties only in the left half
    plain = synth.frame(4, 2, w, h)
    f = _frames(ctx, [img, plain, mixed], 1)
    for k, im in enumerate([img, plain, mixed]):
        got, want = f.corners(k, mc, 0.01, d), checker.shi_tomasi(im, mc, 0.01, d)
        assert got.shape == want.shape and np.array_equal(got, want), (period, k, len(got), len(want))


def test_corners_golden(ctx, g):
    f0 = synth.frame(SEED, 0, W, H)
    f = _frames(ctx, [f0, f0 >> 4 << 4, synth.kat_image(W, H)], 1)
    assert np.array_equal(f.corners(0, 400), g["corners"])
    assert np.array_equal(f.corners(1, 400), g["corners_ties"])
    assert np.array_equal(f.corners(2, 600), g["corners_kat"])


def test_corners_larger_image(ctx, checker):
    img = synth.frame(5, 9, 1280, 720)
    f = _frames(ctx, [img], 1)
    assert np.array_equal(f.corners(0, 3000), checker.shi_tomasi(img, 3000))


# ---- KLT ---------------------------------------------------------------------------------------------------------
def _klt_close(a, b):
    ok = np.array_equal(np.isnan(a), np.isnan(b)) and np.nanmax(np.abs(a - b), initial=0.0) <= KLT_TOL
    if not ok and a.shape == b.shape:
        bad = np.flatnonzero((np.isnan(a) != np.isnan(b)).any(1) | (np.nan_to_num(np.abs(a - b), nan=0.0) > KLT_TOL).any(1))
        print(f"KLT mismatch at {len(bad)} of {len(a)} points, first: " + "; ".join(f"#{i} got {a[i]} want {b[i]}" for i in bad[:6]))
    return ok


@pytest.mark.parametrize("lv,r,it", [(3, 5, 10), (1, 3, 4), (4, 2, 7), (2, 7, 3), (3, 10, 2)])
def test_klt_positions(ctx, checker, lv, r, it):
    rng = np.random.default_rng(5)
    f0, f1 = synth.frame(21, 0, 320, 240), synth.frame(21, 3, 320, 240)
    pts = np.concatenate([checker.shi_tomasi(f0, 150), rng.uniform(-8, 330, (80, 2)) * [1, 0.75],
                          [[0.0, 0.0], [318.0, 238.0], [319.5, 100.25], [127.99999999999999, 64.0], [1e12, 5.0],
                           [np.nan, 3.0], [-1e300, 1e300]]])
    f = _frames(ctx, [f0, f1], lv)
    p1, pb, nit = f.klt_track(0, 1, pts, r, it, count=True)
    w1, wb = checker.klt_track(f0, f1, pts, lv, r, it)
    assert _klt_close(p1, w1) and _klt_close(pb, wb)
    dev = max(np.nanmax(np.abs(p1[:230] - w1[:230])), np.nanmax(np.abs(pb[:230] - wb[:230])))
    print(f"klt max deviation {dev:.3e} px")
    assert dev < 1e-6  # far inside the budget; a regression here means the arithmetic changed


def test_klt_noise_images(ctx, checker):
    rng = np.random.default_rng(8)
    n0, n1 = rng.integers(0, 256, (200, 300), dtype=np.uint8), rng.integers(0, 256, (200, 300), dtype=np.uint8)
    pts = rng.uniform(0, 300, (300, 2)) * [1, 0.66]
    f = _frames(ctx, [n0, n1], 3)
    p1, pb = f.klt_track(0, 1, pts)
    w1, wb = checker.klt_track(n0, n1, pts)
    assert _klt_close(p1, w1) and _klt_close(pb, wb)


def test_klt_golden(ctx, g):
    f = _frames(ctx, [synth.frame(SEED, 0, W, H), synth.frame(SEED, 1, W, H)])
    p1, pb = f.klt_track(0, 1, g["corners"].astype(np.float64)[:200])
    assert _klt_close(p1, g["klt_p1"]) and _klt_close(pb, g["klt_pb"])


def test_klt_iteration_count(ctx, port):
    f0, f1 = synth.frame(21, 0, 320, 240), synth.frame(21, 1, 320, 240)
    pts = port.shi_tomasi(f0, 100)
    f = _frames(ctx, [f0, f1])
    _, _, nit = f.klt_track(0, 1, pts, count=True)
    _, _, want = port.klt_track(f0, f1, pts, count=True)
    assert np.array_equal(nit, want)


@pytest.mark.parametrize("mode", [1, 2, 13])
def test_klt_kernel_modes(ctx, checker, port, mode):
    """The KLT kernels (1: warp-per-feature; 2: lane-per-feature with quadratic forms over integer matrices + deferred border
    features; 13: lane-per-feature with the FP64 window walk) against the checker on
    the same points, including border, out-of-image and non-finite ones; iteration counts must be identical."""
    rng = np.random.default_rng(15)
    f0, f1 = synth.frame(21, 0, 320, 240), synth.frame(21, 3, 320, 240)
    pts = np.concatenate([checker.shi_tomasi(f0, 400), rng.uniform(-8, 330, (200, 2)) * [1, 0.75],
                          [[0.0, 0.0], [318.0, 238.0], [319.5, 100.25], [127.99999999999999, 64.0], [1e12, 5.0],
                           [np.nan, 3.0], [-1e300, 1e300], [160.0, 120.0], [7.0, 7.0], [28.0, 28.0], [27.999, 120.0]]])
    f = _frames(ctx, [f0, f1], 3)
    ctx.klt_set_mode(mode)
    try:
        p1, pb, nit = f.klt_track(0, 1, pts, count=True)
        q1, _ = f.klt_track(0, 1, pts[:77])  # ragged tail of a warp
    finally:
        ctx.klt_set_mode(0)
    w1, wb = checker.klt_track(f0, f1, pts)
    _, _, wn = port.klt_track(f0, f1, pts, count=True)
    assert _klt_close(p1, w1) and _klt_close(pb, wb) and _klt_close(q1, w1[:77])
    assert np.array_equal(nit, wn)
    dev = max(np.nanmax(np.abs(p1[:600] - w1[:600])), np.nanmax(np.abs(pb[:600] - wb[:600])))
    print(f"klt mode {mode} max deviation {dev:.3e} px")
    assert dev < 1e-6


def test_klt_large_batch_takes_the_lane_kernel(ctx, checker):
    """>= 6000 features in one launch: automatic selection of the lane-per-feature kernel (1280x720, 7000 corners)."""
    f0, f1 = synth.frame(31, 0, 1280, 720), synth.frame(31, 2, 1280, 720)
    f = _frames(ctx, [f0, f1], 3)
    rng = np.random.default_rng(16)
    pts = np.concatenate([f.corners(0, 7000), rng.uniform(0, 1280, (6500, 2)) * [1, 0.5625]])
    n0 = ctx.launches()
    p1, pb = f.klt_track(0, 1, pts)
    assert ctx.launches() - n0 == 3  # lane kernel (interior) + masked lane kernel (border) + warp-per-feature (rest)
    sel = np.r_[0:1500, len(pts) - 1500:len(pts)]
    w1, wb = checker.klt_track(f0, f1, pts[sel])
    assert _klt_close(p1[sel], w1) and _klt_close(pb[sel], wb)
    ctx.klt_set_mode(1)
    try:
        r1, rb = f.klt_track(0, 1, pts)
    finally:
        ctx.klt_set_mode(0)
    dev = max(np.abs(p1 - r1).max(), np.abs(pb - rb).max())
    print(f"lane vs warp kernel max difference {dev:.3e} px over {len(pts)} features")
    assert dev < 1e-6


# ---- stateful tracker ---------------------------------------------------------------------------------------------
def test_tracker_sequence(ctx, checker):
    kw = dict(max_tracks=150, min_tracks=120, quality=0.01, min_distance=8, levels=3, radius=5, iters=10, fb=1.0)
    want = checker.tracker(**kw)
    got = ctx.tracker(max_tracks=150, min_tracks=120)
    for t in [0, 1, 2, 40, 41, 42]:
        img = synth.frame(SEED, t, W, H)
        wp, wc, wi = want.step(img)
        gp, gc, gi = got.step(img)
        assert np.array_equal(gi, wi), t
        assert _klt_close(gp, wp) and _klt_close(gc, wc), t
        wxy, wid = want.tracks()
        gxy, gid = got.tracks()
        assert np.array_equal(gid, wid) and _klt_close(gxy, wxy), t


def test_tracker_resident_frames_equals_host_fed(ctx):
    imgs = [synth.frame(SEED, t, W, H) for t in range(4)]
    f = _frames(ctx, imgs)
    a, b = ctx.tracker(max_tracks=150, min_tracks=120), ctx.tracker(max_tracks=150, min_tracks=120)
    for k, img in enumerate(imgs):
        ra, rb = a.step(img), b.step_frames(f, k)
        for x, y in zip(ra, rb):
            assert np.array_equal(x, y)


def test_multitracker_equals_separate_trackers(ctx, checker):
    """BASELINE.json config C5 in lock step: S sequences advanced by ONE batched launch per stage equal S separate
    KLTTracker twins step by step (survivors, ids, track lists incl. replenishment), and the reference tracker."""
    S, T = 5, 7
    seqs = [[synth.frame(200 + s, t, W, H) for t in range(T)] for s in range(S)]
    seqs[3] = [f >> 3 << 3 for f in seqs[3]]  # a sequence with many identical scores
    kw = dict(max_tracks=150, min_tracks=140)  # replenishment triggers within a few frames
    mt = ctx.multitracker(S, W, H, **kw)
    singles = [ctx.tracker(**kw) for _ in range(S)]
    ref = checker.tracker(**kw)
    for t in range(T):
        got = mt.step(np.stack([seqs[s][t] for s in range(S)]))
        for s in range(S):
            want = singles[s].step(seqs[s][t])
            for a, b in zip(got[s], want):
                assert np.array_equal(a, b), (t, s)
            for a, b in zip(mt.tracks(s), singles[s].tracks()):
                assert np.array_equal(a, b), (t, s)
        r = ref.step(seqs[0][t])
        assert np.array_equal(got[0][2], r[2]) and _klt_close(got[0][1], r[1]), t
    assert mt.totals()[0] == sum(tr.totals()[0] for tr in singles)


def test_multitracker_pipelined_equals_plain(ctx):
    """Prefetching the next frames on the copy stream while a step computes does not change any result."""
    S, T = 4, 8
    kw = dict(max_tracks=150, min_tracks=140)
    stack = ctx.pinned_empty((T, S, H, W), np.uint8)
    for t in range(T):
        for s in range(S):
            stack[t, s] = synth.frame(400 + s, t, W, H)
    plain, piped = ctx.multitracker(S, W, H, **kw), ctx.multitracker(S, W, H, **kw)
    piped.prefetch(stack[0])
    for t in range(T):
        want = plain.step(stack[t])
        got = piped.step(None, next_imgs=stack[t + 1] if t + 1 < T else None)
        for s in range(S):
            for a, b in zip(got[s], want[s]):
                assert np.array_equal(a, b), (t, s)
            for a, b in zip(piped.tracks(s), plain.tracks(s)):
                assert np.array_equal(a, b), (t, s)
    with pytest.raises(sfmgpu.SfmGpuError):
        piped.step(None)  # nothing prefetched


def test_multitracker_total_track_loss(ctx):
    """Every track fails the forward-backward test in every step (fb_thresh = -1): the track lists drop to zero and are
    refilled by the replenish rule (:374-389) inside the same step, identically in the lock-step and the single tracker."""
    S, T = 3, 5
    seqs = [[synth.frame(300 + s, t, W, H) for t in range(T)] for s in range(S)]
    kw = dict(max_tracks=120, min_tracks=100, fb_thresh=-1.0)  # fb >= -1 for every finite fb: every track is dropped each step
    mt = ctx.multitracker(S, W, H, **kw)
    singles = [ctx.tracker(**kw) for _ in range(S)]
    for t in range(T):
        got = mt.step(np.stack([seqs[s][t] for s in range(S)]))
        for s in range(S):
            want = singles[s].step(seqs[s][t])
            for a, b in zip(got[s], want):
                assert np.array_equal(a, b), (t, s)
            for a, b in zip(mt.tracks(s), singles[s].tracks()):
                assert np.array_equal(a, b), (t, s)


def test_c5_sequences_in_parallel(ctx):
    """BASELINE.json config C5 (several independent sequences per GPU): one context + tracker + host thread per
    sequence; the results equal the one-by-one run."""
    from sfmgpu import sched
    seqs = [[synth.frame(100 + s, t, W, H) for t in range(5)] for s in range(4)]
    kw = dict(max_tracks=150, min_tracks=120)
    par = sched.run_sequences(seqs, 0, kw, max_workers=4, lockstep=False)
    lock = sched.run_sequences(seqs, 0, kw)
    for s, seq in enumerate(seqs):
        trk = ctx.tracker(**kw)
        for t, img in enumerate(seq):
            want = trk.step(img)
            for a, b, c in zip(par[s][t], want, lock[s][t]):
                assert np.array_equal(a, b) and np.array_equal(c, b), (s, t)


# ---- RANSAC scoring ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,H", [(300, 40), (2200, 250), (10000, 64), (9, 3), (513, 129)])
def test_ransac_counts_bit_exact(ctx, checker, port, n, H):
    pi, pj = two_view_scene(n, seed=n + H)
    xi, xj = port.norm_points(TEMPLE_K, pi), port.norm_points(TEMPLE_K, pj)
    E, _ = checker.ransac_hypotheses(xi, xj, H)
    for thr in (1e-3, 2e-3, 1e-6, 0.0, 1e3):
        counts, bh, inl = ctx.ransac_score(xi, xj, E, thr)
        wc, wb, wi = checker.ransac_score(xi, xj, E, thr)
        assert np.array_equal(counts, wc) and bh == wb and np.array_equal(inl, wi), (n, H, thr)


def test_ransac_counts_c4_full_scale(ctx, checker):
    """BASELINE.json C4 at its largest point: 65,536 hypotheses x 10,000 correspondences, hypotheses from the reference's own
    seeded sampler + eight_point_E (cycled: the solver costs 24 us each on the host), every count against the reference's
    sampson_err loop on all host threads."""
    n, H, Hu = 10000, 65536, 2048
    pi, pj = two_view_scene(n)
    xi, xj = checker.norm_points(TEMPLE_K, pi), checker.norm_points(TEMPLE_K, pj)
    Eu, _ = checker.ransac_hypotheses(xi, xj, Hu)
    # 32 scaled copies: scaling E by s scales numerator^2 and denominator by s^2 except for the +1e-12, so counts differ
    # slightly from copy to copy and every copy exercises different roundings
    scales = np.repeat(1.0 + 0.37 * np.arange(H // Hu), Hu)[:, None]
    E = np.ascontiguousarray(np.tile(Eu, (H // Hu, 1)) * scales)
    counts, bh, inl = ctx.ransac_score(xi, xj, E, 1e-3)
    want = checker.ransac_score_mt(xi, xj, E, 1e-3, os.cpu_count() or 1)
    assert np.array_equal(counts, want)
    wbh = int(np.argmax(want)) if want.max() > 0 else -1
    assert bh == wbh and len(inl) == want[wbh]


def test_ransac_threshold_band_takes_the_literal_division(ctx, port):
    # thresholds placed exactly ON computed errors: the division-free screen must hand over to the exact test
    pi, pj = two_view_scene(400, seed=4)
    xi, xj = port.norm_points(TEMPLE_K, pi), port.norm_points(TEMPLE_K, pj)
    E, _ = port.ransac_hypotheses(xi, xj, 8)
    for h in range(8):
        e = np.array([port.sampson(E[h], xi[i], xj[i]) for i in range(0, 400, 37)])
        for thr in e:
            for t in (thr, np.nextafter(thr, 0), np.nextafter(thr, 1)):
                counts, bh, inl = ctx.ransac_score(xi, xj, E, float(t))
                wc, wb, wi = port.ransac_score(xi, xj, E, float(t))
                assert np.array_equal(counts, wc) and bh == wb and np.array_equal(inl, wi)


@pytest.mark.parametrize("scale_pts,scale_e", [(1.0, 1.0), (1520.0, 1.0), (1.0, 1e-20), (1.0, 1e20), (1e6, 1e-3), (1e-4, 1.0),
                                                (1e25, 1e25)])
def test_ransac_fp32_screen_is_rigorous(ctx, port, scale_pts, scale_e):
    """The FP32 screen decides only what its error bound allows, whatever the magnitudes: pixel-unit coordinates,
    tiny / huge hypotheses, values that overflow FP32, thresholds of every size (incl. <= 0, inf, nan), and thresholds
    placed just beside computed errors.  Counts, winner and inlier list stay bit-exact."""
    pi, pj = two_view_scene(1500, seed=77)
    xi, xj = port.norm_points(TEMPLE_K, pi) * scale_pts, port.norm_points(TEMPLE_K, pj) * scale_pts
    E, _ = port.ransac_hypotheses(port.norm_points(TEMPLE_K, pi), port.norm_points(TEMPLE_K, pj), 96)
    E = E * scale_e
    rng = np.random.default_rng(5)
    E[5] = rng.normal(0, 1, 9)
    E[6] = 0.0
    with np.errstate(all="ignore"):
        errs = np.array([port.sampson(E[h], xi[i], xj[i]) for h in (0, 1, 5) for i in range(0, 1500, 97)])
    errs = errs[np.isfinite(errs) & (errs > 0)]
    near = np.concatenate([errs * f for f in (1.0, 1 - 1e-6, 1 + 1e-6, 1 - 3e-6, 1 + 3e-6, 1 - 1e-4, 1 + 1e-4)]) if len(errs) else np.zeros(0)
    for thr in [1e-3, 1e-9, 1.0, 1e6, 1e-40, 1e35, 0.0, -1.0, np.inf, np.nan] + near[::5].tolist():
        counts, bh, inl = ctx.ransac_score(xi, xj, E, float(thr))
        wc, wb, wi = port.ransac_score(xi, xj, E, float(thr))
        assert np.array_equal(counts, wc) and bh == wb and np.array_equal(inl, wi), (scale_pts, scale_e, thr)


def test_ransac_golden(ctx, g):
    counts, bh, inl = ctx.ransac_score(g["rs_xi"], g["rs_xj"], g["rs_E"], 1e-3)
    assert np.array_equal(counts, g["rs_counts"]) and bh == g["rs_best"][0] and np.array_equal(inl, g["rs_inl"])


def test_ransac_degenerate(ctx):
    counts, bh, inl = ctx.ransac_score(np.zeros((0, 2)), np.zeros((0, 2)), np.zeros((3, 9)), 1e-3)
    assert counts.tolist() == [0, 0, 0] and bh == -1 and len(inl) == 0


# ---- device minimal solver (opt-in, SURVEY.md §8f-1) -------------------------------------------------------------
@pytest.mark.parametrize("n,H", [(300, 200), (2200, 2500), (40, 64)])
def test_device_solver_matches_host_hypotheses(ctx, port, n, H):
    """sfmgpu_ransac_hypotheses: same sampled octets as the reference (its own RNG stream), hypotheses equal to the
    host solver's up to sign and ~1e-9 relative (NOT bit-identical: CUDA vs glibc trig), same winner and inlier set."""
    pi, pj = two_view_scene(n, seed=7 * n + H)
    xi, xj = port.norm_points(TEMPLE_K, pi), port.norm_points(TEMPLE_K, pj)
    Eh, idx = port.ransac_hypotheses(xi, xj, H)  # host solver + the reference's seeded sampling
    assert np.array_equal(idx.ravel(), port.rng_draws(n, 8 * H))
    Ed = ctx.ransac_hypotheses(xi, xj, idx)
    sgn = np.sign((Ed * Eh).sum(1, keepdims=True))
    scale = np.abs(Eh).max(1, keepdims=True)
    err = np.abs(Ed * sgn - Eh) / scale
    # degenerate samples (repeated indices: sampling is with replacement) have a multi-dimensional null space and
    # may legitimately pick a different vector of it; they never win a RANSAC round
    distinct = np.array([len(set(r)) == 8 for r in idx.tolist()])
    print(f"device solver: max rel. deviation {err[distinct].max():.2e} over {distinct.sum()} non-degenerate hypotheses")
    assert np.quantile(err[distinct], 0.99) < 1e-8
    bh, bn = ctx.ransac_score_resident(1e-3)
    counts, inl = ctx.ransac_download(H, n)
    wc, wbh, wi = port.ransac_score(xi, xj, Eh, 1e-3)
    assert bh == wbh and bn == len(wi) and np.array_equal(inl[:bn], wi)
    assert (counts != wc)[distinct].mean() < 0.01  # borderline points may flip on a few hypotheses


# ---- batched DLT triangulation (opt-in, SURVEY.md §8f-4) -----------------------------------------------------------
@pytest.mark.parametrize("n", [1, 333, 5000])
def test_device_triangulation(ctx, checker, n):
    poses, ia, ib, ui, uj, _ = triangulation_scene(n, seed=n)
    got = ctx.triangulate_dlt(TEMPLE_K, poses, ia, ib, ui, uj)
    want = checker.triangulate_dlt(TEMPLE_K, poses, ia, ib, ui, uj)
    rel = np.abs(got - want).max(1) / np.abs(want).max(1)
    print(f"device triangulation: max rel. deviation {rel.max():.2e} over {n} tracks")
    assert rel.max() < 1e-7 and np.quantile(rel, 0.99) < 1e-9


# ---- loop-closure descriptor (SURVEY.md §8f-3) ----------------------------------------------------------------------
@pytest.mark.parametrize("w,h", [(640, 480), (1920, 1080), (33, 70), (20, 15), (64, 64), (32, 32), (517, 129)])
def test_loop_descriptor_bit_exact(ctx, checker, w, h):
    imgs = [synth.frame(9, t, w, h) for t in (0, 5, 30, 31)]
    f = _frames(ctx, imgs, 1)
    got = f.global_desc32(0, 4)
    want = np.stack([checker.global_desc32(i) for i in imgs])
    assert np.array_equal(got, want)
    bid, bs, sc = ctx.desc_search(got[:3], got[3])
    wid, wbs, wsc = checker.desc_search(want[:3], want[3])
    assert bid == wid and bs == wbs and np.array_equal(sc, wsc)
    assert ctx.desc_search(got[:3], -got[0])[0] == -1 or checker.desc_search(want[:3], -want[0])[0] != -1
    assert ctx.desc_search(got[:0], got[3])[:2] == (-1, 0.0)


# ---- batched two-view front end ----------------------------------------------------------------------------------------
def test_pair_frontend_batch(ctx, checker, g):
    imgs = [synth.frame(SEED, t, W, H) for t in range(6)]
    f = _frames(ctx, imgs)
    cfg = sfmgpu.lkcfg(max_tracks=300)
    pairs = ctx.pairs(5, 300)
    pairs.run(f, 0, 5, cfg)
    nc_tot, nk_tot, nit_tot = pairs.totals()
    cs = ks = 0
    for p in range(5):
        li, lj, nc = pairs.download(p)
        wl, wj, wnc = checker.pair_frontend(imgs[p], imgs[p + 1], 300)
        assert nc == wnc and np.array_equal(li, wl) and _klt_close(lj, wj), p
        cs, ks = cs + nc, ks + len(li)
    assert (nc_tot, nk_tot) == (cs, ks) and nit_tot > 0
    li, lj, nc = pairs.download(2)
    assert nc == g["pair_nc"][0] and np.array_equal(li, g["pair_li"]) and _klt_close(lj, g["pair_lj"])


def test_pair_frontend_batch_provisional_list_overflow(ctx, checker):
    """Weak texture everywhere and ONE strong corner in a tile the probe pass does not visit: the fused score pass works
    with a far too low provisional threshold, its list overflows the batch capacity (w*h/6), and the frame is redone
    against the final threshold on the device (score_rescue_kernel).  Plain frames share the batch."""
    rng = np.random.default_rng(8)
    weak = (100 + rng.integers(0, 4, (H, W))).astype(np.uint8)
    strong = weak.copy()
    strong[200:216, 16:32] = 0
    strong[208:216, 24:32] = 255
    imgs = [strong, np.roll(strong, 1, axis=1), synth.frame(41, 0, W, H), synth.frame(41, 1, W, H), weak]
    f = _frames(ctx, imgs)
    cfg = sfmgpu.lkcfg(max_tracks=500)
    pairs = ctx.pairs(4, 500)
    pairs.run(f, 0, 4, cfg)
    for p in range(4):
        li, lj, nc = pairs.download(p)
        wl, wj, wnc = checker.pair_frontend(imgs[p], imgs[p + 1], 500)
        assert nc == wnc and np.array_equal(li, wl) and _klt_close(lj, wj), p
    # the single-frame entry points (capacity w*h) on the same images
    for k, im in enumerate(imgs):
        assert np.array_equal(f.corners(k, 500), checker.shi_tomasi(im, 500)), k


@pytest.mark.parametrize("streaming", [False, True])
def test_pair_frontend_batch_flat_and_weak_frames(ctx, checker, streaming):
    """A flat frame (thr = 0: every pixel incl. the zeroed border is a candidate, :274-285) and a weak-texture frame (almost
    every pixel reaches 1 % of the maximum) inside a batch: their FINAL candidate lists exceed the batch capacity
    (max(w*h/6, 65536) < w*h), so the call redoes them with the full capacity and returns the reference's result -
    no SFMGPU_E_CAPACITY, nothing truncated."""
    rng = np.random.default_rng(21)
    flat = np.full((H, W), 131, np.uint8)
    weak = (90 + rng.integers(0, 3, (H, W))).astype(np.uint8)
    imgs = [synth.frame(51, 0, W, H), flat, synth.frame(51, 1, W, H), weak, np.roll(weak, 1, axis=0), flat, flat]
    cfg = sfmgpu.lkcfg(max_tracks=400)
    pairs = ctx.pairs(6, 400)
    if streaming:
        f = ctx.frames(W, H, len(imgs), 3)
        li, lj = np.full((6, 400, 2), -1.0), np.full((6, 400, 2), -1.0)
        nk, nc = np.zeros(6, np.int32), np.zeros(6, np.int32)
        pairs.run_host(f, np.stack(imgs), cfg, li, lj, nk, nc, chunk=3)
    else:
        f = _frames(ctx, imgs)
        pairs.run(f, 0, 6, cfg)
    tot_c, tot_k, _ = pairs.totals()  # raises if a frame were still marked as overflowed
    cs = ks = 0
    for p in range(6):
        wl, wj, wnc = checker.pair_frontend(imgs[p], imgs[p + 1], 400)
        if streaming:
            gl, gj, gnc = li[p, :nk[p]], lj[p, :nk[p]], int(nc[p])
        else:
            gl, gj, gnc = pairs.download(p)
        assert gnc == wnc and np.array_equal(gl, wl) and _klt_close(gj, wj), p
        cs, ks = cs + gnc, ks + len(gl)
    assert (tot_c, tot_k) == (cs, ks)


def test_pair_frontend_bench_shape_pair(ctx, checker):
    """One pair of bench.py's own C2 sequence (1920x1080, seed 20261018, 2000 corners, frames 500/501) against the
    compiled reference: corner count, survivors, li bit-exact, lj within the KLT tolerance."""
    w, h, nmax = 1920, 1080, 2000
    f0, f1 = synth.frame(SEED, 500, w, h), synth.frame(SEED, 501, w, h)
    f = _frames(ctx, [f0, f1], 3)
    cfg = sfmgpu.lkcfg(max_tracks=nmax)
    pairs = ctx.pairs(1, nmax)
    pairs.run(f, 0, 1, cfg)
    li, lj, nc = pairs.download(0)
    wl, wj, wnc = checker.pair_frontend(f0, f1, nmax)
    assert nc == wnc and len(li) == len(wl) and np.array_equal(li, wl) and _klt_close(lj, wj)


def test_pair_frontend_batch_with_score_ties(ctx, checker):
    """Quantised frames (many identical scores) between plain ones in ONE batch: the bucket selection hands exactly the
    frames whose consumed prefix holds a tie to the exact emulation, inside the batched launch."""
    imgs = [synth.frame(31, t, W, H) for t in range(7)]
    for t in (1, 2, 5):
        imgs[t] = imgs[t] >> 4 << 4
    f = _frames(ctx, imgs)
    cfg = sfmgpu.lkcfg(max_tracks=900)
    pairs = ctx.pairs(6, 900)
    for mode in (0, 1, 16, 1100):
        ctx.select_set_mode(mode)
        try:
            pairs.run(f, 0, 6, cfg)
        finally:
            ctx.select_set_mode(0)
        for p in range(6):
            li, lj, nc = pairs.download(p)
            wl, wj, wnc = checker.pair_frontend(imgs[p], imgs[p + 1], 900)
            assert nc == wnc and np.array_equal(li, wl) and _klt_close(lj, wj), (mode, p)


@pytest.mark.parametrize("chunk,pipe", [(0, 0), (2, 0), (3, 1), (7, 2), (100, 2), (4, 3)])
def test_pair_frontend_streaming_equals_resident(ctx, chunk, pipe):
    """sfmgpu_pair_frontend_host (chunked upload || two compute lanes || download) and the two-lane resident call
    return what the sequential resident call returns."""
    imgs = np.stack([synth.frame(SEED, t, W, H) for t in range(7)])
    cfg = sfmgpu.lkcfg(max_tracks=300)
    f = _frames(ctx, list(imgs))
    pairs = ctx.pairs(6, 300)
    ctx.pipeline_set(0)
    pairs.run(f, 0, 6, cfg)
    want_tot = pairs.totals()
    li, lj = np.zeros((6, 300, 2)), np.zeros((6, 300, 2))
    nk, nc = np.zeros(6, np.int32), np.zeros(6, np.int32)
    pairs.download_all(li, lj, nk, nc)
    f2 = ctx.frames(W, H, 7, 3)  # fresh storage: the streaming call must fill it itself
    p2 = ctx.pairs(6, 300)
    li2, lj2 = np.full((6, 300, 2), -1.0), np.full((6, 300, 2), -1.0)
    nk2, nc2 = np.zeros(6, np.int32), np.zeros(6, np.int32)
    ctx.pipeline_set(pipe)
    try:
        p2.run_host(f2, imgs, cfg, li2, lj2, nk2, nc2, chunk=chunk)
        assert p2.totals() == want_tot
        assert np.array_equal(nk, nk2) and np.array_equal(nc, nc2)
        for p in range(6):
            assert np.array_equal(li[p, :nk[p]], li2[p, :nk[p]]) and np.array_equal(lj[p, :nk[p]], lj2[p, :nk[p]]), p
        # the resident call with the two-lane pipeline
        p3 = ctx.pairs(6, 300)
        p3.run(f, 0, 6, cfg)
        assert p3.totals() == want_tot
        li3, lj3 = np.zeros((6, 300, 2)), np.zeros((6, 300, 2))
        nk3, nc3 = np.zeros(6, np.int32), np.zeros(6, np.int32)
        p3.download_all(li3, lj3, nk3, nc3)
        assert np.array_equal(nk, nk3) and np.array_equal(nc, nc3)
        for p in range(6):
            assert np.array_equal(li[p, :nk[p]], li3[p, :nk[p]]) and np.array_equal(lj[p, :nk[p]], lj3[p, :nk[p]]), p
    finally:
        ctx.pipeline_set(0)


def test_c3_shape_4k_pair(ctx, checker):
    """BASELINE.json config C3 at full size: one 3840x2160 pair, 8000 corners/frame (bit-exact against the checker),
    tracks through the batched front end (lane kernel) within the KLT tolerance on a 1500-point sample."""
    w, h, nmax = 3840, 2160, 8000
    f0, f1 = synth.frame(SEED, 0, w, h), synth.frame(SEED, 1, w, h)
    f = _frames(ctx, [f0, f1], 3)
    cfg = sfmgpu.lkcfg(max_tracks=nmax, min_tracks=3273)
    pairs = ctx.pairs(1, nmax)
    pairs.run(f, 0, 1, cfg)
    li, lj, nc = pairs.download(0)
    want = checker.shi_tomasi(f0, nmax)
    assert nc == len(want) == nmax
    sel = np.r_[0:750, nmax - 750:nmax]
    w1, wb = checker.klt_track(f0, f1, want[sel])
    keep = ~(np.hypot(*(wb - want[sel]).T) >= 1.0)
    # survivors keep corner order: map the sample through the kept mask of the full run
    p1, pb = f.klt_track(0, 1, want)
    kept_all = ~(np.hypot(*(pb - want).T) >= 1.0)
    assert np.array_equal(li, want[kept_all]) and _klt_close(lj, p1[kept_all])
    assert np.array_equal(kept_all[sel], keep) and _klt_close(p1[sel], w1) and _klt_close(pb[sel], wb)


@pytest.mark.parametrize("select_mode", [0, 1300, 3048, 20])
def test_c3_shape_4k_corners_select_modes(ctx, checker, select_mode):
    """One 3840x2160 frame, 8000 corners (~400 k candidates): the bucket selection with its default geometry, with gathers
    of 300 / 2048 words (every bucket oversized: the sub-bucket walk at scale, or the exact emulation) and with 20-bit
    order codes (equal codes by the exact score recomputed from the image): bit-exact corners."""
    w, h, nmax = 3840, 2160, 8000
    f0 = synth.frame(SEED, 3, w, h)
    f = _frames(ctx, [f0], 1)
    ctx.select_set_mode(select_mode)
    try:
        got = f.corners(0, nmax, 0.01, 8)
    finally:
        ctx.select_set_mode(0)
    want = checker.shi_tomasi(f0, nmax, 0.01, 8)
    assert got.shape == want.shape and np.array_equal(got, want), (select_mode, len(got), len(want))


def test_errors_are_loud(ctx):
    f = ctx.frames(64, 48, 2, 3)
    with pytest.raises(sfmgpu.SfmGpuError):
        f.klt_track(0, 5, np.zeros((1, 2)))
    with pytest.raises(sfmgpu.SfmGpuError):
        f.klt_track(0, 1, np.zeros((1, 2)), radius=50)
    with pytest.raises(sfmgpu.SfmGpuError):
        ctx.frames(0, 48, 2, 3)
    with pytest.raises(sfmgpu.SfmGpuError):  # not a selection mode: an error, never a silent default
        ctx.select_set_mode(2)
