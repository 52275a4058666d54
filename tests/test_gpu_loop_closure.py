"""GPU tests of batched loop closure: the device-resident descriptor bank (global_desc_32, cpp/src/templering_sfm.cpp:1100-1122),
the all-query candidate search (dot_desc :1124-1129 inside the loop of :1823-1831) and the two-view unit over explicit
frame pairs (:1836-1857 on (old keyframe, current frame)).

Bars: descriptors, scores, candidates, corners, survivors' first-frame positions, RANSAC status / counts / inlier lists
bit-exact against the CPU checker; second-frame positions within KLT_TOL; the list call byte for byte equal to the
consecutive call on consecutive pairs."""
import ctypes as C

import numpy as np
import pytest

import ring_dataset
import sfmgpu
from conftest import TEMPLE_K
from sfmgpu import synth

pytestmark = pytest.mark.gpu

KLT_TOL = 1e-3  # px
W, H = 320, 240
E_ARG = -1
OK = 2  # SFMGPU_TV_OK
GAP = 6  # keyframes closer than this are not loop candidates (the caller's n_search = k - GAP)


def _frames(ctx, imgs, levels=3):
    imgs = np.ascontiguousarray(np.stack(imgs))
    f = ctx.frames(imgs.shape[2], imgs.shape[1], len(imgs), levels)
    f.upload(0, imgs)
    f.build_pyramid()
    return f


def _klt_close(a, b):
    a, b = np.asarray(a).reshape(-1, 2), np.asarray(b).reshape(-1, 2)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and np.nanmax(np.abs(a - b), initial=0.0) <= KLT_TOL


def _same_f32(a, b):
    return np.asarray(a, np.float32).tobytes() == np.asarray(b, np.float32).tobytes()


def _same_scores(a, b):
    """Bit for bit, except that a NaN only has to be a NaN: a GPU returns the canonical NaN where x86 propagates the input's
    payload (a NaN score never becomes a candidate on either)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


def _code(fn, *a):
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        fn(*a)
    return e.value.code


# ---- 1. the bank holds the reference's descriptors ------------------------------------------------------------------------
@pytest.mark.parametrize("w,h", [(20, 15), (32, 32), (33, 71), (700, 90), (1920, 1080)])
def test_bank_compute_equals_reference(ctx, checker, w, h):
    imgs = [synth.frame(13, t, w, h) for t in (0, 5, 9)]
    f = _frames(ctx, imgs, 1)
    bank = ctx.descs(8)
    bank.compute(f, 0, 3, slot=4)
    bank.compute(f, 1, 1, slot=0)
    got = bank.download()
    host = f.global_desc32(0, 3)
    want = np.stack([checker.global_desc32(i) for i in imgs])
    assert np.array_equal(host, want)
    assert _same_f32(got[4:7], want) and _same_f32(got[0], want[1])
    assert not got[[1, 2, 3, 7]].any()  # untouched slots stay zero


def test_bank_upload_download_round_trip(ctx):
    rng = np.random.default_rng(3)
    d = rng.standard_normal((5, 1024)).astype(np.float32)
    d[2, 17] = np.nan
    d[3, 5] = -0.0
    bank = ctx.descs(9)
    bank.upload(d, slot=3)
    assert _same_f32(bank.download(3, 5), d)
    assert not bank.download(0, 3).any() and not bank.download(8, 1).any()


# ---- 2. the search is the reference's loop --------------------------------------------------------------------------------
def _bank(n, seed):
    """Unit descriptors with close neighbours (scores near the 0.94 gate), duplicates, negated and zero ones, and a NaN."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((max(n // 8, 1), 1024))
    d = base[rng.integers(0, len(base), n)] + 0.3 * rng.standard_normal((n, 1024))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    if n >= 12:
        d[9] = d[5]  # duplicate: the lower slot wins the tie
        d[10] = -d[4]
        d[11] = 0.0  # a flat frame's descriptor
    if n >= 20:
        d[17, 100] = np.nan  # never wins
    return d


def _check_search(checker, d, qs, ns, bid, bs, sc):
    ld = int(ns.max()) if len(ns) else 0
    assert sc.shape == (len(qs), ld)
    for q, (s, n) in enumerate(zip(qs, ns)):
        wid, wbs, wsc = checker.desc_search(d[:n], d[s], n)
        assert bid[q] == wid and _same_f32(bs[q], wbs), (q, s, n, bid[q], wid, bs[q], wbs)
        assert _same_scores(sc[q, :n], wsc) and not sc[q, n:].any(), (q, s, n)


@pytest.mark.parametrize("n,nq", [(1, 1), (63, 63), (65, 40), (257, 257), (1100, 300)])
def test_search_equals_reference_loop(ctx, checker, n, nq):
    d = _bank(n, n)
    bank = ctx.descs(n + 3)
    bank.upload(d)
    rng = np.random.default_rng(n + 1)
    qs = rng.integers(0, n, nq).astype(np.int32)
    ns = rng.integers(0, n + 1, nq).astype(np.int32)
    ns[0] = 0
    if nq > 3:
        ns[1], ns[2], qs[3], ns[3] = n, min(n, 10), min(n - 1, 9), n  # slot 9 duplicates 5: 5 must win against itself
    bid, bs, sc = bank.search(qs, ns, want_scores=True)
    _check_search(checker, d, qs, ns, bid, bs, sc)
    assert bid[0] == -1 and bs[0] == 0.0
    bid2, bs2, none = bank.search(qs, ns)
    assert none is None and np.array_equal(bid2, bid) and _same_f32(bs2, bs)
    neg = ctx.descs(3)  # a negated descriptor against its own direction: every score < 0, no candidate
    neg.upload(np.stack([d[0], 0.5 * d[0], -d[0]]))
    nb, nbs, nsc = neg.search([2], [2], want_scores=True)
    assert nb[0] == -1 and nbs[0] == 0.0 and (nsc < 0).all()


def test_search_triangular_keyframes(ctx, checker):
    """Every keyframe k against the earlier ones minus the gap: slots [0, k - GAP)."""
    n = 1030
    d = _bank(n, 77)
    bank = ctx.descs(n)
    bank.upload(d)
    qs = np.arange(n, dtype=np.int32)
    ns = np.maximum(qs - GAP, 0).astype(np.int32)
    bid, bs, sc = bank.search(qs, ns, want_scores=True)
    _check_search(checker, d, qs, ns, bid, bs, sc)
    assert (bid[:GAP + 1] == -1).all() and (bid[GAP + 2:] >= 0).any()


def test_search_errors_leave_the_bank_usable(ctx):
    bank = ctx.descs(10)
    bank.upload(np.ones((10, 1024), np.float32) / 32)
    for qs, ns in (([10], [3]), ([-1], [3]), ([0], [11]), ([0], [-1])):
        assert _code(bank.search, qs, ns) == E_ARG
    assert _code(bank.upload, np.zeros((2, 1024), np.float32), 9) == E_ARG
    assert _code(bank.download, 8, 3) == E_ARG
    f = _frames(ctx, [synth.frame(1, 0, 64, 48)], 1)
    assert _code(bank.compute, f, 0, 1, 10) == E_ARG
    assert _code(bank.compute, f, 0, 2, 0) == E_ARG
    bid, bs, _ = bank.search([9], [9])
    assert bid[0] == 0 and bs[0] > 0


# ---- 3. the list front end is the reference's pair unit -------------------------------------------------------------------
def _list_images():
    rng = np.random.default_rng(21)
    flat = np.full((H, W), 131, np.uint8)
    weak = (90 + rng.integers(0, 3, (H, W))).astype(np.uint8)
    return [synth.frame(51, t, W, H) for t in (0, 1, 4, 9)] + [flat, weak, np.roll(weak, 1, axis=0)]


def test_list_frontend_equals_reference_pairs(ctx, checker):
    imgs = _list_images()
    f = _frames(ctx, imgs)
    fa = np.array([0, 3, 2, 0, 4, 5, 6, 1, 0], np.int32)  # non-adjacent, reversed, a == b, repeated a, flat, weak
    fb = np.array([3, 1, 2, 2, 0, 6, 5, 1, 1], np.int32)
    cfg = sfmgpu.lkcfg(max_tracks=300)
    pairs = ctx.pairs(12, 300)
    pairs.run_list(f, fa, fb, cfg)
    tot_c, tot_k, tot_it = pairs.totals()
    cs = ks = 0
    for k, (a, b) in enumerate(zip(fa, fb)):
        li, lj, nc = pairs.download(k)
        wl, wj, wnc = checker.pair_frontend(imgs[a], imgs[b], 300)
        assert nc == wnc and np.array_equal(li, wl) and _klt_close(lj, wj), (k, a, b, nc, wnc)
        cs, ks = cs + nc, ks + len(li)
    assert (tot_c, tot_k) == (cs, ks) and tot_it > 0
    nk, nc = np.zeros(len(fa), np.int32), np.zeros(len(fa), np.int32)
    pairs.download_all(None, None, nk, nc)
    assert nc.sum() == cs and nk.sum() == ks


# ---- 4. list = consecutive, byte for byte ------------------------------------------------------------------------------------
def _all_outputs(pairs, n, with_ransac):
    cap = pairs.cap
    li, lj = np.full((n, cap, 2), -7.0), np.full((n, cap, 2), -7.0)
    nk, nc = np.zeros(n, np.int32), np.zeros(n, np.int32)
    pairs.download_all(li, lj, nk, nc)
    out = [nk, nc, pairs.totals()]
    for k in range(n):
        out += [li[k, :nk[k]], lj[k, :nk[k]]]
    if with_ransac:
        st, bn = np.zeros(n, np.int32), np.zeros(n, np.int32)
        inl, R, t = np.zeros((n, cap), np.int32), np.zeros((n, 9)), np.zeros((n, 3))
        pairs.ransac_download_all(st, bn, inl, R, t)
        out += [st, bn] + [inl[k, :max(bn[k], 0)] for k in range(n)] + [R[st == OK], t[st == OK]]
    return out


def _assert_same(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert np.asarray(x).tobytes() == np.asarray(y).tobytes(), i


@pytest.mark.parametrize("with_ransac", [False, True])
def test_list_equals_consecutive(ctx, with_ransac):
    imgs = [ring_dataset.render(np.deg2rad(0.4 * t), W, H) for t in range(6)] + _list_images()
    f = _frames(ctx, imgs)
    n = len(imgs) - 1
    cfg = sfmgpu.lkcfg(max_tracks=500)
    res = []
    for mode in ("run", "list"):
        pairs = ctx.pairs(n, 500)
        if with_ransac:
            pairs.set_ransac(TEMPLE_K, 4000, 2e-3, 80, 120)
        if mode == "run":
            pairs.run(f, 0, n, cfg)
        else:
            pairs.run_list(f, np.arange(n), np.arange(1, n + 1), cfg)
        res.append(_all_outputs(pairs, n, with_ransac))
        pairs.close()
    _assert_same(res[0], res[1])
    if with_ransac:
        assert (res[0][3 + 2 * n] == OK).any()  # status follows counts, totals and the 2n point lists


def test_list_equals_consecutive_over_several_chunks(ctx):
    """More than 1024 pairs: the corner stages run in two chunks."""
    n = 1100
    f = ctx.frames(96, 64, n + 1, 3)
    f.synth(0, n + 1, 4242, 0)
    f.build_pyramid()
    cfg = sfmgpu.lkcfg(max_tracks=40, pyr_levels=3)
    res = []
    for mode in ("run", "list"):
        pairs = ctx.pairs(n, 40)
        pairs.set_ransac(TEMPLE_K, 300, 2e-3, 8, 12)
        if mode == "run":
            pairs.run(f, 0, n, cfg)
        else:
            pairs.run_list(f, np.arange(n), np.arange(1, n + 1), cfg)
        res.append(_all_outputs(pairs, n, True))
        pairs.close()
    _assert_same(res[0], res[1])
    assert res[0][2][1] > 0


# ---- 5. loop closure end to end -------------------------------------------------------------------------------------------
RING_DEG = [0.0, 1.5, 3.0, 4.5, 6.0, 7.5, 9.0, 10.5, 12.0, 10.8, 8.7, 6.6, 4.9, 3.3, 1.7, 0.2]  # out and back near the start


def test_loop_closure_end_to_end(ctx, checker):
    imgs = [ring_dataset.render(np.deg2rad(a), 640, 480) for a in RING_DEG]
    n = len(imgs)
    f = _frames(ctx, imgs)
    bank = ctx.descs(n)
    bank.compute(f, 0, n)
    qs = np.arange(n, dtype=np.int32)
    ns = np.maximum(qs - GAP, 0).astype(np.int32)
    bid, bs, _ = bank.search(qs, ns)
    want = np.stack([checker.global_desc32(i) for i in imgs])
    for k in range(n):
        wid, wbs, _ = checker.desc_search(want[:ns[k]], want[k], int(ns[k]))
        assert bid[k] == wid and _same_f32(bs[k], wbs), (k, bid[k], wid)
    cand = [(int(bid[k]), k) for k in range(n) if bid[k] >= 0]
    assert any(RING_DEG[a] < 1.0 and RING_DEG[b] < 1.0 for a, b in cand), cand  # the revisit finds the start
    fa = np.array([a for a, _ in cand], np.int32)
    fb = np.array([b for _, b in cand], np.int32)
    cfg = sfmgpu.lkcfg(max_tracks=1200)
    pairs = ctx.pairs(len(cand), 1200)
    pairs.set_ransac(TEMPLE_K, 4000, 2e-3, 80, 120)  # :1855-1857
    pairs.run_list(f, fa, fb, cfg)
    statuses, repeated = [], 0
    for k, (a, b) in enumerate(cand):
        li, lj, nc = pairs.download(k)
        wl, wj, wnc = checker.pair_frontend(imgs[a], imgs[b], 1200)
        assert nc == wnc and np.array_equal(li, wl) and _klt_close(lj, wj), (k, a, b)
        st, _, inl, _, R, t = pairs.ransac_download(k)
        statuses.append(st)
        if len(li) < 120:
            assert st == 0, (k, st)
            continue
        r = checker.find_E_ransac(TEMPLE_K, li, lj, 4000, 2e-3, 80)
        if r is None:
            assert st == 1, (k, st)
            continue
        wR, wt, winl = r
        assert st == OK and np.array_equal(inl, winl), (k, st, len(inl), len(winl))
        if np.abs(R - wR).max() >= 1e-6 or np.abs(t - wt).max() >= 1e-6:
            # a winning octet with a repeated index: a two-dimensional null space, another member of it (DESIGN.md §4)
            xi, xj = checker.norm_points(TEMPLE_K, li), checker.norm_points(TEMPLE_K, lj)
            E, idx = checker.ransac_hypotheses(xi, xj, 4000)
            wbh = checker.ransac_score(xi, xj, E, 2e-3)[1]
            assert len(set(idx[wbh])) < 8, (k, np.abs(R - wR).max())
            repeated += 1
    print(f"loop closure: {len(cand)} candidate pairs, statuses {statuses}, {repeated} repeated-index winners")
    assert OK in statuses and repeated <= max(1, statuses.count(OK) // 4)


# ---- 6. errors ----------------------------------------------------------------------------------------------------------------
def test_list_errors_leave_the_pairs_usable(ctx, checker):
    imgs = [synth.frame(8, t, W, H) for t in range(3)]
    f = _frames(ctx, imgs)
    cfg = sfmgpu.lkcfg(max_tracks=200)
    pairs = ctx.pairs(2, 200)
    assert _code(pairs.run_list, f, [0, 3], [1, 1], cfg) == E_ARG
    assert _code(pairs.run_list, f, [-1], [1], cfg) == E_ARG
    assert _code(pairs.run_list, f, [0], [3], cfg) == E_ARG
    assert _code(pairs.run_list, f, [0, 1, 2], [1, 2, 0], cfg) == E_ARG  # more than max_pairs
    assert _code(pairs.run_list, f, [0], [1], sfmgpu.lkcfg(max_tracks=100)) == E_ARG
    assert _code(pairs.run_list, f, [0], [1], sfmgpu.lkcfg(max_tracks=200, pyr_levels=2)) == E_ARG
    assert ctx.lib.sfmgpu_pair_frontend_list(ctx.h, f.h_, None, None, 1, C.byref(cfg), pairs.h_) == E_ARG
    pairs.run_list(f, [2, 0], [0, 2], cfg)
    for k, (a, b) in enumerate(((2, 0), (0, 2))):
        li, lj, nc = pairs.download(k)
        wl, wj, wnc = checker.pair_frontend(imgs[a], imgs[b], 200)
        assert nc == wnc and np.array_equal(li, wl) and _klt_close(lj, wj)
    pairs.run_list(f, [], [], cfg)
    assert pairs.totals() == (0, 0, 0)
