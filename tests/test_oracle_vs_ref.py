"""Pins the restatement (oracle/sfm_oracle.cpp) against the reference (oracle/_ref, the unmodified TU).

The reference ships no tests or golden vectors (SURVEY.md §4); these cases are therefore the pin.  Every case is checked
against tests/golden/oracle_vs_ref.npz (stored outputs of cases(), written by tests/golden/gen_oracle_vs_ref.py) and,
where the compiled reference is built - its sources are not part of this repository - against the reference itself on
the same inputs.  The committed file was recorded with the restatement at commit 170c80d (its "recorded_with" key):
it freezes the restatement as this module compared it with the compiled reference.  Regenerate it where the reference
is built to record from the reference directly.  CPU only.
"""
import os

import numpy as np
import pytest

from conftest import TEMPLE_K, two_view_scene, triangulation_scene
from sfmgpu import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref.npz")


def _images():
    rng = np.random.default_rng(3)
    kat = synth.kat_image(320, 200)
    return {
        "kat": kat,
        "synth": synth.frame(11, 0, 320, 240),
        "ties": (synth.frame(12, 0, 200, 160) >> 4 << 4),  # coarse grey levels -> many tied scores
        "noise": rng.integers(0, 256, (97, 131), dtype=np.uint8),  # odd sizes
        "flat": np.full((24, 40), 77, np.uint8),  # thr = 0: every pixel is a candidate
        "tiny": rng.integers(0, 256, (4, 9), dtype=np.uint8),  # h < 5: all-zero score map
        "one_bright": np.pad(np.full((1, 1), 255, np.uint8), 20),
    }


# ---- the cases: each returns the checker's outputs as a list of arrays --------------------------------------------------
def pyramid(chk, name):
    img, out = _images()[name], []
    for levels in (1, 2, 3, 4):
        p = chk.build_pyr(img, levels)
        assert np.array_equal(p[0], img)  # level 0 is the image itself: not stored
        out += [np.array(len(p))] + p[1:]
    return out


CORNER_CFGS = [(2200, 0.01, 8), (50, 0.2, 3), (0, 0.01, 8), (300, 0.0, 1), (100, 0.01, 0)]


def corners(chk, name, mc, q, d):
    return [chk.shi_tomasi(_images()[name], mc, q, d)]


KLT_CFGS = [(3, 5, 10), (1, 3, 4), (4, 2, 7)]


def klt(chk, pts):
    f0, f1 = synth.frame(21, 0, 320, 240), synth.frame(21, 3, 320, 240)
    return [a for lv, r, it in KLT_CFGS for a in chk.klt_track(f0, f1, pts, lv, r, it)]


def klt_points(port):
    rng = np.random.default_rng(5)
    f0 = synth.frame(21, 0, 320, 240)
    return np.concatenate([port.shi_tomasi(f0, 150), rng.uniform(-8, 330, (80, 2)) * [1, 0.75],
                           [[0.0, 0.0], [318.0, 238.0], [319.5, 100.25], [127.99999999999999, 64.0]]])


def tracker_sequence(chk):
    trk = chk.tracker(max_tracks=120, min_tracks=100, quality=0.01, min_distance=8, levels=3, radius=5, iters=10, fb=1.0)
    out = []
    for t in [0, 1, 2, 40, 41, 42, 43]:  # the jump 2 -> 40 kills tracks and triggers the replenish rule
        out += list(trk.step(synth.frame(31, t, 256, 192))) + list(trk.tracks())
    return out


RNG_NS = (8, 100, 2200, 10000)


def rng_draws(chk):
    return [chk.rng_draws(n, 64) for n in RNG_NS]


def hypotheses_and_scores(chk):
    pi, pj = two_view_scene(500)
    xi, xj = chk.norm_points(TEMPLE_K, pi), chk.norm_points(TEMPLE_K, pj)
    E, idx = chk.ransac_hypotheses(xi, xj, 60)
    out = [xi, xj, E, idx]
    for thr in (1e-3, 1e-6):
        c, bh, inl = chk.ransac_score(xi, xj, E, thr)
        out += [c, np.array(bh), inl]
    return out


FIND_E = [(400, 120, 1e-3, 60), (400, 60, 1e-9, 80), (7, 50, 1e-3, 1), (30, 40, 2e-3, 5)]


def find_E(chk, n, iters, thr, mi):
    pi, pj = two_view_scene(n, seed=n)
    r = chk.find_E_ransac(TEMPLE_K, pi, pj, iters, thr, mi)
    return [] if r is None else list(r)  # [] stands for std::nullopt


def pair_frontend(chk):
    f0, f1 = synth.frame(41, 7, 256, 192), synth.frame(41, 8, 256, 192)
    li, lj, nc = chk.pair_frontend(f0, f1, 150)
    return [li, lj, np.array(nc)]


DESC_SIZES = [(640, 480), (1920, 1080), (33, 70), (20, 15), (64, 64)]


def loop_descriptor(chk, w, h):
    d = [chk.global_desc32(synth.frame(9, t, w, h)) for t in (0, 5, 30)]
    bid, bs, scores = chk.desc_search(np.stack(d[:2]), d[2])
    return d + [np.array(bid), np.array(bs), scores]


def triangulate(chk):
    poses, ia, ib, ui, uj, X = triangulation_scene(400)
    return [chk.triangulate_dlt(TEMPLE_K, poses, ia, ib, ui, uj)]


def two_view_frames():
    return np.stack([synth.frame(20261018, t, 320, 240) for t in range(4)])


def two_view_unit(chk, threads):
    tracks, d = chk.two_view_mt(two_view_frames(), 300, threads, K=TEMPLE_K, rs_iters=150, rs_thr=2e-3, rs_min_inliers=80,
                                min_points=120)
    return [np.array(tracks)] + [d[k] for k in sorted(d)]


def cases(port):
    """key -> outputs(checker): every stored case of this module (the KLT points come from the port's corners)."""
    c = {f"pyramid/{n}": (lambda chk, n=n: pyramid(chk, n)) for n in _images()}
    for n in _images():
        for mc, q, d in CORNER_CFGS:
            c[f"corners/{n}/{mc}/{q}/{d}"] = lambda chk, a=(n, mc, q, d): corners(chk, *a)
    c["klt_points"] = lambda chk: [klt_points(port)]
    c["klt"] = lambda chk: klt(chk, klt_points(port))
    c["tracker"] = tracker_sequence
    c["rng"] = rng_draws
    c["hypotheses_and_scores"] = hypotheses_and_scores
    for a in FIND_E:
        c["find_E/%d/%d/%g/%d" % a] = lambda chk, a=a: find_E(chk, *a)
    c["pair_frontend"] = pair_frontend
    for w, h in DESC_SIZES:
        c[f"loop_descriptor/{w}x{h}"] = lambda chk, s=(w, h): loop_descriptor(chk, *s)
    c["triangulate"] = triangulate
    c["two_view_unit"] = lambda chk: two_view_unit(chk, 2)
    return c


# ---- the comparison ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def reference():
    import oracle
    return oracle.ref()  # None where the compiled reference is not built


def stored(golden, key):
    return [golden[f"{key}#{i}"] for i in range(int(golden[f"{key}#n"]))]


def same(a, b):
    return len(a) == len(b) and all(np.shape(x) == np.shape(y) and np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


def check(key, got, golden, reference, outputs):
    """The port's outputs `got` equal the stored ones and, where the reference is built, the reference's."""
    assert same(got, stored(golden, key)), key
    if reference is not None:
        assert same(got, outputs(reference)), key


@pytest.mark.parametrize("name", list(_images()))
def test_pyramid(name, port, reference, golden):
    check(f"pyramid/{name}", pyramid(port, name), golden, reference, lambda chk: pyramid(chk, name))


@pytest.mark.parametrize("name", list(_images()))
@pytest.mark.parametrize("mc,q,d", CORNER_CFGS)
def test_corners(name, mc, q, d, port, reference, golden):
    check(f"corners/{name}/{mc}/{q}/{d}", corners(port, name, mc, q, d), golden, reference, lambda chk: corners(chk, name, mc, q, d))


def test_kat_corners_match_survey(port, reference):
    # SURVEY.md §8c(3): first six corners of the 640x480 known-answer image
    for chk in (port, reference):
        if chk is not None:
            c = chk.shi_tomasi(synth.kat_image(), 2200)
            assert len(c) == 2200
            assert c[:6].astype(int).tolist() == [[545, 159], [305, 367], [255, 256], [239, 49], [49, 111], [289, 159]]


def test_klt(port, reference, golden):
    pts = klt_points(port)
    assert same([pts], stored(golden, "klt_points"))
    check("klt", klt(port, pts), golden, reference, lambda chk: klt(chk, pts))


def test_tracker_sequence(port, reference, golden):
    check("tracker", tracker_sequence(port), golden, reference, tracker_sequence)


def test_rng_kat(port, reference, golden):
    # SURVEY.md §8c(1)
    for chk in (port, reference):
        if chk is not None:
            assert chk.rng_draws(100, 16).tolist() == [92, 89, 31, 13, 18, 3, 20, 82, 56, 53, 59, 95, 96, 46, 65, 92]
    check("rng", rng_draws(port), golden, reference, rng_draws)


def test_sampson_kat(port, reference):
    E = [0, -0.1, 0.3, 0.12, 0, -0.9, -0.28, 0.91, 0.01]
    for chk in (port, reference):
        if chk is not None:
            assert chk.sampson(E, (0.1, -0.05), (0.11, -0.04)) == 1.7519471550715924e-05  # SURVEY.md §8c(2)


def test_hypotheses_and_scores(port, reference, golden):
    check("hypotheses_and_scores", hypotheses_and_scores(port), golden, reference, hypotheses_and_scores)


@pytest.mark.parametrize("n,iters,thr,mi", FIND_E)
def test_find_E_ransac(n, iters, thr, mi, port, reference, golden):
    check("find_E/%d/%d/%g/%d" % (n, iters, thr, mi), find_E(port, n, iters, thr, mi), golden, reference,
          lambda chk: find_E(chk, n, iters, thr, mi))


def test_pair_frontend(port, reference, golden):
    check("pair_frontend", pair_frontend(port), golden, reference, pair_frontend)


@pytest.mark.parametrize("w,h", DESC_SIZES)
def test_loop_descriptor(w, h, port, reference, golden):
    """global_desc_32 :1100-1122 and the candidate search :1823-1831: restatement == reference, bit for bit."""
    check(f"loop_descriptor/{w}x{h}", loop_descriptor(port, w, h), golden, reference, lambda chk: loop_descriptor(chk, w, h))


def test_triangulate_dlt(port, reference, golden):
    """triangulate_dlt :1477-1516: restatement == reference, bit for bit; and close to the true points."""
    got = triangulate(port)
    check("triangulate", got, golden, reference, triangulate)
    X = triangulation_scene(400)[5]
    assert np.median(np.linalg.norm(got[0] - X, axis=1)) < 0.05


def test_two_view_unit(port, reference, golden):
    """The whole two-view unit (:1836-1857: front end, size guard, find_E_ransac) per pair: restatement == reference, bit
    for bit, whatever the thread count; and equal to the single-pair entry points."""
    check("two_view_unit", two_view_unit(port, 2), golden, reference, lambda chk: two_view_unit(chk, 3))
    fr = two_view_frames()
    for chk in (port, reference):
        if chk is None:
            continue
        _, a = chk.two_view_mt(fr, 300, 3, K=TEMPLE_K, rs_iters=150, rs_thr=2e-3, rs_min_inliers=80, min_points=120)
        for p in range(3):
            li, lj, nc = chk.pair_frontend(fr[p], fr[p + 1], 300)
            assert nc == a["n_corners"][p] and np.array_equal(li, a["li"][p, :len(li)]) and np.array_equal(lj, a["lj"][p, :len(lj)])
            if len(li) < 120:
                assert a["status"][p] == 0
                continue
            r = chk.find_E_ransac(TEMPLE_K, li, lj, 150, 2e-3, 80)
            assert (r is None) == (a["status"][p] == 1)
            if r is not None:
                assert np.array_equal(r[0].reshape(9), a["R"][p]) and np.array_equal(r[1], a["t"][p])
                assert np.array_equal(r[2], a["inliers"][p, :a["n_inl"][p]])
        assert {0, 2} <= set(a["status"].tolist())
