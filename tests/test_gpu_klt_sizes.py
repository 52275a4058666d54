"""KLT between two pyramids of any sizes, and the tracker across image-size changes.

The reference's track_one walks the levels of any two pyramids built with the same level count and samples each image against
its own bounds (:183-198): a tap outside THAT image zeroes the sample.  Its KLTTracker keeps the previous image at its old size
and tracks into the new one (:345-346, :370).  sfmgpu_klt_track_between and the host-image tracker entry points do the same on
the device; these tests compare them with the restatement (oracle/sfm_oracle.cpp: track(Pyr, Pyr) through a flat export built
here, and its Tracker), with the one-batch kernel they generalise, with the reference where it is built, and through the C++
drop-in (KLTTracker, track_one_public)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import sfmgpu
from sfmgpu import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "structure-from-motion-3d-reconstruction_b200", "host")
E_ARG, E_STATE = -1, -4
BUDGET = 1e-3  # px, the parity budget of tests/test_gpu_parity.py
_u8 = np.ctypeslib.ndpointer(np.uint8, flags="C")
_f8 = np.ctypeslib.ndpointer(np.float64, flags="C")
_i4 = np.ctypeslib.ndpointer(np.int32, flags="C")
_i, _d, _vp = C.c_int, C.c_double, C.c_void_p
CXX = ["g++", "-std=c++20", "-O3", "-DNDEBUG", "-fPIC", "-shared", "-pthread", "-ffp-contract=off"]  # oracle/Makefile's flags


@pytest.fixture(scope="module")
def klt2(tmp_path_factory):
    """orc_klt_track2: the restatement's track(A, B) forward then backward, A and B of their own sizes."""
    so = str(tmp_path_factory.mktemp("klt2") / "libklt2.so")
    subprocess.run(CXX + [os.path.join(ROOT, "tests", "cpp", "klt_sizes_oracle.cpp"), "-o", so], check=True)
    lib = C.CDLL(so)
    lib.orc_klt_track2.argtypes = [_u8, _i, _i, _u8, _i, _i, _i, _i, _i, _f8, _i, _f8, _f8]

    def track(im0, im1, p0, levels=3, radius=5, iters=10):
        p0 = np.ascontiguousarray(p0, np.float64).reshape(-1, 2)
        p1, pb = np.zeros_like(p0), np.zeros_like(p0)
        lib.orc_klt_track2(np.ascontiguousarray(im0), im0.shape[1], im0.shape[0], np.ascontiguousarray(im1), im1.shape[1],
                           im1.shape[0], levels, radius, iters, p0, len(p0), p1, pb)
        return p1, pb
    return track


@pytest.fixture(scope="module")
def szshim(tmp_path_factory):
    """The C++ drop-in's KLTTracker and track_one_public behind flat wrappers (tests/cpp/klt_sizes_shim.cpp)."""
    sfmgpu.load_library()  # the shim links the in-tree library
    libdir = os.path.dirname(sfmgpu.LIB_PATH)
    so = str(tmp_path_factory.mktemp("szshim") / "libszshim.so")
    subprocess.run(CXX + ["-I" + HOST, os.path.join(ROOT, "tests", "cpp", "klt_sizes_shim.cpp"), "-o", so, "-L" + libdir,
                          "-lsfmgpu", "-Wl,-rpath," + libdir], check=True)
    lib = C.CDLL(so)
    lib.sz_last_error.restype = C.c_char_p
    lib.sz_tracker_create.restype = _vp
    lib.sz_tracker_create.argtypes = [_i, _i, _i]
    lib.sz_tracker_destroy.argtypes = [_vp]
    lib.sz_tracker_reset.argtypes = [_vp, _u8, _i, _i]
    lib.sz_tracker_step.argtypes = [_vp, _u8, _i, _i, _f8, _f8, _i4, _i]
    lib.sz_tracker_tracks.argtypes = [_vp, _f8, _i4, _i]
    lib.sz_pyr_build.restype = _vp
    lib.sz_pyr_build.argtypes = [_u8, _i, _i, _i]
    lib.sz_pyr_free.argtypes = [_vp]
    lib.sz_same_pool.argtypes = [_vp, _vp]
    lib.sz_track_one.argtypes = [_vp, _vp, _vp, _f8, _i, _f8]
    return lib


def _ck(lib, rc):
    if rc <= -1000:
        raise RuntimeError(lib.sz_last_error().decode())
    return rc


def _frames(ctx, img, levels=3, n=1, slot=0):
    f = ctx.frames(img.shape[1], img.shape[0], n, levels)
    f.upload(slot, img)
    f.build_pyramid(slot, 1)
    return f


def _probe_points(wa, ha, wb, hb, img, seed):
    """Corners of A, random points over the union of both images, and points on / just outside every border of either."""
    rng = np.random.default_rng(seed)
    pts = []
    if wa >= 16 and ha >= 16:
        from oracle import port
        pts += list(port().shi_tomasi(img, 60))
    W, H = max(wa, wb), max(ha, hb)
    pts += list(np.c_[rng.uniform(-3, W + 3, 60), rng.uniform(-3, H + 3, 60)])
    for w, h in ((wa, ha), (wb, hb)):
        for v in (0.0, 0.4, 1.0, 5.3, w - 7.2, w - 2.0, w - 1.5, w - 1.0, w - 0.3, w + 0.5):
            pts += [(v, h / 2 + 0.25), (v, 1.7), (v, h - 1.6)]
        for v in (0.0, 0.6, 5.5, h - 6.8, h - 2.0, h - 1.2, h - 0.5, h + 1.0):
            pts += [(w / 2 + 0.3, v), (2.2, v), (w - 2.7, v)]
    pts += [(-40.0, 10.0), (W + 30.0, H + 30.0), (1e12, 5.0)]
    return np.ascontiguousarray(np.array(pts, np.float64).reshape(-1, 2))


def _keep(p0, pb, thr=1.0):
    return ~(np.hypot(pb[:, 0] - p0[:, 0], pb[:, 1] - p0[:, 1]) >= thr)  # NaN is kept (:362)


def _stable(klt2, im0, im1, p0, w1, wb, *args):
    """Points where the checker itself is well conditioned: shifting p0 by 1e-11 px moves its results by less than 1e-6 px.
    Elsewhere (windows that only a few samples of one image reach, with a near-singular normal matrix) the reference's
    non-contractive update amplifies any rounding difference, so no other operation order can agree with it there."""
    d = np.zeros(len(p0))
    for eps in ((1e-11, 0.0), (0.0, 1e-11), (1e-11, 1e-11)):
        s1, sb = klt2(im0, im1, p0 + np.array(eps), *args)
        with np.errstate(invalid="ignore"):
            dd = np.nan_to_num(np.maximum(np.abs(s1 - w1).max(1), np.abs(sb - wb).max(1)), nan=np.inf)
        d = np.maximum(d, dd)
    both_nan = ~np.isfinite(w1).all(1)
    return (d < 1e-6) | both_nan


SIZE_PAIRS = [((640, 480), (641, 479)), ((640, 480), (320, 240)), ((640, 480), (1280, 720)), ((640, 480), (700, 480)),
              ((320, 240), (9, 7)), ((9, 7), (320, 240))]


@pytest.mark.parametrize("radius", [5, 3, 10])
@pytest.mark.parametrize("sa,sb", SIZE_PAIRS, ids=[f"{a[0]}x{a[1]}-{b[0]}x{b[1]}" for a, b in SIZE_PAIRS])
def test_klt_track_between_matches_checker(ctx, klt2, sa, sb, radius):
    (wa, ha), (wb, hb) = sa, sb
    levels = 3
    im0, im1 = synth.frame(41, 0, wa, ha), synth.frame(41, 1, wb, hb)
    fa, fb = _frames(ctx, im0, levels), _frames(ctx, im1, levels)
    p0 = _probe_points(wa, ha, wb, hb, im0, 5)
    p1, pb = fa.klt_track_between(0, fb, 0, p0, radius=radius)
    w1, wb_ = klt2(im0, im1, p0, levels, radius)
    st = _stable(klt2, im0, im1, p0, w1, wb_, levels, radius)
    assert st.mean() >= 0.75
    fin = np.isfinite(w1).all(1) & np.isfinite(wb_).all(1)
    assert np.array_equal(fin[st], (np.isfinite(p1).all(1) & np.isfinite(pb).all(1))[st])
    c = st & fin
    dev = max(np.abs(p1[c] - w1[c]).max(), np.abs(pb[c] - wb_[c]).max())
    print(f"{wa}x{ha} -> {wb}x{hb}, r={radius}: {st.sum()} of {len(p0)} points well conditioned, "
          f"max |device - checker| = {dev:.3e} px there")
    assert dev <= BUDGET
    assert np.array_equal(_keep(p0, pb)[st], _keep(p0, wb_)[st])


@pytest.mark.parametrize("radius", [5, 3, 7, 10])
def test_klt_track_between_same_size_equals_one_batch_warp_kernel(ctx, radius):
    """Two batches of one size run the two-geometry kernel; one batch with the warp kernel pinned gives the same bytes."""
    w, h = 640, 480
    im0, im1 = synth.frame(43, 0, w, h), synth.frame(43, 1, w, h)
    fa, fb = _frames(ctx, im0), _frames(ctx, im1)
    one = ctx.frames(w, h, 2, 3)
    one.upload(0, np.stack([im0, im1]))
    one.build_pyramid()
    p0 = _probe_points(w, h, w, h, im0, 6)
    got = fa.klt_track_between(0, fb, 0, p0, radius=radius, count=True)
    ctx.klt_set_mode(1)
    try:
        want = one.klt_track(0, 1, p0, radius=radius, count=True)
        same = fa.klt_track_between(0, fa, 0, p0, radius=radius, count=True)  # fa == fb is sfmgpu_klt_track
    finally:
        ctx.klt_set_mode(0)
    for g, x in zip(got, want):
        assert g.tobytes() == x.tobytes()
    for g, x in zip(same, fa.klt_track(0, 0, p0, radius=radius, count=True)):
        assert g.tobytes() == x.tobytes()


def test_klt_track_between_refusals(ctx):
    im = synth.frame(44, 0, 160, 120)
    f3, f2 = _frames(ctx, im, 3), _frames(ctx, im, 2)
    p0 = np.array([[50.0, 40.0]])
    p1, pb, nit = np.zeros((1, 2)), np.zeros((1, 2)), np.zeros(1, np.int32)
    lib = ctx.lib
    assert lib.sfmgpu_klt_track_between(ctx.h, f3.h_, 0, f2.h_, 0, p0, 1, 5, 10, p1, pb, None) == E_ARG  # level counts differ
    assert lib.sfmgpu_klt_track_between(ctx.h, f3.h_, 0, None, 0, p0, 1, 5, 10, p1, pb, None) == E_ARG
    f3b = _frames(ctx, im, 3)
    assert lib.sfmgpu_klt_track_between(ctx.h, f3.h_, 1, f3b.h_, 0, p0, 1, 5, 10, p1, pb, None) == E_ARG  # bad index
    assert lib.sfmgpu_klt_track_between(ctx.h, f3.h_, 0, f3b.h_, 0, p0, -1, 5, 10, p1, pb, None) == E_ARG
    assert lib.sfmgpu_klt_track_between(ctx.h, f3.h_, 0, f3b.h_, 0, p0, 1, 11, 10, p1, pb, None) == E_ARG  # radius
    assert lib.sfmgpu_klt_track_between(ctx.h, f3.h_, 0, f3b.h_, 0, p0, 0, 5, 10, p1, pb, None) == 0  # nothing to do


# Host-fed sequences: (seed, t, w, h): constant size, grow, shrink, back, odd sizes.  The frame of another sequence (seed 5)
# at a new size loses every track; with min_tracks = 0 nothing is replenished, so the next step, at yet another size, resets
# (:341-344).  With min_tracks > 0 the steps after a size change replenish on the new image.  Seed "reset": reset() on frame
# t of sequence 91 instead of step(), at a new size and at the same size.
SEQ = [(91, 0, 320, 240), (91, 1, 320, 240), (91, 2, 400, 300), (91, 3, 256, 200), (91, 4, 320, 240), (91, 5, 321, 239),
       (91, 6, 333, 251), (91, 7, 333, 251), (5, 0, 250, 190), (91, 8, 262, 198), (91, 9, 257, 203), ("reset", 10, 320, 240),
       (91, 11, 320, 240), ("reset", 12, 320, 240), (91, 13, 301, 222)]
CFGS = {"replenish": dict(max_tracks=150, min_tracks=120), "no_replenish": dict(max_tracks=150, min_tracks=0)}


def _image(seed, t, w, h):
    return synth.frame(91 if seed == "reset" else seed, t, w, h)


def _check_step(got, want, what):
    (gp, gc, gi), (wp, wc, wi) = got, want
    assert np.array_equal(gi, wi), what
    if len(gi):
        dev = max(np.abs(gp - wp).max(), np.abs(gc - wc).max())
        assert dev <= BUDGET, (what, dev)


def _check_tracks(got, want, what):
    (gx, gi), (wx, wi) = got, want
    assert np.array_equal(gi, wi), what
    if len(gi):
        assert np.abs(gx - wx).max() <= BUDGET, what


def _follower(ctx, **cfg):
    """A C ABI tracker that follows image-size changes (sfmgpu_tracker_set_size_change)."""
    t = ctx.tracker(**cfg)
    t.set_size_change(True)
    return t


def _run_against(ctx, other, cfg):
    """Steps the C ABI tracker and `other` (a CPU checker) through SEQ and compares every step and tracks()."""
    t = _follower(ctx, **cfg)
    o = other.tracker(**cfg)
    lost_all = resets_at_new_size = 0
    for k, (seed, tt, w, h) in enumerate(SEQ):
        img = _image(seed, tt, w, h)
        what = f"step {k} ({w}x{h})"
        if seed == "reset":
            t.reset(img)
            o.reset(img)
        else:
            n_before = len(o.tracks()[1])
            got, want = t.step(img), o.step(img)
            _check_step(got, want, what)
            lost_all += n_before > 0 and len(want[2]) == 0
            resets_at_new_size += n_before == 0 and k > 0 and (w, h) != SEQ[k - 1][2:]
        _check_tracks(t.tracks(), o.tracks(), what)
    return lost_all, resets_at_new_size


@pytest.mark.parametrize("cfg", list(CFGS), ids=list(CFGS))
def test_tracker_across_sizes_matches_checker(ctx, port, cfg):
    lost_all, resets = _run_against(ctx, port, CFGS[cfg])
    assert lost_all >= 1  # the frame of another sequence took every track
    if cfg == "no_replenish":
        assert resets >= 1  # ... and the next step, at another size, reset


@pytest.mark.parametrize("cfg", list(CFGS), ids=list(CFGS))
def test_tracker_across_sizes_matches_reference(ctx, ref, cfg):
    _run_against(ctx, ref, CFGS[cfg])


def test_tracker_size_change_is_opt_in(ctx):
    """Without sfmgpu_tracker_set_size_change a new size is refused by reset and step and changes nothing; turned on, the same
    tracker follows it; turned off again, it refuses again."""
    kw = dict(max_tracks=150, min_tracks=120)
    t, u = ctx.tracker(**kw), _follower(ctx, **kw)
    for tr in (t, u):
        tr.step(synth.frame(93, 0, 320, 240))
        tr.step(synth.frame(93, 1, 320, 240))
    small = synth.frame(93, 2, 256, 200)
    for call in (t.reset, t.step):
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            call(small)
        assert e.value.code == E_ARG
    for a, b in zip(t.tracks(), u.tracks()):  # the refused calls changed nothing
        assert a.tobytes() == b.tobytes()
    t.set_size_change(True)
    for a, b in zip(t.step(small), u.step(small)):
        assert a.tobytes() == b.tobytes()
    t.set_size_change(False)
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        t.step(synth.frame(93, 3, 320, 240))
    assert e.value.code == E_ARG
    assert ctx.lib.sfmgpu_tracker_set_size_change(ctx.h, t.h_, 2) == E_ARG


def test_tracker_size_change_keeps_the_step_frames_refusal(ctx):
    """A host step at a new size leaves the previous frame in the tracker's own batch: step_frames on another batch is
    still refused, and changes nothing."""
    t, u = _follower(ctx, max_tracks=150, min_tracks=120), _follower(ctx, max_tracks=150, min_tracks=120)
    for tr in (t, u):
        tr.step(synth.frame(92, 0, 320, 240))
        tr.step(synth.frame(92, 1, 400, 300))
    other = _frames(ctx, synth.frame(92, 2, 400, 300))
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        t.step_frames(other, 0)
    assert e.value.code == E_STATE
    img = synth.frame(92, 2, 352, 288)
    for a, b in zip(t.step(img), u.step(img)):
        assert a.tobytes() == b.tobytes()


def test_shim_tracker_across_sizes_equals_c_abi(ctx, szshim):
    cfg = CFGS["replenish"]
    t = _follower(ctx, **cfg)
    s = szshim.sz_tracker_create(cfg["max_tracks"], cfg["min_tracks"], 3)
    assert s, szshim.sz_last_error().decode()
    try:
        cap = t.cap
        for k, (seed, tt, w, h) in enumerate(SEQ):
            img = np.ascontiguousarray(_image(seed, tt, w, h))
            if seed == "reset":
                t.reset(img)
                _ck(szshim, szshim.sz_tracker_reset(s, img, w, h))
            else:
                prev, cur, ids = np.zeros((cap, 2)), np.zeros((cap, 2)), np.zeros(cap, np.int32)
                n = _ck(szshim, szshim.sz_tracker_step(s, img, w, h, prev, cur, ids, cap))
                gp, gc, gi = t.step(img)
                assert n == len(gi)
                assert prev[:n].tobytes() == gp.tobytes() and cur[:n].tobytes() == gc.tobytes() and np.array_equal(ids[:n], gi)
            xy, ids = np.zeros((cap, 2)), np.zeros(cap, np.int32)
            n = szshim.sz_tracker_tracks(s, xy, ids, cap)
            wx, wi = t.tracks()
            assert n == len(wi) and xy[:n].tobytes() == wx.tobytes() and np.array_equal(ids[:n], wi), f"step {k}"
    finally:
        szshim.sz_tracker_destroy(s)


def _shim_track_one(szshim, trk, pa, pb, p0):
    out = np.zeros_like(p0)
    _ck(szshim, szshim.sz_track_one(trk, pa, pb, p0, len(p0), out))
    return out


def _check_track_one(szshim, klt2, trk, a, b, im0, im1, p0, what):
    """track_one_public forward a -> b, then backward b -> a from the result, against the checker's track(A, B), track(B, A)."""
    p1 = _shim_track_one(szshim, trk, a, b, p0)
    pb = _shim_track_one(szshim, trk, b, a, p1)
    w1, wb = klt2(im0, im1, p0)
    st = _stable(klt2, im0, im1, p0, w1, wb) & np.isfinite(w1).all(1) & np.isfinite(wb).all(1)
    assert st.mean() >= 0.75
    dev = max(np.abs(p1[st] - w1[st]).max(), np.abs(pb[st] - wb[st]).max())
    print(f"track_one_public {what}: {st.sum()} of {len(p0)} points well conditioned, max |shim - checker| = {dev:.3e} px")
    assert dev <= BUDGET


def test_shim_track_one_public_between_sizes_and_pools(szshim, klt2):
    trk = szshim.sz_tracker_create(150, 120, 3)
    assert trk, szshim.sz_last_error().decode()
    pyrs = []
    try:
        # different sizes
        im0, im1 = synth.frame(45, 0, 640, 480), synth.frame(45, 1, 320, 240)
        a, b = szshim.sz_pyr_build(im0, 640, 480, 3), szshim.sz_pyr_build(im1, 320, 240, 3)
        pyrs += [a, b]
        assert a and b, szshim.sz_last_error().decode()
        p0 = _probe_points(640, 480, 320, 240, im0, 7)
        _check_track_one(szshim, klt2, trk, a, b, im0, im1, p0, "640x480 -> 320x240")
        # one size, nine live pyramids: a pool holds eight, so two of them sit in different pools
        imgs = [synth.frame(46, t, 352, 288) for t in range(9)]
        same = [szshim.sz_pyr_build(im, 352, 288, 3) for im in imgs]
        pyrs += same
        assert all(same), szshim.sz_last_error().decode()
        k = [i for i in range(1, 9) if not szshim.sz_same_pool(same[i - 1], same[i])]
        assert len(k) == 1
        i = k[0]
        p0 = _probe_points(352, 288, 352, 288, imgs[i - 1], 8)
        _check_track_one(szshim, klt2, trk, same[i - 1], same[i], imgs[i - 1], imgs[i], p0, "352x288, two pools")
    finally:
        for p in pyrs:
            if p:
                szshim.sz_pyr_free(p)
        szshim.sz_tracker_destroy(trk)
