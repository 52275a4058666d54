"""The tracker objects' refusals and their KLT launch sizing.

Both sfmgpu_tracker and sfmgpu_multitracker run on one track-list core; what stays per object is pinned here.  The single
tracker reads its previous frame in place (a frame of another batch is refused), downloads only its survivors into the caller's
capacity (too small: refused before the track list changes), and sizes its KLT launch by its live tracks.  The lock-step
tracker sizes its launch by all S x rows entries.  The automatic KLT choice takes the lane-per-feature kernel for launches of at
least 6000 slots, and the lane and warp kernels agree to within 1e-6 px but not bit for bit, so a byte-for-byte comparison
with a forced kernel family pins the family a launch took."""
import ctypes as C

import numpy as np
import pytest

import sfmgpu
from sfmgpu import synth

pytestmark = pytest.mark.gpu
W, H = 320, 240
KW = dict(max_tracks=150, min_tracks=120)
E_ARG, E_CAPACITY, E_STATE = -1, -3, -4


def _frames(ctx, imgs, levels=3):
    f = ctx.frames(imgs[0].shape[1], imgs[0].shape[0], len(imgs), levels)
    f.upload(0, np.stack(imgs))
    f.build_pyramid()
    return f


def _vp(a):
    return a.ctypes.data_as(C.c_void_p)


def test_tracker_refuses_a_previous_frame_of_another_batch(ctx):
    imgs = [synth.frame(71, t, W, H) for t in range(3)]
    fa, fb = _frames(ctx, imgs[:2]), _frames(ctx, imgs[1:])
    t = ctx.tracker(**KW)
    t.step_frames(fa, 0)  # reset
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        t.step_frames(fb, 0)
    assert e.value.code == E_STATE
    ref = ctx.tracker(**KW)
    ref.step_frames(fa, 0)
    for a, b in zip(t.step_frames(fa, 1), ref.step_frames(fa, 1)):  # the refused call changed nothing
        assert np.array_equal(a, b)


def test_tracker_step_refuses_a_small_cap_before_changing_its_tracks(ctx):
    imgs = [synth.frame(72, t, W, H) for t in range(3)]
    f = _frames(ctx, imgs)
    t = ctx.tracker(**KW)
    t.step_frames(f, 0)
    t.step_frames(f, 1)
    xy0, ids0 = t.tracks()
    assert len(ids0) > 1
    prev, cur, ids = np.zeros((t.cap, 2)), np.zeros((t.cap, 2)), np.zeros(t.cap, np.int32)
    n = C.c_int(-1)
    rc = ctx.lib.sfmgpu_tracker_step_frames(ctx.h, t.h_, f.h_, 2, _vp(prev), _vp(cur), _vp(ids), 1, C.byref(n))
    assert rc == E_CAPACITY
    xy1, ids1 = t.tracks()
    assert np.array_equal(xy1, xy0) and np.array_equal(ids1, ids0)


def test_tracker_tracks_refuses_a_small_cap(ctx):
    t = ctx.tracker(**KW)
    t.step(synth.frame(73, 0, W, H))
    _, want = t.tracks()
    assert len(want) > 1
    xy, ids = np.zeros((t.cap, 2)), np.zeros(t.cap, np.int32)
    n = C.c_int(-1)
    assert ctx.lib.sfmgpu_tracker_tracks(ctx.h, t.h_, xy, ids, 1, C.byref(n)) == E_CAPACITY
    assert n.value == len(want)


def test_tracker_refuses_a_new_image_size(ctx):
    t = ctx.tracker(**KW)
    t.step(synth.frame(74, 0, W, H))
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        t.step(synth.frame(74, 1, W // 2, H // 2))
    assert e.value.code == E_ARG


def _run_modes(ctx, modes, make, step, lists, T):
    """One tracker per KLT mode through the same T steps; per mode and step: (the step's results, the track lists after it)."""
    trackers = [make() for _ in modes]
    out = [[] for _ in modes]
    try:
        for t in range(T):
            for i, (m, tr) in enumerate(zip(modes, trackers)):
                ctx.klt_set_mode(m)
                out[i].append((step(tr, t), lists(tr)))
    finally:
        ctx.klt_set_mode(0)
    return out


def test_tracker_klt_launch_is_sized_by_live_tracks(ctx):
    """rows >= 6000 but fewer live tracks: the automatic choice is the warp kernel, byte-identical to forcing it."""
    w, h, T = 640, 480, 5
    kw = dict(max_tracks=7000, min_tracks=900)
    imgs = [synth.frame(75, t, w, h) for t in range(T)]
    res = _run_modes(ctx, [0, 1], lambda: ctx.tracker(**kw), lambda tr, t: tr.step(imgs[t]), lambda tr: tr.tracks(), T)
    for t in range(T):
        (ga, ta), (gb, tb) = res[0][t], res[1][t]
        assert len(ta[1]) < 6000, len(ta[1])
        for a, b in zip(ga, gb):
            assert np.array_equal(a, b), t
        for a, b in zip(ta, tb):
            assert np.array_equal(a, b), t


def test_multitracker_klt_launch_is_sized_by_all_rows(ctx):
    """S x rows >= 6000 with few live tracks: the automatic choice is the lane kernel, byte-identical to forcing it."""
    S, T = 4, 5
    kw = dict(max_tracks=2000, min_tracks=818)  # S x 2001 rows >= 6000; a 320x240 frame holds far fewer corners
    seqs = [[synth.frame(76 + s, t, W, H) for t in range(T)] for s in range(S)]
    res = _run_modes(ctx, [0, 2], lambda: ctx.multitracker(S, W, H, **kw),
                     lambda tr, t: tr.step(np.stack([seqs[s][t] for s in range(S)])), lambda tr: [tr.tracks(s) for s in range(S)], T)
    for t in range(T):
        (ga, ta), (gb, tb) = res[0][t], res[1][t]
        assert sum(len(x[1]) for x in ta) < 6000
        for s in range(S):
            for a, b in zip(ga[s], gb[s]):
                assert np.array_equal(a, b), (t, s)
            for a, b in zip(ta[s], tb[s]):
                assert np.array_equal(a, b), (t, s)
