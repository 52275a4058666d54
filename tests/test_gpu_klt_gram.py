"""The Gram build of klt_quad_kernel (the default, integer MMA over raw taps) against the FFMA build (klt mode 17): both
compute the same integer matrices, so every KLT output must be byte-identical, including the features deferred to the
border kernels, and so must the two-view unit's results with the RANSAC stage on."""
import numpy as np
import pytest

from conftest import TEMPLE_K
from sfmgpu import synth
import sfmgpu

pytestmark = pytest.mark.gpu

FFMA = 17  # lane path, tuning variant 7: the FFMA build
GRAM = 2   # lane path, default variant: the Gram build


def _frames(ctx, imgs, levels=3):
    h, w = imgs[0].shape
    f = ctx.frames(w, h, len(imgs), levels)
    f.upload(0, np.stack(imgs))
    f.build_pyramid()
    return f


def _track(ctx, f, pts, mode):
    ctx.klt_set_mode(mode)
    try:
        return f.klt_track(0, 1, pts, count=True)
    finally:
        ctx.klt_set_mode(0)


def _noise(rng, w, h):
    a = rng.integers(0, 256, (h, w), dtype=np.uint8)
    return a, np.roll(a, (1, 2), (0, 1))


def _cases():
    rng = np.random.default_rng(20261020)
    flat = np.full((720, 1280), 90, np.uint8)
    return {
        "c2": ([synth.frame(5, 0, 1920, 1080), synth.frame(5, 1, 1920, 1080)], 2000),
        "c3": ([synth.frame(6, 0, 3840, 2160), synth.frame(6, 1, 3840, 2160)], 8000),
        "noise": (list(_noise(rng, 1280, 720)), 0),
        "flat": ([flat, flat], 0),
    }


@pytest.mark.parametrize("case", ["c2", "c3", "noise", "flat"])
def test_klt_gram_build_is_byte_identical(ctx, case):
    imgs, ncorn = _cases()[case]
    h, w = imgs[0].shape
    f = _frames(ctx, imgs)
    rng = np.random.default_rng(len(case))
    pts = [rng.uniform(0, 1, (6000, 2)) * [w, h]]  # random positions, many of them near the border (deferred)
    if ncorn:
        pts.append(f.corners(0, ncorn))
    edge = rng.uniform(0, 14, (1500, 2))  # windows touching each border: deferral to the masked kernel must be unchanged
    pts += [edge, [w, h] - edge, edge * [1, 0] + [0, h / 2], [w - 1, h / 2] - edge * [1, 0]]
    pts = np.concatenate(pts)
    p1, pb, nit = _track(ctx, f, pts, GRAM)
    q1, qb, qit = _track(ctx, f, pts, FFMA)
    assert p1.tobytes() == q1.tobytes() and pb.tobytes() == qb.tobytes() and np.array_equal(nit, qit)
    assert nit.sum() > 0


def test_pairs_with_ransac_byte_identical(ctx):
    """pairs.run with the RANSAC stage on: corners, survivors (the fb keep decision), points and poses."""
    W, H, P = 1920, 1080, 6
    imgs = [synth.frame(20261020, t, W, H) for t in range(P + 1)]
    imgs[4] = np.full((H, W), 90, np.uint8)
    cap = 2000
    cfg = sfmgpu.lkcfg(max_tracks=cap)
    f = _frames(ctx, imgs)
    out = {}
    for mode in (GRAM, FFMA):
        pairs = ctx.pairs(P, cap)
        pairs.set_ransac(TEMPLE_K, 400, 2e-3, 80, 120)
        ctx.klt_set_mode(mode)
        try:
            pairs.run(f, 0, P, cfg)
        finally:
            ctx.klt_set_mode(0)
        li, lj = np.zeros((P, cap, 2)), np.zeros((P, cap, 2))
        nk, nc = np.zeros(P, np.int32), np.zeros(P, np.int32)
        st, bn = np.zeros(P, np.int32), np.zeros(P, np.int32)
        inl, R, t = np.zeros((P, cap), np.int32), np.zeros((P, 9)), np.zeros((P, 3))
        pairs.download_all(li, lj, nk, nc)
        pairs.ransac_download_all(st, bn, inl, R, t)
        out[mode] = (li, lj, nk, nc, st, bn, inl, R, t)
        pairs.close()
    (li, lj, nk, nc, st, bn, inl, R, t), want = out[GRAM], out[FFMA]
    for a, b in zip((nk, nc, st, bn), want[2:6]):
        assert a.tobytes() == b.tobytes()
    ok = st == 2
    assert R[ok].tobytes() == want[7][ok].tobytes() and t[ok].tobytes() == want[8][ok].tobytes()
    for p in range(P):
        assert li[p, :nk[p]].tobytes() == want[0][p, :nk[p]].tobytes() and lj[p, :nk[p]].tobytes() == want[1][p, :nk[p]].tobytes()
        assert np.array_equal(inl[p, :bn[p]], want[6][p, :bn[p]])
    assert (out[GRAM][2] > 0).sum() >= P - 1 and (out[GRAM][4] == 2).any()
