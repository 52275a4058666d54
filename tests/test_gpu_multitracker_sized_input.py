"""Packed and resident input for lock-step trackers whose sequences have different image sizes.

Packed blobs are decoded by one launch over all S frames of a step, each into its own size class's slot, and the pyramids are
built per class; resident frames come from one batch per sequence (sfmgpu_multitracker_step_frames_sized), gathered by one
launch over a (sequence, level) table.  Both must give, byte for byte, what raw steps with the same images give: survivors,
ids, counts, track lists, totals and the per-camera RANSAC stage.  The sizes have partial edge tiles and row padding at every
pyramid level (333 x 251, 200 x 150), one is smaller than a 64 x 64 tile (61 x 45), and the classes are not adjacent
([A, B, A, C, B]).  Sequence 2 shows sequence 0's images, so two sequences read one batch at the same indices."""
import ctypes as C

import numpy as np
import pytest

import frame_codec as fc
import sfmgpu
from sfmgpu import synth

pytestmark = pytest.mark.gpu

E_ARG, E_STATE = -1, -4
OK = 2  # SFMGPU_TV_OK
SIZES = [(333, 251), (61, 45), (333, 251), (200, 150), (61, 45)]
SEEDS = [4100, 4101, 4100, 4103, 4104]
S = len(SIZES)
T = 7
WARP = dict(max_tracks=150, min_tracks=140)     # S x ROWS < 6000: the warp-per-feature kernel
LANE = dict(max_tracks=1300, min_tracks=1250)   # S x ROWS >= 6000: the lane chain
RANSAC = (500, 1e-3, 30, 1)


def _K(w, h, s):
    a, b = w / 640.0, h / 480.0
    return np.array([[1520.4 * a * (1 + 0.01 * s), 0, 302.32 * a + 2 * s], [0, 1525.9 * a * (1 + 0.01 * s), 246.87 * b - s], [0, 0, 1.0]])


@pytest.fixture(scope="module")
def seqs():
    """seqs[s][t]: value noise of sequence s; sequence 4 turns flat for two frames (its tracks are lost and it restarts)."""
    return [[np.full((h, w), 90, np.uint8) if s == 4 and t in (3, 4) else synth.frame(SEEDS[s], t, w, h) for t in range(T)]
            for s, (w, h) in enumerate(SIZES)]


def _tracker(ctx, kw, sizes=SIZES):
    mt = ctx.multitracker(len(sizes), [w for w, _ in sizes], [h for _, h in sizes], **kw)
    mt.set_ransac(np.stack([_K(w, h, s) for s, (w, h) in enumerate(sizes)]), *RANSAC)
    return mt


def _record(mt, surv):
    return (surv, [mt.tracks(s) for s in range(mt.S)], mt.totals(), mt.ransac_results())


def _same(a, b, where):
    surv, trk, tot, rr = a
    surv2, trk2, tot2, rr2 = b
    assert len(surv) == len(surv2), where
    for x, y in zip(surv, surv2):
        for u, v in zip(x, y):
            assert u.dtype == v.dtype and np.array_equal(u, v), where
    for (xy, ids), (xy2, ids2) in zip(trk, trk2):
        assert np.array_equal(xy, xy2) and np.array_equal(ids, ids2), where
    assert tot == tot2, where
    st, bn, inl, R, t = rr
    st2, bn2, inl2, R2, t2 = rr2
    assert np.array_equal(st, st2) and np.array_equal(bn, bn2), where
    for s in range(len(st)):
        assert np.array_equal(inl[s], inl2[s]), (where, s)
    ok = st == OK
    assert np.array_equal(R[ok], R2[ok]) and np.array_equal(t[ok], t2[ok]), where  # R, t are written for poses only


def _same_run(got, want, what):
    assert len(got) == len(want), what
    for t, (a, b) in enumerate(zip(got, want)):
        _same(a, b, (what, t))


def _raw_run(ctx, seqs, kw):
    mt = _tracker(ctx, kw)
    out = [_record(mt, mt.step([sq[t] for sq in seqs])) for t in range(T)]
    mt.close()
    return out


def _pack(ctx, imgs):
    imgs = np.ascontiguousarray(np.stack(imgs))
    f = ctx.frames(imgs.shape[2], imgs.shape[1], len(imgs), 1)
    f.upload(0, imgs)
    blob = f.pack().copy()
    f.close()
    return blob


def _classes():
    """{size: [sequences of that size]} in sequence order."""
    cls = {}
    for s, wh in enumerate(SIZES):
        cls.setdefault(wh, []).append(s)
    return cls


def _per_sequence(ctx, seqs):
    """One blob per sequence; sequence s's frame t is blob frame t."""
    return [_pack(ctx, seqs[s]) for s in range(S)], (lambda t: np.full(S, t))


def _per_class(ctx, seqs):
    """One step-major blob per size class: frame t of the i-th sequence of class c is blob frame t * n_c + i."""
    blobs, pos = [None] * S, np.zeros(S, np.int64)
    n = np.zeros(S, np.int64)
    for members in _classes().values():
        b = _pack(ctx, [seqs[s][t] for t in range(T) for s in members])
        for i, s in enumerate(members):
            blobs[s], pos[s], n[s] = b, i, len(members)
    return blobs, (lambda t: t * n + pos)


def _batches(ctx, seqs):
    """Resident input: one batch per size holding every distinct sequence of that size (pyramids built), and per step the
    batch and frame index of every sequence.  Sequences 0 and 2 read the same frames of one batch."""
    batches, where = {}, [None] * S
    for (w, h), members in _classes().items():
        seeds = sorted({SEEDS[s] for s in members})
        f = ctx.frames(w, h, len(seeds) * T, 3)
        for k, sd in enumerate(seeds):
            s = members[[SEEDS[m] for m in members].index(sd)]
            f.upload(k * T, np.stack(seqs[s]))
        f.build_pyramid()
        batches[(w, h)] = f
        for s in members:
            where[s] = (f, seeds.index(SEEDS[s]) * T)
    fs = [where[s][0] for s in range(S)]
    return batches, fs, (lambda t: np.array([where[s][1] + t for s in range(S)]))


@pytest.mark.parametrize("family", ["warp", "lane"])
def test_resident_equals_raw(ctx, seqs, family):
    kw = WARP if family == "warp" else LANE
    want = _raw_run(ctx, seqs, kw)
    batches, fs, idx = _batches(ctx, seqs)
    mt = _tracker(ctx, kw)
    got = [_record(mt, mt.step_frames(fs, idx(t))) for t in range(T)]
    mt.close()
    _same_run(got, want, "resident")
    for f in batches.values():
        f.close()


@pytest.mark.parametrize("family", ["warp", "lane"])
def test_packed_equals_raw(ctx, seqs, family):
    kw = WARP if family == "warp" else LANE
    want = _raw_run(ctx, seqs, kw)
    layouts = {"per_sequence": _per_sequence(ctx, seqs), "per_class": _per_class(ctx, seqs)}
    for name, (blobs, idx) in layouts.items():
        for mode in ("plain", "prefetch", "next_frames", "pipelined_raw_step"):
            mt = _tracker(ctx, kw)
            got = []
            for t in range(T):
                nxt = idx(t + 1) if t + 1 < T else None
                if mode == "plain":
                    surv = mt.step_packed(blobs, idx(t))
                elif mode == "prefetch":
                    mt.prefetch_packed(blobs, idx(t))
                    surv = mt.step_packed(blobs, None)
                elif mode == "next_frames":
                    surv = mt.step_packed(blobs, idx(t) if t == 0 else None, next_frames=nxt)
                else:  # sfmgpu_multitracker_step_pipelined(host_pix = NULL) consumes a packed prefetch
                    if t == 0:
                        mt.prefetch_packed(blobs, idx(0))
                    surv = mt.step(None)
                    if nxt is not None:
                        mt.prefetch_packed(blobs, nxt)
                got.append(_record(mt, surv))
            mt.close()
            _same_run(got, want, (name, mode))


def test_alternating_raw_packed_resident(ctx, seqs):
    """Raw, packed and resident steps in one run, so that every input form writes every slot group."""
    want = _raw_run(ctx, seqs, WARP)
    blobs, pidx = _per_sequence(ctx, seqs)
    batches, fs, ridx = _batches(ctx, seqs)
    raw = lambda t: [sq[t] for sq in seqs]  # noqa: E731
    mt = _tracker(ctx, WARP)
    got = [_record(mt, mt.step(raw(0))), _record(mt, mt.step_packed(blobs, pidx(1))), _record(mt, mt.step_frames(fs, ridx(2)))]
    mt.prefetch_packed(blobs, pidx(3))
    got.append(_record(mt, mt.step(None, next_imgs=raw(4))))  # packed prefetch consumed, raw prefetch queued
    got.append(_record(mt, mt.step_packed(blobs, None, next_frames=pidx(5))))  # raw prefetch consumed, packed one queued
    got.append(_record(mt, mt.step(None)))
    got.append(_record(mt, mt.step_frames(fs, ridx(6))))
    mt.close()
    _same_run(got, want, "alternating")
    for f in batches.values():
        f.close()


def test_one_size_sized_equals_step_frames(ctx):
    """On a one-size tracker step_frames_sized with every f[s] = f is step_frames byte for byte, and so is the same run with
    the sequences split over two batches of that size."""
    n, w, h = 4, 320, 240
    imgs = np.stack([np.stack([synth.frame(4200 + s, t, w, h) for t in range(T)]) for s in range(n)])  # [s][t]
    f = ctx.frames(w, h, n * T, 3)
    f.upload(0, imgs.reshape(n * T, h, w))
    f.build_pyramid()
    halves = []
    for k in range(2):  # batch k holds sequences k and k + 2
        b = ctx.frames(w, h, 2 * T, 3)
        b.upload(0, imgs[[k, k + 2]].reshape(2 * T, h, w))
        b.build_pyramid()
        halves.append(b)
    idx = lambda t: np.arange(n) * T + t  # noqa: E731
    runs = {}
    for form in ("step_frames", "sized_one_batch", "sized_two_batches"):
        mt = ctx.multitracker(n, w, h, **WARP)
        mt.set_ransac(np.stack([_K(w, h, s) for s in range(n)]), *RANSAC)
        out = []
        for t in range(T):
            if form == "step_frames":
                surv = mt.step_frames(f, idx(t))
            elif form == "sized_one_batch":
                surv = mt.step_frames([f] * n, idx(t))
            else:
                surv = mt.step_frames([halves[0], halves[1], halves[0], halves[1]], np.array([0, 0, T, T]) + t)
            out.append(_record(mt, surv))
        runs[form] = out
        mt.close()
    _same_run(runs["sized_one_batch"], runs["step_frames"], "one batch")
    _same_run(runs["sized_two_batches"], runs["step_frames"], "two batches")
    for b in [f] + halves:
        b.close()


# ---- refusals ---------------------------------------------------------------------------------------------------------------
def _state(mt):
    return ([mt.tracks(s) for s in range(mt.S)], mt.totals(), mt.ransac_results())


def _same_state(a, b, where):
    _same(([],) + a, ([],) + b, where)


def _sized_call(ctx, mt, fs, idx):
    p = None if fs is None else (C.c_void_p * mt.S)(*[None if f is None else f.h_ for f in fs])
    i = None if idx is None else np.ascontiguousarray(idx, np.int32)
    return ctx.lib.sfmgpu_multitracker_step_frames_sized(ctx.h, mt.h_, p, None if i is None else i.ctypes.data_as(C.c_void_p),
                                                         None, None, None, None)


def _packed_call(ctx, mt, blobs, idx, prefetch=False):
    p = (C.c_void_p * mt.S)(*[None if b is None else b.ctypes.data for b in blobs])
    n = (C.c_size_t * mt.S)(*[0 if b is None else b.nbytes for b in blobs])
    i = None if idx is None else np.ascontiguousarray(idx, np.int32)
    vi = None if i is None else i.ctypes.data_as(C.c_void_p)
    if prefetch:
        return ctx.lib.sfmgpu_multitracker_prefetch_packed(ctx.h, mt.h_, p, n, vi)
    return ctx.lib.sfmgpu_multitracker_step_packed(ctx.h, mt.h_, p, n, vi, None, None, None, None, None)


def _corrupt(blob, frame, tile=1):
    """The blob with the k table of one coded tile record of `frame` holding k = 15 (it does not decode)."""
    H = fc.parse_header(blob)
    fb = int(H["frame_off"][frame])
    nt = len(fc.tile_grid(H["w"], H["h"]))
    toff = blob[fb:fb + 4 * (nt + 1)].view("<u4").astype(int)
    out = blob.copy()
    rec = out[fb + toff[tile]:fb + toff[tile + 1]].view("<u4")
    assert rec[0] != 1, "the tile is stored raw"
    rec[1] |= 0xF0000000
    return out


def _grown_last_record(blob, extra):
    """The blob with its last frame record `extra` bytes longer (zeros appended, the frame table moved)."""
    H = fc.parse_header(blob)
    nf = len(H["frame_off"]) - 1
    out = np.concatenate([blob, np.zeros(extra, np.uint8)])
    o = fc.HEADER_BYTES + 8 * nf
    out[o:o + 8] = np.array([int(H["frame_off"][nf]) + extra], "<u8").view(np.uint8)
    return out


def test_resident_refusals(ctx, seqs):
    want = _raw_run(ctx, seqs, WARP)
    batches, fs, idx = _batches(ctx, seqs)
    fewer_levels = ctx.frames(*SIZES[3], T, 2)
    mt = _tracker(ctx, WARP)
    got = []
    for t in range(T):
        if t == 3:
            before = _state(mt)
            wrong_size = list(fs)
            wrong_size[3] = fs[0]  # a 333 x 251 batch for the 200 x 150 sequence 3
            wrong_levels = list(fs)
            wrong_levels[3] = fewer_levels
            outside = idx(t)
            outside[4] = 2 * T  # the 61 x 45 batch holds two sequences of T frames
            negative = idx(t)
            negative[1] = -1
            codes = [_sized_call(ctx, mt, None, idx(t)), _sized_call(ctx, mt, fs, None),
                     _sized_call(ctx, mt, fs[:2] + [None] + fs[3:], idx(t)),
                     _sized_call(ctx, mt, wrong_size, idx(t)), _sized_call(ctx, mt, wrong_levels, idx(t)),
                     _sized_call(ctx, mt, fs, outside), _sized_call(ctx, mt, fs, negative)]
            assert codes == [E_ARG] * 7, codes
            for bad, s in ((wrong_size, 3), (wrong_levels, 3)):
                with pytest.raises(sfmgpu.SfmGpuError) as e:
                    mt.step_frames(bad, idx(t))
                assert e.value.code == E_ARG and f"sequence {s}" in str(e.value)
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                mt.step_frames(fs, outside)
            assert e.value.code == E_ARG and "sequence 4" in str(e.value)
            _same_state(_state(mt), before, "refused")
            mt.prefetch([sq[t] for sq in seqs])
            assert _sized_call(ctx, mt, fs, idx(t)) == E_STATE  # prefetched frames not yet stepped
            got.append(_record(mt, mt.step(None)))
        else:
            got.append(_record(mt, mt.step_frames(fs, idx(t))))
    mt.close()
    _same_run(got, want, "after refusals")
    fewer_levels.close()
    for f in batches.values():
        f.close()


@pytest.mark.parametrize("how", ["given", "prefetched"])
def test_packed_refusals_and_corrupt_records(ctx, seqs, how):
    want = _raw_run(ctx, seqs, WARP)
    blobs, idx = _per_sequence(ctx, seqs)
    wrong_size = list(blobs)
    wrong_size[3] = blobs[0].copy()  # a 333 x 251 blob for the 200 x 150 sequence 3
    shared = [blobs[0]] * S  # one blob for sequences of three sizes
    grown = list(blobs)
    grown[1] = _grown_last_record(blobs[1], 8192)  # above the 61 x 45 bound, below the 333 x 251 one
    corrupt = list(blobs)
    corrupt[2] = _corrupt(blobs[2], 4)  # frame 4 of sequence 2
    pf = how == "prefetched"
    mt = _tracker(ctx, WARP)
    got = []
    for t in range(T):
        if t == 4:
            before = _state(mt)
            assert _packed_call(ctx, mt, blobs, None) == E_STATE  # nothing given, nothing prefetched
            for bad, frame_idx, word in ((wrong_size, idx(t), "sequence 3"), (shared, idx(t), "different image sizes"),
                                         (grown, np.full(S, T - 1), "sequence 1")):
                assert _packed_call(ctx, mt, bad, frame_idx, prefetch=pf) == E_ARG
                with pytest.raises(sfmgpu.SfmGpuError) as e:
                    if pf:
                        mt.prefetch_packed(bad, frame_idx)
                    else:
                        mt.step_packed(bad, frame_idx)
                assert e.value.code == E_ARG and word in str(e.value), (word, str(e.value))
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                if pf:
                    mt.prefetch_packed(corrupt, idx(t))
                    assert _packed_call(ctx, mt, blobs, idx(t)) == E_STATE  # frames given while others are prefetched
                    mt.step_packed(corrupt, None)
                else:
                    mt.step_packed(corrupt, idx(t))
            assert e.value.code == E_ARG and "does not decode" in str(e.value)
            _same_state(_state(mt), before, "refused")
            assert _packed_call(ctx, mt, blobs, None) == E_STATE  # no prefetch pending
        got.append(_record(mt, mt.step_packed(blobs, idx(t))))
    mt.close()
    _same_run(got, want, "after refusals")
