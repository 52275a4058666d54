"""GPU tests of packed frames as the lock-step tracker's input (sfmgpu_multitracker_step_packed / prefetch_packed): blob frames
are copied into the tracker's own staging, decoded on the device and stepped, and every result - survivors, ids, n_out, track
lists, totals and the RANSAC stage's results - equals the same tracker stepped with the raw frames, byte for byte (the codec
is lossless).  Malformed blobs are refused before any work; records that do not decode fail the step and leave the tracker
exactly as it was."""
import ctypes as C

import numpy as np
import pytest

import frame_codec as fc
import ring_dataset
import sfmgpu
from conftest import TEMPLE_K
from sfmgpu import synth

pytestmark = pytest.mark.gpu

KW = dict(max_tracks=400, min_tracks=380)  # replenishment in most steps
RANSAC = (2500, 1e-3, 60, 1)  # find_E_ransac(K, prev, cur, 2500, 1e-3, 60) (:1739), skipped without survivors
OK = 2  # SFMGPU_TV_OK
E_ARG, E_STATE = -1, -4
T = 9  # frames per sequence: 8 steps after the first


def _ring(w, h, deg0, t):
    return ring_dataset.render(np.deg2rad(deg0 + 0.25 * t), w, h)


def _mixed_sequences(w, h):
    """[T, 5, h, w]: the ring scene, value noise, flat frames (every tile coded; no corners, so the sequence is reset on every
    frame), uniform noise (every tile stored raw), and value noise that turns flat for two frames (its tracks are lost, and
    it starts again on the next textured frame)."""
    rng = np.random.default_rng(5)
    seqs = [[_ring(w, h, 0.0, t) for t in range(T)],
            [synth.frame(20261201, t, w, h) for t in range(T)], [np.full((h, w), 77, np.uint8)] * T,
            [rng.integers(0, 256, (h, w), dtype=np.uint8) for _ in range(T)],
            [np.full((h, w), 90, np.uint8) if t in (3, 4) else synth.frame(20261202, t, w, h) for t in range(T)]]
    return np.ascontiguousarray(np.stack([np.stack([s[t] for s in seqs]) for t in range(T)]))


def _device_synth(ctx, w, h, S, seed0=20261203):
    """[T, S, h, w] of the bench's synthetic 1080p content, made on the device and downloaded."""
    out = np.zeros((T, S, h, w), np.uint8)
    for s in range(S):
        f = ctx.frames(w, h, T, 1)
        f.synth(0, T, seed0 + s, 0)
        for t in range(T):
            out[t, s] = f.download(t)
        f.close()
    return out


@pytest.fixture(scope="module")
def small():
    return _mixed_sequences(200, 150)  # not a multiple of the 64 x 64 tile


def _pack(ctx, imgs):
    """Blob of imgs [N, h, w] by the device encoder (byte-identical to tests/frame_codec.encode)."""
    imgs = np.ascontiguousarray(imgs)
    f = ctx.frames(imgs.shape[2], imgs.shape[1], len(imgs), 1)
    f.upload(0, imgs)
    blob = f.pack().copy()
    f.close()
    return blob


def _seq_blobs(ctx, frames):
    return [_pack(ctx, frames[:, s]) for s in range(frames.shape[1])]


def _step_major(ctx, frames):
    T_, S = frames.shape[:2]
    return _pack(ctx, frames.reshape(T_ * S, *frames.shape[2:]))


def _tracker(ctx, frames, ransac):
    mt = ctx.multitracker(frames.shape[1], frames.shape[3], frames.shape[2], **KW)
    if ransac:
        mt.set_ransac(TEMPLE_K, *RANSAC)
    return mt


def _record(mt, surv, ransac):
    return (surv, [mt.tracks(s) for s in range(mt.S)], mt.totals(), mt.ransac_results() if ransac else None)


def _state(mt):
    """Track lists, totals and stage results (what a refused or failed call must leave as it was)."""
    return _record(mt, [], True)


def _raw_run(ctx, frames, ransac=False):
    mt = _tracker(ctx, frames, ransac)
    out = [_record(mt, mt.step(frames[t]), ransac) for t in range(len(frames))]
    mt.close()
    return out


def _same(a, b):
    surv, trk, tot, rr = a
    surv2, trk2, tot2, rr2 = b
    assert len(surv) == len(surv2)
    for x, y in zip(surv, surv2):
        for u, v in zip(x, y):
            assert u.dtype == v.dtype and np.array_equal(u, v)
    for (xy, ids), (xy2, ids2) in zip(trk, trk2):
        assert np.array_equal(xy, xy2) and np.array_equal(ids, ids2)
    assert tot == tot2
    assert (rr is None) == (rr2 is None)
    if rr is not None:
        st, bn, inl, R, t = rr
        st2, bn2, inl2, R2, t2 = rr2
        assert np.array_equal(st, st2) and np.array_equal(bn, bn2)
        for s in range(len(st)):
            assert np.array_equal(inl[s], inl2[s]), s
        ok = st == OK
        assert np.array_equal(R[ok], R2[ok]) and np.array_equal(t[ok], t2[ok])  # R, t are written for poses only


def _same_run(got, want):
    assert len(got) == len(want)
    for t, (a, b) in enumerate(zip(got, want)):
        try:
            _same(a, b)
        except AssertionError as e:
            raise AssertionError(f"step {t}") from e


def _packed_run(ctx, frames, blobs, index, mode="plain", ransac=False):
    """Step a fresh tracker through frames with index(t) = the blob frame of every sequence at step t.  mode: plain steps,
    pipelined (next_frames), or prefetch_packed + step_packed(None)."""
    mt = _tracker(ctx, frames, ransac)
    out = []
    n = len(frames)
    for t in range(n):
        if mode == "plain":
            surv = mt.step_packed(blobs, index(t))
        elif mode == "pipelined":
            surv = mt.step_packed(blobs, index(t) if t == 0 else None, next_frames=index(t + 1) if t + 1 < n else None)
        else:
            mt.prefetch_packed(blobs, index(t))
            surv = mt.step_packed(blobs, None)
        out.append(_record(mt, surv, ransac))
    mt.close()
    return out


@pytest.mark.parametrize("case", ["ring_s1", "mixed_s5", "mixed_s5_ransac"])
def test_per_sequence_blobs(ctx, small, case):
    frames = small[:, :1] if case == "ring_s1" else small
    ransac = case.endswith("ransac")
    want = _raw_run(ctx, frames, ransac)
    got = _packed_run(ctx, frames, _seq_blobs(ctx, frames), lambda t: np.full(frames.shape[1], t), ransac=ransac)
    _same_run(got, want)


def test_1080p_four_sequences(ctx):
    frames = _device_synth(ctx, 1920, 1080, 4)
    want = _raw_run(ctx, frames, ransac=True)
    got = _packed_run(ctx, frames, _seq_blobs(ctx, frames), lambda t: np.full(4, t), ransac=True)
    _same_run(got, want)
    got = _packed_run(ctx, frames, _step_major(ctx, frames), lambda t: t * 4 + np.arange(4), mode="pipelined", ransac=True)
    _same_run(got, want)


def test_step_major_blob(ctx, small):
    frames = small
    S = frames.shape[1]
    want = _raw_run(ctx, frames)
    got = _packed_run(ctx, frames, _step_major(ctx, frames), lambda t: t * S + np.arange(S))
    _same_run(got, want)


def test_shared_blob_offsets_and_repeats(ctx, small):
    """One sequence-major blob read at different start frames, sequences 0 and 3 reading the same blob frames."""
    pool = small[:, 1]  # value noise, T frames
    blob = _pack(ctx, np.concatenate([pool, small[:, 0], small[:, 4]]))  # blob frames: pool, ring, noise turning flat
    starts = np.array([0, T, 2 * T, 0, 2])
    n = T - 2
    frames = np.stack([np.stack([pool[t], small[t, 0], small[t, 4], pool[t], pool[t + 2]]) for t in range(n)])
    want = _raw_run(ctx, frames)
    got = _packed_run(ctx, frames, blob, lambda t: starts + t)
    _same_run(got, want)
    got = _packed_run(ctx, frames, [blob] * 5, lambda t: starts + t, mode="prefetch")
    _same_run(got, want)


@pytest.mark.parametrize("mode", ["pipelined", "prefetch"])
@pytest.mark.parametrize("layout", ["per_sequence", "step_major"])
def test_pipelined_and_prefetch_forms(ctx, small, mode, layout):
    frames = small
    S = frames.shape[1]
    want = _raw_run(ctx, frames, ransac=True)
    if layout == "per_sequence":
        blobs, index = _seq_blobs(ctx, frames), (lambda t: np.full(S, t))
    else:
        blobs, index = _step_major(ctx, frames), (lambda t: t * S + np.arange(S))
    _same_run(_packed_run(ctx, frames, blobs, index, mode=mode, ransac=True), want)


def test_mixing_raw_and_packed(ctx, small):
    frames = small
    S = frames.shape[1]
    want = _raw_run(ctx, frames, ransac=True)
    blobs = _seq_blobs(ctx, frames)
    idx = lambda t: np.full(S, t)  # noqa: E731
    mt = _tracker(ctx, frames, True)
    got = [_record(mt, mt.step(frames[0]), True), _record(mt, mt.step_packed(blobs, idx(1)), True)]
    mt.prefetch(frames[2])
    got.append(_record(mt, mt.step_packed(blobs, None), True))  # a raw prefetch consumed by the packed call
    mt.prefetch_packed(blobs, idx(3))
    got.append(_record(mt, mt.step(None), True))  # a packed prefetch consumed by the raw call
    got.append(_record(mt, mt.step_packed(blobs, idx(4), next_frames=idx(5)), True))
    got.append(_record(mt, mt.step(None, next_imgs=frames[6]), True))
    got.append(_record(mt, mt.step_packed(blobs, None, next_frames=idx(7)), True))
    got.append(_record(mt, mt.step(None), True))
    got.append(_record(mt, mt.step(frames[8]), True))
    mt.close()
    _same_run(got, want)


# ---- refusals and records that do not decode ---------------------------------------------------------------------------
def _set_u32(blob, off, v):
    b = blob.copy()
    b[off:off + 4] = np.array([v], "<u4").view(np.uint8)
    return b


def _set_u64(blob, off, v):
    b = blob.copy()
    b[off:off + 8] = np.array([v], "<u8").view(np.uint8)
    return b


def _corrupt(blob, frame, tile=1):
    """The blob with the k table of one tile record of `frame` holding k = 15 (it does not decode, here or in the reference)."""
    H = fc.parse_header(blob)
    fb = int(H["frame_off"][frame])
    nt = len(fc.tile_grid(H["w"], H["h"]))
    toff = blob[fb:fb + 4 * (nt + 1)].view("<u4").astype(int)
    a, b = fb + toff[tile], fb + toff[tile + 1]
    out = blob.copy()
    rec = out[a:b].view("<u4")
    assert rec[0] != 1, "the tile is stored raw"
    rec[1] |= 0xF0000000
    x, y, tw, th = fc.tile_grid(H["w"], H["h"])[tile]
    with pytest.raises(ValueError):
        fc.decode_tile(rec.copy(), tw, th)
    return out


def _raw_call(ctx, mt, blobs, sizes, idx, nxt=None, prefetch=False):
    """The C entry point with hand-made arguments; returns its code."""
    S = mt.S
    p = None if blobs is None else (C.c_void_p * S)(*blobs)
    n = None if sizes is None else (C.c_size_t * S)(*sizes)
    i = None if idx is None else np.ascontiguousarray(idx, np.int32)
    j = None if nxt is None else np.ascontiguousarray(nxt, np.int32)
    vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    if prefetch:
        return ctx.lib.sfmgpu_multitracker_prefetch_packed(ctx.h, mt.h_, p, n, vp(i))
    return ctx.lib.sfmgpu_multitracker_step_packed(ctx.h, mt.h_, p, n, vp(i), vp(j), None, None, None, None)


def test_refusals_before_any_work(ctx, small):
    frames = small
    S, h, w = frames.shape[1], frames.shape[2], frames.shape[3]
    want = _raw_run(ctx, frames, ransac=True)
    blob = _step_major(ctx, frames)  # blob frame t*S + s
    nf = T * S
    fo = fc.parse_header(blob)["frame_off"]
    other = _pack(ctx, np.stack([synth.frame(7, 0, 208, 150)] * nf))
    oversize = np.concatenate([blob, np.zeros(64 << 10, np.uint8)])
    oversize = _set_u64(oversize, fc.HEADER_BYTES + 8 * nf, int(fo[nf]) + (64 << 10))  # the last frame's record grows
    bad_blobs = {
        "magic": _set_u32(blob, 0, 0x12345678),
        "version": _set_u32(blob, 4, 2),
        "tile": _set_u32(blob, 20, 32),
        "width": _set_u32(blob, 8, w + 1),
        "other_size": other,
        "truncated": blob[:int(fo[nf]) - 8],
        "non_monotonic": _set_u64(blob, fc.HEADER_BYTES + 8 * (nf - 1), int(fo[nf - 2]) - 4),
        "misaligned": _set_u64(blob, fc.HEADER_BYTES + 8 * (nf - 1), int(fo[nf - 1]) + 2),
        "past_the_end": _set_u64(blob, fc.HEADER_BYTES + 8 * nf, len(blob) + 64),
        "oversize_record": oversize,
    }
    mt = _tracker(ctx, frames, True)
    last = (T - 1) * S + np.arange(S)  # the last step's frames: the tests above touch their offsets
    got = []
    for t in range(T):
        idx = t * S + np.arange(S)
        if t >= 2:
            before = _state(mt)
            addr, size = blob.ctypes.data, blob.nbytes
            if t == T - 1:
                for name, b in bad_blobs.items():
                    for pf in (False, True):
                        rc = _raw_call(ctx, mt, [b.ctypes.data] * S, [b.nbytes] * S, idx, prefetch=pf)
                        assert rc == E_ARG, (name, pf, rc)
            codes = [
                _raw_call(ctx, mt, None, [size] * S, idx),  # null blob array
                _raw_call(ctx, mt, [addr] * S, None, idx),  # null size array
                _raw_call(ctx, mt, [addr] * (S - 1) + [None], [size] * S, idx),  # null entry
                _raw_call(ctx, mt, [addr] * S, [size] * S, [0, 1, 2, 3, nf]),  # frame outside the blob
                _raw_call(ctx, mt, [addr] * S, [size] * S, [0, -1, 2, 3, 4]),
                _raw_call(ctx, mt, [addr] * S, [size] * S, idx, nxt=[0, 1, 2, 3, nf]),  # a bad next index: nothing done
                _raw_call(ctx, mt, None, None, idx, nxt=idx),
                _raw_call(ctx, mt, [addr] * S, [size] * S, None, prefetch=True),  # prefetch without indices
                _raw_call(ctx, mt, None, None, None),  # nothing given, nothing prefetched
            ]
            assert codes == [E_ARG] * 8 + [E_STATE], codes
            mt.prefetch_packed(blob, idx)
            assert _raw_call(ctx, mt, [addr] * S, [size] * S, last) == E_STATE  # frames given while others are prefetched
            assert _raw_call(ctx, mt, [addr] * S, [size] * S, last, prefetch=True) == E_STATE
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                mt.step_frames(ctx.frames(w, h, 1, 3), [0] * S)
            assert e.value.code == E_STATE
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                mt.prefetch(frames[t])
            assert e.value.code == E_STATE
            _same(_state(mt), before)  # nothing changed
            got.append(_record(mt, mt.step_packed(blob, None), True))
        else:
            got.append(_record(mt, mt.step_packed(blob, idx), True))
    mt.close()
    _same_run(got, want)


@pytest.mark.parametrize("how", ["given", "prefetched", "pipelined", "prefetched_raw_step"])
def test_corrupt_records(ctx, small, how):
    frames = small
    S = frames.shape[1]
    want = _raw_run(ctx, frames, ransac=True)
    blobs = _seq_blobs(ctx, frames)
    bad = list(blobs)
    bad[1] = _corrupt(blobs[1], 4)  # frame 4 of sequence 1 (value noise)
    idx = lambda t: np.full(S, t)  # noqa: E731
    mt = _tracker(ctx, frames, True)
    got = []
    for t in range(T):
        if t == 4:
            before = _state(mt)
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                if how == "given":
                    mt.step_packed(bad, idx(4))
                elif how == "prefetched":
                    mt.prefetch_packed(bad, idx(4))
                    mt.step_packed(bad, None)
                elif how == "pipelined":
                    mt.step_packed(bad, None)  # prefetched by step 3
                else:
                    mt.prefetch_packed(bad, idx(4))
                    mt.step(None)
            assert e.value.code == E_ARG
            _same(_state(mt), before)  # tracker and stage results as before the call
            assert _raw_call(ctx, mt, None, None, None) == E_STATE  # no prefetch pending
        if how == "pipelined" and t == 3:  # frame 3 of the corrupt blob decodes; frame 4 is its prefetch
            got.append(_record(mt, mt.step_packed(bad, idx(3), next_frames=idx(4)), True))
        else:
            got.append(_record(mt, mt.step_packed(blobs, idx(t)), True))
    mt.close()
    _same_run(got, want)


def test_staging_isolation(ctx, small):
    """Packed calls of the context between a prefetch and its step (other blobs, larger than the prefetch) change nothing."""
    frames = small
    S = frames.shape[1]
    want = _raw_run(ctx, frames, ransac=True)
    blobs = _seq_blobs(ctx, frames)
    rng = np.random.default_rng(9)
    noise = rng.integers(0, 256, (12, 480, 640), dtype=np.uint8)
    other = _pack(ctx, noise)
    fr = ctx.frames(640, 480, 12, 3)
    pairs = ctx.pairs(12, 600)
    cfg = sfmgpu.lkcfg(max_tracks=600, min_tracks=300)
    mt = _tracker(ctx, frames, True)
    got = []
    for t in range(T):
        mt.prefetch_packed(blobs, np.full(S, t))
        fr.upload_packed(0, other)
        pairs.run_host_packed(fr, other, 12, cfg, chunk=4)
        got.append(_record(mt, mt.step_packed(blobs, None), True))
    assert np.array_equal(fr.download(11), noise[11])
    mt.close()
    _same_run(got, want)
