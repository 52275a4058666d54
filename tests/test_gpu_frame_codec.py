"""Packed frame input on the device: the encoder writes the reference codec's bytes (tests/frame_codec.py), the decoder turns
reference blobs back into level 0 exactly as a raw upload writes it, and every consumer of decoded frames - the resident pair
calls and the streaming host call - gives byte-identical results to the raw path.  Malformed blobs are refused before any
work, and tile records that do not decode are reported and not written."""
import ctypes as C

import numpy as np
import pytest

import frame_codec as fc
import sfmgpu
from conftest import TEMPLE_K
from sfmgpu import synth

pytestmark = pytest.mark.gpu

IMAGES = fc.sample_images()
CFG = dict(max_tracks=600, min_tracks=300)


def _frames(ctx, imgs, levels=3):
    imgs = np.asarray(imgs, np.uint8)
    f = ctx.frames(imgs.shape[2], imgs.shape[1], len(imgs), levels)
    f.upload(0, imgs)
    ctx.sync()
    return f


def _level0_with_padding(fr):
    import torch

    class _View:
        def __init__(self, ptr, shape):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": "|u1", "data": (ptr, False), "version": 2}

    ptr, pitch, _ = fr.device_ptr(0)
    return torch.as_tensor(_View(ptr, (fr.n, fr.h, pitch)), device=f"cuda:{fr.ctx.device}")


def _seq(n, w=640, h=480, flat=()):
    out = np.stack([synth.frame(20261018, t, w, h) for t in range(n)])
    for t in flat:
        out[t] = 90
    return out


@pytest.mark.parametrize("name", sorted(IMAGES))
def test_device_encode_matches_reference(ctx, name):
    img = IMAGES[name]
    f = _frames(ctx, img[None], 1)
    assert np.array_equal(f.pack(), fc.encode(img))


def test_device_encode_sequence_and_range(ctx):
    seq = _seq(5, 320, 200, flat=(2,))
    f = _frames(ctx, seq, 1)
    assert np.array_equal(f.pack(), fc.encode(seq))
    assert np.array_equal(f.pack(1, 3), fc.encode(seq[1:4]))
    assert np.array_equal(f.pack(0, 0), fc.encode(np.zeros((0, 200, 320), np.uint8)))


@pytest.mark.parametrize("name", sorted(IMAGES))
def test_decode_reference_blob(ctx, name):
    import torch
    img = IMAGES[name]
    h, w = img.shape
    f = ctx.frames(w, h, 2, 3)
    lv = _level0_with_padding(f)
    lv.fill_(0xAB)
    torch.cuda.synchronize()
    f.upload_packed(1, fc.encode(img))
    ctx.sync()
    got = lv.cpu().numpy()
    assert np.array_equal(got[1, :, :w], img)
    assert (got[1, :, w:] == 0xAB).all() and (got[0] == 0xAB).all()  # row padding and other frames untouched
    r = _frames(ctx, img[None], 3)
    f.build_pyramid(1, 1)
    r.build_pyramid()
    for lvl in range(3):
        assert np.array_equal(f.download(1, lvl), r.download(0, lvl))


def test_decode_hand_built_records(ctx):
    # records the encoder never writes but the format allows (shorter than raw): runs of k = 8 with any values, runs of
    # k = 0 holding a 255 (q = 255), partial tiles
    rng = np.random.default_rng(3)
    w, h = 100, 70
    recs = []
    for x, y, tw, th in fc.tile_grid(w, h):
        n = tw * th
        nr = (n + 31) // 32
        k = np.where(np.arange(nr) % 4 == 0, 8, 0)
        u = np.zeros(nr * 32, np.uint8)
        u[np.repeat(k == 8, 32)] = rng.integers(0, 256, int((k == 8).sum()) * 32)
        u[np.arange(nr)[k == 0][::2] * 32 + 7] = 255
        recs.append(fc.coded_record(u[:n], k))
        assert len(recs[-1]) < 1 + (n + 3) // 4
    blob = fc.blob_from_frames(w, h, [fc.frame_from_records(recs)])
    want = fc.decode(blob)[0]
    f = ctx.frames(w, h, 1, 1)
    f.upload_packed(0, blob)
    assert np.array_equal(f.download(0), want)


def _pair_results(p, npairs, ransac=True):
    li, lj = np.zeros((npairs, p.cap, 2)), np.zeros((npairs, p.cap, 2))
    nk, nc = np.zeros(npairs, np.int32), np.zeros(npairs, np.int32)
    p.download_all(li, lj, nk, nc)
    out = [li, lj, nk, nc]
    if ransac:
        st, bn, inl = np.zeros(npairs, np.int32), np.zeros(npairs, np.int32), np.zeros((npairs, p.cap), np.int32)
        R, t = np.zeros((npairs, 9)), np.zeros((npairs, 3))
        p.ransac_download_all(st, bn, inl, R, t)
        out += [st, bn, inl, R, t]
    return out


def _defined(li, lj, nk, nc, st, bn, inl, R, t):
    """The entries the library defines: survivors up to n_kept, inliers up to best_n, R and t of pairs with a pose (slots past
    the counts keep whatever the pairs object held before)."""
    out = [nk, nc, st, bn]
    for k in range(len(nk)):
        out += [li[k, :nk[k]], lj[k, :nk[k]], inl[k, :max(bn[k], 0)]]
        if st[k] == 2:
            out += [R[k], t[k]]
    return out


def _same(a, b):
    """a, b: lists of 9-array result groups (_pair_results layout), optionally followed by more arrays compared whole."""
    assert len(a) == len(b)
    i = 0
    while i < len(a):
        if i + 9 <= len(a) and a[i].ndim == 3:  # li of a group
            x, y = _defined(*a[i:i + 9]), _defined(*b[i:i + 9])
            i += 9
        else:
            x, y = [a[i]], [b[i]]
            i += 1
        assert len(x) == len(y)
        for u, v in zip(x, y):
            assert u.dtype == v.dtype and u.shape == v.shape and u.tobytes() == v.tobytes()


def test_upload_packed_equals_raw_for_resident_calls(ctx):
    seq = _seq(10, flat=(6,))
    n = len(seq)
    cfg = sfmgpu.lkcfg(**CFG)
    raw = _frames(ctx, seq)
    pk = ctx.frames(640, 480, n, 3)
    pk.upload_packed(0, fc.encode(seq))
    for fr in (raw, pk):
        fr.build_pyramid()
    for t in range(n):
        assert np.array_equal(pk.download(t, 0), seq[t])
    res = []
    for fr in (raw, pk):
        p = ctx.pairs(64, 600)
        p.set_ransac(TEMPLE_K, iters=500, thr=1e-3, min_inliers=60, min_points=1)
        p.run(fr, 0, n - 1, cfg)
        a = _pair_results(p, n - 1)
        p.run_list(fr, [0, 3, 8, 5], [1, 1, 9, 6], cfg)
        b = _pair_results(p, 4)
        q = ctx.pairs(64, 902)
        q.set_ransac(TEMPLE_K, iters=500, thr=1e-3, min_inliers=60, min_points=1)
        q.run_segments(fr, [0, 4], 5, sfmgpu.lkcfg(max_tracks=600, min_tracks=300))
        c = _pair_results(q, 10)
        ids = q.ids_download_all(10)
        c += [np.concatenate([ids[k, :c[2][k]] for k in range(10)])]
        res.append(a + b + c)
    _same(res[0], res[1])


def _host_run(ctx, p, fr, n, cfg, packed=None, chunk=0, blob_first=0, host=None):
    P = n - 1
    li, lj = np.zeros((P, p.cap, 2)), np.zeros((P, p.cap, 2))
    nk, nc = np.zeros(P, np.int32), np.zeros(P, np.int32)
    st, bn, inl = np.zeros(P, np.int32), np.zeros(P, np.int32), np.zeros((P, p.cap), np.int32)
    R, t = np.zeros((P, 9)), np.zeros((P, 3))
    p.ransac_host_outputs(st, bn, inl, R, t)
    if packed is None:
        p.run_host(fr, host, cfg, li, lj, nk, nc, chunk=chunk)
    else:
        p.run_host_packed(fr, packed, n, cfg, li, lj, nk, nc, chunk=chunk, blob_first=blob_first)
    return [li, lj, nk, nc, st, bn, inl, R, t] + _pair_results(p, P)


@pytest.mark.parametrize("chunk,blob_first", [(0, 0), (3, 0), (4, 2)])
def test_host_packed_equals_host(ctx, chunk, blob_first):
    seq = _seq(14, flat=(5, 6))
    n = len(seq) - blob_first
    cfg = sfmgpu.lkcfg(**CFG)
    host = ctx.pinned_empty(seq[blob_first:].shape)
    host[:] = seq[blob_first:]
    blob_np = fc.encode(seq)
    blob = ctx.pinned_empty(blob_np.shape)
    blob[:] = blob_np
    out = []
    for packed in (None, blob):
        fr = ctx.frames(640, 480, n, 3)
        p = ctx.pairs(n, 600)
        p.set_ransac(TEMPLE_K, iters=500, thr=1e-3, min_inliers=60, min_points=1)
        out.append(_host_run(ctx, p, fr, n, cfg, packed, chunk, blob_first, host))
        out[-1] += [np.asarray(p.totals())]
        for t in range(n):
            assert np.array_equal(fr.download(t, 0), seq[blob_first + t])
    _same(out[0], out[1])


def _set_u32(blob, off, v):
    b = blob.copy()
    b[off:off + 4] = np.array([v], "<u4").view(np.uint8)
    return b


def _set_u64(blob, off, v):
    b = blob.copy()
    b[off:off + 8] = np.array([v], "<u8").view(np.uint8)
    return b


def test_refusals_before_any_work(ctx):
    seq = _seq(3, 320, 200)
    blob = fc.encode(seq)
    fo = fc.parse_header(blob)["frame_off"]
    f = ctx.frames(320, 200, 3, 3)
    f.upload(0, seq[::-1])
    ctx.sync()
    before = [f.download(t) for t in range(3)]
    p = ctx.pairs(4, 600)
    cfg = sfmgpu.lkcfg(**CFG)
    bad = {
        "magic": _set_u32(blob, 0, 0x12345678),
        "version": _set_u32(blob, 4, 2),
        "width": _set_u32(blob, 8, 321),
        "height": _set_u32(blob, 12, 100),
        "tile": _set_u32(blob, 20, 32),
        "truncated": blob[:-5],
        "truncated_table": blob[:40],
        "non_monotonic": _set_u64(blob, fc.HEADER_BYTES + 16, int(fo[1]) - 4),
        "past_the_end": _set_u64(blob, fc.HEADER_BYTES + 24, len(blob) + 64),
    }
    for name, b in bad.items():
        for call in (lambda: f.upload_packed(0, b), lambda: p.run_host_packed(f, b, 3, cfg)):
            with pytest.raises(sfmgpu.SfmGpuError) as e:
                call()
            assert e.value.code == -1, name
    for first, count in ((2, 2), (-1, 1), (3, 1)):
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            f.upload_packed(0, blob, first, count)
        assert e.value.code == -1
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        p.run_host_packed(f, blob, 3, cfg, blob_first=1)
    assert e.value.code == -1
    for t in range(3):
        assert np.array_equal(f.download(t), before[t])


def _corrupt_tile(blob, frame, tile, fn):
    """Apply fn to the words of one tile record; the result must not decode in the reference either."""
    H = fc.parse_header(blob)
    fb = int(H["frame_off"][frame])
    nt = len(fc.tile_grid(H["w"], H["h"]))
    toff = blob[fb:fb + 4 * (nt + 1)].view("<u4").astype(int)
    a, b = fb + toff[tile], fb + toff[tile + 1]
    out = blob.copy()
    rec = out[a:b].view("<u4")
    fn(rec)
    x, y, tw, th = fc.tile_grid(H["w"], H["h"])[tile]
    with pytest.raises(ValueError):
        fc.decode_tile(rec.copy(), tw, th)
    return out, (x, y, tw, th)


def test_corrupt_records(ctx):
    seq = _seq(2, 320, 200)
    blob = fc.encode(seq)
    rng = np.random.default_rng(11)

    def k15(r):
        r[1] |= 0xF0000000

    def no_terminator(r):
        r[-1] = 0xFFFFFFFF

    def random_k_table(r):
        r[1:5] = rng.integers(0, 2**32, 4, dtype=np.uint64).astype(np.uint32) | 0x99999999

    def bad_header(r):
        r[0] = 3

    for fn in (k15, no_terminator, random_k_table, bad_header):
        tile = int(rng.integers(0, 20))
        b, (x, y, tw, th) = _corrupt_tile(blob, 1, tile, fn)
        f = ctx.frames(320, 200, 2, 3)  # zero-filled
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            f.upload_packed(0, b)
        assert e.value.code == -1
        got = f.download(1)
        mask = np.zeros_like(got, bool)
        mask[y:y + th, x:x + tw] = True
        assert (got[mask] == 0).all()  # the tile that does not decode is not written
        assert np.array_equal(got[~mask], seq[1][~mask]) and np.array_equal(f.download(0), seq[0])
        p = ctx.pairs(2, 600)
        with pytest.raises(sfmgpu.SfmGpuError) as e:
            p.run_host_packed(f, b, 2, sfmgpu.lkcfg(**CFG))
        assert e.value.code == -1
    # tile offsets out of order inside a frame
    H = fc.parse_header(blob)
    fb = int(H["frame_off"][0])
    b = _set_u32(blob, fb + 4 * 3, int(blob[fb + 4 * 5:fb + 4 * 6].view("<u4")[0]))
    f = ctx.frames(320, 200, 2, 3)
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        f.upload_packed(0, b)
    assert e.value.code == -1


def test_pack_capacity(ctx):
    seq = _seq(2, 320, 200)
    f = _frames(ctx, seq, 1)
    need = len(fc.encode(seq))
    lib = ctx.lib
    nb = C.c_size_t(0)
    small = np.zeros(need - 1, np.uint8)
    rc = lib.sfmgpu_frames_pack(ctx.h, f.h_, 0, 2, small.ctypes.data_as(C.c_void_p), small.nbytes, C.byref(nb))
    assert rc == -3 and nb.value == need
    rc = lib.sfmgpu_frames_pack(ctx.h, f.h_, 0, 2, None, 0, C.byref(nb))
    assert rc == -3 and nb.value == need
    assert need <= sfmgpu.pack_bound(320, 200, 2)
    with pytest.raises(sfmgpu.SfmGpuError) as e:
        f.pack(out=small)
    assert e.value.code == -3
