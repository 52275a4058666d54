"""numpy reference of the packed frame format (include/sfmgpu.h, DESIGN.md §2): the lossless tile codec that
sfmgpu_frames_pack writes and sfmgpu_frames_upload_packed / sfmgpu_pair_frontend_host_packed read.  It pins the format:
the device encoder must produce these bytes, and the device decoder must turn these bytes back into the frames.

Blob (all integers little-endian):
    header   8 x u32: MAGIC, VERSION, w, h, nframes, TILE, 0, 0
    u64 frame_off[nframes + 1]   byte offsets from the blob start; frame k is [frame_off[k], frame_off[k+1])
    frames   per frame: u32 tile_off[ntiles + 1] (byte offsets from the frame start, 4-byte aligned, tile_off[ntiles] =
             the frame's size), then the tile records, tiles in raster order of the tile grid
Tile (TILE x TILE pixels of level 0, edge tiles partial; n = tw * th pixels in raster order inside the tile):
    residual  d = p - left - up + upleft (mod 256), pixels outside the tile taken as 0; u = zig-zag(d as int8) in [0, 255]
    runs      nruns = ceil(n / 32) runs of 32 values, the last one zero-padded; run r codes each u as q = u >> k_r (unary)
              and u & (2^k_r - 1) (k_r bits); k_r in 0..8 = the k with the fewest bits, the smallest on a tie
    coded record (u32 words): hdr = U << 1 (U = unary bits), k table (nibble r = k_r, ceil(nruns / 8) words),
              remainder stream (run r: its 32 remainders of k_r bits LSB-first = k_r words), unary stream (value j:
              q_j one-bits then a zero bit, LSB-first, ceil(U / 32) words, zero padded)
    raw record: hdr = 1, then the n pixels, zero padded to a word; used when the coded record would have at least as
              many words as the raw one (so a coded record is always shorter than the raw one: a decoder refuses others)
Decoding is a 2D inclusive prefix sum of the residuals mod 256.
"""
import numpy as np

MAGIC = 0x504B4653  # "SFKP"
VERSION = 1
TILE = 64
RUN = 32
HEADER_BYTES = 32


def tile_grid(w, h):
    """[(x0, y0, tw, th)] in raster order of the tile grid."""
    return [(x, y, min(TILE, w - x), min(TILE, h - y)) for y in range(0, h, TILE) for x in range(0, w, TILE)]


def _raw_words(n):
    return 1 + (n + 3) // 4


def pack_bound(w, h, nframes):
    """The largest blob nframes frames of w x h can give (every tile raw)."""
    g = tile_grid(w, h)
    frame = 4 * (len(g) + 1) + sum(4 * _raw_words(tw * th) for _, _, tw, th in g)
    return HEADER_BYTES + 8 * (nframes + 1) + nframes * frame


def residuals(tiles):
    """[T, th, tw] uint8 tiles -> zig-zagged planar residuals [T, th, tw] uint8."""
    p = tiles.astype(np.int32)
    left = np.zeros_like(p)
    left[:, :, 1:] = p[:, :, :-1]
    up = np.zeros_like(p)
    up[:, 1:, :] = p[:, :-1, :]
    ul = np.zeros_like(p)
    ul[:, 1:, 1:] = p[:, :-1, :-1]
    d = ((p - left - up + ul) & 255).astype(np.uint8).view(np.int8).astype(np.int32)
    return np.where(d >= 0, 2 * d, -2 * d - 1).astype(np.uint8)


def unzigzag(u):
    u = u.astype(np.int32)
    return (np.where(u & 1, -((u + 1) >> 1), u >> 1) & 255).astype(np.uint8)


def prefix2d(d):
    """2D inclusive prefix sum mod 256 (the inverse of the planar predictor)."""
    return (np.cumsum(np.cumsum(d.astype(np.int64), axis=-1), axis=-2) & 255).astype(np.uint8)


def choose_k(u_runs):
    """[..., RUN] values -> (k [...], unary bits [...]): the k in 0..8 with the fewest bits, the smallest on a tie."""
    q = u_runs[..., None].astype(np.int32) >> np.arange(9)  # [..., RUN, 9]
    qsum = q.sum(axis=-2)  # [..., 9]
    bits = qsum + RUN * (1 + np.arange(9))
    k = np.argmin(bits, axis=-1)  # first minimum
    return k, np.take_along_axis(qsum, k[..., None], -1)[..., 0] + RUN


def _bits(values, widths):
    """Concatenate values[i] in widths[i] bits, LSB first -> flat bit array."""
    b = (values[:, None].astype(np.int64) >> np.arange(8)) & 1
    return b[np.arange(8)[None, :] < widths[:, None]]


def _words(bits):
    nw = (len(bits) + 31) // 32
    pad = np.zeros(nw * 32, np.uint8)
    pad[:len(bits)] = bits
    return np.packbits(pad, bitorder="little").view("<u4")


def encode_tile(tile):
    """One tile [th, tw] uint8 -> record (uint32 words)."""
    th, tw = tile.shape
    n = tw * th
    nruns = (n + RUN - 1) // RUN
    u = np.zeros(nruns * RUN, np.uint8)
    u[:n] = residuals(tile[None])[0].reshape(-1)
    k, ubits = choose_k(u.reshape(nruns, RUN))
    U = int(ubits.sum())
    kw = (nruns + 7) // 8
    coded_words = 1 + kw + int(k.sum()) + (U + 31) // 32
    if coded_words >= _raw_words(n):
        raw = np.zeros(4 * (_raw_words(n) - 1), np.uint8)
        raw[:n] = tile.reshape(-1)
        return np.concatenate([np.array([1], "<u4"), raw.view("<u4")])
    out = coded_record(u, k)
    assert len(out) == coded_words
    return out


def coded_record(u, k):
    """A coded record from chosen values u [n] and run parameters k [nruns] (any k in 0..8, not just the encoder's choice):
    records the encoder never writes but the format allows, such as q = 255 at k = 0."""
    u = np.asarray(u, np.uint8)
    k = np.asarray(k, np.int64)
    nruns = len(k)
    uu = np.zeros(nruns * RUN, np.uint8)
    uu[:len(u)] = u
    kw = (nruns + 7) // 8
    ktab = np.zeros(kw * 8, np.uint32)
    ktab[:nruns] = k
    ktab = (ktab.reshape(kw, 8) << (4 * np.arange(8, dtype=np.uint32))).sum(axis=1, dtype=np.uint32)
    kk = np.repeat(k, RUN)
    q = uu.astype(np.int64) >> kk
    U = int((q + 1).sum())
    ub = np.ones(U, np.uint8)
    ub[np.cumsum(q + 1) - 1] = 0
    return np.concatenate([np.array([U << 1], "<u4"), ktab.astype("<u4"), _words(_bits(uu & ((1 << kk) - 1), kk)), _words(ub)])


def frame_from_records(recs):
    """A frame's bytes (tile table + records) from its tile records."""
    off = np.zeros(len(recs) + 1, np.int64)
    off[0] = 4 * (len(recs) + 1)
    off[1:] = off[0] + 4 * np.cumsum([len(r) for r in recs])
    return np.concatenate([off.astype("<u4")] + list(recs)).view(np.uint8)


def encode_frame(img):
    g = tile_grid(img.shape[1], img.shape[0])
    return frame_from_records([encode_tile(img[y:y + th, x:x + tw]) for x, y, tw, th in g])


def encode(frames):
    """[n, h, w] uint8 -> blob (uint8)."""
    frames = np.asarray(frames, np.uint8)
    if frames.ndim == 2:
        frames = frames[None]
    _, h, w = frames.shape
    return blob_from_frames(w, h, [encode_frame(f) for f in frames])


def blob_from_frames(w, h, body):
    """A blob from its frames' bytes."""
    n = len(body)
    foff = np.zeros(n + 1, np.int64)
    foff[0] = HEADER_BYTES + 8 * (n + 1)
    foff[1:] = foff[0] + np.cumsum([len(b) for b in body])
    hdr = np.array([MAGIC, VERSION, w, h, n, TILE, 0, 0], "<u4").view(np.uint8)
    return np.concatenate([hdr, foff.astype("<u8").view(np.uint8)] + body)


def parse_header(blob):
    hdr = np.frombuffer(blob[:HEADER_BYTES].tobytes(), "<u4")
    magic, version, w, h, n, tile = (int(v) for v in hdr[:6])
    foff = np.frombuffer(blob[HEADER_BYTES:HEADER_BYTES + 8 * (n + 1)].tobytes(), "<u8").astype(np.int64)
    return dict(magic=magic, version=version, w=w, h=h, n=n, tile=tile, frame_off=foff)


def decode_tile(rec, tw, th):
    """Record (uint32 words) -> tile [th, tw] uint8; raises ValueError on a record that does not decode."""
    n = tw * th
    nruns = (n + RUN - 1) // RUN
    kw = (nruns + 7) // 8
    hdr = int(rec[0])
    if hdr == 1:
        if len(rec) != _raw_words(n):
            raise ValueError("raw record size")
        return rec[1:].view(np.uint8)[:n].reshape(th, tw).copy()
    if hdr & 1 or len(rec) >= _raw_words(n):  # a coded record is always shorter than the raw one
        raise ValueError("bad header / record longer than raw")
    U = hdr >> 1
    k = ((rec[1:1 + kw, None] >> (4 * np.arange(8, dtype=np.uint32))) & 15).reshape(-1)[:nruns].astype(np.int64)
    if (k > 8).any() or len(rec) != 1 + kw + int(k.sum()) + (U + 31) // 32:
        raise ValueError("k table / record size")
    rbits = np.unpackbits(rec[1 + kw:1 + kw + int(k.sum())].view(np.uint8), bitorder="little")
    ubits = np.unpackbits(rec[1 + kw + int(k.sum()):].view(np.uint8), bitorder="little")[:U]
    zeros = np.flatnonzero(ubits == 0)
    if len(zeros) != nruns * RUN or U == 0 or ubits[U - 1] != 0:
        raise ValueError("unary stream")
    q = np.diff(np.concatenate([[-1], zeros])) - 1
    kk = np.repeat(k, RUN)
    start = np.concatenate([[0], np.cumsum(kk)[:-1]])
    rem = np.zeros(nruns * RUN, np.int64)
    for b in range(8):
        m = b < kk
        rem[m] |= rbits[start[m] + b].astype(np.int64) << b
    u = (q << kk) | rem
    if (u > 255).any():
        raise ValueError("value out of range")
    return prefix2d(unzigzag(u[:n]).reshape(th, tw))


def decode(blob, first=0, count=None):
    """Blob -> frames [count, h, w] uint8 (frames first .. first+count-1 of the blob)."""
    blob = np.asarray(blob, np.uint8)
    H = parse_header(blob)
    if H["magic"] != MAGIC or H["version"] != VERSION or H["tile"] != TILE:
        raise ValueError("not a packed frame blob")
    w, h, n = H["w"], H["h"], H["n"]
    count = n - first if count is None else count
    g = tile_grid(w, h)
    out = np.zeros((count, h, w), np.uint8)
    for i in range(count):
        a, b = H["frame_off"][first + i], H["frame_off"][first + i + 1]
        fr = blob[a:b]
        toff = fr[:4 * (len(g) + 1)].view("<u4").astype(np.int64)
        for t, (x, y, tw, th) in enumerate(g):
            out[i, y:y + th, x:x + tw] = decode_tile(fr[toff[t]:toff[t + 1]].view("<u4"), tw, th)
    return out


def sample_images():
    """{name: image} of every class the codec tests cover: bench content, the ring scene, the KAT image, noise, flat frames,
    0/255 checkerboards (extreme residuals: q up to 255 at k = 0) and sizes that are not multiples of the tile."""
    import ring_dataset
    from sfmgpu import synth
    rng = np.random.default_rng(20261021)
    yy, xx = np.mgrid[:96, :130]
    return {
        "synth_1080p": synth.frame(20261018, 5, 1920, 1080),
        "ring": ring_dataset.render(0.0),
        "kat": synth.kat_image(640, 480),
        "noise": rng.integers(0, 256, (480, 640), dtype=np.uint8),
        "flat": np.full((480, 640), 77, np.uint8),
        "checker_1px": (((xx + yy) & 1) * 255).astype(np.uint8),
        "checker_2px": ((((xx >> 1) + (yy >> 1)) & 1) * 255).astype(np.uint8),
        "size_1x1": np.array([[200]], np.uint8),
        "size_17x5": rng.integers(0, 256, (5, 17), dtype=np.uint8),
        "size_65x1": (np.arange(65, dtype=np.uint8) * 7)[None],
        "synth_640x480": synth.frame(3, 1, 640, 480),
    }
