"""The packed frame format (tests/frame_codec.py, include/sfmgpu.h): round trips, the encoder's deterministic choices, the
pack bound and compression floors, on the CPU reference."""
import numpy as np
import pytest

import frame_codec as fc
from sfmgpu import synth

IMAGES = fc.sample_images()


@pytest.mark.parametrize("name", sorted(IMAGES))
def test_round_trip(name):
    img = IMAGES[name]
    blob = fc.encode(img)
    assert len(blob) <= fc.pack_bound(img.shape[1], img.shape[0], 1)
    assert np.array_equal(fc.decode(blob)[0], img)


def test_round_trip_4k_sequence_and_frame_ranges():
    frames = np.stack([synth.frame(20261018, t, 3840, 2160) for t in (0, 1)])
    blob = fc.encode(frames)
    H = fc.parse_header(blob)
    assert (H["magic"], H["version"], H["w"], H["h"], H["n"], H["tile"]) == (fc.MAGIC, fc.VERSION, 3840, 2160, 2, 64)
    assert H["frame_off"][0] == fc.HEADER_BYTES + 8 * 3 and H["frame_off"][-1] == len(blob)
    assert np.array_equal(fc.decode(blob), frames)
    assert np.array_equal(fc.decode(blob, 1, 1)[0], frames[1])
    assert frames.nbytes / len(blob) >= 2.8


def test_prefix_sum_of_residuals_is_the_frame():
    for img in (IMAGES["synth_640x480"], IMAGES["checker_1px"], IMAGES["size_17x5"]):
        d = fc.unzigzag(fc.residuals(img[None])[0])
        assert np.array_equal(fc.prefix2d(d), img)


def test_k_tie_rule():
    # all zeros: k = 0 costs 32 bits, every larger k costs more
    k, U = fc.choose_k(np.zeros((1, 32), np.uint8))
    assert k[0] == 0 and U[0] == 32
    # u = 1 everywhere: k = 0 -> 32 + 32 = 64 bits, k = 1 -> 0 + 32 + 32 = 64 bits: the tie goes to k = 0
    k, U = fc.choose_k(np.ones((1, 32), np.uint8))
    assert k[0] == 0 and U[0] == 64
    # u = 255 everywhere: k = 8 (no unary ones) beats k = 7 (one 1-bit each: 32 * (1 + 7 + 1) = 288 = 32 * (1 + 8)): tie -> 7
    k, _ = fc.choose_k(np.full((1, 32), 255, np.uint8))
    assert k[0] == 7
    # brute force over random runs
    rng = np.random.default_rng(5)
    u = rng.integers(0, 256, (200, 32)).astype(np.uint8) >> rng.integers(0, 8, (200, 1)).astype(np.uint8)
    k, U = fc.choose_k(u)
    for r in range(200):
        bits = [int((u[r].astype(int) >> b).sum()) + 32 * (1 + b) for b in range(9)]
        assert k[r] == bits.index(min(bits)) and U[r] == bits[k[r]] - 32 * k[r]


def test_raw_fallback_and_bound():
    noise = IMAGES["noise"]
    blob = fc.encode(noise)
    fr = blob[fc.HEADER_BYTES + 16:]
    toff = fr[:4 * 81].view("<u4")
    hdrs = [int(fr[toff[t]:toff[t] + 4].view("<u4")[0]) for t in range(80)]
    assert all(h == 1 for h in hdrs)  # uniform noise does not compress: every tile is stored raw
    assert len(blob) == fc.pack_bound(640, 480, 1)
    assert len(blob) <= noise.nbytes * 1.003
    # the coded record is used only when it is shorter than the raw one
    flat = fc.encode_tile(np.full((64, 64), 9, np.uint8))
    assert flat[0] != 1 and len(flat) < 1 + 1024
    assert fc.pack_bound(1, 1, 0) == fc.HEADER_BYTES + 8
    assert fc.pack_bound(1920, 1080, 3) == fc.HEADER_BYTES + 32 + 3 * (4 * 511 + 4 * (480 * 1025 + 30 * (1 + 56 * 16)))


def test_q_255_at_k_0_decodes():
    # the encoder never codes u = 255 at k = 0 (k = 1 always costs fewer bits), but the format allows it and the decoder reads
    # it: a unary run of 255 ones
    u = np.zeros(4096, np.uint8)
    u[7::64] = 255
    u[9::64] = 3
    rec = fc.coded_record(u, np.zeros(128, np.int64))
    assert len(rec) < 1 + 1024
    want = fc.prefix2d(fc.unzigzag(u).reshape(64, 64))
    assert np.array_equal(fc.decode_tile(rec, 64, 64), want)
    assert np.array_equal(fc.decode_tile(fc.encode_tile(want), 64, 64), want)


def test_ratio_floors():
    syn = np.stack([synth.frame(20261018, t, 1920, 1080) for t in (0, 37)])
    assert syn.nbytes / len(fc.encode(syn)) >= 2.9
    ring = IMAGES["ring"]
    assert ring.nbytes / len(fc.encode(ring)) >= 1.9


def test_corrupt_records_do_not_decode():
    img = IMAGES["synth_640x480"]
    blob = fc.encode(img)
    fr = blob[fc.HEADER_BYTES + 16:]
    toff = fr[:4 * 81].view("<u4").astype(int)
    rec = fr[toff[0]:toff[1]].view("<u4").copy()
    bad = rec.copy()
    bad[1] |= 0xF  # k = 15
    with pytest.raises(ValueError):
        fc.decode_tile(bad, 64, 64)
    bad = rec.copy()
    bad[-1] = 0xFFFFFFFF  # the last terminator is gone
    with pytest.raises(ValueError):
        fc.decode_tile(bad, 64, 64)
    with pytest.raises(ValueError):
        fc.decode_tile(rec[:-1], 64, 64)
