"""The arg-max rule of the batched loop-closure search (csrc/loopdesc.cu, desc_search_kernel), restated on the CPU.

The reference picks the loop candidate with a sequential scan (cpp/src/templering_sfm.cpp:1823-1831):
    best_id = -1; best_score = 0; for k: if (s[k] > best_score) { best_score = s[k]; best_id = k; }
The kernel instead combines, in any order, the 64-bit keys (float_bits(s) << 32) | (0xFFFFFFFF - k) of the scores s > 0 with
a maximum; key 0 stands for (-1, 0.0f).  These tests pin that the two agree on float32 scores with ties, NaN, +-0, negatives
and denormals, whatever order the keys are reduced in."""
import numpy as np
import pytest


def sequential(s):
    bid, bs = -1, np.float32(0.0)
    for k, v in enumerate(s):
        if v > bs:
            bid, bs = k, v
    return bid, bs


def keys(s):
    s = np.asarray(s, np.float32)
    k = np.arange(len(s), dtype=np.uint64)
    key = (s.view(np.uint32).astype(np.uint64) << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - k)
    return np.where(s > 0, key, np.uint64(0))  # NaN, +-0 and negatives never enter


def packed_argmax(s, rng=None):
    kk = keys(s)
    if rng is not None:  # the kernel reduces per thread, per warp and by atomics in whatever order blocks finish
        kk = kk[rng.permutation(len(kk))]
    best = np.uint64(0)
    for v in kk:
        best = max(best, v)
    if best == 0:
        return -1, np.float32(0.0)
    return int(np.uint64(0xFFFFFFFF) - (best & np.uint64(0xFFFFFFFF))), np.uint32(best >> np.uint64(32)).view(np.float32)


def _cases():
    rng = np.random.default_rng(5)
    tiny = np.float32(1e-45)  # smallest denormal
    yield np.zeros(0, np.float32)
    yield np.zeros(7, np.float32)
    yield -np.abs(rng.standard_normal(50)).astype(np.float32) - tiny
    yield np.array([np.nan, 0.5, np.nan, 0.5, 0.25], np.float32)  # tie: the first 0.5 wins
    yield np.array([-0.0, 0.0, tiny, -tiny, 2 * tiny, 2 * tiny], np.float32)  # denormals order like their bits
    yield np.array([np.nan] * 4, np.float32)
    yield np.array([np.inf, 3.0, np.inf], np.float32)
    yield np.array([-np.inf, -1.0, np.float32(3.4e38)], np.float32)
    for n in (1, 63, 65, 257, 1000, 4096):
        s = rng.choice(np.array([0.9, 0.95, 0.95, -0.2, 0.0, -0.0, np.nan, tiny, 0.5], np.float32), n)
        yield s
        yield rng.uniform(-1, 1, n).astype(np.float32)
        q = np.round(rng.uniform(-1, 1, n) * 8).astype(np.float32) / 8  # many exact ties
        yield q


@pytest.mark.parametrize("case", list(range(len(list(_cases())))))
def test_packed_key_argmax_equals_sequential_scan(case):
    s = list(_cases())[case]
    want = sequential(s)
    for seed in (None, 1, 2):
        got = packed_argmax(s, None if seed is None else np.random.default_rng(seed))
        assert got[0] == want[0] and np.float32(got[1]).tobytes() == np.float32(want[1]).tobytes(), (got, want)


def test_positive_floats_order_like_their_bits():
    rng = np.random.default_rng(9)
    v = np.concatenate([rng.uniform(0, 1, 10000), rng.uniform(0, 1e-38, 1000), [1e-45, 3.4e38, np.inf]]).astype(np.float32)
    v = v[v > 0]
    order_f = np.argsort(v, kind="stable")
    order_b = np.argsort(v.view(np.uint32), kind="stable")
    assert np.array_equal(v[order_f], v[order_b])
