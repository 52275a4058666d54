"""Segment-mode shard (sfmgpu_sched_segment_shard), without a GPU: G segments of L = ceil((T-1)/G) steps over a sequence of T
frames.  Every frame pair must be a step of some segment, the last segment must end on the last frame, fewer than G steps
may be done twice, the ranks' blocks must tile the segments, and each rank's frame range must hold exactly its segments."""
import numpy as np
import pytest

from sfmgpu import sched

T_GRID = sorted({2, 3, 4, 5, 7, 9, 16, 17, 31, 64, 65, 100, 127, 257, 500, 999, 1000, 1001, 1999, 2000})


def g_grid(T):
    gs = {1, 2, 3, T - 1, T - 2, (T - 1) // 2, (T - 1) // 3, 31, 32, 33, 64, 65, 128}
    return sorted(g for g in gs if 1 <= g <= T - 1)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_segment_shard_properties(world):
    for T in T_GRID:
        for G in g_grid(T):
            blocks = []
            for rank in range(world):
                L, a, b, first, f0, f1 = sched.segment_shard(T, G, world, rank)
                assert L == -(-(T - 1) // G)
                assert len(first) == G and first[0] == 0 and np.all(np.diff(first) >= 0)
                covered = np.zeros(T - 1, bool)
                for s in first:
                    assert 0 <= s and s + L <= T - 1, (T, G, s, L)
                    covered[s:s + L] = True
                assert covered.all(), (T, G)  # every pair (t, t+1) is a step of some segment
                assert first[-1] + L == T - 1  # the last segment ends on the last frame
                assert G * L - (T - 1) < G  # duplicated steps
                assert (a, b) == sched.shard_range(G, world, rank)
                if b > a:
                    assert (f0, f1) == (first[a], first[b - 1] + L + 1)
                else:
                    assert f0 == f1 == 0
                blocks.append((a, b))
            assert blocks[0][0] == 0 and blocks[-1][1] == G
            assert all(blocks[r][1] == blocks[r + 1][0] for r in range(world - 1))


def test_segment_shard_first_in_64_bits():
    """j * (T-1-L) overflows 32 bits for long sequences with many segments."""
    T, G = 200001, 100000
    L, _, _, first, _, _ = sched.segment_shard(T, G)
    assert L == 2 and first[-1] == T - 1 - L
    j = np.arange(G, dtype=np.int64)
    assert np.array_equal(first, j * (T - 1 - L) // (G - 1))


@pytest.mark.parametrize("T,G,world,rank", [(1, 1, 1, 0), (2, 0, 1, 0), (2, 2, 1, 0), (10, 10, 1, 0), (10, 3, 0, 0), (10, 3, 2, 2),
                                            (10, 3, 2, -1)])
def test_segment_shard_refusals(T, G, world, rank):
    with pytest.raises(ValueError):
        sched.segment_shard(T, G, world, rank)
