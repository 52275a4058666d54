"""CPU check of the "observable tie" rule behind the default selection (csrc/corner_select.cu: bucket_select_kernel,
DESIGN.md §4).

std::sort may leave a group of candidates with IDENTICAL scores in any order.  The rule: the order inside a group can only
change the result of the greedy min-distance selection if at least TWO members of the group are unblocked (farther than
min_dist from every corner accepted before the group) when the selection reaches the group.  Here every permutation of
every tie group of small random instances is run through the reference's greedy loop (sfm.cpp:288-300) and compared."""
import itertools

import numpy as np
import pytest


def greedy(points, d, cap):
    """shi_tomasi's selection loop: accept iff no accepted corner at squared distance < d^2; cap tested after the push."""
    acc = []
    for (x, y) in points:
        if all((x - ax) ** 2 + (y - ay) ** 2 >= d * d for ax, ay in acc):
            acc.append((x, y))
            if len(acc) >= cap:
                break
    return acc


def observable(groups, d, cap):
    """The device's criterion, evaluated in score order: a group is flagged iff >= 2 of its members are unblocked by the
    corners accepted BEFORE the group (the kernel tests a superset: unblocked by the corners of earlier rounds)."""
    acc = []
    for g in groups:
        free = [p for p in g if all((p[0] - ax) ** 2 + (p[1] - ay) ** 2 >= d * d for ax, ay in acc)]
        if len(g) > 1 and len(free) >= 2 and len(acc) < cap:
            return True
        for p in g:  # continue the greedy walk in the given order
            if len(acc) < cap and all((p[0] - ax) ** 2 + (p[1] - ay) ** 2 >= d * d for ax, ay in acc):
                acc.append(p)
    return False


@pytest.mark.parametrize("seed", range(40))
def test_unobservable_ties_do_not_change_the_selection(seed):
    rng = np.random.default_rng(seed)
    n, d, cap = 14, int(rng.integers(2, 6)), int(rng.integers(2, 9))
    pts = set()
    while len(pts) < n:
        pts.add((int(rng.integers(0, 12)), int(rng.integers(0, 12))))
    pts = list(pts)
    # scores: a few groups of 2-3 equal scores between distinct ones, sorted descending
    sizes = []
    while sum(sizes) < n:
        sizes.append(int(rng.choice([1, 1, 1, 2, 2, 3])))
    sizes[-1] -= sum(sizes) - n
    groups, k = [], 0
    for s in sizes:
        if s > 0:
            groups.append(pts[k:k + s])
            k += s
    base = greedy([p for g in groups for p in g], d, cap)
    outcomes = set()
    for perm in itertools.product(*[list(itertools.permutations(g)) for g in groups]):
        outcomes.add(tuple(greedy([p for g in perm for p in g], d, cap)))
    if not observable(groups, d, cap):
        assert outcomes == {tuple(base)}, (seed, groups, d, cap)


def test_rule_is_not_vacuous():
    """Both outcomes occur in the random instances above: ties that matter are flagged, ties that do not are not."""
    flagged = clean = differing = 0
    for seed in range(200):
        rng = np.random.default_rng(1000 + seed)
        d, cap = 3, 5
        pts = list({(int(rng.integers(0, 9)), int(rng.integers(0, 9))) for _ in range(12)})
        groups = [[p] for p in pts[:5]] + [pts[i:i + 2] for i in range(5, len(pts) - 1, 2)]  # distinct scores first
        outs = {tuple(greedy([p for g in perm for p in g], d, cap))
                for perm in itertools.product(*[list(itertools.permutations(g)) for g in groups])}
        if observable(groups, d, cap):
            flagged += 1
            differing += len(outs) > 1
        else:
            clean += 1
            assert len(outs) == 1
    assert flagged > 20 and clean > 20 and differing > 10, (flagged, clean, differing)
