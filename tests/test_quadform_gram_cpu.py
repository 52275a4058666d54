"""CPU model of the Gram build of klt_quad_kernel (csrc/klt_lane.cu, gram_build): every matrix entry of the five families is an
integer combination of the entries of one 16 x 16 Gram matrix G = sum_p t(p) t(p)^T of raw u8 taps.  Checked entry for
entry against the FFMA build's strip bookkeeping (family() of test_quadform_cpu.py) and the direct window sums, and through
an emulation of the kernel's fragment layout: K order, the zeroed column-12 byte and zero row, PRMT selectors, the
m16n8k32 fragments, the scratch layout of G and the per-lane entry addresses."""
import numpy as np
import pytest

from test_quadform_cpu import ENTRIES, family, family_direct

LIMG, LSTRIDE, ZROW, QM = 224, 464, 448, 50


def tap(j):
    """(image, dr, dc) of tap j (0: I1, 1: I0), offsets from window pixel (r, c)."""
    if j < 8:
        return 0, j >> 2, (j & 3) - 1
    if j < 12:
        return 0, -1 if j < 10 else 2, j & 1
    return 1, (j - 12) >> 1, j & 1


def diff_tap(side, k, plus):
    a, b = k >> 1, k & 1
    if side == 0:
        return a * 4 + b + (2 if plus else 0)
    if side == 1:
        return (10 + b if a else 5 + b) if plus else (1 + b if a else 8 + b)
    return 12 + 2 * a + b if plus else a * 4 + b + 1


SIDES = [(0, 0), (1, 1), (0, 1), (0, 2), (1, 2)]  # XX, YY, XY, XE, YE: sides of A and B


def entries_from_gram(G):
    """The 50 integers of quad_store's layout from G."""
    def d(sa, ka, sb, kb):
        ap, am, bp, bm = diff_tap(sa, ka, True), diff_tap(sa, ka, False), diff_tap(sb, kb, True), diff_tap(sb, kb, False)
        return int(G[ap, bp]) - int(G[ap, bm]) - int(G[am, bp]) + int(G[am, bm])
    out = []
    for sa, sb in SIDES:
        for k, l in ENTRIES:
            out.append(d(sa, k, sb, l) + (d(sa, l, sb, k) if k != l else 0))
    return out


def entries_from_family(t1, t0):
    DX, DY, DE = np.zeros((14, 14), np.int64), np.zeros((14, 14), np.int64), t0 - t1
    DX[:, 1:13] = t1[:, 2:14] - t1[:, 0:12]
    DY[1:13, :] = t1[2:14, :] - t1[0:12, :]
    D = {0: DX, 1: DY, 2: DE}
    out = []
    for sa, sb in SIDES:
        sym = sa == sb
        out += [v + v if sym and k != l else v for v, (k, l) in zip(family(D[sa], D[sb], sym), ENTRIES)]
    return out, D


def gram_direct(t1, t0):
    imgs = (t1, t0)
    R = np.array([[imgs[i][r + dr, c + dc] for i, dr, dc in map(tap, range(16))] for r in range(1, 12) for c in range(1, 12)],
                 np.int64)
    return R.T @ R


def staged(t1, t0):
    """One lane region as klt_quad_kernel stages it: 14 rows of 16 bytes per image, bytes 14 / 15 zero, then the zero row."""
    s = np.zeros(LSTRIDE, np.uint8)
    s[0:LIMG].reshape(14, 16)[:, :14] = t1
    s[LIMG:2 * LIMG].reshape(14, 16)[:, :14] = t0
    return s


def byte_perm(x, y, sel):
    b = list(x.to_bytes(4, "little")) + list(y.to_bytes(4, "little"))
    return bytes(b[(sel >> (4 * i)) & 7] for i in range(4))


def word(s, off):
    return int.from_bytes(bytes(s[off:off + 4]), "little")


def gram_at(i, j):
    if i >= 8 and j < 8:
        i, j = j, i
    return (i * 8 + j) * 4 if i < 8 and j < 8 else (256 + (i * 8 + j - 8) * 4 if i < 8 else 512 + ((i - 8) * 8 + j - 8) * 4)


def emulate_kernel(s):
    """gram_lane_init + gram_build for one feature: fragments per lane, the two m16n8k32 products per k-step, the scratch
    and the entries each lane reads from it."""
    A = np.zeros((16, 160), np.int64)  # rows: taps, columns: K
    for lane in range(32):
        g, t = lane >> 2, lane & 3
        for x in range(2):
            img, dr, dc = tap(g + 8 * x)
            rb = img * LIMG + (dr + t + 1) * 16
            r2 = ZROW if t == 3 else rb + 128
            sel = 0x3210 + 0x1111 * (dc + 1)
            selm = (sel & 0x0FFF) | 0x7000
            for u in range(10):
                kstep, half = u >> 1, u & 1
                if u >= 9:
                    w = bytes(4)
                else:
                    cls, j = u // 3, u % 3
                    rowp = r2 if j == 2 else rb + 64 * j
                    w = byte_perm(word(s, rowp + 4 * cls), word(s, rowp + 4 * cls + 4), selm if cls == 2 else sel)
                k0 = 32 * kstep + 16 * half + 4 * t  # fragment: row g (+8 for x = 1), columns 4t.. (+16 for half 1)
                A[g + 8 * x, k0:k0 + 4] = list(w)
    G = A @ A.T  # B = the same words: B[k][n] = A[n][k]
    scratch = np.zeros(192, np.int64)
    for lane in range(32):  # the three int2 stores of a lane
        g, t = lane >> 2, lane & 3
        o = g * 8 + 2 * t
        scratch[o:o + 2] = G[g, 2 * t:2 * t + 2]
        scratch[64 + o:64 + o + 2] = G[g, 8 + 2 * t:10 + 2 * t]
        scratch[128 + o:128 + o + 2] = G[8 + g, 8 + 2 * t:10 + 2 * t]
    out = []
    for e in range(QM):
        f, q = divmod(e, 10)
        k = 0 if q < 4 else 1 if q < 7 else 2 if q < 9 else 3
        l = k + q - (0 if q < 4 else 4 if q < 7 else 7 if q < 9 else 9)
        sa, sb = SIDES[f]
        v = 0
        for d in range(2):
            if d == 1 and k == l:
                continue  # the kernel reads a zero word
            ka, kb = (l, k) if d else (k, l)
            ap, am, bp, bm = diff_tap(sa, ka, True), diff_tap(sa, ka, False), diff_tap(sb, kb, True), diff_tap(sb, kb, False)
            rd = lambda i, j: int(scratch[gram_at(i, j) // 4])
            v += rd(ap, bp) - rd(ap, bm) - rd(am, bp) + rd(am, bm)
        out.append(v)
    return out, G


def _tiles():
    rng = np.random.default_rng(7)
    cb = (np.indices((14, 14)).sum(0) % 2 * 255).astype(np.int64)
    full, zero = np.full((14, 14), 255, np.int64), np.zeros((14, 14), np.int64)
    cases = [("random", rng.integers(0, 256, (14, 14)), rng.integers(0, 256, (14, 14))),
             ("random_close", *(lambda a: (a, np.clip(a + rng.integers(-30, 31, (14, 14)), 0, 255)))(rng.integers(0, 256, (14, 14)))),
             ("all_255", full, full), ("all_0", zero, zero), ("255_0", full, zero), ("0_255", zero, full),
             ("checker", cb, cb), ("checker_inverted", cb, 255 - cb), ("checker_full", cb, full),
             ("flat", np.full((14, 14), 90, np.int64), np.full((14, 14), 90, np.int64))]
    return cases


@pytest.mark.parametrize("name,t1,t0", _tiles(), ids=[c[0] for c in _tiles()])
def test_gram_entries_equal_the_ffma_build(name, t1, t0):
    want, D = entries_from_family(t1, t0)
    G = gram_direct(t1, t0)
    assert G.max() <= 121 * 255 ** 2 < 2 ** 31
    got = entries_from_gram(G)
    assert got == want
    assert max(abs(v) for v in got) < 2 ** 31
    if name in ("random", "checker_inverted"):  # and the plain 121-pixel accumulation
        direct = []
        for sa, sb in SIDES:
            sym = sa == sb
            direct += [v + v if sym and k != l else v for v, (k, l) in zip(family_direct(D[sa], D[sb], sym), ENTRIES)]
        assert got == direct


@pytest.mark.parametrize("name,t1,t0", _tiles(), ids=[c[0] for c in _tiles()])
def test_fragment_layout_emulation(name, t1, t0):
    """K order (11 rows x 12 columns in groups of 4, column 12 from the zeroed byte 15, 7 zero groups), selectors and the
    zero row give exactly G; the scratch layout and per-lane entry addresses give exactly the 50 integers."""
    s = staged(t1.astype(np.uint8), t0.astype(np.uint8))
    got, G = emulate_kernel(s)
    assert np.array_equal(G, gram_direct(t1, t0))
    assert got == entries_from_family(t1, t0)[0]


def test_the_kernel_reads_the_zeroed_bytes():
    """The column-12 byte of class-2 groups comes from byte 15 of the tile row and window row 12 from the zero row after
    the tiles: the result depends on both being zero (staging and the kernel's preamble make them so)."""
    rng = np.random.default_rng(3)
    t1, t0 = rng.integers(0, 256, (14, 14)), rng.integers(0, 256, (14, 14))
    s = staged(t1.astype(np.uint8), t0.astype(np.uint8))
    got, _ = emulate_kernel(s)
    assert got == entries_from_family(t1, t0)[0]
    for off in (ZROW, 5 * 16 + 15):
        bad = s.copy()
        bad[off] = 1
        assert emulate_kernel(bad)[0] != got
