"""CPU: the numpy restatement of the device's Philox streams (tests/philox_ref.py) against the
Random123 known answers, the locus-key helper of the genome-initialisation tests, and stream
addressing with ids and seeds whose high words are set."""
import numpy as np
import pytest

import philox_ref as pr
from test_cuda_genome_init import _locus_key


@pytest.mark.parametrize('ctr,key,want', [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_random123_known_answers(ctr, key, want):
    got = pr.philox4x32_10(*ctr, *key)
    assert tuple(int(v) for v in got) == want


@pytest.mark.parametrize('seed', [0, 12345, 0xDEADBEEF12345678, (1 << 64) - 1])
def test_word0_of_the_genome_init_stream_is_the_locus_key(seed):
    loci = np.array([0, 1, 2, 31, 1000, 65535, 1 << 20])
    w = pr.stream_words(seed, loci, pr.SITE_GENOME_INIT, 0, 1)[:, 0]
    assert [int(v) for v in w] == [_locus_key(seed, int(l)) for l in loci]


def _scalar_block(seed, i, site, t, block):
    """One block by the definition, from Python integers (no vectorisation)."""
    ctr = (i & 0xFFFFFFFF, ((i >> 32) & 0xFFFFFFFF) ^ ((site << 24) & 0xFFFFFFFF), t & 0xFFFFFFFF, block)
    return [int(v) for v in pr.philox4x32_10(*ctr, seed & 0xFFFFFFFF, seed >> 32)]


def test_ids_and_seeds_with_high_words():
    seed = 0x9E3779B97F4A7C15
    ids = np.array([0, 1, (1 << 32) - 1, 1 << 32, (1 << 32) + 7, (1 << 40) + 3, (1 << 62) + 11], dtype=np.int64)
    w = pr.stream_words(seed, ids, pr.SITE_DISP, (1 << 32) + 5, 11)    # t is taken mod 2^32
    for r, i in enumerate(ids):
        want = sum((_scalar_block(seed, int(i), pr.SITE_DISP, 5, b) for b in range(3)), [])[:11]
        assert [int(v) for v in w[r]] == want
    # the high id word and the site share the second counter word: both must change the stream
    a = pr.stream_words(seed, [5], pr.SITE_MATE, 3, 4)
    assert not np.array_equal(a, pr.stream_words(seed, [5 + (1 << 32)], pr.SITE_MATE, 3, 4))
    assert not np.array_equal(a, pr.stream_words(seed, [5], pr.SITE_DEATH, 3, 4))
    # seed_lo is the first key word, seed_hi the second
    lo, hi = 0x01234567, 0x89ABCDEF
    got = pr.stream_words((hi << 32) | lo, [9], pr.SITE_MOVE, 2, 4)[0]
    assert [int(v) for v in got] == [int(v) for v in pr.philox4x32_10(9, pr.SITE_MOVE << 24, 2, 0, lo, hi)]
    assert not np.array_equal(got, pr.stream_words((lo << 32) | hi, [9], pr.SITE_MOVE, 2, 4)[0])


def test_derived_draws():
    w = np.array([[0, 0, 0xFFFFFFFF, 0xFFFFFFFF, 0x80000000, 0x40000000]], dtype=np.uint32)
    assert pr.uniform(w, 0)[0] == 0.0
    assert pr.uniform(w, 2)[0] == (2.0 ** 53 - 1) / 2.0 ** 53
    assert pr.uniform(w, 4)[0] == 0.5 + 2.0 ** -29      # (2^26 * 2^26 + 2^24) / 2^53
    assert pr.uniform_f32(np.uint32(0xFFFFFFFF)) == np.float32(1 - 2.0 ** -24)
    assert pr.uniform_pos_f32(np.uint32(0)) == np.float32(2.0 ** -32)
    assert pr.uniform_pos_f32(np.uint32(0xFFFFFFFF)) == np.float32(1.0)
    R = np.array([0, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF], dtype=np.uint32)
    assert list(pr.choose_k(R, 10)) == [0, 4, 5, 9]
    # the restated lognormal is a lognormal: median exp(p1), and its error bound stays small
    ws = pr.stream_words(3, np.arange(20000), pr.SITE_MOVE, 0, 3)
    d, rel = pr.lognormal_f32(ws[:, 1], ws[:, 2], 0.0, 0.5)
    assert abs(np.median(d) - 1.0) < 0.02
    assert np.median(rel) < 1e-5 and rel.max() < 1e-3


# ---- the on-the-fly surface direction and the Wald distance --------------------------------------------
def _exact_fma(a, b, c):
    from fractions import Fraction
    return np.array([pr._round_f32(Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z)))
                     for x, y, z in zip(a, b, c)], np.float32)


def test_fma_halfway_cases():
    """Sums whose float64 rounding lands on a float32 midpoint while the exact sum does not: rounding the
    float64 sum (ties to even) would give the wrong neighbour."""
    f = np.float32
    a = np.array([64 * (1 + 2.0 ** -23), 64 * (1 + 2.0 ** -23), -64 * (1 + 2.0 ** -23), 1 + 2.0 ** -23], np.float32)
    b = np.array([1 - 2.0 ** -23, 1 - 2.0 ** -23, 1 - 2.0 ** -23, 1 - 2.0 ** -23], np.float32)
    c = np.array([2.0 ** 30 + 128, 2.0 ** 30, -(2.0 ** 30 + 128), 2.0 ** 24 + 2], np.float32)
    want = _exact_fma(a, b, c)
    naive = (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)
    assert want[0] == f(2.0 ** 30 + 128) and naive[0] == f(2.0 ** 30 + 256)
    assert want[2] == f(-(2.0 ** 30 + 128)) and naive[2] == f(-(2.0 ** 30 + 256))
    assert np.array_equal(pr.fma_f32(a, b, c), want)
    rng = np.random.default_rng(0)
    a = rng.random(2000).astype(np.float32)
    b = (rng.random(2000) * 2.0 ** -rng.integers(0, 30, 2000)).astype(np.float32)
    c = (rng.random(2000) * 3).astype(np.float32)
    assert np.array_equal(pr.fma_f32(a, b, c), _exact_fma(a, b, c))


def _words(*ws):
    return np.array([ws], dtype=np.uint32)


TAB = np.linspace(0, np.pi, pr.VM_TAB_LEN).astype(np.float32)
TAB[pr.VM_TAB_CELLS + 1:] = np.linspace(TAB[pr.VM_TAB_CELLS - 1], np.float32(np.pi), pr.VM_TAB_FINE + 1)


def test_surface_direction_hand_built():
    D = pr.SURF_DIRS
    zero = np.zeros((1, 8), np.float32)
    # all zero, mixture: uniform over the 8 directions; word j 2^29 gives target j, so direction j.  A zero
    # von Mises word gives |theta| = tab[0] = 0.  Direction 3 is pi itself: it wraps to -pi
    for j in range(8):
        h, nw = pr.surface_direction(_words(j << 29, 0), 0, zero, True, 12.0, TAB)
        want = -np.pi if j == 3 else D[j]
        assert h[0] == np.float16(want) and nw[0] == 2
    # all zero, unimodal: the mean of all 8 directions, summed in float32 in order
    s = np.float32(0)
    for d in D:
        s = np.float32(s + d)
    h, nw = pr.surface_direction(_words(0), 0, zero, False, 12.0, TAB)
    assert h[0] == np.float16(s / np.float32(8)) and nw[0] == 1
    # one non-zero neighbour: every mixture draw picks it
    one = zero.copy()
    one[0, 6] = 0.3
    for u in (0, 1 << 31, 0xFFFFFFFF):
        assert pr.surface_direction(_words(u, 0), 0, one, True, 12.0, TAB)[0][0] == np.float16(D[6])
    # ties for the maximum: pi and -3 pi / 4 average to pi / 8, which is neither
    tie = np.full((1, 8), 0.1, np.float32)
    tie[0, 0] = tie[0, 3] = 0.7
    h, _ = pr.surface_direction(_words(0), 0, tie, False, 12.0, TAB)
    assert h[0] == np.float16((D[0] + D[3]) / np.float32(2)) and abs(float(h[0]) - np.pi / 8) < 1e-3
    # the sign of theta is bit 31 of the table word; the cell is bits 30..19, the position bits 18..0
    r = np.uint32((1 << 31) | (5 << 19) | (1 << 18))            # cell 5, f = 1/2, negative
    h, _ = pr.surface_direction(_words(r), 0, one, False, 12.0, TAB)
    want = np.float32(D[6] - (TAB[5] + np.float32(0.5) * (TAB[6] - TAB[5])))
    assert h[0] == np.float16(want)
    # the last cell goes to the fine table: fine cell 3 at f = 1/4
    r = np.uint32((4095 << 19) | (3 << 11) | (1 << 9))
    v = pr.vonmises_tab(np.array([r], np.uint32), TAB)[0]
    a, b = TAB[pr.VM_TAB_CELLS + 4], TAB[pr.VM_TAB_CELLS + 5]
    assert v == pr.fma_f32(np.float32(0.25), b - a, a)[0]
    # kappa < 1e-8: uniform on the circle from one uniform_f32 word, the table unread
    h, nw = pr.surface_direction(_words(0, 0x80000000), 0, zero, True, 0.0, None)
    assert nw[0] == 2 and h[0] == np.float16(D[0])      # target 0 -> direction 0; theta = pi (2 u - 1) = 0
    h, nw = pr.surface_direction(_words(1 << 31, 0), 0, zero, True, 0.0, None)
    assert h[0] == np.float16(-np.pi)                   # direction 0 + theta -pi: -pi stays, it does not wrap
    h, nw = pr.surface_direction(_words(0xC0000000), 0, one, False, 0.0, None)
    assert nw[0] == 1 and h[0] == np.float16(-np.pi)    # pi / 2 + pi (2 * 3/4 - 1) is exactly pi: wraps


def test_wald_restatement_and_bound():
    """wald_f32 against numpy's formula in float64: agreement within the bound, and few ambiguous draws."""
    w = pr.stream_words(99, np.arange(20000), pr.SITE_MOVE, 3, 3)
    d, rel, amb = pr.wald_f32(w[:, 0], w[:, 1], w[:, 2], 1.0, 1.0)
    z, _ = pr.normal_f32(w[:, 0], w[:, 1])
    Y = z * z
    X = 1 + 0.5 * (Y - np.sqrt(4 * Y + Y * Y))
    U = pr.uniform_f32(w[:, 2]).astype(np.float64)
    ref = np.where(U <= 1 / (1 + X), X, 1 / X)
    ok = ~amb
    assert amb.sum() < 20
    assert np.all(np.abs(d[ok] - ref[ok]) <= 1e-9 * ref[ok] + rel[ok] * ref[ok])
    assert np.all(rel[ok] < 1e-3) and np.median(rel) < 1e-5
    assert abs(np.mean(d) - 1.0) < 0.05                  # Wald(1, 1): mean 1
