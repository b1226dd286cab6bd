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
