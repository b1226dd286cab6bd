"""CPU tests of the device genome assignment's host side: the per-locus 1-allele counts, the ctypes
struct of gnx_genome_init_t, and the genome_init option of make_model."""
import os
import re

import numpy as np
import pytest

from geonomics_b200 import _lib, api
from geonomics_b200 import genome_pack as gp

HERE = os.path.dirname(os.path.abspath(__file__))
PARAMS = os.path.join(HERE, 'data', 'params_small.py')


def _host_rule(n, p):
    """The per-locus count of the post-burn-in assignment loop as the reference writes it (genome.py:1127-1136)."""
    out = []
    for freq in p:
        n_mut = int(round(2 * n * freq, 0))
        if n_mut == n * 2 and freq < 1:
            n_mut -= 1
        if n_mut == 0 and freq > 0:
            n_mut = 1
        out.append(n_mut)
    return np.array(out, dtype=np.int64)


@pytest.mark.parametrize('n', [1, 2, 3, 7, 10, 1000, 4097, 10 ** 7])
def test_carrier_counts_follow_the_host_rule_on_edge_cases(n):
    two_n = 2 * n
    p = np.array([0.0, 1.0, 1e-300, 1e-12, 0.4 / two_n, 0.5 / two_n, 1.5 / two_n, 2.5 / two_n,   # tiny and .5 products
                  1 - 1e-12, 1 - 0.4 / two_n, 1 - 0.5 / two_n, np.nextafter(1.0, 0.0),          # just below 1
                  0.5, 0.25, 0.75, 1.0 / 3.0])
    p = np.concatenate([p, np.random.default_rng(n).random(300)])
    got = gp.carrier_counts(n, p)
    assert got.dtype == np.int64
    assert np.array_equal(got, _host_rule(n, p))
    assert got[0] == 0 and got[1] == two_n                  # p = 0: lost; p = 1: fixed
    assert got[2] == 1 and got[3] == 1                      # tiny p > 0 keeps one copy
    assert got[8] == two_n - 1 or two_n == 2                # p just below 1 is never fixed
    assert np.all((got >= 0) & (got <= two_n))


def test_carrier_counts_round_half_to_even():
    # 2n p = k + 0.5 exactly: numpy's (and Python's) rounding goes to the even neighbour
    n = 4
    p = np.array([0.5, 1.5, 2.5, 3.5, 4.5]) / 8.0
    assert list(gp.carrier_counts(n, p)) == [1, 2, 2, 4, 4]
    assert list(gp.carrier_counts(n, p)) == list(_host_rule(n, p))


def test_genome_init_struct_matches_the_header_field_order():
    hdr = open(_lib.HEADER_PATH).read()
    end = hdr.index('} gnx_genome_init_t;')
    body = hdr[hdr.rindex('typedef struct {', 0, end) + len('typedef struct {'):end]
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    names = [d.strip().split()[-1].lstrip('*') for d in body.split(';') if d.strip()]
    assert names == [f[0] for f in _lib.GenomeInit._fields_]


def test_make_model_rejects_an_unknown_genome_init():
    p = api.read_parameters_file(PARAMS)
    with pytest.raises(ValueError, match='genome_init'):
        api.make_model(p, genome_init='gpu')
    with pytest.raises(ValueError, match='genome_init'):
        api.Model('m', p, genome_init=None)
