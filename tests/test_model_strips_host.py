"""Host side of a Model cut into strips: the bookkeeping of the landscape rows that adjacent strips share in
the burn-in spatial statistic (against a numpy tally of the whole landscape), and the refusals that
make_model raises before any device work."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from geonomics_b200 import api, strips  # noqa: E402

PARAMS = os.path.join(HERE, 'data', 'params_small.py')


def _whole_tally(x, y, X, Y):
    """k_burnin_count: the transposed tally counts[iy * X + ix], only for ix < Y and iy < X."""
    ix, iy = x.astype(np.int64), y.astype(np.int64)
    keep = (ix < Y) & (iy < X)
    return np.bincount(iy[keep] * X + ix[keep], minlength=X * Y)


def _band_tally(x, y, X, Y, ly0, ly1):
    """k_strip_burnin_count: the same tally over the band rows [ly0, ly1) only."""
    ix, iy = x.astype(np.int64), y.astype(np.int64)
    assert np.all((iy >= ly0) & (iy < ly1)), 'an individual outside its strip band'
    keep = (ix < Y) & (iy < X)
    return np.bincount((iy[keep] - ly0) * X + ix[keep], minlength=(ly1 - ly0) * X).reshape(ly1 - ly0, X)


@pytest.mark.parametrize('dim, cell_size, world', [
    ((40, 40), 2.0000002, 3),        # boundaries fall inside landscape rows
    ((40, 40), 2.0, 3),              # boundaries on whole landscape rows
    ((64, 24), 1.5, 4),              # non-square, wider than tall
    ((20, 52), 2.5, 5),              # non-square, taller than wide: the tally drops x >= dim_y
    ((30, 30), 0.3, 6),              # bands of one or two landscape rows
])
def test_strip_bands_reproduce_the_whole_landscape_statistic(dim, cell_size, world):
    X, Y = dim
    rng = np.random.default_rng(world)
    ncy = int(Y / cell_size) + 1
    for plan in range(3):                                        # random cuts of the mating grid
        bounds = strips.plan_rows(ncy, world, rng.random(ncy))
        bands = strips.band_rows(bounds, cell_size, Y)
        adds, skip_last = strips.shared_band_rows(bands)
        # the bands cover every landscape row once, apart from the rows they share
        assert sum(b1 - b0 - int(sk) for (b0, b1), sk in zip(bands, skip_last)) == Y
        prev = [np.zeros((b1 - b0, X), np.int64) for b0, b1 in bands]
        prev_whole = np.zeros(X * Y, np.int64)
        for step in range(4):                                    # successive burn-in steps
            n = int(rng.integers(0, 4000))
            x, y = rng.random(n) * X, rng.random(n) * Y
            own = strips.owner_of(y, bounds, cell_size, ncy)
            now = [_band_tally(x[own == r], y[own == r], X, Y, *bands[r]) for r in range(world)]
            lasts = [b[-1].copy() for b in now]
            s1 = s2 = 0
            for r in range(world):
                for q in adds[r]:
                    now[r][0] += lasts[q]
                rows = len(now[r]) - int(skip_last[r])
                d = now[r][:rows] - prev[r][:rows]
                s1, s2 = s1 + int(d.sum()), s2 + int((d * d).sum())
                prev[r][:rows] = now[r][:rows]
            whole = _whole_tally(x, y, X, Y)
            dw = whole - prev_whole
            prev_whole = whole
            assert (s1, s2) == (int(dw.sum()), int((dw * dw).sum())), (plan, step)


def test_shared_rows_follow_the_band_ends():
    cs = 2.0000002
    bounds = np.array([0, 5, 10, 20], np.int32)
    bands = strips.band_rows(bounds, cs, 40)
    assert bands == [(0, 11), (10, 21), (20, 40)]
    adds, skip = strips.shared_band_rows(bands)
    assert adds == [[], [0], [1]] and skip == [True, True, False]
    # a one-row band shared with both neighbours: both lower last rows go to the upper band
    adds, skip = strips.shared_band_rows([(0, 3), (2, 3), (2, 5)])
    assert adds == [[], [0], [0, 1]] and skip == [True, True, False]


def _params(**edit):
    p = api.read_parameters_file(PARAMS)
    spp = p.comm.species.spp_0
    for k, v in edit.items():
        sect, key = k.split('__')
        (spp.gen_arch.traits.trait_0 if sect == 'trait' else spp[sect])[key] = v
    return p


@pytest.mark.parametrize('edit, strips_arg, match', [
    (dict(gen_arch__use_tskit=True), 2, 'use_tskit'),
    (dict(trait__mu=1e-4), 2, 'trait mutation'),
    (dict(mating__mating_radius=None), 2, 'panmictic'),
    ({}, 11, 'mating-grid rows'),                # 40 / 2 -> 21 mating-grid rows: 10 strips at most
    ({}, 1, 'at least 2'),
    ({}, True, 'process group'),
    ({}, 'two', 'process group'),
])
def test_make_model_refuses_what_strips_do_not_carry(edit, strips_arg, match):
    with pytest.raises(ValueError, match=match):
        api.make_model(_params(**edit), strips=strips_arg)
