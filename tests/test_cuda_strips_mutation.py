"""Mutation (by-locus layout, neutral + deleterious) and Poisson births under strip decomposition,
against the undecomposed run with the same seed: after every step the same individuals (ids,
positions, ages, genomes, phenotypes, fitness), the same step records, and -- with mutation -- the
same mutation log and tables on every rank.  Every rank replays the species-wide mutation draws;
Poisson births are keyed by the species-wide pair positions, which the pairs all-gather supplies."""
import numpy as np
import pytest

from test_cuda_strips import _workload, _single, _strips, _same

pytestmark = pytest.mark.gpu

L = 512
NCY = int(44 / 2.0000002) + 1          # mating-grid rows of the (48, 44) landscape at radius 2


def _with(wl, **prm):
    dim, rasters, p, ga, pop, g = wl
    return dim, rasters, dict(p, **prm), ga, pop, g


def _mutation(wl, seed=0, mu=4e-5):
    """Neutral + deleterious mutation over every non-trait locus; the trait loci are the non-neutral ones.
    Deleterious mutations are rarer and milder than the default gamma(0.2, 0.2), so that a few hundred of
    them over a run do not drive the population extinct."""
    ga = wl[3]
    trait_loci = np.sort(np.concatenate([t['loci'] for t in ga['traits']]))
    mutables = [int(v) for v in np.random.default_rng(seed).permutation(np.setdiff1d(np.arange(ga['L']), trait_loci))]
    return dict(mu_neut=mu, mu_delet=mu / 5, mutables=mutables, nonneut_loci=trait_loci, delet_s_scale=0.02)


def _low_population(wl, y_max=30.0):
    """Everyone starts below y_max, so a strip above it has no pairs in the first step."""
    dim, rasters, prm, ga, pop, g = wl
    return dim, rasters, prm, ga, dict(pop, y=pop['y'] * (y_max / dim[1])), g


def _run_single(wl, steps, seed, mut=None, switch=None):
    from geonomics_b200.device import DeviceSpecies
    dim, rasters, prm, ga, pop, g = wl
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=seed)
    try:
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
        if mut:
            dev.set_mutation(**mut)
        out, logs = [], []
        for t in range(steps):
            if switch and t == switch[0]:
                dev.set_life_history(**switch[1])
            dev.step(1)
            dev.sync()
            out.append(dev.download())
            logs.append(dev.read_mutations() if mut else None)
        return dict(states=out, records=dev.step_records(), logs=logs)
    finally:
        dev.close()


def _run_strips(wl, world, steps, seed, mut=None, bounds=None, device_barrier=False, switch=None):
    from geonomics_b200 import strips
    dim, rasters, prm, ga, pop, g = wl
    st = strips.LocalStrips(world, dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=seed, bounds=bounds,
                            device_barrier=device_barrier)
    try:
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
        if mut:
            st.set_mutation(**mut)
        out, logs, recs, local_pairs, holders = [], [], [], [], []
        for t in range(steps):
            if switch and t == switch[0]:
                for r in st.ranks:
                    r.dev.set_life_history(**switch[1])
            st.step(1)
            out.append(st.download())
            per_rank = [r.dev.step_records() for r in st.ranks]
            recs += strips.merge_records(per_rank)
            local_pairs.append([p[-1]['n_pairs'] for p in per_rank])
            holders.append([r.dev.download(genomes=False)['idx'] for r in st.ranks])
            logs.append(st.read_mutations() if mut else None)      # raises unless every rank holds the same
        captures = st.ranks[0].dev.graph_capture_count
        return dict(states=out, records=recs, logs=logs, local_pairs=local_pairs, holders=holders,
                    captures=captures)
    finally:
        st.close()


def _records(recs):
    return [(r['Nt'], r['n_births'], r['n_deaths'], r['n_pairs']) for r in recs]


def _compare(ref, got):
    assert len(ref['states']) == len(got['states'])
    for t, (a, b) in enumerate(zip(ref['states'], got['states'])):
        _same(a, b, t)
    assert _records(ref['records']) == _records(got['records'])
    for t, (la, lb) in enumerate(zip(ref['logs'], got['logs'])):
        if la is None:
            assert lb is None
            continue
        (rows_a, st_a), (rows_b, st_b) = la, lb
        assert rows_a == rows_b, 'mutation log differs at step %d' % t
        assert st_a['n_mutables'] == st_b['n_mutables']
        for k in ('nonneut_loci', 'delet_loci', 'delet_s'):
            assert np.array_equal(st_a[k], st_b[k]), '%s differs at step %d' % (k, t)


def _mutation_was_exercised(got, steps, idle_rank):
    rows = [r for log in got['logs'] for r in log[0]]
    assert len(rows) >= 10 * steps, len(rows)
    assert {r['type'] for r in rows} == {'neut', 'delet'}
    # mutated offspring ended up on more than one rank
    ranks = set()
    for (log, _), holders in zip(got['logs'], got['holders']):
        for r in log:
            ranks |= {k for k, ids in enumerate(holders) if r['individual'] in ids}
    assert len(ranks) >= 2, ranks
    if idle_rank:
        # a rank without pairs (so without births) replayed a step in which other ranks mutated offspring
        assert any(min(pairs) == 0 and len(log[0]) > 0 for pairs, log in zip(got['local_pairs'], got['logs']))


@pytest.mark.parametrize('world', [2, 3, 4])
def test_mutation_under_strips_reproduces_the_undecomposed_run(world):
    wl = _workload(L=L, seed=3)
    bounds = None
    if world > 2:
        # the top strip holds the two top mating-grid rows, which nobody reaches in the first step
        wl = _low_population(wl)
        bounds = np.array([0, 10, NCY - 2, NCY] if world == 3 else [0, 7, 14, NCY - 2, NCY], np.int32)
    mut = _mutation(wl, seed=world)
    ref = _run_single(wl, 6, seed=77, mut=mut)
    got = _run_strips(wl, world, 6, seed=77, mut=mut, bounds=bounds)
    _compare(ref, got)
    _mutation_was_exercised(got, 6, idle_rank=world > 2)


@pytest.mark.parametrize('world', [2, 3, 4])
def test_poisson_births_under_strips(world):
    wl = _with(_workload(seed=5), n_births_fixed=False, lam=2.5)
    ref, ref_recs = _single(wl, 6, seed=31)
    got, recs, _ = _strips(wl, world, 6, seed=31)
    for t, (a, b) in enumerate(zip(ref, got)):
        _same(a, b, t)
    assert _records(ref_recs) == _records(recs)
    assert any(r['n_births'] > r['n_pairs'] > 0 for r in recs)


def test_poisson_births_with_surfaces_sexes_and_uneven_rows():
    wl = _with(_workload(surfaces=True, sex=True, b=0.9, seed=11), n_births_fixed=False, lam=2.5)
    bounds = np.array([0, 2, 9, NCY], dtype=np.int32)
    ref, ref_recs = _single(wl, 5, seed=5)
    got, recs, _ = _strips(wl, 3, 5, seed=5, bounds=bounds)
    for t, (a, b) in enumerate(zip(ref, got)):
        _same(a, b, t)
    assert _records(ref_recs) == _records(recs)
    assert any(r['n_births'] > r['n_pairs'] > 0 for r in recs)


@pytest.mark.timeout(600)
@pytest.mark.parametrize('world', [2, 4])
def test_mutation_and_poisson_births_through_step_graphs_with_device_barriers(world):
    """gnx_step graphs with the peer-memory barriers: phase 3, pairs all-gather, phase 8, births all-gather."""
    wl = _with(_workload(surfaces=True, L=L, seed=21), n_births_fixed=False, lam=2.5)
    mut = _mutation(wl, seed=9, mu=2e-5)
    ref = _run_single(wl, 6, seed=13, mut=mut)
    got = _run_strips(wl, world, 6, seed=13, mut=mut, device_barrier=True)
    _compare(ref, got)
    assert sum(len(log[0]) for log in got['logs']) > 0
    assert any(r['n_births'] > r['n_pairs'] > 0 for r in got['records'])


@pytest.mark.timeout(600)
def test_switch_from_fixed_to_poisson_births_recaptures_the_step():
    """set_life_history(n_births_fixed=False) between graph-launched steps changes the step key, so the next
    step is captured again with the Poisson phase sequence."""
    wl = _workload(L=L, seed=8)
    mut = _mutation(wl, seed=2, mu=2e-5)
    switch = (3, dict(n_births_fixed=False, lam=2.5))
    ref = _run_single(wl, 6, seed=17, mut=mut, switch=switch)
    got = _run_strips(wl, 2, 6, seed=17, mut=mut, device_barrier=True, switch=switch)
    _compare(ref, got)
    assert all(r['n_births'] == r['n_pairs'] for r in got['records'][:3])
    assert any(r['n_births'] > r['n_pairs'] for r in got['records'][3:])
    assert got['captures'] >= 2


def test_burn_in_with_poisson_births():
    from geonomics_b200.device import DeviceSpecies
    from geonomics_b200.strips import LocalStrips
    dim, rasters, prm, ga, pop, g = _with(_workload(seed=4), n_births_fixed=False, lam=2.5)
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=9)
    st = LocalStrips(3, dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=9)
    try:
        dev.set_burn(True)
        st.set_burn(True)
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        dev.step(5)
        dev.sync()
        st.step(5)
        a, b = dev.download(genomes=False), st.download(genomes=False)
        assert np.array_equal(a['idx'], b['idx'])
        for k in ('x', 'y', 'age'):
            assert np.array_equal(a[k], b[k]), k
        ra, rb = dev.step_records(), st.step_records()
        assert _records(ra) == _records(rb)
        assert any(r['n_births'] > r['n_pairs'] for r in rb)
    finally:
        dev.close()
        st.close()


def test_mutables_exhausted_is_an_error_under_strips():
    from geonomics_b200._lib import GnxError
    from geonomics_b200.strips import LocalStrips
    dim, rasters, prm, ga, pop, g = wl = _workload(seed=6)
    st = LocalStrips(2, dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=7)
    try:
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
        st.set_mutation(1e-3, 0.0, [5, 9], _mutation(wl)['nonneut_loci'])
        with pytest.raises(GnxError) as ei:
            st.step(3)
            st.download()
        assert ei.value.code == -6
    finally:
        st.close()


def test_unsupported_combinations_are_refused_at_the_call():
    """The tskit layout, trait mutation, tskit recording and injected draws stay unsupported under strips; each
    is refused by the call that would set it up, and the strips then still run the undecomposed model."""
    from geonomics_b200._lib import GnxError
    from geonomics_b200.strips import LocalStrips
    wl = _workload(seed=12)
    dim, rasters, prm, ga, pop, g = wl
    nonneut = _mutation(wl)['nonneut_loci']
    st = LocalStrips(2, dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=19)
    try:
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
        # the strip guards' own messages: a one-GPU context refuses trait mutation without the tskit layout too,
        # but for another reason (the reference raises for it)
        refused = 'under strip decomposition'
        with pytest.raises(GnxError, match=refused):
            st.set_mutation(1e-5, 0.0, [1, 2, 3], nonneut, tskit_layout=True)
        with pytest.raises(GnxError, match='trait mutation is not supported ' + refused):
            st.set_mutation(1e-5, 0.0, [1, 2, 3], nonneut, trait_mus=[1e-5, 0.0],
                            trait_alpha_distr=[(0.0, 0.1, None), (0.0, 0.1, None)])
        for r in st.ranks:
            with pytest.raises(GnxError, match=refused):
                r.dev.tskit_enable(10000, 10000)
            with pytest.raises(GnxError, match=refused):
                r.dev.set_draws(dict(death_u=np.full(len(pop['x']), 0.5)))
        got = []
        for _ in range(2):
            st.step(1)
            got.append(st.download())
        recs = st.step_records()
    finally:
        st.close()
    ref, ref_recs = _single(wl, 2, seed=19)
    for t, (a, b) in enumerate(zip(ref, got)):
        _same(a, b, t)
    assert _records(ref_recs) == _records(recs)
