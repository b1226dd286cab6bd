"""Device assignment of the starting genomes (gnx_genome_init_*, DeviceSpecies.init_genomes): exact
per-locus 1-allele counts on the homologues with the smallest Philox keys, checked against a numpy
restatement of the keys; the statistics of the draw; independence of entry order and strip cut; the
assignment after a real burn-in and through make_model(genome_init='device')."""
import functools
import os

import numpy as np
import pytest
from scipy import stats

from geonomics_b200 import genome_pack as gp

pytestmark = pytest.mark.gpu

M32 = np.uint64(0xFFFFFFFF)


def _mul(a, b):
    p = np.uint64(a) * np.asarray(b, dtype=np.uint64)
    return p >> np.uint64(32), p & M32


def _locus_key(seed, l):
    """k_l = first word of Philox4x32-10(counter (l, SITE_GENOME_INIT << 24, 0, 0), key = seed)."""
    c = [l & 0xFFFFFFFF, 10 << 24, 0, 0]
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k0, p1 & 0xFFFFFFFF, (p0 >> 32) ^ c[3] ^ k1, p0 & 0xFFFFFFFF]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c[0]


def _keys(ids, h, k):
    """K_l(i, h) = Philox2x32-10(counter 2i + h, key k_l), as uint64."""
    ctr = 2 * np.asarray(ids, dtype=np.uint64) + np.uint64(h)
    c0, c1 = ctr & M32, ctr >> np.uint64(32)
    for _ in range(10):
        hi, lo = _mul(0xD256D193, c0)
        c0, c1 = hi ^ np.uint64(k) ^ c1, lo
        k = (k + 0x9E3779B9) & 0xFFFFFFFF
    return (c0 << np.uint64(32)) | c1


def _expected(ids, counts, seed):
    """int8[n, L, 2]: at every locus the counts[l] homologues with the smallest keys carry the 1-allele."""
    n, L = len(ids), len(counts)
    g = np.zeros((n, L, 2), np.int8)
    for l in range(L):
        if counts[l] == 0:
            continue
        k = _locus_key(seed, l)
        keys = np.concatenate([_keys(ids, 0, k), _keys(ids, 1, k)])
        pick = np.argsort(keys, kind='stable')[:counts[l]]
        g[pick % n, l, pick // n] = 1
    return g


def _edge_p(L, n, rng):
    two_n = 2 * n
    edge = [0.0, 1.0, 1e-12, 0.5 / two_n, 1.5 / two_n, 1 - 1e-12, 1 - 0.5 / two_n, 0.5, 1.0 / two_n]
    return np.concatenate([edge, rng.random(L - len(edge))])


def _species(n, L, seed=3, traits=None, dim=(40, 30), capacity=None):
    from geonomics_b200.device import DeviceSpecies
    rng = np.random.default_rng(seed)
    X, Y = dim
    rasters = np.stack([np.ones((Y, X)), np.tile(np.linspace(0, 1, X), (Y, 1))])
    paths = (np.cumsum(rng.random((64, L)) < 0.05, axis=1) % 2).astype(np.uint8)
    ga = dict(L=L, paths=paths, traits=traits or [], dom=np.zeros(L, np.int8))
    prm = dict(b=0.5, R=0.5, lam=1, n_births_fixed=True, mating_radius=2.0, d_min=0.0, d_max=1.0, sex=False,
               sex_ratio_p=0.5, max_age=None, K_layer=0, K_factor=n / float(X * Y), move=True,
               move_distr=('wald', 1.0, 1.0), disp_distr=('wald', 1.0, 1.0), direction_mu=0.0, direction_kappa=0.0,
               density_grid_window_width=None)
    pop = dict(x=rng.uniform(0, X - 0.001, n), y=rng.uniform(0, Y - 0.001, n), age=rng.integers(0, 3, n).astype(np.int32),
               sex=rng.integers(0, 2, n).astype(np.int8), idx=np.sort(rng.choice(5 * n, n, replace=False)).astype(np.int64))
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=capacity or 4 * n, seed=seed)
    return dev, pop, (dim, rasters, prm, ga)


@pytest.mark.parametrize('L', [129, 1000])
def test_exact_counts_and_carriers(L):
    n = 3000 if L == 129 else 800
    rng = np.random.default_rng(L)
    dev, pop, _ = _species(n, L)
    try:
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        p = _edge_p(L, n, rng)
        counts = gp.carrier_counts(n, p)
        seed = 0x123456789ABCDEF
        dev.init_genomes(p, seed)
        s = dev.download(unpack=False)
        g = gp.unpack_genomes(s['genomes'], L)
        assert np.array_equal(g.sum(axis=(0, 2)), counts)
        assert np.array_equal(g, _expected(s['idx'], counts, seed))
        bits = np.unpackbits(s['genomes'].view(np.uint8), axis=-1, bitorder='little')
        assert not bits[:, :, L:].any()                                   # padding beyond L stays zero
        # the tskit layout: only the non-neutral loci carry bits, the rows list every carrier of every locus
        mask = np.zeros(L, np.uint8)
        nonneut = np.sort(rng.choice(L, L // 3, replace=False))
        mask[nonneut] = 1
        rows = dev.init_genomes(p, seed + 1, write_mask=mask, tskit_rows=True)
        s2 = dev.download()
        exp = _expected(s2['idx'], counts, seed + 1)
        assert np.array_equal(s2['g'][:, mask == 1], exp[:, mask == 1])
        assert not s2['g'][:, mask == 0].any()
        assert np.array_equal(np.bincount(rows['site'], minlength=L), counts)
        k = np.searchsorted(s2['idx'], rows['idx'])
        assert np.array_equal(s2['idx'][k], rows['idx'])
        listed = np.zeros((n, L, 2), np.int8)
        listed[k, rows['site'], rows['homologue']] = 1
        assert np.array_equal(listed, exp)
        node = 2 * k + rows['homologue']
        assert np.all((np.diff(rows['site']) > 0) | ((np.diff(rows['site']) == 0) & (np.diff(node) > 0)))
    finally:
        dev.close()


def test_refusals():
    from geonomics_b200 import _lib
    from geonomics_b200.device import DeviceSpecies
    dev, pop, (dim, rasters, prm, ga) = _species(500, 40)
    try:
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        with pytest.raises(_lib.GnxError, match='n_loci'):
            dev.genome_init_begin(np.ones(39, np.int64), 1)
        with pytest.raises(_lib.GnxError, match=r'\[0, 2n\]'):
            dev.genome_init_begin(np.full(40, 1001, np.int64), 1)
        with pytest.raises(_lib.GnxError, match='wrong state|gnx_genome_init_end'):
            dev.genome_init_end()
    finally:
        dev.close()
    bare = DeviceSpecies(dim, rasters, prm, None, capacity=2000, seed=1)
    try:
        bare.upload(pop['x'], pop['y'])
        with pytest.raises(_lib.GnxError, match='L = 0'):
            bare.genome_init_begin(np.zeros(0, np.int64), 1)
    finally:
        bare.close()


def test_distribution():
    n, L = 50000, 48
    rng = np.random.default_rng(11)
    dev, pop, _ = _species(n, L, dim=(120, 100))
    try:
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        p = np.concatenate([[0.5, 0.1, 0.9, 0.01], rng.random(L - 4)])
        counts = gp.carrier_counts(n, p)
        dev.init_genomes(p, 2024)
        s = dev.download()
        g = s['g'].astype(np.int64)
    finally:
        dev.close()
    N2 = 2 * n
    pvals = []
    for l in range(L):
        c = counts[l]
        p2 = c * (c - 1) / (N2 * (N2 - 1))                    # both homologues, drawn without replacement
        p0 = (N2 - c) * (N2 - c - 1) / (N2 * (N2 - 1))
        exp = n * np.array([p0, 1 - p0 - p2, p2])
        obs = np.bincount(g[:, l, :].sum(axis=1), minlength=3)
        if np.all(exp > 5):
            # the allele count is fixed (n1 + 2 n2 = c): one degree of freedom
            pvals.append(stats.chisquare(obs, exp, ddof=1).pvalue)
        # the two homologues carry the same share
        a, b = g[:, l, 0].sum(), g[:, l, 1].sum()
        assert abs(a - b) <= 6 * np.sqrt(c * (1 - c / N2) + 1)
    assert len(pvals) > 40
    assert stats.kstest(pvals, 'uniform').pvalue > 1e-4
    assert min(pvals) > 1e-5
    # carriers are uniform over the ids
    carriers = np.repeat(s['idx'], g[:, 0, :].sum(axis=1))
    assert stats.kstest(carriers, 'uniform', args=(0, 5 * n)).pvalue > 1e-4
    # loci independent: mean r^2 between pairs of loci is about 1/n
    f = g.sum(axis=2) / 2.0
    f = f[:, np.std(f, axis=0) > 0]
    r = np.corrcoef(f.T)
    iu = np.triu_indices(r.shape[0], 1)
    assert np.mean(r[iu] ** 2) < 3.0 / n


def test_determinism_and_entry_order():
    n, L = 4000, 100
    rng = np.random.default_rng(5)
    p = rng.random(L)
    out = []
    for seed, perm in ((7, False), (7, False), (8, False), (7, True)):
        dev, pop, _ = _species(n, L)
        try:
            o = rng.permutation(n) if perm else np.arange(n)
            dev.upload(pop['x'][o], pop['y'][o], pop['age'][o], pop['sex'][o], pop['idx'][o])
            dev.init_genomes(p, seed)
            out.append(dev.download())
        finally:
            dev.close()
    assert np.array_equal(out[0]['g'], out[1]['g'])
    assert not np.array_equal(out[0]['g'], out[2]['g'])
    assert np.array_equal(out[0]['idx'], out[3]['idx']) and np.array_equal(out[0]['g'], out[3]['g'])


@pytest.mark.parametrize('world', [2, 3])
def test_strips_give_the_single_context_genomes(world):
    from test_cuda_strips import _workload, _same
    from geonomics_b200.device import DeviceSpecies
    from geonomics_b200.strips import LocalStrips
    dim, rasters, prm, ga, pop, _ = _workload(n=6000, L=200, seed=8)
    p = np.random.default_rng(1).random(200)
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=77)
    st = LocalStrips(world, dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=77)
    try:
        for d in (dev, st):
            d.set_burn(True)
            d.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        dev.step(2)
        st.step(2)
        dev.init_genomes(p, 99)
        st.init_genomes(p, 99)
        dev.set_burn(False)
        st.set_burn(False)
        a, b = dev.download(), st.download()
        _same(a, b, -1)
        assert np.array_equal(a['g'].sum(axis=(0, 2)), gp.carrier_counts(len(a['idx']), p))
        for t in range(3):
            dev.step(1)
            st.step(1)
            _same(dev.download(), st.download(), t)
    finally:
        dev.close()
        st.close()


def test_after_a_real_burn_in():
    from oracle import step_oracle as so
    n, L = 3000, 96
    rng = np.random.default_rng(2)
    traits = [dict(loci=np.sort(rng.choice(L, 9, replace=False)), alpha=rng.normal(0, 0.2, 9), phi=0.3, gamma=1.0,
                   lyr_num=1, univ_adv=False)]
    dev, pop, _ = _species(n, L, traits=traits)
    try:
        dev.set_burn(True)
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        dev.step(6)
        n_now = dev.population_size()
        assert (dev.read('GSLOT', 4 * n) == -1).any()            # burn-in newborns own no genome row
        p = rng.random(L)
        dev.init_genomes(p, 31)
        dev.set_burn(False)
        s = dev.download()
        assert len(s['idx']) == n_now
        slots = dev.read('GSLOT', n_now)
        assert len(np.unique(slots)) == n_now and slots.min() == 0 and slots.max() == n_now - 1
        assert np.array_equal(s['g'].sum(axis=(0, 2)), gp.carrier_counts(n_now, p))
        z = so.phenotype(s['g'], traits)
        assert np.allclose(s['z'], z, rtol=0, atol=1e-12)
        dev.step(2)
        dev.sync()
    finally:
        dev.close()


PARAMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'data', 'params_small.py')


def test_make_model_assigns_on_the_device(monkeypatch):
    from geonomics_b200 import api
    orig = api.Species._set_genomes_and_tables
    mod = api.make_model(PARAMS, genome_init='device')
    assert mod.genome_init == 'device'
    spp = mod.comm[0]
    seen = {}

    def spy(self, *a, **k):
        seen['dl'] = []
        dl = self._dev.download

        def no_genomes(genomes=True, **kw):
            seen['dl'].append(genomes)
            return dl(genomes=genomes, **kw)
        self._dev.download = no_genomes
        try:
            return orig(self, *a, **k)
        finally:
            del self._dev.download
    monkeypatch.setattr(api.Species, '_set_genomes_and_tables', spy)
    mod.walk(10000, 'burn')
    assert seen['dl'] == [False]                                  # no genotype download
    n = len(spp)
    g = mod.get_genotypes()
    assert np.array_equal(g.sum(axis=(0, 2)), gp.carrier_counts(n, spp.gen_arch.p))
    mod.walk(5, 'main')
    assert len(spp.Nt) > 5 and spp.Nt[-1] > 0


def test_use_tskit_model_assigned_on_the_device(monkeypatch):
    """The tables invariant of test_use_tskit_model_tables_replay_to_the_genotypes with device genomes."""
    import test_model_gpu
    from geonomics_b200 import api
    monkeypatch.setattr(api, 'make_model', functools.partial(api.make_model, genome_init='device'))
    test_model_gpu.test_use_tskit_model_tables_replay_to_the_genotypes()


def test_rand_genarch_iterations_get_new_genomes(monkeypatch):
    from geonomics_b200 import api
    p = api.read_parameters_file(PARAMS)
    p['model']['its'] = dict(n_its=2, rand_landscape=False, rand_comm=False, rand_genarch=True, repeat_burn=False)
    p['model']['T'] = 3
    got = []
    orig = api.Species._set_genomes_on_device

    def spy(self, *a, **k):
        orig(self, *a, **k)
        s = self._dev.download()
        got.append((s['idx'], s['g']))
    monkeypatch.setattr(api.Species, '_set_genomes_on_device', spy)
    mod = api.make_model(p, genome_init='device')
    mod.run()
    assert len(got) == 2
    (i0, g0), (i1, g1) = got
    assert np.array_equal(i0, i1) and not np.array_equal(g0, g1)
