"""Sort + simplify of the tskit tables on the device (gnx_simplify, DeviceSpecies.simplify_tables) against the
host restatement tables.simplify_columns: every output column must be bitwise equal."""
import copy
import os

import numpy as np
import pytest

from geonomics_b200.tables import TableColumns, simplify_columns

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
PARAMS = os.path.join(HERE, 'data', 'params_small.py')


def grow(tc, alive, steps, rng, t0=0, bp=5.0, birth_frac=0.3):
    """`steps` time steps of model-shaped births appended to `tc`: overlapping generations, both parents drawn
    from the living, ~Poisson(bp) breakpoints per homologue at k - 0.5, each homologue's segments alternating
    between its parent's two homologues from a random start, births at time -t.  alive: int[n, 2] node ids of
    the living; returns the new one (as many die as are born)."""
    L = tc.sequence_length
    for t in range(t0 + 1, t0 + steps + 1):
        B = max(1, int(birth_frac * len(alive)))
        par = rng.integers(len(alive), size=(B, 2))
        first = tc.individuals.append_columns(flags=np.zeros(B, np.int32), location=rng.random((B, tc.n_loc)),
                                              idx=tc.individuals.num_rows + np.arange(B))
        node0 = tc.nodes.append_columns(flags=np.ones(2 * B, np.int32), time=np.full(2 * B, -float(t)),
                                        population=np.zeros(2 * B, np.int32),
                                        individual=np.repeat(first + np.arange(B, dtype=np.int32), 2))
        H = 2 * B                                           # child homologue h = 2 o + j has parent par[o, j]
        k = rng.poisson(bp, size=H)
        hb = np.repeat(np.arange(H), k)
        pos = rng.integers(1, L, size=len(hb))
        o = np.lexsort((pos, hb))
        hb, pos = hb[o], pos[o]
        keep = np.r_[True, (hb[1:] != hb[:-1]) | (pos[1:] != pos[:-1])] if len(hb) else np.zeros(0, bool)
        hb, pos = hb[keep], pos[keep]
        k = np.bincount(hb, minlength=H)
        bo = np.cumsum(k) - k
        seg_h = np.repeat(np.arange(H), k + 1)
        i = np.arange(len(seg_h)) - (np.cumsum(k + 1) - (k + 1))[seg_h]
        bps = pos - 0.5
        left = np.where(i == 0, 0.0, bps[np.maximum(bo[seg_h] + i - 1, 0)] if len(bps) else 0.0)
        right = np.where(i == k[seg_h], float(L), bps[np.minimum(bo[seg_h] + i, max(len(bps) - 1, 0))]
                         if len(bps) else float(L))
        start = rng.integers(2, size=H)
        pind = par.reshape(-1)[seg_h]
        parent = alive[pind, (i + start[seg_h]) % 2]
        tc.edges.append_columns(left=left, right=right, parent=parent.astype(np.int32),
                                child=(node0 + seg_h).astype(np.int32))
        dead = rng.choice(len(alive), size=B, replace=False)
        born = node0 + np.arange(2 * B, dtype=np.int64).reshape(B, 2)
        alive = np.concatenate([np.delete(alive, dead, axis=0), born])
    return alive


def model_tables(n, steps, L=1000, seed=1, n_mut=2000, bp=5.0):
    """Founders at time 1 (2n nodes, n individuals) and `steps` steps of births; mutations on random nodes
    and sites; a few nodes without an individual.  Returns (tables, alive node ids)."""
    rng = np.random.default_rng(seed)
    tc = TableColumns(L, 1)
    tc.sites.append_columns(position=np.arange(L, dtype=np.float64), nonneutral=np.zeros(L, np.int8))
    tc.individuals.append_columns(flags=np.ones(n, np.int32), location=rng.random((n, tc.n_loc)), idx=np.arange(n))
    tc.nodes.append_columns(flags=np.ones(2 * n, np.int32), time=np.ones(2 * n), population=np.zeros(2 * n, np.int32),
                            individual=np.repeat(np.arange(n, dtype=np.int32), 2))
    alive = grow(tc, np.arange(2 * n, dtype=np.int64).reshape(n, 2), steps, rng, bp=bp)
    nn = tc.nodes.num_rows
    ind = tc.nodes.individual
    ind[rng.choice(nn, size=max(1, nn // 50), replace=False)] = -1
    add_mutations(tc, rng, n_mut)
    return tc, alive, rng


def add_mutations(tc, rng, n_mut):
    t = rng.random(n_mut)
    t[::7] = np.nan
    tc.mutations.append_columns(site=rng.integers(tc.sites.num_rows, size=n_mut).astype(np.int32),
                                node=rng.integers(tc.nodes.num_rows, size=n_mut).astype(np.int32), time=t)


def shuffled_samples(alive, rng):
    s = alive.reshape(-1).copy()
    rng.shuffle(s)
    return s


def clone(tc):
    out = TableColumns(tc.sequence_length, 0)
    out.n_loc = tc.n_loc
    out.nodes, out.edges, out.individuals, out.sites, out.mutations = (copy.deepcopy(x) for x in (
        tc.nodes, tc.edges, tc.individuals, tc.sites, tc.mutations))
    return out


def columns(tc):
    return {'%s.%s' % (t, k): v for t in ('nodes', 'edges', 'individuals', 'sites', 'mutations')
            for k, v in getattr(tc, t).asdict().items()}


def assert_tables_equal(a, b):
    ca, cb = columns(a), columns(b)
    assert ca.keys() == cb.keys()
    for k in ca:
        x, y = ca[k], cb[k]
        assert x.dtype == y.dtype and x.shape == y.shape, k
        if x.dtype.kind == 'f':                         # bitwise: NaN in locations and mutation times
            x, y = x.view(np.int64), y.view(np.int64)
        assert np.array_equal(x, y), k


@pytest.fixture(scope='module')
def dev():
    import sys
    sys.path.insert(0, HERE)
    from golden_io import load_case
    from parity_util import make_device
    z, arch, prm, state, draws = load_case('base')
    d = make_device(arch, prm, capacity=4 * len(state['x']) + 256, seed=3)
    yield d
    d.close()


def check(dev, tc, samples):
    host = simplify_columns(clone(tc), samples)
    got = dev.simplify_tables(clone(tc), samples)
    assert_tables_equal(got, host)
    return host


@pytest.mark.parametrize('n,steps,seed', [(60, 5, 1), (2000, 20, 2), (5000, 20, 3)])
def test_model_shaped_tables(dev, n, steps, seed):
    tc, alive, rng = model_tables(n, steps, seed=seed)
    assert tc.edges.num_rows >= 1000
    samples = shuffled_samples(alive, rng)
    # some samples are parents of other samples
    assert np.isin(tc.edges.parent, samples).any()
    out = check(dev, tc, samples)
    # the three kinds of mutation: kept on a retained node, moved off a unary node, dropped
    assert 0 < out.mutations.num_rows < tc.mutations.num_rows
    assert np.isin(tc.mutations.node, samples).any()
    # individuals: some rows dropped, nodes without an individual kept as -1
    assert 0 < out.individuals.num_rows < tc.individuals.num_rows
    assert (out.nodes.individual == -1).any()


def test_a_million_edges(dev):
    tc, alive, rng = model_tables(30000, 12, seed=4, n_mut=20000)
    assert tc.edges.num_rows > 10 ** 6
    check(dev, tc, shuffled_samples(alive, rng))


def test_second_simplification(dev):
    """Simplified tables grown further and simplified again: the retained ancestors span many time levels."""
    tc, alive, rng = model_tables(3000, 15, seed=5)
    samples = shuffled_samples(alive, rng)
    tc = check(dev, tc, samples)
    alive = np.arange(len(samples), dtype=np.int64).reshape(-1, 2)         # sample k is now node k
    for rnd in range(2):
        alive = grow(tc, alive, 12, rng, t0=15 + 12 * rnd)
        add_mutations(tc, rng, 500)
        assert len(np.unique(tc.nodes.time[tc.edges.parent])) > 12
        samples = shuffled_samples(alive, rng)
        tc = check(dev, tc, samples)
        alive = np.arange(len(samples), dtype=np.int64).reshape(-1, 2)


def test_no_edges(dev):
    tc, alive, rng = model_tables(50, 0, seed=6, n_mut=100)
    assert tc.edges.num_rows == 0
    out = check(dev, tc, shuffled_samples(alive, rng)[:40])
    assert out.nodes.num_rows == 40 and out.edges.num_rows == 0


def test_no_samples_no_mutations(dev):
    tc, alive, rng = model_tables(50, 3, seed=7, n_mut=0)
    out = check(dev, tc, np.zeros(0, np.int32))
    assert out.nodes.num_rows == 0 and out.edges.num_rows == 0 and out.individuals.num_rows == 0


@pytest.mark.parametrize('sample_parent', [False, True])
def test_one_parent_with_many_pieces(dev, sample_parent):
    """One parent of 12 000 sample children in one level, over overlapping intervals: more pieces in one
    parent than a warp or a CTA could hold."""
    m, L = 12000, 20000
    rng = np.random.default_rng(8)
    tc = TableColumns(L, 0)
    tc.sites.append_columns(position=np.arange(L, dtype=np.float64) + 0.25, nonneutral=np.zeros(L, np.int8))
    tc.individuals.append_columns(flags=np.zeros(m + 1, np.int32), location=np.zeros((m + 1, 2)),
                                  idx=np.arange(m + 1))
    tc.nodes.append_columns(flags=np.ones(m + 1, np.int32), time=np.r_[np.zeros(m), 5.0],
                            population=np.zeros(m + 1, np.int32), individual=np.arange(m + 1, dtype=np.int32))
    i = np.arange(m)
    tc.edges.append_columns(left=i.astype(np.float64), right=(i + 1 + i % 4).astype(np.float64),
                            parent=np.full(m, m, np.int32), child=i.astype(np.int32))
    add_mutations(tc, rng, 3000)
    samples = rng.permutation(np.r_[i, m] if sample_parent else i)
    out = check(dev, tc, samples)
    assert out.edges.num_rows >= m // 2


def test_refuses_a_parent_not_older_than_its_child(dev):
    from geonomics_b200._lib import GnxError
    tc, alive, rng = model_tables(100, 4, seed=9)
    e = tc.edges.num_rows // 2
    tc.nodes.time[tc.edges.parent[e]] = tc.nodes.time[tc.edges.child[e]]
    with pytest.raises(GnxError) as ei:
        dev.simplify_tables(clone(tc), shuffled_samples(alive, rng))
    assert ei.value.code == -2 and 'older' in str(ei.value)


def test_refuses_a_repeated_sample(dev):
    from geonomics_b200._lib import GnxError
    tc, alive, rng = model_tables(100, 4, seed=10)
    s = shuffled_samples(alive, rng)
    s[-1] = s[0]
    with pytest.raises(GnxError) as ei:
        dev.simplify_tables(clone(tc), s)
    assert ei.value.code == -2
    # and the context still works
    check(dev, tc, shuffled_samples(alive, rng))


def _walk_recording(monkeypatch, host):
    """A use_tskit model with deleterious and trait mutation walked through four simplifications: the tables
    and the device node ids after every step.  On the device path the genotype rows of everyone alive must
    still decode from the tables at the end."""
    from geonomics_b200 import api, tables
    from test_model_gpu import _haplotypes_from_tables
    if host:
        monkeypatch.setattr(tables.TableColumns, 'sort_and_simplify',
                            lambda self, samples, dev=None: simplify_columns(self, samples))
    p = copy.deepcopy(api.read_parameters_file(PARAMS))
    g = p['comm']['species']['spp_0']['gen_arch']
    g.update(use_tskit=True, tskit_simp_interval=5, L=200, r_distr_alpha=None, mu_neut=5e-6, mu_delet=8e-6,
             start_neut_zero=True)
    g['traits']['trait_0'].update(mu=8e-6, n_loci=6)
    p['model']['T'] = 30
    mod = api.make_model(p)
    mod.walk(10000, 'burn')
    spp = mod.comm[0]
    nn0 = np.array(spp.gen_arch.nonneut_loci, dtype=np.int64)
    rec = []
    for _ in range(21):
        mod.walk(1, 'main')
        rec.append((clone(spp._tc), spp._node_ids().copy(), spp._tc_sorted_and_simplified))
    if not host:
        nodes = spp._node_ids()
        H = _haplotypes_from_tables(spp._tc, nn0)
        g_now = mod.get_genotypes()
        rows_of_start = np.searchsorted(np.array(spp.gen_arch.nonneut_loci, dtype=np.int64), nn0)
        for h in (0, 1):
            assert np.array_equal(g_now[:, rows_of_start, h], H[nodes[:, h]])
    monkeypatch.undo()
    return rec


def test_model_walk_matches_the_host_simplification(monkeypatch):
    dev_rec = _walk_recording(monkeypatch, host=False)
    host_rec = _walk_recording(monkeypatch, host=True)
    assert sum(r[2] for r in dev_rec) >= 3
    for (ta, na, sa), (tb, nb, sb) in zip(dev_rec, host_rec):
        assert sa == sb
        assert np.array_equal(na, nb)
        assert_tables_equal(ta, tb)
