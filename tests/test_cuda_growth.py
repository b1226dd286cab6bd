"""A population that outgrows the capacity it started with (gnx_set_growth_guard, gnx_reserve,
gnx_tskit_reserve): with the guard on, a step that could overflow a buffer does not start, the host grows
the buffers and launches it again.  Every case is compared, bit for bit, against the same seed run with
buffers large enough never to stop."""
import copy
import os
import runpy

import numpy as np
import pytest

from parity_util import device_params, synthetic_case

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _workload(lam, fixed, n=2000):
    from geonomics_b200 import workloads
    w = workloads.build(workloads.scaled(workloads.CONFIGS['c2'], n), seed=5)
    w['prm'] = dict(w['prm'], lam=lam, n_births_fixed=fixed)
    return w


def _device(w, capacity, grow):
    from geonomics_b200.device import DeviceSpecies
    from geonomics_b200 import workloads
    d = DeviceSpecies(w['land_dim'], w['rasters'], w['prm'], w['gen_arch'], capacity=capacity, seed=11, grow=grow)
    p = w['pop']
    d.upload(p['x'], p['y'], p['age'], p['sex'], p['idx'],
             genomes_packed=workloads.random_packed_genomes(len(p['x']), w['L'], 12))
    return d


def _same_state(a, b):
    da, db = a.download(e=True), b.download(e=True)
    assert set(da) == set(db)
    for k in da:
        assert np.array_equal(np.asarray(da[k]), np.asarray(db[k])), k


def _grow_and_compare(lam, fixed):
    w = _workload(lam, fixed)
    K = w['rasters'][0] * w['prm']['K_factor']
    ref, dev = _device(w, 1 << 17, False), _device(w, 4096, True)
    try:
        caps = []
        reserve = dev.reserve
        dev.reserve = lambda c: (caps.append(int(c)), reserve(c))
        for d in (ref, dev):
            d.step(3)
            d.set_K(5 * K)
            d.step(40)
        assert dev.step_records() == ref.step_records()
        _same_state(ref, dev)
        st = dev.step_status()
        assert st['steps_run'] > 0 and not st['stopped'] and st['capacity'] == dev.capacity
        assert len(caps) >= 2 and dev.capacity >= 4 * 4096
        assert dev.graph_capture_count > ref.graph_capture_count      # every growth captures the step again
        assert ref.counters()['t'] == dev.counters()['t'] == 43
    finally:
        ref.close()
        dev.close()


def test_fixed_births_grow_bit_identically():
    _grow_and_compare(2, True)


def test_poisson_births_grow_bit_identically():
    _grow_and_compare(3, False)


def test_guard_need_matches_the_bound():
    """The needs the guard reports are n + device.max_births(n) at the population the step starts from."""
    from geonomics_b200.device import max_births
    w = _workload(3, False)
    dev = _device(w, 4096, True)
    try:
        for _ in range(3):                          # the first step is checked on the host, later ones on the device
            n0 = dev.counters()['n']
            assert dev.step(1) is None
            st = dev.step_status()
            assert st['steps_run'] == 1 and not st['stopped']
            assert st['need_entries'] == n0 + max_births(3, False, n0) <= dev.capacity == st['capacity']
        cap = dev.capacity
        dev.reserve(cap // 2)                       # never shrinks
        assert dev.capacity == cap
    finally:
        dev.close()


def _tskit_pair(edge_capacity, birth_capacity, grow_capacity):
    """A use_tskit column-layout species with mutation and tskit rows, small or large buffers."""
    from geonomics_b200.device import DeviceSpecies
    L, n, seed = 1000, 1500, 3
    arch, prm, state, _ = synthetic_case(L=L, n=n, n_traits=1, loci_per_trait=10, seed=seed, max_tries=24)
    trait_loci = np.unique(np.asarray(arch['traits'][0]['loci']))
    rng = np.random.default_rng(seed)
    delet = np.sort(rng.choice(np.setdiff1d(np.arange(L), trait_loci), 4, replace=False))
    nonneut = np.union1d(trait_loci, delet)
    mutables = [int(v) for v in rng.permutation(np.setdiff1d(np.arange(L), nonneut))]
    rasters = np.concatenate([np.array(arch['rasters'], dtype=np.float64), arch['K'][None]], axis=0)
    p = device_params(arch, prm)
    p['K_layer'] = rasters.shape[0] - 1
    p['lam'], p['n_births_fixed'] = 2.0, True
    ga = dict(L=L, paths=arch['paths'], traits=arch['traits'], dom=arch['dom'], cols=nonneut)
    devs = []
    for cap, ecap, bcap, grow in ((1 << 16, 1 << 24, 1 << 18, False),
                                  (grow_capacity, edge_capacity, birth_capacity, True)):
        d = DeviceSpecies(arch['land_dim'], rasters, p, ga, capacity=cap, seed=seed + 11, disp_tries_injected=24,
                          grow=grow)
        d.upload(state['x'], state['y'], state['age'], state['sex'], state['idx'], g=state['g'][:, nonneut, :],
                 max_ind_idx=state['max_ind_idx'])
        # rates low enough that no step draws more than GNX_MUT_MAX_NEW non-neutral mutations
        d.set_mutation(2e-6, 1e-6, mutables, nonneut, delet, np.full(len(delet), 0.002), tskit_layout=True,
                       trait_mus=[1e-6], trait_alpha_distr=[(0.0, 0.1, None)])
        d.tskit_enable(edge_capacity=ecap, birth_capacity=bcap)
        d.tskit_set_nodes(2 * np.arange(n, dtype=np.int32), 2 * np.arange(n, dtype=np.int32) + 1, 2 * n, n)
        devs.append(d)
    return devs[0], devs[1], rasters[-1]


def _cat(chunks):
    out = {}
    for k in ('left', 'right', 'parent', 'child', 'idx', 'x', 'y', 'time', 'node_time', 'node_individual'):
        out[k] = np.concatenate([c[k] for c in chunks])
    out['z'] = np.concatenate([c['z'] for c in chunks], axis=0)
    return out


def _run_tskit(dev, n, drained, counts):
    """Species._step's loop: on a stop, drain, grow the row buffers only if one step still needs more."""
    from geonomics_b200.device import growth_capacity
    stop = dev.step(n)
    while stop is not None:
        counts['stops'] += 1
        drained.append(dev.tskit_drain())
        need_b, need_e = stop['need_births'] - len(drained[-1]['idx']), stop['need_edges'] - len(drained[-1]['left'])
        ecap, bcap = stop['edge_capacity'], stop['born_capacity']
        if need_b > bcap or need_e > ecap:
            counts['reserves'] += 1
            dev.tskit_reserve(growth_capacity(need_e, ecap) if need_e > ecap else ecap,
                              growth_capacity(need_b, bcap) if need_b > bcap else bcap)
        stop = dev.step(stop['steps_left'])


def test_tskit_rows_and_columns_grow_bit_identically():
    ref, dev, K = _tskit_pair(edge_capacity=4096, birth_capacity=512, grow_capacity=4096)
    try:
        ref.step(2)
        ref.set_K(4 * K)
        ref.step(20)
        drained, counts = [], dict(stops=0, reserves=0)
        _run_tskit(dev, 2, drained, counts)
        dev.set_K(4 * K)
        _run_tskit(dev, 20, drained, counts)
        drained.append(dev.tskit_drain())
        assert counts['stops'] >= 1 and counts['reserves'] >= 1 and dev.capacity > 4096
        assert dev.step_records() == ref.step_records()
        a, b = ref.tskit_drain(), _cat(drained)
        for k in b:
            assert np.array_equal(a[k], b[k]), k
        assert drained[0]['first_node_id'] == a['first_node_id']
        assert drained[0]['first_individual_row'] == a['first_individual_row']
        _same_state(ref, dev)
        assert np.array_equal(ref.read_cols(), dev.read_cols())
        r_mut, r_st = ref.read_mutations()
        d_mut, d_st = dev.read_mutations()
        assert r_mut == d_mut
        for k in r_st:
            assert np.array_equal(r_st[k], d_st[k]), k
    finally:
        ref.close()
        dev.close()


def _model_params(T=30):
    p = copy.deepcopy(runpy.run_path(os.path.join(HERE, 'data', 'params_small.py'))['params'])
    spp = p['comm']['species']['spp_0']
    spp['mating']['n_births_distr_lambda'] = 4
    spp['change'] = {'dem': {0: dict(kind='monotonic', start_t=1, end_t=11, rate=1.2)}}
    p['model']['T'] = T
    return p


def _walk(p):
    from geonomics_b200 import api
    mod = api.make_model(copy.deepcopy(p), name='growth')
    mod.walk(10000, 'burn')
    mod.walk(p['model']['T'], 'main')
    return mod


def test_model_outgrows_its_starting_capacity(monkeypatch):
    from geonomics_b200 import api
    from geonomics_b200._lib import GnxError
    p = _model_params()
    grown = _walk(p)
    spp = grown.comm[0]
    assert spp._dev.capacity > 4096                # started at max(4096, 3 sum(K), 2 N0) = 4096; lambda = 4 outgrows it
    attach = api.Species._attach

    def attach_large(self, capacity=None, cols=None):
        return attach(self, capacity=1 << 17, cols=cols)
    monkeypatch.setattr(api.Species, '_attach', attach_large)
    large = _walk(p)
    assert large.comm[0]._dev.capacity == 1 << 17
    assert large.comm[0].Nt == spp.Nt
    assert np.array_equal(large.get_genotypes(), grown.get_genotypes())
    assert np.array_equal(large.get_x(), grown.get_x())

    # without the guard a capacity the population outgrows is the old hard error
    def attach_tight(self, capacity=None, cols=None):
        return attach(self, capacity=1300, cols=cols)
    monkeypatch.setattr(api.Species, '_attach', attach_tight)
    device_species = api.DeviceSpecies
    monkeypatch.setattr(api, 'DeviceSpecies', lambda *a, **kw: device_species(*a, **dict(kw, grow=False)))
    with pytest.raises(GnxError) as e:
        _walk(p)
    assert e.value.code == -3


def test_guard_is_off_by_default_and_refused_on_strips():
    from geonomics_b200._lib import GnxError
    from geonomics_b200.strips import LocalStrips
    w = _workload(2, True)
    dev = _device(w, 4096, False)
    try:
        assert not dev.grow
        dev.step(3)
        dev.set_K(5 * w['rasters'][0] * w['prm']['K_factor'])
        with pytest.raises(GnxError) as e:
            dev.step(40, sync=True)
        assert e.value.code == -3
        with pytest.raises(GnxError) as e:
            dev.step_status()
        assert e.value.code == -5
    finally:
        dev.close()
    p = w['pop']
    st = LocalStrips(2, w['land_dim'], w['rasters'], w['prm'], w['gen_arch'], capacity=4 * len(p['x']), seed=3)
    try:
        d = st.ranks[0].dev
        with pytest.raises(GnxError) as e:
            d.reserve(8 * len(p['x']))
        assert e.value.code == -5
        assert d._L.gnx_set_growth_guard(d._ctx, 1) == -5
    finally:
        st.close()
