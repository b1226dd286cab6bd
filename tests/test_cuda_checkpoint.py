"""Model.save / load_model: a model saved at step k, closed, and resumed (with numpy's global stream disturbed in
between) ends exactly where the same model run without the interruption ends -- the step series, the population
bit for bit (ids, positions, ages, sexes, packed genomes, z, fitness), the mutation log, the VCF bytes and, with
use_tskit, the tables after a simplification past the resume point -- on one context and across strip
decompositions."""
import copy
import os
import random
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from geonomics_b200 import api  # noqa: E402
from geonomics_b200._lib import GnxError  # noqa: E402

pytestmark = pytest.mark.gpu

PARAMS = os.path.join(HERE, 'data', 'params_small.py')
BURN = ('burn', 10000)


def _params(**edit):
    p = copy.deepcopy(api.read_parameters_file(PARAMS))
    spp = p.comm.species.spp_0
    g = spp.gen_arch
    if edit.get('mutation'):
        g.mu_neut, g.mu_delet, g.delet_alpha_distr_scale = 5e-5, 2e-5, 0.02
    if edit.get('tskit'):
        # about 8 non-neutral mutations a step: the 128 starting columns widen near t = 7 and again near t = 23
        g.update(use_tskit=True, tskit_simp_interval=10, L=4000, r_distr_alpha=None, mu_neut=2e-6, mu_delet=4e-6,
                 delet_alpha_distr_scale=0.01, start_neut_zero=True)
        g.traits.trait_0.update(mu=4e-6, n_loci=6)
    if edit.get('changes'):
        spp['change'] = {'dem': {0: dict(kind='custom', timesteps=[3, 9], sizes=[0.6, 1.0])},
                         'life_hist': {'b': {'timesteps': [6], 'vals': [0.3]}}}
    if edit.get('surfaces'):
        mv = spp.movement
        mv['move_surf'] = dict(layer='lyr_1', mixture=True, vm_distr_kappa=12, approx_len=64)
        mv['disp_surf'] = dict(layer='lyr_2', mixture=False, vm_distr_kappa=30, approx_len=64)
    if edit.get('grow'):
        spp.mating.n_births_distr_lambda = 4
        spp['change'] = {'dem': {0: dict(kind='monotonic', start_t=1, end_t=11, rate=1.2)}}
    p.model.T = edit.get('T', 12)
    p.model.its.n_its = edit.get('n_its', 1)
    return p


def _do(model, plan):
    for step in plan:
        if callable(step):
            step(model)
        else:
            model.walk(step[1], step[0])


def _close(model):
    for spp in model.comm.values():
        spp._detach()


def _collect(model, path):
    spp = model.comm[0]
    st = spp._dev.download(genomes=bool(spp.burned and spp.gen_arch is not None), unpack=False)
    out = dict(t=model.t, burn_t=model.burn_t, Nt=list(spp.Nt), n_births=list(spp.n_births),
               n_deaths=list(spp.n_deaths), mutations=repr(spp.mutations), K=spp.K.tobytes(),
               burn_stats=None if spp._burnin_spat_tester is None else repr(spp._burnin_spat_tester.stats),
               iterations=repr({it: {n: {k: v.tolist() for k, v in d.items()} for n, d in v.items()}
                                for it, v in model.iterations.items()}))
    for k in ('idx', 'x', 'y', 'age', 'sex', 'genomes', 'z', 'fit'):
        v = st.get(k)
        out[k] = None if v is None else (v.shape, v.tobytes())
    if spp.burned:
        model.write_gendata(path)
        with open(path, 'rb') as f:
            out['vcf'] = f.read()
    if spp.__dict__.get('_tc') is not None:
        out['tables'] = repr({name: {k: v.tolist() for k, v in getattr(spp._tc, name).asdict().items()}
                              for name in ('nodes', 'edges', 'individuals', 'sites', 'mutations')})
    return out


def _resume_equals_uninterrupted(p, before, after, tmp_path, save_strips=None, load_strips=None, at_save=None,
                                 after_load=None):
    ref = api.make_model(copy.deepcopy(p))
    try:
        _do(ref, before)
        _do(ref, after)
        want = _collect(ref, str(tmp_path / 'ref.vcf'))
    finally:
        _close(ref)
    model = api.make_model(copy.deepcopy(p), strips=save_strips)
    ck = str(tmp_path / 'model.ckpt')
    try:
        _do(model, before)
        saved = at_save(model) if at_save else None
        model.save(ck)
    finally:
        _close(model)
    np.random.seed(12345)                       # the resumed run must not depend on the stream at load time
    np.random.rand(17)
    random.random()
    got_model = api.load_model(ck, strips=load_strips)
    try:
        if after_load:
            after_load(got_model, saved)
        _do(got_model, after)
        got = _collect(got_model, str(tmp_path / 'got.vcf'))
    finally:
        _close(got_model)
    assert want['Nt'] and want['Nt'][-1] > 0
    for k in want:
        assert got.get(k) == want[k], k
    return want


def test_neutral_and_deleterious_mutation(tmp_path):
    want = _resume_equals_uninterrupted(_params(mutation=True), [BURN, ('main', 5)], [('main', 7)], tmp_path)
    assert "'neut'" in want['mutations'] and "'delet'" in want['mutations']


def test_use_tskit_trait_mutation_widening_on_both_sides(tmp_path):
    p = _params(tskit=True, T=40)

    def at_save(model):
        spp = model.comm[0]
        assert spp._dev.col_capacity > 128                        # widened before the save (and again after it)
        return dict(cols=spp._dev.col_capacity, col_locus=spp._dev.read_cols(), paths=spp._dev.read_paths(),
                    subsetters=spp._dev.subsetters())

    def after_load(model, saved):
        spp = model.comm[0]
        assert spp._dev.col_capacity == saved['cols']
        assert np.array_equal(spp._dev.read_cols(), saved['col_locus'])
        assert np.array_equal(spp._dev.read_paths(), saved['paths'])
        # a column a mutation added (every column after the 6 starting trait loci) reads the path in front of its
        # locus, which the paths as simulated, read at the locus, do not always give: the reason the checkpoint
        # carries the paths the device reads
        paths = spp.gen_arch.recombinations._paths
        nn = np.sort(saved['col_locus'])
        added = saved['col_locus'][6:]
        assert len(added)
        pos = np.searchsorted(nn, added)
        assert np.array_equal(saved['subsetters'][:, pos], paths[:, added - 1])
        assert not np.array_equal(paths[:, added - 1], paths[:, added])

    model = {}

    def keep(m):
        model['cols'] = m.comm[0]._dev.col_capacity

    want = _resume_equals_uninterrupted(p, [BURN, ('main', 15)], [('main', 25), keep], tmp_path, at_save=at_save,
                                        after_load=after_load)
    assert "'t0'" in want['mutations'] and 'tables' in want and model['cols'] > 256


def test_landscape_and_demographic_changes_across_the_save(tmp_path):
    _resume_equals_uninterrupted(_params(changes=True), [BURN, ('main', 5)], [('main', 7)], tmp_path)


def test_table_mode_conductance_surfaces(tmp_path):
    # lyr_1 changes at t = 4, 6, 8: its move surface is re-drawn from numpy's stream after the resume
    _resume_equals_uninterrupted(_params(surfaces=True), [BURN, ('main', 5)], [('main', 7)], tmp_path)


def test_saved_mid_burn_in(tmp_path):
    want = _resume_equals_uninterrupted(_params(), [('burn', 3)], [BURN, ('main', 4)], tmp_path)
    assert want['burn_t'] >= 9 and want['burn_stats']


def test_species_that_grew_before_the_save(tmp_path):
    def at_save(model):
        assert model.comm[0]._dev.capacity > 4096

    def after_load(model, saved):
        assert model.comm[0]._dev.capacity > 4096

    _resume_equals_uninterrupted(_params(grow=True, T=30), [BURN, ('main', 20)], [('main', 10)], tmp_path,
                                 at_save=at_save, after_load=after_load)


def _iteration_0_to(k):
    def go(m):                                 # Model._do_next_iteration for iteration 0, up to main step k
        m.it = m.its.pop()
        m._reset()
        m.walk(10 ** 9, 'burn')
        m.orig_comm = {n: spp._snapshot() for n, spp in m.comm.items()}
        m.walk(k, 'main')
    return go


def _finish_and_run(k):
    def go(m):
        m.walk(m.T - k, 'main')
        spp = m.comm[0]
        m.iterations[0] = {0: dict(Nt=np.array(spp.Nt[-m.T:]), n_births=np.array(spp.n_births[-m.T:]),
                                   n_deaths=np.array(spp.n_deaths[-m.T:]))}
        m.run()                                # the remaining iteration, from orig_comm / orig_land
    return go


def test_two_iterations_saved_in_iteration_0(tmp_path):
    want = _resume_equals_uninterrupted(_params(n_its=2), [_iteration_0_to(5)], [_finish_and_run(5)], tmp_path)
    assert '1:' in want['iterations']


@pytest.mark.parametrize('save_strips,load_strips', [(2, None), (2, 3), (None, 2)])
def test_strips(save_strips, load_strips, tmp_path):
    _resume_equals_uninterrupted(_params(mutation=True), [BURN, ('main', 5)], [('main', 7)], tmp_path,
                                 save_strips=save_strips, load_strips=load_strips)


def test_set_clock_continues_the_draws_without_a_new_graph():
    """Two contexts from the same start: one steps 5 times; the other steps twice (its graph is captured), takes
    the first one's population and clock, and from there both make the same draws, on the captured graph."""
    p = _params()
    a, b = api.make_model(copy.deepcopy(p)), api.make_model(copy.deepcopy(p))
    try:
        da, db = a.comm[0]._dev, b.comm[0]._dev
        da.step(1)
        da.step(4)
        db.step(1)
        db.step(1)
        with pytest.raises(GnxError, match='pending'):
            db.set_clock(5)                       # the last step's deaths are only flagged
        st = da.download(genomes=False)
        t, t0 = da.clock()
        assert t == 5
        captures = db.graph_capture_count
        db.upload(st['x'], st['y'], st['age'], st['sex'], st['idx'], z=st.get('z'), fit=st['fit'],
                  max_ind_idx=st['max_ind_idx'])
        db.set_clock(t, t0)
        assert db.clock() == (t, t0)
        da.step(3)
        db.step(3)
        ra, rb = da.download(genomes=False), db.download(genomes=False)
        for k in ('idx', 'x', 'y', 'age', 'sex', 'fit'):
            assert ra[k].tobytes() == rb[k].tobytes(), k
        assert db.graph_capture_count == captures
        assert da.clock() == db.clock() == (8, t0)
    finally:
        _close(a)
        _close(b)
