"""A Model cut into strips (make_model(strips=...)) against the same Model undecomposed with the same seed:
the burn-in (its length and the spatial tester's series), the step series, the getters, the device
statistics, the writers, mutation bookkeeping, species changes and iterations are all equal."""
import copy
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from geonomics_b200 import api  # noqa: E402

pytestmark = pytest.mark.gpu

PARAMS = os.path.join(HERE, 'data', 'params_small.py')


def _params(mutation=False, poisson=False, n_its=1):
    p = api.read_parameters_file(PARAMS)
    spp = p.comm.species.spp_0
    if mutation:
        spp.gen_arch.mu_neut, spp.gen_arch.mu_delet = 5e-5, 2e-5
        spp.gen_arch.delet_alpha_distr_scale = 0.02
    if poisson:
        spp.mating.n_births_fixed = False
        spp.mating.n_births_distr_lambda = 2.5
        spp['change'] = {'life_hist': {'b': {'timesteps': [3], 'vals': [0.15]}},
                         'dem': {0: {'kind': 'custom', 'timesteps': [5, 7], 'sizes': [0.8, 1.0]}}}
    p.model.its.n_its = n_its
    return p


def _run(strips, genome_init='host', tmp=None, **kw):
    """Burn in, assign the genomes, walk the main phase; everything a user can read off the model."""
    model = api.make_model(_params(**kw), strips=strips, genome_init=genome_init)
    try:
        spp = model.comm[0]
        model.walk(10000, 'burn')
        out = dict(burn_t=model.burn_t, burn_stats=copy.deepcopy(spp._burnin_spat_tester.stats))
        model.walk(12, 'main')
        out.update(Nt=list(spp.Nt), n_births=list(spp.n_births), n_deaths=list(spp.n_deaths))
        for g in ('x', 'y', 'age', 'z', 'e', 'fitness', 'genotypes'):
            out[g] = getattr(model, 'get_' + g)()
        out.update(het=spp._calc_het(), maf=spp._calc_maf(), freqs=spp._calc_allele_freqs(), ld=spp._calc_ld(),
                   density=spp._calc_density(), mean_fit=spp._calc_mean_fitness(), n=len(spp))
        ga = spp.gen_arch
        out.update(mutations=list(spp.mutations), nonneut=np.array(ga.nonneut_loci), delet=np.array(ga.delet_loci),
                   delet_s=np.array(ga.delet_loci_s), mutables=list(ga._mutables or []))
        if tmp is not None:
            files = {}
            for ext in ('vcf', 'fasta'):
                f = os.path.join(tmp, '%s_%s.%s' % (strips, genome_init, ext))
                model.write_gendata(f)
                files[ext] = open(f, 'rb').read()
            f = os.path.join(tmp, '%s_%s.csv' % (strips, genome_init))
            model.write_geodata(f)
            files['csv'] = open(f, 'rb').read()
            out['files'] = files
        return out
    finally:
        for s in model.comm.values():
            s._detach()


def _equal(ref, got):
    assert got['burn_t'] == ref['burn_t']
    for k in ('mean', 'std'):
        assert got['burn_stats'][k] == ref['burn_stats'][k], k
    for k in ('Nt', 'n_births', 'n_deaths', 'mutations', 'mutables', 'n'):
        assert got[k] == ref[k], k
    for k in ('x', 'y', 'age', 'z', 'e', 'fitness', 'genotypes', 'het', 'maf', 'freqs', 'ld', 'density',
              'nonneut', 'delet', 'delet_s'):
        assert np.array_equal(got[k], ref[k], equal_nan=k == 'ld'), k
    assert got['mean_fit'] == pytest.approx(ref['mean_fit'], rel=1e-12)
    assert got.get('files') == ref.get('files')


_REF = {}


def _ref(key, **kw):
    if key not in _REF:
        _REF[key] = _run(None, **kw)
    return _REF[key]


@pytest.mark.parametrize('genome_init', ['host', 'device'])
@pytest.mark.parametrize('k', [2, 3])
def test_strip_model_equals_the_undecomposed_model(k, genome_init, tmp_path):
    ref = _ref(('base', genome_init), genome_init=genome_init, tmp=str(tmp_path))
    got = _run(k, genome_init=genome_init, tmp=str(tmp_path))
    assert len(ref['burn_stats']['mean']) > 1 and ref['n'] > 0
    _equal(ref, got)


@pytest.mark.parametrize('k', [2, 3])
def test_strip_model_with_mutation(k):
    ref = _ref('mutation', mutation=True)
    got = _run(k, mutation=True)
    assert len(ref['mutations']) > 0 and {m['type'] for m in ref['mutations']} == {'neut', 'delet'}
    _equal(ref, got)


@pytest.mark.parametrize('k', [2, 3])
def test_strip_model_with_poisson_births_and_species_changes(k):
    ref = _ref('poisson', poisson=True)
    got = _run(k, poisson=True)
    assert any(b > 0 for b in ref['n_births'])
    _equal(ref, got)


@pytest.mark.parametrize('k', [2, 3])
def test_strip_model_iterations(k):
    def run(strips):
        model = api.make_model(_params(n_its=2), strips=strips)
        try:
            model.run()
            return model.iterations
        finally:
            for s in model.comm.values():
                s._detach()
    ref, got = run(None), run(k)
    assert sorted(ref) == sorted(got) == [0, 1]
    for it in ref:
        for key in ('Nt', 'n_births', 'n_deaths'):
            assert np.array_equal(ref[it][0][key], got[it][0][key]), (it, key)


def test_strip_model_refuses_replicate_sharding():
    import torch.distributed as dist
    model = api.make_model(_params(), strips=2)
    try:
        with pytest.raises(ValueError, match='dist'):
            model.run(dist=dist)
    finally:
        for s in model.comm.values():
            s._detach()


def test_one_rank_process_group_equals_the_undecomposed_model(tmp_path):
    """strips=group with one nccl rank: the group code paths (gathers, the device barriers inside the step
    graph, the seed broadcast) on one GPU."""
    import torch
    import torch.distributed as dist
    ref = _ref(('base', 'host'), genome_init='host', tmp=str(tmp_path))
    torch.cuda.set_device(0)
    dist.init_process_group('nccl', init_method='file://' + str(tmp_path / 'pg'), rank=0, world_size=1,
                            device_id=torch.device('cuda', 0))
    try:
        got = _run(dist.group.WORLD, genome_init='host', tmp=str(tmp_path))
    finally:
        dist.destroy_process_group()
    _equal(ref, got)
