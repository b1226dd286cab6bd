"""A use_tskit species at a genome length the by-locus rows cannot carry in practice: 200 000 loci of which 20
are non-neutral, through make_model and Model.walk with mutation on and simplifications in between.  The device
keeps one column per non-neutral locus (gnx_create_cols)."""
import copy
import ctypes as C
import os

import numpy as np
import pytest

from test_model_gpu import PARAMS, _haplotypes_from_tables

pytestmark = pytest.mark.gpu

L = 200000


@pytest.mark.parametrize('genome_init', ['host', 'device'])
def test_long_genome_use_tskit_model(genome_init, tmp_path):
    from geonomics_b200 import api, writers, _lib
    p = copy.deepcopy(api.read_parameters_file(PARAMS))
    s = p['comm']['species']['spp_0']
    s['init'].update(N=5000, K_factor=3.0)
    g = s['gen_arch']
    g.update(use_tskit=True, tskit_simp_interval=5, L=L, r_distr_alpha=None, mu_neut=4e-8, mu_delet=4e-8,
             start_neut_zero=True, n_recomb_sims=300)
    g['traits']['trait_0'].update(mu=2e-8, n_loci=20)
    p['model']['T'] = 20
    np.random.seed(17)
    mod = api.make_model(p, genome_init=genome_init)
    mod.walk(10000, 'burn')
    spp = mod.comm[0]
    dev = spp._dev
    nn0 = np.array(spp.gen_arch.nonneut_loci, dtype=np.int64)
    assert dev.cols and len(nn0) == 20 and dev.col_capacity == 128
    mod.walk(13, 'main')                                      # simplified after t = 4, 9
    assert len(spp.mutations) > 0 and spp._tc.mutations.num_rows > 0
    n = len(spp)
    assert n > 100
    # the genotype buffer: 16 bytes per 128 columns and homologue, not per 128 loci
    ptr, nbytes = C.c_void_p(), C.c_int64()
    _lib.check(dev._L.gnx_device_ptr(dev._ctx, _lib.FIELDS['GENOMES'], C.byref(ptr), C.byref(nbytes)), 'gnx_device_ptr')
    assert nbytes.value == n * 2 * 16 * (dev.col_capacity // 128)
    nn = np.array(spp.gen_arch.nonneut_loci, dtype=np.int64)
    assert np.array_equal(np.sort(dev.read_cols()), nn) and dev.col_capacity < 1024
    # the rows of everyone alive at the starting non-neutral loci decode from the tables
    rows = mod.get_genotypes()
    assert rows.shape == (n, len(nn), 2)
    H = _haplotypes_from_tables(spp._tc, nn0)
    nodes = spp._node_ids()
    start = np.searchsorted(nn, nn0)
    for h in (0, 1):
        assert np.array_equal(rows[:, start, h], H[nodes[:, h]])
    # the VCF is what the by-locus layout writes: the rows scattered into an [n, L, 2] zero array
    path = os.path.join(str(tmp_path), 'out.vcf')
    np.random.seed(5)
    mod.write_gendata(path, n=200, include_fixed_sites=False)
    np.random.seed(5)
    ids = writers.adhoc_sample_ids([*spp], 200)
    full = np.zeros((len(ids), L, 2), np.int8)
    full[:, nn, :] = spp._get_genotypes(individs=ids)
    with open(path) as f:
        got = f.read().split('\n')
    want = writers.format_vcf(ids, full, L, include_fixed_sites=False).split('\n')
    assert got[0] == want[0] and got[2:] == want[2:]           # line 1 is the date
    assert len(got) > 5
