"""The column genotype layout of a use_tskit species (gnx_create_cols) against the by-locus tskit layout it
replaces: the same workload, seed and starting genomes on both, compared after every step.  Integer state is
compared bit for bit; z and fitness to the last bits, because a trait's entries are summed in the order of the
bits they read, and a column added by a trait mutation comes after every older column whatever its locus."""
import numpy as np
import pytest

from parity_util import device_params, synthetic_case

pytestmark = pytest.mark.gpu


def _make(arch, prm, cols, capacity, seed):
    from geonomics_b200.device import DeviceSpecies
    rasters = np.concatenate([np.array(arch['rasters'], dtype=np.float64), arch['K'][None]], axis=0)
    p = device_params(arch, prm)
    p['K_layer'] = rasters.shape[0] - 1
    ga = dict(L=arch['paths'].shape[1], paths=arch['paths'], traits=arch['traits'], dom=arch['dom'])
    if cols is not None:
        ga['cols'] = cols
    return DeviceSpecies(arch['land_dim'], rasters, p, ga, capacity=capacity, seed=seed, disp_tries_injected=24)


def _pair(n_traits=2, dom=False, mono=False, n_delet0=0, mu=(2e-5, 1e-5, 1e-5), seed=3, n=1500, L=1000):
    """(by-locus device, column device, case) on one synthetic workload with mutation and tskit rows on."""
    from geonomics_b200 import genome_pack as gp
    arch, prm, state, draws = synthetic_case(L=L, n=n, n_traits=n_traits, loci_per_trait=10, seed=seed, max_tries=24)
    if mono:                                                   # trait 0 starts monogenic
        arch['traits'][0] = dict(arch['traits'][0], loci=arch['traits'][0]['loci'][:1],
                                 alpha=arch['traits'][0]['alpha'][:1])
    trait_loci = np.unique(np.concatenate([np.asarray(t['loci']) for t in arch['traits']]))
    rng = np.random.default_rng(seed)
    delet = np.sort(rng.choice(np.setdiff1d(np.arange(L), trait_loci), n_delet0, replace=False))
    nonneut = np.union1d(trait_loci, delet)
    if dom:
        arch['dom'] = np.zeros(L, np.int8)
        arch['dom'][trait_loci[::2]] = 1
    rows = state['g'][:, nonneut, :]
    mutables = [int(v) for v in rng.permutation(np.setdiff1d(np.arange(L), nonneut))]
    devs = []
    for cols in (None, nonneut):
        d = _make(arch, prm, cols, capacity=6 * n, seed=seed + 11)
        d.upload(state['x'], state['y'], state['age'], state['sex'], state['idx'],
                 g=rows if cols is not None else gp.rows_to_loci(rows, nonneut, L), max_ind_idx=state['max_ind_idx'])
        d.set_mutation(mu[0], mu[1], mutables, nonneut, delet, np.full(len(delet), 0.002), tskit_layout=True,
                       trait_mus=[mu[2]] * n_traits, trait_alpha_distr=[(0.0, 0.1, None)] * n_traits)
        d.tskit_enable(edge_capacity=1 << 22, birth_capacity=1 << 18)
        d.tskit_set_nodes(2 * np.arange(n, dtype=np.int32), 2 * np.arange(n, dtype=np.int32) + 1, 2 * n, n)
        devs.append(d)
    return devs[0], devs[1], dict(arch=arch, prm=prm, state=state, draws=draws, nonneut=nonneut, L=L)


def _compare(a, b, L):
    da, db = a.download(e=False), b.download(e=False)
    for k in ('idx', 'x', 'y', 'age', 'sex'):
        assert np.array_equal(da[k], db[k]), k
    np.testing.assert_allclose(db['z'], da['z'], rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(db['fit'], da['fit'], rtol=1e-13, atol=1e-15)
    loci = np.sort(db['col_locus'])
    assert len(np.unique(loci)) == len(loci)
    assert np.array_equal(da['g'][:, loci, :], db['g'])
    assert not np.delete(da['g'], loci, axis=1).any()          # by-locus neutral bits stay zero
    assert a.step_records() == b.step_records()
    (la, sa), (lb, sb) = a.read_mutations(), b.read_mutations()
    assert la == lb
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert np.array_equal(sb['nonneut_loci'], loci)            # the columns are the non-neutral loci
    (ta, ia), (tb, ib) = a.read_mutation_tables(), b.read_mutation_tables()
    assert np.array_equal(ia, ib)
    for x, y in zip(ta, tb):
        for k in x:
            assert np.array_equal(x[k], y[k]), k
    ra, rb = a.tskit_drain(), b.tskit_drain()
    for k in ra:
        if k == 'z':
            np.testing.assert_allclose(rb[k], ra[k], rtol=1e-13, atol=1e-15)
        else:
            assert np.array_equal(ra[k], rb[k]), k
    ca, cb = a.stat_counts(), b.stat_counts()
    assert np.array_equal(ca[0], cb[0]) and np.array_equal(ca[1], cb[1]) and ca[3] == cb[3]
    assert cb[2] == pytest.approx(ca[2], rel=1e-12)
    na, nb = a.ld_counts(), b.ld_counts()
    assert np.array_equal(na[0], nb[0]) and na[1] == nb[1]
    return la


@pytest.mark.parametrize('kind', ['mono', 'dom', 'traits3'])
def test_columns_match_by_locus_step_by_step(kind):
    """Neutral, deleterious and trait mutation (trait 0 turning polygenic in 'mono'), dominance on and off,
    2 and 3 traits; free-running draws, one graph-launched step per call."""
    a, b, case = _pair(n_traits=3 if kind == 'traits3' else 2, dom=kind == 'dom', mono=kind == 'mono')
    try:
        assert b.W == 4 and a.W == 4 * 8                        # 128 columns; 1000 loci by locus
        log = []
        for _ in range(8):
            a.step(1)
            b.step(1)
            log += _compare(a, b, case['L'])
        types = {r['type'] for r in log}
        assert {'neut', 'delet', 't0', 't1'} <= types, types
        if kind == 'mono':
            assert len(b.read_mutation_tables()[0][0]['loci']) > 1
    finally:
        a.close()
        b.close()


def test_columns_match_by_locus_multistep_calls():
    """Several steps per gnx_step call: one captured graph re-launched."""
    a, b, case = _pair(seed=5)
    try:
        for k in (1, 3, 4):
            a.step(k)
            b.step(k)
            _compare(a, b, case['L'])
        widenings = int(np.log2(b.col_capacity // 128))
        assert a.graph_capture_count == 1 and b.graph_capture_count == 1 + widenings
        assert b.graph_launch_count == a.graph_launch_count
    finally:
        a.close()
        b.close()


def test_columns_match_by_locus_with_injected_draws():
    a, b, case = _pair(seed=7)
    try:
        d = dict(case['draws'])
        d.pop('move_choice', None)
        d.pop('disp_choice', None)
        rng = np.random.default_rng(9)
        nm = 12
        d.update(mut_n=np.array([nm], np.int32), mut_type_u=rng.random(nm),
                 mut_ind_R=rng.integers(0, 2**32, nm, dtype=np.uint64).astype(np.uint32),
                 mut_homol_u=rng.random(nm), mut_s=rng.gamma(0.2, 0.2, nm), mut_alpha=rng.normal(0, 0.15, nm))
        for dev in (a, b):
            dev.set_draws(d)
            dev.step(1)
        log = _compare(a, b, case['L'])
        assert len(log) == nm and any(r['type'] != 'neut' for r in log)
    finally:
        a.close()
        b.close()


def _delet_per_step(devs, n_mut):
    """Inject n_mut deleterious mutations into every step (same mutation draws each step; everything else
    stays on Philox): a known number of new columns per step, under the GNX_MUT_MAX_NEW limit."""
    d = dict(mut_n=np.array([n_mut], np.int32), mut_type_u=np.full(n_mut, 0.9),
             mut_ind_R=np.arange(n_mut, dtype=np.uint32) * np.uint32(2**32 // n_mut),
             mut_homol_u=np.linspace(0.0, 1.0, n_mut, endpoint=False), mut_s=np.full(n_mut, 1e-3))
    for dev in devs:
        dev.set_draws(d)


def test_columns_widen_between_steps():
    """120 starting non-neutral loci: 256 columns, which 20 deleterious mutations a step fill; the host widens
    the rows between steps (doubling), and every widening costs exactly one more graph capture."""
    a, b, case = _pair(n_delet0=100, mu=(1e-5, 4e-4, 0.0), seed=11)
    try:
        assert len(case['nonneut']) == 120 and b.col_capacity == 256 and b.W == 8
        _delet_per_step((a, b), 20)
        caps = [b.col_capacity]
        for _ in range(12):
            a.step(1)
            b.step(1)
            _compare(a, b, case['L'])
            if b.col_capacity != caps[-1]:
                caps.append(b.col_capacity)
        assert caps == [256, 512], caps
        assert len(b.read_cols()) > 256 and b.W == 16
        assert b.graph_capture_count == a.graph_capture_count + 1
    finally:
        a.close()
        b.close()


def test_no_free_column_is_a_capacity_error():
    """Without the host's widening a non-neutral mutation that finds no free column fails the step
    (GNX_ERR_CAPACITY); it is never dropped."""
    from geonomics_b200._lib import GnxError
    a, b, case = _pair(n_delet0=100, mu=(0.0, 2e-4, 0.0), seed=13)
    try:
        b._col_budget = None                                   # the bare C-ABI: no widening
        _delet_per_step((b,), 20)
        used = len(b.read_cols())
        with pytest.raises(GnxError) as ei:
            for _ in range(12):
                b.step(1)
                b.sync()
                used = len(b.read_cols())
        assert ei.value.code == -3
        assert used <= 256 < used + 20                         # the step that failed had no room for its columns
    finally:
        a.close()
        b.close()
