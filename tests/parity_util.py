"""Shared helpers for the GPU parity tests: drive libgnxb200.so stage by stage on a golden
case and compare with the oracle / the reference-recorded vectors."""
import numpy as np


def device_params(arch, prm, case_cfg=None):
    """Translate the golden-case parameter dicts into DeviceSpecies arguments."""
    p = dict(b=prm['b'], R=prm['R'], lam=prm['lam'], n_births_fixed=prm['n_births_fixed'],
             mating_radius=prm['mating_radius'], d_min=prm['d_min'], d_max=prm['d_max'],
             sex=prm['sex'], sex_ratio_p=prm['sex_ratio_p'], max_age=prm['max_age'],
             K_layer=0, K_factor=1.0, move=True,
             direction_mu=prm.get('direction_mu', 0.0), direction_kappa=prm.get('direction_kappa', 0.0),
             density_grid_window_width=arch['ww'],
             choose_nearest=prm.get('choose_nearest', False), inverse_dist=prm.get('inverse_dist', False))
    if arch.get('move_surf') is not None:
        p['move_surf'] = dict(table=arch['move_surf'], layer=0)
        p['disp_surf'] = dict(table=arch['disp_surf'], layer=0)
    if case_cfg:
        p.update(case_cfg)
    return p


def make_device(arch, prm, capacity=None, seed=0, disp_tries=6, extra=None):
    from geonomics_b200.device import DeviceSpecies
    rasters = np.array(arch['rasters'], dtype=np.float64)
    # the golden K raster already includes K_factor: feed it as an extra layer with factor 1
    rasters = np.concatenate([rasters, arch['K'][None]], axis=0)
    p = device_params(arch, prm, extra)
    p['K_layer'] = rasters.shape[0] - 1
    ga = dict(L=arch['paths'].shape[1], paths=arch['paths'], traits=arch['traits'], dom=arch['dom'])
    return DeviceSpecies(arch['land_dim'], rasters, p, ga, capacity=capacity, seed=seed,
                         disp_tries_injected=disp_tries, res_ratio=tuple(arch.get('res_ratio', (1.0, 1.0))))


def set_device_mutation(dev, mut):
    """arch['mutation'] (golden_io / oracle format) -> DeviceSpecies.set_mutation."""
    kw = {}
    if mut.get('tskit_layout'):
        kw = dict(tskit_layout=True, trait_mus=mut.get('trait_mus'),
                  trait_alpha_distr=[tr['alpha_distr'] for tr in mut['traits']],
                  trait_loci_idxs=[tr['loci_idxs'] for tr in mut['traits']],
                  delet_loci_idxs=mut['delet_loci_idxs'], subsetters=mut['subsetters'])
    dev.set_mutation(mut['mu_neut'], mut['mu_delet'], mut['mutables'], mut['nonneut_loci'],
                     mut['delet_loci'], mut['delet_s'], mut.get('s_shape', 0.2), mut.get('s_scale', 0.2), **kw)


def run_device_step(arch, prm, state, draws, capacity=None, staged=True, debug=True, tskit=None):
    """One main time step on the device with injected draws; returns intermediates.
    A use_tskit = True case (arch['mutation']['tskit_layout']) carries genotype ROWS in state['g']: they are
    spread to their loci for the upload and gathered back from the download (genome_pack.rows_to_loci).
    tskit: dict(node0, node1, next_node_id, next_individual_row) turns the row recording on."""
    from geonomics_b200 import genome_pack as gp
    n0 = len(state['x'])
    tsk_layout = bool(arch.get('mutation') and arch['mutation'].get('tskit_layout'))
    if tsk_layout:
        state = dict(state, g=gp.rows_to_loci(state['g'], arch['mutation']['nonneut_loci'], arch['paths'].shape[1]))
    dev = make_device(arch, prm, capacity=capacity or (2 * n0 + 256),
                      disp_tries=draws['disp_dist'].shape[1])
    try:
        dev.set_debug(debug)
        burn = bool(prm.get('burn', False))
        if burn:
            dev.set_burn(True)
            dev.upload(state['x'], state['y'], state['age'], state['sex'], state['idx'],
                       max_ind_idx=state['max_ind_idx'])
        else:
            dev.upload(state['x'], state['y'], state['age'], state['sex'], state['idx'], g=state['g'],
                       z=state['z'], max_ind_idx=state['max_ind_idx'])
        out_burn = burn
        mut = arch.get('mutation')
        if mut is not None and not burn:
            set_device_mutation(dev, mut)
        if tskit is not None:
            dev.tskit_enable(edge_capacity=tskit.get('edge_capacity', 1 << 20), birth_capacity=4 * n0 + 64)
            dev.tskit_set_nodes(tskit['node0'], tskit['node1'], tskit['next_node_id'], tskit['next_individual_row'])
        d = dict(draws)
        if arch.get('move_surf') is None:
            d.pop('move_choice', None)
            d.pop('disp_choice', None)
        else:
            d.pop('move_dir', None)
            d.pop('disp_dir', None)
        dev.set_draws(d)
        out = {}
        if staged:
            dev.stage('age_step')
            dev.stage('move')
            out['mv_x'] = dev.read('X', n0)
            out['mv_y'] = dev.read('Y', n0)
            out['mv_age'] = dev.read('AGE', n0)
            out['mv_e'] = dev.read('E', n0 * dev.n_layers).reshape(n0, dev.n_layers)[:, :-1]
            dev.stage('bin_cells')
            out['perm'] = dev.read('PERM', n0)
            dev.stage('find_mates')
            out['n_nbrs'] = dev.read('N_NBRS', n0)
            out['mate'] = dev.read('MATE', n0)
            dev.stage('dedup_pairs')
            c = dev.counters()
            out['P'], out['B'] = c['P'], c['B']
            out['pairs'] = dev.read('PAIRS', 2 * c['P']).reshape(-1, 2)
            out['nb'] = dev.read('NB', c['P'])
            dev.stage('make_offspring')
            c = dev.counters()
            npre = c['n_pre']
            out['disp_tries'] = dev.read('DISP_TRIES', c['B'])
            out['pre'] = dict(x=dev.read('X', npre), y=dev.read('Y', npre), age=dev.read('AGE', npre),
                              sex=dev.read('SEX', npre), idx=dev.read('IDX', npre), z=dev.read_z(npre))
            dev.stage('density_counts')
            out['counts_N'] = dev.read('COUNTS_N', len(dev.density.points))
            out['counts_P'] = dev.read('COUNTS_P', len(dev.density.points))
            dev.stage('density_eval')
            out['N_rast'] = dev.raster('N_RAST')
            out['n_pairs_rast'] = dev.raster('NPAIRS_RAST')
            out['d_rast'] = dev.raster('D_RAST')
            out['grad_N'] = dev.read('GRAD_N', 2 * len(dev.density.points)).reshape(-1, 2)
            out['gs_iters'] = dev.counters()['gs_iters']
            dev.stage('death_prob')
            out['death_p'] = dev.read('DEATH_P', npre)
            out['fit_all'] = dev.read('FIT', npre)
            out['alive'] = dev.read('ALIVE', npre)
            dev.stage('mortality')
        else:
            dev.step(1)
            if not debug:
                out['N_rast_on_demand'] = dev.raster('N_RAST')
        dev.sync()
        if mut is not None and not burn:
            out['mut_log'], out['mutation'] = dev.read_mutations()
            out['mut_traits'], out['mut_delet_loci_idxs'] = dev.read_mutation_tables()
        if tskit is not None:
            out['tskit_rows'] = dev.tskit_drain()
        out['new'] = dev.download(e=True, genomes=not out_burn)
        if tsk_layout:
            out['new']['g_loci'] = out['new']['g']
            out['new']['g'] = gp.loci_to_rows(out['new']['g'], out['mutation']['nonneut_loci'])
        out['new']['e'] = out['new']['e'][:, :-1]
        out['burn'] = out_burn
        out['records'] = dev.step_records()
        out['counters'] = dev.counters()
        out['launches'] = dev.launch_count
        return out
    finally:
        dev.close()


def compare_step(out, new_o, im_o, rtol=1e-6, exact_xy_tol=1e-9):
    """Device results vs oracle: integer/index work bit-exact, floating point within rtol
    (north_star: 1e-6 relative on phenotype / fitness / mortality probabilities)."""
    if 'pairs' in out:
        assert np.array_equal(out['mv_age'], im_o['mv_age'])
        np.testing.assert_allclose(out['mv_x'], im_o['mv_x'], rtol=0, atol=exact_xy_tol)
        np.testing.assert_allclose(out['mv_y'], im_o['mv_y'], rtol=0, atol=exact_xy_tol)
        assert np.array_equal(out['mv_e'], im_o['mv_e'])
        assert np.array_equal(out['n_nbrs'], im_o['n_nbrs'])
        if im_o['mate'] is not None:
            assert np.array_equal(out['mate'], im_o['mate'])
        assert np.array_equal(out['pairs'], im_o['pairs'])
        assert np.array_equal(out['nb'], im_o['nb'])
        assert out['B'] == im_o['B']
        assert np.array_equal(out['disp_tries'], im_o['disp_tries'])
        pre_o = im_o['pre']
        assert np.array_equal(out['pre']['idx'], pre_o['idx'])
        assert np.array_equal(out['pre']['sex'], pre_o['sex'])
        assert np.array_equal(out['pre']['age'], pre_o['age'])
        np.testing.assert_allclose(out['pre']['x'], pre_o['x'], rtol=0, atol=exact_xy_tol)
        np.testing.assert_allclose(out['pre']['y'], pre_o['y'], rtol=0, atol=exact_xy_tol)
        if not out.get('burn'):
            np.testing.assert_allclose(out['pre']['z'], pre_o['z'], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(out['N_rast'], im_o['N_rast'], rtol=rtol, atol=1e-9)
        np.testing.assert_allclose(out['n_pairs_rast'], im_o['n_pairs_rast'], rtol=rtol, atol=1e-9)
        np.testing.assert_allclose(out['d_rast'], im_o['d_rast'], rtol=rtol, atol=1e-9)
        if not out.get('burn'):
            np.testing.assert_allclose(out['fit_all'], im_o['fit_all'], rtol=rtol)
        np.testing.assert_allclose(out['death_p'], im_o['death_p'], rtol=rtol, atol=1e-9)
    new = out['new']
    assert np.array_equal(new['idx'], new_o['idx'])
    assert np.array_equal(new['age'], new_o['age'])
    assert np.array_equal(new['sex'], new_o['sex'])
    np.testing.assert_allclose(new['x'], new_o['x'], rtol=0, atol=exact_xy_tol)
    np.testing.assert_allclose(new['y'], new_o['y'], rtol=0, atol=exact_xy_tol)
    if not out.get('burn'):
        assert np.array_equal(new['g'], new_o['g'])
        np.testing.assert_allclose(new['z'], new_o['z'], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(new['fit'], new_o['fit'], rtol=rtol)
    assert np.array_equal(new['e'], new_o['e'])
    assert new['max_ind_idx'] == new_o['max_ind_idx']
    rec = out['records'][-1]
    assert rec['Nt'] == len(new_o['x'])
    assert rec['n_births'] == im_o['B']
    assert rec['n_deaths'] == im_o['n_deaths']


# Genome sizes and trait kinds that reach every k_gametes<GW, NT> instantiation and phenotype mode
# (gnx_api.cu launch_gametes): GW = 1, 2, 4, 8, 16, 32 lanes per offspring; at GW 32 two staged rows
# (L 3000), one staged row (L 12000: two 94-unit rows exceed 44 KB) and no staging (L 17000: one row
# exceeds 32 KB).  Kinds: polygenic; polygenic with dominance; a monogenic trait beside a polygenic
# one; five traits with dominance (the GNX_MAX_TRAITS accumulators).
GAMETE_MATRIX_L = (100, 200, 400, 1000, 1500, 3000, 12000, 17000)
TRAIT_KINDS = ('poly', 'dom', 'mono', 'dom5')


def trait_set(L, kind, seed=0, lyr_nums=(1, 2), phi=0.1):
    """(traits, dom) of one trait kind, with trait loci on the word and unit edges 0, 31, 32, 127,
    128 and L - 1 (those below L) dealt round-robin to the traits; traits hold disjoint loci."""
    rng = np.random.default_rng(seed)
    n_traits = 5 if kind == 'dom5' else 2
    edges = [l for l in (0, 31, 32, 127, 128, L - 1) if l < L]
    edges = list(dict.fromkeys(edges))
    per = max(2, min(9, (L - len(edges)) // (2 * n_traits)))
    rest = rng.permutation(np.setdiff1d(np.arange(L), edges))[:per * n_traits]
    loci = [[] for _ in range(n_traits)]
    for k, l in enumerate(edges):
        loci[k % n_traits].append(l)
    for k, l in enumerate(rest):
        loci[k % n_traits].append(int(l))
    if kind == 'mono':                       # trait 0 keeps one locus (31 where the genome has it)
        one = 31 if 31 in loci[0] else loci[0][0]
        loci[1] += [l for l in loci[0] if l != one]
        loci[0] = [one]
    traits = []
    for t in range(n_traits):
        lc = np.array(sorted(loci[t]), dtype=np.int64)
        traits.append(dict(loci=lc, alpha=rng.normal(0, 0.1, len(lc)), phi=phi, gamma=1.0,
                           lyr_num=lyr_nums[t % len(lyr_nums)], univ_adv=False))
    dom = np.zeros(L, np.int8)
    if kind in ('dom', 'dom5'):
        for tr in traits:
            dom[tr['loci'][::2]] = 1         # every other trait locus, the first (an edge locus) included
    return traits, dom


def synthetic_case(L=1000, n=1500, n_traits=2, loci_per_trait=20, dim=(40, 40), seed=0, max_tries=8, cap=None):
    """A synthetic population in the golden-case format (arch, prm, state, draws), for parity
    of the CUDA path against the (golden-pinned) oracle at genome sizes the reference-recorded
    cases do not cover."""
    from geonomics_b200 import workloads, genome_pack
    from oracle import step_oracle as so
    from oracle import draws as od
    cfg = dict(dim=dim, N=n, L=L, n_traits=n_traits, loci_per_trait=loci_per_trait, mating_radius=2.0, b=0.5,
               lam=1, R=0.5, phi=0.1, gamma=1.0, n_paths=500, recomb_rate=0.05, seed=seed, surfaces=False)
    w = workloads.build(cfg, seed)
    g = genome_pack.unpack_genomes(workloads.random_packed_genomes(n, L, seed + 1), L)
    prm_w = w['prm']
    arch = dict(land_dim=w['land_dim'], rasters=w['rasters'], K=w['rasters'][0] * prm_w['K_factor'], ww=None,
                traits=w['gen_arch']['traits'], dom=np.zeros(L, np.int8), paths=w['gen_arch']['paths'],
                move_surf=None, disp_surf=None)
    arch['ww'] = round(0.1 * max(dim))
    prm = dict(b=prm_w['b'], R=prm_w['R'], lam=1, n_births_fixed=True, mating_radius=2.0, d_min=0.0, d_max=1.0,
               sex=False, sex_ratio_p=0.5, max_age=None, direction_mu=0.0, direction_kappa=0.0)
    z = so.phenotype(g, arch['traits'])
    state = dict(x=w['pop']['x'], y=w['pop']['y'], age=w['pop']['age'], sex=w['pop']['sex'],
                 idx=w['pop']['idx'], g=g, z=z, max_ind_idx=n - 1)
    rng = np.random.default_rng(seed + 5)
    draws = od.make_draws(rng, dict(prm, move_distr=('wald', 1.0, 1.0), disp_distr=('wald', 1.0, 1.0)), n,
                          cap or n, len(arch['paths']), max_tries=max_tries)
    return arch, prm, state, draws
