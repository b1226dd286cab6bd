"""The density rasters in one landscape pass (k_raster_Nd) with a list-driven tail (k_raster_fix_N,
k_raster_fix_d), on a landscape where all three kinds of cell occur:
  * ordinary cells, whose d is written by the fused pass;
  * deferred cells, whose d waits for max(N): a K = 0 patch and a patch where N > K (1 + 1/R);
  * fix cells, whose density is at rounding-noise level: an empty region, evaluated in scipy's exact
    operation order.
Against the oracle (staged), graph-launched steps against the staged path, and strips against the
undecomposed run."""
import numpy as np
import pytest

from parity_util import synthetic_case, make_device, run_device_step, compare_step

pytestmark = pytest.mark.gpu

DIM = (120, 40)
EMPTY_X = 72          # no individual starts left of this column: the interpolant there is at noise level


def _case(seed=5, n=2400):
    arch, prm, state, draws = synthetic_case(L=64, n=n, n_traits=2, loci_per_trait=8, dim=DIM, seed=seed,
                                             max_tries=24)
    X, Y = DIM
    state = dict(state, x=EMPTY_X + state['x'] * (X - 0.001 - EMPTY_X) / X)
    K = np.array(arch['K'], dtype=np.float64)
    K[:, 84:90] = 0.0                 # K = 0: dNdt = -inf
    K[:, 100:106] = 1e-3              # N > K (1 + 1/R)
    arch = dict(arch, K=K)
    return arch, prm, state, draws


def test_three_cell_classes_against_the_oracle():
    from oracle import step_oracle as so
    arch, prm, state, draws = _case()
    new_o, im_o = so.step(state, arch, prm, draws)
    out = run_device_step(arch, prm, state, draws)
    nfix, ndef = out['counters']['density_lists']
    assert nfix > 0 and ndef > 0, (nfix, ndef)
    N = out['N_rast']
    assert (N > 1e-7).sum() > N.size // 4          # ordinary cells too
    compare_step(out, new_o, im_o)


def _device_draws(d):
    d = dict(d)
    d.pop('move_choice', None)
    d.pop('disp_choice', None)
    return d


def test_graph_launched_steps_equal_the_staged_path():
    from oracle import draws as od
    arch, prm, state, _ = _case(seed=6)
    rows = 12000
    rng = np.random.default_rng(17)
    dprm = dict(prm, move_distr=('wald', 1.0, 1.0), disp_distr=('wald', 1.0, 1.0))
    steps = [od.make_draws(rng, dprm, rows // 2, rows // 2, len(arch['paths']), max_tries=24) for _ in range(12)]
    devs = [make_device(arch, prm, capacity=rows, disp_tries=24) for _ in range(2)]
    try:
        for dev in devs:
            dev.upload(state['x'], state['y'], state['age'], state['sex'], state['idx'], g=state['g'], z=state['z'],
                       max_ind_idx=state['max_ind_idx'])
        graph, staged = devs
        lists = []
        for t, d in enumerate(steps):
            for dev in devs:
                dev.set_draws(_device_draws(d))
            graph.step(1)
            for st in ('age_step', 'move', 'bin_cells', 'find_mates', 'dedup_pairs', 'make_offspring',
                       'density_counts', 'density_eval', 'death_prob', 'mortality'):
                staged.stage(st)
            graph.sync()
            staged.sync()
            for f in ('N_RAST', 'D_RAST'):
                assert np.array_equal(graph.raster(f), staged.raster(f), equal_nan=True), (f, t)
            lists.append((graph.counters()['density_lists'], staged.counters()['density_lists']))
            assert lists[-1][0] == lists[-1][1], (t, lists[-1])
            a, b = graph.download(genomes=True), staged.download(genomes=True)
            assert np.array_equal(a['idx'], b['idx']), t
            for k in ('x', 'y', 'age', 'sex', 'g', 'z', 'fit'):
                assert np.array_equal(a[k], b[k]), (k, t)
        assert graph.graph_launch_count >= 10, graph.graph_launch_count
        assert all(l[0][0] > 0 and l[0][1] > 0 for l in lists), lists
    finally:
        for dev in devs:
            dev.close()


def _strip_workload(seed=3, n=4000):
    rng = np.random.default_rng(seed)
    X, Y = DIM
    lyr0 = np.ones((Y, X))
    lyr0[:, 84:90] = 0.0
    lyr0[:, 100:106] = 1e-3
    rasters = np.stack([lyr0, np.tile(np.linspace(0, 1, X), (Y, 1)), np.tile(np.linspace(0, 1, Y)[:, None], (1, X))])
    L = 64
    loci = np.sort(rng.choice(L, 16, replace=False))
    traits = [dict(loci=loci[:8].astype(np.int64), alpha=rng.normal(0, 0.1, 8), phi=0.3, gamma=1.0, lyr_num=1,
                   univ_adv=False),
              dict(loci=loci[8:].astype(np.int64), alpha=rng.normal(0, 0.1, 8), phi=0.2, gamma=1.0, lyr_num=2,
                   univ_adv=False)]
    paths = (np.cumsum(rng.random((200, L)) < 0.3, axis=1) % 2).astype(np.uint8)
    ga = dict(L=L, paths=paths, traits=traits, dom=np.zeros(L, np.int8))
    prm = dict(b=0.5, R=0.5, lam=1, n_births_fixed=True, mating_radius=2.0, d_min=0.0, d_max=1.0, sex=False,
               sex_ratio_p=0.5, max_age=None, K_layer=0, K_factor=n / float(lyr0.sum()), move=True,
               move_distr=('wald', 1.5, 1.0), disp_distr=('wald', 2.0, 1.0), direction_mu=0.0, direction_kappa=0.0,
               density_grid_window_width=None)
    pop = dict(x=rng.uniform(EMPTY_X, X - 0.001, n), y=rng.uniform(0, Y - 0.001, n),
               age=rng.integers(0, 4, n).astype(np.int32), sex=rng.integers(0, 2, n).astype(np.int8),
               idx=np.arange(n, dtype=np.int64))
    g = (rng.random((n, L, 2)) < 0.5).astype(np.int8)
    return DIM, rasters, prm, ga, pop, g


@pytest.mark.parametrize('world', [2, 3])
def test_strips_equal_the_single_context(world):
    from geonomics_b200.device import DeviceSpecies
    from geonomics_b200.strips import LocalStrips
    dim, rasters, prm, ga, pop, g = _strip_workload()
    steps, seed = 5, 29
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=seed)
    try:
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
        ref = []
        for _ in range(steps):
            dev.step(1)
            dev.sync()
            ref.append(dev.download())
        assert all(v > 0 for v in dev.counters()['density_lists'])
    finally:
        dev.close()
    st = LocalStrips(world, dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=seed)
    try:
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
        for t in range(steps):
            st.step(1)
            got = st.download()
            a = ref[t]
            assert np.array_equal(a['idx'], got['idx']), t
            for k in ('x', 'y', 'age', 'sex', 'g', 'z', 'fit'):
                assert np.array_equal(a[k], got[k]), (k, t)
        deferred = [r.dev.counters()['density_lists'][1] for r in st.ranks]
        assert sum(v > 0 for v in deferred) >= 2, deferred
    finally:
        st.close()
