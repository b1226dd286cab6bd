"""GPU parity: libgnxb200.so (through the C-ABI) vs the oracle and vs the vectors recorded
from the reference, with identical injected draws.  Integer / index work must be bit-exact;
floating point within 1e-6 relative (BASELINE.json north_star)."""
import numpy as np
import pytest

from golden_io import case_names, load_case
from parity_util import run_device_step, compare_step

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module', params=case_names())
def stepped(request):
    from oracle import step_oracle as so
    z, arch, prm, state, draws = load_case(request.param)
    new_o, im_o = so.step(state, arch, prm, draws, burn=prm.get('burn', False))
    out = run_device_step(arch, prm, state, draws, staged=True)
    return request.param, z, out, new_o, im_o


def test_staged_step_matches_oracle(stepped):
    _, z, out, new_o, im_o = stepped
    compare_step(out, new_o, im_o)


def test_staged_step_matches_reference_vectors(stepped):
    """Directly against what the reference itself produced (tests/golden/make_golden.py)."""
    _, z, out, new_o, im_o = stepped
    assert np.array_equal(out['n_nbrs'], z['n_nbrs'])
    assert np.array_equal(out['pairs'], z['pairs'])
    assert np.array_equal(out['nb'], z['nb'])
    assert np.array_equal(out['pre']['idx'], z['pre_idx'])
    assert np.array_equal(out['pre']['sex'], z['pre_sex'])
    new = out['new']
    assert np.array_equal(new['idx'], z['out_idx'])
    if out.get('burn'):
        assert np.array_equal(new['sex'], z['out_sex']) and np.array_equal(new['age'], z['out_age'])
        np.testing.assert_allclose(new['x'], z['out_x'], rtol=0, atol=1e-9)
        np.testing.assert_allclose(out['d_rast'], z['d_rast'], rtol=1e-6, atol=1e-9)
        np.testing.assert_allclose(out['death_p'], z['death_p'], rtol=1e-6, atol=1e-9)
        assert out['records'][-1]['n_deaths'] == int(z['out_n_deaths'])
        return
    assert np.array_equal(new['g'], z['out_g'])
    assert np.array_equal(new['sex'], z['out_sex'])
    assert np.array_equal(new['age'], z['out_age'])
    np.testing.assert_allclose(new['x'], z['out_x'], rtol=0, atol=1e-9)
    np.testing.assert_allclose(new['y'], z['out_y'], rtol=0, atol=1e-9)
    np.testing.assert_allclose(new['z'], z['out_z'], rtol=1e-6)
    np.testing.assert_allclose(new['fit'], z['out_fit'], rtol=1e-6)
    np.testing.assert_allclose(out['N_rast'], z['N_rast'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(out['d_rast'], z['d_rast'], rtol=1e-6, atol=1e-9)
    np.testing.assert_allclose(out['death_p'], z['death_p'], rtol=1e-6, atol=1e-9)
    assert out['records'][-1]['Nt'] == int(z['out_Nt'])
    assert out['records'][-1]['n_deaths'] == int(z['out_n_deaths'])


def test_density_counts_exact(stepped):
    from oracle import step_oracle as so
    name, z, out, new_o, im_o = stepped
    _, arch, prm, state, draws = load_case(name)[0:5]
    dgs = so.DensityGridStack(arch['land_dim'], arch['ww'])
    pre = im_o['pre']
    cN = np.concatenate([c.ravel() for c in dgs.counts(pre['x'], pre['y'])])
    assert np.array_equal(out['counts_N'], cN)
    pairs = im_o['pairs']
    x, y = im_o['mv_x'], im_o['mv_y']
    px = (x[pairs[:, 0]] + x[pairs[:, 1]]) / 2
    py = (y[pairs[:, 0]] + y[pairs[:, 1]]) / 2
    cP = np.concatenate([c.ravel() for c in dgs.counts(px, py)])
    assert np.array_equal(out['counts_P'], cP)


@pytest.mark.parametrize('name', case_names())
def test_fused_step_equals_staged(name):
    from oracle import step_oracle as so
    z, arch, prm, state, draws = load_case(name)
    new_o, im_o = so.step(state, arch, prm, draws, burn=prm.get('burn', False))
    out = run_device_step(arch, prm, state, draws, staged=False)
    compare_step(out, new_o, im_o)


@pytest.mark.parametrize('ww', [3, 2.5, 3.7, 7.25])
def test_density_counts_window_widths(ww):
    """Grid-cell assignment (spatial.py:73-97) for integer, dyadic and non-dyadic window widths:
    the one-index-per-axis shortcut (dyadic half-windows) and the four floor divisions as
    written (everything else) both match the oracle bin for bin, including points on cell edges."""
    from oracle import step_oracle as so
    from parity_util import synthetic_case, make_device
    arch, prm, state, draws = synthetic_case(L=32, n=30000, n_traits=0, loci_per_trait=0, dim=(60, 45), seed=77)
    arch['ww'] = ww
    x, y = state['x'].copy(), state['y'].copy()
    # a third of the points exactly on multiples of the half-window
    k = len(x) // 3
    x[:k] = np.minimum(np.round(x[:k] / (ww / 2)) * (ww / 2), 60 - 0.001)
    y[:k] = np.minimum(np.round(y[:k] / (ww / 2)) * (ww / 2), 45 - 0.001)
    dev = make_device(arch, prm, capacity=40000)
    try:
        dev.set_burn(True)
        dev.upload(x, y, state['age'], state['sex'], state['idx'], max_ind_idx=state['max_ind_idx'])
        dev.stage('density_counts')
        dev.sync()
        got = dev.read('COUNTS_N', len(dev.density.points))
    finally:
        dev.close()
    dgs = so.DensityGridStack(arch['land_dim'], ww)
    want = np.concatenate([c.ravel() for c in dgs.counts(x, y)])
    assert np.array_equal(got, want)
    assert got.sum() > 0


@pytest.mark.parametrize('name', case_names())
def test_production_step_matches_oracle(name):
    """The step as it runs in production (fused gnx_step, no debug arrays): the survivors, their
    genotypes, phenotypes and fitness must equal the oracle's, and so must the N raster read
    afterwards (`spp.N`)."""
    from oracle import step_oracle as so
    z, arch, prm, state, draws = load_case(name)
    new_o, im_o = so.step(state, arch, prm, draws, burn=prm.get('burn', False))
    out = run_device_step(arch, prm, state, draws, staged=False, debug=False)
    compare_step(out, new_o, im_o)
    assert np.array_equal(out['new']['idx'], z['out_idx'])
    np.testing.assert_allclose(out['N_rast_on_demand'], im_o['N_rast'], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize('L,n_traits,lpt', [(100, 5, 7), (300, 8, 9), (1000, 3, 40)])
def test_many_traits(L, n_traits, lpt):
    """More than two traits (the reference allows any number, genome.py:826-867): the 8-accumulator
    instantiations of the gamete / phenotype kernels, the per-trait environment reads of k_death and
    the z planes of the compaction, against the oracle -- staged and as the production step."""
    from oracle import step_oracle as so
    from parity_util import synthetic_case
    arch, prm, state, draws = synthetic_case(L=L, n=1800, n_traits=n_traits, loci_per_trait=lpt, seed=50 + n_traits,
                                             max_tries=24)
    for t, tr in enumerate(arch['traits']):                  # spread the traits over the layers and exponents
        tr['gamma'] = (1.0, 2.0, 1.5)[t % 3]
        tr['phi'] = 0.03 + 0.02 * t
    new_o, im_o = so.step(state, arch, prm, draws)
    compare_step(run_device_step(arch, prm, state, draws, staged=True), new_o, im_o)
    compare_step(run_device_step(arch, prm, state, draws, staged=False, debug=False), new_o, im_o)
    assert new_o['z'].shape[1] == n_traits and im_o['B'] > 100
