"""GPU: gamete formation / phenotype of the register-streaming kernel across genome sizes,
against the golden-pinned oracle."""
import pytest

from parity_util import synthetic_case, run_device_step, compare_step, trait_set, GAMETE_MATRIX_L, TRAIT_KINDS

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('L', [1, 64, 129, 300, 512, 1000, 2100, 4500])
def test_full_step_parity_across_genome_sizes(L):
    from oracle import step_oracle as so
    arch, prm, state, draws = synthetic_case(L=L, n=1200, loci_per_trait=min(20, max(1, L // 3)),
                                             n_traits=2 if L >= 4 else 1, seed=L, max_tries=24)
    new_o, im_o = so.step(state, arch, prm, draws)
    assert im_o['B'] > 100
    out = run_device_step(arch, prm, state, draws, staged=True)
    compare_step(out, new_o, im_o)


@pytest.mark.parametrize('kind', TRAIT_KINDS)
@pytest.mark.parametrize('L', GAMETE_MATRIX_L)
def test_full_step_parity_across_gamete_instantiations(L, kind):
    """Every lane width, both trait-accumulator counts and the three phenotype modes of k_gametes
    (paired staged rows, one staged row with the dominance / monogenic branch, unstaged), with
    trait loci on word and unit edges, against the oracle with injected draws."""
    from oracle import step_oracle as so
    arch, prm, state, draws = synthetic_case(L=L, n=1200, n_traits=2, loci_per_trait=4, seed=L + 7, max_tries=24)
    arch['traits'], arch['dom'] = trait_set(L, kind, seed=L)
    state['z'] = so.phenotype(state['g'], arch['traits'], arch['dom'])
    new_o, im_o = so.step(state, arch, prm, draws)
    assert im_o['B'] > 100
    out = run_device_step(arch, prm, state, draws, staged=True)
    compare_step(out, new_o, im_o)
