"""The growth guard's bound on one step's births and the growth policy (geonomics_b200.device), on the CPU:
the bound k_step_guard evaluates, restated as plain functions, and the Poisson bound's tail against
scipy.stats.poisson."""
import numpy as np
import pytest


def test_fixed_births_bound_is_lambda_n():
    from geonomics_b200.device import max_births
    for lam in (1, 2, 5):
        for n in (0, 1, 4096, 10_000_000):
            assert max_births(lam, True, n) == lam * n
    assert max_births(2.7, True, 100) == 200             # the integer litter size, as the kernels take it


@pytest.mark.parametrize('lam', [0.5, 1.0, 3.0, 10.0])
def test_poisson_bound_tail_is_negligible(lam):
    """Births of a step are Poisson(lam * P) with P <= n pairs; P(births > bound) < 1e-15 at every size."""
    from scipy.stats import poisson
    from geonomics_b200.device import max_births
    for n in (0, 1, 10, 1000, 100_000, 10_000_000):
        b = max_births(lam, False, n)
        assert b >= lam * n + 32
        assert poisson.sf(b, lam * n) < 1e-15, (lam, n)


def test_poisson_bound_formula():
    from geonomics_b200.device import max_births
    assert max_births(3.0, False, 0) == 32
    m = 3.0 * 2000
    assert max_births(3.0, False, 2000) == int(np.ceil(m + 10.0 * np.sqrt(m))) + 32


def test_growth_capacity_at_least_doubles():
    from geonomics_b200.device import growth_capacity
    assert growth_capacity(5000, 4096) == 8192
    assert growth_capacity(30000, 4096) == 30000
    caps = [4096]
    while caps[-1] < 10_000_000:
        caps.append(growth_capacity(caps[-1] + 1, caps[-1]))
    assert len(caps) <= 13                               # a logarithmic number of re-allocations
