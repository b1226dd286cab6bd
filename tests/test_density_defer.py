"""The fused density pass (k_raster_Nd) writes the d of a cell before max(N) is known unless the cell is
deferred.  This restates `raster_d_cell` in numpy and checks the deferral rule: a cell that is not deferred
gets the same d for every Nmax >= N, so computing it early cannot change a bit."""
import numpy as np


def raster_d_cell(N, K, np_, Nmax, R, b, lam, d_min, d_max):
    """d of one cell as k_raster_fix_d computes it (demography.py:95-172)."""
    N, K, np_, Nmax, R, b, lam = map(np.float64, (N, K, np_, Nmax, R, b, lam))
    with np.errstate(all='ignore'):
        np_ = 0.0 if np_ < 0.0 else np_
        if np.isnan(np_):
            np_ = 0.0
        dNdt = R * (1 - (N / K)) * N
        if dNdt < -Nmax:
            dNdt = -Nmax
        if np.isnan(dNdt) or np.isinf(dNdt):
            dNdt = -Nmax
        N_b = b * lam * np_
        N_d = N_b - dNdt
        dv = N_d / N
        if np.isnan(dv):
            dv = 0.0
        return d_min if dv < d_min else (d_max if dv > d_max else dv)


def deferred(N, K, R):
    """The rule of raster_d_cell_no_clip: d waits for max(N) unless dNdt is finite and >= -N."""
    N, K, R = map(np.float64, (N, K, R))
    with np.errstate(all='ignore'):
        dNdt = R * (1 - (N / K)) * N
        return not (np.isfinite(dNdt) and dNdt >= -N)


def _draw(rng, special):
    if rng.random() < 0.3:
        return special[rng.integers(len(special))]
    return float(10.0 ** rng.uniform(-9, 4)) * (1.0 if rng.random() < 0.9 else -1.0)


def test_undeferred_cells_do_not_depend_on_nmax():
    rng = np.random.default_rng(0)
    special = [0.0, -0.0, np.inf, -np.inf, np.nan, 1e-300, 5e-324, 1.0]
    n_kept = n_deferred = 0
    for _ in range(20000):
        N = abs(_draw(rng, special))         # N is clipped at 0 before d (NaN stays NaN)
        K = _draw(rng, special)
        np_ = _draw(rng, special)
        R = float(rng.choice([0.5, 1.0, 2.0, 1e-3, 0.0, np.inf]))
        b, lam = 0.2, float(rng.choice([1.0, 2.5]))
        d_min, d_max = (0.0, 1.0) if rng.random() < 0.5 else (0.01, 0.9)
        if deferred(N, K, R):
            n_deferred += 1
            continue
        n_kept += 1
        ref = raster_d_cell(N, K, np_, N, R, b, lam, d_min, d_max)
        for Nmax in (N, np.nextafter(N, np.inf), 2 * N + 1e-3, N + 1e6, 1e308):
            got = raster_d_cell(N, K, np_, Nmax, R, b, lam, d_min, d_max)
            assert np.array_equal(np.float64(got), np.float64(ref), equal_nan=True), (N, K, np_, R, Nmax, got, ref)
    assert n_kept > 5000 and n_deferred > 2000, (n_kept, n_deferred)


def test_deferred_classes():
    """The cells the rule sends to the tail: K = 0, N > K (1 + 1/R), and NaN; not an empty cell."""
    R = 0.5
    assert deferred(1.0, 0.0, R)                  # K = 0: dNdt = -inf
    assert deferred(0.0, 0.0, R)                  # 0/0: NaN
    assert deferred(3.1, 1.0, R)                  # N > K (1 + 1/R) = 3
    assert not deferred(2.9, 1.0, R)
    assert not deferred(0.0, 1.0, R)
    assert not deferred(0.5, 1.0, R)
    assert deferred(np.nan, 1.0, R)
    assert deferred(np.inf, 1.0, R)
