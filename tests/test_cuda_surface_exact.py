"""GPU: the on-the-fly conductance-surface sampler (GNX_SURF_ONTHEFLY, the mode of the c4 workload)
draw for draw, and its von Mises quantile table against the exact quantile.

  * The tables the device built (GNX_F_VM_TAB_MOVE / _DISP) against the von Mises(0, kappa)
    half-distribution quantile computed with scipy in float64, entry by entry, and the distance of
    the distribution the kernel samples from the exact one.
  * Movement and natal dispersal rebuilt from (seed, id, site, t) through tests/philox_ref.py
    (surface_direction, lognormal_f32, wald_f32): the float16 direction is exact, so positions
    with injected distances must equal the restatement bit for bit; free-running distances are
    checked within the float32 samplers' bound, and dispersal tries and sex exactly.
  * A raster change on the movement layer, then on the dispersal layer alone, and a scaled c4 case
    run through graph-launched steps.

The landscape is 37 x 23 (swapping X and Y fails), every cell holds a distinct conductance except
planted patches: a zero block (all-zero neighbourhoods, zero cells next to positive ones), tied
maxima (among them directions pi and -3 pi / 4, whose mean is pi / 8) and the four edges."""
import numpy as np
import pytest

import philox_ref as pr

pytestmark = pytest.mark.gpu

SEED = (0x0C4C4C4C << 32) | 0x13572468            # a seed with a non-zero high word
DIM = (37, 23)                                     # (X, Y)
DIST = 0.25
H = np.pi / (1 << 20)                              # the table builder's trapezoid step
OFFS = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)]     # (di, dj), row-major
MAX_TRIES = 64
GL = 32                                            # loci of the neutral genome the species carry


# ---- landscape and species -----------------------------------------------------------------------------
def landscape(seed=0, X=DIM[0], Y=DIM[1]):
    rng = np.random.default_rng(seed)
    r = (rng.permutation(X * Y) + 1.0).reshape(Y, X) / (X * Y)        # distinct values in (0, 1]
    r[9:14, 14:19] = 0.0                                               # (11, 16): all-zero neighbourhood
    r[4, 24] = r[5, 24] = 5.0                                          # (5, 25): tie of -3 pi / 4 and pi
    r[16, 8] = r[17, 9] = r[18, 8] = 4.0                               # (17, 8): three-way tie
    r[0, 1] = r[1, 0] = 3.0                                            # corner (0, 0): tie on the edges
    r[21, 36] = 2.5                                                    # corner (22, 36): single maximum
    return r


def neighbourhoods(rast, cx, cy):
    """float32[n, 8]: the zero-embedded queen neighbourhoods of cells (cx, cy), as the kernel reads them."""
    Y, X = rast.shape
    r32 = rast.astype(np.float32)
    out = np.zeros((len(cx), 8), np.float32)
    for k, (di, dj) in enumerate(OFFS):
        i, j = cy + di, cx + dj
        ok = (i >= 0) & (i < Y) & (j >= 0) & (j < X)
        out[ok, k] = r32[i[ok], j[ok]]
    return out


def _surf(layer, mixture, kappa):
    return dict(layer=layer, mixture=mixture, kappa=kappa)


def species(rasters, move_surf, disp_surf, move_distr=('lognormal', -1.0, 0.5), disp_distr=('lognormal', -1.0, 0.5),
            capacity=1 << 16, seed=SEED, **kw):
    from geonomics_b200.device import DeviceSpecies
    X, Y = DIM
    prm = dict(b=1.0, R=0.5, lam=1, n_births_fixed=True, mating_radius=1.0, d_min=0.0, d_max=0.0, sex=False,
               K_layer=0, K_factor=1.0, move=True, move_distr=move_distr, disp_distr=disp_distr,
               move_surf=move_surf, disp_surf=disp_surf)
    prm.update(kw)
    paths = (np.cumsum(np.random.default_rng(1).random((16, GL)) < 0.1, axis=1) % 2).astype(np.uint8)
    ga = dict(L=GL, paths=paths, traits=[], dom=np.zeros(GL, np.int8))     # a small neutral genome
    return DeviceSpecies((X, Y), np.asarray(rasters, np.float64), prm, ga, capacity=capacity, seed=seed)


def _upload(dev, x, y, ids):
    dev.upload(x, y, idx=ids, g=np.zeros((len(x), GL, 2), np.int8), max_ind_idx=int(ids.max()))


def population(per_cell, rng, id_base=0, X=DIM[0], Y=DIM[1]):
    """per_cell individuals in every cell, at positions with few mantissa bits (multiples of 1/8), so
    that x + cos * 0.25 is exact wherever it is not clipped."""
    cy, cx = np.divmod(np.repeat(np.arange(X * Y), per_cell), X)
    x = cx + rng.integers(0, 8, len(cx)) / 8.0
    y = cy + rng.integers(0, 8, len(cy)) / 8.0
    return x, y, id_base + np.arange(len(x), dtype=np.int64)


def half_cos_sin(h):
    from oracle import step_oracle as so
    c, s = so._cos_sin(np.asarray(h, np.float16))
    return c.astype(np.float64), s.astype(np.float64)


def _pos_bound(d, rel):
    """|device - float64| of one displacement component with an exact direction: the distance's relative
    error, doubled for the float64 products and sums around it."""
    return 2.0 * d * rel + 1e-12


def _distance(w, k, distr):
    """(distance, relative bound, ambiguous, words used) of sample_distance_f32 from words k, k + 1, ..."""
    name, p1, p2 = distr
    rows = np.arange(len(w))
    if name == 'lognormal':
        d, rel = pr.lognormal_f32(w[rows, k], w[rows, k + 1], p1, p2)
        return d, rel, np.zeros(len(d), bool), 2
    d, rel, amb = pr.wald_f32(w[rows, k], w[rows, k + 1], w[rows, k + 2], p1, p2)
    return d, rel, amb, 3


# ---- 1. the quantile tables ------------------------------------------------------------------------------
def _half_pdf(kappa):
    """The von Mises(0, kappa) density of |theta| on [0, pi]: exp(kappa (cos t - 1)) / (pi i0e(kappa))."""
    from scipy.special import i0e
    A = np.pi * i0e(kappa)
    return lambda t: np.exp(kappa * (np.cos(t) - 1.0)) / A


def _mass(p, a, b):
    from scipy.integrate import quad
    return quad(p, a, b, epsabs=0.0, epsrel=1e-13, limit=200)[0] if b > a else 0.0


def table_nodes():
    """(lower mass u, upper mass 1 - u) of every table entry, both exact: coarse u = k / 4096, fine
    u = 1 - (1 - k / 256) / 4096."""
    k, kf = np.arange(pr.VM_TAB_CELLS + 1), np.arange(pr.VM_TAB_FINE + 1)
    lower = np.concatenate([k / pr.VM_TAB_CELLS, 1 - (1 - kf / pr.VM_TAB_FINE) / pr.VM_TAB_CELLS])
    upper = np.concatenate([(pr.VM_TAB_CELLS - k) / pr.VM_TAB_CELLS, (1 - kf / pr.VM_TAB_FINE) / pr.VM_TAB_CELLS])
    return lower, upper


def entry_bound(tab, kappa, u, p):
    """How far an entry may lie from the exact quantile q(u):
      * one float32 ulp (the entry is the float64 quantile rounded to float32, half an ulp, plus margin);
      * the trapezoid rule: the composite rule's CDF error at node t_i is (h^2 / 12) f'(t_i) / A (the
        end corrections f'(0) = f'(pi) = 0, so the normalising total is exact to far higher order), and
        linear interpolation of the CDF inside a step adds at most (h^2 / 8) max |f'| / A.  Divided by
        the density f / A to become an error in t, with |f' / f| = kappa sin t <= kappa and the density
        changing by at most e^(2 kappa h) inside a step: (1/12 + 1/8) kappa h^2 (1 + 2 kappa h) <= kappa h^2 / 4.
        With h = pi / 2^20 that is 2.2e-12 kappa: about h^2;
      * the float64 rounding of the 2^20-term running sum and its normalisation: lambda sqrt(n) eps
        relative to u (probabilistic bound of recursive summation, lambda = 8), over the density."""
    ulp = np.spacing(np.maximum(tab, np.float32(1e-30))).astype(np.float64)
    trap = kappa * H * H / 4
    rnd = 8 * np.sqrt(1 << 20) * 2.0 ** -53 * u / np.maximum(p, 1e-300)
    return ulp + trap + rnd


def check_table(tab, kappa):
    """Every entry within entry_bound of the exact quantile (the exact quantile is bracketed: the mass
    below tab - B is at most u and the mass below tab + B at least u, counted from whichever end of
    [0, pi] is nearer, so that tail entries keep their relative accuracy); ends exact; monotone."""
    assert tab.dtype == np.float32 and len(tab) == pr.VM_TAB_LEN
    t = tab.astype(np.float64)
    assert tab[0] == 0 and tab[pr.VM_TAB_CELLS] == pr.PI_F and tab[-1] == pr.PI_F
    assert tab[pr.VM_TAB_CELLS + 1] == tab[pr.VM_TAB_CELLS - 1]        # the fine table starts at u = 4095 / 4096
    assert np.all(np.diff(t[:pr.VM_TAB_CELLS + 1]) > 0) and np.all(np.diff(t[pr.VM_TAB_CELLS + 1:]) > 0)
    p = _half_pdf(kappa)
    lower, upper = table_nodes()
    B = entry_bound(tab, kappa, lower, p(t))
    worst = 0.0
    for j in range(len(t)):
        if j in (0, pr.VM_TAB_CELLS, len(t) - 1):
            continue
        lo, hi = t[j] - B[j], min(t[j] + B[j], np.pi)
        if lower[j] <= 0.5:
            ok = _mass(p, 0.0, lo) <= lower[j] <= _mass(p, 0.0, hi)
            r = _mass(p, 0.0, t[j]) - lower[j]
        else:
            ok = _mass(p, lo, np.pi) >= upper[j] >= _mass(p, hi, np.pi)
            r = upper[j] - _mass(p, t[j], np.pi)
        err = abs(r / p(t[j]))                        # one Newton step from the entry: |entry - q(u)|
        worst = max(worst, err / np.spacing(tab[j]))
        assert ok, (kappa, j, lower[j], tab[j], err, B[j])
    return worst


def sampled_distance(tab, kappa):
    """(total variation, Kolmogorov distance) between |theta| as the kernel samples it -- uniform on
    [tab[k], tab[k + 1]] with mass 1 / 4096 for the first 4095 cells, then the last cell's 256 fine cells
    with mass 2^-20 each -- and the exact half-distribution.  The density f is decreasing, so inside a
    cell [a, b] of mass w it crosses the cell's constant c = w / (b - a) once, at t*; with
    D = int_a^t* (f - c) >= 0 (the largest CDF deviation inside the cell) and M = int_a^b f,
    int_a^b |f - c| = 2 D - (M - w)."""
    p = _half_pdf(kappa)
    from scipy.special import i0e
    A = np.pi * i0e(kappa)
    t = tab.astype(np.float64)
    co, fi = t[:pr.VM_TAB_CELLS], t[pr.VM_TAB_CELLS + 1:]
    cells = [(co[k], co[k + 1], 1.0 / pr.VM_TAB_CELLS) for k in range(pr.VM_TAB_CELLS - 1)]
    cells += [(fi[k], fi[k + 1], 1.0 / (pr.VM_TAB_CELLS * pr.VM_TAB_FINE)) for k in range(pr.VM_TAB_FINE)]
    tv, ks = 0.0, 0.0
    for a, b, w in cells:
        c = w / (b - a)
        arg = 1.0 + np.log(c * A) / kappa                          # f(t*) = c
        ts = a if arg >= 1 else (b if arg <= -1 else min(max(np.arccos(arg), a), b))
        D = _mass(p, a, ts) - c * (ts - a)
        tv += 2 * D - (_mass(p, a, b) - w)
        ks = max(ks, D)
    return tv / 2, ks


@pytest.mark.parametrize('kappas', [(0.5, 4.0), (12.0, 60.0), (500.0, 500.0)])
def test_quantile_tables_against_the_exact_quantile(kappas):
    """Both sites' tables (the dispersal table aliases the movement table when the two kappas are equal)."""
    from geonomics_b200 import _lib
    dev = species(landscape()[None], _surf(0, True, kappas[0]), _surf(0, False, kappas[1]))
    try:
        tabs = [dev.read('VM_TAB_MOVE', pr.VM_TAB_LEN), dev.read('VM_TAB_DISP', pr.VM_TAB_LEN)]
    finally:
        dev.close()
    for tab, kappa in zip(tabs, kappas):
        worst = check_table(tab, kappa)
        tv, ks = sampled_distance(tab, kappa)
        print('kappa %g: entries within %.3f ulp of the exact quantile; sampled distribution: TV %.3g, '
              'Kolmogorov %.3g' % (kappa, worst, tv, ks))
        # the linear interpolation inside the 4096 cells is first order in the cell width: TV ~ 1 / 4096 in
        # all; the CDF itself is off by at most ~2e-5, far below what a KS test on 1e6 draws resolves
        assert tv < 3e-4, (kappa, tv)
        assert ks < 3e-5, (kappa, ks)
    if kappas[0] == kappas[1]:
        assert np.array_equal(tabs[0], tabs[1])
    # no table at a site that is not on the fly
    dev = species(landscape()[None], _surf(0, True, 12.0), None)
    try:
        with pytest.raises(_lib.GnxError) as e:
            dev.read('VM_TAB_DISP', pr.VM_TAB_LEN)
        assert e.value.code == -5                                     # GNX_ERR_STATE
        assert len(dev.read('VM_TAB_MOVE', pr.VM_TAB_LEN)) == pr.VM_TAB_LEN
    finally:
        dev.close()


# ---- 2. movement ----------------------------------------------------------------------------------------
def run_move(dev, x, y, ids, dist=None):
    """One movement stage from (x, y); injected distances when `dist` is given.  -> (x', y', t)."""
    _upload(dev, x, y, ids)
    dev.set_draws(None if dist is None else dict(move_dist=np.full(len(x), dist)))
    t = dev.counters()['t']
    dev.stage('move')
    dev.sync()
    n = len(x)
    return dev.read('X', n), dev.read('Y', n), t


def expected_move(rast, x, y, ids, t, mixture, kappa, tab, distr=None):
    """The restated movement: (x, y, tolerance, ambiguous, directions)."""
    X, Y = DIM
    cx, cy = x.astype(np.int64), y.astype(np.int64)
    w = pr.stream_words(SEED, ids, pr.SITE_MOVE, t, 6)
    h, nw = pr.surface_direction(w, 0, neighbourhoods(rast, cx, cy), mixture, kappa, tab)
    cs, sn = half_cos_sin(h)
    if distr is None:
        d, tol, amb = np.full(len(x), DIST), np.zeros(len(x)), np.zeros(len(x), bool)
    else:
        d, rel, amb, _ = _distance(w, nw, distr)
        tol = _pos_bound(d, rel)
    with np.errstate(invalid='ignore'):
        xr = np.clip(x + cs * d, 0, X - 0.001)
        yr = np.clip(y + sn * d, 0, Y - 0.001)
    return xr, yr, tol, amb, h


def _tab(dev, site):
    return dev.read('VM_TAB_' + site, pr.VM_TAB_LEN)


@pytest.mark.parametrize('kappa', [0.0, 12.0, 500.0])
@pytest.mark.parametrize('mixture', [True, False])
def test_movement_directions_exact(mixture, kappa):
    """Injected distance 0.25, free-running directions: every position equals the restatement bit for bit.
    The ids cross 2^32."""
    rng = np.random.default_rng(int(kappa) + 7 * mixture)
    rast = landscape(1)
    x, y, ids = population(24, rng, id_base=(1 << 32) - 5000)
    dev = species(rast[None], _surf(0, mixture, kappa), _surf(0, mixture, kappa))
    try:
        tab = _tab(dev, 'MOVE')
        nx, ny, t = run_move(dev, x, y, ids, dist=DIST)
    finally:
        dev.close()
    xr, yr, _, _, h = expected_move(rast, x, y, ids, t, mixture, kappa, tab)
    bad = np.nonzero((nx != xr) | (ny != yr))[0]
    assert len(bad) == 0, ('%d of %d moves differ' % (len(bad), len(x)), bad[:5], x[bad[:5]], y[bad[:5]],
                           h[bad[:5]], nx[bad[:5]], xr[bad[:5]], ny[bad[:5]], yr[bad[:5]])
    # the draws reached the wrap and, with a table, its fine part
    assert np.any(np.abs(h.astype(np.float64)) > 3.0)
    if kappa > 0:
        r = pr.stream_words(SEED, ids, pr.SITE_MOVE, t, 2)[:, 1 if mixture else 0]
        assert np.any(((r << np.uint32(1)) >> np.uint32(20)) == pr.VM_TAB_CELLS - 1)


def test_direction_pi_wraps_to_minus_pi():
    """loc = pi (the west neighbour is the only maximum) plus a von Mises sample too small to move it:
    the sum is exactly pi and wraps to -pi, as scipy's mod(theta + pi, 2 pi) - pi does."""
    X, Y = DIM
    rast = landscape(2)
    rast[10, 19] = 9.0                                   # the west neighbour of (10, 20)
    n = 200000
    rng = np.random.default_rng(3)
    x, y = 20 + rng.integers(0, 8, n) / 8.0, 10 + rng.integers(0, 8, n) / 8.0
    ids = np.arange(n, dtype=np.int64)
    kappa = 1e6
    dev = species(rast[None], _surf(0, False, kappa), None, capacity=n + 64)
    try:
        tab = _tab(dev, 'MOVE')
        nx, ny, t = run_move(dev, x, y, ids, dist=DIST)
    finally:
        dev.close()
    xr, yr, _, _, h = expected_move(rast, x, y, ids, t, False, kappa, tab)
    assert np.array_equal(nx, xr) and np.array_equal(ny, yr)
    assert np.sum(h == np.float16(-np.pi)) >= 3


@pytest.mark.parametrize('distr', [('lognormal', -1.0, 0.5), ('wald', 1.0, 1.0)])
def test_movement_free_running(distr):
    """Direction and distance both drawn on the device: the distance comes from the words after the
    direction's, within the float32 sampler's bound."""
    rng = np.random.default_rng(21)
    rast = landscape(3)
    x, y, ids = population(12, rng, id_base=(1 << 32) - 3000)
    for mixture, kappa in ((True, 12.0), (False, 60.0)):
        dev = species(rast[None], _surf(0, mixture, kappa), None, move_distr=distr)
        try:
            tab = _tab(dev, 'MOVE')
            nx, ny, t = run_move(dev, x, y, ids)
        finally:
            dev.close()
        xr, yr, tol, amb, _ = expected_move(rast, x, y, ids, t, mixture, kappa, tab, distr)
        ok = ~amb
        assert amb.sum() <= 3, amb.sum()
        ex, ey = np.abs(nx - xr)[ok], np.abs(ny - yr)[ok]
        assert np.all(ex <= tol[ok]), np.max(ex / tol[ok])
        assert np.all(ey <= tol[ok]), np.max(ey / tol[ok])


# ---- 3. dispersal ---------------------------------------------------------------------------------------
def run_dispersal(dev, x, y, ids):
    """Mate search, births and natal dispersal, free-running, from (x, y)."""
    _upload(dev, x, y, ids)
    dev.set_draws(None)
    dev.set_debug(True)
    c0 = dev.counters()
    for st in ('bin_cells', 'find_mates', 'dedup_pairs', 'make_offspring'):
        dev.stage(st)
    dev.sync()
    c = dev.counters()
    n, B, P = len(x), c['B'], c['P']
    S = dict(t=c0['t'], max_idx=c0['max_idx'], B=B, pairs=dev.read('PAIRS', 2 * P).reshape(-1, 2).astype(np.int64),
             nb=dev.read('NB', P).astype(np.int64), tries=dev.read('DISP_TRIES', B))
    S['ox'], S['oy'] = dev.read('X', n + B)[n:], dev.read('Y', n + B)[n:]
    S['sex'], S['idx'] = dev.read('SEX', n + B)[n:], dev.read('IDX', n + B)[n:]
    return S


def check_dispersal(S, rast, x, y, mixture, kappa, tab, distr, sexed=False, sex_ratio_p=0.5):
    """The retry loop restated: each try takes the direction's words, then the distance's, until the
    offspring lands inside the landscape; tries exact wherever no try lands within the bound of the edge,
    the accepted position within its bound, then sex from the words after the last try."""
    X, Y = DIM
    B = S['B']
    assert B > 100
    assert np.array_equal(S['idx'], S['max_idx'] + 1 + np.arange(B))
    pair_of = np.repeat(np.arange(len(S['nb'])), S['nb'])
    a, m = S['pairs'][pair_of, 0], S['pairs'][pair_of, 1]
    mx, my = (x[a] + x[m]) / 2, (y[a] + y[m]) / 2          # exact: the positions are multiples of 1/8
    nv = neighbourhoods(rast, mx.astype(np.int64), my.astype(np.int64))
    per_try = (2 if mixture else 1) + (2 if distr[0] == 'lognormal' else 3)
    w = pr.stream_words(SEED, S['idx'], pr.SITE_DISP, S['t'], per_try * MAX_TRIES + 4)
    tries = S['tries']
    assert tries.min() >= 1 and tries.max() <= MAX_TRIES
    done = np.zeros(B, bool)
    ambiguous = np.zeros(B, bool)
    tries_ref = np.zeros(B, np.int64)
    for k in range(MAX_TRIES):
        h, nw = pr.surface_direction(w, per_try * k, nv, mixture, kappa, tab)
        cs, sn = half_cos_sin(h)
        d, rel, amb, _ = _distance(w, per_try * k + nw, distr)
        tol = _pos_bound(d, rel)
        with np.errstate(invalid='ignore'):
            rx, ry = mx + cs * d, my + sn * d
        ok = (rx > 0) & (ry > 0)
        ambiguous |= ~done & (amb | (np.abs(rx) <= tol) | (np.abs(ry) <= tol))
        last = (k == tries - 1) & ~ambiguous
        xk, yk = np.clip(rx, 0, X - 0.001), np.clip(ry, 0, Y - 0.001)
        assert np.all(np.abs(S['ox'][last] - xk[last]) <= tol[last]), k
        assert np.all(np.abs(S['oy'][last] - yk[last]) <= tol[last]), k
        tries_ref[~done & ok] = k + 1
        done |= ok
    clear = ~ambiguous & done
    bad = np.nonzero(tries[clear] != tries_ref[clear])[0]
    assert len(bad) == 0, (len(bad), tries[clear][bad[:5]], tries_ref[clear][bad[:5]])
    assert clear.mean() > 0.97, clear.mean()
    rows = np.nonzero(clear)[0]
    off = per_try * tries[rows]
    u1 = pr.uniform(np.stack([w[rows, off], w[rows, off + 1]], axis=1), 0)
    u2 = pr.uniform(np.stack([w[rows, off + 2], w[rows, off + 3]], axis=1), 0)
    first = u1 < sex_ratio_p if sexed else np.zeros(len(rows), bool)
    sex = np.where(first, 1, ((u2 if sexed else u1) < 0.5).astype(np.int8))
    assert np.array_equal(S['sex'][rows], sex)
    return tries


def edge_parents(rng, n_pairs):
    """Coincident pairs of parents near the lower and left edges (and some in the interior): the
    offspring's first tries often land below 0."""
    X, Y = DIM
    x = np.concatenate([rng.integers(0, 6, n_pairs // 2) / 8.0, rng.integers(8, 8 * X - 8, n_pairs - n_pairs // 2) / 8.0])
    y = np.concatenate([rng.integers(0, 8 * Y - 8, n_pairs // 2) / 8.0, rng.integers(0, 6, n_pairs - n_pairs // 2) / 8.0])
    return np.repeat(x, 2), np.repeat(y, 2)


@pytest.mark.parametrize('mixture,distr', [(True, ('wald', 0.5, 1.0)), (False, ('lognormal', -1.0, 0.75))])
def test_dispersal_exact(mixture, distr):
    """Movement and dispersal on different layers with different kappas: a swapped or aliased table or
    layer fails."""
    rng = np.random.default_rng(33)
    rasts = np.stack([landscape(4), landscape(5)])
    x, y = edge_parents(rng, 1500)
    ids = 1000 + np.arange(len(x), dtype=np.int64)
    k_move, k_disp = 500.0, 0.5
    dev = species(rasts, _surf(0, not mixture, k_move), _surf(1, mixture, k_disp), disp_distr=distr)
    try:
        tab = _tab(dev, 'DISP')
        S = run_dispersal(dev, x, y, ids)
    finally:
        dev.close()
    tries = check_dispersal(S, rasts[1], x, y, mixture, k_disp, tab, distr)
    assert tries.max() > 2 and (tries > 1).mean() > 0.05


# ---- 4. raster changes ------------------------------------------------------------------------------------
@pytest.mark.parametrize('same_layer', [False, True])
def test_raster_change_reaches_the_sampler(same_layer):
    """set_raster on the movement layer, then on the dispersal layer alone (or, when both sites share a
    layer, the one float32 copy they share): the next draws follow the new raster."""
    rng = np.random.default_rng(44)
    rasts = [landscape(6), landscape(7)]
    disp_layer = 0 if same_layer else 1
    mv, dp = _surf(0, True, 12.0), _surf(disp_layer, False, 4.0)
    distr = ('lognormal', -1.0, 0.75)
    xm, ym, idm = population(4, rng)
    xd, yd = edge_parents(rng, 800)
    idd = 1000 + np.arange(len(xd), dtype=np.int64)
    dev = species(np.stack(rasts), mv, dp, disp_distr=distr)

    def check(cur):
        nx, ny, t = run_move(dev, xm, ym, idm, dist=DIST)
        xr, yr, _, _, _ = expected_move(cur[0], xm, ym, idm, t, True, 12.0, _tab(dev, 'MOVE'))
        assert np.array_equal(nx, xr) and np.array_equal(ny, yr)
        S = run_dispersal(dev, xd, yd, idd)
        check_dispersal(S, cur[disp_layer], xd, yd, False, 4.0, _tab(dev, 'DISP'), distr)

    try:
        cur = list(rasts)
        check(cur)
        cur[0] = landscape(8)
        dev.set_raster(0, cur[0])
        check(cur)
        if not same_layer:
            cur[1] = landscape(9)
            dev.set_raster(1, cur[1])
            check(cur)
    finally:
        dev.close()


# ---- 5. graph-launched steps at c4's settings ----------------------------------------------------------------------
def test_scaled_c4_graph_steps():
    """workloads.CONFIGS['c4'] scaled to ~50 000 individuals (Wald distances, mixture kappa = 12 at both
    sites): after each graph-launched step, every individual that was alive before it moved as the
    restatement says."""
    from geonomics_b200 import workloads
    from geonomics_b200.device import DeviceSpecies
    cfg = workloads.scaled(workloads.CONFIGS['c4'], 50000)
    wl = workloads.build(cfg, cfg['seed'])
    prm = dict(wl['prm'])
    assert prm['move_distr'][0] == 'wald' and prm['move_surf'] == dict(layer=0, mixture=True, kappa=12.0)
    X, Y = wl['land_dim']
    rast = wl['rasters'][0]
    dev = DeviceSpecies(wl['land_dim'], wl['rasters'], prm, wl['gen_arch'], capacity=4 * cfg['N'], seed=SEED)
    pop = wl['pop']
    n_checked = 0
    try:
        tab = _tab(dev, 'MOVE')
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'],
                   genomes_packed=workloads.random_packed_genomes(len(pop['x']), wl['L'], 5))
        dev.set_draws(None)
        dev.set_debug(False)
        before = dev.download(genomes=False)
        for _ in range(4):
            t = dev.counters()['t']
            dev.step(1)
            dev.sync()
            after = dev.download(genomes=False)
            old = np.isin(after['idx'], before['idx'])
            k = np.searchsorted(before['idx'], after['idx'][old])
            x0, y0, ids = before['x'][k], before['y'][k], after['idx'][old]
            cs_h, nw = pr.surface_direction(pr.stream_words(SEED, ids, pr.SITE_MOVE, t, 5), 0,
                                            neighbourhoods(rast, x0.astype(np.int64), y0.astype(np.int64)),
                                            True, 12.0, tab)
            cs, sn = half_cos_sin(cs_h)
            w = pr.stream_words(SEED, ids, pr.SITE_MOVE, t, 5)
            d, rel, amb = pr.wald_f32(w[:, 2], w[:, 3], w[:, 4], 1.0, 1.0)
            tol = _pos_bound(d, rel)
            with np.errstate(invalid='ignore'):
                xr, yr = np.clip(x0 + cs * d, 0, X - 0.001), np.clip(y0 + sn * d, 0, Y - 0.001)
            ok = ~amb
            assert amb.sum() <= 5
            assert np.all(np.abs(after['x'][old][ok] - xr[ok]) <= tol[ok])
            assert np.all(np.abs(after['y'][old][ok] - yr[ok]) <= tol[ok])
            assert old.sum() > 0.5 * len(before['idx']) and (~old).sum() > 1000
            n_checked += int(ok.sum())
            before = after
        assert dev.graph_launch_count >= 3
    finally:
        dev.close()
    assert n_checked > 100000
