"""GPU: the free-running step (set_draws(None): Philox streams keyed by (seed, id, site, t), pair
list in mating-grid order) checked draw for draw against the oracle's stage functions.

Every random number of the step is a pure function of (seed, id, site, t, word), so each stage's
draws are rebuilt on the host (tests/philox_ref.py) from the device's own state before that stage,
in the layout the oracle's stage function reads:

  MOVE       id       w0 direction (uniform_f32), w1-w2 lognormal distance (normal_f32)
  MATE       id       uniform: w0 R, w1-2 u; nearest: w0-1 u; inverse distance: w0-1 u_inv, w2-3 u
  PANMIXIA   id of entry i     w0-1 u, w2 R0, w3 R1 (R0 and R1 pick entries)
  BIRTHS     position of the pair in the device's pair list: products of uniform() (lam < 10)
  GAMETE     newborn id max_idx + 1 + o: w0 k0, w1 k1, w2 bit 0 = h0, bit 1 = h1
  DISP       newborn id       each try: direction, distance as MOVE; then sex from the same stream
  DEATH      entry id         w0-1 u; alive = !(u < p)

Integer work (pairs, births, genomes, sexes, survival) must match exactly; positions match a
float64 restatement within a bound derived from the float32 samplers' documented error (a wrong
word or key is an O(1) error); phenotypes match an exactly rounded sum within a bound derived from
the number of terms."""
import json
import math
import os
import tempfile

import numpy as np
import pytest

import philox_ref as pr
from parity_util import trait_set, GAMETE_MATRIX_L, TRAIT_KINDS

pytestmark = pytest.mark.gpu

SEED = (0x5EED1234 << 32) | 0x9ABCDEF1          # a seed with a non-zero high word
DIST = ('lognormal', 0.0, 0.5)                   # well conditioned in float32; float32-exact parameters
MAX_TRIES_CHECKED = 64                           # dispersal tries restated (parents on the landscape edge need ~20)


# ---- building and driving a species ---------------------------------------------------------------
def _paths(L, n_paths, rng, rate=0.02):
    """Cached recombination paths as simulated: cumsum(Bernoulli(rate)) % 2, rate[0] = 0."""
    br = rng.random((n_paths, L)) < rate
    br[:, 0] = False
    return (np.cumsum(br, axis=1) % 2).astype(np.uint8)


def _species(dim, n, L=128, kind='poly', b=0.6, mode='random', sexed=False, radius=2.0, lam=1, fixed=True,
             d_max=0.3, phi=0.1, capacity=None, n_paths=64, seed=SEED, gseed=0, id_base=0, xy=None, sex_ratio_p=0.5):
    """A DeviceSpecies with lognormal movement and dispersal, plus the population to upload."""
    from geonomics_b200.device import DeviceSpecies
    rng = np.random.default_rng(gseed)
    X, Y = dim
    rasters = np.stack([np.tile(np.linspace(0, 1, X), (Y, 1)), np.tile(np.linspace(0, 1, Y)[:, None], (1, X)),
                        np.ones((Y, X))])
    traits, dom = trait_set(L, kind, seed=gseed, lyr_nums=(0, 1), phi=phi)
    paths = _paths(L, n_paths, rng)
    prm = dict(b=b, R=0.5, lam=lam, n_births_fixed=fixed, mating_radius=radius, d_min=0.0, d_max=d_max, sex=sexed,
               sex_ratio_p=sex_ratio_p, max_age=None, K_layer=2, K_factor=n / float(X * Y), move=True,
               move_distr=DIST, disp_distr=DIST, direction_mu=0.0, direction_kappa=0.0,
               choose_nearest=(mode == 'nearest'), inverse_dist=(mode == 'inverse'))
    ga = dict(L=L, paths=paths, traits=traits, dom=dom)
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=capacity or (3 * n + 256), seed=seed)
    if xy is None:
        x, y = rng.uniform(0, X - 0.001, n), rng.uniform(0, Y - 0.001, n)
    else:
        x, y = xy
    g = (rng.random((n, L, 2)) < 0.5).astype(np.int8)
    pop = dict(x=x, y=y, age=rng.integers(0, 5, n).astype(np.int32), sex=rng.integers(0, 2, n).astype(np.int8),
               idx=id_base + np.arange(n, dtype=np.int64), g=g)
    sp = dict(dim=dim, L=L, traits=traits, dom=dom, paths=paths, rasters=rasters, prm=prm, mode=mode)
    return dev, pop, sp


def _upload(dev, pop):
    from oracle import step_oracle as so
    z = so.phenotype(pop['g'], dev.gen_arch['traits'], dev.gen_arch['dom'])
    dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=pop['g'], z=z,
               max_ind_idx=int(pop['idx'][-1]))


def traced(fn):
    """Run fn under torch.profiler -> the names of the kernels it launched."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory(prefix='gnx_free_') as td:
        path = os.path.join(td, 'trace.json')
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)['traceEvents']
    return {e['name'].split('(')[0].replace('void ', '').strip() for e in events if e.get('cat') == 'kernel'}


def run_stages(dev, pop, debug=True, trace_gametes=False, finish=True):
    """One free-running step stage by stage; the species-order state between the stages."""
    _upload(dev, pop)
    dev.set_draws(None)
    dev.set_debug(debug)
    c = dev.counters()
    S = dict(t=c['t'], max_idx=c['max_idx'], n0=c['n'], ids=dev.read('IDX', c['n']))
    n0 = S['n0']
    assert np.array_equal(S['ids'], pop['idx'])
    dev.stage('age_step')
    dev.stage('move')
    S['x'], S['y'] = dev.read('X', n0), dev.read('Y', n0)
    dev.stage('bin_cells')
    S['perm'] = dev.read('PERM', n0)
    dev.stage('find_mates')
    if debug:
        S['n_nbrs'] = dev.read('N_NBRS', n0)
    dev.stage('dedup_pairs')
    c = dev.counters()
    S['P'], S['B'] = c['P'], c['B']
    S['pairs'] = dev.read('PAIRS', 2 * c['P']).reshape(-1, 2).astype(np.int64)
    S['nb'] = dev.read('NB', c['P']).astype(np.int64)
    if not finish:
        return S
    if trace_gametes:
        S['kernels'] = traced(lambda: dev.stage('make_offspring'))
    else:
        dev.stage('make_offspring')
    c = dev.counters()
    npre = c['n_pre']
    S['npre'] = npre
    if debug:
        S['disp_tries'] = dev.read('DISP_TRIES', c['B'])
    S['pre'] = dict(x=dev.read('X', npre), y=dev.read('Y', npre), age=dev.read('AGE', npre),
                    sex=dev.read('SEX', npre), idx=dev.read('IDX', npre), z=dev.read_z(npre))
    dev.stage('density_counts')
    dev.stage('density_eval')
    dev.stage('death_prob')
    S['d_rast'] = dev.raster('D_RAST')
    if debug:
        S['death_p'] = dev.read('DEATH_P', npre)
    S['alive'] = dev.read('ALIVE', npre)
    dev.stage('mortality')
    dev.sync()
    S['new'] = dev.download(genomes=True)
    return S


# ---- the checks, one per stage ---------------------------------------------------------------------
def _pos_bound(d, rel, e_dir):
    """|device - float64| of one displacement component: the direction's error times the distance plus
    the distance's relative error, doubled for the float64 sums around them."""
    return 2.0 * d * (e_dir + (1.0 + e_dir) * rel) + 1e-12


def check_move(S, pop, sp):
    w = pr.stream_words(SEED, S['ids'], pr.SITE_MOVE, S['t'], 3)
    cs, sn, e_dir = pr.direction_f32(w[:, 0])
    d, rel = pr.lognormal_f32(w[:, 1], w[:, 2], DIST[1], DIST[2])
    X, Y = sp['dim']
    xr = np.clip(pop['x'] + cs * d, 0, X - 0.001)
    yr = np.clip(pop['y'] + sn * d, 0, Y - 0.001)
    tol = _pos_bound(d, rel, e_dir)
    assert np.all(np.abs(S['x'] - xr) <= tol), np.max(np.abs(S['x'] - xr) / tol)
    assert np.all(np.abs(S['y'] - yr) <= tol), np.max(np.abs(S['y'] - yr) / tol)
    assert np.median(np.abs(S['x'] - xr) / d) < 1e-6          # typical error: float32 rounding, not the bound


def mate_draws(ids, t, mode):
    w = pr.stream_words(SEED, ids, pr.SITE_MATE, t, 4)
    if mode == 'random':
        return w[:, 0], pr.uniform(w, 1), None
    if mode == 'nearest':
        return None, pr.uniform(w, 0), None
    return None, pr.uniform(w, 2), pr.uniform(w, 0)


def check_mates(S, pop, sp):
    """The device's pair list equals the oracle's mate search on the restated draws, as (focal, mate)
    pairs, and lists them in mating-grid order of the focal (cell key, id)."""
    from oracle import step_oracle as so
    prm, mode = sp['prm'], sp['mode']
    R, u, u_inv = mate_draws(S['ids'], S['t'], mode)
    if R is None:
        R = np.zeros(len(u), np.uint32)
    pairs_o, nn_o, _ = so.find_mates_radius(S['x'], S['y'], sp['dim'], prm['mating_radius'], prm['b'], R, u,
                                            sex=pop['sex'] if prm['sex'] else None,
                                            choose_nearest=(mode == 'nearest'), inverse_dist=(mode == 'inverse'),
                                            inv_u=u_inv)
    rank, perm_o, _ = so.canonical_rank(S['x'], S['y'], sp['dim'], prm['mating_radius'])
    assert np.array_equal(S['perm'], perm_o)
    if 'n_nbrs' in S:
        assert np.array_equal(S['n_nbrs'], nn_o)
    assert len(S['pairs']) == len(pairs_o)
    want = pairs_o[np.argsort(rank[pairs_o[:, 0]], kind='stable')]
    assert np.array_equal(S['pairs'], want)
    return pairs_o


def check_births(S, sp):
    prm = sp['prm']
    if prm['n_births_fixed']:
        assert np.all(S['nb'] == prm['lam']) and S['B'] == S['P'] * prm['lam']
        return
    nw = 48
    w = pr.stream_words(SEED, np.arange(S['P']), pr.SITE_BIRTHS, S['t'], nw)
    u = np.stack([pr.uniform(w, 2 * k) for k in range(nw // 2)], axis=1)
    prod = np.cumprod(u, axis=1)                      # sequential products, as the device forms them
    enlam = math.exp(-prm['lam'])
    assert np.all(prod[:, -1] <= enlam), 'restated Poisson ran out of words'
    want = np.maximum((prod > enlam).sum(axis=1), 1)
    bad = np.nonzero(want != S['nb'])[0]
    # the one tolerated difference: a product within a few ulp of exp(-lam), where the device's exp()
    # and the host's may round to neighbouring doubles
    near = np.any(np.abs(prod[bad] - enlam) <= 4 * np.spacing(enlam), axis=1)
    assert np.all(near), (bad[~near][:10], want[bad[~near][:10]], S['nb'][bad[~near][:10]])
    assert len(bad) <= 1
    assert S['B'] == int(S['nb'].sum())


def offspring_layout(S):
    nb = S['nb']
    pair_of = np.repeat(np.arange(len(nb)), nb)
    off_start = np.concatenate([[0], np.cumsum(nb)])[:-1]
    return pair_of, off_start


def gamete_draws(S, n_paths):
    """(recomb_keys, start_homs) laid out as the injected branch of load_plan reads them."""
    B = S['B']
    pair_of, off_start = offspring_layout(S)
    w = pr.stream_words(SEED, S['max_idx'] + 1 + np.arange(B), pr.SITE_GAMETE, S['t'], 3)
    k0, k1 = pr.choose_k(w[:, 0], n_paths), pr.choose_k(w[:, 1], n_paths)
    h0, h1 = (w[:, 2] & 1).astype(np.int64), ((w[:, 2] >> 1) & 1).astype(np.int64)
    o = np.arange(B)
    j = o - off_start[pair_of]
    e = 2 * (off_start[pair_of] + S['nb'][pair_of])
    rk = np.zeros(2 * B, np.int64)
    rk[e - 1 - 2 * j] = k0
    rk[e - 2 - 2 * j] = k1
    return rk, np.stack([h0, h1], axis=1)


def z_reference(child, traits, dom):
    """Exactly rounded phenotypes (math.fsum) with the dominance and monogenic rules of so.phenotype, and
    the bound a sum of n terms in another order may differ by: (n + 2) eps (0.5 + sum |geno alpha|)."""
    B = child.shape[0]
    z = np.zeros((B, len(traits)))
    tol = np.zeros((B, len(traits)))
    for t, tr in enumerate(traits):
        loci = np.asarray(tr['loci'], np.int64)
        geno = child[:, loci, :].astype(np.float64).mean(axis=2)
        if np.any(dom):
            geno = np.minimum(geno * (1 + dom[loci]), 1.0)
        if len(loci) == 1:
            z[:, t] = geno[:, 0]
            continue
        terms = geno * np.asarray(tr['alpha'])[None, :]
        z[:, t] = [math.fsum([0.5] + list(r)) for r in terms]
        tol[:, t] = (len(loci) + 2) * np.finfo(np.float64).eps * (0.5 + np.abs(terms).sum(axis=1))
    return z, tol


def check_gametes(S, pop, sp, expect_all=False):
    """Newborn ids follow the device's pair order; every newborn's homologues are so.make_gametes of its
    parents with the restated keys and start homologues; z is the exactly rounded sum within its bound."""
    from oracle import step_oracle as so
    B, n0 = S['B'], S['n0']
    assert B > 0
    ids_new = S['max_idx'] + 1 + np.arange(B)
    assert np.array_equal(S['pre']['idx'][n0:n0 + B], ids_new)
    rk, sh = gamete_draws(S, len(sp['paths']))
    child = so.make_gametes(pop['g'], S['pairs'], S['nb'], rk, sh, sp['paths'])
    z_ref, tol = z_reference(child, sp['traits'], sp['dom'])
    z_dev = S['pre']['z'][n0:n0 + B]
    assert np.all(np.abs(z_dev - z_ref) <= tol), np.max(np.abs(z_dev - z_ref) - tol)
    new = S['new']
    sel = np.nonzero(new['idx'] > S['max_idx'])[0]
    o = new['idx'][sel] - S['max_idx'] - 1
    if expect_all:
        assert len(sel) == B
    assert len(sel) > 0
    assert np.array_equal(new['g'][sel], child[o])


def check_dispersal_and_sex(S, sp):
    """Natal dispersal from the parents' midpoint (float64 restatement within its bound, tries exact where
    no try lands within the bound of the landscape edge) and the sex drawn after the last try."""
    B, n0 = S['B'], S['n0']
    prm = sp['prm']
    X, Y = sp['dim']
    pair_of, _ = offspring_layout(S)
    a, m = S['pairs'][pair_of, 0], S['pairs'][pair_of, 1]
    mx, my = (S['x'][a] + S['x'][m]) / 2, (S['y'][a] + S['y'][m]) / 2
    K = MAX_TRIES_CHECKED
    w = pr.stream_words(SEED, S['max_idx'] + 1 + np.arange(B), pr.SITE_DISP, S['t'], 3 * K + 4)
    tries = S['disp_tries']
    assert tries.min() >= 1 and tries.max() <= K
    ox, oy = np.zeros(B), np.zeros(B)
    done = np.zeros(B, bool)
    tries_ref = np.zeros(B, np.int64)
    ambiguous = np.zeros(B, bool)
    for k in range(K):
        cs, sn, e_dir = pr.direction_f32(w[:, 3 * k])
        d, rel = pr.lognormal_f32(w[:, 3 * k + 1], w[:, 3 * k + 2], DIST[1], DIST[2])
        tol = _pos_bound(d, rel, e_dir)
        rx, ry = mx + cs * d, my + sn * d
        ok = (rx > 0) & (ry > 0)                   # clipped to [0, dim - 0.001]: only 0 is refused
        ambiguous |= ~done & ((np.abs(rx) <= tol) | (np.abs(ry) <= tol))
        last = k == tries - 1
        xk, yk = np.clip(rx, 0, X - 0.001), np.clip(ry, 0, Y - 0.001)
        assert np.all(np.abs(S['pre']['x'][n0:][last] - xk[last]) <= tol[last])
        assert np.all(np.abs(S['pre']['y'][n0:][last] - yk[last]) <= tol[last])
        tries_ref[~done & ok] = k + 1
        done |= ok
    clear = ~ambiguous & done
    assert np.array_equal(tries[clear], tries_ref[clear])
    assert clear.mean() > 0.95
    # sex: from the same stream, at word 3 * tries
    off = 3 * tries
    rows = np.arange(B)
    u1 = pr.uniform(np.stack([w[rows, off], w[rows, off + 1]], axis=1), 0)
    u2 = pr.uniform(np.stack([w[rows, off + 2], w[rows, off + 3]], axis=1), 0)
    if prm['sex']:
        first = u1 < prm['sex_ratio_p']
        redraw = u2
    else:
        first = np.zeros(B, bool)
        redraw = u1
    sex = np.where(first, 1, (redraw < 0.5).astype(np.int8))
    assert np.array_equal(S['pre']['sex'][n0:n0 + B], sex)


def check_mortality(S, sp):
    from oracle import step_oracle as so
    pre = S['pre']
    w = pr.stream_words(SEED, pre['idx'], pr.SITE_DEATH, S['t'], 2)
    u = pr.uniform(w, 0)
    if 'death_p' in S:
        p = S['death_p']
        assert np.array_equal(S['alive'].astype(bool), ~(u < p))
        e = so.sample_env(sp['rasters'], pre['x'], pre['y'])
        cx, cy = so.cells(pre['x'], pre['y'])
        fit = so.fitness(e, pre['z'], sp['traits'], cx, cy)
        p_ref = so.death_probs(S['d_rast'], pre['x'], pre['y'], fit, pre['age'], sp['prm']['max_age'])
        np.testing.assert_allclose(p, p_ref, rtol=1e-6, atol=1e-9)
        assert 0 < (~S['alive'].astype(bool)).sum() < len(p)
    new = S['new']
    assert np.array_equal(new['idx'], pre['idx'][S['alive'].astype(bool)])


def check_all(S, pop, sp):
    check_move(S, pop, sp)
    check_mates(S, pop, sp)
    check_births(S, sp)
    check_gametes(S, pop, sp)
    check_dispersal_and_sex(S, sp)
    check_mortality(S, sp)


# ---- populations (the generators of test_cuda_mates.py) --------------------------------------------
def _positions(kind, rng):
    if kind == 'sparse':
        dim, n = (64, 48), 600
        return dim, rng.uniform(0, dim[0] - 0.001, n), rng.uniform(0, dim[1] - 0.001, n), 2.0
    if kind == 'medium':                                 # row ranges of 33-64 candidates
        dim, n = (20, 20), 1400
        return dim, rng.uniform(0, dim[0] - 0.001, n), rng.uniform(0, dim[1] - 0.001, n), 2.0
    if kind == 'crowded':                                # > 2048 candidates in a 3x3 block: k_find_mates_dense
        dim, n = (12, 12), 4200
        return dim, rng.uniform(0, dim[0] - 0.001, n), rng.uniform(0, dim[1] - 0.001, n), 3.5
    dim, n = (48, 40), 9000                              # clumped: both search kernels
    return dim, dim[0] * rng.beta(0.6, 2.5, n) * 0.9999, dim[1] * rng.beta(2.5, 0.6, n) * 0.9999, 2.0


@pytest.mark.parametrize('mode', ['random', 'nearest', 'inverse'])
@pytest.mark.parametrize('popkind', ['sparse', 'medium', 'crowded', 'clumped'])
def test_mate_search_exact(popkind, mode):
    rng = np.random.default_rng(['sparse', 'medium', 'crowded', 'clumped'].index(popkind))
    dim, x, y, radius = _positions(popkind, rng)
    dev, pop, sp = _species(dim, len(x), L=64, b=0.5, mode=mode, radius=radius, xy=(x, y), gseed=3)
    try:
        S = run_stages(dev, pop, finish=False)
    finally:
        dev.close()
    check_move(S, pop, sp)
    pairs = check_mates(S, pop, sp)
    assert len(pairs) > 20
    if popkind == 'crowded':
        assert S['n_nbrs'].max() > 1000


@pytest.mark.parametrize('mode', ['random', 'nearest', 'inverse'])
def test_debug_off_gives_the_same_pair_list(mode):
    """k_mate_select lists only the focals whose Bernoulli(b) draw lets them mate unless debug is on;
    the pair list must not depend on it."""
    rng = np.random.default_rng(11)
    dim, x, y, radius = _positions('clumped', rng)
    got = []
    for debug in (True, False):
        dev, pop, sp = _species(dim, len(x), L=64, b=0.3, mode=mode, radius=radius, xy=(x, y), gseed=4)
        try:
            got.append(run_stages(dev, pop, debug=debug, finish=False)['pairs'])
        finally:
            dev.close()
    assert len(got[0]) > 100
    assert np.array_equal(got[0], got[1])


@pytest.mark.parametrize('id_base', [0, (1 << 32) - 1000])
@pytest.mark.parametrize('sexed,fixed,mode', [(False, True, 'random'), (True, False, 'random'),
                                              (False, False, 'inverse'), (True, True, 'nearest')])
def test_whole_step_stage_by_stage(sexed, fixed, mode, id_base):
    """Movement, mate search, births (fixed, or Poisson with lam = 2), gametes, phenotypes, dispersal,
    sex and mortality of one step.  id_base 2^32 - 1000: the ids cross 2^32 during the step, so the
    counter's high id word and the fifth byte of the species-order radix sort are exercised."""
    rng = np.random.default_rng(5 + sexed + 2 * fixed)
    dim = (30, 30)
    n = 1800
    # a tenth of the population near the lower edges: dispersal tries beyond the first
    x = np.concatenate([rng.uniform(0, dim[0] - 0.001, n - n // 10), rng.uniform(0, 0.6, n // 10)])
    y = np.concatenate([rng.uniform(0, dim[1] - 0.001, n - n // 10), rng.uniform(0, 0.6, n // 10)])
    dev, pop, sp = _species(dim, n, L=300, kind='dom', b=0.8, mode=mode, sexed=sexed, lam=1 if fixed else 2,
                            fixed=fixed, xy=(x, y), id_base=id_base, gseed=7, sex_ratio_p=0.4)
    try:
        S = run_stages(dev, pop)
    finally:
        dev.close()
    check_all(S, pop, sp)
    assert S['disp_tries'].max() > 1
    if id_base:
        assert S['ids'][0] < (1 << 32) <= S['max_idx'] + 1


@pytest.mark.parametrize('sexed,b', [(False, 0.3), (True, 0.8)])
def test_panmixia_exact(sexed, b):
    """mating_radius = None: slot i is entry i, keyed by its id; R0 and R1 pick entries."""
    from oracle import step_oracle as so
    dim, n = (30, 30), 1500
    dev, pop, sp = _species(dim, n, L=64, b=b, radius=None, sexed=sexed, gseed=9)
    try:
        S = run_stages(dev, pop)
    finally:
        dev.close()
    check_move(S, pop, sp)
    perm = S['perm']                                      # entry -> ordinal
    ids_e = S['ids'][perm]
    w = pr.stream_words(SEED, ids_e, pr.SITE_PANMIXIA, S['t'], 4)
    pe = so.find_mates_panmixia_draws(n, b, pr.uniform(w, 0), np.stack([w[:, 2], w[:, 3]], axis=1),
                                      pop['sex'][perm] if sexed else None)
    assert len(pe) > 100
    assert np.array_equal(S['pairs'], perm[pe])
    check_births(S, sp)
    check_gametes(S, pop, sp)
    check_dispersal_and_sex(S, sp)
    check_mortality(S, sp)


def test_fused_steps_equal_the_stages():
    """Several graph-launched steps give, bit for bit, the population that the same stages run one by
    one give, with the same seed."""
    rng = np.random.default_rng(12)
    dim, n = (40, 40), 3000
    x, y = rng.uniform(0, dim[0] - 0.001, n), rng.uniform(0, dim[1] - 0.001, n)
    outs = []
    for fused in (True, False):
        dev, pop, sp = _species(dim, n, L=200, kind='mono', b=0.5, sexed=True, lam=2, fixed=False, xy=(x, y),
                                gseed=12, d_max=0.5)
        try:
            _upload(dev, pop)
            dev.set_draws(None)
            dev.set_debug(False)
            for _ in range(4):
                if fused:
                    dev.step(1)
                else:
                    for s in ('age_step', 'move', 'bin_cells', 'find_mates', 'dedup_pairs', 'make_offspring',
                              'density_counts', 'density_eval', 'death_prob', 'mortality'):
                        dev.stage(s)
            dev.sync()
            if fused:
                assert dev.graph_launch_count >= 3
            outs.append((dev.download(genomes=True), [(r['Nt'], r['n_births'], r['n_deaths'])
                                                      for r in dev.step_records()]))
        finally:
            dev.close()
    (a, ra), (b, rb) = outs
    assert ra == rb and len(ra) == 4 and ra[-1][1] > 100
    for k in ('x', 'y', 'age', 'sex', 'idx', 'fit', 'z', 'genomes'):
        assert np.array_equal(a[k], b[k]), k
    assert a['max_ind_idx'] == b['max_ind_idx']


# ---- the gamete kernel's dispatch table ------------------------------------------------------------------
def gamete_launch(L, n_traits, pair_phenotype):
    """Host mirror of launch_gametes (gnx_api.cu): (GW, NT, stage_rows)."""
    Wq = (L + 127) // 128
    GW = next(g for g in (1, 2, 4, 8, 16, 32) if Wq <= g or g == 32)
    rows_b = (256 // GW) * 2 * Wq * 16
    stage = 1 if (GW > 1 and n_traits > 0 and rows_b <= 32 * 1024) else 0
    nb = min(2, GW)
    if stage and nb >= 2 and nb * rows_b <= 44 * 1024 and pair_phenotype:
        stage = nb
    return GW, (2 if n_traits <= 2 else 8), stage


def _launch_of(L, kind):
    traits, dom = trait_set(L, kind)
    pair = not np.any(dom) and all(len(t['loci']) > 1 for t in traits)
    return gamete_launch(L, len(traits), pair)


def test_gamete_matrix_reaches_every_instantiation_and_mode():
    cases = {_launch_of(L, k) for L in GAMETE_MATRIX_L for k in TRAIT_KINDS}
    assert {gw for gw, _, _ in cases} == {1, 2, 4, 8, 16, 32}
    assert {nt for _, nt, _ in cases} == {2, 8}
    assert {s for gw, _, s in cases if gw > 1} == {0, 1, 2}


@pytest.mark.parametrize('kind', TRAIT_KINDS)
@pytest.mark.parametrize('L', GAMETE_MATRIX_L)
def test_gametes_exact_across_instantiations(L, kind):
    """Gametes and phenotypes of the free-running step for every k_gametes<GW, NT> instantiation and
    phenotype mode; the case names the instantiation it ran, read from a profiler trace."""
    GW, NT, stage = _launch_of(L, kind)
    rng = np.random.default_rng(L)
    dim, n = (30, 30), 1500
    x, y = rng.uniform(0, dim[0] - 0.001, n), rng.uniform(0, dim[1] - 0.001, n)
    # no deaths (d = 0, phi = 0): every newborn's row is downloaded after the step
    dev, pop, sp = _species(dim, n, L=L, kind=kind, b=1.0, xy=(x, y), gseed=L, d_max=0.0, phi=0.0,
                            n_paths=200)
    try:
        S = run_stages(dev, pop, trace_gametes=True)
    finally:
        dev.close()
    name = 'k_gametes<%d, %d>' % (GW, NT)
    assert name in S['kernels'], (name, sorted(k for k in S['kernels'] if 'gamete' in k))
    print('L %d %s: %s stage_rows %d, %d births' % (L, kind, name, stage, S['B']))
    assert S['B'] > 300
    check_gametes(S, pop, sp, expect_all=True)


# ---- full size --------------------------------------------------------------------------------------
def test_full_size_c2():
    """workloads.CONFIGS['c2'] at full size (1,048,576 individuals): mate search, gametes, phenotypes and
    mortality of one free-running step against the restated draws."""
    from geonomics_b200 import workloads, genome_pack
    from geonomics_b200.device import DeviceSpecies
    cfg = dict(workloads.CONFIGS['c2'])
    w = workloads.build(cfg, cfg['seed'])
    n, L = cfg['N'], w['L']
    g = genome_pack.unpack_genomes(workloads.random_packed_genomes(n, L, cfg['seed'] + 1), L)
    pw = w['prm']
    traits = w['gen_arch']['traits']
    prm = dict(b=pw['b'], R=pw['R'], lam=1, n_births_fixed=True, mating_radius=2.0, d_min=0.0, d_max=1.0,
               sex=False, sex_ratio_p=0.5, max_age=None, K_layer=0, K_factor=pw['K_factor'], move=True,
               move_distr=DIST, disp_distr=DIST, direction_mu=0.0, direction_kappa=0.0)
    dev = DeviceSpecies(w['land_dim'], w['rasters'], prm, dict(L=L, paths=w['gen_arch']['paths'], traits=traits),
                        capacity=int(1.5 * n), seed=SEED)
    pop = dict(x=w['pop']['x'], y=w['pop']['y'], age=w['pop']['age'], sex=w['pop']['sex'], idx=w['pop']['idx'], g=g)
    sp = dict(dim=w['land_dim'], L=L, traits=traits, dom=np.zeros(L, np.int8), paths=w['gen_arch']['paths'],
              rasters=w['rasters'], prm=prm, mode='random')
    try:
        dev.gen_arch = dict(dev.gen_arch, dom=sp['dom'])
        S = run_stages(dev, pop)
    finally:
        dev.close()
    assert S['n0'] == n and S['B'] > 150000
    check_mates(S, pop, sp)
    check_gametes(S, pop, sp)
    check_mortality(S, sp)
