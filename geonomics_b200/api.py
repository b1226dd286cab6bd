"""Host-side mirror of the Geonomics API for the accelerated path.

Same names, argument meaning and attributes as the reference (erthward/geonomics v1.4.9;
`file:line` below are relative to /root/reference/geonomics/): the parameters file
(`sim/params.py`), `read_parameters_file` (`main.py:308`), `make_model` (`main.py:442`),
`Model.walk` / `Model.run` (`sim/model.py:966,866`), `Landscape`/`Layer`
(`structs/landscape.py`), `Community` (`structs/community.py`), `Species`
(`structs/species.py`), `Individual` (`structs/individual.py`), `GenomicArchitecture`,
`Trait`, `Recombinations` (`structs/genome.py`).

What changes is where the state lives and who advances it: individuals are
structure-of-arrays device buffers owned by a `DeviceSpecies`, and one queue pass
(`sim/model.py:603-667`) is one `gnx_step` of libgnxb200.so.  `Species` remains a mapping
of ids to `Individual` objects, materialised lazily from the device when someone looks.

Setup code here (layers, genomic architecture, starting genotypes, conductance tables,
burn-in control) runs on the host with numpy, as it does in the reference; it is not on the
per-timestep path (SURVEY.md section 2, "setup").  There is no CPU implementation of the
time step itself: stepping a Model without libgnxb200.so / a CUDA device raises.
"""
import copy
import os
import warnings
from collections import OrderedDict

import numpy as np

from . import genome_pack as gp
from .device import DeviceSpecies, growth_capacity


# ---------------------------------------------------------------------------------------------
# parameters (sim/params.py:713-760, 1127-1143)
# ---------------------------------------------------------------------------------------------
class ParametersDict(dict):
    """Nested dict with attribute access (`params.model.T`), like params.py:730."""

    def __init__(self, d=None):
        super().__init__()
        for k, v in (d or {}).items():
            self[k] = ParametersDict(v) if isinstance(v, dict) and not isinstance(v, ParametersDict) else v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)

    def __setattr__(self, k, v):
        self[k] = v

    def __deepcopy__(self, memo):
        return ParametersDict(copy.deepcopy(dict(self), memo))


def read_parameters_file(filepath):
    """main.py:308 / params.py:1127-1143: a parameters file is Python source defining `params`."""
    ns = {'np': np}
    with open(filepath) as f:
        exec(compile(f.read(), filepath, 'exec'), ns)
    p = ParametersDict(ns['params'])
    name = os.path.splitext(os.path.basename(filepath))[0]
    p.setdefault('model', ParametersDict())
    p['model']['name'] = name
    return p


def make_params_dict(params, model_name='unnamed_model'):
    """main.py:403."""
    p = ParametersDict(params)
    p.setdefault('model', ParametersDict())
    p['model'].setdefault('name', model_name)
    return p


# ---------------------------------------------------------------------------------------------
# landscape (structs/landscape.py)
# ---------------------------------------------------------------------------------------------
class Layer:
    """landscape.py:34: a 2-D raster in [0, 1] plus georeferencing."""

    def __init__(self, rast, lyr_type, name, dim, res=(1, 1), ulc=(0, 0), prj=None, idx=None):
        self.idx = idx
        self.type = lyr_type
        self.name = str(name)
        self.dim = tuple(dim)
        self.res = res
        self.ulc = ulc
        self.prj = prj
        self.rast = np.array(rast, dtype=np.float64)
        assert self.rast.shape == (self.dim[1], self.dim[0]), (
            'Layer raster must have shape (dim_y, dim_x) = %s, got %s' % ((self.dim[1], self.dim[0]),
                                                                          self.rast.shape))
        self._is_K = []


def _scattered_values_to_raster(dim, pts, vals, method, num_hab_types):
    """Seed values at scattered points -> a [dim_y, dim_x] raster: scipy griddata on the integer lattice
    1..max(dim) of a square, 'nearest' results rounded to habitat classes, 'cubic' results shifted and
    scaled into (0, 1) with two small uniform jitters (drawn in that order), cropped to the layer."""
    from scipy.interpolate import griddata
    side = max(dim)
    axis = np.linspace(1, side, side)
    field = griddata(pts, vals * (num_hab_types - 1) if method == 'nearest' else vals,
                     tuple(np.meshgrid(axis, axis, indexing='ij')), method=method)
    if method == 'nearest':
        field = np.rint(field).astype(float)
    elif method == 'cubic':
        field = field + abs(field.min()) + 0.01 * np.random.rand()
        field = field / (field.max() + 0.01 * np.random.rand())
    return field[:dim[1], :dim[0]]


def _make_random_lyr(dim, n_pts, interp_method='cubic', num_hab_types=2, dist='beta', alpha=0.05, beta=0.05):
    """landscape.py:411-470 ('random' layers): values first, then the seed points -- the reference's
    draw order, so a seeded numpy.random gives the reference's layer."""
    vals = np.random.rand(n_pts) if dist == 'unif' else np.random.beta(alpha, beta, n_pts)
    pts = np.random.normal(max(dim) / 2, max(dim) * 2, [n_pts, 2])
    return _scattered_values_to_raster(dim, pts, vals, interp_method, num_hab_types)


def _make_defined_lyr(dim, rast, pts=None, vals=None, interp_method='cubic', num_hab_types=2):
    """landscape.py:473-519 ('defined' layers): a raster as given, or interpolated from points."""
    if rast is not None:
        return np.array(rast, dtype=np.float64)
    return _scattered_values_to_raster(dim, np.asarray(pts), np.asarray(vals, dtype=np.float64), interp_method,
                                       num_hab_types)


class _LandscapeChanger:
    """ops/change.py:103-152, 302-357: scheduled, linearly interpolated raster series."""

    def __init__(self, land, change_params):
        changes = []
        for lyr_num, events in change_params.items():
            start_rast = land[lyr_num].rast
            for _, ev in sorted(events.items()):
                change_rast = np.array(ev['change_rast'], dtype=np.float64)
                n_steps = int(ev['n_steps'])
                timesteps = np.int64(np.round(np.linspace(ev['start_t'], ev['end_t'], n_steps)))
                # linspace(start, end, n_steps + 1)[1:] per cell (change.py:349-354)
                for k, t in enumerate(timesteps):
                    # numpy.linspace arithmetic, per cell: y_k = k * ((b - a) / n) + a, last = b
                    rast = (k + 1) * ((change_rast - start_rast) / float(n_steps)) + start_rast
                    if k == n_steps - 1:
                        rast = change_rast.copy()
                    changes.append((int(t), lyr_num, rast))
                start_rast = change_rast
        self.changes = sorted(changes, key=lambda c: c[0])
        self.change_info = {k: dict(v) for k, v in change_params.items()}
        self._pos = 0

    def _make_change(self, t, land):
        made = False
        while self._pos < len(self.changes) and self.changes[self._pos][0] == t:
            _, lyr_num, rast = self.changes[self._pos]
            land._set_raster(lyr_num, rast)
            self._pos += 1
            made = True
        return made


class _SpeciesChanger:
    """ops/change.py:155-267 (_SpeciesChanger) with the change functions of change.py:612-742:
    demographic events rewrite the carrying-capacity raster (`spp.K *= size` for 'monotonic',
    `spp.K = base_K * size` for 'stochastic' / 'cyclical' / 'custom', where base_K is spp.K at
    the event's first time step), life-history events `setattr(spp, parameter, val)`.  Conductance
    surfaces that follow a changing layer (change.py:576-606) are re-built when the layer's raster
    is swapped (Species._on_raster_change), at the same time steps as the reference's series."""

    def __init__(self, spp, change_params, land):
        self.base_K = None
        changes = []
        cp = change_params or {}
        for _, ev in sorted((cp.get('dem') or {}).items(), key=lambda kv: str(kv[0])):
            if not any(v is not None for v in dict(ev).values()):
                continue
            changes.extend(self._dem_changes(**dict(ev)))
        for parameter, pp in (cp.get('life_hist') or {}).items():
            pp = dict(pp)
            if not any(v is not None for v in pp.values()):
                continue
            ts, vals = list(pp['timesteps']), list(pp['vals'])
            assert len(ts) == len(vals), ("For custom changes of the '%s' parameter, timesteps and vals "
                                          "must be iterables of equal length.") % parameter
            changes.extend((int(t), 'param', (parameter, v)) for t, v in zip(ts, vals))
        self.changes = sorted(changes, key=lambda c: c[0])          # stable, like the reference's sort
        self._pos = 0

    # change.py:612-731
    @staticmethod
    def _dem_changes(kind, start_t=None, end_t=None, rate=None, interval=None, n_cycles=None, size_range=None,
                     distr='uniform', min_size=None, max_size=None, timesteps=None, sizes=None,
                     increase_first=True):
        if kind == 'monotonic':                                     # change.py:652-661
            ts = list(range(start_t, end_t + 1))
            return [(t, 'K_current', float(rate)) for t in ts]
        if kind == 'stochastic':                                    # change.py:669-688
            ts = list(range(start_t, end_t + 1, 1 if interval is None else interval))
            if distr == 'uniform':
                sz = np.random.uniform(*size_range, len(ts))
            elif distr == 'normal':
                sz = np.random.normal(loc=np.mean(size_range), scale=(size_range[1] - size_range[0]) / 6,
                                      size=len(ts))
            else:
                raise ValueError("Argument 'distr' must be a value among ['uniform', 'normal']")
            sz[-1] = 1
        elif kind == 'cyclical':                                    # change.py:691-731
            if size_range is not None and min_size is None and max_size is None:
                min_size, max_size = size_range
            elif not (size_range is None and min_size is not None and max_size is not None):
                raise ValueError('Must either provide size_range (as a tuple of minimum and maximum sizes), or '
                                 'provide min_size and max_size separately, but not both.')
            assert n_cycles <= (end_t - start_t) / 2
            base = np.sin(np.linspace(0, 2 * np.pi, 1000))
            if not increase_first:
                base = base[::-1]
            sb = np.array([1 + v * (max_size - 1) if v >= 0 else v for v in base])
            sb = np.array([1 + v * (1 - min_size) if v < 0 else v for v in sb])
            cyc_t = np.int32(np.linspace(start_t, end_t, n_cycles + 1))
            sz = np.hstack([sb[np.int32(np.linspace(1, len(sb) - 1, ln))] for ln in np.diff(cyc_t)] + [1])
            ts = list(range(cyc_t[0], cyc_t[-1] + 1))
        elif kind == 'custom':                                      # change.py:734-738
            assert len(timesteps) == len(sizes)
            ts, sz = list(timesteps), list(sizes)
        else:
            raise ValueError("unknown demographic change kind '%s'" % kind)
        t0 = int(ts[0])
        return [(int(t), 'K_base', (float(v), t0)) for t, v in zip(ts, sz)]

    def _next_t(self):
        return self.changes[self._pos][0] if self._pos < len(self.changes) else None

    def _make_change(self, t, spp):
        """change.py:56-84: every change scheduled for time step t, in order."""
        while self._pos < len(self.changes) and self.changes[self._pos][0] == t:
            _, kind, payload = self.changes[self._pos]
            self._pos += 1
            if kind == 'K_current':
                spp._override_K(spp.K * payload)                    # change.py:636-638
            elif kind == 'K_base':
                size, t0 = payload
                if spp.t == t0:
                    self.base_K = spp.K                             # change.py:642-644
                spp._override_K(self.base_K * size)
            else:
                spp._set_parameter(*payload)                        # change.py:737-738


class Landscape(dict):
    """landscape.py:199: dict of Layers keyed by layer number."""

    def __init__(self, lyrs, res=(1, 1), ulc=(0, 0), prj=None):
        super().__init__(lyrs)
        first = next(iter(lyrs.values()))
        self.dim = first.dim
        self.res = res
        self.ulc = ulc
        self.prj = prj
        # landscape.py:277-278: each axis' cell size relative to the larger one
        self._res_ratio = tuple(float(abs(v / max(res))) for v in res)
        self._dim_om = len(str(max(self.dim)))
        self._changer = None
        self._listeners = []        # attached Species (device raster mirrors)
        for n, lyr in self.items():
            lyr.idx = n

    def _set_raster(self, lyr_num, rast):
        """landscape.py:353-354 (+ the device mirror; Species._set_K for the K layer)."""
        self[lyr_num].rast = np.array(rast, dtype=np.float64)
        for spp in self._listeners:
            spp._on_raster_change(lyr_num, self[lyr_num].rast)

    def _make_change(self, t, verbose=False):
        if self._changer is not None:
            self._changer._make_change(t, self)


def _make_landscape(params, num_hab_types=2):
    """landscape.py:522-674 ('random' and 'defined' layers; 'file'/'nlmpy' need rasterio /
    nlmpy, which this image lacks -> they raise)."""
    main = params.landscape.main
    dim = tuple(main.dim)
    res = tuple(main.res) if main.get('res') is not None else (1, 1)
    ulc = tuple(main.ulc) if main.get('ulc') is not None else (0, 0)
    prj = main.get('prj')
    lyrs = {}
    for n, (name, lp) in enumerate(params.landscape.layers.items()):
        init = lp['init']
        keys = list(init.keys())
        if len(keys) != 1:
            raise ValueError("Layer '%s' must have parameters for exactly one layer type" % name)
        lyr_type = keys[0]
        if lyr_type == 'random':
            rast = _make_random_lyr(dim, num_hab_types=num_hab_types, **dict(init[lyr_type]))
        elif lyr_type == 'defined':
            rast = _make_defined_lyr(dim, num_hab_types=num_hab_types, **dict(init[lyr_type]))
        else:
            raise NotImplementedError("layer type '%s' needs rasterio/nlmpy, not available here" % lyr_type)
        rast = np.clip(rast, 0, 1)                              # landscape.py:646-648
        lyrs[n] = Layer(rast, lyr_type, name, dim, res, ulc, prj, idx=n)
    land = Landscape(lyrs, res=res, ulc=ulc, prj=prj)
    change_params = {}
    for n, (name, lp) in enumerate(params.landscape.layers.items()):
        if 'change' in lp:
            change_params[n] = lp['change']
    if change_params:
        land._changer = _LandscapeChanger(land, change_params)
    return land


# ---------------------------------------------------------------------------------------------
# genomic architecture (structs/genome.py)
# ---------------------------------------------------------------------------------------------
class Recombinations:
    """genome.py:47-281: cache of `n` pre-simulated recombination events.  The reference
    stores each as a bitarray 'subsetter' of '10'/'01' units per locus; here only the
    homologue bit per locus is kept (`_paths`, uint8[n, L])."""

    def __init__(self, L, positions, n, r_distr_alpha, r_distr_beta, recomb_rates, jitter_breakpoints=False):
        self._L = L
        self._positions = np.arange(L) if positions is None else np.sort(np.array(positions))
        self._n = n
        self._r_distr_alpha = r_distr_alpha
        self._r_distr_beta = r_distr_beta
        self._jitter_breakpoints = jitter_breakpoints
        if recomb_rates is not None:
            assert len(recomb_rates) == len(self._positions)
            assert recomb_rates[0] == 0
            self._rates = np.array(recomb_rates, dtype=np.float64)
        else:
            self._rates = self._draw_recombination_rates()
        self._paths = None
        self._breakpoints = None

    def _draw_recombination_rates(self):
        """genome.py:163-185."""
        n = len(self._positions)
        if self._r_distr_alpha is not None and self._r_distr_beta is not None:
            rates = np.clip(np.random.beta(a=self._r_distr_alpha, b=self._r_distr_beta, size=n), 0, 0.5)
        elif self._r_distr_alpha is not None:
            rates = np.ones(n) * self._r_distr_alpha
        else:
            rates = np.ones(n) * (1 / self._L)
        rates[0] = 0
        return rates

    def _set_events(self):
        """genome.py:188-230: n x binomial(1, rates); path = cumsum % 2."""
        ev = np.random.random((self._n, len(self._rates))) < self._rates[None, :]
        self._breakpoints = {k: self._positions[np.where(e)] for k, e in enumerate(ev)}
        self._paths = (np.cumsum(ev, axis=1) % 2).astype(np.uint8)

    def _get_subsetter(self, event_key):
        """The reference's '10'/'01' bit pattern for one event, as a bool array of length 2L."""
        p = self._paths[event_key]
        out = np.zeros(2 * len(p), dtype=bool)
        out[0::2] = p == 0
        out[1::2] = p == 1
        return out


class Trait:
    """genome.py:284-437."""

    def __init__(self, idx, name, phi, n_loci, mu, layer, alpha_distr_mu, alpha_distr_sigma, max_alpha_mag,
                 gamma, univ_adv):
        self.idx = idx
        self.name = name
        self.phi = phi
        self.n_loci = n_loci
        self.mu = 0 if mu is None else mu
        self.lyr_num = layer
        self.alpha_distr_mu = alpha_distr_mu
        self.alpha_distr_sigma = alpha_distr_sigma
        self.max_alpha_mag = max_alpha_mag
        self.gamma = gamma
        self.univ_adv = univ_adv
        self.loci = np.int64([])
        self.loci_idxs = None
        self.alpha = np.array([])

    def _set_loci_idxs(self, nonneut_loci, use_tskit):
        """genome.py:405-414: rows of the trait's loci in the (non-neutral-only) genotype arrays."""
        if use_tskit:
            self.loci_idxs = np.array([np.where(nonneut_loci == n)[0][0] for n in self.loci], dtype=np.int64)
        else:
            self.loci_idxs = None

    def _get_phi(self, spp):
        if type(self.phi) in (float, int):
            return np.array([self.phi] * len(spp))
        return self.phi[spp._cells[:, 1], spp._cells[:, 0]]


class MutationRateError(Exception):
    """genome.py:36-37."""


class GenomicArchitecture:
    """genome.py:440-810."""

    def __init__(self, dom, g_params, land, recomb_rates=None, recomb_positions=None):
        self.x = 2
        self.L = g_params.L
        self.p = None
        self.pleiotropy = g_params.get('pleiotropy', False)
        self.dom = dom
        self._use_dom = bool(np.any(self.dom))
        self.sex = g_params.get('sex', False)
        self.use_tskit = bool(g_params.get('use_tskit', False))
        self.tskit_simp_interval = g_params.get('tskit_simp_interval', 100)
        self.mu_neut = g_params.get('mu_neut', 0)
        self.mu_delet = g_params.get('mu_delet', 0)
        self.delet_alpha_distr_shape = g_params.get('delet_alpha_distr_shape', 0.2)
        self.delet_alpha_distr_scale = g_params.get('delet_alpha_distr_scale', 0.2)
        self.neut_loci = np.array(range(self.L))
        self.nonneut_loci = np.array([])
        self.delet_loci = np.int64([])
        self.delet_loci_idxs = np.int64([]) if self.use_tskit else None     # genome.py:590-594
        self.delet_loci_s = np.array([])
        self.traits = None
        if 'traits' in g_params and g_params['traits']:
            self.traits = _make_traits(g_params.traits, land)
        mus = [m for m in (self.mu_neut, self.mu_delet) if m is not None]
        if self.traits is not None:
            mus = mus + [t.mu for t in self.traits.values()]
        self._mu_tot = sum(mus)
        self._mu_nonneut = self._mu_tot - (self.mu_neut or 0)
        self._mutables = None
        self.recombinations = Recombinations(self.L, recomb_positions, g_params.get('n_recomb_sims', 10000),
                                             g_params.get('r_distr_alpha'), g_params.get('r_distr_beta'),
                                             recomb_rates, g_params.get('jitter_breakpoints', False))

    def _draw_trait_alpha(self, trait_num, n=1):
        """genome.py:666-687."""
        trt = self.traits[trait_num]
        if trt.alpha_distr_sigma == 0:
            alpha = trt.alpha_distr_mu * np.array([1 - (i % 2) * 2 for i in range(n)])
        else:
            alpha = np.random.normal(trt.alpha_distr_mu, trt.alpha_distr_sigma, n)
            if trt.max_alpha_mag is not None:
                alpha = np.clip(alpha, -trt.max_alpha_mag, trt.max_alpha_mag)
        if trt.n_loci == 1:
            alpha = np.abs(alpha)
        return alpha

    def _set_trait_loci(self, trait_num, loci=None, alpha=None):
        """genome.py:696-750 (initial assignment)."""
        n = self.traits[trait_num].n_loci
        assert n <= self.L
        if loci is None:
            pool = self.neut_loci if not self.pleiotropy else np.arange(self.L)
            loci = set(np.random.choice(pool, size=n, replace=False))
        trt = self.traits[trait_num]
        trt.loci = np.sort(np.hstack((trt.loci, np.array([*loci])))).astype(np.int64)
        trt.n_loci = trt.loci.size
        self.nonneut_loci = np.array(sorted([*self.nonneut_loci] + [*loci]))
        self.neut_loci = np.array(sorted(set(self.neut_loci).difference(set(self.nonneut_loci))))
        effects = np.array([*np.atleast_1d(alpha)]) if alpha is not None else self._draw_trait_alpha(trait_num, n)
        if n == 1:
            effects = np.array([0.5])
        assert len(loci) == len(effects)
        trt.alpha = np.hstack((trt.alpha, effects))


def _make_traits(traits_params, land):
    """genome.py:826-867."""
    traits = {}
    for n, (name, v) in enumerate(traits_params.items()):
        v = dict(v)
        layer = v.pop('layer')
        if isinstance(layer, str):
            nums = [num for num, lyr in land.items() if lyr.name == layer]
        else:
            nums = [num for num, lyr in land.items() if lyr.idx == layer]
        assert len(nums) == 1, 'Expected a single Layer named %s for Trait %s' % (layer, name)
        traits[n] = Trait(n, name, layer=nums[0], **v)
        if traits[n].n_loci == 1 and traits[n].mu != 0:
            warnings.warn("Coercing Trait %i ('%s') to a 0 mutation rate because it is monogenic." % (n, name))
            traits[n].mu = 0
    return traits


def _make_genomic_architecture(spp_params, land):
    """genome.py:870-1062 (no custom CSV file in this build)."""
    g_params = spp_params.gen_arch
    if g_params.get('gen_arch_file') is not None:
        import pandas as pd
        gaf = pd.read_csv(g_params.gen_arch_file)
        assert len(gaf) == g_params.L
    else:
        gaf = None
    g_params['sex'] = spp_params.mating.sex
    recomb_rates = recomb_positions = None
    if gaf is not None:
        recomb_rates = gaf['r'].values
        recomb_positions = gaf['locus'].values
        dom = gaf['dom'].values
    else:
        dom = np.array([int(g_params.dom)] * g_params.L)
    ga = GenomicArchitecture(dom, g_params, land, recomb_rates, recomb_positions)
    if ga.traits is not None:
        if gaf is not None:
            names = {t.name: n for n, t in ga.traits.items()}
            tcol = [[names[v.strip()] for v in str(row).split(',') if v.strip() in names] for row in gaf['trait']]
            acol = [[float(a) for a in str(row).split(',')] if str(row) != 'nan' else [] for row in gaf['alpha']]
            for tn in ga.traits:
                loci = np.array([l for l, ts in zip(gaf['locus'], tcol) if tn in ts])
                alphas = np.array([a[ts.index(tn)] for ts, a in zip(tcol, acol) if tn in ts])
                ga._set_trait_loci(tn, loci=loci, alpha=alphas)
        else:
            for tn in ga.traits:
                ga._set_trait_loci(tn)
    if gaf is None:
        spf = g_params.get('start_p_fixed')
        if spf is not None:
            if isinstance(spf, bool):
                ga.p = np.array([0.5] * g_params.L) if spf else np.random.beta(1, 1, g_params.L)
            else:
                assert 0 <= spf <= 1
                ga.p = np.array([spf] * g_params.L, dtype=np.float64)
        else:
            ga.p = np.random.beta(1, 1, g_params.L)
        if g_params.get('start_neut_zero') and len(ga.neut_loci) > 0:
            ga.p[ga.neut_loci] = 0
    else:
        ga.p = gaf['p'].values
    ga.recombinations._set_events()
    if ga.traits is not None:                                  # genome.py:1044-1047
        for trt in ga.traits.values():
            trt._set_loci_idxs(ga.nonneut_loci, ga.use_tskit)
    return ga


# ---------------------------------------------------------------------------------------------
# conductance surfaces (utils/spatial.py:149-184, 365-461) -- table mode, built on the host
# ---------------------------------------------------------------------------------------------
class _ConductanceSurface:
    def __init__(self, cond_lyr, mixture=True, approx_len=5000, vm_distr_kappa=12):
        self.dim = cond_lyr.dim
        self.mix = mixture
        self.lyr_num = cond_lyr.idx
        self.approx_len = 5000 if approx_len is None else approx_len
        self.kappa = 12 if vm_distr_kappa is None else vm_distr_kappa
        self.surf = _make_conductance_surface(cond_lyr.rast, self.mix, self.approx_len, self.kappa)


def _make_conductance_surface(rast, mixture=True, approx_len=5000, vm_distr_kappa=12):
    """spatial.py:432-461 (vectorised over cells; same distributions)."""
    pi = np.pi
    dirs = np.array([-3 * pi / 4, -pi / 2, -pi / 4, pi, 0, 3 * pi / 4, pi / 2, pi / 4])
    Y, X = rast.shape
    emb = np.zeros((Y + 2, X + 2))
    emb[1:-1, 1:-1] = rast
    offs = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)]
    neigh = np.stack([emb[1 + di:1 + di + Y, 1 + dj:1 + dj + X] for di, dj in offs], axis=-1)   # [Y, X, 8]
    if mixture:
        s = neigh.sum(axis=-1, keepdims=True)
        probs = np.where(s > 0, neigh / np.where(s > 0, s, 1), 0.125)
        cdf = np.cumsum(probs, axis=-1)
        u = np.random.random((Y, X, approx_len))
        pick = (u[..., None] >= cdf[:, :, None, :]).sum(axis=-1).clip(max=7)
        loc = dirs[pick]
    else:
        mx = neigh.max(axis=-1, keepdims=True)
        is_max = neigh == mx
        loc = ((is_max * dirs).sum(axis=-1) / is_max.sum(axis=-1))[..., None] * np.ones((1, 1, approx_len))
    # scipy.stats.vonmises.rvs(kappa, loc=loc) wraps onto [-pi, pi) (scipy >= 1.11)
    surf = np.mod(loc + np.random.vonmises(0, vm_distr_kappa, size=(Y, X, approx_len)) + pi, 2 * pi) - pi
    return np.float16(surf)


# ---------------------------------------------------------------------------------------------
# individuals and species (structs/individual.py, structs/species.py)
# ---------------------------------------------------------------------------------------------
class Individual:
    """individual.py:26: a *view* of one individual's current state."""
    __slots__ = ('idx', 'x', 'y', 'age', 'sex', 'e', 'z', 'fit', 'g', '_individuals_tab_id', '_nodes_tab_ids')

    def __init__(self, idx, x, y, age=0, new_genome=None, sex=None, e=None, z=None, fit=None):
        self.idx = idx
        self.g = new_genome
        self.x = float(x)
        self.y = float(y)
        self.sex = sex
        self.age = age
        self.e = e
        self.z = [] if z is None else z
        self.fit = fit
        self._individuals_tab_id = None
        self._nodes_tab_ids = {}


class _ParamsVals:
    def __init__(self, spp_name):
        self.spp_name = spp_name


class Species:
    """species.py:77.  Mapping of individual id -> Individual (species order), backed by a
    DeviceSpecies.  Parameter attributes (`spp.b`, `spp.mating_radius`, ...) resolve through
    `_pv` like the reference (species.py:71-74, 405-425)."""

    def __init__(self, name, idx, land, spp_params, genomic_architecture=None, N=0, seed=0, strips=None):
        self.idx = idx
        self.name = str(name)
        self._land = land
        self._land_dim = land.dim
        self._land_res = land.res
        self._land_res_ratio = land._res_ratio
        self.t = -1
        self.burned = False
        self.extinct = False
        self.start_N = N
        self.max_ind_idx = N - 1
        self.N = None
        self.K = None
        self.K_layer = None
        self.K_factor = None
        self.Nt = []
        self.n_births = []
        self.n_deaths = []
        self._move = False
        self._move_surf = None
        self._disp_surf = None
        self._changer = None
        self.sex_ratio = 0.5                      # species.py:399 (shadows the parameter, as there)
        self._pv = _ParamsVals(self.name)
        for section in ('mating', 'mortality', 'movement'):
            if section in spp_params:
                for att, val in spp_params[section].items():
                    if not isinstance(val, dict):
                        if att == 'sex_ratio':
                            val = val / (val + 1)
                        setattr(self._pv, att, val)
                if section == 'movement' and spp_params[section].move:
                    self._move = True
        self.gen_arch = genomic_architecture
        self.selection = (self.gen_arch is not None and
                          ((self.gen_arch.mu_delet or 0) > 0 or self.gen_arch.traits is not None))
        self.mutate = (self.gen_arch is not None and self.gen_arch._mu_tot is not None and
                       self.gen_arch._mu_tot > 0)
        self.mut_log = None
        if 'gen_arch' in spp_params and spp_params['gen_arch'].get('mut_log'):
            self.mut_log = spp_params['gen_arch']['mut_log']
            if self.mut_log is True:
                self.mut_log = '%s_mutations.log' % name
        self.mutations = []                    # drained device mutation log (dict rows)
        self._seed = seed
        self._strips = strips                  # None, a strip count or a process group (strips.LocalStrips, NcclStrips)
        self._tc = None                        # tskit tables as numpy columns (tables.TableColumns), use_tskit only
        self._dev = None
        self._cache = None                     # host copy of the device state (lazy)
        self._inds = None                      # OrderedDict of Individual views (lazy)
        self._init_pop = None

    def __getattr__(self, attr):
        pv = self.__dict__.get('_pv')
        if pv is not None and hasattr(pv, attr):
            return getattr(pv, attr)
        raise AttributeError("Species has no attribute '%s'" % attr)

    # ---- device attachment --------------------------------------------------------------
    def _device_params(self):
        prm = dict(b=self.b, R=self.R, lam=self.n_births_distr_lambda, n_births_fixed=self.n_births_fixed,
                   mating_radius=self.mating_radius, d_min=self.d_min, d_max=self.d_max, sex=self.sex,
                   sex_ratio_p=self.sex_ratio, max_age=self.max_age, K_layer=self.K_layer,
                   K_factor=self.K_factor, move=self._move,
                   choose_nearest=self.choose_nearest_mate, inverse_dist=self.inverse_dist_mating,
                   density_grid_window_width=self.density_grid_window_width)
        if self._move:
            prm['move_distr'] = (self.movement_distance_distr, self.movement_distance_distr_param1,
                                 self.movement_distance_distr_param2)
            prm['direction_mu'] = self.direction_distr_mu
            prm['direction_kappa'] = self.direction_distr_kappa
        prm['disp_distr'] = (self.dispersal_distance_distr, self.dispersal_distance_distr_param1,
                             self.dispersal_distance_distr_param2)
        for nm, surf in (('move_surf', self._move_surf), ('disp_surf', self._disp_surf)):
            if surf is not None:
                prm[nm] = dict(table=surf.surf, layer=surf.lyr_num, mixture=surf.mix, kappa=surf.kappa)
        return prm

    def _attach(self, capacity=None, cols=None):
        """cols: (col_locus, col_capacity) of the column layout to continue from (a snapshot's); a use_tskit
        species otherwise starts its columns at the ascending non-neutral loci."""
        land = self._land
        rasters = np.stack([land[l].rast for l in range(len(land))])
        ga = None
        if self.gen_arch is not None:
            traits = []
            for t in (self.gen_arch.traits or {}).values():
                traits.append(dict(loci=t.loci, alpha=t.alpha, phi=t.phi, gamma=t.gamma, lyr_num=t.lyr_num,
                                   univ_adv=t.univ_adv))
            ga = dict(L=self.gen_arch.L, paths=self.gen_arch.recombinations._paths, traits=traits,
                      dom=np.asarray(self.gen_arch.dom, dtype=np.int8))
            if self.gen_arch.use_tskit:
                # species.py:891-905: genotype rows carry the non-neutral loci only; so do the device's (gnx_create_cols)
                if cols is None:
                    cols = (np.sort(np.asarray(self.gen_arch.nonneut_loci, dtype=np.int64)), None)
                ga['cols'], ga['col_capacity'] = cols
        p = self._init_pop
        if self._strips is not None:
            from .strips import LocalStrips, NcclStrips
            kw = dict(seed=self._seed, res_ratio=self._land_res_ratio, K=self.K, start_y=p['y'])
            if isinstance(self._strips, (int, np.integer)):
                self._dev = LocalStrips(self._strips, land.dim, rasters, self._device_params(), ga, capacity, **kw)
            else:
                self._dev = NcclStrips(land.dim, rasters, self._device_params(), ga, capacity, group=self._strips, **kw)
        else:
            if capacity is None:
                capacity = int(max(4096, 3.0 * float(np.sum(self.K)), 2 * max(self.start_N, len(p['x']))))
            # the population may outgrow the starting capacity (a K raised by a landscape or demographic
            # change, a high lambda): the buffers grow between steps
            self._dev = DeviceSpecies(land.dim, rasters, self._device_params(), ga, capacity=capacity,
                                      seed=self._seed, res_ratio=self._land_res_ratio, grow=True)
        land._listeners.append(self)
        self._dev.set_burn(not self.burned)
        self._upload(p)
        self._init_pop = None
        self._invalidate()
        self._burnin_spat_tester = None
        self._burnin_base = None
        if not self.burned:                                   # species.py:469-470
            from .burnin import SpatialTester
            self._burnin_spat_tester = SpatialTester(self._dev)
            self._burnin_base = (p['x'], p['y'])              # the device compares the next update with these counts

    def _upload(self, p):
        self._dev.upload(p['x'], p['y'], p['age'], p['sex'], p['idx'], max_ind_idx=self.max_ind_idx,
                         genomes_packed=p.get('genomes'), z=p.get('z'), fit=p.get('fit'))

    def _do_spatial_burnin_test(self, num_timesteps_back):
        """species.py:572-578."""
        if self._burnin_spat_tester is None:
            from .burnin import SpatialTester
            self._burnin_spat_tester = SpatialTester(self._dev)
        self._burnin_spat_tester.update(self._dev)
        self._burnin_base = None
        return self._burnin_spat_tester.run_test(num_timesteps_back)

    def _detach(self):
        if self._dev is not None:
            if self in self._land._listeners:
                self._land._listeners.remove(self)
            self._dev.close()
            self._dev = None

    # ---- iterations (model.py:455-506): the reference deep-copies the burned-in Community; here
    # the population lives on the device, so the copy is a download and the reset an upload
    def _snapshot(self):
        st = self._dev.download(genomes=bool(self.burned and self.gen_arch is not None), unpack=False)
        keep = ('Nt', 'n_births', 'n_deaths', 't', 'burned', 'extinct', 'max_ind_idx', 'start_N', 'mutate', 'K_factor')
        snap = {k: copy.deepcopy(getattr(self, k)) for k in keep}
        snap.update(state=st, K=np.array(self.K), gen_arch=copy.deepcopy(self.gen_arch),
                    changer=copy.deepcopy(self._changer), pv=copy.deepcopy(self._pv),
                    inst={k: copy.deepcopy(v) for k, v in self.__dict__.items()
                          if hasattr(self._pv, k) and not k.startswith('_')},        # life-history overrides
                    capacity=self._dev.capacity)
        if getattr(self._dev, 'cols', False):
            snap['cols'] = (self._dev.read_cols(), self._dev.col_capacity)
        return snap

    def _restore(self, snap, land, gen_arch=None):
        """Back to a snapshot (on `land`); with `gen_arch` the genomic architecture is replaced and
        the genomes are left for _set_genomes_and_tables (rand_genarch, model.py:476-494)."""
        self._detach()
        for k in ('Nt', 'n_births', 'n_deaths', 't', 'burned', 'extinct', 'max_ind_idx', 'start_N', 'mutate',
                  'K_factor'):
            setattr(self, k, copy.deepcopy(snap[k]))
        for k in [k for k in self.__dict__ if hasattr(self._pv, k) and not k.startswith('_')]:
            del self.__dict__[k]
        self._pv = copy.deepcopy(snap['pv'])
        for k, v in snap['inst'].items():
            setattr(self, k, copy.deepcopy(v))
        self._changer = copy.deepcopy(snap['changer'])
        self._land = land
        self.K = np.array(snap['K'])
        self._K_overridden = False
        self.gen_arch = copy.deepcopy(snap['gen_arch']) if gen_arch is None else gen_arch
        st = snap['state']
        self._init_pop = dict(x=st['x'], y=st['y'], age=st['age'], sex=st['sex'], idx=st['idx'])
        if gen_arch is None and st.get('genomes') is not None:
            self._init_pop['genomes'] = st['genomes']
        self._attach(capacity=snap['capacity'], cols=snap.get('cols') if gen_arch is None else None)
        if self.burned and gen_arch is None and self.mutate:
            ga = self.gen_arch
            self._dev.set_mutation(ga.mu_neut or 0, ga.mu_delet or 0, ga._mutables,
                                   np.sort(np.asarray(ga.nonneut_loci, dtype=np.int64)), ga.delet_loci, ga.delet_loci_s,
                                   ga.delet_alpha_distr_shape, ga.delet_alpha_distr_scale,
                                   log_capacity=max(ga.L, 16), **self._tskit_mutation_kw())

    # ---- checkpoints (Model.save / load_model) ----------------------------------------------------
    _DEVICE_ATTRS = ('_dev', '_cache', '_inds', '_land', '_strips', '_init_pop')

    def _checkpoint(self):
        """Everything a resumed species needs, at a step boundary, without a device handle: the host attributes
        (life-history overrides, K, changer, burn-in tester, gen_arch with its mutation bookkeeping, surface tables
        as built, tskit tables), the population as downloaded (packed genomes, z, fitness) and the device's clock,
        capacity, column map, path patches and tskit node ids."""
        self._drain_tskit()
        self._sync_mutations()
        ck = dict(attrs={k: v for k, v in self.__dict__.items() if k not in self._DEVICE_ATTRS},
                  state=self._dev.download(genomes=bool(self.burned and self.gen_arch is not None), unpack=False),
                  clock=self._dev.clock(), capacity=int(self._dev.capacity))
        if getattr(self._dev, 'cols', False):
            ck['cols'] = (self._dev.read_cols(), self._dev.col_capacity)
            ck['subsetters'] = self._dev.subsetters()
        if self.burned and self.__dict__.get('_tc') is not None:
            c = self._dev.counters()
            ck['tskit'] = dict(nodes=self._node_ids(), next_node=c['n_nodes'], next_row=c['n_ind_rows'],
                               capacity=self._dev.tskit_capacity)
        return ck

    @classmethod
    def _from_checkpoint(cls, ck, land, strips):
        """The host side of a checkpointed species on `land`, not yet on the device (_resume)."""
        spp = cls.__new__(cls)
        spp.__dict__.update(ck['attrs'])
        spp._land, spp._strips = land, strips
        spp._dev = spp._cache = spp._inds = None
        st = ck['state']
        spp._init_pop = {k: st[k] for k in ('x', 'y', 'age', 'sex', 'idx', 'z', 'fit', 'genomes') if k in st}
        return spp

    def _resume(self, ck, capacity=None):
        """Re-attach from a checkpoint: upload the population, restore the burn-in counts, K, the mutation
        bookkeeping and the tskit node ids, and set the device clock last, so that every later draw is the one
        the saved run would have made."""
        p = self._init_pop
        tester, base = ck['attrs'].get('_burnin_spat_tester'), ck['attrs'].get('_burnin_base')
        self._attach(capacity=capacity, cols=ck.get('cols'))  # life history, rasters, surface tables, burn flag
        if base is not None and not self.burned:
            # the tester's last counts are those of an earlier population (the one it was attached with)
            self._dev.upload(base[0], base[1])
            self._dev.burnin_cell_stats()
            self._upload(p)
        self._burnin_spat_tester, self._burnin_base = tester, base
        if self.__dict__.get('_K_overridden'):
            self._dev.set_K(self.K)
        ga = self.gen_arch
        if self.burned and ga is not None and (self.mutate or ga.use_tskit):
            nn = np.sort(np.asarray(ga.nonneut_loci, dtype=np.int64))
            kw = self._tskit_mutation_kw()
            if ck.get('subsetters') is not None:
                kw['subsetters'] = ck['subsetters']
            if self.mutate:
                self._dev.set_mutation(ga.mu_neut or 0, ga.mu_delet or 0, ga._mutables, nn, ga.delet_loci,
                                       ga.delet_loci_s, ga.delet_alpha_distr_shape, ga.delet_alpha_distr_scale,
                                       log_capacity=max(ga.L, 16), **kw)
            else:
                self._dev.set_mutation(0, 0, [], nn, ga.delet_loci, ga.delet_loci_s, log_capacity=16, **kw)
        tk = ck.get('tskit')
        if tk is not None:
            self._dev.tskit_enable(*tk['capacity'])
            self._dev.tskit_set_nodes(tk['nodes'][:, 0], tk['nodes'][:, 1], tk['next_node'], tk['next_row'])
        self._dev.set_clock(*ck['clock'])
        self._invalidate()

    def _on_raster_change(self, lyr_num, rast):
        if self._dev is not None:
            self._dev.set_raster(lyr_num, rast)        # on-the-fly surfaces follow through the raster itself
            # a table-mode conductance surface over this layer is re-built and swapped in
            # (change.py:576-606: the reference pre-builds one _ConductanceSurface per change step)
            tabs = [None, None]
            for k, nm in enumerate(('_move_surf', '_disp_surf')):
                surf = getattr(self, nm)
                if surf is not None and surf.lyr_num == lyr_num and self._dev._surf_tabs[k] is not None:
                    surf.surf = _make_conductance_surface(self._land[lyr_num].rast, surf.mix, surf.approx_len,
                                                          surf.kappa)
                    tabs[k] = surf.surf
            if tabs[0] is not None or tabs[1] is not None:
                self._dev.set_surface_tables(*tabs)
        if lyr_num == self.K_layer:
            self._set_K(self._land)

    # ---- the queue entries (sim/model.py:603-667) -------------------------------------
    def _set_K(self, land):
        """species.py:546-547.  (The device recomputes its K from the layer whenever the layer
        or K_factor changes; it needs a push only to undo a demographic-change override.)"""
        self.K = land[self.K_layer].rast * self.K_factor
        if self.__dict__.get('_K_overridden') and self._dev is not None:
            self._dev.set_K(self.K)
        self._K_overridden = False

    def _override_K(self, K):
        """A demographic change event rewrote spp.K (change.py:633-649)."""
        self.K = np.asarray(K, dtype=np.float64)
        self._K_overridden = True
        if self._dev is not None:
            self._dev.set_K(self.K)

    _LIFE_HISTORY = {'b': 'b', 'R': 'R', 'n_births_distr_lambda': 'lam', 'n_births_fixed': 'n_births_fixed',
                     'd_min': 'd_min', 'd_max': 'd_max', 'max_age': 'max_age', 'sex_ratio': 'sex_ratio_p',
                     'K_factor': 'K_factor', 'choose_nearest_mate': 'choose_nearest',
                     'inverse_dist_mating': 'inverse_dist', 'direction_distr_mu': 'direction_mu',
                     'direction_distr_kappa': 'direction_kappa'}

    def _set_parameter(self, parameter, val):
        """A life-history change event: setattr(spp, parameter, val) (change.py:737-738)."""
        setattr(self, parameter, val)                  # an instance attribute, shadowing _pv as in the reference
        if self._dev is None:
            return
        prm = self._device_params()
        upd = {}
        if parameter in self._LIFE_HISTORY:
            upd[self._LIFE_HISTORY[parameter]] = prm[self._LIFE_HISTORY[parameter]]
        elif parameter.startswith('movement_distance_distr'):
            upd['move_distr'] = prm['move_distr']
        elif parameter.startswith('dispersal_distance_distr'):
            upd['disp_distr'] = prm['disp_distr']
        elif parameter in ('repro_age',):
            return                                     # never applied by the reference (SURVEY.md quirk 2)
        else:
            raise NotImplementedError("life-history change of '%s' is not supported on the device path "
                                      "(it fixes buffer sizes or the mating grid)" % parameter)
        self._dev.set_life_history(**upd)
        if parameter == 'K_factor' and not self.__dict__.get('_K_overridden'):
            self.K = self._land[self.K_layer].rast * self.K_factor

    def _make_change(self, verbose=False):
        """species.py:836-838."""
        if self._changer is not None:
            self._changer._make_change(self.t, self)

    def _set_t(self):
        self.t += 1

    def _step(self, n=1):
        """_set_age_stage + _do_movement + _do_pop_dynamics + _set_Nt for n time steps
        (species.py:567, 582, 822, 554) on the device."""
        tsk = self.burned and self.gen_arch is not None and self.gen_arch.use_tskit and \
            self.__dict__.get('_tc') is not None
        if tsk and n > self._tsk_steps:
            # the device row buffers hold _tsk_steps steps of births: drain in between
            done = 0
            while done < n and not self.extinct:
                k = min(self._tsk_steps, n - done)
                self._step(k)
                done += k
            return
        stop = self._dev.step(n)
        while stop is not None:
            # a step would overflow the tskit row buffers: drain them, grow them only if one step still
            # needs more, and go on (every step runs: walk's `ran < n` keeps meaning extinction)
            births, edges = self._drain_tskit()
            need_b, need_e = stop['need_births'] - births, stop['need_edges'] - edges
            ecap, bcap = stop['edge_capacity'], stop['born_capacity']
            if need_b > bcap or need_e > ecap:
                self._dev.tskit_reserve(growth_capacity(need_e, ecap) if need_e > ecap else ecap,
                                        growth_capacity(need_b, bcap) if need_b > bcap else bcap)
            stop = self._dev.step(stop['steps_left'])
        recs = self._dev.step_records()
        if tsk:
            self._drain_tskit()
            self._tc_sorted_and_simplified = False
        for k, r in enumerate(recs):
            self.Nt.append(int(r['Nt']))
            self.n_births.append(int(r['n_births']))
            self.n_deaths.append(int(r['n_deaths']))
            if r['Nt'] == 0:                         # extinct: the reference stops here (model.py:704-706);
                recs = recs[:k + 1]                  # later steps of a bulk call were no-ops on an empty population
                break
        if self.mutate and self.burned:
            self._sync_mutations()
        if recs:
            self.max_ind_idx += int(sum(r['n_births'] for r in recs))
            if recs[-1]['Nt'] == 0:
                self.extinct = True                  # demography.py:329
        self._invalidate()

    def _invalidate(self):
        self._cache = None
        self._inds = None
        self.N = None

    # ---- lazy host views -----------------------------------------------------------------
    def _state(self):
        if self._cache is None:
            if self._dev is None:
                p = self._init_pop
                self._cache = dict(x=p['x'], y=p['y'], age=p['age'], sex=p['sex'], idx=p['idx'],
                                   z=np.zeros((len(p['x']), 0)), fit=np.full(len(p['x']), np.nan),
                                   e=None, g=None)
            else:
                # a use_tskit species' rows are the Individuals' own: one per non-neutral locus (species.py:891-905)
                self._cache = self._dev.download(genomes=self.burned and self.gen_arch is not None, e=True)
        return self._cache

    def _individuals(self):
        if self._inds is None:
            s = self._state()
            inds = OrderedDict()
            g = s.get('g')
            has_z = s['z'] is not None and s['z'].shape[1] > 0
            for k in range(len(s['x'])):
                inds[int(s['idx'][k])] = Individual(
                    int(s['idx'][k]), s['x'][k], s['y'][k], int(s['age'][k]),
                    None if g is None else g[k], int(s['sex'][k]),
                    None if s.get('e') is None else list(s['e'][k]),
                    list(s['z'][k]) if has_z else [], None if np.isnan(s['fit'][k]) else float(s['fit'][k]))
            self._inds = inds
        return self._inds

    def __len__(self):
        if self._cache is not None:
            return len(self._cache['x'])
        if self._dev is None:
            return len(self._init_pop['x'])
        return self._dev.population_size()

    def __iter__(self):
        return iter(self._individuals())

    def __getitem__(self, idx):
        return self._individuals()[idx]

    def __contains__(self, idx):
        return idx in self._individuals()

    def keys(self):
        return self._individuals().keys()

    def values(self):
        return self._individuals().values()

    def items(self):
        return self._individuals().items()

    @property
    def _coords(self):
        s = self._state()
        return np.stack([s['x'], s['y']], axis=1)

    @property
    def _cells(self):
        return np.int32(np.floor(self._coords))

    # getters (species.py:1364-1499)
    def _get_x(self, individs=None):
        return self._sel(self._state()['x'], individs)

    def _get_y(self, individs=None):
        return self._sel(self._state()['y'], individs)

    def _get_coords(self, individs=None, as_float=True):
        c = self._sel(self._coords, individs)
        return c if as_float else np.int32(np.floor(c))

    def _get_cells(self, individs=None):
        return self._get_coords(individs, as_float=False)

    def _get_age(self, individs=None):
        return self._sel(self._state()['age'], individs)

    def _get_sex(self, individs=None):
        return self._sel(self._state()['sex'], individs)

    def _get_z(self, trait_num=None, individs=None):
        z = self._sel(self._state()['z'], individs)
        return z if trait_num is None else z[:, trait_num]

    def _get_e(self, lyr_num=None, individs=None):
        e = self._sel(self._state()['e'], individs)
        return e if lyr_num is None else e[:, lyr_num]

    def _get_fit(self, individs=None):
        return self._sel(self._state()['fit'], individs)

    def _get_genotypes(self, loci=None, individs=None, biallelic=True, as_dict=False, all_loci=False):
        """species.py:1364-1448.  For a use_tskit species the arrays are the Individuals' own rows (one
        per non-neutral locus, species.py:891-905); `all_loci=True` gives all L loci, which the
        reference reads off the tree sequence (:1395-1425) and the device holds by locus."""
        s = self._state()
        g = self._sel(s['g'], individs)
        if all_loci and s.get('col_locus') is not None:      # rows of the chosen individuals scattered to their loci
            g = gp.rows_to_loci(g, np.sort(s['col_locus']), self.gen_arch.L)
        if loci is not None:
            g = g[:, loci, :]
        if not biallelic:
            g = g.mean(axis=2)
        if as_dict:
            ids = self._sel(self._state()['idx'], individs)
            return {int(i): gi for i, gi in zip(ids, g)}
        return g

    def _sel(self, arr, individs):
        if individs is None or arr is None:
            return arr
        ids = self._state()['idx']
        pos = {int(v): k for k, v in enumerate(ids)}
        return arr[[pos[int(i)] for i in individs]]

    def _calc_density(self, normalize=False, as_layer=False, set_N=False):
        """species.py:845-882: the N raster of the last completed step (device resident)."""
        dens = self._dev.raster('N_RAST')
        if normalize:
            dens = (dens - dens.min()) / (dens.max() - dens.min())
        if set_N:
            self.N = dens
            return None
        return dens

    # ---- statistics on the device (sim/stats.py:399-435) ---------------------------------
    def _calc_het(self, mean=False):
        """stats.py:399-410: locus-wise (or mean) frequency of heterozygotes."""
        het = self._dev.stats()['het']
        return float(np.mean(het)) if mean else het

    def _calc_maf(self):
        """stats.py:412-425."""
        return self._dev.stats()['maf']

    def _calc_allele_freqs(self):
        return self._dev.stats()['freq']

    def _calc_ld(self):
        """stats.py:359-392: r^2 between every pair of loci (L x L, NaN diagonal); the chromosome
        counts behind it are accumulated on the device from the packed genotypes."""
        return self._dev.ld()

    def _calc_mean_fitness(self):
        """stats.py:428-435: mean of the fitness values of the last completed step."""
        return self._dev.stats()['mean_fit'] if self.gen_arch.traits is not None else np.nan

    # ---- post burn-in genome assignment (species.py:956-1094, genome.py:1108-1157) ----
    def _set_genomes_and_tables(self, burn_T=None, T=None, genome_init='host'):
        s = self._dev.download(genomes=False)
        n = len(s['x'])
        ga = self.gen_arch
        L = ga.L
        tsk = ga.use_tskit
        if genome_init == 'device':
            self._set_genomes_on_device(s, burn_T, T)
            return
        p = ga.p
        # genome.py:1137-1142: a use_tskit species carries the non-neutral rows only, in ascending locus order
        row_of = {int(l): r for r, l in enumerate(np.sort(np.asarray(ga.nonneut_loci, dtype=np.int64)))} if tsk \
            else {l: l for l in range(L)}
        g = np.zeros((n, len(row_of), 2), dtype=np.int8)
        mut_site, mut_node = [], []
        n_muts = gp.carrier_counts(n, p[:L])
        for site in range(L):
            n_mut = int(n_muts[site])
            if n_mut > 0:
                hom = np.random.permutation(2 * n)[:n_mut]
                if site in row_of:
                    g[hom // 2, row_of[site], hom % 2] = 1
                if tsk:                                   # genome.py:1143-1147: node of (individual k, homologue h)
                    mut_site.append(np.full(n_mut, site, np.int32))
                    mut_node.append(hom.astype(np.int32))  # is 2k + h (see below)
        self._dev.set_burn(False)
        self._dev.upload(s['x'], s['y'], s['age'], s['sex'], s['idx'], g=g, max_ind_idx=s['max_ind_idx'])
        self._finish_genome_assignment(s, burn_T, T, mut_site, mut_node)

    def _set_genomes_on_device(self, s, burn_T, T):
        """The same assignment drawn on the device (DeviceSpecies.init_genomes): the same per-locus 1-allele
        counts, no genotype download and no host array.  The device seed comes from numpy's stream, so a
        seeded model stays reproducible and every rand_genarch iteration gets new genomes."""
        ga = self.gen_arch
        seed = int(np.random.randint(0, 2 ** 63 - 1, dtype=np.int64))
        mask = None
        if ga.use_tskit:                                  # genome.py:1137-1142: only non-neutral rows are carried
            mask = np.zeros(ga.L, np.uint8)
            mask[np.asarray(ga.nonneut_loci, dtype=np.int64)] = 1
        rows = self._dev.init_genomes(np.asarray(ga.p, dtype=np.float64)[:ga.L], seed, write_mask=mask,
                                      tskit_rows=ga.use_tskit)
        self._dev.set_burn(False)
        mut_site, mut_node = [], []
        if rows is not None and len(rows['site']):
            # node of (individual k in species order, homologue h) is 2k + h; rows come sorted by (site, node)
            mut_site = [rows['site']]
            mut_node = [(2 * np.searchsorted(s['idx'], rows['idx']) + rows['homologue']).astype(np.int32)]
        self._finish_genome_assignment(s, burn_T, T, mut_site, mut_node)

    def _finish_genome_assignment(self, s, burn_T, T, mut_site, mut_node):
        ga = self.gen_arch
        n = len(s['x'])
        tsk = ga.use_tskit
        # everyone up to this id was alive at the assignment (the FASTA writer tells them apart, writers.py)
        self._genome_assignment_max_idx = int(s['max_ind_idx'])
        self._tc = None
        if tsk:
            self._set_tables(s, mut_site, mut_node)
        self._set_mutation(burn_T, T)
        if tsk:
            # per-birth row buffers on the device, drained at the simplification cadence (model.py:756-768)
            n_bp = max([len(v) for v in ga.recombinations._breakpoints.values()] + [1])
            births = max(1024.0, float(np.sum(self.K)) * self.b * self.n_births_distr_lambda)
            self._tsk_steps = int(max(1, min(ga.tskit_simp_interval or 100, 2.0e8 // (2 * (n_bp + 1) * births))))
            self._dev.tskit_enable(edge_capacity=int(2 * (n_bp + 1) * births * 2 * self._tsk_steps) + 4096,
                                   birth_capacity=int(births * 2 * self._tsk_steps) + 1024)
            self._dev.tskit_set_nodes(2 * np.arange(n, dtype=np.int32), 2 * np.arange(n, dtype=np.int32) + 1,
                                      2 * n, n)
            self._tsk_t0 = self._dev.counters()['t']
            self._tc_sorted_and_simplified = False
        self._invalidate()

    def _set_tables(self, s, mut_site, mut_node):
        """species.py:968-1090 without msprime (absent here): the starting population is 2N unrelated sample
        nodes -- a forest of singletons, which is what msprime's ancestry reduces to for the path (only the
        nodes' flags are read, species.py:1006-1009) -- one individuals row per individual (flags = 1, location
        [x, y, z..., fit], idx), nodes 2k, 2k + 1 for the k-th individual (time 1: born before the main phase,
        species.py:1075-1077), one sites row per locus in order (:994-1002) and the starting mutations
        (genome.py:1143-1147).  Phenotypes / fitness are not known before the first step: NaN."""
        from .tables import TableColumns
        ga = self.gen_arch
        n = len(s['x'])
        nt = len(ga.traits) if ga.traits is not None else 0
        tc = TableColumns(ga.L, nt)
        loc = np.full((n, tc.n_loc), np.nan)
        loc[:, 0], loc[:, 1] = s['x'], s['y']
        tc.individuals.append_columns(flags=np.ones(n, np.int32), location=loc, idx=s['idx'])
        tc.nodes.append_columns(flags=np.ones(2 * n, np.int32), time=np.ones(2 * n), population=np.zeros(2 * n, np.int32),
                                individual=np.repeat(np.arange(n, dtype=np.int32), 2))
        nn = np.zeros(ga.L, np.int8)
        nn[np.asarray(ga.nonneut_loci, dtype=np.int64)] = 1
        tc.sites.append_columns(position=np.arange(ga.L, dtype=np.float64), nonneutral=nn)
        if mut_site:
            ms, mn = np.concatenate(mut_site), np.concatenate(mut_node)
            tc.mutations.append_columns(site=ms, node=mn, time=np.full(len(ms), np.nan))
        self._tc = tc

    def _drain_tskit(self):
        """Device row buffers -> self._tc (species.py:692-736 rows, in the reference's order)."""
        if self._tc is None or self._dev is None:
            return 0, 0
        rows = self._dev.tskit_drain()
        self._tc.append_births(rows)
        return len(rows['idx']), len(rows['left'])

    def _sort_and_simplify_table_collection(self):
        """species.py:1107-1219: sort + simplify on the current nodes, then nodes 2k, 2k + 1 in species order and
        the individuals rows in species order (gnx_tskit_renumber).  sort()/simplify() are tskit's own."""
        self._drain_tskit()
        n = len(self)
        self._tc.sort_and_simplify(self._node_ids().reshape(-1), self._dev)
        # the samples are nodes 0 .. 2N - 1 in the order given (species.py:1148-1152); nodes where their ancestry
        # coalesces follow, with the individuals they belong to, so the NEXT rows continue from the table sizes
        self._dev.tskit_set_nodes(2 * np.arange(n, dtype=np.int32), 2 * np.arange(n, dtype=np.int32) + 1,
                                  self._tc.nodes.num_rows, self._tc.individuals.num_rows)
        self._tc_sorted_and_simplified = True
        self._invalidate()

    def _node_ids(self):
        """int32[N, 2]: the nodes-table ids of every individual's two homologues, species order."""
        n = len(self)
        out = np.stack([self._dev.read('NODE0', n), self._dev.read('NODE1', n)], axis=1)
        return out

    def _set_mutation(self, burn_T, T):
        """species.py:960-967 + genome.py:1060-1104: check the rates against the infinite-sites
        budget, shuffle the mutable loci, hand the bookkeeping to the device (a13)."""
        ga = self.gen_arch
        kw = self._tskit_mutation_kw()
        nonneut = set(int(v) for v in ga.nonneut_loci)
        nn_sorted = np.array(sorted(nonneut), dtype=np.int64)
        if not self.mutate:
            if ga.use_tskit:
                self._dev.set_mutation(0, 0, [], nn_sorted, ga.delet_loci, ga.delet_loci_s, log_capacity=16, **kw)
            return
        if not ga.use_tskit and ga.traits is not None and any(t.mu > 0 for t in ga.traits.values()):
            # genome.py:430: Trait._add_locus indexes loci_idxs, which is None when use_tskit=False
            raise NotImplementedError('trait mutation (Trait.mu > 0) raises in the reference when '
                                      'use_tskit=False (genome.py:416-437)')
        # mutation.py:24-41 _calc_estimated_total_mutations
        mean_births = float(np.sum(self.K)) * self.b * self.n_births_distr_lambda
        est = int(2.5 * mean_births * ga.L * (T or 0) * ga._mu_tot)
        if est > 0.75 * (ga.L - len(nonneut)):
            raise MutationRateError('This species has been parameterized with too few neutral loci to '
                                    'accommodate the expected number of mutations. (Geonomics only uses an '
                                    'infinite sites model.)')
        if len(ga.neut_loci) == 0 and ga._mu_tot > 0:        # genome.py:1082-1094
            warnings.warn('non-zero mutation rates but no neutral loci: mutation switched off')
            ga.mu_neut = ga.mu_delet = 0
            for t in (ga.traits or {}).values():
                t.mu = 0
            self.mutate = False
            if ga.use_tskit:
                kw['trait_mus'] = None
                self._dev.set_mutation(0, 0, [], nn_sorted, ga.delet_loci, ga.delet_loci_s, log_capacity=16, **kw)
            return
        mutables = [*set(range(ga.L)).difference(nonneut)]    # genome.py:1101-1104
        np.random.shuffle(mutables)
        ga._mutables = [*mutables]
        self._dev.set_mutation(ga.mu_neut or 0, ga.mu_delet or 0, ga._mutables, nn_sorted, ga.delet_loci,
                               ga.delet_loci_s, ga.delet_alpha_distr_shape, ga.delet_alpha_distr_scale,
                               log_capacity=max(ga.L, 16), **kw)

    def _tskit_mutation_kw(self):
        """set_mutation's use_tskit arguments: species.py:891-905 layout (rows = non-neutral loci, read through
        the reference's index arrays as written)."""
        ga = self.gen_arch
        if not ga.use_tskit:
            return {}
        traits = list((ga.traits or {}).values())
        return dict(tskit_layout=True,
                    trait_mus=[t.mu or 0 for t in traits] if self.mutate else None,
                    trait_alpha_distr=[(t.alpha_distr_mu, t.alpha_distr_sigma, t.max_alpha_mag) for t in traits],
                    trait_loci_idxs=[t.loci_idxs for t in traits], delet_loci_idxs=ga.delet_loci_idxs)

    def _sync_mutations(self):
        """Pull the device's mutation log and bookkeeping into gen_arch (what mutation.py:199-205
        logs, and genome.py:753-788 maintains, in the reference)."""
        if not self.mutate or self._dev is None or not self.burned:
            return []
        rows, st = self._dev.read_mutations(max_rows=max(self.gen_arch.L, 16))
        ga = self.gen_arch
        ga._mutables = ga._mutables[:st['n_mutables']]
        ga.nonneut_loci = st['nonneut_loci'].astype(np.int64)
        ga.neut_loci = np.array(sorted(set(range(ga.L)).difference(set(int(v) for v in ga.nonneut_loci))))
        ga.delet_loci = st['delet_loci'].astype(np.int64)
        ga.delet_loci_s = st['delet_s']
        if ga.use_tskit and rows:
            traits, di = self._dev.read_mutation_tables()     # genome.py:416-437, 779-782, as written
            ga.delet_loci_idxs = di.astype(np.int64)
            for t, tr in zip((ga.traits or {}).values(), traits):
                t.loci, t.alpha, t.loci_idxs = tr['loci'].astype(np.int64), tr['alpha'], tr['loci_idxs'].astype(np.int64)
                t.n_loci = len(t.loci)
            if self._tc is not None:                           # mutation.py:44-58
                self._tc.mutations.append_columns(site=[r['locus'] for r in rows], node=[r['node'] for r in rows],
                                                  time=[-1.0 * (r['t'] - self._tsk_t0) for r in rows])
                nn = self._tc.sites.nonneutral
                # (the reference leaves the sites metadata as assigned at the start, species.py:994-1002)
        self.mutations.extend(rows)
        if self.mut_log:
            with open(self.mut_log, 'a') as f:
                for r in rows:
                    f.write('MUTATION: %s\n\t INDIVIDUAL %i,  LOCUS %i\n\t timestep %i\n\n'
                            % (r['type'], r['individual'], r['locus'], r['t']))
        return rows


class Community(dict):
    """community.py:25."""

    def __init__(self, land, spps):
        super().__init__(spps)
        self.n_spps = len(spps)
        self.t = -1
        self.burned = False


def _make_species(land, name, idx, spp_params, seed=0, strips=None):
    """species.py:3276-3397."""
    init = dict(spp_params.init)
    ga = _make_genomic_architecture(spp_params, land) if 'gen_arch' in spp_params else None
    N = int(init.pop('N'))
    spp = Species(name, idx, land, spp_params, ga, N=N, seed=seed, strips=strips)
    # individual.py:188-229: uniform positions, Bernoulli(0.5) sex (with the re-draw quirk of
    # Individual.__init__, individual.py:110-115: a drawn 0 is re-drawn)
    xy = np.random.rand(N, 2) * np.array(land.dim)
    x = np.clip(xy[:, 0], 0, land.dim[0] - 0.001)
    y = np.clip(xy[:, 1], 0, land.dim[1] - 0.001)
    sex = np.random.binomial(1, 0.5, N)
    sex = np.where(sex == 1, 1, np.random.binomial(1, 0.5, N)).astype(np.int8)
    spp._init_pop = dict(x=x, y=y, age=np.zeros(N, np.int32), sex=sex, idx=np.arange(N, dtype=np.int64))
    K_layer = [lyr for lyr in land.values() if lyr.name == init['K_layer']]
    assert len(K_layer) == 1, 'K_layer must name a single Layer'
    spp.K_layer = K_layer[0].idx
    spp.K_factor = init['K_factor']
    K_layer[0]._is_K.append(idx)
    spp._set_K(land)
    mv = spp_params.get('movement', {})
    if spp._move and 'move_surf' in mv:
        ms = dict(mv['move_surf'])
        name = ms.pop('layer')
        lyr = [k for k, v in land.items() if v.name == name]
        assert len(lyr) == 1
        spp._move_surf = _ConductanceSurface(land[lyr[0]], **ms)
    if 'disp_surf' in mv:
        ds = dict(mv['disp_surf'])
        name = ds.pop('layer')
        lyr = [k for k, v in land.items() if v.name == name]
        assert len(lyr) == 1
        spp._disp_surf = _ConductanceSurface(land[lyr[0]], **ds)
    if 'change' in spp_params:                               # species.py:3373-3395
        spp._changer = _SpeciesChanger(spp, spp_params['change'], land)
    return spp


# ---------------------------------------------------------------------------------------------
# model (sim/model.py)
# ---------------------------------------------------------------------------------------------
def _check_genome_init(genome_init):
    if genome_init not in ('host', 'device'):
        raise ValueError("genome_init must be 'host' or 'device', not %r" % (genome_init,))


def _strip_world(strips):
    """The number of strips of `strips` (None, an int >= 2 or an initialised nccl process group)."""
    if strips is None:
        return None
    if isinstance(strips, (int, np.integer)) and not isinstance(strips, bool):
        if strips < 2:
            raise ValueError('strips must be at least 2 (or None, or a process group), not %d' % strips)
        return int(strips)
    import torch.distributed as dist
    if not isinstance(strips, dist.ProcessGroup) or not dist.is_initialized():
        raise ValueError('strips must be None, an int >= 2 or an initialised torch.distributed process group')
    if dist.get_backend(strips) != 'nccl':
        raise ValueError('a strip process group needs the nccl backend, not %s' % dist.get_backend(strips))
    return dist.get_world_size(strips)


def _check_strip_species(spp, world):
    """What strip decomposition does not carry, refused before any device work."""
    from .strips import mating_grid
    ga = spp.gen_arch
    if ga is not None and ga.use_tskit:
        raise ValueError("species '%s': use_tskit=True is not supported under strip decomposition" % spp.name)
    if ga is not None and any((t.mu or 0) > 0 for t in (ga.traits or {}).values()):
        raise ValueError("species '%s': trait mutation (Trait.mu > 0) is not supported under strip decomposition"
                         % spp.name)
    if getattr(spp, 'mating_radius', None) is None:
        raise ValueError("species '%s': a panmictic species (no mating radius) cannot be cut into strips" % spp.name)
    ncy = mating_grid(spp._land_dim, spp.mating_radius)[2]
    if ncy < 2 * world:
        raise ValueError("species '%s': %d strips need %d mating-grid rows, the landscape has %d"
                         % (spp.name, world, 2 * world, ncy))


class Model:
    """sim/model.py:47.  `walk` / `run` keep their reference signatures.

    genome_init selects how the starting genomes are assigned after the burn-in: 'host' (the
    default) draws them with numpy's stream exactly as the reference does; 'device' draws them on the
    GPU with the same exact per-locus allele counts (DeviceSpecies.init_genomes) and never builds the
    N x L x 2 host array, which is what makes populations of millions of individuals startable.

    strips cuts every species into horizontal strips of its mating grid (geonomics_b200/strips.py) and
    reproduces the undecomposed model with the same seed: None (the default) keeps each species on one
    context; an int k >= 2 holds k strips as contexts of this process on the current GPU (a check, no
    speed-up); an initialised torch.distributed process group (nccl, one rank per GPU of one node) gives
    every rank its own strip.  Under a group every rank runs the same script and makes the same calls in
    the same order, and builds the same host state from numpy's global stream: without a seed in the
    parameters rank 0 draws one and every rank seeds numpy with it.  Strips refuse use_tskit, trait
    mutation, panmixia, fewer than two mating-grid rows per strip and Model.run(dist=...)."""

    def __init__(self, name, params, verbose=False, genome_init='host', strips=None):
        _check_genome_init(genome_init)
        world = _strip_world(strips)
        self.genome_init = genome_init
        self.strips = strips
        self.params = copy.deepcopy(params)
        m = self.params.model
        self.name = name or 'unnamed_model'
        self._verbose = verbose
        self.seed = None
        if 'seed' in m and m.seed is not None:
            self.seed = m.seed.num if isinstance(m.seed, dict) else m.seed
        if world is not None and not isinstance(strips, (int, np.integer)) and self.seed is None:
            import torch.distributed as dist
            box = [int(np.random.SeedSequence().generate_state(1)[0]) if dist.get_rank(strips) == 0 else None]
            dist.broadcast_object_list(box, group=strips, group_src=0)
            self.seed = box[0]
        if self.seed is not None:
            np.random.seed(self.seed)                       # model.py:362-366
        self.burn_T = m.burn_T
        self.burn_t = -1
        self.T = m.T
        self.t = -1
        its = m.get('its', {'n_its': 1})
        self.n_its = its['n_its']
        self.its = [*range(self.n_its)][::-1]
        self.it = -1
        # model.py:115-131: what is re-drawn from one iteration to the next
        self.rand_landscape = bool(its.get('rand_landscape', False))
        self.rand_comm = bool(its.get('rand_comm', False))
        self.rand_genarch = bool(its.get('rand_genarch', True))
        self.repeat_burn = bool(its.get('repeat_burn', False))
        self.iterations = {}                 # {it: per-step Nt / births / deaths of that iteration's main phase}
        self.land = _make_landscape(self.params)
        spps = {}
        for n, (sname, sp) in enumerate(self.params.comm.species.items()):
            spps[n] = _make_species(self.land, sname, n, sp, seed=(self.seed or 0) * 1000003 + n, strips=strips)
            if world is not None:
                _check_strip_species(spps[n], world)
        self.comm = Community(self.land, spps)
        for spp in self.comm.values():
            spp._attach()
        self.reassign_genomes = True
        self._never_been_run = True
        # model.py:147-163: the originals the later iterations start from
        self.orig_land = None if self.rand_landscape else copy.deepcopy(self._bare_land())
        self.orig_comm = None if self.rand_comm else {n: spp._snapshot() for n, spp in self.comm.items()}

    # ---- one queue pass (model.py:603-667, 699-787); each species is advanced itself (the
    # reference's late-binding lambdas advance only the last species, SURVEY.md quirk 1)
    def _do_timestep(self, mode):
        if mode == 'burn':
            self.burn_t += 1
            for spp in self.comm.values():
                if not any(s.extinct for s in self.comm.values()):
                    spp._step(1)
            self._check_comm_burned()
            if all(spp.burned for spp in self.comm.values()):
                if self.reassign_genomes:
                    for spp in self.comm.values():
                        if spp.gen_arch is not None:
                            spp._set_genomes_and_tables(self.burn_T, self.T, self.genome_init)
                    self.reassign_genomes = False
                self.comm.burned = True
        elif mode == 'main':
            self.t += 1
            self.comm.t += 1
            for spp in self.comm.values():
                if not any(s.extinct for s in self.comm.values()):
                    spp._set_t()
                    spp._step(1)
            self._make_changes()
            self._simplify_if_due()
        return any(spp.extinct for spp in self.comm.values())

    @staticmethod
    def _have_tskit():
        import importlib.util
        import sys
        import types
        mod = sys.modules.get('tskit')
        if mod is not None:                               # a test shim in sys.modules is not tskit
            return isinstance(mod, types.ModuleType) and getattr(mod, '__file__', None) is not None
        try:
            return importlib.util.find_spec('tskit') is not None
        except (ValueError, ImportError):
            return False

    def _next_simplify_t(self, spp):
        """model.py:756-768: the tables are sorted and simplified after the step at every t with
        (t + 1) % tskit_simp_interval == 0 (tskit's own implementation where it is installed, the restated
        algorithm of tables.simplify_columns otherwise)."""
        ga = spp.gen_arch
        if ga is None or not ga.use_tskit or spp.__dict__.get('_tc') is None:
            return None
        k = int(ga.tskit_simp_interval)
        return (self.t + 1) + (k - 1 - (self.t + 1) % k)

    def _simplify_if_due(self):
        for spp in self.comm.values():
            ga = spp.gen_arch
            if (ga is not None and ga.use_tskit and spp.__dict__.get('_tc') is not None and self.t != -1
                    and (self.t + 1) % int(ga.tskit_simp_interval) == 0):
                spp._sort_and_simplify_table_collection()

    def _make_changes(self):
        """The tail of the main queue (model.py:646-656): the landscape change of this time step,
        Species._set_K for every species whenever the landscape has a changer (which also undoes a
        demographic override of K, as in the reference), then the species' own changes."""
        if self.land._changer is not None:
            self.land._make_change(self.t)
            for spp in self.comm.values():
                spp._set_K(self.land)
        for spp in self.comm.values():
            if spp._changer is not None:
                spp._make_change()

    def _check_comm_burned(self):
        """community.py:107-131: after at least burn_T steps, every species must pass the ADF and the
        paired t-test on Nt (burnin.py:93-103) and the spatial test on the per-cell count changes
        (burnin.py:21-90, species.py:572-578; counts and their change come from the device).  As in
        the reference all three are evaluated for every species (no short circuit), so the spatial
        tester sees every step after the burn_T-th."""
        from . import burnin
        ok = all(len(spp.Nt) >= self.burn_T for spp in self.comm.values())
        if ok:
            def safe(fn, spp):
                try:
                    return bool(fn(spp.Nt, self.burn_T))
                except ValueError:                    # a constant series (e.g. K reached exactly): not stationary evidence
                    return False
            adf_tests = all([safe(burnin.test_adf_threshold, spp) for spp in self.comm.values()])
            t_tests = all([safe(burnin.test_t_threshold, spp) for spp in self.comm.values()])
            spat_tests = all([spp._do_spatial_burnin_test(self.burn_T) for spp in self.comm.values()])
            ok = adf_tests and t_tests and spat_tests
        for spp in self.comm.values():
            spp.burned = ok
        self.comm.burned = ok

    def walk(self, T=1, mode='main', verbose=False):
        """model.py:966: run T time steps in 'burn' or 'main' mode."""
        assert mode in ('burn', 'main')
        if mode == 'main' and not self.comm.burned:
            raise ValueError("Model.walk(mode='main') called before the burn-in completed "
                             "(walk(mode='burn') first), as in the reference (model.py:1112).")
        if mode == 'burn' and self.comm.burned:
            return
        # fast path: between two host-side events (a scheduled landscape change, the end of the
        # walk) the steps are enqueued in one call -- no host round trip per time step
        if mode == 'main' and not verbose and len(self.comm) == 1:
            spp = next(iter(self.comm.values()))
            done = 0
            while done < T and not spp.extinct:
                n = min(T - done, 65536)                              # the device holds 65 536 step records
                changer = self.land._changer
                events = []                                           # applied after the step at that t
                if changer is not None and changer._pos < len(changer.changes):
                    events.append(changer.changes[changer._pos][0])
                if spp._changer is not None and spp._changer._next_t() is not None:
                    events.append(spp._changer._next_t())
                simp = self._next_simplify_t(spp)
                if simp is not None:
                    events.append(simp)
                if events:
                    n = max(1, min(n, min(events) - self.t))
                if changer is not None and spp.__dict__.get('_K_overridden'):
                    n = 1                                             # the next _set_K undoes the override
                n_rec0 = len(spp.Nt)
                spp._step(n)
                ran = len(spp.Nt) - n_rec0                           # < n if the species went extinct
                spp.t += ran
                self.t += ran
                self.comm.t += ran
                done += ran
                self._make_changes()                                  # model.py:646-656
                self._simplify_if_due()                               # model.py:756-768
                if ran < n:
                    break
            return
        for t in range(T):
            extinct = self._do_timestep(mode)
            if verbose:
                for spp in self.comm.values():
                    print('%s:\tit=%i:\tt=%i\tspecies: %s N=%s (births=%s deaths=%s)' % (
                        mode, self.it, self.burn_t if mode == 'burn' else self.t, spp.name,
                        spp.Nt[-1] if spp.Nt else np.nan, spp.n_births[-1] if spp.n_births else np.nan,
                        spp.n_deaths[-1] if spp.n_deaths else np.nan))
            if extinct or (mode == 'burn' and self.comm.burned):
                break

    # ---- iterations (model.py:338-339, 410-506, 520-593, 790-858, 866-953) -----------------------
    def _bare_land(self):
        """The landscape without its device listeners (what a deep copy should carry)."""
        land = copy.copy(self.land)
        land._listeners = []
        return land

    def _reset_landscape(self, rand_landscape):
        if rand_landscape:
            self.land = _make_landscape(self.params)               # model.py:436-441
        else:
            self.land = copy.deepcopy(self.orig_land)              # model.py:423-435 (changer included:
            self.land._listeners = []                              #  its schedule starts over)

    def _reset_community(self, rand_comm):
        if rand_comm:                                              # model.py:499-505: a new Community
            for spp in self.comm.values():
                spp._detach()
            spps = {}
            for n, (sname, sp) in enumerate(self.params.comm.species.items()):
                spps[n] = _make_species(self.land, sname, n, sp, seed=(self.seed or 0) * 1000003 + n + 7919 * (self.it + 1),
                                        strips=self.strips)
            self.comm = Community(self.land, spps)
            for spp in self.comm.values():
                spp._attach()
            return
        for n, spp in self.comm.items():                           # model.py:457-494: the original Community
            ga = None
            if self.rand_genarch and spp.gen_arch is not None:
                ga = _make_genomic_architecture(self.params.comm.species[spp.name], self.land)
            spp._restore(self.orig_comm[n], self.land, gen_arch=ga)
            if ga is not None and not self.repeat_burn and spp.burned:
                spp._set_genomes_and_tables(self.burn_T, self.T, self.genome_init)
        self.comm.burned = all(spp.burned for spp in self.comm.values())
        self.comm.t = -1

    def _reset(self):
        """model.py:520-593."""
        if not self._never_been_run:
            self._reset_landscape(self.rand_landscape)
            self._reset_community(self.rand_comm)
        else:
            self._never_been_run = False
        self.t = -1
        if self.repeat_burn:
            self.burn_t = -1
        self.comm.t = -1
        for spp in self.comm.values():
            spp.t = -1
        self.reassign_genomes = any(spp.gen_arch is not None for spp in self.comm.values())

    def _do_next_iteration(self, verbose=False):
        """model.py:808-858."""
        self.it = self.its.pop()                                   # model.py:338-339
        self._reset()
        if self.rand_comm or self.repeat_burn or self.it == 0 or not self.comm.burned:
            if self.repeat_burn and self.orig_comm is not None and self.it > 0:
                for spp in self.comm.values():                     # burn in again from the saved start
                    spp.burned = False
                    spp._dev.set_burn(True)
                self.comm.burned = False
            self.walk(10 ** 9, 'burn', verbose)
            if not self.rand_comm and not self.repeat_burn:
                self.orig_comm = {n: spp._snapshot() for n, spp in self.comm.items()}     # model.py:833-838
        if any(spp.extinct for spp in self.comm.values()):
            return
        n0 = {n: len(spp.Nt) for n, spp in self.comm.items()}
        self.walk(self.T, 'main', verbose)
        self.iterations[self.it] = {n: dict(Nt=np.array(spp.Nt[n0[n]:]), n_births=np.array(spp.n_births[n0[n]:]),
                                            n_deaths=np.array(spp.n_deaths[n0[n]:]))
                                    for n, spp in self.comm.items()}

    def run(self, verbose=False, dist=None):
        """model.py:866-953: every iteration in `its` -- burn-in where the iteration needs one, then
        T main steps; what carries over between iterations follows rand_landscape / rand_comm /
        rand_genarch / repeat_burn.  With an initialised `torch.distributed` handle in `dist` the
        iterations are sharded round-robin over the ranks (they never exchange data,
        geonomics_b200/parallel.py) and rank 0 returns every iteration's trajectories."""
        if dist is not None and self.strips is not None:
            raise ValueError('Model.run(dist=...) shards iterations over the ranks; a strip model already spreads '
                             'each species over them')
        self._verbose = verbose
        mine = None
        if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
            from . import parallel
            mine = set(parallel.shard_iterations(self.n_its, dist.get_rank(), dist.get_world_size()))
        while len(self.its) > 0:
            if mine is not None and self.its[-1] not in mine:
                it = self.its.pop()
                if it == 0:
                    self.its.append(it)                            # every rank needs the burned-in original
                else:
                    continue
            if mine is not None and self.seed is not None:
                np.random.seed(self.seed + 104729 * self.its[-1])  # an iteration's draws do not depend on the sharding
            self._do_next_iteration(verbose)
        self._verbose = False
        if mine is not None:
            from . import parallel
            return parallel.gather_trajectories({it: v for it, v in self.iterations.items() if it in mine}, dist)
        return self.iterations

    # ---- checkpoints ----------------------------------------------------------------------------
    _DEVICE_ATTRS = ('land', 'comm', 'strips')

    def save(self, path):
        """Write the model, at the step boundary it stands at, to one file that load_model resumes from bit for
        bit, on one GPU or on any number of strips: the model's own state (params, clocks, remaining iterations
        and the originals they start from), numpy's and random's global streams, the landscape with its changer,
        and every species (Species._checkpoint).  Under a process group every rank calls save; rank 0 writes
        and the other ranks wait for it."""
        import random
        from . import _lib, checkpoint
        species = {n: spp._checkpoint() for n, spp in self.comm.items()}
        payload = dict(model={k: v for k, v in self.__dict__.items() if k not in self._DEVICE_ATTRS},
                       land=self._bare_land(), comm=dict(t=self.comm.t, burned=self.comm.burned), species=species,
                       strips=_strip_world(self.strips), rng=(np.random.get_state(), random.getstate()))
        group = None if self.strips is None or isinstance(self.strips, (int, np.integer)) else self.strips
        if group is None:
            checkpoint.write(path, payload, _lib.lib().gnx_abi_version())
            return
        import torch.distributed as dist
        try:
            if dist.get_rank(group) == 0:
                checkpoint.write(path, payload, _lib.lib().gnx_abi_version())
        finally:
            dist.barrier(group=group)

    # ---- getters (model.py:2787-3176) ---------------------------------------------------
    def _spp(self, spp):
        return self.comm[spp] if isinstance(spp, int) else [s for s in self.comm.values() if s.name == spp][0]

    def get_x(self, spp=0, individs=None):
        return self._spp(spp)._get_x(individs)

    def get_y(self, spp=0, individs=None):
        return self._spp(spp)._get_y(individs)

    def get_coords(self, spp=0, individs=None, as_float=True):
        return self._spp(spp)._get_coords(individs, as_float)

    def get_cells(self, spp=0, individs=None):
        return self._spp(spp)._get_cells(individs)

    def get_age(self, spp=0, individs=None):
        return self._spp(spp)._get_age(individs)

    def get_z(self, spp=0, trait_num=None, individs=None):
        return self._spp(spp)._get_z(trait_num, individs)

    def get_e(self, spp=0, lyr_num=None, individs=None):
        return self._spp(spp)._get_e(lyr_num, individs)

    def get_fitness(self, spp=0, individs=None):
        return self._spp(spp)._get_fit(individs)

    def get_genotypes(self, spp=0, loci=None, individs=None, biallelic=True, as_dict=False):
        return self._spp(spp)._get_genotypes(loci, individs, biallelic, as_dict)

    def write_gendata(self, filepath, spp=0, n=None, include_fixed_sites=True):
        """model.py:3342-3396: VCF / FASTA of everyone or of n individuals drawn at random, by extension."""
        from . import writers
        return writers.write_gendata(filepath, self._spp(spp), n=n, include_fixed_sites=include_fixed_sites)

    def write_geodata(self, filepath, spp=0, n=None):
        """model.py:3399-3446: idx, z, e, age, sex, x, y of everyone or of n individuals drawn at random (CSV)."""
        from . import writers
        return writers.write_geodata(filepath, self._spp(spp), n=n)


def load_model(path, strips=None):
    """A Model resumed from the file Model.save wrote: walking or running it on gives what the saved model
    would have given.  strips has its meaning in make_model and need not match the decomposition the file was
    written from.  Under a process group every rank reads the file.  A file of another checkpoint format or
    C-ABI version is refused (checkpoint.CheckpointError)."""
    import random
    from . import _lib, checkpoint
    world = _strip_world(strips)
    ck = checkpoint.read(path, _lib.GNX_ABI_VERSION)
    m = Model.__new__(Model)
    m.__dict__.update(ck['model'])
    m.strips = strips
    m.land = ck['land']
    m.land._listeners = []
    spps = {n: Species._from_checkpoint(sc, m.land, strips) for n, sc in ck['species'].items()}
    if world is not None:
        for spp in spps.values():
            _check_strip_species(spp, world)
    # a capacity is per strip under a decomposition: it carries over only between single contexts
    same = world is None and ck['strips'] is None
    for n, spp in spps.items():
        spp._resume(ck['species'][n], capacity=ck['species'][n]['capacity'] if same else None)
    if not same:
        for snap in (m.orig_comm or {}).values():
            snap['capacity'] = None
    m.comm = Community(m.land, spps)
    m.comm.t, m.comm.burned = ck['comm']['t'], ck['comm']['burned']
    np.random.set_state(ck['rng'][0])
    random.setstate(ck['rng'][1])
    return m


def make_model(parameters=None, verbose=False, name=None, genome_init='host', strips=None):
    """main.py:442: a Model from a parameters-file path, a dict or a ParametersDict.  genome_init: how the
    starting genomes are assigned after the burn-in; strips: None, a strip count or a process group (Model)."""
    _check_genome_init(genome_init)
    _strip_world(strips)
    if isinstance(parameters, str):
        params = read_parameters_file(parameters)
    elif isinstance(parameters, ParametersDict):
        params = parameters
    elif isinstance(parameters, dict):
        params = make_params_dict(parameters, name or 'unnamed_model')
    else:
        raise ValueError('parameters must be a filepath, a dict or a ParametersDict')
    return Model(name or params.get('model', {}).get('name', 'unnamed_model'), params, verbose=verbose,
                 genome_init=genome_init, strips=strips)
