"""DeviceSpecies: the structure-of-arrays, HBM-resident state of one Species plus the calls
that advance it, bound to libgnxb200.so through ctypes (include/gnx_b200.h).

This is the thin host layer between the reference-shaped API objects
(geonomics_b200.api: Species / Landscape / GenomicArchitecture / Model) and the CUDA
kernels.  All per-timestep arithmetic happens in the shared library; nothing here computes
on the CPU, and constructing a DeviceSpecies without the library or without a CUDA device
raises.
"""
import ctypes as C

import numpy as np

from . import _lib
from .density import DensityGridSetup
from . import genome_pack as gp

_DT = {
    'X': np.float64, 'Y': np.float64, 'AGE': np.int32, 'SEX': np.int8, 'IDX': np.int64, 'FIT': np.float64,
    'GSLOT': np.int32, 'N_NBRS': np.int32, 'MATE': np.int32, 'PAIRS': np.int32, 'NB': np.int32,
    'PERM': np.int32, 'CELL_START': np.uint32, 'COUNTS_N': np.int32, 'COUNTS_P': np.int32,
    'VALS_N': np.float64, 'VALS_P': np.float64, 'GRAD_N': np.float64, 'GRAD_P': np.float64,
    'N_RAST': np.float64, 'NPAIRS_RAST': np.float64, 'D_RAST': np.float64, 'K_RAST': np.float64,
    'DEATH_P': np.float64, 'ALIVE': np.uint8, 'DISP_TRIES': np.int32, 'E': np.float64, 'Z': np.float64,
    'COUNTERS': np.int32, 'GENOMES': np.uint32, 'NODE0': np.int32, 'NODE1': np.int32,
    'VM_TAB_MOVE': np.float32, 'VM_TAB_DISP': np.float32,
}


def _ptr(a, typ):
    return None if a is None else a.ctypes.data_as(typ)


class _DevArray:
    """A ctx-owned device array as a __cuda_array_interface__ object (zero-copy torch view)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {'shape': (int(n),), 'typestr': typestr, 'data': (int(ptr), False),
                                         'version': 2, 'strides': None}


def stats_from_counts(c1, het, fit_sum, N):
    """DeviceSpecies.stats from the device's counts (summed over the strips of a decomposed species)."""
    Lg = len(c1)
    freq = c1 / float(2 * N) if N else np.zeros(Lg)
    return dict(N=N, freq=freq, het=het / float(N) if N else np.zeros(Lg),
                maf=np.minimum(freq, 1 - freq), mean_fit=float(fit_sum) / N if N else float('nan'))


def ld_from_counts(n11, n):
    """DeviceSpecies.ld from the chromosome counts n11 [L, L] of n individuals."""
    L = n11.shape[0]
    N = 2 * int(n)                                        # chromosomes
    n11 = n11.astype(np.float64)
    n11 = np.triu(n11) + np.triu(n11, 1).T                # only one word-triangle is filled
    f1 = np.diagonal(n11) / N
    with np.errstate(divide='ignore', invalid='ignore'):
        D = n11 / N - f1[:, None] * f1[None, :]
        r2 = (D ** 2) / (((f1 * (1 - f1))[:, None] * f1[None, :]) * (1 - f1)[None, :])
    # the reference fills (i, j) and (j, i) from the i < j evaluation
    r2 = np.triu(r2, 1) + np.triu(r2, 1).T
    r2[np.arange(L), np.arange(L)] = np.nan
    return r2


def cell_stats_from_sums(sum_diff, sum_sq_diff, ncell):
    """(mean, std) of the per-cell count changes over ncell landscape cells from their sum and sum of squares."""
    mean = sum_diff / float(ncell)
    return mean, float(np.sqrt(max(sum_sq_diff / float(ncell) - mean * mean, 0.0)))


def max_births(lam, fixed, n):
    """Most births one step of n individuals can have (k_step_guard): every focal makes at most one pair,
    so fixed births give at most lam * n; Poisson births ceil(lam n + 10 sqrt(lam n)) + 32, whose tail
    probability is below 1e-15."""
    if fixed:
        return int(lam) * int(n)
    m = float(lam) * float(n)
    return int(np.ceil(m + 10.0 * np.sqrt(m))) + 32


def growth_capacity(need, capacity):
    """The size to grow a buffer of `capacity` to when a step needs `need`: at least double, so that a
    population growing steadily re-allocates a logarithmic number of times."""
    return max(int(need), 2 * int(capacity))


class DeviceSpecies:
    """One Species resident on the GPU.

    Parameters mirror what the reference's ops read off `Species`, `Landscape` and
    `GenomicArchitecture` (SURVEY.md section 8b):

    land_dim : (dim_x, dim_y)                       landscape.py:245
    rasters  : float64[n_layers, dim_y, dim_x]      land[l].rast
    prm      : dict with b, R, lam, n_births_fixed, mating_radius, d_min, d_max, sex,
               sex_ratio_p, max_age, K_layer, K_factor, move, move_distr (name, p1, p2),
               disp_distr (name, p1, p2), direction_mu, direction_kappa, choose_nearest,
               inverse_dist, density_grid_window_width, move_surf / disp_surf (dicts or None)
    gen_arch : dict with L, paths (uint8[n_paths, L]), traits (list of dicts loci/alpha/phi/
               gamma/lyr_num/univ_adv), dom (int8[L])   or None (no genomes);
               cols (the starting non-neutral loci, ascending) selects the column layout of a use_tskit
               species (gnx_create_cols): genotype rows hold one column per non-neutral locus, and
               upload(g=...) / download()['g'] take and give the reference's rows [n, n_nonneut, 2] in
               ascending locus order; col_capacity (optional): the starting columns per row
    grow     : let the population outgrow `capacity`: every step first checks that it cannot overflow a
               buffer, and step() grows the buffers in front of a step that could (gnx_set_growth_guard);
               the run is bit-identical to one started at the larger capacity
    """

    def __init__(self, land_dim, rasters, prm, gen_arch=None, capacity=None, seed=0,
                 disp_tries_injected=6, res_ratio=(1.0, 1.0), grow=False):
        L = _lib.lib()
        self._L = L
        self.land_dim = (int(land_dim[0]), int(land_dim[1]))
        rasters = np.ascontiguousarray(rasters, dtype=np.float64)
        assert rasters.ndim == 3 and rasters.shape[1:] == (self.land_dim[1], self.land_dim[0]), \
            'rasters must be [n_layers, dim_y, dim_x]'
        self.n_layers = rasters.shape[0]
        self.prm = dict(prm)
        self.gen_arch = gen_arch
        traits = (gen_arch or {}).get('traits') or []
        self.n_traits = len(traits)
        self.Lg = int(gen_arch['L']) if gen_arch is not None else 0
        cols = None if gen_arch is None else gen_arch.get('cols')
        self.cols = cols is not None
        if self.cols:
            cols = np.ascontiguousarray(cols, dtype=np.int32)
            self.W = gp.words_per_hap(int(gen_arch.get('col_capacity') or gp.col_capacity(len(cols))))
            self.col_capacity = 32 * self.W
        else:
            self.W = gp.words_per_hap(self.Lg)
        self._col_budget = None
        if capacity is None:
            ksum = float(np.sum(rasters[int(prm.get('K_layer', 0))]) * float(prm.get('K_factor', 1.0)))
            capacity = int(max(4096, 3.0 * ksum))
        self.capacity = int(capacity)

        cfg = _lib.Config()
        cfg.abi_version = _lib.GNX_ABI_VERSION
        cfg.dim_x, cfg.dim_y = self.land_dim
        cfg.n_layers = self.n_layers
        cfg.capacity = self.capacity
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.L = self.Lg
        cfg.n_recomb_paths = int(len(gen_arch['paths'])) if gen_arch is not None else 0
        cfg.n_traits = self.n_traits
        dom = None
        if gen_arch is not None and gen_arch.get('dom') is not None and np.any(gen_arch['dom']):
            dom = np.ascontiguousarray(gen_arch['dom'], dtype=np.int8)
        cfg.use_dom = int(dom is not None)
        self._fill_life_history(cfg, prm)
        cfg.res_ratio_x, cfg.res_ratio_y = float(res_ratio[0]), float(res_ratio[1])
        self._surf_tabs = [None, None]
        approx_len = 0
        for k, (name, pre) in enumerate((('move_surf', 'move'), ('disp_surf', 'disp'))):
            s = prm.get(name)
            mode = _lib.SURF_NONE
            if s is not None:
                if s.get('table') is not None:
                    mode = _lib.SURF_TABLE
                    tab = np.ascontiguousarray(s['table'], dtype=np.float16)
                    assert tab.shape[:2] == (self.land_dim[1], self.land_dim[0])
                    assert approx_len in (0, tab.shape[2]), 'surface tables must share approx_len'
                    approx_len = tab.shape[2]
                    self._surf_tabs[k] = tab
                else:
                    mode = _lib.SURF_ONTHEFLY
                setattr(cfg, pre + '_surf_layer', int(s.get('layer', 0)))
                setattr(cfg, pre + '_surf_mixture', int(bool(s.get('mixture', True))))
                setattr(cfg, pre + '_surf_kappa', float(s.get('kappa', 12.0)))
            setattr(cfg, pre + '_surf_mode', mode)
        cfg.surf_approx_len = approx_len
        cfg.disp_max_tries_injected = int(disp_tries_injected)
        self.disp_R = int(disp_tries_injected)
        self._cfg = cfg

        self._ctx = C.c_void_p()
        if self.cols:
            _lib.check(L.gnx_create_cols(C.byref(cfg), self.col_capacity, len(cols), _ptr(cols, _lib.c_int32_p),
                                         C.byref(self._ctx)), 'gnx_create_cols')
        else:
            _lib.check(L.gnx_create(C.byref(cfg), C.byref(self._ctx)), 'gnx_create')
        _lib.check(L.gnx_set_rasters(self._ctx, _ptr(rasters, _lib.c_double_p)), 'gnx_set_rasters')
        self._rasters_host = rasters

        self.density = DensityGridSetup(self.land_dim, prm.get('density_grid_window_width'))
        dstruct = self.density.to_struct()
        _lib.check(L.gnx_set_density(self._ctx, C.byref(dstruct)), 'gnx_set_density')

        if gen_arch is not None:
            packed = gp.pack_paths(gen_arch['paths'])
            _lib.check(L.gnx_set_recomb_paths(self._ctx, _ptr(packed, _lib.c_uint32_p)), 'gnx_set_recomb_paths')
            self.set_traits(traits, dom)
        if self._surf_tabs[0] is not None or self._surf_tabs[1] is not None:
            mv = None if self._surf_tabs[0] is None else self._surf_tabs[0].view(np.uint16)
            dv = None if self._surf_tabs[1] is None else self._surf_tabs[1].view(np.uint16)
            _lib.check(L.gnx_set_surface_tables(self._ctx, _ptr(mv, _lib.c_uint16_p), _ptr(dv, _lib.c_uint16_p)),
                       'gnx_set_surface_tables')
        self._keep = []
        self.tskit_capacity = (0, 0)               # (edge, birth) rows of the tskit buffers, once enabled
        self.grow = bool(grow)
        if self.grow:
            _lib.check(L.gnx_set_growth_guard(self._ctx, 1), 'gnx_set_growth_guard')

    # ---- setup -----------------------------------------------------------------------
    def set_recomb_paths(self, paths):
        """Cached recombination paths uint8[n_paths, L], AS SIMULATED (bit l = homologue at locus l,
        genome.py:209-226); n_paths is fixed at creation."""
        packed = gp.pack_paths(np.asarray(paths, dtype=np.uint8))
        assert len(paths) == self._cfg.n_recomb_paths, 'n_recomb_paths is fixed at creation'
        _lib.check(self._L.gnx_set_recomb_paths(self._ctx, _ptr(packed, _lib.c_uint32_p)), 'gnx_set_recomb_paths')

    def set_traits(self, traits, dom=None):
        if len(traits) != self.n_traits:
            raise ValueError('the number of traits is fixed at creation')
        if dom is not None:
            dom = np.ascontiguousarray(dom, dtype=np.int8)
        arr = (_lib.Trait * max(1, len(traits)))()
        keep = []
        for t, tr in enumerate(traits):
            loci = np.ascontiguousarray(tr['loci'], dtype=np.int32)
            alpha = np.ascontiguousarray(tr['alpha'], dtype=np.float64)
            keep += [loci, alpha]
            arr[t].n_loci = len(loci)
            arr[t].host_loci = _ptr(loci, _lib.c_int32_p)
            arr[t].host_alpha = _ptr(alpha, _lib.c_double_p)
            phi = tr['phi']
            if np.ndim(phi) == 2:
                ph = np.ascontiguousarray(phi, dtype=np.float64)
                keep.append(ph)
                arr[t].host_phi_raster = _ptr(ph, _lib.c_double_p)
                arr[t].phi = 0.0
            else:
                arr[t].host_phi_raster = None
                arr[t].phi = float(phi)
            arr[t].gamma = float(tr['gamma'])
            arr[t].layer = int(tr['lyr_num'])
            arr[t].univ_adv = int(bool(tr['univ_adv']))
        _lib.check(self._L.gnx_set_traits(self._ctx, len(traits), arr, _ptr(dom, _lib.c_int8_p)),
                   'gnx_set_traits')
        self._trait_sizes = [len(tr['loci']) for tr in traits]

    def set_debug(self, on=True):
        """Keep n_nbrs / death_p / disp_tries / n_pairs raster readable (parity tests)."""
        _lib.check(self._L.gnx_set_debug(self._ctx, int(bool(on))), 'gnx_set_debug')

    @staticmethod
    def _fill_life_history(cfg, prm):
        """The scalar parameters the step reads off the Species (species.py:405-425)."""
        mr = prm.get('mating_radius')
        cfg.mating_radius = -1.0 if mr is None else float(mr)
        cfg.b = float(prm['b'])
        cfg.R = float(prm['R'])
        cfg.n_births_lambda = float(prm['lam'])
        cfg.n_births_fixed = int(bool(prm['n_births_fixed']))
        cfg.sex = int(bool(prm.get('sex', False)))
        cfg.sex_ratio_p = float(prm.get('sex_ratio_p', 0.5))
        cfg.choose_nearest = int(bool(prm.get('choose_nearest', False)))
        cfg.inverse_dist = int(bool(prm.get('inverse_dist', False)))
        cfg.d_min = float(prm.get('d_min', 0.0))
        cfg.d_max = float(prm.get('d_max', 1.0))
        cfg.max_age = -1 if prm.get('max_age') is None else int(prm['max_age'])
        cfg.K_layer = int(prm.get('K_layer', 0))
        cfg.K_factor = float(prm.get('K_factor', 1.0))
        cfg.move = int(bool(prm.get('move', True)))
        mname, mp1, mp2 = prm.get('move_distr', ('wald', 1.0, 1.0))
        dname, dp1, dp2 = prm.get('disp_distr', ('wald', 1.0, 1.0))
        cfg.move_distr = _lib.DISTR[mname]
        cfg.disp_distr = _lib.DISTR[dname]
        cfg.move_p1, cfg.move_p2, cfg.disp_p1, cfg.disp_p2 = float(mp1), float(mp2), float(dp1), float(dp2)
        cfg.dir_mu = float(prm.get('direction_mu', 0.0))
        cfg.dir_kappa = float(prm.get('direction_kappa', 0.0))

    def set_life_history(self, **changes):
        """A species life-history change event (`setattr(spp, parameter, val)`, change.py:735-742):
        keys as in the `prm` dict of the constructor (b, R, lam, n_births_fixed, d_min, d_max,
        max_age, sex_ratio_p, K_factor, move_distr, disp_distr, direction_mu, direction_kappa,
        choose_nearest, inverse_dist)."""
        prm = dict(self.prm)
        prm.update(changes)
        self._fill_life_history(self._cfg, prm)
        _lib.check(self._L.gnx_set_life_history(self._ctx, C.byref(self._cfg)), 'gnx_set_life_history')
        self.prm = prm

    def set_K(self, K):
        """A demographic change event rewrote spp.K (change.py:633-649)."""
        k = np.ascontiguousarray(K, dtype=np.float64)
        assert k.shape == (self.land_dim[1], self.land_dim[0])
        _lib.check(self._L.gnx_set_K(self._ctx, _ptr(k, _lib.c_double_p)), 'gnx_set_K')

    def set_surface_tables(self, move_tab=None, disp_tab=None):
        """Swap in re-built float16 direction tables (change.py:597-606: a landscape change on the
        layer behind a conductance surface re-builds the _ConductanceSurface)."""
        tabs = []
        for k, t in enumerate((move_tab, disp_tab)):
            if t is None:
                tabs.append(None)
                continue
            t = np.ascontiguousarray(t, dtype=np.float16)
            assert self._surf_tabs[k] is not None and t.shape == self._surf_tabs[k].shape, \
                'surface table shape must match the one given at construction'
            self._surf_tabs[k] = t
            tabs.append(t.view(np.uint16))
        _lib.check(self._L.gnx_set_surface_tables(
            self._ctx, None if tabs[0] is None else _ptr(tabs[0], _lib.c_uint16_p),
            None if tabs[1] is None else _ptr(tabs[1], _lib.c_uint16_p)), 'gnx_set_surface_tables')

    def set_burn(self, burn):
        _lib.check(self._L.gnx_set_burn(self._ctx, int(bool(burn))), 'gnx_set_burn')

    def set_raster(self, layer, rast):
        """Landscape._set_raster (landscape.py:353) for an environmental-change event."""
        r = np.ascontiguousarray(rast, dtype=np.float64)
        assert r.shape == (self.land_dim[1], self.land_dim[0])
        _lib.check(self._L.gnx_set_raster(self._ctx, int(layer), _ptr(r, _lib.c_double_p)), 'gnx_set_raster')

    def set_draws(self, draws):
        """Inject replayed random draws (dict of arrays, see gnx_draws_t) or None for Philox."""
        if draws is None:
            _lib.check(self._L.gnx_set_draws(self._ctx, None), 'gnx_set_draws')
            return
        d = _lib.Draws()
        keep = []

        # the C struct carries one row count for every array: pad all of them (zeros) to the
        # longest one so no site reads past its buffer
        widths = dict(recomb_keys=2, start_homs=2, pan_R=2, disp_dir=self.disp_R, disp_choice=self.disp_R,
                      disp_dist=self.disp_R)
        n = max([np.asarray(v).size // widths.get(k, 1) for k, v in draws.items()
                 if v is not None and not k.startswith('mut_')] + [0])

        def put(name, key, dtype, typ, width=1):
            a = draws.get(key)
            if a is None:
                return
            a = np.ascontiguousarray(a, dtype=dtype).reshape(-1)
            if a.size < n * width:
                a = np.concatenate([a, np.zeros(n * width - a.size, dtype=dtype)])
            keep.append(a)
            setattr(d, name, _ptr(a, typ))
        R = self.disp_R
        put('move_dir', 'move_dir', np.float64, _lib.c_double_p)
        put('move_choice', 'move_choice', np.int32, _lib.c_int32_p)
        put('move_dist', 'move_dist', np.float64, _lib.c_double_p)
        put('mate_R', 'mate_R', np.uint32, _lib.c_uint32_p)
        put('mate_inv_u', 'mate_inv_u', np.float64, _lib.c_double_p)
        put('mate_u', 'mate_u', np.float64, _lib.c_double_p)
        put('poisson', 'poisson', np.int32, _lib.c_int32_p)
        put('recomb_keys', 'recomb_keys', np.int32, _lib.c_int32_p, 2)
        put('start_homs', 'start_homs', np.int32, _lib.c_int32_p, 2)
        for key in ('disp_dir', 'disp_choice', 'disp_dist'):
            a = draws.get(key)
            if a is not None:
                assert np.asarray(a).shape[1] == R, '%s must have %d columns' % (key, R)
        put('disp_dir', 'disp_dir', np.float64, _lib.c_double_p, R)
        put('disp_choice', 'disp_choice', np.int32, _lib.c_int32_p, R)
        put('disp_dist', 'disp_dist', np.float64, _lib.c_double_p, R)
        put('sex_u', 'sex_u', np.float64, _lib.c_double_p)
        put('sex_redraw_u', 'sex_redraw_u', np.float64, _lib.c_double_p)
        put('death_u', 'death_u', np.float64, _lib.c_double_p)
        put('pan_u', 'pan_u', np.float64, _lib.c_double_p)
        put('pan_R', 'pan_R', np.uint32, _lib.c_uint32_p, 2)
        d.n = int(n)
        # mutation draws (their own row count: one row per mutation)
        if draws.get('mut_n') is not None:
            nm = max([np.asarray(draws[k]).size for k in ('mut_type_u', 'mut_ind_R', 'mut_homol_u', 'mut_s', 'mut_alpha')
                      if draws.get(k) is not None] + [0])
            n, n_rows = nm, n
            keep.append(np.ascontiguousarray(np.asarray(draws['mut_n']).reshape(-1)[:1], dtype=np.int32))
            d.mut_n = _ptr(keep[-1], _lib.c_int32_p)
            put('mut_type_u', 'mut_type_u', np.float64, _lib.c_double_p)
            put('mut_ind_R', 'mut_ind_R', np.uint32, _lib.c_uint32_p)
            put('mut_homol_u', 'mut_homol_u', np.float64, _lib.c_double_p)
            put('mut_s', 'mut_s', np.float64, _lib.c_double_p)
            put('mut_alpha', 'mut_alpha', np.float64, _lib.c_double_p)
            d.n_mut = int(nm)
            n = n_rows
        _lib.check(self._L.gnx_set_draws(self._ctx, C.byref(d)), 'gnx_set_draws')

    # ---- a13 mutation ------------------------------------------------------------------------
    def set_mutation(self, mu_neut, mu_delet, mutables, nonneut_loci, delet_loci=(), delet_s=(),
                     delet_s_shape=0.2, delet_s_scale=0.2, log_capacity=4096, tskit_layout=False,
                     trait_mus=None, trait_alpha_distr=None, trait_loci_idxs=None, delet_loci_idxs=None,
                     subsetters=None):
        """Enable mutation of each step's offspring (ops/mutation.py:169-206).
        mutables: the shuffled list of mutable loci (genome.py:1101-1104), popped from its end.
        tskit_layout: gen_arch.use_tskit = True semantics (genotype rows = non-neutral loci; see
        include/gnx_b200.h); trait_mus [T] with trait_alpha_distr [T][3] (alpha_distr_mu, alpha_distr_sigma,
        max_alpha_mag or None) enables trait mutation; trait_loci_idxs (list of arrays, Trait.loci_idxs),
        delet_loci_idxs and subsetters [n_paths, n_nonneut] carry the reference's arrays as it left them."""
        m = _lib.Mutation()
        m.mu_neut, m.mu_delet = float(mu_neut), float(mu_delet)
        m.delet_s_shape, m.delet_s_scale = float(delet_s_shape), float(delet_s_scale)
        mt = np.ascontiguousarray(mutables, dtype=np.int32)
        nn = np.ascontiguousarray(nonneut_loci, dtype=np.int32)
        dl = np.ascontiguousarray(delet_loci, dtype=np.int32)
        ds = np.ascontiguousarray(delet_s, dtype=np.float64)
        m.n_mutables, m.host_mutables = len(mt), _ptr(mt, _lib.c_int32_p)
        m.n_nonneut, m.host_nonneut_loci = len(nn), _ptr(nn, _lib.c_int32_p)
        m.n_delet, m.host_delet_loci, m.host_delet_s = len(dl), _ptr(dl, _lib.c_int32_p), _ptr(ds, _lib.c_double_p)
        m.log_capacity = int(log_capacity)
        m.tskit_layout = 1 if tskit_layout else 0
        keep = []
        if trait_mus is not None and any(float(v) > 0 for v in trait_mus):
            tm = np.ascontiguousarray(trait_mus, dtype=np.float64)
            assert len(tm) == self.n_traits
            ad = np.array([[a[0], a[1], -1.0 if a[2] is None else a[2]] for a in trait_alpha_distr], dtype=np.float64)
            assert ad.shape == (self.n_traits, 3)
            keep += [tm, ad]
            m.host_trait_mu = _ptr(tm, _lib.c_double_p)
            m.host_trait_alpha_distr = _ptr(ad, _lib.c_double_p)
        elif trait_alpha_distr is not None:
            ad = np.array([[a[0], a[1], -1.0 if a[2] is None else a[2]] for a in trait_alpha_distr], dtype=np.float64)
            keep.append(ad)
            m.host_trait_alpha_distr = _ptr(ad, _lib.c_double_p)
        if trait_loci_idxs is not None:
            if [len(v) for v in trait_loci_idxs] != list(getattr(self, '_trait_sizes', [])):
                raise ValueError('trait_loci_idxs must hold one index per locus of the traits last given to set_traits')
            ti = np.ascontiguousarray(np.concatenate([np.asarray(v, dtype=np.int32).reshape(-1)
                                                      for v in trait_loci_idxs] + [np.zeros(0, np.int32)]), dtype=np.int32)
            keep.append(ti)
            m.host_trait_loci_idxs = _ptr(ti, _lib.c_int32_p)
        if delet_loci_idxs is not None:
            di = np.ascontiguousarray(delet_loci_idxs, dtype=np.int32)
            assert len(di) == len(dl)
            keep.append(di)
            m.host_delet_loci_idxs = _ptr(di, _lib.c_int32_p)
        if subsetters is not None:
            sb = np.ascontiguousarray(subsetters, dtype=np.uint8)
            assert sb.ndim == 2 and sb.shape[1] == len(nn), (sb.shape, len(nn))
            keep.append(sb)
            m.host_subsetters = sb.ctypes.data_as(C.POINTER(C.c_uint8))
        _lib.check(self._L.gnx_set_mutation(self._ctx, C.byref(m)), 'gnx_set_mutation')
        self._mut_tskit = bool(tskit_layout)
        if self.cols:
            nonneutral = float(mu_delet) > 0 or (trait_mus is not None and any(float(v) > 0 for v in trait_mus))
            self._col_budget = gp.ColumnBudget(len(self.read_cols()), self.col_capacity,
                                               gp.MUT_MAX_NEW if nonneutral else 0, 128 * ((self.Lg + 127) // 128))

    # ---- column layout -----------------------------------------------------------------------
    def read_cols(self):
        """int32[n_cols]: the locus of every column, in column order (gnx_read_cols; synchronises)."""
        out = np.zeros(max(1, self.Lg), np.int32)
        n, cap = C.c_int32(), C.c_int32()
        _lib.check(self._L.gnx_read_cols(self._ctx, _ptr(out, _lib.c_int32_p), C.byref(n), C.byref(cap)),
                   'gnx_read_cols')
        return out[:n.value].copy()

    def widen_cols(self, col_capacity):
        """Re-pack the rows to col_capacity columns (between steps; the next step captures its graph again)."""
        _lib.check(self._L.gnx_widen_cols(self._ctx, int(col_capacity)), 'gnx_widen_cols')
        self.W = gp.words_per_hap(col_capacity)
        self.col_capacity = 32 * self.W
        if self._col_budget is not None:
            self._col_budget.capacity = self.col_capacity

    @staticmethod
    def _mut_type_name(t):
        return ('neut', 'delet')[t] if t < 2 else 't%i' % (t - 2)

    def read_mutations(self, max_rows=4096):
        """Drain the mutation log; returns (rows, state) with rows a list of dicts (t, individual,
        locus, row, homologue, type, s, alpha, node) and state the current bookkeeping arrays."""
        rows = (_lib.MutationRow * max_rows)()
        n_rows, n_left, n_nn, n_dl = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
        nn = np.zeros(self.Lg + 1, np.int32)
        dl = np.zeros(self.Lg + 1, np.int32)
        ds = np.zeros(self.Lg + 1, np.float64)
        _lib.check(self._L.gnx_read_mutations(
            self._ctx, rows, max_rows, C.byref(n_rows), C.byref(n_left), _ptr(nn, _lib.c_int32_p), C.byref(n_nn),
            _ptr(dl, _lib.c_int32_p), _ptr(ds, _lib.c_double_p), C.byref(n_dl)), 'gnx_read_mutations')
        out = [dict(t=r.t, individual=r.individual, locus=r.locus, row=r.row, homologue=r.homologue,
                    type=self._mut_type_name(r.type), s=r.s, alpha=r.alpha, node=r.node) for r in rows[:n_rows.value]]
        state = dict(n_mutables=n_left.value, nonneut_loci=nn[:n_nn.value].copy(),
                     delet_loci=dl[:n_dl.value].copy(), delet_s=ds[:n_dl.value].copy())
        return out, state

    def read_mutation_tables(self):
        """(Trait.loci, Trait.alpha, Trait.loci_idxs) per trait and gen_arch.delet_loci_idxs as the mutations
        left them (genome.py:416-437, 753-788)."""
        traits = []
        cap = self.Lg + 1
        di = np.zeros(cap, np.int32)
        for t in range(self.n_traits):
            n = C.c_int32(0)
            lo, al, ix = np.zeros(cap, np.int32), np.zeros(cap, np.float64), np.zeros(cap, np.int32)
            _lib.check(self._L.gnx_read_mutation_tables(
                self._ctx, t, C.byref(n), _ptr(lo, _lib.c_int32_p), _ptr(al, _lib.c_double_p), _ptr(ix, _lib.c_int32_p),
                _ptr(di, _lib.c_int32_p)), 'gnx_read_mutation_tables')
            traits.append(dict(loci=lo[:n.value].copy(), alpha=al[:n.value].copy(), loci_idxs=ix[:n.value].copy()))
        if not self.n_traits:
            _lib.check(self._L.gnx_read_mutation_tables(self._ctx, -1, None, None, None, None, _ptr(di, _lib.c_int32_p)),
                       'gnx_read_mutation_tables')
        n_dl = C.c_int32(0)
        _lib.check(self._L.gnx_read_mutations(self._ctx, None, 0, None, None, None, None, None, None, C.byref(n_dl)),
                   'gnx_read_mutations')
        return traits, di[:n_dl.value].copy()

    # ---- population in / out ---------------------------------------------------------------
    def _pop_struct(self, bufs):
        p = _lib.Population()
        p.n = int(bufs.get('n', 0))
        p.x = _ptr(bufs.get('x'), _lib.c_double_p)
        p.y = _ptr(bufs.get('y'), _lib.c_double_p)
        p.age = _ptr(bufs.get('age'), _lib.c_int32_p)
        p.sex = _ptr(bufs.get('sex'), _lib.c_int8_p)
        p.idx = _ptr(bufs.get('idx'), _lib.c_int64_p)
        p.genomes = _ptr(bufs.get('genomes'), _lib.c_uint32_p)
        p.z = _ptr(bufs.get('z'), _lib.c_double_p)
        p.fit = _ptr(bufs.get('fit'), _lib.c_double_p)
        p.e = _ptr(bufs.get('e'), _lib.c_double_p)
        p.max_ind_idx = int(bufs.get('max_ind_idx', -1))
        return p

    def upload(self, x, y, age=None, sex=None, idx=None, g=None, z=None, max_ind_idx=None,
               genomes_packed=None, fit=None):
        """Upload a population in species order.  g: int8[N, L, 2] (reference layout) or
        genomes_packed: u32[N, 2, W]; z and fit as downloaded (z otherwise follows from the genomes)."""
        n = len(x)
        bufs = dict(n=n, x=np.ascontiguousarray(x, dtype=np.float64), y=np.ascontiguousarray(y, dtype=np.float64))
        if age is not None:
            bufs['age'] = np.ascontiguousarray(age, dtype=np.int32)
        if sex is not None:
            bufs['sex'] = np.ascontiguousarray(sex, dtype=np.int8)
        if idx is not None:
            bufs['idx'] = np.ascontiguousarray(idx, dtype=np.int64)
        if genomes_packed is None and g is not None:
            genomes_packed = gp.rows_to_cols(g, self.read_cols(), self.W) if self.cols else gp.pack_genomes(g)
        if genomes_packed is not None:
            gpk = np.ascontiguousarray(genomes_packed, dtype=np.uint32)
            assert gpk.shape == (n, 2, self.W), (gpk.shape, (n, 2, self.W))
            bufs['genomes'] = gpk
        if z is not None and self.n_traits:
            bufs['z'] = np.ascontiguousarray(z, dtype=np.float64).reshape(n, self.n_traits)
        if fit is not None:
            bufs['fit'] = np.ascontiguousarray(fit, dtype=np.float64)
        if max_ind_idx is None:
            max_ind_idx = int(np.max(idx)) if idx is not None and n else n - 1
        bufs['max_ind_idx'] = max_ind_idx
        p = self._pop_struct(bufs)
        _lib.check(self._L.gnx_upload_population(self._ctx, C.byref(p)), 'gnx_upload_population')

    def population_size(self):
        n = C.c_int64()
        _lib.check(self._L.gnx_population_size(self._ctx, C.byref(n)), 'gnx_population_size')
        return int(n.value)

    def download(self, genomes=True, unpack=True, e=False):
        n = self.population_size()
        bufs = dict(n=n, x=np.empty(n), y=np.empty(n), age=np.empty(n, np.int32), sex=np.empty(n, np.int8),
                    idx=np.empty(n, np.int64), fit=np.empty(n))
        if self.n_traits:
            bufs['z'] = np.empty((n, self.n_traits))
        if genomes and self.gen_arch is not None:
            bufs['genomes'] = np.empty((n, 2, self.W), np.uint32)
        if e:
            bufs['e'] = np.empty((n, self.n_layers))
        p = self._pop_struct(bufs)
        _lib.check(self._L.gnx_download_population(self._ctx, C.byref(p)), 'gnx_download_population')
        out = {k: v for k, v in bufs.items() if k != 'n'}
        out['max_ind_idx'] = int(p.max_ind_idx)
        if 'genomes' in out and self.cols:
            out['col_locus'] = self.read_cols()
            if unpack:
                out['g'] = gp.cols_to_rows(out['genomes'], out['col_locus'])
        elif 'genomes' in out and unpack:
            out['g'] = gp.unpack_genomes(out['genomes'], self.Lg)
        return out

    def walk_host(self, bufs, n_steps):
        """gnx_walk_host: host buffers in, n_steps on the device, host buffers out."""
        p = self._pop_struct(bufs)
        _lib.check(self._L.gnx_walk_host(self._ctx, C.byref(p), int(n_steps)), 'gnx_walk_host')
        bufs['n'] = int(p.n)
        bufs['max_ind_idx'] = int(p.max_ind_idx)
        return bufs

    def walk_host_begin(self, bufs, n_steps):
        """gnx_walk_host_begin: enqueue upload + n_steps; returns at once (bufs must be pinned)."""
        self._inflight = self._pop_struct(bufs)
        _lib.check(self._L.gnx_walk_host_begin(self._ctx, C.byref(self._inflight), int(n_steps)),
                   'gnx_walk_host_begin')

    def walk_host_end(self, bufs):
        """gnx_walk_host_end: wait for the steps and copy the population out into bufs."""
        p = self._pop_struct(bufs)
        _lib.check(self._L.gnx_walk_host_end(self._ctx, C.byref(p)), 'gnx_walk_host_end')
        self._inflight = None
        bufs['n'] = int(p.n)
        bufs['max_ind_idx'] = int(p.max_ind_idx)
        return bufs

    # ---- device assignment of the starting genomes (gnx_genome_init_*) ----------------------
    def genome_init_begin(self, n_carriers, seed, write_mask=None, tskit_rows=False):
        """Start the staged assignment: exactly n_carriers[l] 1-alleles at locus l.  Returns the
        int32[L * 2048] digit histogram of this context as a torch view (summed over the strips of a
        decomposed landscape before every genome_init_pass)."""
        import torch
        nc = np.ascontiguousarray(n_carriers, dtype=np.int64)
        gi = _lib.GenomeInit()
        gi.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        gi.n_loci = len(nc)
        gi.host_n_carriers = _ptr(nc, _lib.c_int64_p)
        wm = None
        if write_mask is not None:
            wm = np.ascontiguousarray(write_mask, dtype=np.uint8)
            assert wm.shape == nc.shape, 'write_mask must hold one flag per locus'
            gi.host_write_mask = wm.ctypes.data_as(C.POINTER(C.c_uint8))
        gi.tskit_rows = int(bool(tskit_rows))
        ptr, n = C.c_void_p(), C.c_int64()
        _lib.check(self._L.gnx_genome_init_begin(self._ctx, C.byref(gi), C.byref(ptr), C.byref(n)),
                   'gnx_genome_init_begin')
        return torch.as_tensor(_DevArray(ptr.value, n.value, '<i4'), device='cuda')

    def genome_init_pass(self):
        """Select from the (summed) histogram; True when every locus is resolved."""
        done = C.c_int32()
        _lib.check(self._L.gnx_genome_init_pass(self._ctx, C.byref(done)), 'gnx_genome_init_pass')
        return bool(done.value)

    def genome_init_end(self):
        _lib.check(self._L.gnx_genome_init_end(self._ctx), 'gnx_genome_init_end')

    def genome_init_rows(self):
        """(site, idx, homologue) of every starting carrier at every locus, sorted by (site, idx, homologue)."""
        n = C.c_int64()
        _lib.check(self._L.gnx_genome_init_rows(self._ctx, None, None, None, 0, C.byref(n)), 'gnx_genome_init_rows')
        site, idx, hom = np.empty(n.value, np.int32), np.empty(n.value, np.int64), np.empty(n.value, np.int8)
        _lib.check(self._L.gnx_genome_init_rows(self._ctx, _ptr(site, _lib.c_int32_p), _ptr(idx, _lib.c_int64_p),
                                                _ptr(hom, _lib.c_int8_p), n.value, C.byref(n)), 'gnx_genome_init_rows')
        o = np.lexsort((hom, idx, site))
        return dict(site=site[o], idx=idx[o], homologue=hom[o])

    def init_genomes(self, p, seed, write_mask=None, tskit_rows=False):
        """Assign the starting genomes on the device (the post-burn-in assignment of species.py:956-1094
        without a host genotype array): locus l gets exactly genome_pack.carrier_counts(n, p)[l] 1-alleles,
        on the homologues with the smallest Philox keys (include/gnx_b200.h).  write_mask [L]: loci whose
        bits are set (the non-neutral loci of the tskit layout), None: all.  tskit_rows: return the
        starting carriers of every locus (genome_init_rows)."""
        self.genome_init_begin(gp.carrier_counts(self.population_size(), p), seed, write_mask, tskit_rows)
        while not self.genome_init_pass():
            pass
        self.genome_init_end()
        return self.genome_init_rows() if tskit_rows else None

    # ---- stepping ------------------------------------------------------------------------
    def step(self, n_steps=1, sync=False):
        """Enqueue n_steps steps.  With grow, the population capacity is grown (reserve) in front of any
        step that could outgrow it, and the call returns None once every step ran, or the step_status()
        dict, with 'steps_left', of a stop on the tskit row buffers (the caller drains them, grows them
        with tskit_reserve if one step still needs more, and steps on)."""
        n_steps = int(n_steps)
        while n_steps > 0:
            k = n_steps
            if self._col_budget is not None:
                # column layout: widen before a step could run out of free columns
                k, cap = self._col_budget.take(n_steps, lambda: len(self.read_cols()))
                if cap > self.col_capacity:
                    self.widen_cols(cap)
            _lib.check(self._L.gnx_step(self._ctx, k), 'gnx_step')
            if not self.grow:
                n_steps -= k
                continue
            st = self.step_status()
            n_steps -= st['steps_run']
            if not st['stopped']:
                continue
            need = max(st['need_entries'], st['need_slots'])
            if need > self.capacity:
                self.reserve(growth_capacity(need, self.capacity))
            else:
                st['steps_left'] = n_steps
                return st
        if sync:
            self.sync()
        return None

    def step_status(self):
        """The last gnx_step batch (grow only; synchronises): steps_run, stopped, and the capacities the
        next step needs (need_entries, need_slots, need_births, need_edges) beside the current ones."""
        s = _lib.StepStatus()
        _lib.check(self._L.gnx_step_status(self._ctx, C.byref(s)), 'gnx_step_status')
        return {name: int(getattr(s, name)) for name, _ in s._fields_}

    def reserve(self, capacity):
        """Grow the population capacity to `capacity` individuals (never shrinks; between steps)."""
        _lib.check(self._L.gnx_reserve(self._ctx, int(capacity)), 'gnx_reserve')
        self.capacity = max(self.capacity, int(capacity))
        self._cfg.capacity = self.capacity

    def tskit_reserve(self, edge_capacity, birth_capacity):
        """Grow the tskit row buffers, keeping the rows buffered since the last drain."""
        _lib.check(self._L.gnx_tskit_reserve(self._ctx, int(edge_capacity), int(birth_capacity)),
                   'gnx_tskit_reserve')
        self.tskit_capacity = (max(self.tskit_capacity[0], int(edge_capacity)),
                               max(self.tskit_capacity[1], int(birth_capacity)))

    # ---- checkpoints ---------------------------------------------------------------------------
    def clock(self):
        """(t, tsk_t0): the step counter that keys every draw and the tskit time origin (synchronises)."""
        c = self.counters()
        return c['t'], c['tsk_t0']

    def set_clock(self, t, tsk_t0=0):
        """Continue the draws of a saved run (gnx_set_clock): after the upload, set_mutation and the tskit
        calls, between steps."""
        _lib.check(self._L.gnx_set_clock(self._ctx, int(t), int(tsk_t0)), 'gnx_set_clock')

    def read_paths(self):
        """uint32[n_paths, 4 * Wq]: the recombination paths the gamete kernel reads, at the genotype bits
        (gnx_read_paths); under the tskit layout they carry the patches of the columns mutations added."""
        out = np.zeros((self._cfg.n_recomb_paths, self.W), np.uint32)
        _lib.check(self._L.gnx_read_paths(self._ctx, _ptr(out, _lib.c_uint32_p), out.size), 'gnx_read_paths')
        return out

    def simplify_tables(self, tc, sample_nodes):
        """TableCollection.sort() + simplify(sample_nodes, filter_individuals=True, filter_sites=False) of a
        tables.TableColumns on this context's device (gnx_simplify), in place; row for row what
        tables.simplify_columns gives.  The columns are copied up, simplified and copied back."""
        cols = {}

        def col(name, a, dtype, typ):
            cols[name] = np.ascontiguousarray(a, dtype=dtype)
            return _ptr(cols[name], typ)

        f8, i4, i8 = (np.float64, _lib.c_double_p), (np.int32, _lib.c_int32_p), (np.int64, _lib.c_int64_p)
        t = _lib.Tables()
        t.sequence_length = float(tc.sequence_length)
        t.n_nodes, t.n_edges = tc.nodes.num_rows, tc.edges.num_rows
        t.n_individuals, t.n_location = tc.individuals.num_rows, tc.n_loc
        t.n_sites, t.n_mutations = tc.sites.num_rows, tc.mutations.num_rows
        t.node_time = col('nt', tc.nodes.time, *f8)
        t.node_population = col('np', tc.nodes.population, *i4)
        t.node_individual = col('ni', tc.nodes.individual, *i4)
        t.edge_left, t.edge_right = col('el', tc.edges.left, *f8), col('er', tc.edges.right, *f8)
        t.edge_parent, t.edge_child = col('ep', tc.edges.parent, *i4), col('ec', tc.edges.child, *i4)
        t.individual_flags = col('if', tc.individuals.flags, *i4)
        t.individual_location = col('il', tc.individuals.location, *f8)
        t.individual_idx = col('ii', tc.individuals.idx, *i8)
        t.site_position = col('sp', tc.sites.position, *f8)
        t.mutation_site, t.mutation_node = col('ms', tc.mutations.site, *i4), col('mn', tc.mutations.node, *i4)
        t.mutation_time = col('mt', tc.mutations.time, *f8)
        samples = np.ascontiguousarray(sample_nodes, dtype=np.int32)
        sizes = np.zeros(4, np.int64)
        _lib.check(self._L.gnx_simplify(self._ctx, C.byref(t), _ptr(samples, _lib.c_int32_p), len(samples),
                                        _ptr(sizes, _lib.c_int64_p)), 'gnx_simplify')
        nn, ne, ni, nm = (int(v) for v in sizes)
        nodes = dict(flags=np.zeros(nn, np.int32), time=np.zeros(nn), population=np.zeros(nn, np.int32),
                     individual=np.zeros(nn, np.int32))
        edges = dict(left=np.zeros(ne), right=np.zeros(ne), parent=np.zeros(ne, np.int32), child=np.zeros(ne, np.int32))
        inds = dict(flags=np.zeros(ni, np.int32), location=np.zeros((ni, tc.n_loc)), idx=np.zeros(ni, np.int64))
        muts = dict(site=np.zeros(nm, np.int32), node=np.zeros(nm, np.int32), time=np.zeros(nm))
        o = _lib.Tables()
        o.sequence_length, o.n_location = t.sequence_length, tc.n_loc
        o.n_nodes, o.n_edges, o.n_individuals, o.n_sites, o.n_mutations = nn, ne, ni, t.n_sites, nm
        o.node_flags, o.node_time = _ptr(nodes['flags'], _lib.c_int32_p), _ptr(nodes['time'], _lib.c_double_p)
        o.node_population = _ptr(nodes['population'], _lib.c_int32_p)
        o.node_individual = _ptr(nodes['individual'], _lib.c_int32_p)
        o.edge_left, o.edge_right = _ptr(edges['left'], _lib.c_double_p), _ptr(edges['right'], _lib.c_double_p)
        o.edge_parent, o.edge_child = _ptr(edges['parent'], _lib.c_int32_p), _ptr(edges['child'], _lib.c_int32_p)
        o.individual_flags = _ptr(inds['flags'], _lib.c_int32_p)
        o.individual_location = _ptr(inds['location'], _lib.c_double_p)
        o.individual_idx = _ptr(inds['idx'], _lib.c_int64_p)
        o.mutation_site, o.mutation_node = _ptr(muts['site'], _lib.c_int32_p), _ptr(muts['node'], _lib.c_int32_p)
        o.mutation_time = _ptr(muts['time'], _lib.c_double_p)
        _lib.check(self._L.gnx_simplify_result(self._ctx, C.byref(o)), 'gnx_simplify_result')
        for tab in (tc.nodes, tc.edges, tc.individuals, tc.mutations):
            tab.truncate(0)
        tc.individuals.append_columns(**inds)
        tc.nodes.append_columns(**nodes)
        tc.edges.append_columns(**edges)
        tc.mutations.append_columns(**muts)
        return tc

    def subsetters(self):
        """uint8[n_paths, n_cols]: the homologue every path reads at each non-neutral locus in ascending locus
        order -- the `subsetters` argument of set_mutation that rebuilds the paths read_paths returns."""
        col_locus = self.read_cols()
        bits = np.argsort(col_locus, kind='stable')                 # the column of each ascending locus
        rows = self.read_paths()
        return ((rows[:, bits >> 5] >> (bits & 31).astype(np.uint32)) & 1).astype(np.uint8)

    def sync(self):
        _lib.check(self._L.gnx_sync(self._ctx), 'gnx_sync')

    def stage(self, name):
        fn = getattr(self._L, 'gnx_' + name)
        _lib.check(fn(self._ctx), 'gnx_' + name)

    def step_records(self, max_records=1 << 16):
        arr = (_lib.StepRecord * max_records)()
        n = C.c_int32()
        _lib.check(self._L.gnx_read_step_records(self._ctx, arr, max_records, C.byref(n)), 'gnx_read_step_records')
        return [dict(t=r.t, Nt=r.Nt, n_births=r.n_births, n_deaths=r.n_deaths, n_pairs=r.n_pairs)
                for r in arr[:n.value]]

    # ---- tskit record buffering (species.py:692-736) ---------------------------------------
    def tskit_enable(self, edge_capacity, birth_capacity):
        _lib.check(self._L.gnx_tskit_enable(self._ctx, int(edge_capacity), int(birth_capacity)), 'gnx_tskit_enable')
        self.tskit_capacity = (int(edge_capacity), int(birth_capacity))

    def tskit_set_nodes(self, node0, node1, next_node_id, next_individual_row):
        a = np.ascontiguousarray(node0, dtype=np.int32)
        b = np.ascontiguousarray(node1, dtype=np.int32)
        _lib.check(self._L.gnx_tskit_set_nodes(self._ctx, _ptr(a, _lib.c_int32_p), _ptr(b, _lib.c_int32_p), len(a),
                                               int(next_node_id), int(next_individual_row)), 'gnx_tskit_set_nodes')

    def tskit_renumber(self):
        _lib.check(self._L.gnx_tskit_renumber(self._ctx), 'gnx_tskit_renumber')

    def tskit_drain(self):
        """Rows buffered since the last drain, as numpy columns ready for
        tskit.TableCollection.{edges,nodes,individuals}.append_columns."""
        q = _lib.TskitRows()
        _lib.check(self._L.gnx_tskit_drain(self._ctx, C.byref(q)), 'gnx_tskit_drain')
        ne, nb, T = int(q.n_edges), int(q.n_births), self.n_traits
        out = dict(left=np.empty(ne), right=np.empty(ne), parent=np.empty(ne, np.int32), child=np.empty(ne, np.int32),
                   idx=np.empty(nb, np.int64), x=np.empty(nb), y=np.empty(nb), z=np.empty((max(1, T), nb)),
                   time=np.empty(nb))
        r = _lib.TskitRows()
        r.n_edges, r.n_births = ne, nb
        r.edge_left, r.edge_right = _ptr(out['left'], _lib.c_double_p), _ptr(out['right'], _lib.c_double_p)
        r.edge_parent, r.edge_child = _ptr(out['parent'], _lib.c_int32_p), _ptr(out['child'], _lib.c_int32_p)
        r.birth_idx = _ptr(out['idx'], _lib.c_int64_p)
        r.birth_x, r.birth_y = _ptr(out['x'], _lib.c_double_p), _ptr(out['y'], _lib.c_double_p)
        r.birth_z, r.birth_time = _ptr(out['z'], _lib.c_double_p), _ptr(out['time'], _lib.c_double_p)
        _lib.check(self._L.gnx_tskit_drain(self._ctx, C.byref(r)), 'gnx_tskit_drain')
        out['z'] = out['z'][:T].T.copy()
        out['first_node_id'] = int(r.first_node_id)
        out['first_individual_row'] = int(r.first_individual_row)
        # nodes table columns of birth k: ids first_node_id + 2k (+1), flags 1, population 0
        out['node_time'] = np.repeat(out['time'], 2)
        out['node_individual'] = np.repeat(out['first_individual_row'] + np.arange(nb), 2)
        return out

    def stat_counts(self, region=None):
        """The integer counts behind `stats` and the fitness sum: (c1 u64[L], het u64[L], fit_sum, n)."""
        c1 = np.zeros(max(1, self.Lg), dtype=np.uint64)
        het = np.zeros(max(1, self.Lg), dtype=np.uint64)
        fs = C.c_double()
        n = C.c_int64()
        x0, x1, y0, y1 = region if region is not None else (-1e300, 1e300, -1e300, 1e300)
        _lib.check(self._L.gnx_stats_genotypes_region(
            self._ctx, float(x0), float(x1), float(y0), float(y1), c1.ctypes.data_as(C.POINTER(C.c_uint64)),
            het.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(fs), C.byref(n)), 'gnx_stats_genotypes_region')
        return c1[:self.Lg], het[:self.Lg], float(fs.value), int(n.value)

    def stats(self, region=None):
        """Per-locus statistics computed on the device from the packed genotypes
        (sim/stats.py:399-435): dict(N, freq, het, maf, mean_fit).  region = (x_min, x_max,
        y_min, y_max) restricts them to the individuals in that half-open rectangle."""
        return stats_from_counts(*self.stat_counts(region))

    def ld_counts(self):
        """(n11 u64[L, L], n): the chromosome counts behind `ld` (gnx_stats_ld)."""
        L = self.Lg
        Lp = 32 * ((L + 31) // 32)
        n11 = np.zeros((Lp, Lp), dtype=np.uint64)
        n = C.c_int64()
        _lib.check(self._L.gnx_stats_ld(self._ctx, n11.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(n)),
                   'gnx_stats_ld')
        return n11[:L, :L], int(n.value)

    def ld(self):
        """r^2 between every pair of loci (sim/stats.py:359-392 _calc_ld): the L x L matrix the
        reference returns (NaN on the diagonal), formed with the reference's own expression from
        the chromosome counts n11[i][j] that the device accumulates (gnx_stats_ld)."""
        return ld_from_counts(*self.ld_counts())

    def burnin_cell_stats(self):
        """(mean, std) of the change of the per-cell individual counts since the previous call
        (sim/burnin.py:41-58 SpatialTester.update: np.mean(diff), np.std(diff))."""
        s1, s2 = C.c_int64(), C.c_int64()
        _lib.check(self._L.gnx_burnin_cell_stats(self._ctx, C.byref(s1), C.byref(s2)), 'gnx_burnin_cell_stats')
        return cell_stats_from_sums(s1.value, s2.value, self.land_dim[0] * self.land_dim[1])

    def fst(self, region_a, region_b, est_Hs=False):
        """Per-locus pairwise Fst = (Ht - Hs) / Ht between two rectangular sub-populations, as in the
        reference's validation suite (tests/validation/island/island_test.py:54-68 calc_Fst_HsHt):
        Ht = 2 pbar (1 - pbar), Hs = mean observed heterozygosity of the two (or p(1-p) summed
        with est_Hs); NaN where the two frequencies are equal.  Allele counts come from the device."""
        a, b = self.stats(region_a), self.stats(region_b)
        f0, f1 = a['freq'], b['freq']
        pbar = (f0 + f1) / 2
        Ht = 2 * pbar * (1 - pbar)
        Hs = (f0 * (1 - f0) + f1 * (1 - f1)) if est_Hs else (a['het'] + b['het']) / 2
        with np.errstate(divide='ignore', invalid='ignore'):
            out = (Ht - Hs) / Ht
        out[f0 == f1] = np.nan
        return out

    def counters(self):
        c = self.read('COUNTERS', 48)
        names = ['n', 'n_pre', 'P', 'B', 'deaths', 'n_free', 'n_slots', 'cur']
        out = {k: int(c[i]) for i, k in enumerate(names)}
        out['max_idx'] = int(c[8:10].view(np.int64)[0])
        out['t'] = int(c[10:12].view(np.int64)[0])
        out['err'] = int(c[12])
        out['n_rec'] = int(c[13])
        out['gs_iters'] = (int(c[14]), int(c[15]))
        out['n_nodes'], out['n_ind_rows'] = int(c[20]), int(c[21])      # next tskit node id / individuals row
        out['tsk_t0'] = int(c[24:26].view(np.int64)[0])
        # lengths of the fix list (exact-order cells) and the deferred list (d waits for max(N)) of the last
        # density evaluation
        out['density_lists'] = (int(c[46]), int(c[47]))
        return out

    def read(self, field, count):
        """Copy `count` elements of a device field to the host (parity tests, API views)."""
        dt = np.dtype(_DT[field])
        out = np.zeros(int(count), dtype=dt)
        _lib.check(self._L.gnx_read_field(self._ctx, _lib.FIELDS[field], out.ctypes.data_as(C.c_void_p),
                                          out.nbytes), 'gnx_read_field')
        return out

    def read_z(self, n):
        """z as [n, n_traits] (device layout is [n_traits][capacity])."""
        if not self.n_traits:
            return np.zeros((n, 0))
        full = self.read('Z', self.capacity * self.n_traits).reshape(self.n_traits, self.capacity)
        return np.ascontiguousarray(full[:, :n].T)

    def raster(self, field):
        return self.read(field, self.land_dim[0] * self.land_dim[1]).reshape(self.land_dim[1], self.land_dim[0])

    def profile(self, enable=True):
        _lib.check(self._L.gnx_profile(self._ctx, int(bool(enable))), 'gnx_profile')

    def profile_report(self):
        """{kernel: (launches, total_ms)} since profile(True)."""
        buf = C.create_string_buffer(1 << 16)
        _lib.check(self._L.gnx_profile_report(self._ctx, buf, len(buf)), 'gnx_profile_report')
        out = {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.split('\t')
            out[name] = (int(cnt), float(ms))
        return out

    @property
    def launch_count(self):
        return int(self._L.gnx_launch_count(self._ctx))

    @property
    def graph_launch_count(self):
        return int(self._L.gnx_graph_launch_count(self._ctx))

    @property
    def graph_capture_count(self):
        return int(self._L.gnx_graph_capture_count(self._ctx))

    @property
    def stream_ptr(self):
        return int(self._L.gnx_stream(self._ctx) or 0)

    def close(self):
        if getattr(self, '_ctx', None) is not None and self._ctx.value is not None:
            self._L.gnx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
