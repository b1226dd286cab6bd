"""Strip domain decomposition of ONE landscape over several GPUs (SURVEY.md section 8e-2,
BASELINE configs[3]): host-side plan and orchestration above the C-ABI (gnx_strip_*).

Each rank owns a horizontal strip of the mating grid (whole rows, so that "owned" is one
contiguous range of the (mating cell, id) order and the rank-major order of pairs, births and
offspring ids is the order of the undecomposed run).  The data path is in the library:
individuals are written by the sender straight into the receiver's buffer (NVLink peer memory
mapped through CUDA IPC) and the device reads every size from device memory, so a time step
is enqueued without a host round trip.  This module supplies the plan (which rows, which
individuals go where at upload) and, where the host sequences the phases, the barrier between
them and the small collectives (births all-gather, density-count sum, max(N), and with Poisson
births the pairs all-gather).

Two transports:
  * `NcclStrips`   one process per GPU (`torch.distributed`, backend nccl, which only exchanges
                   the CUDA IPC handles): the barrier and the collectives are one-CTA kernels
                   over peer memory (gnx_strip_barrier) inside each step's CUDA graph.
  * `LocalStrips`  all ranks as contexts of ONE process on one GPU (tests; a box with fewer GPUs
                   than ranks): the same kernels write into the other contexts' buffers, the
                   host runs each phase on every context before the next and does the
                   collectives with plain device copies.
"""
import ctypes as C

import numpy as np

from . import _lib
from . import genome_pack as gp
from .device import DeviceSpecies, _DevArray, cell_stats_from_sums, ld_from_counts, stats_from_counts


# ---------------------------------------------------------------------------------------------
# the plan (pure host logic; CPU-tested)
# ---------------------------------------------------------------------------------------------
def mating_grid(land_dim, mating_radius):
    """Cell size and shape of the mating grid exactly as the library builds it (gnx_api.cu
    `mating_grid`): square cells of side >= radius * (1 + 1e-7), doubled until <= 2^22 cells."""
    cs = float(mating_radius) * 1.0000001
    while True:
        ncx, ncy = int(land_dim[0] / cs) + 1, int(land_dim[1] / cs) + 1
        if ncx * ncy <= (1 << 22):
            return cs, ncx, ncy
        cs *= 2.0


def plan_rows(ncy, world, weights=None):
    """First mating-grid row of every rank (length world + 1).  `weights` (per-row expected load,
    e.g. the row sums of the carrying-capacity raster) balance the strips; every strip gets at
    least two rows."""
    assert ncy >= 2 * world, 'the mating grid has too few rows for %d strips' % world
    if weights is None:
        weights = np.ones(ncy)
    w = np.maximum(np.asarray(weights, dtype=np.float64), 0) + 1e-12
    cum = np.concatenate([[0.0], np.cumsum(w)])
    bounds = [0]
    for r in range(1, world):
        target = cum[-1] * r / world
        row = int(np.searchsorted(cum, target))
        row = max(row, bounds[-1] + 2)
        row = min(row, ncy - 2 * (world - r))
        bounds.append(row)
    bounds.append(ncy)
    return np.array(bounds, dtype=np.int32)


def row_weights_from_K(K, cell_size, ncy):
    """Expected individuals per mating-grid row from a carrying-capacity raster [Y, X]."""
    rows = np.minimum((np.arange(K.shape[0]) / cell_size).astype(np.int64), ncy - 1)
    return np.bincount(rows, weights=K.sum(axis=1), minlength=ncy)


def owner_of(y, bounds, cell_size, ncy):
    """Rank that owns an individual at ordinate y (its mating-grid row, clamped like the kernel)."""
    row = np.minimum(np.floor(np.asarray(y) / cell_size).astype(np.int64), ncy - 1)
    return np.searchsorted(np.asarray(bounds)[1:-1], row, side='right')


def band_rows(bounds, cell_size, dim_y):
    """Landscape rows [ly0, ly1) that hold each rank's individuals, as gnx_strip_enable sets them: the rows
    of y in [row0, row1) * cell_size.  A band ends on the row its upper neighbour's band starts on."""
    b = np.asarray(bounds)
    world = len(b) - 1
    out = []
    for r in range(world):
        ly0 = max(0, int(np.floor(int(b[r]) * float(cell_size))))
        ly1 = int(dim_y) if r == world - 1 else min(int(dim_y), int(np.floor(int(b[r + 1]) * float(cell_size))) + 1)
        out.append((ly0, ly1))
    return out


def shared_band_rows(bands):
    """The burn-in bookkeeping of rows that adjacent bands share: per rank, the lower ranks whose last band row
    is this rank's first (their counts there are added into this rank's before the diff), and whether this
    rank's last row is an upper rank's first (the row, and its previous counts, belong to the upper rank)."""
    world = len(bands)
    adds = [[q for q in range(r) if bands[q][1] - 1 == bands[r][0]] for r in range(world)]
    skip_last = [any(bands[q][0] == bands[r][1] - 1 for q in range(r + 1, world)) for r in range(world)]
    return adds, skip_last


def phase_sequence(n_births_fixed):
    """The phases of one time step in order, each with the gnx_strip_barrier kind that follows it
    (0 barrier, 1 births all-gather, 2 density-count sum, 3 max(N), 4 pairs all-gather; None: the
    step ends), as the library's gnx_step runs them.  Poisson births are keyed by the species-wide
    position of each pair, so phase 3 publishes the pairs and phase 8 draws the births once the
    pairs of every rank are known."""
    phases, syncs, n = (C.c_int32 * 16)(), (C.c_int32 * 16)(), C.c_int32()
    _lib.check(_lib.lib().gnx_strip_phase_order(int(bool(n_births_fixed)), phases, syncs, C.byref(n)),
               'gnx_strip_phase_order')
    return [(phases[k], None if syncs[k] < 0 else syncs[k]) for k in range(n.value)]


def merge_records(per_rank):
    """Species-wide step records from the ranks' shares (Nt, births, deaths and pairs add up)."""
    out = []
    for recs in zip(*per_rank):
        out.append({'t': recs[0]['t'], 'Nt': sum(r['Nt'] for r in recs), 'n_births': sum(r['n_births'] for r in recs),
                    'n_deaths': sum(r['n_deaths'] for r in recs), 'n_pairs': sum(r['n_pairs'] for r in recs)})
    return out


def merge_states(states):
    """Species order (ascending id) from the ranks' downloads."""
    ids = np.concatenate([s['idx'] for s in states])
    order = np.argsort(ids, kind='stable')
    out = {}
    for k in states[0]:
        v0 = states[0][k]
        if isinstance(v0, np.ndarray) and v0.ndim >= 1 and len(v0) == len(states[0]['idx']):
            out[k] = np.concatenate([s[k] for s in states])[order]
    out['max_ind_idx'] = max(int(s['max_ind_idx']) for s in states)
    return out


# ---------------------------------------------------------------------------------------------
# one rank
# ---------------------------------------------------------------------------------------------
class StripRank:
    """One rank's DeviceSpecies with strip decomposition enabled."""

    def __init__(self, rank, world, bounds, land_dim, rasters, prm, gen_arch, capacity, seed,
                 migrant_capacity=None, halo_capacity=None, res_ratio=(1.0, 1.0)):
        self.rank, self.world = int(rank), int(world)
        self.bounds = np.ascontiguousarray(bounds, dtype=np.int32)
        self.dev = DeviceSpecies(land_dim, rasters, prm, gen_arch, capacity=capacity, seed=seed, res_ratio=res_ratio)
        L = self.dev._L
        sc = _lib.StripConfig()
        sc.rank, sc.world = self.rank, self.world
        sc.first_rows = self.bounds.ctypes.data_as(_lib.c_int32_p)
        sc.migrant_capacity = int(migrant_capacity or max(4096, capacity // 8))
        sc.halo_capacity = int(halo_capacity or max(4096, capacity // 4))
        _lib.check(L.gnx_strip_enable(self.dev._ctx, C.byref(sc)), 'gnx_strip_enable')
        self.endpoints = _lib.StripEndpoints()
        _lib.check(L.gnx_strip_endpoints(self.dev._ctx, C.byref(self.endpoints)), 'gnx_strip_endpoints')
        b, c, n, m = C.c_void_p(), C.c_void_p(), C.c_int64(), C.c_void_p()
        _lib.check(L.gnx_strip_collective_ptrs(self.dev._ctx, C.byref(b), C.byref(c), C.byref(n), C.byref(m)),
                   'gnx_strip_collective_ptrs')
        self.births_ptr, self.counts_ptr, self.n_counts, self.nmax_ptr = b.value, c.value, int(n.value), m.value
        p = C.c_void_p()
        _lib.check(L.gnx_strip_pairs_ptr(self.dev._ctx, C.byref(p)), 'gnx_strip_pairs_ptr')
        self.pairs_ptr = p.value

    def connect(self, peer_rank, endpoints, same_process):
        _lib.check(self.dev._L.gnx_strip_connect(self.dev._ctx, int(peer_rank), C.byref(endpoints),
                                                 int(bool(same_process))), 'gnx_strip_connect')

    def phase(self, k):
        _lib.check(self.dev._L.gnx_strip_phase(self.dev._ctx, int(k)), 'gnx_strip_phase')

    def barrier(self, kind=0):
        """gnx_strip_barrier: the barrier (0) or a collective (1 births, 2 counts, 3 max(N), 4 pairs) over peer
        memory."""
        _lib.check(self.dev._L.gnx_strip_barrier(self.dev._ctx, int(kind)), 'gnx_strip_barrier')

    def check(self):
        _lib.check(self.dev._L.gnx_strip_check(self.dev._ctx), 'gnx_strip_check')

    def burnin_count(self):
        """gnx_strip_burnin_count: (ly0, ly1, first band row, last band row), the rows as int32 torch views."""
        import torch
        a, b, f, l = C.c_int32(), C.c_int32(), C.c_void_p(), C.c_void_p()
        _lib.check(self.dev._L.gnx_strip_burnin_count(self.dev._ctx, C.byref(a), C.byref(b), C.byref(f), C.byref(l)),
                   'gnx_strip_burnin_count')
        X = self.dev.land_dim[0]
        return (a.value, b.value, torch.as_tensor(_DevArray(f.value, X, '<i4'), device='cuda'),
                torch.as_tensor(_DevArray(l.value, X, '<i4'), device='cuda'))

    def burnin_diff(self, skip_last_row):
        s1, s2 = C.c_int64(), C.c_int64()
        _lib.check(self.dev._L.gnx_strip_burnin_diff(self.dev._ctx, int(bool(skip_last_row)), C.byref(s1), C.byref(s2)),
                   'gnx_strip_burnin_diff')
        return int(s1.value), int(s2.value)

    def tensors(self):
        import torch
        births = torch.as_tensor(_DevArray(self.births_ptr, self.world, '<i8'), device='cuda')
        counts = torch.as_tensor(_DevArray(self.counts_ptr, self.n_counts, '<i4'), device='cuda')
        nmax = torch.as_tensor(_DevArray(self.nmax_ptr, 1, '<i8'), device='cuda')      # bits of a double >= 0
        pairs = torch.as_tensor(_DevArray(self.pairs_ptr, self.world, '<i8'), device='cuda')
        return births, counts, nmax, pairs


def _subset(pop, mask):
    return {k: (v[mask] if isinstance(v, np.ndarray) and v.ndim >= 1 and len(v) == len(mask) else v)
            for k, v in pop.items()}


# ---------------------------------------------------------------------------------------------
# all ranks in one process (tests / fewer GPUs than ranks)
# ---------------------------------------------------------------------------------------------
class LocalStrips:
    """`world` strips as contexts of this process on the current GPU."""

    def __init__(self, world, land_dim, rasters, prm, gen_arch, capacity, seed=0, bounds=None, device_barrier=False,
                 **kw):
        import torch
        self.torch = torch
        self.world = int(world)
        # device_barrier: the ranks synchronise through gnx_strip_barrier (no host round trip inside a step);
        # otherwise the host is the barrier and does the three collectives on the ranks' tensors
        self.device_barrier = bool(device_barrier)
        self._warm = False
        self.cs, self.ncx, self.ncy = mating_grid(land_dim, prm['mating_radius'])
        K = np.asarray(rasters)[int(prm.get('K_layer', 0))] * float(prm.get('K_factor', 1.0))
        self.bounds = plan_rows(self.ncy, world, row_weights_from_K(K, self.cs, self.ncy)) if bounds is None \
            else np.asarray(bounds, dtype=np.int32)
        self.ranks = [StripRank(r, world, self.bounds, land_dim, rasters, prm, gen_arch, capacity, seed, **kw)
                      for r in range(world)]
        for a in self.ranks:
            for b in self.ranks:
                if a is not b:
                    a.connect(b.rank, b.endpoints, same_process=True)
        self._t = [r.tensors() for r in self.ranks]

    def set_burn(self, burn):
        for r in self.ranks:
            r.dev.set_burn(burn)

    def set_mutation(self, *args, **kw):
        """Mutation of each step's offspring (DeviceSpecies.set_mutation, by-locus layout): every rank gets
        the same tables and replays the same species-wide draws."""
        for r in self.ranks:
            r.dev.set_mutation(*args, **kw)

    def read_mutations(self, max_rows=4096):
        """Drain every rank's mutation log; each must equal the undecomposed run's, so they must agree.
        Returns rank 0's (rows, state) as DeviceSpecies.read_mutations does."""
        for r in self.ranks:
            r.check()
        out = [r.dev.read_mutations(max_rows) for r in self.ranks]
        rows0, st0 = out[0]
        for rank, (rows, st) in enumerate(out[1:], 1):
            same = rows == rows0 and st['n_mutables'] == st0['n_mutables'] and \
                all(np.array_equal(st[k], st0[k]) for k in ('nonneut_loci', 'delet_loci', 'delet_s'))
            if not same:
                raise RuntimeError('strip rank %d: mutation log or tables differ from rank 0' % rank)
        return rows0, st0

    def init_genomes(self, p, seed, write_mask=None):
        """DeviceSpecies.init_genomes over the strips: the counts follow the species-wide size, the ranks'
        histograms are summed between the passes and every rank makes the same selection, so the genomes
        equal those of the undecomposed population."""
        torch = self.torch
        n = sum(self.population_sizes())
        counts = gp.carrier_counts(n, p)
        hists = [r.dev.genome_init_begin(counts, seed, write_mask) for r in self.ranks]
        while True:
            torch.cuda.synchronize()
            tot = torch.stack(hists).sum(dim=0, dtype=torch.int32)
            for h in hists:
                h.copy_(tot)
            torch.cuda.synchronize()
            done = [r.dev.genome_init_pass() for r in self.ranks]
            assert len(set(done)) == 1, 'strip ranks disagree on the genome selection'
            if done[0]:
                break
        for r in self.ranks:
            r.dev.genome_init_end()

    def upload(self, x, y, age=None, sex=None, idx=None, g=None, genomes_packed=None, max_ind_idx=None):
        n = len(x)
        idx = np.arange(n, dtype=np.int64) if idx is None else np.asarray(idx)
        max_ind_idx = int(idx.max()) if (max_ind_idx is None and n) else max_ind_idx
        own = owner_of(y, self.bounds, self.cs, self.ncy)
        for r in self.ranks:
            m = own == r.rank
            r.dev.upload(x[m], y[m], None if age is None else age[m], None if sex is None else sex[m], idx[m],
                         g=None if g is None else g[m],
                         genomes_packed=None if genomes_packed is None else genomes_packed[m],
                         max_ind_idx=max_ind_idx)

    def _sync(self):
        for r in self.ranks:
            r.dev.sync()

    def step(self, n=1):
        torch = self.torch
        if self.device_barrier and self._warm:
            # whole steps through gnx_step (one CUDA graph per rank and step, spin barriers inside); one step of
            # every rank is enqueued before the next, so no rank's queue fills up while a peer has nothing queued
            for _ in range(n):
                for r in self.ranks:
                    r.dev.step(1)
            return
        if self.device_barrier:
            # The first step of a process loads every kernel (CUDA loads modules lazily, and a load may wait for
            # the device to drain): with all ranks enqueued by ONE host thread, rank 0's spinning barrier would
            # wait for a rank the blocked host has not enqueued yet.  One step with the host as the barrier first.
            # (One process per GPU has no such coupling: a rank's barrier kernel is queued before its host can
            # block on the next phase's kernels.)
            self._warm = True
            self.device_barrier = False
            try:
                self.step(1)
            finally:
                self.device_barrier = True
            return self.step(n - 1) if n > 1 else None
        for _ in range(n):
            for k, sync in phase_sequence(self.ranks[0].dev._cfg.n_births_fixed):
                for r in self.ranks:
                    r.phase(k)
                self._sync()                               # the barrier: every context finished phase k
                if sync in (1, 4):                         # births (pairs) of every rank, everywhere
                    j = 0 if sync == 1 else 3
                    b = torch.stack([t[j][r] for r, t in enumerate(self._t)])
                    for t in self._t:
                        t[j][:self.world] = b
                elif sync == 2:                            # density counts summed over the strips
                    tot = sum(t[1] for t in self._t)
                    for t in self._t:
                        t[1].copy_(tot)
                elif sync == 3:                            # max(N): non-negative doubles order like their bits
                    mx = torch.stack([t[2] for t in self._t]).max()
                    for t in self._t:
                        t[2].fill_(mx)
                if sync:
                    torch.cuda.synchronize()

    def step_records(self):
        return merge_records([r.dev.step_records() for r in self.ranks])

    def download(self, **kw):
        for r in self.ranks:
            r.check()
        return merge_states([r.dev.download(**kw) for r in self.ranks])

    def population_sizes(self):
        return [r.dev.population_size() for r in self.ranks]

    def close(self):
        for r in self.ranks:
            r.dev.close()


# ---------------------------------------------------------------------------------------------
# one process per GPU
# ---------------------------------------------------------------------------------------------
class NcclStrips:
    """This process's strip of a landscape decomposed over the ranks of `torch.distributed`
    (backend nccl, one GPU each, one node: the receive buffers are shared through CUDA IPC)."""

    def __init__(self, land_dim, rasters, prm, gen_arch, capacity, seed=0, bounds=None, group=None, **kw):
        import torch
        import torch.distributed as dist
        # the barriers and the three small collectives of a step run as one-CTA kernels over peer memory
        # (gnx_strip_barrier), never on the host
        self.device_barrier = True
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.group = group
        self.cs, self.ncx, self.ncy = mating_grid(land_dim, prm['mating_radius'])
        K = np.asarray(rasters)[int(prm.get('K_layer', 0))] * float(prm.get('K_factor', 1.0))
        self.bounds = plan_rows(self.ncy, self.world, row_weights_from_K(K, self.cs, self.ncy)) if bounds is None \
            else np.asarray(bounds, dtype=np.int32)
        self.me = StripRank(self.rank, self.world, self.bounds, land_dim, rasters, prm, gen_arch, capacity, seed, **kw)
        # exchange the endpoints (raw bytes of the struct: offsets + the CUDA IPC handle)
        mine = bytes(self.me.endpoints)
        everyone = [None] * self.world
        dist.all_gather_object(everyone, mine, group=group)
        for r, raw in enumerate(everyone):
            if r != self.rank:
                self.me.connect(r, _lib.StripEndpoints.from_buffer_copy(raw), same_process=False)
        self.stream = torch.cuda.ExternalStream(self.me.dev.stream_ptr)
        dist.barrier(group=group)

    @property
    def dev(self):
        return self.me.dev

    def set_burn(self, burn):
        self.me.dev.set_burn(burn)

    def set_mutation(self, *args, **kw):
        """DeviceSpecies.set_mutation on this rank; every rank must make the same call."""
        self.me.dev.set_mutation(*args, **kw)

    def read_mutations(self, max_rows=4096):
        """This rank's mutation log and tables, which equal every other rank's."""
        return self.me.dev.read_mutations(max_rows)

    def init_genomes(self, p, seed, write_mask=None):
        """DeviceSpecies.init_genomes on this rank with the size and the histograms summed over the ranks
        (every rank makes the same call)."""
        import torch.distributed as dist
        self.me.dev.init_genomes(p, seed, write_mask, allreduce=lambda t: dist.all_reduce(t, group=self.group))

    def upload_owned(self, x, y, age=None, sex=None, idx=None, g=None, genomes_packed=None, max_ind_idx=None):
        """Upload this rank's share of a population every rank holds on the host."""
        idx = np.arange(len(x), dtype=np.int64) if idx is None else np.asarray(idx)
        m = owner_of(y, self.bounds, self.cs, self.ncy) == self.rank
        self.me.dev.upload(x[m], y[m], None if age is None else age[m], None if sex is None else sex[m], idx[m],
                           g=None if g is None else g[m],
                           genomes_packed=None if genomes_packed is None else genomes_packed[m],
                           max_ind_idx=int(idx.max()) if max_ind_idx is None else max_ind_idx)

    def step(self, n=1):
        self.me.dev.step(n)            # gnx_step: the phases + gnx_strip_barrier, one graph per step

    def sync(self):
        self.me.check()

    def step_records_local(self):
        return self.me.dev.step_records()

    def close(self):
        self.me.dev.close()


# ---------------------------------------------------------------------------------------------
# one species over strips, behind the DeviceSpecies surface of api.Species
# ---------------------------------------------------------------------------------------------
def band_capacities(K, start_y, bounds, cell_size, ncy):
    """Per-rank capacity: what DeviceSpecies gives a whole species (3 x the carrying capacity, twice the
    starting size, at least 4096), taken over the rank's own band of mating-grid rows."""
    b = np.asarray(bounds, dtype=np.int64)
    kb = np.add.reduceat(row_weights_from_K(np.asarray(K, dtype=np.float64), cell_size, ncy), b[:-1])
    nb = np.bincount(owner_of(start_y, b, cell_size, ncy), minlength=len(b) - 1) if len(start_y) else 0 * kb
    return np.maximum(4096, np.maximum(3.0 * kb, 2.0 * nb)).astype(np.int64)


class StripSpecies:
    """One species cut into strips, with the members of DeviceSpecies that api.Species uses and species-wide
    results.  `strips` is a strip count (LocalStrips: every strip a context of this process on the current
    GPU, the host the barrier between the phases) or an initialised torch.distributed process group
    (NcclStrips: this process's strip, device barriers, one graph per step).  Under a group every rank
    makes the same calls in the same order and sees the whole species."""

    def __init__(self, land_dim, rasters, prm, gen_arch, K, start_y, strips, seed=0, res_ratio=(1.0, 1.0),
                 capacity=None):
        self.land_dim = (int(land_dim[0]), int(land_dim[1]))
        self.group = None if isinstance(strips, (int, np.integer)) else strips
        if self.group is None:
            self.world, self.rank = int(strips), None
        else:
            import torch.distributed as dist
            self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        cs, ncx, ncy = mating_grid(self.land_dim, prm['mating_radius'])
        bounds = plan_rows(ncy, self.world, row_weights_from_K(np.asarray(K, dtype=np.float64), cs, ncy))
        self.bands = band_rows(bounds, cs, self.land_dim[1])
        self._adds, self._skip_last = shared_band_rows(self.bands)
        if capacity is None:
            caps = band_capacities(K, np.asarray(start_y), bounds, cs, ncy)
            capacity = int(caps.max() if self.group is None else caps[self.rank])
        self.capacity = int(capacity)
        kw = dict(seed=seed, bounds=bounds, res_ratio=res_ratio)
        if self.group is None:
            self._st = LocalStrips(self.world, self.land_dim, rasters, prm, gen_arch, self.capacity, **kw)
            self._ranks = self._st.ranks
        else:
            self._st = NcclStrips(self.land_dim, rasters, prm, gen_arch, self.capacity, group=self.group, **kw)
            self._ranks = [self._st.me]
        self.Lg = self._ranks[0].dev.Lg

    def _per_rank(self, fn):
        """[fn(rank 0), ..., fn(rank world - 1)] on every rank (all-gathered under a group)."""
        mine = [fn(r) for r in self._ranks]
        if self.group is None:
            return mine
        import torch.distributed as dist
        out = [None] * self.world
        dist.all_gather_object(out, mine[0], group=self.group)
        return out

    def _each(self, name, *args, **kw):
        for r in self._ranks:
            getattr(r.dev, name)(*args, **kw)

    @property
    def _surf_tabs(self):
        return self._ranks[0].dev._surf_tabs

    # ---- setup: the same call on every strip
    def set_burn(self, burn):
        self._each('set_burn', burn)

    def set_raster(self, layer, rast):
        self._each('set_raster', layer, rast)

    def set_K(self, K):
        self._each('set_K', K)

    def set_life_history(self, **changes):
        self._each('set_life_history', **changes)

    def set_surface_tables(self, move_tab=None, disp_tab=None):
        self._each('set_surface_tables', move_tab, disp_tab)

    def set_mutation(self, *args, **kw):
        self._st.set_mutation(*args, **kw)

    def read_mutations(self, max_rows=4096):
        return self._st.read_mutations(max_rows)

    def read_mutation_tables(self):
        return self._ranks[0].dev.read_mutation_tables()

    def init_genomes(self, p, seed, write_mask=None, tskit_rows=False):
        if tskit_rows:
            raise ValueError('strip decomposition does not carry tskit rows')
        self._st.init_genomes(p, seed, write_mask)

    # ---- population in / out
    def upload(self, x, y, age=None, sex=None, idx=None, g=None, max_ind_idx=None, genomes_packed=None):
        up = self._st.upload if self.group is None else self._st.upload_owned
        up(x, y, age, sex, idx, g=g, genomes_packed=genomes_packed, max_ind_idx=max_ind_idx)

    def _check(self):
        """gnx_strip_check on every strip: a dropped migrant or a barrier timeout raises (on every rank)."""
        if self.group is None:
            for r in self._ranks:
                r.check()
            return
        import torch
        import torch.distributed as dist
        err = None
        try:
            self._st.me.check()
        except _lib.GnxError as e:
            err = e
        flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=self.group)
        if err is not None:
            raise err
        if int(flag.item()):
            raise RuntimeError('a strip rank of this species failed (see that rank\'s error)')

    def step(self, n_steps=1):
        self._st.step(n_steps)
        self._check()

    def step_records(self):
        return merge_records(self._per_rank(lambda r: r.dev.step_records()))

    def population_size(self):
        return sum(self._per_rank(lambda r: r.dev.population_size()))

    def download(self, genomes=True, unpack=True, e=False):
        self._check()
        out = merge_states(self._per_rank(lambda r: r.dev.download(genomes=genomes, unpack=False, e=e)))
        if 'genomes' in out and unpack:
            out['g'] = gp.unpack_genomes(out['genomes'], self.Lg)
        return out

    # ---- statistics: the integer counts add up over the strips, the fitness sum in rank order
    def stats(self, region=None):
        per = self._per_rank(lambda r: r.dev.stat_counts(region))
        c1 = sum(p[0] for p in per)
        het = sum(p[1] for p in per)
        fs = 0.0
        for p in per:
            fs += p[2]
        return stats_from_counts(c1, het, fs, sum(p[3] for p in per))

    def ld(self):
        per = self._per_rank(lambda r: r.dev.ld_counts())
        return ld_from_counts(sum(p[0] for p in per), sum(p[1] for p in per))

    def raster(self, field):
        """A landscape raster of the last step, each band's rows from the rank that computes them (a row two
        bands share from the upper one)."""
        per = self._per_rank(lambda r: r.dev.raster(field)[slice(*self.bands[r.rank])])
        out = None
        for (ly0, ly1), rows in zip(self.bands, per):
            if out is None:
                out = np.zeros((self.land_dim[1],) + rows.shape[1:], dtype=rows.dtype)
            out[ly0:ly1] = rows
        return out

    def burnin_cell_stats(self):
        """DeviceSpecies.burnin_cell_stats of the whole species: every rank counts into its band, the rows two
        bands share are added into the upper band, and each rank sums the change over the rows it accounts for."""
        import torch
        got = {r.rank: r.burnin_count() for r in self._ranks}
        for k, (ly0, ly1, _, _) in got.items():
            assert (ly0, ly1) == self.bands[k], 'strip band rows differ from the host plan'
        if self.group is None:
            lasts = [got[k][3].clone() for k in range(self.world)]
        else:
            import torch.distributed as dist
            X = self.land_dim[0]
            allrows = torch.empty(self.world * X, dtype=torch.int32, device='cuda')
            dist.all_gather_into_tensor(allrows, got[self.rank][3].clone(), group=self.group)
            lasts = list(allrows.view(self.world, X))
        for k, (_, _, first, _) in got.items():
            for q in self._adds[k]:
                first += lasts[q]
        torch.cuda.synchronize()
        per = self._per_rank(lambda r: r.burnin_diff(self._skip_last[r.rank]))
        return cell_stats_from_sums(sum(p[0] for p in per), sum(p[1] for p in per), self.land_dim[0] * self.land_dim[1])

    def close(self):
        self._st.close()
