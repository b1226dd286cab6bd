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

One species over strips is one object: `_Strips` holds the plan and every species-wide operation
(setters, upload, download, step records, statistics, the burn-in statistic, genome assignment),
written once over the ranks that live in this process; two subclasses supply the transport:
  * `NcclStrips`   one process per GPU (`torch.distributed`, backend nccl, which only exchanges
                   the CUDA IPC handles): the barrier and the collectives are one-CTA kernels
                   over peer memory (gnx_strip_barrier) inside each step's CUDA graph; species-wide
                   results are gathered over the group.
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


# ---------------------------------------------------------------------------------------------
# one species over strips: the plan and every species-wide operation
# ---------------------------------------------------------------------------------------------
def band_capacities(K, start_y, bounds, cell_size, ncy):
    """Per-rank capacity: what DeviceSpecies gives a whole species (3 x the carrying capacity, twice the
    starting size, at least 4096), taken over the rank's own band of mating-grid rows."""
    b = np.asarray(bounds, dtype=np.int64)
    kb = np.add.reduceat(row_weights_from_K(np.asarray(K, dtype=np.float64), cell_size, ncy), b[:-1])
    nb = np.bincount(owner_of(start_y, b, cell_size, ncy), minlength=len(b) - 1) if len(start_y) else 0 * kb
    return np.maximum(4096, np.maximum(3.0 * kb, 2.0 * nb)).astype(np.int64)


class _Strips:
    """One species cut into `world` strips, of which `self.ranks` live in this process, with the members of
    DeviceSpecies that api.Species uses and species-wide results.  The subclasses supply the transport: how
    the ranks are connected, how a step is sequenced, and the primitives that combine the ranks' values:
      _gather(fn)        [fn(rank 0), ..., fn(rank world - 1)]
      _sum(tensors)      one tensor per rank of this process, each replaced by the sum over all ranks
                         (on the device when the call returns)
      _gather_rows(rows) one row per rank of this process in, every rank's row out ([world, len(row)])
      _check()           gnx_strip_check on every strip; a failure on any rank raises on every rank
    Where the ranks live in several processes, every process makes the same calls in the same order and sees
    the whole species.

    The plan: the mating grid, the first mating-grid row of every rank (`bounds`: given, or cut by the
    carrying capacity `K`, which defaults to the K layer of `rasters`), the landscape rows of each rank's
    band and the rows that adjacent bands share.  capacity None: each rank's band_capacities from `K` and the
    starting ordinates `start_y`; the ranks of one process share the largest."""

    def __init__(self, world, mine, land_dim, rasters, prm, gen_arch, capacity, seed, bounds=None, K=None,
                 start_y=(), **kw):
        self.world = int(world)
        self.land_dim = (int(land_dim[0]), int(land_dim[1]))
        self.cs, self.ncx, self.ncy = mating_grid(land_dim, prm['mating_radius'])
        K = np.asarray(rasters)[int(prm.get('K_layer', 0))] * float(prm.get('K_factor', 1.0)) if K is None \
            else np.asarray(K, dtype=np.float64)
        self.bounds = plan_rows(self.ncy, self.world, row_weights_from_K(K, self.cs, self.ncy)) if bounds is None \
            else np.asarray(bounds, dtype=np.int32)
        self.bands = band_rows(self.bounds, self.cs, self.land_dim[1])
        self._adds, self._skip_last = shared_band_rows(self.bands)
        if capacity is None:
            capacity = band_capacities(K, np.asarray(start_y), self.bounds, self.cs, self.ncy)[list(mine)].max()
        self.capacity = int(capacity)
        self.ranks = [StripRank(r, self.world, self.bounds, land_dim, rasters, prm, gen_arch, self.capacity, seed,
                                **kw) for r in mine]
        self.Lg = self.ranks[0].dev.Lg

    @property
    def _surf_tabs(self):
        return self.ranks[0].dev._surf_tabs

    # ---- setup: the same call on every strip
    def set_burn(self, burn):
        for r in self.ranks:
            r.dev.set_burn(burn)

    def set_raster(self, layer, rast):
        for r in self.ranks:
            r.dev.set_raster(layer, rast)

    def set_K(self, K):
        for r in self.ranks:
            r.dev.set_K(K)

    def set_life_history(self, **changes):
        for r in self.ranks:
            r.dev.set_life_history(**changes)

    def set_surface_tables(self, move_tab=None, disp_tab=None):
        for r in self.ranks:
            r.dev.set_surface_tables(move_tab, disp_tab)

    def set_mutation(self, *args, **kw):
        """Mutation of each step's offspring (DeviceSpecies.set_mutation, by-locus layout): every rank gets
        the same tables and replays the same species-wide draws."""
        for r in self.ranks:
            r.dev.set_mutation(*args, **kw)

    def set_clock(self, t, tsk_t0=0):
        """DeviceSpecies.set_clock on every strip: the ranks step in lockstep and share one clock."""
        for r in self.ranks:
            r.dev.set_clock(t, tsk_t0)

    def clock(self):
        return self.ranks[0].dev.clock()

    def read_mutations(self, max_rows=4096):
        """Drain the mutation logs; each rank's must equal the undecomposed run's, so the ranks of this
        process must agree.  Returns (rows, state) as DeviceSpecies.read_mutations does."""
        self._check()
        out = [r.dev.read_mutations(max_rows) for r in self.ranks]
        rows0, st0 = out[0]
        for r, (rows, st) in zip(self.ranks[1:], out[1:]):
            same = rows == rows0 and st['n_mutables'] == st0['n_mutables'] and \
                all(np.array_equal(st[k], st0[k]) for k in ('nonneut_loci', 'delet_loci', 'delet_s'))
            if not same:
                raise RuntimeError('strip rank %d: mutation log or tables differ from rank %d'
                                   % (r.rank, self.ranks[0].rank))
        return rows0, st0

    def read_mutation_tables(self):
        return self.ranks[0].dev.read_mutation_tables()

    def init_genomes(self, p, seed, write_mask=None, tskit_rows=False):
        """DeviceSpecies.init_genomes over the strips: the counts follow the species-wide size, the ranks'
        histograms are summed between the passes and every rank makes the same selection, so the genomes
        equal those of the undecomposed population."""
        if tskit_rows:
            raise ValueError('strip decomposition does not carry tskit rows')
        counts = gp.carrier_counts(self.population_size(), p)
        hists = [r.dev.genome_init_begin(counts, seed, write_mask) for r in self.ranks]
        while True:
            self._sum(hists)
            done = [r.dev.genome_init_pass() for r in self.ranks]
            assert len(set(done)) == 1, 'strip ranks disagree on the genome selection'
            if done[0]:
                break
        for r in self.ranks:
            r.dev.genome_init_end()

    # ---- population in / out
    def upload(self, x, y, age=None, sex=None, idx=None, g=None, max_ind_idx=None, genomes_packed=None, z=None,
               fit=None):
        """Upload each rank's share of a population every process holds on the host."""
        idx = np.arange(len(x), dtype=np.int64) if idx is None else np.asarray(idx)
        if max_ind_idx is None and len(idx):
            max_ind_idx = int(idx.max())
        cols = dict(x=x, y=y, age=age, sex=sex, idx=idx, g=g, genomes_packed=genomes_packed, z=z, fit=fit)
        own = owner_of(y, self.bounds, self.cs, self.ncy)
        for r in self.ranks:
            m = own == r.rank
            r.dev.upload(**{k: None if v is None else v[m] for k, v in cols.items()}, max_ind_idx=max_ind_idx)

    def step_records(self):
        """Species-wide records of the steps since the last call, after the strips are checked: a dropped
        migrant or a barrier timeout raises here (on every rank)."""
        self._check()
        return merge_records(self._gather(lambda r: r.dev.step_records()))

    def population_size(self):
        return sum(self._gather(lambda r: r.dev.population_size()))

    def download(self, genomes=True, unpack=True, e=False):
        self._check()
        out = merge_states(self._gather(lambda r: r.dev.download(genomes=genomes, unpack=False, e=e)))
        if 'genomes' in out and unpack:
            out['g'] = gp.unpack_genomes(out['genomes'], self.Lg)
        return out

    # ---- statistics: the integer counts add up over the strips, the fitness sum in rank order
    def stats(self, region=None):
        per = self._gather(lambda r: r.dev.stat_counts(region))
        c1 = sum(p[0] for p in per)
        het = sum(p[1] for p in per)
        fs = 0.0
        for p in per:
            fs += p[2]
        return stats_from_counts(c1, het, fs, sum(p[3] for p in per))

    def ld(self):
        per = self._gather(lambda r: r.dev.ld_counts())
        return ld_from_counts(sum(p[0] for p in per), sum(p[1] for p in per))

    def raster(self, field):
        """A landscape raster of the last step, each band's rows from the rank that computes them (a row two
        bands share from the upper one)."""
        per = self._gather(lambda r: r.dev.raster(field)[slice(*self.bands[r.rank])])
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
        got = [r.burnin_count() for r in self.ranks]
        for r, (ly0, ly1, _, _) in zip(self.ranks, got):
            assert (ly0, ly1) == self.bands[r.rank], 'strip band rows differ from the host plan'
        lasts = self._gather_rows([last for _, _, _, last in got])
        for r, (_, _, first, _) in zip(self.ranks, got):
            for q in self._adds[r.rank]:
                first += lasts[q]
        torch.cuda.synchronize()
        per = self._gather(lambda r: r.burnin_diff(self._skip_last[r.rank]))
        return cell_stats_from_sums(sum(p[0] for p in per), sum(p[1] for p in per), self.land_dim[0] * self.land_dim[1])

    def close(self):
        for r in self.ranks:
            r.dev.close()


# ---------------------------------------------------------------------------------------------
# all ranks in one process (tests / fewer GPUs than ranks)
# ---------------------------------------------------------------------------------------------
class LocalStrips(_Strips):
    """`world` strips as contexts of this process on the current GPU."""

    def __init__(self, world, land_dim, rasters, prm, gen_arch, capacity, seed=0, bounds=None, device_barrier=False,
                 **kw):
        super().__init__(world, range(int(world)), land_dim, rasters, prm, gen_arch, capacity, seed, bounds, **kw)
        # device_barrier: the ranks synchronise through gnx_strip_barrier (no host round trip inside a step);
        # otherwise the host is the barrier and does the three collectives on the ranks' tensors
        self.device_barrier = bool(device_barrier)
        self._warm = False
        for a in self.ranks:
            for b in self.ranks:
                if a is not b:
                    a.connect(b.rank, b.endpoints, same_process=True)
        self._t = [r.tensors() for r in self.ranks]

    def _gather(self, fn):
        return [fn(r) for r in self.ranks]

    def _sum(self, tensors):
        import torch
        torch.cuda.synchronize()
        tot = torch.stack(tensors).sum(dim=0, dtype=tensors[0].dtype)
        for t in tensors:
            t.copy_(tot)
        torch.cuda.synchronize()

    def _gather_rows(self, rows):
        import torch
        return torch.stack(rows)

    def _check(self):
        for r in self.ranks:
            r.check()

    def _sync(self):
        for r in self.ranks:
            r.dev.sync()

    def step(self, n=1):
        import torch
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


# ---------------------------------------------------------------------------------------------
# one process per GPU
# ---------------------------------------------------------------------------------------------
class NcclStrips(_Strips):
    """This process's strip of a landscape decomposed over the ranks of `torch.distributed`
    (backend nccl, one GPU each, one node: the receive buffers are shared through CUDA IPC)."""

    def __init__(self, land_dim, rasters, prm, gen_arch, capacity, seed=0, bounds=None, group=None, **kw):
        import torch
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group)
        super().__init__(dist.get_world_size(group), [self.rank], land_dim, rasters, prm, gen_arch, capacity, seed,
                         bounds, **kw)
        # the barriers and the three small collectives of a step run as one-CTA kernels over peer memory
        # (gnx_strip_barrier), never on the host
        self.device_barrier = True
        # exchange the endpoints (raw bytes of the struct: offsets + the CUDA IPC handle)
        everyone = [None] * self.world
        dist.all_gather_object(everyone, bytes(self.ranks[0].endpoints), group=group)
        for r, raw in enumerate(everyone):
            if r != self.rank:
                self.ranks[0].connect(r, _lib.StripEndpoints.from_buffer_copy(raw), same_process=False)
        self.stream = torch.cuda.ExternalStream(self.dev.stream_ptr)
        dist.barrier(group=group)

    @property
    def dev(self):
        return self.ranks[0].dev

    def _gather(self, fn):
        import torch.distributed as dist
        out = [None] * self.world
        dist.all_gather_object(out, fn(self.ranks[0]), group=self.group)
        return out

    def _sum(self, tensors):
        import torch
        import torch.distributed as dist
        for t in tensors:
            dist.all_reduce(t, group=self.group)
        torch.cuda.synchronize()

    def _gather_rows(self, rows):
        import torch
        import torch.distributed as dist
        out = torch.empty(self.world * len(rows[0]), dtype=rows[0].dtype, device='cuda')
        dist.all_gather_into_tensor(out, rows[0].clone(), group=self.group)
        return out.view(self.world, -1)

    def _check(self):
        """Each rank checks its strip, then the error flags are all-reduced, so every rank raises."""
        import torch
        import torch.distributed as dist
        err = None
        try:
            self.ranks[0].check()
        except _lib.GnxError as e:
            err = e
        flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=self.group)
        if err is not None:
            raise err
        if int(flag.item()):
            raise RuntimeError('a strip rank of this species failed (see that rank\'s error)')

    def step(self, n=1):
        self.dev.step(n)               # gnx_step: the phases + gnx_strip_barrier, one graph per step

    def sync(self):
        self.ranks[0].check()

    def step_records_local(self):
        """This rank's own records, without a check or a gather."""
        return self.dev.step_records()
