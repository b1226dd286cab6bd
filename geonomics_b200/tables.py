"""Host side of the tskit hand-off (species.py:440-445, 692-736, 956-1094, 1107-1219; mutation.py:44-58).

The reference adds one `tskit.TableCollection` row per Python call.  Here the step kernels write
the rows of every birth into device buffers (include/gnx_b200.h, "tskit record buffering"); this
module keeps them on the host as numpy COLUMNS -- the layout `TableCollection.*.append_columns` /
`set_columns` take -- and turns them into a real `tskit.TableCollection` when tskit is importable
(`to_tskit`).  tskit and msprime are absent from the build image: nothing here imports them at module
level; without tskit `sort_and_simplify` runs the restated algorithm on the species' device.
"""
import numpy as np


class _Columns:
    """Append-only numpy columns with amortised growth."""

    def __init__(self, **dtypes):
        self._dt = dtypes
        self._n = 0
        self._c = {k: np.zeros((0,) + tuple(sh), dtype=dt) for k, (dt, sh) in dtypes.items()}

    @property
    def num_rows(self):
        return self._n

    def __len__(self):
        return self._n

    def append_columns(self, **cols):
        n_new = None
        for k, v in cols.items():
            v = np.asarray(v)
            n_new = len(v) if n_new is None else n_new
            assert len(v) == n_new, 'ragged append'
        if not n_new:
            return self._n
        need = self._n + n_new
        for k, (dt, sh) in self._dt.items():
            a = self._c[k]
            if len(a) < need:
                b = np.zeros((max(need, 2 * len(a), 1024),) + tuple(sh), dtype=dt)
                b[:self._n] = a[:self._n]
                self._c[k] = a = b
            a[self._n:need] = cols[k] if k in cols else self._default(k)
        first = self._n
        self._n = need
        return first

    def _default(self, k):
        return -1 if np.issubdtype(self._dt[k][0], np.integer) else 0

    def column(self, k):
        return self._c[k][:self._n]

    def __getattr__(self, k):
        c = self.__dict__.get('_c')
        if c is not None and k in c:
            return c[k][:self._n]
        raise AttributeError(k)

    def truncate(self, n=0):
        self._n = n

    def asdict(self):
        return {k: self.column(k).copy() for k in self._c}


class TableColumns:
    """The five tables the path writes, as columns.

    nodes:       flags, time, population, individual
    edges:       left, right, parent, child
    individuals: flags, location [n, 2 + T + 1] = x, y, z..., fit (species.py:694-697), idx (the reference stores
                 it as 4 little-endian metadata bytes, species.py:703-704)
    sites:       position, nonneutral (metadata 't' / 'n', species.py:994-1002); ancestral_state is '0' for all
    mutations:   site, node, time; derived_state '1', parent -1 (mutation.py:47-57, genome.py:1146-1147)
    """

    def __init__(self, sequence_length, n_traits):
        self.sequence_length = int(sequence_length)
        self.n_loc = 2 + (n_traits + 1 if n_traits else 0)
        f8, i4, i8 = np.float64, np.int32, np.int64
        self.nodes = _Columns(flags=(i4, ()), time=(f8, ()), population=(i4, ()), individual=(i4, ()))
        self.edges = _Columns(left=(f8, ()), right=(f8, ()), parent=(i4, ()), child=(i4, ()))
        self.individuals = _Columns(flags=(i4, ()), location=(f8, (self.n_loc,)), idx=(i8, ()))
        self.sites = _Columns(position=(f8, ()), nonneutral=(np.int8, ()))
        self.mutations = _Columns(site=(i4, ()), node=(i4, ()), time=(f8, ()))

    def append_births(self, rows):
        """Rows drained from the device (DeviceSpecies.tskit_drain), one or several time steps of births
        (species.py:692-736: location = [x, y] + z + [fit], nodes flags = 1, time = -t, population = 0;
        rows['time'] is -t of each birth, t counted from the step recording was enabled in)."""
        nb = len(rows['idx'])
        if nb == 0:
            return
        if self.individuals.num_rows != rows['first_individual_row'] or self.nodes.num_rows != rows['first_node_id']:
            raise AssertionError('tables out of step with the device (rows %i / %i, device %i / %i)' % (
                self.individuals.num_rows, self.nodes.num_rows, rows['first_individual_row'], rows['first_node_id']))
        loc = np.full((nb, self.n_loc), np.nan)
        loc[:, 0], loc[:, 1] = rows['x'], rows['y']
        if self.n_loc > 2:
            loc[:, 2:-1] = rows['z']
        first = self.individuals.append_columns(flags=np.zeros(nb, np.int32), location=loc, idx=rows['idx'])
        time = np.repeat(np.asarray(rows['time'], dtype=np.float64), 2)
        self.nodes.append_columns(flags=np.ones(2 * nb, np.int32), time=time,
                                           population=np.zeros(2 * nb, np.int32),
                                           individual=np.repeat(first + np.arange(nb, dtype=np.int32), 2))
        self.edges.append_columns(left=rows['left'], right=rows['right'], parent=rows['parent'], child=rows['child'])

    def to_tskit(self):
        """A real tskit.TableCollection with these rows (needs tskit)."""
        try:
            import tskit
        except ImportError as e:           # pragma: no cover - tskit is absent from the build image
            raise RuntimeError('tskit is not installed: the tables stay numpy columns (TableColumns)') from e
        tc = tskit.TableCollection(sequence_length=self.sequence_length)
        n = self.individuals.num_rows
        meta = self.individuals.idx.astype('<u4').view(np.int8)
        tc.individuals.set_columns(flags=self.individuals.flags.astype(np.uint32),
                                   location=self.individuals.location.reshape(-1),
                                   location_offset=np.arange(n + 1, dtype=np.uint64) * self.n_loc,
                                   metadata=meta, metadata_offset=np.arange(n + 1, dtype=np.uint64) * 4)
        tc.nodes.set_columns(flags=self.nodes.flags.astype(np.uint32), time=self.nodes.time,
                             population=self.nodes.population, individual=self.nodes.individual)
        tc.edges.set_columns(left=self.edges.left, right=self.edges.right, parent=self.edges.parent,
                             child=self.edges.child)
        ns = self.sites.num_rows
        tc.sites.set_columns(position=self.sites.position, ancestral_state=np.full(ns, ord('0'), np.int8),
                             ancestral_state_offset=np.arange(ns + 1, dtype=np.uint64),
                             metadata=np.where(self.sites.nonneutral == 1, ord('t'), ord('n')).astype(np.int8),
                             metadata_offset=np.arange(ns + 1, dtype=np.uint64))
        nm = self.mutations.num_rows
        tc.mutations.set_columns(site=self.mutations.site, node=self.mutations.node, time=self.mutations.time,
                                 derived_state=np.full(nm, ord('1'), np.int8),
                                 derived_state_offset=np.arange(nm + 1, dtype=np.uint64))
        return tc

    def sort_and_simplify(self, sample_nodes, dev=None):
        """species.py:1107-1152: TableCollection.sort(); simplify(current nodes, filter_individuals=True,
        filter_sites=False).  With tskit installed its own C implementation runs on a real TableCollection
        (`to_tskit`) and the result is read back.  Without it, the published algorithm as `simplify_columns`
        restates it (parity with tskit unpinned, invariants checked by the tests): on the device of `dev`, a
        DeviceSpecies (gnx_simplify, row for row what `simplify_columns` gives), or here when there is none."""
        try:
            import tskit          # noqa: F401
            have = getattr(tskit, '__file__', None) is not None
        except ImportError:
            have = False
        if have:                            # pragma: no cover - tskit is absent from the build image
            tc = self.to_tskit()
            tc.sort()
            tc.simplify(np.asarray(sample_nodes, dtype=np.int32), filter_individuals=True, filter_sites=False)
            self._load(tc)
            return tc
        if dev is not None:
            return dev.simplify_tables(self, sample_nodes)
        simplify_columns(self, sample_nodes)
        return self

    def _load(self, tc):                    # pragma: no cover - needs tskit
        for tab in (self.nodes, self.edges, self.individuals, self.mutations):
            tab.truncate(0)
        self.nodes.append_columns(flags=tc.nodes.flags, time=tc.nodes.time, population=tc.nodes.population,
                                  individual=tc.nodes.individual)
        self.edges.append_columns(left=tc.edges.left, right=tc.edges.right, parent=tc.edges.parent,
                                  child=tc.edges.child)
        n = tc.individuals.num_rows
        loc = tc.individuals.location.reshape(n, self.n_loc) if n else np.zeros((0, self.n_loc))
        idx = tc.individuals.metadata.view('<u4').astype(np.int64) if n else np.zeros(0, np.int64)
        self.individuals.append_columns(flags=tc.individuals.flags, location=loc, idx=idx)
        self.mutations.append_columns(site=tc.mutations.site, node=tc.mutations.node, time=tc.mutations.time)


def simplify_columns(tc, sample_nodes):
    """`TableCollection.sort()` + `simplify(samples, filter_individuals=True, filter_sites=False)` on a
    TableColumns, in place.  tskit (>= 0.2.3 in the reference's requirements.txt) is absent here; this restates
    the published algorithm -- Kelleher, Thornton, Ashander & Ralph 2018, "Efficient pedigree recording for fast
    population genetics simulation", PLoS Comput Biol 14(11): e1006581, Algorithm S -- as tskit's documentation
    describes its effect:
      * the samples become output nodes 0 .. len(samples) - 1 in the order given (what species.py:1148-1152
        relies on), other nodes are kept only where ancestry of the samples coalesces in them;
      * parents are visited youngest first (edges sorted by parent time, then parent, child, left); the
        ancestry segments each child holds over an edge's interval are merged per parent through a priority
        queue; overlapping segments coalesce into the parent's output node and emit output edges, a segment
        on its own passes through unchanged (unary nodes vanish);
      * output edges of a parent are squashed (adjacent intervals to the same child merged);
      * a mutation moves to the output node that carries its node's ancestry at the site, or is dropped when
        nothing of the samples descends from it there; sites are all kept; individuals no retained node
        refers to are dropped, the others keep their relative order.
    Parity with tskit's C implementation is UNPINNED (nothing to run it against here); tests check the
    invariants: the samples' haplotypes replayed from the tables are unchanged, edges of every child tile
    without overlap, parents are older than children."""
    import heapq
    samples = np.asarray(sample_nodes, dtype=np.int64)
    L = float(tc.sequence_length)
    n_in = tc.nodes.num_rows
    time, nind, npop = tc.nodes.time.copy(), tc.nodes.individual.copy(), tc.nodes.population.copy()
    el, er, ep, ec = (tc.edges.left.copy(), tc.edges.right.copy(), tc.edges.parent.astype(np.int64),
                      tc.edges.child.astype(np.int64))
    order = np.lexsort((el, ec, ep, time[ep]))            # TableCollection.sort(): parent time, parent, child, left
    el, er, ep, ec = el[order], er[order], ep[order], ec[order]
    # ancestry of every input node: list of [left, right, output node]
    A = [None] * n_in
    o_time, o_ind, o_pop, o_flags = [], [], [], []
    for u in samples:
        A[u] = [[0.0, L, len(o_time)]]
        o_time.append(time[u]); o_ind.append(nind[u]); o_pop.append(npop[u]); o_flags.append(1)
    oe = [[], [], [], []]                                  # left, right, parent, child
    starts = np.flatnonzero(np.r_[True, ep[1:] != ep[:-1]]) if len(ep) else np.zeros(0, np.int64)
    ends = np.r_[starts[1:], len(ep)] if len(ep) else starts
    cnt = 0
    for s0, s1 in zip(starts, ends):
        u = int(ep[s0])
        Q = []
        for k in range(s0, s1):
            segs = A[ec[k]]
            if not segs:
                continue
            l_e, r_e = el[k], er[k]
            for x in segs:
                if x[1] > l_e and r_e > x[0]:
                    cnt += 1
                    heapq.heappush(Q, (max(x[0], l_e), cnt, min(x[1], r_e), x[2]))
        if not Q:
            continue
        v = -1
        own = A[u] if A[u] is not None else []            # a sample keeps its own node over [0, L)
        is_sample = bool(own)
        out = []
        pe = [[], [], []]                                   # this parent's output edges: left, right, child
        while Q:
            l = Q[0][0]
            r = L
            X = []
            while Q and Q[0][0] == l:
                x = heapq.heappop(Q)
                X.append(x)
                r = min(r, x[2])
            if Q:
                r = min(r, Q[0][0])
            if len(X) == 1 and not is_sample:
                x = X[0]
                if Q and Q[0][0] < x[2]:
                    out.append([x[0], Q[0][0], x[3]])
                    cnt += 1
                    heapq.heappush(Q, (Q[0][0], cnt, x[2], x[3]))
                else:
                    out.append([x[0], x[2], x[3]])
            else:
                if is_sample:
                    v = own[0][2]
                elif v == -1:
                    v = len(o_time)
                    o_time.append(time[u]); o_ind.append(nind[u]); o_pop.append(npop[u]); o_flags.append(0)
                out.append([l, r, v])
                for x in X:
                    pe[0].append(l); pe[1].append(r); pe[2].append(x[3])
                    if x[2] > r:
                        cnt += 1
                        heapq.heappush(Q, (r, cnt, x[2], x[3]))
        if not is_sample:
            A[u] = out
        if pe[0]:
            # squash: adjacent intervals to the same child become one edge
            o = np.lexsort((pe[0], pe[2]))
            l_, r_, c_ = np.asarray(pe[0])[o], np.asarray(pe[1])[o], np.asarray(pe[2])[o]
            keep = np.r_[True, (c_[1:] != c_[:-1]) | (l_[1:] != r_[:-1])]
            first = np.flatnonzero(keep)
            last = np.r_[first[1:], len(l_)] - 1
            oe[0].extend(l_[first]); oe[1].extend(r_[last]); oe[2].extend([v] * len(first)); oe[3].extend(c_[first])
    # mutations: to the output node carrying the ancestry of their node at the site
    ms, mn, mt = tc.mutations.site.copy(), tc.mutations.node.astype(np.int64), tc.mutations.time.copy()
    pos = tc.sites.position
    k_site, k_node, k_time = [], [], []
    for s_, n_, t_ in zip(ms, mn, mt):
        segs = A[n_] if 0 <= n_ < n_in else None
        if not segs:
            continue
        x = pos[s_] if len(pos) else float(s_)
        for a in segs:
            if a[0] <= x < a[1]:
                k_site.append(s_); k_node.append(a[2]); k_time.append(t_)
                break
    # individuals: drop the unreferenced, keep the order
    o_ind = np.asarray(o_ind, dtype=np.int64)
    used = np.zeros(tc.individuals.num_rows, bool)
    used[o_ind[o_ind >= 0]] = True
    remap = np.full(tc.individuals.num_rows, -1, np.int64)
    remap[used] = np.arange(int(used.sum()))
    i_flags, i_loc, i_idx = tc.individuals.flags[used].copy(), tc.individuals.location[used].copy(), \
        tc.individuals.idx[used].copy()
    for tab in (tc.nodes, tc.edges, tc.individuals, tc.mutations):
        tab.truncate(0)
    tc.individuals.append_columns(flags=i_flags, location=i_loc, idx=i_idx)
    tc.nodes.append_columns(flags=np.asarray(o_flags, np.int32), time=np.asarray(o_time, np.float64),
                            population=np.asarray(o_pop, np.int32),
                            individual=np.where(o_ind >= 0, remap[np.maximum(o_ind, 0)], -1).astype(np.int32))
    if oe[0]:
        l_, r_, p_, c_ = (np.asarray(v) for v in oe)
        o = np.lexsort((l_, c_, p_, np.asarray(o_time)[p_]))
        tc.edges.append_columns(left=l_[o], right=r_[o], parent=p_[o].astype(np.int32), child=c_[o].astype(np.int32))
    if k_site:
        tc.mutations.append_columns(site=np.asarray(k_site, np.int32), node=np.asarray(k_node, np.int32),
                                    time=np.asarray(k_time, np.float64))
    return tc
