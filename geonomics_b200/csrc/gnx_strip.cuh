// gnx_strip.cuh -- strip domain decomposition of ONE landscape over several GPUs
// (SURVEY.md section 8e-2; BASELINE configs[3]).  Rank r owns the individuals whose mating-grid
// row lies in [row0, row1); mating-grid rows are contiguous in the (cell, id) order of the
// state, so "owned" is one contiguous entry range and the rank-major order of pairs, births
// and offspring ids equals the order of the undecomposed run: with ids based at
// max_ind_idx + 1 + (births of the lower ranks) every Philox stream, every id and therefore
// every survivor is bit-identical to the single-GPU run, whatever the number of strips.
//
// Exchanges per time step (all device-side: a record is written by the SENDER straight into
// the receiver's buffer over NVLink peer memory, its slot claimed with a system-scope atomic;
// a stream-ordered collective enqueued by the host between the phases is the only barrier):
//   migrants  -- individuals that moved out of the strip (movement.py:34-95), whole record +
//                genome row, to whichever rank owns their new row; they join that rank's re-grid
//   halo      -- copies of the individuals in the strip's first / last row, to the lower / upper
//                neighbour: candidates (and possible parents, hence the genome row) of that
//                rank's mate search (species.py:2157-2215), never focals there
//   choices   -- for a focal on the edge that chose a ghost: (focal, mate) so that the neighbour
//                can apply the reciprocal-pair rule of mating.py:62-63 to its own focal
//   newborns  -- offspring that dispersed out of the strip (movement.py:98-141), before the
//                density counts and the mortality of the same step
// plus three collectives on small arrays: births per rank (id bases, species.py:614-619), the
// 2 x 4 coarse density-count grids (sum, spatial.py:73-97) and max(N) (demography.py:104-119); with
// Poisson births a fourth, pairs per rank, comes first: the birth draws are keyed by the pair's
// species-wide position (mating.py:120-126).  Mutation needs no exchange: every rank replays the
// step's draws and keeps the tables, and the owner of a mutated offspring edits its genome row.
#pragma once
#include "gnx_common.cuh"

// record layout: x f64 | y f64 | id i64 | fit f64 | z[T] f64 | age i32 | sex i32 | pad to 16 | genome row
__host__ __device__ __forceinline__ int strip_header_bytes(int T) { return ((40 + 8 * T) + 15) & ~15; }

__device__ __forceinline__ int strip_owner(const Strip* st, int row) {
  int d = 0;
  for (int r = 1; r < st->world; ++r) d += (row >= st->bounds[r]) ? 1 : 0;
  return d;
}

// list an entry for shipping
__device__ __forceinline__ void strip_list(const Strip* st, int entry, int dest) {
  const int L = atomicAdd(st->list_n, 1);
  if (L < st->list_cap) {
    st->list_entry[L] = entry;
    st->list_dest[L] = dest;
  } else {
    atomicOr(st->err, 1);
  }
}

// One warp per listed individual: claim a slot in the destination's receive buffer and write
// the record there (peer memory over NVLink when the destination is another GPU).
__global__ void __launch_bounds__(256) k_strip_send(Pop pop, const Counters* c, const Strip* st, int which, int with_genome) {
  const int cur = c->cur, T = pop.T, Wq = pop.Wq;
  const int n_list = min(*st->list_n, st->list_cap);
  const int lane = threadIdx.x & 31;
  const int hb = strip_header_bytes(T);
  for (int L = GTID >> 5; L < n_list; L += GSTRIDE >> 5) {
    const int e = st->list_entry[L], d = st->list_dest[L];
    int pos = 0;
    if (lane == 0) pos = atomicAdd_system(st->peer[d].count[which], 1);
    pos = __shfl_sync(0xffffffffu, pos, 0);
    if (pos >= st->cap[which]) {
      if (lane == 0) atomicOr(st->err, 2);
      continue;
    }
    unsigned char* rec = st->peer[d].buf[which] + (size_t)pos * st->rec_bytes;
    if (lane == 0) {
      const double2 xy = pop.xy[cur][e];
      double* h = reinterpret_cast<double*>(rec);
      h[0] = xy.x;
      h[1] = xy.y;
      reinterpret_cast<int64_t*>(rec)[2] = pop.idx[cur][e];
      h[3] = pop.fit[cur][e];
      for (int tt = 0; tt < T; ++tt) h[4 + tt] = pop.z[cur][(size_t)tt * pop.cap + e];
      int32_t* tail = reinterpret_cast<int32_t*>(rec + 32 + 8 * T);
      tail[0] = pop.age[cur][e];
      tail[1] = (int32_t)pop.sex[cur][e];
    }
    if (with_genome) {
      const uint4* src = pop.G + (size_t)pop.gslot[cur][e] * 2 * Wq;
      uint4* dst = reinterpret_cast<uint4*>(rec + hb);
      for (int q = lane; q < 2 * Wq; q += 32) dst[q] = src[q];
    }
    __threadfence_system();
  }
}

// Arrivals (after the barrier): append the records of receive buffer `which` to the population.
//   mode 0: before the re-grid (migrants, halo ghosts): entries [n, n + n_in) of the current half,
//           keyed into the mating grid (key + histogram rank) so that the re-grid places them
//   mode 1: after the births (newborns that dispersed in): tail entries [n + B, n + B + n_in)
// Genome slots: the i-th arrival takes the i-th free slot from the top of the free list, then
// fresh slots -- the same rule as k_gametes; k_strip_recv_finish books them.
__global__ void __launch_bounds__(256) k_strip_recv(Pop pop, Land land, Work w, Counters* c, const Strip* st, int which,
                                                     int mode, int with_genome) {
  const int cur = c->cur, T = pop.T, Wq = pop.Wq;
  const int n_in = min(*st->peer[st->rank].count[which], st->cap[which]);
  const int base = mode == 0 ? c->n : c->n + c->B;
  const int n_free = c->n_free, n_slots = c->n_slots;
  const int lane = threadIdx.x & 31;
  const int hb = strip_header_bytes(T);
  const unsigned char* buf = st->peer[st->rank].buf[which];
  for (int i = GTID >> 5; i < n_in; i += GSTRIDE >> 5) {
    const int dst = base + i;
    if (dst >= pop.cap) {
      if (lane == 0) atomicOr(&c->err, GNX_ERRBIT_CAPACITY);
      continue;
    }
    const unsigned char* rec = buf + (size_t)i * st->rec_bytes;
    int slot = -1;
    if (with_genome) {
      slot = i < n_free ? pop.free_slots[n_free - 1 - i] : n_slots + (i - n_free);
      if (slot >= pop.cap) {
        if (lane == 0) atomicOr(&c->err, GNX_ERRBIT_CAPACITY);
        continue;
      }
      const uint4* src = reinterpret_cast<const uint4*>(rec + hb);
      uint4* row = pop.G + (size_t)slot * 2 * Wq;
      for (int q = lane; q < 2 * Wq; q += 32) row[q] = src[q];
    }
    if (lane == 0) {
      const double* h = reinterpret_cast<const double*>(rec);
      const double x = h[0], y = h[1];
      pop.xy[cur][dst] = make_double2(x, y);
      pop.idx[cur][dst] = reinterpret_cast<const int64_t*>(rec)[2];
      pop.fit[cur][dst] = h[3];
      for (int tt = 0; tt < T; ++tt) pop.z[cur][(size_t)tt * pop.cap + dst] = h[4 + tt];
      const int32_t* tail = reinterpret_cast<const int32_t*>(rec + 32 + 8 * T);
      pop.age[cur][dst] = tail[0];
      pop.sex[cur][dst] = (int8_t)tail[1];
      pop.gslot[cur][dst] = slot;
      w.alive[dst] = 1;
      if (mode == 0) {
        const uint32_t key = mating_cell(land, x, y);
        w.mkey[dst] = key;
        atomicAdd(&w.cell_count[cell_linear(land, key)], 1u);
      } else {
        st->sent[dst] = 0;
      }
    }
  }
}

__global__ void k_strip_recv_finish(Counters* c, const Strip* st, int which, int mode, int with_genome) {
  int32_t* cnt = st->peer[st->rank].count[which];
  const int n_in = min(*cnt, st->cap[which]);
  if (*cnt > st->cap[which]) atomicOr(st->err, 2);
  if (with_genome) {
    const int nf = c->n_free;
    if (n_in <= nf) c->n_free = nf - n_in;
    else { c->n_free = 0; c->n_slots += n_in - nf; }
  }
  if (mode == 0) c->n += n_in;
  else { c->B += n_in; c->n_pre = c->n + c->B; }
  *cnt = 0;                                  // ready for the next time step (several barriers away)
}

// the strip's first and last mating-grid rows go to the lower / upper neighbour as ghosts
__global__ void __launch_bounds__(256) k_strip_halo_list(Work w, const Counters* c, const Strip* st) {
  const int n = c->n;
  for (int p = GTID; p < n; p += GSTRIDE) {
    const uint32_t key = w.mkey[p];
    if (key == GNX_KEY_DEAD) continue;
    const int row = (int)(key >> 16);
    if (row == st->row0 && st->rank > 0) strip_list(st, p, st->rank - 1);
    if (row == st->row1 - 1 && st->rank < st->world - 1) strip_list(st, p, st->rank + 1);
  }
}

// newborns whose natal dispersal (movement.py:98-141) carried them out of the strip
__global__ void __launch_bounds__(256) k_strip_newborn_route(Pop pop, Land land, Counters* c, const Strip* st) {
  const int n = c->n, B = c->B, cur = c->cur;
  int sent = 0;
  for (int o = GTID; o < B; o += GSTRIDE) {
    const double2 xy = pop.xy[cur][n + o];
    const int row = (int)(mating_cell(land, xy.x, xy.y) >> 16);
    const bool out = row < st->row0 || row >= st->row1;
    st->sent[n + o] = out ? 1 : 0;
    if (out) { strip_list(st, n + o, strip_owner(st, row)); sent += 1; }
  }
  if (sent) atomicAdd(&c->tail_sent, sent);
}

// A focal on the strip's edge that chose a ghost: tell the ghost's owner, so that it can apply
// the reciprocal-pair rule (mating.py:62-63: a couple that chose each other is kept once, under
// the focal with the smaller id) to its own focal.  Record: {focal key, mate key, focal id, mate id}.
struct StripChoice { uint32_t key_j, key_m; int64_t id_j, id_m; };
__global__ void __launch_bounds__(256) k_strip_choice_send(Pop pop, Work w, const Counters* c, const Strip* st) {
  const int lo = c->own_lo, hi = c->own_hi, cur = c->cur;
  for (int p = lo + GTID; p < hi; p += GSTRIDE) {
    const int m = w.mate[p];
    if (m < 0 || (m >= lo && m < hi)) continue;
    const int d = m < lo ? st->rank - 1 : st->rank + 1;
    const int pos = atomicAdd_system(st->peer[d].count[STRIP_BUF_CHOICES], 1);
    if (pos >= st->cap[STRIP_BUF_CHOICES]) { atomicOr(st->err, 2); continue; }
    StripChoice r;
    r.key_j = w.skey[p];
    r.key_m = w.skey[m];
    r.id_j = pop.idx[cur][p];
    r.id_m = pop.idx[cur][m];
    reinterpret_cast<StripChoice*>(st->peer[d].buf[STRIP_BUF_CHOICES])[pos] = r;
    __threadfence_system();
  }
}

// entry of individual `id` in mating cell `key` (ids ascend inside a cell), or -1
__device__ __forceinline__ int strip_find(const Pop& pop, const Land& land, const Work& w, int cur, uint32_t key, int64_t id) {
  const uint32_t lin = cell_linear(land, key);
  int lo = (int)w.cell_start[lin], hi = (int)w.cell_start[lin + 1];
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int64_t v = pop.idx[cur][mid];
    if (v == id) return mid;
    if (v < id) lo = mid + 1; else hi = mid;
  }
  return -1;
}

__global__ void __launch_bounds__(256) k_strip_choice_recv(Pop pop, Land land, Work w, const Counters* c, const Strip* st) {
  const int cur = c->cur;
  const int n_in = min(*st->peer[st->rank].count[STRIP_BUF_CHOICES], st->cap[STRIP_BUF_CHOICES]);
  const StripChoice* in = reinterpret_cast<const StripChoice*>(st->peer[st->rank].buf[STRIP_BUF_CHOICES]);
  for (int i = GTID; i < n_in; i += GSTRIDE) {
    const StripChoice r = in[i];
    const int g = strip_find(pop, land, w, cur, r.key_j, r.id_j);      // the ghost of the neighbour's focal
    const int e = strip_find(pop, land, w, cur, r.key_m, r.id_m);      // my own individual it chose
    if (g >= 0 && e >= 0) w.mate[g] = e;
  }
}
__global__ void k_strip_choice_finish(const Strip* st) {
  int32_t* cnt = st->peer[st->rank].count[STRIP_BUF_CHOICES];
  if (*cnt > st->cap[STRIP_BUF_CHOICES]) atomicOr(st->err, 2);
  *cnt = 0;
}

__global__ void k_strip_list_reset(const Strip* st) { *st->list_n = 0; }

// ids of this step's offspring (species.py:614-619): based at max_ind_idx + 1 + the births of the
// lower ranks -- the ids the undecomposed run assigns, since its pair list is in the same
// rank-major (mating cell, id) order.  Counters.max_idx carries the base until the step ends.
__global__ void k_strip_id_base(Counters* c, const Strip* st) {
  long long off = 0, tot = 0;
  for (int r = 0; r < st->world; ++r) {
    if (r < st->rank) off += st->births[r];
    tot += st->births[r];
  }
  c->max_idx_base = c->max_idx;
  c->births_lo = (int32_t)off;
  c->births_all = (int32_t)tot;
  c->max_idx_global = c->max_idx + tot;      // species-wide max_ind_idx once this step's births exist
  c->max_idx += off;
}
// after k_death closed the step (it added this rank's tail to max_idx): back to the species-wide value
__global__ void k_strip_end_step(Counters* c) {
  c->max_idx = c->max_idx_global;
  c->tail_sent = 0;
}
// this rank's births, where the all-gather picks them up
__global__ void k_strip_publish_births(const Counters* c, const Strip* st) { st->births[st->rank] = (long long)c->B; }
// this rank's pairs (Poisson births: the lower ranks' pairs key this rank's draws, k_draw_births)
__global__ void k_strip_publish_pairs(const Counters* c, const Strip* st) { st->pairs[st->rank] = (long long)c->P; }

// ========================================================================================
// Barrier and the three small collectives of a strip time step, over peer memory.
// Every rank owns a synchronisation page inside its receive block (mapped by all peers through
// CUDA IPC / NVLink like the record buffers); rank w writes only slot w of every page, so nothing
// is ever contended: the payload first (kind 1: this rank's births -> all-gather; kind 2: its
// coarse density counts -> sum over the ranks in rank order, so the integers are the same on every
// rank; kind 3: the bits of its max(N) -> maximum; kind 4: its pairs -> all-gather, in a slot of its own
// because the births all-gather of the same step follows it only one phase later), a system-scope
// fence, then the rank's barrier
// epoch with release semantics into every peer's flag word; the lanes then spin (acquire loads) on
// the flags of this rank's own page until every peer has reached the same epoch.  Kernels of a rank
// are stream-ordered, so a peer that reads a slot has finished with it before the writer can get to
// the next barrier of the same kind (there is at least one other barrier in between).  One launch of
// one CTA replaces an NCCL collective (and its launch gap) after seven of the eight phases.  A peer
// that never arrives (a failed rank) ends the wait after ~5 s with the error bit set instead of
// hanging the device.
// ========================================================================================
__device__ __forceinline__ void st_release_sys_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__global__ void __launch_bounds__(256) k_strip_barrier(const Strip* stp, int kind, int32_t* counts, int n_counts,
                                                       unsigned long long* nmax) {
  const Strip& st = *stp;
  __shared__ uint32_t s_epoch;
  if (threadIdx.x == 0) s_epoch = ++(*st.epoch);
  __syncthreads();
  const uint32_t e = s_epoch;
  const int W = st.world, me = st.rank, tid = threadIdx.x;
  if (kind == 1) {
    if (tid < W) reinterpret_cast<int64_t*>(st.peer[tid].sync + STRIP_SYNC_BIRTHS)[me] = st.births[me];
  } else if (kind == 2) {
    for (int k = tid; k < W * n_counts; k += blockDim.x) {
      const int r = k / n_counts, i = k - r * n_counts;
      reinterpret_cast<int32_t*>(st.peer[r].sync + STRIP_SYNC_COUNTS)[(size_t)me * st.counts_cap + i] = counts[i];
    }
  } else if (kind == 3) {
    if (tid < W) reinterpret_cast<unsigned long long*>(st.peer[tid].sync + STRIP_SYNC_NMAX)[me] = *nmax;
  } else if (kind == 4) {
    if (tid < W) reinterpret_cast<int64_t*>(st.peer[tid].sync + STRIP_SYNC_PAIRS)[me] = st.pairs[me];
  }
  __threadfence_system();
  __syncthreads();
  if (tid < W && tid != me) {
    st_release_sys_u32(reinterpret_cast<uint32_t*>(st.peer[tid].sync + STRIP_SYNC_FLAGS) + me, e);
    const uint32_t* f = reinterpret_cast<const uint32_t*>(st.peer[me].sync + STRIP_SYNC_FLAGS) + tid;
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys_u32(f) - e) < 0) {
      if (clock64() - t0 > (10ll << 30)) { atomicOr(st.err, 4); break; }
      __nanosleep(64);
    }
  }
  __syncthreads();
  __threadfence_system();
  const unsigned char* mine = st.peer[me].sync;
  if (kind == 1) {
    if (tid < W) st.births[tid] = reinterpret_cast<const volatile int64_t*>(mine + STRIP_SYNC_BIRTHS)[tid];
  } else if (kind == 2) {
    const volatile int32_t* in = reinterpret_cast<const volatile int32_t*>(mine + STRIP_SYNC_COUNTS);
    for (int i = tid; i < n_counts; i += blockDim.x) {
      int32_t sum = 0;
      for (int r = 0; r < W; ++r) sum += in[(size_t)r * st.counts_cap + i];
      counts[i] = sum;
    }
  } else if (kind == 3) {
    if (tid == 0) {
      const volatile unsigned long long* in = reinterpret_cast<const volatile unsigned long long*>(mine + STRIP_SYNC_NMAX);
      unsigned long long m = 0;                       // non-negative doubles order like their bit patterns
      for (int r = 0; r < W; ++r) m = in[r] > m ? in[r] : m;
      *nmax = m;
    }
  } else if (kind == 4) {
    if (tid < W) st.pairs[tid] = reinterpret_cast<const volatile int64_t*>(mine + STRIP_SYNC_PAIRS)[tid];
  }
}

// Burn-in spatial statistic under strips (gnx_strip_burnin_count): this rank's individuals counted into its
// band of landscape rows [ly0, ly1), row iy - ly0, with k_burnin_count's transposed tally; an individual
// outside the band is counted in *outside (the caller reports it).
__global__ void __launch_bounds__(256) k_strip_burnin_count(Pop pop, Land land, const Counters* c, int ly0, int ly1,
                                                             int32_t* counts, int32_t* outside) {
  const int n = c->n, cur = c->cur;
  for (int p = GTID; p < n; p += GSTRIDE) {
    const double2 xy = pop.xy[cur][p];
    const int ix = (int)xy.x, iy = (int)xy.y;
    if (iy < ly0 || iy >= ly1) {
      atomicAdd(outside, 1);
      continue;
    }
    if (ix < land.Y && iy < land.X) atomicAdd(&counts[(size_t)(iy - ly0) * land.X + ix], 1);
  }
}
