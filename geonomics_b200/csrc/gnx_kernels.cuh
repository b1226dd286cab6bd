// gnx_kernels.cuh -- the per-timestep kernels (sm_100a).  Every kernel is a grid-stride /
// persistent kernel that reads its problem size from the device-resident Counters, so a
// whole time step is launched without a host round trip (and is CUDA-graph capturable).
//
// Order of the state (DESIGN.md section 3): the scalar SoA is kept in MATING-GRID order --
// (cell key, individual id) -- re-established every step by the re-grid that also applies the
// previous step's mortality.  Per-individual raster reads (conductance neighbourhood, K,
// death rate, environment) and the neighbour scan then touch contiguous memory; species
// order (ascending id) is produced on demand for the host (k_species_gather).
#pragma once
#include "gnx_common.cuh"
#include "gnx_scan.cuh"

#define GTID (blockIdx.x * blockDim.x + threadIdx.x)
#define GSTRIDE (gridDim.x * blockDim.x)

// ========================================================================================
// samplers of the movement / dispersal kernels.  Distances and free directions are drawn in
// float32 (the position update itself is float64, movement.py:75-92): a distance is a
// continuous random variable and its 2^-24 relative granularity is far below anything a KS
// test on 10^6 draws resolves (tests/test_cuda_samplers.py), while the float64 log / sqrt /
// cospi chain was the bulk of the 1490 instructions per individual of the round-1 kernel.
// ========================================================================================
__device__ __forceinline__ float uniform_f32(RngStream& g) { return (g.u32() >> 8) * (1.0f / 16777216.0f); }
// (0, 1] with the full 32 random bits near zero, for log(): tails reach 6.6 sigma
__device__ __forceinline__ float uniform_pos_f32(RngStream& g) { return ((float)g.u32() + 1.0f) * (1.0f / 4294967296.0f); }
__device__ __forceinline__ float normal_f32(RngStream& g) {
  const float u1 = uniform_pos_f32(g), u2 = uniform_f32(g);
  return sqrtf(-2.0f * __logf(u1)) * cospif(2.0f * u2);
}
// numpy legacy wald (inverse Gaussian), lognormal; scipy levy (loc + scale / Z^2)
__device__ __forceinline__ double sample_distance_f32(RngStream& g, int distr, double p1, double p2) {
  if (distr == GNX_DISTR_WALD) {
    const float mean = (float)p1, scale = (float)p2;
    const float mu_2l = mean / (2.0f * scale);
    float Y = normal_f32(g);
    Y = mean * Y * Y;
    const float X = mean + mu_2l * (Y - sqrtf(4.0f * scale * Y + Y * Y));
    const float U = uniform_f32(g);
    return (double)((U <= mean / (mean + X)) ? X : mean * mean / X);
  } else if (distr == GNX_DISTR_LOGNORMAL) {
    return (double)expf((float)p1 + (float)p2 * normal_f32(g));
  } else {
    const float Z = normal_f32(g);
    return p1 + p2 / ((double)Z * (double)Z);
  }
}

// von Mises(0, kappa) for the on-the-fly conductance surfaces: kappa is one number per species and
// the sample is about to be quantised to float16, so it is drawn by INVERSE CDF from a table built
// at setup (gnx_api.cu build_vm_table) instead of numpy's Best & Fisher rejection loop (cospif,
// division, logf, acosf and 2-3 uniforms per trip, ~1.5 trips, the trips of a warp's 32 lanes
// serialised).  One 32-bit word: sign | 12-bit cell | 19-bit position in the cell, linear
// inside a cell.  The last cell of the half-distribution -- where the quantile function turns
// steep -- is resolved by a second 256-cell table, so what is left to linear interpolation of
// the far tail is 2^-20 of the mass.  The sampled CDF is within 2.1e-5 of the exact one (for
// kappa from 0.5 to 500), 70x under what a KS test on 10^6 draws resolves; being uniform inside
// each cell, the sampled density is off by first order in the cell width, a total-variation
// distance of about 2.4e-4 (tests/test_cuda_surface_exact.py checks the tables against the exact
// quantile and the sampler draw for draw; tests/test_cuda_surface_onthefly.py checks it against
// the reference's tables).
#define VM_TAB_CELLS 4096
#define VM_TAB_FINE 256
#define VM_TAB_LEN (VM_TAB_CELLS + 1 + VM_TAB_FINE + 1)
__device__ __forceinline__ float vonmises_tab(RngStream& g, const float* __restrict__ tab, float kappa) {
  const float PI_F = 3.14159265358979f;
  if (kappa < 1e-8f) return PI_F * (2.0f * uniform_f32(g) - 1.0f);     // numpy: uniform on the circle
  const uint32_t r = g.u32();
  const uint32_t v = r << 1;                          // 31 random bits, left-aligned
  uint32_t k = v >> 20;                               // 12 bits: cell
  float a, b, f;
  if (k < VM_TAB_CELLS - 1) {
    f = (float)((v >> 1) & 0x7ffffu) * (1.0f / 524288.0f);
    a = __ldg(&tab[k]);
    b = __ldg(&tab[k + 1]);
  } else {
    const uint32_t k2 = (v >> 12) & 0xffu;            // 8 bits: fine cell inside the last cell
    f = (float)((v >> 1) & 0x7ffu) * (1.0f / 2048.0f);
    a = __ldg(&tab[VM_TAB_CELLS + 1 + k2]);
    b = __ldg(&tab[VM_TAB_CELLS + 2 + k2]);
  }
  const float res = fmaf(f, b - a, a);
  return (r >> 31) ? -res : res;
}

// On-the-fly conductance-surface direction.  The reference pre-draws `approx_len` float16
// samples per cell from this same distribution (spatial.py:365-461); at 4096^2 that table
// would be 168 GB, so the sample is drawn here instead.  `nv` = the 8 queen neighbours of the
// zero-embedded raster in row-major order (focal dropped), however they were fetched.
__device__ __forceinline__ __half surface_direction_from_neigh(RngStream& g, const float* nv, int mixture,
                                                               float kappa, const float* __restrict__ vm_tab) {
  const float PI_F = 3.14159265358979f;
  const float dirs[8] = {-3 * PI_F / 4, -PI_F / 2, -PI_F / 4, PI_F, 0.0f, 3 * PI_F / 4, PI_F / 2, PI_F / 4};
  float sum = 0.0f, mx = -1.0f;
#pragma unroll
  for (int k = 0; k < 8; ++k) { sum += nv[k]; mx = fmaxf(mx, nv[k]); }
  float loc;
  if (mixture) {
    // spatial.py:411-419: direction k with probability nv[k] / sum (uniform when all are zero)
    const float target = uniform_f32(g) * (sum > 0.0f ? sum : 8.0f);
    float acc = 0.0f;
    loc = dirs[7];
    bool found = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      acc += sum > 0.0f ? nv[k] : 1.0f;
      if (!found && target < acc) { loc = dirs[k]; found = true; }
    }
  } else {
    // spatial.py:376-381: mean of the directions of the maximum-valued neighbours
    float sacc = 0.0f;
    int cnt = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k)
      if (nv[k] == mx) { sacc += dirs[k]; cnt += 1; }
    loc = sacc / cnt;
  }
  // scipy vonmises.rvs(kappa, loc) = mod(loc + vonmises(0, kappa) + pi, 2 pi) - pi (scipy >= 1.11
  // wraps onto [-pi, pi); that is the scipy the reference runs on here), stored as float16 like
  // the reference table (spatial.py:447)
  float v = loc + vonmises_tab(g, vm_tab, kappa);
  if (v >= PI_F) v -= 2.0f * PI_F;
  else if (v < -PI_F) v += 2.0f * PI_F;
  return __float2half_rn(v);
}

__device__ __forceinline__ __half surface_direction_onthefly(RngStream& g, const float* rast, int X, int Y,
                                                             int cx, int cy, int mixture, float kappa,
                                                             const float* __restrict__ vm_tab) {
  // spatial.py:432-461: 3x3 neighbourhood of the zero-embedded raster, focal cell dropped
  const int di[8] = {-1, -1, -1, 0, 0, 1, 1, 1};
  const int dj[8] = {-1, 0, 1, -1, 1, -1, 0, 1};
  float nv[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int i = cy + di[k], j = cx + dj[k];
    nv[k] = (i >= 0 && i < Y && j >= 0 && j < X) ? __ldg(&rast[(size_t)i * X + j]) : 0.0f;
  }
  return surface_direction_from_neigh(g, nv, mixture, kappa, vm_tab);
}

// cos / sin of a float16 direction exactly as numpy evaluates them on a float16 array (half ->
// float, correctly rounded cosf, -> half; movement.py:75-76 with the float16 `direction` of
// spatial.py:184,447): one lookup in the 256 KB table of all 65536 halves built at setup
__device__ __forceinline__ void sincos_half_tab(const uint32_t* __restrict__ cs_tab, __half h, double* s, double* c) {
  const uint32_t v = __ldg(&cs_tab[__half_as_ushort(h)]);
  *c = (double)__half2float(__ushort_as_half((unsigned short)(v & 0xffffu)));
  *s = (double)__half2float(__ushort_as_half((unsigned short)(v >> 16)));
}

// mating-grid cell of a position, packed (cy << 16 | cx); the grid has < 65536 cells per axis
// floor(fl(x / c)) -- the cell index as numpy computes it -- without the FP64 division wherever the quotient
// is clear of an integer: q = x * fl(1 / c) is within 3 ulp(q) < 2.3e-11 of fl(x / c) for q < 2^16 (a grid has
// fewer than 65536 cells per axis), so outside a 1e-9 band around the integers both floors agree; inside the
// band (one position in ~5e8) the division decides
__device__ __forceinline__ int cell_index(double x, double c, double inv_c) {
  const double q = x * inv_c;
  const double fq = floor(q);
  const double fr = q - fq;
  if (fr > 1e-9 && fr < 1.0 - 1e-9) return (int)fq;
  return (int)floor(x / c);
}
__device__ __forceinline__ uint32_t mating_cell(const Land& land, double x, double y) {
  int cx = cell_index(x, land.cell_size, land.inv_cell_size), cy = cell_index(y, land.cell_size, land.inv_cell_size);
  cx = min(cx, land.ncx - 1);
  cy = min(cy, land.ncy - 1);
  return ((uint32_t)cy << 16) | (uint32_t)cx;
}
__device__ __forceinline__ uint32_t cell_linear(const Land& land, uint32_t packed) {
  return (packed >> 16) * (uint32_t)land.ncx + (packed & 0xffffu);
}

#include "gnx_strip.cuh"

// ========================================================================================
// a1 + a2 + a4 (+ a16 removal): age, movement, mating-grid key + per-cell histogram; entries the
// previous step's mortality flagged dead are dropped here (their genome rows go back to the
// free list) -- the re-grid that follows never copies them.
//   species.py:567-569 (age); movement.py:34-95 (movement); spatial.py:182-184 (surface
//   lookup); species.py:937-939 (cells); demography.py:175-180 (removal).  Flags select which
//   parts run so the stage-level C-ABI entry points and the fused step share one kernel.
// ========================================================================================
__global__ void __launch_bounds__(256) k_move_key(Pop pop, Land land, Params prm, DevDraws dr,
                                                   Work w, Counters* c, int do_age, int do_move,
                                                   int do_key, const Strip* st) {
  const int n = c->n, cur = c->cur, pending = c->pending;
  const int64_t t = c->t;
  double2* __restrict__ XY = pop.xy[cur];
  const int32_t* __restrict__ ord = prm.ordered ? pop.ord[cur] : nullptr;
  const int lane = threadIdx.x & 31;
  __shared__ int s_free_off[9];                         // per-warp offsets of the freed rows + the CTA's base
  // whole CTAs stay in the loop (ballots and barriers below): the tail is masked by `in`
  for (int base = blockIdx.x * blockDim.x; base < n; base += GSTRIDE) {
    const int p = base + threadIdx.x;
    const bool in = p < n;
    const bool dead = in && pending && !w.alive[p];
    if (pending && do_key) {
      // lazy mortality (demography.py:175-180): the dead leave the population here and their genome
      // rows go back to the free list.  ONE atomic on the list cursor per CTA pass (the per-warp
      // form queued ~3e5 same-address atomics per step at c4: a third of this kernel's stall samples)
      const unsigned dm = __ballot_sync(0xffffffffu, dead && !prm.burn);
      __syncthreads();                                    // the previous pass has read s_free_off
      if (lane == 0) s_free_off[threadIdx.x >> 5] = __popc(dm);
      __syncthreads();
      if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int ck = s_free_off[k]; s_free_off[k] = tot; tot += ck; }
        s_free_off[8] = tot ? atomicAdd(&c->n_free, tot) : 0;
      }
      __syncthreads();
      if (dead && !prm.burn)
        pop.free_slots[s_free_off[8] + s_free_off[threadIdx.x >> 5] + __popc(dm & ((1u << lane) - 1u))] = pop.gslot[cur][p];
      if (dead) w.mkey[p] = GNX_KEY_DEAD;
    }
    // no early exit: the whole warp takes part in the cell-count aggregation at the end
    const bool act = in && !dead;
    if (act && do_age) pop.age[cur][p] += 1;
    double x = 0.0, y = 0.0;
    if (act) {
      const double2 xy0 = XY[p];
      x = xy0.x;
      y = xy0.y;
    }
    if (act && do_move) {
      const int io = ord ? ord[p] : p;                  // injected draws are indexed by species ordinal
      RngStream g(prm.seed_lo, prm.seed_hi, pop.idx[cur][p], SITE_MOVE, t);
      double cs, sn;
      if (prm.c.move_surf_mode == GNX_SURF_TABLE) {
        const int cx = (int)x, cy = (int)y;
        const int col = dr.move_choice ? dr.move_choice[io] : (int)choose_k(g.u32(), prm.c.surf_approx_len);
        const __half h = prm.move_tab[((size_t)cy * land.X + cx) * prm.c.surf_approx_len + col];
        sincos_half_tab(prm.cs_tab, h, &sn, &cs);
      } else if (prm.c.move_surf_mode == GNX_SURF_ONTHEFLY) {
        const __half d = surface_direction_onthefly(g, land.surf_f32[0], land.X, land.Y, (int)x, (int)y,
                                                    prm.c.move_surf_mixture, (float)prm.c.move_surf_kappa, prm.vm_tab[0]);
        sincos_half_tab(prm.cs_tab, d, &sn, &cs);
      } else if (dr.move_dir) {
        sincos(dr.move_dir[io], &sn, &cs);
      } else if (prm.c.dir_kappa < 1e-8) {
        // numpy vonmises(mu, kappa < 1e-8) = pi*(2U - 1) (mu ignored): movement.py:55
        float sf, cf;
        sincospif(2.0f * uniform_f32(g) - 1.0f, &sf, &cf);
        sn = (double)sf;
        cs = (double)cf;
      } else {
        sincos(sample_vonmises(g, prm.c.dir_mu, prm.c.dir_kappa), &sn, &cs);
      }
      const double dist = dr.move_dist ? dr.move_dist[io]
                                       : sample_distance_f32(g, prm.c.move_distr, prm.c.move_p1, prm.c.move_p2);
      double dx = __dmul_rn(cs, dist), dy = __dmul_rn(sn, dist);
      if (prm.c.res_ratio_x != 1.0) dx = __dmul_rn(dx, prm.c.res_ratio_x);
      if (prm.c.res_ratio_y != 1.0) dy = __dmul_rn(dy, prm.c.res_ratio_y);
      x = clampd(__dadd_rn(x, dx), 0.0, land.max_x);
      y = clampd(__dadd_rn(y, dy), 0.0, land.max_y);
      XY[p] = make_double2(x, y);
    }
    if (do_key) {
      uint32_t key = 0u;
      uint32_t lin = 0xffffffffu - (uint32_t)lane;       // a value no other lane and no cell has
      bool keyed = false;
      if (act) {
        key = mating_cell(land, x, y);
        keyed = true;
        if (st) {
          // strip decomposition: an individual that moved out of this rank's rows is listed for
          // shipping to the rank that owns its new row and leaves this rank's grid (and gives
          // its genome slot back; the row is read by k_strip_send before any slot is re-used)
          const int row = (int)(key >> 16);
          if (row < st->row0 || row >= st->row1) {
            strip_list(st, p, strip_owner(st, row));
            w.mkey[p] = GNX_KEY_DEAD;
            if (!prm.burn) pop.free_slots[atomicAdd(&c->n_free, 1)] = pop.gslot[cur][p];
            keyed = false;
          }
        }
        if (keyed) lin = cell_linear(land, key);
      }
      // The entries are in last step's grid order and move about one cell, so the lanes of a warp
      // land in few distinct cells: the lanes of one cell share ONE histogram update, and it is a
      // fire-and-forget reduction (nothing here waits for its result: the arrival ranks inside a
      // cell are handed out by k_bucket, which has the residency to hide that round trip).
      const unsigned peers = __match_any_sync(0xffffffffu, lin);
      if (keyed) {
        if (lane == __ffs(peers) - 1) atomicAdd(&w.cell_count[lin], (uint32_t)__popc(peers));
        w.mkey[p] = key;
      }
    }
  }
}

// exclusive scan of the per-cell histogram -> cell_start
struct CellScan {
  uint32_t* cnt;
  uint32_t* start;
  int ncell;
  __device__ int size(const Counters*) const { return ncell; }
  __device__ u64 value(int i) const { return cnt[i]; }
  // the counts become k_bucket's per-cell fill cursors: back to zero once they are scanned
  __device__ void apply(int i, u64 v, u64 ex) const {
    start[i] = (uint32_t)ex;
    if (v) cnt[i] = 0u;
  }
  __device__ void total(Counters* c, u64 tot) const {
    start[ncell] = (uint32_t)tot;
    c->n_regrid = (int)tot;
  }
};

// every surviving entry announces itself in its destination cell's range, in arrival order: the
// slot inside the range comes from the cell's fill cursor (one atomic per (warp, cell), the lanes
// of a cell ranked by lane order); the re-grid orders each range by id whatever the arrival order
__global__ void __launch_bounds__(256) k_bucket(Pop pop, Land land, Work w, const Counters* c) {
  const int n = c->n, cur = c->cur;
  const int lane = threadIdx.x & 31;
  // two entries per thread and pass: the two cursor round trips overlap
  for (int base = blockIdx.x * blockDim.x; base < n; base += 2 * GSTRIDE) {
    int p[2];
    uint32_t key[2], lin[2], slot[2];
    unsigned peers[2];
    bool keyed[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      p[u] = base + u * GSTRIDE + threadIdx.x;
      key[u] = p[u] < n ? w.mkey[p[u]] : GNX_KEY_DEAD;
      keyed[u] = key[u] != GNX_KEY_DEAD;
      lin[u] = keyed[u] ? cell_linear(land, key[u]) : 0xffffffffu - (uint32_t)lane;
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      peers[u] = __match_any_sync(0xffffffffu, lin[u]);
      slot[u] = 0u;
      if (keyed[u] && lane == __ffs(peers[u]) - 1) slot[u] = atomicAdd(&w.cell_count[lin[u]], (uint32_t)__popc(peers[u]));
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (!keyed[u]) continue;
      const uint32_t q = __shfl_sync(peers[u], slot[u], __ffs(peers[u]) - 1) + (uint32_t)__popc(peers[u] & ((1u << lane) - 1u));
      const unsigned long long id = (unsigned long long)pop.idx[cur][p[u]];
      w.bucket[w.cell_start[lin[u]] + q] = make_uint4((uint32_t)p[u], key[u], (uint32_t)id, (uint32_t)(id >> 32));
    }
  }
}

// The re-grid: destination entry q takes the source entry whose id has rank (q - cell start)
// among the ids of its cell -- (cell, id) order whatever order the histogram atomics retired
// in -- and gathers that entry's whole record into the other half.  One pass moves the state:
// it is this step's counting sort AND the previous step's mortality compaction.
__global__ void __launch_bounds__(256) k_regrid(Pop pop, Land land, Work w, Counters* c, int age_inc, int ordered,
                                                 const Strip* st) {
  const int total = c->n_regrid, s = c->cur, d = s ^ 1, T = pop.T;
  for (int q = GTID; q < total; q += GSTRIDE) {
    const uint4 e = w.bucket[q];
    const uint32_t lin = cell_linear(land, e.y);
    const int cs = (int)w.cell_start[lin], ce = (int)w.cell_start[lin + 1];
    const unsigned long long id = ((unsigned long long)e.w << 32) | e.z;
    int r = 0;
    for (int j = cs; j < ce; ++j) {
      const uint4 o = __ldg(&w.bucket[j]);
      r += ((((unsigned long long)o.w << 32) | o.z) < id) ? 1 : 0;
    }
    const int dst = cs + r, src = (int)e.x;
    // all loads of the record before its first store (the halves cannot be proven disjoint)
    const double2 xy = pop.xy[s][src];
    const double fit = pop.fit[s][src];
    const int32_t age = pop.age[s][src], gs = pop.gslot[s][src];
    const int8_t sx = pop.sex[s][src];
    double z[GNX_MAX_TRAITS];
#pragma unroll
    for (int tt = 0; tt < GNX_MAX_TRAITS; ++tt)
      if (tt < T) z[tt] = pop.z[s][(size_t)tt * pop.cap + src];
    int32_t na = 0, nb = 0, od = 0;
    if (pop.node[0][0]) { na = pop.node[0][s][src]; nb = pop.node[1][s][src]; }
    if (ordered) od = pop.ord[s][src];
    pop.xy[d][dst] = xy;
    pop.fit[d][dst] = fit;
    pop.idx[d][dst] = (int64_t)id;
    pop.age[d][dst] = age + age_inc;
    pop.gslot[d][dst] = gs;
    pop.sex[d][dst] = sx;
#pragma unroll
    for (int tt = 0; tt < GNX_MAX_TRAITS; ++tt)
      if (tt < T) pop.z[d][(size_t)tt * pop.cap + dst] = z[tt];
    if (pop.node[0][0]) { pop.node[0][d][dst] = na; pop.node[1][d][dst] = nb; }
    if (ordered) { pop.ord[d][dst] = od; w.inv[od] = dst; }
    w.skey[dst] = e.y;
  }
  // the last block to finish publishes the new population: size, order, buffer parity
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(&c->ticket[0], 1u) == gridDim.x - 1;
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    c->n = total;
    c->n_pre = total;
    c->n_sorted = total;
    c->pending = 0;
    c->cur = d;
    c->ticket[0] = 0u;
    // entries this rank owns: its mating-grid rows are one contiguous range of the (cell, id) order
    c->own_lo = st ? (int)w.cell_start[st->row0 * land.ncx] : 0;
    c->own_hi = st ? (int)w.cell_start[st->row1 * land.ncx] : total;
  }
}

// ========================================================================================
// a5: neighbour scan + mate choice.  species.py:2157-2215, spatial.py:191-245.
//   The state is in (cell, id) order, so the candidates of a focal are three contiguous
//   ranges of pop.xy (its 3x3 cell block, row by row) read with 128-bit loads, consecutive
//   focals share them through L1, and a candidate's position in the arrays IS its canonical
//   rank.  Closed ball on squared distances, products and sum rounded separately (as the
//   reference's cKDTree does).
//   MODE 0: uniform random neighbour (spatial.py:232-242); valid candidates are kept as bit
//           masks and the k-th is picked, k = (R * count) >> 32.  Cells whose 3x3 block is
//           crowded (a row range longer than 64 entries, or focals x candidates >= FM_HEAVY_WORK)
//           are not searched here: k_mate_select appends one work item per 32 focals of such a cell
//           to Work.heavy and k_find_mates_dense takes them, one warp per item with the lanes across
//           candidates.  All three kernels search only the focals whose Bernoulli(b) draw lets them
//           mate (k_mate_select)
//   MODE 1: nearest neighbour (spatial.py:194-203)
//   MODE 2: inverse-distance weighting, p ~ (radius - dist) (spatial.py:209-229)
// ========================================================================================
constexpr int FM_HEAVY_WORK = 4096;   // measured flat from 3072 to 16384 at c4 (t = 300); 256-768 are 10-35 % slower
// position of the (k+1)-th set bit of m: popcount bisection (branch-free; __fns is a software loop)
__device__ __forceinline__ int kth_set_bit(uint32_t m, int k) {
  int bit = 0;
#pragma unroll
  for (int wdt = 16; wdt >= 1; wdt >>= 1) {
    const int cl = __popc(m & ((1u << wdt) - 1u));
    if (k >= cl) { k -= cl; m >>= wdt; bit += wdt; }
  }
  return bit;
}

// the crowded-cell test of MODE 0 (see k_find_mates): l0..l2 = lengths of the three candidate row ranges,
// nf = focals of the cell
__device__ __forceinline__ bool fm_is_heavy(int l0, int l1, int l2, int nf) {
  return max(l0, max(l1, l2)) > 64 || nf * (l0 + l1 + l2) >= FM_HEAVY_WORK;
}

// Bernoulli(b) FIRST.  The reference lists every focal's neighbours, lets each focal pick one and only then
// keeps the pair with probability b (species.py:2212-2214) -- the draw is independent of the search, so a
// focal whose draw fails needs no search at all (b = 0.2 at the BASELINE configs: four searches in five).
// Lanes that skip inside a thread-per-focal loop would save nothing (the warp runs as long as its busiest
// lane), so the focals that may mate are COMPACTED into a list here and only they are searched.  The draws
// come from the same Philox stream positions (or injected arrays) as the pick in the search kernels, so the
// result is the one the search-everything form gave, bit for bit.  With store_debug (the parity tests read
// every focal's neighbour count) everyone is listed.  Also announces the crowded cells' work items (one per
// batch of 32 focals of a cell, by the batch's first entry) for k_find_mates_dense.
// draw order per focal -- MODE 0: R, u; MODE 1: u; MODE 2: u_inv, u (each either injected or from the stream)
template <int MODE>
__device__ __forceinline__ double mate_keep_draw(RngStream& g, const DevDraws& dr, int io, uint32_t* R, double* u_inv) {
  if (MODE == 0) *R = dr.mate_R ? dr.mate_R[io] : g.u32();
  if (MODE == 2) *u_inv = dr.mate_inv_u ? dr.mate_inv_u[io] : g.uniform();
  return dr.mate_u ? dr.mate_u[io] : g.uniform();
}

template <int MODE>
__global__ void __launch_bounds__(256) k_mate_select(Pop pop, Land land, Params prm, DevDraws dr, Work w, Counters* c) {
  const int n = c->n, cur = c->cur;
  const int64_t t = c->t;
  const int32_t* __restrict__ ord = prm.ordered ? pop.ord[cur] : nullptr;
  const int own_lo = c->own_lo, own_hi = c->own_hi;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __shared__ int s_off[9];                              // per-warp offsets of the listed focals + the CTA's base
  __shared__ int s_hoff[9];                             // the same for the crowded-cell work items
  for (int base = blockIdx.x * blockDim.x; base < n; base += GSTRIDE) {      // whole CTAs stay (ballot, barriers)
    const int p = base + threadIdx.x;
    bool act = false, heavy = false;
    uint32_t hkey = 0u;
    if (p < n) {
      if (p >= own_lo && p < own_hi) {             // else a ghost of a neighbouring strip: candidate, never focal
        if (MODE == 0) {
          const uint32_t key = w.skey[p];
          const int cx = (int)(key & 0xffffu), cy = (int)(key >> 16);
          const int fs = (int)w.cell_start[cy * land.ncx + cx];
          if (((p - fs) & 31) == 0) {
            const int x0 = max(cx - 1, 0), x1 = min(cx + 1, land.ncx - 1);
            int len[3];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
              const int row = cy - 1 + r;
              len[r] = (row < 0 || row >= land.ncy) ? 0
                     : (int)w.cell_start[row * land.ncx + x1 + 1] - (int)w.cell_start[row * land.ncx + x0];
            }
            const int nf = (int)w.cell_start[cy * land.ncx + cx + 1] - fs;
            heavy = fm_is_heavy(len[0], len[1], len[2], nf);
            hkey = key;
          }
        }
        RngStream g(prm.seed_lo, prm.seed_hi, pop.idx[cur][p], SITE_MATE, t);
        uint32_t R;
        double u_inv;
        const double u = mate_keep_draw<MODE>(g, dr, ord ? ord[p] : p, &R, &u_inv);
        act = u < prm.c.b || prm.store_debug;
      }
      if (!act) w.mate[p] = -1;
    }
    // ONE atomic on the list cursor per CTA pass: a per-warp atomic is 3.7e5 same-address atomics per step at
    // c4 -- they serialise in one L2 slice and were 75 % of this kernel's time (249 us)
    const unsigned am = __ballot_sync(0xffffffffu, act);
    const unsigned hm = MODE == 0 ? __ballot_sync(0xffffffffu, heavy) : 0u;
    __syncthreads();                                      // the previous pass has read s_off
    if (lane == 0) { s_off[wid] = __popc(am); s_hoff[wid] = __popc(hm); }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0, htot = 0;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int ck = s_off[k], hk = s_hoff[k];
        s_off[k] = tot; tot += ck;
        s_hoff[k] = htot; htot += hk;
      }
      s_off[8] = tot ? atomicAdd(w.fm_count, tot) : 0;
      s_hoff[8] = htot ? atomicAdd(&c->n_heavy, htot) : 0;
    }
    __syncthreads();
    if (act) w.fm_list[s_off[8] + s_off[wid] + __popc(am & ((1u << lane) - 1u))] = p;
    if (heavy) {
      const int pos = s_hoff[8] + s_hoff[wid] + __popc(hm & ((1u << lane) - 1u));
      if (pos < w.heavy_cap) w.heavy[pos] = make_uint2(hkey, (uint32_t)p);
      else atomicOr(&c->err, GNX_ERRBIT_CAPACITY);
    }
  }
}

constexpr int FM_BLOCK = 128;   // threads per CTA of k_find_mates (its launch bound and its launch)
template <int MODE>
__global__ void __launch_bounds__(FM_BLOCK) k_find_mates(Pop pop, Land land, Params prm, DevDraws dr, Work w,
                                                         Counters* c) {
  const int cur = c->cur;
  const int64_t t = c->t;
  const double r2 = prm.r2, radius = prm.c.mating_radius;
  const double2* __restrict__ sxy = pop.xy[cur];
  const int32_t* __restrict__ ord = prm.ordered ? pop.ord[cur] : nullptr;
  const int n_list = *w.fm_count;                  // the focals k_mate_select let through
  for (int li = GTID; li < n_list; li += GSTRIDE) {
    const int p = w.fm_list[li];
    const double2 f = sxy[p];
    const uint32_t key = w.skey[p];
    const int cx = (int)(key & 0xffffu), cy = (int)(key >> 16);
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, land.ncx - 1);
    int lo[3], hi[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      int row = cy - 1 + r;
      if (row < 0 || row >= land.ncy) { lo[r] = hi[r] = 0; continue; }
      lo[r] = w.cell_start[row * land.ncx + x0];
      hi[r] = w.cell_start[row * land.ncx + x1 + 1];
    }
    int cnt = 0;
    if (MODE == 0) {
      // crowded block: the whole cell goes to k_find_mates_dense (the test depends on the cell
      // only, so every focal of the cell takes this exit; the cell's first entry announces it)
      const int l0 = hi[0] - lo[0], l1 = hi[1] - lo[1], l2 = hi[2] - lo[2];
      const int fs = (int)w.cell_start[cy * land.ncx + cx], nf = (int)w.cell_start[cy * land.ncx + cx + 1] - fs;
      // both kernels are bound by the six FP64 operations of a distance test; the warp-per-batch
      // kernel loses lanes to padding (candidates in chunks of 32, focals in batches of 32), this
      // one to trip-count divergence: a cell moves over when its focals x candidates product is
      // large enough for the padding not to matter (or a row range exceeds the masks here)
      if (fm_is_heavy(l0, l1, l2, nf)) continue;      // (its work items were announced by k_mate_select)
    }
    // MODE 0 keeps the valid candidates of each row range as two 32-bit masks in registers
    // (candidates 0-31 and 32-63 of the range)
    uint32_t vm[3] = {0u, 0u, 0u}, vh[3] = {0u, 0u, 0u};
    double best = 1e300, wsum = 0.0;
    int best_q = -1, n_w = 0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int len = hi[r] - lo[r];
      const double2* __restrict__ cand = sxy + lo[r];
      const int self = p - lo[r];                   // position of the focal in this range, if any
      if (MODE == 0) {
        uint32_t m = 0u, mh = 0u;
        const int len0 = min(len, 32);
#pragma unroll 4
        for (int j = 0; j < len0; ++j) {
          const double2 cxy = cand[j];
          const double dx = cxy.x - f.x, dy = cxy.y - f.y;
          const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
          m |= (d2 <= r2 ? 1u : 0u) << j;
        }
        if (len > 32) {
          const int len1 = min(len, 64) - 32;
          for (int j = 0; j < len1; ++j) {
            const double2 cxy = cand[32 + j];
            const double dx = cxy.x - f.x, dy = cxy.y - f.y;
            const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            mh |= (d2 <= r2 ? 1u : 0u) << j;
          }
        }
        if (self >= 0 && self < len) {
          if (self < 32) m &= ~(1u << self);
          else if (self < 64) mh &= ~(1u << (self - 32));
        }
        vm[r] = m;
        vh[r] = mh;
        cnt += __popc(m) + __popc(mh);
      } else {
        for (int j = 0; j < len; ++j) {
          const double2 cxy = cand[j];
          const double dx = cxy.x - f.x, dy = cxy.y - f.y;
          const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
          if (d2 <= r2 && j != self) {
            if (MODE == 1) { if (d2 < best) { best = d2; best_q = lo[r] + j; } }
            if (MODE == 2) { const double d = sqrt(d2); if (d != 0.0) { wsum += radius - d; n_w += 1; } }
            cnt += 1;
          }
        }
      }
    }
    if (prm.store_debug) w.n_nbrs[p] = cnt;
    int mate = -1;
    if (cnt > 0) {
      const int io = ord ? ord[p] : p;
      RngStream g(prm.seed_lo, prm.seed_hi, pop.idx[cur][p], SITE_MATE, t);
      int sel_q = -1;
      if (MODE == 1) {
        sel_q = best_q;
      } else if (MODE == 2) {
        if (n_w > 0) {
          const double u = dr.mate_inv_u ? dr.mate_inv_u[io] : g.uniform();
          const double target = u * wsum;
          double acc = 0.0;
          int last = -1;
#pragma unroll
          for (int r = 0; r < 3; ++r)
            for (int q = lo[r]; q < hi[r] && sel_q < 0; ++q) {
              const double2 cxy = sxy[q];
              const double dx = cxy.x - f.x, dy = cxy.y - f.y;
              const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
              if (d2 <= r2 && q != p) {
                const double d = sqrt(d2);
                acc += (d != 0.0) ? radius - d : 0.0;
                last = q;
                if (target < acc) sel_q = q;
              }
            }
          if (sel_q < 0) sel_q = last;
        }
      } else {
        const uint32_t R = dr.mate_R ? dr.mate_R[io] : g.u32();
        int k = (int)choose_k(R, (uint32_t)cnt);
        uint32_t msel = 0u;
        int base_q = 0;
        bool found = false;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const int cr = __popc(vm[r]);
          if (!found) {
            if (k < cr) { msel = vm[r]; base_q = lo[r]; found = true; }
            else k -= cr;
          }
          const int ch = __popc(vh[r]);
          if (!found) {
            if (k < ch) { msel = vh[r]; base_q = lo[r] + 32; found = true; }
            else k -= ch;
          }
        }
        sel_q = base_q + kth_set_bit(msel, k);
      }
      if (sel_q >= 0) {
        const double u = dr.mate_u ? dr.mate_u[io] : g.uniform();
        if (u < prm.c.b) mate = sel_q;               // species.py:2212-2214
      }
    }
    w.mate[p] = mate;
  }
}

// ----- k_find_mates_dense: the crowded cells of MODE 0, one warp per batch of 32 focals -----
// Evolved populations clump (c4 after 1000 steps: 94 neighbours per individual on average, 350
// at the 99th percentile), and a thread per focal then walks hundreds of candidates with its
// own trip count.  Here the LANES run across the candidates of the cell's 3x3 block (three
// contiguous ranges of pop.xy): each lane keeps up to FMD_CG candidates in registers (coalesced
// 128-bit loads, once per batch of 32 focals), the focals of the batch are broadcast one after
// the other from shared memory, and a ballot per 32 candidates IS the validity mask in
// canonical order.  The masks go to shared memory [focal][chunk]; then the lanes switch to one
// focal each for the count, the draw and the k-th-neighbour pick -- same counts, same canonical
// order, same Philox stream as k_find_mates, so the two kernels are interchangeable bit for bit.
// The distance test is the reference's (products and sum rounded separately, closed ball); the
// comparison itself is done on the bit patterns (non-negative doubles order like integers),
// which takes it off the FP64 pipe that bounds this kernel.
// Blocks of up to 64 chunks (2048 candidates) keep their masks; larger ones are swept twice
// (count, then pick) without storing them.  Work items are handed out by an atomic cursor.
#define FMD_WARPS 4
#define FMD_CHUNKS 64
#define FMD_CG 4                       // chunks of 32 candidates held in registers at a time
#define FMD_STRIDE (FMD_CHUNKS + 4)    // row stride in words: rows stay 16-byte aligned

struct FmdBlock {                      // the 3x3 block of a crowded cell as one candidate sequence
  int lo0, lo1, lo2, e1, e2, K;
  __device__ __forceinline__ int entry(int ci) const {
    return ci < e1 ? lo0 + ci : (ci < e2 ? lo1 + (ci - e1) : lo2 + (ci - e2));
  }
};

// ballots of NC chunks (held in cv) against focal f
template <int NC>
__device__ __forceinline__ void fmd_ballots(const double2* cv, const double2 f, long long r2b, uint32_t* bm) {
#pragma unroll
  for (int j = 0; j < FMD_CG; ++j) {
    if (j < NC) {
      const double dx = cv[j].x - f.x, dy = cv[j].y - f.y;
      const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
      bm[j] = __ballot_sync(0xffffffffu, __double_as_longlong(d2) <= r2b);
    } else {
      bm[j] = 0u;
    }
  }
}

template <int NC>
__device__ __forceinline__ void fmd_group(const double2* __restrict__ sxy, const FmdBlock& blk, const double2* foc,
                                          uint32_t (*mk)[FMD_STRIDE], int nf, int cg, int lane, long long r2b,
                                          uint32_t amask) {
  double2 cv[FMD_CG];
#pragma unroll
  for (int j = 0; j < FMD_CG; ++j) {
    if (j < NC) {
      const int ci = ((cg + j) << 5) + lane;
      // lanes past the end hold a point at infinity: it fails every distance test
      cv[j] = ci < blk.K ? sxy[blk.entry(ci)] : make_double2(1e300, 1e300);
    }
  }
  // only the focals whose Bernoulli(b) draw lets them mate (amask, uniform across the warp)
  for (uint32_t rest = amask; rest; rest &= rest - 1u) {
    const int fi = __ffs(rest) - 1;
    uint32_t bm[FMD_CG];
    fmd_ballots<NC>(cv, foc[fi], r2b, bm);
    if (lane == 0) *reinterpret_cast<uint4*>(&mk[fi][cg]) = make_uint4(bm[0], bm[1], bm[2], bm[3]);
  }
}

__global__ void __launch_bounds__(32 * FMD_WARPS) k_find_mates_dense(Pop pop, Land land, Params prm, DevDraws dr,
                                                                       Work w, Counters* c) {
  __shared__ __align__(16) uint32_t smask[FMD_WARPS][32][FMD_STRIDE];
  __shared__ double2 sfoc[FMD_WARPS][32];
  const int n_heavy = min(c->n_heavy, w.heavy_cap), cur = c->cur;
  const int64_t t = c->t;
  const long long r2b = __double_as_longlong(prm.r2);
  const double2* __restrict__ sxy = pop.xy[cur];
  const int32_t* __restrict__ ord = prm.ordered ? pop.ord[cur] : nullptr;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t (*mk)[FMD_STRIDE] = smask[wid];
  double2* foc = sfoc[wid];
  for (;;) {
    int h = 0;
    if (lane == 0) h = atomicAdd(&c->heavy_next, 1);
    h = __shfl_sync(0xffffffffu, h, 0);
    if (h >= n_heavy) break;
    const uint2 item = w.heavy[h];
    const uint32_t key = item.x;
    const int fb = (int)item.y;
    const int cx = (int)(key & 0xffffu), cy = (int)(key >> 16);
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, land.ncx - 1);
    int lo[3], len[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int row = cy - 1 + r;
      if (row < 0 || row >= land.ncy) { lo[r] = 0; len[r] = 0; continue; }
      lo[r] = (int)w.cell_start[row * land.ncx + x0];
      len[r] = (int)w.cell_start[row * land.ncx + x1 + 1] - lo[r];
    }
    FmdBlock blk;
    blk.lo0 = lo[0]; blk.lo1 = lo[1]; blk.lo2 = lo[2];
    blk.e1 = len[0]; blk.e2 = len[0] + len[1]; blk.K = blk.e2 + len[2];
    const int nch = (blk.K + 31) >> 5;
    const bool keep = nch <= FMD_CHUNKS;
    const int fe = (int)w.cell_start[cy * land.ncx + cx + 1];
    const int nf = min(32, fe - fb);
    const int p = fb + lane;
    const double2 myf = lane < nf ? sxy[p] : make_double2(0.0, 0.0);
    const int self = blk.e1 + (p - lo[1]);             // the focal's own position among the candidates
    foc[lane] = myf;
    __syncwarp();
    int cnt = 0, sel_q = -1, k = 0;
    uint32_t R = 0u;
    double u_keep = 1.0;
    const int io = (lane < nf && ord) ? ord[p] : p;
    // Bernoulli(b) first (see k_mate_select): the draws of this lane's focal, from the stream positions the
    // pick below used to take them from; focals that may not mate are not searched at all
    bool act = false;
    if (lane < nf) {
      RngStream g(prm.seed_lo, prm.seed_hi, pop.idx[cur][p], SITE_MATE, t);
      double u_inv;
      u_keep = mate_keep_draw<0>(g, dr, io, &R, &u_inv);
      act = u_keep < prm.c.b || prm.store_debug;
    }
    const uint32_t amask = __ballot_sync(0xffffffffu, act);
    if (amask == 0u) { __syncwarp(); continue; }       // (k_mate_select has set their mates to -1)
    if (keep) {
      // ---- lanes across candidates: FMD_CG chunks in registers, every listed focal of the batch against them
      int cg = 0;
      for (; cg + FMD_CG <= nch; cg += FMD_CG) fmd_group<FMD_CG>(sxy, blk, foc, mk, nf, cg, lane, r2b, amask);
      const int rem = nch - cg;
      if (rem == 1) fmd_group<1>(sxy, blk, foc, mk, nf, cg, lane, r2b, amask);
      else if (rem == 2) fmd_group<2>(sxy, blk, foc, mk, nf, cg, lane, r2b, amask);
      else if (rem == 3) fmd_group<3>(sxy, blk, foc, mk, nf, cg, lane, r2b, amask);
      __syncwarp();
      // ---- lanes across focals: count, pick (spatial.py:232-242, species.py:2212-2214)
      if (act) {
        const int ngrp = (nch + FMD_CG - 1) / FMD_CG * FMD_CG;
        mk[lane][self >> 5] &= ~(1u << (self & 31));
        for (int ch = 0; ch < ngrp; ++ch) cnt += __popc(mk[lane][ch]);
        if (cnt > 0) {
          k = (int)choose_k(R, (uint32_t)cnt);
          int ch = 0;
          uint32_t m = mk[lane][0];
          for (;;) {
            const int pc = __popc(m);
            if (k < pc) break;
            k -= pc;
            ch += 1;
            m = mk[lane][ch];
          }
          sel_q = blk.entry((ch << 5) + kth_set_bit(m, k));
        }
      }
    } else {
      // ---- more than 2048 candidates: sweep 1 counts, sweep 2 finds each focal's k-th neighbour
      for (int cg = 0; cg < nch; cg += FMD_CG) {
        double2 cv[FMD_CG];
#pragma unroll
        for (int j = 0; j < FMD_CG; ++j) {
          const int ci = ((cg + j) << 5) + lane;
          cv[j] = ci < blk.K ? sxy[blk.entry(ci)] : make_double2(1e300, 1e300);
        }
        for (uint32_t rest = amask; rest; rest &= rest - 1u) {
          const int fi = __ffs(rest) - 1;
          uint32_t bm[FMD_CG];
          fmd_ballots<FMD_CG>(cv, foc[fi], r2b, bm);
          const int sf = blk.e1 + (fb + fi - lo[1]);
          int pc = 0;
#pragma unroll
          for (int j = 0; j < FMD_CG; ++j) {
            if (cg + j == (sf >> 5)) bm[j] &= ~(1u << (sf & 31));
            pc += __popc(bm[j]);
          }
          if (lane == fi) cnt += pc;
        }
      }
      if (act && cnt > 0) k = (int)choose_k(R, (uint32_t)cnt);
      int run = 0;                                     // valid candidates of this lane's focal seen so far
      for (int cg = 0; cg < nch; cg += FMD_CG) {
        double2 cv[FMD_CG];
#pragma unroll
        for (int j = 0; j < FMD_CG; ++j) {
          const int ci = ((cg + j) << 5) + lane;
          cv[j] = ci < blk.K ? sxy[blk.entry(ci)] : make_double2(1e300, 1e300);
        }
        for (uint32_t rest = amask; rest; rest &= rest - 1u) {
          const int fi = __ffs(rest) - 1;
          const int kf = __shfl_sync(0xffffffffu, k, fi), cf = __shfl_sync(0xffffffffu, cnt, fi);
          int rf = __shfl_sync(0xffffffffu, run, fi);
          if (cf == 0 || rf > kf) continue;            // nothing to pick / already picked (uniform)
          uint32_t bm[FMD_CG];
          fmd_ballots<FMD_CG>(cv, foc[fi], r2b, bm);
          const int sf = blk.e1 + (fb + fi - lo[1]);
          int sel = -1;
#pragma unroll
          for (int j = 0; j < FMD_CG; ++j) {
            if (cg + j == (sf >> 5)) bm[j] &= ~(1u << (sf & 31));
            const int pc = __popc(bm[j]);
            if (sel < 0 && kf < rf + pc) sel = ((cg + j) << 5) + kth_set_bit(bm[j], kf - rf);
            rf += pc;
          }
          if (lane == fi) {
            run = sel >= 0 ? kf + 1 : rf;              // past k once picked
            if (sel >= 0) sel_q = blk.entry(sel);
          }
        }
      }
    }
    if (act) {
      if (prm.store_debug) w.n_nbrs[p] = cnt;
      w.mate[p] = (cnt > 0 && u_keep < prm.c.b) ? sel_q : -1;
    }
    __syncwarp();
  }
}

// Panmixia (mating_radius = None), species.py:2178-2194: n_mates ~ Binomial(N, b) mating slots
// (one Bernoulli(b) per individual has exactly that sum), each drawing two individuals with
// replacement; selfing pairs are dropped; with sexes, column 0 must be female and column 1
// male (mating.py:41-55).  No de-duplication (mating.py:64-65).  Slot i belongs to the
// individual of species ordinal i; the drawn numbers are ordinals too (mapped to entries
// through w.inv in ordered mode; without injected draws any bijection is as uniform).
__global__ void __launch_bounds__(256) k_panmixia(Pop pop, Params prm, DevDraws dr, Work w, const Counters* c) {
  const int n = c->n, cur = c->cur;
  const int64_t t = c->t;
  const int32_t* __restrict__ inv = prm.ordered ? w.inv : nullptr;
  for (int i = GTID; i < n; i += GSTRIDE) {
    const int p = inv ? inv[i] : i;
    RngStream g(prm.seed_lo, prm.seed_hi, pop.idx[cur][p], SITE_PANMIXIA, t);
    const double u = dr.pan_u ? dr.pan_u[i] : g.uniform();
    const uint32_t R0 = dr.pan_R ? dr.pan_R[2 * i] : g.u32();
    const uint32_t R1 = dr.pan_R ? dr.pan_R[2 * i + 1] : g.u32();
    const bool active = prm.c.b >= 1.0 || u < prm.c.b;
    int a = (int)choose_k(R0, (uint32_t)n), b2 = (int)choose_k(R1, (uint32_t)n);
    bool ok = active && a != b2;
    if (inv) { a = inv[a]; b2 = inv[b2]; }
    if (ok && prm.c.sex) ok = pop.sex[cur][a] == 0 && pop.sex[cur][b2] == 1;
    w.mate[i] = ok ? a : -1;
    w.perm[i] = b2;
    if (prm.store_debug) w.n_nbrs[p] = n - 1;
  }
}

// ========================================================================================
// a6 + a8: sex filter / reciprocal de-dup (mating.py:41-63), stream compaction into the
// pair list, births per pair (species.py:604-609, mating.py:120-126), offspring table, pair
// midpoints (demography.py:60-72).  Pairs hold ENTRY numbers (positions in the current half).
// The list is built in entry (= mating-grid) order; in ordered mode (injected draws) in
// ascending focal ordinal through w.inv -- the oracle's canonical order.
// ========================================================================================
struct PairScan {
  Pop pop;
  Work w;
  const Counters* cc;
  int32_t sexed;
  int32_t fixed_nb;      // > 0: n_births_fixed
  int32_t panmixia;      // pairs are (mate[i], perm[i]) drawn by k_panmixia, already filtered
  int32_t ordered;
  __device__ int size(const Counters* c) const { return c->n; }
  __device__ int entry(int i) const { return (ordered && !panmixia) ? w.inv[i] : i; }
  __device__ bool keep(int i) const {
    if (panmixia) return w.mate[i] >= 0;
    const int p = entry(i);
    if (p < cc->own_lo || p >= cc->own_hi) return false;     // ghosts found their pairs on their own rank
    const int m = w.mate[p];
    if (m < 0) return false;
    if (sexed) {
      const int8_t* sx = pop.sex[cc->cur];
      return sx[p] == 0 && sx[m] == 1;                 // mating.py:41-55
    }
    // mating.py:62-63: a reciprocal couple is kept once, under the focal with the smaller id
    return !(w.mate[m] == p && pop.idx[cc->cur][m] < pop.idx[cc->cur][p]);
  }
  // the reduce pass evaluates the predicate (dependent gathers) once and leaves it in
  // w.alive, which the mortality stage only rewrites later in the step
  __device__ u64 value_first(int i) const {
    const bool k = keep(i);
    w.alive[i] = k ? 1 : 0;
    return k ? ((u64)1 << 32) : 0;
  }
  __device__ u64 value(int i) const { return w.alive[i] ? ((u64)1 << 32) : 0; }
  static constexpr bool BATCHED = true;
  __device__ void apply_batch(const int* idx, const u64* v, const u64* ex, int n) const {
    const int cur = cc->cur;
    bool on[SCAN_ITEMS];
    int a[SCAN_ITEMS], m[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      on[k] = idx[k] < n && v[k] != 0;
      if (on[k]) {
        if (panmixia) { a[k] = w.mate[idx[k]]; m[k] = w.perm[idx[k]]; }
        else { a[k] = entry(idx[k]); m[k] = w.mate[a[k]]; }
      }
    }
    double2 pa[SCAN_ITEMS], pm[SCAN_ITEMS];
    int sa[SCAN_ITEMS], sm[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      if (on[k]) {
        pa[k] = pop.xy[cur][a[k]];
        pm[k] = pop.xy[cur][m[k]];
        sa[k] = pop.gslot[cur][a[k]]; sm[k] = pop.gslot[cur][m[k]];
      }
    }
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      if (!on[k]) continue;
      const int p = (int)(ex[k] >> 32);
      reinterpret_cast<int2*>(w.pairs)[p] = make_int2(a[k], m[k]);
      w.mid[p] = make_double2((pa[k].x + pm[k].x) / 2, (pa[k].y + pm[k].y) / 2);     // species.py:640-641
      // parents' genome slots, so the gamete kernel's index chain is one load shorter
      reinterpret_cast<int2*>(w.pair_slots)[p] = make_int2(sa[k], sm[k]);
      if (fixed_nb > 0) {
        w.nb[p] = fixed_nb;
        w.off_start[p] = p * fixed_nb;
        for (int j = 0; j < fixed_nb; ++j)
          if ((long long)p * fixed_nb + j < pop.cap) w.off_pair[p * fixed_nb + j] = p;
      }
    }
  }
  __device__ void apply(int, u64, u64) const {}
  __device__ void total(Counters* c, u64 tot) const {
    int P = (int)(tot >> 32);
    c->P = P;
    if (fixed_nb > 0) {
      long long B = (long long)P * fixed_nb;
      if (c->n + B > pop.cap) { B = pop.cap - c->n; c->err |= GNX_ERRBIT_CAPACITY; }
      c->B = (int)B;
    }
  }
};

// Poisson births: second scan over the P pairs.  `st` (strip decomposition, else NULL): this rank's
// pairs are the slice of the species-wide pair list that follows the pairs of the lower ranks.
__global__ void __launch_bounds__(256) k_draw_births(Pop pop, Params prm, DevDraws dr, Work w, const Counters* c,
                                                     const Strip* st) {
  const int P = c->P;
  long long pair_base = 0;
  if (st)
    for (int r = 0; r < st->rank; ++r) pair_base += st->pairs[r];
  for (int p = GTID; p < P; p += GSTRIDE) {
    int nbv;
    if (dr.poisson) nbv = dr.poisson[p];
    else {
      // keyed by the pair's position in the canonical pair list (an individual can belong to
      // several pairs under panmixia)
      RngStream g(prm.seed_lo, prm.seed_hi, (int64_t)(pair_base + p), SITE_BIRTHS, c->t);
      nbv = sample_poisson(g, prm.c.n_births_lambda);
    }
    w.nb[p] = max(nbv, 1);                   // mating.py:125
  }
}
struct BirthScan {
  Work w;
  int32_t cap;
  __device__ int size(const Counters* c) const { return c->P; }
  __device__ u64 value(int p) const { return (u64)w.nb[p]; }
  __device__ void apply(int p, u64 v, u64 ex) const {
    w.off_start[p] = (int)ex;
    for (int j = 0; j < (int)v; ++j)
      if ((long long)ex + j < cap) w.off_pair[ex + j] = p;
  }
  __device__ void total(Counters* c, u64 tot) const {
    long long B = (long long)tot;
    if (c->n + B > cap) { B = cap - c->n; c->err |= GNX_ERRBIT_CAPACITY; }
    c->B = (int)B;
  }
};

// ========================================================================================
// a9 + a12 + a11 + a8: gamete formation over bit-packed genotypes (mating.py:130-172),
// newborn phenotype (selection.py:22-48), natal dispersal (movement.py:98-141), newborn
// record (species.py:638-688, individual.py:100-124).
//   A group of GW lanes (power of two <= 32) owns one offspring; lane q streams the q-th
//   128-bit unit of both parents' homologues and of the two cached recombination paths,
//   forms the two gametes with pure bitwise selects, stores the child's row, and
//   accumulates the trait-locus dosages that fall in its unit.
// ========================================================================================
__device__ __forceinline__ uint4 bitsel(uint4 a0, uint4 a1, uint4 m) {
  return make_uint4((a0.x & ~m.x) | (a1.x & m.x), (a0.y & ~m.y) | (a1.y & m.y),
                    (a0.z & ~m.z) | (a1.z & m.z), (a0.w & ~m.w) | (a1.w & m.w));
}
__device__ __forceinline__ uint32_t unit_bit(const uint4& v, int bit) {
  uint32_t wd = (bit >> 5) == 0 ? v.x : (bit >> 5) == 1 ? v.y : (bit >> 5) == 2 ? v.z : v.w;
  return (wd >> (bit & 31)) & 1u;
}
__device__ __forceinline__ uint4 ld_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(uint4* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}

// phenotype contribution of one 128-bit unit pair (h0, h1) of trait t.  The trait table is
// a CSR over 32-bit words (4 per unit), so the word select is compile-time.
__device__ __forceinline__ int trait_n_loci(const Traits& tr, int t) {
  return tr.n_loci_dev ? __ldg(&tr.n_loci_dev[t]) : tr.n_loci[t];
}
__device__ __forceinline__ double trait_word(const Traits& tr, int s, int e, uint32_t w0, uint32_t w1,
                                             bool polygenic) {
  double acc = 0.0;
  if (!tr.te_dom && polygenic) {
    // common case: geno*alpha = dosage * (0.5*alpha) exactly (power-of-two scaling)
    for (int k = s; k < e; ++k) {
      const int sh = __ldg(&tr.te_locus[k]) & 31;
      const int dosage = (int)((w0 >> sh) & 1u) + (int)((w1 >> sh) & 1u);
      acc += (0.5 * (double)dosage) * __ldg(&tr.te_alpha[k]);              // selection.py:30-33, 43-44
    }
    return acc;
  }
  for (int k = s; k < e; ++k) {
    const int sh = __ldg(&tr.te_locus[k]) & 31;
    const int dosage = (int)((w0 >> sh) & 1u) + (int)((w1 >> sh) & 1u);
    double geno = 0.5 * (double)dosage;                                     // selection.py:30-33
    if (tr.te_dom) geno = fmin(geno * __ldg(&tr.te_dom[k]), 1.0);           // selection.py:35-39
    acc += polygenic ? geno * __ldg(&tr.te_alpha[k]) : geno;                // selection.py:43-47
  }
  return acc;
}
__device__ __forceinline__ double trait_partial(const Traits& tr, int t, int q, int Wq, const uint4& h0,
                                                const uint4& h1) {
  const int* ptr = tr.chunk_ptr + t * (4 * Wq + 1) + 4 * q;
  const int p0 = __ldg(ptr), p4 = __ldg(ptr + 4);
  if (p0 == p4) return 0.0;
  const int p1 = __ldg(ptr + 1), p2 = __ldg(ptr + 2), p3 = __ldg(ptr + 3);
  const bool poly = trait_n_loci(tr, t) > 1;
  return trait_word(tr, p0, p1, h0.x, h1.x, poly) + trait_word(tr, p1, p2, h0.y, h1.y, poly) +
         trait_word(tr, p2, p3, h0.z, h1.z, poly) + trait_word(tr, p3, p4, h0.w, h1.w, poly);
}

// ----- k_gametes: the genotype-streaming kernel -----------------------------------------
// GW lanes per offspring (power of two <= 32), NT = trait accumulators kept in registers
// (instantiated for 2 and GNX_MAX_TRAITS).  Lane 0 of a group walks the index chain
// (offspring -> pair -> parents' genome slots) and draws the two recombination keys and
// start homologues once; the group gets them by shuffle.  Every lane then streams its
// 128-bit units: 4 parental homologue loads + 2 path loads in flight, 2 stores.
struct BirthPlan {
  int s0, s1, cslot, kk0, kk1;     // parents' slots, child slot, key | start << 30
};

constexpr int GAM_NB = 2;     // offspring per trait-table walk in the staged path
constexpr int GAM_MINB = 4;   // 64 registers: 4 CTAs per SM measured fastest (3, 5, 6 are slower)
template <int GW, int NT>
__global__ void __launch_bounds__(256, GAM_MINB) k_gametes(Pop pop, Params prm, Traits tr, DevDraws dr, Work w,
                                                  const Counters* c, int fixed_nb, int stage_rows) {
  // stage_rows: the child's row is also kept in shared memory (2*Wq uint4 per group) and the
  // phenotype is accumulated over the trait table with the entries dealt round-robin to the
  // group's lanes -- balanced, where the per-unit walk leaves most lanes idle.
  extern __shared__ uint4 g_rows[];
  const int n = c->n, B = c->B, cur = c->cur, n_free = c->n_free, n_slots = c->n_slots;
  const int64_t t = c->t, max_idx = c->max_idx;
  const int Wq = pop.Wq, T = pop.T;
  const int lane = threadIdx.x & (GW - 1);
  // the staged row interleaves the homologues word by word ([h0 word w, h1 word w] adjacent),
  // so one 64-bit shared load serves both alleles of a locus
  uint32_t* const row32 = reinterpret_cast<uint32_t*>(g_rows + (size_t)(threadIdx.x / GW) * 2 * Wq);
  const bool fast_trait = !tr.te_dom;
  const int wl = threadIdx.x & 31;
  const int lane0 = wl & ~(GW - 1);
  constexpr int G = 32 / GW;              // offspring groups per warp
  const int grp = wl / GW;
  const unsigned gmask = GW == 32 ? 0xffffffffu : (((1u << GW) - 1u) << lane0);
  // A warp takes chunks of 32 consecutive offspring.  Every lane first resolves ONE offspring
  // of the chunk: offspring -> (parents' genome slots, child slot, recombination keys, start
  // homologues), coalesced and with no idle lanes; the GW iterations that stream the rows then
  // fetch their plan by shuffle.  The next chunk's plans are prefetched under the row stream.
  auto load_plan = [&](int o) -> BirthPlan {
    BirthPlan bp = {0, 0, 0, 0, 0};
    if (o < B) {
      const int p = fixed_nb > 0 ? o / fixed_nb : w.off_pair[o];
      const int2 sl = reinterpret_cast<const int2*>(w.pair_slots)[p];
      bp.s0 = sl.x;
      bp.s1 = sl.y;
      bp.cslot = o < n_free ? pop.free_slots[n_free - 1 - o] : n_slots + (o - n_free);
      int k0, k1, h0, h1;
      RngStream gg(prm.seed_lo, prm.seed_hi, max_idx + 1 + o, SITE_GAMETE, t);
      if (dr.recomb_keys) {
        // mating.py:176-181, 204-209: the pair's key slice is popped from its END
        const int j = o - w.off_start[p];
        const int e = 2 * (w.off_start[p] + w.nb[p]);
        k0 = dr.recomb_keys[e - 1 - 2 * j];
        k1 = dr.recomb_keys[e - 2 - 2 * j];
      } else {
        k0 = (int)choose_k(gg.u32(), prm.n_paths);      // species.py:625-627
        k1 = (int)choose_k(gg.u32(), prm.n_paths);
      }
      if (dr.start_homs) {
        h0 = dr.start_homs[2 * o];
        h1 = dr.start_homs[2 * o + 1];
      } else {
        const uint32_t bits = gg.u32();                  // mating.py:133
        h0 = bits & 1;
        h1 = (bits >> 1) & 1;
      }
      bp.kk0 = k0 | (h0 << 30);
      bp.kk1 = k1 | (h1 << 30);
    }
    return bp;
  };
  const int nwarps = GSTRIDE >> 5, nchunks = (B + 31) >> 5;
  int ch = GTID >> 5;
  BirthPlan next = load_plan(ch * 32 + wl);
  for (; ch < nchunks; ch += nwarps) {
    const BirthPlan mine = next;
    next = load_plan((ch + nwarps) * 32 + wl);
    if (ch * 32 + wl < B) pop.gslot[cur][n + ch * 32 + wl] = mine.cslot;
  if (GW > 1 && stage_rows >= 2) {
    // NB offspring per group and pass: their rows are streamed and staged (one buffer each), then
    // ONE walk over the trait table serves all of them -- entry load, address arithmetic and
    // loop control are paid once per NB offspring.
    constexpr int NB = (GAM_NB < GW) ? GAM_NB : GW;
    const int buf_stride = 8 * Wq * (blockDim.x / GW);       // uint32 words between the staging buffers
#pragma unroll 1
    for (int j = 0; j < GW; j += NB) {
      int oo[NB];
      bool vv[NB];
#pragma unroll
      for (int u = 0; u < NB; ++u) {
        const int src = (j + u) * G + grp;
        const int o = ch * 32 + src;
        BirthPlan bp;
        bp.s0 = __shfl_sync(0xffffffffu, mine.s0, src);
        bp.s1 = __shfl_sync(0xffffffffu, mine.s1, src);
        bp.cslot = __shfl_sync(0xffffffffu, mine.cslot, src);
        bp.kk0 = __shfl_sync(0xffffffffu, mine.kk0, src);
        bp.kk1 = __shfl_sync(0xffffffffu, mine.kk1, src);
        oo[u] = o;
        vv[u] = o < B;
        if (!vv[u]) continue;
        const uint4* P0 = pop.G + (size_t)bp.s0 * 2 * Wq;
        const uint4* P1 = pop.G + (size_t)bp.s1 * 2 * Wq;
        const uint4* M0 = prm.paths + (size_t)(bp.kk0 & 0x3fffffff) * Wq;
        const uint4* M1 = prm.paths + (size_t)(bp.kk1 & 0x3fffffff) * Wq;
        uint4* C = pop.G + (size_t)bp.cslot * 2 * Wq;
        const uint32_t f0 = (bp.kk0 >> 30) ? 0xffffffffu : 0u, f1 = (bp.kk1 >> 30) ? 0xffffffffu : 0u;
        uint4* const stg = reinterpret_cast<uint4*>(row32 + u * buf_stride);
        for (int q = lane; q < Wq; q += GW) {
          const uint4 a0 = ld_stream(P0 + q), a1 = ld_stream(P0 + Wq + q);
          const uint4 b0 = ld_stream(P1 + q), b1 = ld_stream(P1 + Wq + q);
          uint4 m0 = __ldg(M0 + q), m1 = __ldg(M1 + q);
          m0 = make_uint4(m0.x ^ f0, m0.y ^ f0, m0.z ^ f0, m0.w ^ f0);
          m1 = make_uint4(m1.x ^ f1, m1.y ^ f1, m1.z ^ f1, m1.w ^ f1);
          const uint4 g0 = bitsel(a0, a1, m0), g1 = bitsel(b0, b1, m1);
          st_stream(C + q, g0);
          st_stream(C + Wq + q, g1);
          stg[2 * q] = make_uint4(g0.x, g1.x, g0.y, g1.y);
          stg[2 * q + 1] = make_uint4(g0.z, g1.z, g0.w, g1.w);
        }
      }
      if (!vv[0]) continue;                  // uniform over the group (the later ones are then invalid too)
      __syncwarp(gmask);
      const int NW = 4 * Wq;
      double zz[NT][NB];
#pragma unroll
      for (int tt = 0; tt < NT; ++tt) {
#pragma unroll
        for (int u = 0; u < NB; ++u) zz[tt][u] = 0.0;
        if (tt < T) {
          const int ks = __ldg(&tr.chunk_ptr[tt * (NW + 1)]), ke = __ldg(&tr.chunk_ptr[tt * (NW + 1) + NW]);
          const int4* __restrict__ tp = reinterpret_cast<const int4*>(tr.te_pack);
          double h0[NB], h1[NB];             // one accumulator per offspring and homologue
#pragma unroll
          for (int u = 0; u < NB; ++u) h0[u] = h1[u] = 0.0;
          for (int k = ks + lane; k < ke; k += GW) {
            const int4 e = __ldg(tp + k);                 // {byte offset of the word pair, bit mask, alpha/2}
            const double ha = __hiloint2double(e.w, e.z);
            const char* base = reinterpret_cast<const char*>(row32) + e.x;
#pragma unroll
            for (int u = 0; u < NB; ++u) {
              const uint2 ww = *reinterpret_cast<const uint2*>(base + 4 * u * buf_stride);
              if (ww.x & (uint32_t)e.y) h0[u] += ha;      // and + predicate in one LOP3, predicated DADD
              if (ww.y & (uint32_t)e.y) h1[u] += ha;
            }
          }
#pragma unroll
          for (int u = 0; u < NB; ++u) zz[tt][u] = h0[u] + h1[u];
        }
      }
      __syncwarp(gmask);      // the rows are rewritten by the next batch of offspring
#pragma unroll
      for (int tt = 0; tt < NT; ++tt) {
        if (tt < T) {
#pragma unroll
          for (int u = 0; u < NB; ++u) {
            double v = zz[tt][u];
#pragma unroll
            for (int d = GW / 2; d >= 1; d >>= 1) v += __shfl_xor_sync(gmask, v, d);
            if (lane == 0 && vv[u]) pop.z[cur][(size_t)tt * pop.cap + n + oo[u]] = 0.5 + v;
          }
        }
      }
    }
    continue;
  }
#pragma unroll 1
  for (int j = 0; j < GW; ++j) {
    const int src = j * G + grp;
    const int o = ch * 32 + src;
    BirthPlan bp;
    bp.s0 = __shfl_sync(0xffffffffu, mine.s0, src);
    bp.s1 = __shfl_sync(0xffffffffu, mine.s1, src);
    bp.cslot = __shfl_sync(0xffffffffu, mine.cslot, src);
    bp.kk0 = __shfl_sync(0xffffffffu, mine.kk0, src);
    bp.kk1 = __shfl_sync(0xffffffffu, mine.kk1, src);
    if (o >= B) continue;                    // uniform over the group
    const uint4* P0 = pop.G + (size_t)bp.s0 * 2 * Wq;
    const uint4* P1 = pop.G + (size_t)bp.s1 * 2 * Wq;
    const uint4* M0 = prm.paths + (size_t)(bp.kk0 & 0x3fffffff) * Wq;
    const uint4* M1 = prm.paths + (size_t)(bp.kk1 & 0x3fffffff) * Wq;
    uint4* C = pop.G + (size_t)bp.cslot * 2 * Wq;
    const uint32_t f0 = (bp.kk0 >> 30) ? 0xffffffffu : 0u, f1 = (bp.kk1 >> 30) ? 0xffffffffu : 0u;
    double zacc[NT];
#pragma unroll
    for (int tt = 0; tt < NT; ++tt) zacc[tt] = 0.0;
    for (int q = lane; q < Wq; q += GW) {
      const uint4 a0 = ld_stream(P0 + q), a1 = ld_stream(P0 + Wq + q);
      const uint4 b0 = ld_stream(P1 + q), b1 = ld_stream(P1 + Wq + q);
      uint4 m0 = __ldg(M0 + q), m1 = __ldg(M1 + q);
      m0 = make_uint4(m0.x ^ f0, m0.y ^ f0, m0.z ^ f0, m0.w ^ f0);
      m1 = make_uint4(m1.x ^ f1, m1.y ^ f1, m1.z ^ f1, m1.w ^ f1);
      // gamete_c[l] = g_parent_c[l, path[l] XOR start_c]  (mating.py:161-168)
      const uint4 g0 = bitsel(a0, a1, m0), g1 = bitsel(b0, b1, m1);
      st_stream(C + q, g0);
      st_stream(C + Wq + q, g1);
      if (stage_rows) {
        reinterpret_cast<uint4*>(row32)[2 * q] = make_uint4(g0.x, g1.x, g0.y, g1.y);
        reinterpret_cast<uint4*>(row32)[2 * q + 1] = make_uint4(g0.z, g1.z, g0.w, g1.w);
      } else {
#pragma unroll
        for (int tt = 0; tt < NT; ++tt)
          if (tt < T) zacc[tt] += trait_partial(tr, tt, q, Wq, g0, g1);
      }
    }
    if (stage_rows) {
      __syncwarp(gmask);
      const int NW = 4 * Wq;
#pragma unroll
      for (int tt = 0; tt < NT; ++tt) {
        if (tt < T) {
          const int ks = __ldg(&tr.chunk_ptr[tt * (NW + 1)]), ke = __ldg(&tr.chunk_ptr[tt * (NW + 1) + NW]);
          const bool poly = trait_n_loci(tr, tt) > 1;
          double acc = 0.0;
          if (fast_trait && poly) {
            // geno * alpha = (b0 + b1) * (alpha / 2), exact (selection.py:30-33, 43-44)
            const int4* __restrict__ tp = reinterpret_cast<const int4*>(tr.te_pack);
            double acc1 = 0.0;                              // one accumulator per homologue
            for (int k = ks + lane; k < ke; k += GW) {
              const int4 e = __ldg(tp + k);                 // {byte offset of the word pair, bit mask, alpha/2}
              const uint2 ww = *reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(row32) + e.x);
              const double ha = __hiloint2double(e.w, e.z);
              if (ww.x & (uint32_t)e.y) acc += ha;          // and + predicate in one LOP3, predicated DADD
              if (ww.y & (uint32_t)e.y) acc1 += ha;
            }
            acc += acc1;
          } else {
            for (int k = ks + lane; k < ke; k += GW) {
              const int loc = __ldg(&tr.te_locus[k]);
              const int wi = 2 * (loc >> 5), sh = loc & 31;
              const int dosage = (int)((row32[wi] >> sh) & 1u) + (int)((row32[wi + 1] >> sh) & 1u);
              double geno = 0.5 * (double)dosage;                                 // selection.py:30-33
              if (!fast_trait) geno = fmin(geno * __ldg(&tr.te_dom[k]), 1.0);     // selection.py:35-39
              acc += poly ? geno * __ldg(&tr.te_alpha[k]) : geno;                 // selection.py:43-47
            }
          }
          zacc[tt] = acc;
        }
      }
      __syncwarp(gmask);      // the row is rewritten by the next offspring
    }
#pragma unroll
    for (int tt = 0; tt < NT; ++tt) {
      if (tt < T) {
        double v = zacc[tt];
#pragma unroll
        for (int d = GW / 2; d >= 1; d >>= 1) v += __shfl_xor_sync(gmask, v, d);
        if (lane == 0) pop.z[cur][(size_t)tt * pop.cap + n + o] = (trait_n_loci(tr, tt) > 1) ? 0.5 + v : v;
      }
    }
  }
  }
}

// ----- k_newborns: natal dispersal, sex, newborn record (one thread per offspring) -------
constexpr int NB_MINB = 4;   // 64 registers instead of 77: 83 -> 68 us at c4
__global__ void __launch_bounds__(256, NB_MINB) k_newborns(Pop pop, Land land, Params prm, DevDraws dr, Work w,
                                                   Counters* c, Tsk tsk) {
  const int n = c->n, B = c->B, cur = c->cur;
  const int n_nodes = c->n_nodes, n_born = c->n_born;
  const int64_t t = c->t, max_idx = c->max_idx;
  for (int o = GTID; o < B; o += GSTRIDE) {
    const int p = w.off_pair[o];
    const int64_t oid = max_idx + 1 + o;
    const int dst = n + o;
    // ---- natal dispersal (movement.py:98-141)
    const double2 mid = w.mid[p];
    const double mx = mid.x, my = mid.y;
    RngStream g(prm.seed_lo, prm.seed_hi, oid, SITE_DISP, t);
    double ox = 0.0, oy = 0.0;
    int tries = 0;
    const bool injected = dr.disp_dist || dr.disp_dir || dr.disp_choice;
    const int max_tries = injected ? dr.disp_R : 1000;
    bool ok = false;
    while (!ok && tries < max_tries) {
      double cs, sn;
      if (prm.c.disp_surf_mode == GNX_SURF_TABLE) {
        int col = dr.disp_choice ? dr.disp_choice[(size_t)o * dr.disp_R + tries]
                                 : (int)choose_k(g.u32(), prm.c.surf_approx_len);
        __half h = prm.disp_tab[((size_t)((int)my) * land.X + (int)mx) * prm.c.surf_approx_len + col];
        sincos_half_tab(prm.cs_tab, h, &sn, &cs);
      } else if (prm.c.disp_surf_mode == GNX_SURF_ONTHEFLY) {
        const __half d = surface_direction_onthefly(
            g, land.surf_f32[1], land.X, land.Y, (int)mx,
            (int)my, prm.c.disp_surf_mixture, (float)prm.c.disp_surf_kappa, prm.vm_tab[1]);
        sincos_half_tab(prm.cs_tab, d, &sn, &cs);
      } else if (dr.disp_dir) {
        sincos(dr.disp_dir[(size_t)o * dr.disp_R + tries], &sn, &cs);
      } else {
        // NB reference passes mu=0, kappa=0 whatever the species' params (species.py:650-653):
        // vonmises(0, 0) = pi*(2U - 1)
        float sf, cf;
        sincospif(2.0f * uniform_f32(g) - 1.0f, &sf, &cf);
        sn = (double)sf;
        cs = (double)cf;
      }
      double dist = dr.disp_dist ? dr.disp_dist[(size_t)o * dr.disp_R + tries]
                                 : sample_distance_f32(g, prm.c.disp_distr, prm.c.disp_p1, prm.c.disp_p2);
      double dx = __dmul_rn(cs, dist), dy = __dmul_rn(sn, dist);
      if (prm.c.res_ratio_x != 1.0) dx = __dmul_rn(dx, prm.c.res_ratio_x);
      if (prm.c.res_ratio_y != 1.0) dy = __dmul_rn(dy, prm.c.res_ratio_y);
      ox = clampd(__dadd_rn(mx, dx), 0.0, land.max_x);
      oy = clampd(__dadd_rn(my, dy), 0.0, land.max_y);
      ok = (ox > 0.0 && ox < (double)land.X) && (oy > 0.0 && oy < (double)land.Y);
      tries += 1;
    }
    if (!ok) { tries = max_tries + 1; atomicOr((int*)&c->err, GNX_ERRBIT_DRAWS); }
    if (prm.store_debug) w.disp_tries[o] = tries;
    // ---- sex (species.py:657-662 + the re-draw quirk of individual.py:110-115)
    int first = 0;
    if (prm.c.sex) {
      double u = dr.sex_u ? dr.sex_u[o] : g.uniform();
      first = u < prm.c.sex_ratio_p;
    }
    int sex = 1;
    if (!first) {
      double u = dr.sex_redraw_u ? dr.sex_redraw_u[o] : g.uniform();
      sex = u < 0.5;
    }
    pop.xy[cur][dst] = make_double2(ox, oy);
    pop.age[cur][dst] = 0;
    pop.sex[cur][dst] = (int8_t)sex;
    pop.idx[cur][dst] = oid;
    if (prm.burn) pop.gslot[cur][dst] = -1;
    if (prm.ordered) pop.ord[cur][dst] = dst;       // newborns follow everyone in species order (ids ascend)
    if (tsk.enabled) {
      // species.py:692-736: one individuals row (location = [x, y, z...], metadata = idx) and
      // two nodes rows (flags=1, time=-t, population=0) per offspring, in offspring order
      pop.node[0][cur][dst] = n_nodes + 2 * o;
      pop.node[1][cur][dst] = n_nodes + 2 * o + 1;
      const int k = n_born + o;
      if (k < tsk.born_cap) {
        tsk.b_idx[k] = oid;
        tsk.b_x[k] = ox;
        tsk.b_y[k] = oy;
        tsk.b_time[k] = -(double)(t - c->tsk_t0);
        for (int tt = 0; tt < pop.T; ++tt)
          tsk.b_z[(size_t)tt * tsk.born_cap + k] = pop.z[cur][(size_t)tt * pop.cap + dst];
      } else {
        atomicOr((int*)&c->err, GNX_ERRBIT_CAPACITY);
      }
    }
  }
}

// edges of every offspring (species.py:723-729 + Recombinations._get_seg_info
// genome.py:257-281): for homologue h inherited from parent pair[h] through cached path k_h
// started on homologue s_h, segment i spans [bp[i-1]-0.5, bp[i]-0.5) (0 and L at the ends)
// and descends from the parent's node (i + s_h) % 2.
struct TskitScan {
  Pop pop;
  Params prm;
  DevDraws dr;
  Work w;
  Tsk tsk;
  const Counters* cc;
  int32_t fixed_nb;
  __device__ int size(const Counters* c) const { return c->B; }
  __device__ void keys(int o, int* p, int* k0, int* k1, int* h0, int* h1) const {
    // must mirror k_gametes' plan exactly (same keys and start homologues)
    *p = fixed_nb > 0 ? o / fixed_nb : w.off_pair[o];
    RngStream gg(prm.seed_lo, prm.seed_hi, cc->max_idx + 1 + o, SITE_GAMETE, cc->t);
    if (dr.recomb_keys) {
      const int j = o - w.off_start[*p];
      const int e = 2 * (w.off_start[*p] + w.nb[*p]);
      *k0 = dr.recomb_keys[e - 1 - 2 * j];
      *k1 = dr.recomb_keys[e - 2 - 2 * j];
    } else {
      *k0 = (int)choose_k(gg.u32(), prm.n_paths);
      *k1 = (int)choose_k(gg.u32(), prm.n_paths);
    }
    if (dr.start_homs) {
      *h0 = dr.start_homs[2 * o];
      *h1 = dr.start_homs[2 * o + 1];
    } else {
      const uint32_t bits = gg.u32();
      *h0 = bits & 1;
      *h1 = (bits >> 1) & 1;
    }
  }
  __device__ u64 value(int o) const {
    int p, k0, k1, h0, h1;
    keys(o, &p, &k0, &k1, &h0, &h1);
    return (u64)((tsk.bp_ptr[k0 + 1] - tsk.bp_ptr[k0] + 1) + (tsk.bp_ptr[k1 + 1] - tsk.bp_ptr[k1] + 1));
  }
  __device__ void apply(int o, u64, u64 ex) const {
    int p, k[2], h[2];
    keys(o, &p, &k[0], &k[1], &h[0], &h[1]);
    const int cur = cc->cur;
    long long e = (long long)cc->n_edges + (long long)ex;
    for (int hom = 0; hom < 2; ++hom) {
      const int par = w.pairs[2 * p + hom];
      const int pn[2] = {pop.node[0][cur][par], pop.node[1][cur][par]};
      const int child = cc->n_nodes + 2 * o + hom;
      const int s = tsk.bp_ptr[k[hom]], nbp = tsk.bp_ptr[k[hom] + 1] - s;
      for (int i = 0; i <= nbp; ++i, ++e) {
        if (e >= tsk.edge_cap) continue;
        tsk.e_left[e] = i == 0 ? 0.0 : (double)tsk.bp_pos[s + i - 1] - 0.5;
        tsk.e_right[e] = i == nbp ? tsk.L : (double)tsk.bp_pos[s + i] - 0.5;
        tsk.e_parent[e] = pn[(i + h[hom]) & 1];
        tsk.e_child[e] = child;
      }
    }
  }
  __device__ void total(Counters* c, u64 tot) const {
    // stash the step's edge count; k_after_births folds it into n_edges once apply has run
    c->pad[1] = (int)tot;
    if ((long long)c->n_edges + (long long)tot > tsk.edge_cap) c->err |= GNX_ERRBIT_CAPACITY;
  }
};

// ---- growth guard (gnx_set_growth_guard) --------------------------------------------------
// What one step may need, judged from the counters at step start.  Every focal makes at most one
// pair (mating.py:62-63), so P <= n: fixed births give at most lambda * n newborns; Poisson births
// sum to Poisson(lambda * P), bounded by ceil(lambda n + 10 sqrt(lambda n)) + 32 (tail below 1e-15,
// DESIGN.md section 8).  n counts the dead the previous step only flagged, so it is an upper bound.
struct GrowthBound {
  double lambda;
  int32_t fixed;            // n_births_fixed: lambda is the integer litter size
  int32_t genomes;          // genome slots are taken (not in burn-in, which returns none)
  int32_t tsk;              // tskit rows are written
  int32_t edges_per_birth;  // 2 * (largest breakpoint count of a cached path + 1)
  int64_t cap, born_cap, edge_cap;
};

__host__ __device__ inline int64_t growth_max_births(double lambda, int fixed, int64_t n) {
  if (fixed) return (int64_t)(int32_t)lambda * n;
  const double m = lambda * (double)n;
  return (int64_t)ceil(m + 10.0 * sqrt(m)) + 32;
}

// fills the capacities the step needs; 1: they all fit, the step may run
__host__ __device__ inline int growth_check(const GrowthBound& g, int64_t n, int64_t n_slots, int64_t n_free,
                                            int64_t n_born, int64_t n_edges, gnx_step_status_t* need) {
  const int64_t B = growth_max_births(g.lambda, g.fixed, n);
  need->need_entries = n + B;
  need->need_slots = g.genomes ? n_slots + (B > n_free ? B - n_free : 0) : 0;   // newborns take free slots first
  need->need_births = g.tsk ? n_born + B : 0;
  need->need_edges = g.tsk ? n_edges + B * g.edges_per_birth : 0;
  return need->need_entries <= g.cap && need->need_slots <= g.cap && need->need_births <= g.born_cap &&
         need->need_edges <= g.edge_cap;
}

// gnx_set_clock: the step counter and the tskit time origin of a run resumed from a checkpoint
__global__ void k_set_clock(Counters* c, int64_t t, int64_t tsk_t0) {
  c->t = t;
  c->tsk_t0 = tsk_t0;
}

// first node of a guarded step graph: runs the step body (IF conditional) only when it cannot overflow
__global__ void k_step_guard(const Counters* c, GrowthBound g, gnx_step_status_t* st, cudaGraphConditionalHandle h) {
  gnx_step_status_t need;
  const int ok = growth_check(g, c->n, c->n_slots, c->n_free, c->n_born, c->n_edges, &need);
  st->steps_run += ok;
  st->stopped = !ok;
  st->need_entries = need.need_entries;
  st->need_slots = need.need_slots;
  st->need_births = need.need_births;
  st->need_edges = need.need_edges;
  cudaGraphSetConditional(h, ok);
}

__global__ void k_after_births(Counters* c, int tsk_enabled) {
  const int B = c->B;
  if (tsk_enabled) {
    c->n_nodes += 2 * B;
    c->n_ind_rows += B;
    c->n_born += B;
    c->n_edges += c->pad[1];
    c->pad[1] = 0;
  }
  c->n_pre = c->n + B;
  const int nf = c->n_free;
  if (B <= nf) c->n_free = nf - B;
  else { c->n_free = 0; c->n_slots += B - nf; }
}

// phenotype of every live individual from its stored genome (Species._set_z species.py:925;
// used after upload / genome assignment)
__global__ void __launch_bounds__(256) k_phenotype_all(Pop pop, Traits tr, const Counters* c) {
  const int n = c->n, cur = c->cur, Wq = pop.Wq, T = pop.T;
  for (int i = GTID; i < n; i += GSTRIDE) {
    const uint4* Gi = pop.G + (size_t)pop.gslot[cur][i] * 2 * Wq;
    for (int tt = 0; tt < T; ++tt) {
      double acc = 0.0;
      for (int q = 0; q < Wq; ++q) {
        const int s = tr.chunk_ptr[tt * (4 * Wq + 1) + 4 * q], e = tr.chunk_ptr[tt * (4 * Wq + 1) + 4 * q + 4];
        if (s == e) continue;
        uint4 h0 = Gi[q], h1 = Gi[Wq + q];
        acc += trait_partial(tr, tt, q, Wq, h0, h1);
      }
      pop.z[cur][(size_t)tt * pop.cap + i] = (trait_n_loci(tr, tt) > 1) ? 0.5 + acc : acc;
    }
  }
}

// ========================================================================================
// a13: mutation of this step's offspring (ops/mutation.py:169-206).
//   One thread does the bookkeeping: the number of mutations in a run is bounded by the mutable
//   loci (infinite sites, genome.py:1101-1104), and every event edits small sorted tables in order.
//   neutral (mutation.py:62-86): consumes a locus, genotypes untouched.
//   deleterious (mutation.py:90-131, 156-166; genome.py:753-788): locus joins nonneut_loci at
//   idx and (delet_loci, delet_s).
//   trait (mutation.py:135-144; genome.py:666-687, 416-437): locus joins nonneut_loci and the
//   trait's (loci, alpha, loci_idxs); tskit layout only (the reference raises otherwise).
//   use_tskit = False: the offspring's genotype ROW idx of the drawn homologue is set to 1
//   (mutation.py:117 as written).  tskit layout: the reference inserts a zero row at idx into every
//   individual and sets g[idx, homologue]; here rows are bits by locus, so bit `locus` is set, the
//   index arrays are kept as the reference leaves them (loci_idxs shifted only inside the mutated
//   trait, delet_loci_idxs never) and the trait tables are rebuilt to read bit
//   nonneut[idxs[k]].  The whole CTA then patches bit `locus` of every cached path to the
//   homologue the path is on in FRONT of the locus (genome.py:133-160: bisect_left of the
//   breakpoints), which is bit locus - 1 of the path as simulated.  Column layout: the locus takes
//   the next free column, and that column stands for bit `locus` in all of the above.
// ========================================================================================
__device__ inline int lower_bound_i32(const int32_t* a, int n, int v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < v) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// the trait tables of `Traits` from the per-trait (loci, alpha, idxs) arrays: entries of a trait
// sorted by the bit they read, CSR over 32-bit words (same layout as gnx_set_traits builds)
__device__ inline void mut_rebuild_tables(const Mut& mu, Counters* c) {
  const int nn = mu.counts[1];
  int base = 0;
  for (int t = 0; t < mu.T; ++t) {
    const int n = mu.counts[4 + t];
    const int32_t* tl = mu.t_loci + (size_t)t * mu.tcap;
    const double* ta = mu.t_alpha + (size_t)t * mu.tcap;
    const int32_t* ti = mu.t_idxs + (size_t)t * mu.tcap;
    for (int k = 0; k < n; ++k) {
      int eff = tl[k];
      if (mu.tskit_layout) {
        int r = ti[k];
        if (r < 0 || r >= nn) { c->err |= GNX_ERRBIT_MUTIDX; r = r < 0 ? 0 : nn - 1; }   // IndexError in the reference
        eff = mu.nonneut[r];
        if (mu.col_of_locus) eff = mu.col_of_locus[eff];
      }
      const double al = ta[k];
      const double dm = mu.dom1p ? mu.dom1p[tl[k]] : 1.0;      // selection.py:37: dom[trait.loci]
      int j = base + k;                                         // stable insertion by the bit read
      while (j > base && mu.te_locus[j - 1] > eff) {
        mu.te_locus[j] = mu.te_locus[j - 1];
        mu.te_alpha[j] = mu.te_alpha[j - 1];
        if (mu.te_dom) mu.te_dom[j] = mu.te_dom[j - 1];
        --j;
      }
      mu.te_locus[j] = eff;
      mu.te_alpha[j] = al;
      if (mu.te_dom) mu.te_dom[j] = dm;
    }
    int32_t* cp = mu.chunk_ptr + (size_t)t * (mu.NW + 1);
    int q = 0;
    cp[0] = base;
    for (int k = 0; k < n; ++k) {
      const int eff = mu.te_locus[base + k];
      while (q < (eff >> 5)) cp[++q] = base + k;
      const double ha = 0.5 * mu.te_alpha[base + k];
      mu.te_pack[base + k] = make_int4((eff >> 5) * 8, (int)(1u << (eff & 31)), __double2loint(ha), __double2hiint(ha));
    }
    while (q < mu.NW) cp[++q] = base + n;
    base += n;
  }
  // the bit every deleterious entry reads
  const int nd = mu.counts[2];
  for (int k = 0; k < nd; ++k) {
    int eff = mu.delet_loci[k];
    if (mu.tskit_layout) {
      int r = mu.delet_idxs[k];
      if (r < 0 || r >= nn) { c->err |= GNX_ERRBIT_MUTIDX; r = r < 0 ? 0 : nn - 1; }
      eff = mu.nonneut[r];
      if (mu.col_of_locus) eff = mu.col_of_locus[eff];
    }
    mu.delet_eff[k] = eff;
  }
}

__global__ void k_mut_rebuild(Mut mu, Counters* c) {
  if (threadIdx.x == 0 && blockIdx.x == 0) mut_rebuild_tables(mu, c);
}

// Widening of the column layout (gnx_widen_cols): every row of wo 128-bit units becomes a row of
// wn > wo units, the new columns zero (genotype rows of every slot, compact recombination paths).
__global__ void __launch_bounds__(256) k_widen_rows(const uint4* __restrict__ src, uint4* __restrict__ dst,
                                                    long long n_rows, int wo, int wn) {
  const long long total = n_rows * wn;
  for (long long k = GTID; k < total; k += GSTRIDE) {
    const long long r = k / wn;
    const int q = (int)(k - r * wn);
    dst[k] = q < wo ? src[r * wo + q] : make_uint4(0u, 0u, 0u, 0u);
  }
}
// ... and the trait CSR over 32-bit words: no entry reads a new word, so the new word ranges are empty
__global__ void k_widen_csr(const int32_t* __restrict__ src, int32_t* __restrict__ dst, int n_tables, int nwo, int nwn) {
  for (int k = GTID; k < n_tables * (nwn + 1); k += GSTRIDE) {
    const int t = k / (nwn + 1), q = k - t * (nwn + 1);
    dst[k] = src[t * (nwo + 1) + min(q, nwo)];
  }
}

// STRIP: one strip of a decomposed landscape (by-locus layout only: no tskit layout, trait mutation or
// tskit rows).  Every rank replays the species-wide sequence -- the births of all ranks, keyed by the
// species-wide max_ind_idx (k_strip_id_base left both in Counters) -- and so keeps identical tables and
// logs; only the rank that holds offspring o (offspring are rank-major) edits its row and z.
template <bool STRIP>
__global__ void __launch_bounds__(256) k_mutate(Pop pop, Params prm, Traits tr, DevDraws dr, Mut mu, Counters* c, int tsk_on) {
  __shared__ int new_loci[GNX_MUT_MAX_NEW];
  __shared__ int new_bits[GNX_MUT_MAX_NEW];    // the genotype bit of each: the locus, or its column
  __shared__ int n_new;
  if (blockIdx.x != 0) return;
  if (threadIdx.x == 0) {
    n_new = 0;
    // B: births of the species; under strips this rank's newborns are offspring [births_lo, births_lo + c->B)
    const int B = STRIP ? c->births_all : c->B, n = c->n, cur = c->cur, Wq = pop.Wq;
    RngStream g(prm.seed_lo, prm.seed_hi, (STRIP ? c->max_idx_base : c->max_idx) + 1, SITE_MUTATE, c->t);
    const long long n_muts = B == 0 ? 0 : (dr.mut_n ? (long long)dr.mut_n[0]
                                      : sample_binomial_wait(g, (long long)B * mu.L, mu.mu_tot));   // mutation.py:172-173
    for (long long m = 0; m < n_muts; ++m) {
      if (dr.mut_n && m >= dr.n_mut) { c->err |= GNX_ERRBIT_DRAWS; break; }
      // genome.py:650-663: choice(types, p) = searchsorted(cdf, u, side='right')
      const double ut = dr.mut_type_u ? dr.mut_type_u[m] : g.uniform();
      int type = 0;
      while (type < mu.n_types - 1 && ut >= mu.cdf[type]) ++type;
      if (mu.counts[0] == 0) { c->err |= GNX_ERRBIT_MUTABLES; break; }    // list.pop() on an empty list
      if (type >= 1 && mu.tskit_layout && n_new >= GNX_MUT_MAX_NEW) { c->err |= GNX_ERRBIT_CAPACITY; break; }
      // column layout: a non-neutral mutation needs a free column; the host widens the rows between steps
      if (type >= 1 && mu.col_of_locus && *mu.col_n >= mu.col_cap) { c->err |= GNX_ERRBIT_CAPACITY; break; }
      const double s_raw = type == 1 ? (dr.mut_s ? dr.mut_s[m] : sample_gamma(g, mu.s_shape, mu.s_scale)) : 0.0;
      const double sel = fmin(s_raw, 1.0);                                  // genome.py:692
      const int locus = mu.mutables[--mu.counts[0]];                        // mutation.py:73 / :95
      const uint32_t R = dr.mut_ind_R ? dr.mut_ind_R[m] : g.u32();
      // r.choice(offspring): the list holds the new ids in DESCENDING order (species.py:615-622)
      const int o = B - 1 - (int)choose_k(R, (uint32_t)B);
      const int i = STRIP ? n + (o - c->births_lo) : n + o;
      int row = -1;
      double alpha = 0.0;
      if (type >= 1) {
        // genome.py:753-788 _add_nonneut_locus
        int nn = mu.counts[1];
        const int idx = lower_bound_i32(mu.nonneut, nn, locus);
        for (int k = nn; k > idx; --k) mu.nonneut[k] = mu.nonneut[k - 1];
        mu.nonneut[idx] = locus;
        mu.counts[1] = nn + 1;
        if (mu.col_of_locus) {                                              // the next free column
          const int cn = *mu.col_n;
          mu.col_locus[cn] = locus;
          mu.col_of_locus[locus] = cn;
          *mu.col_n = cn + 1;
        }
        if (type == 1) {
          int nd = mu.counts[2];
          const int di = lower_bound_i32(mu.delet_loci, nd, locus);
          for (int k = nd; k > di; --k) {
            mu.delet_loci[k] = mu.delet_loci[k - 1];
            mu.delet_s[k] = mu.delet_s[k - 1];
            if (mu.delet_idxs) mu.delet_idxs[k] = mu.delet_idxs[k - 1];
          }
          mu.delet_loci[di] = locus;
          mu.delet_s[di] = sel;
          if (mu.delet_idxs) mu.delet_idxs[di] = idx;                       // genome.py:779-782: nothing is shifted
          mu.counts[2] = nd + 1;
        } else {
          const int t = type - 2;
          // genome.py:666-687 _draw_trait_alpha(n = 1)
          if (mu.a_sigma[t] == 0.0) {
            alpha = mu.a_mu[t];
          } else {
            alpha = dr.mut_alpha ? dr.mut_alpha[m] : mu.a_mu[t] + mu.a_sigma[t] * g.normal();
            if (mu.a_max[t] >= 0.0) alpha = fmin(fmax(alpha, -mu.a_max[t]), mu.a_max[t]);
          }
          int nt = mu.counts[4 + t];
          if (nt == 1) alpha = fabs(alpha);
          // genome.py:416-437 Trait._add_locus
          int32_t* tl = mu.t_loci + (size_t)t * mu.tcap;
          double* ta = mu.t_alpha + (size_t)t * mu.tcap;
          int32_t* ti = mu.t_idxs + (size_t)t * mu.tcap;
          const int ip = lower_bound_i32(tl, nt, locus);
          for (int k = nt; k > ip; --k) { tl[k] = tl[k - 1]; ta[k] = ta[k - 1]; ti[k] = ti[k - 1] + 1; }
          tl[ip] = locus;
          ta[ip] = alpha;
          ti[ip] = idx;
          mu.counts[4 + t] = nt + 1;
        }
      }
      const double uh = dr.mut_homol_u ? dr.mut_homol_u[m] : g.uniform();
      const int homol = uh < 0.5 ? 1 : 0;                                   // r.binomial(1, 0.5)
      if (type >= 1) {
        if (mu.own_tables) mut_rebuild_tables(mu, c);
        else                                   // use_tskit = False: every entry reads the row of its locus
          for (int k = 0; k < mu.counts[2]; ++k) mu.delet_eff[k] = mu.delet_loci[k];
        // mutation.py:117: spp[individ].g[idx, homol] = 1
        row = lower_bound_i32(mu.nonneut, mu.counts[1], locus);
        const int bit = !mu.tskit_layout ? row : mu.col_of_locus ? mu.col_of_locus[locus] : locus;
        if (!STRIP || (unsigned)(o - c->births_lo) < (unsigned)c->B) {      // this rank holds offspring o
          uint32_t* hw = reinterpret_cast<uint32_t*>(pop.G + ((size_t)pop.gslot[cur][i] * 2 + homol) * Wq);
          hw[bit >> 5] |= 1u << (bit & 31);
          // species.py:929 _set_z_individ
          const uint4* Gi = pop.G + (size_t)pop.gslot[cur][i] * 2 * Wq;
          for (int tt = 0; tt < pop.T; ++tt) {
            double acc = 0.0;
            const int nl = mu.own_tables ? mu.counts[4 + tt] : tr.n_loci[tt];
            for (int q = 0; q < Wq; ++q) {
              const int* ptr = tr.chunk_ptr + tt * (4 * Wq + 1) + 4 * q;
              if (ptr[0] == ptr[4]) continue;
              const uint4 h0 = Gi[q], h1 = Gi[Wq + q];
              const uint32_t w0[4] = {h0.x, h0.y, h0.z, h0.w}, w1[4] = {h1.x, h1.y, h1.z, h1.w};
              for (int ww = 0; ww < 4; ++ww)
                for (int k = ptr[ww]; k < ptr[ww + 1]; ++k) {                 // plain loads: the tables were just rewritten
                  const int sh = tr.te_locus[k] & 31;
                  double geno = 0.5 * (double)((int)((w0[ww] >> sh) & 1u) + (int)((w1[ww] >> sh) & 1u));
                  if (tr.te_dom) geno = fmin(geno * tr.te_dom[k], 1.0);
                  acc += nl > 1 ? geno * tr.te_alpha[k] : geno;
                }
            }
            pop.z[cur][(size_t)tt * pop.cap + i] = nl > 1 ? 0.5 + acc : acc;
          }
        }
        if (mu.tskit_layout) {
          new_loci[n_new] = locus;
          new_bits[n_new++] = bit;
        }
      }
      const int nl = mu.counts[3];
      if (nl < mu.log_cap) {
        gnx_mutation_row_t r;
        r.t = c->t;
        r.individual = (STRIP ? c->max_idx_base : c->max_idx) + 1 + o;
        r.locus = locus;
        r.row = row;
        r.homologue = homol;
        r.type = type;
        r.s = sel;
        r.alpha = alpha;
        r.node = tsk_on ? pop.node[homol][cur][i] : -1;                     // mutation.py:46
        r.reserved = 0;
        mu.log[nl] = r;
        mu.counts[3] = nl + 1;
      } else {
        c->err |= GNX_ERRBIT_MUTLOG;
      }
    }
  }
  __syncthreads();
  // genome.py:133-160 _update_subsetters: the inserted homologue is the one the path is on in front of the locus
  if (mu.tskit_layout && n_new > 0) {
    for (int pth = threadIdx.x; pth < mu.n_paths; pth += blockDim.x) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(mu.paths_orig + (size_t)pth * mu.WqL);
      uint32_t* dst = reinterpret_cast<uint32_t*>(mu.paths + (size_t)pth * mu.Wq);
      for (int k = 0; k < n_new; ++k) {
        const int l = new_loci[k], j = new_bits[k];
        const uint32_t b = l > 0 ? (src[(l - 1) >> 5] >> ((l - 1) & 31)) & 1u : 0u;
        dst[j >> 5] = (dst[j >> 5] & ~(1u << (j & 31))) | (b << (j & 31));
      }
    }
  }
}

// ========================================================================================
// a10 (counts): _DensityGrid._calc_density spatial.py:73-97.  Four offset coarse grids;
// cell = (x - edge*ww/2) // ww + edge.  Per-CTA shared-memory histograms, merged with
// global atomics.
// ========================================================================================
#define DENS_SMEM_BINS 4096
__global__ void __launch_bounds__(512) k_density_counts(Pop pop, Work w, const Counters* c, Dens d, const Strip* st) {
  // blockIdx.y = 0: all individuals alive before mortality; 1: pair midpoints
  const int which = blockIdx.y;
  const double2* __restrict__ pts = which == 0 ? pop.xy[c->cur] : w.mid;
  __shared__ int hist[DENS_SMEM_BINS];
  const bool use_smem = d.npts <= DENS_SMEM_BINS;
  if (use_smem)
    for (int k = threadIdx.x; k < d.npts; k += blockDim.x) hist[k] = 0;
  __syncthreads();
  const int n = which == 0 ? c->n + c->B : c->P;      // = n_pre once the birth bookkeeping has run
  int* gcounts = d.counts + (size_t)which * d.npts;
  const int n0 = c->n, own_lo = c->own_lo, own_hi = c->own_hi;
  for (int i = GTID; i < n; i += GSTRIDE) {       // GTID / GSTRIDE use the x dimension only
    if (st && which == 0) {
      // strip decomposition: ghosts are counted by their owner, shipped newborns by their new owner
      if (i < n0 ? (i < own_lo || i >= own_hi) : (st->sent[i] != 0)) continue;
    }
    const double2 pt = pts[i];
    const double x = pt.x, y = pt.y;
    // Half-window index once per axis: with h = x // (ww/2), x // ww = h >> 1 and
    // (x - ww/2) // ww + 1 = (h + 1) >> 1.  Exact whenever x - ww/2 is exact in binary64, which
    // holds for half-windows that are multiples of 2^-20 (the default window width is an
    // integer: spatial.py:286-289); otherwise the four floor divisions are done as written.
    int hx = 0, hy = 0;
    if (d.half_index_ok) {
      hx = (int)floordiv_exact(x, d.hww);
      hy = (int)floordiv_exact(y, d.hww);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      int xi, yi;
      if (d.half_index_ok) {
        xi = (hx + d.g_xe[g]) >> 1;
        yi = (hy + d.g_ye[g]) >> 1;
      } else {
        xi = (int)(floordiv_exact(x - d.g_xe[g] * d.ww / 2., d.ww) + d.g_xe[g]);
        yi = (int)(floordiv_exact(y - d.g_ye[g] * d.ww / 2., d.ww) + d.g_ye[g]);
      }
      int a = yi - d.g_i0[g], b = xi - d.g_j0[g];
      if (a >= 0 && a < d.g_ni[g] && b >= 0 && b < d.g_nj[g]) {
        int bin = d.g_off[g] + a * d.g_nj[g] + b;
        if (use_smem) atomicAdd(&hist[bin], 1);
        else atomicAdd(&gcounts[bin], 1);
      }
    }
  }
  if (use_smem) {
    __syncthreads();
    for (int k = threadIdx.x; k < d.npts; k += blockDim.x)
      if (hist[k]) atomicAdd(&gcounts[k], hist[k]);
  }
}

// ========================================================================================
// a10 (interpolation): scipy.interpolate.griddata(method='cubic') spatial.py:144 =
// Qhull Delaunay (setup) + global gradient estimate + Clough-Tocher patches
// (scipy/interpolate/interpnd.pyx).
// ========================================================================================
// Gradient estimate (`_estimate_gradients_2d_global`): Gauss-Seidel sweeps in vertex order.
// The 4 offset grids are independent sets of the lattice triangulation, so a sweep is 4
// fully parallel phases with exactly the sequential algorithm's arithmetic.
// Per-vertex update with the data-independent parts hoisted to setup (gnx_set_density):
// the 2x2 matrix Q of `_estimate_gradients_2d_global` depends only on the triangulation,
// so its inverse (v_inv) and the per-edge weights ex/L^3, ey/L^3 are precomputed; a sweep
// then costs 6 flops per edge and no sqrt.
#define GS_DEG 8

// general form (any degree, CSR), used when a vertex has more than GS_DEG neighbours or the
// triangulation is not 4-colourable by grid
__device__ __forceinline__ double gs_vertex_csr(const Dens& d, const double* f, double* yv, int i) {
  double s0 = 0, s1 = 0;
  const double f1 = f[i];
  for (int jj = d.nbr_indptr[i]; jj < d.nbr_indptr[i + 1]; ++jj) {
    const int j = d.nbr_indices[jj];
    const double ex = d.e_ex[jj], ey = d.e_ey[jj];
    const double tt = 6 * (f1 - f[j]) + 2 * (ex * yv[2 * j] + ey * yv[2 * j + 1]);
    s0 += tt * d.e_wx[jj];
    s1 += tt * d.e_wy[jj];
  }
  const double r0 = d.v_inv[3 * i] * s0 + d.v_inv[3 * i + 1] * s1;
  const double r1 = d.v_inv[3 * i + 1] * s0 + d.v_inv[3 * i + 2] * s1;
  double change = fmax(fabs(yv[2 * i] + r0), fabs(yv[2 * i + 1] + r1));
  yv[2 * i] = -r0;
  yv[2 * i + 1] = -r1;
  change /= fmax(1.0, fmax(fabs(r0), fabs(r1)));
  return change;
}

#define GS_BLOCK 256
// Largest lattice of the register-resident solve: one thread per vertex in one CTA.  Its
// edge tables take 64 registers a thread; an SM's four schedulers hold 16384 registers each,
// so up to 20 warps (5 a scheduler) may use 96.  The default window width gives lattices of
// about 23 x 23 = 529 points.
#define GS_REG_PTS 640

// Fast path (lattices of <= GS_REG_PTS points, every vertex of degree <= GS_DEG, 4-colourable
// by grid): thread v owns vertex v for the whole solve.  The vertices are numbered grid by
// grid, so each colour phase is a contiguous range of threads.  The edge vectors and weights
// of the vertex's GS_DEG slots (pad: neighbour = self, weights = 0) do not change during the
// solve and stay in registers; shared memory holds the values and gradients, the 2x2 inverses
// and the neighbour ids, so an update gathers its 8 neighbours' values and gradients, one
// address each.  (Keeping the value differences or the unpacked ids in registers as well
// exceeds the 96 and spills.)  The arithmetic is spelled out with _rn intrinsics: it is the
// contraction nvcc chose for the shared-memory kernel this replaced, and no rounding of the
// solve may change (density feeds the death draws).
__global__ void __launch_bounds__(GS_REG_PTS, 1) k_ct_gradients_reg(Dens d, Counters* c, int maxiter, double tol) {
  const int which = blockIdx.x;          // 0 = species density N, 1 = pair-midpoint density
  const int npts = d.npts;
  const int v = threadIdx.x;
  const bool own = v < npts;
  struct __align__(16) Vert { double2 y; double f; };   // gradient and value: one address per neighbour
  __shared__ Vert sv[GS_REG_PTS];
  __shared__ double sinv[3][GS_REG_PTS];
  __shared__ uint4 snb[GS_REG_PTS];      // neighbour ids of slots 2q, 2q+1 in the low, high half of word q
  double ex[GS_DEG], ey[GS_DEG], wx[GS_DEG], wy[GS_DEG];
  int colour = -1;
  if (own) {
    // table layout is transposed ([(4*k + c)*npts + v], [k*npts + v], [c*npts + v]): coalesced loads
#pragma unroll
    for (int k = 0; k < GS_DEG; ++k) {
      ex[k] = d.p_e[(4 * k + 0) * npts + v];
      ey[k] = d.p_e[(4 * k + 1) * npts + v];
      wx[k] = d.p_e[(4 * k + 2) * npts + v];
      wy[k] = d.p_e[(4 * k + 3) * npts + v];
    }
    uint32_t w[GS_DEG / 2];
#pragma unroll
    for (int q = 0; q < GS_DEG / 2; ++q)
      w[q] = (uint32_t)d.p_j[2 * q * npts + v] | ((uint32_t)d.p_j[(2 * q + 1) * npts + v] << 16);
    snb[v] = make_uint4(w[0], w[1], w[2], w[3]);
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) sinv[cc][v] = d.v_inv_t[cc * npts + v];
#pragma unroll
    for (int g = 0; g < 4; ++g)
      if (v >= d.g_off[g] && v < d.g_off[g] + d.g_ni[g] * d.g_nj[g]) colour = g;
    const double f = (double)d.counts[(size_t)which * npts + v] / d.areas[v];   // spatial.py:95
    sv[v].f = f;
    d.vals[(size_t)which * npts + v] = f;
    sv[v].y = make_double2(0.0, 0.0);
  }
  __syncthreads();
  int it = 0;
  for (; it < maxiter; ++it) {
    double err = 0.0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (colour == g) {
        const double f1 = sv[v].f;
        const uint4 nbw = snb[v];
        const uint32_t nbp[GS_DEG / 2] = {nbw.x, nbw.y, nbw.z, nbw.w};
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int k = 0; k < GS_DEG; ++k) {
          // (6*(f1 - f2) - 2*df2) with df2 = -ex*y_j0 - ey*y_j1
          const Vert& nv = sv[(nbp[k >> 1] >> (16 * (k & 1))) & 0xffff];
          const double2 yj = nv.y;
          const double q = __fma_rn(ex[k], yj.x, __dmul_rn(ey[k], yj.y));
          const double tt = __fma_rn(__dsub_rn(f1, nv.f), 6.0, __dadd_rn(q, q));
          s0 = __fma_rn(tt, wx[k], s0);
          s1 = __fma_rn(tt, wy[k], s1);
        }
        const double i00 = sinv[0][v], i01 = sinv[1][v], i11 = sinv[2][v];
        const double r0 = __fma_rn(i00, s0, __dmul_rn(i01, s1));
        const double r1 = __fma_rn(i01, s0, __dmul_rn(i11, s1));
        const double2 yi = sv[v].y;
        const double change = fmax(fabs(__dadd_rn(yi.x, r0)), fabs(__dadd_rn(yi.y, r1)));
        sv[v].y = make_double2(-r0, -r1);
        err = fmax(err, __ddiv_rn(change, fmax(1.0, fmax(fabs(r0), fabs(r1)))));
      }
      // the barrier that ends the last colour phase also carries the convergence vote:
      // max over vertices of `change` < tol  <=>  every thread's `change` < tol
      if (g < 3) __syncthreads();
    }
    if (__syncthreads_and(err < tol)) break;
  }
  if (own) {
    double* gy = d.grad + (size_t)which * npts * 2;
    gy[2 * v] = sv[v].y.x;
    gy[2 * v + 1] = sv[v].y.y;
  }
  if (threadIdx.x == 0) c->gs_iters[which] = it < maxiter ? it + 1 : 0;     // 0: maxiter reached (scipy only warns)
}

// General path: larger lattices, vertices of degree > 8, or triangulations that are not
// 4-colourable by grid (then one thread runs the sequential sweep).
__global__ void __launch_bounds__(GS_BLOCK) k_ct_gradients(Dens d, Counters* c, int maxiter, double tol) {
  const int which = blockIdx.x;
  const int* counts = d.counts + (size_t)which * d.npts;
  double* f = d.vals + (size_t)which * d.npts;
  double* yv = d.grad + (size_t)which * d.npts * 2;
  for (int k = threadIdx.x; k < d.npts; k += blockDim.x) {
    f[k] = (double)counts[k] / d.areas[k];
    yv[2 * k] = 0.0;
    yv[2 * k + 1] = 0.0;
  }
  __syncthreads();
  int iters = 0;
  for (int it = 0; it < maxiter; ++it) {
    double err = 0.0;
    if (d.colourable) {
      for (int g = 0; g < 4; ++g) {
        const int s = d.g_off[g], e = s + d.g_ni[g] * d.g_nj[g];
        for (int v = s + threadIdx.x; v < e; v += GS_BLOCK) err = fmax(err, gs_vertex_csr(d, f, yv, v));
        if (g < 3) __syncthreads();
      }
    } else if (threadIdx.x == 0) {
      for (int v = 0; v < d.npts; ++v) err = fmax(err, gs_vertex_csr(d, f, yv, v));
    }
    if (__syncthreads_and(err < tol)) { iters = it + 1; break; }
  }
  if (threadIdx.x == 0) c->gs_iters[which] = iters;
}

__constant__ double CT_MONO[3 * 10 * 19];      // set by gnx_set_density
#define CT_STRIDE 49                           // per triangle: 3 x 10 monomial coefficients + 19 Bezier ordinates

// g weights of `_clough_tocher_2d_single` (scipy interpnd): they depend on the triangulation only,
// so they are computed once at setup with the arithmetic the coefficient kernel used to repeat
// every step (9 divisions and ~30 dependent loads per triangle)
__global__ void __launch_bounds__(128) k_ct_setup_g(Dens d, double* tri_g) {
  for (int t = GTID; t < d.ntri; t += GSTRIDE) {
    const double* P = d.points;
    const int v0 = d.simplices[3 * t], v1 = d.simplices[3 * t + 1], v2 = d.simplices[3 * t + 2];
    // barycentric transform of this triangle: b = Ainv (p - v2)
    const double a00 = P[2 * v0] - P[2 * v2], a01 = P[2 * v1] - P[2 * v2];
    const double a10 = P[2 * v0 + 1] - P[2 * v2 + 1], a11 = P[2 * v1 + 1] - P[2 * v2 + 1];
    const double det = a00 * a11 - a01 * a10;
    double g[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int itri = d.neighbors[3 * t + k];
      if (itri == -1) { g[k] = -0.5; continue; }
      const int w0 = d.simplices[3 * itri], w1 = d.simplices[3 * itri + 1], w2 = d.simplices[3 * itri + 2];
      const double y0 = (P[2 * w0] + P[2 * w1] + P[2 * w2]) / 3;
      const double y1 = (P[2 * w0 + 1] + P[2 * w1 + 1] + P[2 * w2 + 1]) / 3;
      const double dx = y0 - P[2 * v2], dy = y1 - P[2 * v2 + 1];
      double cc[3];
      cc[0] = (a11 * dx - a01 * dy) / det;
      cc[1] = (-a10 * dx + a00 * dy) / det;
      cc[2] = 1 - cc[0] - cc[1];
      if (k == 0) g[k] = (2 * cc[2] + cc[1] - 1) / (2 - 3 * cc[2] - 3 * cc[1]);
      else if (k == 1) g[k] = (2 * cc[0] + cc[2] - 1) / (2 - 3 * cc[0] - 3 * cc[2]);
      else g[k] = (2 * cc[1] + cc[0] - 1) / (2 - 3 * cc[1] - 3 * cc[0]);
    }
    tri_g[3 * t] = g[0];
    tri_g[3 * t + 1] = g[1];
    tri_g[3 * t + 2] = g[2];
  }
}

// Bezier ordinates of every triangle (`_clough_tocher_2d_single`, point-independent part) and the
// monomial coefficients of its micro-triangles.  A CTA takes CT_ITEMS (density, triangle) items: one
// thread per item computes the 19 ordinates once and stages them in shared memory, then every thread
// runs ONE of the 30 coefficients' 19-term FMA chains for one item (the chain's order is fixed, so the
// bits are).  Warp w owns coefficient w for all CT_ITEMS items, so its CT_MONO reads are warp-uniform
// (constant-cache broadcasts) and its shared-memory reads are stride-1.
#define CT_ITEMS 32
#define CT_COEF_THREADS (30 * CT_ITEMS)
__global__ void __launch_bounds__(CT_COEF_THREADS) k_ct_coefficients(Dens d) {
  __shared__ double so[19][CT_ITEMS];
  const int total = 2 * d.ntri;
  const int base = blockIdx.x * CT_ITEMS;
  if (threadIdx.x < CT_ITEMS && base + (int)threadIdx.x < total) {
    const int id = base + threadIdx.x;
    const int which = id / d.ntri, t = id - which * d.ntri;
    const double* f = d.vals + (size_t)which * d.npts;
    const double* gr = d.grad + (size_t)which * d.npts * 2;
    const double* P = d.points;
    const int v0 = d.simplices[3 * t], v1 = d.simplices[3 * t + 1], v2 = d.simplices[3 * t + 2];
    const double e12x = P[2 * v1] - P[2 * v0], e12y = P[2 * v1 + 1] - P[2 * v0 + 1];
    const double e23x = P[2 * v2] - P[2 * v1], e23y = P[2 * v2 + 1] - P[2 * v1 + 1];
    const double e31x = P[2 * v0] - P[2 * v2], e31y = P[2 * v0 + 1] - P[2 * v2 + 1];
    const double f1 = f[v0], f2 = f[v1], f3 = f[v2];
    const double df12 = +(gr[2 * v0] * e12x + gr[2 * v0 + 1] * e12y);
    const double df21 = -(gr[2 * v1] * e12x + gr[2 * v1 + 1] * e12y);
    const double df23 = +(gr[2 * v1] * e23x + gr[2 * v1 + 1] * e23y);
    const double df32 = -(gr[2 * v2] * e23x + gr[2 * v2 + 1] * e23y);
    const double df31 = +(gr[2 * v2] * e31x + gr[2 * v2 + 1] * e31y);
    const double df13 = -(gr[2 * v0] * e31x + gr[2 * v0 + 1] * e31y);
    const double c3000 = f1;
    const double c2100 = (df12 + 3 * c3000) / 3;
    const double c2010 = (df13 + 3 * c3000) / 3;
    const double c0300 = f2;
    const double c1200 = (df21 + 3 * c0300) / 3;
    const double c0210 = (df23 + 3 * c0300) / 3;
    const double c0030 = f3;
    const double c1020 = (df31 + 3 * c0030) / 3;
    const double c0120 = (df32 + 3 * c0030) / 3;
    const double c2001 = (c2100 + c2010 + c3000) / 3;
    const double c0201 = (c1200 + c0300 + c0210) / 3;
    const double c0021 = (c1020 + c0120 + c0030) / 3;
    // the neighbour-dependent weights g are static (triangulation only): precomputed by k_ct_setup_g
    const double g[3] = {d.tri_g[3 * t], d.tri_g[3 * t + 1], d.tri_g[3 * t + 2]};
    const double c0111 = (g[0] * (-c0300 + 3 * c0210 - 3 * c0120 + c0030) + (-c0300 + 2 * c0210 - c0120 + c0021 + c0201)) / 2;
    const double c1011 = (g[1] * (-c0030 + 3 * c1020 - 3 * c2010 + c3000) + (-c0030 + 2 * c1020 - c2010 + c2001 + c0021)) / 2;
    const double c1101 = (g[2] * (-c3000 + 3 * c2100 - 3 * c1200 + c0300) + (-c3000 + 2 * c2100 - c1200 + c2001 + c0201)) / 2;
    const double c1002 = (c1101 + c1011 + c2001) / 3;
    const double c0102 = (c1101 + c0111 + c0201) / 3;
    const double c0012 = (c1011 + c0111 + c0021) / 3;
    const double c0003 = (c1002 + c0102 + c0012) / 3;
    const double o[19] = {c3000, c0300, c0030, c0003, c2100, c2010, c2001, c0210, c0201, c0021,
                          c1200, c1020, c1002, c0120, c0102, c0012, c1101, c1011, c0111};
    double* mo = d.coef + (size_t)id * CT_STRIDE;
#pragma unroll
    for (int cidx = 0; cidx < 19; ++cidx) {
      mo[30 + cidx] = o[cidx];
      so[cidx][threadIdx.x] = o[cidx];
    }
  }
  __syncthreads();
  // Bezier ordinates -> monomial coefficients in (b0, b1): coefficient r of micro-triangle k is row
  // k * 10 + r of CT_MONO
  const int item = threadIdx.x % CT_ITEMS, row = threadIdx.x / CT_ITEMS;
  if (base + item < total) {
    double acc = 0.0;
#pragma unroll
    for (int cidx = 0; cidx < 19; ++cidx) acc = fma(CT_MONO[row * 19 + cidx], so[cidx][item], acc);
    d.coef[(size_t)(base + item) * CT_STRIDE + row] = acc;
  }
}

// Exact-order evaluation (scipy's own formula and operation order) from the Bezier ordinates.
// Used where the interpolant is at rounding-noise level (|w| < 1e-7), so that the sign / exact
// zero-ness of empty regions -- which d = N_d / N amplifies -- matches scipy's.
__device__ __noinline__ double ct_eval_exact(const Dens& d, int which, double qi, double qj) {
  int si = (int)floor(qi / d.hww), sj = (int)floor(qj / d.hww);
  si = min(max(si, 0), d.lat_ni - 2);
  sj = min(max(sj, 0), d.lat_nj - 2);
  const int* st = d.square_tri + 2 * (si * (d.lat_nj - 1) + sj);
  const double* P = d.points;
  int t = st[0];
  double b0, b1, b2;
  for (int k = 0; k < 2; ++k) {
    t = st[k];
    const int v0 = d.simplices[3 * t], v1 = d.simplices[3 * t + 1], v2 = d.simplices[3 * t + 2];
    const double a00 = P[2 * v0] - P[2 * v2], a01 = P[2 * v1] - P[2 * v2];
    const double a10 = P[2 * v0 + 1] - P[2 * v2 + 1], a11 = P[2 * v1 + 1] - P[2 * v2 + 1];
    const double det = a00 * a11 - a01 * a10;
    const double dx = qi - P[2 * v2], dy = qj - P[2 * v2 + 1];
    b0 = (a11 * dx - a01 * dy) / det;
    b1 = (-a10 * dx + a00 * dy) / det;
    b2 = 1 - b0 - b1;
    if (fmin(b0, fmin(b1, b2)) >= -1e-12 || k == 1) break;
  }
  const double* cf = d.coef + ((size_t)which * d.ntri + t) * CT_STRIDE + 30;
  const double minval = fmin(b0, fmin(b1, b2));
  const double B1 = b0 - minval, B2 = b1 - minval, B3 = b2 - minval, B4 = 3 * minval;
  const double c3000 = cf[0], c0300 = cf[1], c0030 = cf[2], c0003 = cf[3], c2100 = cf[4], c2010 = cf[5],
               c2001 = cf[6], c0210 = cf[7], c0201 = cf[8], c0021 = cf[9], c1200 = cf[10], c1020 = cf[11],
               c1002 = cf[12], c0120 = cf[13], c0102 = cf[14], c0012 = cf[15], c1101 = cf[16], c1011 = cf[17],
               c0111 = cf[18];
  return (B1 * B1 * B1 * c3000 + 3 * B1 * B1 * B2 * c2100 + 3 * B1 * B1 * B3 * c2010 + 3 * B1 * B1 * B4 * c2001 +
          3 * B1 * B2 * B2 * c1200 + 6 * B1 * B2 * B4 * c1101 + 3 * B1 * B3 * B3 * c1020 + 6 * B1 * B3 * B4 * c1011 +
          3 * B1 * B4 * B4 * c1002 + B2 * B2 * B2 * c0300 + 3 * B2 * B2 * B3 * c0210 + 3 * B2 * B2 * B4 * c0201 +
          3 * B2 * B3 * B3 * c0120 + 6 * B2 * B3 * B4 * c0111 + 3 * B2 * B4 * B4 * c0102 + B3 * B3 * B3 * c0030 +
          3 * B3 * B3 * B4 * c0021 + 3 * B3 * B4 * B4 * c0012 + B4 * B4 * B4 * c0003);
}

// point-dependent part of `_clough_tocher_2d_single` at (qi, qj).  Inside a triangle the
// interpolant is, on each of its three micro-triangles (k = index of the smallest
// barycentric coordinate), a bivariate cubic in (b0, b1); k_ct_coefficients converts the 19
// Bezier ordinates to those 3 x 10 monomial coefficients (CT_MONO, fixed 10x19 matrices built
// at setup), and the barycentric coordinates are an affine map of (qi, qj) precomputed per
// triangle (tri_aff), so one evaluation is ~12 FMAs with no division.
// lattice square index floor(q / hww), clamped: multiplicative estimate corrected to the exact
// floor (the products are exact for the half-windows in use), no division
__device__ __forceinline__ int lattice_index(double q, double hww, double inv_hww, int smax) {
  int s = (int)floor(q * inv_hww);
  if ((double)(s + 1) * hww <= q) s += 1;
  else if ((double)s * hww > q) s -= 1;
  return min(max(s, 0), smax);
}

// the cell's place in the triangulation, shared by both densities: triangle t, micro-triangle k and
// the barycentric coordinates (b0, b1)
struct CtLoc {
  int t, k;
  double b0, b1;
};
__device__ __forceinline__ CtLoc ct_locate(const Dens& d, double qi, double qj, int si, double inv_hww) {
  const int sj = lattice_index(qj, d.hww, inv_hww, d.lat_nj - 2);
  const int2 st = __ldg(reinterpret_cast<const int2*>(d.square_tri) + (si * (d.lat_nj - 1) + sj));
  int t = st.x;
  const double* a = d.tri_aff + 6 * t;
  double b0 = fma(a[2], qj, fma(a[1], qi, a[0]));
  double b1 = fma(a[5], qj, fma(a[4], qi, a[3]));
  double b2 = 1.0 - b0 - b1;
  if (fmin(b0, fmin(b1, b2)) < -1e-12) {
    t = st.y;
    a = d.tri_aff + 6 * t;
    b0 = fma(a[2], qj, fma(a[1], qi, a[0]));
    b1 = fma(a[5], qj, fma(a[4], qi, a[3]));
    b2 = 1.0 - b0 - b1;
  }
  const int k = (b0 <= b1 && b0 <= b2) ? 0 : ((b1 <= b2) ? 1 : 2);
  return CtLoc{t, k, b0, b1};
}

__device__ __forceinline__ double ct_eval_at(const Dens& d, int which, const CtLoc& l) {
  const double* m = d.coef + ((size_t)which * d.ntri + l.t) * CT_STRIDE + l.k * 10;
  const double b0 = l.b0, b1 = l.b1;
  // order: 1, b1, b1^2, b1^3, b0, b0 b1, b0 b1^2, b0^2, b0^2 b1, b0^3
  const double r0 = fma(b1, fma(b1, fma(b1, m[3], m[2]), m[1]), m[0]);
  const double r1 = fma(b1, fma(b1, m[6], m[5]), m[4]);
  const double r2 = fma(b1, m[8], m[7]);
  return fma(b0, fma(b0, fma(b0, m[9], r2), r1), r0);
}

__device__ __forceinline__ double ct_eval_point(const Dens& d, int which, double qi, double qj, int si, double inv_hww) {
  return ct_eval_at(d, which, ct_locate(d, qi, qj, si, inv_hww));
}

// a7 + a14: n_pairs raster (demography.py:60-91) and the logistic d raster
// (demography.py:104-172), never materialising dNdt / N_b / N_d.
__device__ __forceinline__ double raster_np(const Params& prm, const Work& w, int id, double np) {
  np = np < 0.0 ? 0.0 : np;
  if (isnan(np)) np = 0.0;
  if (prm.store_debug) w.NP_rast[id] = np;
  return np;
}

__device__ __forceinline__ void raster_d_store(const Params& prm, const Work& w, int id, double np, double N,
                                               double dNdt) {
  const double N_b = prm.c.b * prm.c.n_births_lambda * np;     // demography.py:142
  const double N_d = N_b - dNdt;                    // demography.py:149
  double dv = N_d / N;                              // demography.py:159-160
  if (isnan(dv)) dv = 0.0;
  dv = dv < prm.c.d_min ? prm.c.d_min : (dv > prm.c.d_max ? prm.c.d_max : dv);
  w.d_rast[id] = dv;                                // its own plane: a full-sector streaming write
}

__device__ __forceinline__ void raster_d_cell(const Land& land, const Params& prm, const Work& w, int id,
                                              double np, double Nmax) {
  np = raster_np(prm, w, id, np);
  const double N = w.N_rast[id], K = land.K[id];
  double dNdt = prm.c.R * (1 - (N / K)) * N;        // demography.py:95-97
  if (dNdt < -Nmax) dNdt = -Nmax;                   // np.clip(a_min=-N.max())
  if (isnan(dNdt) || isinf(dNdt)) dNdt = -Nmax;
  raster_d_store(prm, w, id, np, N, dNdt);
}

// The d of a cell needs max(N) only through the clip of dNdt at -Nmax.  Nmax >= N (N is one of the
// values it is the maximum of, and under strips it is also reduced over the ranks), so when dNdt is
// finite and >= -N neither clip can fire and d is final without Nmax.  Returns false for the other
// cells (K = 0, N > K (1 + 1/R), NaN): they are deferred to k_raster_fix_d.
__device__ __forceinline__ bool raster_d_cell_no_clip(const Land& land, const Params& prm, const Work& w, int id,
                                                      double np, double N) {
  const double K = land.K[id];
  const double dNdt = prm.c.R * (1 - (N / K)) * N;
  if (!(isfinite(dNdt) && dNdt >= -N)) return false;
  raster_d_store(prm, w, id, raster_np(prm, w, id, np), N, dNdt);
  return true;
}

// Both rasters in one pass over the landscape (Species._calc_density species.py:845-882 for N, clip
// >= 0, and the d raster), plus max(N).  Each cell is located once and both interpolants are
// evaluated there.  Two lists share Work.fix_list: from the front the cells whose N is at
// rounding-noise level, from the back the cells whose d waits for max(N) (raster_d_cell_no_clip).
// Rows are dealt to CTAs, columns to threads: no integer division per cell, the lattice row index is
// computed once per row.
__global__ void __launch_bounds__(256) k_raster_Nd(Dens d, Land land, Params prm, Work w, Counters* c, int row_lo,
                                                    int row_hi) {
  double mx = 0.0;
  const double inv_hww = 1.0 / d.hww;
  const int last = land.X * land.Y - 1;
  for (int i = row_lo + blockIdx.x; i < row_hi; i += gridDim.x) {
   const int si = lattice_index(i + 0.5, d.hww, inv_hww, d.lat_ni - 2);
   for (int j = threadIdx.x; j < land.X; j += blockDim.x) {
    const int id = i * land.X + j;
    const CtLoc loc = ct_locate(d, i + 0.5, j + 0.5, si, inv_hww);
    double v = ct_eval_at(d, 0, loc);
    const double np = ct_eval_at(d, 1, loc);
    // where the interpolant is at rounding-noise level its sign / exact zero-ness is what
    // d = N_d / N amplifies: those cells are re-evaluated in scipy's exact operation order
    // by k_raster_fix_N and k_raster_fix_d (none in a populated landscape)
    const bool fix = fabs(v) < 1e-7;
    if (fix) w.fix_list[atomicAdd(&w.fix_count[0], 1)] = id;
    v = v < 0.0 ? 0.0 : v;                    // np.clip(dens, a_min=0)
    w.N_rast[id] = v;
    mx = fmax(mx, v);
    if (!fix && !raster_d_cell_no_clip(land, prm, w, id, np, v)) w.fix_list[last - atomicAdd(&w.fix_count[1], 1)] = id;
   }
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > 0.0) atomicMax(&c->nmax_bits, (unsigned long long)__double_as_longlong(mx));
}

// exact-order N of the fix list, and their part of max(N)
__global__ void __launch_bounds__(256) k_raster_fix_N(Dens d, Land land, Work w, Counters* c) {
  const int nfix = w.fix_count[0];
  double mx = 0.0;
  for (int k = GTID; k < nfix; k += GSTRIDE) {
    const int id = w.fix_list[k];
    const int i = id / land.X, j = id - i * land.X;
    double v = ct_eval_exact(d, 0, i + 0.5, j + 0.5);
    v = v < 0.0 ? 0.0 : v;
    w.N_rast[id] = v;
    mx = fmax(mx, v);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > 0.0) atomicMax(&c->nmax_bits, (unsigned long long)__double_as_longlong(mx));
}

// d of both lists with the final max(N).  On the fix list d = N_d / N turns the noise of the
// pair-density interpolant into 0 or 1, so it too is evaluated in scipy's exact operation order;
// the deferred cells evaluate it as k_raster_Nd did.  The last CTA to finish keeps the list lengths
// in Counters.dens_lists and resets the list cursors for the next evaluation.
__global__ void __launch_bounds__(256) k_raster_fix_d(Dens d, Land land, Params prm, Work w, Counters* c) {
  const int nfix = w.fix_count[0], ndef = w.fix_count[1];
  const int last = land.X * land.Y - 1;
  const double Nmax = __longlong_as_double((long long)c->nmax_bits);
  const double inv_hww = 1.0 / d.hww;
  for (int k = GTID; k < nfix; k += GSTRIDE) {
    const int id = w.fix_list[k];
    const int i = id / land.X, j = id - i * land.X;
    raster_d_cell(land, prm, w, id, ct_eval_exact(d, 1, i + 0.5, j + 0.5), Nmax);
  }
  for (int k = GTID; k < ndef; k += GSTRIDE) {
    const int id = w.fix_list[last - k];
    const int i = id / land.X, j = id - i * land.X;
    const int si = lattice_index(i + 0.5, d.hww, inv_hww, d.lat_ni - 2);
    raster_d_cell(land, prm, w, id, ct_eval_point(d, 1, i + 0.5, j + 0.5, si, inv_hww), Nmax);
  }
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(reinterpret_cast<unsigned int*>(&w.fix_count[2]), 1u) == gridDim.x - 1;
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    c->dens_lists[0] = nfix;
    c->dens_lists[1] = ndef;
    w.fix_count[0] = 0;
    w.fix_count[1] = 0;
    w.fix_count[2] = 0;
  }
}

// ========================================================================================
// a3 + a15 + a16 (draw): environment gather (species.py:913-922), fitness
// (selection.py:51-112), death probability (selection.py:119-125, demography.py:306-321),
// Bernoulli mortality draw (demography.py:175-176).  The first n entries are in mating-grid
// order, so the d and environment raster reads of a warp's 32 individuals share a few
// neighbouring sectors.  With end_step = 1 (fused step) the last block to finish also closes
// the time step (Species._set_Nt species.py:554, the bookkeeping of demography.py:324-329):
// the dead are only FLAGGED here -- the next step's re-grid drops them.
// ========================================================================================
// 8 resident CTAs (<= 32 registers): the kernel waits on its per-individual raster and genome gathers,
// so residency beats registers (measured at c4: 262 us without the bound, 245 at 6, 233 at 8)
constexpr int DEATH_MINB = 8;
__global__ void __launch_bounds__(256, DEATH_MINB) k_death(Pop pop, Land land, Params prm, Traits tr, DevDraws dr, Work w,
                                                Counters* c, Mut mu, int end_step, const Strip* st) {
  const int n0 = c->n, n = c->n + c->B, cur = c->cur, T = pop.T;
  const int64_t t = c->t;
  const int32_t* __restrict__ ord = prm.ordered ? pop.ord[cur] : nullptr;
  const int own_lo = c->own_lo, own_hi = c->own_hi;
  int live = 0;
  for (int i = GTID; i < n; i += GSTRIDE) {
    if (st && (i < n0 ? (i < own_lo || i >= own_hi) : (st->sent[i] != 0))) {
      // a ghost of a neighbouring strip, or a newborn shipped to the strip it dispersed into:
      // not this rank's individual -- the next re-grid drops the entry
      w.alive[i] = 0;
      continue;
    }
    const double2 xy = pop.xy[cur][i];
    const double x = xy.x, y = xy.y;
    const int cx = (int)x, cy = (int)y;
    const size_t cell = (size_t)cy * land.X + cx;
    // d and the environment layers are read as planes: with the state in mating-grid order a warp's
    // 32 individuals sit in a few neighbouring landscape cells, so the plane reads share sectors,
    // and the d raster is written by k_raster_Nd as whole sectors (interleaved with the environment
    // values it was a read-modify-write of 8 bytes in every 24: 2.6x its algorithmic traffic)
    const size_t plane_sz = (size_t)land.X * land.Y;
    double p = w.d_rast[cell];                                     // demography.py:306
    if (prm.selection) {
      double wfit = 1.0;
      for (int tt = 0; tt < T; ++tt) {
        const double e = tr.univ_adv[tt] ? 1.0 : __ldg(&land.rasters[(size_t)tr.layer[tt] * plane_sz + cell]);
        const double z = pop.z[cur][(size_t)tt * pop.cap + i];
        const double phi = tr.phi_rast[tt] ? __ldg(&tr.phi_rast[tt][cell]) : tr.phi[tt];
        const double diff = fabs(e - z);
        const double gm = tr.gamma[tt];
        const double pw = gm == 1.0 ? diff : (gm == 2.0 ? diff * diff : pow(diff, gm));
        wfit *= 1 - phi * pw;                                     // selection.py:51-54
      }
      if (T > 0) wfit = wfit < 0.001 ? 0.001 : wfit;             // selection.py:74
      if (mu.enabled) {
        // selection.py:78-94: prod_k (1 - s_k * dosage(delet_locus_k)); a row gather per
        // individual, only once a deleterious mutation exists
        const int nd = mu.counts[2];
        if (nd > 0) {
          const uint32_t* g0 = reinterpret_cast<const uint32_t*>(pop.G + (size_t)pop.gslot[cur][i] * 2 * pop.Wq);
          const uint32_t* g1 = g0 + 4 * pop.Wq;
          double wd = 1.0;
          for (int k = 0; k < nd; ++k) {
            const int loc = mu.delet_eff[k];        // use_tskit: row delet_loci_idxs[k] (selection.py:86-88)
            const int dosage = (int)((g0[loc >> 5] >> (loc & 31)) & 1u) + (int)((g1[loc >> 5] >> (loc & 31)) & 1u);
            wd *= 1.0 - (double)dosage * mu.delet_s[k];
          }
          wfit *= wd;                                              // selection.py:110-111
        }
      }
      pop.fit[cur][i] = wfit;
      p = 1 - (1 - p) * wfit;                                     // selection.py:122
    }
    if (prm.c.max_age >= 0 && pop.age[cur][i] > prm.c.max_age) p = 1.0;    // demography.py:319-321
    if (prm.store_debug) w.death_p[i] = p;
    double u;
    if (dr.death_u) u = dr.death_u[(ord && i < n0) ? ord[i] : i];          // newborn o has ordinal n0 + o
    else {
      RngStream g(prm.seed_lo, prm.seed_hi, pop.idx[cur][i], SITE_DEATH, t);
      u = g.uniform();
    }
    const bool alive = !(u < p);
    w.alive[i] = alive;
    live += alive ? 1 : 0;
  }
  if (!end_step) return;
  // ---- survivors of the step, then (last block) the end-of-step bookkeeping
  __shared__ int blk_live;
  __shared__ bool is_last;
  if (threadIdx.x == 0) blk_live = 0;
  __syncthreads();
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) live += __shfl_xor_sync(0xffffffffu, live, o);
  if ((threadIdx.x & 31) == 0 && live) atomicAdd(&blk_live, live);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (blk_live) atomicAdd(&c->alive_acc, blk_live);
    __threadfence();
    is_last = atomicAdd(&c->ticket[1], 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    const int survivors = atomicAdd(&c->alive_acc, 0);
    gnx_step_record_t r;
    r.t = c->t;
    r.Nt = survivors;
    // strip decomposition: this rank's share -- the newborns it holds and the deaths among the
    // individuals it holds (the shares of all ranks sum to the species' counts)
    const int held = st ? (own_hi - own_lo) + c->B - c->tail_sent : n;
    r.n_births = st ? c->B - c->tail_sent : c->B;
    r.n_deaths = held - survivors;
    r.n_pairs = c->P;
    if (c->n_rec < w.max_records) w.records[c->n_rec] = r;
    c->n_rec += 1;
    c->n = n;                    // entries, dead ones included until the next re-grid drops them
    c->n_pre = n;
    c->n_alive = survivors;
    c->pending = 1;
    c->max_idx += c->B;
    c->t += 1;
    c->P = 0;
    c->B = 0;
    c->deaths = 0;
    c->nmax_bits = 0ull;
    c->alive_acc = 0;
    c->ticket[1] = 0u;
  }
}

// a16 (removal), explicit form: stable compaction of survivors into the other half of the SoA
// (entry order -- i.e. mating-grid order -- is preserved); the dead hand their genome slots
// back to the free list (no genome bytes move).  Used by the staged gnx_mortality, by panmixia
// (no re-grid to fold the removal into) and whenever the host needs the population between
// steps while deaths are pending.
struct MortalityScan {
  Pop pop;
  Work w;
  const Counters* cc;
  int32_t burn;
  __device__ int size(const Counters* c) const { return c->n_pre; }
  __device__ u64 value(int i) const { return w.alive[i] ? ((u64)1 << 32) : (u64)1; }
  // all loads of the SCAN_ITEMS elements are issued before the first store: source and
  // destination halves cannot be proven disjoint by the compiler, so interleaved copies
  // would serialise on memory latency
  static constexpr bool BATCHED = true;
  __device__ void apply_batch(const int* i, const u64* v, const u64* ex, int n) const {
    const int s = cc->cur, d = s ^ 1;
    bool live[SCAN_ITEMS], dead[SCAN_ITEMS];
    int dst[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      live[k] = i[k] < n && (v[k] >> 32);
      dead[k] = i[k] < n && !(v[k] >> 32);
      dst[k] = (int)(ex[k] >> 32);
    }
    {
      double2 xy[SCAN_ITEMS];
      double fit[SCAN_ITEMS];
      int64_t id[SCAN_ITEMS];
      int32_t age[SCAN_ITEMS], gs[SCAN_ITEMS];
      int8_t sx[SCAN_ITEMS];
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (live[k]) {
          xy[k] = pop.xy[s][i[k]];
          fit[k] = pop.fit[s][i[k]];
          id[k] = pop.idx[s][i[k]];
          age[k] = pop.age[s][i[k]];
          sx[k] = pop.sex[s][i[k]];
        }
        if (live[k] || dead[k]) gs[k] = pop.gslot[s][i[k]];
      }
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (live[k]) {
          pop.xy[d][dst[k]] = xy[k];
          pop.fit[d][dst[k]] = fit[k];
          pop.idx[d][dst[k]] = id[k];
          pop.age[d][dst[k]] = age[k];
          pop.sex[d][dst[k]] = sx[k];
          pop.gslot[d][dst[k]] = gs[k];
        } else if (dead[k] && !burn) {
          // n_free was already lowered by this step's births (k_after_births)
          pop.free_slots[cc->n_free + (int)(ex[k] & 0xffffffffu)] = gs[k];
        }
      }
    }
    for (int tt = 0; tt < pop.T; ++tt) {
      const double* zs = pop.z[s] + (size_t)tt * pop.cap;
      double* zd = pop.z[d] + (size_t)tt * pop.cap;
      double z[SCAN_ITEMS];
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k)
        if (live[k]) z[k] = zs[i[k]];
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k)
        if (live[k]) zd[dst[k]] = z[k];
    }
    if (pop.node[0][0]) {
      int32_t a[SCAN_ITEMS], b[SCAN_ITEMS];
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k)
        if (live[k]) { a[k] = pop.node[0][s][i[k]]; b[k] = pop.node[1][s][i[k]]; }
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k)
        if (live[k]) { pop.node[0][d][dst[k]] = a[k]; pop.node[1][d][dst[k]] = b[k]; }
    }
  }
  __device__ void apply(int, u64, u64) const {}
  __device__ void total(Counters* c, u64 tot) const {
    // spine runs before apply: stash totals where apply does not read them
    c->deaths = (int)(tot & 0xffffffffu);
    c->pad[0] = (int)(tot >> 32);          // survivors
  }
};

// closes an explicit compaction.  record = 1: the staged gnx_mortality, which also ends the time
// step; record = 0: deaths that a fused step had left pending (its k_death already ended the step)
__global__ void k_end_step(Counters* c, Work w, int burn, int record) {
  const int survivors = c->pad[0];
  if (record) {
    gnx_step_record_t r;
    r.t = c->t;
    r.Nt = survivors;
    r.n_births = c->B;
    r.n_deaths = c->deaths;
    r.n_pairs = c->P;
    if (c->n_rec < w.max_records) w.records[c->n_rec] = r;
    c->n_rec += 1;
    c->max_idx += c->B;
    c->t += 1;
  }
  if (!burn) c->n_free += c->deaths;
  c->n = survivors;
  c->n_pre = survivors;
  c->n_alive = survivors;
  c->n_sorted = 0;               // entry order is kept, but cell_start no longer matches the entries
  c->own_lo = 0;
  c->own_hi = survivors;
  c->pending = 0;
  c->cur ^= 1;
  c->P = 0;
  c->B = 0;
  c->deaths = 0;
  c->nmax_bits = 0ull;
}

// ========================================================================================
// Species order on demand.  The reference's Species is an OrderedDict in ascending id; the
// host-facing views (download, field reads, injected draws, tskit renumbering) need each
// entry's rank by id: an LSD radix sort of (id, entry) pairs, 8 bits per pass, only as many
// passes as the largest id has bits.  A pass takes its size from n, or from device memory when
// n_dev is given (the table simplification, gnx_simplify.cuh, sorts arrays the host never sizes).
// ========================================================================================
#define RS_BLOCK 256
#define RS_ITEMS 8
#define RS_TILE (RS_BLOCK * RS_ITEMS)

__global__ void __launch_bounds__(256) k_order_keys(Pop pop, Work w, const Counters* c, int n, int exclude_dead) {
  const int cur = c->cur;
  for (int p = GTID; p < n; p += GSTRIDE) {
    const bool dead = exclude_dead && !w.alive[p];
    w.sort_keys[0][p] = dead ? ~0ull : (unsigned long long)pop.idx[cur][p];
    w.sort_vals[0][p] = p;
  }
}

__device__ __forceinline__ int radix_tiles(int n) { return max(1, (n + RS_TILE - 1) / RS_TILE); }

__global__ void __launch_bounds__(RS_BLOCK) k_radix_hist(const unsigned long long* __restrict__ keys, int n,
                                                          const int* n_dev, int shift, uint32_t* hist) {
  __shared__ uint32_t h[256];
  if (n_dev) n = *n_dev;
  const int ntiles = radix_tiles(n);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    h[threadIdx.x] = 0u;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ITEMS; ++r) {
      const int i = tile * RS_TILE + r * RS_BLOCK + threadIdx.x;
      if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * ntiles + tile] = h[threadIdx.x];       // digit-major: one scan orders everything
    __syncthreads();
  }
}

struct RadixScan {
  uint32_t* hist;
  int n;
  const int* n_dev;
  __device__ int size(const Counters*) const { return 256 * radix_tiles(n_dev ? *n_dev : n); }
  __device__ u64 value(int i) const { return hist[i]; }
  __device__ void apply(int i, u64, u64 ex) const { hist[i] = (uint32_t)ex; }
  __device__ void total(Counters*, u64) const {}
};

__global__ void __launch_bounds__(RS_BLOCK) k_radix_scatter(const unsigned long long* __restrict__ kin,
                                                             const int32_t* __restrict__ vin, unsigned long long* kout,
                                                             int32_t* vout, int n, const int* n_dev, int shift,
                                                             const uint32_t* hist) {
  __shared__ uint32_t base[256];
  if (n_dev) n = *n_dev;
  const int ntiles = radix_tiles(n);
  __shared__ uint32_t wcnt[RS_BLOCK / 32][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    base[threadIdx.x] = hist[(size_t)threadIdx.x * ntiles + tile];
    __syncthreads();
    for (int r = 0; r < RS_ITEMS; ++r) {
      const int i = tile * RS_TILE + r * RS_BLOCK + threadIdx.x;
      const bool valid = i < n;
      const unsigned long long key = valid ? kin[i] : 0ull;
      const uint32_t dgt = (uint32_t)(key >> shift) & 255u;
#pragma unroll
      for (int k = 0; k < RS_BLOCK / 32; ++k) wcnt[k][threadIdx.x] = 0u;
      __syncthreads();
      // stable rank inside the warp: lanes with the same digit, in lane order
      const unsigned same = __match_any_sync(0xffffffffu, valid ? dgt : (256u + lane));
      const int rank_in_warp = __popc(same & ((1u << lane) - 1u));
      if (valid && rank_in_warp == 0) wcnt[warp][dgt] = (uint32_t)__popc(same);
      __syncthreads();
      {                                             // thread d: running offsets of digit d over the warps
        uint32_t run = base[threadIdx.x];
#pragma unroll
        for (int k = 0; k < RS_BLOCK / 32; ++k) {
          const uint32_t cnt = wcnt[k][threadIdx.x];
          wcnt[k][threadIdx.x] = run;
          run += cnt;
        }
        base[threadIdx.x] = run;
      }
      __syncthreads();
      if (valid) {
        const uint32_t dst = wcnt[warp][dgt] + (uint32_t)rank_in_warp;
        kout[dst] = key;
        vout[dst] = vin[i];
      }
      __syncthreads();
    }
  }
}

// sorted (id, entry) pairs -> ord (entry -> ordinal) and inv (ordinal -> entry)
__global__ void __launch_bounds__(256) k_order_finish(Pop pop, Work w, const Counters* c, const int32_t* __restrict__ vals,
                                                       int n_ranked) {
  const int cur = c->cur;
  for (int i = GTID; i < n_ranked; i += GSTRIDE) {
    const int p = vals[i];
    pop.ord[cur][p] = i;
    w.inv[i] = p;
  }
}

// the population in species order, written into the idle half: x | y as two plain arrays in the
// xy buffer ([0, n) and [cap, cap + n)), every other field at its ordinal; z additionally as
// [n][T] rows for the host layout
__global__ void __launch_bounds__(256) k_species_gather(Pop pop, Work w, const Counters* c, int n, double* z_rows) {
  const int s = c->cur, d = s ^ 1;
  double* sx = reinterpret_cast<double*>(pop.xy[d]);
  double* sy = sx + pop.cap;
  for (int i = GTID; i < n; i += GSTRIDE) {
    const int p = w.inv[i];
    const double2 v = pop.xy[s][p];
    sx[i] = v.x;
    sy[i] = v.y;
    pop.age[d][i] = pop.age[s][p];
    pop.sex[d][i] = pop.sex[s][p];
    pop.idx[d][i] = pop.idx[s][p];
    pop.fit[d][i] = pop.fit[s][p];
    pop.gslot[d][i] = pop.gslot[s][p];
    for (int tt = 0; tt < pop.T; ++tt) {
      const double z = pop.z[s][(size_t)tt * pop.cap + p];
      pop.z[d][(size_t)tt * pop.cap + i] = z;
      if (z_rows) z_rows[(size_t)i * pop.T + tt] = z;
    }
  }
}

// one per-entry work array in species order (parity tests): out[i] = src[inv[i]].  For arrays
// of ENTRY numbers (mate, pairs) the values are translated to ordinals as well.
template <class TT>
__global__ void __launch_bounds__(256) k_gather_by_inv(const TT* __restrict__ src, TT* out, const int32_t* __restrict__ inv, int n) {
  for (int i = GTID; i < n; i += GSTRIDE) out[i] = src[inv[i]];
}
__global__ void __launch_bounds__(256) k_gather_mate(const int32_t* __restrict__ mate, int32_t* out,
                                                      const int32_t* __restrict__ inv, const int32_t* __restrict__ ord, int n,
                                                      int by_slot) {
  for (int i = GTID; i < n; i += GSTRIDE) {
    const int m = mate[by_slot ? i : inv[i]];
    out[i] = m < 0 ? -1 : ord[m];
  }
}
__global__ void __launch_bounds__(256) k_translate_entries(const int32_t* __restrict__ src, int32_t* out,
                                                            const int32_t* __restrict__ ord, int n) {
  for (int i = GTID; i < n; i += GSTRIDE) out[i] = src[i] < 0 ? -1 : ord[src[i]];
}

// environment values for every live individual in species order (API view of ind.e, species.py:913-922)
__global__ void __launch_bounds__(256) k_sample_env(Pop pop, Land land, Work w, const Counters* c, int n) {
  const int cur = c->cur;
  const size_t plane = (size_t)land.X * land.Y;
  for (int i = GTID; i < n; i += GSTRIDE) {
    const double2 xy = pop.xy[cur][w.inv[i]];
    const size_t cell = (size_t)((int)xy.y) * land.X + (int)xy.x;
    for (int l = 0; l < land.n_layers; ++l) w.e_out[(size_t)i * land.n_layers + l] = land.rasters[l * plane + cell];
  }
}

// genome rows gathered into species order (download): gslot = the species-ordered slot array
__global__ void __launch_bounds__(256) k_gather_genomes(Pop pop, const int32_t* __restrict__ gslot, uint4* out, int n) {
  const int row = 2 * pop.Wq;
  const long long total = (long long)n * row;
  for (long long k = GTID; k < total; k += GSTRIDE) {
    const int i = (int)(k / row), q = (int)(k - (long long)i * row);
    out[k] = pop.G[(size_t)gslot[i] * row + q];
  }
}

__global__ void __launch_bounds__(256) k_raster_to_f32(const double* src, float* dst, size_t n) {
  for (size_t id = GTID; id < n; id += GSTRIDE) dst[id] = (float)src[id];
}

// upload epilogue: identity genome slots, default ids, z [n][T] -> [T][cap], counters reset
// (time-step counter and record cursor carry over).  The uploaded order is kept as it is: the
// first re-grid sorts it.
__global__ void __launch_bounds__(256) k_upload_finish(Pop pop, Counters* c, int n, long long max_idx, int make_ids,
                                                        const double* z_rows) {
  // x and y arrive as two plain arrays staged in the other half: [0, n) and [cap, cap + n)
  const double* sx = reinterpret_cast<const double*>(pop.xy[1]);
  const double* sy = sx + pop.cap;
  for (int i = GTID; i < n; i += GSTRIDE) {
    pop.xy[0][i] = make_double2(sx[i], sy[i]);
    pop.gslot[0][i] = i;
    if (make_ids) pop.idx[0][i] = i;
    if (pop.node[0][0]) {             // post-simplify convention, species.py:1148-1152
      pop.node[0][0][i] = 2 * i;
      pop.node[1][0][i] = 2 * i + 1;
    }
    if (z_rows)
      for (int tt = 0; tt < pop.T; ++tt) pop.z[0][(size_t)tt * pop.cap + i] = z_rows[(size_t)i * pop.T + tt];
  }
  if (GTID == 0) {
    c->n = n; c->n_pre = n; c->P = 0; c->B = 0; c->deaths = 0; c->n_free = 0; c->n_slots = n; c->cur = 0;
    c->max_idx = max_idx; c->err = 0; c->nmax_bits = 0ull;
    c->n_nodes = 2 * n; c->n_ind_rows = n; c->n_edges = 0; c->n_born = 0;
    c->n_sorted = 0; c->pending = 0; c->n_alive = n; c->alive_acc = 0; c->ticket[0] = c->ticket[1] = 0u;
    c->own_lo = 0; c->own_hi = n; c->tail_sent = 0;
  }
}

// ========================================================================================
// f2 on-device stats (sim/stats.py:399-435): per-locus 1-allele counts and heterozygote
// counts straight from the bit-packed genotypes, and the fitness sum.  A warp takes 32
// individuals; for every 32-bit word column, one ballot per bit turns the 32 lanes' words
// into a per-locus count (vertical popcount), accumulated in shared memory per CTA.
// ========================================================================================
__global__ void __launch_bounds__(256) k_stats_genotypes(Pop pop, const Counters* c, unsigned long long* c1,
                                                          unsigned long long* chet, double* fit_sum,
                                                          double x0, double x1, double y0, double y1,
                                                          unsigned long long* n_in) {
  extern __shared__ unsigned int st_smem[];       // [2][Wwords * 32]
  const int n = c->n, cur = c->cur, Ww = 4 * pop.Wq, nbits = Ww * 32;
  for (int k = threadIdx.x; k < 2 * nbits; k += blockDim.x) st_smem[k] = 0u;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int nwarps = GSTRIDE / 32;
  double fsum = 0.0;
  for (int base = (GTID / 32) * 32; base < n; base += nwarps * 32) {
    const int i = base + lane;
    bool live = i < n;
    if (live) {                      // restrict to the rectangle [x0, x1) x [y0, y1) (sub-population statistics)
      const double2 xy = pop.xy[cur][i];
      live = xy.x >= x0 && xy.x < x1 && xy.y >= y0 && xy.y < y1;
    }
    const unsigned inside = __ballot_sync(0xffffffffu, live);
    if (lane == 0 && inside) atomicAdd(n_in, (unsigned long long)__popc(inside));
    const uint32_t* row = reinterpret_cast<const uint32_t*>(pop.G + (size_t)(live ? pop.gslot[cur][i] : 0) * 2 * pop.Wq);
    if (live) fsum += pop.fit[cur][i];
    for (int wd = 0; wd < Ww; ++wd) {
      const uint32_t h0 = live ? row[wd] : 0u, h1 = live ? row[Ww + wd] : 0u;
      const uint32_t both = h0 & h1, x = h0 ^ h1;
#pragma unroll 4
      for (int b = 0; b < 32; ++b) {
        const unsigned mx = __ballot_sync(0xffffffffu, (x >> b) & 1u);
        const unsigned mb = __ballot_sync(0xffffffffu, (both >> b) & 1u);
        if (lane == b) {          // lane b owns bit b of this word column
          const int nhet = __popc(mx), nhom = __popc(mb);
          if (nhet | nhom) {
            atomicAdd(&st_smem[wd * 32 + b], (unsigned)(nhet + 2 * nhom));
            atomicAdd(&st_smem[nbits + wd * 32 + b], (unsigned)nhet);
          }
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) fsum += __shfl_xor_sync(0xffffffffu, fsum, o);
  if (lane == 0 && fsum != 0.0) atomicAdd(fit_sum, fsum);
  __syncthreads();
  for (int k = threadIdx.x; k < nbits; k += blockDim.x) {
    if (st_smem[k]) atomicAdd(&c1[k], (unsigned long long)st_smem[k]);
    if (st_smem[nbits + k]) atomicAdd(&chet[k], (unsigned long long)st_smem[nbits + k]);
  }
}

// ========================================================================================
// f2 linkage disequilibrium (sim/stats.py:359-392 _calc_ld): for every pair of loci (i, j) the
// number of CHROMOSOMES carrying the 1-allele at both, n11[i][j] = sum_h bit_i(h) & bit_j(h) over
// the 2n haplotypes -- the binary product H^T H of the haplotype matrix; r^2 follows on the host
// from n11 and its diagonal exactly as the reference writes it.  One warp owns one 32 x 32 tile
// (word column wi x word column wj >= wi) over a range of haplotypes, lane = haplotype: the 32
// lanes' words are bit-transposed (5 butterfly stages of shuffles), so that lane l holds the
// membership mask of locus 32*w + l over the 32 haplotypes; every lane then accumulates its own
// locus of the tile's rows against the 32 column masks (broadcast by shuffle) with AND + POPC.
// ========================================================================================
__device__ __forceinline__ uint32_t warp_bit_transpose(uint32_t x, int lane) {
  // 32 x 32 bit-matrix transpose across the warp: afterwards bit h of lane l = bit l of lane h
#pragma unroll
  for (int j = 16; j >= 1; j >>= 1) {
    const uint32_t m = j == 16 ? 0x0000ffffu : j == 8 ? 0x00ff00ffu : j == 4 ? 0x0f0f0f0fu : j == 2 ? 0x33333333u : 0x55555555u;
    const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
    // lanes with bit j clear keep their low halves and take the partner's low halves shifted up
    x = (lane & j) ? ((x & ~m) | ((y >> j) & m)) : ((x & m) | ((y << j) & ~m));
  }
  return x;
}

__global__ void __launch_bounds__(256) k_stats_ld(Pop pop, const Counters* c, unsigned long long* n11, int Wu, int Lp,
                                                   int nsplit) {
  const int n = c->n, cur = c->cur, Ww = 4 * pop.Wq;
  const int lane = threadIdx.x & 31;
  const int ntile = Wu * (Wu + 1) / 2;
  const long long nhap = 2ll * n;
  const long long ngroup = (nhap + 31) / 32;                 // groups of 32 haplotypes
  for (int item = GTID >> 5; item < ntile * nsplit; item += GSTRIDE >> 5) {
    const int tile = item / nsplit, part = item % nsplit;
    int wi = 0, rem = tile;                                    // tile -> (wi, wj), wj >= wi
    while (rem >= Wu - wi) { rem -= Wu - wi; ++wi; }
    const int wj = wi + rem;
    uint32_t acc[32];
#pragma unroll
    for (int b = 0; b < 32; ++b) acc[b] = 0u;
    const long long g0 = ngroup * part / nsplit, g1 = ngroup * (part + 1) / nsplit;
    for (long long g = g0; g < g1; ++g) {
      const long long h = g * 32 + lane;
      uint32_t a = 0u, bw = 0u;
      if (h < nhap) {
        const uint32_t* row = reinterpret_cast<const uint32_t*>(pop.G + (size_t)pop.gslot[cur][(int)(h >> 1)] * 2 * pop.Wq)
                              + (size_t)(h & 1) * Ww;
        a = row[wi];
        bw = row[wj];
      }
      const uint32_t mi = warp_bit_transpose(a, lane);         // haplotypes carrying locus 32*wi + lane
      const uint32_t mj = wi == wj ? mi : warp_bit_transpose(bw, lane);
#pragma unroll
      for (int b = 0; b < 32; ++b) acc[b] += __popc(mi & __shfl_sync(0xffffffffu, mj, b));
    }
#pragma unroll
    for (int b = 0; b < 32; ++b)
      if (acc[b]) atomicAdd(&n11[(size_t)(32 * wi + lane) * Lp + 32 * wj + b], (unsigned long long)acc[b]);
  }
}

// ========================================================================================
// f4 burn-in control (sim/burnin.py:21-58 SpatialTester.update): individuals per landscape cell,
// and the sum and sum of squares of the change of every cell's count since the previous call
// (mean and standard deviation of `diff` follow on the host).  Integer sums: exact.
// ========================================================================================
__global__ void __launch_bounds__(256) k_burnin_count(Pop pop, Land land, const Counters* c, int32_t* counts) {
  const int n = c->n, cur = c->cur;
  for (int p = GTID; p < n; p += GSTRIDE) {
    const double2 xy = pop.xy[cur][p];
    const int ix = (int)xy.x, iy = (int)xy.y;
    // burnin.py:49-52 fills counts[i, j], i < dim[0], j < dim[1], from the (x = j, y = i) tally: on a
    // non-square landscape the individuals with x >= dim[1] or y >= dim[0] are not counted
    if (ix < land.Y && iy < land.X) atomicAdd(&counts[(size_t)iy * land.X + ix], 1);
  }
}

__global__ void __launch_bounds__(256) k_burnin_diff(const int32_t* __restrict__ counts, int32_t* prev, size_t ncell,
                                                      long long* sums) {
  long long s1 = 0, s2 = 0;
  for (size_t k = GTID; k < ncell; k += GSTRIDE) {
    const long long d = (long long)counts[k] - prev[k];
    s1 += d;
    s2 += d * d;
    prev[k] = counts[k];
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  if ((threadIdx.x & 31) == 0 && (s1 | s2)) {
    atomicAdd(reinterpret_cast<unsigned long long*>(&sums[0]), (unsigned long long)s1);
    atomicAdd(reinterpret_cast<unsigned long long*>(&sums[1]), (unsigned long long)s2);
  }
}

// node ids 2k, 2k+1 in species order (after simplify, species.py:1148-1152); reset_t0 marks
// the current step as tskit time 0
__global__ void __launch_bounds__(256) k_tskit_renumber(Pop pop, Counters* c, int reset_t0) {
  const int n = c->n, cur = c->cur;
  for (int i = GTID; i < n; i += GSTRIDE) {
    const int o = pop.ord[cur][i];                  // ordinal in species order (build_order ran just before)
    pop.node[0][cur][i] = 2 * o;
    pop.node[1][cur][i] = 2 * o + 1;
  }
  if (GTID == 0) {
    c->n_nodes = 2 * n;
    c->n_ind_rows = n;
    if (reset_t0) { c->tsk_t0 = c->t; c->n_edges = 0; c->n_born = 0; }
  }
}

__global__ void __launch_bounds__(256) k_scatter_nodes(Pop pop, Work w, const Counters* c, const int32_t* n0,
                                                        const int32_t* n1, int n) {
  const int cur = c->cur;
  for (int i = GTID; i < n; i += GSTRIDE) {
    const int p = w.inv[i];
    pop.node[0][cur][p] = n0[i];
    pop.node[1][cur][p] = n1[i];
  }
}

__global__ void k_K_from_layer(const double* rast, double* K, double factor, int ncell) {
  for (int id = GTID; id < ncell; id += GSTRIDE) K[id] = rast[id] * factor;   // species.py:546-547
}
