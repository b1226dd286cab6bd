// gnx_genome_init.cuh -- device assignment of the starting genomes with exact per-locus allele
// counts (the genome assignment at the end of the burn-in, species.py:956-1094, genome.py:1108-1157,
// done without a host genotype array).  Part of libgnxb200.so (sm_100a); driven by the
// gnx_genome_init_* entry points of gnx_api.cu.
//
// Homologue h of the individual with id i has, at locus l, the 64-bit key
//   K_l(i, h) = Philox2x32-10(counter = 2i + h, key = k_l),  k_l from (seed, l, SITE_GENOME_INIT).
// Philox is a bijection of its counter, so the keys of one locus never tie, and the n_l carriers of
// locus l are exactly the n_l homologues with the smallest keys.  The result depends only on the
// seed, the set of live ids and the counts -- not on the entry order or on how the population is
// cut into strips.  The n_l-th smallest key is found by an MSB-first radix select: keys are
// regenerated in every pass and never stored (2 * 10^10 of them at 10^7 individuals x 1000 loci).
#pragma once
#include "gnx_common.cuh"

#define GI_DIGIT 11                       // bits resolved per pass
#define GI_BINS (1 << GI_DIGIT)
#define GI_TILE 4                         // loci per CTA of the histogram pass (4 x 8 KB of shared memory)

enum { SITE_GENOME_INIT = 10 };

// select state of one locus: the carriers are the keys whose top `bits` bits are < prefix
// (state GI_LT) or <= prefix (GI_LE); GI_ACTIVE loci still have `remaining` carriers to pick among
// the keys whose top `bits` bits equal prefix
enum { GI_ACTIVE = 0, GI_LT = 1, GI_LE = 2, GI_ERR = 3 };
struct GiLocus {
  unsigned long long prefix;
  long long remaining;
  int32_t bits;
  int32_t state;
};

__device__ __forceinline__ unsigned long long philox2x32_10(unsigned long long ctr, uint32_t k) {
  uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32);
  const uint32_t M = 0xD256D193u, W = 0x9E3779B9u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi = __umulhi(M, c0), lo = M * c0;
    c0 = hi ^ k ^ c1;
    c1 = lo;
    k += W;
  }
  return ((unsigned long long)c0 << 32) | c1;
}

__device__ __forceinline__ unsigned long long gi_key(long long id, int h, uint32_t k) {
  return philox2x32_10(2ull * (unsigned long long)id + (unsigned long long)h, k);
}

__device__ __forceinline__ bool gi_carrier(unsigned long long key, const GiLocus& s) {
  if (s.state != GI_LT && s.state != GI_LE) return false;
  const unsigned long long top = s.bits ? (key >> (64 - s.bits)) : 0ull;
  return s.state == GI_LT ? top < s.prefix : top <= s.prefix;
}

// per-locus Philox keys and the starting select state (n_l = 0 or loci left out: no carriers)
__global__ void __launch_bounds__(256) k_gi_setup(GiLocus* st, uint32_t* lkey, const long long* n_carriers,
                                                  const uint8_t* select, int L, uint32_t seed_lo, uint32_t seed_hi) {
  for (int l = GTID; l < L; l += GSTRIDE) {
    lkey[l] = philox4x32_10(make_uint4((uint32_t)l, (uint32_t)SITE_GENOME_INIT << 24, 0u, 0u),
                            make_uint2(seed_lo, seed_hi)).x;
    GiLocus s;
    s.prefix = 0ull;
    s.remaining = n_carriers[l];
    s.bits = 0;
    s.state = (n_carriers[l] > 0 && select[l]) ? GI_ACTIVE : GI_LT;
    st[l] = s;
  }
}

// every live entry gets its own genome row (burn-in newborns have none, k_newborns): slot = entry
__global__ void __launch_bounds__(256) k_gi_slots(Pop pop, Counters* c) {
  const int n = c->n, cur = c->cur;
  for (int i = GTID; i < n; i += GSTRIDE) pop.gslot[cur][i] = i;
  if (GTID == 0) {
    c->n_free = 0;
    c->n_slots = n;
  }
}

// histogram of the next digit of the keys in every active locus's bucket; blockIdx.y = tile of
// GI_TILE loci, blockIdx.x = slice of the entries
__global__ void __launch_bounds__(256) k_gi_hist(Pop pop, const Counters* c, const GiLocus* __restrict__ st,
                                                 const uint32_t* __restrict__ lkey, int32_t* hist, int L) {
  __shared__ uint32_t sh[GI_TILE][GI_BINS];
  __shared__ GiLocus ss[GI_TILE];
  __shared__ uint32_t sk[GI_TILE];
  __shared__ int any;
  const int l0 = blockIdx.y * GI_TILE;
  if (threadIdx.x == 0) any = 0;
  __syncthreads();
  if (threadIdx.x < GI_TILE) {
    const int l = l0 + threadIdx.x;
    GiLocus s;
    s.state = GI_LT;
    if (l < L) s = st[l];
    ss[threadIdx.x] = s;
    sk[threadIdx.x] = l < L ? lkey[l] : 0u;
    if (s.state == GI_ACTIVE) atomicOr(&any, 1);
  }
  __syncthreads();
  if (!any) return;
  for (int k = threadIdx.x; k < GI_TILE * GI_BINS; k += blockDim.x) (&sh[0][0])[k] = 0u;
  __syncthreads();
  const int n = c->n, cur = c->cur;
  const int64_t* ids = pop.idx[cur];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const long long id = ids[i];
#pragma unroll
    for (int t = 0; t < GI_TILE; ++t) {
      const GiLocus s = ss[t];
      if (s.state != GI_ACTIVE) continue;
      const int dbits = min(GI_DIGIT, 64 - s.bits);
      const int shift = 64 - s.bits - dbits;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const unsigned long long key = gi_key(id, h, sk[t]);
        if (s.bits && (key >> (64 - s.bits)) != s.prefix) continue;
        atomicAdd(&sh[t][(uint32_t)(key >> shift) & ((1u << dbits) - 1u)], 1u);
      }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < GI_TILE * GI_BINS; k += blockDim.x) {
    const int t = k / GI_BINS;
    const uint32_t v = (&sh[0][0])[k];
    if (v && ss[t].state == GI_ACTIVE) atomicAdd(&hist[(size_t)(l0 + t) * GI_BINS + (k % GI_BINS)], (int32_t)v);
  }
}

// one CTA per locus: pick the digit that holds the remaining carriers, narrow the bucket, and
// finish the locus when the whole bucket (or none of it) is carried.  counts[0]: loci that need
// another pass; counts[1]: loci asked for more carriers than the population has homologues.
__global__ void __launch_bounds__(256) k_gi_select(GiLocus* st, const int32_t* __restrict__ hist, int32_t* counts) {
  const int l = blockIdx.x;
  GiLocus s = st[l];
  if (s.state != GI_ACTIVE) return;
  const int32_t* hl = hist + (size_t)l * GI_BINS;
  const int per = GI_BINS / 256;
  long long v[GI_BINS / 256], sum = 0;
#pragma unroll
  for (int k = 0; k < per; ++k) {
    v[k] = hl[threadIdx.x * per + k];
    sum += v[k];
  }
  // block inclusive scan of the per-thread sums
  __shared__ long long wsum[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  long long inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) wsum[wid] = inc;
  __syncthreads();
  long long before = 0, total = 0;
  for (int w = 0; w < 8; ++w) {
    if (w < wid) before += wsum[w];
    total += wsum[w];
  }
  inc += before;
  const long long exc = inc - sum;
  const long long r = s.remaining;
  if (r >= total || r == 0) {                      // every key of the bucket, none, or more than it has
    if (threadIdx.x == 0) {
      st[l].state = r == total ? GI_LE : (r == 0 ? GI_LT : GI_ERR);
      if (r > total) atomicAdd(&counts[1], 1);
    }
    return;
  }
  if (!(exc < r && r <= inc)) return;
  long long acc = exc;
  const int dbits = min(GI_DIGIT, 64 - s.bits);
  for (int k = 0; k < per; ++k) {
    if (acc + v[k] >= r) {
      const int d = threadIdx.x * per + k;
      s.prefix = (s.prefix << dbits) | (unsigned long long)d;
      s.bits += dbits;
      s.remaining = r - acc;
      if (s.remaining == v[k]) s.state = GI_LE;
      else if (s.bits >= 64) {                     // a 64-bit bucket holds one key unless ids repeat
        s.state = GI_ERR;
        atomicAdd(&counts[1], 1);
      } else {
        atomicAdd(&counts[0], 1);
      }
      st[l] = s;
      return;
    }
    acc += v[k];
  }
}

// one thread per (entry, 32-bit word): both homologue words of the row.  Loci outside `write`
// (neutral loci of the tskit layout) and the padding beyond L stay zero.  cols (column layout,
// {n_cols, col_locus[]}): bit j of the row is locus col_locus[j], the unused columns stay zero.
__global__ void __launch_bounds__(256) k_gi_write(Pop pop, const Counters* c, const GiLocus* __restrict__ st,
                                                  const uint32_t* __restrict__ lkey, const uint8_t* __restrict__ write,
                                                  int L, const int32_t* __restrict__ cols) {
  const int n = c->n, cur = c->cur, Ww = 4 * pop.Wq;
  const long long total = (long long)n * Ww;
  uint32_t* G = reinterpret_cast<uint32_t*>(pop.G);
  for (long long k = GTID; k < total; k += GSTRIDE) {
    const int i = (int)(k / Ww), w = (int)(k - (long long)i * Ww);
    const long long id = pop.idx[cur][i];
    uint32_t h0 = 0u, h1 = 0u;
    for (int j = 0; j < 32; ++j) {
      int l = 32 * w + j;
      if (cols) {
        if (l >= cols[0]) break;
        l = cols[1 + l];
      }
      if (l >= L) break;
      if (!write[l]) continue;
      const GiLocus s = st[l];
      if (s.state != GI_LT && s.state != GI_LE) continue;
      if (s.state == GI_LT && s.bits == 0) continue;
      const uint32_t kl = lkey[l];
      h0 |= (uint32_t)gi_carrier(gi_key(id, 0, kl), s) << j;
      h1 |= (uint32_t)gi_carrier(gi_key(id, 1, kl), s) << j;
    }
    uint32_t* row = G + (size_t)pop.gslot[cur][i] * 2 * Ww;
    row[w] = h0;
    row[Ww + w] = h1;
  }
}

// (site, id, homologue) of every carrier at every locus, placed at off[site] + a per-site cursor
__global__ void __launch_bounds__(256) k_gi_rows(Pop pop, const Counters* c, const GiLocus* __restrict__ st,
                                                 const uint32_t* __restrict__ lkey, const long long* __restrict__ off,
                                                 unsigned long long* cursor, int32_t* site, long long* id_out,
                                                 int8_t* hom, int L) {
  const int n = c->n, cur = c->cur, Wl = (L + 31) / 32;
  const long long total = (long long)n * Wl;
  for (long long k = GTID; k < total; k += GSTRIDE) {
    const int i = (int)(k / Wl), w = (int)(k - (long long)i * Wl);
    const long long id = pop.idx[cur][i];
    for (int j = 0; j < 32; ++j) {
      const int l = 32 * w + j;
      if (l >= L) break;
      const GiLocus s = st[l];
      if (s.state == GI_LT && s.bits == 0) continue;
      for (int h = 0; h < 2; ++h) {
        if (!gi_carrier(gi_key(id, h, lkey[l]), s)) continue;
        const long long r = off[l] + (long long)atomicAdd(&cursor[l], 1ull);
        site[r] = l;
        id_out[r] = id;
        hom[r] = (int8_t)h;
      }
    }
  }
}
