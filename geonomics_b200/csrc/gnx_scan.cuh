// gnx_scan.cuh -- device-wide exclusive scan of packed (hi, lo) u32 pairs, sized from
// device-resident counters (no host round trip).  Two launches: per-tile reduce (whose last
// block also scans the tile sums), per-tile apply.  The functor supplies:
//   int  size(const Counters*)                     number of elements
//   u64  value(int i)                              packed (hi << 32 | lo) contribution
//   void apply(int i, u64 value, u64 exclusive)    consume the exclusive prefix
//   void total(Counters*, u64 total)               called once by the spine
// Optional:
//   u64  value_first(int i)                        used by the reduce pass instead of value()
//                                                  (e.g. to cache an expensive predicate)
//   static constexpr bool BATCHED = true; void apply_batch(const int* i, const u64* v,
//        const u64* ex, int n)                     consume SCAN_ITEMS elements at once, so the
//                                                  functor can issue all loads before any store
#pragma once
#include <type_traits>
#include "gnx_common.cuh"

#define SCAN_BLOCK 256
#define SCAN_ITEMS 4
#define SCAN_TILE (SCAN_BLOCK * SCAN_ITEMS)

typedef unsigned long long u64;

__device__ __forceinline__ u64 warp_incl_scan(u64 v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u64 o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += o;
  }
  return v;
}

// exclusive scan across the block of one value per thread; returns exclusive prefix and the
// block total through *total.
__device__ __forceinline__ u64 block_excl_scan(u64 v, u64* total) {
  __shared__ u64 warp_tot[SCAN_BLOCK / 32];
  __shared__ u64 blk_tot;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  u64 inc = warp_incl_scan(v);
  if (lane == 31) warp_tot[w] = inc;
  __syncthreads();
  if (w == 0) {
    u64 t = lane < SCAN_BLOCK / 32 ? warp_tot[lane] : 0;
    u64 ti = warp_incl_scan(t);
    if (lane < SCAN_BLOCK / 32) warp_tot[lane] = ti - t;
    if (lane == SCAN_BLOCK / 32 - 1) blk_tot = ti;
  }
  __syncthreads();
  u64 excl = inc - v + warp_tot[w];
  *total = blk_tot;
  __syncthreads();
  return excl;
}

template <class F, class = void>
struct scan_has_value_first : std::false_type {};
template <class F>
struct scan_has_value_first<F, std::void_t<decltype(std::declval<const F&>().value_first(0))>> : std::true_type {};
template <class F, class = void>
struct scan_is_batched : std::false_type {};
template <class F>
struct scan_is_batched<F, std::void_t<decltype(F::BATCHED)>> : std::true_type {};

template <class F>
__device__ __forceinline__ u64 scan_value_first(const F& f, int i) {
  if constexpr (scan_has_value_first<F>::value) return f.value_first(i);
  else return f.value(i);
}

// Pass 1: per-tile sums; the LAST block to finish (atomic ticket, no spinning) also runs the
// spine -- an exclusive scan of the tile sums by one CTA -- and hands the grand total to the
// functor.  That saves the separate single-CTA launch between reduce and apply.
template <class F>
__global__ void __launch_bounds__(SCAN_BLOCK) scan_reduce_kernel(F f, Counters* c, u64* tile_sums,
                                                                 unsigned int* ticket) {
  const int n = f.size(c);
  const int ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    // striped: consecutive threads touch consecutive elements (coalesced)
    const int base = tile * SCAN_TILE + threadIdx.x;
    u64 s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k)
      if (base + k * SCAN_BLOCK < n) s += scan_value_first(f, base + k * SCAN_BLOCK);
    u64 tot;
    block_excl_scan(s, &tot);
    if (threadIdx.x == 0) tile_sums[tile] = tot;
  }
  __shared__ bool is_last;
  __threadfence();
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  u64 carry = 0;
  for (int base = 0; base < ntiles; base += SCAN_BLOCK) {
    const int i = base + threadIdx.x;
    u64 v = i < ntiles ? __ldcg(&tile_sums[i]) : 0;
    u64 tot;
    u64 ex = block_excl_scan(v, &tot);
    if (i < ntiles) tile_sums[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) {
    f.total(c, carry);
    *ticket = 0u;              // ready for the next scan on this stream
  }
}

constexpr int SCAN_MINB = 3;   // 80 registers: measured best of 1, 3, 4, 5 CTAs per SM
template <class F>
__global__ void __launch_bounds__(SCAN_BLOCK, SCAN_MINB) scan_apply_kernel(F f, const Counters* c, const u64* tile_sums) {
  const int n = f.size(c);
  const int ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    // striped rows of SCAN_BLOCK consecutive elements; one block scan per row
    const int base = tile * SCAN_TILE + threadIdx.x;
    u64 v[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) v[k] = (base + k * SCAN_BLOCK < n) ? f.value(base + k * SCAN_BLOCK) : 0;
    u64 carry = tile_sums[tile];
    u64 ex[SCAN_ITEMS];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
      u64 tot;
      ex[k] = block_excl_scan(v[k], &tot) + carry;
      carry += tot;
    }
    // all prefixes first, then all payload moves: the loads of the SCAN_ITEMS elements
    // overlap instead of queueing behind the barriers of the next row's scan
    if constexpr (scan_is_batched<F>::value) {
      int idx[SCAN_ITEMS];
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k) idx[k] = base + k * SCAN_BLOCK;
      f.apply_batch(idx, v, ex, n);
    } else {
#pragma unroll
      for (int k = 0; k < SCAN_ITEMS; ++k)
        if (base + k * SCAN_BLOCK < n) f.apply(base + k * SCAN_BLOCK, v[k], ex[k]);
    }
  }
}
