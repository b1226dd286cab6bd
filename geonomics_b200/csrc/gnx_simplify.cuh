// gnx_simplify.cuh -- sort + simplify of a use_tskit species' tables (gnx_simplify), the level-parallel
// form of tables.simplify_columns that reproduces it row for row.
//
// Every position the algorithm compares (edge ends, 0, L) is replaced by its rank among the distinct
// positions, so interval ends are u32 and nothing is ever computed on a double: the output columns are
// copies of input values.  Edges are sorted as TableCollection.sort() does; the runs of equal parent
// time are the levels, youngest first, and every parent of a level reads only the ancestry of nodes
// finished at earlier levels.  Per level:
//   k_simp_count / PieceScan / k_simp_pieces   the pieces of A[child] inside every edge (binary search
//                                              in the child's sorted, disjoint segments), as +1 / -1
//                                              events keyed (parent in level, position)
//   radix sort of the events, k_simp_event_inv
//   CoverScan     running sum of delta * (2^32 + node + 1): its high word is the coverage when that is 0
//                 or 1 and >= 2 otherwise, its low word the covering node when the coverage is 1
//   BoundScan     one elementary interval per last event of a (parent, position) group inside a parent
//   k_simp_flag / ParentScan   a non-sample parent with coverage >= 2 somewhere gets the next output id
//   SegScan       the parent's new ancestry: one segment per covered elementary interval (A[u])
//   k_simp_runs (count) / RunScan / k_simp_runs (write)   output edges: every piece's maximal runs of
//                 intervals with coverage >= 2 (>= 1 under a sample)
// Sizes the host does not know (pieces, events, intervals, runs) live in Simp.sv and are read by the
// kernels; the host enqueues every level without a round trip.  A pool that would overflow sets
// sv[SV_OVF] and makes every later size 0; the host then runs the levels again with larger pools.
#pragma once
#include "gnx_kernels.cuh"

enum { SV_P = 0, SV_NEV, SV_NB, SV_NEWN, SV_NSEG, SV_NRUN, SV_OUT, SV_ATOP, SV_RTOP, SV_OVF, SV_NEED_P,
       SV_NEED_A, SV_NEED_R, SV_N };
// error bits of the input check (k_simp_check_*)
enum { SE_ID = 1, SE_TIME = 2, SE_INTERVAL = 4, SE_IND = 8, SE_SITE = 16, SE_SAMPLE = 32 };

struct Simp {
  // input columns
  int n_in, n_edges, n_ind, n_sites, n_mut, n_samples;
  double L;
  const double* time;
  const int32_t* ind;
  const double* el;
  const double* er;
  const int32_t* ep;
  const int32_t* ec;
  const double* site_pos;
  const int32_t* m_site;
  const int32_t* m_node;
  const int32_t* samples;
  int32_t* smap;          // [n_in] sample index, -1 for other nodes
  int32_t* err;
  // distinct positions
  double* uniq;
  int32_t* sv;            // [SV_N] device sizes
  int pb;                 // bits of a position rank
  // sorted edges: ranks of left / right, parent, child, group (parent) index
  uint32_t* sl;
  uint32_t* sr;
  int32_t* sp;
  int32_t* sc;
  int32_t* grp_of;
  int32_t* grp_parent;
  int32_t* lvl_start;     // [n_levels + 1] first edge of every level
  int32_t* lvl_g0;        // [n_levels + 1] first group of every level
  // ancestry segments: A[u] = pool[a_off[u] .. a_end[u])
  int32_t* a_off;
  int32_t* a_end;
  uint32_t* a_lo;
  uint32_t* a_hi;
  int32_t* a_node;
  int cap_a;
  // per-level scratch
  int cap_p;
  int32_t* pcnt;          // [E_level] pieces of each edge, then their exclusive offsets
  int32_t* pj;            // [E_level] first segment of each edge's pieces
  int32_t* pc_node;       // [cap_p]
  unsigned long long* ev_key[2];
  int32_t* ev_val[2];
  int32_t* inv;           // [2 cap_p] sorted position of every event
  uint32_t* cover;        // [2 cap_p][2] per sorted event: coverage clamped to 2, covering node + 1
  int32_t* bex;           // [2 cap_p] boundaries before every sorted event
  uint32_t* b_pos;
  uint32_t* b_end;
  int32_t* b_cls;         // 0 gap, 1 one piece, 2 coalescence
  int32_t* b_node;
  int32_t* b_g;
  int32_t* flag;          // [G_level]
  int32_t* vout;          // [G_level] output node of every parent of the level (-1: none)
  int32_t* rcnt;          // [cap_p]
  // output
  int32_t* out_src;       // [n_samples + n_in] input node of every output node
  uint32_t* r_lo;
  uint32_t* r_hi;
  int32_t* r_par;
  int32_t* r_child;
  int cap_r;
};

__device__ __forceinline__ unsigned long long time_key(double t) {
  // order-preserving bits of a double; -0.0 and 0.0 compare equal and must tie
  const unsigned long long b = (unsigned long long)__double_as_longlong(t == 0.0 ? 0.0 : t);
  return (b >> 63) ? ~b : (b | (1ull << 63));
}

// first index in [lo, hi) with a[i] >= x
template <class T>
__device__ __forceinline__ int lower_bound_dev(const T* a, int lo, int hi, T x) {
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (a[m] < x) lo = m + 1; else hi = m;
  }
  return lo;
}

__global__ void __launch_bounds__(256) k_simp_check_edges(Simp S) {
  for (int e = GTID; e < S.n_edges; e += GSTRIDE) {
    const int p = S.ep[e], c = S.ec[e];
    const double l = S.el[e], r = S.er[e];
    int bad = 0;
    if (p < 0 || p >= S.n_in || c < 0 || c >= S.n_in) bad |= SE_ID;
    else if (!(S.time[p] > S.time[c])) bad |= SE_TIME;
    if (!(l >= 0.0 && l < r && r <= S.L) || signbit(l)) bad |= SE_INTERVAL;
    if (bad) atomicOr(S.err, bad);
  }
}

__global__ void __launch_bounds__(256) k_simp_check_rest(Simp S) {
  for (int u = GTID; u < S.n_in; u += GSTRIDE)
    if (S.ind[u] >= S.n_ind) atomicOr(S.err, SE_IND);
  if (S.n_sites > 0)
    for (int m = GTID; m < S.n_mut; m += GSTRIDE)
      if (S.m_site[m] < 0 || S.m_site[m] >= S.n_sites) atomicOr(S.err, SE_SITE);
  for (int i = GTID; i < S.n_samples; i += GSTRIDE) {
    const int s = S.samples[i];
    if (s < 0 || s >= S.n_in) { atomicOr(S.err, SE_SAMPLE); continue; }
    if (atomicCAS(&S.smap[s], -1, i) != -1) atomicOr(S.err, SE_SAMPLE);
  }
}

// every edge end, 0 and L, as the bits of a non-negative double (order-preserving)
__global__ void __launch_bounds__(256) k_simp_pos_keys(Simp S, unsigned long long* key) {
  const int n = S.n_edges;
  for (int e = GTID; e < n; e += GSTRIDE) {
    key[2 * e] = (unsigned long long)__double_as_longlong(S.el[e]);
    key[2 * e + 1] = (unsigned long long)__double_as_longlong(S.er[e]);
  }
  if (GTID == 0) {
    key[2 * n] = 0ull;
    key[2 * n + 1] = (unsigned long long)__double_as_longlong(S.L);
  }
}

struct UniqScan {
  const unsigned long long* key;
  double* uniq;
  int32_t* n_uniq;
  int n;
  __device__ int size(const Counters*) const { return n; }
  __device__ u64 value(int i) const { return (i == 0 || key[i] != key[i - 1]) ? 1u : 0u; }
  __device__ void apply(int i, u64 v, u64 ex) const { if (v) uniq[ex] = __longlong_as_double((long long)key[i]); }
  __device__ void total(Counters*, u64 t) const { *n_uniq = (int)t; }
};

// ranks of both ends; first sort key (child, left rank), value = edge
__global__ void __launch_bounds__(256) k_simp_edge_keys(Simp S, int n_uniq, uint32_t* lr, uint32_t* rr,
                                                       unsigned long long* key, int32_t* val) {
  for (int e = GTID; e < S.n_edges; e += GSTRIDE) {
    const uint32_t l = (uint32_t)lower_bound_dev(S.uniq, 0, n_uniq, S.el[e]);
    lr[e] = l;
    rr[e] = (uint32_t)lower_bound_dev(S.uniq, 0, n_uniq, S.er[e]);
    key[e] = ((unsigned long long)S.ec[e] << S.pb) | l;
    val[e] = e;
  }
}

__global__ void __launch_bounds__(256) k_simp_time_keys(const double* time, const int32_t* src, int n,
                                                       unsigned long long* key, int32_t* val) {
  for (int u = GTID; u < n; u += GSTRIDE) {
    key[u] = time_key(time[src ? src[u] : u]);
    val[u] = u;
  }
}

__global__ void __launch_bounds__(256) k_simp_rank(const int32_t* val, int n, int32_t* rank) {
  for (int i = GTID; i < n; i += GSTRIDE) rank[val[i]] = i;
}

// second sort key of the edges: rank of the parent in (time, id) order
__global__ void __launch_bounds__(256) k_simp_edge_keys2(Simp S, const int32_t* prank, const int32_t* val,
                                                        unsigned long long* key) {
  for (int i = GTID; i < S.n_edges; i += GSTRIDE) key[i] = (unsigned long long)prank[S.ep[val[i]]];
}

__global__ void __launch_bounds__(256) k_simp_edge_gather(Simp S, const int32_t* val, const uint32_t* lr,
                                                         const uint32_t* rr) {
  for (int i = GTID; i < S.n_edges; i += GSTRIDE) {
    const int e = val[i];
    S.sl[i] = lr[e];
    S.sr[i] = rr[e];
    S.sp[i] = S.ep[e];
    S.sc[i] = S.ec[e];
  }
}

// groups (runs of one parent) and levels (runs of one parent time) of the sorted edges, as a packed
// (level starts, group starts) scan
struct LevelScan {
  Simp S;
  int32_t* n_out;   // [2]: levels, groups
  __device__ int size(const Counters*) const { return S.n_edges; }
  __device__ u64 value(int i) const {
    if (i == 0) return (1ull << 32) | 1ull;
    const int p = S.sp[i], q = S.sp[i - 1];
    return ((u64)(S.time[p] != S.time[q]) << 32) | (u64)(p != q);
  }
  __device__ void apply(int i, u64 v, u64 ex) const {
    const u64 inc = ex + v;
    const int g = (int)(inc & 0xffffffffu) - 1, k = (int)(inc >> 32) - 1;
    S.grp_of[i] = g;
    if (v & 1u) S.grp_parent[g] = S.sp[i];
    if (v >> 32) {
      S.lvl_start[k] = i;
      S.lvl_g0[k] = g;
    }
  }
  __device__ void total(Counters*, u64 t) const {
    const int nl = (int)(t >> 32), ng = (int)(t & 0xffffffffu);
    n_out[0] = nl;
    n_out[1] = ng;
    S.lvl_start[nl] = S.n_edges;
    S.lvl_g0[nl] = ng;
  }
};

// the samples' ancestry: [0, L) on their own output node
__global__ void __launch_bounds__(256) k_simp_init_samples(Simp S, uint32_t L_rank) {
  for (int i = GTID; i < S.n_samples; i += GSTRIDE) {
    const int s = S.samples[i];
    S.a_lo[i] = 0u;
    S.a_hi[i] = L_rank;
    S.a_node[i] = i;
    S.a_off[s] = i;
    S.a_end[s] = i + 1;
    S.out_src[i] = s;
  }
  if (GTID == 0) {
    S.sv[SV_OUT] = S.n_samples;
    S.sv[SV_ATOP] = S.n_samples;
  }
}

// ---- one level: edges [e0, e0 + ne), groups [g0, g0 + ng) -----------------------------------------
__global__ void __launch_bounds__(256) k_simp_count(Simp S, int e0, int ne) {
  for (int j = GTID; j < ne; j += GSTRIDE) {
    const int e = e0 + j, c = S.sc[e];
    const int lo = S.a_off[c], hi = S.a_end[c];
    const uint32_t l = S.sl[e], r = S.sr[e];
    const int a = lower_bound_dev(S.a_hi, lo, hi, l + 1u);   // first segment ending after l
    const int b = lower_bound_dev(S.a_lo, a, hi, r);        // first segment starting at or after r
    S.pcnt[j] = b - a;
    S.pj[j] = a;
  }
}

struct PieceScan {
  Simp S;
  int ne;
  __device__ int size(const Counters*) const { return ne; }
  __device__ u64 value(int j) const { return (u64)S.pcnt[j]; }
  __device__ void apply(int j, u64, u64 ex) const { S.pcnt[j] = (int)ex; }
  __device__ void total(Counters*, u64 t) const {
    int P = (int)t;
    if (S.sv[SV_OVF] || t > (u64)S.cap_p) {
      if (t > (u64)S.cap_p) S.sv[SV_NEED_P] = max(S.sv[SV_NEED_P], (int)min(t, (u64)INT32_MAX));
      S.sv[SV_OVF] = 1;
      P = 0;
    }
    S.sv[SV_P] = P;
    S.sv[SV_NEV] = 2 * P;
  }
};

__global__ void __launch_bounds__(256) k_simp_pieces(Simp S, int e0, int ne, int g0) {
  const int P = S.sv[SV_P];
  for (int q = GTID; q < P; q += GSTRIDE) {
    // the edge: last j with pcnt[j] (exclusive offset) <= q
    int lo = 0, hi = ne;
    while (hi - lo > 1) {
      const int m = (lo + hi) >> 1;
      if (S.pcnt[m] <= q) lo = m; else hi = m;
    }
    const int e = e0 + lo, s = S.pj[lo] + (q - S.pcnt[lo]);
    const uint32_t a = max(S.a_lo[s], S.sl[e]), b = min(S.a_hi[s], S.sr[e]);
    const unsigned long long g = (unsigned long long)(S.grp_of[e] - g0) << S.pb;
    S.pc_node[q] = S.a_node[s];
    S.ev_key[0][2 * q] = g | a;
    S.ev_key[0][2 * q + 1] = g | b;
    S.ev_val[0][2 * q] = 2 * q;
    S.ev_val[0][2 * q + 1] = 2 * q + 1;
  }
}

__global__ void __launch_bounds__(256) k_simp_event_inv(Simp S, const int32_t* val) {
  const int n = S.sv[SV_NEV];
  for (int i = GTID; i < n; i += GSTRIDE) S.inv[val[i]] = i;
}

struct CoverScan {
  Simp S;
  const int32_t* val;
  __device__ int size(const Counters*) const { return S.sv[SV_NEV]; }
  __device__ u64 value(int i) const {
    const int ev = val[i];
    const u64 w = (1ull << 32) + (u64)(S.pc_node[ev >> 1] + 1);
    return (ev & 1) ? (u64)0 - w : w;
  }
  __device__ void apply(int i, u64 v, u64 ex) const {
    const u64 inc = ex + v;
    const u64 hi = min(inc >> 32, (u64)2);
    S.cover[2 * i] = (uint32_t)hi;
    S.cover[2 * i + 1] = (uint32_t)(inc & 0xffffffffu);
  }
  __device__ void total(Counters*, u64) const {}
};

struct BoundScan {
  Simp S;
  const unsigned long long* key;
  __device__ int size(const Counters*) const { return S.sv[SV_NEV]; }
  __device__ bool boundary(int i) const {
    if (i + 1 >= S.sv[SV_NEV]) return false;
    const unsigned long long k0 = key[i], k1 = key[i + 1];
    return k0 != k1 && (k0 >> S.pb) == (k1 >> S.pb);
  }
  __device__ u64 value(int i) const { return boundary(i) ? 1u : 0u; }
  __device__ void apply(int i, u64 v, u64 ex) const {
    S.bex[i] = (int)ex;
    if (!v) return;
    const unsigned long long mask = (1ull << S.pb) - 1ull;
    S.b_pos[ex] = (uint32_t)(key[i] & mask);
    S.b_end[ex] = (uint32_t)(key[i + 1] & mask);
    S.b_g[ex] = (int)(key[i] >> S.pb);
    const int cls = (int)S.cover[2 * i];
    S.b_cls[ex] = cls;
    S.b_node[ex] = cls == 1 ? (int)S.cover[2 * i + 1] - 1 : -1;
  }
  __device__ void total(Counters*, u64 t) const { S.sv[SV_NB] = (int)t; }
};

__global__ void __launch_bounds__(256) k_simp_flag(Simp S) {
  const int nb = S.sv[SV_NB];
  for (int k = GTID; k < nb; k += GSTRIDE)
    if (S.b_cls[k] == 2) S.flag[S.b_g[k]] = 1;
}

// output ids of the level's coalescing non-sample parents, in parent-id order, after the last one handed out
struct ParentScan {
  Simp S;
  int g0, ng;
  __device__ int size(const Counters*) const { return ng; }
  __device__ u64 value(int g) const { return (S.flag[g] && S.smap[S.grp_parent[g0 + g]] < 0) ? 1u : 0u; }
  __device__ void apply(int g, u64 v, u64 ex) const {
    const int u = S.grp_parent[g0 + g], s = S.smap[u];
    const int id = S.sv[SV_OUT] + (int)ex;
    S.vout[g] = s >= 0 ? s : (v ? id : -1);
    if (v) S.out_src[id] = u;
  }
  __device__ void total(Counters*, u64 t) const { S.sv[SV_NEWN] = (int)t; }
};

// A[u] of every non-sample parent: its covered elementary intervals, on the covering piece's node
// (coverage 1) or on the parent's output node (coverage >= 2)
struct SegScan {
  Simp S;
  int g0;
  __device__ int size(const Counters*) const { return S.sv[SV_NB]; }
  __device__ bool own(int k) const { return S.smap[S.grp_parent[g0 + S.b_g[k]]] < 0; }
  __device__ u64 value(int k) const { return (own(k) && S.b_cls[k] >= 1) ? 1u : 0u; }
  __device__ void apply(int k, u64 v, u64 ex) const {
    if (S.sv[SV_OVF] || !own(k)) return;
    const int g = S.b_g[k], u = S.grp_parent[g0 + g], nb = S.sv[SV_NB];
    const int at = S.sv[SV_ATOP] + (int)ex;
    if (v) {
      S.a_lo[at] = S.b_pos[k];
      S.a_hi[at] = S.b_end[k];
      S.a_node[at] = S.b_cls[k] == 1 ? S.b_node[k] : S.vout[g];
    }
    if (k == 0 || S.b_g[k - 1] != g) S.a_off[u] = at;
    if (k == nb - 1 || S.b_g[k + 1] != g) S.a_end[u] = at + (int)v;
  }
  __device__ void total(Counters*, u64 t) const {
    const u64 need = (u64)S.sv[SV_ATOP] + t;
    if (need > (u64)S.cap_a) {
      S.sv[SV_NEED_A] = max(S.sv[SV_NEED_A], (int)min(need, (u64)INT32_MAX));
      S.sv[SV_OVF] = 1;
    }
    S.sv[SV_NSEG] = S.sv[SV_OVF] ? 0 : (int)t;
  }
};

// every piece's maximal runs of elementary intervals with coverage >= 2 (>= 1 under a sample):
// counted (write = false) or written at the piece's offset (write = true)
__global__ void __launch_bounds__(256) k_simp_runs(Simp S, int g0, bool write) {
  const int P = S.sv[SV_P];
  const int base = write ? S.sv[SV_RTOP] : 0;
  for (int q = GTID; q < P; q += GSTRIDE) {
    const int a = S.bex[S.inv[2 * q]], b = S.bex[S.inv[2 * q + 1]];
    const int g = S.b_g[a];
    const int thr = S.smap[S.grp_parent[g0 + g]] >= 0 ? 1 : 2;
    int n = 0, at = write ? base + S.rcnt[q] : 0;
    bool in = false;
    for (int k = a; k < b; ++k) {
      const bool ok = S.b_cls[k] >= thr;
      if (ok && !in) {
        if (write) {
          S.r_lo[at] = S.b_pos[k];
          S.r_par[at] = S.vout[g];
          S.r_child[at] = S.pc_node[q];
        }
        ++n;
      }
      if (!ok && in && write) S.r_hi[at++] = S.b_pos[k];
      in = ok;
    }
    if (in && write) S.r_hi[at] = S.b_end[b - 1];
    if (!write) S.rcnt[q] = n;
  }
}

struct RunScan {
  Simp S;
  __device__ int size(const Counters*) const { return S.sv[SV_P]; }
  __device__ u64 value(int q) const { return (u64)S.rcnt[q]; }
  __device__ void apply(int q, u64, u64 ex) const { S.rcnt[q] = (int)ex; }
  __device__ void total(Counters*, u64 t) const {
    const u64 need = (u64)S.sv[SV_RTOP] + t;
    if (need > (u64)S.cap_r) {
      S.sv[SV_NEED_R] = max(S.sv[SV_NEED_R], (int)min(need, (u64)INT32_MAX));
      S.sv[SV_OVF] = 1;
    }
    if (S.sv[SV_OVF]) S.sv[SV_P] = 0;     // k_simp_runs writes nothing
    S.sv[SV_NRUN] = S.sv[SV_OVF] ? 0 : (int)t;
  }
};

__global__ void __launch_bounds__(32) k_simp_level_end(Simp S) {
  if (threadIdx.x != 0) return;
  S.sv[SV_OUT] += S.sv[SV_NEWN];
  S.sv[SV_ATOP] += S.sv[SV_NSEG];
  S.sv[SV_RTOP] += S.sv[SV_NRUN];
}

// ---- after the last level ---------------------------------------------------------------------------
// mutations: the output node carrying the ancestry of their node at the site (-1: dropped)
struct MutScan {
  Simp S;
  const double* m_time;
  int32_t* o_site;
  int32_t* o_node;
  double* o_time;
  int32_t* n_out;
  __device__ int size(const Counters*) const { return S.n_mut; }
  __device__ int find(int m) const {
    const int u = S.m_node[m];
    if (u < 0 || u >= S.n_in) return -1;
    const int lo = S.a_off[u], hi = S.a_end[u];
    if (lo >= hi) return -1;
    const int site = S.m_site[m];
    const double x = S.n_sites ? S.site_pos[site] : (double)site;
    int a = lo, b = hi;                          // last segment whose left end is <= x
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (S.uniq[S.a_lo[mid]] <= x) a = mid + 1; else b = mid;
    }
    if (a == lo) return -1;
    return x < S.uniq[S.a_hi[a - 1]] ? S.a_node[a - 1] : -1;
  }
  __device__ u64 value(int m) const { return find(m) >= 0 ? 1u : 0u; }
  __device__ void apply(int m, u64 v, u64 ex) const {
    if (!v) return;
    o_site[ex] = S.m_site[m];
    o_node[ex] = find(m);
    o_time[ex] = m_time[m];
  }
  __device__ void total(Counters*, u64 t) const { *n_out = (int)t; }
};

__global__ void __launch_bounds__(256) k_simp_mark_ind(Simp S, int n_out, int32_t* used) {
  for (int o = GTID; o < n_out; o += GSTRIDE) {
    const int i = S.ind[S.out_src[o]];
    if (i >= 0) used[i] = 1;
  }
}

// individuals: the referenced rows in their order, and each row's new index
struct IndScan {
  int n_ind, n_loc;
  int32_t* used;                     // in: referenced; out: new index (or -1)
  const int32_t* flags;
  const double* loc;
  const int64_t* idx;
  int32_t* o_flags;
  double* o_loc;
  int64_t* o_idx;
  int32_t* n_out;
  __device__ int size(const Counters*) const { return n_ind; }
  __device__ u64 value(int i) const { return used[i] ? 1u : 0u; }
  __device__ void apply(int i, u64 v, u64 ex) const {
    used[i] = v ? (int)ex : -1;
    if (!v) return;
    o_flags[ex] = flags[i];
    o_idx[ex] = idx[i];
    for (int k = 0; k < n_loc; ++k) o_loc[ex * n_loc + k] = loc[(size_t)i * n_loc + k];
  }
  __device__ void total(Counters*, u64 t) const { *n_out = (int)t; }
};

__global__ void __launch_bounds__(256) k_simp_nodes_out(Simp S, int n_out, const int32_t* pop, const int32_t* remap,
                                                       int32_t* o_flags, double* o_time, int32_t* o_pop,
                                                       int32_t* o_ind) {
  for (int o = GTID; o < n_out; o += GSTRIDE) {
    const int u = S.out_src[o], i = S.ind[u];
    o_flags[o] = o < S.n_samples ? 1 : 0;
    o_time[o] = S.time[u];
    o_pop[o] = pop[u];
    o_ind[o] = i >= 0 ? remap[i] : -1;
  }
}

// final edge order (time of the output parent, parent, child, left): first key (child, left rank)
__global__ void __launch_bounds__(256) k_simp_run_keys(Simp S, int nr, unsigned long long* key, int32_t* val) {
  for (int i = GTID; i < nr; i += GSTRIDE) {
    key[i] = ((unsigned long long)S.r_child[i] << S.pb) | S.r_lo[i];
    val[i] = i;
  }
}

__global__ void __launch_bounds__(256) k_simp_run_keys2(Simp S, int nr, const int32_t* orank, const int32_t* val,
                                                       unsigned long long* key) {
  for (int i = GTID; i < nr; i += GSTRIDE) key[i] = (unsigned long long)orank[S.r_par[val[i]]];
}

// squash: runs of one (parent, child) that abut become one edge
struct SquashScan {
  Simp S;
  int nr;
  const int32_t* val;
  double* o_l;
  double* o_r;
  int32_t* o_p;
  int32_t* o_c;
  int32_t* n_out;
  __device__ int size(const Counters*) const { return nr; }
  __device__ bool start(int i) const {
    if (i == 0) return true;
    const int a = val[i - 1], b = val[i];
    return S.r_par[a] != S.r_par[b] || S.r_child[a] != S.r_child[b] || S.r_hi[a] != S.r_lo[b];
  }
  __device__ u64 value(int i) const { return start(i) ? 1u : 0u; }
  __device__ void apply(int i, u64 v, u64 ex) const {
    const int at = (int)(ex + v) - 1, r = val[i];
    if (v) {
      o_l[at] = S.uniq[S.r_lo[r]];
      o_p[at] = S.r_par[r];
      o_c[at] = S.r_child[r];
    }
    if (i == nr - 1 || start(i + 1)) o_r[at] = S.uniq[S.r_hi[r]];
  }
  __device__ void total(Counters*, u64 t) const { *n_out = (int)t; }
};
