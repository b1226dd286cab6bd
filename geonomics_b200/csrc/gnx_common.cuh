// gnx_common.cuh -- device-side data layout, Philox RNG and distribution samplers.
// Part of libgnxb200.so (sm_100a).  See DESIGN.md for the HBM layout.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <math.h>
#include "../../include/gnx_b200.h"

#define GNX_PI 3.14159265358979323846

// ----------------------------------------------------------------------------------------
// device-resident step counters (one per ctx).  Kernels read sizes from here so a whole
// time step runs without a host round trip.
// ----------------------------------------------------------------------------------------
struct Counters {
  int32_t n;         // entries of the current half at stage entry (all alive unless `pending`)
  int32_t n_pre;     // n + B: individuals alive before mortality
  int32_t P;         // mating pairs this step
  int32_t B;         // births this step
  int32_t deaths;    // deaths this step
  int32_t n_free;    // genome-slot free-list length
  int32_t n_slots;   // genome-slot high-water mark
  int32_t cur;       // which half of the double-buffered scalar SoA is current
  int64_t max_idx;   // species.py:360 max_ind_idx
  int64_t t;         // time-step counter (Philox counter word)
  int32_t err;       // sticky error bits (GNX_ERRBIT_*)
  int32_t n_rec;     // per-step records written
  int32_t gs_iters[2];
  unsigned long long nmax_bits;   // bits of max(N raster) (N >= 0 so unsigned order works)
  int32_t pad[2];
  // tskit record buffering (a18)
  int32_t n_nodes;      // next row id of the tskit nodes table
  int32_t n_ind_rows;   // next row id of the tskit individuals table
  int32_t n_edges;      // edge rows buffered since the last drain
  int32_t n_born;       // newborn (individual + 2 node) rows buffered since the last drain
  int64_t tsk_t0;       // Counters.t when recording was enabled (node time = -(t - tsk_t0))
  // mating-grid order + lazy mortality (DESIGN.md section 3)
  int32_t n_sorted;     // leading entries in (mating cell, id) order with cell_start valid for them
  int32_t pending;      // 1: the last step's deaths are only flagged (w.alive); the next re-grid drops them
  int32_t n_alive;      // survivors of the last step (valid while pending)
  int32_t alive_acc;    // accumulator of k_death's survivor count (zeroed by its last block)
  uint32_t ticket[2];   // last-block elections (k_regrid, k_death); self-resetting
  int32_t n_regrid;     // entries placed by the running re-grid (scan total)
  int32_t pad2;
  // crowded mating cells handed from k_find_mates to k_find_mates_dense (zeroed before every search)
  int32_t n_heavy;      // cells appended to Work.heavy
  int32_t heavy_next;   // work-stealing cursor of k_find_mates_dense
  // strip domain decomposition (gnx_strip.cuh): the entries [own_lo, own_hi) of the grid-ordered
  // half belong to this rank, the rest are ghosts of the neighbouring strips (whole range when
  // the landscape is not decomposed)
  int32_t own_lo, own_hi;
  int32_t tail_sent;    // newborns of this step shipped to the strip they dispersed into
  int32_t pad3;
  int64_t max_idx_global;   // species-wide max_ind_idx while Counters.max_idx carries this rank's id base
  // set by k_strip_id_base for the rest of the step (k_mutate replays the species-wide mutation draws)
  int64_t max_idx_base;     // species-wide max_ind_idx at the start of the step
  int32_t births_lo;        // births of the lower ranks: offspring number of this rank's first newborn
  int32_t births_all;       // births of the species
  int32_t dens_lists[2];    // fix-list and deferred-list lengths of the last density evaluation (k_raster_fix_d)
};
#define GNX_ERRBIT_CAPACITY 1
#define GNX_ERRBIT_DRAWS 2
#define GNX_ERRBIT_GS 4
#define GNX_ERRBIT_MUTABLES 8     // _mutables.pop() on an empty list
#define GNX_ERRBIT_MUTLOG 16      // mutation log full (rows dropped, bookkeeping still exact)
#define GNX_ERRBIT_MUTIDX 32      // a stale loci_idxs / delet_loci_idxs entry addresses a row that does not exist
                                  // (IndexError in the reference)

// Double-buffered scalar SoA + slot-indexed genome rows.  The order of the entries is the
// MATING-GRID order (cell key, then individual id) established by the re-grid of every step;
// species order (ascending id = the reference's OrderedDict order) is materialised only when
// the host reads the population (k_species_gather).
struct Pop {
  double2* xy[2];      // (x, y) interleaved: always used together, and one 16-byte gather
                       // costs one DRAM burst where two 8-byte gathers cost two
  int32_t* age[2];
  int8_t* sex[2];
  int64_t* idx[2];
  int32_t* gslot[2];
  double* z[2];        // [T][cap]
  double* fit[2];
  int32_t* node[2][2]; // [homologue][buffer][cap] tskit node ids (NULL unless recording)
  int32_t* ord[2];     // species-order ordinal of every entry (ordered mode: injected draws / debug reads)
  uint4* G;            // [cap][2][Wq]
  int32_t* free_slots; // [cap]
  int32_t cap;
  int32_t Wq;          // 128-bit units per homologue
  int32_t T;
};

struct Traits {
  // merged trait-locus table sorted by (trait, locus); entries of trait t for 128-bit
  // unit q are [chunk_ptr[t*(Wq+1)+q], chunk_ptr[t*(Wq+1)+q+1])
  const int32_t* te_locus;
  const double* te_alpha;
  const double* te_dom;        // (1 + dom[locus]) factor, or NULL
  const void* te_pack;         // per entry {int32 byte offset of the staged word pair, uint32 bit mask, f64 alpha/2}
  const int32_t* chunk_ptr;
  int32_t n_loci[GNX_MAX_TRAITS];
  const int32_t* n_loci_dev;   // non-NULL once mutation owns the tables (trait mutation / tskit layout): the
                               // loci counts live on the device and grow inside the graph-launched step
  double phi[GNX_MAX_TRAITS];
  const double* phi_rast[GNX_MAX_TRAITS];
  double gamma[GNX_MAX_TRAITS];
  int32_t layer[GNX_MAX_TRAITS];
  int32_t univ_adv[GNX_MAX_TRAITS];
};

struct Land {
  const double* rasters;   // [n_layers][Y][X]
  const double* K;         // [Y][X]
  const float* surf_f32[2]; // float32 copies of the movement / dispersal conductance layers
                            // (on-the-fly surface mode only; half the footprint, L2-resident)
  int32_t X, Y, n_layers;
  double max_x, max_y;     // dim - 0.001 (movement.py:89-92)
  // mating grid
  double cell_size, inv_cell_size;   // inv_cell_size = fl(1 / cell_size), see cell_index
  int32_t ncx, ncy;
};

struct Dens {
  double ww, hww;
  int32_t half_index_ok;   // hww is a multiple of 2^-20: grid cells from one half-window index per axis
  int32_t npts, ntri;
  const double* points;    // [npts][2] (i, j)
  const double* areas;
  int32_t g_ni[4], g_nj[4], g_i0[4], g_j0[4], g_xe[4], g_ye[4], g_off[4];
  const int32_t* simplices;
  const int32_t* neighbors;
  const int32_t* nbr_indptr;
  const int32_t* nbr_indices;
  const double* e_ex;      // per CSR entry: edge vector and ex/L^3, ey/L^3
  const double* e_ey;
  const double* e_wx;
  const double* e_wy;
  const double* v_inv;     // [npts][3] inverse of the per-vertex 2x2 system (i00, i01, i11)
  const int32_t* p_j;      // [8][npts] neighbours padded with self (transposed)
  const double* p_e;       // [8][4][npts] (ex, ey, ex/L^3, ey/L^3), padded with zeros (transposed)
  const double* v_inv_t;   // [3][npts]
  int32_t padded;          // every vertex has <= 8 neighbours
  int32_t lat_ni, lat_nj;
  const int32_t* square_tri;
  const double* tri_aff;   // [ntri][6]: b0 = a0 + a1*qi + a2*qj, b1 = a3 + a4*qi + a5*qj
  const double* tri_g;     // [ntri][3]: static Clough-Tocher neighbour weights (k_ct_setup_g)
  int32_t colourable;
  // work
  int32_t* counts;   // [2][npts]
  double* vals;      // [2][npts]
  double* grad;      // [2][npts][2]
  double* coef;      // [2][ntri][3][10] monomial coefficients per micro-triangle
};

struct Work {
  uint32_t* cell_count;
  uint32_t* cell_start;    // [ncell + 1]
  uint32_t* mkey;          // per source entry: packed mating cell (cy << 16 | cx) after movement; GNX_KEY_DEAD = dropped
  uint4* bucket;           // per destination cell range: {source entry, packed cell, id lo, id hi}
  uint32_t* skey;          // packed mating cell of every entry of the current (grid-ordered) half
  int32_t* inv;            // ordered mode: entry of species-order ordinal i
  int32_t* perm;           // panmixia: second parent of slot i
  unsigned long long* sort_keys[2];   // radix sort by id (species order on demand)
  int32_t* sort_vals[2];
  uint32_t* sort_hist;     // [256][tiles]
  int32_t* mate;
  uint2* heavy;            // work items of k_find_mates_dense: {packed key of a crowded mating cell, first focal of a batch of 32}
  int32_t heavy_cap;
  int32_t* fm_list;        // focals whose Bernoulli(b) draw lets them mate (k_mate_select), the only ones searched
  int32_t* fm_count;       // [1]
  int32_t* n_nbrs;
  int32_t* pairs;          // [cap][2]
  int32_t* pair_slots;     // [cap][2] genome slots of each pair's parents
  int32_t* nb;
  int32_t* off_start;
  int32_t* off_pair;
  double2* mid;            // pair midpoints (x, y)
  uint8_t* alive;
  double* death_p;
  int32_t* disp_tries;
  unsigned long long* tile_sums;
  unsigned int* scan_ticket;   // last-block election of scan_reduce_kernel (self-resetting)
  double* N_rast;
  double* NP_rast;
  double* d_rast;
  double* e_out;
  int32_t* fix_list;       // [Y*X]: from the front the cells whose N needs the exact-order re-evaluation,
                           // from the back the cells whose d waits for max(N) (k_raster_Nd)
  int32_t* fix_count;      // [3]: both list lengths and k_raster_fix_d's last-block ticket; reset by that block
  gnx_step_record_t* records;
  int32_t max_records;
  void* scratch;           // species-order staging of one per-individual field (gnx_read_field)
};
#define GNX_KEY_DEAD 0xffffffffu

// tskit record buffers (species.py:692-736): rows accumulated on the device between drains
struct Tsk {
  int32_t enabled;
  const int32_t* bp_ptr;   // [n_paths + 1] CSR of recombination breakpoints per cached path
  const int32_t* bp_pos;   // locus index of each breakpoint (segment edge = pos - 0.5, genome.py:248-249)
  double L;                // sequence length
  int32_t edge_cap, born_cap;
  double* e_left;
  double* e_right;
  int32_t* e_parent;
  int32_t* e_child;
  int64_t* b_idx;          // individuals-table metadata (gnx individual idx)
  double* b_x;
  double* b_y;
  double* b_z;             // [T][born_cap]
  double* b_time;          // nodes-table time = -t
};

// Strip domain decomposition of one landscape over several GPUs (SURVEY.md section 8e-2): this
// rank owns the individuals whose mating-grid row lies in [row0, row1).  Individuals that leave
// are written straight into the owner's receive buffer over NVLink peer memory (or, when the
// ranks are emulated as contexts of one process, the other context's buffer), a slot claimed
// with a system-scope atomic; a stream-ordered collective between the phases is the barrier.
#define GNX_STRIP_MAX_WORLD 16
enum { STRIP_BUF_MIGRANTS = 0, STRIP_BUF_HALO = 1, STRIP_BUF_NEWBORNS = 2, STRIP_BUF_CHOICES = 3, STRIP_N_BUF = 4 };
struct StripPeer {
  unsigned char* buf[STRIP_N_BUF];   // receive buffers of that rank
  int32_t* count[STRIP_N_BUF];       // records claimed in each
  unsigned char* sync;               // that rank's synchronisation page (k_strip_barrier): one slot per writer
};
// layout of a rank's synchronisation page; rank w writes only slot w of every page
#define STRIP_SYNC_FLAGS 0           // uint32[MAX_WORLD]: barrier epoch each rank has reached
#define STRIP_SYNC_BIRTHS 128        // int64[MAX_WORLD]: births of each rank this step
#define STRIP_SYNC_NMAX 256          // uint64[MAX_WORLD]: bits of each rank's max(N)
#define STRIP_SYNC_PAIRS 384         // int64[MAX_WORLD]: pairs of each rank this step (Poisson births)
#define STRIP_SYNC_COUNTS 512        // int32[MAX_WORLD][counts_cap]: each rank's coarse density counts
struct Strip {
  int32_t enabled;
  int32_t rank, world;
  int32_t row0, row1;                // mating-grid rows owned
  int32_t ly0, ly1;                  // landscape rows that cover the strip
  int32_t bounds[GNX_STRIP_MAX_WORLD + 1];   // first mating-grid row of every rank; bounds[world] = ncy
  int32_t rec_bytes;                 // bytes per individual record (header + genome row)
  int32_t cap[STRIP_N_BUF];          // record capacity of each receive buffer
  StripPeer peer[GNX_STRIP_MAX_WORLD];       // peer[rank] = this rank's own buffers
  uint8_t* sent;                     // [cap] tail entries shipped away this step
  int64_t* births;                   // [world] births of every rank this step (all-gathered)
  int64_t* pairs;                    // [world] pairs of every rank this step (all-gathered; Poisson births only)
  // individuals to ship, listed by the kernel that finds them (k_move_key: leavers; k_strip_halo_list:
  // the strip's edge rows; k_strip_newborn_route: newborns that dispersed out), sent by k_strip_send
  int32_t* list_entry;
  int32_t* list_dest;
  int32_t* list_n;                   // [1]
  int32_t list_cap;
  int32_t* err;                      // [1] sticky: bit 0 a receive buffer or the list overflowed, bit 2 a peer never
                                     //     reached a barrier
  uint32_t* epoch;                   // [1] barriers this rank has entered
  int32_t counts_cap;                // ints per rank slot of the counts exchange
};

struct DevDraws {
  int64_t n;
  const double* move_dir;
  const int32_t* move_choice;
  const double* move_dist;
  const uint32_t* mate_R;
  const double* mate_inv_u;
  const double* mate_u;
  const int32_t* poisson;
  const int32_t* recomb_keys;
  const int32_t* start_homs;
  const double* disp_dir;
  const int32_t* disp_choice;
  const double* disp_dist;
  const double* sex_u;
  const double* sex_redraw_u;
  const double* death_u;
  const double* pan_u;
  const uint32_t* pan_R;
  int32_t disp_R;
  int64_t n_mut;
  const int32_t* mut_n;
  const double* mut_type_u;
  const uint32_t* mut_ind_R;
  const double* mut_homol_u;
  const double* mut_s;
  const double* mut_alpha;
};

// a13 mutation bookkeeping (ops/mutation.py; genome.py:416-437, 753-788).  All arrays are device
// resident and edited by the single thread of k_mutate.
struct Mut {
  int32_t enabled;
  int32_t n_types;                 // neutral, deleterious, then one per trait when any Trait.mu > 0
  int32_t tskit_layout;            // use_tskit = True semantics (include/gnx_b200.h)
  int32_t own_tables;              // k_mutate rebuilds the trait tables of `Traits` (tskit layout / trait mutation)
  double mu_tot;                   // genome.py:599-603
  double cdf[2 + GNX_MAX_TRAITS];  // cumulative type probabilities (genome.py:650-663)
  double s_shape, s_scale;         // genome.py:690-693
  double a_mu[GNX_MAX_TRAITS], a_sigma[GNX_MAX_TRAITS], a_max[GNX_MAX_TRAITS];   // genome.py:666-687
  int32_t* mutables;               // popped from the end
  int32_t* nonneut;                // ascending, capacity L + 1
  int32_t* delet_loci;             // ascending, capacity L + 1
  double* delet_s;
  int32_t* delet_idxs;             // gen_arch.delet_loci_idxs as written (tskit layout), else NULL
  int32_t* delet_eff;              // the bit every deleterious entry reads: nonneut[delet_idxs[k]] / delet_loci[k]
  int32_t* counts;                 // [0] n_mutables [1] n_nonneut [2] n_delet [3] n_log [4 + t] n_loci of trait t
  int32_t* t_loci;                 // [T][tcap] Trait.loci (ascending), Trait.alpha, Trait.loci_idxs (as written)
  double* t_alpha;
  int32_t* t_idxs;
  int32_t tcap, T;
  const double* dom1p;             // [L] 1 + dom[locus], or NULL
  int32_t* te_locus;               // writable aliases of the Traits tables (capacity: all entries + n_mutables)
  double* te_alpha;
  double* te_dom;
  int4* te_pack;
  int32_t* chunk_ptr;
  int32_t NW;                      // 32-bit words per homologue
  uint4* paths;                    // cached recombination paths the gamete kernel reads (patched, tskit layout)
  const uint4* paths_orig;         // as simulated: bit l = (#breakpoints <= l) % 2, [n_paths][WqL]
  int32_t n_paths, Wq, WqL;        // 128-bit units per row of `paths` / of `paths_orig`
  // column layout (gnx_create_cols): genotype bit j holds non-neutral locus col_locus[j]; NULL otherwise
  int32_t* col_n;                  // [1] columns in use
  int32_t* col_locus;              // [L]
  int32_t* col_of_locus;           // [L], -1: no column
  int32_t col_cap;                 // columns a row holds (128 * Wq)
  gnx_mutation_row_t* log;
  int32_t log_cap;
  int32_t L;
};
#define GNX_MUT_MAX_NEW 64          // non-neutral mutations per step whose path bits are patched in one launch

struct Params {
  gnx_config_t c;
  double r2;             // mating_radius^2
  int32_t burn;
  int32_t selection;     // fitness enters death probability (species.py:825)
  int32_t n_paths;
  const uint4* paths;    // [n_paths][Wq]
  const __half* move_tab;
  const __half* disp_tab;
  uint32_t seed_lo, seed_hi;
  int32_t store_debug;   // keep n_nbrs / death_p / NP_rast for parity tests
  int32_t ordered;       // per-individual injected draws are indexed by species-order ordinal (pop.ord),
                         // and the pair list is built in ascending focal ordinal (the oracle's canonical order)
  const float* vm_tab[2];  // inverse-CDF tables of von Mises(0, kappa) for the on-the-fly movement / dispersal
                           // surfaces (vonmises_tab in gnx_kernels.cuh), NULL when unused
  const uint32_t* cs_tab;  // [65536] (half cos | half sin << 16) of every float16 direction: numpy's portable
                           // float16 cos/sin (movement.py:75-76 on a float16 direction), built at setup
};

// ----------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter-based: no state in HBM.
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

enum {
  SITE_MOVE = 1, SITE_MATE = 2, SITE_BIRTHS = 3, SITE_GAMETE = 4, SITE_DISP = 5, SITE_SEX = 6,
  SITE_DEATH = 7, SITE_PANMIXIA = 8, SITE_MUTATE = 9
};

// A stream of random words addressed by (seed; entity id, call site, time step).
struct RngStream {
  uint2 key;
  uint4 ctr;
  uint4 out;
  int pos;
  __device__ __forceinline__ RngStream(uint32_t seed_lo, uint32_t seed_hi, int64_t id, int site,
                                       int64_t t) {
    key = make_uint2(seed_lo, seed_hi);
    ctr = make_uint4((uint32_t)id, (uint32_t)((uint64_t)id >> 32) ^ ((uint32_t)site << 24),
                     (uint32_t)t, 0u);
    pos = 4;
    out = make_uint4(0, 0, 0, 0);
  }
  __device__ __forceinline__ uint32_t u32() {
    if (pos == 4) {
      out = philox4x32_10(ctr, key);
      ctr.w += 1;
      pos = 0;
    }
    // the block is consumed as a shift register: no select chain on a dynamic position
    const uint32_t v = out.x;
    out.x = out.y;
    out.y = out.z;
    out.z = out.w;
    pos += 1;
    return v;
  }
  // uniform in [0, 1), 53 bits (same construction as numpy's legacy double)
  __device__ __forceinline__ double uniform() {
    uint32_t a = u32() >> 5, b = u32() >> 6;
    return (a * 67108864.0 + b) / 9007199254740992.0;
  }
  __device__ __forceinline__ double normal() {
    double u1 = 1.0 - uniform();           // (0, 1]
    double u2 = uniform();
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
  }
};

__device__ __forceinline__ uint32_t choose_k(uint32_t R, uint32_t n) { return __umulhi(R, n); }

// numpy legacy_vonmises (Best & Fisher); distributions.c
__device__ inline double sample_vonmises(RngStream& g, double mu, double kappa) {
  if (kappa < 1e-8) return GNX_PI * (2.0 * g.uniform() - 1.0);
  double s;
  if (kappa < 1e-5) {
    s = 1.0 / kappa + kappa;
  } else {
    double r = 1.0 + sqrt(1.0 + 4.0 * kappa * kappa);
    double rho = (r - sqrt(2.0 * r)) / (2.0 * kappa);
    s = (1.0 + rho * rho) / (2.0 * rho);
  }
  double W;
  for (int it = 0; it < 1000; ++it) {
    double U = g.uniform();
    double Z = cospi(U);
    W = (1.0 + s * Z) / (s + Z);
    double Y = kappa * (s - W);
    double V = g.uniform();
    if ((Y * (2.0 - Y) - V >= 0.0) || (log(Y / V) + 1.0 - Y >= 0.0)) break;
  }
  double U = g.uniform();
  double result = acos(W);
  if (U < 0.5) result = -result;
  result += mu;
  bool neg = result < 0.0;
  double mod = fabs(result);
  mod = fmod(mod + GNX_PI, 2.0 * GNX_PI) - GNX_PI;
  if (neg) mod = -mod;
  return mod;
}

// numpy legacy wald (inverse Gaussian), lognormal; scipy levy (loc + scale / Z^2)
__device__ inline double sample_distance(RngStream& g, int distr, double p1, double p2) {
  if (distr == GNX_DISTR_WALD) {
    double mean = p1, scale = p2;
    double mu_2l = mean / (2.0 * scale);
    double Y = g.normal();
    Y = mean * Y * Y;
    double X = mean + mu_2l * (Y - sqrt(4.0 * scale * Y + Y * Y));
    double U = g.uniform();
    return (U <= mean / (mean + X)) ? X : mean * mean / X;
  } else if (distr == GNX_DISTR_LOGNORMAL) {
    return exp(p1 + p2 * g.normal());
  } else {
    double Z = g.normal();
    return p1 + p2 / (Z * Z);
  }
}

// numpy legacy poisson: multiplication method below lam = 10, PTRS above
// Gamma(shape, scale): Marsaglia & Tsang (2000), with the U^(1/shape) boost below shape 1
// (numpy's legacy generator uses the same method for shape > 1).
__device__ inline double sample_gamma(RngStream& g, double shape, double scale) {
  if (shape <= 0.0) return 0.0;
  double boost = 1.0;
  if (shape < 1.0) {
    boost = pow(1.0 - g.uniform(), 1.0 / shape);
    shape += 1.0;
  }
  const double d = shape - 1.0 / 3.0, cc = 1.0 / sqrt(9.0 * d);
  for (int it = 0; it < 1000; ++it) {
    double x, v;
    do {
      x = g.normal();
      v = 1.0 + cc * x;
    } while (v <= 0.0);
    v = v * v * v;
    const double u = 1.0 - g.uniform();
    if (u < 1.0 - 0.0331 * (x * x) * (x * x)) return d * v * boost * scale;
    if (log(u) < 0.5 * x * x + d * (1.0 - v + log(v))) return d * v * boost * scale;
  }
  return d * boost * scale;
}

// Binomial(n, p) by geometric waiting times between successes: exact, O(n p) -- the count is
// bounded by the number of mutable loci (infinite sites), so it is always small here.
__device__ inline long long sample_binomial_wait(RngStream& g, long long n, double p) {
  if (p <= 0.0 || n <= 0) return 0;
  if (p >= 1.0) return n;
  const double lq = log1p(-p);
  long long pos = 0, k = 0;
  while (true) {
    const double u = 1.0 - g.uniform();                 // (0, 1]
    const double gap = floor(log(u) / lq);              // failures before the next success
    if (gap >= (double)(n - pos)) break;
    pos += (long long)gap + 1;
    if (pos > n) break;
    k += 1;
    if (k > (1 << 24)) break;
  }
  return k;
}

__device__ inline int sample_poisson(RngStream& g, double lam) {
  if (lam <= 0.0) return 0;
  if (lam < 10.0) {
    double enlam = exp(-lam), prod = 1.0;
    int X = 0;
    for (;;) {
      prod *= g.uniform();
      if (prod > enlam) X += 1; else return X;
    }
  }
  double slam = sqrt(lam), loglam = log(lam);
  double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b;
  double invalpha = 1.1239 + 1.1328 / (b - 3.4), vr = 0.9277 - 3.6224 / (b - 2.0);
  for (;;) {
    double U = g.uniform() - 0.5, V = g.uniform();
    double us = 0.5 - fabs(U);
    double kf = floor((2.0 * a / us + b) * U + lam + 0.43);
    if (us >= 0.07 && V <= vr) return (int)kf;
    if (kf < 0 || (us < 0.013 && V > us)) continue;
    if ((log(V) + log(invalpha) - log(a / (us * us) + b)) <= (-lam + kf * loglam - lgamma(kf + 1.0)))
      return (int)kf;
  }
}

// exact floor(a / b) for finite doubles, b > 0 (numpy floor_divide semantics, spatial.py:79-82)
__device__ __forceinline__ double floordiv_exact(double a, double b) {
  double q = floor(a / b);
  double r = fma(-q, b, a);
  if (r < 0.0) q -= 1.0;
  else if (r >= b) q += 1.0;
  return q;
}

__device__ __forceinline__ double clampd(double v, double lo, double hi) {
  return v < lo ? lo : (v > hi ? hi : v);    // NaN-propagating like np.clip is not needed here
}

// cos/sin of a float16 direction exactly as numpy evaluates them on a float16 array:
// half -> float, libm cosf (correctly rounded), -> half (movement.py:75-76 with a
// float16 `direction`, spatial.py:184,447)
__device__ __forceinline__ void sincos_half(__half h, double* s, double* c) {
  double a = (double)__half2float(h);
  float cf = (float)cos(a), sf = (float)sin(a);
  *c = (double)__half2float(__float2half_rn(cf));
  *s = (double)__half2float(__float2half_rn(sf));
}
