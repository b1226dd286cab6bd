/* gnx_b200.h -- C-ABI of libgnxb200.so: the B200-native (sm_100a) implementation of
 * Geonomics' per-timestep individual-based update loop.
 *
 * The reference (erthward/geonomics v1.4.9) is pure Python and has no FFI; its seam for this
 * path is the per-species method set that Model._make_fn_queue (sim/model.py:603-667) queues
 * each time step.  Every entry point below names the reference interface it replaces
 * (file:line relative to /root/reference/geonomics/).  INTEGRATION.md shows the ctypes
 * binding a maintainer would add on the reference side.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (gnx_strerror); no exceptions;
 *   - one gnx_ctx per Species; it owns all device buffers and one CUDA stream; calls on a
 *     ctx must come from one host thread at a time;
 *   - pointers named host_* are caller-owned HOST buffers; nothing in the ABI is a torch
 *     type; device pointers are exposed only through gnx_device_ptr (for zero-copy views);
 *   - step functions are asynchronous on the ctx stream unless stated; gnx_sync waits;
 *   - individuals are held structure-of-arrays in *species order* (iteration order of the
 *     reference's Species OrderedDict); genotypes are bit-packed, one row per individual:
 *     [homologue 0 | homologue 1], each homologue 16*ceil(L/128) bytes, locus l = bit (l%32)
 *     of u32 word l/32;
 *   - randomness is counter-based Philox4x32-10 keyed by (seed; individual id, call site,
 *     time step); every call site can instead replay caller-injected draws (gnx_set_draws),
 *     which is how integer/index parity with the reference is tested.
 */
#ifndef GNX_B200_H
#define GNX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNX_ABI_VERSION 1
#define GNX_MAX_TRAITS 8
#define GNX_MAX_LAYERS 16

typedef struct gnx_ctx gnx_ctx;

enum { GNX_DISTR_WALD = 0, GNX_DISTR_LOGNORMAL = 1, GNX_DISTR_LEVY = 2 };
enum { GNX_SURF_NONE = 0, GNX_SURF_TABLE = 1, GNX_SURF_ONTHEFLY = 2 };

/* error codes */
enum {
  GNX_OK = 0,
  GNX_ERR_CUDA = -1,        /* a CUDA runtime call failed (message in gnx_last_error) */
  GNX_ERR_ARG = -2,         /* invalid argument */
  GNX_ERR_CAPACITY = -3,    /* population outgrew ctx capacity */
  GNX_ERR_DRAWS = -4,       /* an injected draw buffer was exhausted */
  GNX_ERR_STATE = -5,       /* call made in the wrong state (e.g. genomes not set) */
  GNX_ERR_MUTABLES = -6     /* no mutable locus left (the reference raises on _mutables.pop()) */
};

/* Species + landscape parameters the hot path reads.  Mirrors the attributes the reference
 * ops read off the Species (`spp.b`, `spp.mating_radius`, ... species.py:405-425) and the
 * Landscape (`land.dim`, landscape.py:245-314). */
typedef struct {
  int32_t abi_version;        /* GNX_ABI_VERSION */
  int32_t dim_x, dim_y;       /* land.dim = (x, y) = (cols, rows) */
  int32_t n_layers;
  int64_t capacity;           /* max individuals alive at once (incl. newborns) */
  uint64_t seed;
  /* genome */
  int32_t L;                  /* loci carried per individual (gen_arch.L, use_tskit=False) */
  int32_t n_recomb_paths;     /* Recombinations._n (genome.py:69) */
  int32_t n_traits;
  int32_t use_dom;            /* gen_arch._use_dom (genome.py:556) */
  /* mating (species.py:2157-2215, mating.py:24-126) */
  double mating_radius;       /* < 0: panmixia (mating_radius=None) */
  double b;
  double R;
  double n_births_lambda;
  int32_t n_births_fixed;
  int32_t sex;
  double sex_ratio_p;         /* spp.sex_ratio (probability of drawing a male) */
  int32_t choose_nearest;
  int32_t inverse_dist;
  /* mortality (demography.py:153-180, 319-321) */
  double d_min, d_max;
  int32_t max_age;            /* -1: None */
  int32_t K_layer;
  double K_factor;
  /* movement (movement.py:34-141) */
  int32_t move;               /* spp._move */
  int32_t move_distr, disp_distr;
  double move_p1, move_p2, disp_p1, disp_p2;
  double dir_mu, dir_kappa;
  double res_ratio_x, res_ratio_y;
  int32_t move_surf_mode, disp_surf_mode;     /* GNX_SURF_* */
  int32_t move_surf_layer, disp_surf_layer;
  int32_t move_surf_mixture, disp_surf_mixture;
  double move_surf_kappa, disp_surf_kappa;
  int32_t surf_approx_len;    /* table mode: third dim of the float16 tables */
  int32_t disp_max_tries_injected;   /* columns of the injected dispersal draw arrays */
} gnx_config_t;

/* One trait (genome.py:284-437): loci are row indices into the genotype array. */
typedef struct {
  int32_t n_loci;
  const int32_t* host_loci;     /* [n_loci], ascending */
  const double* host_alpha;     /* [n_loci] */
  double phi;                   /* scalar phi; ignored when host_phi_raster != NULL */
  const double* host_phi_raster;/* [dim_y][dim_x] or NULL (genome.py:391-396) */
  double gamma;
  int32_t layer;                /* trait.lyr_num */
  int32_t univ_adv;
} gnx_trait_t;

/* Density-grid stack + its Delaunay triangulation (spatial.py:100-146, 270-360).  The
 * lattice is built by the caller exactly as the reference builds it; the triangulation is
 * the one scipy.interpolate.griddata builds (Qhull) for those points. */
typedef struct {
  double window_width;
  int32_t n_points;
  const double* host_points;        /* [n_points][2] as (i, j) = (y, x) */
  const double* host_areas;         /* [n_points] window-landscape intersection areas */
  int32_t grid_ni[4], grid_nj[4];   /* shape of each of the 4 offset grids */
  int32_t grid_i0[4], grid_j0[4];   /* cell id of each grid's first point */
  int32_t grid_x_edge[4], grid_y_edge[4];
  int32_t n_tri;
  const int32_t* host_simplices;    /* [n_tri][3] */
  const int32_t* host_neighbors;    /* [n_tri][3] */
  const int32_t* host_nbr_indptr;   /* [n_points+1] vertex_neighbor_vertices CSR */
  const int32_t* host_nbr_indices;
  int32_t lat_ni, lat_nj;           /* lattice points per axis (spacing window_width/2) */
  const int32_t* host_square_tri;   /* [(lat_ni-1)*(lat_nj-1)][2] triangles per lattice square */
  int32_t colourable;               /* 1: the 4 grids are independent sets of the triangulation */
} gnx_density_t;

/* Injected draws (all HOST pointers, any may be NULL = use Philox at that site).
 * Sites follow SURVEY.md Appendix A. */
typedef struct {
  int64_t n;                        /* rows available in per-individual arrays */
  const double* move_dir;           /* A1 vonmises outputs [n] */
  const int32_t* move_choice;       /* A1 surface-table column [n] */
  const double* move_dist;          /* A2 [n] */
  const uint32_t* mate_R;           /* A4 [n]: k = (R * n_nbrs) >> 32 */
  const double* mate_inv_u;         /* A4 inverse-distance mode [n] */
  const double* mate_u;             /* A5 [n]: pair kept iff u < b */
  const int32_t* poisson;           /* A6 [n] per canonical pair */
  const int32_t* recomb_keys;       /* A7 [2n] */
  const int32_t* start_homs;        /* A8 [n][2] */
  const double* disp_dir;           /* A9 [n][tries] */
  const int32_t* disp_choice;       /* A9 surface-table column [n][tries] */
  const double* disp_dist;          /* A10 [n][tries] */
  const double* sex_u;              /* A11 [n] */
  const double* sex_redraw_u;       /* A12 [n] */
  const double* death_u;            /* A16 [n] */
  const double* pan_u;              /* A3 panmixia [n]: individual i opens a mating slot iff u < b */
  const uint32_t* pan_R;            /* A3 panmixia [n][2]: the slot's two parents, (R * N) >> 32 */
  /* mutation (ops/mutation.py:169-206); n_mut = length of the per-mutation arrays */
  int64_t n_mut;
  const int32_t* mut_n;             /* [1] number of mutations this step (binomial(B*L, mu_tot) output) */
  const double* mut_type_u;         /* [n_mut] type = searchsorted(cdf(mu_neut, mu_delet, ...), u, 'right') */
  const uint32_t* mut_ind_R;        /* [n_mut] mutated offspring = B - 1 - ((R * B) >> 32): r.choice over the
                                     * descending id list of species.py:615-622 */
  const double* mut_homol_u;        /* [n_mut] homologue = (u < 0.5) */
  const double* mut_s;              /* [n_mut] gamma(shape, scale) output for deleterious s (before min(s, 1)) */
  const double* mut_alpha;          /* [n_mut] normal(alpha_distr_mu, alpha_distr_sigma) output for a trait mutation
                                     * (before the max_alpha_mag clip, genome.py:679-682) */
} gnx_draws_t;

/* Host-side SoA view of a population (upload / download). Any pointer may be NULL. */
typedef struct {
  int64_t n;
  double* x; double* y;             /* individual.py:107-108 */
  int32_t* age; int8_t* sex; int64_t* idx;
  uint32_t* genomes;                /* [n][2][4*ceil(L/128)] packed rows */
  double* z;                        /* [n][n_traits] */
  double* fit;                      /* [n] */
  double* e;                        /* [n][n_layers]  (download only; species.py:913-922) */
  int64_t max_ind_idx;              /* species.py:360 */
} gnx_population_t;

/* Per-step counters (species.py:374-380: Nt, n_births, n_deaths). */
typedef struct {
  int64_t t; int64_t Nt; int64_t n_births; int64_t n_deaths; int64_t n_pairs;
} gnx_step_record_t;

const char* gnx_strerror(int code);
const char* gnx_last_error(void);
int gnx_abi_version(void);

/* ---- lifecycle / setup (replaces the object state the reference keeps on Species /
 *      Landscape / GenomicArchitecture; setup is not on the hot path) -------------------- */
int gnx_create(const gnx_config_t* cfg, gnx_ctx** out);
int gnx_destroy(gnx_ctx* ctx);
int gnx_set_rasters(gnx_ctx* ctx, const double* host_rasters /* [n_layers][dim_y][dim_x] */);
int gnx_set_traits(gnx_ctx* ctx, int32_t n_traits, const gnx_trait_t* traits,
                   const int8_t* host_dom /* [L] or NULL */);
int gnx_set_recomb_paths(gnx_ctx* ctx, const uint32_t* host_packed_paths /* [n_paths][W] */);
int gnx_set_density(gnx_ctx* ctx, const gnx_density_t* dens);
int gnx_set_surface_tables(gnx_ctx* ctx, const uint16_t* host_move_f16, const uint16_t* host_disp_f16);
int gnx_set_draws(gnx_ctx* ctx, const gnx_draws_t* draws /* NULL: clear, back to Philox */);
int gnx_set_burn(gnx_ctx* ctx, int32_t burn);   /* burn-in: no genomes, no selection (species.py:825) */
/* keep per-individual intermediates (n_nbrs, death_p, disp_tries, n_pairs raster) readable
 * through gnx_read_field; off by default (they cost extra HBM writes) */
int gnx_set_debug(gnx_ctx* ctx, int32_t on);
int gnx_upload_population(gnx_ctx* ctx, const gnx_population_t* pop);
int gnx_download_population(gnx_ctx* ctx, gnx_population_t* pop /* buffers sized >= gnx_population_size */);
int gnx_population_size(gnx_ctx* ctx, int64_t* n);          /* synchronises */

/* ---- hot path, stage by stage (each is asynchronous on the ctx stream) ----------------- */
/* Species._set_age_stage  species.py:567-569 */
int gnx_age_step(gnx_ctx* ctx);
/* ops.movement._do_movement  movement.py:34-95 (+ _ConductanceSurface._draw_directions spatial.py:182) */
int gnx_move(gnx_ctx* ctx);
/* Species._set_e  species.py:913-922 (materialises e[n][n_layers] on demand) */
int gnx_sample_env(gnx_ctx* ctx);
/* Species._set_coords_and_cells + cKDTree rebuild  species.py:937-939, 2170: counting-sort binning */
int gnx_bin_cells(gnx_ctx* ctx);
/* Species._get_mating_pairs + _KDTree._get_mating_pairs  species.py:2157-2215, spatial.py:191-245 */
int gnx_find_mates(gnx_ctx* ctx);
/* ops.mating._find_mates (sex filter / de-dup)  mating.py:24-117;  _draw_n_births mating.py:120-126;
 * offspring ids species.py:614-619;  pair-midpoint counts for demography._calc_n_pairs :60-91 */
int gnx_dedup_pairs(gnx_ctx* ctx);
/* ops.mating._do_mating (gametes) mating.py:130-214 + ops.selection._calc_phenotype selection.py:22-48
 * + ops.movement._do_dispersal movement.py:98-141 + newborn records species.py:638-688 */
int gnx_make_offspring(gnx_ctx* ctx);
/* _DensityGridStack._calc_density counts  spatial.py:73-97 */
int gnx_density_counts(gnx_ctx* ctx);
/* scipy griddata(method='cubic') spatial.py:144: gradient estimate + Clough-Tocher evaluation;
 * demography._calc_dNdt/_calc_N_b/_calc_Nd/_calc_d  demography.py:104-172 */
int gnx_density_eval(gnx_ctx* ctx);
/* selection._calc_fitness/_calc_prob_death selection.py:51-125; demography.py:306-321 */
int gnx_death_prob(gnx_ctx* ctx);
/* demography._do_mortality demography.py:175-180 (+ stable compaction, genome-slot recycling) */
int gnx_mortality(gnx_ctx* ctx);
/* Landscape._set_raster landscape.py:353 + Species._set_K species.py:546 (env change, change.py:56-84) */
int gnx_set_raster(gnx_ctx* ctx, int32_t layer, const double* host_raster);
/* Species change events, ops/change.py:612-742 (queue slot model.py:654-656, Species._make_change
 * species.py:836).  gnx_set_K: a demographic change rewrote spp.K (`spp.K *= size`,
 * `spp.K = base_K * size`, change.py:633-649) -- the new [dim_y][dim_x] raster.
 * gnx_set_life_history: `setattr(spp, parameter, val)` (change.py:735-742) -- a full config whose
 * life-history scalars (b, R, births, sex ratio, d_min/d_max, max_age, K_factor, movement and
 * dispersal distributions, direction, mate-choice flags) may differ; sizes, genome, landscape,
 * mating_radius and the surface setup must equal the values given to gnx_create. */
int gnx_set_K(gnx_ctx* ctx, const double* host_K);
int gnx_set_life_history(gnx_ctx* ctx, const gnx_config_t* cfg);

/* ---- whole steps ------------------------------------------------------------------------ */
/* n_steps iterations of the main/burn queue for this species:
 * _set_age_stage -> _do_movement -> _do_pop_dynamics -> _set_Nt  (model.py:603-667).
 * Asynchronous: nothing is read back (sizes live in device counters); errors such as capacity
 * overflow surface at the next synchronising call.  From the second step of a context on, the
 * step is one CUDA-graph launch (23 kernels on two branches: genotype streaming beside the
 * density chain); the graph is re-captured when a setter changed any kernel argument.
 * GNX_NO_GRAPH=1 in the environment keeps plain stream launches. */
int gnx_step(gnx_ctx* ctx, int32_t n_steps);
/* ---- growth between steps ----------------------------------------------------------------
 * gnx_set_growth_guard(ctx, 1): every step first checks, from the device counters, whether it could
 * overflow the population capacity (entries, genome slots) or the tskit row buffers; a step that
 * could does not start (nothing moves, no draws, Counters.t stays) and neither does any later step
 * of the same gnx_step batch.  The caller reads gnx_step_status, grows the buffers (gnx_reserve,
 * gnx_tskit_reserve) and steps again: Philox draws are keyed by (seed, id, site, t), so the run is
 * bit-identical to one that had the larger buffers from the start.  Graph-launched steps check on
 * the device (a guard kernel in front of an IF conditional node holding the step), the first step
 * of a context and GNX_NO_GRAPH steps on the host.  Off by default; GNX_ERR_STATE on a strip. */
typedef struct {
  int32_t steps_run;          /* steps of the last gnx_step batch that ran */
  int32_t stopped;            /* 1: the batch stopped in front of a step that could overflow */
  int64_t need_entries;       /* population capacity the next step needs (n + most births) */
  int64_t need_slots;         /* genome slots it needs (within the population capacity) */
  int64_t need_births;        /* tskit birth rows it needs (0 without recording) */
  int64_t need_edges;         /* tskit edge rows it needs (0 without recording) */
  int64_t capacity, born_capacity, edge_capacity;   /* the current sizes */
} gnx_step_status_t;
int gnx_set_growth_guard(gnx_ctx* ctx, int32_t on);
/* Synchronises; reconciles the host's step bookkeeping with the steps the device skipped. */
int gnx_step_status(gnx_ctx* ctx, gnx_step_status_t* out);
/* Grow the population capacity (never shrinks): every buffer sized from it is re-allocated and its
 * contents copied.  On an allocation failure GNX_ERR_CUDA, and the context keeps its old buffers. */
int gnx_reserve(gnx_ctx* ctx, int64_t capacity);
/* Grow the tskit row buffers; the rows buffered since the last drain are kept. */
int gnx_tskit_reserve(gnx_ctx* ctx, int64_t edge_capacity, int64_t birth_capacity);
/* ---- resuming a checkpoint ----------------------------------------------------------------------
 * gnx_set_clock writes the time-step counter Counters.t (the Philox counter word of every draw) and the
 * tskit time origin Counters.tsk_t0 (node time = -(t - tsk_t0)) on the context's stream, so that a population
 * uploaded from a checkpoint continues the draws of the run it was saved from.  Call it last, after the
 * upload, gnx_set_mutation and the tskit calls (gnx_tskit_enable sets tsk_t0 to the current t).  The step
 * kernels read both values from Counters, never as graph arguments, so a captured step graph stays valid.
 * GNX_ERR_STATE while a step is pending (its deaths are only flagged: download or upload first) or a device
 * genome assignment is under way; on a strip every rank is given the same values. */
int gnx_set_clock(gnx_ctx* ctx, int64_t t, int64_t tsk_t0);
/* The cached recombination paths as the gamete kernel reads them: n_words = n_recomb_paths * 4 * (128-bit
 * units of a genotype row) words, bit j of path p = the homologue path p reads at genotype bit j.  Under the
 * tskit layout these are the reference's subsetters: k_mutate patches the bit of a column a mutation adds with
 * the path in front of its locus (genome.py:133-160), which the paths as simulated do not give back, so a
 * checkpoint carries them into gnx_set_mutation's host_subsetters.  Synchronises. */
int gnx_read_paths(gnx_ctx* ctx, uint32_t* host_paths, int64_t n_words);
/* ---- sort + simplify of the tskit tables (gnx_simplify.cuh) ---------------------------------------
 * The columns of geonomics_b200.tables.TableColumns: nodes (time, population, individual; flags are
 * written, not read), edges, individuals (n_location doubles per row), site positions and mutations.
 * gnx_simplify reads them, does TableCollection.sort() + simplify(samples, filter_individuals=True,
 * filter_sites=False) as tables.simplify_columns restates it, row for row, and returns the output sizes
 * out_sizes[4] = nodes, edges, individuals, mutations (the sites are unchanged).  The result stays on the
 * device until gnx_simplify_result copies it into host columns of exactly those sizes (the n_* fields of
 * `out` say so) and frees it.  Both run on the ctx's stream and synchronise; scratch lives for the call.
 * GNX_ERR_ARG for an edge whose parent is not older than its child, an edge outside 0 <= left < right <=
 * sequence_length, a node id, sample, site or individual out of range, or a repeated sample. */
typedef struct {
  double sequence_length;
  int64_t n_nodes;
  int32_t* node_flags;
  double* node_time;
  int32_t* node_population;
  int32_t* node_individual;
  int64_t n_edges;
  double* edge_left;
  double* edge_right;
  int32_t* edge_parent;
  int32_t* edge_child;
  int64_t n_individuals;
  int32_t n_location;
  int32_t* individual_flags;
  double* individual_location;   /* [n_individuals][n_location] */
  int64_t* individual_idx;
  int64_t n_sites;
  double* site_position;
  int64_t n_mutations;
  int32_t* mutation_site;
  int32_t* mutation_node;
  double* mutation_time;
} gnx_tables_t;
int gnx_simplify(gnx_ctx* ctx, const gnx_tables_t* tables, const int32_t* samples, int64_t n_samples,
                 int64_t* out_sizes);
int gnx_simplify_result(gnx_ctx* ctx, gnx_tables_t* out);
/* ---- strip domain decomposition of one landscape over several GPUs (SURVEY.md section 8e-2) ---
 * What shards (reference file:line): the mate search species.py:2157-2215 / spatial.py:191-245
 * (halo of the individuals within one mating-grid row of a strip edge, with their genome rows),
 * movement movement.py:34-95 and natal dispersal movement.py:98-141 (migrants to the strip they
 * land in), the density counts spatial.py:73-97 (summed over ranks), max(N) demography.py:104-119,
 * offspring ids species.py:614-619 (based at the births of the lower ranks).  Records travel by
 * direct writes into the receiver's buffer (NVLink peer memory through CUDA IPC, or plain device
 * pointers when the ranks are contexts of one process); the caller supplies the barrier between
 * phases (a stream-ordered collective) and the small collectives named at gnx_strip_collective_ptrs
 * and gnx_strip_pairs_ptr, or gnx_strip_barrier does both over peer memory. */
typedef struct {
  int32_t rank, world;
  const int32_t* first_rows;     /* [world + 1] first mating-grid row of every rank, first_rows[world] = rows of the grid */
  int64_t migrant_capacity;      /* records a rank can receive per step as migrants (and as dispersed newborns) */
  int64_t halo_capacity;         /* records a rank can receive per step as ghosts (and as edge mate choices) */
} gnx_strip_config_t;
typedef struct {
  void* base;                    /* device address of the rank's receive block (valid in its own process) */
  int64_t bytes;
  int64_t buf_offset[4];         /* migrants, halo, newborns, choices */
  int64_t count_offset[4];
  unsigned char ipc_handle[64];  /* cudaIpcMemHandle_t of the block, for ranks in other processes */
  int64_t sync_offset;           /* the rank's synchronisation page inside the block (gnx_strip_barrier) */
  int64_t counts_cap;            /* ints per rank slot of the density-count exchange */
} gnx_strip_endpoints_t;
int gnx_strip_enable(gnx_ctx* ctx, const gnx_strip_config_t* cfg);
int gnx_strip_endpoints(gnx_ctx* ctx, gnx_strip_endpoints_t* out);
int gnx_strip_connect(gnx_ctx* ctx, int32_t peer_rank, const gnx_strip_endpoints_t* peer, int32_t same_process);
/* device buffers the caller's collectives act on: births int64[world] (all-gather after phase 3),
 * counts int32[n_counts] (all-reduce sum after phase 5), nmax uint64[1] holding the bits of a
 * non-negative double (all-reduce max after phase 6) */
int gnx_strip_collective_ptrs(gnx_ctx* ctx, void** births, void** counts, int64_t* n_counts, void** nmax);
/* device buffer of the pairs int64[world] (all-gather after phase 3 with Poisson births) */
int gnx_strip_pairs_ptr(gnx_ctx* ctx, void** pairs);
/* one phase of a time step on this rank's stream; every rank must have finished a phase before any
 * rank starts the next.  With n_births_fixed the step is phases 0..7 (births all-gather after phase 3).
 * With Poisson births the births of a rank are keyed by the species-wide positions of its pairs, so
 * phase 3 ends after the pair list and publishes the pairs; the step is then phases 0, 1, 2, 3, 8, 4, 5,
 * 6, 7 with the pairs all-gather after phase 3 and the births all-gather after phase 8 (the Poisson
 * draws).  Phase 8 with n_births_fixed is an error.  Mutation (by-locus layout) runs inside phase 4:
 * every rank replays the species-wide draws, so their tables and mutation logs stay identical. */
int gnx_strip_phase(gnx_ctx* ctx, int32_t phase);
/* That order, as gnx_step runs it: phases[k] then the gnx_strip_barrier kind sync_after[k] (-1: the step
 * ends), for k < *n (at most 9). */
int gnx_strip_phase_order(int32_t n_births_fixed, int32_t* phases, int32_t* sync_after, int32_t* n);
/* The barrier between two phases (kind 0) and the four collectives (1 births all-gather, 2 density-count sum,
 * 3 max(N), 4 pairs all-gather) done by ONE one-CTA kernel over peer memory on the rank's stream: every rank writes its slot of
 * every peer's synchronisation page (NVLink stores), publishes its barrier epoch with release semantics and
 * spins on its own page until every peer has arrived.  Replaces the caller-supplied NCCL collectives; all
 * ranks must make the same sequence of calls; a peer that never arrives sets an error after ~5 s. */
int gnx_strip_barrier(gnx_ctx* ctx, int32_t kind);
/* gnx_step on a context that holds a strip runs WHOLE time steps this way -- the eight phases with
 * gnx_strip_barrier after each of the first seven (nine and eight with Poisson births), captured as one CUDA
 * graph per step like the undecomposed run; the spin barriers inside order the ranks' graphs against each
 * other.  Every rank makes the same call.  Not supported on a strip context, and refused by the call that
 * would set them up: tskit recording, the tskit genotype layout, trait mutation and injected draws. */
int gnx_strip_check(gnx_ctx* ctx);      /* synchronises; exchange overflow -> GNX_ERR_CAPACITY */

int gnx_sync(gnx_ctx* ctx);
/* Same, with HOST buffers in and out: upload pop, run n_steps, download into pop (synchronous). */
int gnx_walk_host(gnx_ctx* ctx, gnx_population_t* pop, int32_t n_steps);
/* The same in two halves, for hosts that keep several replicate populations (model.py:115-117,
 * one context each) in flight: _begin enqueues the copies in and the steps and returns at once
 * (the buffers of `pop` must be pinned and stay untouched until _end returns); _end waits and
 * copies the population out.  Between the two, calls on OTHER contexts overlap with this one. */
int gnx_walk_host_begin(gnx_ctx* ctx, const gnx_population_t* pop, int32_t n_steps);
int gnx_walk_host_end(gnx_ctx* ctx, gnx_population_t* pop);
/* Drain the per-step records accumulated since the last call (synchronises). */
int gnx_read_step_records(gnx_ctx* ctx, gnx_step_record_t* out, int32_t max_records, int32_t* n_out);

/* ---- tskit record buffering (SURVEY.md section 8f rank 1) -----------------------------------
 * Replaces the per-offspring TableCollection.add_row calls of Species._do_mating
 * (species.py:692-736) and Recombinations._get_seg_info (genome.py:257-281): for every birth
 * the step kernels append, to device buffers, one individuals row (location = [x, y, z...],
 * metadata = idx), two nodes rows (flags = 1, time = -t, population = 0) and one edges row
 * per recombination segment and homologue.  The host drains them into tskit with
 * TableCollection.{individuals,nodes,edges}.append_columns at its existing simplify
 * interval (model.py:756-768), then calls gnx_tskit_renumber (species.py:1148-1152). */
typedef struct {
  int64_t n_edges, n_births;        /* in: capacity of the arrays below; out: rows written */
  double* edge_left; double* edge_right; int32_t* edge_parent; int32_t* edge_child;
  int64_t* birth_idx;               /* individuals.metadata (4 LE bytes of idx in the reference) */
  double* birth_x; double* birth_y; /* individuals.location[0:2] */
  double* birth_z;                  /* [n_traits][n_births] individuals.location[2:] */
  double* birth_time;               /* nodes.time of the two nodes of birth k */
  int32_t first_node_id;            /* nodes rows of birth k: first_node_id + 2k, + 2k + 1 */
  int32_t first_individual_row;     /* individuals row of birth k: first_individual_row + k */
} gnx_tskit_rows_t;
int gnx_tskit_enable(gnx_ctx* ctx, int64_t edge_capacity, int64_t birth_capacity);
int gnx_tskit_set_nodes(gnx_ctx* ctx, const int32_t* host_node0, const int32_t* host_node1, int64_t n,
                        int32_t next_node_id, int32_t next_individual_row);
int gnx_tskit_drain(gnx_ctx* ctx, gnx_tskit_rows_t* rows);   /* NULL arrays: query the counts only */
/* nodes 2k, 2k + 1 in species order and the row counters set to 2N / N: right when the simplified tables hold the
 * samples only; tskit's simplify also keeps the nodes (and their individuals) in which the samples' ancestry
 * coalesces, so after a real simplification call gnx_tskit_set_nodes with the sizes of the simplified tables */
int gnx_tskit_renumber(gnx_ctx* ctx);

/* ---- a13 mutation (ops/mutation.py:169-206 _do_mutation; :62-86 neutral; :90-131 + :156-166
 *      deleterious; genome.py:650-663 _draw_mut_types, :690-693 _draw_delet_s, :753-788
 *      _add_nonneut_locus), for both genotype layouts.  Runs inside gnx_make_offspring /
 *      gnx_step right after the newborn records are written (species.py:808-809).
 *      Infinite sites: every mutation pops one locus from the END of the shuffled `mutables`
 *      list (genome.py:1101-1104), so a run has at most n_mutables mutations and the
 *      bookkeeping is one device thread.
 *      - neutral: consumes a locus and the draws; the genotype array is NOT changed
 *        (mutation.py:81-82).
 *      - deleterious: s = min(gamma(shape, scale), 1); the locus joins nonneut_loci at
 *        idx = bisect_left(nonneut_loci, locus) and (delet_loci, delet_s); the offspring's
 *        genotype is set to 1 at ROW idx of the chosen homologue (mutation.py:117 indexes the
 *        L-row genotype array with the nonneut_loci position, not with the locus -- reproduced
 *        as is) and its phenotype is recomputed; fitness is then multiplied by
 *        prod_k (1 - s_k * dosage(delet_locus_k)) (selection.py:78-94).
 *      - trait mutations (Trait.mu > 0; mutation.py:135-144 -> :90-131, genome.py:666-687
 *        _draw_trait_alpha, :416-437 Trait._add_locus): the locus joins nonneut_loci and the
 *        trait's (loci, alpha, loci_idxs) with alpha = clip(normal(mu, sigma), +-max_alpha_mag)
 *        (or mu when sigma = 0; |alpha| while the trait is monogenic).  The reference raises for
 *        them when use_tskit = False (genome.py:430, loci_idxs is None): accepted only with
 *        tskit_layout = 1, rejected with GNX_ERR_ARG otherwise.
 *      tskit_layout = 1 (gen_arch.use_tskit = True, species.py:891-905): the reference's genotype
 *        arrays hold one row per NON-NEUTRAL locus, a non-neutral mutation inserts a zero row at
 *        idx into every individual (species.py:908-910) and sets g[idx, homologue] = 1, and the
 *        recombination subsetters get the path's homologue in front of the locus inserted at
 *        2*idx (genome.py:133-160).  The device keeps one bit per LOCUS (rows never move; row r
 *        of the reference is bit nonneut_loci[r]; neutral bits are zero and never read), sets bit
 *        `locus`, and patches bit `locus` of every cached path to (#breakpoints < locus) % 2.
 *        The reference's index arrays are reproduced AS WRITTEN: Trait.loci_idxs is shifted only
 *        behind the insertion point of the mutated trait itself and delet_loci_idxs never, so
 *        after mutations they may address other rows than the trait's / deleterious loci; the
 *        phenotype (selection.py:30) and the deleterious fitness (selection.py:86-88) read row
 *        idxs[k], i.e. bit nonneut_loci[idxs[k]].  A context of gnx_create_cols keeps the same
 *        semantics on one COLUMN per non-neutral locus: bit col_of_locus[l] stands for bit l above, a
 *        non-neutral mutation takes the next free column, and the path patch goes to that column.  Each log row carries the tskit node of the
 *        mutated homologue (mutations-table row of mutation.py:44-58: site = locus, node,
 *        derived_state '1', time = -t) when tskit recording is enabled.
 *      gnx_set_traits must precede gnx_set_mutation; re-setting the traits disables mutation. */
typedef struct {
  double mu_neut, mu_delet;           /* per-site, per-generation rates (genome.py:596-603) */
  double delet_s_shape, delet_s_scale;
  int32_t n_mutables;
  const int32_t* host_mutables;       /* shuffled list; popped from the end */
  int32_t n_nonneut;
  const int32_t* host_nonneut_loci;   /* ascending (trait loci + earlier deleterious loci) */
  int32_t n_delet;
  const int32_t* host_delet_loci;     /* ascending */
  const double* host_delet_s;
  int32_t log_capacity;               /* rows kept for gnx_read_mutations */
  int32_t tskit_layout;               /* 1: use_tskit = True semantics (see above) */
  const double* host_trait_mu;        /* [n_traits] Trait.mu, or NULL (no trait mutation) */
  const double* host_trait_alpha_distr; /* [n_traits][3]: alpha_distr_mu, alpha_distr_sigma, max_alpha_mag (< 0: None) */
  const int32_t* host_trait_loci_idxs;  /* tskit_layout: Trait.loci_idxs of every trait, concatenated in trait
                                           order, each in the order of Trait.loci; NULL = rows of the loci */
  const int32_t* host_delet_loci_idxs;  /* tskit_layout: gen_arch.delet_loci_idxs [n_delet]; NULL = rows of the loci */
  const uint8_t* host_subsetters;       /* tskit_layout: [n_recomb_paths][n_nonneut] homologue (0/1) each cached path
                                           takes at each genotype row (Recombinations._subsetters, genome.py:215-224,
                                           133-160); NULL = the paths of gnx_set_recomb_paths at the non-neutral loci.
                                           gnx_set_recomb_paths always takes the paths AS SIMULATED. */
} gnx_mutation_t;
typedef struct {
  int64_t t;                          /* time step */
  int64_t individual;                 /* idx of the mutated offspring */
  int32_t locus;
  int32_t row;                        /* genotype row written (= idx), -1 for neutral */
  int32_t homologue;
  int32_t type;                       /* 0 neutral, 1 deleterious, 2 + k: trait k */
  double s;                           /* selection coefficient (deleterious) */
  double alpha;                       /* effect size (trait mutation) */
  int32_t node;                       /* tskit node of the mutated homologue, -1 when not recording */
  int32_t reserved;
} gnx_mutation_row_t;
int gnx_set_mutation(gnx_ctx* ctx, const gnx_mutation_t* m);
int gnx_mutate(gnx_ctx* ctx);         /* stage entry; already part of gnx_make_offspring / gnx_step */
/* drains the mutation log and returns the current bookkeeping arrays (any pointer may be NULL) */
int gnx_read_mutations(gnx_ctx* ctx, gnx_mutation_row_t* rows, int32_t max_rows, int32_t* n_rows,
                       int32_t* n_mutables_left, int32_t* host_nonneut_loci, int32_t* n_nonneut,
                       int32_t* host_delet_loci, double* host_delet_s, int32_t* n_delet);
/* current (Trait.loci, Trait.alpha, Trait.loci_idxs) of one trait and gen_arch.delet_loci_idxs as the
 * mutations left them (genome.py:416-437, 753-788); arrays sized L + 1, any pointer may be NULL.
 * Without tskit_layout the idxs are the rows of the loci themselves. */
int gnx_read_mutation_tables(gnx_ctx* ctx, int32_t trait, int32_t* n_loci, int32_t* host_loci, double* host_alpha,
                             int32_t* host_loci_idxs, int32_t* host_delet_loci_idxs);

/* ---- column genotype layout of a use_tskit species --------------------------------------------
 * The by-locus layout keeps one bit per locus even under tskit_layout, where only the non-neutral loci
 * carry information.  A context created by gnx_create_cols keeps col_capacity COLUMNS per homologue
 * instead (rounded up to a multiple of 128; a homologue is 16 * col_capacity / 128 bytes): column j holds
 * non-neutral locus col_locus[j].  host_col_locus names the starting columns (usually the ascending
 * non-neutral loci); every non-neutral mutation takes the next free column; columns are never freed and no
 * bit ever moves.  Everything observable is as under the by-locus tskit layout (gnx_set_mutation must give
 * tskit_layout = 1 and host_nonneut_loci = the column loci; gnx_set_traits takes loci, all of them columns;
 * gnx_set_recomb_paths takes the paths as simulated, by locus), except that gnx_population_t.genomes,
 * GNX_F_GENOMES and gnx_genome_init_end use column rows [n][2][4 * col_capacity / 128].  gnx_stats_genotypes
 * (_region) and gnx_stats_ld count over the columns and return the by-locus arrays, zero at loci without a
 * column.  A non-neutral mutation that finds no free column inside a step is GNX_ERR_CAPACITY: the caller
 * widens between steps (gnx_widen_cols re-packs the genotype rows, the paths and the trait tables to the
 * wider rows; the next gnx_step captures its graph again).  Not supported under strip decomposition. */
int gnx_create_cols(const gnx_config_t* cfg, int32_t col_capacity, int32_t n_cols, const int32_t* host_col_locus,
                    gnx_ctx** out);
/* the current columns: host_col_locus [L] (column order) or NULL; synchronises */
int gnx_read_cols(gnx_ctx* ctx, int32_t* host_col_locus, int32_t* n_cols, int32_t* col_capacity);
int gnx_widen_cols(gnx_ctx* ctx, int32_t col_capacity);

/* ---- device assignment of the starting genomes (species.py:956-1094, genome.py:1108-1157) -----------
 * An alternative to uploading host-built genotypes after the burn-in.  Locus l gets exactly
 * host_n_carriers[l] 1-alleles (the caller applies the reference's rounding rule to the species-wide
 * live count n and the starting frequencies): homologue h of the individual with id i has the key
 * K_l(i, h) = Philox2x32-10(counter 2i + h, key k_l), k_l derived from (seed, l), and the carriers of
 * locus l are the n_l homologues with the smallest keys (keys never tie).  The genomes therefore depend
 * only on the seed, the set of live ids and the counts -- not on the entry order or on a strip cut.
 * The n_l-th smallest key is found by an MSB-first radix select (11 bits per pass) over keys that are
 * regenerated in every pass; the passes are separate calls so that the ranks of a strip-decomposed
 * landscape can sum their histograms (int32[L][2048]) between them:
 *   gnx_genome_init_begin  applies pending deaths, gives every live individual its own genome row
 *                          (burn-in newborns have none), counts the first digit; returns the histogram
 *   gnx_genome_init_pass   selects from the (summed) histogram; counts the next digit unless *all_done
 *   gnx_genome_init_end    after *all_done: writes every row (both homologues, padding zero, loci outside
 *                          host_write_mask zero) and recomputes the phenotypes, as an upload does
 *   gnx_genome_init_rows   tskit_rows only, before any step: (site, id, homologue) of every carrier at
 *                          every locus with carriers, sum(n_carriers) rows grouped by site (order within
 *                          a site unspecified); NULL arrays: *n_rows only
 * Each call synchronises.  Every rank of a strip makes the same calls with the same arguments.  Refused
 * (GNX_ERR_ARG): L = 0, n_loci != L, n_l outside [0, 2n], tskit_rows under strip decomposition. */
typedef struct {
  uint64_t seed;
  int32_t n_loci;                     /* = L */
  const int64_t* host_n_carriers;     /* [L] 1-alleles per locus */
  const uint8_t* host_write_mask;     /* [L] loci whose bits are set (the non-neutral loci of the tskit
                                         layout), or NULL: every locus */
  int32_t tskit_rows;                 /* 1: keep the selection of every locus for gnx_genome_init_rows */
} gnx_genome_init_t;
int gnx_genome_init_begin(gnx_ctx* ctx, const gnx_genome_init_t* gi, void** dev_hist, int64_t* hist_len);
int gnx_genome_init_pass(gnx_ctx* ctx, int32_t* all_done);
int gnx_genome_init_end(gnx_ctx* ctx);
int gnx_genome_init_rows(gnx_ctx* ctx, int32_t* host_site, int64_t* host_id, int8_t* host_homologue,
                         int64_t capacity, int64_t* n_rows);

/* ---- on-device statistics (sim/stats.py:399-435 _calc_het / _calc_maf / _calc_mean_fitness;
 *      SURVEY.md section 8f rank 2): per-locus 1-allele counts and heterozygote counts by
 *      vertical popcount over the packed genotypes, and the sum of fitness.  Synchronises. */
int gnx_stats_genotypes(gnx_ctx* ctx, uint64_t* host_c1 /* [L] */, uint64_t* host_het /* [L] */,
                        double* fit_sum, int64_t* n);
/* the same restricted to the individuals in [x_min, x_max) x [y_min, y_max): sub-population allele
 * counts for pairwise Fst = (Ht - Hs) / Ht (tests/validation/island/island_test.py:54-68) */
int gnx_stats_genotypes_region(gnx_ctx* ctx, double x_min, double x_max, double y_min, double y_max,
                               uint64_t* host_c1, uint64_t* host_het, double* fit_sum, int64_t* n);
/* Linkage disequilibrium (sim/stats.py:359-392 _calc_ld): host_n11[Lp * Lp] row-major with
 * Lp = 32 * ceil(L / 32); entry (i, j) with j / 32 >= i / 32 = number of chromosomes (of 2n) that
 * carry the 1-allele at both locus i and locus j (the diagonal: 1-allele counts); the other
 * word-triangle stays zero.  r^2 = D^2 / (f_i (1 - f_i) f_j (1 - f_j)), D = n11 / 2n - f_i f_j, is
 * formed by the caller exactly as the reference writes it.  Synchronises. */
int gnx_stats_ld(gnx_ctx* ctx, uint64_t* host_n11, int64_t* n);
/* Burn-in spatial statistic (sim/burnin.py:21-58 SpatialTester.update, species.py:572-578): counts
 * the live individuals of every landscape cell (int(x), int(y)) and returns the sum and the sum of
 * squares of the change of the counts since the previous call on this context (the first call
 * compares with all-zero counts, as SpatialTester.__init__ does).  mean(diff) and std(diff) over the
 * dim_x * dim_y cells follow from the two integers.  Synchronises. */
int gnx_burnin_cell_stats(gnx_ctx* ctx, int64_t* sum_diff, int64_t* sum_sq_diff);
/* The same statistic for a species cut into strips, in two calls per rank and burn-in step.  A rank's
 * individuals lie in its landscape rows [ly0, ly1) (gnx_strip_enable), and the band of a rank ends on the
 * row its upper neighbour's band starts on whenever a mating-grid row boundary falls inside a landscape row.
 * gnx_strip_burnin_count counts this rank's individuals into a band raster of (ly1 - ly0) x dim_x int32
 * with the transposed tally of gnx_burnin_cell_stats (cell (ix, iy) counted at row iy - ly0, column ix, only
 * for ix < dim_y and iy < dim_x), and returns the band and the device addresses of its first and last rows
 * (dim_x int32 each).  Before gnx_strip_burnin_diff the caller adds the lower neighbour's last row into this
 * rank's first row when they are the same landscape row.  gnx_strip_burnin_diff then returns the sum and the
 * sum of squares of the change of the band's counts since the previous call, over every band row except the
 * last one when skip_last_row (a shared row belongs to the upper rank).  The species-wide sums are the sums
 * over the ranks, equal to gnx_burnin_cell_stats of the undecomposed population.  Both synchronise; an
 * individual outside [ly0, ly1) -> GNX_ERR_STATE; GNX_ERR_STATE without strip decomposition. */
int gnx_strip_burnin_count(gnx_ctx* ctx, int32_t* ly0, int32_t* ly1, void** first_row, void** last_row);
int gnx_strip_burnin_diff(gnx_ctx* ctx, int32_t skip_last_row, int64_t* sum_diff, int64_t* sum_sq_diff);

/* ---- introspection (parity tests, lazy API views) -------------------------------------- */
enum {
  GNX_F_X = 1, GNX_F_Y, GNX_F_AGE, GNX_F_SEX, GNX_F_IDX, GNX_F_Z, GNX_F_FIT, GNX_F_GSLOT,
  GNX_F_N_NBRS, GNX_F_MATE, GNX_F_PAIRS, GNX_F_NB, GNX_F_PERM, GNX_F_CELL_START,
  GNX_F_COUNTS_N, GNX_F_COUNTS_P, GNX_F_VALS_N, GNX_F_VALS_P, GNX_F_GRAD_N, GNX_F_GRAD_P,
  GNX_F_N_RAST, GNX_F_NPAIRS_RAST, GNX_F_D_RAST, GNX_F_K_RAST, GNX_F_DEATH_P, GNX_F_ALIVE,
  GNX_F_DISP_TRIES, GNX_F_E, GNX_F_COUNTERS, GNX_F_GENOMES,
  GNX_F_NODE0, GNX_F_NODE1,    /* tskit node id of homologue 0 / 1 (int32, Individual._nodes_tab_ids) */
  GNX_F_VM_TAB_MOVE, GNX_F_VM_TAB_DISP  /* von Mises inverse-CDF table of an on-the-fly surface (float32
                                           [4096 + 1 + 256 + 1]); GNX_ERR_STATE when that site is not on the fly */
};
/* Copies a device field into a host buffer (synchronises).  For per-individual fields the
 * first `count` elements in species order are returned. */
int gnx_read_field(gnx_ctx* ctx, int32_t field, void* host_out, int64_t nbytes);
int gnx_device_ptr(gnx_ctx* ctx, int32_t field, void** dev_ptr, int64_t* nbytes);
void* gnx_stream(gnx_ctx* ctx);     /* cudaStream_t of the ctx */

/* kernel launch accounting (bench.py "gpu_launches") */
int64_t gnx_launch_count(gnx_ctx* ctx);
/* whole-step CUDA-graph launches / (re-)captures since the ctx was created: a multi-step run must
 * re-launch ONE captured graph (tests/test_cuda_multistep.py) */
int64_t gnx_graph_launch_count(gnx_ctx* ctx);
int64_t gnx_graph_capture_count(gnx_ctx* ctx);
/* per-kernel device timing with CUDA events on the ctx stream (bench.py "roofline"):
 * gnx_profile(ctx, 1) starts recording, gnx_profile_report writes one
 * "kernel\tlaunches\ttotal_ms\n" line per kernel, gnx_profile(ctx, 0) stops. */
int gnx_profile(gnx_ctx* ctx, int32_t enable);
int gnx_profile_report(gnx_ctx* ctx, char* buf, int64_t buflen);

#ifdef __cplusplus
}
#endif
#endif /* GNX_B200_H */
