// gnx_api.cu -- C-ABI of libgnxb200.so (see include/gnx_b200.h).  Host-side orchestration
// of the sm_100a kernels in gnx_kernels.cuh: one ctx per Species, all state resident in
// HBM, one stream, no host round trip inside a time step.
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include "gnx_kernels.cuh"
#include "gnx_genome_init.cuh"
#include "gnx_simplify.cuh"

static thread_local std::string g_last_error;

#define CK(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) {                                                                 \
      char buf_[512];                                                                        \
      snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,       \
               cudaGetErrorString(e_));                                                      \
      g_last_error = buf_;                                                                   \
      return GNX_ERR_CUDA;                                                                   \
    }                                                                                        \
  } while (0)

#define ARG(cond, msg)                                                                       \
  do {                                                                                       \
    if (!(cond)) {                                                                           \
      g_last_error = std::string("invalid argument: ") + msg;                                \
      return GNX_ERR_ARG;                                                                    \
    }                                                                                        \
  } while (0)

#define USE_DEVICE(ctx)                                         \
  do {                                                          \
    if (!(ctx)->capturing) CK(cudaSetDevice((ctx)->device));    \
  } while (0)

struct ProfSpan {
  std::string name;
  cudaEvent_t e0, e1;
};

struct gnx_ctx {
  gnx_config_t cfg;
  bool profiling = false;
  std::vector<ProfSpan> spans;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;          // density chain of the fused step (one_step)
  int32_t* burnin_counts = nullptr;        // gnx_burnin_cell_stats: [2][Y][X] counts (now, previous call) + two sums
  int32_t* strip_burnin = nullptr;         // gnx_strip_burnin_*: [2][ly1 - ly0][X] band counts + two sums + outside
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // one fused step captured as a CUDA graph (every kernel reads its sizes from the device
  // counters, so the same graph serves every step); re-captured when any kernel argument changes
  bool use_graph = true;
  cudaGraphExec_t graph_exec = nullptr;
  int graph_kernels = 0;
  int64_t steps_done = 0;
  std::vector<unsigned char> graph_key;
  int device = 0;
  int num_sms = 148;
  int Wq = 0, Wwords = 0;            // 128-bit units / 32-bit words per homologue of a genotype row
  int WqL = 0;                      // 128-bit units of L bits (by-locus rows, recombination paths as simulated)
  // column layout (gnx_create_cols): a row holds col_cap columns, column j = non-neutral locus col_locus[j]
  bool cols = false;
  int col_cap = 0;
  int32_t* d_cols = nullptr;        // [1 + 2L]: n_cols, col_locus[L], col_of_locus[L] (-1: no column)
  int ncell = 0;
  int64_t n_hint = 0;               // last population size seen by the host (grid sizing only)
  Pop pop{};
  Land land{};
  Traits traits{};
  Dens dens{};
  Work work{};
  Params prm{};
  DevDraws draws{};
  Tsk tsk{};
  Mut mut{};
  bool mut_delet = false;
  std::vector<void*> mut_allocs;
  // host copies of what gnx_set_traits was given (Trait.loci / alpha in the caller's order, dom):
  // gnx_set_mutation builds the device-editable trait tables from them
  std::vector<std::vector<int32_t>> host_trait_loci;
  std::vector<std::vector<double>> host_trait_alpha;
  std::vector<int8_t> host_dom;
  Traits traits_as_set{};            // the tables gnx_set_traits built (restored when mutation lets go of them)
  std::vector<uint32_t> host_paths;   // packed recombination paths (breakpoint CSR for tskit records)
  std::vector<void*> tsk_allocs;
  Counters* d_c = nullptr;
  std::vector<void*> allocs;        // everything cudaMalloc'ed for the ctx lifetime
  std::vector<std::pair<void*, size_t>> draw_bufs;   // injected-draw buffers (pointer, capacity), one per site
  std::vector<void*> trait_allocs;
  std::vector<void*> dens_allocs;
  double* d_rasters = nullptr;
  float* d_surf_f32[2] = {nullptr, nullptr};
  double* d_K = nullptr;
  uint4* d_stage_genomes = nullptr;   // species-order staging for upload/download
  double* d_stage_z = nullptr;        // [n][T] row-major staging of phenotypes
  bool pair_phenotype = false;      // every trait polygenic and no dominance: k_gametes may walk the trait table once per two offspring
  bool have_density = false, have_paths = false, have_traits = false, have_rasters = false;
  int64_t launches = 0;
  int burn = 0;
  bool capturing = false;               // inside cudaStreamBeginCapture/EndCapture of the whole-step graph
  bool pending = false;                 // host mirror of Counters.pending (set by the fused step, cleared by materialise / upload)
  bool order_valid = false;             // pop.ord / work.inv describe the current entries
  uint32_t* d_cs_tab = nullptr;
  int64_t records_pending = 0;          // step records written since the last gnx_read_step_records
  int64_t graph_launches = 0, graph_captures = 0;
  // growth guard (gnx_set_growth_guard): the device status block k_step_guard writes, and the last
  // gnx_step batch as the host saw it (steps enqueued, steps run and a stop found by a host check)
  bool grow_guard = false;
  gnx_step_status_t* d_grow = nullptr;
  int32_t tsk_max_bp = 0;               // largest breakpoint count of a cached path (gnx_tskit_enable)
  int64_t grow_enqueued = 0, grow_host_run = 0;
  bool grow_host_stop = false, grow_graph = false;   // grow_graph: the batch launched a guarded graph
  gnx_step_status_t grow_host_need{};
  void* d_paths = nullptr;
  void* d_surf_tab[2] = {nullptr, nullptr};
  // strip domain decomposition (gnx_strip.cuh)
  Strip strip_h{};                      // host copy of the device-resident descriptor
  Strip* d_strip = nullptr;             // nullptr: the landscape is not decomposed
  unsigned char* strip_block = nullptr; // [counters | 4 receive buffers]: one allocation, one IPC handle
  size_t strip_block_bytes = 0;
  int64_t strip_sync_off = 0;
  int strip_connected = 0;            // peers whose synchronisation page is mapped
  int64_t strip_buf_off[STRIP_N_BUF] = {0, 0, 0, 0};
  std::vector<void*> strip_allocs;
  std::vector<void*> strip_ipc_opened;
  // staged device genome assignment (gnx_genome_init_*): 0 idle, 1 selecting, 3 selected, 2 genomes written
  int gi_stage = 0;
  bool gi_tskit = false;
  std::vector<long long> gi_carriers;   // n_carriers as given to gnx_genome_init_begin
  GiLocus* d_gi_state = nullptr;
  uint32_t* d_gi_lkey = nullptr;
  uint8_t* d_gi_write = nullptr;        // [L] loci whose bits are written
  int32_t* d_gi_hist = nullptr;         // [L][GI_BINS]
  int32_t* d_gi_active = nullptr;       // [2]: loci still active, loci with more carriers than keys
  int64_t gi_t = 0;                     // Counters.t when the genomes were written (the rows describe that population)
  std::vector<void*> gi_allocs;
  // the last gnx_simplify result (device columns and their sizes) until gnx_simplify_result copies it out
  gnx_tables_t simp{};
  std::vector<void*> simp_allocs;
};

template <class T>
static int dmalloc(gnx_ctx* ctx, T** p, size_t count, std::vector<void*>* bucket = nullptr) {
  void* q = nullptr;
  size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
  CK(cudaMalloc(&q, bytes));
  CK(cudaMemsetAsync(q, 0, bytes, ctx->stream));
  (bucket ? *bucket : ctx->allocs).push_back(q);
  *p = (T*)q;
  return GNX_OK;
}
#define DM(...)                                   \
  do {                                            \
    int r_ = dmalloc(__VA_ARGS__);                \
    if (r_ != GNX_OK) return r_;                  \
  } while (0)

static inline int grid_for(const gnx_ctx* ctx, int per_sm) { return ctx->num_sms * per_sm; }
// Grid for a grid-stride kernel whose per-item cost varies (mate search, death): many CTAs let
// the hardware even out the load, but never more than ~one item per thread for the population
// the host last saw (n_hint; the kernels read the true size on the device, so an estimate that
// is off only changes the number of passes).  Matters when several small replicate populations
// share a GPU: their launches must not each carry thousands of empty CTAs.
static inline int grid_cap(const gnx_ctx* ctx, int per_sm, int threads, double scale = 1.0) {
  const long long want = (long long)std::ceil((double)ctx->n_hint * 1.25 * scale / threads);
  const long long hi = (long long)ctx->num_sms * per_sm;
  if (ctx->n_hint <= 0) return (int)hi;
  return (int)std::max<long long>(ctx->num_sms, std::min(hi, want));
}
// CTAs per SM of grid-stride kernels whose per-item cost varies
constexpr int MOVE_KEY_GRID = 8;     // k_move_key
constexpr int NEWBORNS_GRID = 8;     // k_newborns
constexpr int DEATH_GRID = 32;       // k_death
constexpr int REGRID_GRID = 8;       // k_bucket, k_regrid
constexpr int SCAN_GRID = 8;         // scan_reduce_kernel, scan_apply_kernel

// ---- optional per-kernel timing (bench.py roofline): CUDA events on the ctx stream around
// every launch, accumulated by kernel name.
static void prof_begin(gnx_ctx* ctx, const char* name) {
  if (!ctx->profiling) return;
  ProfSpan sp;
  sp.name = name;
  cudaEventCreate(&sp.e0);
  cudaEventCreate(&sp.e1);
  cudaEventRecord(sp.e0, ctx->stream);
  ctx->spans.push_back(sp);
}
static void prof_end(gnx_ctx* ctx) {
  if (!ctx->profiling || ctx->spans.empty()) return;
  cudaEventRecord(ctx->spans.back().e1, ctx->stream);
}
#define PROF(ctx, name) prof_begin(ctx, name)
#define LAUNCHED(ctx)        \
  do {                       \
    prof_end(ctx);           \
    (ctx)->launches++;       \
    CK(cudaGetLastError());  \
  } while (0)

extern "C" const char* gnx_strerror(int code) {
  switch (code) {
    case GNX_OK: return "ok";
    case GNX_ERR_CUDA: return "CUDA runtime error";
    case GNX_ERR_ARG: return "invalid argument";
    case GNX_ERR_CAPACITY: return "population outgrew ctx capacity";
    case GNX_ERR_DRAWS: return "injected draw buffer exhausted";
    case GNX_ERR_STATE: return "call made in the wrong state";
    case GNX_ERR_MUTABLES: return "no mutable locus left";
    default: return "unknown error";
  }
}
extern "C" const char* gnx_last_error(void) { return g_last_error.c_str(); }
extern "C" int gnx_abi_version(void) { return GNX_ABI_VERSION; }

static void mating_grid(const gnx_config_t& c, double* cs, int* ncx, int* ncy) {
  // Cells of side >= radius*(1+1e-7), doubled until <= 2^22 cells (DESIGN.md "mating grid")
  double s = c.mating_radius > 0 ? c.mating_radius * 1.0000001 : (double)std::max(c.dim_x, c.dim_y);
  while (((long long)(c.dim_x / s) + 1) * ((long long)(c.dim_y / s) + 1) > (1ll << 22)) s *= 2.0;
  *cs = s;
  *ncx = (int)(c.dim_x / s) + 1;
  *ncy = (int)(c.dim_y / s) + 1;
}

static int create_impl(const gnx_config_t* cfg, gnx_ctx* ctx);
extern "C" int gnx_destroy(gnx_ctx* ctx);

static int create_ctx(const gnx_config_t* cfg, int32_t col_cap, int32_t n_cols, const int32_t* host_col_locus,
                      gnx_ctx** out) {
  ARG(cfg && out, "null cfg/out");
  ARG(cfg->abi_version == GNX_ABI_VERSION, "abi_version mismatch");
  ARG(cfg->dim_x > 0 && cfg->dim_y > 0 && cfg->n_layers > 0 && cfg->n_layers <= GNX_MAX_LAYERS, "landscape dims");
  ARG(cfg->capacity > 0 && cfg->capacity < (1ll << 31) - 4096, "capacity");
  ARG(cfg->n_traits >= 0 && cfg->n_traits <= GNX_MAX_TRAITS, "n_traits");
  ARG(cfg->L >= 0, "L");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (ndev == 0) { g_last_error = "no CUDA device"; return GNX_ERR_CUDA; }
  if (col_cap > 0) {
    ARG(cfg->L > 0 && n_cols >= 0 && n_cols <= col_cap && (n_cols == 0 || host_col_locus), "columns");
    std::vector<uint8_t> seen(cfg->L, 0);
    for (int j = 0; j < n_cols; ++j) {
      ARG(host_col_locus[j] >= 0 && host_col_locus[j] < cfg->L, "column locus out of range");
      ARG(!seen[host_col_locus[j]], "a locus holds two columns");
      seen[host_col_locus[j]] = 1;
    }
  }
  gnx_ctx* ctx = new gnx_ctx();
  ctx->cfg = *cfg;
  ctx->cols = col_cap > 0;
  ctx->col_cap = 128 * ((std::max(col_cap, 0) + 127) / 128);
  int r = create_impl(cfg, ctx);
  if (r == GNX_OK && ctx->cols) {
    const int L = cfg->L;
    std::vector<int32_t> h((size_t)1 + 2 * L, 0);
    h[0] = n_cols;
    for (int l = 0; l < L; ++l) h[1 + L + l] = -1;
    for (int j = 0; j < n_cols; ++j) {
      h[1 + j] = host_col_locus[j];
      h[1 + L + host_col_locus[j]] = j;
    }
    r = dmalloc(ctx, &ctx->d_cols, h.size());
    if (r == GNX_OK &&
        (cudaMemcpyAsync(ctx->d_cols, h.data(), h.size() * 4, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
         cudaStreamSynchronize(ctx->stream) != cudaSuccess)) {
      g_last_error = "copying the column map";
      r = GNX_ERR_CUDA;
    }
  }
  if (r != GNX_OK) {                       // streams, events and every buffer allocated so far
    const std::string keep = g_last_error;
    gnx_destroy(ctx);
    g_last_error = keep;
    return r;
  }
  *out = ctx;
  return GNX_OK;
}

extern "C" int gnx_create(const gnx_config_t* cfg, gnx_ctx** out) { return create_ctx(cfg, 0, 0, nullptr, out); }

extern "C" int gnx_create_cols(const gnx_config_t* cfg, int32_t col_capacity, int32_t n_cols,
                               const int32_t* host_col_locus, gnx_ctx** out) {
  ARG(col_capacity > 0, "col_capacity");
  return create_ctx(cfg, col_capacity, n_cols, host_col_locus, out);
}

// Quantile table of |theta|, theta ~ von Mises(0, kappa): the half-distribution's inverse CDF at
// u = k / VM_TAB_CELLS (k = 0..VM_TAB_CELLS), then the last cell again at VM_TAB_FINE sub-cells.
// pdf ~ exp(kappa (cos t - 1)) integrated by the trapezoid rule on 2^20 points in double.
static void build_vm_table(double kappa, std::vector<float>* out) {
  const int n = 1 << 20;
  std::vector<double> cdf(n + 1);
  const double h = M_PI / n;
  double acc = 0.0, prev = 1.0;
  cdf[0] = 0.0;
  for (int i = 1; i <= n; ++i) {
    const double f = std::exp(kappa * (std::cos(i * h) - 1.0));
    acc += 0.5 * (prev + f) * h;
    prev = f;
    cdf[i] = acc;
  }
  for (int i = 0; i <= n; ++i) cdf[i] /= acc;
  auto quantile = [&](double u) {
    if (u <= 0.0) return 0.0;
    if (u >= 1.0) return M_PI;
    const int i = (int)(std::upper_bound(cdf.begin(), cdf.end(), u) - cdf.begin());      // cdf[i-1] <= u < cdf[i]
    const double c0 = cdf[i - 1], c1 = cdf[i];
    return ((i - 1) + (c1 > c0 ? (u - c0) / (c1 - c0) : 0.0)) * h;
  };
  out->resize(VM_TAB_LEN);
  for (int k = 0; k <= VM_TAB_CELLS; ++k) (*out)[k] = (float)quantile((double)k / VM_TAB_CELLS);
  for (int k = 0; k <= VM_TAB_FINE; ++k)
    (*out)[VM_TAB_CELLS + 1 + k] = (float)quantile(1.0 - (1.0 - (double)k / VM_TAB_FINE) / VM_TAB_CELLS);
}

static int create_impl(const gnx_config_t* cfg, gnx_ctx* ctx) {
  CK(cudaGetDevice(&ctx->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, ctx->device));
  ctx->num_sms = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  if (const char* ng = getenv("GNX_NO_GRAPH")) ctx->use_graph = !(ng[0] && ng[0] != '0');
  const int64_t cap = cfg->capacity;
  ctx->WqL = std::max(1, (cfg->L + 127) / 128);
  ctx->Wq = ctx->cols ? ctx->col_cap / 128 : ctx->WqL;
  ctx->Wwords = 4 * ctx->Wq;
  Pop& P = ctx->pop;
  P.cap = (int)cap;
  P.Wq = ctx->Wq;
  P.T = cfg->n_traits;
  for (int h = 0; h < 2; ++h) {
    DM(ctx, &P.xy[h], cap);
    DM(ctx, &P.age[h], cap);
    DM(ctx, &P.sex[h], cap);
    DM(ctx, &P.idx[h], cap);
    DM(ctx, &P.gslot[h], cap);
    DM(ctx, &P.z[h], cap * std::max(1, cfg->n_traits));
    DM(ctx, &P.fit[h], cap);
  }
  DM(ctx, &P.G, (size_t)cap * 2 * ctx->Wq);
  DM(ctx, &P.free_slots, cap);
  DM(ctx, &ctx->d_stage_genomes, (size_t)cap * 2 * ctx->Wq);
  DM(ctx, &ctx->d_stage_z, (size_t)cap * std::max(1, cfg->n_traits));
  // landscape
  Land& Ld = ctx->land;
  Ld.X = cfg->dim_x;
  Ld.Y = cfg->dim_y;
  Ld.n_layers = cfg->n_layers;
  Ld.max_x = cfg->dim_x - 0.001;
  Ld.max_y = cfg->dim_y - 0.001;
  mating_grid(*cfg, &Ld.cell_size, &Ld.ncx, &Ld.ncy);
  Ld.inv_cell_size = 1.0 / Ld.cell_size;
  ARG(Ld.ncx < 65536 && Ld.ncy < 65536, "mating grid has more than 65535 cells along one axis");
  ctx->ncell = Ld.ncx * Ld.ncy;
  const size_t plane = (size_t)cfg->dim_x * cfg->dim_y;
  DM(ctx, &ctx->d_rasters, plane * cfg->n_layers);
  DM(ctx, &ctx->d_K, plane);
  Ld.rasters = ctx->d_rasters;
  {
    const int mode[2] = {cfg->move ? cfg->move_surf_mode : GNX_SURF_NONE, cfg->disp_surf_mode};
    const int lyr[2] = {cfg->move_surf_layer, cfg->disp_surf_layer};
    for (int k = 0; k < 2; ++k) {
      if (mode[k] != GNX_SURF_ONTHEFLY) continue;
      if (k == 1 && mode[0] == GNX_SURF_ONTHEFLY && lyr[0] == lyr[1]) {
        ctx->d_surf_f32[1] = ctx->d_surf_f32[0];
      } else {
        DM(ctx, &ctx->d_surf_f32[k], plane);
      }
      Ld.surf_f32[k] = ctx->d_surf_f32[k];
    }
  }
  Ld.K = ctx->d_K;
  // work
  Work& W = ctx->work;
  DM(ctx, &W.cell_count, (size_t)ctx->ncell + 1);
  DM(ctx, &W.cell_start, (size_t)ctx->ncell + 1);
  DM(ctx, &W.mkey, cap);
  DM(ctx, &W.bucket, cap);
  DM(ctx, &W.skey, cap);
  DM(ctx, &W.inv, cap);
  DM(ctx, &W.perm, cap);
  for (int h = 0; h < 2; ++h) {
    DM(ctx, &W.sort_keys[h], cap);
    DM(ctx, &W.sort_vals[h], cap);
    DM(ctx, &P.ord[h], cap);
  }
  DM(ctx, &W.sort_hist, (size_t)256 * (cap / RS_TILE + 2));
  {
    double* sc = nullptr;
    DM(ctx, &sc, (size_t)2 * cap * std::max(1, cfg->n_traits));
    W.scratch = sc;
  }
  DM(ctx, &W.mate, cap);
  // a cell is crowded when focals x candidates of its 3x3 block reaches FM_HEAVY_WORK; it
  // contributes one work item per 32 focals, so n / 32 items plus one per crowded cell (few
  // hundred candidates are shared by the at most 9 cells around them): below n / 4 in all
  W.heavy_cap = (int32_t)(cap / 4 + 1024);
  DM(ctx, &W.heavy, (size_t)W.heavy_cap);
  DM(ctx, &W.fm_list, (size_t)cap);
  DM(ctx, &W.fm_count, 4);
  DM(ctx, &W.n_nbrs, cap);
  DM(ctx, &W.pairs, 2 * cap);
  DM(ctx, &W.pair_slots, 2 * cap);
  DM(ctx, &W.nb, cap);
  DM(ctx, &W.off_start, cap);
  DM(ctx, &W.off_pair, cap);
  DM(ctx, &W.mid, cap);
  DM(ctx, &W.alive, cap);
  DM(ctx, &W.death_p, cap);
  DM(ctx, &W.disp_tries, cap);
  DM(ctx, &W.tile_sums, (size_t)std::max<int64_t>(std::max<int64_t>(cap, ctx->ncell),
                                                    (int64_t)256 * (cap / RS_TILE + 2)) / SCAN_TILE + 2);
  DM(ctx, &W.scan_ticket, 4);
  DM(ctx, &W.N_rast, plane);
  DM(ctx, &W.NP_rast, plane);
  DM(ctx, &W.d_rast, plane);
  DM(ctx, &W.e_out, (size_t)cap * cfg->n_layers);
  DM(ctx, &W.fix_list, plane);
  DM(ctx, &W.fix_count, 3);
  W.max_records = 1 << 16;
  DM(ctx, &W.records, (size_t)W.max_records);
  DM(ctx, &ctx->d_c, 1);
  // params
  Params& pr = ctx->prm;
  pr.c = *cfg;
  pr.r2 = cfg->mating_radius * cfg->mating_radius;
  pr.burn = 0;
  pr.selection = cfg->n_traits > 0;
  pr.n_paths = cfg->n_recomb_paths;
  pr.paths = nullptr;
  pr.move_tab = pr.disp_tab = nullptr;
  pr.seed_lo = (uint32_t)cfg->seed;
  pr.seed_hi = (uint32_t)(cfg->seed >> 32);
  pr.store_debug = 0;
  pr.ordered = 0;
  {
    // (half cos, half sin) of every float16 direction, numpy's portable float16 semantics: half ->
    // double, cos, rounded to float32, rounded to half (oracle/step_oracle.py _cos_sin)
    std::vector<uint32_t> tab(65536);
    for (uint32_t b = 0; b < 65536; ++b) {
      const uint32_t sign = b >> 15, ex = (b >> 10) & 31u, man = b & 1023u;
      double v;
      if (ex == 0) v = std::ldexp((double)man, -24);
      else if (ex == 31) v = man ? NAN : INFINITY;
      else v = std::ldexp((double)(man | 1024u), (int)ex - 25);
      if (sign) v = -v;
      const __half hc = __float2half_rn((float)std::cos(v)), hs = __float2half_rn((float)std::sin(v));
      unsigned short uc, us;
      memcpy(&uc, &hc, 2);
      memcpy(&us, &hs, 2);
      tab[b] = (uint32_t)uc | ((uint32_t)us << 16);
    }
    DM(ctx, &ctx->d_cs_tab, 65536);
    CK(cudaMemcpyAsync(ctx->d_cs_tab, tab.data(), 65536 * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    pr.cs_tab = ctx->d_cs_tab;
  }
  {
    const int mode[2] = {cfg->move ? cfg->move_surf_mode : GNX_SURF_NONE, cfg->disp_surf_mode};
    const double kappa[2] = {cfg->move_surf_kappa, cfg->disp_surf_kappa};
    pr.vm_tab[0] = pr.vm_tab[1] = nullptr;
    for (int k = 0; k < 2; ++k) {
      if (mode[k] != GNX_SURF_ONTHEFLY) continue;
      if (k == 1 && pr.vm_tab[0] && kappa[0] == kappa[1]) { pr.vm_tab[1] = pr.vm_tab[0]; continue; }
      std::vector<float> tab;
      build_vm_table(kappa[k], &tab);
      float* d = nullptr;
      DM(ctx, &d, tab.size());
      CK(cudaMemcpyAsync(d, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      pr.vm_tab[k] = d;
    }
  }
  memset(&ctx->draws, 0, sizeof ctx->draws);
  ctx->draws.disp_R = std::max(1, cfg->disp_max_tries_injected);
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

static void free_bucket(std::vector<void*>& b) {
  for (void* p : b) cudaFree(p);
  b.clear();
}

// column layout: the current columns (col_locus[0 .. n_cols)) and the column of every locus (-1: none).
// Synchronises.
static int read_cols(gnx_ctx* ctx, std::vector<int32_t>* col_locus, std::vector<int32_t>* col_of_locus = nullptr) {
  const int L = ctx->cfg.L;
  std::vector<int32_t> h((size_t)1 + 2 * L);
  CK(cudaMemcpyAsync(h.data(), ctx->d_cols, h.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  col_locus->assign(h.begin() + 1, h.begin() + 1 + h[0]);
  if (col_of_locus) col_of_locus->assign(h.begin() + 1 + L, h.end());
  return GNX_OK;
}

// the recombination paths as simulated (host_paths, [n_paths][4 WqL]) at the bits of the genotype rows: the
// same array by locus, bit j = the path at locus col_locus[j] in the column layout
static std::vector<uint32_t> paths_at_rows(const gnx_ctx* ctx, const std::vector<int32_t>& col_locus) {
  if (!ctx->cols) return ctx->host_paths;
  const size_t WL = (size_t)4 * ctx->WqL, W = (size_t)4 * ctx->Wq;
  const int n = ctx->cfg.n_recomb_paths;
  std::vector<uint32_t> out((size_t)n * W, 0u);
  for (int p = 0; p < n; ++p)
    for (size_t j = 0; j < col_locus.size(); ++j) {
      const int l = col_locus[j];
      out[p * W + (j >> 5)] |= ((ctx->host_paths[p * WL + (l >> 5)] >> (l & 31)) & 1u) << (j & 31);
    }
  return out;
}

extern "C" int gnx_destroy(gnx_ctx* ctx) {
  if (!ctx) return GNX_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  free_bucket(ctx->allocs);
  for (auto& b : ctx->draw_bufs) if (b.first) cudaFree(b.first);
  ctx->draw_bufs.clear();
  free_bucket(ctx->trait_allocs);
  free_bucket(ctx->dens_allocs);
  free_bucket(ctx->tsk_allocs);
  free_bucket(ctx->mut_allocs);
  free_bucket(ctx->strip_allocs);
  free_bucket(ctx->gi_allocs);
  free_bucket(ctx->simp_allocs);
  for (void* m : ctx->strip_ipc_opened) cudaIpcCloseMemHandle(m);
  ctx->strip_ipc_opened.clear();
  if (ctx->strip_block) cudaFree(ctx->strip_block);
  if (ctx->d_paths) cudaFree(ctx->d_paths);
  if (ctx->burnin_counts) cudaFree(ctx->burnin_counts);
  if (ctx->strip_burnin) cudaFree(ctx->strip_burnin);
  for (int k = 0; k < 2; ++k) if (ctx->d_surf_tab[k]) cudaFree(ctx->d_surf_tab[k]);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
  delete ctx;
  return GNX_OK;
}

// refresh the float32 conductance copies after `layer` (or every layer, -1) changed
static int refresh_surf_f32(gnx_ctx* ctx, int layer) {
  const size_t plane = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  const int lyr[2] = {ctx->cfg.move_surf_layer, ctx->cfg.disp_surf_layer};
  for (int k = 0; k < 2; ++k) {
    if (!ctx->d_surf_f32[k] || (layer >= 0 && layer != lyr[k])) continue;
    if (k == 1 && ctx->d_surf_f32[1] == ctx->d_surf_f32[0]) continue;
    PROF(ctx, "k_raster_to_f32");
    k_raster_to_f32<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(ctx->d_rasters + plane * lyr[k], ctx->d_surf_f32[k], plane);
    LAUNCHED(ctx);
  }
  return GNX_OK;
}

static int set_K(gnx_ctx* ctx) {
  const int ncell = ctx->cfg.dim_x * ctx->cfg.dim_y;
  PROF(ctx, "k_K_from_layer");
  k_K_from_layer<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(
      ctx->d_rasters + (size_t)ctx->cfg.K_layer * ncell, ctx->d_K, ctx->cfg.K_factor, ncell);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_set_rasters(gnx_ctx* ctx, const double* host_rasters) {
  ARG(ctx && host_rasters, "null");
  USE_DEVICE(ctx);
  const size_t plane = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  CK(cudaMemcpyAsync(ctx->d_rasters, host_rasters, plane * ctx->cfg.n_layers * sizeof(double),
                     cudaMemcpyHostToDevice, ctx->stream));
  ctx->have_rasters = true;
  int r = refresh_surf_f32(ctx, -1);
  if (r != GNX_OK) return r;
  return set_K(ctx);
}

extern "C" int gnx_set_raster(gnx_ctx* ctx, int32_t layer, const double* host_raster) {
  ARG(ctx && host_raster && layer >= 0 && layer < ctx->cfg.n_layers, "layer");
  USE_DEVICE(ctx);
  const size_t plane = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  CK(cudaMemcpyAsync(ctx->d_rasters + plane * layer, host_raster, plane * sizeof(double), cudaMemcpyHostToDevice,
                     ctx->stream));
  int r = refresh_surf_f32(ctx, layer);
  if (r != GNX_OK) return r;
  if (layer == ctx->cfg.K_layer) return set_K(ctx);      // model.py:651-652 (Species._set_K)
  return GNX_OK;
}

// Species change events (ops/change.py:612-742).
// Demographic change: the change functions rewrite the carrying-capacity raster itself
// (`spp.K *= size`, `spp.K = changer.base_K * size`, change.py:633-649); the caller hands the
// new raster over.  It stays until the next gnx_set_K or until Species._set_K runs again
// (gnx_set_raster on the K layer), exactly like the reference's attribute.
extern "C" int gnx_set_K(gnx_ctx* ctx, const double* host_K) {
  ARG(ctx && host_K, "null");
  USE_DEVICE(ctx);
  const size_t plane = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  CK(cudaMemcpyAsync(ctx->d_K, host_K, plane * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));        // the host buffer may be a temporary
  return GNX_OK;
}

// Life-history change: `setattr(spp, parameter, val)` (change.py:735-742) for the scalar
// parameters the step reads.  Everything that fixes a buffer size or the mating grid must be
// unchanged; the next gnx_step re-captures its graph (the parameters are kernel arguments).
extern "C" int gnx_set_life_history(gnx_ctx* ctx, const gnx_config_t* cfg) {
  ARG(ctx && cfg, "null");
  USE_DEVICE(ctx);
  ARG(cfg->abi_version == GNX_ABI_VERSION, "abi_version");
  const gnx_config_t& o = ctx->cfg;
  ARG(cfg->dim_x == o.dim_x && cfg->dim_y == o.dim_y && cfg->n_layers == o.n_layers && cfg->capacity == o.capacity &&
          cfg->L == o.L && cfg->n_recomb_paths == o.n_recomb_paths && cfg->n_traits == o.n_traits &&
          cfg->use_dom == o.use_dom,
      "gnx_set_life_history cannot change the landscape, capacity or genomic architecture");
  ARG(cfg->mating_radius == o.mating_radius, "gnx_set_life_history cannot change mating_radius (it fixes the mating grid)");
  ARG(cfg->move_surf_mode == o.move_surf_mode && cfg->disp_surf_mode == o.disp_surf_mode &&
          cfg->move_surf_layer == o.move_surf_layer && cfg->disp_surf_layer == o.disp_surf_layer &&
          cfg->surf_approx_len == o.surf_approx_len && cfg->disp_max_tries_injected == o.disp_max_tries_injected &&
          cfg->K_layer == o.K_layer && cfg->seed == o.seed,
      "gnx_set_life_history cannot change the conductance-surface setup, K layer or seed");
  ARG(cfg->b >= 0 && cfg->b <= 1 && cfg->d_min <= cfg->d_max, "b / d_min / d_max");
  if (cfg->n_births_fixed) ARG((int32_t)cfg->n_births_lambda >= 1, "n_births_fixed needs n_births_distr_lambda >= 1");
  CK(cudaStreamSynchronize(ctx->stream));
  const bool k_changed = cfg->K_factor != o.K_factor;
  ctx->cfg = *cfg;
  ctx->prm.c = *cfg;
  if (k_changed && ctx->have_rasters) return set_K(ctx);
  return GNX_OK;
}

template <class T>
static int upload_vec(gnx_ctx* ctx, const std::vector<T>& v, const T** dev, std::vector<void*>& bucket) {
  T* d = nullptr;
  int r = dmalloc(ctx, &d, v.size(), &bucket);
  if (r != GNX_OK) return r;
  if (!v.empty()) CK(cudaMemcpyAsync(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *dev = d;
  return GNX_OK;
}

extern "C" int gnx_set_traits(gnx_ctx* ctx, int32_t n_traits, const gnx_trait_t* traits, const int8_t* host_dom) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  ARG(n_traits == ctx->cfg.n_traits, "n_traits differs from config");
  CK(cudaStreamSynchronize(ctx->stream));
  free_bucket(ctx->trait_allocs);
  if (ctx->mut.enabled && ctx->mut.own_tables) {       // the mutation tables alias the old trait tables
    free_bucket(ctx->mut_allocs);
    memset(&ctx->mut, 0, sizeof ctx->mut);
    ctx->mut_delet = false;
  }
  Traits& T = ctx->traits;
  memset(&T, 0, sizeof T);
  const int Wq = ctx->Wq;
  ctx->host_trait_loci.assign(n_traits, {});
  ctx->host_trait_alpha.assign(n_traits, {});
  ctx->host_dom.clear();
  if (host_dom) ctx->host_dom.assign(host_dom, host_dom + ctx->cfg.L);
  std::vector<int32_t> te_locus;
  std::vector<double> te_alpha, te_dom;
  struct TraitEntry { int32_t off, mask; double half_alpha; };    // Traits::te_pack
  static_assert(sizeof(TraitEntry) == 16, "TraitEntry is one 128-bit load");
  std::vector<TraitEntry> te_pack;
  const int NW = 4 * Wq;      // CSR over 32-bit words
  std::vector<int32_t> chunk_ptr((size_t)std::max(1, n_traits) * (NW + 1), 0);
  const size_t plane = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  std::vector<int32_t> col_locus, col_of;                      // column layout: the bit of a locus is its column
  if (ctx->cols) {
    int r = read_cols(ctx, &col_locus, &col_of);
    if (r != GNX_OK) return r;
  }
  for (int t = 0; t < n_traits; ++t) {
    const gnx_trait_t& tr = traits[t];
    ARG(tr.n_loci >= 0 && (tr.n_loci == 0 || (tr.host_loci && tr.host_alpha)), "trait loci");
    ARG(tr.layer >= 0 && tr.layer < ctx->cfg.n_layers, "trait layer");
    std::vector<int> order(tr.n_loci);
    for (int k = 0; k < tr.n_loci; ++k) order[k] = k;
    for (int k = 0; k < tr.n_loci; ++k) {
      ARG(tr.host_loci[k] >= 0 && tr.host_loci[k] < ctx->cfg.L, "trait locus out of range");
      ARG(!ctx->cols || col_of[tr.host_loci[k]] >= 0, "trait locus without a column");
    }
    // Trait.loci order (by locus) for the host copies, the bit read for the tables
    auto bit_of = [&](int k) { return ctx->cols ? col_of[tr.host_loci[k]] : tr.host_loci[k]; };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return tr.host_loci[a] < tr.host_loci[b]; });
    for (int kk = 0; kk < tr.n_loci; ++kk) {
      ctx->host_trait_loci[t].push_back(tr.host_loci[order[kk]]);
      ctx->host_trait_alpha[t].push_back(tr.host_alpha[order[kk]]);
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return bit_of(a) < bit_of(b); });
    int q = 0;
    chunk_ptr[(size_t)t * (NW + 1)] = (int32_t)te_locus.size();
    for (int kk = 0; kk < tr.n_loci; ++kk) {
      const int k = order[kk];
      const int locus = tr.host_loci[k], bit = bit_of(k);
      while (q < bit / 32) chunk_ptr[(size_t)t * (NW + 1) + (++q)] = (int32_t)te_locus.size();
      te_locus.push_back(bit);
      te_alpha.push_back(tr.host_alpha[k]);
      te_dom.push_back(host_dom ? 1.0 + (double)host_dom[locus] : 1.0);
      te_pack.push_back(TraitEntry{(bit >> 5) * 8, (int32_t)(1u << (bit & 31)), 0.5 * tr.host_alpha[k]});
    }
    while (q < NW) chunk_ptr[(size_t)t * (NW + 1) + (++q)] = (int32_t)te_locus.size();
    T.n_loci[t] = tr.n_loci;
    T.phi[t] = tr.phi;
    T.gamma[t] = tr.gamma;
    T.layer[t] = tr.layer;
    T.univ_adv[t] = tr.univ_adv;
    T.phi_rast[t] = nullptr;
    if (tr.host_phi_raster) {
      double* d = nullptr;
      DM(ctx, &d, plane, &ctx->trait_allocs);
      CK(cudaMemcpyAsync(d, tr.host_phi_raster, plane * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
      T.phi_rast[t] = d;
    }
  }
  int r;
  if ((r = upload_vec(ctx, te_locus, &T.te_locus, ctx->trait_allocs)) != GNX_OK) return r;
  if ((r = upload_vec(ctx, te_alpha, &T.te_alpha, ctx->trait_allocs)) != GNX_OK) return r;
  if (ctx->cfg.use_dom && host_dom) {
    if ((r = upload_vec(ctx, te_dom, &T.te_dom, ctx->trait_allocs)) != GNX_OK) return r;
  } else {
    T.te_dom = nullptr;
  }
  if ((r = upload_vec(ctx, chunk_ptr, &T.chunk_ptr, ctx->trait_allocs)) != GNX_OK) return r;
  const TraitEntry* d_pack = nullptr;
  if ((r = upload_vec(ctx, te_pack, &d_pack, ctx->trait_allocs)) != GNX_OK) return r;
  T.te_pack = d_pack;
  ctx->pair_phenotype = !T.te_dom && n_traits > 0;
  for (int t = 0; t < n_traits; ++t) if (traits[t].n_loci <= 1) ctx->pair_phenotype = false;
  ctx->have_traits = true;
  ctx->traits_as_set = T;
  return GNX_OK;
}

extern "C" int gnx_set_recomb_paths(gnx_ctx* ctx, const uint32_t* host_packed_paths) {
  ARG(ctx && host_packed_paths, "null");
  USE_DEVICE(ctx);
  ARG(ctx->cfg.n_recomb_paths > 0, "n_recomb_paths");
  uint4* d = nullptr;
  const size_t n = (size_t)ctx->cfg.n_recomb_paths * ctx->WqL;     // as simulated: by locus
  CK(cudaStreamSynchronize(ctx->stream));
  if (ctx->mut.enabled && ctx->mut.tskit_layout) {     // the mutation bookkeeping patches the old path array
    if (ctx->mut.own_tables) ctx->traits = ctx->traits_as_set;
    free_bucket(ctx->mut_allocs);
    memset(&ctx->mut, 0, sizeof ctx->mut);
    ctx->mut_delet = false;
  }
  if (ctx->d_paths) { cudaFree(ctx->d_paths); ctx->d_paths = nullptr; }
  ctx->host_paths.assign(host_packed_paths, host_packed_paths + n * 4);
  std::vector<int32_t> col_locus;
  if (ctx->cols) {
    int r = read_cols(ctx, &col_locus);
    if (r != GNX_OK) return r;
  }
  const std::vector<uint32_t> rows = paths_at_rows(ctx, col_locus);   // what k_gametes reads
  CK(cudaMalloc((void**)&d, std::max<size_t>(rows.size() / 4, 1) * sizeof(uint4)));
  ctx->d_paths = d;
  CK(cudaMemcpyAsync(d, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->prm.paths = d;
  ctx->have_paths = true;
  return GNX_OK;
}

extern "C" int gnx_set_surface_tables(gnx_ctx* ctx, const uint16_t* host_move_f16, const uint16_t* host_disp_f16) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  const size_t n = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y * std::max(1, ctx->cfg.surf_approx_len);
  CK(cudaStreamSynchronize(ctx->stream));
  const uint16_t* src[2] = {host_move_f16, host_disp_f16};
  for (int k = 0; k < 2; ++k) {
    if (!src[k]) continue;
    // a changed layer re-builds its table (change.py:597-606): the old buffer is released
    if (ctx->d_surf_tab[k]) { cudaFree(ctx->d_surf_tab[k]); ctx->d_surf_tab[k] = nullptr; }
    __half* d = nullptr;
    CK(cudaMalloc((void**)&d, n * 2));
    ctx->d_surf_tab[k] = d;
    CK(cudaMemcpyAsync(d, src[k], n * 2, cudaMemcpyHostToDevice, ctx->stream));
    (k == 0 ? ctx->prm.move_tab : ctx->prm.disp_tab) = d;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

// ---- Clough-Tocher: Bezier ordinates -> monomial coefficients (setup) -----------------
// w on micro-triangle k (b_k = smallest barycentric coordinate), written exactly as
// scipy/interpolate/interpnd.pyx `_clough_tocher_2d_single` evaluates it.
static double ct_w_forced(const double* c, int k, double b0, double b1) {
  const double b[3] = {b0, b1, 1.0 - b0 - b1};
  const double minval = b[k];
  const double b1_ = b[0] - minval, b2 = b[1] - minval, b3 = b[2] - minval, b4 = 3 * minval;
  const double c3000 = c[0], c0300 = c[1], c0030 = c[2], c0003 = c[3], c2100 = c[4], c2010 = c[5], c2001 = c[6],
               c0210 = c[7], c0201 = c[8], c0021 = c[9], c1200 = c[10], c1020 = c[11], c1002 = c[12],
               c0120 = c[13], c0102 = c[14], c0012 = c[15], c1101 = c[16], c1011 = c[17], c0111 = c[18];
  const double B1 = b1_;
  return B1 * B1 * B1 * c3000 + 3 * B1 * B1 * b2 * c2100 + 3 * B1 * B1 * b3 * c2010 + 3 * B1 * B1 * b4 * c2001 +
         3 * B1 * b2 * b2 * c1200 + 6 * B1 * b2 * b4 * c1101 + 3 * B1 * b3 * b3 * c1020 + 6 * B1 * b3 * b4 * c1011 +
         3 * B1 * b4 * b4 * c1002 + b2 * b2 * b2 * c0300 + 3 * b2 * b2 * b3 * c0210 + 3 * b2 * b2 * b4 * c0201 +
         3 * b2 * b3 * b3 * c0120 + 6 * b2 * b3 * b4 * c0111 + 3 * b2 * b4 * b4 * c0102 + b3 * b3 * b3 * c0030 +
         3 * b3 * b3 * b4 * c0021 + 3 * b3 * b4 * b4 * c0012 + b4 * b4 * b4 * c0003;
}

// M_k (10 x 19): w = sum_r (M_k c)_r * mono_r(b0, b1), mono order 1, b1, b1^2, b1^3, b0, b0 b1,
// b0 b1^2, b0^2, b0^2 b1, b0^3.  Obtained by interpolation on the 10 nodes (i/3, j/3).
static void ct_build_mono(double* M /* [3][10][19] */) {
  double pts[10][2];
  int np = 0;
  for (int i = 0; i <= 3; ++i)
    for (int j = 0; i + j <= 3; ++j) { pts[np][0] = i / 3.0; pts[np][1] = j / 3.0; ++np; }
  auto mono = [](double b0, double b1, double* out) {
    out[0] = 1; out[1] = b1; out[2] = b1 * b1; out[3] = b1 * b1 * b1; out[4] = b0; out[5] = b0 * b1;
    out[6] = b0 * b1 * b1; out[7] = b0 * b0; out[8] = b0 * b0 * b1; out[9] = b0 * b0 * b0;
  };
  for (int k = 0; k < 3; ++k) {
    // augmented system V x = W for the 19 unit coefficient vectors at once
    double A[10][10 + 19];
    for (int p = 0; p < 10; ++p) {
      mono(pts[p][0], pts[p][1], A[p]);
      for (int m = 0; m < 19; ++m) {
        double e[19] = {0};
        e[m] = 1.0;
        A[p][10 + m] = ct_w_forced(e, k, pts[p][0], pts[p][1]);
      }
    }
    for (int col = 0; col < 10; ++col) {           // Gauss-Jordan with partial pivoting
      int piv = col;
      for (int r = col + 1; r < 10; ++r) if (fabs(A[r][col]) > fabs(A[piv][col])) piv = r;
      if (piv != col) for (int q = 0; q < 29; ++q) std::swap(A[col][q], A[piv][q]);
      const double inv = 1.0 / A[col][col];
      for (int q = 0; q < 29; ++q) A[col][q] *= inv;
      for (int r = 0; r < 10; ++r) {
        if (r == col) continue;
        const double f = A[r][col];
        if (f != 0.0) for (int q = 0; q < 29; ++q) A[r][q] -= f * A[col][q];
      }
    }
    for (int r = 0; r < 10; ++r)
      for (int m = 0; m < 19; ++m) M[(k * 10 + r) * 19 + m] = A[r][10 + m];
  }
}

extern "C" int gnx_set_density(gnx_ctx* ctx, const gnx_density_t* dn) {
  ARG(ctx && dn, "null");
  USE_DEVICE(ctx);
  ARG(dn->n_points > 0 && dn->n_tri > 0, "empty triangulation");
  CK(cudaStreamSynchronize(ctx->stream));
  free_bucket(ctx->dens_allocs);
  Dens& D = ctx->dens;
  memset(&D, 0, sizeof D);
  D.ww = dn->window_width;
  D.hww = dn->window_width / 2.;
  {
    const double scaled = D.hww * 1048576.0;     // 2^20
    D.half_index_ok = (D.hww > 0 && scaled == std::floor(scaled) && ctx->cfg.dim_x < (1 << 30) &&
                       ctx->cfg.dim_y < (1 << 30)) ? 1 : 0;
  }
  D.npts = dn->n_points;
  D.ntri = dn->n_tri;
  int off = 0;
  for (int g = 0; g < 4; ++g) {
    D.g_ni[g] = dn->grid_ni[g];
    D.g_nj[g] = dn->grid_nj[g];
    D.g_i0[g] = dn->grid_i0[g];
    D.g_j0[g] = dn->grid_j0[g];
    D.g_xe[g] = dn->grid_x_edge[g];
    D.g_ye[g] = dn->grid_y_edge[g];
    D.g_off[g] = off;
    off += dn->grid_ni[g] * dn->grid_nj[g];
  }
  ARG(off == dn->n_points, "grid shapes do not add up to n_points");
  D.lat_ni = dn->lat_ni;
  D.lat_nj = dn->lat_nj;
  D.colourable = dn->colourable;
  auto up = [&](const void* src, size_t bytes, const void** dst) -> int {
    void* d = nullptr;
    CK(cudaMalloc(&d, std::max<size_t>(bytes, 8)));
    ctx->dens_allocs.push_back(d);
    CK(cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dst = d;
    return GNX_OK;
  };
  int r;
  if ((r = up(dn->host_points, sizeof(double) * 2 * D.npts, (const void**)&D.points))) return r;
  if ((r = up(dn->host_areas, sizeof(double) * D.npts, (const void**)&D.areas))) return r;
  if ((r = up(dn->host_simplices, sizeof(int32_t) * 3 * D.ntri, (const void**)&D.simplices))) return r;
  if ((r = up(dn->host_neighbors, sizeof(int32_t) * 3 * D.ntri, (const void**)&D.neighbors))) return r;
  if ((r = up(dn->host_nbr_indptr, sizeof(int32_t) * (D.npts + 1), (const void**)&D.nbr_indptr))) return r;
  const int nnz = dn->host_nbr_indptr[D.npts];
  if ((r = up(dn->host_nbr_indices, sizeof(int32_t) * nnz, (const void**)&D.nbr_indices))) return r;
  {
    // data-independent parts of the gradient solve (interpnd.pyx: Q, L3 per edge)
    std::vector<double> ex(nnz), ey(nnz), wx(nnz), wy(nnz), vinv((size_t)3 * D.npts);
    const double* P = dn->host_points;
    for (int i = 0; i < D.npts; ++i) {
      double Q0 = 0, Q1 = 0, Q3 = 0;
      for (int jj = dn->host_nbr_indptr[i]; jj < dn->host_nbr_indptr[i + 1]; ++jj) {
        const int j = dn->host_nbr_indices[jj];
        const double x = P[2 * j] - P[2 * i], y = P[2 * j + 1] - P[2 * i + 1];
        const double L = sqrt(x * x + y * y), L3 = L * L * L;
        ex[jj] = x; ey[jj] = y; wx[jj] = x / L3; wy[jj] = y / L3;
        Q0 += 4 * x * x / L3; Q1 += 4 * x * y / L3; Q3 += 4 * y * y / L3;
      }
      const double det = Q0 * Q3 - Q1 * Q1;
      vinv[3 * i] = Q3 / det; vinv[3 * i + 1] = -Q1 / det; vinv[3 * i + 2] = Q0 / det;
    }
    if ((r = up(ex.data(), sizeof(double) * nnz, (const void**)&D.e_ex))) return r;
    if ((r = up(ey.data(), sizeof(double) * nnz, (const void**)&D.e_ey))) return r;
    if ((r = up(wx.data(), sizeof(double) * nnz, (const void**)&D.e_wx))) return r;
    if ((r = up(wy.data(), sizeof(double) * nnz, (const void**)&D.e_wy))) return r;
    if ((r = up(vinv.data(), sizeof(double) * 3 * D.npts, (const void**)&D.v_inv))) return r;
    // padded fixed-degree copy for the unrolled per-vertex update
    std::vector<int32_t> pj((size_t)8 * D.npts);
    std::vector<double> pe((size_t)32 * D.npts, 0.0);
    D.padded = 1;
    for (int i = 0; i < D.npts; ++i) {
      const int s0 = dn->host_nbr_indptr[i], deg = dn->host_nbr_indptr[i + 1] - s0;
      if (deg > 8) D.padded = 0;
      const size_t np = (size_t)D.npts;
      for (int k = 0; k < 8; ++k) {
        pj[k * np + i] = k < deg ? dn->host_nbr_indices[s0 + k] : i;
        if (k < deg) {
          pe[(4 * k + 0) * np + i] = ex[s0 + k];
          pe[(4 * k + 1) * np + i] = ey[s0 + k];
          pe[(4 * k + 2) * np + i] = wx[s0 + k];
          pe[(4 * k + 3) * np + i] = wy[s0 + k];
        }
      }
    }
    std::vector<double> vinv_t((size_t)3 * D.npts);
    for (int i = 0; i < D.npts; ++i)
      for (int cc = 0; cc < 3; ++cc) vinv_t[(size_t)cc * D.npts + i] = vinv[3 * i + cc];
    if ((r = up(vinv_t.data(), sizeof(double) * vinv_t.size(), (const void**)&D.v_inv_t))) return r;
    if ((r = up(pj.data(), sizeof(int32_t) * pj.size(), (const void**)&D.p_j))) return r;
    if ((r = up(pe.data(), sizeof(double) * pe.size(), (const void**)&D.p_e))) return r;
    CK(cudaStreamSynchronize(ctx->stream));     // the host vectors go out of scope below
  }
  {
    // per-triangle affine map (qi, qj) -> (b0, b1) and the Bezier -> monomial matrices
    std::vector<double> aff((size_t)6 * D.ntri);
    const double* P = dn->host_points;
    for (int t = 0; t < D.ntri; ++t) {
      const int v0 = dn->host_simplices[3 * t], v1 = dn->host_simplices[3 * t + 1], v2 = dn->host_simplices[3 * t + 2];
      const double a00 = P[2 * v0] - P[2 * v2], a01 = P[2 * v1] - P[2 * v2];
      const double a10 = P[2 * v0 + 1] - P[2 * v2 + 1], a11 = P[2 * v1 + 1] - P[2 * v2 + 1];
      const double det = a00 * a11 - a01 * a10;
      const double i00 = a11 / det, i01 = -a01 / det, i10 = -a10 / det, i11 = a00 / det;
      double* o = &aff[(size_t)6 * t];
      o[1] = i00; o[2] = i01; o[0] = -(i00 * P[2 * v2] + i01 * P[2 * v2 + 1]);
      o[4] = i10; o[5] = i11; o[3] = -(i10 * P[2 * v2] + i11 * P[2 * v2 + 1]);
    }
    if ((r = up(aff.data(), sizeof(double) * aff.size(), (const void**)&D.tri_aff))) return r;
    CK(cudaStreamSynchronize(ctx->stream));
    double* tri_g = nullptr;
    DM(ctx, &tri_g, (size_t)3 * D.ntri, &ctx->dens_allocs);
    k_ct_setup_g<<<std::max(1, (D.ntri + 127) / 128), 128, 0, ctx->stream>>>(D, tri_g);
    CK(cudaGetLastError());
    D.tri_g = tri_g;
    CK(cudaStreamSynchronize(ctx->stream));
    static double mono[3 * 10 * 19];
    ct_build_mono(mono);
    CK(cudaMemcpyToSymbol(CT_MONO, mono, sizeof mono));
  }
  if ((r = up(dn->host_square_tri, sizeof(int32_t) * 2 * (D.lat_ni - 1) * (D.lat_nj - 1),
              (const void**)&D.square_tri)))
    return r;
  DM(ctx, &D.counts, (size_t)2 * D.npts, &ctx->dens_allocs);
  DM(ctx, &D.vals, (size_t)2 * D.npts, &ctx->dens_allocs);
  DM(ctx, &D.grad, (size_t)4 * D.npts, &ctx->dens_allocs);
  DM(ctx, &D.coef, (size_t)2 * D.ntri * CT_STRIDE + 64, &ctx->dens_allocs);
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->have_density = true;
  return GNX_OK;
}

extern "C" int gnx_set_draws(gnx_ctx* ctx, const gnx_draws_t* dr) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  ARG(!(dr && ctx->d_strip), "injected draws are not supported under strip decomposition");
  CK(cudaStreamSynchronize(ctx->stream));
  const int R = ctx->draws.disp_R;
  memset(&ctx->draws, 0, sizeof ctx->draws);
  ctx->draws.disp_R = R;
  // injected draws are indexed by species-order ordinal and offspring number: switch the step to
  // ordered mode (ordinals carried through the re-grid, pair list in ascending focal ordinal)
  ctx->prm.ordered = dr ? 1 : 0;
  ctx->order_valid = false;
  if (!dr) return GNX_OK;
  const size_t n = (size_t)dr->n;
  ctx->draws.n = dr->n;
  // One device buffer per site, kept across calls and re-used while it is large enough: the
  // device pointers (kernel arguments) then stay the same from step to step, so a multi-step
  // injected-draw run keeps re-launching the SAME captured graph (tests/test_cuda_multistep.py).
  int slot = 0;
  auto up = [&](const void* src, size_t bytes, const void** dst) -> int {
    const int k = slot++;
    if (!src) { *dst = nullptr; return GNX_OK; }
    if ((int)ctx->draw_bufs.size() <= k) ctx->draw_bufs.resize(k + 1, {nullptr, 0});
    auto& b = ctx->draw_bufs[k];
    bytes = std::max<size_t>(bytes, 8);
    if (b.second < bytes) {
      if (b.first) cudaFree(b.first);
      b = {nullptr, 0};
      void* d = nullptr;
      CK(cudaMalloc(&d, bytes + bytes / 2));
      b = {d, bytes + bytes / 2};
    }
    CK(cudaMemcpyAsync(b.first, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dst = b.first;
    return GNX_OK;
  };
  DevDraws& D = ctx->draws;
  int r;
  if ((r = up(dr->move_dir, n * 8, (const void**)&D.move_dir))) return r;
  if ((r = up(dr->move_choice, n * 4, (const void**)&D.move_choice))) return r;
  if ((r = up(dr->move_dist, n * 8, (const void**)&D.move_dist))) return r;
  if ((r = up(dr->mate_R, n * 4, (const void**)&D.mate_R))) return r;
  if ((r = up(dr->mate_inv_u, n * 8, (const void**)&D.mate_inv_u))) return r;
  if ((r = up(dr->mate_u, n * 8, (const void**)&D.mate_u))) return r;
  if ((r = up(dr->poisson, n * 4, (const void**)&D.poisson))) return r;
  if ((r = up(dr->recomb_keys, 2 * n * 4, (const void**)&D.recomb_keys))) return r;
  if ((r = up(dr->start_homs, 2 * n * 4, (const void**)&D.start_homs))) return r;
  if ((r = up(dr->disp_dir, n * R * 8, (const void**)&D.disp_dir))) return r;
  if ((r = up(dr->disp_choice, n * R * 4, (const void**)&D.disp_choice))) return r;
  if ((r = up(dr->disp_dist, n * R * 8, (const void**)&D.disp_dist))) return r;
  if ((r = up(dr->sex_u, n * 8, (const void**)&D.sex_u))) return r;
  if ((r = up(dr->sex_redraw_u, n * 8, (const void**)&D.sex_redraw_u))) return r;
  if ((r = up(dr->death_u, n * 8, (const void**)&D.death_u))) return r;
  if ((r = up(dr->pan_u, n * 8, (const void**)&D.pan_u))) return r;
  if ((r = up(dr->pan_R, 2 * n * 4, (const void**)&D.pan_R))) return r;
  const size_t nm = (size_t)std::max<int64_t>(dr->n_mut, 0);
  D.n_mut = (int64_t)nm;
  if ((r = up(dr->mut_n, 4, (const void**)&D.mut_n))) return r;
  if ((r = up(dr->mut_type_u, nm * 8, (const void**)&D.mut_type_u))) return r;
  if ((r = up(dr->mut_ind_R, nm * 4, (const void**)&D.mut_ind_R))) return r;
  if ((r = up(dr->mut_homol_u, nm * 8, (const void**)&D.mut_homol_u))) return r;
  if ((r = up(dr->mut_s, nm * 8, (const void**)&D.mut_s))) return r;
  if ((r = up(dr->mut_alpha, nm * 8, (const void**)&D.mut_alpha))) return r;
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

extern "C" int gnx_set_burn(gnx_ctx* ctx, int32_t burn) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  ctx->burn = burn ? 1 : 0;
  ctx->prm.burn = ctx->burn;
  // species.py:449-451: selection if there are traits or deleterious mutation
  ctx->prm.selection = (!ctx->burn && (ctx->cfg.n_traits > 0 || (ctx->mut.enabled && ctx->mut_delet))) ? 1 : 0;
  return GNX_OK;
}

static int read_counters(gnx_ctx* ctx, Counters* h) {
  CK(cudaMemcpyAsync(h, ctx->d_c, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->n_hint = std::max(h->n, h->n_pre);
  return GNX_OK;
}

static int check_device_err(const Counters& h) {
  if (h.err & GNX_ERRBIT_CAPACITY) { g_last_error = "population outgrew ctx capacity"; return GNX_ERR_CAPACITY; }
  if (h.err & GNX_ERRBIT_DRAWS) { g_last_error = "injected draws exhausted (dispersal tries or mutation rows)"; return GNX_ERR_DRAWS; }
  if (h.err & GNX_ERRBIT_MUTABLES) { g_last_error = "mutation: no mutable locus left (the reference raises IndexError on _mutables.pop())"; return GNX_ERR_MUTABLES; }
  if (h.err & GNX_ERRBIT_MUTIDX) { g_last_error = "mutation: a loci_idxs / delet_loci_idxs entry addresses a genotype row that does not exist (IndexError in the reference)"; return GNX_ERR_STATE; }
  return GNX_OK;
}

// ---- species order on demand, pending deaths -------------------------------------------------
template <class F>
static int run_scan(gnx_ctx* ctx, F f, const char* name);

// Deaths a fused step left flagged are applied now (explicit stable compaction), so that every
// host-facing view sees exactly the live population.
static int materialise(gnx_ctx* ctx) {
  if (ctx->grow_guard && !ctx->capturing) {
    // the guard may have skipped the steps that would have left deaths pending: ask the device
    Counters h;
    int r = read_counters(ctx, &h);
    if (r != GNX_OK) return r;
    ctx->pending = h.pending != 0;
  }
  if (!ctx->pending) return GNX_OK;
  MortalityScan ms{ctx->pop, ctx->work, ctx->d_c, ctx->burn};
  int r = run_scan(ctx, ms, "scan_mortality");
  if (r != GNX_OK) return r;
  PROF(ctx, "k_end_step");
  k_end_step<<<1, 1, 0, ctx->stream>>>(ctx->d_c, ctx->work, ctx->burn, 0);
  LAUNCHED(ctx);
  ctx->pending = false;
  ctx->order_valid = false;
  return GNX_OK;
}

// pop.ord[cur] (entry -> species-order ordinal) and work.inv (ordinal -> entry) for the first
// n entries of the current half: LSD radix sort of (id, entry).  exclude_dead ranks only the
// entries whose pending-death flag is clear (they sort first; *n_ranked = their number).
static int build_order(gnx_ctx* ctx, const Counters& h, bool exclude_dead) {
  const int n = std::max(h.n, h.n_pre);
  cudaStream_t s = ctx->stream;
  Work& W = ctx->work;
  PROF(ctx, "k_order_keys");
  k_order_keys<<<grid_for(ctx, 4), 256, 0, s>>>(ctx->pop, W, ctx->d_c, n, exclude_dead ? 1 : 0);
  LAUNCHED(ctx);
  int bits = 1;
  while (bits < 63 && (h.max_idx >> bits) != 0) ++bits;
  bits += 1;                                     // dead keys (all ones) stay strictly above every id
  const int ntiles = std::max(1, (n + RS_TILE - 1) / RS_TILE);
  int in = 0;
  for (int shift = 0; shift < bits; shift += 8) {
    PROF(ctx, "k_radix_hist");
    k_radix_hist<<<std::min(ntiles, grid_for(ctx, 8)), RS_BLOCK, 0, s>>>(W.sort_keys[in], n, nullptr, shift, W.sort_hist);
    LAUNCHED(ctx);
    RadixScan rs{W.sort_hist, n, nullptr};
    int r = run_scan(ctx, rs, "scan_radix");
    if (r != GNX_OK) return r;
    PROF(ctx, "k_radix_scatter");
    k_radix_scatter<<<std::min(ntiles, grid_for(ctx, 8)), RS_BLOCK, 0, s>>>(W.sort_keys[in], W.sort_vals[in], W.sort_keys[in ^ 1],
                                                                      W.sort_vals[in ^ 1], n, nullptr, shift, W.sort_hist);
    LAUNCHED(ctx);
    in ^= 1;
  }
  const int n_ranked = exclude_dead ? h.n_alive : n;
  PROF(ctx, "k_order_finish");
  k_order_finish<<<grid_for(ctx, 4), 256, 0, s>>>(ctx->pop, W, ctx->d_c, W.sort_vals[in], n_ranked);
  LAUNCHED(ctx);
  ctx->order_valid = true;
  return GNX_OK;
}

// ---- population upload / download -------------------------------------------------------
extern "C" int gnx_phenotype(gnx_ctx* ctx);

static int upload_population(gnx_ctx* ctx, const gnx_population_t* pop, bool wait) {
  ARG(ctx && pop, "null");
  USE_DEVICE(ctx);
  ARG(pop->n >= 0 && pop->n <= ctx->cfg.capacity, "population larger than capacity");
  ARG(pop->x && pop->y, "x/y required");
  const size_t n = (size_t)pop->n;
  ctx->n_hint = pop->n;
  cudaStream_t s = ctx->stream;
  Pop& P = ctx->pop;
  // everything below is asynchronous on the ctx stream: no host-side staging loops
  // x | y staged as plain arrays in the idle half; k_upload_finish interleaves them
  CK(cudaMemcpyAsync(reinterpret_cast<double*>(P.xy[1]), pop->x, n * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(reinterpret_cast<double*>(P.xy[1]) + P.cap, pop->y, n * 8, cudaMemcpyHostToDevice, s));
  if (pop->age) CK(cudaMemcpyAsync(P.age[0], pop->age, n * 4, cudaMemcpyHostToDevice, s));
  else CK(cudaMemsetAsync(P.age[0], 0, n * 4, s));
  if (pop->sex) CK(cudaMemcpyAsync(P.sex[0], pop->sex, n, cudaMemcpyHostToDevice, s));
  else CK(cudaMemsetAsync(P.sex[0], 0, n, s));
  if (pop->idx) CK(cudaMemcpyAsync(P.idx[0], pop->idx, n * 8, cudaMemcpyHostToDevice, s));
  if (pop->genomes) CK(cudaMemcpyAsync(P.G, pop->genomes, n * 2 * ctx->Wq * sizeof(uint4), cudaMemcpyHostToDevice, s));
  if (pop->fit) CK(cudaMemcpyAsync(P.fit[0], pop->fit, n * 8, cudaMemcpyHostToDevice, s));
  const bool have_z = pop->z && ctx->cfg.n_traits > 0;
  if (have_z) CK(cudaMemcpyAsync(ctx->d_stage_z, pop->z, n * ctx->cfg.n_traits * 8, cudaMemcpyHostToDevice, s));
  // slots = identity, ids = 0..n-1 when absent, z transposed to [T][cap], counters reset
  // (the Philox time-step counter and the record cursor carry over)
  int64_t max_idx = pop->max_ind_idx;
  if (!pop->idx && max_idx < (int64_t)n - 1) max_idx = (int64_t)n - 1;
  PROF(ctx, "k_upload_finish");
  k_upload_finish<<<grid_for(ctx, 4), 256, 0, s>>>(P, ctx->d_c, (int)n, max_idx, pop->idx ? 0 : 1,
                                                  have_z ? ctx->d_stage_z : nullptr);
  LAUNCHED(ctx);
  ctx->pending = false;
  ctx->order_valid = false;
  if (!have_z && pop->genomes && ctx->cfg.n_traits > 0 && ctx->have_traits) {
    int r = gnx_phenotype(ctx);
    if (r != GNX_OK) return r;
  }
  if (wait) CK(cudaStreamSynchronize(s));
  return GNX_OK;
}

extern "C" int gnx_upload_population(gnx_ctx* ctx, const gnx_population_t* pop) {
  return upload_population(ctx, pop, true);
}

extern "C" int gnx_population_size(gnx_ctx* ctx, int64_t* n) {
  ARG(ctx && n, "null");
  USE_DEVICE(ctx);
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  *n = h.pending ? h.n_alive : h.n;
  return check_device_err(h);
}

// the live population in species order (ascending id) in the idle half of the state buffers
static int species_view(gnx_ctx* ctx, Counters* h, bool want_z_rows) {
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  if ((r = read_counters(ctx, h)) != GNX_OK) return r;
  if ((r = build_order(ctx, *h, false)) != GNX_OK) return r;
  const int n = std::max(h->n, h->n_pre);
  PROF(ctx, "k_species_gather");
  k_species_gather<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(ctx->pop, ctx->work, ctx->d_c, n,
                                                             want_z_rows ? ctx->d_stage_z : nullptr);
  LAUNCHED(ctx);
  return GNX_OK;
}

static int sample_env_ordered(gnx_ctx* ctx, int n) {
  PROF(ctx, "k_sample_env");
  k_sample_env<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->work, ctx->d_c, n);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_download_population(gnx_ctx* ctx, gnx_population_t* pop) {
  ARG(ctx && pop, "null");
  USE_DEVICE(ctx);
  Counters h;
  const bool want_z = pop->z && ctx->cfg.n_traits > 0;
  int r = species_view(ctx, &h, want_z);
  if (r != GNX_OK) return r;
  const size_t n = (size_t)h.n;
  const int o = h.cur ^ 1;                       // species-ordered copies live in the idle half
  cudaStream_t s = ctx->stream;
  Pop& P = ctx->pop;
  pop->n = h.n;
  pop->max_ind_idx = h.max_idx;
  const double* sx = reinterpret_cast<const double*>(P.xy[o]);
  if (pop->x) CK(cudaMemcpyAsync(pop->x, sx, n * 8, cudaMemcpyDeviceToHost, s));
  if (pop->y) CK(cudaMemcpyAsync(pop->y, sx + P.cap, n * 8, cudaMemcpyDeviceToHost, s));
  if (pop->age) CK(cudaMemcpyAsync(pop->age, P.age[o], n * 4, cudaMemcpyDeviceToHost, s));
  if (pop->sex) CK(cudaMemcpyAsync(pop->sex, P.sex[o], n, cudaMemcpyDeviceToHost, s));
  if (pop->idx) CK(cudaMemcpyAsync(pop->idx, P.idx[o], n * 8, cudaMemcpyDeviceToHost, s));
  if (pop->fit) CK(cudaMemcpyAsync(pop->fit, P.fit[o], n * 8, cudaMemcpyDeviceToHost, s));
  if (pop->genomes && !ctx->burn) {
    PROF(ctx, "k_gather_genomes");
    k_gather_genomes<<<grid_for(ctx, 8), 256, 0, s>>>(P, P.gslot[o], ctx->d_stage_genomes, (int)n);
    LAUNCHED(ctx);
    CK(cudaMemcpyAsync(pop->genomes, ctx->d_stage_genomes, n * 2 * ctx->Wq * sizeof(uint4), cudaMemcpyDeviceToHost, s));
  }
  if (want_z) CK(cudaMemcpyAsync(pop->z, ctx->d_stage_z, n * ctx->cfg.n_traits * 8, cudaMemcpyDeviceToHost, s));
  if (pop->e) {
    r = sample_env_ordered(ctx, (int)n);
    if (r != GNX_OK) return r;
    CK(cudaMemcpyAsync(pop->e, ctx->work.e_out, n * ctx->cfg.n_layers * 8, cudaMemcpyDeviceToHost, s));
  }
  CK(cudaStreamSynchronize(s));
  return check_device_err(h);
}

// ---- stages -----------------------------------------------------------------------------

// tile_sums / ticket: the ctx's own (sized from the capacity) unless a caller scanning something
// larger brings its own
template <class F>
static int run_scan(gnx_ctx* ctx, F f, const char* name, u64* tile_sums, unsigned int* ticket) {
  cudaStream_t s = ctx->stream;
  char nm[64];
  snprintf(nm, sizeof nm, "%s.reduce", name);
  PROF(ctx, nm);
  scan_reduce_kernel<F><<<grid_for(ctx, SCAN_GRID), SCAN_BLOCK, 0, s>>>(f, ctx->d_c, tile_sums, ticket);
  LAUNCHED(ctx);
  snprintf(nm, sizeof nm, "%s.apply", name);
  PROF(ctx, nm);
  scan_apply_kernel<F><<<grid_for(ctx, SCAN_GRID), SCAN_BLOCK, 0, s>>>(f, ctx->d_c, tile_sums);
  LAUNCHED(ctx);
  return GNX_OK;
}
template <class F>
static int run_scan(gnx_ctx* ctx, F f, const char* name) {
  return run_scan(ctx, f, name, ctx->work.tile_sums, ctx->work.scan_ticket);
}

// injected draws are indexed by species-order ordinal: make pop.ord / work.inv current.
// Synchronises (reads the counters), so never called while a graph is being captured.
static int ensure_order(gnx_ctx* ctx) {
  if (!ctx->prm.ordered || ctx->order_valid) return GNX_OK;
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  return build_order(ctx, h, h.pending != 0);
}

static int move_key(gnx_ctx* ctx, int do_age, int do_move, int do_key) {
  if (do_key) CK(cudaMemsetAsync(ctx->work.cell_count, 0, ((size_t)ctx->ncell + 1) * 4, ctx->stream));
  if (do_move && ctx->cfg.move_surf_mode == GNX_SURF_TABLE && !ctx->prm.move_tab) {
    g_last_error = "movement surface table not set";
    return GNX_ERR_STATE;
  }
  PROF(ctx, "k_move_key");
  k_move_key<<<grid_for(ctx, MOVE_KEY_GRID), 256, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->prm, ctx->draws,
                                                                    ctx->work, ctx->d_c, do_age, do_move, do_key,
                                                                    ctx->d_strip);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_age_step(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  return move_key(ctx, 1, 0, 0);
}
extern "C" int gnx_move(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (!ctx->cfg.move) return GNX_OK;
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  if ((r = ensure_order(ctx)) != GNX_OK) return r;
  return move_key(ctx, 0, 1, 0);
}

// cell starts -> arrival buckets -> the one pass that moves the state into (cell, id) order
static int finish_regrid(gnx_ctx* ctx, int age_inc) {
  CellScan cs{ctx->work.cell_count, ctx->work.cell_start, ctx->ncell};
  int r = run_scan(ctx, cs, "scan_cells");
  if (r != GNX_OK) return r;
  cudaStream_t s = ctx->stream;
  PROF(ctx, "k_bucket");
  k_bucket<<<grid_for(ctx, REGRID_GRID), 256, 0, s>>>(ctx->pop, ctx->land, ctx->work, ctx->d_c);
  LAUNCHED(ctx);
  PROF(ctx, "k_regrid");
  k_regrid<<<grid_for(ctx, REGRID_GRID), 256, 0, s>>>(ctx->pop, ctx->land, ctx->work, ctx->d_c, age_inc,
                                                      ctx->prm.ordered, ctx->d_strip);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_bin_cells(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (ctx->cfg.mating_radius <= 0) return GNX_OK;      // panmixia needs no spatial binning
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  if ((r = ensure_order(ctx)) != GNX_OK) return r;
  if ((r = move_key(ctx, 0, 0, 1)) != GNX_OK) return r;
  return finish_regrid(ctx, 0);
}

static int find_mates(gnx_ctx* ctx);
extern "C" int gnx_find_mates(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  if ((r = ensure_order(ctx)) != GNX_OK) return r;
  return find_mates(ctx);
}

// Bernoulli(b) first: list the focals that may mate (and announce the crowded cells' work items),
// then search the listed focals' neighbours on a grid of g CTAs
template <int MODE>
static int launch_mate_search(gnx_ctx* ctx, int g) {
  k_mate_select<MODE><<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->prm, ctx->draws, ctx->work,
                                                                  ctx->d_c);
  LAUNCHED(ctx);
  k_find_mates<MODE><<<g, FM_BLOCK, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->prm, ctx->draws, ctx->work, ctx->d_c);
  LAUNCHED(ctx);
  return GNX_OK;
}

static int find_mates(gnx_ctx* ctx) {
  if (ctx->cfg.mating_radius <= 0) {          // mating_radius = None: Wright-Fisher style panmixia
    PROF(ctx, "k_panmixia");
    k_panmixia<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(ctx->pop, ctx->prm, ctx->draws, ctx->work, ctx->d_c);
    LAUNCHED(ctx);
    return GNX_OK;
  }
  constexpr int FM_GRID = 128, FMD_GRID = 6;   // CTAs per SM of k_find_mates (at most) and k_find_mates_dense
  PROF(ctx, "k_find_mates");
  // the thread-per-focal search walks the list of focals that may mate: a fraction b of the population
  const int g = grid_cap(ctx, FM_GRID, FM_BLOCK, ctx->prm.store_debug ? 1.0 : std::min(1.0, ctx->cfg.b + 0.05));
  // MODE of the search kernels: 0 uniform random neighbour, 1 nearest, 2 inverse-distance weighting
  const int mode = ctx->cfg.choose_nearest ? 1 : ctx->cfg.inverse_dist ? 2 : 0;
  if (mode == 0)     // n_heavy, heavy_next: the crowded-cell list starts empty
    CK(cudaMemsetAsync(&ctx->d_c->n_heavy, 0, 2 * sizeof(int32_t), ctx->stream));
  CK(cudaMemsetAsync(ctx->work.fm_count, 0, sizeof(int32_t), ctx->stream));
  int r;
  switch (mode) {
    case 1: r = launch_mate_search<1>(ctx, g); break;
    case 2: r = launch_mate_search<2>(ctx, g); break;
    default: r = launch_mate_search<0>(ctx, g); break;
  }
  if (r != GNX_OK) return r;
  if (mode == 0) {
    PROF(ctx, "k_find_mates_dense");
    k_find_mates_dense<<<grid_for(ctx, FMD_GRID), 32 * FMD_WARPS, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->prm,
                                                                               ctx->draws, ctx->work, ctx->d_c);
    LAUNCHED(ctx);
  }
  return GNX_OK;
}

// the pair list (and, with n_births_fixed, the births)
static int scan_pairs(gnx_ctx* ctx) {
  const bool fixed = ctx->cfg.n_births_fixed != 0;
  PairScan ps{ctx->pop, ctx->work, ctx->d_c, ctx->cfg.sex, fixed ? (int32_t)ctx->cfg.n_births_lambda : 0,
              ctx->cfg.mating_radius <= 0 ? 1 : 0, ctx->prm.ordered};
  if (fixed) ARG(ps.fixed_nb >= 1, "n_births_fixed needs n_births_distr_lambda >= 1");
  return run_scan(ctx, ps, "scan_pairs");
}

// Poisson births of the pairs (under strips keyed by the pairs' species-wide positions: the pair
// counts of the lower ranks must have been all-gathered)
static int draw_births(gnx_ctx* ctx) {
  PROF(ctx, "k_draw_births");
  k_draw_births<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(ctx->pop, ctx->prm, ctx->draws, ctx->work, ctx->d_c,
                                                           ctx->d_strip);
  LAUNCHED(ctx);
  BirthScan bs{ctx->work, ctx->pop.cap};
  return run_scan(ctx, bs, "scan_births");
}

extern "C" int gnx_dedup_pairs(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r = scan_pairs(ctx);
  if (r != GNX_OK) return r;
  return ctx->cfg.n_births_fixed ? GNX_OK : draw_births(ctx);
}

extern "C" int gnx_mutate(gnx_ctx* ctx);

// gnx_make_offspring in three parts, so the fused step can overlap the density chain (which
// needs only the newborns' positions) with the genotype streaming
static int offspring_check(gnx_ctx* ctx) {
  if (!ctx->burn) {
    if (!ctx->have_paths) { g_last_error = "recombination paths not set"; return GNX_ERR_STATE; }
    if (ctx->cfg.n_traits > 0 && !ctx->have_traits) { g_last_error = "traits not set"; return GNX_ERR_STATE; }
  }
  return GNX_OK;
}

// k_gametes with GW lanes per offspring (fnb: births per pair when fixed, else 0)
template <int GW>
static void launch_gametes(gnx_ctx* ctx, int fnb) {
  const int g = grid_for(ctx, 8);
  // child rows staged in shared memory for the phenotype when they fit (32 KB per block)
  const size_t rows_b = (size_t)(256 / GW) * 2 * ctx->Wq * 16;
  int stage = (GW > 1 && ctx->cfg.n_traits > 0 && rows_b <= 32 * 1024) ? 1 : 0;
  // 2 = two staged rows per group and one trait-table walk for both: every trait polygenic, no dominance
  constexpr int NB = (GAM_NB < GW) ? GAM_NB : GW;
  if (stage && NB >= 2 && NB * rows_b <= 44 * 1024 && ctx->pair_phenotype) stage = NB;
  const size_t smem = stage ? stage * rows_b : 0;
  if (ctx->cfg.n_traits <= 2)
    k_gametes<GW, 2><<<g, 256, smem, ctx->stream>>>(ctx->pop, ctx->prm, ctx->traits, ctx->draws, ctx->work, ctx->d_c,
                                                    fnb, stage);
  else
    k_gametes<GW, GNX_MAX_TRAITS><<<g, 256, smem, ctx->stream>>>(ctx->pop, ctx->prm, ctx->traits, ctx->draws,
                                                                 ctx->work, ctx->d_c, fnb, stage);
}

static int offspring_gametes(gnx_ctx* ctx) {
  if (!ctx->burn) {
    const int Wq = ctx->Wq;
    const int fnb = ctx->cfg.n_births_fixed ? (int)ctx->cfg.n_births_lambda : 0;
    PROF(ctx, "k_gametes");
    if (Wq <= 1) launch_gametes<1>(ctx, fnb);
    else if (Wq <= 2) launch_gametes<2>(ctx, fnb);
    else if (Wq <= 4) launch_gametes<4>(ctx, fnb);
    else if (Wq <= 8) launch_gametes<8>(ctx, fnb);
    else if (Wq <= 16) launch_gametes<16>(ctx, fnb);
    else launch_gametes<32>(ctx, fnb);
    LAUNCHED(ctx);
  }
  return GNX_OK;
}

static int offspring_newborns(gnx_ctx* ctx) {
  PROF(ctx, "k_newborns");
  k_newborns<<<grid_for(ctx, NEWBORNS_GRID), 256, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->prm, ctx->draws,
                                                                    ctx->work, ctx->d_c, ctx->tsk);
  LAUNCHED(ctx);
  return GNX_OK;
}

static int offspring_finish(gnx_ctx* ctx) {
  cudaStream_t s = ctx->stream;
  if (ctx->tsk.enabled && !ctx->burn) {
    TskitScan ts{ctx->pop, ctx->prm, ctx->draws, ctx->work, ctx->tsk, ctx->d_c,
                 ctx->cfg.n_births_fixed ? (int)ctx->cfg.n_births_lambda : 0};
    int r = run_scan(ctx, ts, "scan_tskit_edges");
    if (r != GNX_OK) return r;
  }
  if (ctx->mut.enabled && !ctx->burn) {
    int r = gnx_mutate(ctx);                       // species.py:808-809
    if (r != GNX_OK) return r;
  }
  PROF(ctx, "k_after_births");
  k_after_births<<<1, 1, 0, s>>>(ctx->d_c, (ctx->tsk.enabled && !ctx->burn) ? 1 : 0);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_make_offspring(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r;
  if ((r = offspring_check(ctx))) return r;
  if ((r = offspring_gametes(ctx))) return r;
  if ((r = offspring_newborns(ctx))) return r;
  return offspring_finish(ctx);
}

// ---- a13 mutation -------------------------------------------------------------------------
extern "C" int gnx_set_mutation(gnx_ctx* ctx, const gnx_mutation_t* m) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (ctx->d_strip && m) {
    // every rank replays the species-wide draws on by-locus rows; the tskit layout would also need the path
    // patches and node ids of offspring held by other ranks
    ARG(!m->tskit_layout, "the tskit genotype layout is not supported under strip decomposition");
    for (int t = 0; m->host_trait_mu && t < ctx->cfg.n_traits; ++t)
      ARG(!(m->host_trait_mu[t] > 0), "trait mutation is not supported under strip decomposition");
  }
  // the column layout carries the use_tskit = True semantics: its genotype bits are non-neutral loci only
  ARG(!ctx->cols || (m && m->tskit_layout), "a context with the column layout needs tskit_layout = 1");
  CK(cudaStreamSynchronize(ctx->stream));
  std::vector<int32_t> col_locus, col_of;
  if (ctx->cols) {
    int r = read_cols(ctx, &col_locus, &col_of);
    if (r != GNX_OK) return r;
  }
  if (ctx->mut.enabled && ctx->mut.own_tables) {
    ctx->traits = ctx->traits_as_set;                  // back to the tables gnx_set_traits built
    if (ctx->mut.tskit_layout && ctx->d_paths && !ctx->host_paths.empty()) {   // undo the path patches
      const std::vector<uint32_t> rows = paths_at_rows(ctx, col_locus);
      CK(cudaMemcpyAsync(ctx->d_paths, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
  }
  free_bucket(ctx->mut_allocs);
  memset(&ctx->mut, 0, sizeof ctx->mut);
  ctx->mut_delet = false;
  const int nT = ctx->cfg.n_traits;
  double trait_mu_sum = 0;
  if (m && m->host_trait_mu)
    for (int t = 0; t < nT; ++t) {
      ARG(m->host_trait_mu[t] >= 0, "negative trait mutation rate");
      trait_mu_sum += m->host_trait_mu[t];
    }
  const bool tskit_layout = m && m->tskit_layout;
  if (!m || (m->mu_neut <= 0 && m->mu_delet <= 0 && trait_mu_sum <= 0 && !tskit_layout)) return gnx_set_burn(ctx, ctx->burn);
  ARG(m->mu_neut >= 0 && m->mu_delet >= 0, "negative mutation rate");
  // genome.py:430: Trait._add_locus indexes loci_idxs, which is None when use_tskit = False
  ARG(trait_mu_sum == 0 || tskit_layout, "trait mutation (Trait.mu > 0) raises in the reference when use_tskit = False");
  ARG(trait_mu_sum == 0 || m->host_trait_alpha_distr, "trait mutation needs host_trait_alpha_distr");
  ARG(m->n_mutables >= 0 && (m->n_mutables == 0 || m->host_mutables), "mutables");
  ARG(m->n_nonneut >= 0 && m->n_nonneut <= ctx->cfg.L && (m->n_nonneut == 0 || m->host_nonneut_loci), "nonneut_loci");
  ARG(m->n_delet >= 0 && m->n_delet <= ctx->cfg.L && (m->n_delet == 0 || (m->host_delet_loci && m->host_delet_s)),
      "delet_loci");
  ARG(!ctx->cols || (int)col_locus.size() == m->n_nonneut, "the columns must be the non-neutral loci");
  for (int k = 0; ctx->cols && k < m->n_nonneut; ++k)
    ARG(m->host_nonneut_loci[k] >= 0 && m->host_nonneut_loci[k] < ctx->cfg.L && col_of[m->host_nonneut_loci[k]] >= 0,
        "a non-neutral locus without a column");
  const bool own = tskit_layout || trait_mu_sum > 0;
  if (own) {
    if (nT > 0 && !ctx->have_traits) { g_last_error = "gnx_set_traits must precede gnx_set_mutation"; return GNX_ERR_STATE; }
    if (tskit_layout && !ctx->have_paths) { g_last_error = "gnx_set_recomb_paths must precede gnx_set_mutation"; return GNX_ERR_STATE; }
  }
  const int L = ctx->cfg.L;
  Mut& M = ctx->mut;
  M.enabled = 1;
  M.tskit_layout = tskit_layout ? 1 : 0;
  M.own_tables = own ? 1 : 0;
  M.n_types = 2 + (trait_mu_sum > 0 ? nT : 0);
  M.mu_tot = m->mu_neut + m->mu_delet + trait_mu_sum;   // genome.py:599-603
  // genome.py:657-662: probs = mu / sum(mu); numpy choice: cdf = cumsum(p); cdf /= cdf[-1]
  {
    double mus[2 + GNX_MAX_TRAITS] = {m->mu_neut, m->mu_delet};
    for (int t = 0; t < nT && trait_mu_sum > 0; ++t) mus[2 + t] = m->host_trait_mu[t];
    double tot = 0;
    for (int k = 0; k < M.n_types; ++k) tot += mus[k];
    ARG(tot > 0 || tskit_layout, "all mutation rates are zero");
    double run = 0;
    for (int k = 0; k < M.n_types; ++k) { run += tot > 0 ? mus[k] / tot : 0.0; M.cdf[k] = run; }
    for (int k = 0; k < M.n_types; ++k) M.cdf[k] = run > 0 ? M.cdf[k] / run : 1.0;
  }
  for (int t = 0; t < nT; ++t) {
    M.a_mu[t] = m->host_trait_alpha_distr ? m->host_trait_alpha_distr[3 * t] : 0.0;
    M.a_sigma[t] = m->host_trait_alpha_distr ? m->host_trait_alpha_distr[3 * t + 1] : 0.0;
    M.a_max[t] = m->host_trait_alpha_distr ? m->host_trait_alpha_distr[3 * t + 2] : -1.0;
  }
  M.s_shape = m->delet_s_shape;
  M.s_scale = m->delet_s_scale;
  M.L = L;
  M.T = nT;
  M.NW = 4 * ctx->Wq;
  M.Wq = ctx->Wq;
  M.WqL = ctx->WqL;
  if (ctx->cols) {
    M.col_n = ctx->d_cols;
    M.col_locus = ctx->d_cols + 1;
    M.col_of_locus = ctx->d_cols + 1 + L;
    M.col_cap = ctx->col_cap;
  }
  M.log_cap = std::max(m->log_capacity, 1);
  DM(ctx, &M.mutables, (size_t)std::max(L, m->n_mutables), &ctx->mut_allocs);
  DM(ctx, &M.nonneut, (size_t)L + 1, &ctx->mut_allocs);
  DM(ctx, &M.delet_loci, (size_t)L + 1, &ctx->mut_allocs);
  DM(ctx, &M.delet_s, (size_t)L + 1, &ctx->mut_allocs);
  DM(ctx, &M.delet_eff, (size_t)L + 1, &ctx->mut_allocs);
  if (tskit_layout) DM(ctx, &M.delet_idxs, (size_t)L + 1, &ctx->mut_allocs);
  DM(ctx, &M.counts, 4 + GNX_MAX_TRAITS, &ctx->mut_allocs);
  DM(ctx, &M.log, (size_t)M.log_cap, &ctx->mut_allocs);
  cudaStream_t s = ctx->stream;
  if (m->n_mutables) CK(cudaMemcpyAsync(M.mutables, m->host_mutables, (size_t)m->n_mutables * 4, cudaMemcpyHostToDevice, s));
  if (m->n_nonneut) CK(cudaMemcpyAsync(M.nonneut, m->host_nonneut_loci, (size_t)m->n_nonneut * 4, cudaMemcpyHostToDevice, s));
  if (m->n_delet) {
    CK(cudaMemcpyAsync(M.delet_loci, m->host_delet_loci, (size_t)m->n_delet * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(M.delet_eff, m->host_delet_loci, (size_t)m->n_delet * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(M.delet_s, m->host_delet_s, (size_t)m->n_delet * 8, cudaMemcpyHostToDevice, s));
  }
  int32_t counts[4 + GNX_MAX_TRAITS] = {m->n_mutables, m->n_nonneut, m->n_delet, 0};
  std::vector<int32_t> keep_i;
  std::vector<double> keep_d;
  std::vector<uint32_t> patched;
  if (own) {
    // rows addressed by the host's idx arrays: position of each locus in nonneut_loci when not given
    auto row_of = [&](int locus) {
      const int32_t* b = m->host_nonneut_loci;
      return (int32_t)(std::lower_bound(b, b + m->n_nonneut, locus) - b);
    };
    if (tskit_layout) {
      std::vector<int32_t> di(std::max(m->n_delet, 1));
      for (int k = 0; k < m->n_delet; ++k) di[k] = m->host_delet_loci_idxs ? m->host_delet_loci_idxs[k] : row_of(m->host_delet_loci[k]);
      for (int k = 0; k < m->n_delet; ++k) ARG(di[k] >= 0 && di[k] < m->n_nonneut, "delet_loci_idxs out of range");
      if (m->n_delet) CK(cudaMemcpyAsync(M.delet_idxs, di.data(), (size_t)m->n_delet * 4, cudaMemcpyHostToDevice, s));
      CK(cudaStreamSynchronize(s));
    }
    // per-trait tables in Trait order, room for every mutable locus
    size_t n_entries = 0;
    for (int t = 0; t < nT; ++t) n_entries += ctx->host_trait_loci[t].size();
    M.tcap = 1;
    for (int t = 0; t < nT; ++t) M.tcap = std::max<int>(M.tcap, (int)ctx->host_trait_loci[t].size());
    M.tcap += m->n_mutables + 1;
    const size_t ecap = n_entries + (size_t)m->n_mutables + 1;
    DM(ctx, &M.t_loci, (size_t)std::max(nT, 1) * M.tcap, &ctx->mut_allocs);
    DM(ctx, &M.t_alpha, (size_t)std::max(nT, 1) * M.tcap, &ctx->mut_allocs);
    DM(ctx, &M.t_idxs, (size_t)std::max(nT, 1) * M.tcap, &ctx->mut_allocs);
    DM(ctx, &M.te_locus, ecap, &ctx->mut_allocs);
    DM(ctx, &M.te_alpha, ecap, &ctx->mut_allocs);
    if (ctx->traits_as_set.te_dom) DM(ctx, &M.te_dom, ecap, &ctx->mut_allocs);
    DM(ctx, &M.te_pack, ecap, &ctx->mut_allocs);
    DM(ctx, &M.chunk_ptr, (size_t)std::max(nT, 1) * (M.NW + 1), &ctx->mut_allocs);
    if (ctx->traits_as_set.te_dom && !ctx->host_dom.empty()) {
      std::vector<double> d1(L);
      for (int l = 0; l < L; ++l) d1[l] = 1.0 + (double)ctx->host_dom[l];
      double* dd = nullptr;
      DM(ctx, &dd, (size_t)L, &ctx->mut_allocs);
      CK(cudaMemcpyAsync(dd, d1.data(), (size_t)L * 8, cudaMemcpyHostToDevice, s));
      CK(cudaStreamSynchronize(s));
      M.dom1p = dd;
    }
    size_t off = 0;
    for (int t = 0; t < nT; ++t) {
      const auto& hl = ctx->host_trait_loci[t];      // sorted by locus in gnx_set_traits = Trait.loci order
      const auto& ha = ctx->host_trait_alpha[t];
      const int n = (int)hl.size();
      counts[4 + t] = n;
      std::vector<int32_t> idxs(std::max(n, 1));
      for (int k = 0; k < n; ++k) {
        idxs[k] = (tskit_layout && m->host_trait_loci_idxs) ? m->host_trait_loci_idxs[off + k] : row_of(hl[k]);
        ARG(!tskit_layout || (idxs[k] >= 0 && idxs[k] < m->n_nonneut), "trait loci_idxs out of range");
      }
      off += n;
      if (n) {
        CK(cudaMemcpyAsync(M.t_loci + (size_t)t * M.tcap, hl.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(M.t_alpha + (size_t)t * M.tcap, ha.data(), (size_t)n * 8, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(M.t_idxs + (size_t)t * M.tcap, idxs.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));
      }
    }
    if (tskit_layout) {
      // cached paths: as simulated (the source of later patches) and, at the current genotype rows, the
      // reference's subsetters (genome.py:133-160 leaves them different from the path where a breakpoint
      // sits on a mutated locus)
      const size_t nw = ctx->host_paths.size();
      uint4* orig = nullptr;
      DM(ctx, &orig, nw / 4, &ctx->mut_allocs);
      CK(cudaMemcpyAsync(orig, ctx->host_paths.data(), nw * 4, cudaMemcpyHostToDevice, s));
      M.paths_orig = orig;
      M.paths = (uint4*)ctx->d_paths;
      M.n_paths = ctx->cfg.n_recomb_paths;
      patched = paths_at_rows(ctx, col_locus);
      if (m->host_subsetters) {
        const size_t W32 = (size_t)4 * ctx->Wq;
        for (int pth = 0; pth < M.n_paths; ++pth)
          for (int j = 0; j < m->n_nonneut; ++j) {
            const int l = m->host_nonneut_loci[j], bit = ctx->cols ? col_of[l] : l;
            const uint32_t b = m->host_subsetters[(size_t)pth * m->n_nonneut + j] & 1u;
            uint32_t& w = patched[(size_t)pth * W32 + (bit >> 5)];
            w = (w & ~(1u << (bit & 31))) | (b << (bit & 31));
          }
      }
      CK(cudaMemcpyAsync(ctx->d_paths, patched.data(), patched.size() * 4, cudaMemcpyHostToDevice, s));
      CK(cudaStreamSynchronize(s));
    }
  }
  CK(cudaMemcpyAsync(M.counts, counts, sizeof counts, cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));
  if (own) {
    // the device-editable tables replace the ones gnx_set_traits built
    k_mut_rebuild<<<1, 32, 0, s>>>(M, ctx->d_c);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s));
    Traits& T = ctx->traits;
    T.te_locus = M.te_locus;
    T.te_alpha = M.te_alpha;
    T.te_dom = M.te_dom;
    T.te_pack = M.te_pack;
    T.chunk_ptr = M.chunk_ptr;
    T.n_loci_dev = M.counts + 4;
    // a monogenic trait may turn polygenic inside a graph-launched step: the per-pair phenotype walk of
    // k_gametes assumes polygenic traits, which stays true (loci are only ever added)
  }
  ctx->mut_delet = m->mu_delet > 0 || m->n_delet > 0;
  return gnx_set_burn(ctx, ctx->burn);                 // refresh prm.selection
}

extern "C" int gnx_mutate(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (!ctx->mut.enabled || ctx->burn) return GNX_OK;
  if (ctx->mut.mu_tot <= 0) return GNX_OK;             // tskit layout without mutation: nothing to draw
  PROF(ctx, "k_mutate");
  if (ctx->d_strip)
    k_mutate<true><<<1, 256, 0, ctx->stream>>>(ctx->pop, ctx->prm, ctx->traits, ctx->draws, ctx->mut, ctx->d_c, 0);
  else
    k_mutate<false><<<1, 256, 0, ctx->stream>>>(ctx->pop, ctx->prm, ctx->traits, ctx->draws, ctx->mut, ctx->d_c,
                                                ctx->tsk.enabled ? 1 : 0);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_read_mutation_tables(gnx_ctx* ctx, int32_t trait, int32_t* n_loci, int32_t* host_loci,
                                        double* host_alpha, int32_t* host_loci_idxs, int32_t* host_delet_loci_idxs) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (!ctx->mut.enabled) { g_last_error = "mutation not enabled"; return GNX_ERR_STATE; }
  Mut& M = ctx->mut;
  cudaStream_t s = ctx->stream;
  int32_t counts[4 + GNX_MAX_TRAITS];
  CK(cudaMemcpyAsync(counts, M.counts, sizeof counts, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (trait >= 0) {
    ARG(trait < ctx->cfg.n_traits, "trait index");
    if (M.own_tables) {
      const int n = counts[4 + trait];
      if (n_loci) *n_loci = n;
      if (host_loci && n) CK(cudaMemcpyAsync(host_loci, M.t_loci + (size_t)trait * M.tcap, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
      if (host_alpha && n) CK(cudaMemcpyAsync(host_alpha, M.t_alpha + (size_t)trait * M.tcap, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
      if (host_loci_idxs && n) CK(cudaMemcpyAsync(host_loci_idxs, M.t_idxs + (size_t)trait * M.tcap, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    } else {
      const auto& hl = ctx->host_trait_loci[trait];
      const int n = (int)hl.size();
      if (n_loci) *n_loci = n;
      for (int k = 0; k < n; ++k) {
        if (host_loci) host_loci[k] = hl[k];
        if (host_alpha) host_alpha[k] = ctx->host_trait_alpha[trait][k];
        if (host_loci_idxs) host_loci_idxs[k] = hl[k];
      }
    }
  }
  if (host_delet_loci_idxs && counts[2] > 0)
    CK(cudaMemcpyAsync(host_delet_loci_idxs, M.tskit_layout ? M.delet_idxs : M.delet_loci, (size_t)counts[2] * 4,
                       cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return GNX_OK;
}

// ---- column layout ---------------------------------------------------------------------------
extern "C" int gnx_read_cols(gnx_ctx* ctx, int32_t* host_col_locus, int32_t* n_cols, int32_t* col_capacity) {
  ARG(ctx, "null ctx");
  if (!ctx->cols) { g_last_error = "the context does not hold the column layout"; return GNX_ERR_STATE; }
  USE_DEVICE(ctx);
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  std::vector<int32_t> col_locus;
  if ((r = read_cols(ctx, &col_locus)) != GNX_OK) return r;
  if (n_cols) *n_cols = (int32_t)col_locus.size();
  if (col_capacity) *col_capacity = ctx->col_cap;
  if (host_col_locus && !col_locus.empty()) memcpy(host_col_locus, col_locus.data(), col_locus.size() * 4);
  return check_device_err(h);
}

// a fresh [n_rows][wn] copy of the rows of *p ([n_rows][wo]), new units zero; *p is freed (and replaced in bucket)
static int widen_rows(gnx_ctx* ctx, std::vector<void*>* bucket, uint4** p, size_t n_rows, int wo, int wn) {
  uint4* q = nullptr;
  CK(cudaMalloc((void**)&q, std::max<size_t>(n_rows * wn, 1) * sizeof(uint4)));
  PROF(ctx, "k_widen_rows");
  k_widen_rows<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(*p, q, (long long)n_rows, wo, wn);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  if (bucket) std::replace(bucket->begin(), bucket->end(), (void*)*p, (void*)q);
  CK(cudaFree(*p));
  *p = q;
  return GNX_OK;
}

static int widen_csr(gnx_ctx* ctx, std::vector<void*>& bucket, int32_t** p, int nwo, int nwn) {
  const int nt = std::max(1, ctx->cfg.n_traits);
  int32_t* q = nullptr;
  CK(cudaMalloc((void**)&q, (size_t)nt * (nwn + 1) * sizeof(int32_t)));
  k_widen_csr<<<grid_for(ctx, 1), 256, 0, ctx->stream>>>(*p, q, nt, nwo, nwn);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  std::replace(bucket.begin(), bucket.end(), (void*)*p, (void*)q);
  CK(cudaFree(*p));
  *p = q;
  return GNX_OK;
}

extern "C" int gnx_widen_cols(gnx_ctx* ctx, int32_t col_capacity) {
  ARG(ctx, "null ctx");
  if (!ctx->cols) { g_last_error = "the context does not hold the column layout"; return GNX_ERR_STATE; }
  ARG(col_capacity > ctx->col_cap, "col_capacity must exceed the current one");
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  const int wo = ctx->Wq, wn = (col_capacity + 127) / 128;
  int r;
  Pop& P = ctx->pop;
  // genotype rows of every slot; the staging buffer of upload / download only needs the new size
  if ((r = widen_rows(ctx, &ctx->allocs, &P.G, (size_t)P.cap * 2, wo, wn)) != GNX_OK) return r;
  if ((r = widen_rows(ctx, &ctx->allocs, &ctx->d_stage_genomes, (size_t)P.cap * 2, wo, wn)) != GNX_OK) return r;
  if (ctx->d_paths) {
    uint4* d = (uint4*)ctx->d_paths;
    if ((r = widen_rows(ctx, nullptr, &d, (size_t)ctx->cfg.n_recomb_paths, wo, wn)) != GNX_OK) return r;
    ctx->d_paths = d;
    ctx->prm.paths = d;
  }
  // the trait CSR over words: the tables of gnx_set_traits and those the mutation bookkeeping owns
  const bool mut_tables = ctx->mut.enabled && ctx->mut.own_tables;
  if (ctx->have_traits && ctx->traits_as_set.chunk_ptr) {
    int32_t* cp = const_cast<int32_t*>(ctx->traits_as_set.chunk_ptr);
    if ((r = widen_csr(ctx, ctx->trait_allocs, &cp, 4 * wo, 4 * wn)) != GNX_OK) return r;
    ctx->traits_as_set.chunk_ptr = cp;
    if (!mut_tables) ctx->traits.chunk_ptr = cp;
  }
  Mut& M = ctx->mut;
  if (mut_tables) {
    if ((r = widen_csr(ctx, ctx->mut_allocs, &M.chunk_ptr, 4 * wo, 4 * wn)) != GNX_OK) return r;
    ctx->traits.chunk_ptr = M.chunk_ptr;
  }
  ctx->Wq = wn;
  ctx->Wwords = 4 * wn;
  ctx->col_cap = 128 * wn;
  P.Wq = wn;
  if (M.enabled) {
    M.Wq = wn;
    M.NW = 4 * wn;
    M.paths = (uint4*)ctx->d_paths;
    if (M.col_of_locus) M.col_cap = ctx->col_cap;
  }
  return GNX_OK;
}

extern "C" int gnx_read_mutations(gnx_ctx* ctx, gnx_mutation_row_t* rows, int32_t max_rows, int32_t* n_rows,
                                  int32_t* n_mutables_left, int32_t* host_nonneut_loci, int32_t* n_nonneut,
                                  int32_t* host_delet_loci, double* host_delet_s, int32_t* n_delet) {
  ARG(ctx, "null ctx");
  if (!ctx->mut.enabled) {
    if (n_rows) *n_rows = 0;
    if (n_mutables_left) *n_mutables_left = 0;
    if (n_nonneut) *n_nonneut = 0;
    if (n_delet) *n_delet = 0;
    return GNX_OK;
  }
  Mut& M = ctx->mut;
  cudaStream_t s = ctx->stream;
  int32_t counts[4];
  CK(cudaMemcpyAsync(counts, M.counts, sizeof counts, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  const int nr = std::min(counts[3], std::max(max_rows, 0));
  if (rows && nr > 0) CK(cudaMemcpyAsync(rows, M.log, (size_t)nr * sizeof(gnx_mutation_row_t), cudaMemcpyDeviceToHost, s));
  if (host_nonneut_loci && counts[1] > 0)
    CK(cudaMemcpyAsync(host_nonneut_loci, M.nonneut, (size_t)counts[1] * 4, cudaMemcpyDeviceToHost, s));
  if (host_delet_loci && counts[2] > 0)
    CK(cudaMemcpyAsync(host_delet_loci, M.delet_loci, (size_t)counts[2] * 4, cudaMemcpyDeviceToHost, s));
  if (host_delet_s && counts[2] > 0)
    CK(cudaMemcpyAsync(host_delet_s, M.delet_s, (size_t)counts[2] * 8, cudaMemcpyDeviceToHost, s));
  if (rows) {                       // drained: reset the log cursor
    const int32_t zero = 0;
    CK(cudaMemcpyAsync(M.counts + 3, &zero, 4, cudaMemcpyHostToDevice, s));
  }
  CK(cudaStreamSynchronize(s));
  if (n_rows) *n_rows = rows ? nr : counts[3];
  if (n_mutables_left) *n_mutables_left = counts[0];
  if (n_nonneut) *n_nonneut = counts[1];
  if (n_delet) *n_delet = counts[2];
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  return check_device_err(h);
}

extern "C" int gnx_phenotype(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (ctx->cfg.n_traits == 0) return GNX_OK;
  if (!ctx->have_traits) { g_last_error = "traits not set"; return GNX_ERR_STATE; }
  PROF(ctx, "k_phenotype_all");
  k_phenotype_all<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(ctx->pop, ctx->traits, ctx->d_c);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_density_counts(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (!ctx->have_density) { g_last_error = "density grids not set"; return GNX_ERR_STATE; }
  cudaStream_t s = ctx->stream;
  CK(cudaMemsetAsync(ctx->dens.counts, 0, (size_t)2 * ctx->dens.npts * 4, s));
  PROF(ctx, "k_density_counts");
  // one launch: blockIdx.y = 0 counts all individuals, 1 counts pair midpoints
  k_density_counts<<<dim3(2 * ctx->num_sms, 2), 512, 0, s>>>(ctx->pop, ctx->work, ctx->d_c, ctx->dens, ctx->d_strip);
  LAUNCHED(ctx);
  return GNX_OK;
}

// gnx_density_eval in two parts: both rasters in one pass and the exact-order N of the fix list, then the d
// of the cells that need max(N) -- under strip decomposition each rank evaluates its own landscape rows and
// the maximum is reduced over the ranks in between
static void raster_grid(const gnx_ctx* ctx, int* row_lo, int* row_hi, int* rgrid) {
  *row_lo = ctx->d_strip ? ctx->strip_h.ly0 : 0;
  *row_hi = ctx->d_strip ? ctx->strip_h.ly1 : ctx->cfg.dim_y;
  // rows per CTA: the smallest whole number that fits the resident grid (no ragged last pass)
  const int rows = std::max(1, *row_hi - *row_lo);
  const int rg_max = grid_for(ctx, 8);
  const int rows_per_cta = (rows + rg_max - 1) / rg_max;
  *rgrid = (rows + rows_per_cta - 1) / rows_per_cta;
}

static int density_eval_rasters(gnx_ctx* ctx) {
  if (!ctx->have_density) { g_last_error = "density grids not set"; return GNX_ERR_STATE; }
  cudaStream_t s = ctx->stream;
  // scipy defaults reached through griddata: CloughTocher2DInterpolator(tol=1e-6, maxiter=400)
  PROF(ctx, "k_ct_gradients");
  if (ctx->dens.colourable && ctx->dens.padded && ctx->dens.npts <= GS_REG_PTS) {
    k_ct_gradients_reg<<<2, (ctx->dens.npts + 31) / 32 * 32, 0, s>>>(ctx->dens, ctx->d_c, 400, 1e-6);
  } else {
    k_ct_gradients<<<2, GS_BLOCK, 0, s>>>(ctx->dens, ctx->d_c, 400, 1e-6);
  }
  LAUNCHED(ctx);
  PROF(ctx, "k_ct_coefficients");
  k_ct_coefficients<<<(2 * ctx->dens.ntri + CT_ITEMS - 1) / CT_ITEMS, CT_COEF_THREADS, 0, s>>>(ctx->dens);
  LAUNCHED(ctx);
  int row_lo, row_hi, rgrid;
  raster_grid(ctx, &row_lo, &row_hi, &rgrid);
  PROF(ctx, "k_raster_Nd");
  k_raster_Nd<<<rgrid, 256, 0, s>>>(ctx->dens, ctx->land, ctx->prm, ctx->work, ctx->d_c, row_lo, row_hi);
  LAUNCHED(ctx);
  PROF(ctx, "k_raster_fix_N");
  k_raster_fix_N<<<grid_for(ctx, 2), 256, 0, s>>>(ctx->dens, ctx->land, ctx->work, ctx->d_c);
  LAUNCHED(ctx);
  return GNX_OK;
}

static int density_eval_deferred(gnx_ctx* ctx) {
  PROF(ctx, "k_raster_fix_d");
  k_raster_fix_d<<<grid_for(ctx, 2), 256, 0, ctx->stream>>>(ctx->dens, ctx->land, ctx->prm, ctx->work, ctx->d_c);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_density_eval(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r = density_eval_rasters(ctx);
  if (r != GNX_OK) return r;
  return density_eval_deferred(ctx);
}

static int death_prob(gnx_ctx* ctx, int end_step) {
  PROF(ctx, "k_death");
  k_death<<<grid_cap(ctx, DEATH_GRID, 256, 1.0 + ctx->cfg.b * ctx->cfg.n_births_lambda), 256, 0, ctx->stream>>>(
      ctx->pop, ctx->land, ctx->prm, ctx->traits, ctx->draws, ctx->work, ctx->d_c, ctx->mut, end_step, ctx->d_strip);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_death_prob(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  if ((r = ensure_order(ctx)) != GNX_OK) return r;
  return death_prob(ctx, 0);
}

// explicit removal of the flagged dead + end-of-step bookkeeping
static int mortality(gnx_ctx* ctx) {
  MortalityScan ms{ctx->pop, ctx->work, ctx->d_c, ctx->burn};
  int r = run_scan(ctx, ms, "scan_mortality");
  if (r != GNX_OK) return r;
  PROF(ctx, "k_end_step");
  k_end_step<<<1, 1, 0, ctx->stream>>>(ctx->d_c, ctx->work, ctx->burn, 1);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_mortality(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (ctx->pending) { g_last_error = "gnx_mortality after a fused step: the step already ended"; return GNX_ERR_STATE; }
  int r = mortality(ctx);
  if (r != GNX_OK) return r;
  ctx->records_pending += 1;
  ctx->order_valid = false;
  return GNX_OK;
}

extern "C" int gnx_sample_env(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  Counters h;
  if ((r = read_counters(ctx, &h)) != GNX_OK) return r;
  if ((r = build_order(ctx, h, false)) != GNX_OK) return r;
  return sample_env_ordered(ctx, std::max(h.n, h.n_pre));
}

// One time step for this species = the reference's queue (model.py:603-667):
//   _set_age_stage -> _do_movement -> _do_pop_dynamics -> _set_Nt
// With a mating radius the removal of the previous step's dead, this step's ageing and the
// counting sort into mating-grid order are ONE pass over the state (k_move_key flags and keys,
// k_regrid moves); under panmixia there is no grid, so the dead are compacted away at the end
// of the step as the staged entry points do.
static int strip_whole_step(gnx_ctx* ctx);
static int one_step(gnx_ctx* ctx) {
  int r;
  if (ctx->d_strip) return strip_whole_step(ctx);     // one strip of a decomposed landscape: eight phases + barriers
  const bool panmixia = ctx->cfg.mating_radius <= 0;
  if (panmixia) {
    if ((r = move_key(ctx, 1, ctx->cfg.move ? 1 : 0, 0))) return r;
  } else {
    if ((r = move_key(ctx, 0, ctx->cfg.move ? 1 : 0, 1))) return r;
    if ((r = finish_regrid(ctx, 1))) return r;
  }
  if ((r = find_mates(ctx))) return r;
  if ((r = gnx_dedup_pairs(ctx))) return r;
  if (ctx->stream2 && !ctx->profiling && !(ctx->tsk.enabled && !ctx->burn)) {
    // Newborn records first (positions do not depend on genotypes), then two branches:
    //   stream  : gametes -> mutation -> birth bookkeeping
    //   stream2 : gradients -> Clough-Tocher coefficients -> N and d rasters -> fix-list N -> fix and deferred d
    // The density chain is a string of small latency-bound kernels; it hides under the
    // genotype streaming.  They join before the death probabilities.
    if ((r = offspring_check(ctx))) return r;
    if ((r = offspring_newborns(ctx))) return r;
    // The counts stay on the main stream, IN FRONT of the gamete kernel: the gradient solve that follows them
    // is two CTAs that each need a whole SM's register file (one thread per lattice vertex, its tables in
    // registers), and once the gamete kernel's CTAs hold the SMs it cannot start before they are all gone.  Forking after the counts makes the gradient solve and the gamete
    // kernel eligible at the same moment, the solve's two CTAs are placed first, and the chain's latency-bound
    // head runs UNDER the genotype streaming instead of behind it.
    if ((r = gnx_density_counts(ctx))) return r;
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
    cudaStream_t main_stream = ctx->stream;
    ctx->stream = ctx->stream2;
    r = gnx_density_eval(ctx);
    ctx->stream = main_stream;
    if (r != GNX_OK) return r;
    CK(cudaEventRecord(ctx->ev_join, ctx->stream2));
    if ((r = offspring_gametes(ctx))) return r;
    if ((r = offspring_finish(ctx))) return r;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
  } else {
    if ((r = gnx_make_offspring(ctx))) return r;
    if ((r = gnx_density_counts(ctx))) return r;
    if ((r = gnx_density_eval(ctx))) return r;
  }
  if (panmixia) {
    if ((r = death_prob(ctx, 0))) return r;
    if ((r = mortality(ctx))) return r;
  } else {
    if ((r = death_prob(ctx, 1))) return r;       // flags the dead and ends the step
  }
  return GNX_OK;
}

// everything the step's kernels take by value: if it changes, the captured graph is stale
static void step_key(const gnx_ctx* ctx, std::vector<unsigned char>* key) {
  key->clear();
  auto put = [&](const void* p, size_t n) {
    const unsigned char* b = static_cast<const unsigned char*>(p);
    key->insert(key->end(), b, b + n);
  };
  put(&ctx->pop, sizeof ctx->pop);
  put(&ctx->land, sizeof ctx->land);
  put(&ctx->prm, sizeof ctx->prm);
  put(&ctx->traits, sizeof ctx->traits);
  put(&ctx->draws, sizeof ctx->draws);
  put(&ctx->work, sizeof ctx->work);
  put(&ctx->dens, sizeof ctx->dens);
  put(&ctx->tsk, sizeof ctx->tsk);
  put(&ctx->mut, sizeof ctx->mut);
  const int flags[5] = {ctx->burn, ctx->have_density ? 1 : 0, ctx->mut_delet ? 1 : 0, ctx->grow_guard ? 1 : 0,
                        ctx->tsk_max_bp};
  put(flags, sizeof flags);
}

static GrowthBound growth_bound(const gnx_ctx* ctx) {
  GrowthBound g;
  g.lambda = ctx->cfg.n_births_lambda;
  g.fixed = ctx->cfg.n_births_fixed ? 1 : 0;
  g.genomes = ctx->burn ? 0 : 1;
  g.tsk = (ctx->tsk.enabled && !ctx->burn) ? 1 : 0;
  g.edges_per_birth = 2 * (ctx->tsk_max_bp + 1);
  g.cap = ctx->pop.cap;
  g.born_cap = ctx->tsk.born_cap;
  g.edge_cap = ctx->tsk.edge_cap;
  return g;
}

// The guarded step: k_step_guard -> IF node whose body holds the captured step as a child graph.
// Nothing is captured into the conditional body; `step` is cloned into it (the caller destroys it).
static int guard_graph(gnx_ctx* ctx, cudaGraph_t step, cudaGraph_t* out) {
  cudaGraph_t g = nullptr;
  CK(cudaGraphCreate(&g, 0));
  cudaGraphConditionalHandle h;
  GrowthBound gb = growth_bound(ctx);
  const Counters* c = ctx->d_c;
  void* args[4] = {&c, &gb, &ctx->d_grow, &h};
  cudaKernelNodeParams kp = {};
  kp.func = (void*)k_step_guard;
  kp.gridDim = dim3(1);
  kp.blockDim = dim3(1);
  kp.kernelParams = args;
  cudaGraphNodeParams cp = {};
  cp.type = cudaGraphNodeTypeConditional;
  cp.conditional.type = cudaGraphCondTypeIf;
  cp.conditional.size = 1;
  cudaGraphNode_t guard, cond, child;
  cudaError_t e = cudaGraphConditionalHandleCreate(&h, g, 0, 0);
  if (e == cudaSuccess) e = cudaGraphAddKernelNode(&guard, g, nullptr, 0, &kp);
  cp.conditional.handle = h;
  if (e == cudaSuccess) e = cudaGraphAddNode(&cond, g, &guard, 1, &cp);
  if (e == cudaSuccess) e = cudaGraphAddChildGraphNode(&child, cp.conditional.phGraph_out[0], nullptr, 0, step);
  if (e != cudaSuccess) {
    cudaGraphDestroy(g);
    g_last_error = std::string("building the guarded step graph: ") + cudaGetErrorString(e);
    return GNX_ERR_CUDA;
  }
  *out = g;
  return GNX_OK;
}

static void drop_graph(gnx_ctx* ctx) {
  if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
  ctx->graph_exec = nullptr;
}

static int capture_step(gnx_ctx* ctx) {
  drop_graph(ctx);
  const int64_t launches0 = ctx->launches;
  CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  ctx->capturing = true;
  int r = one_step(ctx);
  ctx->capturing = false;
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
  ctx->graph_kernels = (int)(ctx->launches - launches0);
  ctx->launches = launches0;                 // nothing ran yet
  if (r != GNX_OK) { if (graph) cudaGraphDestroy(graph); return r; }
  if (e != cudaSuccess) { g_last_error = cudaGetErrorString(e); return GNX_ERR_CUDA; }
  if (ctx->grow_guard) {
    cudaGraph_t guarded = nullptr;
    r = guard_graph(ctx, graph, &guarded);
    cudaGraphDestroy(graph);
    if (r != GNX_OK) return r;
    graph = guarded;
    ctx->graph_kernels += 1;
  }
  e = cudaGraphInstantiate(&ctx->graph_exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) { ctx->graph_exec = nullptr; g_last_error = cudaGetErrorString(e); return GNX_ERR_CUDA; }
  step_key(ctx, &ctx->graph_key);
  ctx->graph_captures += 1;
  return GNX_OK;
}

extern "C" int gnx_step(gnx_ctx* ctx, int32_t n_steps) {
  ARG(ctx && n_steps >= 0, "n_steps");
  USE_DEVICE(ctx);
  if (ctx->d_strip) {
    // one strip of a decomposed landscape: whole steps with the barriers and collectives over peer memory
    // (gnx_strip_barrier) -- every rank makes the same call; one CUDA graph per step like the undecomposed run
    ARG(!ctx->prm.ordered, "injected per-individual draws are not supported under strip decomposition");
    if (ctx->strip_connected != ctx->strip_h.world - 1) { g_last_error = "gnx_step on a strip: not every peer is connected"; return GNX_ERR_STATE; }
  }
  if (ctx->records_pending + n_steps > ctx->work.max_records) {
    // never drop a step record: the caller drains them (gnx_read_step_records) at least every
    // max_records steps; nothing has been launched when this is returned
    g_last_error = "step-record buffer would overflow (65536 records): call gnx_read_step_records first";
    return GNX_ERR_STATE;
  }
  const bool lazy = ctx->cfg.mating_radius > 0;
  if (ctx->grow_guard) {                     // a new batch for gnx_step_status
    ctx->grow_enqueued = ctx->grow_host_run = 0;
    ctx->grow_host_stop = ctx->grow_graph = false;
    CK(cudaMemsetAsync(ctx->d_grow, 0, sizeof(gnx_step_status_t), ctx->stream));
  }
  std::vector<unsigned char> key;
  for (int k = 0; k < n_steps; ++k) {
    if (ctx->prm.ordered) {
      // injected draws: ordinals of the entries alive at step start (outside the captured graph)
      ctx->order_valid = false;
      int r = ensure_order(ctx);
      if (r != GNX_OK) return r;
    }
    // the first step of a context runs un-captured (validates state, sets kernel attributes)
    if (ctx->use_graph && !ctx->profiling && ctx->steps_done >= 1) {
      if (k == 0 || !ctx->graph_exec || ctx->prm.ordered) {
        step_key(ctx, &key);
        if (!ctx->graph_exec || key != ctx->graph_key) {
          int r = capture_step(ctx);
          if (r != GNX_OK) return r;
        }
      }
      CK(cudaGraphLaunch(ctx->graph_exec, ctx->stream));
      ctx->grow_graph = ctx->grow_guard;
      ctx->launches += ctx->graph_kernels;
      ctx->graph_launches += 1;
    } else {
      if (ctx->grow_guard) {                 // the same check as k_step_guard, on the host
        Counters h;
        int r = read_counters(ctx, &h);
        if (r != GNX_OK) return r;
        if (!growth_check(growth_bound(ctx), h.n, h.n_slots, h.n_free, h.n_born, h.n_edges, &ctx->grow_host_need)) {
          ctx->grow_host_stop = true;
          break;                             // every later step would stop as well
        }
        ctx->grow_host_run += 1;
      }
      int r = one_step(ctx);
      if (r != GNX_OK) return r;
    }
    ctx->grow_enqueued += 1;
    ctx->records_pending += 1;
    ctx->steps_done += 1;
    ctx->pending = lazy;
    ctx->order_valid = false;
  }
  return GNX_OK;
}

extern "C" int gnx_set_growth_guard(gnx_ctx* ctx, int32_t on) {
  ARG(ctx, "null ctx");
  if (ctx->d_strip) { g_last_error = "the growth guard is not supported under strip decomposition"; return GNX_ERR_STATE; }
  USE_DEVICE(ctx);
  if (on && !ctx->d_grow) DM(ctx, &ctx->d_grow, 1);
  ctx->grow_guard = on != 0;
  ctx->grow_enqueued = ctx->grow_host_run = 0;
  ctx->grow_host_stop = ctx->grow_graph = false;
  return GNX_OK;
}

extern "C" int gnx_set_clock(gnx_ctx* ctx, int64_t t, int64_t tsk_t0) {
  ARG(ctx && t >= 0, "t must be >= 0");
  USE_DEVICE(ctx);
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  if (ctx->grow_guard) ctx->pending = h.pending != 0;     // the guard may have skipped the step that left deaths
  if (ctx->pending || ctx->gi_stage != 0) {
    g_last_error = "gnx_set_clock: a step or a genome assignment is pending (download or upload the population first)";
    return GNX_ERR_STATE;
  }
  PROF(ctx, "k_set_clock");
  k_set_clock<<<1, 1, 0, ctx->stream>>>(ctx->d_c, t, tsk_t0);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  return check_device_err(h);
}

extern "C" int gnx_read_paths(gnx_ctx* ctx, uint32_t* host_paths, int64_t n_words) {
  ARG(ctx && host_paths, "null");
  if (!ctx->have_paths) { g_last_error = "recombination paths not set"; return GNX_ERR_STATE; }
  ARG(n_words == (int64_t)ctx->cfg.n_recomb_paths * 4 * ctx->Wq, "n_words must be n_recomb_paths * 4 * Wq");
  USE_DEVICE(ctx);
  CK(cudaMemcpyAsync(host_paths, ctx->d_paths, (size_t)n_words * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

// ---- sort + simplify of the tskit tables (gnx_simplify.cuh) ------------------------------------------
#define TRY(call)                        \
  do {                                   \
    int r_ = (call);                     \
    if (r_ != GNX_OK) return r_;         \
  } while (0)

static int bits_for(long long x) {          // bits of the largest value x (at least 1)
  int b = 1;
  while (b < 62 && (x >> b) != 0) ++b;
  return b;
}

template <class T>
static int simp_upload(gnx_ctx* ctx, std::vector<void*>& bucket, const T* host, int64_t n, T** dev) {
  DM(ctx, dev, (size_t)n, &bucket);
  if (n > 0) CK(cudaMemcpyAsync(*dev, host, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return GNX_OK;
}

// scratch of one radix sort / scan family: ping-pong pairs, histogram and scan tile sums for n_cap items
struct SimpSort {
  unsigned long long* key[2];
  int32_t* val[2];
  uint32_t* hist;
  u64* tile_sums;
  unsigned int* ticket;
  int n_cap;
};

static int simp_sort_alloc(gnx_ctx* ctx, std::vector<void*>& bucket, int64_t n_cap, int64_t scan_cap, SimpSort* z) {
  n_cap = std::max<int64_t>(n_cap, 1);
  const int64_t ntiles = (n_cap + RS_TILE - 1) / RS_TILE;
  scan_cap = std::max<int64_t>(std::max<int64_t>(scan_cap, n_cap), 256 * ntiles);
  for (int k = 0; k < 2; ++k) {
    DM(ctx, &z->key[k], (size_t)n_cap, &bucket);
    DM(ctx, &z->val[k], (size_t)n_cap, &bucket);
  }
  DM(ctx, &z->hist, (size_t)256 * ntiles, &bucket);
  DM(ctx, &z->tile_sums, (size_t)(scan_cap / SCAN_TILE + 2), &bucket);
  DM(ctx, &z->ticket, 1, &bucket);
  z->n_cap = (int)n_cap;
  return GNX_OK;
}

// LSD radix sort of z->key[0] / z->val[0] on the low `bits` key bits; n items, or *n_dev when given.
// *in = the buffer holding the result.
static int simp_sort(gnx_ctx* ctx, SimpSort& z, int n, const int* n_dev, int bits, int* in) {
  const int grid = std::max(1, std::min((z.n_cap + RS_TILE - 1) / RS_TILE, grid_for(ctx, 8)));
  *in = 0;
  for (int shift = 0; shift < bits; shift += 8) {
    PROF(ctx, "k_radix_hist");
    k_radix_hist<<<grid, RS_BLOCK, 0, ctx->stream>>>(z.key[*in], n, n_dev, shift, z.hist);
    LAUNCHED(ctx);
    TRY(run_scan(ctx, RadixScan{z.hist, n, n_dev}, "scan_radix", z.tile_sums, z.ticket));
    PROF(ctx, "k_radix_scatter");
    k_radix_scatter<<<grid, RS_BLOCK, 0, ctx->stream>>>(z.key[*in], z.val[*in], z.key[*in ^ 1], z.val[*in ^ 1], n,
                                                        n_dev, shift, z.hist);
    LAUNCHED(ctx);
    *in ^= 1;
  }
  return GNX_OK;
}

template <class F>
static int simp_scan(gnx_ctx* ctx, const SimpSort& z, F f, const char* name) {
  return run_scan(ctx, f, name, z.tile_sums, z.ticket);
}

static int read_ints(gnx_ctx* ctx, const int32_t* dev, int32_t* host, size_t n) {
  CK(cudaMemcpyAsync(host, dev, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

static int simplify_impl(gnx_ctx* ctx, const gnx_tables_t* T, const int32_t* samples, int64_t n_samples,
                         std::vector<void*>& B, std::vector<void*>& A, int64_t* out_sizes) {
  const int64_t lim = 1ll << 29;
  ARG(T->n_nodes >= 0 && T->n_nodes < lim && T->n_edges >= 0 && T->n_edges < lim && T->n_individuals >= 0 &&
      T->n_individuals < lim && T->n_sites >= 0 && T->n_sites < lim && T->n_mutations >= 0 && T->n_mutations < lim,
      "table sizes");
  ARG(n_samples >= 0 && n_samples <= T->n_nodes && (n_samples == 0 || samples), "samples");
  ARG(T->n_location >= 0 && T->sequence_length >= 0, "n_location / sequence_length");
  ARG((T->n_nodes == 0 || (T->node_time && T->node_population && T->node_individual)) &&
      (T->n_edges == 0 || (T->edge_left && T->edge_right && T->edge_parent && T->edge_child)) &&
      (T->n_individuals == 0 || (T->individual_flags && T->individual_idx &&
                                 (T->n_location == 0 || T->individual_location))) &&
      (T->n_sites == 0 || T->site_position) &&
      (T->n_mutations == 0 || (T->mutation_site && T->mutation_node && T->mutation_time)), "null column");
  cudaStream_t st = ctx->stream;
  const int n_in = (int)T->n_nodes, E = (int)T->n_edges, ns = (int)n_samples;
  const int GD = grid_for(ctx, 4);
  auto gr = [&](int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, grid_for(ctx, 8))); };

  Simp S{};
  S.n_in = n_in;
  S.n_edges = E;
  S.n_ind = (int)T->n_individuals;
  S.n_sites = (int)T->n_sites;
  S.n_mut = (int)T->n_mutations;
  S.n_samples = ns;
  S.L = T->sequence_length;
  int32_t *d_pop, *d_iflags;
  double *d_mtime, *d_iloc;
  int64_t* d_iidx;
  TRY(simp_upload(ctx, B, T->node_time, n_in, (double**)&S.time));
  TRY(simp_upload(ctx, B, T->node_population, n_in, &d_pop));
  TRY(simp_upload(ctx, B, T->node_individual, n_in, (int32_t**)&S.ind));
  TRY(simp_upload(ctx, B, T->edge_left, E, (double**)&S.el));
  TRY(simp_upload(ctx, B, T->edge_right, E, (double**)&S.er));
  TRY(simp_upload(ctx, B, T->edge_parent, E, (int32_t**)&S.ep));
  TRY(simp_upload(ctx, B, T->edge_child, E, (int32_t**)&S.ec));
  TRY(simp_upload(ctx, B, T->site_position, T->n_sites, (double**)&S.site_pos));
  TRY(simp_upload(ctx, B, T->mutation_site, T->n_mutations, (int32_t**)&S.m_site));
  TRY(simp_upload(ctx, B, T->mutation_node, T->n_mutations, (int32_t**)&S.m_node));
  TRY(simp_upload(ctx, B, T->mutation_time, T->n_mutations, &d_mtime));
  TRY(simp_upload(ctx, B, T->individual_flags, T->n_individuals, &d_iflags));
  TRY(simp_upload(ctx, B, T->individual_location, T->n_individuals * T->n_location, &d_iloc));
  TRY(simp_upload(ctx, B, T->individual_idx, T->n_individuals, &d_iidx));
  TRY(simp_upload(ctx, B, samples, ns, (int32_t**)&S.samples));
  DM(ctx, &S.smap, (size_t)n_in, &B);
  CK(cudaMemsetAsync(S.smap, 0xff, (size_t)n_in * 4, st));
  int32_t* hsz;                        // sizes the host reads back
  DM(ctx, &S.err, 1, &B);
  DM(ctx, &hsz, 4, &B);

  // ---- refuse what the algorithm cannot take
  PROF(ctx, "k_simp_check_edges");
  k_simp_check_edges<<<gr(E), 256, 0, st>>>(S);
  LAUNCHED(ctx);
  PROF(ctx, "k_simp_check_rest");
  k_simp_check_rest<<<gr(std::max<int64_t>({(int64_t)n_in, T->n_mutations, n_samples})), 256, 0, st>>>(S);
  LAUNCHED(ctx);
  int32_t err = 0;
  TRY(read_ints(ctx, S.err, &err, 1));
  ARG(!(err & SE_ID), "an edge names a node that does not exist");
  ARG(!(err & SE_TIME), "an edge whose parent is not older than its child");
  ARG(!(err & SE_INTERVAL), "an edge outside 0 <= left < right <= sequence_length");
  ARG(!(err & SE_IND), "a node names an individual that does not exist");
  ARG(!(err & SE_SITE), "a mutation names a site that does not exist");
  ARG(!(err & SE_SAMPLE), "a sample is out of range or repeated");

  // ---- distinct positions; edges sorted as TableCollection.sort(); levels and groups
  const int n_pos = 2 * E + 2;
  SimpSort z;
  TRY(simp_sort_alloc(ctx, B, std::max(n_pos, n_in), std::max<int64_t>(T->n_individuals, T->n_mutations), &z));
  int in = 0;
  PROF(ctx, "k_simp_pos_keys");
  k_simp_pos_keys<<<gr(E), 256, 0, st>>>(S, z.key[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, z, n_pos, nullptr, 64, &in));
  DM(ctx, &S.uniq, (size_t)n_pos, &B);
  TRY(simp_scan(ctx, z, UniqScan{z.key[in], S.uniq, hsz, n_pos}, "scan_simp_uniq"));
  int32_t n_uniq = 0;
  TRY(read_ints(ctx, hsz, &n_uniq, 1));
  S.pb = bits_for(n_uniq - 1);
  const int nb_node = bits_for(std::max(n_in - 1, 0));

  int32_t* prank;
  DM(ctx, &prank, (size_t)n_in, &B);
  PROF(ctx, "k_simp_time_keys");
  k_simp_time_keys<<<gr(n_in), 256, 0, st>>>(S.time, nullptr, n_in, z.key[0], z.val[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, z, n_in, nullptr, 64, &in));
  PROF(ctx, "k_simp_rank");
  k_simp_rank<<<gr(n_in), 256, 0, st>>>(z.val[in], n_in, prank);
  LAUNCHED(ctx);
  uint32_t *lr, *rr;
  DM(ctx, &lr, (size_t)E, &B);
  DM(ctx, &rr, (size_t)E, &B);
  PROF(ctx, "k_simp_edge_keys");
  k_simp_edge_keys<<<gr(E), 256, 0, st>>>(S, n_uniq, lr, rr, z.key[0], z.val[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, z, E, nullptr, nb_node + S.pb, &in));
  if (in) {                                          // the second pass starts from buffer 0
    CK(cudaMemcpyAsync(z.val[0], z.val[1], (size_t)E * 4, cudaMemcpyDeviceToDevice, st));
  }
  PROF(ctx, "k_simp_edge_keys2");
  k_simp_edge_keys2<<<gr(E), 256, 0, st>>>(S, prank, z.val[0], z.key[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, z, E, nullptr, nb_node, &in));
  DM(ctx, &S.sl, (size_t)E, &B);
  DM(ctx, &S.sr, (size_t)E, &B);
  DM(ctx, &S.sp, (size_t)E, &B);
  DM(ctx, &S.sc, (size_t)E, &B);
  DM(ctx, &S.grp_of, (size_t)E, &B);
  DM(ctx, &S.grp_parent, (size_t)E, &B);
  DM(ctx, &S.lvl_start, (size_t)E + 1, &B);
  DM(ctx, &S.lvl_g0, (size_t)E + 1, &B);
  PROF(ctx, "k_simp_edge_gather");
  k_simp_edge_gather<<<gr(E), 256, 0, st>>>(S, z.val[in], lr, rr);
  LAUNCHED(ctx);
  TRY(simp_scan(ctx, z, LevelScan{S, hsz}, "scan_simp_levels"));
  int32_t lg[2] = {0, 0};
  TRY(read_ints(ctx, hsz, lg, 2));
  const int n_levels = lg[0];
  std::vector<int32_t> lvl_start(n_levels + 1), lvl_g0(n_levels + 1);
  TRY(read_ints(ctx, S.lvl_start, lvl_start.data(), n_levels + 1));
  TRY(read_ints(ctx, S.lvl_g0, lvl_g0.data(), n_levels + 1));
  int max_ne = 1, max_ng = 1;
  for (int k = 0; k < n_levels; ++k) {
    max_ne = std::max(max_ne, lvl_start[k + 1] - lvl_start[k]);
    max_ng = std::max(max_ng, lvl_g0[k + 1] - lvl_g0[k]);
  }

  // ---- the levels, youngest first; pools that overflow are grown and the levels run again
  int64_t cap_p = std::max<int64_t>(4096, 2 * (int64_t)max_ne);
  int64_t cap_a = (int64_t)ns + 2 * (int64_t)E + 4096, cap_r = 2 * (int64_t)E + 4096;
  int32_t sv[SV_N];
  SimpSort ze{};
  for (;;) {
    ARG(cap_p < lim && cap_a < 2 * lim && cap_r < 2 * lim, "the simplification needs more than 2^29 pieces");
    S.cap_p = (int)cap_p;
    S.cap_a = (int)cap_a;
    S.cap_r = (int)cap_r;
    const size_t P2 = 2 * (size_t)cap_p;
    DM(ctx, &S.sv, SV_N, &A);
    DM(ctx, &S.a_off, (size_t)n_in, &A);
    DM(ctx, &S.a_end, (size_t)n_in, &A);
    DM(ctx, &S.a_lo, (size_t)cap_a, &A);
    DM(ctx, &S.a_hi, (size_t)cap_a, &A);
    DM(ctx, &S.a_node, (size_t)cap_a, &A);
    DM(ctx, &S.pcnt, (size_t)max_ne, &A);
    DM(ctx, &S.pj, (size_t)max_ne, &A);
    DM(ctx, &S.pc_node, (size_t)cap_p, &A);
    DM(ctx, &S.rcnt, (size_t)cap_p, &A);
    DM(ctx, &S.inv, P2, &A);
    DM(ctx, &S.cover, 2 * P2, &A);
    DM(ctx, &S.bex, P2, &A);
    DM(ctx, &S.b_pos, P2, &A);
    DM(ctx, &S.b_end, P2, &A);
    DM(ctx, &S.b_cls, P2, &A);
    DM(ctx, &S.b_node, P2, &A);
    DM(ctx, &S.b_g, P2, &A);
    DM(ctx, &S.flag, (size_t)max_ng, &A);
    DM(ctx, &S.vout, (size_t)max_ng, &A);
    DM(ctx, &S.out_src, (size_t)ns + n_in, &A);
    DM(ctx, &S.r_lo, (size_t)cap_r, &A);
    DM(ctx, &S.r_hi, (size_t)cap_r, &A);
    DM(ctx, &S.r_par, (size_t)cap_r, &A);
    DM(ctx, &S.r_child, (size_t)cap_r, &A);
    TRY(simp_sort_alloc(ctx, A, (int64_t)P2, max_ne, &ze));
    for (int k = 0; k < 2; ++k) {
      S.ev_key[k] = ze.key[k];
      S.ev_val[k] = ze.val[k];
    }
    // rank of L among the positions: the last one
    PROF(ctx, "k_simp_init_samples");
    k_simp_init_samples<<<gr(ns), 256, 0, st>>>(S, (uint32_t)(n_uniq - 1));
    LAUNCHED(ctx);
    for (int k = 0; k < n_levels; ++k) {
      const int e0 = lvl_start[k], ne = lvl_start[k + 1] - e0, g0 = lvl_g0[k], ng = lvl_g0[k + 1] - g0;
      PROF(ctx, "k_simp_count");
      k_simp_count<<<gr(ne), 256, 0, st>>>(S, e0, ne);
      LAUNCHED(ctx);
      TRY(simp_scan(ctx, ze, PieceScan{S, ne}, "scan_simp_pieces"));
      PROF(ctx, "k_simp_pieces");
      k_simp_pieces<<<GD, 256, 0, st>>>(S, e0, ne, g0);
      LAUNCHED(ctx);
      int ein = 0;
      TRY(simp_sort(ctx, ze, 0, S.sv + SV_NEV, bits_for(std::max(ng - 1, 0)) + S.pb, &ein));
      PROF(ctx, "k_simp_event_inv");
      k_simp_event_inv<<<GD, 256, 0, st>>>(S, ze.val[ein]);
      LAUNCHED(ctx);
      TRY(simp_scan(ctx, ze, CoverScan{S, ze.val[ein]}, "scan_simp_cover"));
      TRY(simp_scan(ctx, ze, BoundScan{S, ze.key[ein]}, "scan_simp_bounds"));
      CK(cudaMemsetAsync(S.flag, 0, (size_t)ng * 4, st));
      PROF(ctx, "k_simp_flag");
      k_simp_flag<<<GD, 256, 0, st>>>(S);
      LAUNCHED(ctx);
      TRY(simp_scan(ctx, ze, ParentScan{S, g0, ng}, "scan_simp_parents"));
      TRY(simp_scan(ctx, ze, SegScan{S, g0}, "scan_simp_segments"));
      PROF(ctx, "k_simp_runs");
      k_simp_runs<<<GD, 256, 0, st>>>(S, g0, false);
      LAUNCHED(ctx);
      TRY(simp_scan(ctx, ze, RunScan{S}, "scan_simp_runs"));
      PROF(ctx, "k_simp_runs");
      k_simp_runs<<<GD, 256, 0, st>>>(S, g0, true);
      LAUNCHED(ctx);
      PROF(ctx, "k_simp_level_end");
      k_simp_level_end<<<1, 32, 0, st>>>(S);
      LAUNCHED(ctx);
    }
    TRY(read_ints(ctx, S.sv, sv, SV_N));
    if (!sv[SV_OVF]) break;
    cap_p = std::max<int64_t>(2 * cap_p, sv[SV_NEED_P]);
    cap_a = std::max<int64_t>(2 * cap_a, sv[SV_NEED_A]);
    cap_r = std::max<int64_t>(2 * cap_r, sv[SV_NEED_R]);
    CK(cudaStreamSynchronize(st));
    free_bucket(A);
  }
  const int n_out = sv[SV_OUT], R = sv[SV_RTOP];

  // ---- the result: nodes, individuals, mutations, edges in final order
  std::vector<void*>& Rb = ctx->simp_allocs;
  gnx_tables_t& O = ctx->simp;
  O = gnx_tables_t{};
  O.sequence_length = T->sequence_length;
  O.n_location = T->n_location;
  DM(ctx, &O.node_flags, (size_t)n_out, &Rb);
  DM(ctx, &O.node_time, (size_t)n_out, &Rb);
  DM(ctx, &O.node_population, (size_t)n_out, &Rb);
  DM(ctx, &O.node_individual, (size_t)n_out, &Rb);
  DM(ctx, &O.individual_flags, (size_t)T->n_individuals, &Rb);
  DM(ctx, &O.individual_location, (size_t)(T->n_individuals * T->n_location), &Rb);
  DM(ctx, &O.individual_idx, (size_t)T->n_individuals, &Rb);
  DM(ctx, &O.mutation_site, (size_t)T->n_mutations, &Rb);
  DM(ctx, &O.mutation_node, (size_t)T->n_mutations, &Rb);
  DM(ctx, &O.mutation_time, (size_t)T->n_mutations, &Rb);
  DM(ctx, &O.edge_left, (size_t)R, &Rb);
  DM(ctx, &O.edge_right, (size_t)R, &Rb);
  DM(ctx, &O.edge_parent, (size_t)R, &Rb);
  DM(ctx, &O.edge_child, (size_t)R, &Rb);
  int32_t* remap;
  DM(ctx, &remap, (size_t)T->n_individuals, &B);
  PROF(ctx, "k_simp_mark_ind");
  k_simp_mark_ind<<<gr(n_out), 256, 0, st>>>(S, n_out, remap);
  LAUNCHED(ctx);
  TRY(simp_scan(ctx, z, IndScan{S.n_ind, (int)T->n_location, remap, d_iflags, d_iloc, d_iidx, O.individual_flags,
                                O.individual_location, O.individual_idx, hsz}, "scan_simp_individuals"));
  PROF(ctx, "k_simp_nodes_out");
  k_simp_nodes_out<<<gr(n_out), 256, 0, st>>>(S, n_out, d_pop, remap, O.node_flags, O.node_time, O.node_population,
                                              O.node_individual);
  LAUNCHED(ctx);
  TRY(simp_scan(ctx, z, MutScan{S, d_mtime, O.mutation_site, O.mutation_node, O.mutation_time, hsz + 1},
                "scan_simp_mutations"));
  SimpSort zr;
  TRY(simp_sort_alloc(ctx, B, std::max(n_out, R), 0, &zr));
  int32_t* orank;
  DM(ctx, &orank, (size_t)n_out, &B);
  PROF(ctx, "k_simp_time_keys");
  k_simp_time_keys<<<gr(n_out), 256, 0, st>>>(S.time, S.out_src, n_out, zr.key[0], zr.val[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, zr, n_out, nullptr, 64, &in));
  PROF(ctx, "k_simp_rank");
  k_simp_rank<<<gr(n_out), 256, 0, st>>>(zr.val[in], n_out, orank);
  LAUNCHED(ctx);
  const int nb_out = bits_for(std::max(n_out - 1, 0));
  PROF(ctx, "k_simp_run_keys");
  k_simp_run_keys<<<gr(R), 256, 0, st>>>(S, R, zr.key[0], zr.val[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, zr, R, nullptr, nb_out + S.pb, &in));
  if (in) CK(cudaMemcpyAsync(zr.val[0], zr.val[1], (size_t)R * 4, cudaMemcpyDeviceToDevice, st));
  PROF(ctx, "k_simp_run_keys2");
  k_simp_run_keys2<<<gr(R), 256, 0, st>>>(S, R, orank, zr.val[0], zr.key[0]);
  LAUNCHED(ctx);
  TRY(simp_sort(ctx, zr, R, nullptr, nb_out, &in));
  TRY(simp_scan(ctx, zr, SquashScan{S, R, zr.val[in], O.edge_left, O.edge_right, O.edge_parent, O.edge_child,
                                    hsz + 2}, "scan_simp_squash"));
  int32_t outn[3];
  TRY(read_ints(ctx, hsz, outn, 3));
  O.n_nodes = n_out;
  O.n_individuals = outn[0];
  O.n_mutations = outn[1];
  O.n_edges = outn[2];
  O.n_sites = T->n_sites;
  out_sizes[0] = O.n_nodes;
  out_sizes[1] = O.n_edges;
  out_sizes[2] = O.n_individuals;
  out_sizes[3] = O.n_mutations;
  return GNX_OK;
}

extern "C" int gnx_simplify(gnx_ctx* ctx, const gnx_tables_t* tables, const int32_t* samples, int64_t n_samples,
                            int64_t* out_sizes) {
  ARG(ctx && tables && out_sizes, "null");
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  free_bucket(ctx->simp_allocs);
  ctx->simp = gnx_tables_t{};
  std::vector<void*> scratch, pools;            // pools: the level pass's, grown and replaced on overflow
  int r = simplify_impl(ctx, tables, samples, n_samples, scratch, pools, out_sizes);
  cudaStreamSynchronize(ctx->stream);
  free_bucket(scratch);
  free_bucket(pools);
  if (r != GNX_OK) {
    free_bucket(ctx->simp_allocs);
    ctx->simp = gnx_tables_t{};
  }
  return r;
}

extern "C" int gnx_simplify_result(gnx_ctx* ctx, gnx_tables_t* out) {
  ARG(ctx && out, "null");
  const gnx_tables_t& O = ctx->simp;
  if (ctx->simp_allocs.empty()) { g_last_error = "no gnx_simplify result to copy"; return GNX_ERR_STATE; }
  ARG(out->n_nodes == O.n_nodes && out->n_edges == O.n_edges && out->n_individuals == O.n_individuals &&
      out->n_mutations == O.n_mutations && out->n_location == O.n_location, "sizes differ from gnx_simplify's");
  USE_DEVICE(ctx);
  cudaStream_t st = ctx->stream;
  auto get = [&](void* h, const void* d, size_t bytes) -> int {
    if (bytes == 0) return GNX_OK;
    ARG(h, "null column");
    CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, st));
    return GNX_OK;
  };
  const size_t nn = (size_t)O.n_nodes, ne = (size_t)O.n_edges, ni = (size_t)O.n_individuals, nm = (size_t)O.n_mutations;
  TRY(get(out->node_flags, O.node_flags, nn * 4));
  TRY(get(out->node_time, O.node_time, nn * 8));
  TRY(get(out->node_population, O.node_population, nn * 4));
  TRY(get(out->node_individual, O.node_individual, nn * 4));
  TRY(get(out->edge_left, O.edge_left, ne * 8));
  TRY(get(out->edge_right, O.edge_right, ne * 8));
  TRY(get(out->edge_parent, O.edge_parent, ne * 4));
  TRY(get(out->edge_child, O.edge_child, ne * 4));
  TRY(get(out->individual_flags, O.individual_flags, ni * 4));
  TRY(get(out->individual_location, O.individual_location, ni * (size_t)O.n_location * 8));
  TRY(get(out->individual_idx, O.individual_idx, ni * 8));
  TRY(get(out->mutation_site, O.mutation_site, nm * 4));
  TRY(get(out->mutation_node, O.mutation_node, nm * 4));
  TRY(get(out->mutation_time, O.mutation_time, nm * 8));
  CK(cudaStreamSynchronize(st));
  free_bucket(ctx->simp_allocs);
  ctx->simp = gnx_tables_t{};
  return GNX_OK;
}

extern "C" int gnx_step_status(gnx_ctx* ctx, gnx_step_status_t* out) {
  ARG(ctx && out, "null");
  if (!ctx->grow_guard) { g_last_error = "the growth guard is off"; return GNX_ERR_STATE; }
  USE_DEVICE(ctx);
  gnx_step_status_t st;
  CK(cudaMemcpyAsync(&st, ctx->d_grow, sizeof st, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  st.steps_run += (int32_t)ctx->grow_host_run;
  if (ctx->grow_host_stop || !ctx->grow_graph) {       // the last check of the batch ran on the host
    st.stopped = ctx->grow_host_stop ? 1 : 0;
    st.need_entries = ctx->grow_host_need.need_entries;
    st.need_slots = ctx->grow_host_need.need_slots;
    st.need_births = ctx->grow_host_need.need_births;
    st.need_edges = ctx->grow_host_need.need_edges;
  }
  // launches the guard skipped wrote no record and did not advance the step counter
  const int64_t skipped = ctx->grow_enqueued - st.steps_run;
  ctx->records_pending -= skipped;
  ctx->steps_done -= skipped;
  ctx->grow_enqueued = st.steps_run;
  st.capacity = ctx->pop.cap;
  st.born_capacity = ctx->tsk.enabled ? ctx->tsk.born_cap : 0;
  st.edge_capacity = ctx->tsk.enabled ? ctx->tsk.edge_cap : 0;
  *out = st;
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  return check_device_err(h);
}

// ---- re-allocation of the buffers sized from a capacity ----------------------------------------
// One buffer to grow: rows x (old -> new) bytes, row r at r * old / r * new (a [rows][cap] array);
// rows = 1 for everything laid out by entry.
struct Regrow {
  void** p;
  size_t old_bytes, new_bytes;
  size_t rows;
  std::vector<void*>* bucket;
  void* q;
};

// Allocates every new buffer before it frees an old one: a failed allocation leaves the context on its
// old buffers.  The old contents are copied (state and scratch alike) and the rest is zeroed.
static int regrow(gnx_ctx* ctx, std::vector<Regrow>& v) {
  for (auto& g : v) {
    g.q = nullptr;
    if (cudaMalloc(&g.q, std::max<size_t>(g.new_bytes, 1)) != cudaSuccess) {
      cudaGetLastError();
      for (auto& f : v) if (f.q) cudaFree(f.q);
      g_last_error = "out of device memory growing the buffers (the context keeps its old ones)";
      return GNX_ERR_CUDA;
    }
  }
  cudaStream_t s = ctx->stream;
  for (auto& g : v) {
    CK(cudaMemsetAsync(g.q, 0, std::max<size_t>(g.new_bytes, 1), s));
    const size_t po = g.old_bytes / g.rows, pn = g.new_bytes / g.rows;
    for (size_t r = 0; r < g.rows; ++r)
      CK(cudaMemcpyAsync((char*)g.q + r * pn, (const char*)*g.p + r * po, po, cudaMemcpyDeviceToDevice, s));
  }
  CK(cudaStreamSynchronize(s));
  for (auto& g : v) {
    std::replace(g.bucket->begin(), g.bucket->end(), *g.p, g.q);
    CK(cudaFree(*g.p));
    *g.p = g.q;
  }
  return GNX_OK;
}

template <class T>
static void regrow_add(std::vector<Regrow>& v, T** p, size_t n_old, size_t n_new, std::vector<void*>* bucket,
                       size_t rows = 1) {
  v.push_back(Regrow{reinterpret_cast<void**>(p), std::max<size_t>(n_old, 1) * rows * sizeof(T),
                     std::max<size_t>(n_new, 1) * rows * sizeof(T), rows, bucket, nullptr});
}

extern "C" int gnx_reserve(gnx_ctx* ctx, int64_t capacity) {
  ARG(ctx, "null ctx");
  if (ctx->d_strip) { g_last_error = "gnx_reserve: a strip keeps its capacity"; return GNX_ERR_STATE; }
  ARG(capacity < (1ll << 31) - 4096, "capacity");
  if (capacity <= ctx->pop.cap) return GNX_OK;
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  Pop& P = ctx->pop;
  Work& W = ctx->work;
  const size_t co = (size_t)P.cap, cn = (size_t)capacity;
  const size_t T1 = std::max(1, ctx->cfg.n_traits), row = (size_t)2 * ctx->Wq;
  auto hist = [](size_t c) { return (size_t)256 * (c / RS_TILE + 2); };
  auto tiles = [&](size_t c) { return std::max(std::max(c, (size_t)ctx->ncell), hist(c)) / SCAN_TILE + 2; };
  auto heavy = [](size_t c) { return c / 4 + 1024; };
  std::vector<Regrow> v;
  std::vector<void*>* A = &ctx->allocs;
  for (int h = 0; h < 2; ++h) {
    regrow_add(v, &P.xy[h], co, cn, A);
    regrow_add(v, &P.age[h], co, cn, A);
    regrow_add(v, &P.sex[h], co, cn, A);
    regrow_add(v, &P.idx[h], co, cn, A);
    regrow_add(v, &P.gslot[h], co, cn, A);
    regrow_add(v, &P.z[h], co, cn, A, T1);              // [T][cap]
    regrow_add(v, &P.fit[h], co, cn, A);
    regrow_add(v, &P.ord[h], co, cn, A);
    regrow_add(v, &W.sort_keys[h], co, cn, A);
    regrow_add(v, &W.sort_vals[h], co, cn, A);
    if (ctx->tsk.enabled)
      for (int b = 0; b < 2; ++b) regrow_add(v, &P.node[h][b], co, cn, &ctx->tsk_allocs);
  }
  regrow_add(v, &P.G, co * row, cn * row, A);
  regrow_add(v, &P.free_slots, co, cn, A);
  regrow_add(v, &ctx->d_stage_genomes, co * row, cn * row, A);
  regrow_add(v, &ctx->d_stage_z, co * T1, cn * T1, A);
  regrow_add(v, &W.mkey, co, cn, A);
  regrow_add(v, &W.bucket, co, cn, A);
  regrow_add(v, &W.skey, co, cn, A);
  regrow_add(v, &W.inv, co, cn, A);
  regrow_add(v, &W.perm, co, cn, A);
  regrow_add(v, &W.sort_hist, hist(co), hist(cn), A);
  double* scratch = static_cast<double*>(W.scratch);
  regrow_add(v, &scratch, 2 * co * T1, 2 * cn * T1, A);
  regrow_add(v, &W.mate, co, cn, A);
  regrow_add(v, &W.heavy, heavy(co), heavy(cn), A);
  regrow_add(v, &W.fm_list, co, cn, A);
  regrow_add(v, &W.n_nbrs, co, cn, A);
  regrow_add(v, &W.pairs, 2 * co, 2 * cn, A);
  regrow_add(v, &W.pair_slots, 2 * co, 2 * cn, A);
  regrow_add(v, &W.nb, co, cn, A);
  regrow_add(v, &W.off_start, co, cn, A);
  regrow_add(v, &W.off_pair, co, cn, A);
  regrow_add(v, &W.mid, co, cn, A);
  regrow_add(v, &W.alive, co, cn, A);
  regrow_add(v, &W.death_p, co, cn, A);
  regrow_add(v, &W.disp_tries, co, cn, A);
  regrow_add(v, &W.tile_sums, tiles(co), tiles(cn), A);
  regrow_add(v, &W.e_out, co * ctx->cfg.n_layers, cn * ctx->cfg.n_layers, A);
  int r = regrow(ctx, v);
  if (r != GNX_OK) return r;
  W.scratch = scratch;
  W.heavy_cap = (int32_t)heavy(cn);
  P.cap = (int32_t)capacity;
  ctx->cfg.capacity = capacity;
  ctx->prm.c.capacity = capacity;
  return GNX_OK;                       // the pointers changed: the next gnx_step captures its graph again
}

extern "C" int gnx_tskit_reserve(gnx_ctx* ctx, int64_t edge_capacity, int64_t birth_capacity) {
  ARG(ctx, "null ctx");
  if (!ctx->tsk.enabled) { g_last_error = "tskit recording not enabled"; return GNX_ERR_STATE; }
  ARG(edge_capacity < (1ll << 31) && birth_capacity < (1ll << 31), "capacities");
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  Tsk& T = ctx->tsk;
  const size_t T1 = std::max(1, ctx->cfg.n_traits);
  const size_t eo = (size_t)T.edge_cap, en = (size_t)std::max<int64_t>(edge_capacity, T.edge_cap);
  const size_t bo = (size_t)T.born_cap, bn = (size_t)std::max<int64_t>(birth_capacity, T.born_cap);
  std::vector<Regrow> v;
  std::vector<void*>* B = &ctx->tsk_allocs;
  if (en > eo) {
    regrow_add(v, &T.e_left, eo, en, B);
    regrow_add(v, &T.e_right, eo, en, B);
    regrow_add(v, &T.e_parent, eo, en, B);
    regrow_add(v, &T.e_child, eo, en, B);
  }
  if (bn > bo) {
    regrow_add(v, &T.b_idx, bo, bn, B);
    regrow_add(v, &T.b_x, bo, bn, B);
    regrow_add(v, &T.b_y, bo, bn, B);
    regrow_add(v, &T.b_z, bo, bn, B, T1);               // [T][born_cap]
    regrow_add(v, &T.b_time, bo, bn, B);
  }
  int r = regrow(ctx, v);
  if (r != GNX_OK) return r;
  T.edge_cap = (int32_t)en;
  T.born_cap = (int32_t)bn;
  return GNX_OK;
}

// ---- strip domain decomposition of one landscape (gnx_strip.cuh; SURVEY.md section 8e-2) -------
static int strip_upload(gnx_ctx* ctx) {
  CK(cudaMemcpyAsync(ctx->d_strip, &ctx->strip_h, sizeof(Strip), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

extern "C" int gnx_strip_enable(gnx_ctx* ctx, const gnx_strip_config_t* sc) {
  ARG(ctx && sc && sc->first_rows, "null");
  USE_DEVICE(ctx);
  ARG(!ctx->d_strip, "strip decomposition is already enabled for this context");
  ARG(sc->world >= 1 && sc->world <= GNX_STRIP_MAX_WORLD && sc->rank >= 0 && sc->rank < sc->world, "rank / world");
  ARG(ctx->cfg.mating_radius > 0, "strip decomposition needs a mating radius (panmixia has no locality)");
  ARG(!ctx->tsk.enabled, "strip decomposition does not carry tskit rows");
  ARG(!ctx->grow_guard, "a strip keeps its capacity: turn the growth guard off first");
  ARG(!ctx->cols, "strip decomposition does not carry the column genotype layout");
  ARG(!ctx->mut.enabled || !ctx->mut.own_tables,
      "strip decomposition does not carry the tskit genotype layout or trait mutation");
  ARG(!ctx->prm.ordered, "injected draws are not supported under strip decomposition");
  Strip& S = ctx->strip_h;
  memset(&S, 0, sizeof S);
  S.enabled = 1;
  S.rank = sc->rank;
  S.world = sc->world;
  for (int r = 0; r <= sc->world; ++r) S.bounds[r] = sc->first_rows[r];
  ARG(S.bounds[0] == 0 && S.bounds[sc->world] == ctx->land.ncy, "first_rows must span the mating grid [0, ncy]");
  for (int r = 0; r < sc->world; ++r) ARG(S.bounds[r + 1] - S.bounds[r] >= 2, "every strip needs at least two mating-grid rows");
  S.row0 = S.bounds[S.rank];
  S.row1 = S.bounds[S.rank + 1];
  // landscape rows that contain the strip's individuals: y in [row0, row1) * cell_size
  S.ly0 = std::max(0, (int)std::floor(S.row0 * ctx->land.cell_size));
  S.ly1 = S.rank == S.world - 1 ? ctx->cfg.dim_y
                                : std::min(ctx->cfg.dim_y, (int)std::floor(S.row1 * ctx->land.cell_size) + 1);
  S.rec_bytes = strip_header_bytes(ctx->cfg.n_traits) + 32 * ctx->Wq;
  S.cap[STRIP_BUF_MIGRANTS] = (int32_t)std::max<int64_t>(1024, sc->migrant_capacity);
  S.cap[STRIP_BUF_HALO] = (int32_t)std::max<int64_t>(1024, sc->halo_capacity);
  S.cap[STRIP_BUF_NEWBORNS] = (int32_t)std::max<int64_t>(1024, sc->migrant_capacity);
  S.cap[STRIP_BUF_CHOICES] = (int32_t)std::max<int64_t>(1024, sc->halo_capacity);
  // one block: 256 bytes of counters, then the four receive buffers (a single CUDA IPC handle exports it)
  size_t off = 256;
  for (int k = 0; k < STRIP_N_BUF; ++k) {
    ctx->strip_buf_off[k] = (int64_t)off;
    const size_t rec = k == STRIP_BUF_CHOICES ? sizeof(StripChoice) : (size_t)S.rec_bytes;
    off += ((size_t)S.cap[k] * rec + 255) & ~(size_t)255;
  }
  // ... and the synchronisation page (k_strip_barrier): flags, births, max(N) and counts slots, one per rank
  S.counts_cap = ctx->have_density ? ((2 * ctx->dens.npts + 63) & ~63) : 0;
  ctx->strip_sync_off = (int64_t)off;
  const size_t sync_bytes = STRIP_SYNC_COUNTS + (size_t)GNX_STRIP_MAX_WORLD * S.counts_cap * 4;
  off += (sync_bytes + 255) & ~(size_t)255;
  ctx->strip_block_bytes = off;
  CK(cudaMalloc((void**)&ctx->strip_block, off));
  CK(cudaMemsetAsync(ctx->strip_block, 0, 256, ctx->stream));
  CK(cudaMemsetAsync(ctx->strip_block + ctx->strip_sync_off, 0, sync_bytes, ctx->stream));
  for (int k = 0; k < STRIP_N_BUF; ++k) {
    S.peer[S.rank].buf[k] = ctx->strip_block + ctx->strip_buf_off[k];
    S.peer[S.rank].count[k] = reinterpret_cast<int32_t*>(ctx->strip_block) + 16 * k;
  }
  S.peer[S.rank].sync = ctx->strip_block + ctx->strip_sync_off;
  ctx->strip_connected = 0;
  S.list_cap = S.cap[STRIP_BUF_MIGRANTS] + 2 * S.cap[STRIP_BUF_HALO];
  DM(ctx, &S.list_entry, (size_t)S.list_cap, &ctx->strip_allocs);
  DM(ctx, &S.list_dest, (size_t)S.list_cap, &ctx->strip_allocs);
  DM(ctx, &S.list_n, 4, &ctx->strip_allocs);
  S.err = S.list_n + 1;
  DM(ctx, &S.sent, (size_t)ctx->pop.cap, &ctx->strip_allocs);
  DM(ctx, &S.births, GNX_STRIP_MAX_WORLD, &ctx->strip_allocs);
  DM(ctx, &S.pairs, GNX_STRIP_MAX_WORLD, &ctx->strip_allocs);
  DM(ctx, &S.epoch, 4, &ctx->strip_allocs);
  CK(cudaMemsetAsync(S.epoch, 0, 16, ctx->stream));
  DM(ctx, &ctx->d_strip, 1, &ctx->strip_allocs);
  drop_graph(ctx);
  return strip_upload(ctx);
}

extern "C" int gnx_strip_endpoints(gnx_ctx* ctx, gnx_strip_endpoints_t* out) {
  ARG(ctx && out && ctx->d_strip, "strip decomposition is not enabled");
  USE_DEVICE(ctx);
  memset(out, 0, sizeof *out);
  out->base = ctx->strip_block;
  out->bytes = (int64_t)ctx->strip_block_bytes;
  for (int k = 0; k < STRIP_N_BUF; ++k) {
    out->buf_offset[k] = ctx->strip_buf_off[k];
    out->count_offset[k] = 64 * k;
  }
  out->sync_offset = ctx->strip_sync_off;
  out->counts_cap = ctx->strip_h.counts_cap;
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, ctx->strip_block));
  static_assert(sizeof(h) == sizeof(out->ipc_handle), "CUDA IPC handle is 64 bytes");
  memcpy(out->ipc_handle, &h, sizeof h);
  return GNX_OK;
}

extern "C" int gnx_strip_connect(gnx_ctx* ctx, int32_t peer_rank, const gnx_strip_endpoints_t* ep, int32_t same_process) {
  ARG(ctx && ep && ctx->d_strip, "strip decomposition is not enabled");
  USE_DEVICE(ctx);
  Strip& S = ctx->strip_h;
  ARG(peer_rank >= 0 && peer_rank < S.world && peer_rank != S.rank, "peer_rank");
  unsigned char* base = static_cast<unsigned char*>(ep->base);
  if (!same_process) {
    // another process on this node: map its block (NVLink peer memory) through CUDA IPC
    cudaIpcMemHandle_t h;
    memcpy(&h, ep->ipc_handle, sizeof h);
    void* mapped = nullptr;
    CK(cudaIpcOpenMemHandle(&mapped, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->strip_ipc_opened.push_back(mapped);
    base = static_cast<unsigned char*>(mapped);
  }
  for (int k = 0; k < STRIP_N_BUF; ++k) {
    S.peer[peer_rank].buf[k] = base + ep->buf_offset[k];
    S.peer[peer_rank].count[k] = reinterpret_cast<int32_t*>(base + ep->count_offset[k]);
  }
  ARG(ep->counts_cap == S.counts_cap, "the peer's density lattice differs from this rank's");
  if (!S.peer[peer_rank].sync) ctx->strip_connected += 1;
  S.peer[peer_rank].sync = base + ep->sync_offset;
  return strip_upload(ctx);
}

// Barrier (kind 0) or one of the small collectives of a time step (1: births all-gather after phase 3, or
// after phase 8 with Poisson births; 2: density-count sum after phase 5; 3: max(N) after phase 6; 4: pairs
// all-gather after phase 3 with Poisson births) over peer memory, enqueued on the rank's stream: see
// k_strip_barrier.  Every rank must make the same sequence of calls.
static int strip_barrier_launch(gnx_ctx* ctx, int kind);
extern "C" int gnx_strip_barrier(gnx_ctx* ctx, int32_t kind) {
  ARG(ctx && ctx->d_strip, "strip decomposition is not enabled");
  USE_DEVICE(ctx);
  ARG(kind >= 0 && kind <= 4, "kind");
  if (ctx->strip_connected != ctx->strip_h.world - 1) { g_last_error = "gnx_strip_barrier: not every peer is connected"; return GNX_ERR_STATE; }
  if (kind == 2 && (!ctx->have_density || ctx->strip_h.counts_cap < 2 * ctx->dens.npts)) {
    g_last_error = "gnx_strip_barrier: the density lattice was set after gnx_strip_enable";
    return GNX_ERR_STATE;
  }
  return strip_barrier_launch(ctx, kind);
}

extern "C" int gnx_strip_collective_ptrs(gnx_ctx* ctx, void** births, void** counts, int64_t* n_counts, void** nmax) {
  ARG(ctx && ctx->d_strip, "strip decomposition is not enabled");
  if (births) *births = ctx->strip_h.births;
  if (counts) *counts = ctx->dens.counts;
  if (n_counts) *n_counts = 2 * (int64_t)ctx->dens.npts;
  if (nmax) *nmax = &ctx->d_c->nmax_bits;
  return GNX_OK;
}

extern "C" int gnx_strip_pairs_ptr(gnx_ctx* ctx, void** pairs) {
  ARG(ctx && pairs && ctx->d_strip, "strip decomposition is not enabled");
  *pairs = ctx->strip_h.pairs;
  return GNX_OK;
}

static int strip_send(gnx_ctx* ctx, int which) {
  PROF(ctx, "k_strip_send");
  k_strip_send<<<grid_for(ctx, 2), 256, 0, ctx->stream>>>(ctx->pop, ctx->d_c, ctx->d_strip, which, ctx->burn ? 0 : 1);
  LAUNCHED(ctx);
  k_strip_list_reset<<<1, 1, 0, ctx->stream>>>(ctx->d_strip);
  LAUNCHED(ctx);
  return GNX_OK;
}
static int strip_recv(gnx_ctx* ctx, int which, int mode) {
  PROF(ctx, "k_strip_recv");
  k_strip_recv<<<grid_for(ctx, 2), 256, 0, ctx->stream>>>(ctx->pop, ctx->land, ctx->work, ctx->d_c, ctx->d_strip, which,
                                                        mode, ctx->burn ? 0 : 1);
  LAUNCHED(ctx);
  k_strip_recv_finish<<<1, 1, 0, ctx->stream>>>(ctx->d_c, ctx->d_strip, which, mode, ctx->burn ? 0 : 1);
  LAUNCHED(ctx);
  return GNX_OK;
}

// One time step in eight phases; between two phases EVERY rank must have finished the earlier
// one (the caller enqueues a stream-ordered collective -- or, with all ranks in one process,
// runs the phase on every context first):
//   0 move, list and send the leavers                          | barrier
//   1 receive migrants; list and send the halo                 | barrier
//   2 receive ghosts; re-grid; mate search; send edge choices  | barrier
//   3 receive choices; pair list; publish the births           | all-gather of `births`
//   4 id base; offspring, mutation; route and send dispersed newborns | barrier
//   5 receive newborns; density counts                         | all-reduce (sum) of `counts`
//   6 N and d rasters over the strip's rows (d of the cells that need max(N) deferred) | all-reduce (max) of `nmax`
//   7 deferred d cells; death probabilities and mortality draw; end of step
// With Poisson births (n_births_fixed = 0) the births of a rank depend on the pairs of the lower ranks, so
// phase 3 ends after the pair list and publishes the pairs, and a ninth phase follows the pairs all-gather:
//   3 receive choices; pair list; publish the pairs            | all-gather of `pairs`
//   8 Poisson births keyed by the species-wide pair positions; publish the births | all-gather of `births`
// and then phases 4 to 7 as above.
static int strip_phase_launch(gnx_ctx* ctx, int phase) {
  cudaStream_t s = ctx->stream;
  int r;
  switch (phase) {
    case 0:
      if ((r = move_key(ctx, 0, ctx->cfg.move ? 1 : 0, 1))) return r;
      return strip_send(ctx, STRIP_BUF_MIGRANTS);
    case 1:
      if ((r = strip_recv(ctx, STRIP_BUF_MIGRANTS, 0))) return r;
      PROF(ctx, "k_strip_halo_list");
      k_strip_halo_list<<<grid_for(ctx, 4), 256, 0, s>>>(ctx->work, ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      return strip_send(ctx, STRIP_BUF_HALO);
    case 2:
      if ((r = strip_recv(ctx, STRIP_BUF_HALO, 0))) return r;
      if ((r = finish_regrid(ctx, 1))) return r;
      if ((r = find_mates(ctx))) return r;
      PROF(ctx, "k_strip_choice_send");
      k_strip_choice_send<<<grid_for(ctx, 4), 256, 0, s>>>(ctx->pop, ctx->work, ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      return GNX_OK;
    case 3:
      PROF(ctx, "k_strip_choice_recv");
      k_strip_choice_recv<<<grid_for(ctx, 2), 256, 0, s>>>(ctx->pop, ctx->land, ctx->work, ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      k_strip_choice_finish<<<1, 1, 0, s>>>(ctx->d_strip);
      LAUNCHED(ctx);
      if ((r = scan_pairs(ctx))) return r;
      if (!ctx->cfg.n_births_fixed) {
        k_strip_publish_pairs<<<1, 1, 0, s>>>(ctx->d_c, ctx->d_strip);
        LAUNCHED(ctx);
        return GNX_OK;
      }
      k_strip_publish_births<<<1, 1, 0, s>>>(ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      return GNX_OK;
    case 8:
      ARG(!ctx->cfg.n_births_fixed, "phase 8 (Poisson births) with n_births_fixed");
      if ((r = draw_births(ctx))) return r;
      k_strip_publish_births<<<1, 1, 0, s>>>(ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      return GNX_OK;
    case 4:
      k_strip_id_base<<<1, 1, 0, s>>>(ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      if ((r = gnx_make_offspring(ctx))) return r;
      PROF(ctx, "k_strip_newborn_route");
      k_strip_newborn_route<<<grid_for(ctx, 4), 256, 0, s>>>(ctx->pop, ctx->land, ctx->d_c, ctx->d_strip);
      LAUNCHED(ctx);
      return strip_send(ctx, STRIP_BUF_NEWBORNS);
    case 5:
      if ((r = strip_recv(ctx, STRIP_BUF_NEWBORNS, 1))) return r;
      return gnx_density_counts(ctx);
    case 6:
      return density_eval_rasters(ctx);
    case 7:
      if ((r = density_eval_deferred(ctx))) return r;
      if ((r = death_prob(ctx, 1))) return r;
      k_strip_end_step<<<1, 1, 0, s>>>(ctx->d_c);
      LAUNCHED(ctx);
      return GNX_OK;
    default:
      ARG(false, "phase must be 0..8");
  }
  return GNX_OK;
}

static int strip_barrier_launch(gnx_ctx* ctx, int kind) {
  PROF(ctx, "k_strip_barrier");
  k_strip_barrier<<<1, 256, 0, ctx->stream>>>(ctx->d_strip, kind, ctx->dens.counts, 2 * ctx->dens.npts,
                                              reinterpret_cast<unsigned long long*>(&ctx->d_c->nmax_bits));
  LAUNCHED(ctx);
  return GNX_OK;
}

// The phases of one strip time step in order and the gnx_strip_barrier kind after each (-1: the step ends);
// gnx_strip_phase_order hands the same table to callers that sequence the phases themselves.
static void strip_step_plan(bool fixed, const int** phase, const int** sync_after, int* n) {
  static const int fixed_phase[8] = {0, 1, 2, 3, 4, 5, 6, 7}, fixed_sync[8] = {0, 0, 0, 1, 0, 2, 3, -1};
  static const int poisson_phase[9] = {0, 1, 2, 3, 8, 4, 5, 6, 7}, poisson_sync[9] = {0, 0, 0, 4, 1, 0, 2, 3, -1};
  *phase = fixed ? fixed_phase : poisson_phase;
  *sync_after = fixed ? fixed_sync : poisson_sync;
  *n = fixed ? 8 : 9;
}

extern "C" int gnx_strip_phase_order(int32_t n_births_fixed, int32_t* phases, int32_t* sync_after, int32_t* n) {
  ARG(phases && sync_after && n, "null");
  const int *ph, *sy;
  int k;
  strip_step_plan(n_births_fixed != 0, &ph, &sy, &k);
  for (int i = 0; i < k; ++i) { phases[i] = ph[i]; sync_after[i] = sy[i]; }
  *n = k;
  return GNX_OK;
}

// the whole time step of one strip: phase, then the barrier / collective that follows it (gnx_step captures
// this into one CUDA graph; the spin barriers inside it order the ranks' graphs against each other).  The
// sequence is fixed when the step is captured: a change of n_births_fixed changes prm, hence the step key.
static int strip_whole_step(gnx_ctx* ctx) {
  const int *phase, *sync_after;
  int n;
  strip_step_plan(ctx->cfg.n_births_fixed != 0, &phase, &sync_after, &n);
  for (int k = 0; k < n; ++k) {
    int r = strip_phase_launch(ctx, phase[k]);
    if (r != GNX_OK) return r;
    if (sync_after[k] >= 0 && (r = strip_barrier_launch(ctx, sync_after[k])) != GNX_OK) return r;
  }
  return GNX_OK;
}

extern "C" int gnx_strip_phase(gnx_ctx* ctx, int32_t phase) {
  ARG(ctx && ctx->d_strip, "strip decomposition is not enabled");
  USE_DEVICE(ctx);
  ARG(!ctx->prm.ordered, "injected per-individual draws are not supported under strip decomposition");
  if (phase == 0 && ctx->records_pending + 1 > ctx->work.max_records) {
    g_last_error = "step-record buffer would overflow: call gnx_read_step_records first";
    return GNX_ERR_STATE;
  }
  int r = strip_phase_launch(ctx, phase);
  if (r != GNX_OK) return r;
  if (phase == 7) {
    ctx->records_pending += 1;
    ctx->steps_done += 1;
    ctx->pending = true;
    ctx->order_valid = false;
  }
  return GNX_OK;
}

// sticky overflow flags of the exchange (list or a receive buffer too small); synchronises
extern "C" int gnx_strip_check(gnx_ctx* ctx) {
  ARG(ctx && ctx->d_strip, "strip decomposition is not enabled");
  USE_DEVICE(ctx);
  int32_t e = 0;
  CK(cudaMemcpyAsync(&e, ctx->strip_h.err, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (e & 4) {
    g_last_error = "strip barrier: a peer rank never arrived (gnx_strip_barrier timed out)";
    return GNX_ERR_STATE;
  }
  if (e) {
    g_last_error = (e & 2) ? "strip exchange: a receive buffer overflowed (raise migrant_capacity / halo_capacity)"
                           : "strip exchange: the send list overflowed";
    return GNX_ERR_CAPACITY;
  }
  return gnx_sync(ctx);
}

extern "C" int gnx_sync(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  return check_device_err(h);
}

extern "C" int gnx_walk_host(gnx_ctx* ctx, gnx_population_t* pop, int32_t n_steps) {
  int r = gnx_upload_population(ctx, pop);
  if (r != GNX_OK) return r;
  r = gnx_step(ctx, n_steps);
  if (r != GNX_OK) return r;
  return gnx_download_population(ctx, pop);
}

// The same call split in two so that the host can keep several replicate populations in flight
// (each on its own context = its own stream): _begin only ENQUEUES the copies in and the steps,
// _end waits for them and copies the population out.  While one context's result travels to the
// host, the next one's input travels to the device (PCIe is full duplex) and a third one steps.
extern "C" int gnx_walk_host_begin(gnx_ctx* ctx, const gnx_population_t* pop, int32_t n_steps) {
  int r = upload_population(ctx, pop, false);
  if (r != GNX_OK) return r;
  return gnx_step(ctx, n_steps);
}

extern "C" int gnx_walk_host_end(gnx_ctx* ctx, gnx_population_t* pop) {
  return gnx_download_population(ctx, pop);
}

extern "C" int gnx_read_step_records(gnx_ctx* ctx, gnx_step_record_t* out, int32_t max_records, int32_t* n_out) {
  ARG(ctx && n_out, "null");
  USE_DEVICE(ctx);
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  int n = std::min(h.n_rec, ctx->work.max_records);
  n = std::min(n, max_records);
  if (n > 0 && out)
    CK(cudaMemcpyAsync(out, ctx->work.records, (size_t)n * sizeof(gnx_step_record_t), cudaMemcpyDeviceToHost,
                       ctx->stream));
  h.n_rec = 0;
  ctx->records_pending = 0;
  CK(cudaMemcpyAsync(&ctx->d_c->n_rec, &h.n_rec, sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *n_out = n;
  return check_device_err(h);
}

// Per-individual fields are returned in SPECIES order (ascending id): the entries are ranked by
// id (radix sort) and the field is gathered into a staging area -- the idle half of the state
// buffers for the state fields, work.scratch for work arrays; entry-valued arrays (mate, pairs)
// are translated to ordinals.  The pointer stays valid until the next call on the ctx.
extern "C" int gnx_device_ptr(gnx_ctx* ctx, int32_t field, void** dev_ptr, int64_t* nbytes) {
  ARG(ctx && dev_ptr && nbytes, "null");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  Counters h;
  if ((r = read_counters(ctx, &h)) != GNX_OK) return r;
  const int ne = std::max(h.n, h.n_pre);
  const size_t n = (size_t)ne, cap = (size_t)ctx->pop.cap;
  const size_t plane = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  Pop& P = ctx->pop;
  Work& W = ctx->work;
  Dens& D = ctx->dens;
  cudaStream_t s = ctx->stream;
  const int o = h.cur ^ 1;
  void* p = nullptr;
  size_t b = 0;
  const bool state_field = field == GNX_F_X || field == GNX_F_Y || field == GNX_F_AGE || field == GNX_F_SEX ||
                           field == GNX_F_IDX || field == GNX_F_Z || field == GNX_F_FIT || field == GNX_F_GSLOT ||
                           field == GNX_F_GENOMES;
  const bool work_field = field == GNX_F_N_NBRS || field == GNX_F_MATE || field == GNX_F_PAIRS || field == GNX_F_PERM ||
                          field == GNX_F_DEATH_P || field == GNX_F_ALIVE || field == GNX_F_E ||
                          field == GNX_F_NODE0 || field == GNX_F_NODE1;
  if (state_field || work_field) {
    if ((r = build_order(ctx, h, false)) != GNX_OK) return r;
  }
  if (state_field) {
    PROF(ctx, "k_species_gather");
    k_species_gather<<<grid_for(ctx, 8), 256, 0, s>>>(P, W, ctx->d_c, ne, nullptr);
    LAUNCHED(ctx);
  }
  const int g4 = grid_for(ctx, 4);
  switch (field) {
    case GNX_F_X: p = reinterpret_cast<double*>(P.xy[o]); b = n * 8; break;
    case GNX_F_Y: p = reinterpret_cast<double*>(P.xy[o]) + cap; b = n * 8; break;
    case GNX_F_AGE: p = P.age[o]; b = n * 4; break;
    case GNX_F_SEX: p = P.sex[o]; b = n; break;
    case GNX_F_IDX: p = P.idx[o]; b = n * 8; break;
    case GNX_F_Z: p = P.z[o]; b = cap * std::max(1, ctx->cfg.n_traits) * 8; break;
    case GNX_F_FIT: p = P.fit[o]; b = n * 8; break;
    case GNX_F_GSLOT: p = P.gslot[o]; b = n * 4; break;
    case GNX_F_GENOMES:
      PROF(ctx, "k_gather_genomes");
      k_gather_genomes<<<grid_for(ctx, 8), 256, 0, s>>>(P, P.gslot[o], ctx->d_stage_genomes, h.n);
      LAUNCHED(ctx);
      p = ctx->d_stage_genomes;
      b = (size_t)h.n * 2 * ctx->Wq * sizeof(uint4);
      break;
    case GNX_F_NODE0:
    case GNX_F_NODE1:
      if (!ctx->tsk.enabled) { g_last_error = "tskit recording not enabled"; return GNX_ERR_STATE; }
      k_gather_by_inv<int32_t><<<g4, 256, 0, s>>>(P.node[field == GNX_F_NODE1 ? 1 : 0][h.cur], (int32_t*)W.scratch, W.inv, ne);
      p = W.scratch; b = n * 4; break;
    case GNX_F_N_NBRS:
      k_gather_by_inv<int32_t><<<g4, 256, 0, s>>>(W.n_nbrs, (int32_t*)W.scratch, W.inv, ne);
      p = W.scratch; b = n * 4; break;
    case GNX_F_MATE:
      k_gather_mate<<<g4, 256, 0, s>>>(W.mate, (int32_t*)W.scratch, W.inv, P.ord[h.cur], ne,
                                       ctx->cfg.mating_radius <= 0 ? 1 : 0);
      p = W.scratch; b = n * 4; break;
    case GNX_F_PAIRS:
      k_translate_entries<<<g4, 256, 0, s>>>(W.pairs, (int32_t*)W.scratch, P.ord[h.cur], 2 * h.P);
      p = W.scratch; b = (size_t)h.P * 8; break;
    case GNX_F_PERM: p = P.ord[h.cur]; b = n * 4; break;     /* ordinal of the individual at each grid position */
    case GNX_F_DEATH_P:
      k_gather_by_inv<double><<<g4, 256, 0, s>>>(W.death_p, (double*)W.scratch, W.inv, ne);
      p = W.scratch; b = n * 8; break;
    case GNX_F_ALIVE:
      k_gather_by_inv<uint8_t><<<g4, 256, 0, s>>>(W.alive, (uint8_t*)W.scratch, W.inv, ne);
      p = W.scratch; b = n; break;
    case GNX_F_E:
      if ((r = sample_env_ordered(ctx, ne)) != GNX_OK) return r;
      p = W.e_out; b = n * ctx->cfg.n_layers * 8; break;
    case GNX_F_NB: p = W.nb; b = (size_t)h.P * 4; break;
    case GNX_F_CELL_START: p = W.cell_start; b = ((size_t)ctx->ncell + 1) * 4; break;
    case GNX_F_COUNTS_N: p = D.counts; b = (size_t)D.npts * 4; break;
    case GNX_F_COUNTS_P: p = D.counts + D.npts; b = (size_t)D.npts * 4; break;
    case GNX_F_VALS_N: p = D.vals; b = (size_t)D.npts * 8; break;
    case GNX_F_VALS_P: p = D.vals + D.npts; b = (size_t)D.npts * 8; break;
    case GNX_F_GRAD_N: p = D.grad; b = (size_t)D.npts * 16; break;
    case GNX_F_GRAD_P: p = D.grad + 2 * (size_t)D.npts; b = (size_t)D.npts * 16; break;
    case GNX_F_N_RAST: p = W.N_rast; b = plane * 8; break;
    case GNX_F_NPAIRS_RAST: p = W.NP_rast; b = plane * 8; break;
    case GNX_F_D_RAST: p = W.d_rast; b = plane * 8; break;
    case GNX_F_K_RAST: p = ctx->d_K; b = plane * 8; break;
    case GNX_F_DISP_TRIES: p = W.disp_tries; b = (size_t)h.B * 4; break;
    case GNX_F_COUNTERS: p = ctx->d_c; b = sizeof(Counters); break;
    case GNX_F_VM_TAB_MOVE:
    case GNX_F_VM_TAB_DISP: {
      const int k = field == GNX_F_VM_TAB_DISP ? 1 : 0;
      if (!ctx->prm.vm_tab[k]) { g_last_error = "that site's conductance surface is not on the fly"; return GNX_ERR_STATE; }
      p = const_cast<float*>(ctx->prm.vm_tab[k]); b = (size_t)VM_TAB_LEN * 4; break;
    }
    default: g_last_error = "unknown field"; return GNX_ERR_ARG;
  }
  CK(cudaGetLastError());
  *dev_ptr = p;
  *nbytes = (int64_t)b;
  return GNX_OK;
}

extern "C" int gnx_read_field(gnx_ctx* ctx, int32_t field, void* host_out, int64_t nbytes) {
  ARG(ctx && host_out, "null");
  USE_DEVICE(ctx);
  void* p;
  int64_t avail;
  int r = gnx_device_ptr(ctx, field, &p, &avail);
  if (r != GNX_OK) return r;
  const int64_t b = std::min(avail, nbytes);
  if (b > 0) CK(cudaMemcpyAsync(host_out, p, (size_t)b, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

extern "C" void* gnx_stream(gnx_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" int64_t gnx_launch_count(gnx_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" int64_t gnx_graph_launch_count(gnx_ctx* ctx) { return ctx ? ctx->graph_launches : 0; }
extern "C" int64_t gnx_graph_capture_count(gnx_ctx* ctx) { return ctx ? ctx->graph_captures : 0; }


// ---- per-kernel timing ------------------------------------------------------------------
extern "C" int gnx_profile(gnx_ctx* ctx, int32_t enable) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  for (auto& sp : ctx->spans) { cudaEventDestroy(sp.e0); cudaEventDestroy(sp.e1); }
  ctx->spans.clear();
  ctx->profiling = enable != 0;
  return GNX_OK;
}

// Writes "name\tlaunches\ttotal_ms\n" lines for every kernel launched since gnx_profile(ctx, 1).
extern "C" int gnx_profile_report(gnx_ctx* ctx, char* buf, int64_t buflen) {
  ARG(ctx && buf && buflen > 0, "null");
  USE_DEVICE(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  std::vector<std::string> names;
  std::vector<double> ms;
  std::vector<int64_t> cnt;
  for (auto& sp : ctx->spans) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, sp.e0, sp.e1) != cudaSuccess) continue;
    size_t k = 0;
    for (; k < names.size(); ++k) if (names[k] == sp.name) break;
    if (k == names.size()) { names.push_back(sp.name); ms.push_back(0); cnt.push_back(0); }
    ms[k] += t;
    cnt[k] += 1;
  }
  std::string out;
  char line[256];
  for (size_t k = 0; k < names.size(); ++k) {
    snprintf(line, sizeof line, "%s\t%lld\t%.6f\n", names[k].c_str(), (long long)cnt[k], ms[k]);
    out += line;
  }
  if ((int64_t)out.size() + 1 > buflen) { g_last_error = "profile buffer too small"; return GNX_ERR_ARG; }
  memcpy(buf, out.c_str(), out.size() + 1);
  return GNX_OK;
}


/* keep per-individual intermediates (n_nbrs, death_p, disp_tries, n_pairs raster) for parity tests */
extern "C" int gnx_set_debug(gnx_ctx* ctx, int32_t on) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  ctx->prm.store_debug = on ? 1 : 0;
  return GNX_OK;
}


// ---- on-device stats (sim/stats.py:399-435) -----------------------------------------------
// host_c1[L]: number of 1-alleles per locus; host_het[L]: number of heterozygous individuals
// per locus; *fit_sum: sum of the fitness values of the last completed step; *n: population
// size.  (het = host_het / n, freq_1 = host_c1 / 2n, maf = min(freq_1, 1 - freq_1).)
extern "C" int gnx_stats_genotypes(gnx_ctx* ctx, uint64_t* host_c1, uint64_t* host_het, double* fit_sum, int64_t* n) {
  return gnx_stats_genotypes_region(ctx, -1e300, 1e300, -1e300, 1e300, host_c1, host_het, fit_sum, n);
}

extern "C" int gnx_stats_genotypes_region(gnx_ctx* ctx, double x_min, double x_max, double y_min, double y_max,
                                          uint64_t* host_c1, uint64_t* host_het, double* fit_sum, int64_t* n) {
  ARG(ctx && host_c1 && host_het && fit_sum && n, "null");
  USE_DEVICE(ctx);
  if (ctx->burn || ctx->cfg.L == 0) { g_last_error = "no genomes on the device"; return GNX_ERR_STATE; }
  {
    int rm = materialise(ctx);
    if (rm != GNX_OK) return rm;
  }
  const int nbits = ctx->Wwords * 32;
  unsigned long long* d = nullptr;
  CK(cudaMalloc(&d, (size_t)(2 * nbits + 2) * 8));
  CK(cudaMemsetAsync(d, 0, (size_t)(2 * nbits + 2) * 8, ctx->stream));
  const size_t smem = (size_t)2 * nbits * 4;
  if (smem > 48 * 1024)
    CK(cudaFuncSetAttribute(k_stats_genotypes, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  PROF(ctx, "k_stats_genotypes");
  k_stats_genotypes<<<grid_for(ctx, 2), 256, smem, ctx->stream>>>(ctx->pop, ctx->d_c, d, d + nbits,
                                                                  reinterpret_cast<double*>(d + 2 * nbits),
                                                                  x_min, x_max, y_min, y_max, d + 2 * nbits + 1);
  LAUNCHED(ctx);
  std::vector<unsigned long long> h((size_t)2 * nbits + 2);
  CK(cudaMemcpyAsync(h.data(), d, h.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  Counters hc;
  int r = read_counters(ctx, &hc);
  cudaFree(d);
  if (r != GNX_OK) return r;
  if (ctx->cols) {                                    // column j counts locus col_locus[j]; no column: zero
    std::vector<int32_t> col_locus;
    if ((r = read_cols(ctx, &col_locus)) != GNX_OK) return r;
    memset(host_c1, 0, (size_t)ctx->cfg.L * 8);
    memset(host_het, 0, (size_t)ctx->cfg.L * 8);
    for (size_t j = 0; j < col_locus.size(); ++j) { host_c1[col_locus[j]] = h[j]; host_het[col_locus[j]] = h[nbits + j]; }
  } else {
    for (int l = 0; l < ctx->cfg.L; ++l) { host_c1[l] = h[l]; host_het[l] = h[nbits + l]; }
  }
  memcpy(fit_sum, &h[2 * nbits], 8);
  *n = (int64_t)h[2 * nbits + 1];
  return check_device_err(hc);
}


// Linkage disequilibrium counts (sim/stats.py:359-392): host_n11[Lp * Lp], Lp = 32 * ceil(L / 32),
// row-major; entry (i, j), j's word >= i's word, = chromosomes carrying the 1-allele at both loci
// (the diagonal = 1-allele counts); the other word-triangle stays zero.  *n = population size.
extern "C" int gnx_stats_ld(gnx_ctx* ctx, uint64_t* host_n11, int64_t* n) {
  ARG(ctx && host_n11 && n, "null");
  USE_DEVICE(ctx);
  if (ctx->burn || ctx->cfg.L == 0) { g_last_error = "no genomes on the device"; return GNX_ERR_STATE; }
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  std::vector<int32_t> col_locus;
  if (ctx->cols && (r = read_cols(ctx, &col_locus)) != GNX_OK) return r;
  // the column layout counts over its columns and scatters the pairs to their loci below
  const int Wu = ctx->cols ? std::max<int>(1, ((int)col_locus.size() + 31) / 32) : (ctx->cfg.L + 31) / 32, Lp = 32 * Wu;
  const int ntile = Wu * (Wu + 1) / 2;
  // enough (tile, haplotype range) items to fill the machine a few times over
  const int nsplit = std::max(1, std::min(4096, (ctx->num_sms * 64 + ntile - 1) / ntile));
  unsigned long long* d = nullptr;
  CK(cudaMalloc(&d, (size_t)Lp * Lp * 8));
  CK(cudaMemsetAsync(d, 0, (size_t)Lp * Lp * 8, ctx->stream));
  PROF(ctx, "k_stats_ld");
  k_stats_ld<<<grid_for(ctx, 8), 256, 0, ctx->stream>>>(ctx->pop, ctx->d_c, d, Wu, Lp, nsplit);
  LAUNCHED(ctx);
  std::vector<unsigned long long> hcols(ctx->cols ? (size_t)Lp * Lp : 0);
  cudaError_t e = cudaMemcpyAsync(ctx->cols ? hcols.data() : (unsigned long long*)host_n11, d, (size_t)Lp * Lp * 8,
                                  cudaMemcpyDeviceToHost, ctx->stream);
  Counters hc;
  r = read_counters(ctx, &hc);
  cudaFree(d);
  if (e != cudaSuccess) { g_last_error = cudaGetErrorString(e); return GNX_ERR_CUDA; }
  if (r != GNX_OK) return r;
  if (ctx->cols) {
    // the by-locus answer: entry (i, j) of loci i, j with j / 32 >= i / 32, from the column pair (a, b) -- the
    // device filled the column word-triangle b / 32 >= a / 32 of the symmetric counts
    const size_t LpL = (size_t)32 * ((ctx->cfg.L + 31) / 32);
    memset(host_n11, 0, LpL * LpL * 8);
    const int nc = (int)col_locus.size();
    for (int a = 0; a < nc; ++a)
      for (int b = 0; b < nc; ++b) {
        const int i = col_locus[a], j = col_locus[b];
        if (j / 32 < i / 32) continue;
        host_n11[(size_t)i * LpL + j] = b / 32 >= a / 32 ? hcols[(size_t)a * Lp + b] : hcols[(size_t)b * Lp + a];
      }
  }
  *n = hc.n;
  return check_device_err(hc);
}

// Burn-in spatial statistic (sim/burnin.py:41-58): counts the individuals of every landscape cell
// and returns the sum and the sum of squares of the change of the counts since the previous call
// (the first call compares with all-zero counts, as SpatialTester.__init__ does).
extern "C" int gnx_burnin_cell_stats(gnx_ctx* ctx, int64_t* sum_diff, int64_t* sum_sq_diff) {
  ARG(ctx && sum_diff && sum_sq_diff, "null");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  const size_t ncell = (size_t)ctx->cfg.dim_x * ctx->cfg.dim_y;
  cudaStream_t s = ctx->stream;
  if (!ctx->burnin_counts) {
    CK(cudaMalloc((void**)&ctx->burnin_counts, (2 * ncell + 4) * sizeof(int32_t)));
    CK(cudaMemsetAsync(ctx->burnin_counts, 0, (2 * ncell + 4) * sizeof(int32_t), s));
  }
  int32_t* cur = ctx->burnin_counts;
  int32_t* prev = cur + ncell;
  long long* sums = reinterpret_cast<long long*>(prev + ncell);      // 16 bytes behind the two rasters
  CK(cudaMemsetAsync(cur, 0, ncell * sizeof(int32_t), s));
  CK(cudaMemsetAsync(sums, 0, 16, s));
  PROF(ctx, "k_burnin_count");
  k_burnin_count<<<grid_for(ctx, 8), 256, 0, s>>>(ctx->pop, ctx->land, ctx->d_c, cur);
  LAUNCHED(ctx);
  PROF(ctx, "k_burnin_diff");
  k_burnin_diff<<<grid_for(ctx, 8), 256, 0, s>>>(cur, prev, ncell, sums);
  LAUNCHED(ctx);
  long long h[2] = {0, 0};
  CK(cudaMemcpyAsync(h, sums, 16, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  *sum_diff = h[0];
  *sum_sq_diff = h[1];
  return GNX_OK;
}

// The statistic under strip decomposition: the rank's individuals counted into its band of landscape rows
// [ly0, ly1) only (the host folds the row shared with the lower neighbour in between the two calls).
// Layout of ctx->strip_burnin: cur [rows][X] | prev [rows][X] | two int64 sums | the out-of-band count.
extern "C" int gnx_strip_burnin_count(gnx_ctx* ctx, int32_t* ly0, int32_t* ly1, void** first_row, void** last_row) {
  ARG(ctx && ly0 && ly1 && first_row && last_row, "null");
  USE_DEVICE(ctx);
  if (!ctx->d_strip) { g_last_error = "gnx_strip_burnin_count: strip decomposition is not enabled"; return GNX_ERR_STATE; }
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  const Strip& S = ctx->strip_h;
  const int X = ctx->cfg.dim_x;
  const size_t nband = (size_t)(S.ly1 - S.ly0) * X;
  cudaStream_t s = ctx->stream;
  if (!ctx->strip_burnin) {
    CK(cudaMalloc((void**)&ctx->strip_burnin, (2 * nband + 6) * sizeof(int32_t)));
    CK(cudaMemsetAsync(ctx->strip_burnin, 0, (2 * nband + 6) * sizeof(int32_t), s));
  }
  int32_t* cur = ctx->strip_burnin;
  int32_t* outside = cur + 2 * nband + 4;
  CK(cudaMemsetAsync(cur, 0, nband * sizeof(int32_t), s));
  CK(cudaMemsetAsync(outside, 0, sizeof(int32_t), s));
  PROF(ctx, "k_strip_burnin_count");
  k_strip_burnin_count<<<grid_for(ctx, 8), 256, 0, s>>>(ctx->pop, ctx->land, ctx->d_c, S.ly0, S.ly1, cur, outside);
  LAUNCHED(ctx);
  int32_t h_out = 0;
  CK(cudaMemcpyAsync(&h_out, outside, sizeof h_out, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (h_out) {
    g_last_error = "gnx_strip_burnin_count: an individual lies outside the strip's landscape rows";
    return GNX_ERR_STATE;
  }
  *ly0 = S.ly0;
  *ly1 = S.ly1;
  *first_row = cur;
  *last_row = cur + (size_t)(S.ly1 - S.ly0 - 1) * X;
  return GNX_OK;
}

extern "C" int gnx_strip_burnin_diff(gnx_ctx* ctx, int32_t skip_last_row, int64_t* sum_diff, int64_t* sum_sq_diff) {
  ARG(ctx && sum_diff && sum_sq_diff, "null");
  USE_DEVICE(ctx);
  if (!ctx->d_strip || !ctx->strip_burnin) {
    g_last_error = "gnx_strip_burnin_diff: no band counts (gnx_strip_burnin_count first)";
    return GNX_ERR_STATE;
  }
  const Strip& S = ctx->strip_h;
  const int X = ctx->cfg.dim_x;
  const size_t nband = (size_t)(S.ly1 - S.ly0) * X;
  const size_t ncell = nband - (skip_last_row ? (size_t)X : 0);
  int32_t* cur = ctx->strip_burnin;
  int32_t* prev = cur + nband;
  long long* sums = reinterpret_cast<long long*>(prev + nband);
  cudaStream_t s = ctx->stream;
  CK(cudaMemsetAsync(sums, 0, 16, s));
  PROF(ctx, "k_burnin_diff");
  k_burnin_diff<<<grid_for(ctx, 8), 256, 0, s>>>(cur, prev, ncell, sums);
  LAUNCHED(ctx);
  long long h[2] = {0, 0};
  CK(cudaMemcpyAsync(h, sums, 16, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  *sum_diff = h[0];
  *sum_sq_diff = h[1];
  return GNX_OK;
}

// ---- tskit record buffering (species.py:692-736, genome.py:234-281; SURVEY.md 8f rank 1) --
// Node / edge / individual rows of every birth are written to device buffers by the step
// kernels and handed to the host (tskit's TableCollection.append_columns) at the simplify
// interval (model.py:756-768).
// node ids 2k, 2k+1 by species-order ordinal k: the entries are ranked by id first
static int tskit_renumber(gnx_ctx* ctx, int reset_t0) {
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  Counters h;
  if ((r = read_counters(ctx, &h)) != GNX_OK) return r;
  if ((r = build_order(ctx, h, false)) != GNX_OK) return r;
  PROF(ctx, "k_tskit_renumber");
  k_tskit_renumber<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(ctx->pop, ctx->d_c, reset_t0);
  LAUNCHED(ctx);
  return GNX_OK;
}

extern "C" int gnx_tskit_enable(gnx_ctx* ctx, int64_t edge_capacity, int64_t birth_capacity) {
  ARG(ctx && edge_capacity > 0 && birth_capacity > 0, "capacities");
  USE_DEVICE(ctx);
  ARG(!ctx->d_strip, "tskit recording is not supported under strip decomposition");
  ARG(edge_capacity < (1ll << 31) && birth_capacity < (1ll << 31), "capacities");
  if (!ctx->have_paths) { g_last_error = "recombination paths not set"; return GNX_ERR_STATE; }
  CK(cudaStreamSynchronize(ctx->stream));
  free_bucket(ctx->tsk_allocs);
  Tsk& T = ctx->tsk;
  memset(&T, 0, sizeof T);
  // breakpoints of every cached path: loci where the path switches homologue (genome.py:194-199)
  const int L = ctx->cfg.L, W = 4 * ctx->WqL, np = ctx->cfg.n_recomb_paths;   // paths as simulated: by locus
  std::vector<int32_t> ptr(np + 1, 0), pos;
  for (int k = 0; k < np; ++k) {
    const uint32_t* row = &ctx->host_paths[(size_t)k * W];
    int prev = 0;                                   // rate[0] == 0: every path starts on homologue 0
    for (int l = 0; l < L; ++l) {
      const int b = (row[l >> 5] >> (l & 31)) & 1;
      if (b != prev) pos.push_back(l);
      prev = b;
    }
    ptr[k + 1] = (int32_t)pos.size();
  }
  int r;
  if ((r = upload_vec(ctx, ptr, &T.bp_ptr, ctx->tsk_allocs)) != GNX_OK) return r;
  if ((r = upload_vec(ctx, pos, &T.bp_pos, ctx->tsk_allocs)) != GNX_OK) return r;
  ctx->tsk_max_bp = 0;
  for (int k = 0; k < np; ++k) ctx->tsk_max_bp = std::max(ctx->tsk_max_bp, ptr[k + 1] - ptr[k]);
  T.L = (double)L;
  T.edge_cap = (int32_t)edge_capacity;
  T.born_cap = (int32_t)birth_capacity;
  DM(ctx, &T.e_left, edge_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.e_right, edge_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.e_parent, edge_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.e_child, edge_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.b_idx, birth_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.b_x, birth_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.b_y, birth_capacity, &ctx->tsk_allocs);
  DM(ctx, &T.b_z, birth_capacity * std::max(1, ctx->cfg.n_traits), &ctx->tsk_allocs);
  DM(ctx, &T.b_time, birth_capacity, &ctx->tsk_allocs);
  const int64_t cap = ctx->cfg.capacity;
  for (int h = 0; h < 2; ++h)
    for (int b = 0; b < 2; ++b) DM(ctx, &ctx->pop.node[h][b], cap, &ctx->tsk_allocs);
  T.enabled = 1;
  // node ids 2k, 2k+1 in species order (species.py:1148-1152); time origin = now
  if ((r = tskit_renumber(ctx, 1)) != GNX_OK) return r;
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

// after TableCollection.simplify(): nodes become 2k, 2k+1 in species order and the
// individuals table holds exactly the live individuals (species.py:1140-1164)
extern "C" int gnx_tskit_renumber(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  USE_DEVICE(ctx);
  if (!ctx->tsk.enabled) { g_last_error = "tskit recording not enabled"; return GNX_ERR_STATE; }
  return tskit_renumber(ctx, 0);
}

// explicit node ids (e.g. the msprime-seeded start, species.py:1060-1063), species order
extern "C" int gnx_tskit_set_nodes(gnx_ctx* ctx, const int32_t* host_node0, const int32_t* host_node1, int64_t n,
                                   int32_t next_node_id, int32_t next_individual_row) {
  ARG(ctx && host_node0 && host_node1, "null");
  if (!ctx->tsk.enabled) { g_last_error = "tskit recording not enabled"; return GNX_ERR_STATE; }
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  Counters h;
  if ((r = read_counters(ctx, &h)) != GNX_OK) return r;
  ARG(n == h.n, "n differs from the population size");
  if ((r = build_order(ctx, h, false)) != GNX_OK) return r;
  // host arrays are in species order: staged, then scattered to the entries through work.inv
  int32_t* st = reinterpret_cast<int32_t*>(ctx->work.scratch);
  CK(cudaMemcpyAsync(st, host_node0, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(st + n, host_node1, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  k_scatter_nodes<<<grid_for(ctx, 4), 256, 0, ctx->stream>>>(ctx->pop, ctx->work, ctx->d_c, st, st + n, (int)n);
  CK(cudaGetLastError());
  h.n_nodes = next_node_id;
  h.n_ind_rows = next_individual_row;
  CK(cudaMemcpyAsync(ctx->d_c, &h, sizeof h, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return GNX_OK;
}

// Copies the rows buffered since the last drain into host column arrays and empties the
// buffers.  Pass NULL arrays (with rows->n_* = 0) to query the counts first.
extern "C" int gnx_tskit_drain(gnx_ctx* ctx, gnx_tskit_rows_t* rows) {
  ARG(ctx && rows, "null");
  USE_DEVICE(ctx);
  if (!ctx->tsk.enabled) { g_last_error = "tskit recording not enabled"; return GNX_ERR_STATE; }
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  if ((r = check_device_err(h)) != GNX_OK) return r;
  const bool query = rows->edge_left == nullptr && rows->birth_idx == nullptr;
  if (!query) {
    ARG(rows->n_edges >= h.n_edges && rows->n_births >= h.n_born, "host buffers too small");
    Tsk& T = ctx->tsk;
    cudaStream_t s = ctx->stream;
    const size_t ne = (size_t)h.n_edges, nb = (size_t)h.n_born;
    CK(cudaMemcpyAsync(rows->edge_left, T.e_left, ne * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->edge_right, T.e_right, ne * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->edge_parent, T.e_parent, ne * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->edge_child, T.e_child, ne * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->birth_idx, T.b_idx, nb * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->birth_x, T.b_x, nb * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->birth_y, T.b_y, nb * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(rows->birth_time, T.b_time, nb * 8, cudaMemcpyDeviceToHost, s));
    for (int t = 0; t < ctx->cfg.n_traits; ++t)
      CK(cudaMemcpyAsync(rows->birth_z + (size_t)t * nb, T.b_z + (size_t)t * T.born_cap, nb * 8,
                         cudaMemcpyDeviceToHost, s));
    rows->first_node_id = h.n_nodes - 2 * h.n_born;
    rows->first_individual_row = h.n_ind_rows - h.n_born;
    const int32_t zero2[2] = {0, 0};
    CK(cudaMemcpyAsync(&ctx->d_c->n_edges, zero2, 8, cudaMemcpyHostToDevice, s));   // n_edges, n_born
    CK(cudaStreamSynchronize(s));
  }
  rows->n_edges = h.n_edges;
  rows->n_births = h.n_born;
  return GNX_OK;
}

// ---- device assignment of the starting genomes (gnx_genome_init.cuh) ---------------------------
// One histogram pass over the keys of every still-active locus; synchronises (the caller may sum the
// histograms of several strips before the next gnx_genome_init_pass).
static int gi_hist_pass(gnx_ctx* ctx) {
  const int L = ctx->cfg.L;
  cudaStream_t s = ctx->stream;
  CK(cudaMemsetAsync(ctx->d_gi_hist, 0, (size_t)L * GI_BINS * sizeof(int32_t), s));
  const int tiles = (L + GI_TILE - 1) / GI_TILE;
  const long long n = std::max<long long>(ctx->n_hint, 1);
  const int gx = (int)std::max<long long>(1, std::min<long long>((n + 2047) / 2048, (8ll * ctx->num_sms + tiles - 1) / tiles));
  PROF(ctx, "k_gi_hist");
  k_gi_hist<<<dim3(gx, tiles), 256, 0, s>>>(ctx->pop, ctx->d_c, ctx->d_gi_state, ctx->d_gi_lkey, ctx->d_gi_hist, L);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(s));
  return GNX_OK;
}

extern "C" int gnx_genome_init_begin(gnx_ctx* ctx, const gnx_genome_init_t* gi, void** dev_hist, int64_t* hist_len) {
  ARG(ctx && gi && dev_hist && hist_len, "null");
  const int L = ctx->cfg.L;
  ARG(L > 0, "the context carries no genomes (L = 0)");
  ARG(gi->n_loci == L, "n_loci differs from the L of the context");
  ARG(gi->host_n_carriers, "host_n_carriers is required");
  ARG(!(gi->tskit_rows && ctx->d_strip), "tskit rows are not supported under strip decomposition");
  ARG((L + GI_TILE - 1) / GI_TILE <= 65535, "L too large for the device genome assignment");
  USE_DEVICE(ctx);
  int r = materialise(ctx);
  if (r != GNX_OK) return r;
  Counters h;
  if ((r = read_counters(ctx, &h)) != GNX_OK) return r;
  if ((r = check_device_err(h)) != GNX_OK) return r;
  // a strip holds part of the species: its k_gi_select checks the counts against the summed histogram
  for (int l = 0; l < L; ++l)
    ARG(gi->host_n_carriers[l] >= 0 && (ctx->d_strip || gi->host_n_carriers[l] <= 2ll * h.n),
        "n_carriers must lie in [0, 2n]");
  ctx->gi_stage = 0;
  free_bucket(ctx->gi_allocs);
  ctx->d_gi_hist = nullptr;
  long long* d_nc = nullptr;
  uint8_t* d_sel = nullptr;
  DM(ctx, &ctx->d_gi_state, (size_t)L, &ctx->gi_allocs);
  DM(ctx, &ctx->d_gi_lkey, (size_t)L, &ctx->gi_allocs);
  DM(ctx, &ctx->d_gi_write, (size_t)L, &ctx->gi_allocs);
  DM(ctx, &ctx->d_gi_hist, (size_t)L * GI_BINS, &ctx->gi_allocs);
  DM(ctx, &ctx->d_gi_active, (size_t)2, &ctx->gi_allocs);
  DM(ctx, &d_nc, (size_t)L, &ctx->gi_allocs);
  DM(ctx, &d_sel, (size_t)L, &ctx->gi_allocs);
  ctx->gi_carriers.assign(gi->host_n_carriers, gi->host_n_carriers + L);
  ctx->gi_tskit = gi->tskit_rows != 0;
  // select: loci whose carriers are needed -- the written ones, and every locus for the tskit listing
  std::vector<uint8_t> wr(L), sel(L);
  for (int l = 0; l < L; ++l) {
    wr[l] = gi->host_write_mask ? (gi->host_write_mask[l] ? 1 : 0) : 1;
    sel[l] = ctx->gi_tskit ? 1 : wr[l];
  }
  cudaStream_t s = ctx->stream;
  CK(cudaMemcpyAsync(d_nc, ctx->gi_carriers.data(), (size_t)L * 8, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(d_sel, sel.data(), (size_t)L, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(ctx->d_gi_write, wr.data(), (size_t)L, cudaMemcpyHostToDevice, s));
  PROF(ctx, "k_gi_slots");
  k_gi_slots<<<grid_for(ctx, 4), 256, 0, s>>>(ctx->pop, ctx->d_c);
  LAUNCHED(ctx);
  PROF(ctx, "k_gi_setup");
  k_gi_setup<<<std::max(1, std::min((L + 255) / 256, grid_for(ctx, 4))), 256, 0, s>>>(
      ctx->d_gi_state, ctx->d_gi_lkey, d_nc, d_sel, L, (uint32_t)gi->seed, (uint32_t)(gi->seed >> 32));
  LAUNCHED(ctx);
  if ((r = gi_hist_pass(ctx)) != GNX_OK) return r;
  ctx->gi_stage = 1;
  *dev_hist = ctx->d_gi_hist;
  *hist_len = (int64_t)L * GI_BINS;
  return GNX_OK;
}

extern "C" int gnx_genome_init_pass(gnx_ctx* ctx, int32_t* all_done) {
  ARG(ctx && all_done, "null");
  if (ctx->gi_stage != 1) { g_last_error = "gnx_genome_init_pass outside gnx_genome_init_begin / _end"; return GNX_ERR_STATE; }
  USE_DEVICE(ctx);
  cudaStream_t s = ctx->stream;
  CK(cudaMemsetAsync(ctx->d_gi_active, 0, 2 * sizeof(int32_t), s));
  PROF(ctx, "k_gi_select");
  k_gi_select<<<ctx->cfg.L, 256, 0, s>>>(ctx->d_gi_state, ctx->d_gi_hist, ctx->d_gi_active);
  LAUNCHED(ctx);
  int32_t act[2];
  CK(cudaMemcpyAsync(act, ctx->d_gi_active, sizeof act, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (act[1]) {
    ctx->gi_stage = 0;
    g_last_error = "invalid argument: n_carriers exceeds the 2n homologues of the population at some locus (or ids repeat)";
    return GNX_ERR_ARG;
  }
  *all_done = act[0] == 0;
  if (act[0]) return gi_hist_pass(ctx);
  ctx->gi_stage = 3;                               // selected, not yet written
  return GNX_OK;
}

extern "C" int gnx_genome_init_end(gnx_ctx* ctx) {
  ARG(ctx, "null ctx");
  if (ctx->gi_stage != 3) {
    g_last_error = "gnx_genome_init_end before gnx_genome_init_pass reported every locus selected";
    return GNX_ERR_STATE;
  }
  USE_DEVICE(ctx);
  cudaStream_t s = ctx->stream;
  PROF(ctx, "k_gi_write");
  k_gi_write<<<grid_for(ctx, 8), 256, 0, s>>>(ctx->pop, ctx->d_c, ctx->d_gi_state, ctx->d_gi_lkey, ctx->d_gi_write,
                                              ctx->cfg.L, ctx->d_cols);
  LAUNCHED(ctx);
  if (ctx->cfg.n_traits > 0 && ctx->have_traits) {
    int r = gnx_phenotype(ctx);
    if (r != GNX_OK) return r;
  }
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  // the histograms are not needed any more (L x 8 KB)
  auto it = std::find(ctx->gi_allocs.begin(), ctx->gi_allocs.end(), (void*)ctx->d_gi_hist);
  if (it != ctx->gi_allocs.end()) ctx->gi_allocs.erase(it);
  CK(cudaFree(ctx->d_gi_hist));
  ctx->d_gi_hist = nullptr;
  ctx->gi_stage = 2;
  ctx->gi_t = h.t;
  return check_device_err(h);
}

extern "C" int gnx_genome_init_rows(gnx_ctx* ctx, int32_t* host_site, int64_t* host_id, int8_t* host_homologue,
                                    int64_t capacity, int64_t* n_rows) {
  ARG(ctx && n_rows, "null");
  USE_DEVICE(ctx);
  Counters h;
  int r = read_counters(ctx, &h);
  if (r != GNX_OK) return r;
  if (ctx->gi_stage != 2 || !ctx->gi_tskit || ctx->pending || h.t != ctx->gi_t) {
    g_last_error = "gnx_genome_init_rows needs a finished assignment begun with tskit_rows, before any step";
    return GNX_ERR_STATE;
  }
  const int L = ctx->cfg.L;
  std::vector<long long> off(L + 1, 0);
  for (int l = 0; l < L; ++l) off[l + 1] = off[l] + ctx->gi_carriers[l];
  const long long total = off[L];
  *n_rows = total;
  if (!host_site && !host_id && !host_homologue) return GNX_OK;
  ARG(host_site && host_id && host_homologue && capacity >= total, "host buffers missing or too small");
  std::vector<void*> tmp;
  long long* d_off = nullptr;
  unsigned long long* d_cur = nullptr;
  int32_t* d_site = nullptr;
  long long* d_id = nullptr;
  int8_t* d_h = nullptr;
  auto run = [&]() -> int {
    DM(ctx, &d_off, (size_t)L, &tmp);
    DM(ctx, &d_cur, (size_t)L, &tmp);
    DM(ctx, &d_site, (size_t)total, &tmp);
    DM(ctx, &d_id, (size_t)total, &tmp);
    DM(ctx, &d_h, (size_t)total, &tmp);
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(d_off, off.data(), (size_t)L * 8, cudaMemcpyHostToDevice, s));
    PROF(ctx, "k_gi_rows");
    k_gi_rows<<<grid_for(ctx, 8), 256, 0, s>>>(ctx->pop, ctx->d_c, ctx->d_gi_state, ctx->d_gi_lkey, d_off, d_cur,
                                               d_site, d_id, d_h, L);
    LAUNCHED(ctx);
    CK(cudaMemcpyAsync(host_site, d_site, (size_t)total * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(host_id, d_id, (size_t)total * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(host_homologue, d_h, (size_t)total, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return GNX_OK;
  };
  r = run();
  free_bucket(tmp);
  return r;
}
