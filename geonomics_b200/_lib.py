"""ctypes binding of libgnxb200.so (C-ABI declared in include/gnx_b200.h).

There is no CPU fallback: if the shared library is missing the import of this module's
`lib()` raises, and every op in the package fails loudly.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# GNX_B200_LIB selects another build of the same library (kernel experiments); never a fallback
LIB_PATH = os.environ.get('GNX_B200_LIB') or os.path.join(HERE, 'libgnxb200.so')
HEADER_PATH = os.path.join(os.path.dirname(HERE), 'include', 'gnx_b200.h')

GNX_ABI_VERSION = 1
GNX_MAX_TRAITS = 8
GNX_MAX_LAYERS = 16

DISTR = {'wald': 0, 'lognormal': 1, 'levy': 2}
SURF_NONE, SURF_TABLE, SURF_ONTHEFLY = 0, 1, 2

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_uint32_p = C.POINTER(C.c_uint32)
c_int64_p = C.POINTER(C.c_int64)
c_int8_p = C.POINTER(C.c_int8)
c_uint16_p = C.POINTER(C.c_uint16)


class Config(C.Structure):
    _fields_ = [
        ('abi_version', C.c_int32),
        ('dim_x', C.c_int32), ('dim_y', C.c_int32),
        ('n_layers', C.c_int32),
        ('capacity', C.c_int64),
        ('seed', C.c_uint64),
        ('L', C.c_int32), ('n_recomb_paths', C.c_int32), ('n_traits', C.c_int32), ('use_dom', C.c_int32),
        ('mating_radius', C.c_double), ('b', C.c_double), ('R', C.c_double),
        ('n_births_lambda', C.c_double),
        ('n_births_fixed', C.c_int32), ('sex', C.c_int32),
        ('sex_ratio_p', C.c_double),
        ('choose_nearest', C.c_int32), ('inverse_dist', C.c_int32),
        ('d_min', C.c_double), ('d_max', C.c_double),
        ('max_age', C.c_int32), ('K_layer', C.c_int32),
        ('K_factor', C.c_double),
        ('move', C.c_int32), ('move_distr', C.c_int32), ('disp_distr', C.c_int32),
        ('move_p1', C.c_double), ('move_p2', C.c_double), ('disp_p1', C.c_double), ('disp_p2', C.c_double),
        ('dir_mu', C.c_double), ('dir_kappa', C.c_double),
        ('res_ratio_x', C.c_double), ('res_ratio_y', C.c_double),
        ('move_surf_mode', C.c_int32), ('disp_surf_mode', C.c_int32),
        ('move_surf_layer', C.c_int32), ('disp_surf_layer', C.c_int32),
        ('move_surf_mixture', C.c_int32), ('disp_surf_mixture', C.c_int32),
        ('move_surf_kappa', C.c_double), ('disp_surf_kappa', C.c_double),
        ('surf_approx_len', C.c_int32), ('disp_max_tries_injected', C.c_int32),
    ]


class Trait(C.Structure):
    _fields_ = [
        ('n_loci', C.c_int32),
        ('host_loci', c_int32_p),
        ('host_alpha', c_double_p),
        ('phi', C.c_double),
        ('host_phi_raster', c_double_p),
        ('gamma', C.c_double),
        ('layer', C.c_int32), ('univ_adv', C.c_int32),
    ]


class Density(C.Structure):
    _fields_ = [
        ('window_width', C.c_double),
        ('n_points', C.c_int32),
        ('host_points', c_double_p),
        ('host_areas', c_double_p),
        ('grid_ni', C.c_int32 * 4), ('grid_nj', C.c_int32 * 4),
        ('grid_i0', C.c_int32 * 4), ('grid_j0', C.c_int32 * 4),
        ('grid_x_edge', C.c_int32 * 4), ('grid_y_edge', C.c_int32 * 4),
        ('n_tri', C.c_int32),
        ('host_simplices', c_int32_p),
        ('host_neighbors', c_int32_p),
        ('host_nbr_indptr', c_int32_p),
        ('host_nbr_indices', c_int32_p),
        ('lat_ni', C.c_int32), ('lat_nj', C.c_int32),
        ('host_square_tri', c_int32_p),
        ('colourable', C.c_int32),
    ]


class Draws(C.Structure):
    _fields_ = [
        ('n', C.c_int64),
        ('move_dir', c_double_p), ('move_choice', c_int32_p), ('move_dist', c_double_p),
        ('mate_R', c_uint32_p), ('mate_inv_u', c_double_p), ('mate_u', c_double_p),
        ('poisson', c_int32_p), ('recomb_keys', c_int32_p), ('start_homs', c_int32_p),
        ('disp_dir', c_double_p), ('disp_choice', c_int32_p), ('disp_dist', c_double_p),
        ('sex_u', c_double_p), ('sex_redraw_u', c_double_p), ('death_u', c_double_p),
        ('pan_u', c_double_p), ('pan_R', c_uint32_p),
        ('n_mut', C.c_int64),
        ('mut_n', c_int32_p), ('mut_type_u', c_double_p), ('mut_ind_R', c_uint32_p),
        ('mut_homol_u', c_double_p), ('mut_s', c_double_p), ('mut_alpha', c_double_p),
    ]


class Population(C.Structure):
    _fields_ = [
        ('n', C.c_int64),
        ('x', c_double_p), ('y', c_double_p),
        ('age', c_int32_p), ('sex', c_int8_p), ('idx', c_int64_p),
        ('genomes', c_uint32_p),
        ('z', c_double_p), ('fit', c_double_p), ('e', c_double_p),
        ('max_ind_idx', C.c_int64),
    ]


class StripConfig(C.Structure):
    _fields_ = [
        ('rank', C.c_int32), ('world', C.c_int32),
        ('first_rows', c_int32_p),
        ('migrant_capacity', C.c_int64), ('halo_capacity', C.c_int64),
    ]


class StripEndpoints(C.Structure):
    _fields_ = [
        ('base', C.c_void_p),
        ('bytes', C.c_int64),
        ('buf_offset', C.c_int64 * 4),
        ('count_offset', C.c_int64 * 4),
        ('ipc_handle', C.c_ubyte * 64),
        ('sync_offset', C.c_int64),
        ('counts_cap', C.c_int64),
    ]


class Mutation(C.Structure):
    _fields_ = [
        ('mu_neut', C.c_double), ('mu_delet', C.c_double),
        ('delet_s_shape', C.c_double), ('delet_s_scale', C.c_double),
        ('n_mutables', C.c_int32), ('host_mutables', c_int32_p),
        ('n_nonneut', C.c_int32), ('host_nonneut_loci', c_int32_p),
        ('n_delet', C.c_int32), ('host_delet_loci', c_int32_p), ('host_delet_s', c_double_p),
        ('log_capacity', C.c_int32), ('tskit_layout', C.c_int32),
        ('host_trait_mu', c_double_p), ('host_trait_alpha_distr', c_double_p),
        ('host_trait_loci_idxs', c_int32_p), ('host_delet_loci_idxs', c_int32_p),
        ('host_subsetters', C.POINTER(C.c_uint8)),
    ]


class MutationRow(C.Structure):
    _fields_ = [('t', C.c_int64), ('individual', C.c_int64), ('locus', C.c_int32), ('row', C.c_int32),
                ('homologue', C.c_int32), ('type', C.c_int32), ('s', C.c_double), ('alpha', C.c_double),
                ('node', C.c_int32), ('reserved', C.c_int32)]


class StepRecord(C.Structure):
    _fields_ = [('t', C.c_int64), ('Nt', C.c_int64), ('n_births', C.c_int64),
                ('n_deaths', C.c_int64), ('n_pairs', C.c_int64)]


class TskitRows(C.Structure):
    _fields_ = [
        ('n_edges', C.c_int64), ('n_births', C.c_int64),
        ('edge_left', c_double_p), ('edge_right', c_double_p), ('edge_parent', c_int32_p), ('edge_child', c_int32_p),
        ('birth_idx', c_int64_p),
        ('birth_x', c_double_p), ('birth_y', c_double_p),
        ('birth_z', c_double_p),
        ('birth_time', c_double_p),
        ('first_node_id', C.c_int32),
        ('first_individual_row', C.c_int32),
    ]


class StepStatus(C.Structure):
    _fields_ = [('steps_run', C.c_int32), ('stopped', C.c_int32),
                ('need_entries', C.c_int64), ('need_slots', C.c_int64), ('need_births', C.c_int64),
                ('need_edges', C.c_int64), ('capacity', C.c_int64), ('born_capacity', C.c_int64),
                ('edge_capacity', C.c_int64)]


class Tables(C.Structure):
    _fields_ = [
        ('sequence_length', C.c_double),
        ('n_nodes', C.c_int64),
        ('node_flags', c_int32_p), ('node_time', c_double_p), ('node_population', c_int32_p),
        ('node_individual', c_int32_p),
        ('n_edges', C.c_int64),
        ('edge_left', c_double_p), ('edge_right', c_double_p), ('edge_parent', c_int32_p), ('edge_child', c_int32_p),
        ('n_individuals', C.c_int64), ('n_location', C.c_int32),
        ('individual_flags', c_int32_p), ('individual_location', c_double_p), ('individual_idx', c_int64_p),
        ('n_sites', C.c_int64), ('site_position', c_double_p),
        ('n_mutations', C.c_int64),
        ('mutation_site', c_int32_p), ('mutation_node', c_int32_p), ('mutation_time', c_double_p),
    ]


class GenomeInit(C.Structure):
    _fields_ = [
        ('seed', C.c_uint64),
        ('n_loci', C.c_int32),
        ('host_n_carriers', c_int64_p),
        ('host_write_mask', C.POINTER(C.c_uint8)),
        ('tskit_rows', C.c_int32),
    ]


FIELDS = dict(
    X=1, Y=2, AGE=3, SEX=4, IDX=5, Z=6, FIT=7, GSLOT=8, N_NBRS=9, MATE=10, PAIRS=11, NB=12,
    PERM=13, CELL_START=14, COUNTS_N=15, COUNTS_P=16, VALS_N=17, VALS_P=18, GRAD_N=19, GRAD_P=20,
    N_RAST=21, NPAIRS_RAST=22, D_RAST=23, K_RAST=24, DEATH_P=25, ALIVE=26, DISP_TRIES=27, E=28,
    COUNTERS=29, GENOMES=30, NODE0=31, NODE1=32, VM_TAB_MOVE=33, VM_TAB_DISP=34)

# every exported entry point: name -> (restype, argtypes)
_ctx = C.c_void_p
SIGNATURES = {
    'gnx_strerror': (C.c_char_p, [C.c_int]),
    'gnx_last_error': (C.c_char_p, []),
    'gnx_abi_version': (C.c_int, []),
    'gnx_create': (C.c_int, [C.POINTER(Config), C.POINTER(_ctx)]),
    'gnx_destroy': (C.c_int, [_ctx]),
    'gnx_set_rasters': (C.c_int, [_ctx, c_double_p]),
    'gnx_set_traits': (C.c_int, [_ctx, C.c_int32, C.POINTER(Trait), c_int8_p]),
    'gnx_set_recomb_paths': (C.c_int, [_ctx, c_uint32_p]),
    'gnx_set_density': (C.c_int, [_ctx, C.POINTER(Density)]),
    'gnx_set_surface_tables': (C.c_int, [_ctx, c_uint16_p, c_uint16_p]),
    'gnx_set_draws': (C.c_int, [_ctx, C.POINTER(Draws)]),
    'gnx_set_burn': (C.c_int, [_ctx, C.c_int32]),
    'gnx_set_debug': (C.c_int, [_ctx, C.c_int32]),
    'gnx_upload_population': (C.c_int, [_ctx, C.POINTER(Population)]),
    'gnx_download_population': (C.c_int, [_ctx, C.POINTER(Population)]),
    'gnx_population_size': (C.c_int, [_ctx, c_int64_p]),
    'gnx_age_step': (C.c_int, [_ctx]),
    'gnx_move': (C.c_int, [_ctx]),
    'gnx_sample_env': (C.c_int, [_ctx]),
    'gnx_bin_cells': (C.c_int, [_ctx]),
    'gnx_find_mates': (C.c_int, [_ctx]),
    'gnx_dedup_pairs': (C.c_int, [_ctx]),
    'gnx_make_offspring': (C.c_int, [_ctx]),
    'gnx_density_counts': (C.c_int, [_ctx]),
    'gnx_density_eval': (C.c_int, [_ctx]),
    'gnx_death_prob': (C.c_int, [_ctx]),
    'gnx_mortality': (C.c_int, [_ctx]),
    'gnx_set_raster': (C.c_int, [_ctx, C.c_int32, c_double_p]),
    'gnx_strip_enable': (C.c_int, [_ctx, C.POINTER(StripConfig)]),
    'gnx_strip_endpoints': (C.c_int, [_ctx, C.POINTER(StripEndpoints)]),
    'gnx_strip_connect': (C.c_int, [_ctx, C.c_int32, C.POINTER(StripEndpoints), C.c_int32]),
    'gnx_strip_collective_ptrs': (C.c_int, [_ctx, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_int64), C.POINTER(C.c_void_p)]),
    'gnx_strip_pairs_ptr': (C.c_int, [_ctx, C.POINTER(C.c_void_p)]),
    'gnx_strip_phase': (C.c_int, [_ctx, C.c_int32]),
    'gnx_strip_phase_order': (C.c_int, [C.c_int32, c_int32_p, c_int32_p, c_int32_p]),
    'gnx_strip_barrier': (C.c_int, [_ctx, C.c_int32]),
    'gnx_strip_check': (C.c_int, [_ctx]),
    'gnx_set_K': (C.c_int, [_ctx, c_double_p]),
    'gnx_set_life_history': (C.c_int, [_ctx, C.POINTER(Config)]),
    'gnx_step': (C.c_int, [_ctx, C.c_int32]),
    'gnx_sync': (C.c_int, [_ctx]),
    'gnx_set_growth_guard': (C.c_int, [_ctx, C.c_int32]),
    'gnx_step_status': (C.c_int, [_ctx, C.POINTER(StepStatus)]),
    'gnx_reserve': (C.c_int, [_ctx, C.c_int64]),
    'gnx_tskit_reserve': (C.c_int, [_ctx, C.c_int64, C.c_int64]),
    'gnx_walk_host': (C.c_int, [_ctx, C.POINTER(Population), C.c_int32]),
    'gnx_walk_host_begin': (C.c_int, [_ctx, C.POINTER(Population), C.c_int32]),
    'gnx_walk_host_end': (C.c_int, [_ctx, C.POINTER(Population)]),
    'gnx_read_step_records': (C.c_int, [_ctx, C.POINTER(StepRecord), C.c_int32, c_int32_p]),
    'gnx_tskit_enable': (C.c_int, [_ctx, C.c_int64, C.c_int64]),
    'gnx_tskit_set_nodes': (C.c_int, [_ctx, c_int32_p, c_int32_p, C.c_int64, C.c_int32, C.c_int32]),
    'gnx_tskit_drain': (C.c_int, [_ctx, C.POINTER(TskitRows)]),
    'gnx_tskit_renumber': (C.c_int, [_ctx]),
    'gnx_set_mutation': (C.c_int, [_ctx, C.POINTER(Mutation)]),
    'gnx_mutate': (C.c_int, [_ctx]),
    'gnx_read_mutations': (C.c_int, [_ctx, C.POINTER(MutationRow), C.c_int32, c_int32_p, c_int32_p, c_int32_p,
                                     c_int32_p, c_int32_p, c_double_p, c_int32_p]),
    'gnx_read_mutation_tables': (C.c_int, [_ctx, C.c_int32, c_int32_p, c_int32_p, c_double_p, c_int32_p, c_int32_p]),
    'gnx_create_cols': (C.c_int, [C.POINTER(Config), C.c_int32, C.c_int32, c_int32_p, C.POINTER(_ctx)]),
    'gnx_set_clock': (C.c_int, [_ctx, C.c_int64, C.c_int64]),
    'gnx_read_paths': (C.c_int, [_ctx, c_uint32_p, C.c_int64]),
    'gnx_simplify': (C.c_int, [_ctx, C.POINTER(Tables), c_int32_p, C.c_int64, c_int64_p]),
    'gnx_simplify_result': (C.c_int, [_ctx, C.POINTER(Tables)]),
    'gnx_read_cols': (C.c_int, [_ctx, c_int32_p, c_int32_p, c_int32_p]),
    'gnx_widen_cols': (C.c_int, [_ctx, C.c_int32]),
    'gnx_genome_init_begin': (C.c_int, [_ctx, C.POINTER(GenomeInit), C.POINTER(C.c_void_p), c_int64_p]),
    'gnx_genome_init_pass': (C.c_int, [_ctx, c_int32_p]),
    'gnx_genome_init_end': (C.c_int, [_ctx]),
    'gnx_genome_init_rows': (C.c_int, [_ctx, c_int32_p, c_int64_p, c_int8_p, C.c_int64, c_int64_p]),
    'gnx_stats_genotypes': (C.c_int, [_ctx, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), c_double_p, c_int64_p]),
    'gnx_stats_genotypes_region': (C.c_int, [_ctx, C.c_double, C.c_double, C.c_double, C.c_double,
                                             C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), c_double_p, c_int64_p]),
    'gnx_stats_ld': (C.c_int, [_ctx, C.POINTER(C.c_uint64), c_int64_p]),
    'gnx_burnin_cell_stats': (C.c_int, [_ctx, c_int64_p, c_int64_p]),
    'gnx_strip_burnin_count': (C.c_int, [_ctx, c_int32_p, c_int32_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    'gnx_strip_burnin_diff': (C.c_int, [_ctx, C.c_int32, c_int64_p, c_int64_p]),
    'gnx_read_field': (C.c_int, [_ctx, C.c_int32, C.c_void_p, C.c_int64]),
    'gnx_device_ptr': (C.c_int, [_ctx, C.c_int32, C.POINTER(C.c_void_p), c_int64_p]),
    'gnx_stream': (C.c_void_p, [_ctx]),
    'gnx_launch_count': (C.c_int64, [_ctx]),
    'gnx_graph_launch_count': (C.c_int64, [_ctx]),
    'gnx_graph_capture_count': (C.c_int64, [_ctx]),
    'gnx_profile': (C.c_int, [_ctx, C.c_int32]),
    'gnx_profile_report': (C.c_int, [_ctx, C.c_char_p, C.c_int64]),
}

_LIB = None


class GnxError(RuntimeError):
    def __init__(self, code, what, detail):
        super().__init__('%s failed: %s (%d)%s' % (what, detail[0], code, (': ' + detail[1]) if detail[1] else ''))
        self.code = code


def lib():
    """Load libgnxb200.so (built in-tree by __graft_entry__.build()).  No fallback."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError('geonomics_b200: %s is missing -- build it with '
                              '`python -c "import __graft_entry__ as g; g.build()"`; there is '
                              'no CPU fallback for this package' % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.gnx_abi_version() != GNX_ABI_VERSION:
            raise ImportError('libgnxb200.so ABI version mismatch')
        _LIB = L
    return _LIB


def check(code, what):
    if code != 0:
        L = lib()
        raise GnxError(code, what, (L.gnx_strerror(code).decode(), L.gnx_last_error().decode()))
