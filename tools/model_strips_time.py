"""Time the Model layer over strips: Model.walk(T, 'main') of a c4-shaped model made with
make_model(strips=group) against NcclStrips driven directly (as bench.py's strips_block drives it), same
landscape, seed and steps.

    torchrun --nproc-per-node W tools/model_strips_time.py [--presteps 50] [--steps 200] [--out profiles/...]

The c4 shape (workloads.CONFIGS['c4']: 4096^2, 10 M individuals, 1000 loci, radius 2) without its
conductance surfaces: the Model builds table-mode surfaces on the host, which at 4096^2 would not fit, so both
sides run without them.  The Model's burn-in is cut at --presteps steps (its genomes are then assigned on the
device as at the end of a burn-in); the direct side steps --presteps times before timing.  Writes the GPU name,
its power limit and both ms/step (the slowest rank's) as JSON."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def c4_params(w, cfg, T):
    """A parameters dict of the workload: layer 0 is K, layers 1 and 2 the trait gradients."""
    from geonomics_b200 import api
    X, Y = w['land_dim']
    layers = {'lyr_%d' % k: {'init': {'defined': {'rast': w['rasters'][k], 'pts': None, 'vals': None,
                                                  'interp_method': None}}} for k in range(3)}
    traits = {'trait_%d' % t: {'layer': 'lyr_%d' % (1 + t % 2), 'phi': cfg['phi'], 'n_loci': cfg['loci_per_trait'],
                               'mu': 0, 'alpha_distr_mu': 0, 'alpha_distr_sigma': 0.1, 'max_alpha_mag': 0.25,
                               'gamma': cfg['gamma'], 'univ_adv': False} for t in range(cfg['n_traits'])}
    spp = {'init': {'N': cfg['N'], 'K_layer': 'lyr_0', 'K_factor': w['prm']['K_factor']},
           'mating': {'repro_age': 0, 'sex': False, 'sex_ratio': 1, 'R': cfg['R'], 'b': cfg['b'],
                      'n_births_distr_lambda': cfg['lam'], 'n_births_fixed': True,
                      'mating_radius': cfg['mating_radius'], 'choose_nearest_mate': False,
                      'inverse_dist_mating': False},
           'mortality': {'max_age': None, 'd_min': 0, 'd_max': 1, 'density_grid_window_width': None},
           'movement': {'move': True, 'direction_distr_mu': 0, 'direction_distr_kappa': 0,
                        'movement_distance_distr': 'wald', 'movement_distance_distr_param1': 1.0,
                        'movement_distance_distr_param2': 1.0, 'dispersal_distance_distr': 'wald',
                        'dispersal_distance_distr_param1': 1.0, 'dispersal_distance_distr_param2': 1.0},
           'gen_arch': {'gen_arch_file': None, 'L': cfg['L'], 'start_p_fixed': 0.5, 'start_neut_zero': False,
                        'mu_neut': 0, 'mu_delet': 0, 'r_distr_alpha': cfg['recomb_rate'], 'r_distr_beta': None,
                        'dom': False, 'pleiotropy': False, 'n_recomb_sims': cfg['n_paths'], 'use_tskit': False,
                        'traits': traits}}
    return api.make_params_dict({'landscape': {'main': {'dim': (X, Y), 'res': (1, 1), 'ulc': (0, 0), 'prj': None},
                                               'layers': layers},
                                 'comm': {'species': {'spp_0': spp}},
                                 'model': {'T': T, 'burn_T': 50, 'seed': {'num': cfg['seed']},
                                           'its': {'n_its': 1}}}, 'c4_strips')


def timed(dist, fn):
    import torch
    torch.cuda.synchronize()
    dist.barrier()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    dist.barrier()
    return (time.perf_counter() - t0) * 1e3


def model_ms(dist, group, w, cfg, presteps, steps):
    from geonomics_b200 import api
    model = api.make_model(c4_params(w, cfg, steps), strips=group, genome_init='device')
    spp = model.comm[0]
    model.walk(presteps, 'burn')
    if not model.comm.burned:                      # the end of a burn-in, without waiting for its tests
        spp.burned = True
        spp._set_genomes_and_tables(model.burn_T, model.T, 'device')
        model.reassign_genomes = False
        model.comm.burned = True
    model.walk(5, 'main')                          # warm-up: the step graph is captured
    ms = timed(dist, lambda: model.walk(steps, 'main'))
    n = spp.Nt[-1]
    spp._detach()
    return ms / steps, n


def direct_ms(dist, w, cfg, presteps, steps, rank, world):
    from geonomics_b200 import strips, workloads
    N0 = cfg['N']
    cap = int(2.0 * N0 / world) + 65536
    st = strips.NcclStrips(w['land_dim'], w['rasters'], w['prm'], w['gen_arch'], capacity=cap, seed=cfg['seed'],
                           migrant_capacity=max(65536, cap // 8), halo_capacity=max(65536, cap // 4))
    p = w['pop']
    own = strips.owner_of(p['y'], st.bounds, st.cs, st.ncy) == rank
    st.dev.upload(p['x'][own], p['y'][own], p['age'][own], p['sex'][own], p['idx'][own],
                  genomes_packed=workloads.random_packed_genomes(int(own.sum()), w['L'], cfg['seed'] + 1 + rank),
                  max_ind_idx=N0 - 1)
    st.step(presteps + 5)
    st.sync()
    st.step_records_local()

    def run():
        st.step(steps)
        st.sync()
        st.step_records_local()
    ms = timed(dist, run)
    st.close()
    return ms / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--presteps', type=int, default=50)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from geonomics_b200 import workloads
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank, world = dist.get_rank(), dist.get_world_size()
    cfg = dict(workloads.CONFIGS['c4'], surfaces=False)
    w = workloads.build(cfg, cfg['seed'])
    direct = direct_ms(dist, w, cfg, args.presteps, args.steps, rank, world)
    model, n = model_ms(dist, dist.group.WORLD, w, cfg, args.presteps, args.steps)
    t = torch.tensor([direct, model], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', str(local)],
                           capture_output=True, text=True).stdout.strip()
        res = dict(workload='c4 without conductance surfaces, %d strips' % world, gpus=world, gpu_and_power_limit=q,
                   steps=args.steps, presteps=args.presteps, direct_ms_per_step=float(t[0]),
                   model_ms_per_step=float(t[1]), model_overhead=float(t[1] / t[0] - 1), model_final_N=int(n))
        out = args.out or os.path.join(ROOT, 'profiles', 'model_strips_time_%dgpu.json' % world)
        with open(out, 'w') as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res))
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
