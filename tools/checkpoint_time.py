"""Cost of a checkpoint on the GPU (writes one JSON file): host-clock time of Model.save and of load_model (both
end in a device synchronise) and the file size, for a Model of the c2 shape (1 M individuals, 100 loci) and of
the c4 shape (10 M individuals, 1000 loci; without c4's conductance surfaces, which a Model holds as tables of
approx_len directions per cell).  The model is built with make_model from the workload's rasters and sizes,
marked burned in with its genomes assigned on the device, walked --steps main steps, then saved and loaded
--reps times in a temporary directory.

    python tools/checkpoint_time.py            # writes profiles/r07_checkpoint_time.json
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def params(cfg):
    """Model parameters of a workload shape: its three rasters, N, L, traits and mating radius."""
    from geonomics_b200 import api, workloads
    w = workloads.build(cfg, cfg['seed'])
    dim = w['land_dim']
    layers = {'lyr_%d' % k: {'init': {'defined': {'rast': w['rasters'][k], 'pts': None, 'vals': None,
                                                  'interp_method': None}}} for k in range(3)}
    prm = w['prm']
    traits = {'trait_%d' % t: dict(layer='lyr_%d' % (1 + t % 2), phi=cfg['phi'], n_loci=cfg['loci_per_trait'],
                                   mu=0, alpha_distr_mu=0, alpha_distr_sigma=0.1, max_alpha_mag=0.25,
                                   gamma=cfg['gamma'], univ_adv=False) for t in range(cfg['n_traits'])}
    spp = {'init': {'N': cfg['N'], 'K_layer': 'lyr_0', 'K_factor': prm['K_factor']},
           'mating': dict(repro_age=0, sex=False, sex_ratio=1.0, R=cfg['R'], b=cfg['b'], n_births_distr_lambda=cfg['lam'],
                          n_births_fixed=True, mating_radius=cfg['mating_radius'], choose_nearest_mate=False,
                          inverse_dist_mating=False),
           'mortality': dict(max_age=None, d_min=0, d_max=1, density_grid_window_width=None),
           'movement': dict(move=True, direction_distr_mu=0, direction_distr_kappa=0,
                            movement_distance_distr_param1=1.0, movement_distance_distr_param2=1.0,
                            movement_distance_distr='wald', dispersal_distance_distr_param1=1.0,
                            dispersal_distance_distr_param2=1.0, dispersal_distance_distr='wald'),
           'gen_arch': dict(gen_arch_file=None, L=cfg['L'], start_p_fixed=None, start_neut_zero=False, mu_neut=0,
                            mu_delet=0, delet_alpha_distr_shape=0.2, delet_alpha_distr_scale=0.2,
                            r_distr_alpha=cfg['recomb_rate'], r_distr_beta=None, dom=False, pleiotropy=False,
                            n_recomb_sims=cfg['n_paths'], jitter_breakpoints=False, mut_log=False, use_tskit=False,
                            tskit_simp_interval=100, traits=traits)}
    return api.make_params_dict({
        'landscape': {'main': {'dim': dim, 'res': (1, 1), 'ulc': (0, 0), 'prj': None}, 'layers': layers},
        'comm': {'species': {'spp_0': spp}},
        'model': {'T': 100, 'burn_T': 30, 'seed': {'num': cfg['seed']},
                  'its': {'n_its': 1, 'rand_landscape': False, 'rand_comm': False, 'rand_genarch': False,
                          'repeat_burn': False}}}, 'checkpoint_time')


def burned_model(cfg, steps):
    from geonomics_b200 import api
    m = api.make_model(params(cfg), genome_init='device')
    spp = m.comm[0]
    # what the end of a burn-in does (Model._do_timestep), without the stationarity tests
    spp.burned = m.comm.burned = True
    spp._burnin_base = None
    spp._set_genomes_and_tables(m.burn_T, m.T, 'device')
    m.reassign_genomes = False
    m.walk(steps, 'main')
    return m


def close(m):
    for spp in m.comm.values():
        spp._detach()


def measure(name, cfg, steps, reps, tmp):
    from geonomics_b200 import api
    path = os.path.join(tmp, name + '.ckpt')
    m = burned_model(cfg, steps)
    out = dict(N=len(m.comm[0]), L=cfg['L'], dim=list(cfg['dim']), steps=steps, save_s=[], load_s=[])
    try:
        for _ in range(reps):
            t0 = time.perf_counter()
            m.save(path)
            out['save_s'].append(time.perf_counter() - t0)
    finally:
        close(m)
    out['file_bytes'] = os.path.getsize(path)
    for _ in range(reps):
        t0 = time.perf_counter()
        r = api.load_model(path)
        out['load_s'].append(time.perf_counter() - t0)
        close(r)
    os.remove(path)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r07_checkpoint_time.json'))
    ap.add_argument('--configs', default='c2,c4')
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--reps', type=int, default=2)
    a = ap.parse_args()
    from geonomics_b200 import workloads
    out = dict(gpu=gpu_info())
    tmp = tempfile.mkdtemp(prefix='gnx_ckpt_time_')
    try:
        out['tmp_free_bytes'] = shutil.disk_usage(tmp).free
        for name in a.configs.split(','):
            cfg = dict(workloads.CONFIGS[name], surfaces=False)
            np.random.seed(cfg['seed'])
            out[name] = measure(name, cfg, a.steps, a.reps, tmp)
            print(name, json.dumps(out[name]), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
