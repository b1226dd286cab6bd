"""Time a use_tskit species with mutation on in the by-locus tskit layout and in the column layout
(gnx_create_cols), alternating the two in one run: the c5 workload (500k individuals, 10 000 loci, 20 of them
trait loci), ms per step, k_gametes ms per step (gnx_profile, a separate profiled run) and k_gametes'
algorithmic bytes per birth (two parents' rows read, one child row written; the cached paths stay in L2).
Then a shape the by-locus layout cannot allocate -- c4's 10M individuals at 100 000 loci, 100 of them
non-neutral, starting neutral loci zero -- in the column layout only.  Step times are taken by the host clock
around steps that end in a device synchronise.  Writes one JSON file with the card's name and power limit
read in the same run.

  python tools/cols_time.py [--out profiles/r06_cols_time.json] [--steps 200] [--big-steps 300] [--reps 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [v.strip() for v in q.split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def _species(w, cols, mu, seed=1):
    """A use_tskit species of workload w after its genome assignment (non-neutral loci at p = 0.5, neutral
    loci zero), mutation on in the tskit layout; cols: the column layout."""
    from geonomics_b200.device import DeviceSpecies
    ga = dict(w['gen_arch'])
    L = ga['L']
    nonneut = np.unique(np.concatenate([np.asarray(t['loci']) for t in ga['traits']]))
    if cols:
        ga['cols'] = nonneut
    n = len(w['pop']['x'])
    dev = DeviceSpecies(w['land_dim'], w['rasters'], w['prm'], ga, capacity=3 * n, seed=seed)
    pop = w['pop']
    dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
    p = np.zeros(L)
    p[nonneut] = 0.5
    mask = np.zeros(L, np.uint8)
    mask[nonneut] = 1
    dev.init_genomes(p, seed + 1, write_mask=mask)
    T = len(ga['traits'])
    mutables = [int(v) for v in np.random.default_rng(seed).permutation(np.setdiff1d(np.arange(L), nonneut))]
    dev.set_mutation(mu[0], mu[1], mutables, nonneut, tskit_layout=True, trait_mus=[mu[2]] * T,
                     trait_alpha_distr=[(0.0, 0.1, None)] * T, log_capacity=1 << 16)
    return dev


def _time_steps(dev, steps, warmup):
    dev.step(warmup, sync=True)
    dev.read_mutations(1 << 16)
    t0 = time.perf_counter()
    dev.step(steps, sync=True)
    ms = 1e3 * (time.perf_counter() - t0) / steps
    recs = dev.step_records()[-steps:]
    log, _ = dev.read_mutations(1 << 16)
    return ms, float(np.mean([r['n_births'] for r in recs])), recs[-1]['Nt'], len(log)


def _gametes_ms(dev, steps):
    dev.profile(True)
    dev.step(steps, sync=True)
    rep = dev.profile_report()
    dev.profile(False)
    dev.step_records()
    dev.read_mutations(1 << 16)
    k = rep.get('k_gametes')
    return None if k is None else k[1] / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r06_cols_time.json'))
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--big-steps', type=int, default=300)
    a = ap.parse_args()
    from geonomics_b200 import workloads
    out = dict(card=_card(), c5=[], big=None,
               note='use_tskit, c5: mu_neut = mu_delet = 1e-9, trait mu = 1e-9 (big: 1e-11 each); ms_per_step by the host clock around '
                    'gnx_step calls that end in a synchronise (the column layout also reads its column count when '
                    'the bound of GNX_MUT_MAX_NEW per step would pass the capacity); k_gametes_ms from a separate '
                    'profiled run (gnx_profile: CUDA events around every launch)')
    mu = (1e-9, 1e-9, 1e-9)
    w = workloads.build(workloads.CONFIGS['c5'])
    for rep in range(a.reps):
        for cols in (False, True):
            dev = _species(w, cols, mu)
            try:
                ms, births, Nt, n_mut = _time_steps(dev, a.steps, a.warmup)
                kg = _gametes_ms(dev, 50)
                wq = dev.W // 4
                row = dict(layout='columns' if cols else 'by_locus', rep=rep, ms_per_step=ms, births_per_step=births,
                           Nt=Nt, mutations=n_mut, row_bytes_per_homologue=16 * wq, k_gametes_ms_per_step=kg,
                           k_gametes_bytes_per_birth=6 * 16 * wq,
                           columns=len(dev.read_cols()) if cols else None, col_capacity=dev.col_capacity if cols else None)
            finally:
                dev.close()
            print(json.dumps(row), flush=True)
            out['c5'].append(row)
    del w
    cfg = dict(workloads.CONFIGS['c4'], L=100_000, n_paths=1000)
    w = workloads.build(cfg)
    dev = _species(w, True, (1e-11, 1e-11, 1e-11))      # ~1 M births a step: a few mutations a step, as at c5
    try:
        t0 = time.perf_counter()
        ms, births, Nt, n_mut = _time_steps(dev, a.big_steps, a.warmup)
        out['big'] = dict(config='c4 with L = 100000 (100 non-neutral), n_paths = 1000', N0=cfg['N'],
                          capacity=dev.capacity, ms_per_step=ms, births_per_step=births, Nt=Nt, mutations=n_mut,
                          steps=a.big_steps, columns=len(dev.read_cols()), col_capacity=dev.col_capacity,
                          genome_buffer_GB=dev.capacity * 2 * 4 * dev.W / 1e9,
                          by_locus_genome_buffer_GB=dev.capacity * 2 * 16 * ((cfg['L'] + 127) // 128) / 1e9,
                          wall_s=time.perf_counter() - t0)
    finally:
        dev.close()
    print(json.dumps(out['big']), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
