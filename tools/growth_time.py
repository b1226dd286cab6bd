"""Cost of letting a population outgrow its capacity, on the GPU (writes one JSON file):

  * c2 resident ms/step with the growth guard off and on (CUDA events around 200 graph-launched steps after
    50 warm-up steps; off and on alternate over --reps rounds, each on a fresh context of the same seed);
  * the time of one gnx_reserve from 10 M to 20 M individuals at c4 (1000 loci), host clock around the call
    (it synchronises before and after).

    python tools/growth_time.py            # writes profiles/r06_growth_time.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def species(cfg, capacity, grow):
    from geonomics_b200 import workloads
    from geonomics_b200.device import DeviceSpecies
    w = workloads.build(cfg, cfg['seed'])
    dev = DeviceSpecies(w['land_dim'], w['rasters'], w['prm'], w['gen_arch'], capacity=capacity, seed=cfg['seed'],
                        grow=grow)
    dev.upload(w['pop']['x'], w['pop']['y'], w['pop']['age'], w['pop']['sex'], w['pop']['idx'],
               genomes_packed=workloads.random_packed_genomes(cfg['N'], w['L'], cfg['seed'] + 1))
    return dev


def step_ms(cfg, grow, warmup, steps):
    import torch
    dev = species(cfg, int(1.5 * cfg['N']) + 4096, grow)
    try:
        stream = torch.cuda.ExternalStream(dev.stream_ptr)
        dev.step(warmup)
        dev.sync()
        dev.step_records()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        stop = dev.step(steps)
        e1.record(stream)
        dev.sync()
        torch.cuda.synchronize()
        assert stop is None
        recs = dev.step_records()
        assert len(recs) == steps
        return e0.elapsed_time(e1) / steps, recs[-1]['Nt']
    finally:
        dev.close()


def reserve_s(cfg, n_from, n_to):
    dev = species(dict(cfg, N=n_from), n_from, False)      # full: the uploaded population fills the capacity
    try:
        dev.sync()
        t0 = time.perf_counter()
        dev.reserve(n_to)
        t1 = time.perf_counter()
        return t1 - t0
    finally:
        dev.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r06_growth_time.json'))
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--skip-reserve', action='store_true')
    a = ap.parse_args()
    from geonomics_b200 import workloads
    out = dict(gpu=gpu_info(), warmup=a.warmup, steps=a.steps, c2=dict(off=[], on=[]))
    c2 = dict(workloads.CONFIGS['c2'])
    for _ in range(a.reps):
        for key, grow in (('off', False), ('on', True)):
            ms, nt = step_ms(c2, grow, a.warmup, a.steps)
            out['c2'][key].append(ms)
            out['c2']['Nt_' + key] = nt
    off, on = min(out['c2']['off']), min(out['c2']['on'])
    out['c2']['overhead_pct'] = 100.0 * (on - off) / off
    if not a.skip_reserve:
        c4 = dict(workloads.CONFIGS['c4'])
        out['c4_reserve_10M_to_20M_s'] = reserve_s(c4, 10_000_000, 20_000_000)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
