"""Time the device assignment of the starting genomes (DeviceSpecies.init_genomes) at the population
shapes of the c2, c4 and c5 workloads, and the host assignment (numpy permutations, host array, upload)
at c2 for comparison.  Device times are CUDA events on the context's stream around the whole staged
call (every stage ends in a stream synchronise); the host path is timed by the host clock around work
that ends with the synchronous upload.  Writes one JSON file with the card's name and power limit read
in the same run.

  python tools/genome_init_time.py [--out profiles/r03_genome_init_time.json] [--configs c2,c4,c5] [--reps 3]
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


def _host_assign(dev, n, p):
    """The host path of Species._set_genomes_and_tables: one permutation per locus into an int8[n, L, 2]
    array, packed and uploaded."""
    from geonomics_b200 import genome_pack as gp
    s = dev.download(genomes=False)
    L = len(p)
    g = np.zeros((n, L, 2), dtype=np.int8)
    counts = gp.carrier_counts(n, p)
    for site in range(L):
        if counts[site] > 0:
            hom = np.random.permutation(2 * n)[:counts[site]]
            g[hom // 2, site, hom % 2] = 1
    dev.upload(s['x'], s['y'], s['age'], s['sex'], s['idx'], g=g, max_ind_idx=s['max_ind_idx'])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r03_genome_init_time.json'))
    ap.add_argument('--configs', default='c2,c4,c5')
    ap.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    import torch
    from geonomics_b200 import workloads
    from geonomics_b200 import genome_pack as gp
    from geonomics_b200.device import DeviceSpecies
    if not torch.cuda.is_available():
        raise SystemExit('genome_init_time.py needs a CUDA device')
    out = dict(card=_card(), results={})
    for name in a.configs.split(','):
        cfg = dict(workloads.CONFIGS[name])
        cfg['n_paths'] = 16                                  # the paths play no part in the assignment
        w = workloads.build(cfg)
        pop, L = w['pop'], w['L']
        n = len(pop['x'])
        p = np.full(L, 0.5)                                   # start_p_fixed = 0.5
        dev = DeviceSpecies(w['land_dim'], w['rasters'], w['prm'], w['gen_arch'], capacity=n + 4096, seed=1)
        try:
            dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
            stream = torch.cuda.ExternalStream(dev.stream_ptr)
            times, passes = [], 0
            for rep in range(a.reps + 1):                     # rep 0 loads the kernels
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                dev.genome_init_begin(gp.carrier_counts(n, p), 1000 + rep)
                passes = 1
                while not dev.genome_init_pass():
                    passes += 1
                dev.genome_init_end()
                e1.record(stream)
                e1.synchronize()
                if rep:
                    times.append(e0.elapsed_time(e1) / 1e3)
            g_sum = dev.stats()['freq'] * 2 * n
            exact = bool(np.array_equal(np.rint(g_sum).astype(np.int64), gp.carrier_counts(n, p)))
            res = dict(N=n, L=L, device_s=times, device_s_min=min(times), histogram_passes=passes,
                       keys_per_pass=2 * n * L, exact_counts=exact)
            if name == 'c2':
                np.random.seed(0)
                t0 = time.perf_counter()
                _host_assign(dev, n, p)
                res['host_s'] = time.perf_counter() - t0
                res['speedup_over_host'] = res['host_s'] / res['device_s_min']
            out['results'][name] = res
            print(name, json.dumps(res), flush=True)
        finally:
            dev.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out['card']))


if __name__ == '__main__':
    main()
