"""Cost of a table simplification on the GPU against the host restatement (writes one JSON file).

Model-shaped tables from the seeded generator of tests/test_cuda_simplify.py (overlapping generations, ~5
breakpoints per homologue, founders at time 1, births at -t) are simplified on the current nodes:
  * DeviceSpecies.simplify_tables: host clock around the call (uploads, kernels, result copy, all ending in a
    device synchronise), then once more with per-kernel CUDA events on (gnx_profile) for the kernel time; the
    rest of the first call's time is copies and host work;
  * tables.simplify_columns on the same tables where the host can finish (--host-max edges), and the two
    results compared column for column, bitwise.
The card's name and power limit are read in the same run.

    python tools/simplify_time.py            # writes profiles/r08_simplify_time.json
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
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def make_dev():
    from golden_io import load_case
    from parity_util import make_device
    z, arch, prm, state, draws = load_case('base')
    return make_device(arch, prm, capacity=4 * len(state['x']) + 256, seed=3)


def shape_for(edges):
    """(individuals, steps) whose tables hold about `edges` edges (about 3.6 edges per individual per step)."""
    n = max(1000, int(round(edges / 20 / 3.6)))
    return n, 20


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--edges', default='1e6,1e7,1e8,2e8')
    ap.add_argument('--host-max', type=float, default=1.5e7)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'r08_simplify_time.json'))
    a = ap.parse_args()
    import test_cuda_simplify as T
    from geonomics_b200.tables import simplify_columns
    info = gpu_info()
    dev = make_dev()
    rows = []
    for target in (float(x) for x in a.edges.split(',')):
        n, steps = shape_for(target)
        t0 = time.perf_counter()
        tc, alive, rng = T.model_tables(n, steps, seed=11, n_mut=max(1000, int(target // 100)))
        gen_s = time.perf_counter() - t0
        samples = T.shuffled_samples(alive, rng)
        row = dict(individuals=n, steps=steps, edges_in=tc.edges.num_rows, nodes_in=tc.nodes.num_rows,
                   mutations_in=tc.mutations.num_rows, samples=len(samples), generate_s=round(gen_s, 2))
        d_tc = T.clone(tc)
        t0 = time.perf_counter()
        dev.simplify_tables(d_tc, samples)
        row['device_s'] = time.perf_counter() - t0
        dev.profile(True)
        t0 = time.perf_counter()
        dev.simplify_tables(T.clone(tc), samples)
        row['device_profiled_s'] = time.perf_counter() - t0
        rep = dev.profile_report()
        dev.profile(False)
        row['kernel_s'] = sum(ms for _, ms in rep.values()) / 1e3
        row['copies_and_host_s'] = row['device_s'] - row['kernel_s']
        row['launches'] = sum(c for c, _ in rep.values())
        row['top_kernels_ms'] = dict(sorted(((k, round(ms, 3)) for k, (c, ms) in rep.items()),
                                            key=lambda kv: -kv[1])[:8])
        row.update(edges_out=d_tc.edges.num_rows, nodes_out=d_tc.nodes.num_rows,
                   levels=int(len(np.unique(tc.nodes.time[tc.edges.parent]))))
        if tc.edges.num_rows <= a.host_max:
            t0 = time.perf_counter()
            h_tc = simplify_columns(T.clone(tc), samples)
            row['host_s'] = time.perf_counter() - t0
            T.assert_tables_equal(d_tc, h_tc)
            row['equal'] = True
        print(json.dumps(row), flush=True)
        rows.append(row)
        del tc, d_tc
    dev.close()
    out = dict(gpu=info, note='one process; device_s = host clock around DeviceSpecies.simplify_tables '
               '(uploads, kernels, result copy and numpy appends); kernel_s = sum of per-kernel CUDA events of a '
               'second, profiled call; host_s = tables.simplify_columns on the same tables', rows=rows)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
