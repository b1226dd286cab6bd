#!/usr/bin/env python
"""DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) of every kernel in an
`ncu --set full` capture, under the names bench.py uses -> profiles/r02_traffic.json.

  python tools/make_traffic.py REPORT.ncu-rep WORKLOAD [--out profiles/r02_traffic.json]

bench.py copies the figure of the dominant kernel into `roofline.traffic`.
"""
import argparse
import csv
import io
import json
import os
import re
import subprocess

SCAN = {'CellScan': 'scan_cells', 'PairScan': 'scan_pairs', 'BirthScan': 'scan_births',
        'MortalityScan': 'scan_mortality', 'TskitScan': 'scan_tskit_edges'}


def bench_name(ncu_name):
    n = ncu_name.replace('void ', '').split('(')[0]
    m = re.match(r'scan_(reduce|apply|spine)_kernel<(\w+)>', n)
    if m:
        return '%s.%s' % (SCAN.get(m.group(2), m.group(2)), m.group(1))
    n = re.sub(r'<.*>', '', n)
    return {'k_ct_gradients_reg': 'k_ct_gradients'}.get(n, n)


def to_bytes(v, unit):
    return float(v.replace(',', '')) * {'byte': 1, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9, 'Tbyte': 1e12}.get(unit, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('report')
    ap.add_argument('workload')
    ap.add_argument('--out', default='profiles/r02_traffic.json')
    a = ap.parse_args()
    txt = subprocess.run(['ncu', '-i', a.report, '--page', 'raw', '--csv'], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(txt)))
    h, units = rows[0], rows[1]
    ix = {n: i for i, n in enumerate(h)}
    acc = {}
    for r in rows[2:]:
        name = bench_name(r[ix['Kernel Name']])
        b = sum(to_bytes(r[ix[c]], units[ix[c]]) for c in ('dram__bytes_read.sum', 'dram__bytes_write.sum'))
        t = float(r[ix['gpu__time_duration.sum']].replace(',', ''))
        t *= {'ns': 1e-3, 'us': 1.0, 'ms': 1e3}.get(units[ix['gpu__time_duration.sum']], 1.0)
        if name in ('k_find_mates_dense', 'k_mate_select'):   # parts of the same search: one row, as in bench.py
            d = acc.setdefault('k_find_mates', [0, 0.0, 0.0])
            d[1] += b
            d[2] += t
            continue
        d = acc.setdefault(name, [0, 0.0, 0.0])
        d[0] += 1
        d[1] += b
        d[2] += t
    out = {}
    if os.path.exists(a.out):
        out = json.load(open(a.out))
    out[a.workload] = {'source': os.path.basename(a.report),
                       'kernels': {k: {'launches': v[0], 'dram_bytes_per_launch': v[1] / v[0],
                                       'ncu_us_per_launch': v[2] / v[0]} for k, v in sorted(acc.items())}}
    with open(a.out, 'w') as f:
        json.dump(out, f, indent=1, sort_keys=True)
    for k, v in sorted(acc.items(), key=lambda kv: -kv[1][2]):
        print('%-26s x%d  %8.1f MB/launch  %7.1f us/launch' % (k, v[0], v[1] / v[0] / 1e6, v[2] / v[0]))


if __name__ == '__main__':
    main()
