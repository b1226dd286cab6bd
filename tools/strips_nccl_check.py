"""Multi-process check of the strip decomposition (run under torchrun, one rank per GPU):
the ranks jointly advance one landscape through NcclStrips (records written into the peers'
buffers over NVLink through CUDA IPC, barriers and collectives by gnx_strip_barrier over peer
memory); rank 0 also runs the same population undecomposed and compares -- ids, positions,
ages, genomes, phenotypes, fitness and the step records must be identical.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
      --master-port 29511 tools/strips_nccl_check.py [steps] [--mutation] [--poisson] [--genome-init]

--mutation adds neutral + deleterious mutation (the mutation logs must be identical as well);
--poisson draws the births per pair from Poisson(2.5) instead of one per pair;
--genome-init assigns the starting genomes on the device (NcclStrips.init_genomes, histograms summed by
all_reduce) instead of uploading them; they must equal the undecomposed assignment before the first step too.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def _run_single_device_genomes(wl, steps, seed, mut, p, genome_seed):
    """_run_single with the starting genomes assigned on the device instead of uploaded."""
    from geonomics_b200.device import DeviceSpecies
    dim, rasters, prm, ga, pop, _ = wl
    dev = DeviceSpecies(dim, rasters, prm, ga, capacity=4 * len(pop['x']), seed=seed)
    try:
        dev.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        dev.init_genomes(p, genome_seed)
        start = dev.download()
        if mut:
            dev.set_mutation(**mut)
        out, logs = [], []
        for _ in range(steps):
            dev.step(1)
            dev.sync()
            out.append(dev.download())
            logs.append(dev.read_mutations() if mut else None)
        return dict(start=start, states=out, records=dev.step_records(), logs=logs)
    finally:
        dev.close()


def main():
    import torch
    import torch.distributed as dist
    from test_cuda_strips import _workload
    from test_cuda_strips_mutation import _mutation, _run_single
    from geonomics_b200 import strips
    pos = [a for a in sys.argv[1:] if not a.startswith('--')]
    steps = int(pos[0]) if pos else 8
    mutation, poisson = '--mutation' in sys.argv, '--poisson' in sys.argv
    genome_init = '--genome-init' in sys.argv
    rank, local = int(os.environ['RANK']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    world = dist.get_world_size()
    wl = _workload(surfaces=True, n=20000, dim=(128, 96), L=200, seed=21)
    dim, rasters, prm, ga, pop, g = wl
    if poisson:
        prm = dict(prm, n_births_fixed=False, lam=2.5)
        wl = (dim, rasters, prm, ga, pop, g)
    mut = _mutation(wl, seed=5, mu=1e-5) if mutation else None
    st = strips.NcclStrips(dim, rasters, prm, ga, capacity=4 * len(pop['x']) // world + 4096, seed=77)
    p = np.random.default_rng(3).random(ga['L'])
    start = None
    if genome_init:
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'])
        st.init_genomes(p, 1234)
        start = st.dev.download()
    else:
        st.upload(pop['x'], pop['y'], pop['age'], pop['sex'], pop['idx'], g=g)
    if mut:
        st.set_mutation(**mut)
    st.step(steps)
    st.sync()
    mine = st.dev.download()
    recs = st.step_records_local()
    log = st.read_mutations() if mut else None
    shares = [None] * world
    dist.all_gather_object(shares, (mine, recs, log, start))
    ok = True
    if rank == 0:
        got = strips.merge_states([s[0] for s in shares])
        got_recs = strips.merge_records([s[1] for s in shares])
        if genome_init:
            single = _run_single_device_genomes(wl, steps, 77, mut, p, 1234)
            got0 = strips.merge_states([s[3] for s in shares])
            ok = all(np.array_equal(single['start'][k], got0[k]) for k in ('idx', 'g', 'z'))
            print('starting genomes assigned on the device over %d GPUs: %s' % (
                world, 'IDENTICAL to the undecomposed assignment' if ok else 'MISMATCH'), flush=True)
        else:
            single = _run_single(wl, steps, seed=77, mut=mut)
        ref, ref_recs = single['states'][-1], single['records']
        ok = ok and np.array_equal(ref['idx'], got['idx'])
        for k in ('x', 'y', 'age', 'sex', 'g', 'z', 'fit'):
            ok = ok and np.array_equal(ref[k], got[k])
        ok = ok and all((a['Nt'], a['n_births'], a['n_deaths'], a['n_pairs']) ==
                        (b['Nt'], b['n_births'], b['n_deaths'], b['n_pairs']) for a, b in zip(ref_recs, got_recs))
        if mut:
            ref_rows = [r for rows, _ in single['logs'] for r in rows]
            ref_state = single['logs'][-1][1]
            for _, _, (rows, state), _ in shares:
                ok = ok and rows == ref_rows and state['n_mutables'] == ref_state['n_mutables']
                ok = ok and all(np.array_equal(state[k], ref_state[k]) for k in ('nonneut_loci', 'delet_loci', 'delet_s'))
        print('strips over %d GPUs (CUDA IPC peer writes; barriers and collectives by gnx_strip_barrier over '
              'peer memory), %d steps: %s; N %d -> %d; per-rank shares %s'
              % (world, steps, 'IDENTICAL to the undecomposed run' if ok else 'MISMATCH', len(pop['x']),
                 len(got['idx']), [len(s[0]['idx']) for s in shares]), flush=True)
    st.close()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()
