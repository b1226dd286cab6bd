"""Check that a Model cut into strips over the ranks of a process group reproduces the undecomposed Model.

    torchrun --nproc-per-node W tools/model_strips_check.py [--params tests/data/params_small.py] [--T 12]
                                                             [--checkpoint-at K]

Every rank builds the parameters with make_model(strips=group) and runs the burn-in and T main steps; the
species-wide series and final state every rank sees are then compared, on rank 0, with the same parameters
run with strips=None.  With --checkpoint-at K the strip model is saved after K main steps instead (Model.save on
every rank), and rank 0 resumes the file on one GPU (load_model, strips=None) for the remaining T - K steps
before the comparison.  Exits non-zero on any difference (on every rank)."""
import argparse
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def observe(model):
    spp = model.comm[0]
    out = dict(burn_t=model.burn_t, burn_mean=spp._burnin_spat_tester.stats['mean'],
               burn_std=spp._burnin_spat_tester.stats['std'], Nt=spp.Nt, n_births=spp.n_births,
               n_deaths=spp.n_deaths)
    for g in ('x', 'y', 'age', 'z', 'fitness', 'genotypes'):
        out[g] = getattr(model, 'get_' + g)()
    out.update(het=spp._calc_het(), ld=spp._calc_ld(), density=spp._calc_density())
    return {k: np.asarray(v) for k, v in out.items()}


def run(params, strips, T, genome_init, save_at=None, path=None):
    """The model after T main steps, or None once it is saved to `path` after save_at of them."""
    from geonomics_b200 import api
    model = api.make_model(params, strips=strips, genome_init=genome_init)
    try:
        model.walk(10 ** 6, 'burn')
        if save_at is None:
            model.walk(T, 'main')
            return observe(model)
        model.walk(save_at, 'main')
        model.save(path)
        return None
    finally:
        for s in model.comm.values():
            s._detach()


def resume(path, steps):
    from geonomics_b200 import api
    model = api.load_model(path)
    try:
        model.walk(steps, 'main')
        return observe(model)
    finally:
        for s in model.comm.values():
            s._detach()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--params', default=os.path.join(ROOT, 'tests', 'data', 'params_small.py'))
    ap.add_argument('--T', type=int, default=12)
    ap.add_argument('--genome-init', default='device', choices=('host', 'device'))
    ap.add_argument('--checkpoint-at', type=int, default=None, metavar='K',
                    help='save the strip model after K main steps and resume it on one GPU')
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from geonomics_b200 import api
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank, world = dist.get_rank(), dist.get_world_size()
    params = api.read_parameters_file(args.params)
    k = args.checkpoint_at
    if k is None:
        got = run(params, dist.group.WORLD, args.T, args.genome_init)
    else:
        assert 0 <= k <= args.T, '--checkpoint-at must lie in [0, T]'
        box = [os.path.join(tempfile.mkdtemp(prefix='gnx_ckpt_'), 'model.ckpt') if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        run(params, dist.group.WORLD, args.T, args.genome_init, save_at=k, path=box[0])
        got = resume(box[0], args.T - k) if rank == 0 else None
        if rank == 0:
            os.remove(box[0])
            os.rmdir(os.path.dirname(box[0]))
    bad = []
    if rank == 0:
        ref = run(api.read_parameters_file(args.params), None, args.T, args.genome_init)
        bad = [k for k in ref if ref[k].shape != got[k].shape or not np.array_equal(ref[k], got[k], equal_nan=True)]
    if k is None:
        # every rank's species-wide view must be rank 0's
        views = [None] * world
        dist.all_gather_object(views, got)
        for r, v in enumerate(views):
            bad += ['rank %d: %s' % (r, k) for k in got if not np.array_equal(v[k], views[0][k], equal_nan=True)]
    verdict = [bad]
    dist.broadcast_object_list(verdict, src=0)
    if rank == 0:
        print('model_strips_check: %d ranks%s, burn_t %d, N %d: %s' % (
            world, '' if k is None else ', saved after %d main steps and resumed on one GPU' % k, int(got['burn_t']),
            int(got['Nt'][-1]), 'equal' if not verdict[0] else 'DIFFER: %s' % verdict[0]))
    dist.destroy_process_group()
    sys.exit(1 if verdict[0] else 0)


if __name__ == '__main__':
    main()
