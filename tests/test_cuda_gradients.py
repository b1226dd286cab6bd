"""The gradient solve of the density interpolant (`_estimate_gradients_2d_global` as griddata calls it), bit for
bit.  Density feeds the death draws, so no rounding of the solve may change; the oracle parity tests compare
with rtol = 1e-6 and would not see one.  The sweep is restated here in Python with the device's exact
operation sequence (every FMA rounded once, emulated in integer arithmetic), and the device's values,
gradients and iteration counts must equal it exactly:
  * on the c2 lattice (23 x 23) and the c4 lattice (21 x 21) with counts of a real population after a
    few steps;
  * with an empty region, so that some counts are zero;
  * on the largest lattice the register-resident kernel accepts (GS_REG_PTS = 640 vertices: 3 x 213 = 639
    points, as lattices are odd x odd), where its CTA has 20 warps at 96 registers, the whole register file.
The next lattice (3 x 215 = 645 points) goes to the general CSR kernel, checked against scipy.  Every case
also asserts, from a profiler trace of the last step, which of the two kernels ran."""
import json
import math
import os
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MAXITER, TOL = 400, 1e-6          # CloughTocher2DInterpolator defaults, as griddata reaches them


def fma(a, b, c):
    """a*b + c rounded once to nearest (IEEE 754 fusedMultiplyAdd) for finite doubles."""
    na, da = a.as_integer_ratio()
    nb, db = b.as_integer_ratio()
    nc, dc = c.as_integer_ratio()
    num = na * nb * dc + nc * da * db
    if num == 0:                  # exact zero: -0 only when the product and c are both -0
        neg = a * b == 0 and c == 0 and math.copysign(1.0, a) * math.copysign(1.0, b) < 0 \
            and math.copysign(1.0, c) < 0
        return -0.0 if neg else 0.0
    return num / (da * db * dc)   # int / int is correctly rounded


def tables(dens):
    """The host's per-vertex tables (gnx_set_density): 8 slots padded with (self, zero weights), 2x2 inverse."""
    P = dens.points
    ip, ix = dens.nbr_indptr, dens.nbr_indices
    n = len(P)
    nb = [[i] * 8 for i in range(n)]
    E = [[(0.0, 0.0, 0.0, 0.0)] * 8 for _ in range(n)]
    inv = []
    for i in range(n):
        Q0 = Q1 = Q3 = 0.0
        for k, jj in enumerate(range(ip[i], ip[i + 1])):
            j = int(ix[jj])
            x, y = float(P[j, 0]) - float(P[i, 0]), float(P[j, 1]) - float(P[i, 1])
            L = math.sqrt(x * x + y * y)
            L3 = L * L * L
            nb[i][k] = j
            E[i][k] = (x, y, x / L3, y / L3)
            Q0 += 4 * x * x / L3
            Q1 += 4 * x * y / L3
            Q3 += 4 * y * y / L3
        det = Q0 * Q3 - Q1 * Q1
        inv.append((Q3 / det, -Q1 / det, Q0 / det))
    return nb, E, inv


def solve(dens, counts, tab):
    """Gauss-Seidel in vertex order (= the 4 colour phases), in the kernel's rounding sequence."""
    nb, E, inv = tab
    f = (counts.astype(np.float64) / dens.areas).tolist()
    y = [(0.0, 0.0)] * len(f)
    offs = np.concatenate([[0], np.cumsum([a * b for a, b in dens.grid_shape])]).tolist()
    for it in range(MAXITER):
        err = 0.0
        for v in range(offs[4]):
            f1, s0, s1 = f[v], 0.0, 0.0
            for k in range(8):
                j = nb[v][k]
                ex, ey, wx, wy = E[v][k]
                q = fma(ex, y[j][0], ey * y[j][1])
                tt = fma(f1 - f[j], 6.0, q + q)
                s0 = fma(tt, wx, s0)
                s1 = fma(tt, wy, s1)
            i00, i01, i11 = inv[v]
            r0 = fma(i00, s0, i01 * s1)
            r1 = fma(i01, s0, i11 * s1)
            change = max(abs(y[v][0] + r0), abs(y[v][1] + r1))
            y[v] = (-r0, -r1)
            err = max(err, change / max(1.0, abs(r0), abs(r1)))
        if err < TOL:
            return np.array(f), np.array(y), it + 1
    return np.array(f), np.array(y), 0


def traced_kernels(dev):
    """One step under torch.profiler -> the names of the kernels it launched."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.step(1, sync=True)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory(prefix='gnx_grad_') as td:
        path = os.path.join(td, 'trace.json')
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)['traceEvents']
    return {e['name'].split('(')[0].replace('void ', '').strip() for e in events if e.get('cat') == 'kernel'}


def device_solve(cfg, steps, window_width=None, x_min=None):
    """A workload's population after `steps` graph-launched steps (the last one traced): the counts, values,
    gradients and iteration counts of the last step's solve, and which gradient kernel it ran."""
    from geonomics_b200 import workloads
    from geonomics_b200.device import DeviceSpecies
    w = workloads.build(cfg, cfg['seed'])
    prm = dict(w['prm'], density_grid_window_width=window_width)
    x = w['pop']['x']
    if x_min is not None:                 # nobody left of x_min: zero counts there
        x = x_min + x * (cfg['dim'][0] - 0.001 - x_min) / cfg['dim'][0]
    N0 = cfg['N']
    dev = DeviceSpecies(w['land_dim'], w['rasters'], prm, w['gen_arch'], capacity=int(1.5 * N0) + 4096,
                        seed=cfg['seed'])
    try:
        dev.upload(x, w['pop']['y'], w['pop']['age'], w['pop']['sex'], w['pop']['idx'],
                   genomes_packed=workloads.random_packed_genomes(N0, w['L'], cfg['seed'] + 1))
        dev.step(steps - 1, sync=True)
        names = traced_kernels(dev)
        n = len(dev.density.points)
        out = {'dens': dev.density, 'iters': dev.counters()['gs_iters'],
               'gradient_kernels': sorted(k for k in names if k.startswith('k_ct_gradients'))}
        for k, name in enumerate(('N', 'P')):
            out['counts_' + name] = dev.read('COUNTS_' + name, n)
            out['vals_' + name] = dev.read('VALS_' + name, n)
            out['grad_' + name] = dev.read('GRAD_' + name, 2 * n).reshape(n, 2)
        return out
    finally:
        dev.close()


def assert_bitwise(out):
    assert out['gradient_kernels'] == ['k_ct_gradients_reg'], out['gradient_kernels']
    tab = tables(out['dens'])
    for k, name in enumerate(('N', 'P')):
        f, y, iters = solve(out['dens'], out['counts_' + name], tab)
        assert iters > 0 and out['iters'][k] == iters, (name, out['iters'], iters)
        assert np.array_equal(out['vals_' + name].view(np.uint64), f.view(np.uint64)), name
        assert np.array_equal(out['grad_' + name].view(np.uint64), y.view(np.uint64)), name


def _cfg(name, **kw):
    from geonomics_b200 import workloads
    return dict(workloads.CONFIGS[name], **kw)


def test_c2_lattice():
    out = device_solve(_cfg('c2'), 3)
    assert len(out['dens'].points) == 529
    assert_bitwise(out)
    # the restatement itself is scipy's solve
    from scipy.interpolate import CloughTocher2DInterpolator
    d = out['dens']
    ref = CloughTocher2DInterpolator(d.points, out['vals_N'], tol=TOL, maxiter=MAXITER).grad.reshape(-1, 2)
    np.testing.assert_allclose(out['grad_N'], ref, rtol=1e-9, atol=1e-12 * np.abs(ref).max())


def test_c4_lattice():
    # c4's landscape and window with a lighter population and genome: the lattice depends on the dimensions only
    out = device_solve(_cfg('c4', N=1_000_000, L=100, surfaces=False), 3)
    assert len(out['dens'].points) == 441
    assert_bitwise(out)


def test_empty_region():
    out = device_solve(_cfg('c2', dim=(600, 300), N=100_000), 2, x_min=300.0)
    assert (out['counts_N'] == 0).sum() > len(out['counts_N']) // 4
    assert (out['counts_N'] > 0).sum() > len(out['counts_N']) // 4
    assert_bitwise(out)


def test_largest_register_lattice():
    out = device_solve(_cfg('c2', dim=(1060, 10), N=20_000), 2, window_width=10)
    d = out['dens']
    assert len(d.points) == 639 and d.colourable and np.diff(d.nbr_indptr).max() <= 8
    assert_bitwise(out)


def test_first_lattice_beyond_the_register_kernel_uses_the_csr_kernel():
    from scipy.interpolate import CloughTocher2DInterpolator
    out = device_solve(_cfg('c2', dim=(1070, 10), N=20_000), 2, window_width=10)
    d = out['dens']
    # colourable and of degree <= 8: only the vertex count sends it to the general kernel
    assert len(d.points) == 645 and d.colourable and np.diff(d.nbr_indptr).max() <= 8
    assert out['gradient_kernels'] == ['k_ct_gradients'], out['gradient_kernels']
    for name in ('N', 'P'):
        assert np.array_equal(out['vals_' + name], out['counts_' + name] / d.areas)
        ref = CloughTocher2DInterpolator(d.points, out['vals_' + name], tol=TOL, maxiter=MAXITER).grad.reshape(-1, 2)
        np.testing.assert_allclose(out['grad_' + name], ref, rtol=1e-9, atol=1e-12 * max(np.abs(ref).max(), 1.0))
