"""Gauss-Newton Hessian diagonal on one GPU: the two new kernels alone, and on bench.py's C4 workload the four calls
gauss_newton_diagonal, misfit_gradient_and_gauss_newton_diagonal, misfit_and_adjoint_gradient and
misfit_gradient_and_pseudo_hessian, alternated in one run.

    python tools/gauss_newton_diagonal_probe.py [--nfreq 16 --nsrc 256 --reps 3] --out profiles/<name>.json

Kernels: CUDA events around hz_wavefield_lagcorr4 on a random N x S complex128 panel (3.1 GB at C4, far above the 126 MB
L2), once more on an L2-resident panel (40 depths of the same width, 82 MB, repeated) to name the bound, and around
hz_gauss_newton_diag for c (the sparse column: rho is given in the C4 recipe) and for rho (the full column).
Algorithmic bytes: lag correlation N S 16 B read + 41 N 16 B written; contraction 41 N 16 B of C + 13 N 16 B of Gam +
56 N B of model planes read + 8 N B per parameter written.  FLOPs: 8 per complex multiply-add; the lag correlation forms
40 lag products and one |u|^2 per (node, source) (324 flops); the contraction forms, per interior node, 189 complex
products for the sparse c column (81 for row n with itself, 9 for each of the 8 pairs of row n with a neighbour, 1 for
each of the 36 neighbour pairs) and 45 x 81 for a full column, plus one per row pair with Gam.  End to end (workload and
regimes as tools/pseudo_hessian_probe.py): 'refreshed' = updateModel before every call (all frequencies refactored),
'resident' = unchanged model, factors kept; the methods alternated, the first round untimed, host clock around each
call with a device synchronise.  Card name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

import numpy as np  # noqa: E402
from adjoint_gradient_probe import card, events_ms  # noqa: E402

HBM_PEAK_GBS = 7700.          # HGX B200 data sheet, one GPU
HBM_MEASURED_GBS = 6546.      # DESIGN.md §4
FLOP_PER_NODE_SOURCE = 8 * 40 + 4
PRODUCTS_PER_NODE = {'c': 189 + 45, 'rho': 45 * 81 + 45}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--nfreq', type=int, default=16)
    ap.add_argument('--nsrc', type=int, default=256)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--kernel-reps', type=int, default=10)
    ap.add_argument('--out', required=True)
    a = ap.parse_args()
    import torch
    import bench
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    assert torch.cuda.is_available(), 'needs a CUDA device'
    sc, c_true = bench.c4_config(a.nfreq, a.nsrc, a.nsrc)
    nx, nz, S = sc['nx'], sc['nz'], a.nsrc
    N = nx * nz
    rec = {'card': card(), 'workload': 'C4 recipe %dx%d, %d frequencies x %d sources, %d receivers' % (nx, nz, a.nfreq, S, S),
           'hbm_peak_GB_per_s': HBM_PEAK_GBS, 'hbm_measured_GB_per_s': HBM_MEASURED_GBS}
    lib = _lib.get_lib()

    # ---- the kernels alone ----
    g = torch.Generator(device='cuda').manual_seed(0)
    u = torch.randn((N, S), dtype=torch.complex128, device='cuda', generator=g)
    C = torch.empty((41 * N,), dtype=torch.complex128, device='cuda')

    def lag_rate(nz_, u_):
        def lag():
            _lib.check(lib.hz_wavefield_lagcorr4(_lib.ptr(u_), nx, nz_, S, _lib.ptr(C), None))
        events_ms(torch, lag, 2)
        ms = events_ms(torch, lag, a.kernel_reps)
        n_ = nx * nz_
        nbytes, flops = n_ * S * 16 + 41 * n_ * 16, FLOP_PER_NODE_SOURCE * n_ * S
        return {'ms': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms / 1e6, 'flop': flops, 'TFLOP_per_s': flops / ms / 1e9,
                'ns_per_node_source': ms * 1e6 / (n_ * S),
                'roofline_ms_at_measured_hbm': nbytes / HBM_MEASURED_GBS / 1e6}
    rec['wavefield_lagcorr4'] = lag_rate(nz, u)
    rec['wavefield_lagcorr4_l2_resident'] = lag_rate(40, u[:nx * 40])
    hbm, l2 = rec['wavefield_lagcorr4'], rec['wavefield_lagcorr4_l2_resident']
    rec['wavefield_lagcorr4']['bound'] = (
        'HBM' if hbm['ns_per_node_source'] > 1.3 * l2['ns_per_node_source'] else
        'issue (FP64 vector pipe and warp shuffles): the L2-resident panel runs at %.0f%% of the HBM-sized panel\'s '
        'time per (node, source)' % (100 * l2['ns_per_node_source'] / hbm['ns_per_node_source']))
    del u
    torch.cuda.empty_cache()
    d = zb.MiniZephyr(dict({k: v for k, v in sc.items() if k not in ('freqs', 'geom')}, freq=sc['freqs'][0]))
    C.copy_(torch.randn((41 * N,), dtype=torch.complex128, device='cuda', generator=g))
    Gam = torch.randn((13 * N,), dtype=torch.complex128, device='cuda', generator=g)
    h = torch.zeros(N, dtype=torch.float64, device='cuda')
    for k in ('c', 'rho'):
        def gn():
            _lib.check(lib.hz_gauss_newton_diag(d.handle, _lib.ptr(C), _lib.ptr(Gam), None, None,
                                                _lib.ptr(h) if k == 'c' else None, _lib.ptr(h) if k == 'rho' else None), d.handle)
        events_ms(torch, gn, 2)
        ms = events_ms(torch, gn, a.kernel_reps)
        nbytes = 41 * N * 16 + 13 * N * 16 + 56 * N + 8 * N
        flops = 8 * PRODUCTS_PER_NODE[k] * N
        rec['gauss_newton_diag_kernel_' + k] = {'ms': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms / 1e6, 'flop': flops,
                                                'TFLOP_per_s': flops / ms / 1e9,
                                                'roofline_ms_at_measured_hbm': nbytes / HBM_MEASURED_GBS / 1e6}
    d.close()
    del C, Gam, h
    torch.cuda.empty_cache()

    # ---- end to end, alternated ----
    sv_t, pr_t = zb.Helm2DSurvey(dict(sc, c=c_true, Disc=zb.MiniZephyr)), zb.Helm2DProblem(dict(sc, c=c_true, Disc=zb.MiniZephyr))
    pr_t.pair(sv_t)
    dobs = sv_t.dpred().reshape((S, S, a.nfreq))
    pr_t.clearCache()
    del sv_t, pr_t
    torch.cuda.empty_cache()
    sv, pr = zb.Helm2DSurvey(dict(sc, Disc=zb.MiniZephyr)), zb.Helm2DProblem(dict(sc, Disc=zb.MiniZephyr))
    pr.pair(sv)
    dobs_dev = pr.upload_dobs(dobs)
    c0 = sc['c']
    calls = {'gauss_newton_diagonal': lambda: pr.gauss_newton_diagonal(),
             'gradient_and_gauss_newton_diagonal': lambda: pr.misfit_gradient_and_gauss_newton_diagonal(dobs_dev),
             'adjoint_gradient': lambda: pr.misfit_and_adjoint_gradient(dobs_dev),
             'gradient_and_pseudo_hessian': lambda: pr.misfit_gradient_and_pseudo_hessian(dobs_dev)}
    step = [0]
    for regime in ('refreshed', 'resident'):
        times = {k: [] for k in calls}
        for rep in range(a.reps + 1):
            for k, fn in calls.items():
                if regime == 'refreshed':
                    step[0] += 1
                    pr.updateModel(c0 * (1. + 1e-6 * step[0]))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = fn()
                torch.cuda.synchronize()
                if rep:
                    times[k].append(time.perf_counter() - t0)
                if k == 'gauss_newton_diagonal':
                    hc = res['c']
                    rec.setdefault('H_c_min_over_max_' + regime, float(hc.min() / hc.max()))
        rec['step_s_' + regime] = {k: {'s': v, 'median_s': float(np.median(v)), 'spread_s': float(max(v) - min(v))}
                                   for k, v in times.items()}
        med = {k: v['median_s'] for k, v in rec['step_s_' + regime].items()}
        rec['ratio_fused_over_gradient_' + regime] = med['gradient_and_gauss_newton_diagonal'] / med['adjoint_gradient']
    rec['note'] = ('kernels: CUDA events over %d launches after 2 untimed ones; step_s_*: host clock around the calls with '
                   'device synchronise, methods alternated, first round untimed' % a.kernel_reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: rec[k] for k in ('card', 'wavefield_lagcorr4', 'wavefield_lagcorr4_l2_resident',
                                          'gauss_newton_diag_kernel_c', 'gauss_newton_diag_kernel_rho')}))
    for regime in ('refreshed', 'resident'):
        print(regime, json.dumps({k: v['median_s'] for k, v in rec['step_s_' + regime].items()}),
              'fused/gradient', rec['ratio_fused_over_gradient_' + regime])


if __name__ == '__main__':
    main()
