"""Born modelling and Gauss-Newton products on one GPU: gauss_newton_hvec against misfit_and_adjoint_gradient and
born_dpred on bench.py's C4 workload, alternated in one run; the two new kernels alone; a per-phase breakdown of one
frequency.

    python tools/born_probe.py [--nfreq 16 --nsrc 256 --reps 3] --out profiles/<name>.json

Workload: bench.py's C4 (MiniZephyr 500 x 1500, seed-0 layered model, 16 frequencies, 256 sources and receivers);
observed data from the model with bench's -10 % blob; dm a smooth velocity perturbation.  Two end-to-end regimes, each
with the three methods alternated and the first round untimed, host clock around the call and a device synchronise:
'refreshed': updateModel with a new velocity before every call (every call refactors all frequencies, as bench.py's C4
step and the gradient probe); 'resident': the model is unchanged and the factors stay in HBM (the inner loop of a
truncated Gauss-Newton / CG solve).  Kernels: CUDA events around hz_stencil_apply on two N x S complex128 panels (2 x
3.1 GB at C4, far above the 126 MB L2) and around hz_assemble_jvp; achieved bandwidth = algorithmic bytes over kernel
time (apply: N S 16 B read + N S 16 B written + 9 N 16 B of dcoef; JVP: 9 N 16 B written + 56 N B of model and
perturbation planes read).  Card name and power limit are read in the same run.
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
           'hbm_peak_GB_per_s': HBM_PEAK_GBS}
    lib = _lib.get_lib()

    # ---- the kernels alone ----
    g = torch.Generator(device='cuda').manual_seed(0)
    u = torch.randn((N, S), dtype=torch.complex128, device='cuda', generator=g)
    P = torch.randn((9 * N,), dtype=torch.complex128, device='cuda', generator=g)
    out = torch.empty((N, S), dtype=torch.complex128, device='cuda')

    def apply():
        _lib.check(lib.hz_stencil_apply(_lib.ptr(P), _lib.ptr(u), nx, nz, S, -1., 0., _lib.ptr(out), None))
    events_ms(torch, apply, 2)
    ms = events_ms(torch, apply, a.kernel_reps)
    nbytes = 2 * N * S * 16 + 9 * N * 16
    rec['stencil_apply'] = {'ms': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms / 1e6, 'roofline_ms_at_hbm_peak': nbytes / HBM_PEAK_GBS / 1e6}
    del u, out
    torch.cuda.empty_cache()
    d = zb.MiniZephyr(dict({k: v for k, v in sc.items() if k not in ('freqs', 'geom')}, freq=sc['freqs'][0]))
    dc = torch.randn((N,), dtype=torch.float64, device='cuda', generator=g)
    dr = torch.randn((N,), dtype=torch.float64, device='cuda', generator=g)

    def jvp():
        _lib.check(lib.hz_assemble_jvp(d.handle, _lib.ptr(dc), _lib.ptr(dr), None, _lib.ptr(P)), d.handle)
    events_ms(torch, jvp, 2)
    ms = events_ms(torch, jvp, a.kernel_reps)
    nbytes = 9 * N * 16 + (16 + 16 + 8 + 8 + 8) * N
    rec['assemble_jvp'] = {'ms': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms / 1e6, 'roofline_ms_at_hbm_peak': nbytes / HBM_PEAK_GBS / 1e6}
    d.close()
    del P, dc, dr
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
    zz, xx = np.mgrid[0:nz, 0:nx]
    dm = {'c': (50. * np.sin(np.pi * zz / nz * 3.) * np.cos(np.pi * xx / nx * 2.)).ravel()}
    calls = {'adjoint_gradient': lambda: pr.misfit_and_adjoint_gradient(dobs_dev, to_host=False),
             'born_dpred': lambda: pr.born_dpred(dm),
             'gauss_newton_hvec': lambda: pr.gauss_newton_hvec(dm)}
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
                fn()
                torch.cuda.synchronize()
                if rep:
                    times[k].append(time.perf_counter() - t0)
        rec['step_s_' + regime] = {k: {'s': v, 'median_s': float(np.median(v)), 'spread_s': float(max(v) - min(v))}
                                   for k, v in times.items()}
        med = {k: v['median_s'] for k, v in rec['step_s_' + regime].items()}
        rec['ratio_gn_over_gradient_' + regime] = med['gauss_newton_hvec'] / med['adjoint_gradient']

    # ---- per-phase breakdown of one frequency, factors resident, one stream ----
    ifreq = pr.system.localFreqIndices[0]
    sub = pr.system.subProblems[ifreq]
    ops = pr._device_ops()
    uF = pr.forward_device(ifreq)
    dU, lam = torch.empty_like(uF), torch.empty_like(uF)
    P = torch.empty((9 * N,), dtype=torch.complex128, device='cuda')
    dct = torch.from_numpy(dm['c']).cuda()
    gc = torch.zeros((N,), dtype=torch.float64, device='cuda')
    v = pr.extract_device(uF)
    taps = pr._adjoint_taps(ifreq)

    def born_jvp():
        sub._bind_stream()
        _lib.check(lib.hz_assemble_jvp(sub.handle, _lib.ptr(dct), None, None, _lib.ptr(P)), sub.handle)
    phases = {
        'forward_solve': lambda: pr.forward_device(ifreq, out=uF),
        'assemble_jvp': born_jvp,
        'stencil_apply': lambda: _lib.check(lib.hz_stencil_apply(_lib.ptr(P), _lib.ptr(uF), nx, nz, S, -1., 0., _lib.ptr(dU), None)),
        'born_N_solve_full_depth': lambda: sub.solve_device(dU, (-1, -1)),
        'adjoint_source_T_solve': lambda: pr.backproject_device(ifreq, v, out=lam, vals=taps, conjugate=False, trans='T'),
        'xcorr': lambda: _lib.check(lib.hz_stencil_xcorr(_lib.ptr(lam), _lib.ptr(uF), nx, nz, S, _lib.ptr(P), None)),
        'vjp': lambda: _lib.check(lib.hz_assemble_vjp(sub.handle, _lib.ptr(P), None, _lib.ptr(gc), None), sub.handle),
    }
    ph = {k: [] for k in phases}
    for rnd in range(4):
        for k, fn in phases.items():
            t = events_ms(torch, fn, 1)
            if rnd:
                ph[k].append(t)
    rec['phases_ms_one_frequency'] = {k: {'ms': v_, 'median_ms': float(np.median(v_))} for k, v_ in ph.items()}
    rec['source_depth_range'] = list(ops['s_z'])
    rec['note'] = ('step_s_*: host clock around the calls with device synchronise, methods alternated, first round untimed; '
                   'refreshed = updateModel before every call (all frequencies refactored), resident = unchanged model, '
                   'factors kept; kernels: CUDA events over %d launches after 2 untimed ones; phases: CUDA events around '
                   'each phase of the first frequency on one stream, factors resident, 3 timed rounds; the end-to-end calls '
                   'run up to 4 frequencies concurrently, so phase sums are not call times' % a.kernel_reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: rec[k] for k in ('card', 'stencil_apply', 'assemble_jvp')}))
    for regime in ('refreshed', 'resident'):
        print(regime, json.dumps({k: v['median_s'] for k, v in rec['step_s_' + regime].items()}),
              'GN/gradient', rec['ratio_gn_over_gradient_' + regime])
    print(json.dumps({k: v['median_ms'] for k, v in rec['phases_ms_one_frequency'].items()}))


if __name__ == '__main__':
    main()
