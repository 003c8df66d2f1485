"""Adjoint-state gradient on one GPU: misfit_and_adjoint_gradient against misfit_and_gradient (the reference's Jtvec
formula) on bench.py's C4 workload, alternated in one run; the two new kernels alone; a Taylor test at C4.

    python tools/adjoint_gradient_probe.py [--nfreq 16 --nsrc 256 --reps 8] --out profiles/<name>.json

Workload: bench.py's C4 (MiniZephyr 500 x 1500, seed-0 layered model, 16 frequencies, 256 sources and receivers);
observed data from the model with bench's -10 % blob.  Each timed call follows bench.py's C4 step: updateModel with a
new velocity (so every call refactors all frequencies), then the gradient call with the observed data resident on the
device (upload_dobs), host clock around the call and a device synchronise.  The two methods alternate.  Kernels: CUDA
events around hz_stencil_xcorr on two random N x S complex128 panels (2 x 3.1 GB at C4, far above the 126 MB L2) and
around hz_assemble_vjp; achieved bandwidth = algorithmic bytes (2 N S 16 B read + 9 N 16 B written; VJP: 9 N 16 B of
G + 40 N B of model planes read, 16 N B written) over kernel time.  Per-phase breakdown of one frequency with its factors
resident (forward solve; back-projection + A solve + gradient_kernel of the reference formula; adjoint source + A^T
solve + cross-correlation + VJP of the adjoint-state gradient), CUDA events, phases alternated.  Card name and power
limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

import numpy as np  # noqa: E402


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(',')]
        return {'name': name, 'power_limit': plim, 'max_sm_clock': clk}
    except Exception as e:                                   # noqa: BLE001 -- the record says what failed
        import torch
        return {'name': torch.cuda.get_device_name(0), 'power_limit': 'unknown (%s)' % e}


def events_ms(torch, fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--nfreq', type=int, default=16)
    ap.add_argument('--nsrc', type=int, default=256)
    ap.add_argument('--reps', type=int, default=8)
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
    rec = {'card': card(), 'workload': 'C4 recipe %dx%d, %d frequencies x %d sources, %d receivers' % (nx, nz, a.nfreq, S, S)}
    lib = _lib.get_lib()

    # ---- the kernels alone ----
    g = torch.Generator(device='cuda').manual_seed(0)
    lam = torch.randn((N, S), dtype=torch.complex128, device='cuda', generator=g)
    u = torch.randn((N, S), dtype=torch.complex128, device='cuda', generator=g)
    G = torch.empty((9 * N,), dtype=torch.complex128, device='cuda')

    def xcorr():
        _lib.check(lib.hz_stencil_xcorr(_lib.ptr(lam), _lib.ptr(u), nx, nz, S, _lib.ptr(G), None))
    events_ms(torch, xcorr, 2)
    ms = events_ms(torch, xcorr, a.kernel_reps)
    nbytes = 2 * N * S * 16 + 9 * N * 16
    rec['xcorr'] = {'ms': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms / 1e6}
    del lam, u
    torch.cuda.empty_cache()
    d = zb.MiniZephyr(dict({k: v for k, v in sc.items() if k not in ('freqs', 'geom')}, freq=sc['freqs'][0]))
    gc, gr = torch.zeros(N, dtype=torch.float64, device='cuda'), torch.zeros(N, dtype=torch.float64, device='cuda')

    def vjp():
        _lib.check(lib.hz_assemble_vjp(d.handle, _lib.ptr(G), None, _lib.ptr(gc), _lib.ptr(gr)), d.handle)
    events_ms(torch, vjp, 2)
    ms = events_ms(torch, vjp, a.kernel_reps)
    nbytes = 9 * N * 16 + 40 * N + 16 * N
    rec['vjp'] = {'ms': ms, 'bytes': nbytes, 'GB_per_s': nbytes / ms / 1e6}
    d.close()
    del G, gc, gr
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
    calls = {'reference_formula': lambda: pr.misfit_and_gradient(dobs_dev, to_host=False),
             'adjoint_state': lambda: pr.misfit_and_adjoint_gradient(dobs_dev, to_host=False)}
    times = {k: [] for k in calls}
    step = [0]
    for rep in range(a.reps + 1):
        for k, fn in calls.items():
            step[0] += 1
            pr.updateModel(c0 * (1. + 1e-6 * step[0]))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            if rep:
                times[k].append(time.perf_counter() - t0)
    rec['step_s'] = {k: {'s': v, 'median_s': float(np.median(v))} for k, v in times.items()}
    rec['ratio_adjoint_over_reference'] = rec['step_s']['adjoint_state']['median_s'] / rec['step_s']['reference_formula']['median_s']

    # ---- Taylor test at C4 ----
    pr.updateModel(c0)
    phi0, grad = pr.misfit_and_adjoint_gradient(dobs_dev)
    zz, xx = np.mgrid[0:nz, 0:nx]
    dc = 50. * np.sin(np.pi * zz / nz * 3.) * np.cos(np.pi * xx / nx * 2.)
    gd = float(grad['c'] @ dc.ravel())
    hs = [0.4, 0.2, 0.1, 0.05]
    rem = []
    for h in hs:
        pr.updateModel(c0 + h * dc)
        rem.append(abs(pr.misfit_and_adjoint_gradient(dobs_dev)[0] - phi0 - h * gd))
    rec['taylor'] = {'h': hs, 'remainder': rem, 'phi0': phi0, 'g_dot_dc': gd,
                     'slopes': list(np.diff(np.log(rem)) / np.diff(np.log(hs)))}
    # ---- per-phase breakdown of one frequency, factors resident, one stream ----
    ifreq = pr.system.localFreqIndices[0]
    lib = _lib.get_lib()
    uF = pr.forward_device(ifreq)
    v = pr.extract_device(uF) - dobs_dev[0]
    uB, lam = torch.empty_like(uF), torch.empty_like(uF)
    G = torch.empty((9 * N,), dtype=torch.complex128, device='cuda')
    scaler = torch.ones((N,), dtype=torch.complex128, device='cuda')
    acc = torch.zeros((N,), dtype=torch.complex128, device='cuda')
    gc = torch.zeros((N,), dtype=torch.float64, device='cuda')
    sub = pr.system.subProblems[ifreq]
    taps = pr._adjoint_taps(ifreq)
    phases = {
        'forward_solve': lambda: pr.forward_device(ifreq, out=uF),
        'backproject_N_solve': lambda: pr.backproject_device(ifreq, v, out=uB),
        'gradient_kernel': lambda: _lib.check(lib.hz_gradient(_lib.ptr(uF), _lib.ptr(uB), N, S, _lib.ptr(scaler), _lib.ptr(acc), None)),
        'adjoint_source_T_solve': lambda: pr.backproject_device(ifreq, v, out=lam, vals=taps, conjugate=False, trans='T'),
        'xcorr': lambda: _lib.check(lib.hz_stencil_xcorr(_lib.ptr(lam), _lib.ptr(uF), nx, nz, S, _lib.ptr(G), None)),
        'vjp': lambda: _lib.check(lib.hz_assemble_vjp(sub.handle, _lib.ptr(G), None, _lib.ptr(gc), None), sub.handle),
    }
    ph = {k: [] for k in phases}
    for rnd in range(4):
        for k, fn in phases.items():
            t = events_ms(torch, fn, 1)
            if rnd:
                ph[k].append(t)
    rec['phases_ms_one_frequency'] = {k: {'ms': v_, 'median_ms': float(np.median(v_))} for k, v_ in ph.items()}
    m = {k: float(np.median(v_)) for k, v_ in ph.items()}
    rec['phase_extra_ms_per_frequency'] = (m['adjoint_source_T_solve'] + m['xcorr'] + m['vjp']) - (m['backproject_N_solve'] + m['gradient_kernel'])
    rec['note'] = ('step_s: host clock around updateModel-refreshed gradient calls with device synchronise, methods alternated, '
                   'first round untimed; kernels: CUDA events over %d launches after 2 untimed ones; phases: CUDA events around '
                   'each phase of the first frequency on one stream, factors resident, phases alternated over 3 timed rounds; the '
                   'end-to-end steps run up to 4 frequencies concurrently, so phase sums are not step times' % a.kernel_reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: rec[k] for k in ('card', 'xcorr', 'vjp', 'ratio_adjoint_over_reference')}))
    print(json.dumps({k: v['median_s'] for k, v in rec['step_s'].items()}), 'taylor slopes', rec['taylor']['slopes'])
    print(json.dumps({k: v['median_ms'] for k, v in rec['phases_ms_one_frequency'].items()}), 'extra ms/freq',
          rec['phase_extra_ms_per_frequency'])
    del out


if __name__ == '__main__':
    main()
