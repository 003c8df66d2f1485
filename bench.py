#!/usr/bin/env python
"""Benchmark of the Helmholtz forward hot path on B200 (contract: see the build brief, section 4).

A "step" = one pass of the hot path over one batch of synthetic input for this rank's frequency:
assemble stencil+PML coefficients -> block factorisation -> substitution for ALL sources at once
-> conjugate -> receiver extraction.  Workload (SURVEY.md 8(d) "C3", the configuration
BASELINE.json's target is quoted on): MiniZephyr 1000x3000 grid, dx=dz=10 m, random-layered
velocity, 512 sources / 512 receivers, one frequency per GPU (weak scaling: N GPUs run the first
N of linspace(2,9,8) Hz).  `value` = source-frequency wavefields per second, whole job.

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--nx --nz --nsrc] [--dump-outputs DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault('OPENBLAS_NUM_THREADS', '1')
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')      # see zephyr_b200/__init__.py: must precede CUDA context creation

import numpy as np  # noqa: E402

METRIC = 'source-frequency wavefields/sec'
UNIT = 'wavefields/s'
NOMINAL_FP64_TFLOPS = 148 * 128 * 1.965e9 / 1e12      # 148 SMs x 128 flop/clk x max SM clock
DUMP_BYTES = 64 << 20                                 # --dump-outputs: at most this much per rank


def layered_model(nx, nz, rng, lo=1500., hi=4500., tmin=5, tmax=50):
    c = np.empty((nz, nx))
    z = 0
    while z < nz:
        t = int(rng.integers(tmin, tmax + 1))
        c[z:z + t, :] = rng.uniform(lo, hi)
        z += t
    return c


def c3_config(nx, nz, nsrc, nrec, nfreq, npml=20):
    """SURVEY.md 8(d) C3 recipe (seed 0)."""
    rng = np.random.default_rng(0)
    dx = 10.
    c = layered_model(nx, nz, rng)
    xs = np.round(np.linspace(0.025 * nx, 0.975 * nx, nsrc)) * dx
    xr = np.round(np.linspace(0.025 * nx, 0.975 * nx, nrec)) * dx
    zs = float(min(npml + 5, nz - 2)) * dx
    src = np.stack([xs, np.full(nsrc, zs)], 1)
    rec = np.stack([xr, np.full(nrec, zs + dx)], 1)
    freqs = list(np.linspace(2., 9., 8)[:nfreq]) if nfreq <= 8 else list(np.linspace(2., 9., nfreq))
    return {'nx': nx, 'nz': nz, 'dx': dx, 'dz': dx, 'c': c, 'rho': 1., 'nPML': npml, 'freqs': freqs,
            'geom': {'src': src, 'rec': rec, 'mode': 'fixed'}}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port: numpy assembly + scipy SuperLU) on a bounded sample
# ------------------------------------------------------------------------------------------------
def _cpu_sample(args):
    """One frequency of the sample workload on one core; returns (t_assemble+factor, t_per_rhs, nrhs)."""
    nx, nz_s, nrhs, freq, npml = args
    from oracle import helm_oracle as ho
    sc = c3_config(nx, nz_s, nrhs, nrhs, 1, npml)
    sc['freq'] = freq
    q = ho.sparse_kaiser_source(sc, sc['geom']['src'])
    t0 = time.perf_counter()
    d = ho.OracleDisc(sc, 'MiniZephyr')
    d.factor()
    t1 = time.perf_counter()
    u = d * q
    t2 = time.perf_counter()
    assert np.isfinite(u).all()
    return (t1 - t0, (t2 - t1) / nrhs, nrhs)


def cpu_throughput(nx, nz, nsrc, freqs, nz_sample, nrhs, npml, procs, ratios=(1., 1.)):
    """Extrapolated whole-workload CPU throughput: costs scaled linearly in nz (optimistic for the
    CPU: SuperLU fill grows faster than linearly) and in the number of sources.  `ratios` = measured cost per row
    of a >= 1000-row slab relative to the nz_sample-row slab (factor, solve), see cpu_depth_calibration."""
    import multiprocessing as mp
    jobs = [(nx, nz_sample, nrhs, f, npml) for f in freqs]
    t0 = time.perf_counter()
    if procs > 1:
        with mp.get_context('fork').Pool(procs) as pool:
            res = pool.map(_cpu_sample, jobs)
    else:
        res = [_cpu_sample(j) for j in jobs]
    wall = time.perf_counter() - t0
    scale = nz / float(nz_sample)
    per_freq = [scale * (ratios[0] * tf + nsrc * ratios[1] * ts) for tf, ts, _ in res]
    waves = (len(freqs) + procs - 1) // procs
    t_full = waves * max(per_freq)
    return len(freqs) * nsrc / t_full, wall, res


SURVEY_FULL_C3 = (242.7, 1.60)      # SURVEY.md section 6: splu factor s, solve s per RHS at 1000 x 3000, measured in the build container


def cpu_depth_calibration(nx, nz, freq, npml, nz_small, nz_big=1000, nrhs=16):
    """BASELINE.md section 3 asks for the full factorisation of one frequency (243 s, 26 GB at C3) -- too long for a
    bench that must end within minutes.  The steps therefore time an nz_small-row slab and scale linearly in depth,
    which flatters SuperLU (its fill grows faster than linearly).  This calibration times ONE slab of >= 1000 rows
    with a 16-column panel and returns how much more a row costs there than in the small slab:
    (factor ratio, per-RHS solve ratio, seconds spent, the big-slab timings)."""
    t0 = time.perf_counter()
    tf_b, ts_b, _ = _cpu_sample((nx, nz_big, nrhs, freq, npml))
    tf_s, ts_s, _ = _cpu_sample((nx, nz_small, min(nrhs, 8), freq, npml))
    per_row = lambda t, n: t / float(n)
    return (per_row(tf_b, nz_big) / per_row(tf_s, nz_small), per_row(ts_b, nz_big) / per_row(ts_s, nz_small),
            time.perf_counter() - t0, (tf_b, ts_b))


def run_reference(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    n = a.gpus
    nfreq = n
    freqs = list(np.linspace(2., 9., 8)[:nfreq])
    procs = max(1, min(nfreq, os.cpu_count() or 1))
    for _ in range(a.warmup if a.warmup < 2 else 1):           # one warm pass is enough for a CPU code
        cpu_throughput(a.nx, a.nz, a.nsrc, freqs, max(40, a.ref_nz // 2), 4, a.npml, procs)
    # depth calibration (once, before the steps): cost per row in a >= 1000-row slab relative to the ref_nz-row slab
    big = min(1000, a.nz)
    cal, ratios = None, (1., 1.)
    if not a.no_calibration and big > a.ref_nz:
        rf, rs, cal_s, (tf_b, ts_b) = cpu_depth_calibration(a.nx, a.nz, freqs[0], a.npml, a.ref_nz, big)
        ratios = (rf, rs)
        t_survey = SURVEY_FULL_C3[0] + a.nsrc * SURVEY_FULL_C3[1]
        cal = {'rows': big, 'nrhs': 16, 'factor_s': tf_b, 'solve_s_per_rhs': ts_b, 'per_row_cost_vs_step_slab': {'factor': rf, 'solve': rs}, 'cpu_s': cal_s,
               'remaining_bias': ('linear from %d to %d rows; SURVEY.md section 6 measured the full operator in the build container at %.1f s factor '
                                  '+ %.2f s per RHS = %.2f wavefields/s per core' % (big, a.nz, SURVEY_FULL_C3[0], SURVEY_FULL_C3[1], a.nsrc / t_survey))
               if (a.nx, a.nz) == (1000, 3000) else 'linear beyond the calibrated slab'}
    vals, walls, lin = [], [], []
    for _ in range(a.steps):
        v, w, res = cpu_throughput(a.nx, a.nz, a.nsrc, freqs, a.ref_nz, a.ref_nrhs, a.npml, procs, ratios)
        vals.append(v)
        walls.append(w)
        lin.append(v * max(ratios[0] * tf + a.nsrc * ratios[1] * ts for tf, ts, _ in res) / max(tf + a.nsrc * ts for tf, ts, _ in res))
    v = float(np.mean(vals))
    if cal is not None:
        cal['value_without_calibration'] = float(np.mean(lin))
    sample = ('oracle port (numpy assembly + scipy SuperLU splu), nx=%d; each step times an nz=%d slab (of %d) with %d RHS per frequency; per-row costs '
              'are corrected by the ratio measured once on a %d-row slab with a 16-column panel (BASELINE.md section 3), then scaled linearly to nz=%d '
              'and %d sources (extrapolated; still optimistic for the CPU); %d process(es): the reference\'s only parallel axis is the frequency Pool '
              '(backend/distributors.py:74-96), SuperLU itself is serial' % (a.nx, a.ref_nz, a.nz, a.ref_nrhs, big, a.nz, a.nsrc, procs))
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': n, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': 1e3 * nfreq * a.nsrc / v, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'c128', 'data': 'synthetic', 'config': workload_config(a, nfreq),
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': procs, 'kind': 'port', 'sample': sample,
                             'sample_wall_s': float(np.mean(walls)), 'calibration': cal},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line))
    return 0


def c2_config(nfreq_per_rank, world):
    """SURVEY.md 8(d) C2 recipe: Eurus 200x400, dx=dz=10 m, layered TTI model, freqs 4..10 Hz, 64 sources."""
    rng = np.random.default_rng(0)
    nx, nz, dx = 200, 400, 10.
    c = layered_model(nx, nz, rng, 2000., 3500., 5, 40)
    th = layered_model(nx, nz, rng, 0., 0.3, 5, 40)
    ep = layered_model(nx, nz, rng, 0., 0.2, 5, 40)
    de = layered_model(nx, nz, rng, 0., 0.1, 5, 40)
    xs = np.round(np.linspace(20, 180, 64)) * dx
    xr = np.round(np.linspace(20, 180, 128)) * dx
    freqs = [4., 6., 8., 10.] * world
    return {'nx': nx, 'nz': nz, 'dx': dx, 'dz': dx, 'c': c, 'theta': th, 'eps': ep, 'delta': de, 'nPML': 10, 'cPML': 1e3,
            'freqs': freqs[:nfreq_per_rank * world],
            'geom': {'src': np.stack([xs, np.full(64, 150.)], 1), 'rec': np.stack([xr, np.full(128, 160.)], 1), 'mode': 'fixed'}}


def c4_config(nfreq=16, nsrc=256, nrec=256, nx=500, nz=1500, npml=20):
    """SURVEY.md 8(d) C4 recipe: MiniZephyr 500x1500, C3's model recipe (seed 0), freqs linspace(2,12,16), sources
    and receivers on grid nodes just below the top PML.  Returns (systemConfig, c_true): observed data come from
    the same model with a -10 % Gaussian velocity blob (sigma = 20 cells) at the centre."""
    rng = np.random.default_rng(0)
    dx = 10.
    c = layered_model(nx, nz, rng)
    xs = np.round(np.linspace(0.025 * nx, 0.975 * nx, nsrc)) * dx
    xr = np.round(np.linspace(0.025 * nx, 0.975 * nx, nrec)) * dx
    zs = float(min(npml + 5, nz - 2)) * dx
    blob = np.exp(-(((np.arange(nx)[None, :] - nx / 2) ** 2 + (np.arange(nz)[:, None] - nz / 2) ** 2) / (2 * 20. ** 2)))
    sc = {'nx': nx, 'nz': nz, 'dx': dx, 'dz': dx, 'c': c, 'rho': 1., 'nPML': npml, 'freqs': list(np.linspace(2., 12., 16)[:nfreq]),
          'geom': {'src': np.stack([xs, np.full(nsrc, zs)], 1), 'rec': np.stack([xr, np.full(nrec, zs + dx)], 1), 'mode': 'fixed'}}
    return sc, c * (1. - 0.1 * blob)


def dump_outputs(dirname, outputs, rank, world):
    """--dump-outputs: write what the timed path returned in its last step as DIR/<name>.npy, so that two builds can be
    compared output for output.  `outputs` maps name -> (device tensor, byte budget).  Complex tensors are stored as
    real arrays with a trailing (re, im) axis: float64, or float32 for complex64.  A tensor larger than its budget is
    cut to a fixed sample of its rows (first axis; seed 0, sorted), the same rows in every run with the same arguments.
    With several ranks each writes its own frequencies as <name>.rank<r>.npy."""
    import torch
    assert sum(b for _, b in outputs.values()) <= DUMP_BYTES
    os.makedirs(dirname, exist_ok=True)
    for name, (t, budget) in outputs.items():
        if t.is_complex():
            t = torch.view_as_real(t)
        row_bytes = t[0].numel() * t.element_size()
        if t.numel() * t.element_size() > budget:
            keep = np.sort(np.random.default_rng(0).choice(t.shape[0], budget // row_bytes, replace=False))
            t = t[torch.from_numpy(keep).to(t.device)]
        np.save(os.path.join(dirname, name + ('' if world == 1 else '.rank%d' % rank) + '.npy'), t.cpu().numpy())


def workload_config(a, nfreq):
    if getattr(a, 'config', 'c3') == 'c2':
        return {'workload': 'C2: Eurus 2D TTI 200x400, dx=dz=10 m, nPML=10, 64 sources, 128 receivers, 4 frequencies (4,6,8,10 Hz) '
                            'per GPU, one refinement step', 'nx': 200, 'nz': 400, 'nsrc': 64, 'nrec': 128, 'nfreq': nfreq,
                'parallelism': 'freq-shard x%d' % max(nfreq // 4, 1),
                'l2': 'L2 flushed between steps by rewriting the 1 GB of block inverses (> 126 MB L2) each step'}
    return {'workload': 'C3: MiniZephyr 2D random-layered %dx%d (nx x nz), dx=dz=10 m, nPML=%d, %d sources, %d receivers, '
                        '%d frequenc%s of linspace(2,9,8) Hz, one per GPU' % (a.nx, a.nz, a.npml, a.nsrc, a.nsrc, nfreq,
                                                                               'y' if nfreq == 1 else 'ies'),
            'nx': a.nx, 'nz': a.nz, 'nsrc': a.nsrc, 'nrec': a.nsrc, 'nfreq': nfreq, 'parallelism': 'freq-shard x%d' % nfreq,
            'l2': 'inputs larger than L2: every step rewrites %.1f GB of block inverses and a %.1f GB wavefield panel'
                  % (a.nz * a.nx * a.nx * 16 / 1e9, a.nz * a.nx * a.nsrc * 16 / 1e9)}


# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                       '-lms', '200'], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, smax, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.f.read().splitlines():
            parts = [x.strip() for x in ln.split(',')]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        return out


def fp64_peak_tflops(torch, dev):
    """Measured FP64 GEMM rate (cuBLAS DGEMM via torch.matmul) -- the roofline denominator for the
    tensor-bound kernels; MEASURED_PEAKS.json has no FP64 figure (BASELINE.md section 4)."""
    n = 6144
    a = torch.randn((n, n), dtype=torch.float64, device=dev)
    b = torch.randn((n, n), dtype=torch.float64, device=dev)
    c = torch.empty_like(a)
    best = 1e30
    for i in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        e1.synchronize()
        if i:
            best = min(best, e0.elapsed_time(e1))
    del a, b, c
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def gradient_check(zb, parallel, world, rank):
    """N-GPU check of the one data-path collective (the NCCL all-reduce of the gradient and misfit): a reduced C4
    (MiniZephyr 120x200, 2 frequencies per rank, 16 sources / receivers) is evaluated with its frequencies sharded over
    the ranks and compared, on rank 0, with the oracle's Jtvec (middleware/problem.py:125-164 restated and pinned to the
    reference by tests/golden/gradient_*.npz).  The oracle is the checker here, never the thing measured."""
    nfreq = 2 * world
    sc, c_true = c4_config(nfreq=16, nsrc=16, nrec=16, nx=120, nz=200, npml=10)
    sc['freqs'] = list(np.linspace(3., 9., nfreq))
    sc['Disc'] = zb.MiniZephyr
    sv, pr = zb.Helm2DSurvey(sc), zb.Helm2DProblem(sc)
    pr.pair(sv)
    svt, prt = zb.Helm2DSurvey(dict(sc, c=c_true)), zb.Helm2DProblem(dict(sc, c=c_true))
    prt.pair(svt)
    dobs = svt.dpred()                                   # all-gathered data cube of the perturbed model
    prt.clearCache()
    phi, g = pr.misfit_and_gradient(dobs)                # frequencies sharded, one all-reduce
    pr.clearCache()
    if rank != 0:
        return None
    from oracle import helm_oracle as ho
    osv = ho.OracleSurvey(sc, sc['freqs'], sc['geom']['src'], sc['geom']['rec'])
    u = osv.fields()
    phi_ref, v = osv.misfit(dobs, u)
    g_ref = osv.Jtvec(v, u=u)
    return {'gradient_rel_l2': float(np.linalg.norm(g - g_ref) / np.linalg.norm(g_ref)), 'misfit_rel': float(abs(phi - phi_ref) / phi_ref),
            'tolerance': 1e-8, 'ranks': world, 'frequencies': nfreq,
            'workload': 'reduced C4: MiniZephyr 120x200, %d frequencies sharded over %d ranks, 16 sources, 16 receivers; NCCL all-reduce of N+1 doubles' % (nfreq, world)}


def run_c4(a, torch, zb, _lib, parallel, rank, world, dev, local):
    """BASELINE config 4: FWI misfit + gradient (forward + adjoint) on MiniZephyr 500x1500, 16 frequencies x 256 sources,
    frequencies sharded round-robin over the ranks (strong scaling: the job is fixed), gradient and misfit summed by one
    NCCL all-reduce INSIDE the timed region.  A step = new model -> assemble + factor every local frequency -> forward
    solve, extraction, misfit, back-projection, adjoint solve, gradient correlation -> all-reduce."""
    import ctypes as C
    lib = _lib.get_lib()
    sc, c_true = c4_config()
    F, S = len(sc['freqs']), sc['geom']['src'].shape[0]
    sc['Disc'] = zb.MiniZephyr
    if a.dtype == 'c64':
        sc['dtype'] = 'complex64'
    if a.twist == -2:
        sc['twist'] = 'source'
    elif a.twist >= 0:
        sc['twist'] = a.twist
    if a.workers > 0:
        sc['factorWorkers'] = sc['solveWorkers'] = a.workers
    sv, pr = zb.Helm2DSurvey(sc), zb.Helm2DProblem(sc)
    pr.pair(sv)
    svt, prt = zb.Helm2DSurvey(dict(sc, c=c_true)), zb.Helm2DProblem(dict(sc, c=c_true))
    prt.pair(svt)
    dobs = svt.dpred()
    prt.clearCache()
    torch.cuda.empty_cache()
    mine = pr.system.localFreqIndices
    subs = pr.system.subProblems
    for kv in a.opt:
        key, val = kv.split('=')
        for i in mine:
            _lib.check(lib.hz_set_option(subs[i].handle, key.encode(), float(val)), subs[i].handle)
    peak = fp64_peak_tflops(torch, dev)
    dobs_dev = pr.upload_dobs(dobs)
    nx, nz = sc['nx'], sc['nz']
    N = nx * nz

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def step():
        for i in mine:                                   # "new model": same values, re-assembled, factors invalidated
            _lib.check(lib.hz_assemble(subs[i].handle, *subs[i]._assemble_args()), subs[i].handle)
        return pr.misfit_and_gradient(dobs_dev, to_host=False)
    for _ in range(a.warmup):
        red = step()
    barrier()
    n0 = C.c_int64(0)
    lib.hz_launch_count(C.byref(n0))
    sampler = ClockSampler(local) if rank == 0 else None
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(a.steps):
        red = step()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    clocks = sampler.stop() if sampler else None
    n1 = C.c_int64(0)
    lib.hz_launch_count(C.byref(n1))
    barrier()
    tt = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
    ms_per_step = float(tt.item()) / a.steps
    value = 2 * F * S / (ms_per_step * 1e-3)             # forward + adjoint wavefields
    assert bool(torch.isfinite(red).all())
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {'gradient': (red[:-1], DUMP_BYTES - (1 << 20)), 'misfit': (red[-1:], 1 << 20)}, rank, world)
    # end to end: host model in, host gradient + misfit out
    c_host = torch.from_numpy(np.ascontiguousarray(sc['c'], dtype=np.complex128)).pin_memory()
    e2e = None
    if a.e2e_steps > 0:
        def e2e_step(k):
            pr.updateModel({'c': c_host.numpy() * (1. + 1e-6 * k)})      # a genuinely new model every evaluation
            return pr.misfit_and_gradient(dobs)
        e2e_step(0)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for k in range(a.e2e_steps):
            phi, g = e2e_step(k + 1)
        s1.record()
        torch.cuda.synchronize()
        et = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(et, op=torch.distributed.ReduceOp.MAX)
        ems = float(et.item()) / a.e2e_steps
        assert np.isfinite(g).all() and np.isfinite(phi)
        e2e = {'value': 2 * F * S / (ems * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': int(N * 16 + N * 8 + dobs.size * 16 + N * 16),
               'd2h_bytes_per_step': int((N + 1) * 8), 'ms_per_step': ems,
               'call': 'problem.updateModel({c: host array}); problem.misfit_and_gradient(host dobs) -> (phi, host gradient)'}
    gcheck = None
    if world > 1 and not a.no_gradient_check:
        gcheck = gradient_check(zb, parallel, world, rank)
    if rank != 0:
        return 0
    # roofline of the step: algorithmic flops (factor 8 b^3 nz per frequency; two substitution passes of
    # 2 nz 8 b^2 S each) against the measured FP64 GEMM rate
    per_rank_f = max(len(parallel.shard_indices(F, r, world)) for r in range(world))
    flops = per_rank_f * (8.0 * nx ** 3 * nz + 2 * 2 * nz * 8.0 * nx * nx * S)
    ach = flops / (ms_per_step * 1e-3) / 1e12
    roof = {'bound': 'tensor', 'kernel': 'whole gradient step of the busiest rank (gj_step_kernel + zgemm_dmma_kernel; b = %d blocks are latency-bound, '
                                         'so co-resident frequencies are factored and swept concurrently)' % nx,
            'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak, 'traffic': None,
            'peak_source': 'cuBLAS DGEMM 6144^3 measured in this run', 'flops_per_step_busiest_rank': flops}
    cpu = None
    if not a.no_cpu_baseline and world == 1:
        from oracle import helm_oracle as ho
        sub = {k: v for k, v in sc.items() if k not in ('freqs', 'geom', 'Disc')}
        sub['freq'] = sc['freqs'][8]
        q = ho.sparse_kaiser_source(sub, sc['geom']['src'][:8])
        t0_ = time.perf_counter()
        od = ho.OracleDisc(sub)
        od.factor()
        t1_ = time.perf_counter()
        od * q
        t2_ = time.perf_counter()
        per_f = (t1_ - t0_) + 2 * S * (t2_ - t1_) / 8
        cpu = {'value': 2 * S / per_f, 'unit': UNIT, 'cores': 1, 'kind': 'port',
               'sample': 'oracle port (numpy assembly + scipy SuperLU), MiniZephyr 500x1500: one of the 16 frequencies factored in full (%.1f s) + 8 of '
                         '2 x 256 right-hand sides (%.3f s each), solve time scaled to forward + adjoint of 256 sources; %.1f s of CPU work'
                         % (t1_ - t0_, (t2_ - t1_) / 8, t2_ - t0_)}
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': ms_per_step,
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': a.dtype, 'data': 'synthetic',
            'config': {'workload': 'C4: FWI misfit + gradient (forward + adjoint, MultiFreq), MiniZephyr 500x1500, 16 frequencies x 256 sources / receivers, '
                                   'frequencies sharded over %d GPU(s), gradient + misfit all-reduced (NCCL) inside the timed region; wavefields counted: '
                                   '2 x 16 x 256 per step' % world, 'nx': nx, 'nz': nz, 'nsrc': S, 'nrec': S, 'nfreq': F,
                       'parallelism': 'freq-shard x%d' % world,
                       'l2': 'inputs larger than L2: every step rewrites %.1f GB of block inverses per frequency' % (nz * nx * nx * 16 / 1e9)},
            'roofline': roof, 'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': int(n1.value - n0.value), 'clocks': clocks,
            's_per_gradient': ms_per_step * 1e-3, 'gradient_check': gcheck, 'fp64_peak_tflops_measured': peak}
    print(json.dumps(line))
    return 0


def c5_config(nx=2000, nz=6000, nsrc=16, npml=20):
    """SURVEY.md 8(d) C5 recipe: MiniZephyr 2000x6000, dx=dz=7.5 m, C3's model recipe (seed 0), 32 frequencies
    linspace(2,20,32) Hz, 16 sources on grid nodes just below the top PML."""
    rng = np.random.default_rng(0)
    dx = 7.5
    c = layered_model(nx, nz, rng)
    xs = np.round(np.linspace(0.025 * nx, 0.975 * nx, nsrc)) * dx
    zs = float(min(npml + 5, nz - 2)) * dx
    return {'nx': nx, 'nz': nz, 'dx': dx, 'dz': dx, 'c': c, 'rho': 1., 'nPML': npml, 'freqs': list(np.linspace(2., 20., 32)),
            'geom': {'src': np.stack([xs, np.full(nsrc, zs)], 1), 'rec': np.stack([xs, np.full(nsrc, zs + dx)], 1), 'mode': 'fixed'}}


def run_c5(a, torch, zb, _lib, parallel, rank, world, dev, local):
    """BASELINE config 5: multiscale sweep on 2000x6000, complex64-vs-complex128 tolerance study.  The block inverses of
    one frequency are 384 GB (complex128) / 192 GB (complex64): more than one GPU holds, so factors are CHECKPOINTED
    (storeEvery='auto': every k-th block inverse kept, the rest recomputed inside the sweeps).  A step = one frequency:
    assemble + factor + solve 16 sources, once in complex128 and once in complex64; reported per frequency: seconds,
    store_every, factor HBM, the complex128 stencil residual and rel-L2(complex64 vs complex128).  --steps K runs K of
    the 32 frequencies per rank (spread over the sweep; rank r takes every world-th of them)."""
    import ctypes as C
    lib = _lib.get_lib()
    nx, nz = (a.nx, a.nz) if (a.nx, a.nz) != (1000, 3000) else (2000, 6000)
    sc = c5_config(nx, nz, 16, a.npml)
    S = 16
    pick = [int(round(i)) for i in np.linspace(0, 31, a.steps * world)][rank::world]
    freqs = [sc['freqs'][i] for i in pick]
    q = zb.SparseKaiserSource(sc)(sc['geom']['src'])
    # warm-up: load every kernel on a small problem of the same kind (both dtypes, checkpointed)
    for dt in (None, 'complex64'):
        w = c3_config(256, 96, 4, 4, 1)
        wsub = {k: v for k, v in w.items() if k not in ('freqs', 'geom')}
        wsub.update(freq=5., storeEvery=3)
        if dt:
            wsub['dtype'] = dt
        for _ in range(max(a.warmup, 1)):
            zb.MiniZephyr(wsub) * zb.SparseKaiserSource(wsub)(w['geom']['src'])
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    n0 = C.c_int64(0)
    lib.hz_launch_count(C.byref(n0))
    sampler = ClockSampler(local) if rank == 0 else None
    rows = []
    tot = {'c128': 0.0, 'c64': 0.0}
    peak_mem = 0
    for f in freqs:
        row = {'freq_hz': float(f)}
        u128 = None
        for name, dt in (('c128', None), ('c64', 'complex64')):
            sub = {k: v for k, v in sc.items() if k not in ('freqs', 'geom')}
            sub.update(freq=f, storeEvery='auto')
            if dt:
                sub['dtype'] = dt
            d = zb.MiniZephyr(sub)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            X, zr = d.rhs_to_device(q)
            ev[0].record()
            _lib.check(lib.hz_assemble(d.handle, *d._assemble_args()), d.handle)
            d._ensure_factors(*zr)
            ev[1].record()
            d.solve_device(X, zr, want_residual=(dt is None))
            ev[2].record()
            ev[2].synchronize()
            peak_mem = max(peak_mem, torch.cuda.mem_get_info(dev)[1] - torch.cuda.mem_get_info(dev)[0])
            row[name] = {'factor_s': ev[0].elapsed_time(ev[1]) * 1e-3, 'solve_s': ev[1].elapsed_time(ev[2]) * 1e-3,
                         'store_every': d._store_every_used, 'factor_gb': d.factor_bytes() / 1e9}
            tot[name] += ev[0].elapsed_time(ev[2]) * 1e-3
            if dt is None:
                row['c128']['stencil_residual'] = d.last_residual
                u128 = X
            else:
                rel = torch.linalg.vector_norm(X.to(torch.complex128) - u128, dim=0) / torch.linalg.vector_norm(u128, dim=0)
                row['rel_l2_c64_vs_c128'] = float(rel.max())
                assert bool(torch.isfinite(torch.view_as_real(u128)).all())
            d.close()
            del d
            torch.cuda.empty_cache()
        rows.append(row)
        del u128, X
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    n1 = C.c_int64(0)
    lib.hz_launch_count(C.byref(n1))
    tt = torch.tensor([tot['c128'], tot['c64']], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        gathered = [None] * world
        torch.distributed.all_gather_object(gathered, rows)
        rows = sorted([r for g in gathered for r in g], key=lambda r: r['freq_hz'])
    if rank != 0:
        return 0
    t128, t64 = float(tt[0]), float(tt[1])
    nfreq = a.steps * world
    peak = fp64_peak_tflops(torch, dev)
    k128 = rows[0]['c128']['store_every']
    flops = a.steps * 8.0 * nx ** 3 * nz * (1 + 2.0 * (k128 - 1) / k128)      # executed: factor + recomputation in both sweeps
    line = {'metric': METRIC, 'value': nfreq * S / t128, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': 1e3 * t128 / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'c128',
            'data': 'synthetic',
            'config': {'workload': 'C5: multiscale sweep, MiniZephyr %dx%d, dx=dz=7.5 m, %d of the 32 frequencies of linspace(2,20,32) Hz per GPU, 16 sources; '
                                   'complex128 (value) and complex64 per frequency; checkpointed factors (store_every auto)' % (nx, nz, a.steps),
                       'nx': nx, 'nz': nz, 'nsrc': S, 'nfreq': nfreq, 'parallelism': 'freq-shard x%d' % world,
                       'l2': 'inputs larger than L2: every frequency writes > 90 GB of block inverses'},
            'roofline': {'bound': 'tensor', 'kernel': 'gj_step_kernel, b = %d (factorisation + recomputation between checkpoints)' % nx,
                         'achieved': flops / t128 / 1e12, 'peak': peak, 'unit': 'TFLOP/s', 'frac': flops / t128 / 1e12 / peak, 'traffic': None,
                         'peak_source': 'cuBLAS DGEMM 6144^3 measured in this run', 'note': 'executed flops incl. recomputation; algorithmic 8 b^3 nz per frequency'},
            'cpu_baseline': None, 'e2e': None, 'gpu_launches': int(n1.value - n0.value), 'clocks': clocks,
            'value_c64': nfreq * S / t64, 'seconds_per_frequency': {'c128': t128 / a.steps, 'c64': t64 / a.steps},
            'hbm_peak_gb': peak_mem / 1e9, 'tolerance_study': rows, 'tolerance': {'c64_vs_c128': 1e-4}}
    print(json.dumps(line))
    return 0


def tf32_peak_tflops(torch, dev):
    """Measured TF32 GEMM rate (cuBLAS via torch.matmul with TF32 allowed): the denominator for the tcgen05 contraction of
    the complex64 variant (MEASURED_PEAKS.json has no TF32 figure; nominal dense 1100 TFLOP/s)."""
    n = 8192
    a = torch.randn((n, n), dtype=torch.float32, device=dev)
    b = torch.randn((n, n), dtype=torch.float32, device=dev)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    best = 1e30
    for i in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        e1.synchronize()
        if i:
            best = min(best, e0.elapsed_time(e1))
    torch.backends.cuda.matmul.allow_tf32 = old
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--config', default='c3', choices=['c3', 'c2', 'c4', 'c5'], help='c3: MiniZephyr 1000x3000 x 512 src (default, headline); c2: Eurus 200x400, 4 freqs x 64 src; c4: FWI gradient 500x1500, 16 freqs x 256 src; c5: 2000x6000 sweep, c64-vs-c128 study with checkpointed factors')
    ap.add_argument('--nx', type=int, default=1000)
    ap.add_argument('--nz', type=int, default=3000)
    ap.add_argument('--nsrc', type=int, default=512)
    ap.add_argument('--npml', type=int, default=20)
    ap.add_argument('--e2e-steps', type=int, default=2)
    ap.add_argument('--ref-nz', type=int, default=240)
    ap.add_argument('--ref-nrhs', type=int, default=8)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-calibration', action='store_true', help='reference arm: skip the >= 1000-row depth calibration')
    ap.add_argument('--no-gradient-check', action='store_true', help='N > 1: skip the NCCL-summed gradient check against the oracle')
    ap.add_argument('--no-operator-e2e', action='store_true', help='skip the one-off timing of Disc * q -> host (N, S) wavefield')
    ap.add_argument('--dtype', default='c128', choices=['c128', 'c64'], help='c64: complex64 storage of the block inverses + complex64 substitution')
    ap.add_argument('--opt', action='append', default=[], help='library option key=value (hz_set_option), e.g. gj_pdl=1')
    ap.add_argument('--workers', type=int, default=0, help='c2/c4: host threads (frequencies in flight) per GPU for factorisation and sweeps (0: library default 4)')
    ap.add_argument('--twist', type=int, default=-1, help='block row where the elimination chains meet (-1: nz/2 (default policy), -2: source depth)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last step returned as DIR/<name>.npy '
                    '(c3: receiver data + a fixed row sample of the wavefield panel; c2: receiver data; c4: gradient + misfit)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and (a.impl == 'reference' or a.config == 'c5'):
        ap.error('--dump-outputs covers the c2, c3 and c4 GPU paths')
    if a.impl == 'reference':
        return run_reference(a)

    import ctypes as C
    import torch
    import zephyr_b200 as zb
    from zephyr_b200 import _lib, parallel

    rank, world = parallel.init_from_env()
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    nfreq = max(world, 1)
    lib = _lib.get_lib()
    if a.config == 'c4':
        return run_c4(a, torch, zb, _lib, parallel, rank, world, dev, local)
    if a.config == 'c5':
        return run_c5(a, torch, zb, _lib, parallel, rank, world, dev, local)

    if a.config == 'c2':
        nfreq = 4 * max(world, 1)
        sc = c2_config(4, max(world, 1))
        sc['Disc'] = zb.Eurus
        a.nx, a.nz, a.nsrc = sc['nx'], sc['nz'], 64
    else:
        sc = c3_config(a.nx, a.nz, a.nsrc, a.nsrc, nfreq, a.npml)
        sc['Disc'] = zb.MiniZephyr
    if a.dtype == 'c64':
        sc['dtype'] = 'complex64'
    sc['twist'] = 'mid' if a.twist == -1 else ('source' if a.twist == -2 else a.twist)
    c_host = torch.from_numpy(np.ascontiguousarray(sc['c'], dtype=np.complex128)).pin_memory()
    sc['c'] = c_host.numpy()
    sv, pr = zb.Helm2DSurvey(sc), zb.Helm2DProblem(sc)
    pr.pair(sv)
    mine = pr.system.localFreqIndices
    subs = pr.system.subProblems
    ops = pr._device_ops()
    for kv in a.opt:
        key, val = kv.split('=')
        for i in mine:
            _lib.check(lib.hz_set_option(subs[i].handle, key.encode(), float(val)), subs[i].handle)
    nf_ = 2 if a.config == 'c2' else 1
    N, S, b = a.nx * a.nz, a.nsrc, nf_ * a.nx
    X = torch.empty((nf_ * N, S), dtype=torch.complex64 if a.dtype == 'c64' else torch.complex128, device=dev)
    peak = fp64_peak_tflops(torch, dev)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    tms = {'assemble': 0.0, 'factor': 0.0, 'solve': 0.0, 'extract': 0.0}
    last = {}

    def step(record=False):
        if len(mine) > 1:
            # several frequencies on this GPU: assemble all, factor them concurrently (MultiFreq.prefactor), then sweep
            # them concurrently too (MultiFreq.run_local: one stream + host thread per frequency in flight)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
            for i in mine:
                _lib.check(lib.hz_assemble(subs[i].handle, *subs[i]._assemble_args()), subs[i].handle)
            ev[1].record()
            dd = pr.dpred_device()        # each worker factors and sweeps its own frequencies: phases of different frequencies overlap
            ev[2].record()
            last['data'] = dd
            if record:
                ev[2].synchronize()
                tms['assemble'] += ev[0].elapsed_time(ev[1])
                tms['factor'] += ev[1].elapsed_time(ev[2])          # factor + solve + extract, overlapped across frequencies
            return dd[mine[-1]]
        for i in mine:
            sub = subs[i]
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record()
            _lib.check(lib.hz_assemble(sub.handle, *sub._assemble_args()), sub.handle)
            ev[1].record()
            sub._ensure_factors(*ops['s_z'])
            ev[2].record()
            pr.forward_device(i, out=X)
            ev[3].record()
            d = pr.extract_device(X)
            ev[4].record()
            if record:
                ev[4].synchronize()
                for k, nm in enumerate(['assemble', 'factor', 'solve', 'extract']):
                    tms[nm] += ev[k].elapsed_time(ev[k + 1])
        return d

    for _ in range(a.warmup):
        step()
    barrier()
    for i in mine:
        _lib.check(lib.hz_profile(subs[i].handle, 1, None), subs[i].handle)
    n0 = C.c_int64(0)
    lib.hz_launch_count(C.byref(n0))
    sampler = ClockSampler(local) if rank == 0 else None
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(a.steps):
        d = step(record=True)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    clocks = sampler.stop() if sampler else None
    n1 = C.c_int64(0)
    lib.hz_launch_count(C.byref(n1))
    prof = (C.c_double * 6)()
    _lib.check(lib.hz_profile(subs[mine[0]].handle, 0, prof), subs[mine[0]].handle)
    for i in mine[1:]:
        lib.hz_profile(subs[i].handle, 0, None)
    barrier()
    tt = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
    ms = float(tt.item())
    ms_per_step = ms / a.steps
    value = nfreq * S / (ms_per_step * 1e-3)
    assert bool(torch.isfinite(torch.view_as_real(d)).all())
    if a.dump_outputs:
        if 'data' in last:                # several frequencies: the (R, S) data of each, the wavefield panels stay internal
            out = {'data': (torch.stack([last['data'][i] for i in mine]), DUMP_BYTES)}
        else:                             # receiver data and the (N, S) wavefield panel the last step solved for
            out = {'data': (d, 16 << 20), 'wavefield': (X, DUMP_BYTES - (16 << 20))}
        dump_outputs(a.dump_outputs, out, rank, world)
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12      # nominal FP32 FFMA peak (no measured figure in MEASURED_PEAKS.json)

    # ---- end to end through the reference-facing call: host model in, host data out ----------
    e2e = None
    if a.e2e_steps > 0:
        def e2e_step():
            pr.updateModel({'c': c_host.numpy()})       # H2D of the model, re-assembly; factors invalidated
            return sv.dpred()                            # sources -> solve -> extraction -> D2H of the data cube
        e2e_step()
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(a.e2e_steps):
            dh = e2e_step()
        s1.record()
        torch.cuda.synchronize()
        et = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(et, op=torch.distributed.ReduceOp.MAX)
        ems = float(et.item()) / a.e2e_steps
        assert np.isfinite(dh).all()
        h2d = N * 16 + N * 8 * (4 if a.config == 'c2' else 1) + sum(ops[k].numel() * ops[k].element_size() for k in ops if hasattr(ops[k], 'numel'))
        e2e = {'value': nfreq * S / (ems * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': int(h2d),
               'd2h_bytes_per_step': int(sv.nrec * S * 16), 'ms_per_step': ems,
               'call': 'problem.updateModel({c: host array}); survey.dpred() -> host (nrec, nsrc, nfreq) data'}

    # ---- second end-to-end figure: the reference's own operator call, Disc * q -> dense host (N, S) wavefield
    # (backend/discretization.py:101-106); 24.6 GB of D2H at C3.  Timed once (N = 1 only), factors reused.
    op_e2e = None
    if world == 1 and a.config == 'c3' and not a.no_operator_e2e:
        q = zb.SparseKaiserSource(sc)(sc['geom']['src'])
        sub0 = subs[mine[0]]
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        uh = sub0 * q
        w1 = time.perf_counter()
        assert uh.shape == (N, S) and np.isfinite(uh[::997]).all()
        op_e2e = {'value': S / (w1 - w0), 'unit': UNIT, 'seconds': w1 - w0, 'd2h_bytes': int(uh.nbytes), 'factors': 'reused',
                  'call': 'MiniZephyr(systemConfig) * q -> host ndarray (N, S) complex128 (wall clock: sparse rhs injection, substitution, D2H)'}
        del uh
    gcheck = None
    if world > 1 and not a.no_gradient_check:
        for i in mine:                                   # make room: the check allocates its own small handles
            del subs[i].factors
        gcheck = gradient_check(zb, parallel, world, rank)

    if rank != 0:
        return 0

    # ---- rooflines.  Both hot kernels are bound by the FP64 tensor pipe (DMMA).  The two elimination
    # chains run on two streams, so single-launch durations overlap; `achieved` is therefore the
    # algorithmic flops of ALL launches of the kernel in a step divided by the phase time measured with
    # CUDA events on the launching stream.  The sampled per-launch durations are reported beside it.
    solve_ms, solve_n, solve_all, upd_ms, upd_n, upd_all = list(prof)
    per = {k: v / a.steps / max(len(mine), 1) for k, v in tms.items()}
    nsteps_gj = (b + 31) // 32
    flop_upd = 8.0 * b * b * b / nsteps_gj       # complex MAC = 8 real flops; mean over the panel steps of one block
    refine_note = ' (x2 sweeps: one refinement step)' if a.config == 'c2' else ''
    flop_solve = 8.0 * b * b * S                 # one launch = (b x b) . (b x S)
    peak_src = ('cuBLAS DGEMM 6144^3 measured in this run = %.1f TFLOP/s (MEASURED_PEAKS.json has no FP64 figure); nominal '
                'FP64 tensor = %.1f TFLOP/s' % (peak, NOMINAL_FP64_TFLOPS))
    combined = len(mine) > 1              # several frequencies per GPU: factorisations and sweeps overlap, one combined phase
    sweeps = 2 if a.config == 'c2' else 1                       # Eurus: one refinement step = a second pair of sweeps
    solve_flops_all = sweeps * 2 * a.nz * 8.0 * b * b * S       # SURVEY 8(d): forward + backward sweeps over all block rows
    fac_ach = (8.0 * b ** 3 * a.nz + (solve_flops_all if combined else 0.0)) / (per['factor'] * 1e-3) / 1e12 if per['factor'] > 0 else 0.0
    # DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full` capture of
    # this kernel at b=1000, complex128; not re-measured here (ncu cannot run inside a timed bench) and null for other shapes
    c3_shape = a.config != 'c2' and b == 1000 and a.dtype != 'c64'
    traffic_gj = 16.617e6 if c3_shape else None
    traffic_src = ('profiles/r2z_ncu_summary.md: 16.62 MB read + 0 written per launch (cold-cache under ncu; algorithmic '
                   '32 MB = 16 MB block read + 16 MB written -- the ping-pong partner stays in the 126 MB L2)') if c3_shape else None
    roof = {'bound': 'tensor', 'kernel': ('gj_step_kernel + zgemm_dmma_kernel, factorisation and substitution of co-resident frequencies overlapped (b = %d)' % b) if combined
            else 'gj_step_kernel (fused Gauss-Jordan step: rank-32 DMMA update of the %dx%d block + look-ahead panel)' % (b, b),
            'achieved': fac_ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': fac_ach / peak, 'traffic': traffic_gj,
            'traffic_source': traffic_src, 'peak_source': peak_src,
            'flops_per_launch': flop_upd, 'launches_per_step': upd_all / a.steps / max(len(mine), 1),
            'avg_launch_ms_sampled': (upd_ms / upd_n) if upd_n else None, 'sampled_launches': int(upd_n),
            'share_of_step': per['factor'] / sum(per.values())}
    launches_solve = solve_all / a.steps / max(len(mine), 1)
    sol_ach = flop_solve * launches_solve / (per['solve'] * 1e-3) / 1e12 if per['solve'] > 0 else 0.0
    sol_peak = tf32_peak_tflops(torch, dev) if a.dtype == 'c64' else peak
    if a.dtype == 'c64':
        sol_ach *= 3.0                        # executed TF32 flops: every real product is three MMAs (3xTF32 split)
    m3 = not any(kv.split('=')[0] == 'gemm_3m' and int(float(kv.split('=')[1])) % 2 == 0 for kv in a.opt)
    sol_kernel = 'cgemm_tf32_kernel (complex64, tcgen05 kind::tf32 3xTF32 + TMA + TMEM; one refinement step = a second, full-depth pair of sweeps; ' if a.dtype == 'c64' else 'zgemm_dmma_kernel ('
    extra = {} if combined else {'roofline_solve': {'bound': 'tensor',
                                'kernel': '%ssubstitution sweep, M=%d N=%d K=%d)%s' % (sol_kernel, b, S, b, refine_note),
                                'achieved': sol_ach, 'peak': sol_peak, 'unit': 'TFLOP/s', 'frac': sol_ach / sol_peak,
                                'traffic': 32.435e6 if (c3_shape and S == 512) else None,
                                'traffic_source': 'profiles/r2z_ncu_summary.md: 32.4 MB read + 0 written per launch (16 MB block '
                                                  'inverse + 2 x 8 MB panel; the written panel is still in L2)' if (c3_shape and S == 512) else None,
                                'flops_per_launch': flop_solve, 'launches_per_step': launches_solve,
                                'avg_launch_ms_sampled': (solve_ms / solve_n) if solve_n else None,
                                'share_of_step': per['solve'] / sum(per.values())}}
    if not combined and a.dtype != 'c64' and m3:
        # `achieved` counts ALGORITHMIC flops (8 per complex MAC); with the three-multiplication products (option gemm_3m,
        # default) the kernel EXECUTES 6 per complex MAC on the tensor pipe, so the pipe itself runs at 3/4 of `frac`
        extra['roofline_solve']['executed_frac'] = 0.75 * sol_ach / sol_peak
        extra['roofline_solve']['note'] = ('three real DMMAs per complex MAC (Re = ar br - ai bi, Im = (ar + ai)(br + bi) - ar br - ai bi): achieved/frac count '
                                           'the algorithmic 8 flops per complex MAC, executed_frac the 6 the tensor pipe actually performs')
    extra['phase_ms'] = per
    extra['factor_ms'] = per['factor']
    extra['fp64_peak_tflops_measured'] = peak

    cpu = None
    if not a.no_cpu_baseline and world == 1 and a.config == 'c2':
        from oracle import helm_oracle as ho
        sub_sc = {k: v for k, v in sc.items() if k not in ('freqs', 'geom', 'Disc', 'twist')}
        sub_sc['freq'] = sc['freqs'][0]
        q = ho.sparse_kaiser_source(sub_sc, sc['geom']['src'][:8])
        t0 = time.perf_counter()
        od = ho.OracleDisc(sub_sc, 'Eurus')
        od.factor()
        t1 = time.perf_counter()
        od * q
        t2 = time.perf_counter()
        v = S / ((t1 - t0) + S * (t2 - t1) / 8)
        cpu = {'value': v, 'unit': UNIT, 'cores': 1, 'kind': 'port',
               'sample': 'oracle port (numpy assembly + scipy SuperLU), Eurus 200x400, one of the 4 frequencies in full '
                         '(factor %.1f s) + 8 of 64 RHS (%.3f s each), solve time scaled to 64 sources; %.1f s of CPU work'
                         % (t1 - t0, (t2 - t1) / 8, t2 - t0)}
    elif not a.no_cpu_baseline and world == 1:
        # BASELINE.md section 3: a >= 1000-row slab with a 16-column panel (the full operator costs 243 s and 26 GB)
        big = min(1000, a.nz)
        v, wall, res = cpu_throughput(a.nx, a.nz, S, [sc['freqs'][0]], big, 16, a.npml, 1)
        t_survey = SURVEY_FULL_C3[0] + S * SURVEY_FULL_C3[1]
        cpu = {'value': v, 'unit': UNIT, 'cores': 1, 'kind': 'port',
               'sample': 'oracle port (numpy assembly + scipy SuperLU) on nx=%d, nz=%d of %d, 16 RHS (factor %.1f s, %.3f s per RHS); scaled '
                         'linearly to the full depth and %d sources (extrapolated; optimistic for the CPU: SURVEY.md section 6 measured the full '
                         'operator in the build container at %.1f s + %.2f s per RHS = %.2f wavefields/s per core); %.1f s of CPU work'
                         % (a.nx, big, a.nz, res[0][0], res[0][1], S, SURVEY_FULL_C3[0], SURVEY_FULL_C3[1], S / t_survey, wall)}

    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': a.dtype,
            'data': 'synthetic', 'config': workload_config(a, nfreq), 'roofline': roof, 'cpu_baseline': cpu, 'e2e': e2e,
            'gpu_launches': int(n1.value - n0.value), 'clocks': clocks}
    line.update(extra)
    line['e2e_operator'] = op_e2e
    line['gradient_check'] = gcheck
    print(json.dumps(line))
    return 0


if __name__ == '__main__':
    sys.exit(main())
