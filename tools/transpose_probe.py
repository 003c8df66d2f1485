"""Transposed solves on one GPU: time of the N, T and H substitution sweeps on the same factors, and of the op(A) tiles
of the DMMA contraction (hz_zgemm_op) at the sweep's shape, all alternated in one run.

    python tools/transpose_probe.py [--nx 1000 --nz 3000 --nsrc 512 --reps 5] --out profiles/<name>.json

Workload: bench.py's C3 (MiniZephyr 1000 x 3000, its seed-0 layered model, 512 Kaiser sources at bench's depth, first
frequency).  Sweeps: `solve_device` on a panel restored from a saved copy before every call (the copy is outside the
timed window), CUDA events around each solve, after one untimed solve per op (the first one also runs the accuracy
probe).  GEMM: b x S x b with twelve different A operands cycled (192 MB > the 126 MB L2, as in the sweep, where every
block inverse comes from HBM).  For scale, the copy a transposed-scratch design would add per GEMM is timed too
(torch's transpose copy of one b x b complex128 block; not a library kernel).  Card name and power limit are read
in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

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
    ap.add_argument('--nx', type=int, default=1000)
    ap.add_argument('--nz', type=int, default=3000)
    ap.add_argument('--nsrc', type=int, default=512)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--gemm-reps', type=int, default=60)
    ap.add_argument('--out', required=True)
    a = ap.parse_args()
    import torch
    import bench
    import zephyr_b200 as zb
    from oracle import helm_oracle as ho
    from zephyr_b200 import _lib
    assert torch.cuda.is_available(), 'needs a CUDA device'
    rec = {'card': card(), 'workload': 'C3 recipe %dx%d, %d sources, f = 2 Hz' % (a.nx, a.nz, a.nsrc)}

    # ---- sweeps on one set of factors ----
    sc = bench.c3_config(a.nx, a.nz, a.nsrc, a.nsrc, 1)
    sc['freq'] = sc.pop('freqs')[0]
    geom = sc.pop('geom')
    d = zb.MiniZephyr(sc)
    X0, zr = d.rhs_to_device(ho.sparse_kaiser_source(sc, geom['src']))
    X = torch.empty_like(X0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {t: [] for t in 'NTH'}
    for rep in range(a.reps + 1):
        for t in 'NTH':
            X.copy_(X0)
            e0.record()
            d.solve_device(X, zr, trans=t)
            e1.record()
            e1.synchronize()
            if rep:
                times[t].append(e0.elapsed_time(e1))
    sweep = {t: {'ms': times[t], 'median_ms': float(np.median(times[t]))} for t in 'NTH'}
    rec['sweep'] = sweep
    rec['sweep_ratio_T_N'] = sweep['T']['median_ms'] / sweep['N']['median_ms']
    rec['sweep_ratio_H_N'] = sweep['H']['median_ms'] / sweep['N']['median_ms']
    rec['probe'] = d.last_probe
    rec['depth_range'] = list(zr)
    d.close()
    del X, X0
    torch.cuda.empty_cache()

    # ---- the contraction at the sweep's shape ----
    lib = _lib.get_lib()
    b, S = a.nx, a.nsrc
    g = torch.Generator(device='cuda').manual_seed(0)
    As = [torch.randn((b, b), dtype=torch.complex128, device='cuda', generator=g) for _ in range(12)]
    B = torch.randn((b, S), dtype=torch.complex128, device='cuda', generator=g)
    Cm = torch.empty((b, S), dtype=torch.complex128, device='cuda')
    gemm = {}
    for m3 in (1, 0):
        ts = {op: [] for op in 'NTC'}
        for rnd in range(4):
            for op, code in (('N', 0), ('T', 1), ('C', 2)):
                k = [0]

                def one():
                    A = As[k[0] % len(As)]
                    k[0] += 1
                    _lib.check(lib.hz_zgemm_op(b, S, b, 1.0, _lib.ptr(A), b, code, _lib.ptr(B), S, 0, _lib.ptr(Cm), S, -1, m3, None))
                events_ms(torch, one, 5)
                ts[op].append(events_ms(torch, one, a.gemm_reps) * 1e3)
        key = 'gemm_3m' if m3 else 'gemm_4m'
        gemm[key] = {op: {'us': ts[op], 'median_us': float(np.median(ts[op]))} for op in 'NTC'}
        gemm[key]['ratio_T_N'] = gemm[key]['T']['median_us'] / gemm[key]['N']['median_us']
        gemm[key]['ratio_C_N'] = gemm[key]['C']['median_us'] / gemm[key]['N']['median_us']
    for op, code in (('T', 1), ('C', 2)):                  # op(A) product against torch's complex128 matmul
        _lib.check(lib.hz_zgemm_op(b, S, b, 1.0, _lib.ptr(As[0]), b, code, _lib.ptr(B), S, 0, _lib.ptr(Cm), S, -1, 1, None))
        ref = (As[0].t() if op == 'T' else As[0].conj().t()) @ B
        torch.cuda.synchronize()
        gemm['rel_err_' + op] = float(torch.linalg.norm(Cm - ref) / torch.linalg.norm(ref))
    rec['gemm'] = gemm
    rec['gemm_shape'] = [b, S, b]
    k = [0]
    Tbuf = torch.empty((b, b), dtype=torch.complex128, device='cuda')

    def tcopy():
        Tbuf.copy_(As[k[0] % len(As)].t())
        k[0] += 1
    events_ms(torch, tcopy, 5)
    rec['transpose_copy_us'] = events_ms(torch, tcopy, a.gemm_reps) * 1e3
    rec['note'] = ('sweep: CUDA events around solve_device (premul 1, conjugation on) on the same factors, N/T/H alternated; '
                   'gemm: CUDA events over %d launches per op, A cycled through 12 operands; transpose_copy_us: torch copy '
                   'of one transposed %dx%d complex128 block (the per-GEMM extra of a transposed-scratch design)' % (a.gemm_reps, b, b))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: rec[k] for k in ('card', 'sweep_ratio_T_N', 'sweep_ratio_H_N', 'probe')}))
    print(json.dumps({k: {kk: (vv['median_us'] if isinstance(vv, dict) else vv) for kk, vv in v.items()} for k, v in gemm.items()
                      if isinstance(v, dict)}))
    print('sweep median ms: ' + ', '.join('%s %.1f' % (t, sweep[t]['median_ms']) for t in 'NTH') + '; transpose copy %.1f us' % rec['transpose_copy_us'])


if __name__ == '__main__':
    main()
