"""Pseudo-Hessian diagonal (Helm*Problem.pseudo_hessian, misfit_gradient_and_pseudo_hessian, hz_wavefield_lagcorr,
hz_pseudo_hessian) against numpy, against the JVP + stencil-apply route of the Born kernels node by node, and against
the oracle: sum_f sum_s ||dA_f/dm_n w_{f,s}||^2 with splu forward fields and a finite-difference dA.  Also the fused
call against the separate ones, refusals and a 2-rank gloo run.  Every test runs on the CPU through the emulation shim
(tests/emu) and, marked gpu, through the CUDA library; the C4 grid runs on the GPU only.  Run as a script, the file is
one rank of the gloo test."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == '__main__':                                 # one rank of test_two_rank_gloo_pseudo_hessian
    sys.path[:0] = [os.path.dirname(HERE), HERE]

from emu_util import emu, emu_cdll  # noqa: F401,E402
from helpers import layered, rel_l2  # noqa: E402
from oracle import helm_oracle as ho  # noqa: E402
from test_adjoint_gradient import (case, crand, fd5, free_port, observed, oracle_survey, problem, smooth,  # noqa: E402
                                   sub_config)

LAGS = [(0, 0), (0, 1), (0, 2)] + [(1, dx) for dx in range(-2, 3)] + [(2, dx) for dx in range(-2, 3)]


@pytest.fixture(params=['emu', pytest.param('gpu', marks=pytest.mark.gpu)])
def lib(request, monkeypatch):
    """The library the package binds: the CPU-emulated kernels (panels are CPU tensors) or the CUDA build."""
    from zephyr_b200 import _lib
    if request.param == 'emu':
        import torch
        cdll = request.getfixturevalue('emu_cdll')
        monkeypatch.setattr(_lib, 'get_lib', lambda: cdll)
        monkeypatch.setattr(_lib, 'torch_device', lambda index=None: torch.device('cpu'))
        return cdll
    return _lib.get_lib()


@pytest.fixture()
def cuda_lib():
    from zephyr_b200 import _lib
    return _lib.get_lib()


def lagcorr_numpy(u, nx, nz):
    """C(p, delta) = sum_s conj(u_s[p]) u_s[p + delta], zero where p + delta is outside the grid; (13, N)."""
    S = u.shape[1]
    g = u.reshape((nz, nx, S))
    out = np.zeros((13, nz, nx), dtype=np.complex128)
    for l, (dz, dx) in enumerate(LAGS):
        x0, x1 = max(0, -dx), min(nx, nx - dx)
        out[l, :nz - dz, x0:x1] = np.sum(np.conj(g[:nz - dz, x0:x1]) * g[dz:, x0 + dx:x1 + dx], axis=2)
    return out.reshape((13, nz * nx))


# 1. hz_wavefield_lagcorr alone --------------------------------------------------------------------------------------
def test_lagcorr_kernel(lib):
    import torch
    from zephyr_b200 import _lib
    rng = np.random.default_rng(201)
    dev = _lib.torch_device()
    for nx, nz, S in ((7, 5, 3), (19, 6, 37), (5, 11, 291), (40, 4, 70), (9, 5, 600)):    # 600: several passes over S
        N = nx * nz
        u = crand(rng, N, S)
        Ut = torch.from_numpy(u).to(dev)
        Ct = torch.full((13 * N,), 7. + 7j, dtype=torch.complex128, device=dev)
        assert lib.hz_wavefield_lagcorr(_lib.ptr(Ut), nx, nz, S, _lib.ptr(Ct), None) == 0
        ref = lagcorr_numpy(u, nx, nz)
        out = Ct.cpu().numpy().reshape((13, N))
        assert np.abs(out - ref).max() <= 1e-13 * np.abs(ref).max()
        assert np.all(out[ref == 0] == 0)                               # partners outside the grid, edges and corners
    p = _lib.ptr(Ct)                                                    # rejected before any access
    assert lib.hz_wavefield_lagcorr(None, 4, 4, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr(p, 4, 4, 1, None, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr(p, 2, 4, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr(p, 4, 2, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr(p, 4, 4, 0, p, None) == _lib.HZ_EINVAL


# 2. against the JVP + stencil-apply route, node by node -------------------------------------------------------------
def jvp_apply_diag(lib, pr, wrt, nodes=None):
    """sum_f sum_s ||hz_stencil_apply(hz_assemble_jvp(e_n), u_f)||^2 for each node n (all nodes, or ``nodes``).  The
    column of the c derivative is alpha_n dA/dc_n + drho_dc[n] dA/drho_n under Gardner's rule.  With all nodes, the nodes
    go nine colours at a time: the rows a node's column touches (its 3 x 3 neighbourhood) do not overlap within one
    colour (iz mod 3, ix mod 3), so each row of the applied panel belongs to one node and the sums split exactly."""
    import torch
    from zephyr_b200 import _lib
    ops = pr._device_ops()
    dev, N, S = ops['dev'], pr.nrow, pr.survey.nsrc
    nx, nz = int(pr.nx), int(pr.nz)
    gardner = pr.systemConfig.get('rho', None) is None
    iz, ix = np.divmod(np.arange(N), nx)
    if nodes is None:
        groups = [np.flatnonzero((iz % 3 == a) & (ix % 3 == b)) for a in range(3) for b in range(3)]
    else:
        groups = [np.array([n]) for n in nodes]
    out = {k: np.zeros(N) for k in wrt}
    subs = pr.system.subProblems
    for ifreq in pr.system.localFreqIndices:
        pr._ensure_factors(ifreq, ops['s_z'])
        uF = pr.forward_device(ifreq)
        sub = subs[ifreq]
        a = pr._adjoint_alpha(ifreq)
        at = None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.complex128).ravel()).to(dev)
        cr = np.real(np.asarray(pr.systemConfig['c'], dtype=np.complex128)) * np.ones((nz, nx))
        g = (0.25 * np.asarray(sub.rho, dtype=np.float64).reshape((nz, nx)) / cr).ravel()
        P = torch.empty((9 * N,), dtype=torch.complex128, device=dev)
        O = torch.empty((N, S), dtype=torch.complex128, device=dev)
        for k in wrt:
            for grp in groups:
                e = np.zeros(N)
                e[grp] = 1.
                dc = torch.from_numpy(e).to(dev) if k == 'c' else None
                dr = torch.from_numpy(e * g if k == 'c' else e).to(dev) if (k == 'rho' or gardner) else None
                sub._bind_stream()
                _lib.check(lib.hz_assemble_jvp(sub.handle, _lib.ptr(dc), _lib.ptr(dr), _lib.ptr(at if k == 'c' else None),
                                               _lib.ptr(P)), sub.handle)
                _lib.check(lib.hz_stencil_apply(_lib.ptr(P), _lib.ptr(uF), nx, nz, S, 1., 0., _lib.ptr(O), None))
                rows = np.sum(np.abs(O.cpu().numpy()) ** 2, axis=1).reshape((nz, nx))
                for n in grp:
                    out[k][n] += rows[max(iz[n] - 1, 0):iz[n] + 2, max(ix[n] - 1, 0):ix[n] + 2].sum()
    return out


JVP_CASES = [(211, None, False, 'random', ('c',)),
             (212, None, False, 'random', ('rho',)),
             (213, (True, False, False, True), False, 'random', ('c', 'rho')),
             (214, None, True, 'random', ('c', 'rho')),
             (215, (True, False, False, False), False, None, ('c', 'rho')),
             (216, None, True, None, ('c',))]


@pytest.mark.parametrize('seed,freeSurf,visco,rho,wrt', JVP_CASES)
def test_against_jvp_apply(lib, seed, freeSurf, visco, rho, wrt):
    rng = np.random.default_rng(seed)
    sc = case(rng, model='random', freeSurf=freeSurf, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    sv, pr = problem(sc, visco=visco)
    P = pr.pseudo_hessian(wrt=wrt)
    assert list(P) == list(wrt)
    ref = jvp_apply_diag(lib, pr, wrt)
    for k in wrt:
        assert P[k].dtype == np.float64 and P[k].shape == (pr.nrow,)
        assert np.all(np.abs(P[k] - ref[k]) <= 1e-11 * ref[k]), k          # boundary nodes where w = 0: both exactly 0


# 3. against the oracle: splu forward fields and a finite-difference dA per node ---------------------------------------
def oracle_pseudo_hessian(sc, wrt, visco=False):
    osv = oracle_survey(sc, visco)
    c0 = np.asarray(sc['c']) * np.ones((int(sc['nz']), int(sc['nx'])))
    rho0 = None if sc.get('rho') is None else np.asarray(sc['rho']) * np.ones(c0.shape)
    N = c0.size
    qs = osv.getSources()
    out = {k: np.zeros(N) for k in wrt}
    for i, f in enumerate(sc['freqs']):
        sub = sub_config(sc, f, c0, rho0, visco)
        lu = spla.splu(sp.csc_matrix(ho.mz_matrix(sub)))
        w = lu.solve(np.asarray(ho.premul(sub, sc.get('hd', False)) * qs[i].toarray(), dtype=np.complex128))
        for k in wrt:
            for n in range(N):
                e = np.zeros(N)
                e[n] = 1.
                e = e.reshape(c0.shape)

                def A_at(t):
                    c = c0 + t * e if k == 'c' else c0
                    if rho0 is not None:
                        r = rho0 + t * e if k == 'rho' else rho0
                    else:                                  # Gardner's rule on c_f, plus drho when it is perturbed
                        r = 310. * np.real(sub_config(sc, f, c, None, visco)['c']) ** 0.25 + t * e if k == 'rho' else None
                    return ho.mz_matrix(sub_config(sc, f, c, r, visco))
                h = 1e-3 * (np.abs(c0).max() if k == 'c' else (rho0.max() if rho0 is not None else 500.))
                dA = sp.csr_matrix(fd5(A_at, h))
                out[k][n] += np.sum(np.abs(dA @ w) ** 2)
    return out


@pytest.mark.parametrize('seed,mode,visco,rho,wrt,hd', [(221, 'fixed', False, 'random', ('c', 'rho'), True),
                                                        (222, 'fixed', True, None, ('c', 'rho'), False)])
def test_oracle(lib, seed, mode, visco, rho, wrt, hd):
    rng = np.random.default_rng(seed)
    sc = case(rng, nx=9, nz=8, mode=mode, rho=rho)
    sc['geom']['src'] = np.array([[25., 22.], [55., 30.]])
    sc['geom']['rec'] = np.array([[15., 46.], [45., 40.], [65., 42.]])
    if hd:
        sc['hd'] = True
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    import zephyr_b200 as zb
    sv, pr = problem(sc, visco=visco, disc=zb.MiniZephyrHD if hd else None)
    P = pr.pseudo_hessian(wrt=wrt)
    ref = oracle_pseudo_hessian(sc, wrt, visco=visco)
    for k in wrt:
        assert np.abs(P[k] - ref[k]).max() <= 1e-8 * np.abs(ref[k]).max(), k


# 4. the fused call --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('visco,rho,wrt', [(False, 'random', ('c', 'rho')), (True, None, ('c',)), (False, None, ('rho', 'c'))])
def test_fused(lib, visco, rho, wrt):
    rng = np.random.default_rng(231 + visco)
    sc = case(rng, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    dobs = observed(sc, rng, visco=visco)
    sv, pr = problem(sc, visco=visco)
    Wd = 1.3
    phi, g, P = pr.misfit_gradient_and_pseudo_hessian(dobs, Wd=Wd, wrt=wrt)
    phi0, g0 = pr.misfit_and_adjoint_gradient(dobs, Wd=Wd, wrt=wrt)
    P0 = pr.pseudo_hessian(wrt=wrt)
    assert list(g) == list(wrt) and list(P) == list(wrt)
    assert abs(phi - phi0) <= 1e-13 * phi0
    for k in wrt:
        assert rel_l2(g[k], g0[k]) <= 1e-13, k
        assert rel_l2(P[k], P0[k]) <= 1e-13, k
        assert np.all(P[k] >= 0), k


# 5. refusals --------------------------------------------------------------------------------------------------------
def test_refusals(lib):
    import torch
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(241)
    sc = case(rng)
    v = observed(sc, rng)
    for extra in ({'Disc': zb.Eurus, 'theta': 0.1, 'eps': 0.05, 'delta': 0.02}, {'dtype': 'complex64'},
                  {'Disc': zb.MiniZephyr25D, 'nky': 2}):
        sv, pr = problem(dict(sc, **extra), disc=extra.get('Disc'))
        for call in (lambda: pr.pseudo_hessian(), lambda: pr.misfit_gradient_and_pseudo_hessian(v)):
            with pytest.raises(NotImplementedError):
                call()
    sv, pr = problem(sc)
    for bad in ((), ('c', 'c'), ('vp',)):
        for call in (lambda: pr.pseudo_hessian(wrt=bad), lambda: pr.misfit_gradient_and_pseudo_hessian(v, wrt=bad)):
            with pytest.raises(ValueError):
                call()
    # the C ABI
    N = sc['nx'] * sc['nz']
    dev = _lib.torch_device()
    C = torch.zeros(13 * N, dtype=torch.complex128, device=dev)
    p = torch.zeros(N, dtype=torch.float64, device=dev)
    for d in (zb.MiniZephyr(dict(sc, freq=6., dtype='complex64')), zb.Eurus(dict(sc, freq=6., theta=0.1, eps=0.05, delta=0.02))):
        assert lib.hz_pseudo_hessian(d.handle, _lib.ptr(C), None, None, _lib.ptr(p), None) == _lib.HZ_ENOTIMPL
    d = zb.MiniZephyr(dict(sc, freq=6.))
    assert lib.hz_pseudo_hessian(None, _lib.ptr(C), None, None, _lib.ptr(p), None) == _lib.HZ_EINVAL
    assert lib.hz_pseudo_hessian(d.handle, None, None, None, _lib.ptr(p), None) == _lib.HZ_EINVAL
    assert lib.hz_pseudo_hessian(d.handle, _lib.ptr(C), None, None, None, None) == _lib.HZ_EINVAL
    assert lib.hz_pseudo_hessian(d.handle, _lib.ptr(C), None, None, None, _lib.ptr(p)) == 0
    _lib.check(lib.hz_set_coefficients(d.handle, _lib.ptr(d.coefficients())), d.handle)
    assert lib.hz_pseudo_hessian(d.handle, _lib.ptr(C), None, None, _lib.ptr(p), None) == _lib.HZ_ESTATE


# 6. two gloo ranks shard the frequencies and give the single-rank results ---------------------------------------------
def gloo_case():
    rng = np.random.default_rng(251)
    sc = case(rng, model='random', freqs=(5., 7., 10.))
    return sc, observed(sc, rng)


def gloo_results(pr, v):
    wrt = ('c', 'rho')
    P = pr.pseudo_hessian(wrt=wrt)
    phi, g, P2 = pr.misfit_gradient_and_pseudo_hessian(v, wrt=wrt)
    return {'P_c': P['c'], 'P_rho': P['rho'], 'phi': np.array([phi]), 'g_c': g['c'], 'P2_rho': P2['rho']}


def test_two_rank_gloo_pseudo_hessian(emu, tmp_path):
    import emu_util
    emu_util.load_emu()                                    # build once, before the ranks race for it
    sc, v = gloo_case()
    sv, pr = problem(sc)
    ref = gloo_results(pr, v)
    out = str(tmp_path / 'res')
    port = free_port()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE='2', MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port),
                   OPENBLAS_NUM_THREADS='1', OMP_NUM_THREADS='1')
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), out], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        o, _ = p.communicate(timeout=600)
        assert p.returncode == 0, o.decode()[-2000:]
    seen = []
    for r in range(2):
        z = np.load(out + '.rank%d.npz' % r)
        seen += list(z['local'])
        for k in ref:
            assert rel_l2(z[k], ref[k]) <= 1e-13, (r, k)
    assert sorted(seen) == [0, 1, 2]


def gloo_rank(out_path):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(HERE, 'emu'))
    from emu_util import load_emu
    from zephyr_b200 import _lib, parallel
    cdll = load_emu()
    _lib.get_lib = lambda: cdll
    _lib.torch_device = lambda index=None: torch.device('cpu')
    rank, _ = parallel.init_from_env(backend='gloo')
    sc, v = gloo_case()
    sv, pr = problem(sc)
    res = gloo_results(pr, v)
    np.savez(out_path + '.rank%d.npz' % rank, local=np.array(pr.system.localFreqIndices), **res)
    dist.barrier()
    dist.destroy_process_group()


# 7. the GPU at size: the C4 grid -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_c4_grid_pseudo_hessian(cuda_lib):
    rng = np.random.default_rng(261)
    nx, nz = 500, 1500
    c = layered(nx, nz, 1500., 4500., rng, 5, 50)
    xs = np.linspace(500., 4500., 8)
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': c, 'rho': 1., 'nPML': 20, 'freqs': [3., 7.],
          'geom': {'src': np.stack([xs, np.full(8, 300.)], 1), 'rec': np.stack([np.linspace(250., 4750., 32), np.full(32, 14500.)], 1),
                   'mode': 'fixed', 'rterms': np.exp(1j * np.linspace(0., 2., 32))}}
    sv, pr = problem(sc)
    wrt = ('c', 'rho')
    P = pr.pseudo_hessian(wrt=wrt)
    # PML corners, rows next to each boundary, the PML's inner edge and the interior
    pts = [(0, 0), (0, nx - 1), (nz - 1, 0), (nz - 1, nx - 1), (1, 1), (1, nx - 2), (nz - 2, 1), (nz - 2, nx - 2),
           (0, 250), (1, 250), (nz - 1, 250), (nz - 2, 250), (750, 0), (750, 1), (750, nx - 1), (750, nx - 2),
           (19, 19), (20, 20), (nz - 21, nx - 21), (30, 120)]
    pts += [tuple(rng.integers([0, 0], [nz, nx])) for _ in range(64 - len(pts))]
    nodes = [iz * nx + ix for iz, ix in pts]
    ref = jvp_apply_diag(cuda_lib, pr, wrt, nodes=nodes)
    for k in wrt:
        assert np.all(np.abs(P[k][nodes] - ref[k][nodes]) <= 1e-10 * ref[k][nodes]), k
        assert np.all(P[k] >= 0)
    dobs = 0.9 * sv.dpred().reshape((32, 8, 2))
    phi, g, P2 = pr.misfit_gradient_and_pseudo_hessian(dobs, wrt=wrt)
    phi0, g0 = pr.misfit_and_adjoint_gradient(dobs, wrt=wrt)
    assert abs(phi - phi0) <= 1e-13 * phi0
    for k in wrt:
        assert rel_l2(g[k], g0[k]) <= 1e-13 and rel_l2(P2[k], P[k]) <= 1e-13, k


if __name__ == '__main__':
    gloo_rank(sys.argv[1])
