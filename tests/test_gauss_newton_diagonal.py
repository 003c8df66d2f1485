"""Gauss-Newton Hessian diagonal (Helm*Problem.gauss_newton_diagonal, misfit_gradient_and_gauss_newton_diagonal,
hz_wavefield_lagcorr4, hz_gauss_newton_diag) against numpy, against the pseudo-Hessian with the receiver correlation set to
the identity, against G^T (JVP + stencil apply) node by node with G from the library's A^T solve, against born_dpred and
gauss_newton_hvec, and against the oracle: splu forward fields and Green's functions and a finite-difference dA.  Also
the fused call against the separate ones, refusals and a 2-rank gloo run.  Every test runs on the CPU through the
emulation shim (tests/emu) and, marked gpu, through the CUDA library; the C4 grid runs on the GPU only.  Run as a
script, the file is one rank of the gloo test."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == '__main__':                                 # one rank of test_two_rank_gloo_gauss_newton_diagonal
    sys.path[:0] = [os.path.dirname(HERE), HERE]

from emu_util import emu, emu_cdll  # noqa: F401,E402
from helpers import layered, rel_l2  # noqa: E402
from oracle import helm_oracle as ho  # noqa: E402
from test_adjoint_gradient import case, crand, fd5, free_port, observed, oracle_survey, problem, sub_config  # noqa: E402


def lags(R):
    """The stored lags of radius R in the order of the library: (0,0), (0, 1..R), (1, -R..R), ..., (R, -R..R)."""
    return [(0, dx) for dx in range(R + 1)] + [(dz, dx) for dz in range(1, R + 1) for dx in range(-R, R + 1)]


LAGS2, LAGS4 = lags(2), lags(4)


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


def lagcorr_numpy(u, nx, nz, lag_list):
    """C(p, delta) = sum_s conj(u_s[p]) u_s[p + delta], zero where p + delta is outside the grid; (len(lag_list), N)."""
    S = u.shape[1]
    g = u.reshape((nz, nx, S))
    out = np.zeros((len(lag_list), nz, nx), dtype=np.complex128)
    for l, (dz, dx) in enumerate(lag_list):
        x0, x1 = max(0, -dx), min(nx, nx - dx)
        if dz < nz and x1 > x0:
            out[l, :nz - dz, x0:x1] = np.sum(np.conj(g[:nz - dz, x0:x1]) * g[dz:, x0 + dx:x1 + dx], axis=2)
    return out.reshape((len(lag_list), nz * nx))


# 1. hz_wavefield_lagcorr4 alone --------------------------------------------------------------------------------------
def test_lagcorr4_kernel(lib):
    import torch
    from zephyr_b200 import _lib
    rng = np.random.default_rng(301)
    dev = _lib.torch_device()
    # odd sizes, S < 32, S above two passes of a CTA (128 threads, one source per lane), nx < 16, fewer depths than lags
    for nx, nz, S in ((7, 5, 3), (19, 6, 37), (5, 11, 291), (40, 4, 70), (9, 5, 600), (13, 9, 1)):
        N = nx * nz
        u = crand(rng, N, S)
        Ut = torch.from_numpy(u).to(dev)
        C4 = torch.full((41 * N,), 7. + 7j, dtype=torch.complex128, device=dev)
        C2 = torch.full((13 * N,), 7. + 7j, dtype=torch.complex128, device=dev)
        assert lib.hz_wavefield_lagcorr4(_lib.ptr(Ut), nx, nz, S, _lib.ptr(C4), None) == 0
        assert lib.hz_wavefield_lagcorr(_lib.ptr(Ut), nx, nz, S, _lib.ptr(C2), None) == 0
        ref = lagcorr_numpy(u, nx, nz, LAGS4)
        out = C4.cpu().numpy().reshape((41, N))
        assert np.abs(out - ref).max() <= 1e-13 * np.abs(ref).max()
        assert np.all(out[ref == 0] == 0)                               # partners outside the grid, edges and corners
        two = C2.cpu().numpy().reshape((13, N))
        sel = [LAGS4.index(d) for d in LAGS2]                          # the radius-2 lags inside the radius-4 planes
        assert np.abs(out[sel] - two).max() <= 1e-13 * np.abs(two).max()
    p = _lib.ptr(C4)                                                    # rejected before any access
    assert lib.hz_wavefield_lagcorr4(None, 4, 4, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr4(p, 4, 4, 1, None, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr4(p, 2, 4, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr4(p, 4, 2, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_wavefield_lagcorr4(p, 4, 4, 0, p, None) == _lib.HZ_EINVAL


# 2. with the receiver correlation the identity, the contraction is the pseudo-Hessian -------------------------------
def column_inputs(pr, ifreq, dev):
    """alpha (viscous) and drho_dc (Gardner's rule) of one frequency as _derivative_sweep forms them."""
    import torch
    nx, nz = int(pr.nx), int(pr.nz)
    a = pr._adjoint_alpha(ifreq)
    at = None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.complex128).ravel()).to(dev)
    g = None
    if pr.systemConfig.get('rho', None) is None:
        cr = np.real(np.asarray(pr.systemConfig['c'], dtype=np.complex128)) * np.ones((nz, nx))
        rho = np.asarray(pr.system.subProblems[ifreq].rho, dtype=np.float64).reshape((nz, nx))
        g = torch.from_numpy((0.25 * rho / cr).ravel()).to(dev)
    return at, g


@pytest.mark.parametrize('seed,freeSurf,visco,rho', [(311, None, False, 'random'), (312, (True, False, False, True), False, None),
                                                    (313, None, True, 'random'), (314, None, True, None)])
def test_identity_receivers_is_pseudo_hessian(lib, seed, freeSurf, visco, rho):
    import torch
    from zephyr_b200 import _lib
    rng = np.random.default_rng(seed)
    sc = case(rng, model='random', freeSurf=freeSurf, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    sv, pr = problem(sc, visco=visco)
    ops = pr._device_ops()
    dev, N, S, nx, nz = ops['dev'], pr.nrow, sv.nsrc, int(pr.nx), int(pr.nz)
    gam = torch.zeros((13 * N,), dtype=torch.complex128, device=dev)
    gam[:N] = 1.
    C2 = torch.empty((13 * N,), dtype=torch.complex128, device=dev)
    C4 = torch.empty((41 * N,), dtype=torch.complex128, device=dev)
    for ifreq in pr.system.localFreqIndices:
        pr._ensure_factors(ifreq, ops['s_z'])
        uF = pr.forward_device(ifreq)
        sub = pr.system.subProblems[ifreq]
        at, g = column_inputs(pr, ifreq, dev)
        _lib.check(lib.hz_wavefield_lagcorr(_lib.ptr(uF), nx, nz, S, _lib.ptr(C2), None))
        _lib.check(lib.hz_wavefield_lagcorr4(_lib.ptr(uF), nx, nz, S, _lib.ptr(C4), None))
        out = {}
        for name, fn, args in (('P', lib.hz_pseudo_hessian, (C2,)), ('H', lib.hz_gauss_newton_diag, (C4, gam))):
            pc = torch.zeros(N, dtype=torch.float64, device=dev)
            prho = torch.zeros(N, dtype=torch.float64, device=dev)
            sub._bind_stream()
            _lib.check(fn(sub.handle, *[_lib.ptr(a) for a in args], _lib.ptr(at), _lib.ptr(g), _lib.ptr(pc), _lib.ptr(prho)),
                       sub.handle)
            out[name] = (pc.cpu().numpy(), prho.cpu().numpy())
        for P, H in zip(out['P'], out['H']):
            assert np.all(np.abs(H - P) <= 1e-12 * P.max())
            assert P.max() > 0


# 3. node by node against G^T (JVP + stencil apply) with G from the library's A^T solve ------------------------------
def green_apply_diag(lib, pr, wrt, Wd, nodes):
    """Wd^2 sum_f ||G^T hz_stencil_apply(hz_assemble_jvp(e_n), u_f)||_F^2 for each node n of ``nodes``, with
    G = A^-T conj(Rv)^T from Disc.solve(., 'T').  The column of the c derivative is alpha_n dA/dc_n + drho_dc[n]
    dA/drho_n under Gardner's rule.  Only the 3 x 3 rows around n of the applied panel are nonzero."""
    import torch
    from zephyr_b200 import _lib
    ops = pr._device_ops()
    dev, N, S = ops['dev'], pr.nrow, pr.survey.nsrc
    nx, nz = int(pr.nx), int(pr.nz)
    gardner = pr.systemConfig.get('rho', None) is None
    Rv = pr.survey.rVec().tocsr()
    out = {k: np.zeros(len(nodes)) for k in wrt}
    for ifreq in pr.system.localFreqIndices:
        pr._ensure_factors(ifreq, ops['s_z'])
        uF = pr.forward_device(ifreq)
        sub = pr.system.subProblems[ifreq]
        G = np.conj(sub.solve(np.asarray(Rv.conj().T.toarray() / complex(sub.premul), dtype=np.complex128), 'T'))
        at, g = column_inputs(pr, ifreq, dev)
        P = torch.empty((9 * N,), dtype=torch.complex128, device=dev)
        O = torch.empty((N, S), dtype=torch.complex128, device=dev)
        for j, n in enumerate(nodes):
            iz, ix = divmod(n, nx)
            rows = np.array([z * nx + x for z in range(max(iz - 1, 0), min(iz + 2, nz)) for x in range(max(ix - 1, 0), min(ix + 2, nx))])
            for k in wrt:
                e = torch.zeros(N, dtype=torch.float64, device=dev)
                e[n] = 1.
                dc = e if k == 'c' else None
                dr = (e * g if k == 'c' else e) if (k == 'rho' or gardner) else None
                sub._bind_stream()
                _lib.check(lib.hz_assemble_jvp(sub.handle, _lib.ptr(dc), _lib.ptr(dr), _lib.ptr(at if k == 'c' else None),
                                               _lib.ptr(P)), sub.handle)
                _lib.check(lib.hz_stencil_apply(_lib.ptr(P), _lib.ptr(uF), nx, nz, S, 1., 0., _lib.ptr(O), None))
                Dw = O[torch.from_numpy(rows).to(dev)].cpu().numpy()
                out[k][j] += np.sum(np.abs(G[rows].T @ Dw) ** 2)
    return {k: Wd * Wd * v for k, v in out.items()}


NODE_CASES = [(321, None, False, 'random', ('c',)),
              (322, None, False, 'random', ('rho',)),
              (323, (True, False, False, True), False, 'random', ('c', 'rho')),
              (324, None, True, 'random', ('c', 'rho')),
              (325, (True, False, False, False), False, None, ('c', 'rho')),
              (326, None, True, None, ('c',))]


@pytest.mark.parametrize('seed,freeSurf,visco,rho,wrt', NODE_CASES)
def test_every_node(lib, seed, freeSurf, visco, rho, wrt):
    rng = np.random.default_rng(seed)
    sc = case(rng, model='random', freeSurf=freeSurf, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    sv, pr = problem(sc, visco=visco)
    Wd = 1.7
    H = pr.gauss_newton_diagonal(Wd=Wd, wrt=wrt)
    assert list(H) == list(wrt)
    ref = green_apply_diag(lib, pr, wrt, Wd, list(range(pr.nrow)))
    for k in wrt:
        assert H[k].dtype == np.float64 and H[k].shape == (pr.nrow,)
        assert np.all(np.abs(H[k] - ref[k]) <= 1e-11 * ref[k].max()), k
        assert H[k].min() >= -1e-12 * H[k].max(), k


# 4. end to end: born_dpred and gauss_newton_hvec along e_n ------------------------------------------------------------
@pytest.mark.parametrize('seed,freeSurf,visco,rho,wrt', [(331, (True, False, False, False), False, 'random', ('c', 'rho')),
                                                         (332, (True, False, False, False), True, None, ('c',))])
def test_born_and_hvec(lib, seed, freeSurf, visco, rho, wrt):
    rng = np.random.default_rng(seed)
    sc = case(rng, model='random', freeSurf=freeSurf, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    sv, pr = problem(sc, visco=visco)
    nx, nz, N = sc['nx'], sc['nz'], pr.nrow
    Wd = 1.3
    H = pr.gauss_newton_diagonal(Wd=Wd, wrt=wrt)
    # interior, inside the PML, its inner edge, the boundary column and row, a corner, right under the free surface
    pts = [(5, 6), (1, 1), (3, 3), (4, 0), (nz - 1, 7), (0, 0), (1, 5), (nz - 2, nx - 2)]
    for iz, ix in pts:
        n = iz * nx + ix
        for k in wrt:
            dm = {q: np.zeros(N) for q in wrt}
            dm[k][n] = 1.
            born = Wd * Wd * np.sum(np.abs(pr.born_dpred(dm, wrt=wrt)) ** 2)
            hv = pr.gauss_newton_hvec(dm, Wd=Wd, wrt=wrt)[k][n]
            scale = max(H[k].max(), 1e-300)
            assert abs(H[k][n] - born) <= 1e-10 * scale, (k, iz, ix)
            assert abs(H[k][n] - hv) <= 1e-10 * scale, (k, iz, ix)


# 5. against the oracle: splu fields and Green's functions, a finite-difference dA per node ----------------------------
def oracle_gauss_newton_diagonal(sc, wrt, Wd, visco=False):
    osv = oracle_survey(sc, visco)
    c0 = np.asarray(sc['c']) * np.ones((int(sc['nz']), int(sc['nx'])))
    rho0 = None if sc.get('rho') is None else np.asarray(sc['rho']) * np.ones(c0.shape)
    N = c0.size
    qs = osv.getSources()
    Rv = osv.rVec()
    out = {k: np.zeros(N) for k in wrt}
    for i, f in enumerate(sc['freqs']):
        sub = sub_config(sc, f, c0, rho0, visco)
        lu = spla.splu(sp.csc_matrix(ho.mz_matrix(sub)))
        w = lu.solve(np.asarray(ho.premul(sub, sc.get('hd', False)) * qs[i].toarray(), dtype=np.complex128))
        G = lu.solve(np.asarray(Rv.conj().T.toarray(), dtype=np.complex128), trans='T')
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
                out[k][n] += np.sum(np.abs(G.T @ (dA @ w)) ** 2)
    return {k: Wd * Wd * v for k, v in out.items()}


@pytest.mark.parametrize('seed,visco,rho,wrt,hd', [(341, False, 'random', ('c', 'rho'), True),
                                                   (342, True, None, ('c', 'rho'), False)])
def test_oracle(lib, seed, visco, rho, wrt, hd):
    rng = np.random.default_rng(seed)
    sc = case(rng, nx=9, nz=8, rho=rho)
    sc['geom']['src'] = np.array([[25., 22.], [55., 30.]])
    sc['geom']['rec'] = np.array([[15., 46.], [45., 40.], [65., 42.]])
    if hd:
        sc['hd'] = True
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    import zephyr_b200 as zb
    sv, pr = problem(sc, visco=visco, disc=zb.MiniZephyrHD if hd else None)
    Wd = 0.8
    H = pr.gauss_newton_diagonal(Wd=Wd, wrt=wrt)
    ref = oracle_gauss_newton_diagonal(sc, wrt, Wd, visco=visco)
    for k in wrt:
        assert np.abs(H[k] - ref[k]).max() <= 1e-8 * np.abs(ref[k]).max(), k


# 6. the fused call --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('visco,rho,wrt', [(False, 'random', ('c', 'rho')), (True, None, ('c',)), (False, None, ('rho', 'c'))])
def test_fused(lib, visco, rho, wrt):
    rng = np.random.default_rng(351 + visco)
    sc = case(rng, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    dobs = observed(sc, rng, visco=visco)
    sv, pr = problem(sc, visco=visco)
    Wd = 1.3
    phi, g, H = pr.misfit_gradient_and_gauss_newton_diagonal(dobs, Wd=Wd, wrt=wrt)
    phi0, g0 = pr.misfit_and_adjoint_gradient(dobs, Wd=Wd, wrt=wrt)
    H0 = pr.gauss_newton_diagonal(Wd=Wd, wrt=wrt)
    assert list(g) == list(wrt) and list(H) == list(wrt)
    assert abs(phi - phi0) <= 1e-13 * phi0
    for k in wrt:
        assert rel_l2(g[k], g0[k]) <= 1e-13, k
        assert rel_l2(H[k], H0[k]) <= 1e-13, k
        assert H[k].min() >= -1e-12 * H[k].max(), k


# 7. refusals --------------------------------------------------------------------------------------------------------
def test_refusals(lib):
    import torch
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(361)
    sc = case(rng)
    v = observed(sc, rng)
    for extra in ({'Disc': zb.Eurus, 'theta': 0.1, 'eps': 0.05, 'delta': 0.02}, {'dtype': 'complex64'},
                  {'Disc': zb.MiniZephyr25D, 'nky': 2}):
        sv, pr = problem(dict(sc, **extra), disc=extra.get('Disc'))
        for call in (lambda: pr.gauss_newton_diagonal(), lambda: pr.misfit_gradient_and_gauss_newton_diagonal(v)):
            with pytest.raises(NotImplementedError):
                call()
    rel = case(rng, mode='relative')
    sv, pr = problem(rel)
    for call in (lambda: pr.gauss_newton_diagonal(), lambda: pr.misfit_gradient_and_gauss_newton_diagonal(observed(rel, rng))):
        with pytest.raises(NotImplementedError):
            call()
    sv, pr = problem(sc)
    for bad in ((), ('c', 'c'), ('vp',)):
        for call in (lambda: pr.gauss_newton_diagonal(wrt=bad), lambda: pr.misfit_gradient_and_gauss_newton_diagonal(v, wrt=bad)):
            with pytest.raises(ValueError):
                call()
    # the C ABI
    N = sc['nx'] * sc['nz']
    dev = _lib.torch_device()
    C = torch.zeros(41 * N, dtype=torch.complex128, device=dev)
    G = torch.zeros(13 * N, dtype=torch.complex128, device=dev)
    p = torch.zeros(N, dtype=torch.float64, device=dev)
    pc, pg, pp = _lib.ptr(C), _lib.ptr(G), _lib.ptr(p)
    for d in (zb.MiniZephyr(dict(sc, freq=6., dtype='complex64')), zb.Eurus(dict(sc, freq=6., theta=0.1, eps=0.05, delta=0.02))):
        assert lib.hz_gauss_newton_diag(d.handle, pc, pg, None, None, pp, None) == _lib.HZ_ENOTIMPL
    d = zb.MiniZephyr(dict(sc, freq=6.))
    assert lib.hz_gauss_newton_diag(None, pc, pg, None, None, pp, None) == _lib.HZ_EINVAL
    assert lib.hz_gauss_newton_diag(d.handle, None, pg, None, None, pp, None) == _lib.HZ_EINVAL
    assert lib.hz_gauss_newton_diag(d.handle, pc, None, None, None, pp, None) == _lib.HZ_EINVAL
    assert lib.hz_gauss_newton_diag(d.handle, pc, pg, None, None, None, None) == _lib.HZ_EINVAL
    assert lib.hz_gauss_newton_diag(d.handle, pc, pg, None, None, None, pp) == 0
    _lib.check(lib.hz_set_coefficients(d.handle, _lib.ptr(d.coefficients())), d.handle)
    assert lib.hz_gauss_newton_diag(d.handle, pc, pg, None, None, pp, None) == _lib.HZ_ESTATE


# 8. two gloo ranks shard the frequencies and give the single-rank results ---------------------------------------------
def gloo_case():
    rng = np.random.default_rng(371)
    sc = case(rng, model='random', freqs=(5., 7., 10.))
    return sc, observed(sc, rng)


def gloo_results(pr, v):
    wrt = ('c', 'rho')
    H = pr.gauss_newton_diagonal(Wd=1.2, wrt=wrt)
    phi, g, H2 = pr.misfit_gradient_and_gauss_newton_diagonal(v, Wd=1.2, wrt=wrt)
    return {'H_c': H['c'], 'H_rho': H['rho'], 'phi': np.array([phi]), 'g_c': g['c'], 'H2_rho': H2['rho']}


def test_two_rank_gloo_gauss_newton_diagonal(emu, tmp_path):
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


# 9. the GPU at size: the C4 grid -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_c4_grid_gauss_newton_diagonal(cuda_lib):
    rng = np.random.default_rng(381)
    nx, nz = 500, 1500
    c = layered(nx, nz, 1500., 4500., rng, 5, 50)
    xs = np.linspace(500., 4500., 8)
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': c, 'rho': 1., 'nPML': 20, 'freqs': [3., 7.],
          'geom': {'src': np.stack([xs, np.full(8, 300.)], 1), 'rec': np.stack([np.linspace(250., 4750., 32), np.full(32, 14500.)], 1),
                   'mode': 'fixed', 'rterms': np.exp(1j * np.linspace(0., 2., 32))}}
    sv, pr = problem(sc)
    wrt = ('c', 'rho')
    H = pr.gauss_newton_diagonal(wrt=wrt)
    # PML corners, rows next to each boundary, the PML's inner edge, the receiver depth and the interior
    pts = [(0, 0), (0, nx - 1), (nz - 1, 0), (nz - 1, nx - 1), (1, 1), (1, nx - 2), (nz - 2, 1), (nz - 2, nx - 2),
           (0, 250), (1, 250), (nz - 1, 250), (nz - 2, 250), (750, 0), (750, 1), (750, nx - 1), (750, nx - 2),
           (19, 19), (20, 20), (nz - 21, nx - 21), (30, 120), (1450, 100), (1449, 101)]
    pts += [tuple(int(v) for v in rng.integers([0, 0], [nz, nx])) for _ in range(64 - len(pts))]
    nodes = [iz * nx + ix for iz, ix in pts]
    ref = green_apply_diag(cuda_lib, pr, wrt, 1., nodes)
    for k in wrt:
        assert np.all(np.abs(H[k][nodes] - ref[k]) <= 1e-10 * ref[k].max()), k
        assert H[k].min() >= -1e-12 * H[k].max(), k
    dobs = 0.9 * sv.dpred().reshape((32, 8, 2))
    phi, g, H2 = pr.misfit_gradient_and_gauss_newton_diagonal(dobs, wrt=wrt)
    phi0, g0 = pr.misfit_and_adjoint_gradient(dobs, wrt=wrt)
    assert abs(phi - phi0) <= 1e-13 * phi0
    for k in wrt:
        assert rel_l2(g[k], g0[k]) <= 1e-13 and rel_l2(H2[k], H[k]) <= 1e-13, k


if __name__ == '__main__':
    gloo_rank(sys.argv[1])
