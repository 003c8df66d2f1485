"""Adjoint-state FWI gradient (Helm*Problem.misfit_and_adjoint_gradient, hz_stencil_xcorr, hz_assemble_vjp) against
the oracle and scipy: the adjoint identity -Re sum lambda^T dA w with splu solves and finite-difference dA, finite
differences and Taylor tests of the misfit, the two kernels alone, the viscous problem, refusals and a 2-rank gloo run.
Every test runs on the CPU through the emulation shim (tests/emu) and, marked gpu, through the CUDA library; the C4 grid
runs on the GPU only.  Run as a script, the file is one rank of the gloo test."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == '__main__':                                 # one rank of test_two_rank_gloo
    sys.path[:0] = [os.path.dirname(HERE), HERE]

from emu_util import emu, emu_cdll  # noqa: F401,E402
from helpers import layered, rel_l2  # noqa: E402
from oracle import helm_oracle as ho  # noqa: E402


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


def crand(rng, *s):
    return rng.normal(size=s) + 1j * rng.normal(size=s)


def smooth(rng, nz, nx, k=3):
    """A smooth random field (sum of a few low-order sines), unit scale."""
    z, x = np.mgrid[0:nz, 0:nx]
    out = np.zeros((nz, nx))
    for _ in range(k):
        a, b, p, q = rng.uniform(0.5, 2.5, 4)
        out += rng.normal() * np.sin(np.pi * a * z / nz + p) * np.cos(np.pi * b * x / nx + q)
    return out / np.abs(out).max()


def fd5(f, h):
    """Fourth-order central difference of f at 0."""
    return (8 * (f(h) - f(-h)) - (f(2 * h) - f(-2 * h))) / (12 * h)


# ---- oracle side -------------------------------------------------------------------------------------------------
def sub_config(sc, f, c, rho, visco):
    sub = {k: v for k, v in sc.items() if k not in ('geom', 'sterms', 'Disc', 'freqs', 'Q', 'freqBase')}
    sub['freq'] = f
    sub['c'] = ho.visco_c(np.real(c), sc.get('Q', np.inf), f, sc.get('freqBase', 0.)).reshape(np.shape(c)) if visco else c
    if rho is not None:
        sub['rho'] = rho
    return sub


def oracle_survey(sc, visco=False):
    g = sc['geom']
    return ho.OracleSurvey(sc, sc['freqs'], g['src'], g['rec'], ssTerms=g.get('sterms'), srTerms=g.get('rterms'),
                           tsTerms=sc.get('sterms'), mode=g.get('mode', 'fixed'), visco=visco)


def oracle_phi(sc, dobs, Wd=1., visco=False, c=None, rho=None):
    sc = dict(sc)
    if c is not None:
        sc['c'] = c
    if rho is not None:
        sc['rho'] = rho
    return oracle_survey(sc, visco).misfit(dobs, Wd=Wd)[0]


def oracle_adjoint_dot(sc, dobs, dc, drho, Wd=1., visco=False):
    """-Re sum_f sum_s lambda_s^T dA_f w_s with w = splu(A) (premul q), lambda = splu(A).solve(Rv^H v, trans='T') and dA
    the fourth-order central difference of ho.mz_matrix along (dc, drho)."""
    osv = oracle_survey(sc, visco)
    c0 = np.asarray(sc['c']) * np.ones((int(sc['nz']), int(sc['nx'])))
    rho0 = ho.model_rho(sc_for_rho(sc, c0)) if sc.get('rho') is None else np.asarray(sc['rho']) * np.ones(c0.shape)
    gardner = sc.get('rho') is None
    dobs = np.asarray(dobs).reshape((osv.nrec, osv.nsrc, osv.nfreq))
    qs = osv.getSources()
    total = 0.
    for i, f in enumerate(sc['freqs']):
        sub = sub_config(sc, f, c0, None if gardner else rho0, visco)
        A = ho.mz_matrix(sub)
        lu = spla.splu(sp.csc_matrix(A))
        w = lu.solve(np.asarray(ho.premul(sub, sc.get('hd', False)) * qs[i].toarray(), dtype=np.complex128))
        u = np.conj(w)
        if osv.mode == 'fixed':
            Rv = osv.rVec()
            d = Rv @ u
            v = Wd * Wd * (d - dobs[:, :, i])
            rhs = Rv.conj().T @ v
        else:
            rhs = np.empty_like(u)
            for s in range(osv.nsrc):
                Rv = osv.rVec(s)
                v = Wd * Wd * (Rv @ u[:, s] - dobs[:, s, i])
                rhs[:, s] = Rv.conj().T @ v
        lam = lu.solve(np.asarray(rhs, dtype=np.complex128), trans='T')

        def A_at(h):
            c = c0 + h * dc
            r = None if gardner else rho0 + h * drho
            return ho.mz_matrix(sub_config(sc, f, c, r, visco))
        h = 1e-3 * np.abs(c0).max() / max(np.abs(dc).max(), 1e-300) if np.any(dc) else 1e-3 * rho0.max() / np.abs(drho).max()
        dA = (8 * (A_at(h) - A_at(-h)) - (A_at(2 * h) - A_at(-2 * h))) / (12 * h)
        total += -np.real(np.sum(lam * (dA @ w)))
    return total


def sc_for_rho(sc, c):
    return {'nx': sc['nx'], 'nz': sc['nz'], 'c': c}


def case(rng, nx=12, nz=10, model='layered', rho='random', freeSurf=None, mode='fixed', nPML=3, freqs=(6., 9.)):
    c = layered(nx, nz, 1800., 3600., rng, 2, 4) if model == 'layered' else 2000. + 1200. * rng.uniform(size=(nz, nx))
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 8., 'c': c, 'nPML': nPML, 'freqs': list(freqs),
          'geom': {'src': np.array([[35., 22.], [75., 30.]]), 'rec': np.array([[25., 46.], [55., 50.], [85., 42.]]), 'mode': mode,
                   'sterms': np.array([1. + 0.3j, 0.7 - 0.2j]), 'rterms': np.array([1., 0.5 + 1j, -0.4j])},
          'sterms': np.array([1. + 0.5j, 0.8 - 0.3j, 1.1 + 0.1j])[:len(freqs)]}
    if mode == 'relative':
        sc['geom']['rec'] = np.array([[-10., 16.], [10., 12.], [20., 20.]])
    if rho == 'random':
        sc['rho'] = 1800. + 600. * rng.uniform(size=(nz, nx))
    elif rho is not None:
        sc['rho'] = rho
    if freeSurf is not None:
        sc['freeSurf'] = freeSurf
    return sc


def problem(sc, visco=False, disc=None):
    import zephyr_b200 as zb
    sc = dict(sc, Disc=disc or zb.MiniZephyr)
    sv = zb.Helm2DSurvey(sc)
    pr = (zb.Helm2DViscoProblem if visco else zb.Helm2DProblem)(sc)
    pr.pair(sv)
    return sv, pr


def observed(sc, rng, visco=False):
    d = oracle_survey(sc, visco).dpred()
    return (0.7 * d + 0.05 * np.abs(d).max() * crand(rng, d.size)).reshape((len(sc['geom']['rec']), len(sc['geom']['src']), -1))


# 4. the kernels alone ------------------------------------------------------------------------------------------------
def test_stencil_xcorr_kernel(lib):
    import torch
    from zephyr_b200 import _lib
    rng = np.random.default_rng(1)
    for nx, nz, S in ((7, 5, 3), (9, 6, 37)):
        N = nx * nz
        lam, u = crand(rng, N, S), crand(rng, N, S)
        dev = _lib.torch_device()
        Lt, Ut = (torch.from_numpy(a).to(dev) for a in (lam, u))
        Gt = torch.full((9 * N,), 7. + 7j, dtype=torch.complex128, device=dev)
        assert lib.hz_stencil_xcorr(_lib.ptr(Lt), _lib.ptr(Ut), nx, nz, S, _lib.ptr(Gt), None) == 0
        G = Gt.cpu().numpy().reshape((9, nz, nx))
        wp = np.conj(u).reshape((nz, nx, S))
        L = lam.reshape((nz, nx, S))
        ref = np.zeros((9, nz, nx), dtype=np.complex128)
        for k in range(9):
            a, q = k // 3 - 1, k % 3 - 1
            ref[k, 1:-1, 1:-1] = np.einsum('zxs,zxs->zx', L[1:-1, 1:-1], wp[1 + a:nz - 1 + a, 1 + q:nx - 1 + q])
        assert np.abs(G - ref).max() <= 1e-13 * np.abs(ref).max()
    p = _lib.ptr(Gt)                                                    # rejected before any access
    assert lib.hz_stencil_xcorr(None, p, 4, 4, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_xcorr(p, p, 2, 4, 1, p, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_xcorr(p, p, 4, 4, 0, p, None) == _lib.HZ_EINVAL


@pytest.mark.parametrize('freeSurf', [None, (True, False, False, True)])
@pytest.mark.parametrize('cplx_c,with_alpha', [(False, False), (True, True)])
def test_assemble_vjp_dot(lib, freeSurf, cplx_c, with_alpha):
    """sum Re(G dcoef) against -(g_c . dc) and -(g_rho . drho), dcoef by a fourth-order difference of the oracle planes."""
    import torch
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(3 + 2 * cplx_c + (freeSurf is not None))
    nx, nz = 11, 9
    c = 1800. + 1500. * rng.uniform(size=(nz, nx)) + (1j * 80. * rng.uniform(size=(nz, nx)) if cplx_c else 0.)
    rho = 1700. + 800. * rng.uniform(size=(nz, nx))
    sc = {'nx': nx, 'nz': nz, 'dx': 9., 'dz': 11., 'c': c, 'rho': rho, 'freq': 7. + 0.2j, 'tau': 0.8, 'ky': 0.004, 'nPML': 3}
    if freeSurf:
        sc['freeSurf'] = freeSurf
    d = zb.MiniZephyr(sc)
    dev = d.device
    N = nx * nz
    G = crand(rng, 9, N)
    alpha = (1. + 0.3 * crand(rng, N)) if with_alpha else None
    gc, gr = torch.zeros(N, dtype=torch.float64, device=dev), torch.zeros(N, dtype=torch.float64, device=dev)
    Gt = torch.from_numpy(G.ravel().copy()).to(dev)
    at = None if alpha is None else torch.from_numpy(alpha).to(dev)
    assert lib.hz_assemble_vjp(d.handle, _lib.ptr(Gt), _lib.ptr(at), _lib.ptr(gc), _lib.ptr(gr)) == 0
    gc, gr = gc.cpu().numpy(), gr.cpu().numpy()
    dc, drho = smooth(rng, nz, nx) + 0.3 * rng.normal(size=(nz, nx)), smooth(rng, nz, nx) + 0.3 * rng.normal(size=(nz, nx))
    a2 = np.ones((nz, nx)) if alpha is None else alpha.reshape((nz, nx))

    def planes(c_, r_):
        dd = ho.mz_diagonals(dict(sc, c=c_, rho=r_))
        return np.stack([dd[k].ravel() for k in ho.MZ_KEYS])
    dP_c = fd5(lambda h: planes(c + h * a2 * dc, rho), 1e-3 * 3000.)
    dP_r = fd5(lambda h: planes(c, rho + h * drho), 1e-3 * 2500.)
    lhs_c, lhs_r = np.sum(np.real(G * dP_c)), np.sum(np.real(G * dP_r))
    assert abs(-gc @ dc.ravel() - lhs_c) <= 1e-8 * np.sum(np.abs(G * dP_c))
    assert abs(-gr @ drho.ravel() - lhs_r) <= 1e-8 * np.sum(np.abs(G * dP_r))
    # accumulation, one output only, and the argument checks
    gc2 = torch.from_numpy(gc.copy()).to(dev)
    assert lib.hz_assemble_vjp(d.handle, _lib.ptr(Gt), _lib.ptr(at), _lib.ptr(gc2), None) == 0
    assert np.allclose(gc2.cpu().numpy(), 2 * gc, rtol=1e-14, atol=0)
    assert lib.hz_assemble_vjp(d.handle, _lib.ptr(Gt), None, None, None) == _lib.HZ_EINVAL
    assert lib.hz_assemble_vjp(d.handle, None, None, _lib.ptr(gc2), None) == _lib.HZ_EINVAL
    assert lib.hz_assemble_vjp(None, _lib.ptr(Gt), None, _lib.ptr(gc2), None) == _lib.HZ_EINVAL
    _lib.check(lib.hz_set_coefficients(d.handle, _lib.ptr(d.coefficients())), d.handle)
    assert lib.hz_assemble_vjp(d.handle, _lib.ptr(Gt), None, _lib.ptr(gc2), None) == _lib.HZ_ESTATE


# 1. the oracle adjoint identity on small grids ------------------------------------------------------------------------
@pytest.mark.parametrize('seed,model,freeSurf,mode', [(11, 'layered', None, 'fixed'), (12, 'random', (True, False, False, False), 'fixed'),
                                                      (13, 'layered', (True, True, False, True), 'relative'), (14, 'random', None, 'relative')])
def test_adjoint_identity(lib, seed, model, freeSurf, mode):
    rng = np.random.default_rng(seed)
    sc = case(rng, model=model, freeSurf=freeSurf, mode=mode)
    dobs = observed(sc, rng)
    sv, pr = problem(sc)
    Wd = 1.7
    phi, g = pr.misfit_and_adjoint_gradient(dobs, Wd=Wd, wrt=('c', 'rho'))
    assert sorted(g) == ['c', 'rho']
    assert abs(phi - oracle_phi(sc, dobs, Wd=Wd)) <= 1e-11 * phi
    nz, nx = sc['c'].shape
    for k in range(2):
        dc, drho = 50. * smooth(rng, nz, nx), 40. * smooth(rng, nz, nx)
        ref_c = oracle_adjoint_dot(sc, dobs, dc, 0 * drho, Wd=Wd)
        ref_r = oracle_adjoint_dot(sc, dobs, 0 * dc, drho, Wd=Wd)
        assert abs(g['c'] @ dc.ravel() - ref_c) <= 1e-8 * abs(ref_c)
        assert abs(g['rho'] @ drho.ravel() - ref_r) <= 1e-8 * abs(ref_r)
    phi2, g2 = pr.misfit_and_adjoint_gradient(dobs, Wd=Wd, wrt=('rho',))
    assert phi2 == phi and list(g2) == ['rho'] and np.array_equal(g2['rho'], g['rho'])


# 2. finite differences of phi: directions and single nodes ------------------------------------------------------------
def test_finite_differences(lib):
    rng = np.random.default_rng(21)
    sc = case(rng, nx=13, nz=11, model='random', freeSurf=(True, False, False, False))
    dobs = observed(sc, rng)
    sv, pr = problem(sc)
    phi, g = pr.misfit_and_adjoint_gradient(dobs, wrt=('c', 'rho'))
    c0, r0 = sc['c'], sc['rho']
    nz, nx = c0.shape
    for k in range(3):
        dc, drho = smooth(rng, nz, nx), smooth(rng, nz, nx) * (k > 0)
        fd = fd5(lambda h: oracle_phi(sc, dobs, c=c0 + 30. * h * dc, rho=r0 + 20. * h * drho), 1.)
        ad = 30. * g['c'] @ dc.ravel() + 20. * g['rho'] @ drho.ravel()
        assert abs(ad - fd) <= 1e-6 * abs(fd), k
    # interior, inside the PML, on the identity boundary next to the first interior column, under the free surface
    for (iz, ix) in [(6, 6), (1, 5), (8, 11), (5, 0), (1, 7), (0, 6)]:
        e = np.zeros((nz, nx))
        e[iz, ix] = 1.
        fd_c = fd5(lambda h: oracle_phi(sc, dobs, c=c0 + h * e), 5.)
        fd_r = fd5(lambda h: oracle_phi(sc, dobs, rho=r0 + h * e), 5.)
        scale = max(abs(fd_c), 1e-3 * np.abs(g['c']).max())
        assert abs(g['c'][iz * nx + ix] - fd_c) <= 1e-6 * scale, (iz, ix)
        scale = max(abs(fd_r), 1e-3 * np.abs(g['rho']).max())
        assert abs(g['rho'][iz * nx + ix] - fd_r) <= 1e-6 * scale, (iz, ix)


# 3. Taylor test: the remainder falls at rate 2 ------------------------------------------------------------------------
def taylor_slopes(pr, sc, dobs, dc, hs):
    phi0, g = pr.misfit_and_adjoint_gradient(dobs)
    gd = g['c'] @ dc.ravel()
    rem = []
    for h in hs:
        pr.updateModel(sc['c'] + h * dc)
        rem.append(abs(pr.misfit_and_adjoint_gradient(dobs)[0] - phi0 - h * gd))
    pr.updateModel(sc['c'])
    return np.diff(np.log(rem)) / np.diff(np.log(hs))


def test_taylor(lib):
    rng = np.random.default_rng(31)
    sc = case(rng, nx=14, nz=12, model='layered')
    dobs = observed(sc, rng)
    sv, pr = problem(sc)
    slopes = taylor_slopes(pr, sc, dobs, 100. * smooth(rng, 12, 14), [0.1, 0.05, 0.025, 0.0125])
    assert np.all((slopes > 1.9) & (slopes < 2.1)), slopes


# 5. the viscous problem, Gardner density and the half-differentiated source -------------------------------------------
@pytest.mark.parametrize('freqBase', [0., 5.])
def test_visco(lib, freqBase):
    import zephyr_b200 as zb
    rng = np.random.default_rng(41)
    sc = case(rng, model='layered')
    sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=freqBase)
    dobs = observed(sc, rng, visco=True)
    sv, pr = problem(sc, visco=True)
    phi, g = pr.misfit_and_adjoint_gradient(dobs, wrt=('rho', 'c'))
    assert list(g) == ['rho', 'c']
    assert abs(phi - oracle_phi(sc, dobs, visco=True)) <= 1e-11 * phi
    nz, nx = sc['c'].shape
    dc = smooth(rng, nz, nx)
    fd = fd5(lambda h: oracle_phi(sc, dobs, visco=True, c=sc['c'] + 30. * h * dc), 1.)
    assert abs(30. * g['c'] @ dc.ravel() - fd) <= 1e-6 * abs(fd)
    assert abs(30. * g['c'] @ dc.ravel() - oracle_adjoint_dot(sc, dobs, 30. * dc, 0 * dc, visco=True)) <= 1e-8 * abs(fd)
    # premul of the half-differentiated operator is divided out of the adjoint source
    sc_hd = dict(sc, hd=True)
    sv, pr = problem(sc_hd, visco=True, disc=zb.MiniZephyrHD)
    phi, g = pr.misfit_and_adjoint_gradient(dobs)
    ref = oracle_adjoint_dot(sc_hd, dobs, 30. * dc, 0 * dc, visco=True)
    assert abs(30. * g['c'] @ dc.ravel() - ref) <= 1e-8 * abs(ref)


def test_gardner_density(lib):
    """rho not given: rho = 310 Re(c)^0.25 follows c, and g_c is the total derivative."""
    rng = np.random.default_rng(51)
    sc = case(rng, model='random', rho=None)
    dobs = observed(sc, rng)
    sv, pr = problem(sc)
    phi, g = pr.misfit_and_adjoint_gradient(dobs, wrt=('c', 'rho'))
    nz, nx = sc['c'].shape
    dc = smooth(rng, nz, nx)
    fd = fd5(lambda h: oracle_phi(sc, dobs, c=sc['c'] + 30. * h * dc), 1.)
    assert abs(30. * g['c'] @ dc.ravel() - fd) <= 1e-6 * abs(fd)
    r0 = 310. * sc['c'] ** 0.25
    fd_r = fd5(lambda h: oracle_phi(sc, dobs, rho=r0 + 20. * h * dc), 1.)
    assert abs(20. * g['rho'] @ dc.ravel() - fd_r) <= 1e-6 * abs(fd_r)


# 7. refusals ----------------------------------------------------------------------------------------------------------
def test_refusals(lib):
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(61)
    sc = case(rng)
    dobs = observed(sc, rng)
    for extra in ({'Disc': zb.Eurus, 'theta': 0.1, 'eps': 0.05, 'delta': 0.02}, {'dtype': 'complex64'},
                  {'Disc': zb.MiniZephyr25D, 'nky': 2}):
        s = dict(sc, **extra)
        sv, pr = problem(s, disc=extra.get('Disc'))
        with pytest.raises(NotImplementedError):
            pr.misfit_and_adjoint_gradient(dobs)
    sv, pr = problem(sc)
    for bad in ((), ('c', 'c'), ('vp',)):
        with pytest.raises(ValueError):
            pr.misfit_and_adjoint_gradient(dobs, wrt=bad)
    # the ABI: complex64 and Eurus handles are refused
    import torch
    dev = _lib.torch_device()
    N = sc['nx'] * sc['nz']
    G = torch.zeros(9 * N, dtype=torch.complex128, device=dev)
    g = torch.zeros(N, dtype=torch.float64, device=dev)
    for d in (zb.MiniZephyr(dict(sc, freq=6., dtype='complex64')), zb.Eurus(dict(sc, freq=6., theta=0.1, eps=0.05, delta=0.02))):
        assert lib.hz_assemble_vjp(d.handle, _lib.ptr(G), None, _lib.ptr(g), None) == _lib.HZ_ENOTIMPL


# 6. the GPU at size: the C4 grid -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_c4_grid(cuda_lib):
    rng = np.random.default_rng(71)
    nx, nz = 500, 1500
    c = layered(nx, nz, 1500., 4500., rng, 5, 50)
    xs = np.linspace(500., 4500., 8)
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': c, 'rho': 1., 'nPML': 20, 'freqs': [3., 7.],
          'geom': {'src': np.stack([xs, np.full(8, 300.)], 1), 'rec': np.stack([np.linspace(250., 4750., 32), np.full(32, 14500.)], 1),
                   'mode': 'fixed', 'rterms': np.exp(1j * np.linspace(0., 2., 32))}}
    dobs = observed(sc, rng)
    sv, pr = problem(sc)
    phi, g = pr.misfit_and_adjoint_gradient(dobs)
    phi_ref, _ = pr.misfit_and_gradient(dobs)
    assert abs(phi - phi_ref) <= 1e-12 * phi_ref
    dc = 50. * smooth(rng, nz, nx)
    ref = oracle_adjoint_dot(dict(sc, rho=np.ones((nz, nx))), dobs, dc, 0 * dc)
    assert abs(g['c'] @ dc.ravel() - ref) <= 1e-8 * abs(ref)


@pytest.mark.gpu
def test_taylor_gpu(cuda_lib):
    rng = np.random.default_rng(32)
    sc = case(rng, nx=120, nz=200, model='layered', nPML=10, freqs=(4., 7., 9.))
    sc['geom'] = {'src': np.array([[300., 100.], [800., 150.]]), 'rec': np.stack([np.linspace(100., 1100., 12), np.full(12, 1500.)], 1)}
    dobs = observed(sc, rng)
    sv, pr = problem(sc)
    slopes = taylor_slopes(pr, sc, dobs, 100. * smooth(rng, 200, 120), [0.1, 0.05, 0.025, 0.0125])
    assert np.all((slopes > 1.9) & (slopes < 2.1)), slopes


@pytest.mark.gpu
def test_concurrent_workers_gpu(cuda_lib):
    """Four frequencies swept on four worker streams give the gradient of one stream, on the first call of a problem
    (when the shared adjoint-source taps are formed) and on the next one; both geometries, HD premul."""
    import zephyr_b200 as zb
    rng = np.random.default_rng(33)
    for mode in ('fixed', 'relative'):
        sc = case(rng, nx=60, nz=80, model='layered', nPML=8, freqs=(4., 5., 6.5, 8.), mode=mode)
        sc['sterms'] = np.ones(4, dtype=np.complex128)
        sc['geom']['src'] = np.array([[150., 100.], [350., 120.], [450., 90.]])
        sc['geom']['sterms'] = np.ones(3, dtype=np.complex128)
        if mode == 'fixed':
            sc['geom']['rec'] = np.stack([np.linspace(60., 540., 8), np.full(8, 560.)], 1)
        else:
            sc['geom']['rec'] = np.stack([np.linspace(-40., 40., 8), np.full(8, 300.)], 1)
        sc['geom']['rterms'] = np.exp(1j * np.linspace(0., 1., 8))
        dobs = observed(sc, rng)
        ref = problem(dict(sc, solveWorkers=1, factorWorkers=1), disc=zb.MiniZephyrHD)[1].misfit_and_adjoint_gradient(dobs, wrt=('c', 'rho'))
        pr = problem(sc, disc=zb.MiniZephyrHD)[1]
        assert pr._workers(pr._device_ops()['s_z']) == 4
        for _ in range(2):
            phi, g = pr.misfit_and_adjoint_gradient(dobs, wrt=('c', 'rho'))
            assert abs(phi - ref[0]) <= 1e-12 * ref[0]
            assert rel_l2(g['c'], ref[1]['c']) <= 1e-12 and rel_l2(g['rho'], ref[1]['rho']) <= 1e-12


# 6. two gloo ranks shard the frequencies and all-reduce the same gradient --------------------------------------------
def gloo_case():
    rng = np.random.default_rng(81)
    sc = case(rng, model='random', freqs=(5., 7., 10.))
    return sc, observed(sc, rng)


def free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_rank_gloo(emu, tmp_path):
    import emu_util
    emu_util.load_emu()                                    # build once, before the ranks race for it
    sc, dobs = gloo_case()
    sv, pr = problem(sc)
    phi, g = pr.misfit_and_adjoint_gradient(dobs, wrt=('c', 'rho'))
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
        assert abs(float(z['phi']) - phi) <= 1e-13 * phi
        assert rel_l2(z['g_c'], g['c']) <= 1e-13 and rel_l2(z['g_rho'], g['rho']) <= 1e-13
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
    sc, dobs = gloo_case()
    sv, pr = problem(sc)
    phi, g = pr.misfit_and_adjoint_gradient(dobs, wrt=('c', 'rho'))
    np.savez(out_path + '.rank%d.npz' % rank, phi=phi, g_c=g['c'], g_rho=g['rho'], local=np.array(pr.system.localFreqIndices))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    gloo_rank(sys.argv[1])
