"""Born modelling, its adjoint and Gauss-Newton products (Helm*Problem.born_dpred, born_adjoint, gauss_newton_hvec,
hz_assemble_jvp, hz_stencil_apply) against the oracle and scipy: -Rv conj(splu(A).solve(dA w)) with finite-difference dA,
finite differences of survey.dpred, the dot-product test, consistency with the adjoint-state gradient, symmetry and
positivity of the Gauss-Newton product, the two kernels alone, refusals and a 2-rank gloo run.  Every test runs on the
CPU through the emulation shim (tests/emu) and, marked gpu, through the CUDA library; the C4 grid runs on the GPU only.
Run as a script, the file is one rank of the gloo test."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == '__main__':                                 # one rank of test_two_rank_gloo_born
    sys.path[:0] = [os.path.dirname(HERE), HERE]

from emu_util import emu, emu_cdll  # noqa: F401,E402
from helpers import layered, rel_l2  # noqa: E402
from oracle import helm_oracle as ho  # noqa: E402
from test_adjoint_gradient import (case, crand, fd5, free_port, observed, oracle_survey, problem, smooth,  # noqa: E402
                                   sub_config)


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


def dot(a, b):
    """The real inner product of the data space, Re sum conj(a) b."""
    return float(np.real(np.vdot(np.ravel(a), np.ravel(b))))


def model_dot(a, b):
    return float(sum(np.dot(a[k], b[k]) for k in a))


def perturbation(rng, nz, nx, wrt):
    return {k: (50. if k == 'c' else 40.) * (smooth(rng, nz, nx) + 0.2 * rng.normal(size=(nz, nx))).ravel() for k in wrt}


# ---- oracle side -------------------------------------------------------------------------------------------------
def base_model(sc):
    c0 = np.asarray(sc['c']) * np.ones((int(sc['nz']), int(sc['nx'])))
    gardner = sc.get('rho') is None
    return c0, (None if gardner else np.asarray(sc['rho']) * np.ones(c0.shape))


def oracle_born(sc, dm, visco=False):
    """J dm per frequency: du = conj(-splu(A).solve(dA w)), w = splu(A).solve(premul q), dA the fourth-order central
    difference of ho.mz_matrix along dm, then the receiver taps.  Returns (R, S, F)."""
    osv = oracle_survey(sc, visco)
    c0, rho0 = base_model(sc)
    dc = np.reshape(dm.get('c', np.zeros(c0.size)), c0.shape)
    drho = np.reshape(dm.get('rho', np.zeros(c0.size)), c0.shape)
    qs = osv.getSources()
    hs = [1e-3 * np.abs(c0).max() / np.abs(dc).max()] if np.any(dc) else []
    if np.any(drho):
        hs.append(1e-3 * (rho0.max() if rho0 is not None else 500.) / np.abs(drho).max())
    h = min(hs)
    out = np.zeros((osv.nrec, osv.nsrc, osv.nfreq), dtype=np.complex128)
    for i, f in enumerate(sc['freqs']):
        sub = sub_config(sc, f, c0, rho0, visco)
        lu = spla.splu(sp.csc_matrix(ho.mz_matrix(sub)))
        w = lu.solve(np.asarray(ho.premul(sub, sc.get('hd', False)) * qs[i].toarray(), dtype=np.complex128))

        def A_at(t):
            c = c0 + t * dc
            if rho0 is not None:
                r = rho0 + t * drho
            else:                                          # Gardner's rule on c_f, plus drho when it is perturbed
                r = 310. * np.real(sub_config(sc, f, c, None, visco)['c']) ** 0.25 + t * drho if np.any(drho) else None
            return ho.mz_matrix(sub_config(sc, f, c, r, visco))
        dA = fd5(A_at, h)
        du = np.conj(-lu.solve(np.asarray(dA @ w, dtype=np.complex128)))
        if osv.mode == 'fixed':
            out[:, :, i] = osv.rVec() @ du
        else:
            for s in range(osv.nsrc):
                out[:, s, i] = osv.rVec(s) @ du[:, s]
    return out


def dpred_at(pr, sv, sc, dm, t):
    """survey.dpred at the model sc + t dm, as (R, S, F).  Under Gardner's rule a density perturbation is added to
    310 Re(c)^0.25 (problems without attenuation only)."""
    c0, rho0 = base_model(sc)
    m = {'c': c0 + t * dm['c'].reshape(c0.shape) if 'c' in dm else c0}
    if rho0 is None and 'rho' in dm:
        rho0 = 310. * np.real(m['c']) ** 0.25
    if rho0 is not None:
        m['rho'] = rho0 + t * dm['rho'].reshape(c0.shape) if 'rho' in dm else rho0
    pr.updateModel(m)
    return sv.dpred().reshape((sv.nrec, sv.nsrc, sv.nfreq))


# 1. hz_assemble_jvp alone ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('freeSurf', [None, (True, False, False, True)])
@pytest.mark.parametrize('cplx_c,with_alpha', [(False, False), (True, False), (True, True)])
def test_assemble_jvp(lib, freeSurf, cplx_c, with_alpha):
    """dcoef against a fourth-order difference of the oracle planes, and the exact transpose of hz_assemble_vjp."""
    import torch
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(101 + 4 * cplx_c + 2 * with_alpha + (freeSurf is not None))
    nx, nz = 11, 9
    N = nx * nz
    c = 1800. + 1500. * rng.uniform(size=(nz, nx)) + (1j * 80. * rng.uniform(size=(nz, nx)) if cplx_c else 0.)
    rho = 1700. + 800. * rng.uniform(size=(nz, nx))
    sc = {'nx': nx, 'nz': nz, 'dx': 9., 'dz': 11., 'c': c, 'rho': rho, 'freq': 7. + 0.2j, 'tau': 0.8, 'ky': 0.004, 'nPML': 3}
    if freeSurf:
        sc['freeSurf'] = freeSurf
    d = zb.MiniZephyr(sc)
    dev = d.device
    alpha = (1. + 0.3 * crand(rng, N)) if with_alpha else None
    a2 = np.ones((nz, nx)) if alpha is None else alpha.reshape((nz, nx))
    at = None if alpha is None else torch.from_numpy(alpha).to(dev)
    dc, drho = smooth(rng, nz, nx) + 0.3 * rng.normal(size=(nz, nx)), smooth(rng, nz, nx) + 0.3 * rng.normal(size=(nz, nx))
    dct, drt = (torch.from_numpy(a.ravel().copy()).to(dev) for a in (dc, drho))

    def jvp(dc_t, dr_t):
        out = torch.full((9 * N,), 5. - 3j, dtype=torch.complex128, device=dev)
        assert lib.hz_assemble_jvp(d.handle, _lib.ptr(dc_t), _lib.ptr(dr_t), _lib.ptr(at), _lib.ptr(out)) == 0
        return out.cpu().numpy().reshape((9, N))
    both, only_c, only_r = jvp(dct, drt), jvp(dct, None), jvp(None, drt)

    def planes(c_, r_):
        dd = ho.mz_diagonals(dict(sc, c=c_, rho=r_))
        return np.stack([dd[k].ravel() for k in ho.MZ_KEYS])
    ref = fd5(lambda h: planes(c + h * a2 * dc, rho + h * drho), 2.)
    scale = np.abs(ref).max()
    assert np.abs(both - ref).max() <= 1e-8 * scale
    assert np.abs(only_c + only_r - both).max() <= 1e-14 * scale
    bnd = np.zeros((nz, nx), dtype=bool)
    bnd[0], bnd[-1], bnd[:, 0], bnd[:, -1] = True, True, True, True
    assert not np.any(both[:, bnd.ravel()])                               # identity rows have no tangent
    # the exact transpose of hz_assemble_vjp: Re sum G dcoef = -(g_c . dc + g_rho . drho)
    for _ in range(2):
        G = crand(rng, 9, N)
        Gt = torch.from_numpy(G.ravel().copy()).to(dev)
        gc, gr = torch.zeros(N, dtype=torch.float64, device=dev), torch.zeros(N, dtype=torch.float64, device=dev)
        assert lib.hz_assemble_vjp(d.handle, _lib.ptr(Gt), _lib.ptr(at), _lib.ptr(gc), _lib.ptr(gr)) == 0
        lhs = np.sum(np.real(G * both))
        rhs = -(gc.cpu().numpy() @ dc.ravel() + gr.cpu().numpy() @ drho.ravel())
        assert abs(lhs - rhs) <= 1e-12 * np.sum(np.abs(G * both))


def test_assemble_jvp_refusals(lib):
    import torch
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(111)
    sc = case(rng)
    N = sc['nx'] * sc['nz']
    dev = _lib.torch_device()
    P = torch.zeros(9 * N, dtype=torch.complex128, device=dev)
    dc = torch.zeros(N, dtype=torch.float64, device=dev)
    for d in (zb.MiniZephyr(dict(sc, freq=6., dtype='complex64')), zb.Eurus(dict(sc, freq=6., theta=0.1, eps=0.05, delta=0.02))):
        assert lib.hz_assemble_jvp(d.handle, _lib.ptr(dc), None, None, _lib.ptr(P)) == _lib.HZ_ENOTIMPL
    d = zb.MiniZephyr(dict(sc, freq=6.))
    assert lib.hz_assemble_jvp(None, _lib.ptr(dc), None, None, _lib.ptr(P)) == _lib.HZ_EINVAL
    assert lib.hz_assemble_jvp(d.handle, None, None, None, _lib.ptr(P)) == _lib.HZ_EINVAL
    assert lib.hz_assemble_jvp(d.handle, _lib.ptr(dc), None, None, None) == _lib.HZ_EINVAL
    assert lib.hz_assemble_jvp(d.handle, _lib.ptr(dc), _lib.ptr(dc), None, _lib.ptr(P)) == 0
    _lib.check(lib.hz_set_coefficients(d.handle, _lib.ptr(d.coefficients())), d.handle)
    assert lib.hz_assemble_jvp(d.handle, _lib.ptr(dc), None, None, _lib.ptr(P)) == _lib.HZ_ESTATE


# 2. hz_stencil_apply alone -------------------------------------------------------------------------------------------
def test_stencil_apply_kernel(lib):
    import torch
    from zephyr_b200 import _lib
    rng = np.random.default_rng(121)
    dev = _lib.torch_device()
    for nx, nz, S in ((7, 5, 3), (9, 6, 37), (5, 11, 291)):
        N = nx * nz
        P, u, lam = crand(rng, 9, N), crand(rng, N, S), crand(rng, N, S)
        scale = -0.7 + 0.4j
        Pt, Ut, Lt = (torch.from_numpy(a.copy()).to(dev) for a in (P.ravel(), u, lam))
        Ot = torch.full((N, S), 7. + 7j, dtype=torch.complex128, device=dev)
        assert lib.hz_stencil_apply(_lib.ptr(Pt), _lib.ptr(Ut), nx, nz, S, scale.real, scale.imag, _lib.ptr(Ot), None) == 0
        out = Ot.cpu().numpy()
        wp = np.conj(u).reshape((nz, nx, S))
        Pp = P.reshape((9, nz, nx))
        ref = np.zeros((nz, nx, S), dtype=np.complex128)
        for k in range(9):
            a, q = k // 3 - 1, k % 3 - 1
            ref[1:-1, 1:-1] += Pp[k, 1:-1, 1:-1, None] * wp[1 + a:nz - 1 + a, 1 + q:nx - 1 + q]
        ref *= scale
        assert np.abs(out - ref.reshape((N, S))).max() <= 1e-13 * np.abs(ref).max()
        # duality with hz_stencil_xcorr: sum lam .* apply(P, u) = scale sum G .* P
        Gt = torch.empty(9 * N, dtype=torch.complex128, device=dev)
        assert lib.hz_stencil_xcorr(_lib.ptr(Lt), _lib.ptr(Ut), nx, nz, S, _lib.ptr(Gt), None) == 0
        lhs, rhs = np.sum(lam * out), scale * np.sum(Gt.cpu().numpy() * P.ravel())
        assert abs(lhs - rhs) <= 1e-12 * np.sum(np.abs(lam * out))
    p = _lib.ptr(Pt)                                                    # rejected before any access
    assert lib.hz_stencil_apply(None, p, 4, 4, 1, 1., 0., p, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_apply(p, None, 4, 4, 1, 1., 0., p, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_apply(p, p, 4, 4, 1, 1., 0., None, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_apply(p, p, 2, 4, 1, 1., 0., p, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_apply(p, p, 4, 2, 1, 1., 0., p, None) == _lib.HZ_EINVAL
    assert lib.hz_stencil_apply(p, p, 4, 4, 0, 1., 0., p, None) == _lib.HZ_EINVAL


# 3. born_dpred against the oracle and finite differences of survey.dpred ----------------------------------------------
BORN_CASES = [(131, 'layered', None, 'fixed', False, 'random', ('c',)),
              (132, 'random', (True, False, False, False), 'fixed', False, 'random', ('c', 'rho')),
              (133, 'layered', (True, True, False, True), 'relative', False, 'random', ('rho',)),
              (134, 'layered', None, 'fixed', True, 'random', ('c', 'rho')),
              (135, 'random', (True, False, False, False), 'relative', False, None, ('c', 'rho'))]


def born_case(seed, model, freeSurf, mode, visco, rho):
    rng = np.random.default_rng(seed)
    sc = case(rng, model=model, freeSurf=freeSurf, mode=mode, rho=rho)
    if visco:
        sc.update(Q=30. + 60. * rng.uniform(size=sc['c'].shape), freqBase=5.)
    return rng, sc


@pytest.mark.parametrize('seed,model,freeSurf,mode,visco,rho,wrt', BORN_CASES)
def test_born_dpred_oracle(lib, seed, model, freeSurf, mode, visco, rho, wrt):
    rng, sc = born_case(seed, model, freeSurf, mode, visco, rho)
    sv, pr = problem(sc, visco=visco)
    nz, nx = sc['c'].shape
    dm = perturbation(rng, nz, nx, wrt)
    jd = pr.born_dpred(dm, wrt=wrt)
    assert jd.shape == (sv.nrec, sv.nsrc, sv.nfreq) and jd.dtype == np.complex128
    ref = oracle_born(sc, dm, visco=visco)
    assert np.abs(jd - ref).max() <= 1e-8 * np.abs(ref).max()


@pytest.mark.parametrize('seed,model,freeSurf,mode,visco,rho,wrt', [BORN_CASES[1], BORN_CASES[3], BORN_CASES[4]])
def test_born_dpred_finite_differences(lib, seed, model, freeSurf, mode, visco, rho, wrt):
    rng, sc = born_case(seed, model, freeSurf, mode, visco, rho)
    sv, pr = problem(sc, visco=visco)
    nz, nx = sc['c'].shape
    dm = perturbation(rng, nz, nx, wrt)
    jd = pr.born_dpred(dm, wrt=wrt)
    fd = fd5(lambda t: dpred_at(pr, sv, sc, dm, t), 0.2)
    assert np.abs(jd - fd).max() <= 1e-6 * np.abs(fd).max()


# 4-6. the dot-product test, consistency with the gradient and the Gauss-Newton product ---------------------------------
@pytest.mark.parametrize('seed,model,freeSurf,mode,visco,rho,wrt', [BORN_CASES[1], BORN_CASES[2], BORN_CASES[3], BORN_CASES[4]])
def test_dot_product_and_gauss_newton(lib, seed, model, freeSurf, mode, visco, rho, wrt):
    rng, sc = born_case(seed, model, freeSurf, mode, visco, rho)
    sv, pr = problem(sc, visco=visco)
    nz, nx = sc['c'].shape
    dm1, dm2 = perturbation(rng, nz, nx, wrt), perturbation(rng, nz, nx, wrt)
    jd1 = pr.born_dpred(dm1, wrt=wrt)
    v = np.abs(jd1).max() * crand(rng, *jd1.shape)
    jtv = pr.born_adjoint(v, wrt=wrt)
    assert list(jtv) == list(wrt)
    lhs, rhs = dot(jd1, v), model_dot(dm1, jtv)
    assert abs(lhs - rhs) <= 1e-10 * np.linalg.norm(jd1) * np.linalg.norm(v)
    # the device-resident form of v is accepted as well
    assert all(rel_l2(pr.born_adjoint(pr.upload_dobs(v), wrt=wrt)[k], jtv[k]) <= 1e-14 for k in wrt)
    # H_GN dm = J^H Wd^2 J dm, symmetric, <dm, H dm> = ||Wd J dm||^2
    Wd = 1.3
    h1 = pr.gauss_newton_hvec(dm1, Wd=Wd, wrt=wrt)
    h2 = pr.gauss_newton_hvec(dm2, Wd=Wd, wrt=wrt)
    ref1 = pr.born_adjoint(Wd * Wd * jd1, wrt=wrt)
    for k in wrt:
        assert rel_l2(h1[k], ref1[k]) <= 1e-10, k
    s12, s21 = model_dot(dm1, h2), model_dot(dm2, h1)
    assert abs(s12 - s21) <= 1e-10 * np.sqrt(model_dot(dm1, h1) * model_dot(dm2, h2))
    q = model_dot(dm1, h1)
    assert q > 0 and abs(q - Wd * Wd * dot(jd1, jd1)) <= 1e-10 * q


@pytest.mark.parametrize('visco,rho,wrt', [(False, 'random', ('c', 'rho')), (True, None, ('c',))])
def test_adjoint_is_the_gradient(lib, visco, rho, wrt):
    """born_adjoint(Wd^2 (dpred - dobs)) is the gradient of misfit_and_adjoint_gradient(dobs, Wd)."""
    rng, sc = born_case(141 + visco, 'layered', None, 'fixed', visco, rho)
    dobs = observed(sc, rng, visco=visco)
    sv, pr = problem(sc, visco=visco)
    Wd = 1.7
    phi, g = pr.misfit_and_adjoint_gradient(dobs, Wd=Wd, wrt=wrt)
    d = sv.dpred().reshape(dobs.shape)
    jtv = pr.born_adjoint(Wd * Wd * (d - dobs), wrt=wrt)
    for k in wrt:
        assert rel_l2(jtv[k], g[k]) <= 1e-12, k


def test_factors_reused(lib, monkeypatch):
    """Three solves per frequency on one set of factors: with keepFactors and an unchanged model nothing is refactored."""
    rng, sc = born_case(151, 'layered', None, 'fixed', False, 'random')
    sv, pr = problem(sc)
    nz, nx = sc['c'].shape
    dm = perturbation(rng, nz, nx, ('c',))
    factor, calls = lib.hz_factor, []

    def counting(*a):
        calls.append(a)
        return factor(*a)
    monkeypatch.setattr(lib, 'hz_factor', counting)
    h = pr.gauss_newton_hvec(dm)
    assert len(calls) == len(sc['freqs'])
    h2 = pr.gauss_newton_hvec(dm)
    assert len(calls) == len(sc['freqs'])
    assert np.array_equal(h2['c'], h['c'])
    pr.updateModel(sc['c'] + 10.)
    pr.gauss_newton_hvec(dm)
    assert len(calls) == 2 * len(sc['freqs'])


# 7. refusals ---------------------------------------------------------------------------------------------------------
def test_refusals(lib):
    import zephyr_b200 as zb
    rng = np.random.default_rng(161)
    sc = case(rng)
    nz, nx = sc['c'].shape
    dm = perturbation(rng, nz, nx, ('c',))
    v = observed(sc, rng)
    for extra in ({'Disc': zb.Eurus, 'theta': 0.1, 'eps': 0.05, 'delta': 0.02}, {'dtype': 'complex64'},
                  {'Disc': zb.MiniZephyr25D, 'nky': 2}):
        sv, pr = problem(dict(sc, **extra), disc=extra.get('Disc'))
        for call in (lambda: pr.born_dpred(dm), lambda: pr.born_adjoint(v), lambda: pr.gauss_newton_hvec(dm)):
            with pytest.raises(NotImplementedError):
                call()
    sv, pr = problem(sc)
    for bad in ((), ('c', 'c'), ('vp',)):
        for call in (lambda: pr.born_dpred(dm, wrt=bad), lambda: pr.born_adjoint(v, wrt=bad),
                     lambda: pr.gauss_newton_hvec(dm, wrt=bad)):
            with pytest.raises(ValueError):
                call()
    N = nx * nz
    for bad_dm, wrt in (({}, ('c',)), ({'c': np.ones(N)}, ('c', 'rho')), ({'c': np.ones(N), 'rho': np.ones(N)}, ('c',)),
                        ({'c': np.ones(N - 1)}, ('c',)), ({'c': np.ones(N) + 1j}, ('c',)), (np.ones(N), ('c',))):
        for call in (lambda: pr.born_dpred(bad_dm, wrt=wrt), lambda: pr.gauss_newton_hvec(bad_dm, wrt=wrt)):
            with pytest.raises(ValueError):
                call()
    # a (nz, nx) array is N values too
    a = pr.born_dpred({'c': dm['c'].reshape((nz, nx))})
    assert np.array_equal(a, pr.born_dpred(dm))


# 8. two gloo ranks shard the frequencies and give the single-rank results ---------------------------------------------
def gloo_case():
    rng = np.random.default_rng(171)
    sc = case(rng, model='random', freqs=(5., 7., 10.))
    nz, nx = sc['c'].shape
    dm = perturbation(rng, nz, nx, ('c', 'rho'))
    v = observed(sc, rng)
    return sc, dm, v


def gloo_results(pr, dm, v):
    wrt = ('c', 'rho')
    jd = pr.born_dpred(dm, wrt=wrt)
    jtv = pr.born_adjoint(v, wrt=wrt)
    h = pr.gauss_newton_hvec(dm, Wd=0.8, wrt=wrt)
    return {'jd': jd, 'jtv_c': jtv['c'], 'jtv_rho': jtv['rho'], 'h_c': h['c'], 'h_rho': h['rho']}


def test_two_rank_gloo_born(emu, tmp_path):
    import emu_util
    emu_util.load_emu()                                    # build once, before the ranks race for it
    sc, dm, v = gloo_case()
    sv, pr = problem(sc)
    ref = gloo_results(pr, dm, v)
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
    sc, dm, v = gloo_case()
    sv, pr = problem(sc)
    res = gloo_results(pr, dm, v)
    np.savez(out_path + '.rank%d.npz' % rank, local=np.array(pr.system.localFreqIndices), **res)
    dist.barrier()
    dist.destroy_process_group()


# 9. the GPU at size: the C4 grid -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_c4_grid_born(cuda_lib):
    rng = np.random.default_rng(181)
    nx, nz = 500, 1500
    c = layered(nx, nz, 1500., 4500., rng, 5, 50)
    xs = np.linspace(500., 4500., 8)
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': c, 'rho': 1., 'nPML': 20, 'freqs': [3., 7.],
          'geom': {'src': np.stack([xs, np.full(8, 300.)], 1), 'rec': np.stack([np.linspace(250., 4750., 32), np.full(32, 14500.)], 1),
                   'mode': 'fixed', 'rterms': np.exp(1j * np.linspace(0., 2., 32))}}
    sv, pr = problem(sc)
    dm1, dm2 = {'c': 20. * smooth(rng, nz, nx).ravel()}, {'c': 20. * smooth(rng, nz, nx).ravel()}
    # the dot-product test
    jd1 = pr.born_dpred(dm1)
    v = np.abs(jd1).max() * crand(rng, *jd1.shape)
    assert abs(dot(jd1, v) - model_dot(dm1, pr.born_adjoint(v))) <= 1e-10 * np.linalg.norm(jd1) * np.linalg.norm(v)
    # symmetry of the Gauss-Newton product
    h1, h2 = pr.gauss_newton_hvec(dm1), pr.gauss_newton_hvec(dm2)
    s12, s21 = model_dot(dm1, h2), model_dot(dm2, h1)
    assert abs(s12 - s21) <= 1e-10 * np.sqrt(model_dot(dm1, h1) * model_dot(dm2, h2))
    # at zero residual the Hessian of the misfit is H_GN: a central difference of the gradient along dm
    dobs = sv.dpred().reshape(jd1.shape)
    base = np.asarray(c)

    def grad_at(t):
        pr.updateModel(base + t * dm1['c'].reshape((nz, nx)) / 200.)
        return pr.misfit_and_adjoint_gradient(dobs)[1]['c']
    fd = fd5(grad_at, 1.) * 200.
    pr.updateModel(base)
    assert rel_l2(fd, h1['c']) <= 1e-6


if __name__ == '__main__':
    gloo_rank(sys.argv[1])
