"""Transposed and conjugate-transposed solves (A^T x = b, A^H x = b) from the block factors of A: the op(A) tiles of the
DMMA contraction, Disc.solve(rhs, trans), Solver(A).solve(rhs, trans) and hz_solve_op, against numpy / scipy's splu.
Every test runs on the CPU through the emulation shim (tests/emu) and, marked gpu, through the CUDA library; the large
sizes run on the GPU only."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from emu_util import emu_cdll  # noqa: F401
from helpers import SC_KEYS, layered, max_col_rel_l2, rel_l2, sc_from_golden
from oracle import helm_oracle as ho

OPS = {'N': 0, 'T': 1, 'H': 2}


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
    """The CUDA build only: sizes the emulation cannot run in test time."""
    from zephyr_b200 import _lib
    return _lib.get_lib()


def crand(rng, *s):
    return rng.normal(size=s) + 1j * rng.normal(size=s)


def op_dense(A, trans):
    return {'N': A, 'T': A.T, 'H': A.conj().T}[trans]


def zgemm_op(lib, M, N, K, alpha, A, lda, opa, B, beta, Cm, tile, m3):
    """hz_zgemm_op on device copies of the numpy operands; returns the new C."""
    import torch
    from zephyr_b200 import _lib
    dev = _lib.torch_device()
    At, Bt, Ct = (torch.from_numpy(np.array(x, dtype=np.complex128)).to(dev) for x in (A, B, Cm))      # copies: C is written
    assert lib.hz_zgemm_op(M, N, K, alpha, _lib.ptr(At), lda, opa, _lib.ptr(Bt), N, beta, _lib.ptr(Ct), N, tile, m3, None) == 0
    if dev.type == 'cuda':
        torch.cuda.synchronize()
    return Ct.cpu().numpy()


# 1. every tile the host can pick (0..6 of kGemmTiles, -1 = its own pick) x op(A) x product form, odd M / N / K included
@pytest.mark.parametrize('tile,M,N,K', [(0, 70, 45, 37), (1, 60, 66, 16), (2, 50, 64, 16), (3, 81, 64, 40), (4, 33, 70, 9), (5, 32, 32, 32),
                                        (6, 17, 35, 50), (-1, 40, 24, 40)])
@pytest.mark.parametrize('m3', [0, 1])
@pytest.mark.parametrize('trans', ['N', 'T', 'H'])
def test_zgemm_op(lib, trans, m3, tile, M, N, K):
    rng = np.random.default_rng(100 + tile)
    opa = OPS[trans]
    pad = 3                                                              # row stride of the stored A > its width
    stored = crand(rng, M, K + pad) if trans == 'N' else crand(rng, K, M + pad)
    A = op_dense(stored[:, :K] if trans == 'N' else stored[:, :M], trans)   # op(A), M x K
    B, C0 = crand(rng, K, N), crand(rng, M, N)
    lda = stored.shape[1]
    Cm = zgemm_op(lib, M, N, K, -1.0, stored, lda, opa, B, 1, C0, tile, m3)
    assert np.abs(Cm - (C0 - A @ B)).max() < 1e-12
    Cm = zgemm_op(lib, M, N, K, 1.0, stored, lda, opa, B, 0, Cm, tile, m3)
    assert np.abs(Cm - A @ B).max() < 1e-12


def test_zgemm_op_rejects(lib):
    from zephyr_b200 import _lib
    z = np.zeros(16, dtype=np.complex128)
    p = _lib.ptr(z)
    assert lib.hz_zgemm_op(2, 2, 2, 1.0, p, 2, 3, p, 2, 0, p, 2, -1, 1, None) == _lib.HZ_EINVAL      # op
    assert lib.hz_zgemm_op(2, 2, 2, 1.0, p, 2, 1, p, 2, 0, p, 2, 7, 1, None) == _lib.HZ_EINVAL       # tile
    assert lib.hz_zgemm_op(2, 2, 2, 1.0, p, 2, 1, p, 2, 0, p, 2, -1, 2, None) == _lib.HZ_EINVAL      # product form


@pytest.mark.gpu
@pytest.mark.parametrize('m3', [0, 1])
@pytest.mark.parametrize('trans', ['N', 'T', 'H'])
def test_zgemm_op_large(cuda_lib, trans, m3):
    """The substitution shape of C3 (b = 1000, S = 512) with the host's tile pick."""
    rng = np.random.default_rng(7)
    M, N, K = 1000, 512, 1000
    stored = crand(rng, M, K)
    B = crand(rng, K, N)
    ref = op_dense(stored, trans) @ B
    Cm = zgemm_op(cuda_lib, M, N, K, 1.0, stored, K, OPS[trans], B, 0, np.zeros((M, N), dtype=np.complex128), -1, m3)
    assert np.abs(Cm - ref).max() < 1e-11 * np.abs(ref).max()


# 2. Disc.solve(rhs, trans) against splu(A).solve(rhs, trans), A from the golden coefficient planes
def golden_matrix(g, eurus):
    nx, nz = int(g['nx']), int(g['nz'])
    if not eurus:
        return ho._diags_to_csr({k: g['planes'][s] for s, k in enumerate(ho.MZ_KEYS)}, ho.MZ_KEYS, ho.mz_offsets(nx), nx * nz)
    M = [ho._diags_to_csr({k: q[s] for s, k in enumerate(ho.EU_KEYS)}, ho.EU_KEYS, ho.eurus_offsets(nx), nx * nz) for q in g['quads']]
    return sp.bmat([[M[0], M[1]], [M[2], M[3]]])


def splu_disc(lu, rhs, trans, premul, nrows):
    """What Disc.solve(rhs, trans) returns: conj(splu(A).solve(premul * rhs, trans)), N-row Eurus rhs zero-padded."""
    rhs = rhs.toarray() if sp.issparse(rhs) else np.asarray(rhs)
    pad = rhs.shape[0] < nrows
    if pad:
        rhs = np.vstack([rhs, np.zeros(rhs.shape, dtype=np.complex128)])
    u = lu.solve(np.asarray(premul * rhs, dtype=np.complex128), trans=trans).conjugate()
    return u[:nrows // 2] if pad else u


@pytest.mark.parametrize('name,disc', [('mz_plain', 'MiniZephyr'), ('mz_freesurf_all', 'MiniZephyrHD'), ('mz_tau_ky', 'MiniZephyr'),
                                       ('eurus_iso', 'EurusHD'), ('eurus_tti', 'Eurus')])
def test_disc_solve_trans_golden(lib, golden, name, disc):
    import zephyr_b200 as zb
    g = golden(name)
    eurus = disc.startswith('Eurus')
    A = golden_matrix(g, eurus)
    assert sp.linalg.norm(A - A.T) > 1e-6 * sp.linalg.norm(A)          # the operator is not symmetric
    lu = spla.splu(sp.csc_matrix(A))
    sc = sc_from_golden(g, SC_KEYS)
    d = getattr(zb, disc)(sc)
    rng = np.random.default_rng(5)
    n = int(g['nx']) * int(g['nz'])                                    # Eurus: N-row right-hand sides, zero-padded to 2N
    rhs = np.hstack([ho.sparse_kaiser_source(sc, g['locs']).toarray(), crand(rng, n, 1)])
    for trans in ('T', 'H', 'N'):
        ref = splu_disc(lu, rhs, trans, d.premul, A.shape[0])
        assert max_col_rel_l2(d.solve(rhs, trans), ref) <= 1e-10, trans
        if eurus:
            assert d.last_residual < 1e-12                              # the refinement step ran on the op(A) residual


# 3. twist, checkpointed factors and right-hand sides confined to a depth range (sweep skipping)
@pytest.mark.parametrize('k,twist', [(1, 'mid'), (1, 'source'), (1, 3), (2, 'mid'), (3, 'source'), (3, 15)])
def test_trans_twist_checkpoints_depth_range(lib, k, twist):
    import zephyr_b200 as zb
    rng = np.random.default_rng(4)
    nx, nz = 8, 21
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': 2000. + 800. * rng.uniform(size=(nz, nx)), 'rho': 1., 'freq': 11., 'nPML': 3,
          'storeEvery': k, 'twist': twist}
    lu = spla.splu(sp.csc_matrix(ho.mz_matrix(sc)))
    d = zb.MiniZephyr(sc)
    shallow = ho.sparse_kaiser_source(sc, np.array([[40., 20.], [50., 30.]]))       # block rows 0..7
    deep = ho.sparse_kaiser_source(sc, np.array([[30., 180.]]))                     # block rows 14..20
    assert d.rhs_depth_range(shallow)[1] < nz // 2 < d.rhs_depth_range(deep)[0]
    for trans in ('T', 'H'):
        for rhs in (shallow, deep, crand(rng, nx * nz, 2)):
            assert max_col_rel_l2(d.solve(rhs, trans), splu_disc(lu, rhs, trans, 1.0, nx * nz)) <= 1e-10, (trans, rhs.shape)
    if k > 1:
        assert d.factor_bytes() < 0.8 * zb.MiniZephyr(dict(sc, storeEvery=1)).factor_bytes()


# 4. the Solver shim: SuperLU.solve(rhs, trans) semantics
def test_solver_shim_trans(lib):
    import zephyr_b200 as zb
    rng = np.random.default_rng(3)
    nx, nz = 9, 7
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': 2000. + 500. * rng.uniform(size=(nz, nx)), 'rho': 1., 'freq': 9., 'nPML': 3}
    for A, nxa, tol in ((ho.mz_matrix(sc), None, 1e-12), (ho.eurus_matrix(dict(sc, theta=0.2, eps=0.1, delta=0.05)), nx, 1e-9)):
        lu = spla.splu(A.tocsc())
        s = zb.BlockTridiagonalSolver(A, nx=nxa)
        rhs = crand(rng, A.shape[0], 2)
        for trans in ('N', 'T', 'H'):
            assert max_col_rel_l2(s.solve(rhs, trans), lu.solve(rhs, trans=trans)) < tol, trans
            assert max_col_rel_l2(s.solve(rhs[:, 0], trans=trans), lu.solve(rhs[:, 0], trans=trans)) < tol
        assert np.array_equal(s * rhs, s.solve(rhs))
        with pytest.raises(ValueError):
            s.solve(rhs, 'X')


# 5. the accuracy probe after a factorisation runs for a transposed first solve, on the op(A) residual
@pytest.mark.parametrize('trans', ['T', 'H'])
def test_probe_on_transposed_solve(lib, trans):
    import zephyr_b200 as zb
    rng = np.random.default_rng(2)
    nx, nz = 14, 12
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 8., 'c': layered(nx, nz, 1500., 4000., rng, 2, 4),
          'rho': layered(nx, nz, 1800., 2600., rng, 2, 4), 'freq': 11., 'nPML': 3}
    d = zb.MiniZephyr(sc)
    assert d.last_probe == -1.0
    q = ho.sparse_kaiser_source(sc, np.array([[40., 24.]]))
    u = d.solve(q, trans)
    # an A residual of this solution would be ~ the asymmetry of A (> 1e-7: the probe would have failed)
    assert 0. <= d.last_probe < 1e-12
    x = np.conj(u[:, 0])
    A = ho.mz_matrix(sc)
    assert rel_l2(A @ x, q.toarray()[:, 0]) > 1e-6
    assert rel_l2(op_dense(A, trans) @ x, q.toarray()[:, 0]) < 1e-12


# 6. complex64 handles: N only
def test_complex64_trans_not_implemented(lib):
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    rng = np.random.default_rng(8)
    nx, nz = 10, 8
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': layered(nx, nz, 1500., 4000., rng, 2, 3), 'rho': 1., 'freq': 9., 'nPML': 3,
          'dtype': 'complex64'}
    d = zb.MiniZephyr(sc)
    q = crand(rng, nx * nz, 1)
    for trans in ('T', 'H'):
        with pytest.raises(NotImplementedError):
            d.solve(q, trans)
    assert max_col_rel_l2(d.solve(q), ho.OracleDisc(sc) * q) < 1e-4
    s = zb.BlockTridiagonalSolver(ho.mz_matrix(sc), dtype='complex64')
    with pytest.raises(NotImplementedError):
        s.solve(q, 'T')
    with pytest.raises(ValueError):
        d.solve(q, 'X')
    assert lib.hz_solve_op(d.handle, 3, _lib.ptr(np.zeros(1)), 1, 1., 0., 0, -1, -1, 0, None) == _lib.HZ_EINVAL


# 7. solve(rhs) is Disc * rhs, bit for bit
@pytest.mark.parametrize('disc', ['MiniZephyrHD', 'EurusHD'])
def test_solve_n_is_mul(lib, disc):
    import zephyr_b200 as zb
    rng = np.random.default_rng(9)
    nx, nz = 9, 10
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': layered(nx, nz, 2000., 3500., rng, 2, 4), 'rho': 1., 'freq': 9., 'nPML': 3,
          'theta': 0.2, 'eps': 0.1, 'delta': 0.05}
    d = getattr(zb, disc)(sc)
    q = ho.sparse_kaiser_source(sc, np.array([[40., 30.], [60., 50.]]))
    assert np.array_equal(d.solve(q), d * q)
    qd = crand(rng, d.shape[0] if disc.startswith('Eurus') else nx * nz, 2)
    assert np.array_equal(d.solve(qd), d * qd)
    with pytest.raises(NotImplementedError):
        zb.MiniZephyr25D(dict(sc, nky=2)).solve(q, 'T')


# 8/9/10. large grids on the GPU: op(A) stencil residual and the bilinear identities between the N and T / H paths
@pytest.mark.gpu
@pytest.mark.parametrize('disc,nx,nz', [('MiniZephyr', 1000, 3000), ('Eurus', 200, 400)])
def test_trans_large_residual_and_identity(cuda_lib, disc, nx, nz):
    import torch
    import zephyr_b200 as zb
    rng = np.random.default_rng(0)
    sc = {'nx': nx, 'nz': nz, 'dx': 10., 'dz': 10., 'c': layered(nx, nz, 1500., 4500., rng, 5, 50), 'rho': 1., 'freq': 4., 'nPML': 20}
    if disc == 'Eurus':
        sc.update(theta=layered(nx, nz, 0., 0.4, rng, 5, 50), eps=layered(nx, nz, 0., 0.2, rng, 5, 50), delta=layered(nx, nz, 0., 0.1, rng, 5, 50))
    d = getattr(zb, disc)(sc)
    A = d.A                                                             # op(A) from hz_get_coefficients
    n = A.shape[0]
    b = crand(rng, n, 2)
    w, c = crand(rng, n), crand(rng, n)

    def solve(rhs, trans):                                              # op(A)^-1 rhs: no premul (1), no conjugation
        X = torch.from_numpy(np.ascontiguousarray(rhs.reshape((n, -1)))).to(d.device)
        d.solve_device(X, conjugate=False, trans=trans)
        return X.cpu().numpy()
    x_n = solve(c, 'N')[:, 0]
    for trans in ('T', 'H'):
        x = solve(b, trans)
        opA = A.T if trans == 'T' else A.conj().T
        for j in range(2):
            assert rel_l2(opA @ x[:, j], b[:, j]) <= 1e-10, (trans, j)
        y = solve(w, trans)[:, 0]
        if trans == 'T':                                                # w^T (A^-1 c) = (A^-T w)^T c
            lhs, rhs = w @ x_n, y @ c
        else:                                                           # w^H (A^-1 c) = (A^-H w)^H c
            lhs, rhs = np.conj(w) @ x_n, np.conj(y) @ c
        assert abs(lhs - rhs) <= 1e-10 * abs(lhs), trans


def test_eurus_transposed_refinement_default():
    """Eurus refines transposed solves twice unless systemConfig sets `refine` (DESIGN §2); N keeps its one step."""
    import zephyr_b200 as zb
    from zephyr_b200 import _lib
    sc = {'nx': 9, 'nz': 10, 'dx': 10., 'dz': 10., 'c': 2500., 'rho': 1., 'freq': 9., 'nPML': 3, 'theta': 0.2, 'eps': 0.1, 'delta': 0.05}
    d = zb.Eurus(sc)
    assert [d._refine_steps(op) for op in (_lib.HZ_OP_N, _lib.HZ_OP_T, _lib.HZ_OP_H)] == [1, 2, 2]
    d1 = zb.Eurus(dict(sc, refine=1))
    assert [d1._refine_steps(op) for op in (_lib.HZ_OP_N, _lib.HZ_OP_T, _lib.HZ_OP_H)] == [1, 1, 1]
    m = zb.MiniZephyr(sc)
    assert m._refine_steps(_lib.HZ_OP_T) == m.refine == -1
