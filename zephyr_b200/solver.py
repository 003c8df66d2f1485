"""``Solver``-compatible shim: the reference's third plug-in point.

``systemConfig['Solver']`` is a class handed to ``problemo.BestSolver`` (zephyr/backend/discretization.py:28,83;
zephyr/frontend/jobs.py:27-32 tries pymatsolver's MUMPS, notebooks pass ``scipy.sparse.linalg.splu``): it is called
with the assembled sparse matrix and must return an object with ``solve(rhs)``.  ``BlockTridiagonalSolver(A)`` accepts
the 9-diagonal matrices MiniZephyr builds (and Eurus' 2N x 2N block form) and solves with the GPU block
factorisation -- for A/B runs of the factorisation alone: assembly stays in the reference (SURVEY.md 8(b) explains
why the full path plugs in at 'Disc' instead).  No conjugation and no premul here: that is the caller's job
(discretization.py:103), exactly as with splu.  ``solve(rhs, trans)`` takes SuperLU's ``trans`` ('N', 'T', 'H': solve
with A, A^T or A^H) and runs all three from the same factors (complex128 only for 'T' / 'H').
"""
import ctypes as C

import numpy as np
import scipy.sparse as sp

from . import _lib


class BlockTridiagonalSolver(object):

    def __init__(self, A, nx=None, device=None, dtype='complex128'):
        A = sp.csr_matrix(A)
        n = A.shape[0]
        if A.shape[0] != A.shape[1]:
            raise ValueError('square matrix expected')
        coo = A.tocoo()
        offs = np.unique(coo.col - coo.row)
        nf = 1
        if offs.size and np.abs(offs).max() > n // 2 - 2:      # Eurus: [[M1, M2], [M3, M4]], coupling offsets +-N
            nf = 2
        N = n // nf
        if nx is None:                                           # the largest in-quadrant offset is nx + 1
            inq = np.abs(((coo.col % N) - (coo.row % N)))
            nx = int(inq.max()) - 1
        nx = int(nx)
        if nx < 3 or N % nx:
            raise ValueError('cannot infer the grid from the matrix; pass nx')
        nz = N // nx
        planes = np.zeros((nf, nf, 9, nz, nx), dtype=np.complex128)
        fr, fc = coo.row // N, coo.col // N
        rr, cc = coo.row % N, coo.col % N
        d = cc - rr
        dz = np.rint(d / float(nx)).astype(np.int64)
        dx = d - dz * nx
        if np.any(np.abs(dz) > 1) or np.any(np.abs(dx) > 1):
            raise ValueError('matrix is not a 9-point stencil operator on a %d x %d grid' % (nx, nz))
        np.add.at(planes, (fr, fc, (dz + 1) * 3 + (dx + 1), rr // nx, rr % nx), coo.data)
        self.shape, self.nf, self.nx, self.nz, self.N = A.shape, nf, nx, nz, N
        self._c64 = np.dtype(dtype) == np.complex64
        lib = _lib.get_lib()
        dev = _lib.torch_device(device)
        h = C.c_void_p()
        _lib.check(lib.hz_create(C.byref(h), dev.index or 0, _lib.HZ_C64 if self._c64 else _lib.HZ_C128,
                                 _lib.HZ_DISC_EURUS if nf == 2 else _lib.HZ_DISC_MINIZEPHYR, nx, nz, 1., 1., 2, 1e3, None,
                                 _lib.current_stream_ptr(dev)))
        self._handle, self._dev = h, dev
        _lib.check(lib.hz_set_coefficients(h, _lib.ptr(np.ascontiguousarray(planes))), h)
        _lib.check(lib.hz_factor(h, -1), h)

    def solve(self, rhs, trans='N'):
        import torch
        lib = _lib.get_lib()
        op = _lib.trans_op(trans)
        rhs = np.asarray(rhs.toarray() if sp.issparse(rhs) else rhs, dtype=np.complex128)
        squeeze = rhs.ndim < 2
        if squeeze:
            rhs = rhs.reshape((rhs.size, 1))
        if rhs.shape[0] != self.shape[0]:
            raise ValueError('dimension mismatch')
        X = torch.from_numpy(np.ascontiguousarray(rhs)).to(self._dev, copy=True).to(torch.complex64 if self._c64 else torch.complex128)
        _lib.check(lib.hz_set_stream(self._handle, _lib.current_stream_ptr(self._dev)), self._handle)
        _lib.check(lib.hz_solve_op(self._handle, op, _lib.ptr(X), X.shape[1], 1.0, 0.0, 0, -1, -1, -1, None), self._handle)
        out = X.to(torch.complex128).cpu().numpy()
        return out[:, 0] if squeeze else out

    __mul__ = solve

    def close(self):
        if getattr(self, '_handle', None) is not None:
            _lib.get_lib().hz_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
