"""Host mirror of the reference's discretisation operators, backed by the sm_100a library.

Drop-in for ``zephyr.backend.{MiniZephyr, MiniZephyrHD, Eurus, EurusHD}``
(zephyr/backend/discretization.py:18-106, minizephyr.py:27-343, eurus.py:14-552): same
``systemConfig`` keys, ``Disc * rhs`` / ``Disc(rhs)`` returning the conjugated dense wavefield,
``.A``, ``.shape``, ``.c``, ``.rho``, ``.premul``, ``.factors`` and ``del disc.factors``.

What differs underneath: assembly, the block factorisation, and the multi-RHS substitution run
on the GPU (include/zephyr_b200.h); ``systemConfig['Solver']`` is accepted and ignored (the
factorisation *is* the product).  Extra optional keys: ``device`` (CUDA ordinal), ``twist``
(block row where the two elimination chains meet: an int, ``'mid'`` = nz/2 (default: the two
chains factor concurrently) or ``'source'`` = centre of the first right-hand side's depth range,
which minimises substitution work when factors are reused for many solves), ``refine`` (iterative-refinement steps; default 0 for MiniZephyr, 1 for
Eurus whose diagonal blocks are ill-conditioned, see DESIGN.md), ``dtype`` ('complex128' / 'complex64'), ``storeEvery``
(checkpointed factors: keep only every k-th block inverse per elimination chain and recompute the ones in between
during the substitution sweeps -- 1/k of the HBM for 2 (k-1)/k extra factorisations per solve; ``'auto'`` picks the
smallest k whose checkpoints fit in free HBM; this is how 2000 x 6000 grids run on one GPU).
"""
import ctypes as C

import numpy as np
import scipy.sparse as sp

from . import _lib
from .base import AttributeMapper, BaseAnisotropic, BaseModelDependent

MZ_KEYS = ['AD', 'DD', 'CD', 'AA', 'BE', 'CC', 'AF', 'FF', 'CF']


def _panel_to_host(X, chunk_bytes=128 << 20, nbuf=8):
    """Device panel -> complex128 ndarray.  The reference's operator returns the dense (N, S) wavefield to the host
    (discretization.py:101-106) -- 24.6 GB at 1000 x 3000 x 512 sources.  A plain .cpu() goes through pageable memory
    at ~2 GB/s; large panels are copied in chunks through a ring of pinned staging buffers (PCIe rate) while `nbuf`
    host threads move finished chunks into the result array (first-touch page faults of the fresh 24.6 GB array are
    what limits one thread to ~7 GB/s).  Measured at C3 with the factors resident (tools/d2h_probe.py): 2 buffers 3.50 s,
    4 buffers 2.06 s, 8 buffers 1.71 s per `Disc * q` (0.6 s of which is the substitution)."""
    import torch
    nbytes = X.numel() * 16
    if X.device.type != 'cuda' or nbytes < 4 * chunk_bytes:
        return X.cpu().numpy().astype(np.complex128, copy=False)
    from concurrent.futures import ThreadPoolExecutor
    rows, S = X.shape
    res = np.empty((rows, S), dtype=np.complex128)
    rpc = max(1, chunk_bytes // (S * 16))
    stage = [torch.empty((rpc, S), dtype=torch.complex128).pin_memory() for _ in range(nbuf)]
    events = [torch.cuda.Event() for _ in range(nbuf)]
    stream = torch.cuda.current_stream(X.device)
    pending = [None] * nbuf

    def drain(buf, r0, r1):
        events[buf].synchronize()
        np.copyto(res[r0:r1], stage[buf][:r1 - r0].numpy())
    with ThreadPoolExecutor(max_workers=nbuf) as pool:
        for k, r0 in enumerate(range(0, rows, rpc)):
            buf, r1 = k % nbuf, min(r0 + rpc, rows)
            if pending[buf] is not None:
                pending[buf].result()                      # the staging buffer is free again
            stage[buf][:r1 - r0].copy_(X[r0:r1], non_blocking=True)      # converts complex64 panels on the fly
            events[buf].record(stream)
            pending[buf] = pool.submit(drain, buf, r0, r1)
        for f in pending:
            if f is not None:
                f.result()
    return res


class BaseDiscretization(BaseModelDependent):

    initMap = {
        #   Argument        Required    Rename as ...   Store as type
        'c':            (True,      '_c',           np.complex128),
        'rho':          (False,     '_rho',         np.float64),
        'freq':         (True,      None,           np.complex128),
        'Solver':       (False,     '_Solver',      None),
        'tau':          (False,     '_tau',         np.float64),
        'premul':       (False,     '_premul',      np.complex128),
        'nPML':         (False,     '_nPML',        np.int64),
        'mord':         (False,     '_mord',        tuple),
        'device':       (False,     '_device',      None),
        'twist':        (False,     '_twist',       None),
        'refine':       (False,     '_refine',      np.int64),
        'dtype':        (False,     '_dtype',       None),
        'storeEvery':   (False,     '_storeEvery',  None),
    }

    _disc_id = _lib.HZ_DISC_MINIZEPHYR
    _nf = 1

    def __init__(self, systemConfig):
        super(BaseDiscretization, self).__init__(systemConfig)
        if hasattr(self, 'ny'):
            raise NotImplementedError('3D grids are not supported')
        if hasattr(self, '_mord') and tuple(self._mord) != tuple(self._default_mord()):
            raise NotImplementedError('only the default matrix ordering mord=%r is built' % (self._default_mord(),))
        self._handle = None
        self._twist_used = None
        self.last_residual = None

    def reconfigure(self, systemConfig):
        """Re-read the configuration (new model and/or frequency) while keeping the device handle and
        its HBM allocations; factors are invalidated.  This is what a model update in an inversion
        loop costs here, instead of the reference's rebuild-everything clearCache()
        (middleware/problem.py:51-66)."""
        old = (int(self.nx), int(self.nz), float(self.dx), float(self.dz), int(self.nPML), tuple(self.freeSurf))
        for attr in ('_c', '_rho', '_tau', '_premul', '_theta', '_eps', '_delta', '_ky', '_twist'):
            if hasattr(self, attr):
                delattr(self, attr)
        AttributeMapper.__init__(self, systemConfig)
        self._A = None
        new = (int(self.nx), int(self.nz), float(self.dx), float(self.dz), int(self.nPML), tuple(self.freeSurf))
        if self._handle is not None:
            if new != old:
                self.close()
            else:
                lib = _lib.get_lib()
                arrs = self._model_arrays()
                arrs += [None] * (5 - len(arrs))
                _lib.check(lib.hz_set_model(self._handle, *[_lib.ptr(a) for a in arrs], 0), self._handle)
                _lib.check(lib.hz_assemble(self._handle, *self._assemble_args()), self._handle)

    # ---- reference attributes (discretization.py:33-76) --------------------------------------
    @property
    def tau(self):
        return getattr(self, '_tau', np.inf)

    @property
    def dampCoeff(self):
        return 1j / self.tau

    @property
    def premul(self):
        return getattr(self, '_premul', 1.)

    @property
    def c(self):
        if isinstance(self._c, np.ndarray):
            return self._c
        return self._c * np.ones((self.nz, self.nx), dtype=np.complex128)

    @property
    def rho(self):
        if hasattr(self, '_rho'):
            if not isinstance(self._rho, np.ndarray):
                return self._rho * np.ones((self.nz, self.nx), dtype=np.float64)
        else:
            self._rho = 310. * self.c.real ** 0.25          # Gardner default (discretization.py:66-72)
        return self._rho

    @property
    def nPML(self):
        return getattr(self, '_nPML', 10)

    @property
    def mord(self):
        return getattr(self, '_mord', self._default_mord())

    @property
    def refine(self):
        return int(getattr(self, '_refine', -1))            # -1: library default (hz_solve)

    def _refine_steps(self, op):
        """Refinement steps of a solve with op(A) (HZ_OP_N / T / H)."""
        return self.refine

    @property
    def shape(self):
        n = self._nf * self.nrow
        return (n, n)

    @property
    def c64(self):
        """True for the complex64 variant (``dtype='complex64'``): block inverses stored and
        substitution carried out in complex64; wavefields are still returned as complex128."""
        dt = getattr(self, '_dtype', None)
        if dt is None:
            return False
        dt = np.dtype(dt)
        if dt == np.complex64:
            return True
        if dt == np.complex128:
            return False
        raise ValueError('dtype must be complex128 or complex64')

    @property
    def panel_dtype(self):
        import torch
        return torch.complex64 if self.c64 else torch.complex128

    # ---- device objects ----------------------------------------------------------------------
    @property
    def device(self):
        return _lib.torch_device(getattr(self, '_device', None))

    def _model_arrays(self):
        return [np.ascontiguousarray(self.c.reshape((self.nz, self.nx)), dtype=np.complex128),
                np.ascontiguousarray(np.asarray(self.rho, dtype=np.float64).reshape((self.nz, self.nx)))]

    def _assemble_args(self):
        freq = complex(self.freq)
        return freq.real, freq.imag, float(self.tau), 0.0

    def _create_args(self):
        return float(1e3)

    @property
    def handle(self):
        """Opaque library handle; created, loaded with the model and assembled on first use."""
        if self._handle is None:
            import torch
            lib = _lib.get_lib()
            dev = self.device
            fs = (C.c_int32 * 4)(*[int(bool(v)) for v in self.freeSurf])
            h = C.c_void_p()
            _lib.check(lib.hz_create(C.byref(h), dev.index or 0, _lib.HZ_C64 if self.c64 else _lib.HZ_C128, self._disc_id, int(self.nx), int(self.nz),
                                     float(self.dx), float(self.dz), int(self.nPML), self._create_args(), fs,
                                     _lib.current_stream_ptr(dev)))
            self._handle = h
            arrs = self._model_arrays()
            arrs += [None] * (5 - len(arrs))
            _lib.check(lib.hz_set_model(h, *[_lib.ptr(a) for a in arrs], 0), h)
            _lib.check(lib.hz_assemble(h, *self._assemble_args()), h)
        return self._handle

    def coefficients(self):
        """Device-assembled stencil planes [nf, nf, 9, nz, nx]; slot = (dz+1)*3 + (dx+1)."""
        out = np.empty((self._nf, self._nf, 9, int(self.nz), int(self.nx)), dtype=np.complex128)
        _lib.check(_lib.get_lib().hz_get_coefficients(self.handle, _lib.ptr(out)), self.handle)
        return out

    @property
    def A(self):
        """The sparse system matrix as scipy CSR, built from the device-assembled coefficients
        (minizephyr.py:300-306 / eurus.py:487-492); used for ``.shape`` and parity checks."""
        if getattr(self, '_A', None) is None:
            coef = self.coefficients()
            nx, n = int(self.nx), self.nrow
            quads = []
            for fr in range(self._nf):
                row = []
                for fc in range(self._nf):
                    diags, offs = [], []
                    for slot in range(9):
                        off = (slot // 3 - 1) * nx + (slot % 3 - 1)
                        v = coef[fr, fc, slot].ravel()
                        diags.append(v[-off:] if off < 0 else (v[:n - off] if off > 0 else v))
                        offs.append(off)
                    row.append(sp.diags(diags, offs, shape=(n, n), format='csr', dtype=np.complex128))
                quads.append(row)
            self._A = quads[0][0] if self._nf == 1 else sp.bmat(quads).tocsr()
        return self._A

    # ---- factors (discretization.py:78-99) ------------------------------------------------------
    def _bind_stream(self):
        """The handle follows the caller's current stream (and host thread): factor / solve work is issued on the
        same stream as the torch operations and helper kernels around it."""
        _lib.check(_lib.get_lib().hz_set_stream(self.handle, _lib.current_stream_ptr(self.device)), self.handle)

    def _apply_store_every(self):
        lib = _lib.get_lib()
        k = getattr(self, '_storeEvery', None)
        if k is None:
            return
        if k == 'auto':
            import torch
            _lib.check(lib.hz_set_option(self.handle, b'store_every', 1.0), self.handle)
            full = self.factor_bytes()
            free = torch.cuda.mem_get_info(self.device)[0] if self.device.type == 'cuda' else 8 << 30
            budget = 0.85 * free - 4 * full / int(self.nz)           # leave room for workspaces and a few panels
            k = 1
            while k < 64 and full / k > budget:
                k += 1
        _lib.check(lib.hz_set_option(self.handle, b'store_every', float(int(k))), self.handle)
        self._store_every_used = int(k)

    def _ensure_factors(self, zf=-1, zl=-1):
        lib = _lib.get_lib()
        self._bind_stream()
        flag = C.c_int32(0)
        _lib.check(lib.hz_has_factors(self.handle, C.byref(flag)), self.handle)
        if not flag.value:
            self._apply_store_every()
            tw = getattr(self, '_twist', 'mid')
            if tw == 'source' and zf >= 0 and zl >= 0:
                twist = int((zf + zl) // 2)      # chains meet at the source depth: fewest substitution GEMMs
            elif tw in ('mid', 'source'):
                twist = int(self.nz) // 2        # two equally long chains factor concurrently (default)
            else:
                twist = int(tw)
            _lib.check(lib.hz_factor(self.handle, twist), self.handle)
            self._twist_used = twist

    @property
    def Ainv(self):
        self._ensure_factors()
        return self

    @property
    def factors(self):
        if self._handle is None:
            return False
        flag = C.c_int32(0)
        _lib.check(_lib.get_lib().hz_has_factors(self._handle, C.byref(flag)), self._handle)
        return bool(flag.value)

    @factors.deleter
    def factors(self):
        if getattr(self, '_handle', None) is not None:
            _lib.get_lib().hz_free_factors(self._handle)

    @property
    def last_probe(self):
        """Stencil residual measured by the library's accuracy probe on the first solve after the last
        factorisation (include/zephyr_b200.h: hz_last_probe); -1 before any solve."""
        v = C.c_double(-1.0)
        _lib.check(_lib.get_lib().hz_last_probe(self.handle, C.byref(v)), self.handle)
        return v.value

    def factor_bytes(self):
        n = C.c_int64(0)
        _lib.check(_lib.get_lib().hz_factor_bytes(self.handle, C.byref(n)), self.handle)
        return n.value

    def factor_bytes_missing(self):
        """HBM a factorisation of this handle still has to allocate (0 after a model update: the block-inverse store is kept)."""
        n = C.c_int64(0)
        _lib.check(_lib.get_lib().hz_factor_resident_bytes(self.handle, C.byref(n)), self.handle)
        return max(0, self.factor_bytes() - n.value)

    def close(self):
        if getattr(self, '_handle', None) is not None:
            try:
                _lib.get_lib().hz_destroy(self._handle)
            except Exception:
                pass
            self._handle = None

    def __del__(self):
        self.close()

    # ---- the operator (discretization.py:101-106) ----------------------------------------------
    def _rows_ok(self, nrows):
        """returns clip flag; raises ValueError('dimension mismatch') like eurus.py:516-526."""
        if nrows == self.shape[1]:
            return False
        raise ValueError('dimension mismatch')

    def rhs_depth_range(self, rhs):
        """(first, last) block row holding a non-zero of an ndarray / scipy.sparse right-hand side; (-1, -1) if none."""
        nx, N = int(self.nx), self.nrow
        if sp.issparse(rhs):
            rows = np.unique(rhs.tocoo().row)
        else:
            rhs = np.asarray(rhs)
            rows = np.flatnonzero(np.any(rhs.reshape((rhs.shape[0], -1)) != 0, axis=1))
        if rows.size == 0:
            return (-1, -1)
        iz = (rows % N) // nx
        return (int(iz.min()), int(iz.max()))

    def rhs_to_device(self, rhs):
        """Build the (nf*N, S) device panel from an ndarray / scipy.sparse right-hand side.
        Returns (X, (z_first, z_last)) with the depth range (block rows) holding non-zeros."""
        import torch
        lib = _lib.get_lib()
        dev = self.device
        rows_total = self.shape[1]
        nx, N = int(self.nx), self.nrow
        if sp.issparse(rhs):
            q = rhs.tocoo()
            q.sum_duplicates()
            S = q.shape[1]
            X = torch.zeros((rows_total, S), dtype=self.panel_dtype, device=dev)
            if q.nnz:
                row = torch.from_numpy(np.ascontiguousarray(q.row, dtype=np.int64)).to(dev)
                col = torch.from_numpy(np.ascontiguousarray(q.col, dtype=np.int64)).to(dev)
                val = torch.from_numpy(np.ascontiguousarray(q.data, dtype=np.complex128)).to(dev)
                _lib.check(_lib.panel_fn('hz_scatter_coo', self.c64)(_lib.ptr(X), S, q.nnz, _lib.ptr(row), _lib.ptr(col), _lib.ptr(val),
                                              1.0, 0.0, _lib.current_stream_ptr(dev)))
                iz = (q.row % N) // nx
                zr = (int(iz.min()), int(iz.max()))
            else:
                zr = (-1, -1)
            return X, zr
        rhs = np.asarray(rhs, dtype=np.complex128)
        S = rhs.shape[1]
        if rhs.shape[0] == rows_total:
            X = torch.from_numpy(np.ascontiguousarray(rhs)).to(dev, copy=True).to(self.panel_dtype)
        else:
            X = torch.zeros((rows_total, S), dtype=self.panel_dtype, device=dev)
            X[:rhs.shape[0]] = torch.from_numpy(np.ascontiguousarray(rhs)).to(dev).to(self.panel_dtype)
        nzr = np.flatnonzero(np.any(rhs != 0, axis=1))
        if nzr.size:
            iz = (nzr % N) // nx
            zr = (int(iz.min()), int(iz.max()))
        else:
            zr = (-1, -1)
        return X, zr

    def solve_device(self, X, zrange=(-1, -1), conjugate=True, want_residual=False, trans='N'):
        """In place on a device panel X (nf*N, S): X <- conj(premul * op(A)^-1 X) with op(A) = A, A^T or A^H for
        ``trans`` = 'N', 'T' or 'H' (all three from the same factors; 'T' / 'H' need complex128).  Fast path for
        callers that keep wavefields in HBM (survey / bench)."""
        lib = _lib.get_lib()
        op = _lib.trans_op(trans)
        if X.dtype != self.panel_dtype or not X.is_contiguous():
            raise ValueError('panel must be a contiguous %s tensor' % (self.panel_dtype,))
        self._ensure_factors(*zrange)
        self._bind_stream()
        pm = complex(self.premul)
        res = C.c_double(-1.0)
        refine = self._refine_steps(op)
        _lib.check(lib.hz_solve_op(self.handle, op, _lib.ptr(X), X.shape[1], pm.real, pm.imag, int(bool(conjugate)),
                                   int(zrange[0]), int(zrange[1]), refine,
                                   C.byref(res) if (want_residual or refine > 0) else None), self.handle)
        if want_residual or refine > 0:
            self.last_residual = res.value
        return X

    def solve(self, rhs, trans='N'):
        """conj(premul * op(A)^-1 rhs) for an ndarray / scipy.sparse right-hand side, op(A) = A, A^T, A^H for
        ``trans`` = 'N', 'T', 'H' (scipy's ``SuperLU.solve`` convention), with the conventions of ``Disc * rhs``
        (premul, conjugation, Eurus' zero padding of N-row right-hand sides and clipping of the result).
        ``solve(rhs)`` is ``Disc * rhs``."""
        _lib.trans_op(trans)
        squeeze = False
        if not sp.issparse(rhs):
            rhs = np.asarray(rhs)
            if rhs.ndim < 2:
                rhs = rhs.reshape((rhs.size, 1))
                squeeze = True
        clip = self._rows_ok(rhs.shape[0])
        X, zr = self.rhs_to_device(rhs)
        self.solve_device(X, zr, trans=trans)
        out = X[:self.nrow] if clip else X
        res = _panel_to_host(out)
        return res[:, 0] if squeeze else res

    def __mul__(self, rhs):
        return self.solve(rhs)

    def __call__(self, value):
        return self * value


class MiniZephyr(BaseDiscretization):
    """2D (visco)acoustic 9-point mixed-grid stencil with PML (zephyr/backend/minizephyr.py:27-324)."""

    initMap = {
        'ky':           (False,     '_ky',          np.float64),
    }

    def _default_mord(self):
        return (self.nx, +1)

    @property
    def ky(self):
        return getattr(self, '_ky', 0.)

    def _assemble_args(self):
        freq = complex(self.freq)
        return freq.real, freq.imag, float(self.tau), float(self.ky)


class MiniZephyrHD(MiniZephyr):
    """MiniZephyr with half-differentiation of the source (minizephyr.py:327-343)."""

    @property
    def premul(self):
        return getattr(self, '_premul', np.sqrt(2j * np.pi * self.freq))


class MiniZephyr25D(BaseDiscretization):
    """2.5-D modelling: Fourier summation of 2-D solves over cross-line wavenumbers ky
    (zephyr/backend/minizephyr.py:346-460).  Each ky is its own operator (own factorisation); the
    partial wavefields are accumulated on the device and only the sum is copied back.  ``parallel``
    is accepted and ignored; factors are released after each ky unless ``keepFactors`` is set.  Transposed solves
    (``solve(rhs, trans='T' / 'H')``) are not built for the 2.5-D sum; ``solve(rhs)`` is ``self * rhs``."""

    initMap = {
        'Disc':         (False,     '_Disc',        None),
        'nky':          (True,      '_nky',         np.int64),
        'parallel':     (False,     '_parallel',    bool),
        'cmin':         (False,     '_cmin',        np.float64),
        'scaleTerm':    (False,     '_scaleTerm',   np.complex128),
        'keepFactors':  (False,     '_keepFactors', bool),
    }
    maskKeys = {'nky', 'Disc', 'parallel', 'scaleTerm', 'keepFactors'}

    def __init__(self, systemConfig):
        super(MiniZephyr25D, self).__init__(systemConfig)
        self.systemConfig = {k: systemConfig[k] for k in systemConfig if k not in self.maskKeys}
        self._subProblems = None

    def _default_mord(self):
        return (self.nx, +1)

    def solve(self, rhs, trans='N'):
        if _lib.trans_op(trans) != _lib.HZ_OP_N:
            raise NotImplementedError('MiniZephyr25D: transposed solves are not built for the 2.5-D sum')
        return self * rhs

    @property
    def Disc(self):
        return getattr(self, '_Disc', None) or MiniZephyr

    @property
    def nky(self):
        return int(getattr(self, '_nky', 1) or 1)

    @property
    def cmin(self):
        return getattr(self, '_cmin', None) if getattr(self, '_cmin', None) is not None else np.min(self.c)

    @property
    def pkys(self):
        indices = np.arange(self.nky)
        dky = self.freq / (self.cmin * (self.nky - 1)) if self.nky > 1 else 0.
        return indices * dky

    @property
    def kyweights(self):
        return 1. + (np.arange(self.nky) > 0)

    @property
    def spUpdates(self):
        weightfac = 1. / (2 * self.nky - 1) if self.nky > 1 else 1.
        return [{'ky': np.real(ky), 'premul': weightfac * (1. + (np.real(ky) > 0))} for ky in self.pkys]

    @property
    def subProblems(self):
        if self._subProblems is None:
            self._subProblems = []
            for spu in self.spUpdates:
                sc = dict(self.systemConfig)
                sc.update(spu)
                self._subProblems.append(self.Disc(sc))
        return self._subProblems

    @property
    def scaleTerm(self):
        return getattr(self, '_scaleTerm', 1.) * np.exp(1j * np.pi) / (4 * np.pi)

    @property
    def factors(self):
        return self._subProblems is not None and any(sub.factors for sub in self._subProblems)

    @factors.deleter
    def factors(self):
        if self._subProblems is not None:
            for sub in self._subProblems:
                del sub.factors

    def close(self):
        if getattr(self, '_subProblems', None):
            for sub in self._subProblems:
                sub.close()
        self._subProblems = None

    def __mul__(self, rhs):
        squeeze = False
        if not sp.issparse(rhs):
            rhs = np.asarray(rhs)
            if rhs.ndim < 2:
                rhs = rhs.reshape((rhs.size, 1))
                squeeze = True
        total = None
        for sub in self.subProblems:
            sub._rows_ok(rhs.shape[0])
            X, zr = sub.rhs_to_device(rhs)
            sub.solve_device(X, zr)
            total = X if total is None else total.add_(X)
            if not getattr(self, '_keepFactors', False):
                del sub.factors
        res = (total * complex(self.scaleTerm)).cpu().numpy().astype(np.complex128, copy=False)
        return res[:, 0] if squeeze else res


class Eurus(BaseDiscretization, BaseAnisotropic):
    """TTI anisotropic mixed-grid stencil, Operto et al. 2009 (zephyr/backend/eurus.py:14-533)."""

    initMap = {
        'cPML':         (False,     '_cPML',        np.float64),
    }

    _disc_id = _lib.HZ_DISC_EURUS
    _nf = 2

    def _default_mord(self):
        return (-self.nx, +1)

    @property
    def cPML(self):
        return getattr(self, '_cPML', 1e3)

    @property
    def refine(self):
        return int(getattr(self, '_refine', 1))

    def _refine_steps(self, op):
        """Transposed solves (A^T, A^H) refine twice by default: on ill-conditioned TTI operators the transposed sweep
        leaves about five times the N sweep's residual after one step (measured at 200 x 400: 5e-11 - 1.2e-10 against
        1.3e-11 - 1.7e-11), two steps bring it to ~1.5e-12.  A `refine` set in systemConfig is used as given."""
        if op != _lib.HZ_OP_N and not hasattr(self, '_refine'):
            return 2
        return self.refine

    def _create_args(self):
        return float(self.cPML)

    def _model_arrays(self):
        base = super(Eurus, self)._model_arrays()
        return base + [np.ascontiguousarray(a, dtype=np.float64) for a in (self.theta, self.eps, self.delta)]

    def _rows_ok(self, nrows):
        if 2 * nrows == self.shape[1]:                        # eurus.py:516-524: pad with zeros, clip the result
            return True
        if nrows != self.shape[1]:
            raise ValueError('dimension mismatch')
        return False


class EurusHD(Eurus):
    """Eurus with half-differentiation of the source (eurus.py:536-552)."""

    @property
    def premul(self):
        return getattr(self, '_premul', np.sqrt(2j * np.pi * self.freq))
