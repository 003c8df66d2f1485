"""Survey / problem layer for the hot path: sources, receiver extraction, residual sources,
misfit and the FWI gradient.

Restates, without SimPEG, the semantics of zephyr/middleware/survey.py:29-198 (HelmBaseSurvey)
and zephyr/middleware/problem.py:17-199 (HelmBaseProblem) for the calls on the forward/adjoint
path: ``survey.getSources()``, ``survey.rVec()``, ``survey.projectFields`` /
``_lazyProjectFields``, ``survey.getResidualSources``, ``survey.dpred``, ``problem.fields`` /
``lazyFields``, ``problem.gradientScaler``, ``problem.Jtvec``.  Host-array signatures match the
reference; ``Helm2DProblem.misfit_and_gradient`` is the device-resident pipeline (wavefields never
leave HBM; one all-reduce of N+1 doubles per evaluation, SURVEY.md 8(e)).
"""
import numpy as np
import scipy.sparse as sp

from . import _lib, parallel
from .base import AttributeMapper, BaseModelDependent
from .discretization import MiniZephyr
from .distributors import MultiFreq, ViscoMultiFreq
from .source import SparseKaiserSource


class HelmBaseSurvey(AttributeMapper):

    initMap = {
        #   Argument        Required    Rename as ...   Store as type
        'geom':         (True,      '_geom',        dict),
        'freqs':        (True,      None,           tuple),
        'sterms':       (False,     '_sterms',      np.complex128),
    }

    def __init__(self, systemConfig):
        super(HelmBaseSurvey, self).__init__(systemConfig)
        if self._geom.get('mode', 'fixed') not in {'fixed', 'relative'}:
            raise Exception('%s objects only work with \'fixed\' or \'relative\' receiver arrays' % (self.__class__.__name__,))
        self.systemConfig = dict(systemConfig)
        self.prob = None

    # ---- geometry (survey.py:48-107) ---------------------------------------------------------
    @property
    def geom(self):
        return self._geom

    @property
    def nfreq(self):
        return len(self.freqs)

    @property
    def mode(self):
        return self.geom.get('mode', 'fixed')

    @property
    def sLocs(self):
        return self.geom.get('src')

    @property
    def rLocs(self):
        return self.geom.get('rec')

    @property
    def nsrc(self):
        return 0 if self.sLocs is None else self.sLocs.shape[0]

    @property
    def nrec(self):
        return 0 if self.rLocs is None else self.rLocs.shape[0]

    @property
    def ssTerms(self):
        return self.geom.get('sterms', np.ones((self.nsrc,), dtype=np.complex128))

    @property
    def srTerms(self):
        return self.geom.get('rterms', np.ones((self.nrec,), dtype=np.complex128))

    @property
    def tsTerms(self):
        return getattr(self, '_sterms', np.ones(self.nfreq, dtype=np.complex128))

    @property
    def RHSGenerator(self):
        if not hasattr(self, '_RHSGenerator'):
            self._RHSGenerator = self.geom.get('GeneratorClass', SparseKaiserSource)
        return self._RHSGenerator

    @property
    def nD(self):
        return self.nsrc * self.nrec * self.nfreq

    # ---- operators (survey.py:109-125) -------------------------------------------------------
    def sVecs(self):
        if not hasattr(self, '_sVecs'):
            self._sVecs = sp.csc_matrix(self.RHSGenerator(self.systemConfig)(self.sLocs) * sp.diags((self.ssTerms,), (0,)))
        return self._sVecs

    def rVec(self, isrc=0):
        if self.mode == 'fixed':
            if not hasattr(self, '_rVecs'):
                self._rVecs = sp.csr_matrix((self.RHSGenerator(self.systemConfig)(self.rLocs) * sp.diags((self.srTerms,), (0,))).T)
            return self._rVecs
        if not hasattr(self, '_rVecs'):
            self._rVecs = {}
        if isrc not in self._rVecs:
            self._rVecs[isrc] = sp.csr_matrix((self.RHSGenerator(self.systemConfig)(self.rLocs + self.sLocs[isrc])
                                               * sp.diags((self.srTerms,), (0,))).T)
        return self._rVecs[isrc]

    def rVecs(self, ifreq=None):
        return (self.rVec(i) for i in range(self.nsrc))

    def getSources(self):
        'survey.py:162-169'
        qs = self.sVecs()
        ts = np.asarray(self.tsTerms)
        if ts.ndim < 2:
            return [qs * sterm.conjugate() for sterm in ts]
        return [qs * sp.diags((sterm.conjugate(),), (0,)) for sterm in ts]

    def getResidualSources(self, resid):
        'survey.py:171-188: per frequency, hstack over sources of rVec(isrc).T * resid[:, isrc, ifreq]'
        if self.mode == 'fixed':
            RvT = self.rVec().T.tocsr()
            return [sp.csc_matrix(RvT * resid[:, :, ifreq]) for ifreq in range(self.nfreq)]
        return [sp.hstack([self.rVec(isrc).T * sp.csc_matrix(resid[:, isrc, ifreq].reshape((self.nrec, 1)))
                           for isrc in range(self.nsrc)]) for ifreq in range(self.nfreq)]

    # ---- projection (survey.py:141-160) ------------------------------------------------------
    def projectFields(self, u):
        """u: iterable over frequencies of (N, S) wavefields -> data (R, S, F).  Frequencies not
        owned by this rank (None entries) are left zero; see ``gatherData``."""
        data = np.zeros((self.nrec, self.nsrc, self.nfreq), dtype=np.complex128)
        for ifreq, uFreq in enumerate(u):
            if uFreq is None:
                continue
            uFreq = np.asarray(uFreq)[:self.rVec(0).shape[1]]
            if self.mode == 'fixed':
                data[:, :, ifreq] = self.rVec() * uFreq
            else:
                for isrc in range(self.nsrc):
                    data[:, isrc, ifreq] = self.rVec(isrc) * uFreq[:, isrc]
        return data

    _lazyProjectFields = projectFields

    def pair(self, prob):
        self.prob = prob
        prob.survey = self

    def dpred(self, m=None, u=None):
        'survey.py:190-198'
        if self.prob is None:
            raise Exception('%s instance is not paired to a problem' % (self.__class__.__name__,))
        if u is None:
            if hasattr(self.prob, 'dpred_device'):
                # same result as projecting lazyFields(m); the wavefields stay in HBM and only the
                # (nrec, nsrc, nfreq) data cube crosses PCIe (summed over frequency shards)
                self.prob.updateModel(m)
                return self._gather_freqs(self.prob.dpred_device()).cpu().numpy().ravel()
            u = self.prob.lazyFields(m)
        return self.projectFields(u).ravel()

    def _gather_freqs(self, dd):
        """{ifreq: (R, S) device tensor} of this rank's frequencies -> the (R, S, F) complex128 device cube on every rank.
        Every rank contributes only the (R, S) slabs of its own frequencies: all-gather of ceil(F / world) slabs per
        rank instead of all-reducing a cube that is zero elsewhere."""
        import torch
        dev = self.prob._device_ops()['dev']
        rank, world = parallel.rank_world()
        per = -(-self.nfreq // world)
        mine = torch.zeros((per, self.nrec, self.nsrc), dtype=torch.complex128, device=dev)
        for k, ifreq in enumerate(sorted(dd)):
            mine[k] = dd[ifreq].to(torch.complex128)
        slabs = parallel.allgather(mine)                  # list over ranks of (per, R, S)
        cube = torch.empty((self.nrec, self.nsrc, self.nfreq), dtype=torch.complex128, device=dev)
        for r, slab in enumerate(slabs):
            for k, ifreq in enumerate(parallel.shard_indices(self.nfreq, r, world)):
                cube[:, :, ifreq] = slab[k]
        return cube

    @property
    def postProcessors(self):
        return [lambda x: x for _ in self.freqs]

    @property
    def preProcessors(self):
        return [lambda x: x for _ in self.freqs]


class Helm2DSurvey(HelmBaseSurvey):
    pass


class HelmBaseProblem(BaseModelDependent):

    initMap = {
        'SystemWrapper':    (False,     '_SystemWrapper',   None),
    }
    SystemWrapper = MultiFreq

    def __init__(self, systemConfig):
        super(HelmBaseProblem, self).__init__(systemConfig)
        self.systemConfig = dict(systemConfig)
        if hasattr(self, '_SystemWrapper'):
            self.SystemWrapper = self._SystemWrapper
        self.survey = None
        self._system = None

    @property
    def ispaired(self):
        return self.survey is not None

    def pair(self, survey):
        self.survey = survey
        survey.prob = self

    def clearCache(self):
        if self._system is not None:
            self._system.clearCache()
        self._system = None

    def _refresh(self):
        """The reference drops every cached object on a model change (clearCache); here the
        sub-problems keep their device handles and HBM and only re-assemble / re-factor."""
        if self._system is not None:
            sc = dict(self.systemConfig)
            sc['freqs'] = list(sc.get('freqs', self.survey.freqs if self.survey is not None else []))
            self._system.reconfigure(sc)

    def updateModel(self, m, loneKey='c'):
        'problem.py:51-66'
        if m is None:
            return
        if isinstance(m, dict):
            self.systemConfig.update(m)
            self._refresh()
        elif isinstance(m, (np.ndarray, np.inexact, complex, float)):
            old = np.asarray(self.systemConfig.get(loneKey, 0.))
            if old.size != np.asarray(m).size or not np.linalg.norm(np.asarray(m).ravel() - old.ravel()) < 1e-15:
                self.systemConfig[loneKey] = m
                self._refresh()
        else:
            raise Exception('Class %s doesn\'t know how to update with model of type %s' % (self.__class__.__name__, type(m)))

    @property
    def system(self):
        if self._system is None:
            sc = dict(self.systemConfig)
            sc.setdefault('freqs', list(self.survey.freqs) if self.survey is not None else None)
            sc['freqs'] = list(sc['freqs'])
            self._system = self.SystemWrapper(sc)
        return self._system

    def scaledTerms(self, ifreq):
        omega = 2 * np.pi * self.survey.freqs[ifreq]
        c = self.system.subProblems[ifreq].c
        return omega, c

    def gradientScaler(self, ifreq):
        'problem.py:74-81'
        omega, c = self.scaledTerms(ifreq)
        return self.survey.postProcessors[ifreq](-(omega ** 2 / c ** 3).ravel())

    def sensScaler(self, ifreq):
        'problem.py:83-85'
        omega, c = self.scaledTerms(ifreq)
        return self.survey.postProcessors[ifreq](-(c ** 3 / omega ** 2).ravel())

    def Jvec(self, m=None, v=None, u=None):
        """Forward sensitivity, as written in problem.py:88-122: one virtual-source solve per
        frequency, then the outer product of its receiver and source projections.  Entries of
        frequencies owned by other ranks are zero (all-reduce to complete)."""
        if not self.ispaired:
            raise Exception('%s instance is not paired to a survey' % (self.__class__.__name__,))
        if v is None:
            raise Exception('Actually, Jvec requires a perturbation vector')
        self.updateModel(m)
        sv = self.survey
        pqShape = (self.nz * self.nx, 1)
        perturb = np.asarray(v).reshape(pqShape)
        qv = [sv.preProcessors[i](perturb * self.sensScaler(i).reshape(pqShape)) for i in range(sv.nfreq)]
        qf = sv.getSources()
        dpert = np.zeros((sv.nrec, sv.nsrc, sv.nfreq), dtype=np.complex128)
        for ifreq, uFreq in zip(self.system.localFreqIndices, self.system * qv):
            uFreq = uFreq[:self.nrow]
            srcTerms = qf[ifreq].T * uFreq
            if sv.mode == 'fixed':
                recTerms = sv.rVec() * uFreq
                dpert[:, :, ifreq] = recTerms.reshape((sv.nrec, 1)) * srcTerms.reshape((1, sv.nsrc))
            else:
                for isrc in range(sv.nsrc):
                    dpert[:, isrc, ifreq] = srcTerms[isrc] * (sv.rVec(isrc) * uFreq)[:, 0]
        return dpert.ravel()

    def _expand(self, local_list):
        """local results (frequency order over localFreqIndices) -> list over all frequencies."""
        out = [None] * self.survey.nfreq
        for i, u in zip(self.system.localFreqIndices, local_list):
            out[i] = u
        return out

    def lazyFields(self, m=None):
        'problem.py:166-179; entries of frequencies owned by other ranks are None'
        if not self.ispaired:
            raise Exception('%s instance is not paired to a survey' % (self.__class__.__name__,))
        self.updateModel(m)
        qf = self.survey.getSources()
        return self._expand(list(self.system * qf))

    fields = lazyFields

    def Jtvec(self, m=None, v=None, u=None):
        """problem.py:125-164.  Returns the rank-local partial sum when frequencies are sharded;
        ``parallel.allreduce_sum_`` (or ``misfit_and_gradient``) completes it."""
        if not self.ispaired:
            raise Exception('%s instance is not paired to a survey' % (self.__class__.__name__,))
        if v is None:
            raise Exception('Actually, Jtvec requires a residual vector')
        self.updateModel(m)
        sv = self.survey
        resid = np.asarray(v).reshape((sv.nrec, sv.nsrc, sv.nfreq))
        qb = sv.getResidualSources(resid)
        local = self.system.localFreqIndices
        g = 0
        if u is None:                                            # mux path: no .real (problem.py:142-152)
            qf = sv.getSources()
            qm = [sp.hstack((qFi, qBi)) for qFi, qBi in zip(qf, qb)]
            for ifreq, uM in zip(local, self.system * qm):
                g = g + self.gradientScaler(ifreq) * (uM[:, :sv.nsrc] * uM[:, sv.nsrc:]).sum(axis=1)
            return g
        for ifreq, uB in zip(local, self.system * qb):
            g = g + self.gradientScaler(ifreq) * (np.asarray(u[ifreq]) * uB).sum(axis=1)
        return np.real(g)

    @property
    def factors(self):
        return self._system is not None and self._system.factors

    @factors.deleter
    def factors(self):
        if self._system is not None:
            del self._system.factors

    # ---- device-resident pipeline -----------------------------------------------------------
    def _device_ops(self):
        """Source taps and receiver operators as device arrays (built once).  'fixed' geometry: one receiver
        operator shared by all sources (CSR, and its transpose restricted to the touched nodes).  'relative'
        geometry (survey.py:120-125): one operator per source, stacked as a CSR over rows i = r*nsrc + s."""
        if getattr(self, '_dev_ops', None) is None:
            import torch
            sv = self.survey
            gen = sv.RHSGenerator(sv.systemConfig)
            dev = gen.device
            nx, N = int(self.nx), self.nrow
            qs = sv.sVecs().tocoo()

            def t(a, dt):
                return torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
            ops = {'dev': dev, 'mode': sv.mode,
                   's_row': t(qs.row, np.int64), 's_col': t(qs.col, np.int64), 's_val': t(qs.data, np.complex128),
                   's_z': (int((qs.row // nx).min()), int((qs.row // nx).max()))}
            if sv.mode == 'fixed':
                Rv = sv.rVec().tocsr()                                # (R, N)
                RvT = sp.csr_matrix(Rv.T)                             # (N, R)
                nodes = np.flatnonzero(np.diff(RvT.indptr)).astype(np.int64)
                RvTc = RvT[nodes]
                ops.update({'r_ptr': t(Rv.indptr, np.int64), 'r_col': t(Rv.indices, np.int64), 'r_val': t(Rv.data, np.complex128),
                            'b_ptr': t(RvTc.indptr, np.int64), 'b_col': t(RvTc.indices, np.int64), 'b_val': t(RvTc.data, np.complex128),
                            'b_nodes': t(nodes, np.int64), 'b_z': (int((nodes // nx).min()), int((nodes // nx).max()))})
            else:
                per_src = [sv.rVec(isrc).tocsr() for isrc in range(sv.nsrc)]      # each (R, N)
                counts = np.stack([np.diff(m.indptr) for m in per_src], 1)       # (R, S): taps of row i = r*S + s
                ptr = np.concatenate([[0], np.cumsum(counts.ravel())]).astype(np.int64)
                col = np.empty(ptr[-1], dtype=np.int64)
                val = np.empty(ptr[-1], dtype=np.complex128)
                for isrc, m in enumerate(per_src):
                    for r in range(sv.nrec):
                        a, b = ptr[r * sv.nsrc + isrc], ptr[r * sv.nsrc + isrc + 1]
                        col[a:b] = m.indices[m.indptr[r]:m.indptr[r + 1]]
                        val[a:b] = m.data[m.indptr[r]:m.indptr[r + 1]]
                ops.update({'r_ptr': t(ptr, np.int64), 'r_col': t(col, np.int64), 'r_val': t(val, np.complex128),
                            'b_z': (int((col // nx).min()), int((col // nx).max()))})
            self._dev_ops = ops
        return self._dev_ops

    def forward_device(self, ifreq, out=None):
        """uF for one frequency as a device panel (nf*N, S); sources injected on the device."""
        import torch
        lib = _lib.get_lib()
        ops = self._device_ops()
        sub = self.system.subProblems[ifreq]
        sv = self.survey
        rows = sub.shape[1]
        X = out if out is not None else torch.empty((rows, sv.nsrc), dtype=sub.panel_dtype, device=ops['dev'])
        X.zero_()
        tf = np.conj(np.asarray(sv.tsTerms)[ifreq]).ravel()
        vals = ops['s_val']
        if tf.size == 1:
            ts = complex(tf[0])
        else:                                       # per-source signature terms (survey.py:166-167): scale column s by ts[f, s]
            vals = vals * torch.from_numpy(np.ascontiguousarray(tf, dtype=np.complex128)).to(ops['dev'])[ops['s_col']]
            ts = 1. + 0j
        _lib.check(_lib.panel_fn('hz_scatter_coo', sub.c64)(_lib.ptr(X), sv.nsrc, ops['s_row'].numel(), _lib.ptr(ops['s_row']), _lib.ptr(ops['s_col']),
                                      _lib.ptr(vals), ts.real, ts.imag, _lib.current_stream_ptr(ops['dev'])))
        sub.solve_device(X, ops['s_z'])
        return X

    def extract_device(self, X, out=None):
        """data[:, :, f] = rVec * uF on the device -> (R, S) tensor."""
        import torch
        ops = self._device_ops()
        sv = self.survey
        c64 = X.dtype == torch.complex64
        d = out if out is not None else torch.empty((sv.nrec, sv.nsrc), dtype=X.dtype, device=ops['dev'])
        if ops['mode'] != 'fixed':
            _lib.check(_lib.panel_fn('hz_spmm_percol', c64)(0, sv.nrec * sv.nsrc, _lib.ptr(ops['r_ptr']), _lib.ptr(ops['r_col']), _lib.ptr(ops['r_val']),
                                                         sv.nsrc, _lib.ptr(X), _lib.ptr(d), X.shape[1], _lib.current_stream_ptr(ops['dev'])))
            return d
        _lib.check(_lib.panel_fn('hz_spmm_csr', c64)(sv.nrec, _lib.ptr(ops['r_ptr']), _lib.ptr(ops['r_col']), _lib.ptr(ops['r_val']), None,
                                              _lib.ptr(X), X.shape[1], sv.nsrc, _lib.ptr(d), sv.nsrc, 1, 0,
                                              _lib.current_stream_ptr(ops['dev'])))
        return d

    def backproject_device(self, ifreq, v, out=None, vals=None, conjugate=True, trans='N'):
        """uB = Disc * (rVec.T v) for one frequency; v is the (R, S) device residual.  `vals` replaces the receiver
        taps (the CSR values of the back-projection operator); `conjugate` and `trans` are passed to solve_device."""
        import torch
        ops = self._device_ops()
        sub = self.system.subProblems[ifreq]
        sv = self.survey
        X = out if out is not None else torch.empty((sub.shape[1], sv.nsrc), dtype=sub.panel_dtype, device=ops['dev'])
        X.zero_()
        if ops['mode'] != 'fixed':
            _lib.check(_lib.panel_fn('hz_spmm_percol', sub.c64)(1, sv.nrec * sv.nsrc, _lib.ptr(ops['r_ptr']), _lib.ptr(ops['r_col']),
                                                             _lib.ptr(ops['r_val'] if vals is None else vals),
                                                             sv.nsrc, _lib.ptr(v), _lib.ptr(X), sv.nsrc, _lib.current_stream_ptr(ops['dev'])))
            sub.solve_device(X, ops['b_z'], conjugate=conjugate, trans=trans)
            return X
        _lib.check(_lib.panel_fn('hz_spmm_csr', sub.c64)(ops['b_nodes'].numel(), _lib.ptr(ops['b_ptr']), _lib.ptr(ops['b_col']),
                                              _lib.ptr(ops['b_val'] if vals is None else vals),
                                              _lib.ptr(ops['b_nodes']), _lib.ptr(v), sv.nsrc, sv.nsrc, _lib.ptr(X), sv.nsrc, 1, 0,
                                              _lib.current_stream_ptr(ops['dev'])))
        sub.solve_device(X, ops['b_z'], conjugate=conjugate, trans=trans)
        return X

    def _panel_bytes(self):
        sub = self.system.subProblems[self.system.localFreqIndices[0]]
        return sub.shape[1] * self.survey.nsrc * (8 if sub.c64 else 16)

    def _ensure_factors(self, ifreq, zrange, evict=True):
        """Factor one frequency; if HBM is exhausted because other frequencies' factors are resident (keepFactors
        with more local frequencies than fit), release those and retry once -- the reference's Pool mode never keeps
        factors (SURVEY.md App. B-10) and would complete.  (Only when frequencies run one at a time.)"""
        subs = self.system.subProblems
        try:
            subs[ifreq]._ensure_factors(*zrange)
        except MemoryError:
            others = [s for j, s in enumerate(subs) if j != ifreq and s.factors]
            if not others or not evict:
                raise
            for s in others:
                del s.factors
            subs[ifreq]._ensure_factors(*zrange)

    def _workers(self, zrange):
        """Frequencies in flight at once.  When the factors of all local frequencies fit in HBM together they are
        factored first, several at a time (MultiFreq.prefactor), and the sweeps then run MultiFreq.solveWorkers
        frequencies at a time; otherwise one frequency at a time, factors evicted as needed.  (Factorisations are not
        mixed with sweeps of other frequencies: measured on C4, 6.5 s instead of 3.1 s per gradient -- the sweeps'
        one-CTA-per-SM GEMMs starve the inverter-service CTAs, which need an SM to themselves.)"""
        import torch
        system = self.system
        local = system.localFreqIndices
        subs = system.subProblems
        if len(local) < 2 or not system.keepFactors or subs[local[0]].device.type != 'cuda':
            return 1
        for i in local:
            subs[i].handle                                # create handles / upload models on the caller's thread
        free, _ = torch.cuda.mem_get_info(subs[local[0]].device)
        need = sum(subs[i].factor_bytes_missing() for i in local if not subs[i].factors)     # (a model update keeps the allocations)
        if need > 0.8 * free:
            return 1
        system.prefactor(zrange)
        return system.solveWorkers

    def dpred_device(self):
        """Forward modelling with everything on the device; returns {ifreq: (R, S) tensor} for the
        frequencies this rank owns.  Several frequencies of one GPU are swept concurrently
        (MultiFreq.run_local: one stream and host thread per frequency in flight)."""
        ops = self._device_ops()
        workers = self._workers(ops['s_z'])
        panels = {}

        def one(ifreq, slot):
            self._ensure_factors(ifreq, ops['s_z'], evict=workers == 1)
            panels[slot] = self.forward_device(ifreq, out=panels.get(slot))
            d = self.extract_device(panels[slot])
            if not self.system.keepFactors:
                del self.system.subProblems[ifreq].factors
            return d
        return self.system.run_local(one, workers=workers, bytes_per_worker=self._panel_bytes())

    def upload_dobs(self, dobs):
        """Observed data (R, S, F) -> device tensor (F_local, R, S) holding this rank's frequencies, in the panel
        dtype; pass it to misfit_and_gradient to keep the data resident across evaluations."""
        import torch
        sv = self.survey
        local = self.system.localFreqIndices
        dobs = np.asarray(dobs, dtype=np.complex128).reshape((sv.nrec, sv.nsrc, sv.nfreq))
        pdt = self.system.subProblems[local[0]].panel_dtype if local else torch.complex128
        return torch.from_numpy(np.ascontiguousarray(np.moveaxis(dobs[:, :, local], 2, 0))).to(self._device_ops()['dev']).to(pdt)

    def misfit_and_gradient(self, dobs, Wd=1., to_host=True):
        """phi = 0.5 ||Wd (dpred - dobs)||^2 and g = Jtvec(Wd*Wd*(dpred - dobs), u) with wavefields
        resident in HBM; both are all-reduced over the frequency shards.  dobs: (R, S, F) array.
        Returns (phi: float, g: ndarray (N,) float64).  Observed data and the gradient scalers are uploaded once
        per call; co-resident frequencies run forward + adjoint concurrently, each into its own accumulator.
        dobs may also be the device tensor from ``upload_dobs``; to_host=False returns the all-reduced device
        tensor [g (N), phi] (float64) instead of host values."""
        import torch
        ops = self._device_ops()
        dev, sv, N = ops['dev'], self.survey, self.nrow
        local = self.system.localFreqIndices
        subs = self.system.subProblems
        # observed data of the local frequencies, (Fl, R, S), in one transfer
        do_all = dobs if isinstance(dobs, torch.Tensor) else self.upload_dobs(dobs)
        workers = self._workers(ops['s_z'])
        # gradient scalers -omega^2 / c^3 (problem.py:74-81) formed on the device; c is shared by all
        # frequencies unless the problem is viscous (per-frequency complex c)
        cinv3 = {}

        def scaler_for(ifreq):
            c = subs[ifreq].c
            key = ifreq if isinstance(self.system, ViscoMultiFreq) else -1
            if key not in cinv3:
                cinv3[key] = torch.from_numpy(np.ascontiguousarray(c, dtype=np.complex128).ravel()).to(dev).pow(-3)
            omega = 2 * np.pi * sv.freqs[ifreq]
            return cinv3[key] * (-(omega ** 2))
        if not isinstance(self.system, ViscoMultiFreq) and local:
            scaler_for(local[0])                       # upload on the caller's stream, before the workers start
        accs, phis, panels = {}, {}, {}

        def one(ifreq, slot):
            stream = _lib.current_stream_ptr(dev)
            if slot not in accs:
                accs[slot] = torch.zeros((N,), dtype=torch.complex128, device=dev)
                phis[slot] = torch.zeros((1,), dtype=torch.float64, device=dev)
                panels[slot] = [None, None]
            self._ensure_factors(ifreq, ops['s_z'], evict=workers == 1)
            uF = panels[slot][0] = self.forward_device(ifreq, out=panels[slot][0])
            d = self.extract_device(uF)
            c64 = d.dtype == torch.complex64
            do = do_all[local.index(ifreq)]
            v = torch.empty_like(d)
            _lib.check(_lib.panel_fn('hz_misfit', c64)(_lib.ptr(d), _lib.ptr(do), d.numel(), float(Wd), _lib.ptr(v), _lib.ptr(phis[slot]), stream))
            uB = panels[slot][1] = self.backproject_device(ifreq, v, out=panels[slot][1])
            scaler = scaler_for(ifreq)
            _lib.check(_lib.panel_fn('hz_gradient', c64)(_lib.ptr(uF), _lib.ptr(uB), N, sv.nsrc, _lib.ptr(scaler), _lib.ptr(accs[slot]), stream))
            if not self.system.keepFactors:
                del subs[ifreq].factors
            return None
        self.system.run_local(one, workers=workers, bytes_per_worker=2 * self._panel_bytes() if local else 0)
        red = torch.zeros((N + 1,), dtype=torch.float64, device=dev)
        for slot in accs:
            red[:N] += accs[slot].real
            red[N] += phis[slot][0]
        parallel.allreduce_sum_(red)
        if not to_host:
            return red
        host = red.cpu().numpy()
        return float(host[N]), host[:N].copy()

    # ---- adjoint-state gradient (DESIGN.md §2) ------------------------------------------------
    def _adjoint_alpha(self, ifreq):
        """dc_f/dc at every node for frequency ifreq as a host complex array, or None when c_f = c."""
        return None

    def _check_adjoint_supported(self, name='misfit_and_adjoint_gradient'):
        subs = self.system.subProblems
        for i in self.system.localFreqIndices:
            sub = subs[i]
            if not isinstance(sub, MiniZephyr):
                raise NotImplementedError('%s is built for the MiniZephyr operator only, not %s' % (name, type(sub).__name__))
            if sub.c64:
                raise NotImplementedError("%s needs complex128 factors (A^T solves); dtype='complex64' has no transposed solve"
                                          % name)

    def _adjoint_taps(self, ifreq):
        """Receiver taps of the adjoint source of one frequency: conjugated (rterms may be complex) and divided by
        premul, so that the premultiplied, unconjugated A^T solve of the back-projection returns lambda = A^-T (Rv^H v)
        itself.  Formed on the caller's stream, before any worker stream reads them."""
        ops = self._device_ops()
        key = 'b_val' if ops['mode'] == 'fixed' else 'r_val'
        if key + '_conj' not in ops:
            ops[key + '_conj'] = ops[key].conj().resolve_conj()
        pm = complex(self.system.subProblems[ifreq].premul)
        return ops[key + '_conj'] if pm == 1 else ops[key + '_conj'] / pm

    @staticmethod
    def _check_wrt(wrt):
        wrt = tuple(wrt)
        if not wrt or len(set(wrt)) != len(wrt) or any(k not in ('c', 'rho') for k in wrt):
            raise ValueError("wrt must name 'c' and/or 'rho', each at most once")
        return wrt

    def _check_dm(self, dm, wrt):
        """A model perturbation {name: N float64 values} over exactly the names of ``wrt`` -> host float64 arrays of N."""
        if not isinstance(dm, dict) or set(dm) != set(wrt):
            raise ValueError('dm must be a dict with exactly the keys %s' % (wrt,))
        out = {}
        for k in wrt:
            a = np.asarray(dm[k])
            if np.iscomplexobj(a) or a.size != self.nrow:
                raise ValueError("dm['%s'] must hold %d real values" % (k, self.nrow))
            out[k] = np.ascontiguousarray(a, dtype=np.float64).ravel()
        return out

    def _derivative_sweep(self, wrt, adjoint_data, dm=None, back=True, nextra=0):
        """The per-frequency device pipeline of the exact derivatives (DESIGN.md §2).  For every local frequency:

        1. the forward panel uF (``forward_device``);
        2. if ``dm`` is given, the Born panel dU = conj(-A^-1 dA w) in a second panel: ``hz_assemble_jvp`` along dm,
           ``hz_stencil_apply`` with scale -1/premul and an N solve over the whole depth range;
        3. v = adjoint_data(ifreq, uF, dU, extra), an (R, S) device tensor (extra: this worker's float64 accumulator
           of ``nextra`` values);
        4. if ``back``: lambda = A^-T (Rv^H v) (back-projection with the adjoint taps, A^T solve), ``hz_stencil_xcorr``
           of lambda and uF and ``hz_assemble_vjp`` into per-worker accumulators of -Re sum lambda^T (dA/dm) w.

        The caller checks that the operators are supported.  ``dm`` holds float64 device tensors of N over ``wrt``.  Where rho is not given (Gardner's rule), the tangent
        and the gradient both carry density's dependence on c.  Returns {ifreq: v} if not ``back``; otherwise the
        float64 device tensor [g_wrt[0] (N), g_wrt[1] (N), ..., extra] summed over the workers of this rank (the
        caller all-reduces it)."""
        import torch
        ops = self._device_ops()
        dev, sv, N = ops['dev'], self.survey, self.nrow
        nx, nz = int(self.nx), int(self.nz)
        local = self.system.localFreqIndices
        subs = self.system.subProblems
        workers = self._workers(ops['s_z'])
        gardner = self.systemConfig.get('rho', None) is None
        want_c, want_rho = 'c' in wrt, 'rho' in wrt
        rho_scratch = back and (want_rho or (gardner and want_c))
        tan_rho = dm is not None and gardner and want_c          # the tangent's drho_f = drho_f/dc dc (+ drho)
        lib = _lib.get_lib()

        def to_dev(a, dt):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=dt).ravel()).to(dev)
        # everything the workers share or only read is formed here, on the caller's stream, which every worker stream
        # waits for when it starts (MultiFreq.run_local)
        taps = {i: self._adjoint_taps(i) for i in local} if back else {}
        alphas = {i: (None if self._adjoint_alpha(i) is None else to_dev(self._adjoint_alpha(i), np.complex128)) for i in local}
        drho_dc = {}
        if gardner and want_c:
            # rho_f = 310 Re(c_f)^0.25 and Re(c_f) = Re(alpha_f) c  =>  drho_f/dc = rho_f / (4 Re(c))
            cr = np.real(np.asarray(self.systemConfig['c'], dtype=np.complex128)) * np.ones((nz, nx))
            drho_dc = {i: to_dev(0.25 * np.asarray(subs[i].rho, dtype=np.float64).reshape((nz, nx)) / cr, np.float64) for i in local}
        accs, extras, panels = {}, {}, {}

        def one(ifreq, slot):
            stream = _lib.current_stream_ptr(dev)
            if slot not in panels:
                if back:
                    accs[slot] = {k: torch.zeros((N,), dtype=torch.float64, device=dev) for k in wrt}
                extras[slot] = torch.zeros((nextra,), dtype=torch.float64, device=dev)
                panels[slot] = {'uF': None, 'lam': None, 'G': torch.empty((9 * N,), dtype=torch.complex128, device=dev),
                                'grho': torch.empty((N,), dtype=torch.float64, device=dev) if rho_scratch else None,
                                'drho': torch.empty((N,), dtype=torch.float64, device=dev) if tan_rho else None}
            pn = panels[slot]
            sub = subs[ifreq]
            self._ensure_factors(ifreq, ops['s_z'], evict=workers == 1)
            uF = pn['uF'] = self.forward_device(ifreq, out=pn['uF'])
            dU = None
            if dm is not None:
                dc, drho = dm.get('c'), dm.get('rho')
                if tan_rho:
                    drho = torch.mul(drho_dc[ifreq], dc, out=pn['drho']) if drho is None else \
                        torch.addcmul(drho, drho_dc[ifreq], dc, out=pn['drho'])
                sub._bind_stream()
                _lib.check(lib.hz_assemble_jvp(sub.handle, _lib.ptr(dc), _lib.ptr(drho), _lib.ptr(alphas[ifreq]), _lib.ptr(pn['G'])),
                           sub.handle)
                if pn['lam'] is None:
                    pn['lam'] = torch.empty_like(uF)
                scale = -1. / complex(sub.premul)
                _lib.check(lib.hz_stencil_apply(_lib.ptr(pn['G']), _lib.ptr(uF), nx, nz, sv.nsrc, scale.real, scale.imag,
                                                _lib.ptr(pn['lam']), stream))
                dU = sub.solve_device(pn['lam'], (-1, -1))          # the secondary source fills every depth
            v = adjoint_data(ifreq, uF, dU, extras[slot])
            if back:
                lam = pn['lam'] = self.backproject_device(ifreq, v, out=pn['lam'], vals=taps[ifreq], conjugate=False, trans='T')
                _lib.check(lib.hz_stencil_xcorr(_lib.ptr(lam), _lib.ptr(uF), nx, nz, sv.nsrc, _lib.ptr(pn['G']), stream))
                sub._bind_stream()
                g_c = accs[slot]['c'] if want_c else None
                if rho_scratch:
                    pn['grho'].zero_()
                _lib.check(lib.hz_assemble_vjp(sub.handle, _lib.ptr(pn['G']), _lib.ptr(alphas[ifreq]), _lib.ptr(g_c), _lib.ptr(pn['grho'])),
                           sub.handle)
                if want_rho:
                    accs[slot]['rho'] += pn['grho']
                if drho_dc:
                    accs[slot]['c'] += pn['grho'] * drho_dc[ifreq]
            if not self.system.keepFactors:
                del sub.factors
            return None if back else v
        per_worker = 2 * self._panel_bytes() + 160 * N + (8 * N if tan_rho else 0)
        res = self.system.run_local(one, workers=workers, bytes_per_worker=per_worker if local else 0)
        if not back:
            return res
        nk = len(wrt)
        red = torch.zeros((nk * N + nextra,), dtype=torch.float64, device=dev)
        for slot in accs:
            for j, k in enumerate(wrt):
                red[j * N:(j + 1) * N] += accs[slot][k]
            red[nk * N:] += extras[slot]
        return red

    def misfit_and_adjoint_gradient(self, dobs, Wd=1., wrt=('c',), to_host=True):
        """phi = 0.5 ||Wd (dpred - dobs)||^2 and its exact gradient with respect to the model parameters named in
        ``wrt`` ('c', 'rho'), by the adjoint-state method: per frequency a forward solve, an A^T solve of the
        back-projected residual, the stencil cross-correlation of the two panels and the vector-Jacobian product of
        the assembly (DESIGN.md §2).  Unlike ``misfit_and_gradient``, which follows the reference's Jtvec formula,
        this is the derivative of phi: what a line search or a quasi-Newton method needs.

        Returns (phi, {'c': g_c, 'rho': g_rho}) with the requested keys only (float64 arrays of N).  For the viscous
        problem g_c is with respect to the real base velocity; where rho is not given (Gardner's rule rho = 310
        Re(c)^0.25), g_c includes the change of rho with c and g_rho is the partial derivative at fixed c.  dobs: the
        (R, S, F) data or the device tensor from ``upload_dobs``.  to_host=False returns the all-reduced device
        tensor [g_wrt[0] (N), g_wrt[1] (N), ..., phi] (float64) instead.  MiniZephyr operators in complex128 only."""
        import torch
        wrt = self._check_wrt(wrt)
        self._check_adjoint_supported()
        local = self.system.localFreqIndices
        do_all = dobs if isinstance(dobs, torch.Tensor) else self.upload_dobs(dobs)
        lib = _lib.get_lib()
        dev = self._device_ops()['dev']

        def residual(ifreq, uF, dU, phi):
            d = self.extract_device(uF)
            do = do_all[local.index(ifreq)]
            v = torch.empty_like(d)
            _lib.check(lib.hz_misfit(_lib.ptr(d), _lib.ptr(do), d.numel(), float(Wd), _lib.ptr(v), _lib.ptr(phi),
                                     _lib.current_stream_ptr(dev)))
            return v
        red = self._derivative_sweep(wrt, residual, nextra=1)
        parallel.allreduce_sum_(red)
        if not to_host:
            return red
        nk, N = len(wrt), self.nrow
        host = red.cpu().numpy()
        return float(host[nk * N]), {k: host[j * N:(j + 1) * N].copy() for j, k in enumerate(wrt)}

    # ---- Born modelling, its adjoint and Gauss-Newton products (DESIGN.md §2) ------------------------------------
    def _dm_to_device(self, dm, wrt, name):
        import torch
        self._check_adjoint_supported(name)
        dev = self._device_ops()['dev']
        return {k: torch.from_numpy(a).to(dev) for k, a in self._check_dm(dm, wrt).items()}

    def born_dpred(self, dm, wrt=('c',)):
        """J dm: the exact linearised ("Born") data of a real model perturbation dm = {'c': dc, 'rho': drho} (the
        keys of ``wrt``, each N float64 values, the layout ``misfit_and_adjoint_gradient`` returns).  Per frequency a
        forward solve, the tangent of the assembled planes (``hz_assemble_jvp``), the Born secondary source
        -dA w (``hz_stencil_apply``), an N solve and the receiver extraction.  Returns the (R, S, F) complex128 data,
        gathered over the frequency shards as ``survey.dpred`` does.  For the viscous problem dc perturbs the real base
        velocity; where rho is not given (Gardner's rule) density follows dc.  MiniZephyr operators in complex128 only."""
        wrt = self._check_wrt(wrt)
        dmd = self._dm_to_device(dm, wrt, 'born_dpred')
        dd = self._derivative_sweep(wrt, lambda ifreq, uF, dU, extra: self.extract_device(dU), dm=dmd, back=False)
        return self.survey._gather_freqs(dd).cpu().numpy()

    def born_adjoint(self, v, wrt=('c',)):
        """J^H v: the exact adjoint of ``born_dpred`` under the real inner products Re sum conj(a) b on data and the
        dot product on the model, as a dict of N float64 arrays over ``wrt``, all-reduced over the frequency shards.
        v: (R, S, F) data or the device tensor of ``upload_dobs``.  Per frequency a forward solve, the A^T solve of the
        back-projected v, ``hz_stencil_xcorr`` and ``hz_assemble_vjp``: the adjoint path of
        ``misfit_and_adjoint_gradient``, which is born_adjoint(Wd^2 (dpred - dobs))."""
        import torch
        wrt = self._check_wrt(wrt)
        self._check_adjoint_supported('born_adjoint')
        local = self.system.localFreqIndices
        v_all = v if isinstance(v, torch.Tensor) else self.upload_dobs(v)
        red = self._derivative_sweep(wrt, lambda ifreq, uF, dU, extra: v_all[local.index(ifreq)])
        return self._reduce_model(red, wrt)

    def gauss_newton_hvec(self, dm, Wd=1., wrt=('c',)):
        """H_GN dm = J^H Wd^2 J dm, the Gauss-Newton Hessian of 0.5 ||Wd (dpred - dobs)||^2 applied to dm, as a dict of
        N float64 arrays over ``wrt``, with one all-reduce.  Per frequency, all on the device and on one set of
        factors: the forward solve, the Born solve, the extraction scaled by Wd^2, the A^T solve of its
        back-projection, ``hz_stencil_xcorr`` and ``hz_assemble_vjp``.  With keepFactors and an unchanged model,
        nothing is refactored.  Symmetric and positive semi-definite: <dm, H dm> = ||Wd J dm||^2."""
        wrt = self._check_wrt(wrt)
        dmd = self._dm_to_device(dm, wrt, 'gauss_newton_hvec')
        w2 = float(Wd) ** 2

        def weighted(ifreq, uF, dU, extra):
            return self.extract_device(dU).mul_(w2)
        red = self._derivative_sweep(wrt, weighted, dm=dmd)
        return self._reduce_model(red, wrt)

    def _reduce_model(self, red, wrt):
        parallel.allreduce_sum_(red)
        N = self.nrow
        host = red.cpu().numpy()
        return {k: host[j * N:(j + 1) * N].copy() for j, k in enumerate(wrt)}

class Helm2DProblem(HelmBaseProblem):
    SystemWrapper = MultiFreq


class Helm2DViscoProblem(HelmBaseProblem):
    SystemWrapper = ViscoMultiFreq

    def _adjoint_alpha(self, ifreq):
        """c_f = fact_f c (1 + i/(2Q)) (ViscoMultiFreq.spUpdates), so dc_f/dc = fact_f (1 + i/(2Q))."""
        system = self.system
        Q = np.asarray(system.Q, dtype=np.float64).reshape((int(self.nz), int(self.nx)))
        alpha = 1. + 0.5j / Q
        if system.disperseFreqs:
            alpha = alpha * (1. + (np.log(system.freqs[ifreq] / system.freqBase) / (np.pi * Q)))
        return alpha
