/* zephyr_b200 -- C ABI of the B200-native Helmholtz forward/adjoint hot path.
 *
 * This is the drop-in boundary for uwoseis/zephyr's frequency-domain solve path (SURVEY.md 8(b)).
 * The reference is pure Python and has no FFI of its own; the entry points below are what a
 * ctypes binding on the reference side would call in place of the numpy/scipy internals of the
 * cited functions (paths relative to /root/reference/zephyr/).  INTEGRATION.md shows that binding.
 *
 * Conventions
 *  - every function returns an int status (HZ_OK == 0); no exception or abort crosses the ABI;
 *    hz_last_error(handle) returns a message for the last failure on that handle
 *    (hz_last_error(NULL): last failure of a handle-less call on this thread);
 *  - all array arguments are DEVICE pointers unless the name ends in `_host`; the caller owns
 *    every buffer it passes; the library owns what it allocates (factors, workspaces) and frees
 *    it in hz_free_factors / hz_destroy (both idempotent);
 *  - complex arrays are interleaved (re, im) float64 pairs, row-major: numpy complex128 C order;
 *  - a handle is bound to one device and one stream; not thread-safe per handle, re-entrant
 *    across handles.  `stream` arguments are cudaStream_t passed as void* (NULL: default stream);
 *  - wavefield / right-hand-side panels X are (nf*N) x S with row(f, iz, ix) = f*N + iz*nx + ix,
 *    N = nx*nz, nf = 1 (MiniZephyr) or 2 (Eurus) -- the reference's own ordering
 *    (backend/minizephyr.py:308-312, backend/eurus.py:463).
 */
#ifndef ZEPHYR_B200_H
#define ZEPHYR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hz_ctx* hz_handle_t;

enum {
    HZ_OK = 0,
    HZ_EINVAL = 1,      /* bad argument                     -> Python ValueError            */
    HZ_EDIM = 2,        /* 'dimension mismatch'             -> ValueError (eurus.py:526)     */
    HZ_ENOMEM = 3,      /* device allocation failed         -> MemoryError                   */
    HZ_ECUDA = 4,       /* CUDA runtime error               -> RuntimeError                  */
    HZ_ESINGULAR = 5,   /* zero / non-finite pivot detected -> numpy.linalg.LinAlgError      */
    HZ_ESTATE = 6,      /* call out of order (e.g. solve before factor) -> RuntimeError      */
    HZ_ENOTIMPL = 7,    /* feature not built                -> NotImplementedError           */
    HZ_EACCURACY = 8    /* accuracy probe of a solve failed -> numpy.linalg.LinAlgError      */
};
enum { HZ_C128 = 0, HZ_C64 = 1 };
enum { HZ_DISC_MINIZEPHYR = 0, HZ_DISC_EURUS = 1 };
enum { HZ_OP_N = 0, HZ_OP_T = 1, HZ_OP_H = 2 };   /* which operator a solve inverts: A, A^T, A^H (conjugate transpose) */

const char* hz_version(void);
const char* hz_last_error(hz_handle_t h);

/* ---- discretisation object: backend/discretization.py:18-106 (BaseDiscretization), with the
 *      grid attributes of backend/base.py:11-109.  freeSurf_host[4] as base.py:61-65. ------------- */
int hz_create(hz_handle_t* out, int device, int dtype, int disc, int64_t nx, int64_t nz, double dx, double dz,
              int nPML, double cPML, const int32_t* freeSurf_host, void* stream);
int hz_destroy(hz_handle_t h);                       /* discretization.py:98-99 (__del__)          */
/* Rebind the handle to another stream of its device (the stream given to hz_create is only the initial
 * binding).  Work already queued on the old stream is ordered before anything issued afterwards.  The host
 * classes call it with the caller's current stream before every factor / solve, so a handle follows the
 * stream context (and the host thread) it is used from.                                            */
int hz_set_stream(hz_handle_t h, void* stream);

/* model arrays (nz, nx): c complex128, the rest float64; theta/eps/delta only for Eurus
 * (base.py:112-149).  on_device = 0: the pointers are host pointers and are copied.            */
int hz_set_model(hz_handle_t h, const void* c, const double* rho, const double* theta, const double* eps,
                 const double* delta, int on_device);

/* a1/a2: stencil + PML coefficients on device, block-tridiagonal layout.  Replaces
 * MiniZephyr._initHelmholtzNinePoint (minizephyr.py:40-298) / Eurus._initHelmholtzNinePoint
 * (eurus.py:28-485).  omega_damped = 2*pi*freq - i/tau (discretization.py:33-41).            */
int hz_assemble(hz_handle_t h, double freq_re, double freq_im, double tau, double ky);
/* coefficient planes to host: out[(fr*nf+fc)*9 + slot][iz][ix], slot = (dz+1)*3 + (dx+1) -- the
 * entries of `Disc.A` (minizephyr.py:300-306), for parity tests.                              */
int hz_get_coefficients(hz_handle_t h, void* out_host);
/* The inverse: load caller-assembled coefficient planes (same layout) instead of calling hz_assemble.  This is
 * the entry behind the `Solver`-compatible shim -- systemConfig['Solver'](A_csc).solve(rhs), the third plug-in point
 * of the reference (backend/discretization.py:83 via problemo) -- which receives an already assembled matrix.      */
int hz_set_coefficients(hz_handle_t h, const void* planes_host);

/* a3 (factor): block LU of the block-tridiagonal operator with explicit block inverses held in
 * HBM.  Replaces BaseDiscretization.Ainv (discretization.py:78-85) + problemo.BestSolver +
 * scipy.sparse.linalg.splu.  `twist` = block row where the two elimination chains meet
 * (-1: nz/2); choosing the source depth halves the substitution work for shallow sources.      */
int hz_factor(hz_handle_t h, int64_t twist);
int hz_has_factors(hz_handle_t h, int32_t* out);     /* discretization.py:91-93 (.factors)          */
int hz_free_factors(hz_handle_t h);                  /* discretization.py:94-96 (del .factors)      */
int hz_factor_bytes(hz_handle_t h, int64_t* bytes);  /* HBM the factors of this handle need          */
int hz_factor_resident_bytes(hz_handle_t h, int64_t* bytes);  /* ... and how much of it the handle already holds (valid or
                                                       * invalidated factors: a model update keeps the allocation) */
int hz_get_block_inverse(hz_handle_t h, int64_t iz, void* out_host);   /* (b x b), tests only       */

/* a3 (solve): X <- conj(premul * A^{-1} X) in place for all S columns at once
 * (discretization.py:101-106: `(self.Ainv * (self.premul * rhs)).conjugate()`).
 * z_first/z_last: first/last block row (iz) holding a non-zero right-hand side, or -1 when
 * unknown; refine: iterative-refinement steps with the stencil residual (0 = none; -1 = library default: 0,
 * or 1 for complex64 handles on the tensor-core path, whose TF32 accumulation needs it to stay within 1e-4);
 * resid_host (optional): ||q - A x||_F / ||q||_F of the final solution.                          */
int hz_solve(hz_handle_t h, void* X, int64_t S, double premul_re, double premul_im, int conjugate,
             int64_t z_first, int64_t z_last, int refine, double* resid_host);
/* X <- conj(premul * op(A)^{-1} X), op = HZ_OP_N (== hz_solve), HZ_OP_T (A^T) or HZ_OP_H (A^H), from the same factors:
 * the Schur complements of A^T are the transposes of those of A, so the sweeps apply the stored block inverses as
 * S_i^{-T} / S_i^{-H} with the transposed (conjugated) stencil -- scipy's SuperLU.solve(rhs, trans='N'|'T'|'H').  Other
 * arguments, the accuracy probe (the first solve after hz_factor probes, whatever its op) and the refinement use the
 * op(A) residual and otherwise behave as in hz_solve.  Bad op -> HZ_EINVAL; T / H on a complex64 handle -> HZ_ENOTIMPL. */
int hz_solve_op(hz_handle_t h, int op, void* X, int64_t S, double premul_re, double premul_im, int conjugate,
                int64_t z_first, int64_t z_last, int refine, double* resid_host);

/* Accuracy probe.  The reference's SuperLU pivots; the block elimination here does not pivot across
 * 32-wide panels.  The first hz_solve / hz_solve_op (refine = 0) after every hz_factor therefore measures, in FP64,
 * the 9-point stencil residual ||q - op(A) x|| / ||q|| of the first right-hand-side column and returns
 * HZ_EACCURACY when it exceeds 1e-7 (complex128) / 1e-2 (complex64) instead of a silently inaccurate
 * wavefield.  hz_last_probe returns the last measured value (-1: none yet); option "probe_check" = 0
 * disables the probe.  With refine >= 1 the refinement loop's own residual takes its place.        */
int hz_last_probe(hz_handle_t h, double* out);

int hz_synchronize(hz_handle_t h);

/* Measurement support (no reference counterpart).  hz_profile: enable/disable sampled CUDA-event
 * timing of the contraction kernel on this handle and read+reset the counters: out_host[6] =
 * {substitution-GEMM sampled ms, sampled launches, all launches, update-GEMM ditto} (may be NULL).
 * hz_launch_count: kernels launched by this library in this process so far.                     */
int hz_profile(hz_handle_t h, int enable, double* out_host);
/* Tuning knobs, key/value (defaults first).
 *   "gemm_3m"    1: the substitution GEMMs form complex products with THREE real tensor-core products
 *                (Re = ar br - ai bi, Im = (ar + ai)(br + bi) - ar br - ai bi) instead of four: 16-18 % faster
 *                (the kernel is bound by the FP64 tensor pipe), normwise as accurate (1.5e-13 between the two
 *                at 1000 x 3000); bit 1 (values 2, 3): the same for the Gauss-Jordan update tiles (measured
 *                slower there: that kernel is not bound by its DMMA count); 0: four products everywhere.
 *   "gj_mode"    1: fused Gauss-Jordan step, rank-32 update every step; 2: delayed rank-64 updates;
 *                0: separate panel + update launches; 3: one launch per block row (dependence counters);
 *                4: one persistent grid pulling runnable work items of both chains (3, 4: measured slower).
 *   "gj_service" 2: the 32x32 pivot-block inverses run in a persistent one-CTA-per-chain service
 *                kernel that owns its SM and walks the steps of a block row on its own (it forms
 *                the one panel piece it needs itself, from a tile the step kernel hands over);
 *                1: same service, one request per step posted by the step kernel; 0: inverter
 *                CTA inside the step kernel.  The library falls back to 0 by itself if the
 *                service cannot run beside the step kernels (e.g. under a profiler that
 *                serialises launches).
 *   "gj_tile"    update-tile variant of the step kernel (3: 64x64 tile in four rolled row passes;
 *                0..11: the other measured variants, see gj_variants in hz_api.cu).
 *   "gj_order", "gj_inv"  CTA role order / inverter block index inside the step kernel (studies).
 *   "gj_colper"  1; 2: each column-block CTA owns two column blocks (study: slower).
 *   "gj_colpair" 0; 1: two column blocks per CTA processed side by side, four warps each (study: slower).
 *   "gj_lean"    0; 1: service-mode launches use an instance of the step kernel without the in-kernel inverter and the
 *                alternative column-block paths (2 976 instead of 11 888 SASS instructions; study: no gain).
 *   "gj_colslow" 0; 1: column-block CTAs stage their operands in dependent rounds (the code before r2p, for A/B runs).
 *   "gj_coltile" 0; 1: the column-block CTAs process the last update tiles while they wait for the
 *                inverse (study: slower, they then pick the inverse up late).
 *   "gj_pdl"     0/1 programmatic dependent launch between steps.
 *   "gj_trace"   1: record per-CTA timestamps for every block; t >= 2: only for block t-2 of the top
 *                chain and its mirror image in the bottom chain; "gj_trace_chain" selects which
 *                chain hz_get_trace returns.
 *   "c64_fp64_factor" 1: complex64 handles factorise in FP64 and round each finished inverse;
 *                0: the whole complex64 factorisation runs in FP32 (study option; not accurate
 *                enough at 1000 x 3000: up to 5e-3 vs complex128).                                */
int hz_set_option(hz_handle_t h, const char* key, double value);
/* Diagnostics ("gj_trace" = 1): per-CTA (start, end) globaltimer ns for every Gauss-Jordan step of
 * the block factored last; out_host[steps][grid][16].                                             */
int hz_get_trace(hz_handle_t h, int64_t* out_host, int64_t cap, int64_t* steps, int64_t* grid);
int hz_launch_count(int64_t* out);
/* Option "factor_graph" (0 never = default, 1 always, -1 from the second factorisation of a handle on when the launch
 * sequence has at most 16384 kernels): the factorisation's launch sequence is captured once into a CUDA graph and
 * replayed by later hz_factor calls on the same buffers.  Measured: no gain (the steps are bound by dependent-kernel
 * latency on the device, not by the host launch rate), hence off.  out2 = {kernels in the graph (0: none), replays}. */
int hz_factor_graph_info(hz_handle_t h, int64_t* out2);
/* Diagnostics of the pivot-block inverter (FP32 Gauss-Jordan + Newton-Schulz on DMMA, hz_factor.cuh): out4 = {inverses,
 * fallbacks to the FP64 Gauss-Jordan, Newton steps, 0} on the current device since the library was loaded.              */
int hz_newton_stats_get(int64_t* out4);

/* ---- right-hand sides: X[row[j]*S + col[j]] += val[j]*scale.  Injects SparseKaiserSource
 *      columns (backend/source.py:305-317) or residual sources (middleware/survey.py:171-188). -- */
int hz_scatter_coo(void* X, int64_t S, int64_t nnz, const int64_t* row, const int64_t* col, const void* val,
                   double scale_re, double scale_im, void* stream);

/* a5: SimpleSource.linIndexOf (backend/source.py:56-88), bit-exact.  locs (nloc, 2) = [x, z].     */
int hz_nearest_index(int64_t nx, int64_t nz, double dx, double dz, double xorig, double zorig,
                     const double* locs, int64_t nloc, int64_t* out_idx, void* stream);
/* a6: SparseKaiserSource.__call__ (backend/source.py:213-317).  Per location up to (2*ireg+1)^2
 * entries (rows, real values) in the reference's emission order; counts[s] of them are valid.  */
int hz_kaiser_taps(int64_t nx, int64_t nz, double dx, double dz, double xorig, double zorig, int ireg,
                   const int32_t* freeSurf_host, const double* locs, const int64_t* idx, int64_t nloc,
                   int64_t* rows, double* vals, int32_t* counts, void* stream);

/* a8/a9: Out[orow(i)*ldout + s] (stride ostride) = sum_j val[j] * In[col[j]*ldin + s] over CSR row
 * i.  Receiver extraction (middleware/survey.py:141-160) and residual back-projection
 * (survey.py:171-188).  orow may be NULL (identity).                                            */
int hz_spmm_csr(int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, const int64_t* orow,
                const void* In, int64_t ldin, int64_t S, void* Out, int64_t ldout, int64_t ostride,
                int accumulate, void* stream);

/* a8/a9 with 'relative' receiver geometry (middleware/survey.py:120-125: one receiver operator per source).
 * CSR row i = r*S + s holds the taps of receiver r of source s.  transpose = 0 (extraction):
 * Out[i] = sum_j val[j] * In[col[j]*ld + s]; transpose = 1 (back-projection, survey.py:171-188):
 * Out[col[j]*ld + s] += val[j] * In[i] (Out must be zeroed by the caller).                       */
int hz_spmm_percol(int transpose, int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, int64_t S,
                   const void* In, void* Out, int64_t ld, void* stream);

/* a10: g[n] += scaler[n] * sum_s uF[n,s]*uB[n,s]  (middleware/problem.py:74-81,125-164).         */
int hz_gradient(const void* uF, const void* uB, int64_t N, int64_t S, const void* scaler, void* g, void* stream);
/* a11: phi += 0.5*||wd (d - dobs)||^2 ; v = wd*wd*(d - dobs) (v may be NULL).                    */
int hz_misfit(const void* d, const void* dobs, int64_t n, double wd, void* v, double* phi, void* stream);

/* Adjoint-state gradient of MiniZephyr (DESIGN.md §2).  hz_stencil_xcorr: the stencil cross-correlation of an adjoint
 * panel lam and a forward panel u (both complex128, N x S, N = nx*nz, row-major), u as the forward solve returns it
 * (conjugated):  G[slot*N + i] = sum_s lam[i*S + s] * conj(u[(i + off(slot))*S + s]),  off(slot) = (slot/3 - 1)*nx +
 * (slot%3 - 1); G is 9*N complex128, overwritten, zero on boundary rows.
 * hz_assemble_vjp: the vector-Jacobian product of the handle's last hz_assemble with G, added into g_c and g_rho
 * (float64, N; either may be NULL, not both):  g_c[n] -= Re(alpha[n] sum_{slot,i} G[slot][i] d coef[slot][i] / d c[n]),
 * g_rho[n] -= Re(sum G d coef / d rho[n]).  alpha (complex128, N) may be NULL (1).  On the handle's stream.  Complex64
 * and Eurus handles: HZ_ENOTIMPL; coefficients loaded with hz_set_coefficients: HZ_ESTATE.                        */
int hz_stencil_xcorr(const void* lam, const void* u, int64_t nx, int64_t nz, int64_t S, void* G, void* stream);
int hz_assemble_vjp(hz_handle_t h, const void* G, const void* alpha, double* g_c, double* g_rho);

/* Born modelling of MiniZephyr (DESIGN.md §2, "Born modelling and Gauss-Newton products"); the exact transposes of the
 * two entries above.  hz_assemble_jvp: the Jacobian-vector product of the handle's last hz_assemble along a real model
 * perturbation dc, drho (float64, N; either may be NULL, not both):  dcoef[slot*N + i] = sum_n (d coef[slot][i] / d c[n])
 * alpha[n] dc[n] + (d coef[slot][i] / d rho[n]) drho[n], 9*N complex128 in the layout of the assembled planes,
 * overwritten, zero on boundary rows.  alpha (complex128, N) may be NULL (1).  For any G,
 * Re sum G dcoef = -(g_c . dc + g_rho . drho) with g_c, g_rho from hz_assemble_vjp.  On the handle's stream; the same
 * refusals as hz_assemble_vjp.
 * hz_stencil_apply: the tangent stencil applied to a forward panel u (complex128, N x S, as the forward solve returns it):
 * out[i*S + s] = scale * sum_slot dcoef[slot*N + i] * conj(u[(i + off(slot))*S + s]), zero on boundary rows; out must
 * not overlap u.  With scale = -1/premul, the conjugating solve (hz_solve, conjugate = 1) of out returns the Born field
 * conj(-A^-1 dA w).  Duality with hz_stencil_xcorr: sum lam .* out = scale sum G .* dcoef.                         */
int hz_assemble_jvp(hz_handle_t h, const double* dc, const double* drho, const void* alpha, void* dcoef);
int hz_stencil_apply(const void* dcoef, const void* u, int64_t nx, int64_t nz, int64_t S, double scale_re, double scale_im,
                     void* out, void* stream);

/* Pseudo-Hessian diagonal of MiniZephyr (DESIGN.md §2, "Pseudo-Hessian").  hz_wavefield_lagcorr: the lag correlation of
 * a forward panel u (complex128, N x S, as the forward solve returns it):  C[l*N + p] = sum_s conj(u[p*S + s]) *
 * u[(p + delta_l)*S + s] for the 13 lags delta_l = (dz, dx) in the order (0,0), (0,1), (0,2), (1,-2..2), (2,-2..2), zero
 * where p + delta_l lies outside the grid; C is 13*N complex128, overwritten.
 * hz_pseudo_hessian: P_m[n] = sum_s ||(d A / d m_n) w_s||^2 (w = conj(u)) of the handle's last hz_assemble, contracted
 * from C and added into p_c and p_rho (float64, N; either may be NULL, not both).  The c column is
 * alpha[n] dA/dc_n (alpha complex128, N, may be NULL: 1) plus drho_dc[n] dA/drho_n when drho_dc (float64, N) is given
 * (Gardner's rule), combined before squaring: the column hz_assemble_jvp applies along e_n.  On the handle's stream;
 * the same refusals as hz_assemble_vjp.                                                                              */
int hz_wavefield_lagcorr(const void* u, int64_t nx, int64_t nz, int64_t S, void* C, void* stream);
int hz_pseudo_hessian(hz_handle_t h, const void* C, const void* alpha, const double* drho_dc, double* p_c, double* p_rho);

/* Gauss-Newton Hessian diagonal of MiniZephyr, H_nn = sum_r,s |(J e_n)_{r,s}|^2 without the data weight (DESIGN.md §2,
 * "Gauss-Newton diagonal").  hz_wavefield_lagcorr4: the lag correlation of radius 4 of a panel u (complex128, N x S):
 * C41[l*N + p] = sum_s conj(u[p*S + s]) * u[(p + delta_l)*S + s] for the 41 lags delta_l = (dz, dx) in the order
 * (0,0), (0,1..4), (1,-4..4), (2,-4..4), (3,-4..4), (4,-4..4), zero where p + delta_l lies outside the grid; C41 is
 * 41*N complex128, overwritten.  Its planes of the 13 lags of hz_wavefield_lagcorr hold the same values.
 * hz_gauss_newton_diag: with C41 from the forward panel u (C(p, p') = sum_s w_s[p] conj(w_s[p']), w = conj(u)) and
 * Gam13 = hz_wavefield_lagcorr of the conjugated receiver Green's functions conj(g_r), g_r = A^-T conj(Rv[r, .])^T
 * (Gam(i, i') = sum_r g_r[i] conj(g_r[i'])), adds
 *     H_m[n] = sum_{i,i'} Gam(i, i') sum_{a,b} (dA/dm_n)[i, i + off(a)] conj((dA/dm_n)[i', i' + off(b)]) C(i + off(a), i' + off(b))
 * into p_c and p_rho (float64, N; either may be NULL, not both), for the derivative of the handle's last hz_assemble
 * with alpha and drho_dc as in hz_pseudo_hessian.  With Gam the identity (zero-lag plane 1, the others 0) this is
 * hz_pseudo_hessian.  On the handle's stream; the same refusals as hz_pseudo_hessian.                                 */
int hz_wavefield_lagcorr4(const void* u, int64_t nx, int64_t nz, int64_t S, void* C41, void* stream);
int hz_gauss_newton_diag(hz_handle_t h, const void* C41, const void* Gam13, const void* alpha, const double* drho_dc, double* p_c,
                         double* p_rho);

/* complex64 variant (hz_create(dtype = HZ_C64)): block inverses are stored in complex64 (planar: a real and an
 * imaginary float32 plane per block) and applied by the tcgen05 tensor cores: kind::tf32 MMAs with 3xTF32 operand
 * splitting (FP32-like products), tiles staged by TMA, accumulators in TMEM, split-K partial sums combined with
 * red.global.add (option "c64_tf32" = 0 selects the round-1 path: interleaved storage + FP32 FFMA contraction; handles
 * with checkpointed factors use that path by default, because the refinement sweep the tensor-core contraction needs
 * would repeat the recomputation between checkpoints -- "c64_tf32" = 2 forces the tensor cores there too).  X panels
 * of hz_solve are complex64; the factorisation arithmetic is FP64 by default (see "c64_fp64_factor"); assembly,
 * Schur-complement formation and the O(b S) coupling keep FP64 arithmetic.  Panel-typed helpers for complex64 panels
 * (val / scaler / g stay complex128):                                                                                  */
int hz_scatter_coo_c64(void* X, int64_t S, int64_t nnz, const int64_t* row, const int64_t* col, const void* val,
                       double scale_re, double scale_im, void* stream);
int hz_spmm_csr_c64(int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, const int64_t* orow,
                    const void* In, int64_t ldin, int64_t S, void* Out, int64_t ldout, int64_t ostride,
                    int accumulate, void* stream);
int hz_spmm_percol_c64(int transpose, int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, int64_t S,
                       const void* In, void* Out, int64_t ld, void* stream);
int hz_gradient_c64(const void* uF, const void* uB, int64_t N, int64_t S, const void* scaler, void* g, void* stream);
int hz_misfit_c64(const void* d, const void* dobs, int64_t n, double wd, void* v, double* phi, void* stream);

/* Test hook for the tcgen05 contraction of the complex64 variant (hz_tf32.cuh): C += alpha * A * Y with A (M x K) and
 * Y TRANSPOSED (N x K) as PLANAR float32 (real plane followed by imaginary plane, row strides lda / ldy floats,
 * multiples of 4: both operands K-major) and C interleaved complex64 (ldc).  kind::tf32 MMAs with 3xTF32 operand splitting, TMA-staged tiles, TMEM accumulators.   */
int hz_cgemm_tf32(int64_t M, int64_t N, int64_t K, double alpha, const float* A_planes, int64_t lda, const float* Y_planes, int64_t ldy,
                  void* C, int64_t ldc, void* stream, float* dbg /* NULL, or >= 160 KB of floats: tile / accumulator dump of CTA 0 */,
                  int variant /* 0; studies: bits 0-7 mode (1: plain TF32), bits 8-15 tile N (32/64/128), bits 16-23 split-K factor */);
/* Test hook for the DMMA contraction: C = beta*C + alpha*A*B (row-major complex128).            */
int hz_zgemm(int64_t M, int64_t N, int64_t K, double alpha, const void* A, int64_t lda, const void* B,
             int64_t ldb, int beta, void* C, int64_t ldc, int tile, void* stream);
/* ... with op(A): C = beta*C + alpha*op(A)*B, opA = HZ_OP_N (A is M x K), HZ_OP_T or HZ_OP_H (A is K x M, applied
 * transposed / conjugate-transposed); tile: -1 = the host's pick for (M, N), 0..6 = candidate tiling 64x64, 56x64,
 * 48x64, 40x64, 32x64, 32x32, 16x32; gemm_3m: 0 four, 1 three real products per complex product -- every kernel
 * instance the substitution sweeps can run.                                                     */
int hz_zgemm_op(int64_t M, int64_t N, int64_t K, double alpha, const void* A, int64_t lda, int opA, const void* B,
                int64_t ldb, int beta, void* C, int64_t ldc, int tile, int gemm_3m, void* stream);

#ifdef __cplusplus
}
#endif
#endif
