// Born modelling of the MiniZephyr operator: the Jacobian-vector product of the assembly and the tangent stencil applied
// to a forward panel (DESIGN.md §2, "Born modelling and Gauss-Newton products").
//
// Per frequency, with w = A^-1 p (the forward field before its conjugation) and a real model perturbation dm = (dc, drho):
//     dA = sum_n (dA/dc_n) alpha_n dc_n + (dA/drho_n) drho_n ,   dw = -A^-1 dA w ,   J dm = Rv conj(dw) .
// dA has the nine-plane layout of A, so the secondary source -dA w is
//   1. assemble_mz_jvp_kernel:  dcoef[slot][i] = sum_n dcoef[slot][i]/dc_n alpha_n dc_n + dcoef[slot][i]/drho_n drho_n
//   2. stencil_apply_kernel:    out[i, s] = scale sum_slot dcoef[slot][i] w_s[i + off(slot)]
// followed by an N solve of the library.  Both are the exact transposes of the two adjoint-gradient kernels
// (hz_adjoint.cuh): assemble_mz_jvp_kernel of assemble_mz_vjp_kernel, stencil_apply_kernel of stencil_xcorr_kernel.
#pragma once
#include "hz_platform.h"
#include "hz_assemble.cuh"
#include "hz_adjoint.cuh"

// ------------------------------------------------------------------------------------------------
// T_s(b, X) for s = 0..8: the stencil part of an interior row of assemble_mz_kernel (everything but the mass term
// w_s K[i + off(s)]), with the neighbour buoyancy averages b[k] and the PML terms X of the row.  The expressions are
// those of assemble_mz_kernel, term by term; T is linear in b and linear in X (mz_h is its transpose in G).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mz_t(const double b[9], const MzPml& X, const MzGridConst& g, cplx out[9]) {
    const double ac = 0.5461, bc = 0.4539;
    const double bMM = b[0], bME = b[1], bMP = b[2], bEM = b[3], bEP = b[5], bPM = b[6], bPE = b[7], bPP = b[8];
    const cplx lap = (X.r1zsq + X.r1xsq) * g.i4dxz;
    const cplx g_p = (X.r2z + X.r2x) * g.i4dd, g_m = (X.r2z - X.r2x) * g.i4dd;
    const cplx ez = (X.r1zsq * g.idz_ - X.r2z * 0.5) * g.idz_, fz = (X.r1zsq * g.idz_ + X.r2z * 0.5) * g.idz_;
    const cplx ex = (X.r1xsq * g.idx_ - X.r2x * 0.5) * g.idx_, fx = (X.r1xsq * g.idx_ + X.r2x * 0.5) * g.idx_;
    const cplx mz_ = (bc * g.i4dxz) * (X.r1zsq - X.r1xsq), mx_ = (bc * g.i4dxz) * (X.r1xsq - X.r1zsq);
    out[0] = (bc * bMM) * (lap - g_p);
    out[1] = (ac * bME) * ez + mz_ * (bMP + bMM);
    out[2] = (bc * bMP) * (lap - g_m);
    out[3] = (ac * bEM) * ex + mx_ * (bPM + bMM);
    out[4] = ac * (X.r2x * ((bEM - bEP) * g.i2dx) + X.r2z * ((bME - bPE) * g.i2dz)
                   - X.r1xsq * ((bEM + bEP) * g.idxx) - X.r1zsq * ((bME + bPE) * g.idzz))
           + bc * (g_p * (bMM - bPP) + g_m * (bMP - bPM) - lap * (bMM + bPP + bPM + bMP));
    out[5] = (ac * bEP) * fx + mx_ * (bMP + bPP);
    out[6] = (bc * bPM) * (lap + g_m);
    out[7] = (ac * bPE) * fz + mz_ * (bPM + bPP);
    out[8] = (bc * bPP) * (lap + g_p);
}

// ------------------------------------------------------------------------------------------------
// Jacobian-vector product of assemble_mz_kernel.  Interior row i is coef[s][i] = w_s K[i + off(s)] + T_s(b_i, X_i), so
//     dcoef[s][i] = w_s dK[i + off(s)] + T_s(db_i, X_i) + T_s(b_i, dX_i)
//     dK_n = -2 omd^2 binv_n / c_n^3 alpha_n dc_n - K_n binv_n drho_n,   db_i[k] = (dbinv_i + dbinv_{i+off(k)})/2,
//     dbinv_n = -binv_n^2 drho_n,   dX_i = dX/dc_i alpha_i dc_i .
// Boundary rows are identity rows: their tangent is zero.  One thread per row; dc, drho (either may be NULL) and alpha
// (NULL: 1) are read at the nine neighbours through the caches.  Algorithmic traffic: 9*16 B written per node, plus
// the model planes read once.
// ------------------------------------------------------------------------------------------------
__global__ void assemble_mz_jvp_kernel(const cplx* __restrict__ c, const cplx* __restrict__ Kp, const double* __restrict__ binv,
                                       const double* __restrict__ dc, const double* __restrict__ drho,
                                       const cplx* __restrict__ alpha, AsmParams p, cplx* __restrict__ dcoef) {
    const i64 N = (i64)p.nx * p.nz;
    const i64 n = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int nx = p.nx, nz = p.nz;
    const int iz = (int)(n / nx), ix = (int)(n % nx);
    cplx out[9];
#pragma unroll
    for (int s = 0; s < 9; ++s) out[s] = mk(0.0);
    if (ix > 0 && ix < nx - 1 && iz > 0 && iz < nz - 1) {
        const MzGridConst g = mz_grid_const(p);
        const double wK[9] = {0.000001297, 0.09381, 0.000001297, 0.09381, 0.6248, 0.09381, 0.000001297, 0.09381, 0.000001297};
        const double bn = binv[n];
        const double dbn = drho ? -bn * bn * drho[n] : 0.0;
        double b[9], db[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) {
            const i64 j = n + (i64)(k / 3 - 1) * nx + (k % 3 - 1);
            const double bj = binv[j];
            b[k] = (bn + bj) * 0.5;
            cplx dK = mk(0.0);
            if (dc) {
                // K = (omd^2/c^2 - aky^2) binv  =>  dK/dc = -2 omd^2 binv / c^3   (as assemble_mz_vjp_kernel)
                const cplx cj = c[j];
                const cplx dKdc = (p.omd * p.omd) * crecip_fast(cj * cj * cj) * (-2.0 * bj);
                dK = alpha ? dKdc * (alpha[j] * dc[j]) : dKdc * dc[j];
            }
            db[k] = 0.0;
            if (drho) {
                // dK/drho = -K binv ;  dbinv/drho = -binv^2
                dK = dK + Kp[j] * (-bj * drho[j]);
                db[k] = (dbn - bj * bj * drho[j]) * 0.5;
            }
            out[k] = wK[k] * dK;
        }
        MzPml X, dX;
        mz_pml_terms(p, g, ix, iz, c[n], X, dX);
        cplx T[9];
        if (drho) {
            mz_t(db, X, g, T);
#pragma unroll
            for (int s = 0; s < 9; ++s) out[s] = out[s] + T[s];
        }
        if (dc) {
            const cplx dcn = alpha ? alpha[n] * dc[n] : mk(dc[n]);
            dX.r1xsq = dX.r1xsq * dcn; dX.r1zsq = dX.r1zsq * dcn; dX.r2x = dX.r2x * dcn; dX.r2z = dX.r2z * dcn;
            mz_t(b, dX, g, T);
#pragma unroll
            for (int s = 0; s < 9; ++s) out[s] = out[s] + T[s];
        }
    }
#pragma unroll
    for (int s = 0; s < 9; ++s) dcoef[(i64)s * N + n] = out[s];
}

// ------------------------------------------------------------------------------------------------
// out[i*S + s] = scale * sum_slot dcoef[slot*N + i] * conj(u[(i + off(slot))*S + s]),  zero on boundary rows.
// u is the conjugated forward panel (what the forward solve returns), so w = conj(u) on load.  There is no reduction
// over sources, so threads run along s: every neighbour load and the store are coalesced, and the nine coefficients of
// a row are one broadcast load per warp.  blockDim.x (a multiple of 32) covers sources, blockDim.y rows; a CTA takes
// STENCIL_APPLY_RUN * blockDim.y consecutive rows (a short run of x at one z), so the three u rows it reads come
// through L1 and the rows of the adjacent depths, read by the CTAs of the previous and next grid row, through L2.
// Algorithmic traffic: one panel read, one written, 9*N*16 B of dcoef; measured at C4 (S = 256, B200 at 1000 W): 2.75 ms
// = 2.27 TB/s of that traffic, 30% of HBM peak (DESIGN.md §4, §8).
// ------------------------------------------------------------------------------------------------
#define STENCIL_APPLY_RUN 4

__global__ void stencil_apply_kernel(const cplx* __restrict__ dcoef, const cplx* __restrict__ u, int nx, int nz, i64 S,
                                     cplx scale, cplx* __restrict__ out) {
    const i64 N = (i64)nx * nz;
    const i64 rows = (i64)STENCIL_APPLY_RUN * blockDim.y;
    for (i64 i0 = (i64)blockIdx.x * rows; i0 < N; i0 += (i64)gridDim.x * rows) {
#pragma unroll
        for (int r = 0; r < STENCIL_APPLY_RUN; ++r) {
            const i64 i = i0 + (i64)r * blockDim.y + threadIdx.y;
            if (i >= N) break;
            const int iz = (int)(i / nx), ix = (int)(i % nx);
            cplx* o = out + i * S;
            if (ix > 0 && ix < nx - 1 && iz > 0 && iz < nz - 1) {
                cplx cf[9];
#pragma unroll
                for (int k = 0; k < 9; ++k) cf[k] = dcoef[(i64)k * N + i] * scale;
                for (i64 s = threadIdx.x; s < S; s += blockDim.x) {
                    cplx acc = mk(0.0);
#pragma unroll
                    for (int k = 0; k < 9; ++k) {
                        const i64 j = i + (i64)(k / 3 - 1) * nx + (k % 3 - 1);
                        cfma(acc, cf[k], cconj(u[j * S + s]));
                    }
                    o[s] = acc;
                }
            } else {
                for (i64 s = threadIdx.x; s < S; s += blockDim.x) o[s] = mk(0.0);
            }
        }
    }
}
