// Adjoint-state FWI gradient of the MiniZephyr operator (DESIGN.md §2, "Adjoint-state gradient").
//
// Per frequency, with w = A^-1 p (the forward field before its conjugation), lambda = A^-T (Rv^H v) and
// phi = 0.5 sum |Wd (Rv conj(w) - dobs)|^2:
//     dphi/dm = -Re sum_s lambda_s^T (dA/dm) w_s .
// A depends on the model only through the nine coefficient planes of assemble_mz_kernel, so the contraction is
//   1. stencil_xcorr_kernel:   G[slot][i] = sum_s lambda_s[i] * w_s[i + off(slot)]    (9 complex planes of N)
//   2. assemble_mz_vjp_kernel: g_c[n]   -= Re(alpha_n sum_{slot,i} G[slot][i] dcoef[slot][i]/dc_n)
//                              g_rho[n] -= Re(        sum_{slot,i} G[slot][i] dcoef[slot][i]/drho_n)
// Boundary rows of A are constant, so their G is zero and the VJP skips them.
#pragma once
#include "hz_platform.h"
#include "hz_assemble.cuh"

// ------------------------------------------------------------------------------------------------
// G[slot*N + i] = sum_s lam[i*S + s] * conj(u[(i + off(slot))*S + s]),  off(slot) = (slot/3 - 1)*nx + (slot%3 - 1).
// u is the conjugated forward panel (what the forward solve returns), so w = conj(u) on load.  One warp per grid row
// i, lanes over the sources, warp-shuffle reduction (as gradient_kernel).  Consecutive warps of a block take
// consecutive x at fixed z, so the nine neighbour rows of u that adjacent warps read overlap, and the blocks of
// adjacent depths run at about the same time; how much of that reuse the caches actually deliver is not measured.
// Algorithmic traffic is 2*N*S*16 B read + 9*N*16 B written; measured at C4 (S = 256, B200): 4.74 ms = 1.32 TB/s of
// that traffic, 20% of HBM peak (DESIGN.md §4, §8).
// ------------------------------------------------------------------------------------------------
__global__ void stencil_xcorr_kernel(const cplx* __restrict__ lam, const cplx* __restrict__ u, int nx, int nz, i64 S,
                                     cplx* __restrict__ G) {
    const int lane = hz_lane();
    const i64 N = (i64)nx * nz;
    const i64 wpb = blockDim.x >> 5;
    for (i64 n = (i64)blockIdx.x * wpb + (threadIdx.x >> 5); n < N; n += (i64)gridDim.x * wpb) {
        const int iz = (int)(n / nx), ix = (int)(n % nx);
        cplx acc[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) acc[k] = mk(0.0);
        if (ix > 0 && ix < nx - 1 && iz > 0 && iz < nz - 1) {          // warp-uniform: one row per warp
            const cplx* l = lam + n * S;
            for (i64 s = lane; s < S; s += 32) {
                const cplx a = l[s];
#pragma unroll
                for (int k = 0; k < 9; ++k) {
                    const i64 j = n + (i64)(k / 3 - 1) * nx + (k % 3 - 1);
                    cfma(acc[k], a, cconj(u[j * S + s]));
                }
            }
#pragma unroll
            for (int k = 0; k < 9; ++k)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    acc[k].re += __shfl_xor_sync(0xffffffffu, acc[k].re, o);
                    acc[k].im += __shfl_xor_sync(0xffffffffu, acc[k].im, o);
                }
        }
#pragma unroll
        for (int k = 0; k < 9; ++k)
            if (lane == k) G[(i64)k * N + n] = acc[k];
    }
}

// ------------------------------------------------------------------------------------------------
// Vector-Jacobian product of assemble_mz_kernel.
//
// Row i of A (interior) is  coef[s][i] = w_s K[i + off(s)] + T_s(b_i, X_i)  with the mass weights w_s, the nine
// neighbour buoyancy averages b_i[k] = (binv[i] + binv[i + off(k)])/2 and the PML terms X_i = (r1xsq, r1zsq, r2x, r2z),
// functions of c[i] only.  T is linear in b and linear in X, so
//     sum_s G[s][i] T_s(b, X) = sum_{k != 4} b[k] H_k(G[.][i], X)
// with H below (the transpose of the stencil formula in assemble_mz_kernel, term by term).  Hence, for node n:
//   c:   K[n] is read by rows n - off(k) through slot k;  X_n by row n only:
//        dphi/dc_n = -Re alpha_n ( dK_n/dc_n sum_k w_k G[k][n - off(k)] + sum_k b_n[k] H_k(G[.][n], dX_n/dc_n) )
//   rho: K[n] as above, and binv[n] in b_n[k] (all k) and in b_i[k] of rows i = n - off(k), each with weight 1/2:
//        dphi/drho_n = -Re ( dK_n/drho_n sum_k w_k G[k][n - off(k)]
//                           + dbinv_n/drho_n / 2 ( sum_k H_k(G[.][n], X_n) + sum_k H_k(G[.][n - off(k)], X_{n - off(k)}) ) )
// Rows on the grid boundary are identity rows (constant) and contribute nothing.
// ------------------------------------------------------------------------------------------------
struct MzPml {
    cplx r1xsq, r1zsq, r2x, r2z;
};

struct MzGridConst {
    double i4dxz, i4dd, idx_, idz_, i2dx, i2dz, idxx, idzz, pmlfx, pmlfz;
    cplx iom;
};

__device__ __forceinline__ MzGridConst mz_grid_const(const AsmParams& p) {
    MzGridConst g;
    const double dx = p.dx, dz = p.dz;
    const double dxx = dx * dx, dzz = dz * dz, dxz = (dxx + dzz) / 2, dd = sqrt(dxz);
    g.i4dxz = 1.0 / (4 * dxz); g.i4dd = 1.0 / (4 * dd); g.idx_ = 1.0 / dx; g.idz_ = 1.0 / dz;
    g.i2dx = 1.0 / (2 * dx); g.i2dz = 1.0 / (2 * dz); g.idxx = 1.0 / dxx; g.idzz = 1.0 / dzz;
    const double pdx = dx * (double)(p.nPML - 1), pdz = dz * (double)(p.nPML - 1);
    const double lg = log(1.0 / 1e-3);
    g.pmlfx = 3.0 * lg / (2 * pdx * pdx * pdx);
    g.pmlfz = 3.0 * lg / (2 * pdz * pdz * pdz);
    g.iom = mk(-p.omd.im, p.omd.re);
    return g;
}

// one axis of the Roecker PML (as assemble_mz_kernel) and its derivative in c:
//   r1 = iom/den, den = pmlf c dp^2 + iom;  r2 = sn r1^2 (2 pmlf c dp)/den
//   dr1/dc = -r1 pmlf dp^2/den;  d(c/den)/dc = iom/den^2 = r1/den
__device__ __forceinline__ void mz_pml_axis(double pmlf, double dp, double sn, cplx iom, cplx c, cplx& r1sq, cplx& r2,
                                            cplx& dr1sq, cplx& dr2) {
    const cplx rden = crecip_fast((pmlf * c) * (dp * dp) + iom);
    const cplx r1 = iom * rden;
    r1sq = r1 * r1;
    const cplx cr = c * rden;
    const double k2 = sn * (2 * pmlf * dp);
    r2 = (r1sq * k2) * cr;
    const cplx dr1 = (r1 * rden) * (-(pmlf * dp * dp));
    dr1sq = (2.0 * r1) * dr1;
    dr2 = (dr1sq * cr + r1sq * (r1 * rden)) * k2;
}

__device__ __forceinline__ void mz_pml_terms(const AsmParams& p, const MzGridConst& g, int ix, int iz, cplx c, MzPml& X,
                                             MzPml& dX) {
    const int nx = p.nx, nz = p.nz, nP = p.nPML;
    double dpx = 0.0, dpz = 0.0, snx = 0.0, snz = 0.0;
    if (ix >= nx - nP) dpx = (double)(ix - (nx - nP) + 1) * p.dx; else if (ix < nP) dpx = (double)(nP - ix) * p.dx;
    if (iz >= nz - nP) dpz = (double)(iz - (nz - nP) + 1) * p.dz; else if (iz < nP) dpz = (double)(nP - iz) * p.dz;
    if (!p.fs[3] && ix < nP) snx = 1.0; else if (!p.fs[1] && ix >= nx - nP) snx = -1.0;
    if (!p.fs[0] && iz < nP) snz = 1.0; else if (!p.fs[2] && iz >= nz - nP) snz = -1.0;
    mz_pml_axis(g.pmlfx, dpx, snx, g.iom, c, X.r1xsq, X.r2x, dX.r1xsq, dX.r2x);
    mz_pml_axis(g.pmlfz, dpz, snz, g.iom, c, X.r1zsq, X.r2z, dX.r1zsq, dX.r2z);
}

// H_k(G[.][i], X) for k = 0..8 (H_4 = 0): the coefficient of b[k] in sum_s G[s][i] T_s(b, X).  Callers that use only
// some H_k let the compiler drop the G loads the others need.
__device__ __forceinline__ void mz_h(const cplx* __restrict__ G, i64 N, i64 i, const MzPml& X, const MzGridConst& g,
                                     cplx H[9]) {
    const double ac = 0.5461, bc = 0.4539;
    const cplx lap = (X.r1zsq + X.r1xsq) * g.i4dxz;
    const cplx g_p = (X.r2z + X.r2x) * g.i4dd, g_m = (X.r2z - X.r2x) * g.i4dd;
    const cplx ez = (X.r1zsq * g.idz_ - X.r2z * 0.5) * g.idz_, fz = (X.r1zsq * g.idz_ + X.r2z * 0.5) * g.idz_;
    const cplx ex = (X.r1xsq * g.idx_ - X.r2x * 0.5) * g.idx_, fx = (X.r1xsq * g.idx_ + X.r2x * 0.5) * g.idx_;
    const cplx mz_ = (bc * g.i4dxz) * (X.r1zsq - X.r1xsq), mx_ = -mz_;
    const cplx G0 = G[i], G1 = G[N + i], G2 = G[2 * N + i], G3 = G[3 * N + i], G4 = G[4 * N + i];
    const cplx G5 = G[5 * N + i], G6 = G[6 * N + i], G7 = G[7 * N + i], G8 = G[8 * N + i];
    H[0] = G0 * (bc * (lap - g_p)) + G1 * mz_ + G3 * mx_ + G4 * (bc * (g_p - lap));
    H[1] = G1 * (ac * ez) + G4 * (ac * (X.r2z * g.i2dz - X.r1zsq * g.idzz));
    H[2] = G1 * mz_ + G2 * (bc * (lap - g_m)) + G4 * (bc * (g_m - lap)) + G5 * mx_;
    H[3] = G3 * (ac * ex) + G4 * (ac * (X.r2x * g.i2dx - X.r1xsq * g.idxx));
    H[4] = mk(0.0);
    H[5] = G4 * (-ac * (X.r2x * g.i2dx + X.r1xsq * g.idxx)) + G5 * (ac * fx);
    H[6] = G3 * mx_ - G4 * (bc * (g_m + lap)) + G6 * (bc * (lap + g_m)) + G7 * mz_;
    H[7] = G4 * (-ac * (X.r2z * g.i2dz + X.r1zsq * g.idzz)) + G7 * (ac * fz);
    H[8] = G4 * (-bc * (g_p + lap)) + G5 * mx_ + G7 * mz_ + G8 * (bc * (lap + g_p));
}

// One thread per node n.  g_c / g_rho (either may be NULL) are accumulated (+=); alpha (NULL: 1) scales dc_f/dc.
__global__ void assemble_mz_vjp_kernel(const cplx* __restrict__ c, const cplx* __restrict__ Kp, const double* __restrict__ binv,
                                       const cplx* __restrict__ G, const cplx* __restrict__ alpha, AsmParams p,
                                       double* __restrict__ g_c, double* __restrict__ g_rho) {
    const i64 N = (i64)p.nx * p.nz;
    const i64 n = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int nx = p.nx, nz = p.nz;
    const int iz = (int)(n / nx), ix = (int)(n % nx);
    const MzGridConst g = mz_grid_const(p);
    const double wK[9] = {0.000001297, 0.09381, 0.000001297, 0.09381, 0.6248, 0.09381, 0.000001297, 0.09381, 0.000001297};

    cplx accK = mk(0.0);     // sum_k w_k G[k][n - off(k)]: every row that reads K[n]
    cplx accB = mk(0.0);     // sum of H_k over the rows whose b[k] holds binv[n]
    cplx accC = mk(0.0);     // sum_k b_n[k] H_k(G[.][n], dX_n)
    const double bn = binv[n];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        const int a = k / 3 - 1, q = k % 3 - 1;
        const int rz = iz - a, rx = ix - q;                 // row i = n - off(k) reads node n through slot k
        if (rz < 1 || rz > nz - 2 || rx < 1 || rx > nx - 2) continue;
        const i64 i = (i64)rz * nx + rx;
        accK = accK + wK[k] * G[(i64)k * N + i];
        MzPml X, dX;
        mz_pml_terms(p, g, rx, rz, c[i], X, dX);
        cplx H[9];
        mz_h(G, N, i, X, g, H);
        if (k != 4) {
            accB = accB + H[k];
        } else {                                            // row n itself: all its b[k] hold binv[n]; X_n holds c[n]
#pragma unroll
            for (int t = 0; t < 9; ++t) accB = accB + H[t];
            mz_h(G, N, i, dX, g, H);
#pragma unroll
            for (int t = 0; t < 9; ++t)
                if (t != 4) accC = accC + H[t] * ((bn + binv[n + (i64)(t / 3 - 1) * nx + (t % 3 - 1)]) * 0.5);
        }
    }
    if (g_c) {
        // K = (omd^2/c^2 - aky^2) binv  =>  dK/dc = -2 omd^2 binv / c^3
        const cplx cn = c[n];
        const cplx dKdc = (p.omd * p.omd) * crecip_fast(cn * cn * cn) * (-2.0 * bn);
        cplx t = accK * dKdc + accC;
        if (alpha) t = alpha[n] * t;
        g_c[n] -= t.re;
    }
    if (g_rho) {
        // dK/drho = -K binv ;  dbinv/drho = -binv^2
        const cplx t = accK * (Kp[n] * (-bn)) + accB * (-0.5 * bn * bn);
        g_rho[n] -= t.re;
    }
}
