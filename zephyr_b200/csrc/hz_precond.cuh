// Pseudo-Hessian diagonal of the MiniZephyr operator (Shin, Jang & Min 2001; DESIGN.md §2, "Pseudo-Hessian").
//
// Per frequency, with w_s = A^-1 p_s (the forward field before its conjugation) and m one of c, rho:
//     P_m[n] = sum_s || (dA/dm_n) w_s ||^2 = sum_{i in rows(n)} sum_{a,b} d_{n,i,a} conj(d_{n,i,b}) C(i + off(a), off(b) - off(a))
// where d_{n,i,.} are the nine derivatives of row i's coefficients and C is the lag correlation of the source wavefield
//     C(p, delta) = sum_s w_s[p] conj(w_s[p + delta]) = sum_s conj(u_s[p]) u_s[p + delta],   delta in {-2..2}^2.
// C(p, -delta) = conj(C(p - delta, delta)), so 13 planes hold it: the zero lag and the half-plane
//     lag 0: (0,0);  1..2: (0, 1..2);  3..7: (1, -2..2);  8..12: (2, -2..2)      (delta = (dz, dx))
// which are exactly the lags off(b) - off(a) of the slot pairs a < b.  C does not depend on the model derivative, so
// one pass over the panel serves c, rho and the Gardner combination, and the contraction has no S in its cost:
//   1. wavefield_lagcorr_kernel:  u (N x S) -> C (13 complex planes of N)
//   2. pseudo_hessian_mz_kernel:  C -> p_c[n], p_rho[n] (+=)
// The exact Gauss-Newton diagonal (DESIGN.md §2, "Gauss-Newton diagonal") adds the receiver side: the same lag kernel at
// radius 4 on the forward panel (41 planes), at radius 2 on the receiver Green's functions, and
//   3. gauss_newton_diag_mz_kernel:  C41, Gam13 -> h_c[n], h_rho[n] (+=)
// which forms the rows' derivatives with the helper of pseudo_hessian_mz_kernel.
#pragma once
#include "hz_platform.h"
#include "hz_assemble.cuh"
#include "hz_adjoint.cuh"
#include "hz_born.cuh"

// One template serves every lag radius R: the lags delta = (dz, dx) of the Hermitian half-plane of {-R..R}^2 in the order
//     (0,0), (0, 1..R), (1, -R..R), ..., (R, -R..R)          -> LagShape<R>::lags = 1 + R + R (2R + 1) planes
// R = 2: the 13 planes of the pseudo-Hessian (and of the receiver Green's functions of the Gauss-Newton diagonal);
// R = 4: the 41 planes of the Gauss-Newton diagonal's source side (its row pairs reach lags in {-4..4}^2).
template <int R>
struct LagShape {
    static constexpr int lags = 1 + R + R * (2 * R + 1);
    static constexpr int vals = 2 * lags;                   // doubles per node
    static constexpr int chunks = (vals + 31) / 32;         // warp transpose-reductions per node
};

// instances: <R, consecutive x per CTA (the register window slides along them), sources per lane in one pass (partial
// sums over them are added before the warp reduction), threads per CTA at most, CTAs per SM>
#define LAGCORR_RUN 16
#define LAGCORR_SPL 2
#define LAGCORR2_ARGS 2, LAGCORR_RUN, LAGCORR_SPL, 256, 2
#define LAGCORR4_RUN 16
#define LAGCORR4_SPL 1
#define LAGCORR4_THREADS 128
#define LAGCORR4_ARGS 4, LAGCORR4_RUN, LAGCORR4_SPL, LAGCORR4_THREADS, 3

template <int R>
__host__ __device__ __forceinline__ int lag_slot(int dz, int dx) { return dz == 0 ? dx : R + 1 + (2 * R + 1) * (dz - 1) + (dx + R); }
__device__ __forceinline__ int lag_index(int dz, int dx) { return lag_slot<2>(dz, dx); }

__device__ __forceinline__ cplx lag_load(const cplx* __restrict__ u, int nx, int nz, i64 S, int z, int x, i64 s, bool ok) {
    return (ok && x >= 0 && x < nx && z < nz) ? u[((i64)z * nx + x) * S + s] : mk(0.0);
}

// ------------------------------------------------------------------------------------------------
// C[l*N + p] = sum_s conj(u[p*S + s]) u[(p + delta_l)*S + s], zero where p + delta_l lies outside the grid.
// A CTA takes RUN consecutive x at one depth z; threads run along the sources (blockDim.x, a multiple of 32), so every
// load is coalesced.  Each lane walks x with a register window of the rows z (x..x+R) and z+1..z+R (x-R..x+R): R+1
// loads per node and source, and the rows it reads are re-read by the CTAs of the R depths above through L2.  Per
// node a lane forms the lag products of its SPL sources, 32 doubles (16 lags) at a time, and one transpose-reduction
// over the warp per 32 doubles (31 shuffles, 16+8+4+2+1) leaves lane l with the warp's sum of value l; the warps of the
// CTA are summed through shared memory.
//   R = 2 (wavefield_lagcorr_kernel<LAGCORR2_ARGS>, hz_wavefield_lagcorr): 13 lags in one reduction, 2 sources per lane,
//     two CTAs of 256 threads per SM.  Algorithmic traffic: one panel read, 13*N*16 B written; measured at C4 (S = 256,
//     B200 at 1000 W): 2.60 ms = 1.24 TB/s and 7.4 TFLOP/s, bound by issue (FP64 vector pipe and shuffles), not by
//     HBM: an L2-resident panel is no faster per (node, source) (DESIGN.md §4, §8).
//   R = 4 (wavefield_lagcorr_kernel<LAGCORR4_ARGS>, hz_wavefield_lagcorr4): 41 lags in three reductions, 1 source per
//     lane (the window alone is 41 complex registers), CTAs of 128 threads.  One panel read, 41*N*16 B written.
// ------------------------------------------------------------------------------------------------
template <int R, int RUN, int SPL, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) wavefield_lagcorr_kernel(const cplx* __restrict__ u, int nx, int nz, i64 S, cplx* __restrict__ C) {
    constexpr int W = 2 * R + 1, NL = LagShape<R>::lags, NV = LagShape<R>::vals, NCH = LagShape<R>::chunks;
    HZ_SMEM(smem);
    double* red = reinterpret_cast<double*>(smem);      // [warps][RUN][NCH][32]
    const i64 N = (i64)nx * nz;
    const int runs = (nx + RUN - 1) / RUN;
    const int z = (int)(blockIdx.x / runs), x0 = (int)(blockIdx.x % runs) * RUN;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    double* mine = red + (i64)warp * RUN * NCH * 32 + lane;   // this lane's running sums, NCH per node of the run
    for (int r = 0; r < RUN * NCH; ++r) mine[r * 32] = 0.0;
    for (i64 s0 = 0; s0 < S; s0 += (i64)blockDim.x * SPL) {
        // window per source: w0[0..R] = row z at x..x+R, wd[d][0..2R] = row z+1+d at x-R..x+R
        cplx w0[SPL][R + 1], wd[SPL][R][W];
        i64 src[SPL];
        bool ok[SPL];
#pragma unroll
        for (int j = 0; j < SPL; ++j) {
            src[j] = s0 + (i64)j * blockDim.x + threadIdx.x;
            ok[j] = src[j] < S;
#pragma unroll
            for (int q = 1; q <= R; ++q) w0[j][q] = lag_load(u, nx, nz, S, z, x0 + q - 1, src[j], ok[j]);
#pragma unroll
            for (int q = 1; q < W; ++q)
#pragma unroll
                for (int d = 0; d < R; ++d) wd[j][d][q] = lag_load(u, nx, nz, S, z + 1 + d, x0 + q - 1 - R, src[j], ok[j]);
        }
#pragma unroll 1
        for (int r = 0; r < RUN; ++r) {
            const int x = x0 + r;
#pragma unroll
            for (int j = 0; j < SPL; ++j) {
#pragma unroll
                for (int q = 0; q < R; ++q) w0[j][q] = w0[j][q + 1];
                w0[j][R] = lag_load(u, nx, nz, S, z, x + R, src[j], ok[j]);
#pragma unroll
                for (int d = 0; d < R; ++d) {
#pragma unroll
                    for (int q = 0; q < W - 1; ++q) wd[j][d][q] = wd[j][d][q + 1];
                    wd[j][d][W - 1] = lag_load(u, nx, nz, S, z + 1 + d, x + R, src[j], ok[j]);
                }
            }
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                double v[32];
#pragma unroll
                for (int t = 0; t < 32; ++t) v[t] = 0.0;
#pragma unroll
                for (int j = 0; j < SPL; ++j) {
                    // the products of all lags (those outside this chunk are dead code); each is formed from the window
                    // entry itself, not through a select, which keeps the FMA contraction of the radius-2 instance
                    const cplx a = cconj(w0[j][0]);
                    cplx prod[NL];
#pragma unroll
                    for (int q = 0; q <= R; ++q) prod[q] = a * w0[j][q];
#pragma unroll
                    for (int q = 0; q < W; ++q)
#pragma unroll
                        for (int d = 0; d < R; ++d) prod[R + 1 + W * d + q] = a * wd[j][d][q];
#pragma unroll
                    for (int t = 0; t < 16; ++t) {
                        const int l = 16 * ch + t;
                        if (l < NL) { v[2 * t] += prod[l].re; v[2 * t + 1] += prod[l].im; }
                    }
                }
                // transpose-reduction: after the level of offset o, lane keeps the half of its values selected by (lane & o)
#pragma unroll
                for (int o = 16, h = 16; o > 0; o >>= 1, h >>= 1) {
                    const bool up = lane & o;
#pragma unroll
                    for (int t = 0; t < h; ++t) {
                        const double send = up ? v[t] : v[t + h];
                        const double keep = up ? v[t + h] : v[t];
                        v[t] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                    }
                }
                mine[(r * NCH + ch) * 32] += v[0];              // lane l: value 32 ch + l of node x
            }
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < NV * RUN; t += blockDim.x) {
        const int l = t / RUN, r = t % RUN, x = x0 + r;
        if (x >= nx) continue;
        double sum = 0.0;
        for (int w = 0; w < warps; ++w) sum += red[(((i64)w * RUN + r) * NCH + (l >> 5)) * 32 + (l & 31)];
        reinterpret_cast<double*>(C + (i64)(l >> 1) * N + (i64)z * nx + x)[l & 1] = sum;
    }
}

// ------------------------------------------------------------------------------------------------
// sum_{a,b} d_a conj(d_b) C(i + off(a), off(b) - off(a)) for interior row i: the diagonal a = b from the zero lag, each
// pair a < b and its conjugate twin as 2 Re of the stored half-plane lag.  Both loops are unrolled with explicit counts:
// otherwise d[] is indexed at run time and goes to local memory.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double lag_quad(const cplx* __restrict__ C, i64 N, int nx, i64 i, const cplx d[9]) {
    double out = 0.0;
#pragma unroll 9
    for (int a = 0; a < 9; ++a) {
        const i64 pa = i + (i64)(a / 3 - 1) * nx + (a % 3 - 1);
        out += (d[a].re * d[a].re + d[a].im * d[a].im) * C[pa].re;
        cplx cross = mk(0.0);
#pragma unroll 8
        for (int b = a + 1; b < 9; ++b) cfma(cross, cconj(d[b]), C[(i64)lag_index(b / 3 - a / 3, b % 3 - a % 3) * N + pa]);
        out += 2.0 * (d[a] * cross).re;
    }
    return out;
}

// ------------------------------------------------------------------------------------------------
// Column n of dA/dm (the JVP of assemble_mz_jvp_kernel along e_n): row i = n - off(k) reads node n through slot k.
//   c:   slot k: w_k dK_n/dc_n;  row n also T(b_n, dX_n/dc_n)                                     (times alpha_n)
//   rho: slot k: w_k dK_n/drho_n;  T(db_i, X_i) with db_i[k] = dbinv_n/2 (row n: db_n[k'] = dbinv_n/2 for all k')
// Without rho (Gardner's rule) the c column is alpha_n d^c + drho_dc[n] d^rho, combined before any contraction.
// Boundary rows are identity rows: their derivative is zero and callers skip them.  mz_node_deriv holds what does not
// depend on the row; mz_row_deriv forms row i's nine derivatives: dr (rho) if need_rho, dcv (the c column) if want_c.
// The pseudo-Hessian and the Gauss-Newton diagonal both call it.
// ------------------------------------------------------------------------------------------------
struct MzNodeDeriv {
    double bn, gn, hdb;
    cplx an, dKdc, dKdr;
};

__device__ __forceinline__ MzNodeDeriv mz_node_deriv(const cplx* __restrict__ c, const cplx* __restrict__ Kp, const double* __restrict__ binv,
                                                     const cplx* __restrict__ alpha, const double* __restrict__ drho_dc,
                                                     const AsmParams& p, i64 n, bool gardner) {
    MzNodeDeriv nd;
    nd.bn = binv[n];
    const cplx cn = c[n];
    nd.an = alpha ? alpha[n] : mk(1.0);
    nd.gn = gardner ? drho_dc[n] : 0.0;
    // K = (omd^2/c^2 - aky^2) binv  =>  dK/dc = -2 omd^2 binv / c^3 ;  dK/drho = -K binv ;  dbinv/drho = -binv^2
    nd.dKdc = (p.omd * p.omd) * crecip_fast(cn * cn * cn) * (-2.0 * nd.bn);
    nd.dKdr = Kp[n] * (-nd.bn);
    nd.hdb = -0.5 * nd.bn * nd.bn;
    return nd;
}

// the mass weight of slot k (assemble_mz_kernel's wK)
__device__ __forceinline__ double mz_mass_weight(int k) { return k == 4 ? 0.6248 : (k & 1) ? 0.09381 : 0.000001297; }

__device__ __forceinline__ void mz_row_deriv(const cplx* __restrict__ c, const double* __restrict__ binv, const AsmParams& p,
                                             const MzGridConst& g, const MzNodeDeriv& nd, i64 n, int k, int rx, int rz,
                                             bool need_rho, bool want_c, bool gardner, cplx dr[9], cplx dcv[9]) {
    const int nx = p.nx;
    const i64 i = (i64)rz * nx + rx;
    // slot entries are set by compare-and-select over the unrolled t so that the nine-entry arrays stay in registers
    // (k is a runtime loop index)
    const double wk = mz_mass_weight(k);
    MzPml X, dX;
    mz_pml_terms(p, g, rx, rz, c[i], X, dX);
    if (need_rho) {
        double db[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) db[t] = (k == 4 || t == k) ? nd.hdb : 0.0;
        mz_t(db, X, g, dr);
#pragma unroll
        for (int t = 0; t < 9; ++t)
            if (t == k) dr[t] = dr[t] + wk * nd.dKdr;
    }
    if (want_c) {
#pragma unroll
        for (int t = 0; t < 9; ++t) dcv[t] = mk(0.0);
        if (k == 4) {
            double b[9];
#pragma unroll
            for (int t = 0; t < 9; ++t) b[t] = (nd.bn + binv[n + (i64)(t / 3 - 1) * nx + (t % 3 - 1)]) * 0.5;
            mz_t(b, dX, g, dcv);
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            if (t == k) dcv[t] = dcv[t] + wk * nd.dKdc;
            dcv[t] = gardner ? nd.an * dcv[t] + nd.gn * dr[t] : nd.an * dcv[t];
        }
    }
}

__device__ __forceinline__ bool mz_interior_row(int rz, int rx, int nx, int nz) { return rz >= 1 && rz <= nz - 2 && rx >= 1 && rx <= nx - 2; }

// ------------------------------------------------------------------------------------------------
// One thread per node n: p_c[n] += P_c[n], p_rho[n] += P_rho[n] (either may be NULL), with the column of
// mz_row_deriv contracted row by row against C by lag_quad.
// ------------------------------------------------------------------------------------------------
__global__ void pseudo_hessian_mz_kernel(const cplx* __restrict__ c, const cplx* __restrict__ Kp, const double* __restrict__ binv,
                                         const cplx* __restrict__ C, const cplx* __restrict__ alpha,
                                         const double* __restrict__ drho_dc, AsmParams p, double* __restrict__ p_c,
                                         double* __restrict__ p_rho) {
    const i64 N = (i64)p.nx * p.nz;
    const i64 n = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int nx = p.nx, nz = p.nz;
    const int iz = (int)(n / nx), ix = (int)(n % nx);
    const MzGridConst g = mz_grid_const(p);
    const bool gardner = p_c && drho_dc;
    const bool need_rho = p_rho || gardner;
    const MzNodeDeriv nd = mz_node_deriv(c, Kp, binv, alpha, drho_dc, p, n, gardner);
    double sc = 0.0, sr = 0.0;
#pragma unroll 1
    for (int k = 0; k < 9; ++k) {
        const int rz = iz - (k / 3 - 1), rx = ix - (k % 3 - 1);
        if (!mz_interior_row(rz, rx, nx, nz)) continue;
        const i64 i = (i64)rz * nx + rx;
        cplx dr[9], dcv[9];
        mz_row_deriv(c, binv, p, g, nd, n, k, rx, rz, need_rho, p_c != nullptr, gardner, dr, dcv);
        if (p_c) sc += lag_quad(C, N, nx, i, dcv);
        if (p_rho) sr += lag_quad(C, N, nx, i, dr);
    }
    if (p_c) p_c[n] += sc;
    if (p_rho) p_rho[n] += sr;
}

// ------------------------------------------------------------------------------------------------
// Gauss-Newton Hessian diagonal (Pratt, Shin & Hicks 1998; DESIGN.md §2, "Gauss-Newton diagonal").  With g_r = A^-T b_r
// the receiver Green's functions (b_r = conj(Rv[r, .])) and D_n = dA/dm_n the column above,
//     H_nn = sum_{i,i' in rows(n)} Gam(i,i') sum_{a,b} d_{i,a} conj(d_{i',b}) C(i + off(a), i' + off(b))
//     Gam(i,i') = sum_r g_r[i] conj(g_r[i']),     C(p,p') = sum_s w_s[p] conj(w_s[p']) = sum_s conj(u_s[p]) u_s[p'].
// Both are stored as lag planes of their first point: Gam in the 13 planes of lag radius 2 (i' - i in {-2..2}^2) and C
// in the 41 planes of radius 4 (p' - p in {-4..4}^2), the half-plane of each; the other half is the conjugate read at
// the partner point.  The unordered row pairs {i, i'} are summed once each as 2 Re(Gam q) (the diagonal pairs once).
// ------------------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ cplx lag_get(const cplx* __restrict__ P, i64 N, int nx, i64 p, int dz, int dx) {
    if (dz > 0 || (dz == 0 && dx >= 0)) return P[(i64)lag_slot<R>(dz, dx) * N + p];
    return cconj(P[(i64)lag_slot<R>(-dz, -dx) * N + p + (i64)dz * nx + dx]);
}

// q = sum_{a,b} d1[a] conj(d2[b]) C(i1 + off(a), i2 + off(b)) with i2 - i1 = (Dz, Dx).  A row whose derivative has one
// entry (the c column without Gardner's rule away from row n) passes only = its slot and the value in d[0].
__device__ __forceinline__ cplx gn_pair(const cplx* __restrict__ C, i64 N, int nx, i64 i1, int Dz, int Dx,
                                        const cplx d1[9], int only1, const cplx d2[9], int only2) {
    cplx q = mk(0.0);
    if (only1 >= 0 && only2 >= 0) {
        const i64 p = i1 + (i64)(only1 / 3 - 1) * nx + (only1 % 3 - 1);
        return d1[0] * cconj(d2[0]) * lag_get<4>(C, N, nx, p, Dz + only2 / 3 - only1 / 3, Dx + only2 % 3 - only1 % 3);
    }
    if (only1 >= 0) {
        const i64 p = i1 + (i64)(only1 / 3 - 1) * nx + (only1 % 3 - 1);
#pragma unroll
        for (int b = 0; b < 9; ++b) cfma(q, cconj(d2[b]), lag_get<4>(C, N, nx, p, Dz + b / 3 - only1 / 3, Dx + b % 3 - only1 % 3));
        return d1[0] * q;
    }
    if (only2 >= 0) {
#pragma unroll
        for (int a = 0; a < 9; ++a) {
            const i64 p = i1 + (i64)(a / 3 - 1) * nx + (a % 3 - 1);
            cfma(q, d1[a], lag_get<4>(C, N, nx, p, Dz + only2 / 3 - a / 3, Dx + only2 % 3 - a % 3));
        }
        return q * cconj(d2[0]);
    }
#pragma unroll 9
    for (int a = 0; a < 9; ++a) {
        const i64 p = i1 + (i64)(a / 3 - 1) * nx + (a % 3 - 1);
        cplx cross = mk(0.0);
#pragma unroll 9
        for (int b = 0; b < 9; ++b) cfma(cross, cconj(d2[b]), lag_get<4>(C, N, nx, p, Dz + b / 3 - a / 3, Dx + b % 3 - a % 3));
        cfma(q, d1[a], cross);
    }
    return q;
}

// row k of node n's column for one parameter: the nine derivatives, or (sparse) the one entry in d[0] and its slot
__device__ __forceinline__ int gn_row(const cplx* __restrict__ c, const double* __restrict__ binv, const AsmParams& p,
                                      const MzGridConst& g, const MzNodeDeriv& nd, i64 n, int k, int rx, int rz, bool want_c,
                                      bool gardner, cplx d[9]) {
    if (want_c && !gardner && k != 4) {
        d[0] = nd.an * (mz_mass_weight(k) * nd.dKdc);
        return k;
    }
    cplx other[9];
    if (want_c) mz_row_deriv(c, binv, p, g, nd, n, k, rx, rz, gardner, true, gardner, other, d);
    else mz_row_deriv(c, binv, p, g, nd, n, k, rx, rz, true, false, false, d, other);
    return -1;
}

// One thread per node n: h_c[n] += H_c[n], h_rho[n] += H_rho[n] (either may be NULL), without the data weight.  Per
// parameter, an outer loop over the interior rows i holds d_i, an inner loop over the rows i' >= i recomputes d_{i'}
// (45 row pairs at most); C and Gam are read through L1/L2.  The c column with rho given is sparse (row n full, each
// other row one entry), which gn_pair exploits: 81 + 72 + 36 complex products at most instead of 45 x 81.
__global__ void gauss_newton_diag_mz_kernel(const cplx* __restrict__ c, const cplx* __restrict__ Kp, const double* __restrict__ binv,
                                            const cplx* __restrict__ C, const cplx* __restrict__ Gam, const cplx* __restrict__ alpha,
                                            const double* __restrict__ drho_dc, AsmParams p, double* __restrict__ h_c,
                                            double* __restrict__ h_rho) {
    const i64 N = (i64)p.nx * p.nz;
    const i64 n = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const int nx = p.nx, nz = p.nz;
    const int iz = (int)(n / nx), ix = (int)(n % nx);
    const MzGridConst g = mz_grid_const(p);
    const bool gardner = h_c && drho_dc;
    const MzNodeDeriv nd = mz_node_deriv(c, Kp, binv, alpha, drho_dc, p, n, gardner);
#pragma unroll 1
    for (int m = 0; m < 2; ++m) {
        double* out = m == 0 ? h_c : h_rho;
        if (!out) continue;
        const bool want_c = m == 0;
        double h = 0.0;
#pragma unroll 1
        for (int k1 = 0; k1 < 9; ++k1) {
            const int rz1 = iz - (k1 / 3 - 1), rx1 = ix - (k1 % 3 - 1);
            if (!mz_interior_row(rz1, rx1, nx, nz)) continue;
            const i64 i1 = (i64)rz1 * nx + rx1;
            cplx d1[9];
            const int only1 = gn_row(c, binv, p, g, nd, n, k1, rx1, rz1, want_c, gardner, d1);
#pragma unroll 1
            for (int k2 = k1; k2 < 9; ++k2) {
                const int rz2 = iz - (k2 / 3 - 1), rx2 = ix - (k2 % 3 - 1);
                if (!mz_interior_row(rz2, rx2, nx, nz)) continue;
                cplx d2[9];
                const int only2 = gn_row(c, binv, p, g, nd, n, k2, rx2, rz2, want_c, gardner, d2);
                const int Dz = rz2 - rz1, Dx = rx2 - rx1;
                const cplx q = gn_pair(C, N, nx, i1, Dz, Dx, d1, only1, d2, only2);
                const cplx gam = lag_get<2>(Gam, N, nx, i1, Dz, Dx);
                h += (k1 == k2 ? 1.0 : 2.0) * (gam * q).re;
            }
        }
        out[n] += h;
    }
}
