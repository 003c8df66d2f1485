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
#pragma once
#include "hz_platform.h"
#include "hz_assemble.cuh"
#include "hz_adjoint.cuh"
#include "hz_born.cuh"

#define LAGCORR_RUN 16      // consecutive x of one depth per CTA (the register window slides along them)
#define LAGCORR_SPL 2       // sources per lane in one pass: partial sums over them are added before the warp reduction

__device__ __forceinline__ int lag_index(int dz, int dx) { return dz == 0 ? dx : 3 + 5 * (dz - 1) + (dx + 2); }

__device__ __forceinline__ cplx lag_load(const cplx* __restrict__ u, int nx, int nz, i64 S, int z, int x, i64 s, bool ok) {
    return (ok && x >= 0 && x < nx && z < nz) ? u[((i64)z * nx + x) * S + s] : mk(0.0);
}

// ------------------------------------------------------------------------------------------------
// C[l*N + p] = sum_s conj(u[p*S + s]) u[(p + delta_l)*S + s], zero where p + delta_l lies outside the grid.
// A CTA takes LAGCORR_RUN consecutive x at one depth z; threads run along the sources (blockDim.x, a multiple of 32),
// so every load is coalesced.  Each lane walks x with a register window of the rows z (x..x+2), z+1 and z+2
// (x-2..x+2): three loads per node and source, and the three rows it reads are re-read by the CTAs of the two depths
// above through L2.  Per node a lane forms the 13 lag products (26 doubles) of its LAGCORR_SPL sources, and one
// transpose-reduction over the warp (31 shuffles, 16+8+4+2+1) leaves lane l with the warp's sum of value l; the
// warps of the CTA are summed through shared memory.  Two CTAs of 256 threads fit an SM.  Algorithmic traffic: one
// panel read, 13*N*16 B written; measured at C4 (S = 256, B200 at 1000 W): 2.60 ms = 1.24 TB/s and 7.4 TFLOP/s, bound by
// issue (FP64 vector pipe and shuffles), not by HBM: an L2-resident panel is no faster per (node, source) (DESIGN.md §4, §8).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 2) wavefield_lagcorr_kernel(const cplx* __restrict__ u, int nx, int nz, i64 S, cplx* __restrict__ C) {
    HZ_SMEM(smem);
    double* red = reinterpret_cast<double*>(smem);      // [warps][LAGCORR_RUN][32]
    const i64 N = (i64)nx * nz;
    const int runs = (nx + LAGCORR_RUN - 1) / LAGCORR_RUN;
    const int z = (int)(blockIdx.x / runs), x0 = (int)(blockIdx.x % runs) * LAGCORR_RUN;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    double* mine = red + (i64)warp * LAGCORR_RUN * 32 + lane;   // this lane's running sums, one per node of the run
    for (int r = 0; r < LAGCORR_RUN; ++r) mine[r * 32] = 0.0;
    for (i64 s0 = 0; s0 < S; s0 += (i64)blockDim.x * LAGCORR_SPL) {
        // window per source: w0[0..2] = row z at x..x+2, w1[0..4] / w2[0..4] = rows z+1 / z+2 at x-2..x+2
        cplx w0[LAGCORR_SPL][3], w1[LAGCORR_SPL][5], w2[LAGCORR_SPL][5];
        i64 src[LAGCORR_SPL];
        bool ok[LAGCORR_SPL];
#pragma unroll
        for (int j = 0; j < LAGCORR_SPL; ++j) {
            src[j] = s0 + (i64)j * blockDim.x + threadIdx.x;
            ok[j] = src[j] < S;
            w0[j][1] = lag_load(u, nx, nz, S, z, x0, src[j], ok[j]);
            w0[j][2] = lag_load(u, nx, nz, S, z, x0 + 1, src[j], ok[j]);
#pragma unroll
            for (int q = 1; q < 5; ++q) {
                w1[j][q] = lag_load(u, nx, nz, S, z + 1, x0 + q - 3, src[j], ok[j]);
                w2[j][q] = lag_load(u, nx, nz, S, z + 2, x0 + q - 3, src[j], ok[j]);
            }
        }
#pragma unroll 1
        for (int r = 0; r < LAGCORR_RUN; ++r) {
            const int x = x0 + r;
            double v[32];
#pragma unroll
            for (int t = 0; t < 32; ++t) v[t] = 0.0;
#pragma unroll
            for (int j = 0; j < LAGCORR_SPL; ++j) {
                w0[j][0] = w0[j][1]; w0[j][1] = w0[j][2];
                w0[j][2] = lag_load(u, nx, nz, S, z, x + 2, src[j], ok[j]);
#pragma unroll
                for (int q = 0; q < 4; ++q) { w1[j][q] = w1[j][q + 1]; w2[j][q] = w2[j][q + 1]; }
                w1[j][4] = lag_load(u, nx, nz, S, z + 1, x + 2, src[j], ok[j]);
                w2[j][4] = lag_load(u, nx, nz, S, z + 2, x + 2, src[j], ok[j]);
                const cplx a = cconj(w0[j][0]);
                cplx prod[13];
                prod[0] = a * w0[j][0]; prod[1] = a * w0[j][1]; prod[2] = a * w0[j][2];
#pragma unroll
                for (int q = 0; q < 5; ++q) { prod[3 + q] = a * w1[j][q]; prod[8 + q] = a * w2[j][q]; }
#pragma unroll
                for (int l = 0; l < 13; ++l) { v[2 * l] += prod[l].re; v[2 * l + 1] += prod[l].im; }
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
            mine[r * 32] += v[0];                             // lane l: value l of node x (l < 26)
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 26 * LAGCORR_RUN; t += blockDim.x) {
        const int l = t / LAGCORR_RUN, r = t % LAGCORR_RUN, x = x0 + r;
        if (x >= nx) continue;
        double sum = 0.0;
        for (int w = 0; w < warps; ++w) sum += red[((i64)w * LAGCORR_RUN + r) * 32 + l];
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
// One thread per node n: p_c[n] += P_c[n], p_rho[n] += P_rho[n] (either may be NULL).  Row i = n - off(k) reads node n
// through slot k (the JVP of assemble_mz_jvp_kernel along e_n, column by column):
//   c:   slot k: w_k dK_n/dc_n;  row n also T(b_n, dX_n/dc_n)                                     (times alpha_n)
//   rho: slot k: w_k dK_n/drho_n;  T(db_i, X_i) with db_i[k] = dbinv_n/2 (row n: db_n[k'] = dbinv_n/2 for all k')
// Without rho (Gardner's rule) the c column is alpha_n d^c + drho_dc[n] d^rho, combined before the contraction.
// Boundary rows are identity rows and contribute nothing.
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
    const double bn = binv[n];
    const cplx cn = c[n];
    const cplx an = alpha ? alpha[n] : mk(1.0);
    const bool gardner = p_c && drho_dc;
    const double gn = gardner ? drho_dc[n] : 0.0;
    const bool need_rho = p_rho || gardner;
    // K = (omd^2/c^2 - aky^2) binv  =>  dK/dc = -2 omd^2 binv / c^3 ;  dK/drho = -K binv ;  dbinv/drho = -binv^2
    const cplx dKdc = (p.omd * p.omd) * crecip_fast(cn * cn * cn) * (-2.0 * bn);
    const cplx dKdr = Kp[n] * (-bn);
    const double hdb = -0.5 * bn * bn;
    double sc = 0.0, sr = 0.0;
#pragma unroll 1
    for (int k = 0; k < 9; ++k) {
        const int rz = iz - (k / 3 - 1), rx = ix - (k % 3 - 1);
        if (rz < 1 || rz > nz - 2 || rx < 1 || rx > nx - 2) continue;
        const i64 i = (i64)rz * nx + rx;
        // the mass weight of slot k (assemble_mz_kernel's wK); slot entries are set by compare-and-select over the unrolled
        // t so that the nine-entry arrays stay in registers (k is a runtime loop index)
        const double wk = k == 4 ? 0.6248 : (k & 1) ? 0.09381 : 0.000001297;
        MzPml X, dX;
        mz_pml_terms(p, g, rx, rz, c[i], X, dX);
        cplx dr[9], dcv[9];
        if (need_rho) {
            double db[9];
#pragma unroll
            for (int t = 0; t < 9; ++t) db[t] = (k == 4 || t == k) ? hdb : 0.0;
            mz_t(db, X, g, dr);
#pragma unroll
            for (int t = 0; t < 9; ++t)
                if (t == k) dr[t] = dr[t] + wk * dKdr;
        }
        if (p_c) {
#pragma unroll
            for (int t = 0; t < 9; ++t) dcv[t] = mk(0.0);
            if (k == 4) {
                double b[9];
#pragma unroll
                for (int t = 0; t < 9; ++t) b[t] = (bn + binv[n + (i64)(t / 3 - 1) * nx + (t % 3 - 1)]) * 0.5;
                mz_t(b, dX, g, dcv);
            }
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                if (t == k) dcv[t] = dcv[t] + wk * dKdc;
                dcv[t] = gardner ? an * dcv[t] + gn * dr[t] : an * dcv[t];
            }
            sc += lag_quad(C, N, nx, i, dcv);
        }
        if (p_rho) sr += lag_quad(C, N, nx, i, dr);
    }
    if (p_c) p_c[n] += sc;
    if (p_rho) p_rho[n] += sr;
}
