// Substitution-side kernels: block coupling (tridiagonal L/U application to a panel), the
// stencil residual, finalisation (premul + conjugate), and small utilities.  The dense part of
// every sweep step, X_i <- S_i^{-1} Y, is zgemm_dmma_kernel.
//
// Panel layout (HBM): X is (nf*N) x S row-major complex128 in the reference's external ordering,
// row(f, iz, ix) = f*N + iz*nx + ix  (zephyr/backend/eurus.py:463 stacks the two fields), so the
// finished wavefield is already the (N, S) array `Disc * q` returns
// (zephyr/backend/discretization.py:101-106).
#pragma once
#include "hz_platform.h"
#include "hz_factor.cuh"
#include "hz_c64.cuh"

// Entry of op(A) (OP: 0 = N, 1 = T, 2 = H) in row (fr, node), column (fc, nbr = node + dz*nx + dx), slot = (dz+1)*3 + dx+1.
// The transposed stencil is a gather: A^T[r][c] = A[c][r] is stored at the neighbour node, in the mirrored slot (8 - slot)
// of the swapped field pair (fc, fr); H conjugates it.  Block-wise this makes (A^T)_{i,i-1} = U_{i-1}^T and
// (A^T)_{i,i+1} = L_{i+1}^T, so the sweeps below keep their structure for every op.
template <int OP>
__device__ __forceinline__ cplx op_coef(const cplx* __restrict__ coef, int nf, int fr, int fc, int slot, i64 node, i64 nbr, i64 N) {
    if constexpr (OP == 0) return coef_plane(coef, nf, fr, fc, slot, N)[node];
    const cplx v = coef_plane(coef, nf, fc, fr, 8 - slot, N)[nbr];
    return OP == 2 ? cconj(v) : v;
}

// Y[rl][s] = use_self * X_i[rl][s] + sgn_lo * (op(A)_{i,i-1} X_{i-1})[rl][s] + sgn_hi * (op(A)_{i,i+1} X_{i+1})[rl][s]
// rl = f*nx + ix indexes the block-local row; Y is a dense b x S buffer (ld = S).
template <class TP, int OP = 0>
__global__ void couple_kernel(const cplx* __restrict__ coef, int nf, int nx, int nz, int i,
                              const TP* __restrict__ X, i64 S, TP* __restrict__ Y,
                              int use_self, double sgn_lo, double sgn_hi) {
    const i64 s = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    const int rl = blockIdx.y;
    if (s >= S) return;
    const i64 N = (i64)nx * nz;
    const int fr = rl / nx, ix = rl % nx;
    const i64 node = (i64)i * nx + ix;
    cplx acc = mk(0.0);
    if (use_self) acc = ldp(&X[((i64)fr * N + node) * S + s]);
    for (int side = 0; side < 2; ++side) {
        const double sg = side == 0 ? sgn_lo : sgn_hi;
        if (sg == 0.0) continue;
        const int dzs = side == 0 ? -1 : 1;
        cplx part = mk(0.0);
        for (int fc = 0; fc < nf; ++fc) {
#pragma unroll
            for (int a = -1; a <= 1; ++a) {
                if (ix + a < 0 || ix + a >= nx) continue;
                const i64 nbr = (i64)(i + dzs) * nx + ix + a;
                const cplx cf = op_coef<OP>(coef, nf, fr, fc, (dzs + 1) * 3 + a + 1, node, nbr, N);
                cfma(part, cf, ldp(&X[((i64)fc * N + nbr) * S + s]));
            }
        }
        acc = acc + sg * part;
    }
    stp(&Y[(i64)rl * S + s], acc);
}

// R = Q - op(A) X over the whole panel (stencil SpMM); one thread per (row, s)
template <class TP, int OP = 0>
__global__ void residual_kernel(const cplx* __restrict__ coef, int nf, int nx, int nz,
                                const TP* __restrict__ X, const TP* __restrict__ Q, i64 S,
                                TP* __restrict__ R) {
    const i64 s = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const i64 N = (i64)nx * nz;
    const i64 row = (i64)blockIdx.y + (i64)blockIdx.z * 65535;
    if (row >= (i64)nf * N) return;
    const int fr = (int)(row / N);
    const i64 node = row % N;
    const int iz = (int)(node / nx), ix = (int)(node % nx);
    cplx acc = ldp(&Q[row * S + s]);
    for (int fc = 0; fc < nf; ++fc)
#pragma unroll
        for (int dzs = -1; dzs <= 1; ++dzs) {
            if (iz + dzs < 0 || iz + dzs >= nz) continue;
#pragma unroll
            for (int a = -1; a <= 1; ++a) {
                if (ix + a < 0 || ix + a >= nx) continue;
                const i64 nbr = node + (i64)dzs * nx + a;
                const cplx cf = op_coef<OP>(coef, nf, fr, fc, (dzs + 1) * 3 + a + 1, node, nbr, N);
                const cplx xv = ldp(&X[((i64)fc * N + nbr) * S + s]);
                acc = acc - cf * xv;
            }
        }
    stp(&R[row * S + s], acc);
}

// Accuracy probe (one column): out[row] = X[row*S + col] before the solve ...
template <class TP>
__global__ void gather_col_kernel(const TP* __restrict__ X, i64 S, i64 col, i64 rows, cplx* __restrict__ out) {
    for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (i64)gridDim.x * blockDim.x) out[r] = ldp(&X[r * S + col]);
}
// ... and afterwards out[0] += ||q - op(A) x||^2, out[1] += ||q||^2 for that column (9-point stencil residual in FP64)
template <class TP, int OP = 0>
__global__ void residual_col_kernel(const cplx* __restrict__ coef, int nf, int nx, int nz, const TP* __restrict__ X, i64 S, i64 col,
                                    const cplx* __restrict__ q, double* __restrict__ out) {
    const i64 N = (i64)nx * nz, rows = (i64)nf * N;
    double sr = 0.0, sq = 0.0;
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < rows; row += (i64)gridDim.x * blockDim.x) {
        const int fr = (int)(row / N);
        const i64 node = row % N;
        const int iz = (int)(node / nx), ix = (int)(node % nx);
        const cplx qv = q[row];
        cplx acc = qv;
        for (int fc = 0; fc < nf; ++fc)
#pragma unroll
            for (int dzs = -1; dzs <= 1; ++dzs) {
                if (iz + dzs < 0 || iz + dzs >= nz) continue;
#pragma unroll
                for (int a = -1; a <= 1; ++a) {
                    if (ix + a < 0 || ix + a >= nx) continue;
                    const i64 nbr = node + (i64)dzs * nx + a;
                    const cplx cf = op_coef<OP>(coef, nf, fr, fc, (dzs + 1) * 3 + a + 1, node, nbr, N);
                    acc = acc - cf * ldp(&X[((i64)fc * N + nbr) * S + col]);
                }
            }
        sr += cabs2(acc);
        sq += cabs2(qv);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sr += __shfl_xor_sync(0xffffffffu, sr, o);
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
    }
    if (hz_lane() == 0) {
        atomicAdd(out, sr);
        atomicAdd(out + 1, sq);
    }
}

// out[0] += sum |a|^2 ; out[1] += sum |b|^2   (diagnostic norms; block reduce + one atomic each)
template <class TP>
__global__ void norm2_kernel(const TP* __restrict__ a, const TP* __restrict__ b, i64 n, double* out) {
    double sa = 0.0, sb = 0.0;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        sa += cabs2(ldp(&a[i]));
        if (b) sb += cabs2(ldp(&b[i]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sa += __shfl_xor_sync(0xffffffffu, sa, o);
        sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
    if (hz_lane() == 0) {
        atomicAdd(out, sa);
        atomicAdd(out + 1, sb);
    }
}

// X += D
template <class TP>
__global__ void axpy_kernel(TP* __restrict__ X, const TP* __restrict__ D, i64 n) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x)
        stp(&X[i], ldp(&X[i]) + ldp(&D[i]));
}

// X <- conj(premul * X)    (zephyr/backend/discretization.py:103; premul folded in by linearity)
template <class TP>
__global__ void finalize_kernel(TP* __restrict__ X, i64 n, cplx pm, int do_conj) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        cplx v = pm * ldp(&X[i]);
        if (do_conj) v.im = -v.im;
        stp(&X[i], v);
    }
}

// X[row[j]*S + col[j]] += val[j] * scale   (sparse right-hand sides: Kaiser taps, residual sources)
__device__ __forceinline__ void atomic_add_c(cplx* dst, cplx v) { atomicAdd(&dst->re, v.re); atomicAdd(&dst->im, v.im); }
__device__ __forceinline__ void atomic_add_c(cplxf* dst, cplx v) { atomicAdd(&dst->re, (float)v.re); atomicAdd(&dst->im, (float)v.im); }

template <class TP>
__global__ void scatter_coo_kernel(TP* __restrict__ X, i64 S, i64 nnz, const i64* __restrict__ row,
                                   const i64* __restrict__ col, const cplx* __restrict__ val, cplx scale) {
    const i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    const cplx v = val[j] * scale;
    atomic_add_c(X + row[j] * S + col[j], v);
}
