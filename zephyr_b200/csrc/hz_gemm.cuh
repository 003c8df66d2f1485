// Complex128 GEMM on the FP64 tensor pipe (DMMA.8x8x4), the contraction behind both the block
// factorisation (Schur / Gauss-Jordan rank-nb updates) and the multi-RHS substitution sweeps.
//
//   C[crow(r)][c] = beta * Cin[r][c] + alpha * sum_k A[r][k] * B[k][c]
//
// A (M x K), B (K x N), C (M x N) are row-major interleaved complex128.  A complex MAC is four
// real DMMAs on (re, im) fragments: Cre += Are*Bre + (-Aim)*Bim ; Cim += Are*Bim + Aim*Bre.
//
// Design notes (B200): the DMMA pipe retires one 8x8x4 per 4 clk per SM (128 flop/clk/SM), so
// the kernel is tensor-pipe bound with a wide margin everywhere else: operands are staged
// global->shared with 16-byte LDGSTS in a multi-stage ring, one LDS.128 fetches a (re, im)
// fragment, and the shared layouts are padded so that every quarter-warp LDS.128 phase is
// bank-conflict free (A row stride == 4 mod 8 units of 16 B; B row stride == 2 mod 8).
// Tiles are deliberately small (<= 64x64) so that M x N = 1000 x 512 still fills 144 of 148 SMs.
//
// op(A) (template OPA, 0 = N, 1 = T, 2 = C = conjugate transpose): for T and C the stored A is K x M and the kernel
// computes with op(A)[r][k] = A[k][r] (conjugated for C) -- the transposed / adjoint substitution sweeps apply the
// stored block inverses S_i^{-1} as S_i^{-T} / S_i^{-H} without a transposed copy.  The A tile is then staged from
// rows k of the stored A: consecutive threads copy consecutive m of one row (coalesced LDGSTS), into a k-major shared
// layout sA[k][m] with row stride TM + 2 == 2 (mod 8), the layout of B, so the fragment loads A[g][t] stay conflict
// free (a quarter-warp phase reads units t*(TM+2) + g, eight distinct banks of 16 B).  C only flips the sign of the
// imaginary part of the A fragment where it already enters: the -Aim of the four-product form moves to the other
// term, and the three-product form sums ar - ai instead of ar + ai (epilogue: Re = t1 + t2, Im = s - t1 + t2).
#pragma once
#include "hz_platform.h"

struct GemmParams {
    const cplx* A; i64 lda;
    const cplx* B; i64 ldb;
    cplx* C; i64 ldc;
    int M, N, K;
    double alpha;
    int beta;                 // 0: overwrite, 1: accumulate onto Cin
    int sub_c0, sub_c1;       // Gauss-Jordan: for columns in [sub_c0, sub_c1) Cin is the identity
    int row_nx; i64 row_fs;   // C row map: crow(r) = (r / row_nx) * row_fs + r % row_nx  (row_nx = 0: identity)
};

constexpr int GEMM_KB = 32;           // k-depth of one shared-memory stage (one barrier per stage: 16 cost ~18% at K=1000)
constexpr int GEMM_LDA = GEMM_KB + 4; // 36 == 4 (mod 8)

template <int MI, int NI, int WM, int WN, int STAGES, int KS = 1>
struct GemmCfg {
    static constexpr int TM = 8 * MI * WM, TN = 8 * NI * WN, THREADS = 32 * WM * WN * KS;
    static constexpr int LDB = TN + 2;                                // == 2 (mod 8)
    static constexpr int A_ELEMS = TM * GEMM_LDA, B_ELEMS = GEMM_KB * LDB;
    static constexpr int SMEM = STAGES * (A_ELEMS + B_ELEMS) * (int)sizeof(cplx);
};

// KS > 1: intra-CTA split-K.  KS groups of WM x WN warps each take every KS-th k4 step of a stage and the
// partial accumulators are summed through shared memory before the epilogue: twice the warps per scheduler
// for the same tile and the same staging traffic (the 8-warp kernel stalls on fixed-latency DMMA
// dependencies with only two warps per scheduler, profiles/r1c_ncu_zgemm_solve.md).
// M3: three real DMMAs per complex MAC (Re = ar br - ai bi, Im = (ar + ai)(br + bi) - ar br - ai bi) instead of four; the
// operand sums cost one vector-FP64 add per fragment on a pipe this kernel does not otherwise use.  The kernel is bound
// by the tensor pipe, so a quarter fewer DMMAs is a quarter less time; normwise accuracy is that of the 4-product form.
template <int MI, int NI, int WM, int WN, int STAGES, int KS = 1, bool M3 = false, int OPA = 0>
__global__ void __launch_bounds__(32 * WM * WN * KS, 1) zgemm_dmma_kernel(GemmParams p) {
    typedef GemmCfg<MI, NI, WM, WN, STAGES, KS> Cfg;
    constexpr int TM = Cfg::TM, TN = Cfg::TN, NT = Cfg::THREADS, LDB = Cfg::LDB;
    constexpr bool AT = OPA != 0, ACONJ = OPA == 2;
    constexpr int LDAT = TM + 2;                                                  // k-major A tile (T, C): == 2 (mod 8)
    static_assert(OPA >= 0 && OPA <= 2, "op(A) is N, T or C");
    static_assert(!AT || GEMM_KB * LDAT <= Cfg::A_ELEMS, "the k-major A tile must fit the A stage");
    HZ_SMEM(smem_raw);
    cplx* sA = reinterpret_cast<cplx*>(smem_raw);
    cplx* sB = sA + STAGES * Cfg::A_ELEMS;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wk = warp / (WM * WN), w2 = warp % (WM * WN);
    const int wm = w2 / WN, wn = w2 % WN;
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
    const int KT = (p.K + GEMM_KB - 1) / GEMM_KB;

    // ---- operand staging.  One stage is NA + NBL 16-byte LDGSTS per thread.  Measured: issuing them
    // all right after the stage barrier idles the tensor pipe for ~13% of the loop (every warp does address
    // arithmetic at the same moment; the same loop without loads runs at 100% of the DMMA peak), so the
    // copies of the next stage are spread over the k4 steps of the current one, where they fill the issue
    // slot that follows each DMMA, and the addresses are strength-reduced to one base pointer per operand.
    static_assert(NT % GEMM_KB == 0 && NT % TN == 0, "staging assumes whole rows per thread stride");
    // A, op N: rows a_r0 + u*RA of the tile, fixed column a_kk.  A, op T/C: k rows a_r0 + u*RA of the stored A, fixed
    // column a_kk (an m of the tile); RA = NT / TM whole rows per pass, threads past RA * TM rows idle.
    constexpr int RA = AT ? NT / TM : NT / GEMM_KB, RB = NT / TN;   // row stride between a thread's consecutive copies
    constexpr int NA = AT ? (GEMM_KB + RA - 1) / RA : (TM * GEMM_KB + NT - 1) / NT, NBL = (GEMM_KB * TN + NT - 1) / NT;
    const int a_r0 = AT ? tid / TM : tid / GEMM_KB, a_kk = AT ? tid % TM : tid % GEMM_KB;
    const int b_k0 = tid / TN, b_c = tid % TN;                // B: rows b_k0 + u*RB, fixed column b_c
    const cplx* a_base = AT ? p.A + (i64)a_r0 * p.lda + (m0 + a_kk) : p.A + (i64)(m0 + a_r0) * p.lda + a_kk;
    const cplx* b_base = p.B + (i64)b_k0 * p.ldb + (n0 + b_c);
    const i64 a_step = (i64)RA * p.lda, b_step = (i64)RB * p.ldb;
    const bool a_col_ok = AT && a_r0 < RA && m0 + a_kk < p.M;
    const bool b_col_ok = n0 + b_c < p.N;
    auto stage_op = [&](int op, int k0, cplx* a, cplx* b) {   // op in [0, NA + NBL); everything but k0 folds at compile time
        if (op < NA) {
            const int u = op, r = a_r0 + u * RA;
            if constexpr (AT) {
                if (a_r0 < RA && r < GEMM_KB) {
                    const bool ok = a_col_ok && (k0 + r < p.K);
                    cp_async16(a + r * LDAT + a_kk, ok ? a_base + (i64)k0 * p.lda + u * a_step : p.A, ok);
                }
            } else if (u * NT + tid < TM * GEMM_KB) {
                const bool ok = (m0 + r < p.M) && (k0 + a_kk < p.K);
                cp_async16(a + r * GEMM_LDA + a_kk, ok ? a_base + u * a_step + k0 : p.A, ok);
            }
        } else {
            const int u = op - NA, kk = b_k0 + u * RB;
            if (u * NT + tid < GEMM_KB * TN) {
                const bool ok = b_col_ok && (k0 + kk < p.K);
                cp_async16(b + kk * LDB + b_c, ok ? b_base + (i64)k0 * p.ldb + u * b_step : p.B, ok);
            }
        }
    };
    auto load_stage = [&](int kt, int st) {
#pragma unroll
        for (int op = 0; op < NA + NBL; ++op) stage_op(op, kt * GEMM_KB, sA + st * Cfg::A_ELEMS, sB + st * Cfg::B_ELEMS);
    };

    double cre[MI][NI][2], cim[MI][NI][2];       // M3: cre = sum ar br, cim = sum (ar + ai)(br + bi), c2 = sum ai bi
    double c2[M3 ? MI : 1][M3 ? NI : 1][2];
#pragma unroll
    for (int mi = 0; mi < MI; ++mi)
#pragma unroll
        for (int ni = 0; ni < NI; ++ni) {
            cre[mi][ni][0] = cre[mi][ni][1] = cim[mi][ni][0] = cim[mi][ni][1] = 0.0;
            if constexpr (M3) c2[mi][ni][0] = c2[mi][ni][1] = 0.0;
        }

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < KT) load_stage(s, s);
        cp_async_commit();
    }

    constexpr int S4 = GEMM_KB / 4 / KS;                       // k4 steps a warp executes per stage
    constexpr int OPS = (NA + NBL + S4 - 1) / S4;              // staging copies issued after each of them
    for (int kt = 0; kt < KT; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        const int nk = kt + STAGES - 1;                        // stage refilled during this iteration (consumed in kt - 1)
        const bool refill = nk < KT;
        cplx* na = sA + (nk % STAGES) * Cfg::A_ELEMS;
        cplx* nb = sB + (nk % STAGES) * Cfg::B_ELEMS;
        const cplx* a = AT ? sA + (kt % STAGES) * Cfg::A_ELEMS + t * LDAT + wm * MI * 8 + g
                           : sA + (kt % STAGES) * Cfg::A_ELEMS + (wm * MI * 8 + g) * GEMM_LDA + t;
        const cplx* b = sB + (kt % STAGES) * Cfg::B_ELEMS + t * LDB + wn * NI * 8 + g;
#pragma unroll
        for (int k4s = 0; k4s < S4; ++k4s) {
            const int k4 = k4s * KS + wk;
            cplx af[MI], bf[NI];
#pragma unroll
            for (int mi = 0; mi < MI; ++mi) af[mi] = AT ? a[k4 * 4 * LDAT + mi * 8] : a[mi * 8 * GEMM_LDA + k4 * 4];
#pragma unroll
            for (int ni = 0; ni < NI; ++ni) bf[ni] = b[k4 * 4 * LDB + ni * 8];
            // two passes so that consecutive DMMAs never touch the same accumulator
            if constexpr (M3) {
                double as[MI], bs[NI];
#pragma unroll
                for (int mi = 0; mi < MI; ++mi) as[mi] = ACONJ ? af[mi].re - af[mi].im : af[mi].re + af[mi].im;
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) bs[ni] = bf[ni].re + bf[ni].im;
#pragma unroll
                for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni) {
                        dmma884(cre[mi][ni][0], cre[mi][ni][1], af[mi].re, bf[ni].re);
                        dmma884(c2[mi][ni][0], c2[mi][ni][1], af[mi].im, bf[ni].im);
                    }
                if (refill) {
#pragma unroll
                    for (int op = k4s * OPS; op < (k4s + 1) * OPS && op < NA + NBL; ++op) stage_op(op, nk * GEMM_KB, na, nb);
                }
#pragma unroll
                for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                    for (int ni = 0; ni < NI; ++ni) dmma884(cim[mi][ni][0], cim[mi][ni][1], as[mi], bs[ni]);
            } else {
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) {
                    dmma884(cre[mi][ni][0], cre[mi][ni][1], af[mi].re, bf[ni].re);
                    dmma884(cim[mi][ni][0], cim[mi][ni][1], af[mi].re, bf[ni].im);
                }
            if (refill) {
#pragma unroll
                for (int op = k4s * OPS; op < (k4s + 1) * OPS && op < NA + NBL; ++op) stage_op(op, nk * GEMM_KB, na, nb);
            }
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) {
                    dmma884(cre[mi][ni][0], cre[mi][ni][1], ACONJ ? af[mi].im : -af[mi].im, bf[ni].im);
                    dmma884(cim[mi][ni][0], cim[mi][ni][1], ACONJ ? -af[mi].im : af[mi].im, bf[ni].re);
                }
            }
        }
        cp_async_commit();
    }
    cp_async_wait<0>();
    if constexpr (M3) {
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < NI; ++ni)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const double t1 = cre[mi][ni][j], t2 = c2[mi][ni][j];
                    cre[mi][ni][j] = ACONJ ? t1 + t2 : t1 - t2;
                    cim[mi][ni][j] = ACONJ ? cim[mi][ni][j] - t1 + t2 : cim[mi][ni][j] - t1 - t2;
                }
    }
    if (KS > 1) {
        // sum the KS partial tiles: groups wk > 0 park their fragments in the (now idle) staging buffers
        static_assert(KS == 1 || KS == 2, "split-K reduction is written for two groups");
        static_assert(KS == 1 || TM * TN <= STAGES * (Cfg::A_ELEMS + Cfg::B_ELEMS), "partial tile must fit the staging buffers");
        __syncthreads();
        cplx* red = sA + (size_t)w2 * MI * NI * 64 + lane * 2;
        if (wk > 0) {
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < NI; ++ni) {
                    red[(mi * NI + ni) * 64] = mk(cre[mi][ni][0], cim[mi][ni][0]);
                    red[(mi * NI + ni) * 64 + 1] = mk(cre[mi][ni][1], cim[mi][ni][1]);
                }
        }
        __syncthreads();
        if (wk > 0) return;
#pragma unroll
        for (int mi = 0; mi < MI; ++mi)
#pragma unroll
            for (int ni = 0; ni < NI; ++ni)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const cplx v = red[(mi * NI + ni) * 64 + j];
                    cre[mi][ni][j] += v.re;
                    cim[mi][ni][j] += v.im;
                }
    }

    // epilogue: lane (g,t) owns C[8*.. + g][8*.. + 2t, 2t+1] of every 8x8 sub-tile
#pragma unroll
    for (int mi = 0; mi < MI; ++mi) {
        const int r = m0 + (wm * MI + mi) * 8 + g;
        if (r >= p.M) continue;
        const i64 crow = p.row_nx ? (i64)(r / p.row_nx) * p.row_fs + (r % p.row_nx) : (i64)r;
        cplx* crp = p.C + crow * p.ldc;
#pragma unroll
        for (int ni = 0; ni < NI; ++ni) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int cidx = n0 + (wn * NI + ni) * 8 + 2 * t + j;
                if (cidx >= p.N) continue;
                cplx v = mk(p.alpha * cre[mi][ni][j], p.alpha * cim[mi][ni][j]);
                if (p.beta) {
                    cplx cin;
                    if (cidx >= p.sub_c0 && cidx < p.sub_c1) cin = mk(r == cidx ? 1.0 : 0.0);
                    else cin = crp[cidx];
                    v = v + cin;
                }
                crp[cidx] = v;
            }
        }
    }
}

// ---- host-side dispatch -------------------------------------------------------------------
template <int MI, int NI, int WM, int WN, int STAGES, int KS = 1, bool M3 = false, int OPA = 0>
static inline int zgemm_launch_cfg(const GemmParams& p, cudaStream_t stream) {
    typedef GemmCfg<MI, NI, WM, WN, STAGES, KS> Cfg;
    auto kfn = zgemm_dmma_kernel<MI, NI, WM, WN, STAGES, KS, M3, OPA>;
    static std::atomic<unsigned long long> configured{0};
    hz_once_per_device(configured, [&]() { cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM); });
    dim3 grid((p.N + Cfg::TN - 1) / Cfg::TN, (p.M + Cfg::TM - 1) / Cfg::TM, 1);
    HZ_LAUNCH_IND(kfn, grid, dim3(Cfg::THREADS), Cfg::SMEM, stream, p);
    return 0;
}

// candidate tilings; the host picks the one with the best SM fill for (M, N)
struct GemmTile { int tm, tn; };
static const GemmTile kGemmTiles[] = {{64, 64}, {56, 64}, {48, 64}, {40, 64}, {32, 64}, {32, 32}, {16, 32}};
constexpr int kNumGemmTiles = sizeof(kGemmTiles) / sizeof(kGemmTiles[0]);

static inline int zgemm_pick(int M, int N, int num_sms) {
    double best = -1.0;
    int besti = 0;
    for (int i = 0; i < kNumGemmTiles; ++i) {
        const i64 tiles = (i64)((M + kGemmTiles[i].tm - 1) / kGemmTiles[i].tm) * ((N + kGemmTiles[i].tn - 1) / kGemmTiles[i].tn);
        const i64 waves = (tiles + num_sms - 1) / num_sms;
        // useful work / (waves * full-machine tile work); mild preference for larger tiles
        double eff = (double)M * N / ((double)waves * num_sms * kGemmTiles[i].tm * kGemmTiles[i].tn);
        eff *= 1.0 + 0.02 * (kGemmTiles[i].tm * kGemmTiles[i].tn) / 4096.0;
        if (eff > best) { best = eff; besti = i; }
    }
    return besti;
}

// kernel instance (tile id of zgemm_launch) for candidate tiling `cand` of kGemmTiles and the product form; m3 ids are
// 16 + cand, except 56 x 64: warps of 56 x 16 need fewer operand sums per DMMA (109 vs 111 us at 1000 x 512 x 1000)
static inline int zgemm_tile_id(int cand, bool m3) {
    const int which = cand + (m3 ? 16 : 0);
    return which == 17 ? 24 : which;
}

// every instance zgemm_launch can pick for op(A) = OPA (for OPA = 0 also the study tiles), for the eager kernel preload
// (hz_api.cu: preload_all_kernels)
template <int OPA, class F>
static inline void zgemm_for_each_instance(F f) {
    f(zgemm_dmma_kernel<4, 2, 2, 4, 3, 1, false, OPA>); f(zgemm_dmma_kernel<7, 1, 1, 8, 3, 1, false, OPA>);
    f(zgemm_dmma_kernel<6, 1, 1, 8, 3, 1, false, OPA>); f(zgemm_dmma_kernel<5, 1, 1, 8, 3, 1, false, OPA>);
    f(zgemm_dmma_kernel<2, 2, 2, 4, 4, 1, false, OPA>); f(zgemm_dmma_kernel<2, 1, 2, 4, 4, 1, false, OPA>);
    f(zgemm_dmma_kernel<1, 1, 2, 4, 4, 1, false, OPA>);
    // three-multiplication twins of the tiles zgemm_pick chooses from
    f(zgemm_dmma_kernel<4, 2, 2, 4, 3, 1, true, OPA>); f(zgemm_dmma_kernel<6, 1, 1, 8, 3, 1, true, OPA>);
    f(zgemm_dmma_kernel<5, 1, 1, 8, 3, 1, true, OPA>); f(zgemm_dmma_kernel<2, 2, 2, 4, 4, 1, true, OPA>);
    f(zgemm_dmma_kernel<2, 1, 2, 4, 4, 1, true, OPA>); f(zgemm_dmma_kernel<1, 1, 2, 4, 4, 1, true, OPA>);
    f(zgemm_dmma_kernel<7, 2, 1, 4, 3, 2, true, OPA>);
    if constexpr (OPA == 0) {
        f(zgemm_dmma_kernel<7, 1, 1, 8, 3, 2>); f(zgemm_dmma_kernel<4, 2, 2, 4, 3, 2>); f(zgemm_dmma_kernel<6, 1, 1, 8, 3, 2>);
        f(zgemm_dmma_kernel<5, 1, 1, 8, 3, 2>); f(zgemm_dmma_kernel<7, 2, 1, 4, 3>); f(zgemm_dmma_kernel<7, 2, 1, 4, 3, 2>);
        f(zgemm_dmma_kernel<7, 1, 1, 8, 3, 1, true>); f(zgemm_dmma_kernel<7, 2, 1, 4, 3, 1, true>); f(zgemm_dmma_kernel<7, 1, 1, 8, 3, 2, true>);
    }
}

// m3: three-multiplication complex products (tiles 16 + i are the M3 twins of the auto-picked tiles 0..6).  op(A) T and C
// (OPA 1, 2) exist for the tiles the host picks (zgemm_tile_id); the study tiles 7..12, 17, 23, 25 are op N only.
template <int OPA = 0>
static inline int zgemm_launch(const GemmParams& p, cudaStream_t stream, int num_sms, int force_tile = -1, bool m3 = false) {
    const int which = force_tile >= 0 ? force_tile : zgemm_tile_id(zgemm_pick(p.M, p.N, num_sms), m3);
    switch (which) {
        case 16: return zgemm_launch_cfg<4, 2, 2, 4, 3, 1, true, OPA>(p, stream);
        case 18: return zgemm_launch_cfg<6, 1, 1, 8, 3, 1, true, OPA>(p, stream);
        case 19: return zgemm_launch_cfg<5, 1, 1, 8, 3, 1, true, OPA>(p, stream);
        case 20: return zgemm_launch_cfg<2, 2, 2, 4, 4, 1, true, OPA>(p, stream);
        case 21: return zgemm_launch_cfg<2, 1, 2, 4, 4, 1, true, OPA>(p, stream);
        case 22: return zgemm_launch_cfg<1, 1, 2, 4, 4, 1, true, OPA>(p, stream);
        case 24: return zgemm_launch_cfg<7, 2, 1, 4, 3, 2, true, OPA>(p, stream);   // M3 twin of 12 (56 x 64, warps of 56 x 16, split-K)
        case 0: return zgemm_launch_cfg<4, 2, 2, 4, 3, 1, false, OPA>(p, stream);   // 64 x 64
        case 1: return zgemm_launch_cfg<7, 1, 1, 8, 3, 1, false, OPA>(p, stream);   // 56 x 64
        case 2: return zgemm_launch_cfg<6, 1, 1, 8, 3, 1, false, OPA>(p, stream);   // 48 x 64
        case 3: return zgemm_launch_cfg<5, 1, 1, 8, 3, 1, false, OPA>(p, stream);   // 40 x 64
        case 4: return zgemm_launch_cfg<2, 2, 2, 4, 4, 1, false, OPA>(p, stream);   // 32 x 64
        case 5: return zgemm_launch_cfg<2, 1, 2, 4, 4, 1, false, OPA>(p, stream);   // 32 x 32
        case 6: return zgemm_launch_cfg<1, 1, 2, 4, 4, 1, false, OPA>(p, stream);   // 16 x 32
        default: break;
    }
    if constexpr (OPA == 0) {
        switch (which) {
            case 17: return zgemm_launch_cfg<7, 1, 1, 8, 3, 1, true>(p, stream);
            case 23: return zgemm_launch_cfg<7, 2, 1, 4, 3, 1, true>(p, stream);   // M3 twins of 11 and 7 (fewer operand sums per DMMA / split-K)
            case 25: return zgemm_launch_cfg<7, 1, 1, 8, 3, 2, true>(p, stream);
            case 7: return zgemm_launch_cfg<7, 1, 1, 8, 3, 2>(p, stream);   // 56 x 64, 16 warps (split-K)
            case 8: return zgemm_launch_cfg<4, 2, 2, 4, 3, 2>(p, stream);   // 64 x 64, 16 warps (split-K)
            case 9: return zgemm_launch_cfg<6, 1, 1, 8, 3, 2>(p, stream);   // 48 x 64, 16 warps
            case 10: return zgemm_launch_cfg<5, 1, 1, 8, 3, 2>(p, stream);  // 40 x 64, 16 warps
            case 11: return zgemm_launch_cfg<7, 2, 1, 4, 3>(p, stream);     // 56 x 64, 4 warps of 56 x 16
            case 12: return zgemm_launch_cfg<7, 2, 1, 4, 3, 2>(p, stream);  // 56 x 64, 8 warps of 56 x 16 (split-K)
            default: break;
        }
    }
    return zgemm_launch_cfg<1, 1, 2, 4, 4, 1, false, OPA>(p, stream);
}
