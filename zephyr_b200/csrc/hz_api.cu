// C ABI of zephyr_b200 (include/zephyr_b200.h): handle management and host orchestration of the
// sm_100a kernels.  One translation unit; built by zephyr_b200/build.py with
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -shared -Xcompiler -fPIC
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "hz_platform.h"
#include "hz_assemble.cuh"
#include "hz_gemm.cuh"
#include "hz_factor.cuh"
#include "hz_factor_f32.cuh"
#include "hz_c64.cuh"
#include "hz_tf32.cuh"
#include "hz_solve.cuh"
#include "hz_survey.cuh"
#include "hz_adjoint.cuh"
#include "hz_born.cuh"
#include "../../include/zephyr_b200.h"

// sampled device timing of the contraction kernel (every PROF_EVERY-th launch is bracketed by
// CUDA events on its own stream); kind 0 = substitution GEMM, 1 = Gauss-Jordan update GEMM
constexpr int PROF_EVERY = 16, PROF_MAX = 4096;

struct hz_ctx {
    int device = 0, dtype = 0, disc = 0, nf = 1;
    int nx = 0, nz = 0, b = 0, nPML = 10;
    i64 N = 0;
    double dx = 1, dz = 1, cPML = 1e3;
    int fs[4] = {0, 0, 0, 0};
    int num_sms = 148;
    cudaStream_t stream = nullptr, stream2 = nullptr;
    cudaStream_t stream1 = nullptr;                                       // top elimination chain (so that handles sharing the caller's stream can factor concurrently)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join0 = nullptr;
    // model + operator
    cplx* c = nullptr;
    double *rho = nullptr, *theta = nullptr, *eps = nullptr, *delta = nullptr;
    cplx* coef = nullptr;
    cplx* Kp = nullptr;          // per-node mass term (assembly pre-pass)
    double* binv = nullptr;      // per-node buoyancy 1/rho
    cplx* pmltab = nullptr;      // Eurus: 3*nx + 3*nz PML reciprocal tables
    bool have_model = false, assembled = false, factored = false;
    AsmParams asm_p;             // parameters of the last hz_assemble (the adjoint-gradient VJP recomputes from them)
    bool asm_from_model = false; // false after hz_set_coefficients: the planes are no longer a function of the model
    // factors and workspaces
    cplx* Sinv = nullptr;        // complex128 block inverses (HZ_C128)
    cplxf* Sinv64 = nullptr;     // complex64 block inverses (HZ_C64)
    cplxf* Scratch64[2] = {nullptr, nullptr};   // HZ_C64 fp32 factorisation: ping-pong partner, panels, published pivot inverse
    cplxf *Rf[2] = {nullptr, nullptr}, *Cf[2] = {nullptr, nullptr}, *Pgf[2] = {nullptr, nullptr};
    // complex64 on the tcgen05 tensor cores (hz_tf32.cuh): planar storage of the block inverses + TMA/TMEM 3xTF32 substitution GEMM
    int c64_tf32 = 1;                             // option; 0: interleaved storage + FP32 FFMA contraction (round-1 path)
    int tf32_sms = 0;                             // option: SMs one contraction is spread over by split-K (0: all; 74 lets the two sweep chains overlap)
    bool tf32_active = false;                     // decided when the factors are allocated
    int ldb64 = 0;                                // row stride (floats) of a planar block plane
    i64 y_S = -1;                                 // number of columns the Y tensor maps were built for
#ifndef HZ_EMU
    alignas(64) CUtensorMap mapA;
    alignas(64) CUtensorMap mapY[2];
#endif
    int c64_fp64_factor = 1;                      // HZ_C64: 1 (default) = factorise in FP64 and round each finished inverse; 0 = all-FP32 factorisation (study option: loses accuracy at nx = 1000, see profiles/r1d_tolerance_study_fp32_factor.json)
    cplx* Ring[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // HZ_C64: per chain, complex128 window of the last two blocks
    i64 mid = -1;
    // Checkpointed factors (option "store_every" = k > 1): only every k-th block inverse of each elimination chain
    // is kept (plus the last block of each chain and the middle block); the k-1 blocks in between are recomputed,
    // segment by segment, from the preceding checkpoint whenever a substitution sweep needs them (2 (k-1)/k extra
    // factorisations per solve, 1/k of the HBM).  This is what lets 2000 x 6000 (384 GB of complex128 inverses) run
    // on one 180 GB GPU.  slot_of() maps a block row to its slot in Sinv / Sinv64.
    int store_every = 1;
    int store_used = 1;          // the k the current allocation / factors were made with
    i64 nslots = 0;
    cplx *Rbuf[2] = {nullptr, nullptr}, *Cbuf[2] = {nullptr, nullptr};   // per chain: two panel parities each
    cplx* Pg[2] = {nullptr, nullptr};                                     // per chain: 2 parities of the published pivot inverse
    int* d_flag = nullptr;                                                // per chain flag (2 ints)
    int gj_seq = 0;
    // inverter service (gj_service): one persistent CTA per chain on its own stream, a mailbox and a
    // completion counter per chain
    int gj_service = 2;                                                   // 2: self-driven inverter service (default); 1: request per step; 0: inverter CTA inside the step kernel
    int gj_colper = 1;                                                    // column blocks per column-block CTA in launches with update tiles (2: measured slower, the pre-work then outlasts the inverse)
    int gj_coltile = 0;                                                   // 1: column-block CTAs also process update tiles while they wait for the inverse (measured slower: they pick the inverse up late)
    int service_fallbacks = 0;
    bool svc_on[2] = {false, false};
    cudaStream_t svc_stream[2] = {nullptr, nullptr};
    cudaEvent_t ev_svc[2] = {nullptr, nullptr};
    GjJob* d_mail = nullptr;                                              // [2]
    GjBlockJob* d_mail2 = nullptr;                                        // [2] self-driven service (gj_service = 2)
    cplx* d_Tg = nullptr;                                                 // [2 chains][2 parities] T tiles handed to the service
    int* d_cflag = nullptr;                                               // [2 chains][colflag, tileflag]
    int* d_mail_flag = nullptr;                                           // [2]
    unsigned long long* d_done = nullptr;                                 // [2]
    unsigned long long done_total[2] = {0, 0};
    int seq_chain[2] = {0, 0};
    cplx* Scratch[2] = {nullptr, nullptr};                               // per chain: ping-pong partner of the block slot
    int* d_sync[2] = {nullptr, nullptr};                                  // gj_mode 3: per chain, ticket + dependence counters of one block row
    size_t sync_bytes = 0;
    int gj_lean = 0;                                                      // 1: service-mode launches use the lean instance of the step kernel (hz_factor.cuh: gj_step_kernel LEAN; measured: no gain)
    int gemm_3m = 1;                                                      // complex products with three real DMMAs instead of four: bit 0 substitution GEMMs, bit 1 Gauss-Jordan update tiles
    int gj_colpair = 0;                                                   // column-block CTAs own two column blocks, processed side by side (hz_factor.cuh: gj_panel_pair)
    int gj_colslow = 0;                                                   // A/B option: column-block CTAs load their operands in dependent rounds (pre-r2p)
    int gj_crit = 1;                                                      // dispatch the update tile that feeds the inverter service first
    int gj_pdl = 0;                                                       // programmatic dependent launch between GJ steps
    int gj_order = 0;                                                     // 1: block order inverter | update tiles | column blocks
    int gj_inv = -1;                                                      // block index of the inverter CTA (-1: 147 when it has no SM partner, else 0)
    int gj_tile = 3;                                                      // update-tile variant of the fused step kernel (table gj_variants)
    int gj_trace = 0;                                                     // record per-CTA timestamps of the last block's steps
    long long* d_trace[2] = {nullptr, nullptr};                          // per elimination chain
    bool trace_now = false;                                               // set per block by factor_block
    int trace_chain = 0;                                                  // which chain hz_get_trace returns
    int trace_steps = 0, trace_grid = 0;
    // Option "factor_graph": the launch sequence of a factorisation is static (same buffers, same sequence numbers once the
    // flags are reset at the head), so it can be captured ONCE into a CUDA graph -- both chain streams, the inverter-service
    // streams and their fork/join events -- and replayed by later factorisations of the handle.  Measured (profiles/
    // r2r_graph_and_workers.md): no gain on C2 (b = 400) or C4 (b = 500) -- a step there is bound by the dependent-kernel
    // latency on the device (16 us per Gauss-Jordan step, pivot inverse + column-block path), not by the host's launch
    // rate -- and the end-to-end numbers get worse (capture + instantiation after a model update).  So it is off by default.
    int factor_graph = 0;                                                 // option: 0 never (default), 1 always, -1 from the second factorisation on when the sequence has <= 16384 launches
#ifndef HZ_EMU
    cudaGraphExec_t fgraph = nullptr;
#endif
    unsigned long long fgraph_key = 0, fgraph_seen = 0, fgraph_want = 0;
    long long fgraph_launches = 0;                                        // kernels in the graph (added to the launch count on every replay)
    int fgraph_replays = 0;
    unsigned opt_epoch = 0;                                               // bumped by hz_set_option: options change the launch sequence
    cudaEvent_t ev_svc_join[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork2 = nullptr;
    int gj_mode = 1;                                                      // 3: one launch per block row (dependence counters instead of launch boundaries), 1: one fused look-ahead launch per step, 2: delayed rank-64 updates, 0: v1 panel+update
    cplx* Ybuf[2] = {nullptr, nullptr};
    i64 ycap = 0;
    cplx *Qsave = nullptr, *Rres = nullptr;
    i64 qcap = 0;
    // accuracy probe: the block inverses come from a Gauss-Jordan elimination without pivoting across panels, so
    // the first solve after every factorisation measures the stencil residual of one right-hand-side column
    // (in FP64) and fails loudly (HZ_EACCURACY) instead of returning a silently inaccurate wavefield
    int probe_check = 1;
    double probe_limit = 0.0;       // 0: default limits (1e-7 complex128, 1e-2 complex64)
    bool probe_pending = false;
    cplx* Qprobe = nullptr;
    double last_probe = -1.0;
    int* d_err = nullptr;
    double* d_norm = nullptr;
    // profiling
    bool prof_on = false;
    long long prof_tick[2] = {0, 0};
    std::vector<cudaEvent_t> prof_ev[2];     // start/stop pairs
    long long prof_launches[2] = {0, 0};
    std::string err;
};

static void prof_begin(hz_ctx* h, int kind, cudaStream_t st, bool& armed) {
    armed = false;
    if (!h->prof_on) return;
    ++h->prof_launches[kind];
    if ((h->prof_tick[kind]++ % PROF_EVERY) != 0 || (int)h->prof_ev[kind].size() >= 2 * PROF_MAX) return;
    cudaEvent_t e0, e1;
    if (cudaEventCreate(&e0) != cudaSuccess) return;
    if (cudaEventCreate(&e1) != cudaSuccess) { cudaEventDestroy(e0); return; }
    h->prof_ev[kind].push_back(e0);
    h->prof_ev[kind].push_back(e1);
    cudaEventRecord(e0, st);
    armed = true;
}
static void prof_end(hz_ctx* h, int kind, cudaStream_t st, bool armed) {
    if (armed) cudaEventRecord(h->prof_ev[kind].back(), st);
}

static thread_local std::string g_err;
// inverter-service health, process-wide: consecutive factorisations in which the service failed to co-run with the step
// kernels.  One failure can be a scheduling accident (the factorisation is simply redone with the in-kernel inverter);
// two in a row mean something serialises the launches (a profiler, CUDA_LAUNCH_BLOCKING, a sanitizer): the service is
// then switched off for the rest of the process instead of costing a device-side timeout per factorisation.
static std::atomic<int> g_service_failures{0};
static std::atomic<int> g_service_unavailable{0};
std::atomic<long long> g_hz_launches{0};

static int fail(hz_ctx* h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_err = msg;
    return code;
}

#define HZ_CUDA(h, call)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(h, e_ == cudaErrorMemoryAllocation ? HZ_ENOMEM : HZ_ECUDA,                \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                      \
    } while (0)

#define HZ_CHECK_LAUNCH(h) HZ_CUDA(h, cudaGetLastError())

template <class T>
static void free_dev(T*& p) {
    if (p) cudaFree(p);
    p = nullptr;
}

static inline unsigned blocks_for(i64 n, int threads, i64 cap = 148 * 32) {
    i64 nb = (n + threads - 1) / threads;
    if (nb > cap) nb = cap;
    if (nb < 1) nb = 1;
    return (unsigned)nb;
}

// Every exported function below is declared extern "C" in include/zephyr_b200.h and takes that linkage.

const char* hz_version(void) {
#ifdef HZ_EMU
    return "zephyr_b200 0.1.0 (cpu-emulation test build)";
#else
    return "zephyr_b200 0.1.0 (sm_100a)";
#endif
}

const char* hz_last_error(hz_handle_t h) { return h ? h->err.c_str() : g_err.c_str(); }

int hz_create(hz_handle_t* out, int device, int dtype, int disc, int64_t nx, int64_t nz, double dx, double dz,
              int nPML, double cPML, const int32_t* freeSurf_host, void* stream) {
    if (!out) return fail(nullptr, HZ_EINVAL, "hz_create: out is NULL");
    *out = nullptr;
    if (nx < 3 || nz < 3 || nx > 32768 || nz > (1 << 24)) return fail(nullptr, HZ_EINVAL, "hz_create: nx, nz out of range");
    if (!(dx > 0) || !(dz > 0)) return fail(nullptr, HZ_EINVAL, "hz_create: dx, dz must be positive");
    if (disc != HZ_DISC_MINIZEPHYR && disc != HZ_DISC_EURUS) return fail(nullptr, HZ_EINVAL, "hz_create: unknown discretisation");
    if (dtype != HZ_C128 && dtype != HZ_C64) return fail(nullptr, HZ_EINVAL, "hz_create: unknown dtype");
    if (nPML < 2 || nPML > nx || nPML > nz) return fail(nullptr, HZ_EINVAL, "hz_create: nPML out of range");
    hz_ctx* h = new (std::nothrow) hz_ctx();
    if (!h) return fail(nullptr, HZ_ENOMEM, "hz_create: host allocation failed");
    h->device = device; h->dtype = dtype; h->disc = disc;
    h->nf = disc == HZ_DISC_EURUS ? 2 : 1;
    h->nx = (int)nx; h->nz = (int)nz; h->N = nx * nz; h->b = h->nf * (int)nx;
    h->dx = dx; h->dz = dz; h->nPML = nPML; h->cPML = cPML;
    for (int i = 0; i < 4; ++i) h->fs[i] = freeSurf_host ? (freeSurf_host[i] != 0) : 0;
    h->stream = (cudaStream_t)stream;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) {
        cudaDeviceProp prop;
        e = cudaGetDeviceProperties(&prop, device);
        if (e == cudaSuccess) h->num_sms = prop.multiProcessorCount;
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream1, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join0, cudaEventDisableTiming);
    for (int k = 0; k < 2; ++k)
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->svc_stream[k], cudaStreamNonBlocking);
    for (int k = 0; k < 2; ++k)
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_svc[k], cudaEventDisableTiming);
    for (int k = 0; k < 2; ++k)
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_svc_join[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc((void**)&h->d_err, sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void**)&h->d_norm, 2 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemsetAsync(h->d_err, 0, sizeof(int), h->stream);
    if (e != cudaSuccess) {
        std::string m = std::string("hz_create: ") + cudaGetErrorString(e);
        hz_destroy(h);
        return fail(nullptr, HZ_ECUDA, m);
    }
    *out = h;
    return HZ_OK;
}

int hz_free_factors(hz_handle_t h) {
    if (!h) return HZ_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (h->stream2) cudaStreamSynchronize(h->stream2);
    if (h->stream1) cudaStreamSynchronize(h->stream1);
    free_dev(h->Sinv);
    free_dev(h->Sinv64);
    for (int k = 0; k < 2; ++k) { free_dev(h->Ring[k][0]); free_dev(h->Ring[k][1]); free_dev(h->Scratch64[k]); free_dev(h->Rf[k]); free_dev(h->Cf[k]); free_dev(h->Pgf[k]); }
    for (int k = 0; k < 2; ++k) { free_dev(h->Rbuf[k]); free_dev(h->Cbuf[k]); free_dev(h->Ybuf[k]); free_dev(h->Scratch[k]); free_dev(h->Pg[k]); }
    free_dev(h->Qsave); free_dev(h->Rres); free_dev(h->Qprobe);
    h->ycap = h->qcap = 0;
    h->factored = false;
    return HZ_OK;
}

int hz_destroy(hz_handle_t h) {
    if (!h) return HZ_OK;
    hz_free_factors(h);
    free_dev(h->c); free_dev(h->rho); free_dev(h->theta); free_dev(h->eps); free_dev(h->delta);
    free_dev(h->coef); free_dev(h->Kp); free_dev(h->binv); free_dev(h->pmltab); free_dev(h->d_err); free_dev(h->d_norm); free_dev(h->d_trace[0]); free_dev(h->d_trace[1]); free_dev(h->d_flag);
    free_dev(h->d_sync[0]); free_dev(h->d_sync[1]);
    free_dev(h->d_mail); free_dev(h->d_mail_flag); free_dev(h->d_done); free_dev(h->d_mail2); free_dev(h->d_Tg); free_dev(h->d_cflag);
    for (int k = 0; k < 2; ++k) if (h->svc_stream[k]) cudaStreamDestroy(h->svc_stream[k]);
    for (int k = 0; k < 2; ++k) if (h->ev_svc[k]) cudaEventDestroy(h->ev_svc[k]);
    for (int k = 0; k < 2; ++k) for (cudaEvent_t e : h->prof_ev[k]) cudaEventDestroy(e);
#ifndef HZ_EMU
    if (h->fgraph) cudaGraphExecDestroy(h->fgraph);
#endif
    for (int k = 0; k < 2; ++k) if (h->ev_svc_join[k]) cudaEventDestroy(h->ev_svc_join[k]);
    if (h->ev_fork2) cudaEventDestroy(h->ev_fork2);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->ev_join0) cudaEventDestroy(h->ev_join0);
    if (h->stream2) cudaStreamDestroy(h->stream2);
    if (h->stream1) cudaStreamDestroy(h->stream1);
    delete h;
    return HZ_OK;
}

int hz_has_factors(hz_handle_t h, int32_t* out) {
    if (!h || !out) return fail(h, HZ_EINVAL, "hz_has_factors: NULL argument");
    *out = h->factored ? 1 : 0;
    return HZ_OK;
}

static i64 slots_needed(i64 nz, i64 mid, int k);
int hz_factor_bytes(hz_handle_t h, int64_t* bytes) {
    if (!h || !bytes) return fail(h, HZ_EINVAL, "hz_factor_bytes: NULL argument");
    const int k = h->store_every < 1 ? 1 : h->store_every;
    const i64 mid = h->factored ? h->mid : (i64)h->nz / 2;
    *bytes = slots_needed(h->nz, mid, k) * h->b * h->b * (i64)(h->dtype == HZ_C64 ? sizeof(cplxf) : sizeof(cplx));   // (planar storage pads rows to 4 floats)
    return HZ_OK;
}

int hz_factor_resident_bytes(hz_handle_t h, int64_t* bytes) {
    if (!h || !bytes) return fail(h, HZ_EINVAL, "hz_factor_resident_bytes: NULL argument");
    *bytes = (h->Sinv || h->Sinv64) ? h->nslots * h->b * h->b * (i64)(h->dtype == HZ_C64 ? sizeof(cplxf) : sizeof(cplx)) : 0;
    return HZ_OK;
}

int hz_set_stream(hz_handle_t h, void* stream) {
    if (!h) return fail(h, HZ_EINVAL, "hz_set_stream: NULL handle");
    cudaStream_t st = (cudaStream_t)stream;
    if (st == h->stream) return HZ_OK;
    HZ_CUDA(h, cudaSetDevice(h->device));
    // work already queued on the old stream stays ordered before anything issued on the new one
    HZ_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
    HZ_CUDA(h, cudaStreamWaitEvent(st, h->ev_fork, 0));
    h->stream = st;
    return HZ_OK;
}

int hz_last_probe(hz_handle_t h, double* out) {
    if (!h || !out) return fail(h, HZ_EINVAL, "hz_last_probe: NULL argument");
    *out = h->last_probe;
    return HZ_OK;
}

int hz_synchronize(hz_handle_t h) {
    if (!h) return fail(h, HZ_EINVAL, "hz_synchronize: NULL handle");
    HZ_CUDA(h, cudaSetDevice(h->device));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream2));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream1));
    return HZ_OK;
}

int hz_set_model(hz_handle_t h, const void* c, const double* rho, const double* theta, const double* eps,
                 const double* delta, int on_device) {
    if (!h) return fail(h, HZ_EINVAL, "hz_set_model: NULL handle");
    if (!c || !rho) return fail(h, HZ_EINVAL, "hz_set_model: c and rho are required");
    if (h->disc == HZ_DISC_EURUS && (!theta || !eps || !delta))
        return fail(h, HZ_EINVAL, "hz_set_model: Eurus needs theta, eps and delta");
    HZ_CUDA(h, cudaSetDevice(h->device));
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const size_t nd = (size_t)h->N * sizeof(double);
    if (!h->c) HZ_CUDA(h, cudaMalloc((void**)&h->c, 2 * nd));
    if (!h->rho) HZ_CUDA(h, cudaMalloc((void**)&h->rho, nd));
    HZ_CUDA(h, cudaMemcpyAsync(h->c, c, 2 * nd, kind, h->stream));
    HZ_CUDA(h, cudaMemcpyAsync(h->rho, rho, nd, kind, h->stream));
    if (h->disc == HZ_DISC_EURUS) {
        if (!h->theta) HZ_CUDA(h, cudaMalloc((void**)&h->theta, nd));
        if (!h->eps) HZ_CUDA(h, cudaMalloc((void**)&h->eps, nd));
        if (!h->delta) HZ_CUDA(h, cudaMalloc((void**)&h->delta, nd));
        HZ_CUDA(h, cudaMemcpyAsync(h->theta, theta, nd, kind, h->stream));
        HZ_CUDA(h, cudaMemcpyAsync(h->eps, eps, nd, kind, h->stream));
        HZ_CUDA(h, cudaMemcpyAsync(h->delta, delta, nd, kind, h->stream));
    }
    if (!on_device) HZ_CUDA(h, cudaStreamSynchronize(h->stream));   // host buffers may be released
    h->have_model = true;
    h->assembled = false;
    h->factored = false;
    return HZ_OK;
}

int hz_assemble(hz_handle_t h, double freq_re, double freq_im, double tau, double ky) {
    if (!h) return fail(h, HZ_EINVAL, "hz_assemble: NULL handle");
    if (!h->have_model) return fail(h, HZ_ESTATE, "hz_assemble: call hz_set_model first");
    HZ_CUDA(h, cudaSetDevice(h->device));
    if (!h->coef) HZ_CUDA(h, cudaMalloc((void**)&h->coef, (size_t)h->nf * h->nf * 9 * h->N * sizeof(cplx)));
    AsmParams p;
    p.nx = h->nx; p.nz = h->nz; p.nPML = h->nPML; p.dx = h->dx; p.dz = h->dz;
    const double two_pi = 2 * 3.14159265358979323846;
    // omega - i/tau ; tau = inf gives 0 damping (discretization.py:33-41)
    const double damp = std::isinf(tau) ? 0.0 : 1.0 / tau;
    p.omd = mk(two_pi * freq_re, two_pi * freq_im - damp);
    p.aky = two_pi * ky;
    p.cPML = h->cPML;
    for (int i = 0; i < 4; ++i) p.fs[i] = h->fs[i];
    const int threads = 128;
    const unsigned grid = (unsigned)((h->N + threads - 1) / threads);
    if (!h->Kp) HZ_CUDA(h, cudaMalloc((void**)&h->Kp, (size_t)h->N * sizeof(cplx)));
    if (!h->binv) HZ_CUDA(h, cudaMalloc((void**)&h->binv, (size_t)h->N * sizeof(double)));
    HZ_LAUNCH_EW(node_terms_kernel, dim3(grid), dim3(threads), 0, h->stream, (const cplx*)h->c, (const double*)h->rho, h->N, p.omd * p.omd,
                 p.aky * p.aky, h->disc == HZ_DISC_EURUS ? 1 : 0, h->Kp, h->binv);
    HZ_CHECK_LAUNCH(h);
    if (h->disc == HZ_DISC_EURUS) {
        if (!h->pmltab) HZ_CUDA(h, cudaMalloc((void**)&h->pmltab, (size_t)3 * (h->nx + h->nz) * sizeof(cplx)));
        cplx* tabx = h->pmltab;
        cplx* tabz = h->pmltab + 3 * h->nx;
        HZ_LAUNCH_EW(eurus_pml_tables_kernel, dim3((h->nx + 127) / 128), dim3(128), 0, h->stream, h->nx, h->nPML, h->dx, h->cPML, p.omd, tabx);
        HZ_LAUNCH_EW(eurus_pml_tables_kernel, dim3((h->nz + 127) / 128), dim3(128), 0, h->stream, h->nz, h->nPML, h->dz, h->cPML, p.omd, tabz);
        HZ_LAUNCH_EW(assemble_eurus_kernel, dim3(grid), dim3(threads), 0, h->stream, (const cplx*)h->Kp, (const double*)h->binv,
                     (const cplx*)tabx, (const cplx*)tabz, (const double*)h->theta, (const double*)h->eps, (const double*)h->delta, h->coef, p);
    } else {
        HZ_LAUNCH_EW(assemble_mz_kernel, dim3(grid), dim3(threads), 0, h->stream, (const cplx*)h->c, (const cplx*)h->Kp,
                     (const double*)h->binv, h->coef, p);
    }
    HZ_CHECK_LAUNCH(h);
    h->assembled = true;
    h->factored = false;
    h->asm_p = p;
    h->asm_from_model = true;
    return HZ_OK;
}

int hz_set_coefficients(hz_handle_t h, const void* planes_host) {
    if (!h || !planes_host) return fail(h, HZ_EINVAL, "hz_set_coefficients: NULL argument");
    HZ_CUDA(h, cudaSetDevice(h->device));
    const size_t bytes = (size_t)h->nf * h->nf * 9 * h->N * sizeof(cplx);
    if (!h->coef) HZ_CUDA(h, cudaMalloc((void**)&h->coef, bytes));
    HZ_CUDA(h, cudaMemcpyAsync(h->coef, planes_host, bytes, cudaMemcpyHostToDevice, h->stream));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream));
    h->assembled = true;
    h->factored = false;
    h->asm_from_model = false;
    return HZ_OK;
}

int hz_get_coefficients(hz_handle_t h, void* out_host) {
    if (!h || !out_host) return fail(h, HZ_EINVAL, "hz_get_coefficients: NULL argument");
    if (!h->assembled) return fail(h, HZ_ESTATE, "hz_get_coefficients: call hz_assemble first");
    HZ_CUDA(h, cudaSetDevice(h->device));
    HZ_CUDA(h, cudaMemcpyAsync(out_host, h->coef, (size_t)h->nf * h->nf * 9 * h->N * sizeof(cplx), cudaMemcpyDeviceToHost, h->stream));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream));
    return HZ_OK;
}

// ---- factorisation ---------------------------------------------------------------------------
template <class TB>
static int launch_schur(hz_ctx* h, i64 i, const TB* Xa, const TB* Xb, TB* dst, cudaStream_t st) {
    dim3 grid((h->nx + SCHUR_TC - 1) / SCHUR_TC, h->b, 1);       // one row, SCHUR_TC x positions of every field per CTA
    auto kfn = schur_form_kernel<TB>;
    HZ_LAUNCH_IND(kfn, grid, dim3(SCHUR_TC), SCHUR_SMEM, st, (const cplx*)h->coef, h->nf, h->nx, h->nz, (int)i, Xa, Xb, dst);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

static int launch_invert_v1(hz_ctx* h, cplx* A, int chain, cudaStream_t st) {
    const int b = h->b;
    const int nsteps = (b + GJ_NB - 1) / GJ_NB;
    const size_t smem = 2 * GJ_NB * (GJ_NB + 1) * sizeof(cplx);
    for (int k = 0; k < nsteps; ++k) {
        const int k0 = k * GJ_NB, kb = (b - k0) < GJ_NB ? (b - k0) : GJ_NB;
        HZ_LAUNCH(gj_panel_kernel, dim3(nsteps), dim3(256), smem, st, (const cplx*)A, b, k0, kb, h->Rbuf[chain], h->Cbuf[chain], h->d_err);
        HZ_CHECK_LAUNCH(h);
        GemmParams p;
        p.A = h->Cbuf[chain]; p.lda = GJ_NB;
        p.B = h->Rbuf[chain]; p.ldb = b;
        p.C = A; p.ldc = b;
        p.M = b; p.N = b; p.K = kb;
        p.alpha = -1.0; p.beta = 1;
        p.sub_c0 = k0; p.sub_c1 = k0 + kb;
        p.row_nx = 0; p.row_fs = 0;
        bool armed;
        prof_begin(h, 1, st, armed);
        zgemm_launch(p, st, h->num_sms);
        prof_end(h, 1, st, armed);
        HZ_CHECK_LAUNCH(h);
    }
    return HZ_OK;
}

// v2: one fused launch per panel step (update k + look-ahead panel k+1), block ping-pongs between
// its HBM slot and a scratch buffer; `start` says which of the two holds S (see hz_factor).
typedef GjStepCfg<4, 2, 2, 4> GjCfg;      // 64 x 64 update tiles: 256 tiles + 32 column-block CTAs (+ inverter) fit one wave at 2 CTAs/SM

static int gj_start_buffer(const hz_ctx* h) { return ((h->b + GJ_NB - 1) / GJ_NB) % 2; }   // 0: slot, 1: scratch

// Selectable variants of the fused step kernel (option gj_tile).  <MI, NI, WM, WN, MP, NP, DEPTH, OCC>: CTA tile
// 8*MI*WM x 8*NI*WN, each warp's MI x NI sub-tiles of 8x8 processed MP x NP at a time, DEPTH-stage register
// prefetch ring, OCC CTAs per SM targeted.
typedef void (*gj_kernel_t)(GjStepParams);
struct GjVariant {
    int id;
    gj_kernel_t fn;
    int TM, TN, smem_full, smem_ext, m3;
    gj_kernel_t fn_lean;          // instance without the in-kernel inverter and the alternative column-block paths (default variants only)
    int smem_lean;
};
template <int MI, int NI, int WM, int WN, int MP, int NP, int DEPTH, int OCC, bool M3 = false>
static GjVariant gj_variant(int id) {
    typedef GjStepCfg<MI, NI, WM, WN> C;
    static_assert(C::THREADS == GjCfg::THREADS, "all variants use 256 threads");
    return {id, gj_step_kernel<MI, NI, WM, WN, MP, NP, DEPTH, OCC, M3>, C::TM, C::TN, M3 ? C::SMEM3 : C::SMEM, M3 ? C::SMEM_EXT3 : C::SMEM_EXT, M3 ? 1 : 0,
            (id == 3 || id == 12 || id == 4) ? gj_step_kernel<MI, NI, WM, WN, MP, NP, DEPTH, OCC, M3, true> : (gj_kernel_t) nullptr,
            M3 ? C::SMEM_LEAN3 : C::SMEM_LEAN};
}
static const std::vector<GjVariant>& gj_variants() {
    static const std::vector<GjVariant> v = {
        gj_variant<4, 2, 2, 4, 1, 2, 1, 2>(3),     // default: 64x64 tile, 4 row passes, rolled pass and k loops
        gj_variant<4, 2, 2, 4, 2, 2, 1, 2>(0),     // 2 row passes (1.3% slower with the self-driven service, 1.3% faster without)
        gj_variant<2, 2, 2, 4, 2, 2, 1, 2>(1),     // 32x64 tiles (512 CTAs)
        gj_variant<4, 2, 2, 4, 4, 2, 1, 2>(2),     // whole warp tile in one pass (round-1 original)
        gj_variant<4, 2, 2, 4, 1, 2, 1, 3>(4),     // default shape at 3 CTAs/SM
        gj_variant<4, 2, 2, 4, 1, 1, 4, 3>(5),     // 8 passes, 4-deep prefetch
        gj_variant<4, 2, 2, 4, 1, 2, 2, 2>(6),     // 4 passes, 2-deep prefetch
        gj_variant<4, 2, 2, 4, 1, 1, 2, 3>(7),
        gj_variant<4, 2, 2, 4, 1, 1, 1, 2>(8),     // 8 passes
        gj_variant<4, 2, 2, 4, 2, 1, 1, 2>(9),     // 4 column-split passes
        gj_variant<8, 2, 2, 4, 1, 2, 1, 2>(10),    // 128x64 tiles
        gj_variant<8, 2, 2, 4, 2, 2, 1, 2>(11),
        gj_variant<4, 2, 2, 4, 1, 2, 1, 2, true>(12),     // default shape, three-multiplication complex products (6 DMMAs per k-step instead of 8)
        gj_variant<4, 2, 2, 4, 2, 2, 1, 2, true>(13),     // 2 row passes, three-multiplication products
    };
    return v;
}
static const GjVariant& gj_pick(int id) {
    for (const GjVariant& v : gj_variants())
        if (v.id == id) return v;
    return gj_variants()[0];
}

static void configure_gj_variants() {
    static std::atomic<unsigned long long> configured{0};
    hz_once_per_device(configured, [&]() {
        for (const GjVariant& v : gj_variants()) {
            cudaFuncSetAttribute(v.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, v.smem_full);
            cudaFuncSetAttribute(v.fn, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            if (v.fn_lean) {
                cudaFuncSetAttribute(v.fn_lean, cudaFuncAttributeMaxDynamicSharedMemorySize, v.smem_full);
                cudaFuncSetAttribute(v.fn_lean, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
            }
        }
    });
}

static int launch_invert_fused(hz_ctx* h, cplx* slot, int chain, cudaStream_t st) {
    const int b = h->b;
    const int nsteps = (b + GJ_NB - 1) / GJ_NB;
    // option gemm_3m: the three-multiplication twins of the default (12) and the 2-row-pass (13) update tile
    const GjVariant& var = gj_pick((h->gemm_3m & 2) && h->gj_tile == 3 ? 12 : ((h->gemm_3m & 2) && h->gj_tile == 0 ? 13 : h->gj_tile));
    gj_kernel_t kfn = var.fn;
    configure_gj_variants();
    const int TMr = var.TM, TNr = var.TN;
    const int smem_full = var.smem_full, smem_ext = var.smem_ext;
    cplx* X[2] = {slot, h->Scratch[chain]};
    int cur = gj_start_buffer(h);
    cplx* Rb[2] = {h->Rbuf[chain], h->Rbuf[chain] + (size_t)GJ_NB * b};
    cplx* Cb[2] = {h->Cbuf[chain], h->Cbuf[chain] + (size_t)GJ_NB * b};
    const int tiles_m = (b + TMr - 1) / TMr, tiles_n = (b + TNr - 1) / TNr;
    GjStepParams p = {};
    p.b = b; p.err = h->d_err; p.tiles_n = tiles_n;
    p.trace = nullptr;
    const int max_grid = nsteps + 1 + tiles_m * tiles_n;
    const bool tracing = h->gj_trace && h->trace_now;
    if (tracing) {
        if (!h->d_trace[chain]) HZ_CUDA(h, cudaMalloc((void**)&h->d_trace[chain], (size_t)(nsteps + 1) * max_grid * 16 * sizeof(long long)));
        HZ_CUDA(h, cudaMemsetAsync(h->d_trace[chain], 0, (size_t)(nsteps + 1) * max_grid * 16 * sizeof(long long), st));
        h->trace_steps = nsteps + 1;
        h->trace_grid = max_grid;
    }
    for (int k = -1; k < nsteps; ++k) {
        if (tracing) p.trace = h->d_trace[chain] + (size_t)(k + 1) * max_grid * 16;
        p.k = k;
        p.Ain = X[cur];
        p.Aout = X[1 - cur];
        p.R = Rb[k & 1]; p.C = Cb[k & 1];
        p.Rn = Rb[(k + 1) & 1]; p.Cn = Cb[(k + 1) & 1];
        if (var.m3) {
            // operand-sum planes of the three-multiplication tiles: in the (otherwise unused) third panel slot of this chain
            p.lds = (b + 1) & ~1;
            double* Rs0 = reinterpret_cast<double*>(h->Rbuf[chain] + (size_t)2 * GJ_NB * b);
            double* Cs0 = reinterpret_cast<double*>(h->Cbuf[chain] + (size_t)2 * GJ_NB * b);
            double* RsP[2] = {Rs0, Rs0 + (size_t)GJ_NB * p.lds};
            double* CsP[2] = {Cs0, Cs0 + (size_t)GJ_NB * b};
            p.Rs = RsP[k & 1]; p.Cs = CsP[k & 1];
            p.Rns = RsP[(k + 1) & 1]; p.Cns = CsP[(k + 1) & 1];
        }
        p.npanel = (k + 1 < nsteps) ? nsteps + 1 : 0;      // inverter CTA + one CTA per column block
        p.Pg = h->Pg[chain] + (size_t)((k + 1) & 1) * GJ_TILE;
        p.flag = h->d_flag + chain;
        p.seq = ++h->seq_chain[chain];
        const int ntiles = k >= 0 ? tiles_m * tiles_n : 0;
        // inverter service: launches k >= 0 leave the pivot-block inverse to the service CTA; the request for
        // launch k+1 (inputs = this launch's outputs) is posted by this launch's last CTA to finish
        const bool svc = h->svc_on[chain];
        const bool self_driven = svc && h->gj_service == 2;       // the service walks the steps of a block row on its own
        p.ext_inverter = (svc && k >= 0 && p.npanel > 0) ? 1 : 0;
        p.post_next = (svc && k + 2 < nsteps && (!self_driven || k < 0)) ? 1 : 0;
        p.mailbox = nullptr; p.mailbox2 = nullptr; p.mail_flag = nullptr; p.done_ctr = nullptr; p.done_target = 0;
        p.Tg = nullptr; p.colflag = nullptr; p.tileflag = nullptr;
        if (self_driven && k >= 0 && k + 2 < nsteps) {            // launch k feeds the request for pivot k+2
            p.Tg = h->d_Tg + ((size_t)chain * 2 + (k & 1)) * GJ_TILE;
            p.colflag = h->d_cflag + chain * 2;
            p.tileflag = h->d_cflag + chain * 2 + 1;
        }
        // column-block CTAs spend most of their life waiting for the inverse: let them process the last update tiles
        // meanwhile (needs the full shared-memory layout: T + a tile's staging buffers)
        p.ntiles = ntiles;
        p.col_per = (h->gj_colper > 1 && k >= 0) ? 2 : 1;       // column blocks per column-block CTA (the k = -1 launch has slots to spare)
        p.col_pair = (h->gj_colpair && k >= 0 && p.npanel > 0 && !h->gj_coltile && h->gj_order == 0) ? 1 : 0;      // two blocks per CTA, side by side
        if (p.col_pair) p.col_per = 2;
        const int ncolcta = p.npanel > 0 ? (p.npanel - 1 + p.col_per - 1) / p.col_per : 0;
        p.col_tiles = (h->gj_coltile && k >= 0 && p.npanel > 0 && h->gj_order == 0 && p.col_per == 1) ? 1 : 0;
        p.crit_first = (h->gj_crit && self_driven && !p.col_tiles) ? 1 : 0;
        p.col_slow = h->gj_colslow;
        const int nfused = p.col_tiles ? std::min(ncolcta, ntiles) : 0;
        const int grid_k = (p.npanel > 0 ? 1 - p.ext_inverter + ncolcta : 0) + ntiles - nfused;
        if (p.post_next) {
            p.next.Ain = k >= 0 ? X[1 - cur] : X[cur];
            p.next.C = Cb[(k + 1) & 1];
            p.next.R = Rb[(k + 1) & 1];
            p.next.Pg = h->Pg[chain] + (size_t)((k + 2) & 1) * GJ_TILE;
            p.next.flag = h->d_flag + chain;
            p.next.b = b; p.next.k = k + 1; p.next.seq = h->seq_chain[chain] + 1; p.next.quit = 0;
            // diagnostics: the service stamps its phases into the slot the (absent) inverter CTA of launch k+1 would use
            p.next.trace = tracing ? h->d_trace[chain] + ((size_t)(k + 2) * max_grid + (max_grid - 1)) * 16 : nullptr;
            p.mailbox = h->d_mail + chain;
            if (self_driven) {
                GjBlockJob& j = p.next2;
                j.X[0] = X[0]; j.X[1] = X[1];
                j.Cb[0] = Cb[0]; j.Cb[1] = Cb[1]; j.Rb[0] = Rb[0]; j.Rb[1] = Rb[1];
                j.Pg = h->Pg[chain];
                j.Tg = h->d_Tg + (size_t)chain * 2 * GJ_TILE;
                j.flag = h->d_flag + chain;
                j.colflag = h->d_cflag + chain * 2;
                j.tileflag = h->d_cflag + chain * 2 + 1;
                j.b = b; j.nsteps = nsteps; j.cur0 = cur; j.seq_m1 = h->seq_chain[chain];
                j.seq = h->seq_chain[chain]; j.quit = 0;            // mailbox sequence: the k = -1 launch's own (unique per block row)
                // diagnostics: request L is stamped into the slot the (absent) inverter CTA of launch L would use
                j.trace = tracing ? h->d_trace[chain] + ((size_t)max_grid + (max_grid - 1)) * 16 : nullptr;
                j.trace_stride = (long long)max_grid * 16;
                p.mailbox2 = h->d_mail2 + chain;
            }
            p.mail_flag = h->d_mail_flag + chain;
            p.done_ctr = h->d_done + chain;
            h->done_total[chain] += (unsigned long long)grid_k;
            p.done_target = h->done_total[chain];
        }
        {
            const int grid = grid_k;
            p.order = h->gj_order;
            p.inv_bid = h->gj_inv >= 0 ? (h->gj_inv < grid ? h->gj_inv : 0) : (grid > 148 && grid <= 295) ? 147 : 0;
        }
        bool armed = false;
        if (k >= 0) prof_begin(h, 1, st, armed);
        p.pdl = (h->gj_pdl && k >= 0) ? 1 : 0;
        int smem_bytes = ((p.ext_inverter || p.npanel == 0) && !p.col_tiles) ? smem_ext : smem_full;   // no inverter CTA and no fused tiles: 4 tiles suffice
        if (p.col_pair && smem_bytes < GJ_COLPAIR_SMEM) smem_bytes = GJ_COLPAIR_SMEM;
        // the lean instance serves the launches of the default configuration that have no inverter CTA
        const bool lean = h->gj_lean && var.fn_lean && (p.ext_inverter || p.npanel == 0) && !tracing && p.col_per == 1 && !p.col_pair && !p.col_slow &&
                          !p.col_tiles && p.order == 0 && !p.pdl;
        gj_kernel_t kuse = lean ? var.fn_lean : kfn;
        if (lean) smem_bytes = var.smem_lean;
        if (p.pdl) HZ_LAUNCH_PDL(kuse, dim3(grid_k), dim3(GjCfg::THREADS), smem_bytes, st, p);
        else HZ_LAUNCH(kuse, dim3(grid_k), dim3(GjCfg::THREADS), smem_bytes, st, p);
        if (k >= 0) prof_end(h, 1, st, armed);
        HZ_CHECK_LAUNCH(h);
        if (k >= 0) cur ^= 1;
    }
    return HZ_OK;
}

// gj_mode 3 / 4: the dependence-counter kernels (hz_factor.cuh: gj_block_kernel, gj_pair_kernel)
typedef GjStepCfg<4, 2, 2, 4> GjBlkCfg;

static int fill_block_params(hz_ctx* h, cplx* slot, int chain, cudaStream_t st, GjBlockParams& q) {
    const int b = h->b;
    const int nsteps = (b + GJ_NB - 1) / GJ_NB;
    const int tiles_m = (b + GjBlkCfg::TM - 1) / GjBlkCfg::TM, tiles_n = (b + GjBlkCfg::TN - 1) / GjBlkCfg::TN, ntiles = tiles_m * tiles_n;
    const size_t need = sizeof(int) * (size_t)(4 + 4 * (nsteps + 2) + ntiles);
    if (h->sync_bytes < need) {
        HZ_CUDA(h, cudaStreamSynchronize(h->stream1));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream2));
        for (int c = 0; c < 2; ++c) { free_dev(h->d_sync[c]); HZ_CUDA(h, cudaMalloc((void**)&h->d_sync[c], need)); }
        h->sync_bytes = need;
    }
    HZ_CUDA(h, cudaMemsetAsync(h->d_sync[chain], 0, need, st));
    const bool svc = h->svc_on[chain] && h->gj_service == 2;
    q = GjBlockParams();
    q.X[0] = slot; q.X[1] = h->Scratch[chain];
    for (int i = 0; i < 3; ++i) { q.Rb[i] = h->Rbuf[chain] + (size_t)i * GJ_NB * b; q.Cb[i] = h->Cbuf[chain] + (size_t)i * GJ_NB * b; }
    q.Pg = h->Pg[chain];
    q.flag = h->d_flag + chain;
    q.cur0 = gj_start_buffer(h);
    q.seq_m1 = ++h->seq_chain[chain];
    h->seq_chain[chain] += nsteps;                       // step k publishes / waits for seq_m1 + 1 + k
    q.b = b; q.nsteps = nsteps; q.tiles_m = tiles_m; q.tiles_n = tiles_n;
    q.svc = svc ? 2 : 0;
    q.err = h->d_err;
    q.ticket = (unsigned*)h->d_sync[chain];
    q.hint = h->d_sync[chain] + 1;
    q.st = h->d_sync[chain] + 4;                          // 16-byte aligned: 4 ints per step, entry k + 1 = step k
    q.panel_done = q.st; q.tiles_finished = q.st + 3;     // (aliases, stride 4)
    q.tile_done = q.st + 4 * (nsteps + 2);
    if (svc) {
        GjBlockJob& j = q.job;
        j.X[0] = q.X[0]; j.X[1] = q.X[1];
        for (int i = 0; i < 3; ++i) { j.Cb[i] = q.Cb[i]; j.Rb[i] = q.Rb[i]; }
        j.nbuf = 3;
        j.Pg = h->Pg[chain];
        j.Tg = h->d_Tg + (size_t)chain * 2 * GJ_TILE;
        j.flag = h->d_flag + chain;
        j.colflag = h->d_cflag + chain * 2;
        j.tileflag = h->d_cflag + chain * 2 + 1;
        j.b = b; j.nsteps = nsteps; j.cur0 = q.cur0; j.seq_m1 = q.seq_m1; j.seq = q.seq_m1; j.quit = 0;
        q.mailbox2 = h->d_mail2 + chain;
        q.mail_flag = h->d_mail_flag + chain;
        q.Tg = h->d_Tg + (size_t)chain * 2 * GJ_TILE;
        q.colflag = j.colflag; q.tileflag = j.tileflag;
    }
    return HZ_OK;
}

// gj_mode 3: ONE launch per block row and chain
static int launch_invert_block(hz_ctx* h, cplx* slot, int chain, cudaStream_t st) {
    auto kfn = gj_block_kernel<4, 2, 2, 4, 1, 2, 1, 2>;
    static std::atomic<unsigned long long> configured{0};
    hz_once_per_device(configured, [&]() {
        cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, GjBlkCfg::SMEM);
        cudaFuncSetAttribute(kfn, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    });
    GjBlockParams q;
    int rc = fill_block_params(h, slot, chain, st, q);
    if (rc) return rc;
    const int ninv = q.svc ? 0 : 1, ntiles = q.tiles_m * q.tiles_n;
    const int grid = (q.nsteps + 1) + (q.nsteps - 1) * (ninv + q.nsteps + ntiles) + ntiles;
    bool armed = false;
    prof_begin(h, 1, st, armed);
    HZ_LAUNCH(kfn, dim3(grid), dim3(GjBlkCfg::THREADS), GjBlkCfg::SMEM, st, q);
    prof_end(h, 1, st, armed);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

// gj_mode 4: one persistent grid for the current block rows of BOTH chains (slot1 == nullptr: one chain only)
static int launch_invert_pair(hz_ctx* h, cplx* slot0, int chain0, cplx* slot1, int chain1, cudaStream_t st) {
    auto kfn = gj_pair_kernel<4, 2, 2, 4, 1, 2, 1, 2>;
    const int smem = GjBlkCfg::SMEM + 16;
    static std::atomic<unsigned long long> configured{0};
    hz_once_per_device(configured, [&]() {
        cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        cudaFuncSetAttribute(kfn, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    });
    GjPairParams pp;
    pp.nchains = slot1 ? 2 : 1;
    int rc = fill_block_params(h, slot0, chain0, st, pp.q[0]);
    if (rc) return rc;
    if (slot1 && (rc = fill_block_params(h, slot1, chain1, st, pp.q[1]))) return rc;
    if (!slot1) pp.q[1] = pp.q[0];
#ifdef HZ_EMU
    const int grid = 1;                                  // the emulation runs CTAs one after the other: one CTA walks the whole item list
#else
    const int grid = 2 * h->num_sms;                     // two CTAs per SM; the service CTAs' SMs take none, the surplus CTAs simply find the queues empty
#endif
    bool armed = false;
    prof_begin(h, 1, st, armed);
    HZ_LAUNCH(kfn, dim3(grid), dim3(GjBlkCfg::THREADS), smem, st, pp);
    prof_end(h, 1, st, armed);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

// v3: delayed updates -- launch sequence P0 | E O | E O ... (see gj_step2_kernel)
typedef GjStep2Cfg<4, 2, 2, 4, 3> Gj2Cfg;

static int gj2_start_buffer(const hz_ctx* h) {
    const int nsteps = (h->b + GJ_NB - 1) / GJ_NB;
    return ((nsteps + 1) / 2) % 2;                  // one ping-pong per O launch; 0: slot, 1: scratch
}

static int launch_invert_delayed(hz_ctx* h, cplx* slot, int chain, cudaStream_t st) {
    const int b = h->b, NB = GJ_NB;
    const int nsteps = (b + NB - 1) / NB, npairs = (nsteps + 1) / 2;
    auto kfn = gj_step2_kernel<4, 2, 2, 4, 3>;
    static std::atomic<unsigned long long> configured{0};
    hz_once_per_device(configured, [&]() { cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Gj2Cfg::SMEM); });
    cplx* X[2] = {slot, h->Scratch[chain]};
    int cur = gj2_start_buffer(h);
    cplx* RRp[2] = {h->Rbuf[chain], h->Rbuf[chain] + (size_t)2 * NB * b};
    cplx* CCp[2] = {h->Cbuf[chain], h->Cbuf[chain] + (size_t)2 * NB * b};
    const int tiles_m = (b + Gj2Cfg::TM - 1) / Gj2Cfg::TM, tiles_n = (b + Gj2Cfg::TN - 1) / Gj2Cfg::TN;
    const int ntiles = tiles_m * tiles_n, npan = nsteps + 1;
    auto kb_of = [&](int k) { return (b - k * NB) < NB ? (b - k * NB) : NB; };
    int panel_seq = 0, launch_idx = 0;
    const int max_grid = npan + ntiles;
    const bool tracing = h->gj_trace && h->trace_now;
    if (tracing) {
        const size_t n = (size_t)(2 * npairs + 1) * max_grid * 16 * sizeof(long long);
        if (!h->d_trace[chain]) HZ_CUDA(h, cudaMalloc((void**)&h->d_trace[chain], n));
        HZ_CUDA(h, cudaMemsetAsync(h->d_trace[chain], 0, n, st));
        h->trace_steps = 2 * npairs + 1;
        h->trace_grid = max_grid;
    }
    auto launch = [&](GjStep2Params& p, bool count_prof) -> int {
        p.b = b; p.err = h->d_err; p.tiles_n = tiles_n;
        p.npanel = p.do_panel ? npan : 0;
        const int grid = p.npanel + (p.do_update ? ntiles : 0);
        p.inv_bid = (grid > 148 && grid <= 295) ? 147 : 0;
        p.Pg = h->Pg[chain] + (size_t)(panel_seq & 1) * GJ_TILE;
        p.flag = h->d_flag + chain;
        p.seq = ++h->seq_chain[chain];
        p.pdl = (h->gj_pdl && launch_idx > 0) ? 1 : 0;
        p.trace = tracing ? h->d_trace[chain] + (size_t)launch_idx * max_grid * 16 : nullptr;
        if (p.do_panel) ++panel_seq;
        ++launch_idx;
        bool armed = false;
        if (count_prof) prof_begin(h, 1, st, armed);
        if (p.pdl) HZ_LAUNCH_PDL(kfn, dim3(grid), dim3(Gj2Cfg::THREADS), Gj2Cfg::SMEM, st, p);
        else HZ_LAUNCH(kfn, dim3(grid), dim3(Gj2Cfg::THREADS), Gj2Cfg::SMEM, st, p);
        if (count_prof) prof_end(h, 1, st, armed);
        HZ_CHECK_LAUNCH(h);
        return HZ_OK;
    };
    int rc;
    {   // P0: panel 0 from the freshly formed S, nothing pending
        GjStep2Params p = {};
        p.Ain = X[cur]; p.Aout = nullptr; p.RR = RRp[0]; p.CC = CCp[0]; p.npend = 0;
        p.do_panel = 1; p.kn0 = 0; p.kbn = kb_of(0); p.Rn = RRp[0]; p.Cn = CCp[0]; p.do_update = 0;
        if ((rc = launch(p, false))) return rc;
    }
    for (int m = 0; m < npairs; ++m) {
        const int a = 2 * m, par = m & 1;
        const bool have_b = a + 1 < nsteps;
        if (have_b) {   // E: panel a+1 with one pending panel (a)
            GjStep2Params p = {};
            p.Ain = X[cur]; p.Aout = nullptr; p.RR = RRp[par]; p.CC = CCp[par];
            p.npend = 1; p.pk0[0] = a * NB; p.pkb[0] = kb_of(a);
            p.do_panel = 1; p.kn0 = (a + 1) * NB; p.kbn = kb_of(a + 1);
            p.Rn = RRp[par] + (size_t)NB * b; p.Cn = CCp[par] + NB; p.do_update = 0;
            if ((rc = launch(p, false))) return rc;
        }
        {   // O: rank-(kb_a + kb_b) trailing update + look-ahead panel a+2
            GjStep2Params p = {};
            p.Ain = X[cur]; p.Aout = X[1 - cur]; p.RR = RRp[par]; p.CC = CCp[par];
            p.npend = have_b ? 2 : 1;
            p.pk0[0] = a * NB; p.pkb[0] = kb_of(a);
            if (have_b) { p.pk0[1] = (a + 1) * NB; p.pkb[1] = kb_of(a + 1); }
            p.do_panel = (a + 2 < nsteps) ? 1 : 0;
            if (p.do_panel) { p.kn0 = (a + 2) * NB; p.kbn = kb_of(a + 2); }
            p.Rn = RRp[1 - par]; p.Cn = CCp[1 - par]; p.do_update = 1;
            if ((rc = launch(p, true))) return rc;
            cur ^= 1;
        }
    }
    return HZ_OK;
}

// ---- checkpointed storage -------------------------------------------------------------------------
struct ChainPos { int chain; i64 p, len; };      // chain 0: rows < mid (p = i), chain 1: rows > mid (p = nz-1-i), chain 2: the middle row
static ChainPos chain_pos(const hz_ctx* h, i64 i) {
    if (i < h->mid) return {0, i, h->mid};
    if (i > h->mid) return {1, (i64)h->nz - 1 - i, (i64)h->nz - 1 - h->mid};
    return {2, 0, 1};
}
static i64 chain_row(const hz_ctx* h, int chain, i64 p) { return chain == 0 ? p : (i64)h->nz - 1 - p; }
static bool is_stored(const hz_ctx* h, i64 i) {
    const int k = h->store_used;
    if (k <= 1) return true;
    const ChainPos c = chain_pos(h, i);
    return c.chain == 2 || c.p % k == k - 1 || c.p == c.len - 1;
}
static i64 slots_needed(i64 nz, i64 mid, int k) {
    if (k <= 1) return nz;
    const i64 ntop = mid, nbot = nz - 1 - mid;
    return (ntop + k - 1) / k + (nbot + k - 1) / k + 1 + 2 * (k - 1);
}
static i64 slot_of(const hz_ctx* h, i64 i) {
    const int k = h->store_used;
    if (k <= 1) return i;
    const i64 ntop = h->mid, nbot = (i64)h->nz - 1 - h->mid;
    const i64 ctop = (ntop + k - 1) / k, cbot = (nbot + k - 1) / k;
    const ChainPos c = chain_pos(h, i);
    if (c.chain == 2) return ctop + cbot;
    if (c.p % k == k - 1 || c.p == c.len - 1) return (c.chain == 0 ? 0 : ctop) + c.p / k;
    return ctop + cbot + 1 + c.chain * (k - 1) + c.p % k;                 // recomputed on demand: the chain's temporaries
}

// complex64 storage of block i: interleaved (b*b cplxf) or, in tf32 mode, planar (re plane | im plane, b x ldb64 floats each)
static i64 slot64_elems(const hz_ctx* h) { return h->tf32_active ? (i64)h->b * h->ldb64 : (i64)h->b * h->b; }   // in cplxf units (8 bytes)
static cplxf* block64(const hz_ctx* h, i64 i) { return h->Sinv64 + slot_of(h, i) * slot64_elems(h); }

// complex128 home of block i: its HBM slot (HZ_C128) or a slot of the chain's two-block window (HZ_C64)
static cplx* block128(hz_ctx* h, i64 i, int chain) {
    if (h->dtype == HZ_C64) return h->Ring[chain][i & 1];
    return h->Sinv + slot_of(h, i) * (i64)h->b * h->b;
}

// complex64 factorisation of one block: fused look-ahead Gauss-Jordan steps in FP32 (hz_factor_f32.cuh)
static int launch_invert_f32(hz_ctx* h, cplxf* slot, int chain, cudaStream_t st) {
    const int b = h->b;
    const int nsteps = (b + GJ_NB - 1) / GJ_NB;
    static std::atomic<unsigned long long> configured{0};
    hz_once_per_device(configured, [&]() { cudaFuncSetAttribute(gj_step_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GJF_SMEM); });
    cplxf* X[2] = {slot, h->Scratch64[chain]};
    int cur = gj_start_buffer(h);
    cplxf* Rb[2] = {h->Rf[chain], h->Rf[chain] + (size_t)GJ_NB * b};
    cplxf* Cb[2] = {h->Cf[chain], h->Cf[chain] + (size_t)GJ_NB * b};
    const int tiles_m = (b + GJF_TM - 1) / GJF_TM, tiles_n = (b + GJF_TN - 1) / GJF_TN;
    GjStepF32Params p;
    p.b = b; p.err = h->d_err; p.tiles_n = tiles_n;
    for (int k = -1; k < nsteps; ++k) {
        p.k = k;
        p.Ain = X[cur];
        p.Aout = X[1 - cur];
        p.R = Rb[k & 1]; p.C = Cb[k & 1];
        p.Rn = Rb[(k + 1) & 1]; p.Cn = Cb[(k + 1) & 1];
        p.npanel = (k + 1 < nsteps) ? nsteps + 1 : 0;
        p.Pg = h->Pgf[chain] + (size_t)((k + 1) & 1) * GJF_TILE;
        p.flag = h->d_flag + chain;
        p.seq = ++h->seq_chain[chain];
        const int ntiles = k >= 0 ? tiles_m * tiles_n : 0;
        const int grid = p.npanel + ntiles;
        p.inv_bid = (grid > 148 && grid <= 295) ? 147 : 0;
        bool armed = false;
        if (k >= 0) prof_begin(h, 1, st, armed);
        HZ_LAUNCH(gj_step_f32_kernel, dim3(grid), dim3(256), GJF_SMEM, st, p);
        if (k >= 0) prof_end(h, 1, st, armed);
        HZ_CHECK_LAUNCH(h);
        if (k >= 0) cur ^= 1;
    }
    return HZ_OK;
}

// Form S_i from its already-eliminated neighbour(s) ia / ib (block indices, -1: none) into the buffer
// the inversion starts from, and invert it into its home.  complex64 variant: everything in FP32 on
// the complex64 store, or (option c64_fp64_factor) in FP64 with the finished inverse rounded.
static int factor_block(hz_ctx* h, i64 i, i64 ia, i64 ib, int chain, cudaStream_t st) {
    const i64 nb2 = (i64)h->b * h->b;
    int rc;
    if (h->dtype == HZ_C64 && !h->c64_fp64_factor) {
        cplxf* slot = block64(h, i);
        cplxf* start = gj_start_buffer(h) ? h->Scratch64[chain] : slot;
        if ((rc = launch_schur<cplxf>(h, i, ia >= 0 ? block64(h, ia) : (const cplxf*)nullptr,
                                      ib >= 0 ? block64(h, ib) : (const cplxf*)nullptr, start, st))) return rc;
        return launch_invert_f32(h, slot, chain, st);
    }
    // gj_trace: 1 = trace every block (the last one of each chain is kept); t >= 2 = only block t-2 of the top
    // chain and its mirror image nz-1-(t-2) in the bottom chain (a concurrent pair in mid-factorisation)
    h->trace_now = h->gj_trace == 1 || (h->gj_trace >= 2 && (i == h->gj_trace - 2 || i == h->nz - 1 - (h->gj_trace - 2)));
    const cplx* Xa = ia >= 0 ? block128(h, ia, 0) : nullptr;      // top-chain blocks live in chain 0's window
    const cplx* Xb = ib >= 0 ? block128(h, ib, 1) : nullptr;
    cplx* slot = block128(h, i, chain);
    if (h->gj_mode == 2) {
        cplx* start = gj2_start_buffer(h) ? h->Scratch[chain] : slot;
        if ((rc = launch_schur<cplx>(h, i, Xa, Xb, start, st))) return rc;
        rc = launch_invert_delayed(h, slot, chain, st);
    } else if (h->gj_mode == 1 || h->gj_mode == 3 || h->gj_mode == 4) {      // (mode 4 reaches here only for single blocks: recomputation between checkpoints)
        cplx* start = gj_start_buffer(h) ? h->Scratch[chain] : slot;
        if ((rc = launch_schur<cplx>(h, i, Xa, Xb, start, st))) return rc;
        // one launch per block row unless tracing / a non-default tile variant / a one-step-per-launch service was asked for
        const bool block_mode = h->gj_mode == 3 && !h->gj_trace && h->gj_tile == 3 && h->gj_service != 1 && !h->gj_pdl && !h->gj_coltile && h->gj_colper <= 1 && !h->gj_order && h->gj_inv < 0;
        rc = block_mode ? launch_invert_block(h, slot, chain, st) : launch_invert_fused(h, slot, chain, st);
    } else {
        if ((rc = launch_schur<cplx>(h, i, Xa, Xb, slot, st))) return rc;
        rc = launch_invert_v1(h, slot, chain, st);
    }
    if (rc) return rc;
    if (h->dtype == HZ_C64) {
#ifndef HZ_EMU
        if (h->tf32_active)
            HZ_LAUNCH_EW(convert_planar_kernel, dim3(blocks_for(nb2, 256)), dim3(256), 0, st, (const cplx*)slot, (float*)block64(h, i), h->b, h->ldb64);
        else
#endif
        HZ_LAUNCH_EW(convert_c64_kernel, dim3(blocks_for(nb2, 256)), dim3(256), 0, st, (const cplx*)slot, block64(h, i), nb2);
        HZ_CHECK_LAUNCH(h);
    }
    return HZ_OK;
}

// gj_mode 4: Schur complements of the current block row of one or both chains, then ONE persistent grid inverts them together
static bool pair_mode(const hz_ctx* h) {
    return h->gj_mode == 4 && !(h->dtype == HZ_C64 && !h->c64_fp64_factor) && !h->gj_trace && h->gj_tile == 3 && h->gj_service != 1 && !h->gj_pdl &&
           !h->gj_coltile && h->gj_colper <= 1 && !h->gj_order && h->gj_inv < 0;
}
static int factor_pair(hz_ctx* h, i64 i0, i64 ia0, i64 ib0, int chain0, i64 i1, i64 ia1, i64 ib1, int chain1, cudaStream_t st) {
    const i64 nb2 = (i64)h->b * h->b;
    int rc;
    cplx* slot[2] = {nullptr, nullptr};
    const i64 ii[2] = {i0, i1}, ia[2] = {ia0, ia1}, ib[2] = {ib0, ib1};
    const int ch[2] = {chain0, chain1};
    for (int c = 0; c < 2; ++c) {
        if (ii[c] < 0) continue;
        const cplx* Xa = ia[c] >= 0 ? block128(h, ia[c], 0) : nullptr;
        const cplx* Xb = ib[c] >= 0 ? block128(h, ib[c], 1) : nullptr;
        slot[c] = block128(h, ii[c], ch[c]);
        cplx* start = gj_start_buffer(h) ? h->Scratch[ch[c]] : slot[c];
        if ((rc = launch_schur<cplx>(h, ii[c], Xa, Xb, start, st))) return rc;
    }
    if ((rc = launch_invert_pair(h, slot[0], ch[0], slot[1], ch[1], st))) return rc;
    if (h->dtype == HZ_C64)
        for (int c = 0; c < 2; ++c) {
            if (ii[c] < 0) continue;
#ifndef HZ_EMU
            if (h->tf32_active)
                HZ_LAUNCH_EW(convert_planar_kernel, dim3(blocks_for(nb2, 256)), dim3(256), 0, st, (const cplx*)slot[c], (float*)block64(h, ii[c]), h->b, h->ldb64);
            else
#endif
            HZ_LAUNCH_EW(convert_c64_kernel, dim3(blocks_for(nb2, 256)), dim3(256), 0, st, (const cplx*)slot[c], block64(h, ii[c]), nb2);
            HZ_CHECK_LAUNCH(h);
        }
    return HZ_OK;
}

int hz_set_option(hz_handle_t h, const char* key, double value) {
    if (!h || !key) return fail(h, HZ_EINVAL, "hz_set_option: NULL argument");
    if (!strcmp(key, "store_every") && (int)value == h->store_every) return HZ_OK;
    // every other option may change the launch sequence a captured factorisation graph holds
    if (strcmp(key, "probe_check") && strcmp(key, "probe_limit") && strcmp(key, "gj_trace_chain") && strcmp(key, "factor_graph")) ++h->opt_epoch;
    if (!strcmp(key, "factor_graph")) { h->factor_graph = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_mode")) { h->gj_mode = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_colslow")) { h->gj_colslow = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_colpair")) { h->gj_colpair = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_lean")) { h->gj_lean = (int)value; return HZ_OK; }
    if (!strcmp(key, "gemm_3m")) { h->gemm_3m = (int)value; h->factored = false; return HZ_OK; }
    if (!strcmp(key, "gj_trace")) { h->gj_trace = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_trace_chain")) { h->trace_chain = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_crit")) { h->gj_crit = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_pdl")) { h->gj_pdl = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_tile")) { h->gj_tile = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_colper")) { h->gj_colper = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_coltile")) { h->gj_coltile = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_service")) { h->gj_service = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_order")) { h->gj_order = (int)value; return HZ_OK; }
    if (!strcmp(key, "gj_inv")) { h->gj_inv = (int)value; return HZ_OK; }
    if (!strcmp(key, "store_every")) {
        if (value < 1 || value > 64) return fail(h, HZ_EINVAL, "hz_set_option: store_every must be in [1, 64]");
        if ((int)value != h->store_every) h->factored = false;
        h->store_every = (int)value;
        return HZ_OK;
    }
    if (!strcmp(key, "probe_check")) { h->probe_check = (int)value; return HZ_OK; }
    if (!strcmp(key, "probe_limit")) { h->probe_limit = value; return HZ_OK; }
    if (!strcmp(key, "gj_newton")) {
        const int v = (int)value;
#ifdef HZ_EMU
        hz_gj_newton = v;
#else
        HZ_CUDA(h, cudaSetDevice(h->device));
        HZ_CUDA(h, cudaMemcpyToSymbol(hz_gj_newton, &v, sizeof(int)));
#endif
        h->factored = false;
        return HZ_OK;
    }
    if (!strcmp(key, "tf32_sms")) { h->tf32_sms = (int)value; return HZ_OK; }
    if (!strcmp(key, "c64_tf32")) { h->c64_tf32 = (int)value; h->factored = false; return HZ_OK; }
    if (!strcmp(key, "c64_fp64_factor")) { h->c64_fp64_factor = (int)value; h->factored = false; return HZ_OK; }
    return fail(h, HZ_EINVAL, std::string("hz_set_option: unknown key ") + key);
}

#ifndef HZ_EMU
// CUDA loads kernels lazily, and loading one may wait for the device to drain -- which never happens while a
// persistent inverter-service CTA is resident (of this handle or, with several frequencies per GPU, of another handle
// being factored from another host thread).  So EVERY kernel of the library is force-loaded, once per device, before
// the first service starts: a kernel missing from this list shows up as "service did not answer" + a 4 s stall.
template <class K>
static void preload_kernel(K kfn) {
    cudaFuncAttributes attr;
    cudaFuncGetAttributes(&attr, kfn);
}
template <class TP>
static void preload_panel_kernels() {
    preload_kernel(couple_kernel<TP, 0>); preload_kernel(residual_kernel<TP, 0>); preload_kernel(gather_col_kernel<TP>);
    preload_kernel(residual_col_kernel<TP, 0>); preload_kernel(norm2_kernel<TP>); preload_kernel(axpy_kernel<TP>);
    preload_kernel(couple_kernel<TP, 1>); preload_kernel(residual_kernel<TP, 1>); preload_kernel(residual_col_kernel<TP, 1>);
    preload_kernel(couple_kernel<TP, 2>); preload_kernel(residual_kernel<TP, 2>); preload_kernel(residual_col_kernel<TP, 2>);
    preload_kernel(finalize_kernel<TP>); preload_kernel(scatter_coo_kernel<TP>); preload_kernel(spmm_csr_kernel<TP>);
    preload_kernel(spmm_percol_kernel<TP>); preload_kernel(spmm_percol_t_kernel<TP>); preload_kernel(gradient_kernel<TP>);
    preload_kernel(misfit_kernel<TP>);
}
static void preload_factor_kernels() {
    static std::atomic<unsigned long long> done{0};
    hz_once_per_device(done, []() {
    for (const GjVariant& v : gj_variants()) {
        preload_kernel(v.fn);
        if (v.fn_lean) preload_kernel(v.fn_lean);
    }
    preload_kernel(gj_block_kernel<4, 2, 2, 4, 1, 2, 1, 2>);
    preload_kernel(gj_pair_kernel<4, 2, 2, 4, 1, 2, 1, 2>);
    preload_kernel(schur_form_kernel<cplx>);
    preload_kernel(schur_form_kernel<cplxf>);
    preload_kernel(convert_c64_kernel); preload_kernel(convert_c128_kernel);
    preload_kernel(convert_planar_kernel); preload_kernel(unconvert_planar_kernel); preload_kernel(couple_planar_kernel);
    preload_kernel(cgemm_tf32_kernel<32>); preload_kernel(cgemm_tf32_kernel<64>); preload_kernel(cgemm_tf32_kernel<128>);
    preload_kernel(cgemm_f32_kernel); preload_kernel(gj_step_f32_kernel); preload_kernel(gj_panel_kernel);
    preload_kernel(gj_step2_kernel<4, 2, 2, 4, 3>);
    preload_kernel(gj_post_quit_kernel);
    preload_kernel(gj_inverter_service);
    preload_kernel(gj_inverter_service2);
    preload_kernel(gj_post_quit2_kernel);
    preload_kernel(node_terms_kernel); preload_kernel(assemble_mz_kernel); preload_kernel(eurus_pml_tables_kernel); preload_kernel(assemble_eurus_kernel);
    preload_kernel(nearest_index_kernel); preload_kernel(kaiser_taps_kernel);
    preload_kernel(stencil_xcorr_kernel); preload_kernel(assemble_mz_vjp_kernel);
    preload_kernel(stencil_apply_kernel); preload_kernel(assemble_mz_jvp_kernel);
    preload_panel_kernels<cplx>();
    preload_panel_kernels<cplxf>();
    zgemm_for_each_instance<0>([](auto kfn) { preload_kernel(kfn); });
    zgemm_for_each_instance<1>([](auto kfn) { preload_kernel(kfn); });
    zgemm_for_each_instance<2>([](auto kfn) { preload_kernel(kfn); });
    // the service kernels request > 48 KB of dynamic shared memory: a per-device attribute as well
    cudaFuncSetAttribute(gj_inverter_service, cudaFuncAttributeMaxDynamicSharedMemorySize, GJ_SERVICE_SMEM);
    cudaFuncSetAttribute(gj_inverter_service2, cudaFuncAttributeMaxDynamicSharedMemorySize, GJ_SERVICE_SMEM);
    cudaGetLastError();
    });
}
#endif

static int factor_attempt(hz_ctx* h, int64_t twist, int* herr_out) {
    if (!h) return fail(h, HZ_EINVAL, "hz_factor: NULL handle");
    if (!h->assembled) return fail(h, HZ_ESTATE, "hz_factor: call hz_assemble first");
    HZ_CUDA(h, cudaSetDevice(h->device));
    const int nz = h->nz, b = h->b;
    i64 mid = twist < 0 ? nz / 2 : twist;
    if (mid >= nz) mid = nz - 1;
    const size_t blk = (size_t)b * b * sizeof(cplx);
    const int kst = h->store_every < 1 ? 1 : h->store_every;
    const i64 nslots = slots_needed(nz, mid, kst);
    if ((h->Sinv || h->Sinv64) && nslots != h->nslots) {          // another twist / store_every than the allocation was made for
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream1));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream2));
        free_dev(h->Sinv);
        free_dev(h->Sinv64);
    }
    bool want_tf32 = false;
#ifndef HZ_EMU
    // With checkpointed factors (store_every > 1) the sweeps are dominated by the recomputation between checkpoints, and the
    // refinement sweep the tensor-core contraction needs would double it (C5: 49 s instead of 31 s per frequency): those
    // handles use the FFMA contraction, which stays within 1e-4 without refinement (c64_tf32 = 2 forces the tensor cores).
    want_tf32 = h->dtype == HZ_C64 && h->c64_fp64_factor && h->c64_tf32 && (kst == 1 || h->c64_tf32 >= 2) && t32_encoder() != nullptr;
#endif
    if (h->Sinv64 && want_tf32 != h->tf32_active) {
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        free_dev(h->Sinv64);
    }
    h->tf32_active = want_tf32;
    h->ldb64 = (b + 3) & ~3;
    h->nslots = nslots;
    h->store_used = kst;
    h->mid = mid;
    if (h->dtype == HZ_C64 && !h->Sinv64) {
        cudaError_t e = cudaMalloc((void**)&h->Sinv64, (size_t)slot64_elems(h) * sizeof(cplxf) * nslots);
#ifndef HZ_EMU
        if (e == cudaSuccess && h->tf32_active &&
            !t32_make_map(&h->mapA, (const float*)h->Sinv64, b, b, 2 * nslots, h->ldb64, T32_KS, T32_TM, false)) {
            free_dev(h->Sinv64);
            return fail(h, HZ_ECUDA, "hz_factor: cuTensorMapEncodeTiled failed for the block-inverse planes");
        }
#endif
        if (e != cudaSuccess) {
            char msg[256];
            snprintf(msg, sizeof msg, "hz_factor: cannot allocate %.2f GB of HBM for %lld complex64 block inverses of order %d (%s); option store_every > 1 keeps only every k-th",
                     (double)b * b * sizeof(cplxf) * nslots / 1e9, (long long)nslots, b, cudaGetErrorString(e));
            cudaGetLastError();
            return fail(h, HZ_ENOMEM, msg);
        }
        for (int k = 0; k < 2; ++k) {
            for (int q = 0; q < 2; ++q) HZ_CUDA(h, cudaMalloc((void**)&h->Ring[k][q], blk));
            HZ_CUDA(h, cudaMalloc((void**)&h->Scratch64[k], (size_t)b * b * sizeof(cplxf)));
            HZ_CUDA(h, cudaMalloc((void**)&h->Rf[k], 2 * (size_t)GJ_NB * b * sizeof(cplxf)));
            HZ_CUDA(h, cudaMalloc((void**)&h->Cf[k], 2 * (size_t)GJ_NB * b * sizeof(cplxf)));
            HZ_CUDA(h, cudaMalloc((void**)&h->Pgf[k], 2 * (size_t)GJF_TILE * sizeof(cplxf)));
        }
    }
    if (h->dtype == HZ_C128 && !h->Sinv) {
        cudaError_t e = cudaMalloc((void**)&h->Sinv, blk * nslots);
        if (e != cudaSuccess) {
            char msg[256];
            snprintf(msg, sizeof msg, "hz_factor: cannot allocate %.2f GB of HBM for %lld block inverses of order %d (%s); option store_every > 1 keeps only every k-th",
                     (double)blk * nslots / 1e9, (long long)nslots, b, cudaGetErrorString(e));
            cudaGetLastError();
            return fail(h, HZ_ENOMEM, msg);
        }
    }
    for (int k = 0; k < 2; ++k) {
        if (!h->Rbuf[k]) HZ_CUDA(h, cudaMalloc((void**)&h->Rbuf[k], 4 * (size_t)GJ_NB * b * sizeof(cplx)));   // 2 parities x 64 x b
        if (!h->Cbuf[k]) HZ_CUDA(h, cudaMalloc((void**)&h->Cbuf[k], 4 * (size_t)GJ_NB * b * sizeof(cplx)));
        if (!h->Scratch[k]) HZ_CUDA(h, cudaMalloc((void**)&h->Scratch[k], blk));
        if (!h->Pg[k]) HZ_CUDA(h, cudaMalloc((void**)&h->Pg[k], 2 * (size_t)GJ_TILE * sizeof(cplx)));
    }
    if (!h->d_flag) {
        HZ_CUDA(h, cudaMalloc((void**)&h->d_flag, 2 * sizeof(int)));
        HZ_CUDA(h, cudaMemsetAsync(h->d_flag, 0, 2 * sizeof(int), h->stream));
    }
    HZ_CUDA(h, cudaMemsetAsync(h->d_err, 0, sizeof(int), h->stream));
    h->factored = false;
    h->mid = mid;

    // fork: both chains run on internal streams (top: stream1, bottom: stream2) behind an event on the
    // caller's stream, launches interleaved so that neither chain starves behind the other's launch
    // queue.  The caller's stream only waits for the join, so several handles bound to the same caller
    // stream can be factored concurrently from different host threads (MultiFreq.prefactor).
    cudaStream_t s0 = h->stream1;
    HZ_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
    HZ_CUDA(h, cudaStreamWaitEvent(s0, h->ev_fork, 0));
    HZ_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
    const i64 ntop = mid, nbot = nz - 1 - mid;
    const i64 nmax = ntop > nbot ? ntop : nbot;
    const bool pairs = pair_mode(h);                                 // both chains' launches then go to s0
    cudaStream_t chain_stream[2] = {s0, pairs ? s0 : h->stream2};
    // inverter service: one persistent CTA per active chain (not under CPU emulation: it needs real concurrency;
    // not once this process has seen it fail to run beside the step kernels, e.g. under a profiler)
    bool want_svc = false;
#ifndef HZ_EMU
    want_svc = h->gj_service && !g_service_unavailable.load() && (h->gj_mode == 1 || h->gj_mode == 3 || h->gj_mode == 4) && (h->dtype == HZ_C128 || h->c64_fp64_factor) &&
               (b + GJ_NB - 1) / GJ_NB > 1;
    if (want_svc) {
        preload_factor_kernels();
        if (!h->d_mail) {
            HZ_CUDA(h, cudaMalloc((void**)&h->d_mail, 2 * sizeof(GjJob)));
            HZ_CUDA(h, cudaMalloc((void**)&h->d_mail_flag, 2 * sizeof(int)));
            HZ_CUDA(h, cudaMalloc((void**)&h->d_done, 2 * sizeof(unsigned long long)));
            HZ_CUDA(h, cudaMemsetAsync(h->d_mail, 0, 2 * sizeof(GjJob), h->stream));
            HZ_CUDA(h, cudaMemsetAsync(h->d_mail_flag, 0, 2 * sizeof(int), h->stream));
            HZ_CUDA(h, cudaMemsetAsync(h->d_done, 0, 2 * sizeof(unsigned long long), h->stream));
            HZ_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
            HZ_CUDA(h, cudaStreamWaitEvent(s0, h->ev_fork, 0));
            HZ_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
        }
        if (h->gj_service == 2 && !h->d_mail2) {
            HZ_CUDA(h, cudaMalloc((void**)&h->d_mail2, 2 * sizeof(GjBlockJob)));
            HZ_CUDA(h, cudaMalloc((void**)&h->d_Tg, 4 * (size_t)GJ_TILE * sizeof(cplx)));
            HZ_CUDA(h, cudaMalloc((void**)&h->d_cflag, 4 * sizeof(int)));
            HZ_CUDA(h, cudaMemsetAsync(h->d_mail2, 0, 2 * sizeof(GjBlockJob), h->stream));
            HZ_CUDA(h, cudaMemsetAsync(h->d_cflag, 0, 4 * sizeof(int), h->stream));
            HZ_CUDA(h, cudaEventRecord(h->ev_fork, h->stream));
            HZ_CUDA(h, cudaStreamWaitEvent(s0, h->ev_fork, 0));
            HZ_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork, 0));
        }
    }
#endif
    // A chain's service CTA is started behind an event on that chain's stream (so it cannot idle away its 4 s
    // budget while earlier work is queued) and only while the chain has blocks to factor: with unequal chains
    // (twist = 'source', or a small explicit twist) the top chain's service is stopped when the top chain
    // ends and restarted just before the middle block, instead of idling beside the longer bottom chain.
    auto start_service = [&](int c) -> int {
#ifndef HZ_EMU
        if (!want_svc || h->svc_on[c]) return HZ_OK;
        HZ_CUDA(h, cudaEventRecord(h->ev_svc[c], chain_stream[c]));
        HZ_CUDA(h, cudaStreamWaitEvent(h->svc_stream[c], h->ev_svc[c], 0));
        if (h->gj_service == 2)
            HZ_LAUNCH(gj_inverter_service2, dim3(1), dim3(256), GJ_SERVICE_SMEM, h->svc_stream[c], h->d_mail2 + c, h->d_mail_flag + c,
                      h->d_err, h->seq_chain[c]);
        else
            HZ_LAUNCH(gj_inverter_service, dim3(1), dim3(256), GJ_SERVICE_SMEM, h->svc_stream[c], h->d_mail + c, h->d_mail_flag + c,
                      h->d_err, h->seq_chain[c]);
        HZ_CHECK_LAUNCH(h);
        h->svc_on[c] = true;
#endif
        return HZ_OK;
    };
    auto stop_service = [&](int c) {                 // posted in stream order behind the chain's last launch
        if (!h->svc_on[c]) return;
        if (h->gj_service == 2)
            HZ_LAUNCH_EW(gj_post_quit2_kernel, dim3(1), dim3(1), 0, chain_stream[c], h->d_mail2 + c, h->d_mail_flag + c, ++h->seq_chain[c]);
        else
            HZ_LAUNCH_EW(gj_post_quit_kernel, dim3(1), dim3(1), 0, chain_stream[c], h->d_mail + c, h->d_mail_flag + c, ++h->seq_chain[c]);
        h->svc_on[c] = false;
    };
    auto run_chains = [&]() -> int {
        int rcs;
        if (ntop > 0 && (rcs = start_service(0))) return rcs;
        if (nbot > 0 && (rcs = start_service(1))) return rcs;
        for (i64 t = 0; t < nmax && pairs; ++t) {
            if (t == ntop && nbot > ntop + 8) stop_service(0);
            const bool h0 = t < ntop, h1 = t < nbot;
            const i64 i0 = t, i1 = nz - 1 - t;
            int rc;
            if (h0 && h1) rc = factor_pair(h, i0, i0 > 0 ? i0 - 1 : -1, -1, 0, i1, -1, i1 < nz - 1 ? i1 + 1 : -1, 1, s0);
            else if (h0) rc = factor_pair(h, i0, i0 > 0 ? i0 - 1 : -1, -1, 0, -1, -1, -1, 1, s0);
            else rc = factor_pair(h, i1, -1, i1 < nz - 1 ? i1 + 1 : -1, 1, -1, -1, -1, 0, s0);
            if (rc) return rc;
        }
        for (i64 t = 0; t < nmax && !pairs; ++t) {
            if (t == ntop && nbot > ntop + 8) stop_service(0);      // the top chain is done long before the bottom chain
            if (t < ntop) {
                const i64 i = t;
                int rc = factor_block(h, i, i > 0 ? i - 1 : -1, -1, 0, s0);
                if (rc) return rc;
            }
            if (t < nbot) {
                const i64 i = nz - 1 - t;
                int rc = factor_block(h, i, -1, i < nz - 1 ? i + 1 : -1, 1, h->stream2);
                if (rc) return rc;
            }
        }
        stop_service(1);
        HZ_CUDA(h, cudaEventRecord(h->ev_join, h->stream2));
        HZ_CUDA(h, cudaStreamWaitEvent(s0, h->ev_join, 0));
        if ((rcs = start_service(0))) return rcs;                    // no-op when it is still running
        if (pairs) return factor_pair(h, mid, mid > 0 ? mid - 1 : -1, mid < nz - 1 ? mid + 1 : -1, 0, -1, -1, -1, 1, s0);
        return factor_block(h, mid, mid > 0 ? mid - 1 : -1, mid < nz - 1 ? mid + 1 : -1, 0, s0);
    };
    // ---- CUDA graph (see hz_ctx::factor_graph): capture the launch sequence once, replay it afterwards ----------------------
    bool use_graph = false;
#ifndef HZ_EMU
    {
        const i64 nlaunch = (i64)nz * ((b + GJ_NB - 1) / GJ_NB + 2);
        const bool eligible = h->gj_mode == 1 && (h->dtype == HZ_C128 || h->c64_fp64_factor) && !h->gj_trace && !h->prof_on && !h->gj_pdl && kst == 1;
        use_graph = eligible && (h->factor_graph == 1 || (h->factor_graph < 0 && nlaunch <= 16384));
    }
    if (use_graph) {
        unsigned long long key = 1469598103934665603ULL;
        auto mix = [&](unsigned long long v) { key = (key ^ v) * 1099511628211ULL; };
        mix((unsigned long long)(uintptr_t)h->Sinv); mix((unsigned long long)(uintptr_t)h->Sinv64); mix((unsigned long long)(uintptr_t)h->coef);
        for (int c = 0; c < 2; ++c) {
            mix((unsigned long long)(uintptr_t)h->Scratch[c]); mix((unsigned long long)(uintptr_t)h->Rbuf[c]); mix((unsigned long long)(uintptr_t)h->Cbuf[c]);
            mix((unsigned long long)(uintptr_t)h->Pg[c]); mix((unsigned long long)(uintptr_t)h->Ring[c][0]); mix((unsigned long long)(uintptr_t)h->Ring[c][1]);
        }
        mix((unsigned long long)mid); mix((unsigned long long)nz); mix((unsigned long long)b); mix(h->opt_epoch); mix(want_svc ? 1 : 0);
        mix(h->tf32_active ? 1 : 0); mix((unsigned long long)h->dtype);
        h->fgraph_want = key;
        if (h->fgraph && key != h->fgraph_key) {
            cudaGraphExecDestroy(h->fgraph);
            h->fgraph = nullptr;
        }
        // auto: a handle that is factored once gains nothing from a capture (instantiating costs more than the launches it saves);
        // the second factorisation of the same buffers (a model update, the next iteration) is what gets captured
        if (h->factor_graph < 0 && key != h->fgraph_seen) {
            h->fgraph_seen = key;
            use_graph = false;
        }
    }
    if (use_graph) {
        const unsigned long long key = h->fgraph_want;
        if (!h->fgraph) {
            preload_factor_kernels();
            configure_gj_variants();
            HZ_CUDA(h, cudaStreamSynchronize(s0));                  // (pending work of the internal streams is not part of the graph)
            HZ_CUDA(h, cudaStreamBeginCapture(s0, cudaStreamCaptureModeThreadLocal));
            const long long launches_before = g_hz_launches.load();
            bool svc_used[2] = {false, false};
            auto body = [&]() -> int {
                // sequence numbers and completion counters restart from zero with every replay
                h->seq_chain[0] = h->seq_chain[1] = 0;
                h->done_total[0] = h->done_total[1] = 0;
                HZ_CUDA(h, cudaMemsetAsync(h->d_flag, 0, 2 * sizeof(int), s0));
                if (h->d_mail_flag) HZ_CUDA(h, cudaMemsetAsync(h->d_mail_flag, 0, 2 * sizeof(int), s0));
                if (h->d_done) HZ_CUDA(h, cudaMemsetAsync(h->d_done, 0, 2 * sizeof(unsigned long long), s0));
                if (h->d_cflag) HZ_CUDA(h, cudaMemsetAsync(h->d_cflag, 0, 4 * sizeof(int), s0));
                HZ_CUDA(h, cudaEventRecord(h->ev_fork2, s0));
                HZ_CUDA(h, cudaStreamWaitEvent(h->stream2, h->ev_fork2, 0));
                const int rc = run_chains();
                svc_used[0] = want_svc; svc_used[1] = want_svc && nbot > 0;
                stop_service(1);
                stop_service(0);
                if (rc) return rc;
                for (int c = 0; c < 2; ++c)
                    if (svc_used[c]) {
                        HZ_CUDA(h, cudaEventRecord(h->ev_svc_join[c], h->svc_stream[c]));
                        HZ_CUDA(h, cudaStreamWaitEvent(s0, h->ev_svc_join[c], 0));
                    }
                return HZ_OK;
            };
            const int rc = body();
            cudaGraph_t graph = nullptr;
            const cudaError_t ce = cudaStreamEndCapture(s0, &graph);
            const long long captured = g_hz_launches.load() - launches_before;
            g_hz_launches -= captured;                                   // nothing ran yet: replays add them
            if (rc) {
                if (graph) cudaGraphDestroy(graph);
                cudaGetLastError();
                return rc;
            }
            if (ce != cudaSuccess || !graph) {
                cudaGetLastError();
                return fail(h, HZ_ECUDA, (std::string("hz_factor: capturing the factorisation into a CUDA graph failed: ") + cudaGetErrorString(ce)).c_str());
            }
            const cudaError_t ie = cudaGraphInstantiate(&h->fgraph, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) {
                h->fgraph = nullptr;
                cudaGetLastError();
                return fail(h, HZ_ECUDA, (std::string("hz_factor: cudaGraphInstantiate failed: ") + cudaGetErrorString(ie)).c_str());
            }
            h->fgraph_key = key;
            h->fgraph_launches = captured;
            h->fgraph_replays = 0;
        }
        HZ_CUDA(h, cudaGraphLaunch(h->fgraph, s0));
        g_hz_launches += h->fgraph_launches;
        ++h->fgraph_replays;
    }
#endif
    if (!use_graph) {
        const int rc = run_chains();
        stop_service(1);
        stop_service(0);
        if (rc) {
            cudaStreamSynchronize(h->stream2);
            cudaStreamSynchronize(s0);
            cudaStreamSynchronize(h->stream);
            for (int c = 0; c < 2; ++c) cudaStreamSynchronize(h->svc_stream[c]);
            return rc;
        }
    }
    HZ_CUDA(h, cudaEventRecord(h->ev_join0, s0));
    HZ_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_join0, 0));
    int herr = 0;
    HZ_CUDA(h, cudaMemcpyAsync(&herr, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int c = 0; c < 2; ++c) HZ_CUDA(h, cudaStreamSynchronize(h->svc_stream[c]));
    *herr_out = herr;
    if (herr == 2) return fail(h, HZ_ECUDA, "hz_factor: the pivot-block inverter service did not answer (device-side wait timed out)");
    if (herr) return fail(h, HZ_ESINGULAR, "hz_factor: zero or non-finite pivot in a diagonal block (singular operator or NaN in the model)");
    h->factored = true;
    h->probe_pending = true;
    return HZ_OK;
}

int hz_factor(hz_handle_t h, int64_t twist) {
    int herr = 0;
    int rc = factor_attempt(h, twist, &herr);
    if (rc == HZ_ECUDA && herr == 2 && h && h->gj_service) {
        // The service CTA never got to run beside the step kernels (e.g. its stream shares a hardware
        // queue with the chain's stream).  Every device-side wait is bounded, so nothing hangs: fall back
        // to the in-kernel inverter for this handle and factor again.
        // Remembered for the whole process: whatever serialises the launches (a profiler, CUDA_LAUNCH_BLOCKING,
        // a sanitizer) will do so for every handle, and each failed attempt costs a device-side timeout.
        h->service_fallbacks += 1;
        const int fails = ++g_service_failures;
        const int saved = g_service_unavailable.exchange(1);       // this retry runs without the service
        if (fails == 1) fprintf(stderr, "zephyr_b200: pivot-block inverter service did not answer; this factorisation is redone with the in-kernel inverter\n");
        rc = factor_attempt(h, twist, &herr);
        if (fails < 2 && !saved) g_service_unavailable.store(0);
        else if (fails == 2) fprintf(stderr, "zephyr_b200: pivot-block inverter service failed twice in a row; using the in-kernel inverter in this process\n");
    } else if (rc == HZ_OK && h && h->gj_service && !g_service_unavailable.load()) {
        g_service_failures.store(0);
    }
    return rc;
}

int hz_get_block_inverse(hz_handle_t h, int64_t iz, void* out_host) {
    if (!h || !out_host) return fail(h, HZ_EINVAL, "hz_get_block_inverse: NULL argument");
    if (!h->factored) return fail(h, HZ_ESTATE, "hz_get_block_inverse: no factors");
    if (iz < 0 || iz >= h->nz) return fail(h, HZ_EINVAL, "hz_get_block_inverse: iz out of range");
    if (!is_stored(h, iz)) return fail(h, HZ_ESTATE, "hz_get_block_inverse: this block is not kept (store_every > 1); only checkpoints are");
    HZ_CUDA(h, cudaSetDevice(h->device));
    const i64 nb2 = (i64)h->b * h->b;
    if (h->dtype == HZ_C64 && h->tf32_active) {          // planar storage: interleave on the host
        std::vector<float> tmp((size_t)2 * h->b * h->ldb64);
        HZ_CUDA(h, cudaMemcpyAsync(tmp.data(), block64(h, iz), tmp.size() * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        float* o = (float*)out_host;
        const size_t plane = (size_t)h->b * h->ldb64;
        for (int r = 0; r < h->b; ++r)
            for (int c = 0; c < h->b; ++c) {
                o[2 * ((size_t)r * h->b + c)] = tmp[(size_t)r * h->ldb64 + c];
                o[2 * ((size_t)r * h->b + c) + 1] = tmp[plane + (size_t)r * h->ldb64 + c];
            }
        return HZ_OK;
    }
    if (h->dtype == HZ_C64)
        HZ_CUDA(h, cudaMemcpyAsync(out_host, block64(h, iz), (size_t)nb2 * sizeof(cplxf), cudaMemcpyDeviceToHost, h->stream));
    else
        HZ_CUDA(h, cudaMemcpyAsync(out_host, h->Sinv + slot_of(h, iz) * nb2, (size_t)nb2 * sizeof(cplx), cudaMemcpyDeviceToHost, h->stream));
    HZ_CUDA(h, cudaStreamSynchronize(h->stream));
    return HZ_OK;
}

// ---- substitution ----------------------------------------------------------------------------
// op: HZ_OP_N / T / H -- which operator's off-diagonal blocks couple (complex64 panels: N only, hz_solve_op)
template <class TP>
static int launch_couple(hz_ctx* h, i64 i, TP* X, i64 S, TP* Y, int use_self, double lo, double hi, cudaStream_t st, int zero_self, int op) {
    const int threads = S >= 128 ? 128 : (S >= 64 ? 64 : 32);
    dim3 grid((unsigned)((S + threads - 1) / threads), h->b, 1);
#ifndef HZ_EMU
    if (std::is_same<TP, cplxf>::value && h->tf32_active) {
        // planar, transposed FP32 right-hand side for the tensor-core GEMM; X_i zeroed when the GEMM's result replaces it
        const i64 ldk = h->ldb64;
        ++g_hz_launches;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)((S + 31) / 32), (unsigned)((h->b + 31) / 32), 1); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        cudaLaunchKernelEx(&cfg, couple_planar_kernel, (const cplx*)h->coef, h->nf, h->nx, h->nz, (int)i, (cplxf*)X, S, (float*)Y, ldk, (i64)S * ldk,
                           use_self, lo, hi, zero_self);
        HZ_CHECK_LAUNCH(h);
        return HZ_OK;
    }
#endif
    auto kfn = op == HZ_OP_T ? couple_kernel<TP, 1> : (op == HZ_OP_H ? couple_kernel<TP, 2> : couple_kernel<TP, 0>);
    HZ_LAUNCH_EW(kfn, grid, dim3(threads), 0, st, (const cplx*)h->coef, h->nf, h->nx, h->nz, (int)i, X, S, Y, use_self, lo, hi);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

// X_i <- beta X_i + alpha op(S_i^{-1}) Y on the FP64 tensor pipe (complex128; op N, T or H: S_i(A^T) = S_i(A)^T) ...
static int launch_block_gemm(hz_ctx* h, i64 i, const cplx* Y, cplx* X, i64 S, double alpha, int beta, cudaStream_t st, int op) {
    GemmParams p;
    p.A = h->Sinv + slot_of(h, i) * (i64)h->b * h->b; p.lda = h->b;
    p.B = Y; p.ldb = S;
    p.C = X + i * (i64)h->nx * S; p.ldc = S;
    p.M = h->b; p.N = (int)S; p.K = h->b;
    p.alpha = alpha; p.beta = beta;
    p.sub_c0 = p.sub_c1 = 0;
    p.row_nx = h->nf > 1 ? h->nx : 0;
    p.row_fs = h->N;
    bool armed;
    prof_begin(h, 0, st, armed);
    const bool m3 = (h->gemm_3m & 1) != 0;
    if (op == HZ_OP_T) zgemm_launch<1>(p, st, h->num_sms, -1, m3);
    else if (op == HZ_OP_H) zgemm_launch<2>(p, st, h->num_sms, -1, m3);
    else zgemm_launch<0>(p, st, h->num_sms, -1, m3);
    prof_end(h, 0, st, armed);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}
// ... or in FP32 on complex64 factors and panels (op N only: hz_solve_op rejects T / H for complex64 handles)
static int launch_block_gemm(hz_ctx* h, i64 i, const cplxf* Y, cplxf* X, i64 S, double alpha, int beta, cudaStream_t st, int /*op*/) {
#ifndef HZ_EMU
    if (h->tf32_active) {
        Tf32Params tp;
        tp.M = h->b; tp.N = (int)S; tp.K = h->b;
        tp.a_plane0 = (int)(2 * slot_of(h, i));
        tp.y_plane0 = 0;
        tp.C = X + i * (i64)h->nx * S; tp.ldc = S;
        tp.alpha = (float)alpha;
        tp.row_nx = h->nf > 1 ? h->nx : 0;
        tp.row_fs = h->N;
        tp.k_per_split = 0;
        tp.dbg = nullptr; tp.mode = 0; tp.force_split = 0;
        bool armed;
        prof_begin(h, 0, st, armed);
        cgemm_tf32_launch(h->mapA, h->mapY[(const cplx*)Y == h->Ybuf[1] ? 1 : 0], tp, h->tf32_sms > 0 ? h->tf32_sms : h->num_sms, st);     // beta: X_i already holds beta * X_i
        prof_end(h, 0, st, armed);
        HZ_CHECK_LAUNCH(h);
        return HZ_OK;
    }
#endif
    CGemmParams p;
    p.A = block64(h, i); p.lda = h->b;
    p.B = Y; p.ldb = S;
    p.C = X + i * (i64)h->nx * S; p.ldc = S;
    p.M = h->b; p.N = (int)S; p.K = h->b;
    p.alpha = (float)alpha; p.beta = beta;
    p.row_nx = h->nf > 1 ? h->nx : 0;
    p.row_fs = h->N;
    bool armed;
    prof_begin(h, 0, st, armed);
    cgemm_f32_launch(p, st);
    prof_end(h, 0, st, armed);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

// Checkpointed factors: recompute the block inverses of segment j of `chain` that are not kept (all but the segment's
// last block) from the checkpoint preceding the segment, into the chain's temporaries.  Runs on the sweep's own
// stream with the in-kernel inverter (the service is a factorisation-time helper).
static int recompute_segment(hz_ctx* h, int chain, i64 j, cudaStream_t st) {
    const int k = h->store_used;
    const i64 len = chain == 0 ? h->mid : (i64)h->nz - 1 - h->mid;
    const i64 p0 = j * k, p1 = std::min<i64>((j + 1) * k - 1, len - 1);       // p1: the segment's checkpoint
    const i64 nb2 = (i64)h->b * h->b;
    for (i64 p = p0; p < p1; ++p) {
        const i64 i = chain_row(h, chain, p), prev = p > 0 ? chain_row(h, chain, p - 1) : -1;
        if (h->dtype == HZ_C64 && h->c64_fp64_factor && p == p0 && prev >= 0) {
            // the chain continues in complex128: widen the preceding (complex64) checkpoint into the chain's window
#ifndef HZ_EMU
            if (h->tf32_active)
                HZ_LAUNCH_EW(unconvert_planar_kernel, dim3(blocks_for(nb2, 256)), dim3(256), 0, st, (const float*)block64(h, prev), h->Ring[chain][prev & 1], h->b, h->ldb64);
            else
#endif
            HZ_LAUNCH_EW(convert_c128_kernel, dim3(blocks_for(nb2, 256)), dim3(256), 0, st, (const cplxf*)block64(h, prev), h->Ring[chain][prev & 1], nb2);
            HZ_CHECK_LAUNCH(h);
        }
        const int rc = factor_block(h, i, chain == 0 ? prev : -1, chain == 1 ? prev : -1, chain, st);
        if (rc) return rc;
    }
    return HZ_OK;
}

// X <- op(A)^{-1} X (no premul / conjugation); zf/zl: first/last block row with non-zero rhs.  The Schur complements of
// A^T (A^H) are S_i^T (S_i^H) for both chains and the middle block, so every op runs the same two sweeps on the same
// factors: op(S_i^{-1}) in the GEMMs and the op(A) stencil in the coupling.
template <class TP>
static int solve_inplace(hz_ctx* h, TP* X, i64 S, i64 zf, i64 zl, int op) {
    const i64 nz = h->nz, mid = h->mid;
    const int k = h->store_used;
    if (zf < 0 || zf >= nz) zf = 0;
    if (zl < 0 || zl >= nz) zl = nz - 1;
    if (zl < zf) { zf = 0; zl = nz - 1; }
    cudaStream_t st[2] = {h->stream, h->stream2};
    TP* Y[2] = {(TP*)h->Ybuf[0], (TP*)h->Ybuf[1]};
    const i64 len[2] = {mid, nz - 1 - mid};
    int rc;
    HZ_CUDA(h, cudaEventRecord(h->ev_fork, st[0]));
    HZ_CUDA(h, cudaStreamWaitEvent(st[1], h->ev_fork, 0));
    // forward elimination, top chain (downwards) and bottom chain (upwards); chain position p = i (top), nz-1-i (bottom)
    const bool top_fwd = zf < mid, bot_fwd = zl > mid;
    const i64 pfirst[2] = {zf, nz - 1 - zl};
    for (int c = 0; c < 2; ++c) {
        for (i64 p = pfirst[c]; p < len[c]; ++p) {
            if (k > 1 && (p == pfirst[c] || p % k == 0) && (rc = recompute_segment(h, c, p / k, st[c]))) return rc;
            const i64 i = chain_row(h, c, p);
            const double sg = p > pfirst[c] ? -1.0 : 0.0;
            if ((rc = launch_couple<TP>(h, i, X, S, Y[c], 1, c == 0 ? sg : 0.0, c == 0 ? 0.0 : sg, st[c], 1, op))) return rc;
            if ((rc = launch_block_gemm(h, i, (const TP*)Y[c], X, S, 1.0, 0, st[c], op))) return rc;
        }
    }
    HZ_CUDA(h, cudaEventRecord(h->ev_join, st[1]));
    HZ_CUDA(h, cudaStreamWaitEvent(st[0], h->ev_join, 0));
    // middle block
    if ((rc = launch_couple<TP>(h, mid, X, S, Y[0], 1, top_fwd ? -1.0 : 0.0, bot_fwd ? -1.0 : 0.0, st[0], 1, op))) return rc;
    if ((rc = launch_block_gemm(h, mid, (const TP*)Y[0], X, S, 1.0, 0, st[0], op))) return rc;
    // back substitution outwards from the middle
    HZ_CUDA(h, cudaEventRecord(h->ev_fork, st[0]));
    HZ_CUDA(h, cudaStreamWaitEvent(st[1], h->ev_fork, 0));
    const i64 nmax = len[0] > len[1] ? len[0] : len[1];
    for (i64 t = 1; t <= nmax; ++t) {
        for (int c = 0; c < 2; ++c) {
            if (t > len[c]) continue;
            const i64 p = len[c] - t, i = chain_row(h, c, p);
            if (k > 1 && (t == 1 || p % k == k - 1) && (rc = recompute_segment(h, c, p / k, st[c]))) return rc;
            if ((rc = launch_couple<TP>(h, i, X, S, Y[c], 0, c == 0 ? 0.0 : 1.0, c == 0 ? 1.0 : 0.0, st[c], 0, op))) return rc;
            if ((rc = launch_block_gemm(h, i, (const TP*)Y[c], X, S, -1.0, 1, st[c], op))) return rc;
        }
    }
    HZ_CUDA(h, cudaEventRecord(h->ev_join, st[1]));
    HZ_CUDA(h, cudaStreamWaitEvent(st[0], h->ev_join, 0));
    if (k > 1) {                                  // the recomputation can hit the same pivot failures as the factorisation
        int herr = 0;
        HZ_CUDA(h, cudaMemcpyAsync(&herr, h->d_err, sizeof(int), cudaMemcpyDeviceToHost, st[0]));
        HZ_CUDA(h, cudaStreamSynchronize(st[0]));
        if (herr) return fail(h, HZ_ESINGULAR, "hz_solve: zero or non-finite pivot while recomputing block inverses between checkpoints");
    }
    return HZ_OK;
}

template <class TP>
static int launch_residual(hz_ctx* h, const TP* X, const TP* Q, i64 S, TP* R, int op) {
    const int threads = S >= 128 ? 128 : (S >= 64 ? 64 : 32);
    const i64 rows = (i64)h->nf * h->N;
    dim3 grid((unsigned)((S + threads - 1) / threads), (unsigned)(rows < 65535 ? rows : 65535), (unsigned)((rows + 65534) / 65535));
    auto kfn = op == HZ_OP_T ? residual_kernel<TP, 1> : (op == HZ_OP_H ? residual_kernel<TP, 2> : residual_kernel<TP, 0>);
    HZ_LAUNCH_EW(kfn, grid, dim3(threads), 0, h->stream, (const cplx*)h->coef, h->nf, h->nx, h->nz, X, Q, S, R);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

template <class TP>
static int solve_impl(hz_ctx* h, int op, TP* X, int64_t S, double premul_re, double premul_im, int conjugate,
                      int64_t z_first, int64_t z_last, int refine, double* resid_host) {
    const i64 rows = (i64)h->nf * h->N, n = rows * S;
    if (h->ycap < S) {
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream2));
        for (int k = 0; k < 2; ++k) {
            free_dev(h->Ybuf[k]);
            HZ_CUDA(h, cudaMalloc((void**)&h->Ybuf[k], (size_t)h->b * S * sizeof(cplx)));
        }
        h->ycap = S;
        h->y_S = -1;
    }
#ifndef HZ_EMU
    if (std::is_same<TP, cplxf>::value && h->tf32_active && h->y_S != S) {
        for (int k = 0; k < 2; ++k)
            if (!t32_make_map(&h->mapY[k], (const float*)h->Ybuf[k], h->b, S, 2, h->ldb64, T32_KS, t32_tile_n(S), false))
                return fail(h, HZ_ECUDA, "hz_solve: cuTensorMapEncodeTiled failed for the right-hand-side planes");
        h->y_S = S;
    }
#endif
    const bool want_resid = refine > 0 || resid_host != nullptr;
    if (want_resid && h->qcap < S) {
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        free_dev(h->Qsave); free_dev(h->Rres);
        HZ_CUDA(h, cudaMalloc((void**)&h->Qsave, (size_t)n * sizeof(TP)));
        HZ_CUDA(h, cudaMalloc((void**)&h->Rres, (size_t)n * sizeof(TP)));
        h->qcap = S;
    }
    TP* Qs = (TP*)h->Qsave;
    TP* Rr = (TP*)h->Rres;
    if (want_resid) HZ_CUDA(h, cudaMemcpyAsync(Qs, X, (size_t)n * sizeof(TP), cudaMemcpyDeviceToDevice, h->stream));
    const bool probe = h->probe_check && h->probe_pending && refine == 0;
    if (probe) {
        if (!h->Qprobe) HZ_CUDA(h, cudaMalloc((void**)&h->Qprobe, (size_t)rows * sizeof(cplx)));
        auto gfn = gather_col_kernel<TP>;
        HZ_LAUNCH_EW(gfn, dim3(blocks_for(rows, 256)), dim3(256), 0, h->stream, (const TP*)X, (i64)S, (i64)0, rows, h->Qprobe);
        HZ_CHECK_LAUNCH(h);
    }
    int rc = solve_inplace<TP>(h, X, S, z_first, z_last, op);
    if (rc) return rc;
    h->probe_pending = false;
    if (probe) {
        HZ_CUDA(h, cudaMemsetAsync(h->d_norm, 0, 2 * sizeof(double), h->stream));
        auto rfn = op == HZ_OP_T ? residual_col_kernel<TP, 1> : (op == HZ_OP_H ? residual_col_kernel<TP, 2> : residual_col_kernel<TP, 0>);
        HZ_LAUNCH_IND(rfn, dim3(blocks_for(rows, 256, 148 * 8)), dim3(256), 0, h->stream, (const cplx*)h->coef, h->nf, h->nx, h->nz, (const TP*)X, (i64)S,
                  (i64)0, (const cplx*)h->Qprobe, h->d_norm);
        HZ_CHECK_LAUNCH(h);
        double nrm[2];
        HZ_CUDA(h, cudaMemcpyAsync(nrm, h->d_norm, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        h->last_probe = nrm[1] > 0 ? std::sqrt(nrm[0] / nrm[1]) : 0.0;
        const double limit = h->probe_limit > 0 ? h->probe_limit : (sizeof(TP) == sizeof(cplxf) ? 1e-2 : 1e-7);
        if (!(h->last_probe <= limit)) {
            char msg[320];
            snprintf(msg, sizeof msg, "hz_solve: accuracy probe failed: stencil residual %.3e of the first right-hand side exceeds %.0e -- the unpivoted "
                     "block elimination lost accuracy on this operator; solve with refine >= 1 (iterative refinement) or another twist", h->last_probe, limit);
            return fail(h, HZ_EACCURACY, msg);
        }
    }
    double ratio = -1.0;
    for (int it = 0; want_resid; ++it) {
        if ((rc = launch_residual<TP>(h, X, Qs, S, Rr, op))) return rc;
        HZ_CUDA(h, cudaMemsetAsync(h->d_norm, 0, 2 * sizeof(double), h->stream));
        auto nfn = norm2_kernel<TP>;
        HZ_LAUNCH_IND(nfn, dim3(blocks_for(n, 256)), dim3(256), 0, h->stream, (const TP*)Rr, (const TP*)Qs, n, h->d_norm);
        HZ_CHECK_LAUNCH(h);
        double nrm[2];
        HZ_CUDA(h, cudaMemcpyAsync(nrm, h->d_norm, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        ratio = nrm[1] > 0 ? std::sqrt(nrm[0] / nrm[1]) : 0.0;
        if (it >= refine || ratio < 1e-15) break;
        if ((rc = solve_inplace<TP>(h, Rr, S, -1, -1, op))) return rc;
        auto afn = axpy_kernel<TP>;
        HZ_LAUNCH_EW(afn, dim3(blocks_for(n, 256)), dim3(256), 0, h->stream, X, (const TP*)Rr, n);
        HZ_CHECK_LAUNCH(h);
    }
    if (resid_host) *resid_host = ratio;
    if (want_resid) {
        h->last_probe = ratio;
        const double limit = h->probe_limit > 0 ? h->probe_limit : (sizeof(TP) == sizeof(cplxf) ? 1e-2 : 1e-7);
        if (!(ratio <= limit)) {
            char msg[256];
            snprintf(msg, sizeof msg, "hz_solve: stencil residual %.3e after %d refinement step(s) exceeds %.0e -- the block elimination lost "
                     "accuracy on this operator", ratio, refine, limit);
            return fail(h, HZ_EACCURACY, msg);
        }
    }
    if (conjugate || premul_re != 1.0 || premul_im != 0.0) {
        auto ffn = finalize_kernel<TP>;
        HZ_LAUNCH_EW(ffn, dim3(blocks_for(n, 256)), dim3(256), 0, h->stream, X, n, mk(premul_re, premul_im), conjugate);
        HZ_CHECK_LAUNCH(h);
    }
    return HZ_OK;
}

int hz_solve_op(hz_handle_t h, int op, void* Xv, int64_t S, double premul_re, double premul_im, int conjugate,
                int64_t z_first, int64_t z_last, int refine, double* resid_host) {
    if (!h || !Xv) return fail(h, HZ_EINVAL, "hz_solve: NULL argument");
    if (op != HZ_OP_N && op != HZ_OP_T && op != HZ_OP_H) return fail(h, HZ_EINVAL, "hz_solve_op: op must be HZ_OP_N, HZ_OP_T or HZ_OP_H");
    if (!h->factored) return fail(h, HZ_ESTATE, "hz_solve: call hz_factor first");
    if (S < 1 || S > (1 << 24)) return fail(h, HZ_EINVAL, "hz_solve: S out of range");
    if (refine < -1 || refine > 8) return fail(h, HZ_EINVAL, "hz_solve: refine out of range");
    if (op != HZ_OP_N && h->dtype == HZ_C64)
        return fail(h, HZ_ENOTIMPL, "hz_solve_op: transposed solves (HZ_OP_T / HZ_OP_H) are built for complex128 handles only");
    // -1: library default.  The tensor-core (TF32) contraction of the complex64 variant accumulates in the tensor core's
    // truncating FP32 adder (measured ~3.5e-6 per 1000-deep contraction against 3e-7 for FFMA), which over hundreds of
    // block rows exceeds the 1e-4 bound: one refinement step with the FP64 stencil residual restores it.
    if (refine < 0) refine = (h->dtype == HZ_C64 && h->tf32_active) ? 1 : 0;
    HZ_CUDA(h, cudaSetDevice(h->device));
    if (h->dtype == HZ_C64)
        return solve_impl<cplxf>(h, op, (cplxf*)Xv, S, premul_re, premul_im, conjugate, z_first, z_last, refine, resid_host);
    return solve_impl<cplx>(h, op, (cplx*)Xv, S, premul_re, premul_im, conjugate, z_first, z_last, refine, resid_host);
}

int hz_solve(hz_handle_t h, void* Xv, int64_t S, double premul_re, double premul_im, int conjugate,
             int64_t z_first, int64_t z_last, int refine, double* resid_host) {
    return hz_solve_op(h, HZ_OP_N, Xv, S, premul_re, premul_im, conjugate, z_first, z_last, refine, resid_host);
}

int hz_profile(hz_handle_t h, int enable, double* out_host) {
    // out_host[6] = {solve-GEMM sampled ms, sampled launches, all launches,
    //                update-GEMM sampled ms, sampled launches, all launches}; reading resets.
    if (!h) return fail(h, HZ_EINVAL, "hz_profile: NULL handle");
    HZ_CUDA(h, cudaSetDevice(h->device));
    if (out_host) {
        HZ_CUDA(h, cudaStreamSynchronize(h->stream));
        HZ_CUDA(h, cudaStreamSynchronize(h->stream2));
        for (int k = 0; k < 2; ++k) {
            double ms = 0.0;
            for (size_t i = 0; i + 1 < h->prof_ev[k].size(); i += 2) {
                float t = 0.f;
                if (cudaEventElapsedTime(&t, h->prof_ev[k][i], h->prof_ev[k][i + 1]) == cudaSuccess) ms += t;
            }
            out_host[3 * k] = ms;
            out_host[3 * k + 1] = (double)(h->prof_ev[k].size() / 2);
            out_host[3 * k + 2] = (double)h->prof_launches[k];
        }
    }
    for (int k = 0; k < 2; ++k) {
        for (cudaEvent_t e : h->prof_ev[k]) cudaEventDestroy(e);
        h->prof_ev[k].clear();
        h->prof_tick[k] = 0;
        h->prof_launches[k] = 0;
    }
    h->prof_on = enable != 0;
    return HZ_OK;
}

int hz_get_trace(hz_handle_t h, int64_t* out_host, int64_t cap, int64_t* steps, int64_t* grid) {
    // diagnostics: per-CTA (start, end) globaltimer ns of every Gauss-Jordan step of the block factored last
    if (!h || !steps || !grid) return fail(h, HZ_EINVAL, "hz_get_trace: NULL argument");
    *steps = h->trace_steps;
    *grid = h->trace_grid;
    const i64 n = (i64)h->trace_steps * h->trace_grid * 16;
    long long* src = h->d_trace[h->trace_chain & 1];
    if (out_host && src && cap >= n) {
        HZ_CUDA(h, cudaSetDevice(h->device));
        HZ_CUDA(h, cudaDeviceSynchronize());
        HZ_CUDA(h, cudaMemcpy(out_host, src, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost));
    }
    return HZ_OK;
}

int hz_factor_graph_info(hz_handle_t h, int64_t* out2) {
    if (!h || !out2) return fail(h, HZ_EINVAL, "hz_factor_graph_info: NULL argument");
#ifndef HZ_EMU
    out2[0] = h->fgraph ? h->fgraph_launches : 0;
    out2[1] = h->fgraph ? h->fgraph_replays : 0;
#else
    out2[0] = out2[1] = 0;
#endif
    return HZ_OK;
}

int hz_newton_stats_get(int64_t* out4) {
    if (!out4) return fail(nullptr, HZ_EINVAL, "hz_newton_stats_get: NULL argument");
    unsigned long long v[4] = {0, 0, 0, 0};
#ifdef HZ_EMU
    for (int i = 0; i < 4; ++i) v[i] = hz_newton_stats[i];
#else
    if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpyFromSymbol(v, hz_newton_stats, sizeof v) != cudaSuccess)
        return fail(nullptr, HZ_ECUDA, "hz_newton_stats_get: cudaMemcpyFromSymbol failed");
#endif
    for (int i = 0; i < 4; ++i) out4[i] = (int64_t)v[i];
    return HZ_OK;
}

int hz_launch_count(int64_t* out) {
    if (!out) return fail(nullptr, HZ_EINVAL, "hz_launch_count: NULL argument");
    *out = g_hz_launches.load();
    return HZ_OK;
}

// ---- handle-less helpers ---------------------------------------------------------------------
template <class TP>
static int scatter_impl(void* X, int64_t S, int64_t nnz, const int64_t* row, const int64_t* col, const void* val,
                        double scale_re, double scale_im, void* stream) {
    if (nnz == 0) return HZ_OK;
    if (!X || !row || !col || !val || nnz < 0 || S < 1) return fail(nullptr, HZ_EINVAL, "hz_scatter_coo: bad argument");
    auto kfn = scatter_coo_kernel<TP>;
    HZ_LAUNCH_EW(kfn, dim3((unsigned)((nnz + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, (TP*)X, (i64)S, (i64)nnz,
                 (const i64*)row, (const i64*)col, (const cplx*)val, mk(scale_re, scale_im));
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}
int hz_scatter_coo(void* X, int64_t S, int64_t nnz, const int64_t* row, const int64_t* col, const void* val,
                   double scale_re, double scale_im, void* stream) {
    return scatter_impl<cplx>(X, S, nnz, row, col, val, scale_re, scale_im, stream);
}
int hz_scatter_coo_c64(void* X, int64_t S, int64_t nnz, const int64_t* row, const int64_t* col, const void* val,
                       double scale_re, double scale_im, void* stream) {
    return scatter_impl<cplxf>(X, S, nnz, row, col, val, scale_re, scale_im, stream);
}

int hz_nearest_index(int64_t nx, int64_t nz, double dx, double dz, double xorig, double zorig,
                     const double* locs, int64_t nloc, int64_t* out_idx, void* stream) {
    if (nloc == 0) return HZ_OK;
    if (!locs || !out_idx || nloc < 0 || nx < 1 || nz < 1) return fail(nullptr, HZ_EINVAL, "hz_nearest_index: bad argument");
    const int threads = 256;
    HZ_LAUNCH(nearest_index_kernel, dim3((unsigned)nloc), dim3(threads), threads * (sizeof(double) + sizeof(i64)), (cudaStream_t)stream,
              (int)nx, (int)nz, dx, dz, xorig, zorig, locs, (i64*)out_idx);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}

int hz_kaiser_taps(int64_t nx, int64_t nz, double dx, double dz, double xorig, double zorig, int ireg,
                   const int32_t* freeSurf_host, const double* locs, const int64_t* idx, int64_t nloc,
                   int64_t* rows, double* vals, int32_t* counts, void* stream) {
    static const double HC[11] = {0.0, 1.24, 2.94, 4.53, 6.31, 7.91, 9.42, 10.95, 12.53, 14.09, 14.18};  // source.py:138-149
    if (nloc == 0) return HZ_OK;
    if (ireg < 0 || ireg > KWS_MAX_IREG) return fail(nullptr, HZ_EINVAL, "hz_kaiser_taps: Kaiser windowed sinc function not implemented for this half-width");
    if (!locs || !idx || !rows || !vals || !counts || nloc < 0) return fail(nullptr, HZ_EINVAL, "hz_kaiser_taps: bad argument");
    int fs[4] = {0, 0, 0, 0};
    if (freeSurf_host) for (int i = 0; i < 4; ++i) fs[i] = freeSurf_host[i] != 0;
    HZ_LAUNCH_EW(kaiser_taps_kernel, dim3((unsigned)((nloc + 63) / 64)), dim3(64), 0, (cudaStream_t)stream, (int)nx, (int)nz, dx, dz, xorig, zorig,
              ireg, HC[ireg], fs[0], fs[1], fs[2], fs[3], locs, (const i64*)idx, (int)nloc, (i64*)rows, vals, (int*)counts);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}

template <class TP>
static int spmm_impl(int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, const int64_t* orow,
                     const void* In, int64_t ldin, int64_t S, void* Out, int64_t ldout, int64_t ostride,
                     int accumulate, void* stream) {
    if (nrows == 0 || S == 0) return HZ_OK;
    if (!rowptr || !col || !val || !In || !Out || nrows < 0 || S < 0 || nrows > 65535LL * 65535LL)
        return fail(nullptr, HZ_EINVAL, "hz_spmm_csr: bad argument");
    const int threads = S >= 128 ? 128 : (S >= 64 ? 64 : 32);
    auto kfn = spmm_csr_kernel<TP>;
    for (i64 r0 = 0; r0 < nrows; r0 += 65535) {       // gridDim.y limit
        const i64 nr = nrows - r0 < 65535 ? nrows - r0 : 65535;
        dim3 grid((unsigned)((S + threads - 1) / threads), (unsigned)nr, 1);
        HZ_LAUNCH_EW(kfn, grid, dim3(threads), 0, (cudaStream_t)stream, (i64)nr, (const i64*)rowptr + r0, (const i64*)col,
                     (const cplx*)val, orow ? (const i64*)orow + r0 : (const i64*)nullptr, (const TP*)In, (i64)ldin, (i64)S,
                     (TP*)Out + (orow ? 0 : r0 * ldout * ostride), (i64)ldout, (i64)ostride, accumulate);
        HZ_CHECK_LAUNCH(nullptr);
    }
    return HZ_OK;
}
int hz_spmm_csr(int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, const int64_t* orow,
                const void* In, int64_t ldin, int64_t S, void* Out, int64_t ldout, int64_t ostride,
                int accumulate, void* stream) {
    return spmm_impl<cplx>(nrows, rowptr, col, val, orow, In, ldin, S, Out, ldout, ostride, accumulate, stream);
}
int hz_spmm_csr_c64(int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, const int64_t* orow,
                    const void* In, int64_t ldin, int64_t S, void* Out, int64_t ldout, int64_t ostride,
                    int accumulate, void* stream) {
    return spmm_impl<cplxf>(nrows, rowptr, col, val, orow, In, ldin, S, Out, ldout, ostride, accumulate, stream);
}

template <class TP>
static int percol_impl(int transpose, int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, int64_t S,
                       const void* In, void* Out, int64_t ld, void* stream) {
    if (nrows == 0) return HZ_OK;
    if (!rowptr || !col || !val || !In || !Out || nrows < 0 || S < 1 || ld < S) return fail(nullptr, HZ_EINVAL, "hz_spmm_percol: bad argument");
    const dim3 grid((unsigned)((nrows + 255) / 256)), block(256);
    if (transpose) {
        auto kfn = spmm_percol_t_kernel<TP>;
        HZ_LAUNCH_EW(kfn, grid, block, 0, (cudaStream_t)stream, (i64)nrows, (const i64*)rowptr, (const i64*)col, (const cplx*)val, (i64)S,
                     (const TP*)In, (TP*)Out, (i64)ld);
    } else {
        auto kfn = spmm_percol_kernel<TP>;
        HZ_LAUNCH_EW(kfn, grid, block, 0, (cudaStream_t)stream, (i64)nrows, (const i64*)rowptr, (const i64*)col, (const cplx*)val, (i64)S,
                     (const TP*)In, (i64)ld, (TP*)Out);
    }
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}
int hz_spmm_percol(int transpose, int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, int64_t S,
                   const void* In, void* Out, int64_t ld, void* stream) {
    return percol_impl<cplx>(transpose, nrows, rowptr, col, val, S, In, Out, ld, stream);
}
int hz_spmm_percol_c64(int transpose, int64_t nrows, const int64_t* rowptr, const int64_t* col, const void* val, int64_t S,
                       const void* In, void* Out, int64_t ld, void* stream) {
    return percol_impl<cplxf>(transpose, nrows, rowptr, col, val, S, In, Out, ld, stream);
}

template <class TP>
static int gradient_impl(const void* uF, const void* uB, int64_t N, int64_t S, const void* scaler, void* g, void* stream) {
    if (!uF || !uB || !scaler || !g || N < 1 || S < 1) return fail(nullptr, HZ_EINVAL, "hz_gradient: bad argument");
    const int threads = 256;
    const i64 wpb = threads / 32;
    auto kfn = gradient_kernel<TP>;
    HZ_LAUNCH_IND(kfn, dim3(blocks_for((N + wpb - 1) / wpb * threads, threads, 148 * 16)), dim3(threads), 0, (cudaStream_t)stream,
              (const TP*)uF, (const TP*)uB, (i64)N, (i64)S, (const cplx*)scaler, (cplx*)g);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}
int hz_gradient(const void* uF, const void* uB, int64_t N, int64_t S, const void* scaler, void* g, void* stream) {
    return gradient_impl<cplx>(uF, uB, N, S, scaler, g, stream);
}
int hz_gradient_c64(const void* uF, const void* uB, int64_t N, int64_t S, const void* scaler, void* g, void* stream) {
    return gradient_impl<cplxf>(uF, uB, N, S, scaler, g, stream);
}

template <class TP>
static int misfit_impl(const void* d, const void* dobs, int64_t n, double wd, void* v, double* phi, void* stream) {
    if (!d || !dobs || !phi || n < 1) return fail(nullptr, HZ_EINVAL, "hz_misfit: bad argument");
    auto kfn = misfit_kernel<TP>;
    HZ_LAUNCH_IND(kfn, dim3(blocks_for(n, 256, 148 * 4)), dim3(256), 0, (cudaStream_t)stream, (const TP*)d, (const TP*)dobs, (i64)n, wd,
              (TP*)v, phi);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}
int hz_misfit(const void* d, const void* dobs, int64_t n, double wd, void* v, double* phi, void* stream) {
    return misfit_impl<cplx>(d, dobs, n, wd, v, phi, stream);
}
int hz_misfit_c64(const void* d, const void* dobs, int64_t n, double wd, void* v, double* phi, void* stream) {
    return misfit_impl<cplxf>(d, dobs, n, wd, v, phi, stream);
}

int hz_stencil_xcorr(const void* lam, const void* u, int64_t nx, int64_t nz, int64_t S, void* G, void* stream) {
    if (!lam || !u || !G) return fail(nullptr, HZ_EINVAL, "hz_stencil_xcorr: NULL argument");
    if (nx < 3 || nz < 3 || nx > 32768 || nz > (1 << 24) || S < 1) return fail(nullptr, HZ_EINVAL, "hz_stencil_xcorr: nx, nz or S out of range");
    const int threads = 256;
    const i64 wpb = threads / 32, N = nx * nz;
    HZ_LAUNCH_IND(stencil_xcorr_kernel, dim3(blocks_for((N + wpb - 1) / wpb * threads, threads, 148 * 16)), dim3(threads), 0, (cudaStream_t)stream,
                  (const cplx*)lam, (const cplx*)u, (int)nx, (int)nz, (i64)S, (cplx*)G);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}

int hz_assemble_vjp(hz_handle_t h, const void* G, const void* alpha, double* g_c, double* g_rho) {
    if (!h) return fail(h, HZ_EINVAL, "hz_assemble_vjp: NULL handle");
    if (h->disc != HZ_DISC_MINIZEPHYR || h->dtype != HZ_C128)
        return fail(h, HZ_ENOTIMPL, "hz_assemble_vjp: built for complex128 MiniZephyr handles only");
    if (!G || (!g_c && !g_rho)) return fail(h, HZ_EINVAL, "hz_assemble_vjp: G and at least one of g_c, g_rho are required");
    if (!h->assembled || !h->asm_from_model)
        return fail(h, HZ_ESTATE, "hz_assemble_vjp: the coefficients must come from hz_assemble of the current model");
    HZ_CUDA(h, cudaSetDevice(h->device));
    const int threads = 128;
    HZ_LAUNCH_EW(assemble_mz_vjp_kernel, dim3((unsigned)((h->N + threads - 1) / threads)), dim3(threads), 0, h->stream, (const cplx*)h->c,
                 (const cplx*)h->Kp, (const double*)h->binv, (const cplx*)G, (const cplx*)alpha, h->asm_p, g_c, g_rho);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

int hz_stencil_apply(const void* dcoef, const void* u, int64_t nx, int64_t nz, int64_t S, double scale_re, double scale_im, void* out,
                     void* stream) {
    if (!dcoef || !u || !out) return fail(nullptr, HZ_EINVAL, "hz_stencil_apply: NULL argument");
    if (nx < 3 || nz < 3 || nx > 32768 || nz > (1 << 24) || S < 1) return fail(nullptr, HZ_EINVAL, "hz_stencil_apply: nx, nz or S out of range");
    const int tx = S >= 256 ? 256 : (int)((S + 31) / 32 * 32), ty = 256 / tx;
    const i64 N = nx * nz;
    HZ_LAUNCH_IND(stencil_apply_kernel, dim3(blocks_for(N, STENCIL_APPLY_RUN * ty, (i64)1 << 24)), dim3(tx, ty), 0, (cudaStream_t)stream,
                  (const cplx*)dcoef, (const cplx*)u, (int)nx, (int)nz, (i64)S, mk(scale_re, scale_im), (cplx*)out);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}

int hz_assemble_jvp(hz_handle_t h, const double* dc, const double* drho, const void* alpha, void* dcoef) {
    if (!h) return fail(h, HZ_EINVAL, "hz_assemble_jvp: NULL handle");
    if (h->disc != HZ_DISC_MINIZEPHYR || h->dtype != HZ_C128)
        return fail(h, HZ_ENOTIMPL, "hz_assemble_jvp: built for complex128 MiniZephyr handles only");
    if (!dcoef || (!dc && !drho)) return fail(h, HZ_EINVAL, "hz_assemble_jvp: dcoef and at least one of dc, drho are required");
    if (!h->assembled || !h->asm_from_model)
        return fail(h, HZ_ESTATE, "hz_assemble_jvp: the coefficients must come from hz_assemble of the current model");
    HZ_CUDA(h, cudaSetDevice(h->device));
    const int threads = 128;
    HZ_LAUNCH_EW(assemble_mz_jvp_kernel, dim3((unsigned)((h->N + threads - 1) / threads)), dim3(threads), 0, h->stream, (const cplx*)h->c,
                 (const cplx*)h->Kp, (const double*)h->binv, dc, drho, (const cplx*)alpha, h->asm_p, (cplx*)dcoef);
    HZ_CHECK_LAUNCH(h);
    return HZ_OK;
}

int hz_cgemm_tf32(int64_t M, int64_t N, int64_t K, double alpha, const float* A_planes, int64_t lda, const float* Y_planes, int64_t ldy,
                  void* C, int64_t ldc, void* stream, float* dbg, int variant) {
#ifdef HZ_EMU
    return fail(nullptr, HZ_ENOTIMPL, "hz_cgemm_tf32: tcgen05 kernels are not part of the CPU-emulation test build");
#else
    if (!A_planes || !Y_planes || !C || M < 1 || N < 1 || K < 1 || (lda & 3) || (ldy & 3) || lda < K || ldy < K || ldc < N)
        return fail(nullptr, HZ_EINVAL, "hz_cgemm_tf32: bad argument (plane row strides must be multiples of 4 floats)");
    alignas(64) CUtensorMap mapA, mapY;
    const int force_tn = (variant >> 8) & 0xff;
    if (!t32_make_map(&mapA, A_planes, K, M, 2, lda, T32_KS, T32_TM, false) ||
        !t32_make_map(&mapY, Y_planes, K, N, 2, ldy, T32_KS, force_tn ? force_tn : t32_tile_n(N), false))
        return fail(nullptr, HZ_ECUDA, "hz_cgemm_tf32: cuTensorMapEncodeTiled failed");
    Tf32Params tp;
    tp.M = (int)M; tp.N = (int)N; tp.K = (int)K;
    tp.a_plane0 = 0; tp.y_plane0 = 0;
    tp.C = (cplxf*)C; tp.ldc = ldc;
    tp.alpha = (float)alpha;
    tp.row_nx = 0; tp.row_fs = 0; tp.k_per_split = 0;
    tp.dbg = dbg;
    tp.mode = variant & 0xff; tp.force_split = (variant >> 16) & 0xff;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cgemm_tf32_launch(mapA, mapY, tp, sms, (cudaStream_t)stream, force_tn);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
#endif
}

int hz_zgemm(int64_t M, int64_t N, int64_t K, double alpha, const void* A, int64_t lda, const void* B,
             int64_t ldb, int beta, void* C, int64_t ldc, int tile, void* stream) {
    if (!A || !B || !C || M < 1 || N < 1 || K < 1) return fail(nullptr, HZ_EINVAL, "hz_zgemm: bad argument");
    if (tile > 25 || (tile > 12 && tile < 16)) return fail(nullptr, HZ_EINVAL, "hz_zgemm: unknown tile id");
    GemmParams p;
    p.A = (const cplx*)A; p.lda = lda;
    p.B = (const cplx*)B; p.ldb = ldb;
    p.C = (cplx*)C; p.ldc = ldc;
    p.M = (int)M; p.N = (int)N; p.K = (int)K;
    p.alpha = alpha; p.beta = beta;
    p.sub_c0 = p.sub_c1 = 0;
    p.row_nx = 0; p.row_fs = 0;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    zgemm_launch(p, (cudaStream_t)stream, sms, tile);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}

int hz_zgemm_op(int64_t M, int64_t N, int64_t K, double alpha, const void* A, int64_t lda, int opA, const void* B,
                int64_t ldb, int beta, void* C, int64_t ldc, int tile, int gemm_3m, void* stream) {
    if (!A || !B || !C || M < 1 || N < 1 || K < 1) return fail(nullptr, HZ_EINVAL, "hz_zgemm_op: bad argument");
    if (opA != HZ_OP_N && opA != HZ_OP_T && opA != HZ_OP_H) return fail(nullptr, HZ_EINVAL, "hz_zgemm_op: opA must be HZ_OP_N, HZ_OP_T or HZ_OP_H");
    if (tile < -1 || tile >= kNumGemmTiles || (gemm_3m != 0 && gemm_3m != 1)) return fail(nullptr, HZ_EINVAL, "hz_zgemm_op: unknown tile or product form");
    GemmParams p;
    p.A = (const cplx*)A; p.lda = lda;
    p.B = (const cplx*)B; p.ldb = ldb;
    p.C = (cplx*)C; p.ldc = ldc;
    p.M = (int)M; p.N = (int)N; p.K = (int)K;
    p.alpha = alpha; p.beta = beta;
    p.sub_c0 = p.sub_c1 = 0;
    p.row_nx = 0; p.row_fs = 0;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int which = zgemm_tile_id(tile >= 0 ? tile : zgemm_pick(p.M, p.N, sms), gemm_3m != 0);
    if (opA == HZ_OP_T) zgemm_launch<1>(p, (cudaStream_t)stream, sms, which);
    else if (opA == HZ_OP_H) zgemm_launch<2>(p, (cudaStream_t)stream, sms, which);
    else zgemm_launch<0>(p, (cudaStream_t)stream, sms, which);
    HZ_CHECK_LAUNCH(nullptr);
    return HZ_OK;
}
