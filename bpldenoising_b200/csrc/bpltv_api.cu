// bpltv_api.cu — C ABI of libbpltv.so (see include/bpltv.h).
//
// Host side of the hot path: context / buffer management, image sharding over the
// devices of one process, kernel dispatch.  No CPU fallback: every numerical
// operation below is a CUDA kernel for sm_100a.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include <cstddef>

#include "../../include/bpltv.h"
#include "env_switches.h"
#include "common.cuh"
#include "pdps_generic.cuh"
#include "pdps_march.cuh"
#include "tblock_kernels.h"
#include "pdps_resident.cuh"
#include "pdps_sumregs.cuh"
#include "gradient.cuh"
#include "gradient_sumregs.cuh"
#include "gradient_lu.cuh"
#include "gradient_nd.h"
#include "selftest.cuh"
#include "nccl_dyn.h"

// the option structs are mirrored field by field in bpldenoising_b200/_lib.py (ctypes) and julia/BPLTV.jl
static_assert(sizeof(bpltv_pdps_opts) == 72, "bpltv_pdps_opts layout");
static_assert(sizeof(bpltv_eval_opts) == 144 && offsetof(bpltv_eval_opts, gamma_patch) == 128, "bpltv_eval_opts layout");
static_assert(sizeof(bpltv_stats) == 120, "bpltv_stats layout");

using namespace bpltv;

// ---------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------
static thread_local std::string g_last_error;

static int fail(int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

#define CU_TRY(expr)                                                                          \
    do {                                                                                      \
        cudaError_t e_ = (expr);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(BPLTV_ERR_CUDA, "%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,  \
                        cudaGetErrorString(e_));                                              \
    } while (0)

#define RC_TRY(expr)             \
    do {                         \
        int rc_ = (expr);        \
        if (rc_ != 0) return rc_; \
    } while (0)

// ---------------------------------------------------------------------------
// device buffers (grow-only)
// ---------------------------------------------------------------------------
struct DBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need)
    {
        if (need <= bytes) return 0;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(BPLTV_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e));
        }
        bytes = need;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <typename T> T *as() const { return static_cast<T *>(p); }
};

// ---------------------------------------------------------------------------
// Pageable host buffers.  What a caller hands in is usually pageable memory (a Julia Array, a numpy array):
// cudaMemcpyAsync then goes through the driver's single staging thread — measured 11 GB/s up and 18 GB/s down on the B200
// box against 55 GB/s from pinned memory, i.e. 19 ms of copies beside a 95 ms solve at BASELINE config 4.  Registering the
// caller's buffer for the duration of the call (cudaHostRegister) costs more than it saves (page pinning ≈ the copy).
// Instead NT host threads move 4 MiB chunks through their own pinned slots: thread t owns chunks t, t+NT, … and two
// slots, copies chunk k into a slot while the DMA of chunk k-1 drains the other (and the reverse for downloads).
// The caller's buffers stay untouched and unpinned; the slots belong to the context (ownership rule of SURVEY §8b).
// ---------------------------------------------------------------------------
struct HostStage {
    static constexpr int MAXT = 16, NSLOT = 2;
    static constexpr size_t SLOT = (size_t)4 << 20;
    static constexpr size_t MIN_BYTES = (size_t)8 << 20;     // below this the driver's path is as good
    char *pin = nullptr;
    cudaEvent_t ev[MAXT * NSLOT] = {nullptr};
    bool used[MAXT * NSLOT] = {false};
    int nt = 0;
    bool init()
    {
        if (pin) return true;
        const unsigned hc = std::thread::hardware_concurrency();
        nt = (int)std::max(1u, std::min<unsigned>(8, hc ? hc / 2 : 2));
        {   // BPLTV_STAGE_THREADS overrides (1..16); read here, once per context and device
            const char *e = bpltv::env_get("BPLTV_STAGE_THREADS");
            if (e && *e) nt = std::max(1, std::min((int)MAXT, atoi(e)));
        }
        if (cudaHostAlloc((void **)&pin, (size_t)nt * NSLOT * SLOT, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError(); pin = nullptr; return false;
        }
        for (int i = 0; i < nt * NSLOT; ++i)
            if (cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); release(); return false; }
        return true;
    }
    void release()
    {
        for (auto &e : ev) { if (e) cudaEventDestroy(e); e = nullptr; }
        for (auto &u : used) u = false;
        if (pin) cudaFreeHost(pin);
        pin = nullptr;
    }
};

static bool host_is_pageable(const void *h)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, h) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

// host ↔ device copy of `bytes` through the pinned slots, enqueued on `st`.  to_device: returns when the caller's
// buffer has been read (the last DMAs may still be in flight on `st`); otherwise returns when the data is in `host`.
static cudaError_t staged_copy(HostStage &hs, int device, char *dev, char *host, size_t bytes, cudaStream_t st, bool to_device)
{
    const size_t SLOT = HostStage::SLOT;
    const size_t nchunks = (bytes + SLOT - 1) / SLOT;
    const int nt = (int)std::min<size_t>((size_t)hs.nt, nchunks);
    std::atomic<int> err{(int)cudaSuccess};
    auto fail_with = [&](cudaError_t e) { int ok = (int)cudaSuccess; err.compare_exchange_strong(ok, (int)e); };
    auto worker = [&](int t) {
        cudaError_t e = cudaSetDevice(device);
        if (e != cudaSuccess) { fail_with(e); return; }
        auto span = [&](size_t c, size_t &off, size_t &len) { off = c * SLOT; len = std::min(SLOT, bytes - off); };
        if (to_device) {
            size_t k = 0;
            for (size_t c = (size_t)t; c < nchunks; c += (size_t)nt, ++k) {
                const int s = t * HostStage::NSLOT + (int)(k % HostStage::NSLOT);
                char *slot = hs.pin + (size_t)s * SLOT;
                if (hs.used[s] && (e = cudaEventSynchronize(hs.ev[s])) != cudaSuccess) { fail_with(e); return; }
                size_t off, len;
                span(c, off, len);
                std::memcpy(slot, host + off, len);
                if ((e = cudaMemcpyAsync(dev + off, slot, len, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
                    (e = cudaEventRecord(hs.ev[s], st)) != cudaSuccess) { fail_with(e); return; }
                hs.used[s] = true;
            }
        } else {
            // chunk k of this thread lands in slot k % NSLOT; keep NSLOT DMAs in flight ahead of the host copy
            auto issue = [&](size_t k) -> cudaError_t {
                const size_t c = (size_t)t + k * (size_t)nt;
                const int s = t * HostStage::NSLOT + (int)(k % HostStage::NSLOT);
                size_t off, len;
                span(c, off, len);
                if (hs.used[s]) { cudaError_t w = cudaEventSynchronize(hs.ev[s]); if (w != cudaSuccess) return w; }
                cudaError_t r = cudaMemcpyAsync(hs.pin + (size_t)s * SLOT, dev + off, len, cudaMemcpyDeviceToHost, st);
                if (r == cudaSuccess) r = cudaEventRecord(hs.ev[s], st);
                hs.used[s] = true;
                return r;
            };
            const size_t mine = nchunks > (size_t)t ? (nchunks - (size_t)t + (size_t)nt - 1) / (size_t)nt : 0;
            for (size_t k = 0; k < std::min<size_t>(HostStage::NSLOT, mine); ++k)
                if ((e = issue(k)) != cudaSuccess) { fail_with(e); return; }
            for (size_t k = 0; k < mine; ++k) {
                const int s = t * HostStage::NSLOT + (int)(k % HostStage::NSLOT);
                if ((e = cudaEventSynchronize(hs.ev[s])) != cudaSuccess) { fail_with(e); return; }
                size_t off, len;
                span((size_t)t + k * (size_t)nt, off, len);
                std::memcpy(host + off, hs.pin + (size_t)s * SLOT, len);
                hs.used[s] = false;                                // consumed: the slot is free without a wait
                if (k + HostStage::NSLOT < mine && (e = issue(k + HostStage::NSLOT)) != cudaSuccess) { fail_with(e); return; }
            }
        }
    };
    // chunks are dealt by thread index, so a thread that could not be started (std::system_error: no exception may cross
    // the C ABI) has its chunks done by the caller's thread afterwards
    std::vector<std::thread> th;
    std::vector<int> orphan;
    for (int t = 1; t < nt; ++t) {
        try { th.emplace_back(worker, t); } catch (...) { orphan.push_back(t); }
    }
    worker(0);
    for (int t : orphan) worker(t);
    for (auto &x : th) x.join();
    return (cudaError_t)err.load();
}

struct StepKey {
    double tau0 = -1, sigma0 = -1, opnorm = -1;
    int accel = -1, maxiter = -1, prec = 0;
    bool operator==(const StepKey &o) const
    {
        return tau0 == o.tau0 && sigma0 == o.sigma0 && opnorm == o.opnorm && accel == o.accel &&
               maxiter == o.maxiter && prec == o.prec;
    }
};

struct Dev {
    int id = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8] = {nullptr};   // phase marks of the current call (Mark below)
    unsigned marked = 0;             // … which of them it has recorded
    // resident dataset shard
    int M = 0, N = 0, O = 0;  // O = images on this device
    int o_begin = 0;          // first global image index of the shard
    DBuf truth, noisy;
    // solve state (ping-pong) and scratch
    DBuf x[2], y1[2], y2[2], fbuf, amap, steps, partials, scalars, stage, lam_dev, ubuf, sry;
    GradWork grad;            // gradient.cuh
    GradWork grad3;           // gradient_sumregs.cuh
    NdWork *nd = nullptr;     // gradient_nd.cuh (nested-dissection adjoint solver), created on first use
    NdWork *nd3 = nullptr;    // the same solver at coupling radius 2 (scalar sumregs_gradient_reg); a plan of its own
    // the solver of the last gradient on this device: its worst backward error is in its workspace (device memory)
    enum LastGrad { GRAD_NONE, GRAD_TV_ND, GRAD_TV_BAND, GRAD_SR_ND, GRAD_SR_BAND } last_grad = GRAD_NONE;
    StepKey steps_key;
    std::vector<unsigned char> steps_host;
    long long launches = 0;
    HostStage hstage;         // pinned slots for pageable caller buffers
    // denoise with pinned host buffers: the copies of image chunks run on a second stream under the first and the last
    // passes of the streaming solve (PipeIO below)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t pipe_ev[2 * 8 + 2] = {nullptr};
};

// Host↔device copies of a denoise call overlapped with its solve.  The stack is cut into `chunks` groups of images; the
// first `q` passes of the temporally blocked kernel run chunk by chunk as the uploads arrive, the middle passes on the
// whole stack, the last `q` passes chunk by chunk again with each chunk's download following it on the copy stream.
// Images are independent and every range cut of the kernel is bit-identical, so the result does not change.
struct PipeIO {
    const double *h_in = nullptr;     // this device's shard of the caller's noisy stack (pinned)
    double *h_out = nullptr;          // … of the caller's result (pinned)
    bool stage_in = false, stage_out = false;   // pageable buffers: through the context's pinned slots
    int chunks = 3, q = 6;           // measured on config 4 (e2e Gpixel-iter/s): K×q = 3×6 190.1, 4×6 189.1, 6×4 189.4, 8×3 188.5; serial 185.2
};

struct bpltv_ctx {
    int prec = 64;
    std::vector<Dev> devs;
    int M = 0, N = 0, O = 0;  // resident dataset shape (global)
    bool have_dataset = false;
    bpltv_stats stats;
    // one-process-per-GPU jobs: the communicator of bpltv_comm_init (nullptr: this process is the whole job)
    void *comm = nullptr;
    int comm_ranks = 1, comm_rank = 0;
};

// [cost, grad…] summed over the ranks of the job, in place, on `st` (one ncclAllReduce per evaluation); no-op without
// a communicator.  Every rank receives the same bits.
static int allreduce_costgrad(bpltv_ctx *ctx, double *d_costgrad, int count, cudaStream_t st)
{
    if (!ctx->comm) return 0;
    NcclApi &api = nccl_api();
    const int rc = api.AllReduce(d_costgrad, d_costgrad, (size_t)count, /*ncclDouble*/ 8, /*ncclSum*/ 0, ctx->comm, st);
    if (rc != 0) return fail(BPLTV_ERR_CUDA, "ncclAllReduce of [cost, grad]: %s", api.what(rc));
    return 0;
}

static void shard_range(int O, int ndev, int d, int &begin, int &count)
{
    // contiguous blocks of ceil(O/ndev) images (SURVEY §8e)
    const int per = (O + ndev - 1) / ndev;
    begin = std::min(O, d * per);
    count = std::min(O, begin + per) - begin;
}

// ---------------------------------------------------------------------------
// step-size recursion (S1, S2): σ=σ₀/R_K, τ=τ₀/R_K, γ=1, ω=1/√(1+2γτ), τ←τω, σ←σ/ω
// ---------------------------------------------------------------------------
template <typename Real>
static int upload_steps(Dev &d, const bpltv_pdps_opts &o, cudaStream_t st)
{
    StepKey key;
    key.tau0 = o.tau0; key.sigma0 = o.sigma0; key.opnorm = o.opnorm; key.accel = o.accel;
    key.maxiter = o.maxiter; key.prec = (int)sizeof(Real);
    if (key == d.steps_key) return 0;
    const size_t n = (size_t)std::max(o.maxiter, 1);
    d.steps_host.resize(n * sizeof(StepConsts<Real>));
    StepConsts<Real> *h = reinterpret_cast<StepConsts<Real> *>(d.steps_host.data());
    double sigma = o.sigma0 / o.opnorm;
    double tau = o.tau0 / o.opnorm;
    const double gamma = 1.0;
    for (int k = 0; k < o.maxiter; ++k) {
        double omega = 1.0;
        if (o.accel) omega = 1.0 / std::sqrt(1.0 + 2.0 * gamma * tau);
        StepConsts<Real> s;
        s.tau = (Real)tau; s.sigma = (Real)sigma; s.omega = (Real)omega;
        // (1+τ), (1+ω) are formed in the compute type from the rounded τ, ω, as the
        // reference's broadcast would form them per element
        s.one_p_tau = (Real)1 + s.tau;
        s.one_p_omega = (Real)1 + s.omega;
        s.inv_one_p_tau = (Real)(1.0 / (1.0 + tau));
        s.tau_over_one_p_tau = (Real)(tau / (1.0 + tau));
        s.rcp_one_p_tau = (Real)1 / s.one_p_tau;  // correctly rounded in the compute type
        h[k] = s;
        if (o.accel) { tau = tau * omega; sigma = sigma / omega; }
    }
    RC_TRY(d.steps.ensure(n * sizeof(StepConsts<Real>)));
    // stream-ordered w.r.t. kernels still reading the previous table
    CU_TRY(cudaMemcpyAsync(d.steps.p, h, n * sizeof(StepConsts<Real>), cudaMemcpyHostToDevice, st));
    CU_TRY(cudaStreamSynchronize(st));
    d.steps_key = key;
    return 0;
}

// ---------------------------------------------------------------------------
// PDPS driver
// ---------------------------------------------------------------------------
static int env_int(const char *name, int dflt)
{
    const char *s = bpltv::env_get(name);
    return (s && *s) ? atoi(s) : dflt;
}

template <typename Real>
static int march_vec(int M)
{
    int forced = env_int("BPLTV_MARCH_VEC", 0);
    const int cands64[3] = {2, 4, 1}, cands32[3] = {4, 2, 1};
    const int *c = sizeof(Real) == 8 ? cands64 : cands32;
    if (forced == 1 || forced == 2 || forced == 4) {
        if (M % forced == 0 && (M / forced + 31) / 32 * 32 <= 1024) return forced;
    }
    // prefer 16-byte accesses with <= 256 threads per column (no register cap), then
    // wider rows per thread for tall images, then anything that fits one CTA
    for (int pass = 0; pass < 2; ++pass)
        for (int k = 0; k < 3; ++k) {
            const int v = c[k];
            if (M % v) continue;
            const int nt = (M / v + 31) / 32 * 32;
            if (nt <= (pass == 0 ? 256 : 1024)) return v;
        }
    return 0;
}

// kernel pointer of one march instantiation
template <typename Real>
using MarchFn = void (*)(const MarchArgs<Real>);

template <typename Real, int VEC, int MAXT, int MINB>
static MarchFn<Real> march_fn_cfg(bool map, bool strict)
{
    if (map) return strict ? pdps_march_kernel<Real, VEC, true, true, MAXT, MINB>
                           : pdps_march_kernel<Real, VEC, true, false, MAXT, MINB>;
    return strict ? pdps_march_kernel<Real, VEC, false, true, MAXT, MINB>
                  : pdps_march_kernel<Real, VEC, false, false, MAXT, MINB>;
}

template <typename Real, int VEC>
static MarchFn<Real> march_fn_vec(int nthreads, int minb, bool map, bool strict)
{
    // ≤256 threads: ask for `minb` resident CTAs per SM (register cap 65536/(256·minb))
    if (nthreads <= 256) {
        if (minb >= 4) return march_fn_cfg<Real, VEC, 256, 4>(map, strict);
        if (minb == 3) return march_fn_cfg<Real, VEC, 256, 3>(map, strict);
        return march_fn_cfg<Real, VEC, 256, 2>(map, strict);
    }
    return march_fn_cfg<Real, VEC, 1024, 1>(map, strict);
}

template <typename Real>
static MarchFn<Real> march_fn(int vec, int nthreads, int minb, bool map, bool strict)
{
    if (vec == 4) return march_fn_vec<Real, 4>(nthreads, minb, map, strict);
    if (vec == 2) return march_fn_vec<Real, 2>(nthreads, minb, map, strict);
    return march_fn_vec<Real, 1>(nthreads, minb, map, strict);
}

template <typename Real>
static void launch_generic(const GenericArgs<Real> &a, bool map, bool strict, cudaStream_t st)
{
    const int bt = a.M >= 256 ? 256 : std::max(32, (a.M + 31) / 32 * 32);
    dim3 grid((a.M + bt - 1) / bt, a.N, a.O);
    if (map) {
        if (strict) pdps_generic_kernel<Real, true, true><<<grid, bt, 0, st>>>(a);
        else pdps_generic_kernel<Real, true, false><<<grid, bt, 0, st>>>(a);
    } else {
        if (strict) pdps_generic_kernel<Real, false, true><<<grid, bt, 0, st>>>(a);
        else pdps_generic_kernel<Real, false, false><<<grid, bt, 0, st>>>(a);
    }
}

// ---- temporally blocked march (kernel C): T iterations per launch ---------------------
// (the kernels are instantiated in tblock_f{64,32}_t{2,3,4}.cu so that they compile in parallel)
// vector width of the temporally blocked kernel for column height M (0 = shape not taken):
// 16-byte accesses when M allows, one column per CTA of at most 256 threads
template <typename Real>
static int tblock_vec(int M)
{
    const int forced = env_int("BPLTV_MARCH_VEC", 0);
    const int cands64[2] = {2, 1}, cands32[3] = {4, 2, 1};
    const int *c = sizeof(Real) == 8 ? cands64 : cands32;
    const int nc = sizeof(Real) == 8 ? 2 : 3;
    for (int k = 0; k < nc; ++k) {
        const int v = c[k];
        if (forced && v != forced) continue;
        if (M % v) continue;
        if ((M / v + 31) / 32 * 32 <= 256) return v;
    }
    return 0;
}

// Launches floor(iters/T) T-iteration passes starting at iteration `it0`; returns the number
// of iterations done (the caller finishes the remainder with kernel A).
template <typename Real, int T>
static int run_tblock_passes(Dev &d, const Real *f, int M, int N, int O, Real alpha_s, const Real *alpha_map,
                             bool strict, int it0, int iters, cudaStream_t st, int *buf, const BatchMap<Real> &bm,
                             int o0 = 0, int oc = -1)      // images [o0, o0 + oc) of the stack only (oc < 0: all)
{
    const size_t img_off = (size_t)o0 * M * N;
    if (oc >= 0) { f += img_off; O = oc; }
    const int vec = tblock_vec<Real>(M);
    const int nthreads = (M / vec + 31) / 32 * 32;
    const bool batch = bm.alpha_vec != nullptr || bm.f_mod != 0 || bm.lam_div != 0;
    TBlockFn<Real, T> fn = tblock_kernel<Real, T>(vec, alpha_map != nullptr, strict, batch);
    if (!fn) return -2;
    const size_t smem = (vec * sizeof(Real) == 16) ? tblock_ring_bytes<Real, T>(M) : 0;
    if (smem > d.smem_optin) return -1;
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -1;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, nthreads, smem) != cudaSuccess) return -1;
    per_sm = std::max(1, per_sm);
    const long long cols = (long long)N * O;
    long long grid = (long long)d.sm_count * per_sm;
    // a range shorter than the 2(T-1) halo columns it recomputes is not worth a CTA
    const int min_cols = std::max(1, env_int("BPLTV_TBLOCK_MIN_COLS", 4 * T));
    grid = std::max<long long>(1, std::min<long long>(grid, (cols + min_cols - 1) / min_cols));
    if (env_int("BPLTV_MARCH_CHUNK", 0) > 0)  // test hook: force a range length
        grid = (cols + env_int("BPLTV_MARCH_CHUNK", 0) - 1) / env_int("BPLTV_MARCH_CHUNK", 0);
    TBlockArgs<Real, T> a;
    a.f = f; a.alpha_map = alpha_map; a.M = M; a.N = N; a.O = O; a.total_cols = cols; a.alpha_s = alpha_s; a.bm = bm;
    const StepConsts<Real> *hsteps = reinterpret_cast<const StepConsts<Real> *>(d.steps_host.data());
    int done = 0;
    for (int it = it0; it + T <= it0 + iters; it += T) {
        const int bi = *buf, bo = bi ^ 1;
        a.x_in = d.x[bi].as<Real>() + img_off; a.y1_in = d.y1[bi].as<Real>() + img_off; a.y2_in = d.y2[bi].as<Real>() + img_off;
        a.x_out = d.x[bo].as<Real>() + img_off; a.y1_out = d.y1[bo].as<Real>() + img_off; a.y2_out = d.y2[bo].as<Real>() + img_off;
        for (int s = 0; s < T; ++s) a.sc[s] = hsteps[it + s];
        fn<<<(unsigned)grid, nthreads, smem, st>>>(a);
        *buf = bo;
        done += T;
        d.launches += 1;
    }
    return done;
}

// Which lower-level kernel a solve of O images of M×N takes (bpltv_pdps_opts.kernel, AUTO rules) and, for the
// temporally blocked one, its depth.
template <typename Real>
static int choose_pdps_kernel(Dev &d, int M, int N, int O, const bpltv_pdps_opts &o, int *kernel_out, int *tdepth_out)
{
    const bool strict = o.arith == BPLTV_ARITH_STRICT;
    const bool rho = o.rho != 0.0;
    int kernel = o.kernel;
    if (kernel == BPLTV_KERNEL_AUTO) kernel = env_int("BPLTV_PDPS_KERNEL", 0);
    if (kernel == BPLTV_KERNEL_AUTO) {
        if (resident_eligible<Real>(d.smem_optin, M, N) && !rho &&
            O * resident_cluster_size<Real>(d.smem_optin, M, N) <= env_int("BPLTV_RESIDENT_MAX_WAVES", 4) * d.sm_count)
            kernel = BPLTV_KERNEL_RESIDENT;
        else if (tblock_vec<Real>(M) && !rho && o.maxiter >= 2 && env_int("BPLTV_AUTO_TBLOCK", 1))
            kernel = BPLTV_KERNEL_TBLOCK;   // streaming, T iterations per HBM pass
        else
            kernel = march_vec<Real>(M) ? BPLTV_KERNEL_MARCH : BPLTV_KERNEL_GENERIC;
    }
    if (kernel == BPLTV_KERNEL_RESIDENT && (!resident_eligible<Real>(d.smem_optin, M, N) || rho))
        return fail(BPLTV_ERR_ARG, "resident PDPS kernel does not take %dx%d (rho=%g) at this precision", M, N, o.rho);
    if (kernel == BPLTV_KERNEL_MARCH && !march_vec<Real>(M))
        return fail(BPLTV_ERR_ARG, "march PDPS kernel does not take M=%d", M);
    int tdepth = 1;
    if (kernel == BPLTV_KERNEL_TBLOCK) {
        // depth when the caller leaves it open (measured, config 4, Gpixel-iter/s T = 2 / 3 / 4): fp64 strict 189 / 183 /
        // 197 and — sustained, where T = 2's HBM traffic runs the chip into its power cap — 182 vs 196; fp64 fast 189 /
        // 206 / 220; fp32 strict 370 / 346 / 331 (its four-pixel stages spill at depth 4); fp32 fast 370 / 444 / 486
        // Strict fp64 stacks that leave a depth-4 CTA (255 registers: 256 threads per SM) fewer than 160 columns go at
        // depth 2: 128 images of 256² (110 columns per CTA) 180.6 / 172.3 / 170.2 — the 2(T−1) halo columns and the
        // pipeline fill weigh more on short ranges.
        int auto_depth = (strict && sizeof(Real) == 4) ? 2 : 4;
        if (strict && sizeof(Real) == 8 && tblock_vec<Real>(M)) {
            const int nthreads = (M / tblock_vec<Real>(M) + 31) / 32 * 32;
            const long long cols_per_cta = (long long)N * O * nthreads / ((long long)d.sm_count * 256);
            if (cols_per_cta < 160) auto_depth = 2;
        }
        tdepth = o.tblock > 0 ? o.tblock : env_int("BPLTV_TBLOCK_T", auto_depth);
        if (tdepth < 1 || tdepth > 4) return fail(BPLTV_ERR_ARG, "temporal blocking depth must be 1..4 (got %d)", tdepth);
        if (!tblock_vec<Real>(M) || rho)
            return fail(BPLTV_ERR_ARG, "temporally blocked PDPS kernel does not take M=%d (rho=%g)", M, o.rho);
    }
    *kernel_out = kernel; *tdepth_out = tdepth;
    return 0;
}

// The pipelined form of a denoise call with host buffers (PipeIO): decided before the upload.  fp64 contexts, pinned
// caller buffers (pageable ones go through the staging threads), the temporally blocked kernel with a whole number of
// passes, a stack large enough for the copies to matter.  BPLTV_PIPE_IO=0 switches it off; BPLTV_PIPE_MIN_MB,
// BPLTV_PIPE_CHUNKS, BPLTV_PIPE_PASSES tune it (tests).
template <typename Real>
static bool pipe_eligible(Dev &d, int M, int N, int O, const bpltv_pdps_opts &o, int kernel, int tdepth, const double *h_in,
                          double *h_out, bool allow_pageable, PipeIO *pio)
{
    if (sizeof(Real) != 8 || !h_in || !h_out || !env_int("BPLTV_PIPE_IO", 1)) return false;
    if (kernel != BPLTV_KERNEL_TBLOCK || tdepth < 2 || o.maxiter % tdepth != 0) return false;
    // Pageable caller buffers (a Julia Array) travel through the pinned slots (HostStage) chunk by chunk on the copy
    // stream.  There the staging threads bind the copies (≈ 1.5-1.9 ms per third of config 4's stack against 0.8 ms of
    // DMA), so a chunk phase has to be longer to cover them: 14 passes per chunk instead of 6.  Measured at config 4
    // (e2e Gpixel-iter/s): pageable K×q = 3×6 175.5 (= serial), 3×14 181.7, 3×18 179.1, 4×12 180.0, 6×8 172.9; pinned 3×6
    // 190.1, 3×14 186.5.  BPLTV_PIPE_PAGEABLE=0 keeps pageable buffers on the serial path.
    const bool pg_in = host_is_pageable(h_in), pg_out = host_is_pageable(h_out);
    // (a staged copy occupies the calling thread: in a context of several devices it would hold back the other devices'
    // work, so pageable buffers are pipelined in single-device contexts only)
    if ((pg_in || pg_out) && (!allow_pageable || !env_int("BPLTV_PIPE_PAGEABLE", 1))) return false;
    const int K = std::max(2, std::min(8, env_int("BPLTV_PIPE_CHUNKS", 3)));
    const int q = std::max(1, env_int("BPLTV_PIPE_PASSES", (pg_in || pg_out) ? 14 : 6));
    if (o.maxiter / tdepth < 4 * q || O < 2 * K) return false;
    if ((size_t)M * N * O * 8 < ((size_t)env_int("BPLTV_PIPE_MIN_MB", 32) << 20)) return false;
    pio->stage_in = pg_in && env_int("BPLTV_HOST_STAGING", 1) && d.hstage.init();
    pio->stage_out = pg_out && env_int("BPLTV_HOST_STAGING", 1) && d.hstage.init();
    if ((pg_in && !pio->stage_in) || (pg_out && !pio->stage_out)) return false;
    if (!d.copy_stream && cudaStreamCreateWithFlags(&d.copy_stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return false; }
    for (auto &e : d.pipe_ev)
        if (!e && cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return false; }
    pio->h_in = h_in; pio->h_out = h_out; pio->chunks = K; pio->q = q;
    return true;
}

// All passes of a pipelined denoise call (see PipeIO).  f = d.fbuf (filled here, chunk by chunk, on the copy stream).
template <typename Real, int T>
static int run_tblock_pipelined(Dev &d, Real *f, int M, int N, int O, Real alpha_s, const Real *alpha_map, bool strict,
                                int maxiter, int init_mode, cudaStream_t st, int *buf, const BatchMap<Real> &bm, const PipeIO &pio)
{
    const int K = pio.chunks, q = pio.q, P = maxiter / T;
    const size_t plane = (size_t)M * N;
    cudaStream_t cs = d.copy_stream;
    cudaEvent_t ev_start = d.pipe_ev[16], ev_end = d.pipe_ev[17];
    // the copy stream joins: nothing enqueued earlier on `st` may still read the buffers the uploads overwrite
    if (cudaEventRecord(ev_start, st) != cudaSuccess || cudaStreamWaitEvent(cs, ev_start, 0) != cudaSuccess) return -1;
    // (a staged upload occupies the calling thread until the caller's chunk has been read: the passes of the chunks that
    // are already on the device were enqueued before and run meanwhile)
    auto upload = [&](size_t off, size_t cnt) -> cudaError_t {
        char *dst = reinterpret_cast<char *>(reinterpret_cast<double *>(f) + off);
        char *src = reinterpret_cast<char *>(const_cast<double *>(pio.h_in + off));
        if (pio.stage_in && cnt * 8 >= HostStage::MIN_BYTES) return staged_copy(d.hstage, d.id, dst, src, cnt * 8, cs, true);
        return cudaMemcpyAsync(dst, src, cnt * 8, cudaMemcpyHostToDevice, cs);
    };
    auto download = [&](size_t off, size_t cnt, const Real *u) -> cudaError_t {
        char *src = reinterpret_cast<char *>(const_cast<double *>(reinterpret_cast<const double *>(u) + off));
        char *dst = reinterpret_cast<char *>(pio.h_out + off);
        if (pio.stage_out && cnt * 8 >= HostStage::MIN_BYTES) return staged_copy(d.hstage, d.id, src, dst, cnt * 8, cs, false);
        return cudaMemcpyAsync(dst, src, cnt * 8, cudaMemcpyDeviceToHost, cs);
    };
    const int b0 = *buf;
    int b_end = b0;
    for (int k = 0; k < K; ++k) {
        const int o0 = (int)((long long)O * k / K), o1 = (int)((long long)O * (k + 1) / K);
        const size_t off = plane * o0, cnt = plane * (o1 - o0);
        if (upload(off, cnt) != cudaSuccess) return -1;
        if (cudaEventRecord(d.pipe_ev[k], cs) != cudaSuccess) return -1;
        if (cudaStreamWaitEvent(st, d.pipe_ev[k], 0) != cudaSuccess) return -1;
        if (init_mode && cudaMemcpyAsync(d.x[b0].as<Real>() + off, f + off, cnt * sizeof(Real), cudaMemcpyDeviceToDevice, st) != cudaSuccess) return -1;
        int b = b0;
        const int rc = run_tblock_passes<Real, T>(d, f, M, N, O, alpha_s, alpha_map, strict, 0, q * T, st, &b, bm, o0, o1 - o0);
        if (rc < 0) return rc;
        b_end = b;
    }
    *buf = b_end;
    {
        const int rc = run_tblock_passes<Real, T>(d, f, M, N, O, alpha_s, alpha_map, strict, q * T, (P - 2 * q) * T, st, buf, bm);
        if (rc < 0) return rc;
    }
    const int b1 = *buf;
    for (int k = 0; k < K; ++k) {
        const int o0 = (int)((long long)O * k / K), o1 = (int)((long long)O * (k + 1) / K);
        const size_t off = plane * o0, cnt = plane * (o1 - o0);
        int b = b1;
        const int rc = run_tblock_passes<Real, T>(d, f, M, N, O, alpha_s, alpha_map, strict, (P - q) * T, q * T, st, &b, bm, o0, o1 - o0);
        if (rc < 0) return rc;
        b_end = b;
        if (cudaEventRecord(d.pipe_ev[8 + k], st) != cudaSuccess) return -1;
    }
    *buf = b_end;
    // the downloads follow their chunks (all passes are enqueued by now: a staged download may occupy this thread)
    for (int k = 0; k < K; ++k) {
        const int o0 = (int)((long long)O * k / K), o1 = (int)((long long)O * (k + 1) / K);
        const size_t off = plane * o0, cnt = plane * (o1 - o0);
        if (cudaStreamWaitEvent(cs, d.pipe_ev[8 + k], 0) != cudaSuccess) return -1;
        if (download(off, cnt, d.x[b_end].as<Real>()) != cudaSuccess) return -1;
    }
    // `st` ends behind the last download: whoever synchronises the context's stream has the result in the caller's buffer
    if (cudaEventRecord(ev_end, cs) != cudaSuccess || cudaStreamWaitEvent(st, ev_end, 0) != cudaSuccess) return -1;
    return P * T;
}

// Runs opts.maxiter iterations on `f` (device, M×N×O Reals).  On return (stream
// order) the denoised stack is in *u_result (one of the ping-pong buffers).
template <typename Real>
static int run_pdps(Dev &d, const Real *f, int M, int N, int O, double alpha_s, const Real *alpha_map,
                    const bpltv_pdps_opts &o, cudaStream_t st, const Real **u_result, int *kernel_used,
                    int *depth_used = nullptr, const BatchMap<Real> *bmap = nullptr, const PipeIO *pipe = nullptr)
{
    if (O == 0) { *u_result = nullptr; return 0; }
    const size_t n = (size_t)M * N * O;
    for (int b = 0; b < 2; ++b) {
        RC_TRY(d.x[b].ensure(n * sizeof(Real)));
        RC_TRY(d.y1[b].ensure(n * sizeof(Real)));
        RC_TRY(d.y2[b].ensure(n * sizeof(Real)));
    }
    const bool strict = o.arith == BPLTV_ARITH_STRICT;
    const bool rho = o.rho != 0.0;
    const bool map = alpha_map != nullptr;
    const BatchMap<Real> bm = bmap ? *bmap : BatchMap<Real>();

    int kernel = 0, tdepth = 1;
    RC_TRY(choose_pdps_kernel<Real>(d, M, N, O, o, &kernel, &tdepth));
    *kernel_used = kernel;
    if (depth_used) *depth_used = tdepth;

    RC_TRY(upload_steps<Real>(d, o, st));
    const StepConsts<Real> *steps = d.steps.as<StepConsts<Real>>();

    if (kernel == BPLTV_KERNEL_RESIDENT) {
        // whole solve in one launch; x⁰/y⁰ are formed on chip
        ResidentArgs<Real> a;
        a.f = f; a.u_out = d.x[0].as<Real>(); a.alpha_map = alpha_map; a.steps = steps;
        a.maxiter = o.maxiter; a.M = M; a.N = N; a.O = O; a.NC = 0; a.alpha_s = (Real)alpha_s;
        a.init_mode = o.init_mode; a.bm = bm;
        cudaError_t e = launch_resident<Real>(a, d.smem_optin, map, strict, st);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(BPLTV_ERR_CUDA, "resident PDPS launch failed: %s", cudaGetErrorString(e));
        }
        d.launches += 1;
        *u_result = d.x[0].as<Real>();
        return 0;
    }

    // x⁰ = 0 | f (S3), y⁰ = 0
    if (o.init_mode && pipe) {
        // x⁰ = f chunk by chunk, as the uploads arrive (run_tblock_pipelined)
    } else if (o.init_mode) {
        const int Of = bm.f_mod ? bm.f_mod : O;   // a sweep's virtual stack repeats the Of images of f
        for (int v0 = 0; v0 < O; v0 += Of)
            CU_TRY(cudaMemcpyAsync(d.x[0].as<Real>() + (size_t)v0 * M * N, f,
                                   (size_t)std::min(Of, O - v0) * M * N * sizeof(Real), cudaMemcpyDeviceToDevice, st));
    } else CU_TRY(cudaMemsetAsync(d.x[0].p, 0, n * sizeof(Real), st));
    CU_TRY(cudaMemsetAsync(d.y1[0].p, 0, n * sizeof(Real), st));
    CU_TRY(cudaMemsetAsync(d.y2[0].p, 0, n * sizeof(Real), st));

    int buf = 0;       // ping-pong buffer holding the current state
    int it_begin = 0;  // iterations already done
    if (kernel == BPLTV_KERNEL_TBLOCK && tdepth > 1) {
        int done = 0;
        if (pipe) {
            Real *fw = const_cast<Real *>(f);
            if (tdepth == 2) done = run_tblock_pipelined<Real, 2>(d, fw, M, N, O, (Real)alpha_s, alpha_map, strict, o.maxiter, o.init_mode, st, &buf, bm, *pipe);
            else if (tdepth == 3) done = run_tblock_pipelined<Real, 3>(d, fw, M, N, O, (Real)alpha_s, alpha_map, strict, o.maxiter, o.init_mode, st, &buf, bm, *pipe);
            else done = run_tblock_pipelined<Real, 4>(d, fw, M, N, O, (Real)alpha_s, alpha_map, strict, o.maxiter, o.init_mode, st, &buf, bm, *pipe);
        }
        else if (tdepth == 2) done = run_tblock_passes<Real, 2>(d, f, M, N, O, (Real)alpha_s, alpha_map, strict, 0, o.maxiter, st, &buf, bm);
        else if (tdepth == 3) done = run_tblock_passes<Real, 3>(d, f, M, N, O, (Real)alpha_s, alpha_map, strict, 0, o.maxiter, st, &buf, bm);
        else done = run_tblock_passes<Real, 4>(d, f, M, N, O, (Real)alpha_s, alpha_map, strict, 0, o.maxiter, st, &buf, bm);
        if (done == -2) return fail(BPLTV_ERR_ARG, "λ-sweeps through the temporally blocked kernel are built for depths 2 and 4 only");
        if (done < 0) { cudaGetLastError(); return fail(BPLTV_ERR_CUDA, "temporally blocked PDPS kernel: occupancy query failed"); }
        it_begin = done;  // the remainder (< T iterations) runs as single-iteration passes below
    }

    if (kernel == BPLTV_KERNEL_MARCH || kernel == BPLTV_KERNEL_TBLOCK) {
        const int vec = march_vec<Real>(M);
        const int nthreads = (M / vec + 31) / 32 * 32;
        const int minb = env_int("BPLTV_MARCH_MINB", 4);
        MarchFn<Real> fn = march_fn<Real>(vec, nthreads, minb, map, strict);
        // one balanced wave: grid = #SM × resident CTAs per SM, never more CTAs than columns
        int per_sm = 0;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, nthreads, 0));
        per_sm = std::max(1, per_sm);
        const long long cols = (long long)N * O;
        long long grid = (long long)d.sm_count * per_sm;
        const int min_cols = std::max(1, env_int("BPLTV_MARCH_MIN_COLS", 4));
        grid = std::max<long long>(1, std::min<long long>(grid, (cols + min_cols - 1) / min_cols));
        if (env_int("BPLTV_MARCH_CHUNK", 0) > 0)  // test hook: force a range length
            grid = (cols + env_int("BPLTV_MARCH_CHUNK", 0) - 1) / env_int("BPLTV_MARCH_CHUNK", 0);
        MarchArgs<Real> a;
        a.f = f; a.alpha_map = alpha_map; a.M = M; a.N = N; a.O = O; a.total_cols = cols;
        a.prefetch_dist = env_int("BPLTV_MARCH_PREFETCH", 0);
        a.alpha_s = (Real)alpha_s; a.rho = (Real)o.rho; a.bm = bm;
        const StepConsts<Real> *hsteps = reinterpret_cast<const StepConsts<Real> *>(d.steps_host.data());
        for (int it = it_begin; it < o.maxiter; ++it) {
            const int bi = buf, bo = bi ^ 1;
            a.x_in = d.x[bi].as<Real>(); a.y1_in = d.y1[bi].as<Real>(); a.y2_in = d.y2[bi].as<Real>();
            a.x_out = d.x[bo].as<Real>(); a.y1_out = d.y1[bo].as<Real>(); a.y2_out = d.y2[bo].as<Real>();
            a.sc = hsteps[it];
            fn<<<(unsigned)grid, nthreads, 0, st>>>(a);
            buf = bo;
        }
        d.launches += o.maxiter - it_begin;
    } else {
        GenericArgs<Real> a;
        a.f = f; a.alpha_map = alpha_map; a.steps = steps; a.M = M; a.N = N; a.O = O;
        a.alpha_s = (Real)alpha_s; a.rho = (Real)o.rho; a.bm = bm;
        if (N > 65535 || O > 65535) return fail(BPLTV_ERR_ARG, "generic kernel: N and O must be <= 65535");
        for (int it = 0; it < o.maxiter; ++it) {
            const int bi = it & 1, bo = bi ^ 1;
            a.x_in = d.x[bi].as<Real>(); a.y1_in = d.y1[bi].as<Real>(); a.y2_in = d.y2[bi].as<Real>();
            a.x_out = d.x[bo].as<Real>(); a.y1_out = d.y1[bo].as<Real>(); a.y2_out = d.y2[bo].as<Real>();
            a.it = it;
            launch_generic<Real>(a, map, strict, st);
        }
        buf = o.maxiter & 1;
        d.launches += o.maxiter;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BPLTV_ERR_CUDA, "PDPS kernel launch failed: %s", cudaGetErrorString(e));
    *u_result = d.x[buf].as<Real>();
    return 0;
}

// λ handling: scalar → alpha_s; grid → device map (PatchOp up-sampling, S7)
template <typename Real>
static int prepare_lambda(Dev &d, const double *lam, int lm, int ln, int M, int N, cudaStream_t st,
                          double *alpha_s, const Real **alpha_map)
{
    if (lm == 1 && ln == 1) {
        *alpha_s = lam[0];
        *alpha_map = nullptr;
        return 0;
    }
    RC_TRY(d.lam_dev.ensure((size_t)lm * ln * sizeof(double)));
    RC_TRY(d.amap.ensure((size_t)M * N * sizeof(Real)));
    CU_TRY(cudaMemcpyAsync(d.lam_dev.p, lam, (size_t)lm * ln * sizeof(double), cudaMemcpyHostToDevice, st));
    const int n = M * N;
    patch_upsample_kernel<Real><<<(n + 255) / 256, 256, 0, st>>>(d.lam_dev.as<double>(), lm, ln, d.amap.as<Real>(), M, N);
    d.launches += 1;
    *alpha_s = 0.0;
    *alpha_map = d.amap.as<Real>();
    return 0;
}

static int check_lambda(const double *lam, int lm, int ln)
{
    if (!lam || lm < 1 || ln < 1) return fail(BPLTV_ERR_ARG, "lambda grid must be at least 1x1");
    for (int k = 0; k < lm * ln; ++k)
        if (!(lam[k] >= 0.0) || !std::isfinite(lam[k]))
            return fail(BPLTV_ERR_ARG, "lambda[%d] = %g must be finite and >= 0", k, lam[k]);
    return 0;
}

static int check_pdps_opts(const bpltv_pdps_opts &o)
{
    if (!(o.tau0 > 0) || !(o.sigma0 > 0) || !(o.opnorm > 0) || o.maxiter < 0 || o.rho < 0)
        return fail(BPLTV_ERR_ARG, "invalid PDPS options (tau0=%g sigma0=%g opnorm=%g rho=%g maxiter=%d)", o.tau0,
                    o.sigma0, o.opnorm, o.rho, o.maxiter);
    if (!(o.tau0 * o.sigma0 < 1.0))
        return fail(BPLTV_ERR_ARG, "PDPS step condition tau0*sigma0 < 1 violated (%g)", o.tau0 * o.sigma0);
    if (o.arith != BPLTV_ARITH_STRICT && o.arith != BPLTV_ARITH_FAST) return fail(BPLTV_ERR_ARG, "bad arith mode");
    return 0;
}

// host double stack (M×N×count) → device Real buffer
template <typename Real>
static int upload_stack(Dev &d, const double *h, size_t n, DBuf &dst, cudaStream_t st)
{
    RC_TRY(dst.ensure(std::max<size_t>(n, 1) * sizeof(Real)));
    if (n == 0) return 0;
    if (sizeof(Real) != 8) RC_TRY(d.stage.ensure(n * 8));
    void *target = sizeof(Real) == 8 ? dst.p : d.stage.p;
    const bool staged = n * 8 >= HostStage::MIN_BYTES && env_int("BPLTV_HOST_STAGING", 1) && host_is_pageable(h) && d.hstage.init();
    if (staged) CU_TRY(staged_copy(d.hstage, d.id, static_cast<char *>(target), reinterpret_cast<char *>(const_cast<double *>(h)), n * 8, st, true));
    else CU_TRY(cudaMemcpyAsync(target, h, n * 8, cudaMemcpyHostToDevice, st));
    if (sizeof(Real) != 8) {
        const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
        convert_kernel<Real, double><<<blocks, 256, 0, st>>>(d.stage.as<double>(), dst.as<Real>(), n);
        d.launches += 1;
    }
    return 0;
}

template <typename Real>
static int download_stack(Dev &d, const Real *src, size_t n, double *h, cudaStream_t st)
{
    if (n == 0) return 0;
    const void *source = src;
    if (sizeof(Real) != 8) {
        RC_TRY(d.stage.ensure(n * 8));
        const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
        convert_kernel<double, Real><<<blocks, 256, 0, st>>>(src, d.stage.as<double>(), n);
        d.launches += 1;
        source = d.stage.p;
    }
    // a pageable destination: through the pinned slots (the call then returns with the data in `h`, which every
    // host-pointer entry point guarantees at its end anyway)
    const bool staged = n * 8 >= HostStage::MIN_BYTES && env_int("BPLTV_HOST_STAGING", 1) && host_is_pageable(h) && d.hstage.init();
    if (staged) CU_TRY(staged_copy(d.hstage, d.id, static_cast<char *>(const_cast<void *>(source)), reinterpret_cast<char *>(h), n * 8, st, false));
    else CU_TRY(cudaMemcpyAsync(h, source, n * 8, cudaMemcpyDeviceToHost, st));
    return 0;
}

// cost of this device's shard into scalars[0] (device double)
template <typename Real>
static int run_cost(Dev &d, const Real *u, const Real *ubar, size_t n, double *d_out, cudaStream_t st)
{
    const int blocks = (int)std::max<size_t>(1, std::min<size_t>((n + 256 * 8 - 1) / (256 * 8), 1024));
    RC_TRY(d.partials.ensure(1024 * sizeof(double)));
    cost_partial_kernel<Real><<<blocks, 256, 0, st>>>(u, ubar, n, d.partials.as<double>());
    sum_partials_kernel<<<1, 256, 0, st>>>(d.partials.as<double>(), blocks, 0.5, d_out);
    d.launches += 2;
    return 0;
}

// ---------------------------------------------------------------------------
// per-precision implementations of the entry points
// ---------------------------------------------------------------------------
static float ev_ms(cudaEvent_t a, cudaEvent_t b)
{
    float ms = 0;
    if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); return 0; }
    return ms;
}

// Phase boundaries of one call on one device, recorded as Dev::ev[mark] on the stream the work goes to.  A call marks
// the boundaries it passes; a phase runs from the previous mark to its own, and a phase that is not marked stays 0 in
// the stats.  ms_total runs from MARK_BEGIN to MARK_DOWNLOAD.
enum Mark { MARK_BEGIN, MARK_UPLOAD, MARK_SOLVE, MARK_COST, MARK_GRADIENT, MARK_DOWNLOAD, N_MARKS };

static int mark(Dev &d, Mark m, cudaStream_t st)
{
    CU_TRY(cudaEventRecord(d.ev[m], st));
    d.marked |= 1u << m;
    return 0;
}

// kernel launches and phase times (maxima over the devices) of one device's part of a call, after its stream has
// been synchronised
static void fold_device_stats(bpltv_stats &s, const Dev &d)
{
    double *ms[N_MARKS] = {nullptr, &s.ms_upload, &s.ms_pdps, &s.ms_cost, &s.ms_gradient, &s.ms_download};
    int prev = -1;
    for (int m = 0; m < N_MARKS; ++m) {
        if (!(d.marked >> m & 1)) continue;
        if (prev >= 0) *ms[m] = std::max<double>(*ms[m], ev_ms(d.ev[prev], d.ev[m]));
        prev = m;
    }
    const unsigned ends = 1u << MARK_BEGIN | 1u << MARK_DOWNLOAD;
    if ((d.marked & ends) == ends) s.ms_total = std::max<double>(s.ms_total, ev_ms(d.ev[MARK_BEGIN], d.ev[MARK_DOWNLOAD]));
    s.kernel_launches += d.launches;
}

// The three passes of a host-pointer entry point over the context's devices, each in device order:
//  1. enqueue(d, di): the shard's uploads, solve, cost and gradient, the all-reduce and the D2H copy of [cost, grad];
//  2. download(d, di): the downloads of u.  A pass of their own: a pageable destination makes a download wait for its
//     device, which must not hold back the other devices' work;
//  3. fold(d, di), once the device's stream has been synchronised: the host sums (in device order, hence
//     deterministic) and the stats.
// skip_empty: devices whose shard of the resident dataset has no images take no part.
template <class Enqueue, class Download, class Fold>
static int run_sharded(bpltv_ctx *ctx, bool skip_empty, Enqueue &&enqueue, Download &&download, Fold &&fold)
{
    auto each = [&](auto &&pass) {
        for (int di = 0; di < (int)ctx->devs.size(); ++di) {
            Dev &d = ctx->devs[di];
            if (skip_empty && d.O == 0) continue;
            CU_TRY(cudaSetDevice(d.id));
            RC_TRY(pass(d, di));
        }
        return 0;
    };
    RC_TRY(each([&](Dev &d, int di) {
        d.launches = 0;
        d.marked = 0;
        d.last_grad = Dev::GRAD_NONE;
        return enqueue(d, di);
    }));
    RC_TRY(each(download));
    return each([&](Dev &d, int di) {
        CU_TRY(cudaStreamSynchronize(d.stream));
        fold(d, di);
        return 0;
    });
}

static int no_download(Dev &, int) { return 0; }

// second pass of the evaluations: this device's shard of the resident dataset's u (u_out may be NULL)
template <typename Real>
static int download_resident_u(Dev &d, const Real *u, double *u_out)
{
    const size_t plane = (size_t)d.M * d.N;
    if (u_out && d.O > 0) RC_TRY(download_stack<Real>(d, u, plane * d.O, u_out + plane * d.o_begin, d.stream));
    return mark(d, MARK_DOWNLOAD, d.stream);
}

template <typename Real>
static int denoise_impl(bpltv_ctx *ctx, const double *noisy, int M, int N, int O, const double *lam, int lm, int ln,
                        const bpltv_pdps_opts &o, double *u_out)
{
    const int ndev = (int)ctx->devs.size();
    const size_t plane = (size_t)M * N;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    std::vector<const Real *> us(ndev, nullptr);
    std::vector<int> obs(ndev, 0), ocs(ndev, 0);
    std::vector<char> piped(ndev, 0);      // the solve carried its own copies (PipeIO)
    auto enqueue = [&](Dev &d, int di) {
        int &ob = obs[di], &oc = ocs[di];
        if (noisy) shard_range(O, ndev, di, ob, oc);
        else { ob = d.o_begin; oc = d.O; }
        cudaStream_t st = d.stream;
        RC_TRY(mark(d, MARK_BEGIN, st));
        PipeIO pio;
        if (noisy && oc > 0) {
            int k_ = 0, t_ = 1;
            RC_TRY(choose_pdps_kernel<Real>(d, M, N, oc, o, &k_, &t_));
            piped[di] = pipe_eligible<Real>(d, M, N, oc, o, k_, t_, noisy + plane * ob, u_out + plane * ob, ndev == 1, &pio);
        }
        const Real *f = d.noisy.as<Real>();
        if (noisy) {
            if (piped[di]) RC_TRY(d.fbuf.ensure(plane * oc * sizeof(Real)));      // filled chunk by chunk under the first passes
            else RC_TRY(upload_stack<Real>(d, noisy + plane * ob, plane * oc, d.fbuf, st));
            f = d.fbuf.as<Real>();
        }
        RC_TRY(mark(d, MARK_UPLOAD, st));
        double alpha_s; const Real *amap;
        RC_TRY(prepare_lambda<Real>(d, lam, lm, ln, M, N, st, &alpha_s, &amap));
        int used = 0, depth = 1;
        RC_TRY(run_pdps<Real>(d, f, M, N, oc, alpha_s, amap, o, st, &us[di], &used, &depth, nullptr, piped[di] ? &pio : nullptr));
        ctx->stats.pdps_kernel_used = used;
        ctx->stats.tblock_depth = depth;
        return mark(d, MARK_SOLVE, st);
    };
    auto download = [&](Dev &d, int di) {
        if (ocs[di] > 0 && !piped[di]) RC_TRY(download_stack<Real>(d, us[di], plane * ocs[di], u_out + plane * obs[di], d.stream));
        return mark(d, MARK_DOWNLOAD, d.stream);
    };
    RC_TRY(run_sharded(ctx, false, enqueue, download, [&](Dev &d, int) { fold_device_stats(ctx->stats, d); }));
    ctx->stats.pdps_iterations = o.maxiter;
    ctx->stats.pixel_iterations = (long long)plane * O * o.maxiter;
    ctx->stats.n_devices = ndev;
    return 0;
}

// ---------------------------------------------------------------------------
// sum-of-regularisers path (SumRegsLearningFunction.jl): lower-level solve
// ---------------------------------------------------------------------------
// λ handling: lm = ln = 1 → three scalars; otherwise lm×ln×3 grids up-sampled to three M×N maps
template <typename Real>
static int prepare_lambda3(Dev &d, const double *lam, int lm, int ln, int M, int N, cudaStream_t st, Real (&alpha)[3],
                           const Real **amap)
{
    if (lm == 1 && ln == 1) {
        for (int k = 0; k < 3; ++k) alpha[k] = (Real)lam[k];
        *amap = nullptr;
        return 0;
    }
    const size_t ng = (size_t)lm * ln;
    RC_TRY(d.lam_dev.ensure(3 * ng * sizeof(double)));
    RC_TRY(d.amap.ensure((size_t)3 * M * N * sizeof(Real)));
    CU_TRY(cudaMemcpyAsync(d.lam_dev.p, lam, 3 * ng * sizeof(double), cudaMemcpyHostToDevice, st));
    const size_t tot = (size_t)3 * M * N;
    patch_upsample_sets_kernel<Real><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d.lam_dev.as<double>(), 3, lm, ln,
                                                                                d.amap.as<Real>(), M, N);
    d.launches += 1;
    for (int k = 0; k < 3; ++k) alpha[k] = 0;
    *amap = d.amap.as<Real>();
    return 0;
}

// Runs o.maxiter iterations of the three-operator PDPS on `f`; the result is d.x[0].
template <typename Real>
static int run_sumregs_pdps(Dev &d, const Real *f, int M, int N, int O, const Real (&alpha)[3], const Real *amap,
                            const bpltv_pdps_opts &o, cudaStream_t st, const Real **u_result)
{
    if (O == 0) { *u_result = nullptr; return 0; }
    if (o.rho != 0.0) return fail(BPLTV_ERR_ARG, "the sum-of-regularisers solve has no rho path (the reference fixes rho = 0)");
    const size_t n = (size_t)M * N * O;
    RC_TRY(d.x[0].ensure(n * sizeof(Real)));
    RC_TRY(d.x[1].ensure(n * sizeof(Real)));
    RC_TRY(d.sry.ensure(6 * n * sizeof(Real)));
    RC_TRY(upload_steps<Real>(d, o, st));
    const bool strict = o.arith == BPLTV_ARITH_STRICT;
    // Few images of a size that fits on chip: the whole solve in ONE launch, one image per thread-block
    // cluster (sumregs_resident_kernel); otherwise two streaming launches per iteration.  o.kernel:
    // GENERIC / MARCH force the streaming pair, RESIDENT requires the resident kernel, AUTO decides.
    int kern = o.kernel;
    if (kern == BPLTV_KERNEL_AUTO) kern = env_int("BPLTV_PDPS_KERNEL", 0);
    const bool want_res = kern == BPLTV_KERNEL_RESIDENT ||
                          (kern == BPLTV_KERNEL_AUTO && (long long)O * 8 <= (long long)env_int("BPLTV_RESIDENT_MAX_WAVES", 4) * d.sm_count);
    if (want_res && o.maxiter > 0) {
        SumRegsResArgs<Real> ra;
        ra.f = f; ra.u_out = d.x[0].as<Real>(); ra.amap = amap; ra.steps = d.steps.as<StepConsts<Real>>();
        for (int k = 0; k < 3; ++k) ra.alpha[k] = alpha[k];
        ra.maxiter = o.maxiter; ra.M = M; ra.N = N; ra.O = O; ra.init_mode = o.init_mode; ra.NC = 0;
        cudaError_t re = launch_sumregs_resident<Real>(ra, d.smem_optin, amap != nullptr, strict, st);
        if (re == cudaSuccess) {
            d.launches += 1;
            *u_result = d.x[0].as<Real>();
            return 0;
        }
        cudaGetLastError();
        if (kern == BPLTV_KERNEL_RESIDENT)
            return fail(BPLTV_ERR_ARG, "the resident sum-of-regularisers kernel does not take this shape: %s", cudaGetErrorString(re));
    }
    if (o.init_mode) CU_TRY(cudaMemcpyAsync(d.x[0].p, f, n * sizeof(Real), cudaMemcpyDeviceToDevice, st));
    else CU_TRY(cudaMemsetAsync(d.x[0].p, 0, n * sizeof(Real), st));
    CU_TRY(cudaMemsetAsync(d.sry.p, 0, 6 * n * sizeof(Real), st));
    SumRegsArgs<Real> a;
    a.x = d.x[0].as<Real>(); a.xb = d.x[1].as<Real>(); a.f = f; a.y = d.sry.as<Real>(); a.amap = amap;
    for (int k = 0; k < 3; ++k) a.alpha[k] = alpha[k];
    a.M = M; a.N = N; a.O = O;
    const unsigned grid = (unsigned)((n + 255) / 256);
    const StepConsts<Real> *hsteps = reinterpret_cast<const StepConsts<Real> *>(d.steps_host.data());
    for (int it = 0; it < o.maxiter; ++it) {
        a.sc = hsteps[it];
        if (strict) sumregs_primal_kernel<Real, true><<<grid, 256, 0, st>>>(a);
        else sumregs_primal_kernel<Real, false><<<grid, 256, 0, st>>>(a);
        if (amap) {
            if (strict) sumregs_dual_kernel<Real, true, true><<<grid, 256, 0, st>>>(a);
            else sumregs_dual_kernel<Real, true, false><<<grid, 256, 0, st>>>(a);
        } else {
            if (strict) sumregs_dual_kernel<Real, false, true><<<grid, 256, 0, st>>>(a);
            else sumregs_dual_kernel<Real, false, false><<<grid, 256, 0, st>>>(a);
        }
    }
    d.launches += 2LL * o.maxiter;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(BPLTV_ERR_CUDA, "sumregs PDPS kernel launch failed: %s", cudaGetErrorString(e));
    *u_result = d.x[0].as<Real>();
    return 0;
}

template <typename Real>
static int sumregs_denoise_impl(bpltv_ctx *ctx, const double *noisy, int M, int N, int O, const double *lam, int lm,
                                int ln, const bpltv_pdps_opts &o, double *u_out)
{
    const int ndev = (int)ctx->devs.size();
    const size_t plane = (size_t)M * N;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    std::vector<const Real *> us(ndev, nullptr);
    std::vector<int> obs(ndev, 0), ocs(ndev, 0);
    auto enqueue = [&](Dev &d, int di) {
        int &ob = obs[di], &oc = ocs[di];
        if (noisy) shard_range(O, ndev, di, ob, oc);
        else { ob = d.o_begin; oc = d.O; }
        cudaStream_t st = d.stream;
        RC_TRY(mark(d, MARK_BEGIN, st));
        const Real *f = d.noisy.as<Real>();
        if (noisy) {
            RC_TRY(upload_stack<Real>(d, noisy + plane * ob, plane * oc, d.fbuf, st));
            f = d.fbuf.as<Real>();
        }
        RC_TRY(mark(d, MARK_UPLOAD, st));
        Real alpha[3]; const Real *amap;
        RC_TRY(prepare_lambda3<Real>(d, lam, lm, ln, M, N, st, alpha, &amap));
        RC_TRY(run_sumregs_pdps<Real>(d, f, M, N, oc, alpha, amap, o, st, &us[di]));
        return mark(d, MARK_SOLVE, st);
    };
    auto download = [&](Dev &d, int di) {
        if (ocs[di] > 0) RC_TRY(download_stack<Real>(d, us[di], plane * ocs[di], u_out + plane * obs[di], d.stream));
        return mark(d, MARK_DOWNLOAD, d.stream);
    };
    RC_TRY(run_sharded(ctx, false, enqueue, download, [&](Dev &d, int) { fold_device_stats(ctx->stats, d); }));
    ctx->stats.pdps_iterations = o.maxiter;
    ctx->stats.pixel_iterations = (long long)plane * O * o.maxiter;
    ctx->stats.n_devices = ndev;
    ctx->stats.tblock_depth = 1;
    return 0;
}

template <typename Real>
static int set_dataset_impl(bpltv_ctx *ctx, const double *truth, const double *noisy, int M, int N, int O)
{
    const int ndev = (int)ctx->devs.size();
    const size_t plane = (size_t)M * N;
    auto enqueue = [&](Dev &d, int di) {
        int ob, oc;
        shard_range(O, ndev, di, ob, oc);
        d.M = M; d.N = N; d.O = oc; d.o_begin = ob;
        RC_TRY(upload_stack<Real>(d, truth + plane * ob, plane * oc, d.truth, d.stream));
        return upload_stack<Real>(d, noisy + plane * ob, plane * oc, d.noisy, d.stream);
    };
    RC_TRY(run_sharded(ctx, false, enqueue, no_download, [](Dev &, int) {}));
    ctx->M = M; ctx->N = N; ctx->O = O; ctx->have_dataset = true;
    return 0;
}

// ---------------------------------------------------------------------------
// gradients: which solver takes the adjoint systems
// ---------------------------------------------------------------------------
// gradient / gradient_reg of the TV learning function.  The regularised branch has two implementations:
// the multiplier-space banded Cholesky of gradient.cuh and the node-space band LU of lu_band.cuh
// (n² unknowns with half-bandwidth n instead of ≤ 2n² modes with half-bandwidth ≤ 2n+1; its cost does not grow
// with the number of flat pixels, each of which is two modes of the multiplier form).  Measured on B200
// (tools/time_tv_grad_reg.py, tools/time_c5_reg.py), LU vs Cholesky: 25.4 vs 34.6 ms (1 image 128²), 29.6 vs 38.2
// (10), 31.6 vs 37.0 (148), 25.5 vs 25.5 / 29.7 vs 35.1 (2×2 patch parameter, 1 / 10 images), 144 vs 337 (32 images
// of 256², 4-CTA clusters), 253 vs 590 (BASELINE config 5's share of one GPU: 128 images of 256², 5000 inner
// iterations).  Hence the LU whenever it takes the shape; BPLTV_GRAD_REG_LU=0/1 overrides.
// Solver of the adjoint systems (bpltv_eval_opts.solver): 0 / 2 — nested-dissection multifrontal Cholesky
// (gradient_nd.cuh: O(n³) operations, the whole GPU per image); 1 — the banded factorisations of round 1 (multiplier-
// space Cholesky for `gradient`, node-space LU for `gradient_reg`), kept as an independent second implementation.
// BPLTV_GRAD_SOLVER overrides option 0.
// A shape that neither the shared-memory front kernels nor the band solvers take goes back to the nested-dissection
// solver with its large-front variants (fronts beyond shared memory).
template <typename Real>
static int run_tv_gradient(Dev &d, const GradProblem<Real> &gp, cudaStream_t st, double *d_grad_out)
{
    int solver = gp.solver;
    if (solver == 0) solver = env_int("BPLTV_GRAD_SOLVER", 0);
    d.last_grad = Dev::GRAD_NONE;
    auto nd = [&](bool large) {
        if (!d.nd) d.nd = nd_work_create();
        NdProblem np;
        np.u = gp.u; np.ubar = gp.ubar; np.prec = (int)sizeof(Real) * 8; np.M = gp.M; np.N = gp.N; np.O = gp.O;
        np.alpha_s = gp.alpha_s; np.alpha_map = gp.alpha_map; np.lm = gp.lm; np.ln = gp.ln; np.regularised = gp.regularised;
        np.gamma = gp.gamma; np.act_tol = gp.act_tol; np.eps_act = gp.eps_act; np.tol = gp.tol; np.maxit = gp.maxit;
        np.large_fronts = large;
        const int rc = nd_run_gradient(d.nd, np, d.sm_count, d.smem_optin, st, d_grad_out, &d.launches);
        if (rc == 0) d.last_grad = Dev::GRAD_TV_ND;
        else if (rc != -1) d.grad.err = nd_work_error(d.nd);
        return rc;
    };
    if (solver != 1) {
        const int rc = nd(false);
        if (rc != -1) return rc;
        // -1: fronts beyond shared memory for this image size — the band solver takes over
    }
    int rc = -1;
    const char *lu_env = bpltv::env_get("BPLTV_GRAD_REG_LU");
    const bool lu = lu_env && *lu_env ? atoi(lu_env) != 0 : true;
    if (gp.regularised && lu && gp.M == gp.N && gp.M >= 4) {
        LuProblem<Real> lp;
        lp.u = gp.u; lp.ubar = gp.ubar; lp.M = gp.M; lp.N = gp.N; lp.O = gp.O;
        lp.alpha[0] = gp.alpha_s; lp.alpha[1] = lp.alpha[2] = 0.0;
        lp.alpha_maps = gp.alpha_map; lp.lm = gp.lm; lp.ln = gp.ln; lp.gamma = gp.gamma; lp.nops = 1;
        rc = run_gradient_lu<Real>(d.grad, lp, d.sm_count, d.smem_optin, st, d_grad_out, &d.launches);
        if (rc == 0) d.last_grad = Dev::GRAD_TV_BAND;
        // -1: the LU does not take this shape (panels beyond shared memory): Cholesky
    }
    if (rc == -1) {
        rc = run_gradient<Real>(d.grad, gp, d.sm_count, d.smem_optin, st, d_grad_out, &d.launches);
        if (rc == 0) d.last_grad = Dev::GRAD_TV_BAND;
    }
    if (rc == -1 && solver != 1 && gp.M == gp.N) return nd(true);
    return rc;
}

// The sum-of-regularisers gradient (eval_opts.solver as above).  Scalar sumregs_gradient_reg (:112-167) is symmetric
// positive definite in node space with coupling radius 2, and sumregs_gradient (non-regularised, scalar :264-327 and
// patch :330-407) is the same in multiplier space (3-6 unknowns per pixel): both take the nested-dissection
// multifrontal Cholesky.  Solver 1, a shape the fronts do not take (-1) or one that does not fit in memory go to the
// node-space band LU / compliance-form band Cholesky of run_gradient3, which needs less memory per image.  A shape the
// band solvers refuse as well (above 430² for the band LU, 136² for the band Cholesky) goes back to the fronts with their
// large-front variants; a failure there is final, and an image whose workspace does not fit returns BPLTV_ERR_ALLOC with
// the size it needs.
// The patch sumregs_gradient_reg (:195-262, row-scaled, not symmetric) takes the band LU first, as it always has; a shape
// the band LU refuses goes to the LU form of the fronts (shared-memory fronts, then the large-front variants).  Solver 1
// keeps it on the band LU; BPLTV_SUMREGS_PATCH_REG_ND=1 sends it to the fronts' LU at every size they take.
template <typename Real>
static int run_sumregs_gradient(Dev &d, const Grad3Problem<Real> &gp, int solver, int maxit, cudaStream_t st,
                                double *d_grad_out)
{
    if (solver == 0) solver = env_int("BPLTV_GRAD_SOLVER", 0);
    d.last_grad = Dev::GRAD_NONE;
    const bool patch_reg = gp.regularised && gp.alpha_maps;
    const bool fronts = solver != 1 && gp.M == gp.N && !patch_reg;
    auto nd = [&](bool large) {
        if (!d.nd3) d.nd3 = nd_work_create();
        int rc;
        if (gp.regularised) {
            Nd3Problem np;
            np.u = gp.u; np.ubar = gp.ubar; np.prec = (int)sizeof(Real) * 8; np.M = gp.M; np.N = gp.N; np.O = gp.O;
            for (int k = 0; k < 3; ++k) np.alpha[k] = gp.alpha[k];
            np.gamma = gp.gamma; np.tol = 0.0; np.maxit = maxit; np.large_fronts = large;
            np.alpha_maps = gp.alpha_maps; np.lm = gp.lm; np.ln = gp.ln;
            rc = nd_run_gradient3_reg(d.nd3, np, d.sm_count, d.smem_optin, st, d_grad_out, &d.launches);
        } else {
            Nd3mProblem np;
            np.u = gp.u; np.ubar = gp.ubar; np.alpha_maps = gp.alpha_maps; np.prec = (int)sizeof(Real) * 8;
            np.M = gp.M; np.N = gp.N; np.O = gp.O; np.lm = gp.lm; np.ln = gp.ln;
            for (int k = 0; k < 3; ++k) np.alpha[k] = gp.alpha[k];
            np.act_tol = gp.act_tol; np.eps_act = gp.eps_act; np.tol = 0.0; np.maxit = maxit; np.large_fronts = large;
            rc = nd_run_gradient3(d.nd3, np, d.sm_count, d.smem_optin, st, d_grad_out, &d.launches);
        }
        if (rc == 0) d.last_grad = Dev::GRAD_SR_ND;
        return rc;
    };
    auto band = [&]() {
        const int rc = run_gradient3<Real>(d.grad3, gp, d.sm_count, d.smem_optin, st, d_grad_out, &d.launches);
        if (rc == 0) d.last_grad = Dev::GRAD_SR_BAND;
        return rc;
    };
    if (patch_reg && solver != 1 && gp.M == gp.N) {
        const bool nd_first = env_int("BPLTV_SUMREGS_PATCH_REG_ND", 0) != 0;
        int rc = nd_first ? -1 : band();
        if (rc == -1) {
            rc = nd(false);
            if (rc == -1) rc = nd(true);
            if (rc != 0 && rc != -1) d.grad3.err = nd_work_error(d.nd3);
        }
        if (rc == -1 && nd_first) rc = band();      // images the fronts do not take (below 8²)
        return rc;
    }
    int nd_rc = -1;
    if (fronts) {
        nd_rc = nd(false);
        if (nd_rc == 0) return 0;
        if (nd_rc != -1 && nd_rc != BPLTV_ERR_ALLOC) { d.grad3.err = nd_work_error(d.nd3); return nd_rc; }
    }
    int rc = band();
    if (rc == -1 && fronts) {
        if (nd_rc == -1) rc = nd(true);
        else rc = nd_rc;        // the fronts took the shape but their workspace did not fit: say so, with its size
        if (rc != 0 && rc != -1) d.grad3.err = nd_work_error(d.nd3);
    }
    return rc;
}

// worst backward error of the adjoint solves of the last gradient on this device (device pointer) or nullptr
static const double *relres_of_last_gradient(const Dev &d)
{
    switch (d.last_grad) {
    case Dev::GRAD_TV_ND: return nd_work_relres_max(d.nd);
    case Dev::GRAD_TV_BAND: return static_cast<const double *>(d.grad.relres_max);
    case Dev::GRAD_SR_ND: return nd_work_relres_max(d.nd3);
    case Dev::GRAD_SR_BAND: return static_cast<const double *>(d.grad3.relres_max);
    default: return nullptr;
    }
}

// end of an evaluation's first pass: [cost, grad] (`count` doubles in d.scalars) summed over the ranks of the job and
// copied to `host`, with the worst backward error of the device's gradient
static int fetch_costgrad(bpltv_ctx *ctx, Dev &d, int count, double *host, double *relres)
{
    RC_TRY(allreduce_costgrad(ctx, d.scalars.as<double>(), count, d.stream));
    CU_TRY(cudaMemcpyAsync(host, d.scalars.p, count * sizeof(double), cudaMemcpyDeviceToHost, d.stream));
    if (relres_of_last_gradient(d))
        CU_TRY(cudaMemcpyAsync(relres, relres_of_last_gradient(d), sizeof(double), cudaMemcpyDeviceToHost, d.stream));
    return 0;
}

// the TV gradient of u against the device's resident truth
template <typename Real>
static GradProblem<Real> tv_grad_problem(const Dev &d, const Real *u, double alpha_s, const Real *amap, int lm, int ln,
                                         bool regularised, const bpltv_eval_opts &eo)
{
    GradProblem<Real> gp;
    gp.u = u; gp.ubar = d.truth.as<Real>(); gp.M = d.M; gp.N = d.N; gp.O = d.O;
    gp.alpha_s = alpha_s; gp.alpha_map = amap; gp.lm = lm; gp.ln = ln; gp.regularised = regularised;
    gp.gamma = eo.gamma; gp.act_tol = eo.act_tol;
    gp.eps_act = eo.eps_act > 0 ? eo.eps_act : (lm * ln == 1 ? 2.220446049250313e-16 : 1.4901161193847656e-08);
    gp.tol = eo.solver_tol; gp.maxit = eo.solver_maxit; gp.solver = eo.solver;
    return gp;
}

// ---------------------------------------------------------------------------
// evaluations of the learning functions on the resident dataset
// ---------------------------------------------------------------------------
// Enqueue one evaluation on one device: u = denoise; scalars[0] = cost;
// scalars[1..] = gradient.  Everything asynchronous on `st`.
template <typename Real>
static int eval_on_device(bpltv_ctx *ctx, Dev &d, const double *lam, int lm, int ln, double Delta,
                          const bpltv_eval_opts &eo, cudaStream_t st, const Real **u_res, double *d_costgrad)
{
    const int M = d.M, N = d.N, O = d.O;
    const size_t n = (size_t)M * N * O;
    const int ng = lm * ln;
    RC_TRY(mark(d, MARK_BEGIN, st));
    double alpha_s; const Real *amap;
    RC_TRY(prepare_lambda<Real>(d, lam, lm, ln, M, N, st, &alpha_s, &amap));
    const Real *u = nullptr; int used = 0, depth = 1;
    RC_TRY(run_pdps<Real>(d, d.noisy.as<Real>(), M, N, O, alpha_s, amap, eo.pdps, st, &u, &used, &depth));
    ctx->stats.pdps_kernel_used = used;
    ctx->stats.tblock_depth = depth;
    RC_TRY(mark(d, MARK_SOLVE, st));
    CU_TRY(cudaMemsetAsync(d_costgrad, 0, (1 + ng) * sizeof(double), st));
    if (O > 0) RC_TRY(run_cost<Real>(d, u, d.truth.as<Real>(), n, d_costgrad, st));
    RC_TRY(mark(d, MARK_COST, st));
    if (O > 0 && eo.force_branch != 3) {
        const bool reg = eo.force_branch == 2 || (eo.force_branch == 0 && !(Delta > eo.delta_t));
        const int rc = run_tv_gradient<Real>(d, tv_grad_problem<Real>(d, u, alpha_s, amap, lm, ln, reg, eo), st, d_costgrad + 1);
        if (rc != 0) return fail(rc, "gradient: %s", d.grad.err.c_str());
    }
    RC_TRY(mark(d, MARK_GRADIENT, st));
    *u_res = u;
    return 0;
}

template <typename Real>
static int learn_eval_impl(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                           const bpltv_eval_opts &eo, double *u_out, double *cost_out, double *grad_out)
{
    const int ndev = (int)ctx->devs.size();
    const int ng = lm * ln;
    const size_t plane = (size_t)ctx->M * ctx->N;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    std::vector<std::vector<double>> host(ndev, std::vector<double>(1 + ng, 0.0));
    std::vector<double> relres(ndev, 0.0);
    std::vector<const Real *> us(ndev, nullptr);
    double cost = 0.0;
    std::vector<double> grad(ng, 0.0);
    auto enqueue = [&](Dev &d, int di) {
        RC_TRY(d.scalars.ensure((1 + ng) * sizeof(double)));
        RC_TRY(eval_on_device<Real>(ctx, d, lam, lm, ln, Delta, eo, d.stream, &us[di], d.scalars.as<double>()));
        return fetch_costgrad(ctx, d, 1 + ng, host[di].data(), &relres[di]);
    };
    auto fold = [&](Dev &d, int di) {
        cost += host[di][0];
        for (int k = 0; k < ng; ++k) grad[k] += host[di][1 + k];
        fold_device_stats(ctx->stats, d);
        ctx->stats.solver_iterations += d.grad.last_iterations;
        ctx->stats.solver_max_relres = std::max(ctx->stats.solver_max_relres, relres[di]);
    };
    RC_TRY(run_sharded(ctx, false, enqueue, [&](Dev &d, int di) { return download_resident_u<Real>(d, us[di], u_out); }, fold));
    ctx->stats.pdps_iterations = eo.pdps.maxiter;
    ctx->stats.pixel_iterations = (long long)plane * ctx->O * eo.pdps.maxiter;
    ctx->stats.n_devices = ndev;
    if (!std::isfinite(cost)) return fail(BPLTV_ERR_NUMERIC, "non-finite cost");
    for (int k = 0; k < ng; ++k)
        if (!std::isfinite(grad[k]))
            return fail(BPLTV_ERR_NUMERIC, "non-finite gradient entry %d (adjoint solve: worst backward error %.3g, tolerance %.3g)", k,
                        ctx->stats.solver_max_relres, eo.solver_tol);
    *cost_out = cost;
    for (int k = 0; k < ng; ++k) grad_out[k] = grad[k];
    return 0;
}

// one sum-of-regularisers evaluation on one device: u, scalars[0] = cost, scalars[1..3·ng] = gradient
template <typename Real>
static int sumregs_eval_on_device(bpltv_ctx *ctx, Dev &d, const double *lam, int lm, int ln, double Delta,
                                  const bpltv_eval_opts &eo, const Real *u_given, cudaStream_t st, const Real **u_res,
                                  double *d_costgrad)
{
    const int M = d.M, N = d.N, O = d.O;
    const size_t n = (size_t)M * N * O;
    const int ng = lm * ln;
    RC_TRY(mark(d, MARK_BEGIN, st));
    Real alpha[3]; const Real *amap;
    RC_TRY(prepare_lambda3<Real>(d, lam, lm, ln, M, N, st, alpha, &amap));
    const Real *u = u_given;
    if (!u) RC_TRY(run_sumregs_pdps<Real>(d, d.noisy.as<Real>(), M, N, O, alpha, amap, eo.pdps, st, &u));
    RC_TRY(mark(d, MARK_SOLVE, st));
    CU_TRY(cudaMemsetAsync(d_costgrad, 0, (1 + 3 * ng) * sizeof(double), st));
    if (O > 0) RC_TRY(run_cost<Real>(d, u, d.truth.as<Real>(), n, d_costgrad, st));
    RC_TRY(mark(d, MARK_COST, st));
    if (O > 0 && eo.force_branch != 3) {
        Grad3Problem<Real> gp;
        gp.u = u; gp.ubar = d.truth.as<Real>(); gp.M = M; gp.N = N; gp.O = O;
        for (int k = 0; k < 3; ++k) gp.alpha[k] = ng == 1 ? lam[k] : 0.0;
        gp.alpha_maps = amap; gp.lm = lm; gp.ln = ln;
        gp.regularised = eo.force_branch == 2 || (eo.force_branch == 0 && !(Delta > eo.delta_t));
        gp.gamma = (gp.regularised && amap && eo.gamma_patch > 0) ? eo.gamma_patch : eo.gamma;   // :200 vs :117
        gp.act_tol = eo.act_tol;
        gp.eps_act = eo.eps_act > 0 ? eo.eps_act : 2.220446049250313e-16;   // eps() in both variants (:318-320, :387-389)
        const int rc = run_sumregs_gradient<Real>(d, gp, eo.solver, eo.solver_maxit, st, d_costgrad + 1);
        if (rc != 0) return fail(rc == -1 ? BPLTV_ERR_ARG : rc, "sumregs gradient: %s", d.grad3.err.c_str());
    }
    RC_TRY(mark(d, MARK_GRADIENT, st));
    *u_res = u;
    return 0;
}

// u_host != NULL: gradient of the caller's u (no solve; its upload lies outside the timed phases); else the full
// learning function
template <typename Real>
static int sumregs_learn_eval_impl(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                                   const bpltv_eval_opts &eo, const double *u_host, double *u_out, double *cost_out,
                                   double *grad_out)
{
    const int ndev = (int)ctx->devs.size();
    const int ng = 3 * lm * ln;
    const size_t plane = (size_t)ctx->M * ctx->N;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    std::vector<std::vector<double>> host(ndev, std::vector<double>(1 + ng, 0.0));
    std::vector<const Real *> us(ndev, nullptr);
    std::vector<double> relres(ndev, 0.0);
    double cost = 0.0;
    std::vector<double> grad(ng, 0.0);
    auto enqueue = [&](Dev &d, int di) {
        RC_TRY(d.scalars.ensure((1 + ng) * sizeof(double)));
        const Real *ug = nullptr;
        if (u_host) {
            RC_TRY(upload_stack<Real>(d, u_host + plane * d.o_begin, plane * d.O, d.ubuf, d.stream));
            ug = d.ubuf.as<Real>();
        }
        RC_TRY(sumregs_eval_on_device<Real>(ctx, d, lam, lm, ln, Delta, eo, ug, d.stream, &us[di], d.scalars.as<double>()));
        return fetch_costgrad(ctx, d, 1 + ng, host[di].data(), &relres[di]);
    };
    auto fold = [&](Dev &d, int di) {
        cost += host[di][0];
        ctx->stats.solver_max_relres = std::max(ctx->stats.solver_max_relres, relres[di]);
        for (int k = 0; k < ng; ++k) grad[k] += host[di][1 + k];
        fold_device_stats(ctx->stats, d);
    };
    RC_TRY(run_sharded(ctx, false, enqueue, [&](Dev &d, int di) { return download_resident_u<Real>(d, us[di], u_out); }, fold));
    ctx->stats.pdps_iterations = u_host ? 0 : eo.pdps.maxiter;
    ctx->stats.pixel_iterations = u_host ? 0 : (long long)plane * ctx->O * eo.pdps.maxiter;
    ctx->stats.n_devices = ndev;
    ctx->stats.tblock_depth = 1;
    if (!std::isfinite(cost)) return fail(BPLTV_ERR_NUMERIC, "non-finite cost");
    for (int k = 0; k < ng; ++k)
        if (!std::isfinite(grad[k])) return fail(BPLTV_ERR_NUMERIC, "non-finite gradient entry %d", k);
    if (cost_out) *cost_out = cost;
    for (int k = 0; k < ng; ++k) grad_out[k] = grad[k];
    return 0;
}

// λ-sweep: L parameter sets × the resident images as ONE batch of independent solves
// (virtual image v = l·O_dev + o on each device), then 0.5‖u-ū‖² per set.
template <typename Real>
static int sweep_impl(bpltv_ctx *ctx, const double *lams, int L, int lm, int ln, const bpltv_pdps_opts &o,
                      double *cost_out, double *sqerr_out, double *u_out)
{
    const int ndev = (int)ctx->devs.size();
    const int M = ctx->M, N = ctx->N, O = ctx->O, ng = lm * ln;
    const size_t plane = (size_t)M * N;
    const bool scalar = ng == 1;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    std::vector<std::vector<double>> host(ndev);
    std::vector<const Real *> us(ndev, nullptr);
    std::vector<double> cost(L, 0.0);
    auto enqueue = [&](Dev &d, int di) {
        const int V = L * d.O;
        host[di].assign((size_t)V, 0.0);
        cudaStream_t st = d.stream;
        RC_TRY(mark(d, MARK_BEGIN, st));
        RC_TRY(d.lam_dev.ensure((size_t)L * ng * sizeof(double)));
        CU_TRY(cudaMemcpyAsync(d.lam_dev.p, lams, (size_t)L * ng * sizeof(double), cudaMemcpyHostToDevice, st));
        BatchMap<Real> bm;
        bm.f_mod = d.O; bm.lam_div = d.O;
        const Real *amap = nullptr;
        if (scalar) {
            RC_TRY(d.amap.ensure((size_t)L * sizeof(Real)));
            convert_kernel<Real, double><<<(L + 255) / 256, 256, 0, st>>>(d.lam_dev.as<double>(), d.amap.as<Real>(), (size_t)L);
            bm.alpha_vec = d.amap.as<Real>();
        } else {
            RC_TRY(d.amap.ensure((size_t)L * plane * sizeof(Real)));
            const size_t tot = (size_t)L * plane;
            patch_upsample_sets_kernel<Real><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d.lam_dev.as<double>(), L, lm, ln,
                                                                                        d.amap.as<Real>(), M, N);
            bm.map_stride = (long long)plane;
            amap = d.amap.as<Real>();
        }
        d.launches += 1;
        RC_TRY(mark(d, MARK_UPLOAD, st));
        int used = 0, depth = 1;
        RC_TRY(run_pdps<Real>(d, d.noisy.as<Real>(), M, N, V, 0.0, amap, o, st, &us[di], &used, &depth, &bm));
        ctx->stats.pdps_kernel_used = used;
        ctx->stats.tblock_depth = depth;
        RC_TRY(mark(d, MARK_SOLVE, st));
        RC_TRY(d.partials.ensure(std::max<size_t>((size_t)V, 1024) * sizeof(double)));
        sqerr_image_kernel<Real><<<V, 256, 0, st>>>(us[di], d.truth.as<Real>(), (int)plane, d.O, d.partials.as<double>());
        d.launches += 1;
        CU_TRY(cudaMemcpyAsync(host[di].data(), d.partials.p, (size_t)V * sizeof(double), cudaMemcpyDeviceToHost, st));
        return mark(d, MARK_COST, st);
    };
    auto download = [&](Dev &d, int di) {
        if (u_out)
            for (int l = 0; l < L; ++l)
                RC_TRY(download_stack<Real>(d, us[di] + (size_t)l * d.O * plane, plane * d.O,
                                            u_out + ((size_t)l * O + d.o_begin) * plane, d.stream));
        return mark(d, MARK_DOWNLOAD, d.stream);
    };
    auto fold = [&](Dev &d, int di) {      // image order within the device: deterministic sums
        for (int l = 0; l < L; ++l)
            for (int oo = 0; oo < d.O; ++oo) {
                const double v = host[di][(size_t)l * d.O + oo];
                cost[l] += v;
                if (sqerr_out) sqerr_out[(size_t)l * O + d.o_begin + oo] = v;
            }
        fold_device_stats(ctx->stats, d);
    };
    RC_TRY(run_sharded(ctx, true, enqueue, download, fold));
    for (int l = 0; l < L; ++l) {
        cost_out[l] = 0.5 * cost[l];
        if (!std::isfinite(cost_out[l])) return fail(BPLTV_ERR_NUMERIC, "non-finite cost for parameter set %d", l);
    }
    ctx->stats.pdps_iterations = o.maxiter;
    ctx->stats.pixel_iterations = (long long)plane * O * L * o.maxiter;
    ctx->stats.n_devices = ndev;
    return 0;
}

template <typename Real>
static int gradient_impl(bpltv_ctx *ctx, const double *u_host, const double *lam, int lm, int ln, int regularised,
                         const bpltv_eval_opts &eo, double *grad_out)
{
    const int ndev = (int)ctx->devs.size();
    const int ng = lm * ln;
    const size_t plane = (size_t)ctx->M * ctx->N;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    std::vector<std::vector<double>> host(ndev, std::vector<double>(ng, 0.0));
    std::vector<double> relres(ndev, 0.0);
    std::vector<double> grad(ng, 0.0);
    auto enqueue = [&](Dev &d, int di) {
        cudaStream_t st = d.stream;
        RC_TRY(d.scalars.ensure((1 + ng) * sizeof(double)));
        RC_TRY(upload_stack<Real>(d, u_host + plane * d.o_begin, plane * d.O, d.ubuf, st));
        double alpha_s; const Real *amap;
        RC_TRY(prepare_lambda<Real>(d, lam, lm, ln, d.M, d.N, st, &alpha_s, &amap));
        RC_TRY(mark(d, MARK_BEGIN, st));
        const GradProblem<Real> gp = tv_grad_problem<Real>(d, d.ubuf.as<Real>(), alpha_s, amap, lm, ln, regularised != 0, eo);
        CU_TRY(cudaMemsetAsync(d.scalars.p, 0, (1 + ng) * sizeof(double), st));
        const int rc = run_tv_gradient<Real>(d, gp, st, d.scalars.as<double>() + 1);
        if (rc != 0) return fail(rc, "gradient: %s", d.grad.err.c_str());
        RC_TRY(mark(d, MARK_GRADIENT, st));
        CU_TRY(cudaMemcpyAsync(host[di].data(), d.scalars.as<double>() + 1, ng * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (relres_of_last_gradient(d))
            CU_TRY(cudaMemcpyAsync(&relres[di], relres_of_last_gradient(d), sizeof(double), cudaMemcpyDeviceToHost, st));
        return 0;
    };
    auto fold = [&](Dev &d, int di) {
        for (int k = 0; k < ng; ++k) grad[k] += host[di][k];
        fold_device_stats(ctx->stats, d);
        ctx->stats.solver_iterations += d.grad.last_iterations;
        ctx->stats.solver_max_relres = std::max(ctx->stats.solver_max_relres, relres[di]);
    };
    RC_TRY(run_sharded(ctx, true, enqueue, no_download, fold));
    ctx->stats.n_devices = ndev;
    for (int k = 0; k < ng; ++k) {
        if (!std::isfinite(grad[k]))
            return fail(BPLTV_ERR_NUMERIC, "non-finite gradient entry %d (adjoint solve: worst backward error %.3g, tolerance %.3g)", k,
                        ctx->stats.solver_max_relres, eo.solver_tol);
        grad_out[k] = grad[k];
    }
    return 0;
}

template <typename Real>
static int denoise_device_impl(bpltv_ctx *ctx, const void *d_noisy, int M, int N, int O, const double *lam, int lm,
                               int ln, const bpltv_pdps_opts &o, void *d_u_out, cudaStream_t st)
{
    Dev &d = ctx->devs[0];
    CU_TRY(cudaSetDevice(d.id));
    d.launches = 0;
    double alpha_s; const Real *amap;
    RC_TRY(prepare_lambda<Real>(d, lam, lm, ln, M, N, st, &alpha_s, &amap));
    const Real *u = nullptr; int used = 0, depth = 1;
    RC_TRY(run_pdps<Real>(d, static_cast<const Real *>(d_noisy), M, N, O, alpha_s, amap, o, st, &u, &used, &depth));
    if (O > 0)
        CU_TRY(cudaMemcpyAsync(d_u_out, u, (size_t)M * N * O * sizeof(Real), cudaMemcpyDeviceToDevice, st));
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    ctx->stats.pdps_kernel_used = used;
    ctx->stats.tblock_depth = depth;
    ctx->stats.kernel_launches = d.launches;
    ctx->stats.pdps_iterations = o.maxiter;
    ctx->stats.pixel_iterations = (long long)M * N * O * o.maxiter;
    ctx->stats.n_devices = 1;
    return 0;
}

template <typename Real>
static int learn_eval_device_impl(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                                  const bpltv_eval_opts &eo, void *d_u_out, double *d_costgrad, cudaStream_t st)
{
    Dev &d = ctx->devs[0];
    CU_TRY(cudaSetDevice(d.id));
    d.launches = 0;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    const Real *u = nullptr;
    RC_TRY(eval_on_device<Real>(ctx, d, lam, lm, ln, Delta, eo, st, &u, d_costgrad));
    RC_TRY(allreduce_costgrad(ctx, d_costgrad, 1 + lm * ln, st));
    if (d_u_out && d.O > 0)
        CU_TRY(cudaMemcpyAsync(d_u_out, u, (size_t)d.M * d.N * d.O * sizeof(Real), cudaMemcpyDeviceToDevice, st));
    ctx->stats.kernel_launches = d.launches;
    ctx->stats.pdps_iterations = eo.pdps.maxiter;
    ctx->stats.pixel_iterations = (long long)d.M * d.N * d.O * eo.pdps.maxiter;
    ctx->stats.n_devices = 1;
    return 0;
}

// ---------------------------------------------------------------------------
// C entry points
// ---------------------------------------------------------------------------
extern "C" {

int bpltv_version(void) { return BPLTV_VERSION; }

void bpltv_reload_env(void) { bpltv::env_reload(); }

const char *bpltv_last_error(void) { return g_last_error.c_str(); }

void bpltv_default_pdps_opts(bpltv_pdps_opts *o)
{
    if (!o) return;
    std::memset(o, 0, sizeof *o);
    o->tau0 = 5.0;           // /root/reference/src/TVLearningFunctionVec.jl:36
    o->sigma0 = 0.99 / 5;    // :37
    o->rho = 0.0;            // :34
    o->opnorm = std::sqrt(8.0);
    o->accel = 1;            // :38
    o->maxiter = 5000;       // :40
    o->init_mode = 0;
    o->arith = BPLTV_ARITH_STRICT;
    o->kernel = BPLTV_KERNEL_AUTO;
    o->tblock = 0;
}

void bpltv_default_eval_opts(bpltv_eval_opts *o)
{
    if (!o) return;
    std::memset(o, 0, sizeof *o);
    bpltv_default_pdps_opts(&o->pdps);
    o->delta_t = 1e-6;   // :14
    o->gamma = 1e8;      // :142, :197
    o->act_tol = 1e-12;  // :109, :231
    o->eps_act = 0.0;    // → eps() scalar (:128) / sqrt(eps()) patch (:245)
    o->solver_tol = 1e-9;
    o->solver_maxit = 0;
    o->solver = 0;
    o->force_branch = 0;
}

int bpltv_create(const int *device_ids, int ndev, int precision, bpltv_ctx **out)
{
    if (!out) return fail(BPLTV_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (precision != 64 && precision != 32) return fail(BPLTV_ERR_ARG, "precision must be 64 or 32");
    if (ndev < 1) return fail(BPLTV_ERR_ARG, "ndev must be >= 1");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count < 1) {
        cudaGetLastError();
        return fail(BPLTV_ERR_NODEVICE, "no CUDA device (%s); libbpltv has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    bpltv::env_get("BPLTV_PDPS_KERNEL");      // takes the snapshot of the BPLTV_* switches if none exists yet
    bpltv_ctx *ctx = new bpltv_ctx();
    ctx->prec = precision;
    std::memset(&ctx->stats, 0, sizeof ctx->stats);
    ctx->devs.resize(ndev);
    for (int k = 0; k < ndev; ++k) {
        Dev &d = ctx->devs[k];
        d.id = device_ids ? device_ids[k] : k;
        if (d.id < 0 || d.id >= count) {
            delete ctx;
            return fail(BPLTV_ERR_ARG, "device id %d out of range (have %d devices)", d.id, count);
        }
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d.id) != cudaSuccess || prop.major != 10) {
            cudaGetLastError();
            int major = prop.major, minor = prop.minor;
            delete ctx;
            return fail(BPLTV_ERR_NODEVICE, "device %d is sm_%d%d; libbpltv is built for sm_100a only", d.id, major, minor);
        }
        d.sm_count = prop.multiProcessorCount;
        d.smem_optin = prop.sharedMemPerBlockOptin;
        if (cudaSetDevice(d.id) != cudaSuccess || cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError();
            delete ctx;
            return fail(BPLTV_ERR_CUDA, "cannot create stream on device %d", d.id);
        }
        for (auto &ev : d.ev) cudaEventCreate(&ev);
    }
    *out = ctx;
    return 0;
}

int bpltv_comm_unique_id(unsigned char *id_out)
{
    if (!id_out) return fail(BPLTV_ERR_ARG, "NULL argument");
    NcclApi &api = nccl_api();
    if (!api.load()) return fail(BPLTV_ERR_STATE, "NCCL library not available (%s); set BPLTV_NCCL_LIB", api.err.c_str());
    NcclId id;
    const int rc = api.GetUniqueId(&id);
    if (rc != 0) return fail(BPLTV_ERR_CUDA, "ncclGetUniqueId: %s", api.what(rc));
    std::memcpy(id_out, id.internal, BPLTV_COMM_ID_BYTES);
    return 0;
}

int bpltv_comm_destroy(bpltv_ctx *ctx)
{
    if (!ctx) return fail(BPLTV_ERR_ARG, "NULL argument");
    if (ctx->comm) {
        cudaSetDevice(ctx->devs[0].id);
        cudaStreamSynchronize(ctx->devs[0].stream);
        nccl_api().CommDestroy(ctx->comm);
        ctx->comm = nullptr;
    }
    ctx->comm_ranks = 1; ctx->comm_rank = 0;
    return 0;
}

int bpltv_comm_init(bpltv_ctx *ctx, int nranks, int rank, const unsigned char *id)
{
    if (!ctx || !id) return fail(BPLTV_ERR_ARG, "NULL argument");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(BPLTV_ERR_ARG, "bad rank %d of %d", rank, nranks);
    if (ctx->devs.size() != 1)
        return fail(BPLTV_ERR_ARG, "a communicator joins single-device contexts (one process per GPU); this context shards over %d devices itself",
                    (int)ctx->devs.size());
    NcclApi &api = nccl_api();
    if (!api.load()) return fail(BPLTV_ERR_STATE, "NCCL library not available (%s); set BPLTV_NCCL_LIB", api.err.c_str());
    bpltv_comm_destroy(ctx);
    CU_TRY(cudaSetDevice(ctx->devs[0].id));
    NcclId nid;
    std::memcpy(nid.internal, id, BPLTV_COMM_ID_BYTES);
    void *comm = nullptr;
    const int rc = api.CommInitRank(&comm, nranks, nid, rank);
    if (rc != 0) return fail(BPLTV_ERR_CUDA, "ncclCommInitRank(%d of %d): %s", rank, nranks, api.what(rc));
    ctx->comm = comm; ctx->comm_ranks = nranks; ctx->comm_rank = rank;
    return 0;
}

int bpltv_destroy(bpltv_ctx *ctx)
{
    if (!ctx) return 0;
    bpltv_comm_destroy(ctx);
    for (Dev &d : ctx->devs) {
        cudaSetDevice(d.id);
        if (d.stream) cudaStreamSynchronize(d.stream);
        DBuf *bufs[] = {&d.truth, &d.noisy, &d.x[0], &d.x[1], &d.y1[0], &d.y1[1], &d.y2[0], &d.y2[1], &d.fbuf,
                        &d.amap, &d.steps, &d.partials, &d.scalars, &d.stage, &d.lam_dev, &d.ubuf, &d.sry};
        for (DBuf *b : bufs) b->release();
        d.grad.release();
        d.grad3.release();
        nd_work_destroy(d.nd);
        nd_work_destroy(d.nd3);
        d.nd = nullptr;
        d.hstage.release();
        for (auto &ev : d.ev) if (ev) cudaEventDestroy(ev);
        for (auto &ev : d.pipe_ev) if (ev) cudaEventDestroy(ev);
        if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    delete ctx;
    return 0;
}

static int check_shape(int M, int N, int O)
{
    if (M < 1 || N < 1 || O < 0) return fail(BPLTV_ERR_ARG, "bad stack shape %dx%dx%d", M, N, O);
    if ((double)M * N * std::max(O, 1) > 4.0e9) return fail(BPLTV_ERR_ARG, "stack too large");
    return 0;
}

// denoise(noisy = NULL) takes the resident dataset: there must be one, of the call's shape
static int check_resident_shape(const bpltv_ctx *ctx, const double *noisy, int M, int N, int O)
{
    if (noisy) return 0;
    if (!ctx->have_dataset) return fail(BPLTV_ERR_STATE, "denoise(noisy=NULL) needs bpltv_set_dataset first");
    if (M != ctx->M || N != ctx->N || O != ctx->O)
        return fail(BPLTV_ERR_ARG, "shape %dx%dx%d does not match the resident dataset %dx%dx%d", M, N, O, ctx->M,
                    ctx->N, ctx->O);
    return 0;
}

// the sum-of-regularisers parameter: three lm×ln grids, one after the other
static int check_lambda3(const double *lam, int lm, int ln)
{
    if (!lam || lm < 1 || ln < 1) return fail(BPLTV_ERR_ARG, "lambda grid must be at least 1x1(x3)");
    for (int k = 0; k < 3; ++k) RC_TRY(check_lambda(lam + (size_t)k * lm * ln, lm, ln));
    return 0;
}

int bpltv_set_dataset(bpltv_ctx *ctx, const double *truth, const double *noisy, int M, int N, int O)
{
    if (!ctx || !truth || !noisy) return fail(BPLTV_ERR_ARG, "NULL argument");
    RC_TRY(check_shape(M, N, O));
    return ctx->prec == 64 ? set_dataset_impl<double>(ctx, truth, noisy, M, N, O)
                           : set_dataset_impl<float>(ctx, truth, noisy, M, N, O);
}

int bpltv_denoise(bpltv_ctx *ctx, const double *noisy, int M, int N, int O, const double *lam, int lm, int ln,
                  const bpltv_pdps_opts *opts, double *u_out)
{
    if (!ctx || !u_out) return fail(BPLTV_ERR_ARG, "NULL argument");
    RC_TRY(check_shape(M, N, O));
    RC_TRY(check_lambda(lam, lm, ln));
    bpltv_pdps_opts o;
    if (opts) o = *opts; else bpltv_default_pdps_opts(&o);
    RC_TRY(check_pdps_opts(o));
    RC_TRY(check_resident_shape(ctx, noisy, M, N, O));
    return ctx->prec == 64 ? denoise_impl<double>(ctx, noisy, M, N, O, lam, lm, ln, o, u_out)
                           : denoise_impl<float>(ctx, noisy, M, N, O, lam, lm, ln, o, u_out);
}

// Arguments of an evaluation on the resident dataset: the TV learning function (sets = 1) or the sum of regularisers
// (sets = 3 λ grids).  force_branch == 3 evaluates the loss alone (λ-sweeps, validation): no gradient is formed, so
// λ > 0 does not apply, nor, on the TV path, the reference's square-image precondition.
static int check_eval(bpltv_ctx *ctx, const double *lam, int lm, int ln, int sets, const bpltv_eval_opts *opts,
                      bpltv_eval_opts &eo)
{
    if (!ctx) return fail(BPLTV_ERR_ARG, "NULL context");
    if (!ctx->have_dataset) return fail(BPLTV_ERR_STATE, "no resident dataset: call bpltv_set_dataset first");
    RC_TRY(sets == 1 ? check_lambda(lam, lm, ln) : check_lambda3(lam, lm, ln));
    if (opts) eo = *opts;
    else if (sets == 1) bpltv_default_eval_opts(&eo);
    else bpltv_default_sumregs_eval_opts(&eo);
    RC_TRY(check_pdps_opts(eo.pdps));
    const bool grad_needed = eo.force_branch != 3;
    if ((grad_needed || sets == 3) && ctx->M != ctx->N)
        return fail(BPLTV_ERR_ARG, "the gradient assumes square images like the reference (%s); got %dx%d",
                    sets == 1 ? "TVLearningFunctionVec.jl:102" : "SumRegsLearningFunction.jl:116", ctx->M, ctx->N);
    if (lm > ctx->M || ln > ctx->N) return fail(BPLTV_ERR_ARG, "lambda grid larger than the image");
    if (grad_needed)
        for (int k = 0; k < sets * lm * ln; ++k)
            if (!(lam[k] > 0.0)) return fail(BPLTV_ERR_ARG, "lambda[%d] must be > 0 for the gradient", k);
    if (!(eo.gamma > 0) || !(eo.act_tol >= 0)) return fail(BPLTV_ERR_ARG, "bad gamma / act_tol");
    return 0;
}

int bpltv_learn_eval(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta, const bpltv_eval_opts *opts,
                     double *u_out, double *cost_out, double *grad_out)
{
    bpltv_eval_opts eo;
    RC_TRY(check_eval(ctx, lam, lm, ln, 1, opts, eo));
    if (!cost_out || !grad_out) return fail(BPLTV_ERR_ARG, "NULL output");
    return ctx->prec == 64 ? learn_eval_impl<double>(ctx, lam, lm, ln, Delta, eo, u_out, cost_out, grad_out)
                           : learn_eval_impl<float>(ctx, lam, lm, ln, Delta, eo, u_out, cost_out, grad_out);
}

int bpltv_gradient(bpltv_ctx *ctx, const double *u, const double *lam, int lm, int ln, int regularised,
                   const bpltv_eval_opts *opts, double *grad_out)
{
    bpltv_eval_opts eo;
    RC_TRY(check_eval(ctx, lam, lm, ln, 1, opts, eo));
    if (!u || !grad_out) return fail(BPLTV_ERR_ARG, "NULL argument");
    return ctx->prec == 64 ? gradient_impl<double>(ctx, u, lam, lm, ln, regularised, eo, grad_out)
                           : gradient_impl<float>(ctx, u, lam, lm, ln, regularised, eo, grad_out);
}

int bpltv_sweep(bpltv_ctx *ctx, const double *lams, int L, int lm, int ln, const bpltv_pdps_opts *opts,
                double *cost_out, double *sqerr_out, double *u_out)
{
    if (!ctx || !lams || !cost_out) return fail(BPLTV_ERR_ARG, "NULL argument");
    if (!ctx->have_dataset) return fail(BPLTV_ERR_STATE, "no resident dataset: call bpltv_set_dataset first");
    if (L < 1) return fail(BPLTV_ERR_ARG, "need at least one parameter set");
    for (int l = 0; l < L; ++l) RC_TRY(check_lambda(lams + (size_t)l * lm * ln, lm, ln));
    if (lm > ctx->M || ln > ctx->N) return fail(BPLTV_ERR_ARG, "lambda grid larger than the image");
    bpltv_pdps_opts o;
    if (opts) o = *opts; else bpltv_default_pdps_opts(&o);
    RC_TRY(check_pdps_opts(o));
    if ((double)ctx->M * ctx->N * std::max(ctx->O, 1) * L > 4.0e9) return fail(BPLTV_ERR_ARG, "sweep too large: split the parameter range");
    return ctx->prec == 64 ? sweep_impl<double>(ctx, lams, L, lm, ln, o, cost_out, sqerr_out, u_out)
                           : sweep_impl<float>(ctx, lams, L, lm, ln, o, cost_out, sqerr_out, u_out);
}

void bpltv_default_sumregs_eval_opts(bpltv_eval_opts *o)
{
    if (!o) return;
    bpltv_default_eval_opts(o);
    o->pdps.opnorm = std::sqrt(18.0);   // S12: R_K of (∇ᶠ; ∇ᵇ; ∇ᶜ)
    o->delta_t = 1e-3;                  // /root/reference/src/SumRegsLearningFunction.jl:8
    o->gamma = 1e3;                     // :117 (scalar sumregs_gradient_reg)
    o->gamma_patch = 1e8;               // :200 (patch sumregs_gradient_reg)
}

int bpltv_sumregs_denoise(bpltv_ctx *ctx, const double *noisy, int M, int N, int O, const double *lam, int lm, int ln,
                          const bpltv_pdps_opts *opts, double *u_out)
{
    if (!ctx || !u_out) return fail(BPLTV_ERR_ARG, "NULL argument");
    RC_TRY(check_shape(M, N, O));
    RC_TRY(check_lambda3(lam, lm, ln));
    bpltv_pdps_opts o;
    if (opts) o = *opts;
    else { bpltv_eval_opts e; bpltv_default_sumregs_eval_opts(&e); o = e.pdps; }
    RC_TRY(check_pdps_opts(o));
    RC_TRY(check_resident_shape(ctx, noisy, M, N, O));
    return ctx->prec == 64 ? sumregs_denoise_impl<double>(ctx, noisy, M, N, O, lam, lm, ln, o, u_out)
                           : sumregs_denoise_impl<float>(ctx, noisy, M, N, O, lam, lm, ln, o, u_out);
}

int bpltv_sumregs_learn_eval(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                             const bpltv_eval_opts *opts, double *u_out, double *cost_out, double *grad_out)
{
    bpltv_eval_opts eo;
    RC_TRY(check_eval(ctx, lam, lm, ln, 3, opts, eo));
    if (!cost_out || !grad_out) return fail(BPLTV_ERR_ARG, "NULL output");
    return ctx->prec == 64
               ? sumregs_learn_eval_impl<double>(ctx, lam, lm, ln, Delta, eo, nullptr, u_out, cost_out, grad_out)
               : sumregs_learn_eval_impl<float>(ctx, lam, lm, ln, Delta, eo, nullptr, u_out, cost_out, grad_out);
}

int bpltv_sumregs_gradient(bpltv_ctx *ctx, const double *u, const double *lam, int lm, int ln, int regularised,
                           const bpltv_eval_opts *opts, double *grad_out)
{
    bpltv_eval_opts eo;
    RC_TRY(check_eval(ctx, lam, lm, ln, 3, opts, eo));
    if (!u || !grad_out) return fail(BPLTV_ERR_ARG, "NULL argument");
    eo.force_branch = regularised ? 2 : 1;
    return ctx->prec == 64
               ? sumregs_learn_eval_impl<double>(ctx, lam, lm, ln, 0.0, eo, u, nullptr, nullptr, grad_out)
               : sumregs_learn_eval_impl<float>(ctx, lam, lm, ln, 0.0, eo, u, nullptr, nullptr, grad_out);
}

// ---- device-resident variants (single device) --------------------------------
static int single_dev(bpltv_ctx *ctx)
{
    if (!ctx) return fail(BPLTV_ERR_ARG, "NULL context");
    if (ctx->devs.size() != 1) return fail(BPLTV_ERR_ARG, "device-pointer entry points need a single-device context");
    return 0;
}

static int check_aligned16(const void *a, const void *b)
{
    if (((uintptr_t)a | (uintptr_t)b) & 15)
        return fail(BPLTV_ERR_ARG, "device pointers must be 16-byte aligned (vector and TMA accesses)");
    return 0;
}

int bpltv_denoise_device(bpltv_ctx *ctx, const void *d_noisy, int M, int N, int O, const double *lam, int lm, int ln,
                         const bpltv_pdps_opts *opts, void *d_u_out, void *stream)
{
    RC_TRY(single_dev(ctx));
    if (!d_noisy || !d_u_out) return fail(BPLTV_ERR_ARG, "NULL device pointer");
    RC_TRY(check_aligned16(d_noisy, d_u_out));
    RC_TRY(check_shape(M, N, O));
    RC_TRY(check_lambda(lam, lm, ln));
    bpltv_pdps_opts o;
    if (opts) o = *opts; else bpltv_default_pdps_opts(&o);
    RC_TRY(check_pdps_opts(o));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->devs[0].stream;
    return ctx->prec == 64 ? denoise_device_impl<double>(ctx, d_noisy, M, N, O, lam, lm, ln, o, d_u_out, st)
                           : denoise_device_impl<float>(ctx, d_noisy, M, N, O, lam, lm, ln, o, d_u_out, st);
}

int bpltv_set_dataset_device(bpltv_ctx *ctx, const void *d_truth, const void *d_noisy, int M, int N, int O,
                             void *stream)
{
    RC_TRY(single_dev(ctx));
    if (!d_truth || !d_noisy) return fail(BPLTV_ERR_ARG, "NULL device pointer");
    RC_TRY(check_aligned16(d_truth, d_noisy));
    RC_TRY(check_shape(M, N, O));
    Dev &d = ctx->devs[0];
    CU_TRY(cudaSetDevice(d.id));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d.stream;
    const size_t bytes = (size_t)M * N * O * (ctx->prec == 64 ? 8 : 4);
    RC_TRY(d.truth.ensure(std::max<size_t>(bytes, 8)));
    RC_TRY(d.noisy.ensure(std::max<size_t>(bytes, 8)));
    if (bytes) {
        CU_TRY(cudaMemcpyAsync(d.truth.p, d_truth, bytes, cudaMemcpyDeviceToDevice, st));
        CU_TRY(cudaMemcpyAsync(d.noisy.p, d_noisy, bytes, cudaMemcpyDeviceToDevice, st));
    }
    d.M = M; d.N = N; d.O = O; d.o_begin = 0;
    ctx->M = M; ctx->N = N; ctx->O = O; ctx->have_dataset = true;
    return 0;
}


int bpltv_learn_eval_device(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                            const bpltv_eval_opts *opts, void *d_u_out, double *d_costgrad, void *stream)
{
    RC_TRY(single_dev(ctx));
    bpltv_eval_opts eo;
    RC_TRY(check_eval(ctx, lam, lm, ln, 1, opts, eo));
    if (!d_costgrad) return fail(BPLTV_ERR_ARG, "NULL d_costgrad");
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : ctx->devs[0].stream;
    return ctx->prec == 64 ? learn_eval_device_impl<double>(ctx, lam, lm, ln, Delta, eo, d_u_out, d_costgrad, st)
                           : learn_eval_device_impl<float>(ctx, lam, lm, ln, Delta, eo, d_u_out, d_costgrad, st);
}

int bpltv_get_stats(bpltv_ctx *ctx, bpltv_stats *out)
{
    if (!ctx || !out) return fail(BPLTV_ERR_ARG, "NULL argument");
    *out = ctx->stats;
    return 0;
}

int bpltv_selftest(bpltv_ctx *ctx, int what, int mode, unsigned long long count, unsigned long long seed,
                   unsigned long long *result)
{
    if (!ctx || !result) return fail(BPLTV_ERR_ARG, "NULL argument");
    if (what != 0 || mode < 0 || mode > 3) return fail(BPLTV_ERR_ARG, "selftest: unknown test %d / mode %d", what, mode);
    Dev &d = ctx->devs[0];
    CU_TRY(cudaSetDevice(d.id));
    unsigned long long *dres = nullptr;
    CU_TRY(cudaMalloc(&dres, 4 * sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(dres, 0, 4 * sizeof(unsigned long long), d.stream);
    if (e == cudaSuccess) {
        const unsigned grid = (unsigned)(d.sm_count * 8);
        if (ctx->prec == 64) selftest_ball_scale_kernel<double><<<grid, 256, 0, d.stream>>>(mode, count, seed, dres);
        else selftest_ball_scale_kernel<float><<<grid, 256, 0, d.stream>>>(mode, count, seed, dres);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(result, dres, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(d.stream);
    cudaFree(dres);
    if (e != cudaSuccess) return fail(BPLTV_ERR_CUDA, "selftest: %s", cudaGetErrorString(e));
    return 0;
}

}  // extern "C"
