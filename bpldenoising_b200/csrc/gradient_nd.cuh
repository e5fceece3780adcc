// gradient_nd.cuh — host driver of the nested-dissection adjoint solver (nd_symbolic.h, nd_solver.cuh, nd_tv.cuh).
//
// gradient (/root/reference/src/TVLearningFunctionVec.jl:98-135, :219-254) runs in multiplier space (MULT: 1-2
// unknowns per pixel, sizes known only after the classification → one small device→host read per wave of images);
// gradient_reg (:137-161, :192-215) in node space (NODE: one unknown per node, every size static).
// Images are processed in waves of `slots`; inside a wave every kernel has a grid (work items, images), so one image
// spreads over the SMs level by level and many images fill the GPU together.
#pragma once
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>

#include "env_switches.h"
#include "gradient_nd.h"
#include "nd_sumregs.cuh"
#include "nd_tv.cuh"

namespace bpltv {

// grad[g] = Σ_o out_img[o][g] in image order (the reference's serial `for i = 1:O`, TVLearningFunctionVec.jl:76-81),
// and the worst backward error over the images
__global__ void nd_reduce_kernel(const double *out_img, const double *relres_img, int O, int ng, double *grad, double *relres_max)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < ng) {
        double s = 0.0;
        for (int o = 0; o < O; ++o) s += out_img[(size_t)o * ng + g];
        grad[g] = s;
    }
    if (g == 0) {
        double m = 0.0;
        for (int o = 0; o < O; ++o) m = fmax(m, relres_img[o]);
        relres_max[0] = m;
    }
}

struct NdPlan {      // symbolic structure of one image size, on the device
    NdSymbolic sym;
    int n = 0;
    void *d_fronts = nullptr, *d_pixlist = nullptr, *d_nbr = nullptr, *d_cmap = nullptr, *d_step_start = nullptr;
    void *d_posg1 = nullptr, *d_foff1 = nullptr;       // static tables of the one-unknown-per-pixel case
    long long tot1[4] = {0, 0, 0, 0};
    size_t posg_len = 0;
    void release()
    {
        void **all[] = {&d_fronts, &d_pixlist, &d_nbr, &d_cmap, &d_step_start, &d_posg1, &d_foff1};
        for (void **p : all) { if (*p) cudaFree(*p); *p = nullptr; }
        n = 0;
    }
};

struct NdBuf {
    void *p = nullptr; size_t bytes = 0;
    // grows by at least half of what it had: the pools of the multiplier form follow the data (unknowns per pixel change
    // with λ from one evaluation of a learn run to the next), and a cudaFree + cudaMalloc per evaluation synchronises
    cudaError_t ensure(size_t need)
    {
        if (need <= bytes) return cudaSuccess;
        const size_t want = std::max(need, bytes + bytes / 2);
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) { bytes = want; return e; }
        cudaGetLastError();
        e = cudaMalloc(&p, need);
        if (e == cudaSuccess) bytes = need; else cudaGetLastError();
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

struct NdWork {
    std::string err;
    NdPlan plan;
    NdBuf pix, off, off3, lvl, vec, posg, foff, totals, ast, L, U0, U1, UV0, UV1, scr, info, out_img, relres, relres_max;
    std::vector<long long> h_totals;
    size_t budget_cached = 0;
    // what the last call saw (statistics)
    double last_relres = 0.0;
    long long last_guarded = 0;
    size_t last_bytes_per_image = 0;
    // images per wave decided for (image size, form, images wanted): asked of the driver once
    int slots_key_n = -1, slots_key_node = -1, slots_key_want = -1, slots_cached = 0;
    void release()
    {
        slots_key_n = slots_key_node = slots_key_want = -1;
        plan.release();
        NdBuf *all[] = {&pix, &off, &off3, &lvl, &vec, &posg, &foff, &totals, &ast, &L, &U0, &U1, &UV0, &UV1, &scr, &info, &out_img, &relres, &relres_max};
        for (NdBuf *b : all) b->release();
    }
};

constexpr int ND_LEAF = 4;

static inline int nd_build_plan(NdPlan &pl, int n, int W, cudaStream_t st, std::string &err)
{
    if (pl.n == n && pl.sym.W == W) return 0;
    pl.release();
    pl.sym.build(n, W, ND_LEAF);
    const NdSymbolic &s = pl.sym;
    const int nf = (int)s.fronts.size();
    pl.posg_len = s.pixlist.size() + nf;
    std::vector<int> posg1(pl.posg_len);
    std::vector<long long> foff1((size_t)4 * nf);
    long long run[3] = {0, 0, 0}, lvl_max[2] = {0, 0};
    for (int stp = 0; stp < s.nsteps(); ++stp) {
        run[1] = run[2] = 0;
        for (int t = s.step_start[stp]; t < s.step_start[stp + 1]; ++t) {
            const NdFront &f = s.fronts[t];
            for (int k = 0; k <= f.npiv + f.nring; ++k) posg1[(size_t)f.pix0 + t + k] = k;
            long long sz[3];
            nd_front_sizes(f.npiv, f.nring, sz);
            for (int k = 0; k < 3; ++k) { foff1[4 * (size_t)t + k] = run[k]; run[k] += sz[k]; }
        }
        lvl_max[0] = std::max(lvl_max[0], run[1]); lvl_max[1] = std::max(lvl_max[1], run[2]);
    }
    pl.tot1[0] = run[0]; pl.tot1[1] = lvl_max[0]; pl.tot1[2] = lvl_max[1]; pl.tot1[3] = 0;
    auto up = [&](void **dst, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(dst, std::max<size_t>(bytes, 16));
        if (e == cudaSuccess) e = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, st);
        return e;
    };
    cudaError_t e = up(&pl.d_fronts, s.fronts.data(), s.fronts.size() * sizeof(NdFront));
    if (e == cudaSuccess) e = up(&pl.d_pixlist, s.pixlist.data(), s.pixlist.size() * sizeof(int));
    if (e == cudaSuccess) e = up(&pl.d_nbr, s.nbr.data(), s.nbr.size() * sizeof(int));
    if (e == cudaSuccess) e = up(&pl.d_cmap, s.cmap.data(), s.cmap.size() * sizeof(int));
    if (e == cudaSuccess) e = up(&pl.d_step_start, s.step_start.data(), s.step_start.size() * sizeof(int));
    if (e == cudaSuccess) e = up(&pl.d_posg1, posg1.data(), posg1.size() * sizeof(int));
    if (e == cudaSuccess) e = up(&pl.d_foff1, foff1.data(), foff1.size() * sizeof(long long));
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);     // the host vectors go out of scope
    if (e != cudaSuccess) { cudaGetLastError(); pl.release(); err = std::string("nested-dissection plan upload: ") + cudaGetErrorString(e); return -6; }
    pl.n = n;
    return 0;
}

static inline int nd_fail(NdWork &w, int code, const std::string &msg) { w.err = msg; return code; }

// Opt-in shared memory of the front kernels.  -1: a front does not fit (the caller falls back to a band solver).
static int nd_kernel_attributes(NdWork &w, size_t fsmem, size_t ssmem, size_t fsmem_small, size_t ssmem_small, size_t smem_optin,
                                size_t fsmem8 = 0,      // fsmem8: of the levels that take 8-column block steps
                                size_t fsmem_large = 0, size_t ssmem_large = 0)     // of the levels on the large-front variants
{
    if (fsmem > smem_optin || ssmem > smem_optin || fsmem_small > smem_optin || ssmem_small > smem_optin || fsmem8 > smem_optin ||
        fsmem_large > smem_optin || ssmem_large > smem_optin)
        return -1;      // the caller falls back to the band solver
    {
        // the opt-in shared-memory size is an attribute of the KERNEL on the current device, shared by every workspace
        // that launches it (the TV solver and the sum-of-regularisers one): raised to the largest any of them asked for
        static std::mutex mu;
        static int have[64][8] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        dev = std::max(0, std::min(63, dev));
        std::lock_guard<std::mutex> lock(mu);
        cudaError_t e = cudaSuccess;
        if (have[dev][0] < (int)fsmem) {
            e = cudaFuncSetAttribute(nd_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem);
            if (e == cudaSuccess) have[dev][0] = (int)fsmem;
        }
        if (e == cudaSuccess && have[dev][4] < (int)fsmem) {
            e = cudaFuncSetAttribute(nd_factor_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(nd_factor_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) have[dev][4] = (int)fsmem;
        }
        if (e == cudaSuccess && fsmem8 > 0 && have[dev][5] < (int)fsmem8) {
            e = cudaFuncSetAttribute(nd_factor8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem8);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(nd_factor8_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem8);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(nd_factor8_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) have[dev][5] = (int)fsmem8;
        }
        if (e == cudaSuccess && fsmem_large > 0 && have[dev][6] < (int)fsmem_large) {
            for (auto k : {nd_factor_large_kernel, nd_factor8_large_kernel, nd_factor_large_cluster_kernel, nd_factor8_large_cluster_kernel})
                if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem_large);
            for (auto k : {nd_factor_large_cluster_kernel, nd_factor8_large_cluster_kernel})
                if (e == cudaSuccess) e = cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e == cudaSuccess) have[dev][6] = (int)fsmem_large;
        }
        if (e == cudaSuccess && ssmem_large > 0 && have[dev][7] < (int)ssmem_large) {
            e = cudaFuncSetAttribute(nd_fwd_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem_large);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(nd_bwd_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem_large);
            if (e == cudaSuccess) have[dev][7] = (int)ssmem_large;
        }
        if (e == cudaSuccess && have[dev][1] < (int)ssmem) {
            e = cudaFuncSetAttribute(nd_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(nd_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem);
            if (e == cudaSuccess) have[dev][1] = (int)ssmem;
        }
        if (e == cudaSuccess && have[dev][2] < (int)fsmem_small) {
            e = cudaFuncSetAttribute(nd_factor_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem_small);
            if (e == cudaSuccess) have[dev][2] = (int)fsmem_small;
        }
        if (e == cudaSuccess && have[dev][3] < (int)ssmem_small) {
            e = cudaFuncSetAttribute(nd_fwd_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem_small);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(nd_bwd_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem_small);
            if (e == cudaSuccess) have[dev][3] = (int)ssmem_small;
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            char buf[160];
            snprintf(buf, sizeof buf, " (dynamic shared memory: factor %zu / %zu / %zu B, solves %zu / %zu B)", fsmem, fsmem8,
                     fsmem_large, ssmem, ssmem_large);
            return nd_fail(w, -2, std::string("nested-dissection kernel attributes: ") + cudaGetErrorString(e) + buf);
        }
    }
    return 0;
}

// Dynamic shared memory a front kernel may ask for: the opt-in maximum per block less the static shared memory of the
// factorisation kernels (their block-step flags, 16 B), which the opt-in maximum also has to hold.
static size_t nd_dynamic_optin(size_t smem_optin)
{
    static const size_t stat = [] {
        size_t m = 0;
        for (auto k : {nd_factor_kernel, nd_factor8_kernel, nd_factor_cluster_kernel, nd_factor8_cluster_kernel, nd_factor_large_kernel,
                       nd_factor8_large_kernel, nd_factor_large_cluster_kernel, nd_factor8_large_cluster_kernel}) {
            cudaFuncAttributes a;
            if (cudaFuncGetAttributes(&a, k) == cudaSuccess) m = std::max(m, a.sharedSizeBytes);
            else cudaGetLastError();
        }
        return m;
    }();
    return smem_optin > stat ? smem_optin - stat : 0;
}

// Shared memory (bytes) beyond which a level takes the large-front variants: the opt-in maximum.  Test hook:
// BPLTV_ND_LARGE_KB lowers it, so that small images run the variants where the shared-memory kernels can be compared.
static size_t nd_large_limit(size_t smem_optin)
{
    const char *e = bpltv::env_get("BPLTV_ND_LARGE_KB");
    return e && *e ? std::min<size_t>(smem_optin, (size_t)std::max(0, atoi(e)) << 10) : smem_optin;
}

// Launch plan of every level of the tree for `mb` unknowns per pixel at most (`fsz` typical): CTA sizes, shared memory of
// the largest front (worst case: mb unknowns on every pixel), kernel attributes.  -1: a front does not fit in shared
// memory and `large` is not set (the caller lets a band solver try first); with `large`, such levels take the
// large-front variants.
static int nd_prepare_levels(NdWork &w, const NdSymbolic &sym, int mb, double fsz, int O, size_t smem_optin, bool large,
                             std::vector<NdLevelPlan> &plan, std::vector<char> &plan_small)
{
    const int nsteps = sym.nsteps();
    // CTA size of the generic front factorisation: a stack of many images has fronts for every SM several times over, and
    // 4-warp CTAs (several per SM) beat 16-warp ones by 5–12 % (148 × 128²: 16.9 → 14.7 ms, 128 × 256²: 81.2 → 77.5 ms; the
    // kernel is bound by the barriers of its block steps, not by threads); few images keep the wide CTAs.  The CTA size of
    // the solves makes no measurable difference.  BPLTV_ND_WARPS_F / BPLTV_ND_THREADS_S override.
    const char *e1 = bpltv::env_get("BPLTV_ND_WARPS_F"), *e2 = bpltv::env_get("BPLTV_ND_THREADS_S");
    // (the width is now decided per level at launch time, nd_factor_cta_threads: the plan carries the widest CTA)
    const int cta_warps_f = e1 && *e1 ? std::max(2, std::min(16, atoi(e1))) : 16;
    (void)O;
    const int cta_threads_s = e2 && *e2 ? std::max(64, std::min(512, atoi(e2))) : 512;
    plan.assign(nsteps, NdLevelPlan());
    plan_small.assign(nsteps, 0);
    size_t fsmem = 0, ssmem = 0, fsmem_small = 0, ssmem_small = 0, fsmem_large = 0, ssmem_large = 0;
    const size_t limit = nd_large_limit(smem_optin);
    for (int s = 0; s < nsteps; ++s) {
        plan[s] = nd_level_plan(sym, s, mb, fsz, cta_warps_f, cta_threads_s);
        plan_small[s] = plan[s].small;
        if (plan[s].small) { fsmem_small = std::max(fsmem_small, plan[s].smem_f); ssmem_small = std::max(ssmem_small, plan[s].smem_s); }
        // every level can also run on the generic kernels
        if (!nd_level_large(plan[s], limit, smem_optin, large)) return -1;
        size_t &f = plan[s].large_f ? fsmem_large : fsmem, &g = plan[s].large_s ? ssmem_large : ssmem;
        f = std::max(f, nd_level_smem_f(plan[s]));
        g = std::max(g, nd_level_smem_s(plan[s]));
    }
    return nd_kernel_attributes(w, fsmem, ssmem, fsmem_small, ssmem_small, smem_optin, 0, fsmem_large, ssmem_large);
}

using NdFactorKernel = void (*)(NdDev, int, int, double, int);
// the generic factorisation kernel of a level: block width, where the panel lives, alone or shared by a cluster
static NdFactorKernel nd_factor_kernel_of(const NdLevelPlan &lp, bool cluster)
{
    if (lp.large_f)
        return lp.nb != ND_NB ? (cluster ? nd_factor8_large_cluster_kernel : nd_factor8_large_kernel)
                              : (cluster ? nd_factor_large_cluster_kernel : nd_factor_large_kernel);
    return lp.nb != ND_NB ? (cluster ? nd_factor8_cluster_kernel : nd_factor8_kernel) : (cluster ? nd_factor_cluster_kernel : nd_factor_kernel);
}

// CTAs per front of a level (a thread-block cluster shares the front: nd_factor_body<true>): the top levels of the tree
// have fewer fronts than the GPU has SMs, and their fronts are the large ones.  As many as leave every front of the
// wave its own cluster, while every warp of the cluster still has a tile of the trailing update.  BPLTV_ND_CLUSTER = 1
// switches it off, 2 / 4 / 8 / 16 caps the size; BPLTV_ND_CLUSTER_MINF: smallest front (unknowns) that is shared.
static int nd_cluster_size(const NdLevelPlan &lp, int cnt, int sm_count)
{
    const char *e1 = bpltv::env_get("BPLTV_ND_CLUSTER"), *e2 = bpltv::env_get("BPLTV_ND_CLUSTER_MINF");
    const int cap = e1 && *e1 ? std::max(1, std::min(16, atoi(e1))) : 16;
    const int minf = e2 && *e2 ? atoi(e2) : 256;
    if (lp.small || lp.nFw < minf || cap < 2) return 1;
    const long long fronts = (long long)lp.nfr * cnt;
    const int nt = (lp.nFw + 31) / 32, ntiles = nt * (nt + 1) / 2, warps = lp.threads_f / 32;
    long long C = std::min<long long>(cap, sm_count / std::max<long long>(1, fronts));
    C = std::min<long long>(C, ntiles / (2 * warps));       // two tiles per warp of the cluster at least
    return (int)std::max<long long>(1, C);
}

// how many clusters of C CTAs (threads, dynamic shared memory) of kernel k the device runs at once: asked of the driver
// once per shape
static int nd_active_clusters(NdFactorKernel k, int C, int threads, size_t smem)
{
    static std::mutex mu;
    static std::map<std::tuple<int, int, int, size_t, NdFactorKernel>, int> memo;
    int dev = 0;
    cudaGetDevice(&dev);
    const auto key = std::make_tuple(dev, C, threads, smem, k);
    std::lock_guard<std::mutex> lock(mu);
    auto it = memo.find(key);
    if (it != memo.end()) return it->second;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)C); cfg.blockDim = dim3((unsigned)threads); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int nclusters = 0;
    const cudaError_t qe = cudaOccupancyMaxActiveClusters(&nclusters, k, &cfg);
    if (qe != cudaSuccess) { cudaGetLastError(); nclusters = 0; }
    memo[key] = nclusters;
    return nclusters;
}

// launch of the cluster-shared front factorisation; the cluster shrinks until the device runs all fronts of the level at once
static cudaError_t nd_launch_factor_cluster(const NdDev &nd, const NdLevelPlan &lp, int s, int cnt, int C, double guard, cudaStream_t st)
{
    const size_t smem = nd_level_smem_f(lp);
    const long long fronts = (long long)lp.nfr * cnt;
    const NdFactorKernel kc = nd_factor_kernel_of(lp, true);
    while (C > 1 && nd_active_clusters(kc, C, lp.threads_f, smem) < fronts) --C;
    if (C > 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(lp.nfr * C), (unsigned)cnt);
        cfg.blockDim = dim3((unsigned)lp.threads_f);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, kc, nd, lp.t0, s & 1, guard, lp.nFw);
    }
    nd_factor_kernel_of(lp, false)<<<dim3(lp.nfr, cnt), lp.threads_f, smem, st>>>(nd, lp.t0, s & 1, guard, lp.nFw);
    return cudaGetLastError();
}

// scratch of the large-front variants (doubles per image): enough for any wave, whose clusters are at most as large as
// those of a single image
static size_t nd_scratch_doubles(const std::vector<NdLevelPlan> &plan, int sm_count)
{
    size_t m = 0;
    for (NdLevelPlan lp : plan) {
        lp.small = false;
        m = std::max(m, nd_level_scratch(lp, nd_cluster_size(lp, 1, sm_count)));
    }
    return nd_even((long long)m);
}

// the workspace could not be allocated: what one image needs, for the message
static int nd_alloc_fail(NdWork &w, const char *what, size_t bytes, size_t per_image, cudaError_t e)
{
    char buf[256];
    snprintf(buf, sizeof buf, "nested-dissection workspace (%s): %.3g GB could not be allocated, %.3g GB per image: %s", what,
             bytes * 1e-9, per_image * 1e-9, cudaGetErrorString(e));
    w.slots_key_n = -1;      // memory got tighter since the wave size was decided: ask again next time
    return nd_fail(w, -6, buf);
}

// CTA width of the generic front factorisation of one level.  A level with several fronts per SM runs narrow CTAs (4
// warps, four CTAs per SM: more independent fronts in flight hide the latency chain of a block step), a level with about
// one front per SM gives each front the whole SM (16 warps).  Measured as a global choice in round 2 (4 warps won by
// 5-12 % on stacks); per level the top of the tree no longer pays for it (ncu, 128 × 256²: the root level ran 128 CTAs of
// 4 warps, 43 tile rounds per block step).
static int nd_factor_cta_threads(const NdLevelPlan &lp, int cnt, int sm_count)
{
    const long long fronts = (long long)lp.nfr * cnt;
    const int cap = 2 * fronts <= 3LL * sm_count ? 16 : (fronts <= 3LL * sm_count ? 8 : 4);
    return std::min(lp.threads_f, 32 * cap);
}

// one launch per level: assemble + partial Cholesky of every front of the wave's `cnt` images
static void nd_launch_factor(const NdDev &nd, std::vector<NdLevelPlan> &plan, const std::vector<char> &plan_small,
                             const NdSymbolic &sym, int mb, int cnt, int sm_count, double guard, cudaStream_t st, long long *launches)
{
    const int nsteps = sym.nsteps();
    // the warp-per-front kernels pay off when the level has warps for every scheduler of the GPU; with few fronts (the
    // upper small levels of a single image) a CTA per front is faster (ncu, 1 image of 128²: 48 vs 117 µs at 256 fronts)
    for (int s = 0; s < nsteps; ++s) plan[s].small = plan_small[s] && (long long)plan[s].nfr * cnt >= 4LL * sm_count;
    for (int s = 0; s < nsteps; ++s) {
        const NdLevelPlan &lp = plan[s];
        if (lp.small)
            nd_factor_small_kernel<<<dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, cnt), 32 * ND_SMALL_WARPS, lp.smem_f, st>>>(
                nd, lp.t0, lp.nfr, s & 1, guard, lp.arena_f);
        else {
            const int C = nd_cluster_size(lp, cnt, sm_count);
            if (C > 1) nd_launch_factor_cluster(nd, lp, s, cnt, C, guard, st);
            else
                nd_factor_kernel_of(lp, false)<<<dim3(lp.nfr, cnt), nd_factor_cta_threads(lp, cnt, sm_count), nd_level_smem_f(lp), st>>>(
                    nd, lp.t0, s & 1, guard, lp.nFw);
        }
    }
    *launches += nsteps;
}

// L y = b up the tree, Lᵀ x = y down: `vec` (per image, `stride` doubles apart) is overwritten by the solution
static void nd_launch_solve(const NdDev &nd, const std::vector<NdLevelPlan> &plan, int cnt, double *vec, size_t stride,
                            cudaStream_t st, long long *launches)
{
    const int nsteps = (int)plan.size();
    for (int s = 0; s < nsteps; ++s) {
        const NdLevelPlan &lp = plan[s];
        if (lp.small)
            nd_fwd_small_kernel<<<dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, cnt), 32 * ND_SMALL_WARPS, lp.smem_s, st>>>(
                nd, lp.t0, lp.nfr, s & 1, vec, stride, lp.arena_s);
        else if (lp.large_s)
            nd_fwd_large_kernel<<<dim3(lp.nfr, cnt), lp.threads_s, nd_level_smem_s(lp), st>>>(nd, lp.t0, s & 1, vec, stride, lp.nFw);
        else
            nd_fwd_kernel<<<dim3(lp.nfr, cnt), lp.threads_s, nd_solve_smem(lp.nFw), st>>>(nd, lp.t0, s & 1, vec, stride);
    }
    for (int s = nsteps - 1; s >= 0; --s) {
        const NdLevelPlan &lp = plan[s];
        if (lp.small)
            nd_bwd_small_kernel<<<dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, cnt), 32 * ND_SMALL_WARPS, lp.smem_s, st>>>(
                nd, lp.t0, lp.nfr, vec, stride, lp.arena_s);
        else if (lp.large_s)
            nd_bwd_large_kernel<<<dim3(lp.nfr, cnt), lp.threads_s, nd_level_smem_s(lp), st>>>(nd, lp.t0, vec, stride, lp.nFw);
        else
            nd_bwd_kernel<<<dim3(lp.nfr, cnt), lp.threads_s, nd_solve_smem(lp.nFw), st>>>(nd, lp.t0, vec, stride);
    }
    *launches += 2 * nsteps;
}

template <typename Real>
static int run_gradient_nd(NdWork &w, const NdProblem &gp, int sm_count, size_t smem_optin,
                           cudaStream_t st, double *d_grad_out, long long *launches)
{
    NdWork &gw = w;
    smem_optin = nd_dynamic_optin(smem_optin);
    const Real *gp_u = static_cast<const Real *>(gp.u), *gp_ubar = static_cast<const Real *>(gp.ubar),
               *gp_amap = static_cast<const Real *>(gp.alpha_map);
    const int n = gp.M, N = gp.M * gp.N, ng = gp.lm * gp.ln;
    if (gp.M != gp.N) return nd_fail(gw, -1, "square images required");
    if (ng > 65536) return nd_fail(gw, -1, "lambda grid larger than 65536 entries is not supported");
    const bool node = gp.regularised;
    const int mb = node ? 1 : 2;
    {
        const int rc = nd_build_plan(w.plan, n, 1, st, gw.err);
        if (rc != 0) return rc;
    }
    const NdSymbolic &sym = w.plan.sym;
    const int nf = (int)sym.fronts.size(), nsteps = sym.nsteps();
    if (nsteps > 62) return nd_fail(gw, -1, "image too large for the nested-dissection level table");
    // launch plan of every level (CTA sizes, shared memory, kernel attributes)
    const double fsz = node ? 1.0 : 1.25;        // typical unknowns per pixel, for CTA sizes and arenas only
    std::vector<NdLevelPlan> plan;
    std::vector<char> plan_small;
    {
        const int rc = nd_prepare_levels(w, sym, mb, fsz, gp.O, smem_optin, gp.large_fronts, plan, plan_small);
        if (rc != 0) return rc;
    }
    const size_t scr_stride = nd_scratch_doubles(plan, sm_count);

    // ---- per-slot sizes.  Pools of the MULT form are estimated at 2.2× the one-unknown-per-pixel sizes (≈ 1.5
    // unknowns per pixel) and grown when a wave needs more.
    const long long *t1 = w.plan.tot1;
    const double est = node ? 1.0 : 2.2;
    const size_t fix_bytes = (size_t)NDTV_PLANES * N * 8 + (size_t)5 * mb * mb * N * 8 +
                             (node ? 0 : ((size_t)N + 2) * 4 + (size_t)6 * N * 8 + w.plan.posg_len * 4 + (size_t)4 * nf * 8 + 32) + 16;
    const size_t pool_bytes = (size_t)(est * (double)(t1[0] + 2 * t1[1] + 2 * t1[2])) * 8 + scr_stride * 8;
    const size_t per_slot = fix_bytes + pool_bytes;
    w.last_bytes_per_image = per_slot;
    int slots = std::min(gp.O, 256);      // 256 images already give every level thousands of fronts
    if (w.slots_key_n == n && w.slots_key_node == (int)node && w.slots_key_want == slots) {
        slots = w.slots_cached;           // the same question as last time: no free-memory query on the evaluation path
    } else {
        const int want = slots;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t have = w.pix.bytes + w.ast.bytes + w.L.bytes + w.U0.bytes + w.U1.bytes + w.vec.bytes + w.posg.bytes + w.foff.bytes;
        const size_t budget = (free_b + have) / 2;
        slots = (int)std::min<size_t>((size_t)slots, std::max<size_t>(1, budget / per_slot));
        w.slots_key_n = n; w.slots_key_node = (int)node; w.slots_key_want = want; w.slots_cached = slots;
    }
    auto need = [&](NdBuf &b, size_t bytes, const char *what) -> int {
        const cudaError_t e = b.ensure(bytes);
        return e == cudaSuccess ? 0 : nd_alloc_fail(gw, what, bytes, w.last_bytes_per_image, e);
    };
    int rc = 0;
    NdTvSlots ws;
    ws.n = n; ws.N = N;
    ws.pix_stride = (size_t)NDTV_PLANES * N;
    ws.off_stride = (size_t)N + 2;
    ws.vec_stride = (size_t)6 * N;
    const size_t ast_stride = (size_t)5 * mb * mb * N;
    if ((rc = need(w.pix, ws.pix_stride * 8 * slots, "pixel planes"))) return rc;
    if ((rc = need(w.ast, ast_stride * 8 * slots, "stencil matrix"))) return rc;
    if ((rc = need(w.info, (size_t)16 * slots, "info"))) return rc;
    if ((rc = need(w.out_img, (size_t)gp.O * ng * 8, "per-image gradients"))) return rc;
    if ((rc = need(w.relres, (size_t)gp.O * 8, "residuals"))) return rc;
    if ((rc = need(w.relres_max, 16, "residual maximum"))) return rc;
    if (!node) {
        if ((rc = need(w.off, ws.off_stride * 4 * slots, "mode offsets"))) return rc;
        if ((rc = need(w.vec, ws.vec_stride * 8 * slots, "mode vectors"))) return rc;
        if ((rc = need(w.posg, w.plan.posg_len * 4 * slots, "front offsets"))) return rc;
        if ((rc = need(w.foff, (size_t)4 * nf * 8 * slots, "pool offsets"))) return rc;
        if ((rc = need(w.totals, (size_t)32 * slots, "pool totals"))) return rc;
    }
    ws.pix = (double *)w.pix.p; ws.off = (int *)w.off.p; ws.vec = (double *)w.vec.p; ws.info = (int *)w.info.p;

    NdDev nd;
    nd.n = n; nd.N = N; nd.W = 1; nd.nnb = sym.nnb; nd.nh = nd_nh(1); nd.mb = mb;
    nd.nfronts = nf; nd.nsteps = nsteps;
    nd.fronts = (const NdFront *)w.plan.d_fronts; nd.pixlist = (const int *)w.plan.d_pixlist;
    nd.nbr = (const int *)w.plan.d_nbr; nd.cmap = (const int *)w.plan.d_cmap; nd.step_start = (const int *)w.plan.d_step_start;
    if (node) {
        nd.off = nullptr; nd.off_stride = 0;
        nd.posg = (int *)w.plan.d_posg1; nd.posg_stride = 0;
        nd.foff = (long long *)w.plan.d_foff1; nd.foff_stride = 0;
        nd.totals = nullptr;
    } else {
        nd.off = ws.off; nd.off_stride = ws.off_stride;
        nd.posg = (int *)w.posg.p; nd.posg_stride = w.plan.posg_len;
        nd.foff = (long long *)w.foff.p; nd.foff_stride = (size_t)4 * nf;
        nd.totals = (long long *)w.totals.p;
    }
    nd.ast = (const double *)w.ast.p; nd.ast_stride = ast_stride;
    nd.info = ws.info;

    NdTvVariant gv;
    gv.patch = gp.alpha_map != nullptr; gv.lm = gp.lm; gv.ln = gp.ln;
    gv.alpha_s = gp.alpha_s; gv.gamma = gp.gamma; gv.act_tol = gp.act_tol; gv.eps_act = gp.eps_act;
    gv.relres_tol = gp.tol > 0 ? gp.tol : 1e300;
    const double guard = node ? 0.0 : 1e-13;
    const int refine = gp.maxit > 0 ? std::min(gp.maxit, 8) : 1;
    const int chunks = std::max(1, std::min(64, (N + 255) / 256));
    const int pgroups = std::max(1, std::min(ng, 32));

    for (int img0 = 0; img0 < gp.O; img0 += slots) {
        const int cnt = std::min(slots, gp.O - img0);
        size_t Ls, Us, UVs;
        if (node) {
            ndtv_classify_node_kernel<Real><<<dim3(cnt, chunks), 256, 0, st>>>(ws, gv, gp_u, gp_ubar, gp_amap, img0);
            ndtv_stencil_node_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, (double *)w.ast.p, ast_stride);
            *launches += 2;
            Ls = (size_t)t1[0]; Us = (size_t)t1[1]; UVs = (size_t)t1[2];
        } else {
            ndtv_classify_mult_kernel<Real><<<cnt, 1024, 0, st>>>(ws, gv, gp_u, gp_ubar, gp_amap, img0);
            nd_dims_kernel<<<dim3((nf + 7) / 8, cnt), 256, 0, st>>>(nd);
            nd_scan_kernel<<<cnt, 256, 0, st>>>(nd);
            ndtv_stencil_mult_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, (double *)w.ast.p, ast_stride);
            *launches += 4;
            w.h_totals.resize((size_t)4 * cnt);
            cudaError_t e = cudaMemcpyAsync(w.h_totals.data(), w.totals.p, (size_t)32 * cnt, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { cudaGetLastError(); return nd_fail(gw, -2, std::string("nested-dissection sizes: ") + cudaGetErrorString(e)); }
            long long m[4] = {0, 0, 0, 0};
            for (int s = 0; s < cnt; ++s)
                for (int k = 0; k < 4; ++k) m[k] = std::max(m[k], w.h_totals[4 * (size_t)s + k]);
            Ls = (size_t)m[0]; Us = (size_t)m[1]; UVs = (size_t)m[2];
        }
        Ls = (Ls + 1) & ~(size_t)1; Us = (Us + 1) & ~(size_t)1; UVs = (UVs + 1) & ~(size_t)1;
        w.last_bytes_per_image = fix_bytes + (Ls + 2 * Us + 2 * UVs + scr_stride) * 8;
        if ((rc = need(w.L, Ls * 8 * cnt, "factors"))) return rc;
        if ((rc = need(w.U0, Us * 8 * cnt, "update matrices"))) return rc;
        if ((rc = need(w.U1, Us * 8 * cnt, "update matrices"))) return rc;
        if ((rc = need(w.UV0, UVs * 8 * cnt, "update vectors"))) return rc;
        if ((rc = need(w.UV1, UVs * 8 * cnt, "update vectors"))) return rc;
        if (scr_stride && (rc = need(w.scr, scr_stride * 8 * cnt, "large-front scratch"))) return rc;
        nd.L = (double *)w.L.p; nd.L_stride = Ls;
        nd.U[0] = (double *)w.U0.p; nd.U[1] = (double *)w.U1.p; nd.U_stride = Us;
        nd.UV[0] = (double *)w.UV0.p; nd.UV[1] = (double *)w.UV1.p; nd.UV_stride = UVs;
        nd.scr = (double *)w.scr.p; nd.scr_stride = scr_stride;
        w.last_bytes_per_image = fix_bytes + (Ls + 2 * Us + 2 * UVs + scr_stride) * 8;

        nd_launch_factor(nd, plan, plan_small, sym, mb, cnt, sm_count, guard, st, launches);
        auto solve = [&](double *vec, size_t stride) { nd_launch_solve(nd, plan, cnt, vec, stride, st, launches); };
        if (node) {
            double *p = ws.pix + 7 * (size_t)N, *work = ws.pix + 8 * (size_t)N;
            solve(p, ws.pix_stride);
            ndtv_residual_node_kernel<<<cnt, 1024, 0, st>>>(ws, (double *)w.relres.p, img0);
            for (int it = 0; it < refine; ++it) {
                solve(work, ws.pix_stride);
                ndtv_axpy_node_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, 7, 8);
                ndtv_residual_node_kernel<<<cnt, 1024, 0, st>>>(ws, (double *)w.relres.p, img0);
            }
            ndtv_finish_node_kernel<<<dim3(cnt, pgroups), 512, 0, st>>>(ws, gv, (const double *)w.relres.p, (double *)w.out_img.p, img0);
            *launches += 2 + 2 * refine;
        } else {
            double *zeta = ws.vec + 2 * (size_t)N, *work = ws.vec + 4 * (size_t)N;
            ndtv_copy_mult_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, 1, 0);
            solve(zeta, ws.vec_stride);
            ndtv_residual_mult_kernel<<<cnt, 1024, 0, st>>>(ws, (double *)w.relres.p, img0);
            for (int it = 0; it < refine; ++it) {
                solve(work, ws.vec_stride);
                ndtv_axpy_mult_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, 1, 2);
                ndtv_residual_mult_kernel<<<cnt, 1024, 0, st>>>(ws, (double *)w.relres.p, img0);
            }
            ndtv_finish_mult_kernel<<<dim3(cnt, pgroups), 512, 0, st>>>(ws, gv, (const double *)w.relres.p, (double *)w.out_img.p, img0);
            *launches += 3 + 2 * refine;
        }
    }
    nd_reduce_kernel<<<(ng + 255) / 256, 256, 0, st>>>((double *)w.out_img.p, (double *)w.relres.p, gp.O, ng, d_grad_out,
                                                         (double *)w.relres_max.p);
    *launches += 1;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return nd_fail(gw, -2, std::string("nested-dissection kernel launch failed: ") + cudaGetErrorString(e));
    return 0;
}

// ---------------------------------------------------------------------------
// scalar sumregs_gradient_reg on the same solver (nd_sumregs.cuh): node space, one unknown per node, W = 2
// ---------------------------------------------------------------------------
template <typename Real>
static int run_gradient3_nd_reg(NdWork &w, const Nd3Problem &gp, int sm_count, size_t smem_optin, cudaStream_t st,
                                double *d_grad_out, long long *launches)
{
    const Real *gp_u = static_cast<const Real *>(gp.u), *gp_ubar = static_cast<const Real *>(gp.ubar);
    const int n = gp.M, N = gp.M * gp.N, nops = 3, ng = 1;
    smem_optin = nd_dynamic_optin(smem_optin);
    if (gp.M != gp.N) return nd_fail(w, -1, "square images required");
    if (n < 8) return -1;                                   // tiny images: the band LU
    {
        const int rc = nd_build_plan(w.plan, n, ND3_W, st, w.err);
        if (rc != 0) return rc;
    }
    const NdSymbolic &sym = w.plan.sym;
    const int nf = (int)sym.fronts.size(), nsteps = sym.nsteps();
    if (nsteps > 62) return nd_fail(w, -1, "image too large for the nested-dissection level table");
    std::vector<NdLevelPlan> plan;
    std::vector<char> plan_small;
    {
        const int rc = nd_prepare_levels(w, sym, 1, 1.0, gp.O, smem_optin, gp.large_fronts, plan, plan_small);
        if (rc != 0) return rc;
    }
    const long long *t1 = w.plan.tot1;
    const size_t pix_stride = (size_t)LU_PLANES * N, ast_stride = (size_t)ND3_NH * N;
    const size_t Ls = ((size_t)t1[0] + 1) & ~(size_t)1, Us = ((size_t)t1[1] + 1) & ~(size_t)1, UVs = ((size_t)t1[2] + 1) & ~(size_t)1;
    const size_t scr_stride = nd_scratch_doubles(plan, sm_count);
    const size_t per_slot = (pix_stride + ast_stride + Ls + 2 * Us + 2 * UVs + scr_stride) * 8 + 16;
    w.last_bytes_per_image = per_slot;
    int slots = std::min(gp.O, 256);
    if (w.slots_key_n == n && w.slots_key_node == 3 && w.slots_key_want == slots) {
        slots = w.slots_cached;
    } else {
        const int want = slots;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t have = w.pix.bytes + w.ast.bytes + w.L.bytes + w.U0.bytes + w.U1.bytes;
        const size_t budget = (free_b + have) / 2;
        slots = (int)std::min<size_t>((size_t)slots, std::max<size_t>(1, budget / per_slot));
        w.slots_key_n = n; w.slots_key_node = 3; w.slots_key_want = want; w.slots_cached = slots;
    }
    auto need = [&](NdBuf &b, size_t bytes, const char *what) -> int {
        const cudaError_t e = b.ensure(bytes);
        return e == cudaSuccess ? 0 : nd_alloc_fail(w, what, bytes, w.last_bytes_per_image, e);
    };
    int rc = 0;
    if ((rc = need(w.pix, pix_stride * 8 * slots, "pixel planes"))) return rc;
    if ((rc = need(w.ast, ast_stride * 8 * slots, "stencil matrix"))) return rc;
    if ((rc = need(w.info, (size_t)16 * slots, "info"))) return rc;
    if ((rc = need(w.out_img, (size_t)gp.O * nops * ng * 8, "per-image gradients"))) return rc;
    if ((rc = need(w.relres, (size_t)gp.O * 8, "residuals"))) return rc;
    if ((rc = need(w.relres_max, 16, "residual maximum"))) return rc;
    if ((rc = need(w.L, Ls * 8 * slots, "factors"))) return rc;
    if ((rc = need(w.U0, Us * 8 * slots, "update matrices"))) return rc;
    if ((rc = need(w.U1, Us * 8 * slots, "update matrices"))) return rc;
    if ((rc = need(w.UV0, UVs * 8 * slots, "update vectors"))) return rc;
    if ((rc = need(w.UV1, UVs * 8 * slots, "update vectors"))) return rc;
    if (scr_stride && (rc = need(w.scr, scr_stride * 8 * slots, "large-front scratch"))) return rc;

    LuSlots ws;
    ws.ab = nullptr; ws.ab_stride = 0; ws.pix = (double *)w.pix.p; ws.pix_stride = pix_stride; ws.info = (int *)w.info.p;
    ws.n = n; ws.N = N; ws.bw = 0; ws.bwx = 0; ws.LD = 0; ws.use_pin = 0; ws.nops = nops;
    Lu3Params pr;
    for (int k = 0; k < 3; ++k) pr.alpha[k] = gp.alpha[k];
    pr.gamma = gp.gamma; pr.lm = 1; pr.ln = 1; pr.refine = 0;

    NdDev nd;
    nd.n = n; nd.N = N; nd.W = ND3_W; nd.nnb = sym.nnb; nd.nh = nd_nh(ND3_W); nd.mb = 1;
    nd.nfronts = nf; nd.nsteps = nsteps;
    nd.fronts = (const NdFront *)w.plan.d_fronts; nd.pixlist = (const int *)w.plan.d_pixlist;
    nd.nbr = (const int *)w.plan.d_nbr; nd.cmap = (const int *)w.plan.d_cmap; nd.step_start = (const int *)w.plan.d_step_start;
    nd.off = nullptr; nd.off_stride = 0;
    nd.posg = (int *)w.plan.d_posg1; nd.posg_stride = 0;
    nd.foff = (long long *)w.plan.d_foff1; nd.foff_stride = 0;
    nd.totals = nullptr;
    nd.L = (double *)w.L.p; nd.L_stride = Ls;
    nd.U[0] = (double *)w.U0.p; nd.U[1] = (double *)w.U1.p; nd.U_stride = Us;
    nd.UV[0] = (double *)w.UV0.p; nd.UV[1] = (double *)w.UV1.p; nd.UV_stride = UVs;
    nd.ast = (const double *)w.ast.p; nd.ast_stride = ast_stride;
    nd.info = (int *)w.info.p;
    nd.scr = (double *)w.scr.p; nd.scr_stride = scr_stride;

    const double tol = gp.tol > 0 ? gp.tol : 1e300;
    const int refine = gp.maxit > 0 ? std::min(gp.maxit, 8) : 1;
    const int chunks = std::max(1, std::min(64, (N + 255) / 256));
    for (int img0 = 0; img0 < gp.O; img0 += slots) {
        const int cnt = std::min(slots, gp.O - img0);
        cudaMemsetAsync(w.ast.p, 0, ast_stride * 8 * cnt, st);
        cudaMemsetAsync(w.info.p, 0, (size_t)16 * cnt, st);
        lu3_classify_kernel<Real><<<dim3(cnt, chunks), 256, 0, st>>>(ws, pr.gamma, gp_u, gp_ubar, img0);
        nd3_stencil_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, pr, (double *)w.ast.p, ast_stride);
        *launches += 2;
        nd_launch_factor(nd, plan, plan_small, sym, 1, cnt, sm_count, 0.0, st, launches);
        double *p = ws.pix + (size_t)LU_PL_P * N, *work = ws.pix + (size_t)LU_PL_WORK * N;
        nd_launch_solve(nd, plan, cnt, p, pix_stride, st, launches);
        nd3_residual_kernel<Real><<<cnt, 1024, 0, st>>>(ws, pr, (double *)w.relres.p, img0);
        for (int it = 0; it < refine; ++it) {
            nd_launch_solve(nd, plan, cnt, work, pix_stride, st, launches);
            nd3_axpy_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws);
            nd3_residual_kernel<Real><<<cnt, 1024, 0, st>>>(ws, pr, (double *)w.relres.p, img0);
        }
        nd3_finish_kernel<<<cnt, 1024, 0, st>>>(ws, pr, (const int *)w.info.p, tol, (double *)w.out_img.p, (double *)w.relres.p, img0);
        *launches += 2 + 2 * refine;
    }
    nd_reduce_kernel<<<1, 32, 0, st>>>((double *)w.out_img.p, (double *)w.relres.p, gp.O, nops * ng, d_grad_out,
                                       (double *)w.relres_max.p);
    *launches += 1;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return nd_fail(w, -2, std::string("nested-dissection kernel launch failed: ") + cudaGetErrorString(e));
    return 0;
}

// ---------------------------------------------------------------------------
// sumregs_gradient (non-regularised) on the same solver: multiplier space, 3-6 unknowns per pixel, W = 2.  Front sizes
// are data: measured per level on the device (nd_level_sizes_kernel) and read back with the pool totals, one
// synchronisation per wave; a front beyond shared memory sends the call back to the band Cholesky (-1), or, with
// gp.large_fronts (the band Cholesky refused the shape too), to the large-front variants.
// ---------------------------------------------------------------------------
template <typename Real>
static int run_gradient3_nd_mult(NdWork &w, const Nd3mProblem &gp, int sm_count, size_t smem_optin, cudaStream_t st,
                                 double *d_grad_out, long long *launches)
{
    const Real *gp_u = static_cast<const Real *>(gp.u), *gp_ubar = static_cast<const Real *>(gp.ubar),
               *gp_amaps = static_cast<const Real *>(gp.alpha_maps);
    const int n = gp.M, N = gp.M * gp.N, ng = gp.lm * gp.ln, mb = ND3M_MB;
    smem_optin = nd_dynamic_optin(smem_optin);
    if (gp.M != gp.N) return nd_fail(w, -1, "square images required");
    if (n < 8) return -1;
    if (3 * ng > 65536) return nd_fail(w, -1, "lambda grid too large");
    {
        const int rc = nd_build_plan(w.plan, n, ND3_W, st, w.err);
        if (rc != 0) return rc;
    }
    const NdSymbolic &sym = w.plan.sym;
    const int nf = (int)sym.fronts.size(), nsteps = sym.nsteps();
    if (nsteps > 62) return nd_fail(w, -1, "image too large for the nested-dissection level table");
    const char *e1 = bpltv::env_get("BPLTV_ND_WARPS_F");
    const int cta_warps_f = e1 && *e1 ? std::max(2, std::min(16, atoi(e1))) : 16;

    const long long *t1 = w.plan.tot1;
    const size_t pix_stride = (size_t)ND3M_PLANES * N, ast_stride = (size_t)ND3_NH * mb * mb * N;
    const size_t off3_stride = (size_t)3 * N + 1, poff_stride = (size_t)N + 2, vec_stride = (size_t)3 * mb * N;
    const size_t fix_bytes = (pix_stride + ast_stride + vec_stride) * 8 + (off3_stride + poff_stride + w.plan.posg_len) * 4 +
                             (size_t)4 * nf * 8 + 32 + 16;
    // pools grow with the square of the unknowns per pixel: estimated at 4 per pixel, checked against the measured sizes
    const size_t pool_est = (size_t)(16.0 * (double)(t1[0] + 2 * t1[1]) + 4.0 * (double)(2 * t1[2])) * 8;
    int slots = std::min(gp.O, 64);
    if (w.slots_key_n == n && w.slots_key_node == 4 && w.slots_key_want == slots) {
        slots = w.slots_cached;
    } else {
        const int want = slots;
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t have = w.pix.bytes + w.ast.bytes + w.L.bytes + w.U0.bytes + w.U1.bytes + w.vec.bytes + w.posg.bytes + w.foff.bytes;
        w.budget_cached = (free_b + have) / 2;
        {   // test hook: BPLTV_ND3_BUDGET_MB replaces the memory budget of a wave (exercises the smaller-wave retry)
            const char *bm = bpltv::env_get("BPLTV_ND3_BUDGET_MB");
            if (bm && *bm) w.budget_cached = (size_t)atoll(bm) << 20;
        }
        slots = (int)std::min<size_t>((size_t)slots, std::max<size_t>(1, w.budget_cached / (fix_bytes + pool_est)));
        w.slots_key_n = n; w.slots_key_node = 4; w.slots_key_want = want; w.slots_cached = slots;
    }
    auto need = [&](NdBuf &b, size_t bytes, const char *what) -> int {
        const cudaError_t e = b.ensure(bytes);
        return e == cudaSuccess ? 0 : nd_alloc_fail(w, what, bytes, w.last_bytes_per_image, e);
    };
    int rc = 0;
    if ((rc = need(w.out_img, (size_t)gp.O * 3 * ng * 8, "per-image gradients"))) return rc;
    if ((rc = need(w.relres, (size_t)gp.O * 8, "residuals"))) return rc;
    if ((rc = need(w.relres_max, 16, "residual maximum"))) return rc;
    if ((rc = need(w.lvl, 512, "level sizes"))) return rc;

    Nd3mVariant gv;
    gv.patch = gp.alpha_maps != nullptr; gv.lm = gp.lm; gv.ln = gp.ln;
    for (int k = 0; k < 3; ++k) gv.alpha[k] = gp.alpha[k];
    gv.act_tol = gp.act_tol; gv.eps_act = gp.eps_act; gv.relres_tol = gp.tol > 0 ? gp.tol : 1e300;
    const double guard = 1e-13;
    const int refine = gp.maxit > 0 ? std::min(gp.maxit, 8) : 1;
    const int chunks = std::max(1, std::min(64, (N + 255) / 256));
    const int chunks_st = std::max(1, std::min(512, (int)(((long long)N * ND3_NH + 255) / 256)));
    std::vector<NdLevelPlan> plan(nsteps);
    const std::vector<char> plan_small(nsteps, 0);
    int h_lvl[128];

    for (int img0 = 0; img0 < gp.O;) {
        const int cnt = std::min(slots, gp.O - img0);
        if ((rc = need(w.pix, pix_stride * 8 * slots, "pixel planes"))) return rc;
        if ((rc = need(w.ast, ast_stride * 8 * slots, "stencil matrix"))) return rc;
        if ((rc = need(w.info, (size_t)16 * slots, "info"))) return rc;
        if ((rc = need(w.off, poff_stride * 4 * slots, "mode offsets"))) return rc;
        if ((rc = need(w.off3, off3_stride * 4 * slots, "mode offsets"))) return rc;
        if ((rc = need(w.vec, vec_stride * 8 * slots, "mode vectors"))) return rc;
        if ((rc = need(w.posg, w.plan.posg_len * 4 * slots, "front offsets"))) return rc;
        if ((rc = need(w.foff, (size_t)4 * nf * 8 * slots, "pool offsets"))) return rc;
        if ((rc = need(w.totals, (size_t)32 * slots, "pool totals"))) return rc;
        Nd3mSlots ws;
        ws.n = n; ws.N = N; ws.pix = (double *)w.pix.p; ws.pix_stride = pix_stride;
        ws.off3 = (int *)w.off3.p; ws.off3_stride = off3_stride; ws.poff = (int *)w.off.p; ws.poff_stride = poff_stride;
        ws.vec = (double *)w.vec.p; ws.vec_stride = vec_stride; ws.info = (int *)w.info.p;
        NdDev nd;
        nd.n = n; nd.N = N; nd.W = ND3_W; nd.nnb = sym.nnb; nd.nh = nd_nh(ND3_W); nd.mb = mb;
        nd.nfronts = nf; nd.nsteps = nsteps;
        nd.fronts = (const NdFront *)w.plan.d_fronts; nd.pixlist = (const int *)w.plan.d_pixlist;
        nd.nbr = (const int *)w.plan.d_nbr; nd.cmap = (const int *)w.plan.d_cmap; nd.step_start = (const int *)w.plan.d_step_start;
        nd.off = ws.poff; nd.off_stride = poff_stride;
        nd.posg = (int *)w.posg.p; nd.posg_stride = w.plan.posg_len;
        nd.foff = (long long *)w.foff.p; nd.foff_stride = (size_t)4 * nf;
        nd.totals = (long long *)w.totals.p;
        nd.ast = (const double *)w.ast.p; nd.ast_stride = ast_stride;
        nd.info = ws.info;

        cudaMemsetAsync(w.lvl.p, 0, 512, st);
        nd3m_classify_kernel<Real><<<cnt, 1024, 0, st>>>(ws, gv, gp_u, gp_ubar, gp_amaps, img0);
        nd_dims_kernel<<<dim3((nf + 7) / 8, cnt), 256, 0, st>>>(nd);
        nd_scan_kernel<<<cnt, 256, 0, st>>>(nd);
        nd_level_sizes_kernel<<<dim3((nf + 255) / 256, cnt), 256, 0, st>>>(nd, (int *)w.lvl.p);
        nd3m_stencil_kernel<<<dim3(cnt, chunks_st), 256, 0, st>>>(ws, (double *)w.ast.p, ast_stride);
        *launches += 5;
        w.h_totals.resize((size_t)4 * cnt);
        cudaError_t e = cudaMemcpyAsync(w.h_totals.data(), w.totals.p, (size_t)32 * cnt, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_lvl, w.lvl.p, 512, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { cudaGetLastError(); return nd_fail(w, -2, std::string("nested-dissection sizes: ") + cudaGetErrorString(e)); }
        long long m[4] = {0, 0, 0, 0};
        for (int s = 0; s < cnt; ++s)
            for (int k = 0; k < 4; ++k) m[k] = std::max(m[k], w.h_totals[4 * (size_t)s + k]);
        const size_t Ls = ((size_t)m[0] + 1) & ~(size_t)1, Us = ((size_t)m[1] + 1) & ~(size_t)1, UVs = ((size_t)m[2] + 1) & ~(size_t)1;
        const size_t pool_bytes = (Ls + 2 * Us + 2 * UVs) * 8;
        w.last_bytes_per_image = fix_bytes + pool_bytes;
        if (cnt > 1 && (fix_bytes + pool_bytes) * cnt > w.budget_cached && w.budget_cached > 0) {
            // the images carry more unknowns than estimated: a smaller wave, classified again
            slots = (int)std::max<size_t>(1, std::min<size_t>((size_t)cnt - 1, w.budget_cached / (fix_bytes + pool_bytes)));
            w.slots_cached = slots;
            continue;
        }
        size_t fsmem = 0, fsmem8 = 0, ssmem = 0, fsmem_large = 0, ssmem_large = 0;
        // test hook: BPLTV_ND3_SMEM_KB lowers the shared memory the 16-column panel may take (sends fronts to the 8-column kernels)
        const char *skb = bpltv::env_get("BPLTV_ND3_SMEM_KB");
        const size_t smem_plan = skb && *skb ? std::min<size_t>(smem_optin, (size_t)atoi(skb) << 10) : smem_optin;
        const size_t limit = nd_large_limit(smem_optin);
        for (int s = 0; s < nsteps; ++s) {
            plan[s] = nd_level_plan_sized(sym, s, h_lvl[2 * s], s > 0 ? h_lvl[2 * (s - 1) + 1] : 0, smem_plan, cta_warps_f, 512);
            if (!nd_level_large(plan[s], limit, smem_optin, gp.large_fronts)) return -1;      // the band Cholesky first
            if (plan[s].large_f) fsmem_large = std::max(fsmem_large, plan[s].smem_f);
            else if (plan[s].nb == ND_NB) fsmem = std::max(fsmem, plan[s].smem_f);
            else fsmem8 = std::max(fsmem8, plan[s].smem_f);
            size_t &g = plan[s].large_s ? ssmem_large : ssmem;
            g = std::max(g, plan[s].smem_s);
        }
        const size_t scr_stride = nd_scratch_doubles(plan, sm_count);
        w.last_bytes_per_image += scr_stride * 8;
        {   // test hook: BPLTV_ND3_MAXF caps the front size this path takes (exercises the fall-back below)
            const char *mf = bpltv::env_get("BPLTV_ND3_MAXF");
            if (mf && *mf)
                for (int s = 0; s < nsteps; ++s)
                    if (h_lvl[2 * s] > atoi(mf)) return -1;
        }
        if ((rc = nd_kernel_attributes(w, fsmem, ssmem, 0, 0, smem_optin, fsmem8, fsmem_large, ssmem_large))) return rc;
        if ((rc = need(w.L, Ls * 8 * cnt, "factors"))) return rc;
        if ((rc = need(w.U0, Us * 8 * cnt, "update matrices"))) return rc;
        if ((rc = need(w.U1, Us * 8 * cnt, "update matrices"))) return rc;
        if ((rc = need(w.UV0, UVs * 8 * cnt, "update vectors"))) return rc;
        if ((rc = need(w.UV1, UVs * 8 * cnt, "update vectors"))) return rc;
        if (scr_stride && (rc = need(w.scr, scr_stride * 8 * cnt, "large-front scratch"))) return rc;
        nd.L = (double *)w.L.p; nd.L_stride = Ls;
        nd.U[0] = (double *)w.U0.p; nd.U[1] = (double *)w.U1.p; nd.U_stride = Us;
        nd.UV[0] = (double *)w.UV0.p; nd.UV[1] = (double *)w.UV1.p; nd.UV_stride = UVs;
        nd.scr = (double *)w.scr.p; nd.scr_stride = scr_stride;

        nd_launch_factor(nd, plan, plan_small, sym, mb, cnt, sm_count, guard, st, launches);
        double *zeta = ws.vec + (size_t)mb * N, *work = ws.vec + (size_t)2 * mb * N;
        nd3m_axpy_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, 1, 0, 0);
        nd_launch_solve(nd, plan, cnt, zeta, vec_stride, st, launches);
        nd3m_residual_kernel<<<cnt, 1024, 0, st>>>(ws, (double *)w.relres.p, img0);
        for (int it = 0; it < refine; ++it) {
            nd_launch_solve(nd, plan, cnt, work, vec_stride, st, launches);
            nd3m_axpy_kernel<<<dim3(cnt, chunks), 256, 0, st>>>(ws, 1, 2, 1);
            nd3m_residual_kernel<<<cnt, 1024, 0, st>>>(ws, (double *)w.relres.p, img0);
        }
        nd3m_finish_kernel<<<cnt, 1024, 0, st>>>(ws, gv, (const double *)w.relres.p, (double *)w.out_img.p, img0);
        *launches += 3 + 2 * refine;
        img0 += cnt;
    }
    nd_reduce_kernel<<<(3 * ng + 255) / 256, 256, 0, st>>>((double *)w.out_img.p, (double *)w.relres.p, gp.O, 3 * ng, d_grad_out,
                                                           (double *)w.relres_max.p);
    *launches += 1;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return nd_fail(w, -2, std::string("nested-dissection kernel launch failed: ") + cudaGetErrorString(e));
    return 0;
}

NdWork *nd_work_create() { return new NdWork(); }
void nd_work_destroy(NdWork *w) { if (w) { w->release(); delete w; } }
const char *nd_work_error(const NdWork *w) { return w->err.c_str(); }
size_t nd_work_bytes_per_image(const NdWork *w) { return w->last_bytes_per_image; }
const double *nd_work_relres_max(const NdWork *w) { return (const double *)w->relres_max.p; }
int nd_run_gradient(NdWork *w, const NdProblem &gp, int sm_count, size_t smem_optin, cudaStream_t st, double *d_grad_out,
                    long long *launches)
{
    return gp.prec == 64 ? run_gradient_nd<double>(*w, gp, sm_count, smem_optin, st, d_grad_out, launches)
                         : run_gradient_nd<float>(*w, gp, sm_count, smem_optin, st, d_grad_out, launches);
}
int nd_run_gradient3_reg(NdWork *w, const Nd3Problem &gp, int sm_count, size_t smem_optin, cudaStream_t st, double *d_grad_out,
                         long long *launches)
{
    return gp.prec == 64 ? run_gradient3_nd_reg<double>(*w, gp, sm_count, smem_optin, st, d_grad_out, launches)
                         : run_gradient3_nd_reg<float>(*w, gp, sm_count, smem_optin, st, d_grad_out, launches);
}
int nd_run_gradient3(NdWork *w, const Nd3mProblem &gp, int sm_count, size_t smem_optin, cudaStream_t st, double *d_grad_out,
                     long long *launches)
{
    return gp.prec == 64 ? run_gradient3_nd_mult<double>(*w, gp, sm_count, smem_optin, st, d_grad_out, launches)
                         : run_gradient3_nd_mult<float>(*w, gp, sm_count, smem_optin, st, d_grad_out, launches);
}

}  // namespace bpltv
