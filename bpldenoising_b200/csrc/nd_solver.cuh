// nd_solver.cuh — multifrontal Cholesky on a nested-dissection ordering of a pixel grid (fp64, device code).
//
// The adjoint systems of /root/reference/src/TVLearningFunctionVec.jl:98-161, :192-254 are sparse SPD matrices
// whose unknowns sit on the pixels of an n×n image and couple only across ≤ W pixels.  nd_symbolic.h cuts the
// grid into an elimination tree of "fronts"; this header factorises and solves on it:
//
//   nd_dims_kernel     unknowns before each pixel of every front (a scan over the front's pixel list)
//   nd_scan_kernel     where every front's factor / update matrix / update vector lives in the pools
//   nd_factor_kernel   one tree level per launch, one CTA per (front, image):
//                        assemble  F = original entries of the pivot columns  (+)  children's update matrices
//                        factor    [F11 F21ᵀ; F21 F22] → L11 L11ᵀ, L21 = F21 L11⁻ᵀ, U = F22 − L21 L21ᵀ
//                                  blocked right-looking, NB = 16: the diagonal block by one warp in registers,
//                                  the panel by forward substitution with one thread per row, the rank-16 update
//                                  of the trailing matrix in 32×32 warp tiles (4×8 per thread) fed from shared memory
//                        U stays in the level's pool for the parent; L11 and L21 are kept
//   nd_fwd_kernel      L y = b   up the tree (children's update vectors are summed in a fixed order)
//   nd_bwd_kernel      Lᵀ x = y  down the tree
//   nd_lu_factor_*     the same for an unsymmetric matrix of the same sparsity: partial LU without pivoting, L and
//                      Uᵀ in the column layout of L, so that nd_fwd / nd_bwd solve with them unchanged
//
// Every sum has a fixed order: results are deterministic, independent of the grid shape of the launch.
// Fronts live in global memory (the working set of a level is L2-resident); a front of the top levels of a
// 256×256 image has ≈ 400-800 unknowns and does not fit in shared memory.
//
// The matrix comes in "pixel stencil" form: for pixel p and forward offset h (nd_symbolic.h) the dense block
//   ast[(p·NH + h)·MB² + β·MB + α] = A[(p + d_h, β), (p, α)]        (h = 0: the pixel's own symmetric block).
// Device code only; tests/emu compiles it with g++ on the thread emulation (-DBPLTV_EMU).
#pragma once
#ifndef BPLTV_EMU
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#endif
#include "nd_symbolic.h"

namespace bpltv {

constexpr int ND_NB = 16;
constexpr double ND_LTRIG = 8.0;    // a consistent SPD front has |l| ≤ √a_jj < 3: beyond this the pivot is raised and the block redone
constexpr double ND_LMAX = 1e6;     // a multiplier of the factor beyond this flags the factorisation as broken

struct NdDev {
    int n, N, W, nnb, nh, mb;
    int nfronts, nsteps;
    const NdFront *fronts;
    const int *pixlist, *nbr, *cmap, *step_start;
    // unknown numbering: off[q] = first unknown of pixel q in pixel order (N+1 per slot), nullptr: one per pixel
    const int *off; size_t off_stride;
    // per slot (stride 0: static, one unknown per pixel): prefix of the unknown counts along each front's pixel
    // list — front t uses posg[pix0_t + t + k], k = 0..npix_t
    int *posg; size_t posg_stride;
    // per slot (stride 0: static): 4 per front — offsets of L, of U and of the update vector (one spare)
    long long *foff; size_t foff_stride;
    long long *totals;                    // per slot: L doubles, max U doubles of a level, max UV doubles (one spare)
    double *L;  size_t L_stride;
    double *U[2];  size_t U_stride;       // by level parity
    double *UV[2]; size_t UV_stride;
    const double *ast; size_t ast_stride;
    int *info;                            // per slot: [0] pivots raised (floor / bound), [1] ≠ 0: the factorisation broke down
    double *scr = nullptr;                // per slot: scratch of the large-front variants (nd_level_scratch)
    size_t scr_stride = 0;
};

#ifdef BPLTV_EMU
#define ND_DYN_SMEM(name) double *name = emu::dyn_smem()
#else
#define ND_DYN_SMEM(name) extern __shared__ __align__(16) double name[]
#endif

static __device__ __forceinline__ int nd_count(const NdDev &nd, const int *off, int q) { return off ? off[q + 1] - off[q] : 1; }
static __host__ __device__ __forceinline__ long long nd_even(long long v) { return (v + 1) & ~1LL; }

// ---------------------------------------------------------------------------
// unknowns before each pixel of each front: one warp per front
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nd_dims_kernel(NdDev nd)
{
    const int slot = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int t = blockIdx.x * nw + warp;
    // (no early return: the emulation's warp barriers expect all 32 lanes of every warp)
    const bool live = t < nd.nfronts;
    const NdFront f = nd.fronts[live ? t : 0];
    const int npix = live ? f.npiv + f.nring : 0;
    const int *off = nd.off ? nd.off + nd.off_stride * slot : nullptr;
    int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + (live ? t : 0);
    int run = 0;
    for (int k0 = 0; k0 < npix; k0 += 32) {
        const int k = k0 + lane;
        const int c = k < npix ? nd_count(nd, off, nd.pixlist[f.pix0 + k]) : 0;
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (k < npix) pos[k] = run + incl - c;
        run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (live && lane == 0) pos[npix] = run;
}

// sizes of a front's blocks in the pools (doubles, even → every block starts 16-byte aligned): L, U, update vector
static __host__ __device__ __forceinline__ void nd_front_sizes(int nP, int nR, long long sz[3])
{
    sz[0] = nd_even((long long)(nP + nR) * nP);
    sz[1] = nd_even((long long)nR * nR);
    sz[2] = nd_even(nR);
}

// ---------------------------------------------------------------------------
// pool offsets: exclusive prefix over the fronts (sorted by level); U and UV restart at every level
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nd_scan_kernel(NdDev nd)
{
    __shared__ long long s_part[256][3];
    __shared__ long long s_base[64][2], s_lvl[64][2];
    const int slot = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const int *posg = nd.posg + nd.posg_stride * slot;
    long long *foff = nd.foff + nd.foff_stride * slot;
    const int per = (nd.nfronts + T - 1) / T;
    const int a = min(nd.nfronts, tid * per), b = min(nd.nfronts, a + per);
    long long acc[3] = {0, 0, 0};
    for (int t = a; t < b; ++t) {
        const NdFront f = nd.fronts[t];
        const int *pos = posg + f.pix0 + t;
        const int nP = pos[f.npiv], nR = pos[f.npiv + f.nring] - nP;
        long long sz[3];
        nd_front_sizes(nP, nR, sz);
        for (int k = 0; k < 3; ++k) acc[k] += sz[k];
    }
    for (int k = 0; k < 3; ++k) s_part[tid][k] = acc[k];
    __syncthreads();
    if (tid < 3) {      // serial scan of the 256 partial sums, one quantity per thread
        long long run = 0;
        for (int i = 0; i < T; ++i) { const long long v = s_part[i][tid]; s_part[i][tid] = run; run += v; }
        if (tid == 0) nd.totals[4 * slot] = run;
        else s_base[nd.nsteps][tid - 1] = run;          // grand totals of U, UV = prefix at the end of the last level
    }
    __syncthreads();
    for (int k = 0; k < 3; ++k) acc[k] = s_part[tid][k];
    for (int t = a; t < b; ++t) {
        const NdFront f = nd.fronts[t];
        const int *pos = posg + f.pix0 + t;
        const int nP = pos[f.npiv], nR = pos[f.npiv + f.nring] - nP;
        long long sz[3];
        nd_front_sizes(nP, nR, sz);
        for (int k = 0; k < 3; ++k) { foff[4 * (size_t)t + k] = acc[k]; acc[k] += sz[k]; }
    }
    __syncthreads();
    if (tid < nd.nsteps) {
        const int t = nd.step_start[tid];      // every level has at least one front
        s_base[tid][0] = foff[4 * (size_t)t + 1];
        s_base[tid][1] = foff[4 * (size_t)t + 2];
    }
    __syncthreads();
    if (tid < nd.nsteps) {
        s_lvl[tid][0] = s_base[tid + 1][0] - s_base[tid][0];
        s_lvl[tid][1] = s_base[tid + 1][1] - s_base[tid][1];
    }
    for (int t = tid; t < nd.nfronts; t += T) {
        const int s = nd.nsteps - 1 - nd.fronts[t].depth;
        foff[4 * (size_t)t + 1] -= s_base[s][0];
        foff[4 * (size_t)t + 2] -= s_base[s][1];
    }
    __syncthreads();
    if (tid == 0) {
        long long m0 = 0, m1 = 0;
        for (int s = 0; s < nd.nsteps; ++s) { m0 = max(m0, s_lvl[s][0]); m1 = max(m1, s_lvl[s][1]); }
        nd.totals[4 * slot + 1] = m0;
        nd.totals[4 * slot + 2] = m1;
        nd.totals[4 * slot + 3] = 0;
    }
}

// ---------------------------------------------------------------------------
// dense building blocks
// ---------------------------------------------------------------------------
// One warp: S0 (NB×NB row-major, lower, identity padded beyond nb) → L11 in S (row-major, lower) and the reciprocals
// of its diagonal in dinv.  Rows across lanes, columns through shuffles.
// Pivot rule (guard > 0, the multiplier form).  The matrix is SPD with eigenvalues down to eps(): redundant
// constraints of flat regions give pivots that are pure rounding noise.  (a) d ≤ guard → d = guard: the constraint is
// implied by those already eliminated, its column is noise as well, and the floor keeps 1/√d from amplifying it.
// (b) d < a²/16 for the largest entry a of its column inside the block: impossible for a positive semidefinite
// matrix whose diagonal is ≤ 8 (a² ≤ d·a_jj), so it only triggers when accumulated rounding made the Schur
// complement indefinite (barely sloped regions, |∇u| ≈ 1e-12, where compliances of 1e-11 sit next to eps()):
// raising d to a²/16 bounds the multipliers by 4 instead of letting 1/√guard blow the factorisation up.  Rows below
// the block are covered after the fact: nd_factor_kernel repeats the block step with a raised floor dfl[c] when a
// multiplier of the panel exceeds ND_LTRIG.  All are counted in `guarded`; iterative refinement against the true
// residual follows.
// guard == 0 (node form, well conditioned): a non-positive pivot sets `bad`.
// No explicit inverse of L11 anywhere: with pivots from 1 down to √guard the block has a condition number of 1e6 and
// multiplying by its inverse loses what substitution keeps (measured: Schur complements of barely sloped regions
// turned indefinite).
template <int NB>
static __device__ void nd_diag_block(const double *S0, double *S, double *dinv, const double *dfl, int nb, double guard, int lane,
                                     int &guarded, int &bad)
{
    double row[NB];
    const int lr = lane < NB ? lane : NB - 1;
#pragma unroll
    for (int c = 0; c < NB; ++c) row[c] = S0[lr * NB + c];
    guarded = 0;
    double dinv_own = 1.0;
#pragma unroll
    for (int c = 0; c < NB; ++c) {
        double d = __shfl_sync(0xffffffffu, row[c], c);
        if (guard > 0.0) {
            double am = (lane > c && lane < NB) ? fabs(row[c]) : 0.0;
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) am = fmax(am, __shfl_xor_sync(0xffffffffu, am, o));
            am = __shfl_sync(0xffffffffu, am, 0);           // lanes 0-15 hold the maximum of the block's column
            const double floor_ = fmax(dfl[c], am * am * 0.0625);
            if (!(d >= floor_)) { d = floor_; if (lane == 0 && c < nb) ++guarded; }
        } else if (!(d > 0.0)) {
            if (lane == 0 && c < nb) bad = 1;
            d = 1.0;
        }
        const double inv = rsqrt(d);
        const double l = row[c] * inv;
        if (lane == c) { row[c] = d * inv; dinv_own = inv; }
        else if (lane > c) row[c] = l;
#pragma unroll
        for (int c2 = c + 1; c2 < NB; ++c2) {
            const double lc2 = __shfl_sync(0xffffffffu, l, c2);
            if (lane >= c2) row[c2] = fma(-l, lc2, row[c2]);
        }
    }
    if (lane < NB) {
#pragma unroll
        for (int c = 0; c < NB; ++c) S[lane * NB + c] = (c <= lane) ? row[c] : 0.0;
        dinv[lane] = dinv_own;
    }
    __syncwarp();
}

// One warp: v ← L11⁻¹ v (forward) or L11⁻ᵀ v (backward) by substitution; L11 row-major NB×NB in shared memory
// (identity beyond nb), v[0..NB) in shared memory.  Lane r holds entry r.
static __device__ __forceinline__ void nd_block_subst(const double *S, double *v, bool transposed, int lane)
{
    constexpr int NB = ND_NB;
    const int lr = lane < NB ? lane : NB - 1;
    double x = v[lr];
    const double dinv = 1.0 / S[lr * NB + lr];
    if (!transposed) {
#pragma unroll
        for (int c = 0; c < NB; ++c) {
            const double yc = __shfl_sync(0xffffffffu, x * dinv, c);      // lane c: final value of entry c
            if (lr == c) x = yc;
            else if (lr > c) x = fma(-S[lr * NB + c], yc, x);
        }
    } else {
#pragma unroll
        for (int c = NB - 1; c >= 0; --c) {
            const double yc = __shfl_sync(0xffffffffu, x * dinv, c);
            if (lr == c) x = yc;
            else if (lr < c) x = fma(-S[c * NB + lr], yc, x);
        }
    }
    if (lane < NB) v[lane] = x;
    __syncwarp();
}

// column c of the front: rows are addressed with the FRONT index r ≥ c
static __device__ __forceinline__ double *nd_col(double *L, double *U, int nP, int nF, int nR, int c)
{
    return c < nP ? L + (size_t)c * nF : U + (size_t)(c - nP) * nR - nP;
}

static __host__ __device__ __forceinline__ int nd_panel_pitch(int nFmax) { return (nFmax + 31) & ~31; }
// dynamic shared memory of nd_factor_kernel (bytes): S0, S, reciprocal diagonal, column floors, panel P (NB × pitch;
// not on the large-front variants, which keep it in global memory), the child map (ints).  lu: nd_lu_factor_body, whose
// two panels (L21 and U12ᵀ) take twice the room.
static inline size_t nd_factor_smem(int nFmax, int nRchild_max, int nb = ND_NB, bool panel_global = false, bool lu = false)
{
    return (size_t)(2 * nb * nb + 2 * nb + (panel_global ? 0 : (lu ? 2 : 1) * nb * nd_panel_pitch(nFmax))) * sizeof(double) +
           (((size_t)nRchild_max * sizeof(int) + 15) & ~(size_t)15);
}

// ---------------------------------------------------------------------------
// assemble + partial Cholesky of the fronts of one level.  grid (fronts of the level, slots)
// ---------------------------------------------------------------------------
// CL: the front is shared by the CTAs of a thread-block cluster (the top levels of the tree, where a level has fewer
// fronts than the GPU has SMs): assembly and write-back are dealt over all threads of the cluster, the diagonal block and
// the panel are formed redundantly by every CTA in its own shared memory (same operations in the same order: the same
// pivots and the same bits), the tiles of the trailing update are dealt over all warps of the cluster, and one cluster
// barrier per phase / block step publishes them through global memory.  Results do not depend on the cluster size.
// NB: columns per block step.  16 everywhere, except for fronts whose 16-column panel exceeds shared memory (the
// sum-of-regularisers multiplier form of a large or mostly flat image: > ≈ 1700 unknowns), which take 8 — twice the steps
// for half the panel.  (The factor does not depend on NB beyond the order of the updates; the solves use blocks of 16.)
// PG (large fronts, whose panel does not fit in shared memory even at 8 columns): the panel lives in global memory, in
// the CTA's own slice of nd.scr (NB × pitch doubles at blockIdx.x; a cluster's CTAs each form their own copy, as in
// shared memory).  Nothing else changes: the same operations in the same order, the same bits.
template <bool CL, int NB, bool PG = false>
static __device__ __forceinline__ void nd_factor_body(const NdDev &nd, int t0, int par, double guard, int nFmax)
{
    ND_DYN_SMEM(sm);
    const int PR = nd_panel_pitch(nFmax);
    double *S0 = sm, *S = sm + NB * NB, *dinv = sm + 2 * NB * NB, *dfl = dinv + NB;
    double *P = PG ? nd.scr + nd.scr_stride * blockIdx.y + (size_t)blockIdx.x * NB * PR : dfl + NB;
    __shared__ int s_cbad;
    __shared__ unsigned long long s_amax2;
    int *umap = reinterpret_cast<int *>(PG ? dfl + NB : P + (size_t)NB * PR);
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
    int crank = 0, csize = 1;
    if (CL) {
        cooperative_groups::cluster_group cluster = cooperative_groups::this_cluster();
        crank = (int)cluster.block_rank(); csize = (int)cluster.num_blocks();
    }
    auto csync = [&]() { if (CL) cooperative_groups::this_cluster().sync(); else __syncthreads(); };
    const int gtid = crank * T + tid, GT = csize * T;       // thread index / count over the cluster
    const int t = t0 + blockIdx.x / csize, slot = blockIdx.y;
    const NdFront f = nd.fronts[t];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + t;
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int nP = pos[f.npiv], nF = pos[f.npiv + f.nring], nR = nF - nP;
    double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
    double *U = nd.U[par] + nd.U_stride * slot + foff[4 * (size_t)t + 1];
    const double *ast = nd.ast + nd.ast_stride * slot;
    const int MB = nd.mb, MB2 = MB * MB;

    // ---- zero
    for (size_t k = gtid; k < (size_t)nF * nP; k += GT) L[k] = 0.0;
    for (size_t k = gtid; k < (size_t)nR * nR; k += GT) U[k] = 0.0;
    csync();
    // ---- original entries of the pivot columns (each pixel pair once: by the earlier pixel of the front)
    {
        const int ne = nd.nnb + 1;
        for (int idx = gtid; idx < f.npiv * ne; idx += GT) {
            const int kp = idx / ne, e = idx - kp * ne;
            const int p = nd.pixlist[f.pix0 + kp];
            const int a0 = pos[kp], mp = pos[kp + 1] - a0;
            if (e == 0) {
                const double *blk = ast + (size_t)p * nd.nh * MB2;
                for (int al = 0; al < mp; ++al)
                    for (int be = al; be < mp; ++be) L[(size_t)(a0 + al) * nF + a0 + be] = blk[be * MB + al];
            } else {
                const int kq = nd.nbr[f.nbr0 + kp * nd.nnb + (e - 1)];
                if (kq <= kp) continue;
                const int q = nd.pixlist[f.pix0 + kq];
                const int b0 = pos[kq], mq = pos[kq + 1] - b0;
                const int h = 1 + ((e - 1) >> 1);
                const bool fwd = ((e - 1) & 1) == 0;       // q = p + d_h, else p = q + d_h
                const double *blk = ast + ((size_t)(fwd ? p : q) * nd.nh + h) * MB2;
                for (int al = 0; al < mp; ++al)
                    for (int be = 0; be < mq; ++be)
                        L[(size_t)(a0 + al) * nF + b0 + be] = fwd ? blk[be * MB + al] : blk[al * MB + be];
            }
        }
    }
    csync();
    // ---- extend-add: the children's update matrices, one child after the other (fixed order)
    for (int ci = 0; ci < 2; ++ci) {
        const int c = ci == 0 ? f.child0 : f.child1;
        if (c < 0) continue;
        const NdFront cf = nd.fronts[c];
        const int *cpos = nd.posg + nd.posg_stride * slot + cf.pix0 + c + cf.npiv;
        const int cnP = cpos[0], cnR = cpos[cf.nring] - cnP;
        for (int k = tid; k < cf.nring; k += T) {
            const int r0 = cpos[k] - cnP, m = cpos[k + 1] - cpos[k];
            const int R0 = pos[nd.cmap[cf.cmap0 + k]];
            for (int al = 0; al < m; ++al) umap[r0 + al] = R0 + al;
        }
        __syncthreads();
        const double *cU = nd.U[par ^ 1] + nd.U_stride * slot + foff[4 * (size_t)c + 1];
        const size_t tot = (size_t)cnR * cnR;
        // four entries per thread and pass, loads before stores (distinct targets: the map is injective)
        for (size_t idx0 = gtid; idx0 < tot; idx0 += (size_t)4 * GT) {
            double *dst[4];
            double v[4], a[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const size_t idx = idx0 + (size_t)k * GT;
                dst[k] = nullptr;
                if (idx < tot) {
                    const int r = (int)(idx % cnR), cc = (int)(idx / cnR);
                    if (r >= cc) {
                        int R = umap[r], C = umap[cc];
                        if (R < C) { const int s = R; R = C; C = s; }
                        dst[k] = nd_col(L, U, nP, nF, nR, C) + R;
                        a[k] = cU[idx];
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = dst[k] ? *dst[k] : 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (dst[k]) *dst[k] = v[k] + a[k];
        }
        csync();
    }
    // ---- blocked partial Cholesky of the first nP columns
    int guarded = 0, bad = 0;
    for (int kb = 0; kb < nP; kb += NB) {
        const int nb = min(NB, nP - kb), k1 = kb + nb, ntr = nF - k1;
        for (int idx = tid; idx < NB * NB; idx += T) {
            const int r = idx / NB, c = idx - r * NB;
            S0[idx] = (r < nb && c <= r) ? L[(size_t)(kb + c) * nF + kb + r] : (r == c ? 1.0 : 0.0);
        }
        if (tid < NB) dfl[tid] = guard;
        if (tid == 0) { s_cbad = NB; s_amax2 = 0ULL; }
        const int ntr32 = (ntr + 31) & ~31;
        int blk_guarded = 0;
        for (int attempt = 0;; ++attempt) {
            __syncthreads();
            if (warp == 0) nd_diag_block<NB>(S0, S, dinv, dfl, nb, guard, lane, blk_guarded, bad);
            __syncthreads();
            // panel: L21 = A21 · L11⁻ᵀ by forward substitution, one thread per row, into P; rows up to the next
            // multiple of 32 are zero
            for (int rr = tid; rr < ntr32; rr += T) {
                double x[NB];
                if (rr < ntr) {
#pragma unroll
                    for (int c = 0; c < NB; ++c) x[c] = c < nb ? L[(size_t)(kb + c) * nF + k1 + rr] : 0.0;
                    int cb = NB;
#pragma unroll
                    for (int c = 0; c < NB; ++c) {
                        double s0 = x[c], s1 = 0.0;
#pragma unroll
                        for (int k = 0; k < c; k += 2) {
                            s0 = fma(-S[c * NB + k], x[k], s0);
                            if (k + 1 < c) s1 = fma(-S[c * NB + k + 1], x[k + 1], s1);
                        }
                        x[c] = (s0 + s1) * dinv[c];
                        P[c * PR + rr] = c < nb ? x[c] : 0.0;
                        if (cb == NB && c < nb && !(fabs(x[c]) <= ND_LTRIG)) cb = c;
                    }
                    if (cb < NB && guard > 0.0) atomicMin(&s_cbad, cb);
                } else {
#pragma unroll
                    for (int c = 0; c < NB; ++c) P[c * PR + rr] = 0.0;
                }
            }
            __syncthreads();
            const int cb = s_cbad;
            if (cb >= NB) break;
            if (attempt >= 4 * NB) { bad = 1; break; }      // (NaN input: nothing to tame)
            // a multiplier beyond any consistent SPD front in column cb: raise that pivot so that the largest becomes 4
            // (a = l·√d recovers the column entry), and redo the block step
            const double sd = S[cb * NB + cb];
            for (int rr = tid; rr < ntr; rr += T) {
                const double a = fabs(P[cb * PR + rr]) * sd;
                if (a == a && a < 1e150) atomicMax(&s_amax2, (unsigned long long)__double_as_longlong(a * a));
                else atomicMax(&s_amax2, (unsigned long long)__double_as_longlong(1e300));
            }
            __syncthreads();
            if (tid == 0) {
                dfl[cb] = fmax(2.0 * dfl[cb], __longlong_as_double((long long)s_amax2) * 0.0625);
                s_cbad = NB; s_amax2 = 0ULL;
            }
        }
        guarded += blk_guarded;
        if (CL) csync();        // every CTA has read the block's columns (its own S0 and panel) before they are overwritten
        if (crank == 0)
            for (int idx = tid; idx < NB * NB; idx += T) {
                const int r = idx / NB, c = idx - r * NB;
                if (r < nb && c <= r) L[(size_t)(kb + c) * nF + kb + r] = S[idx];
            }
        for (int idx = gtid; idx < ntr * nb; idx += GT) {
            const int c = idx / ntr, rr = idx - c * ntr;
            const double v = P[c * PR + rr];
            L[(size_t)(kb + c) * nF + k1 + rr] = v;
            if (!(fabs(v) <= ND_LMAX)) bad = 1;      // NaN, or a multiplier no raised pivot could tame
        }
        // trailing update F22 -= P Pᵀ (lower triangle) in 32×32 warp tiles, 4 rows × 8 columns per thread
        const int nt = ntr32 >> 5, ntiles = nt * (nt + 1) / 2;
        const int li = lane & 7, lj = lane >> 3;
        for (int wt = crank * nwarps + warp; wt < ntiles; wt += csize * nwarps) {
            // wt = ti(ti+1)/2 + tj, tj ≤ ti
            int ti = (int)((sqrt(8.0 * wt + 1.0) - 1.0) * 0.5);
            while ((ti + 1) * (ti + 2) / 2 <= wt) ++ti;
            while (ti * (ti + 1) / 2 > wt) --ti;
            const int tj = wt - ti * (ti + 1) / 2;
            const int i0 = 32 * ti + 4 * li, j0 = 32 * tj + 8 * lj;
            if (j0 > i0 + 3 || j0 >= ntr || i0 >= ntr) continue;      // nothing of this thread's patch in the lower triangle
            // The tile's old entries are the initial values of the accumulators: their loads are issued before the
            // rank-16 loop and fly under it (an update after the loop — load, subtract, store per element, or in batches
            // — exposes L2 round trips the block step's chain has to wait for: ncu, 20 % of the kernel's stall samples).
            double acc[4][8];
#pragma unroll
            for (int y = 0; y < 8; ++y) {
                const int cc = j0 + y;
                const double *col = nd_col(L, U, nP, nF, nR, k1 + (cc < ntr ? cc : 0)) + k1;
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const int r = i0 + x;
                    acc[x][y] = (cc < ntr && r >= cc && r < ntr) ? col[r] : 0.0;
                }
            }
#pragma unroll 4
            for (int c = 0; c < NB; ++c) {
                const double *pc = P + c * PR;
                const double2 a0 = *reinterpret_cast<const double2 *>(pc + i0);
                const double2 a1 = *reinterpret_cast<const double2 *>(pc + i0 + 2);
                const double2 b0 = *reinterpret_cast<const double2 *>(pc + j0);
                const double2 b1 = *reinterpret_cast<const double2 *>(pc + j0 + 2);
                const double2 b2 = *reinterpret_cast<const double2 *>(pc + j0 + 4);
                const double2 b3 = *reinterpret_cast<const double2 *>(pc + j0 + 6);
                const double pi[4] = {-a0.x, -a0.y, -a1.x, -a1.y};
                const double pj[8] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, b3.x, b3.y};
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 8; ++y) acc[x][y] = fma(pi[x], pj[y], acc[x][y]);
            }
#pragma unroll
            for (int y = 0; y < 8; ++y) {
                const int cc = j0 + y;
                double *col = nd_col(L, U, nP, nF, nR, k1 + (cc < ntr ? cc : 0)) + k1;
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const int r = i0 + x;
                    if (cc < ntr && r >= cc && r < ntr) col[r] = acc[x][y];
                }
            }
        }
        csync();
    }
    if (guarded && crank == 0) atomicAdd(nd.info + 4 * slot, guarded);
    if (bad) atomicAdd(nd.info + 4 * slot + 1, 1);
}

__global__ void __launch_bounds__(512) nd_factor_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<false, ND_NB>(nd, t0, par, guard, nFmax); }
// grid (fronts of the level × cluster size, slots), launched with the cluster dimension
__global__ void __launch_bounds__(512) nd_factor_cluster_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<true, ND_NB>(nd, t0, par, guard, nFmax); }
// the same with 8-column block steps (fronts whose 16-column panel does not fit in shared memory)
__global__ void __launch_bounds__(512) nd_factor8_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<false, 8>(nd, t0, par, guard, nFmax); }
__global__ void __launch_bounds__(512) nd_factor8_cluster_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<true, 8>(nd, t0, par, guard, nFmax); }
// large fronts: the panel in global memory (nd.scr).  16-column block steps for fronts beyond the 8-column panel, and for
// levels sent here by BPLTV_ND_LARGE_KB, the block width their shared-memory kernel would have used
__global__ void __launch_bounds__(512) nd_factor_large_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<false, ND_NB, true>(nd, t0, par, guard, nFmax); }
__global__ void __launch_bounds__(512) nd_factor_large_cluster_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<true, ND_NB, true>(nd, t0, par, guard, nFmax); }
__global__ void __launch_bounds__(512) nd_factor8_large_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<false, 8, true>(nd, t0, par, guard, nFmax); }
__global__ void __launch_bounds__(512) nd_factor8_large_cluster_kernel(NdDev nd, int t0, int par, double guard, int nFmax) { nd_factor_body<true, 8, true>(nd, t0, par, guard, nFmax); }

// ===========================================================================
// LU form: the same fronts for an UNSYMMETRIC matrix with the sparsity of the symmetric one (the row-scaled patch
// sum-of-regularisers system, nd_sumregs.cuh).  No pivoting: every term of that matrix is a positive diagonal times a
// PSD matrix; with equal maps it is D·SPD, and a symmetric reordering P(D·S)Pᵀ keeps that form, so its leading minors
// stay positive.  A zero or non-finite pivot sets the breakdown flag; the caller's backward-error test does the rest.
//
// Storage: F = L U with L unit lower.  L (nd.L) holds L's first nP columns, its unit diagonal written out; Ut holds U's
// first nP ROWS, transposed, in the same nF × nP column layout (column c = row c of U, entries r ≥ c, diagonal
// included); the update matrix is the whole nR × nR Schur complement.  A slot's factor pool is twice the Cholesky's:
// L in its first half, Ut at the same offsets in its second (nd.L_stride / 2 further).  The forward sweep of nd_fwd_body
// on L solves L y = b (its pivots are exactly 1), the backward sweep of nd_bwd_body on Ut solves U x = y: the solve
// kernels are the Cholesky's, launched with nd.L moved to the second half for the backward sweep.
// The ast of this form has 2·nh − 1 blocks per pixel: [0] A[p, p] (the whole block), [h] A[p + d_h, p] as in the
// symmetric form, [nh − 1 + h] A[p, p + d_h].
// ===========================================================================
constexpr double ND_DMAX = 1.7976931348623157e308;

// entry (R, C) of the front while it is factorised: pivot columns on or below the diagonal in L, pivot rows right of
// the diagonal in Ut, the rest in the update matrix
static __device__ __forceinline__ double *nd_lu_at(double *L, double *Ut, double *U, int nP, int nF, int nR, int R, int C)
{
    if (C < nP && R >= C) return L + (size_t)C * nF + R;
    if (R < nP) return Ut + (size_t)R * nF + C;
    return U + (size_t)(C - nP) * nR + (R - nP);
}

// One warp: S0 (NB×NB row-major, identity padded beyond nb) → its LU without pivoting in S (row-major: the multipliers
// of L below the diagonal, U on and above it) and the reciprocals of U's diagonal in dinv.  Rows across lanes, columns
// through shuffles.  A zero or non-finite pivot sets `bad` and is replaced by 1, so that the step completes.
template <int NB>
static __device__ void nd_lu_diag_block(const double *S0, double *S, double *dinv, int nb, int lane, int &bad)
{
    double row[NB];
    const int lr = lane < NB ? lane : NB - 1;
#pragma unroll
    for (int c = 0; c < NB; ++c) row[c] = S0[lr * NB + c];
    double dinv_own = 1.0;
#pragma unroll
    for (int c = 0; c < NB; ++c) {
        double d = __shfl_sync(0xffffffffu, row[c], c);
        if (!(fabs(d) > 0.0 && fabs(d) <= ND_DMAX)) {
            if (lane == 0 && c < nb) bad = 1;
            d = 1.0;
        }
        const double inv = 1.0 / d;
        const double l = row[c] * inv;
#pragma unroll
        for (int c2 = c + 1; c2 < NB; ++c2) {
            const double uc2 = __shfl_sync(0xffffffffu, row[c2], c);
            if (lane > c) row[c2] = fma(-l, uc2, row[c2]);
        }
        if (lane == c) { row[c] = d; dinv_own = inv; }
        else if (lane > c) row[c] = l;
    }
    if (lane < NB) {
#pragma unroll
        for (int c = 0; c < NB; ++c) S[lane * NB + c] = row[c];
        dinv[lane] = dinv_own;
    }
    __syncwarp();
}

// assemble + partial LU of the fronts of one level; CL, NB and PG as nd_factor_body (a cluster's CTAs form the diagonal
// block and both panels redundantly and share the tiles of the trailing update: the same bits for every cluster size;
// the panels in global memory give the bits of the shared-memory kernel at the same NB).  Blocked right-looking, per step:
// the diagonal block by one warp (nd_lu_diag_block), L21 = F21 U11⁻¹ and U12ᵀ = (L11⁻¹ F12)ᵀ by substitution with one
// thread per row of both panels, F22 −= L21 U12 over ALL 32×32 tiles of the trailing matrix.
template <bool CL, int NB, bool PG = false>
static __device__ __forceinline__ void nd_lu_factor_body(const NdDev &nd, int t0, int par, int nFmax)
{
    ND_DYN_SMEM(sm);
    const int PR = nd_panel_pitch(nFmax);
    double *S0 = sm, *S = sm + NB * NB, *dinv = sm + 2 * NB * NB;
    double *PL = PG ? nd.scr + nd.scr_stride * blockIdx.y + (size_t)blockIdx.x * 2 * NB * PR : dinv + 2 * NB;
    double *PU = PL + (size_t)NB * PR;
    int *umap = reinterpret_cast<int *>(PG ? dinv + 2 * NB : PU + (size_t)NB * PR);
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
    int crank = 0, csize = 1;
    if (CL) {
        cooperative_groups::cluster_group cluster = cooperative_groups::this_cluster();
        crank = (int)cluster.block_rank(); csize = (int)cluster.num_blocks();
    }
    auto csync = [&]() { if (CL) cooperative_groups::this_cluster().sync(); else __syncthreads(); };
    const int gtid = crank * T + tid, GT = csize * T;
    const int t = t0 + blockIdx.x / csize, slot = blockIdx.y;
    const NdFront f = nd.fronts[t];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + t;
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int nP = pos[f.npiv], nF = pos[f.npiv + f.nring], nR = nF - nP;
    double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
    double *Ut = L + nd.L_stride / 2;
    double *U = nd.U[par] + nd.U_stride * slot + foff[4 * (size_t)t + 1];
    const double *ast = nd.ast + nd.ast_stride * slot;
    const int MB = nd.mb, MB2 = MB * MB, NH2 = 2 * nd.nh - 1;

    // ---- zero
    for (size_t k = gtid; k < (size_t)nF * nP; k += GT) { L[k] = 0.0; Ut[k] = 0.0; }
    for (size_t k = gtid; k < (size_t)nR * nR; k += GT) U[k] = 0.0;
    csync();
    // ---- original entries of the pivot rows and columns (each pixel pair once: by the earlier pixel of the front)
    {
        const int ne = nd.nnb + 1;
        for (int idx = gtid; idx < f.npiv * ne; idx += GT) {
            const int kp = idx / ne, e = idx - kp * ne;
            const int p = nd.pixlist[f.pix0 + kp];
            const int a0 = pos[kp], mp = pos[kp + 1] - a0;
            if (e == 0) {
                const double *blk = ast + (size_t)p * NH2 * MB2;       // blk[be·MB + al] = F(a0 + be, a0 + al)
                for (int al = 0; al < mp; ++al)
                    for (int be = 0; be < mp; ++be) {
                        if (be >= al) L[(size_t)(a0 + al) * nF + a0 + be] = blk[be * MB + al];
                        else Ut[(size_t)(a0 + be) * nF + a0 + al] = blk[be * MB + al];
                    }
            } else {
                const int kq = nd.nbr[f.nbr0 + kp * nd.nnb + (e - 1)];
                if (kq <= kp) continue;
                const int q = nd.pixlist[f.pix0 + kq];
                const int b0 = pos[kq], mq = pos[kq + 1] - b0;
                const int h = 1 + ((e - 1) >> 1);
                const bool fwd = ((e - 1) & 1) == 0;       // q = p + d_h, else p = q + d_h
                const double *lo = ast + ((size_t)(fwd ? p : q) * NH2 + h) * MB2;              // A[· + d_h, ·]
                const double *up = ast + ((size_t)(fwd ? p : q) * NH2 + nd.nh - 1 + h) * MB2;  // A[·, · + d_h]
                const double *bqp = fwd ? lo : up, *bpq = fwd ? up : lo;   // A[q, p], A[p, q]: [row unknown · MB + column unknown]
                for (int al = 0; al < mp; ++al)
                    for (int be = 0; be < mq; ++be) {
                        L[(size_t)(a0 + al) * nF + b0 + be] = bqp[be * MB + al];
                        Ut[(size_t)(a0 + al) * nF + b0 + be] = bpq[al * MB + be];
                    }
            }
        }
    }
    csync();
    // ---- extend-add: the children's whole update matrices, one child after the other (fixed order)
    for (int ci = 0; ci < 2; ++ci) {
        const int c = ci == 0 ? f.child0 : f.child1;
        if (c < 0) continue;
        const NdFront cf = nd.fronts[c];
        const int *cpos = nd.posg + nd.posg_stride * slot + cf.pix0 + c + cf.npiv;
        const int cnP = cpos[0], cnR = cpos[cf.nring] - cnP;
        for (int k = tid; k < cf.nring; k += T) {
            const int r0 = cpos[k] - cnP, m = cpos[k + 1] - cpos[k];
            const int R0 = pos[nd.cmap[cf.cmap0 + k]];
            for (int al = 0; al < m; ++al) umap[r0 + al] = R0 + al;
        }
        __syncthreads();
        const double *cU = nd.U[par ^ 1] + nd.U_stride * slot + foff[4 * (size_t)c + 1];
        const size_t tot = (size_t)cnR * cnR;
        for (size_t idx0 = gtid; idx0 < tot; idx0 += (size_t)4 * GT) {
            double *dst[4];
            double v[4], a[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const size_t idx = idx0 + (size_t)k * GT;
                dst[k] = nullptr;
                if (idx < tot) {
                    const int r = (int)(idx % cnR), cc = (int)(idx / cnR);
                    dst[k] = nd_lu_at(L, Ut, U, nP, nF, nR, umap[r], umap[cc]);
                    a[k] = cU[idx];
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = dst[k] ? *dst[k] : 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (dst[k]) *dst[k] = v[k] + a[k];
        }
        csync();
    }
    // ---- blocked partial LU of the first nP rows and columns
    int bad = 0;
    for (int kb = 0; kb < nP; kb += NB) {
        const int nb = min(NB, nP - kb), k1 = kb + nb, ntr = nF - k1;
        for (int idx = tid; idx < NB * NB; idx += T) {
            const int r = idx / NB, c = idx - r * NB;
            S0[idx] = (r < nb && c < nb) ? *nd_lu_at(L, Ut, U, nP, nF, nR, kb + r, kb + c) : (r == c ? 1.0 : 0.0);
        }
        __syncthreads();
        if (warp == 0) nd_lu_diag_block<NB>(S0, S, dinv, nb, lane, bad);
        __syncthreads();
        // panels, one thread per trailing index rr: row k1+rr of L21 = F21 U11⁻¹ into PL, column k1+rr of U12 = L11⁻¹ F12
        // into PU; entries up to the next multiple of 32 are zero
        const int ntr32 = (ntr + 31) & ~31;
        for (int rr = tid; rr < ntr32; rr += T) {
            double x[NB];
            if (rr < ntr) {
#pragma unroll
                for (int c = 0; c < NB; ++c) x[c] = c < nb ? L[(size_t)(kb + c) * nF + k1 + rr] : 0.0;
#pragma unroll
                for (int c = 0; c < NB; ++c) {
                    double s0 = x[c], s1 = 0.0;
#pragma unroll
                    for (int k = 0; k < c; k += 2) {
                        s0 = fma(-S[k * NB + c], x[k], s0);
                        if (k + 1 < c) s1 = fma(-S[(k + 1) * NB + c], x[k + 1], s1);
                    }
                    x[c] = (s0 + s1) * dinv[c];
                    PL[c * PR + rr] = c < nb ? x[c] : 0.0;
                }
#pragma unroll
                for (int c = 0; c < NB; ++c) x[c] = c < nb ? Ut[(size_t)(kb + c) * nF + k1 + rr] : 0.0;
#pragma unroll
                for (int c = 0; c < NB; ++c) {
                    double s0 = x[c], s1 = 0.0;
#pragma unroll
                    for (int k = 0; k < c; k += 2) {
                        s0 = fma(-S[c * NB + k], x[k], s0);
                        if (k + 1 < c) s1 = fma(-S[c * NB + k + 1], x[k + 1], s1);
                    }
                    x[c] = s0 + s1;
                    PU[c * PR + rr] = c < nb ? x[c] : 0.0;
                }
            } else {
#pragma unroll
                for (int c = 0; c < NB; ++c) { PL[c * PR + rr] = 0.0; PU[c * PR + rr] = 0.0; }
            }
        }
        __syncthreads();
        if (CL) csync();        // every CTA has read the block's rows and columns before they are overwritten
        if (crank == 0)
            for (int idx = tid; idx < NB * NB; idx += T) {
                const int r = idx / NB, c = idx - r * NB;
                if (r < nb && c < nb) {
                    if (c < r) L[(size_t)(kb + c) * nF + kb + r] = S[idx];
                    else {
                        Ut[(size_t)(kb + r) * nF + kb + c] = S[idx];
                        if (c == r) L[(size_t)(kb + c) * nF + kb + r] = 1.0;
                    }
                }
            }
        for (int idx = gtid; idx < ntr * nb; idx += GT) {
            const int c = idx / ntr, rr = idx - c * ntr;
            const double vl = PL[c * PR + rr], vu = PU[c * PR + rr];
            L[(size_t)(kb + c) * nF + k1 + rr] = vl;
            Ut[(size_t)(kb + c) * nF + k1 + rr] = vu;
            if (!(fabs(vl) <= ND_DMAX) || !(fabs(vu) <= ND_DMAX)) bad = 1;
        }
        // trailing update F22 −= PL PUᵀ over all 32×32 warp tiles, 4 rows × 8 columns per thread
        const int nt = ntr32 >> 5, ntiles = nt * nt;
        const int li = lane & 7, lj = lane >> 3;
        for (int wt = crank * nwarps + warp; wt < ntiles; wt += csize * nwarps) {
            const int ti = wt / nt, tj = wt - ti * nt;
            const int i0 = 32 * ti + 4 * li, j0 = 32 * tj + 8 * lj;
            if (i0 >= ntr || j0 >= ntr) continue;
            double acc[4][8];
#pragma unroll
            for (int y = 0; y < 8; ++y)
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const int r = i0 + x, cc = j0 + y;
                    acc[x][y] = (r < ntr && cc < ntr) ? *nd_lu_at(L, Ut, U, nP, nF, nR, k1 + r, k1 + cc) : 0.0;
                }
#pragma unroll 4
            for (int c = 0; c < NB; ++c) {
                const double *pl = PL + c * PR, *pu = PU + c * PR;
                const double2 a0 = *reinterpret_cast<const double2 *>(pl + i0);
                const double2 a1 = *reinterpret_cast<const double2 *>(pl + i0 + 2);
                const double2 b0 = *reinterpret_cast<const double2 *>(pu + j0);
                const double2 b1 = *reinterpret_cast<const double2 *>(pu + j0 + 2);
                const double2 b2 = *reinterpret_cast<const double2 *>(pu + j0 + 4);
                const double2 b3 = *reinterpret_cast<const double2 *>(pu + j0 + 6);
                const double pi[4] = {-a0.x, -a0.y, -a1.x, -a1.y};
                const double pj[8] = {b0.x, b0.y, b1.x, b1.y, b2.x, b2.y, b3.x, b3.y};
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 8; ++y) acc[x][y] = fma(pi[x], pj[y], acc[x][y]);
            }
#pragma unroll
            for (int y = 0; y < 8; ++y)
#pragma unroll
                for (int x = 0; x < 4; ++x) {
                    const int r = i0 + x, cc = j0 + y;
                    if (r < ntr && cc < ntr) *nd_lu_at(L, Ut, U, nP, nF, nR, k1 + r, k1 + cc) = acc[x][y];
                }
        }
        csync();
    }
    if (bad) atomicAdd(nd.info + 4 * slot + 1, 1);
}

// the LU kernels, one per (cluster, block width, panel place) as the Cholesky's; `guard` is unused (no pivot is raised)
__global__ void __launch_bounds__(512) nd_lu_factor_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<false, ND_NB>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor_cluster_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<true, ND_NB>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor8_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<false, 8>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor8_cluster_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<true, 8>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor_large_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<false, ND_NB, true>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor_large_cluster_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<true, ND_NB, true>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor8_large_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<false, 8, true>(nd, t0, par, nFmax); }
__global__ void __launch_bounds__(512) nd_lu_factor8_large_cluster_kernel(NdDev nd, int t0, int par, double, int nFmax) { nd_lu_factor_body<true, 8, true>(nd, t0, par, nFmax); }

// dynamic shared memory of the solve kernels (bytes): the front's vector, the ring sums of the backward sweep (both in
// global memory on the large-front variants), two diagonal blocks (the next one is fetched while the current one is
// used), NB scratch
static inline size_t nd_solve_smem(int nFmax, bool vec_global = false)
{
    return (size_t)((vec_global ? 0 : 2 * ((nFmax + 1) & ~1)) + 2 * ND_NB * ND_NB + 2 * ND_NB + 2) * sizeof(double);
}

// diagonal block kb of the factor → registers (≤ 4 per thread, CTAs of ≥ 64 threads) → shared memory, so that the global
// latency of the NEXT block hides behind the substitution of the current one
static __device__ __forceinline__ void nd_diag_fetch(const double *L, int nF, int nP, int kb, int tid, int T, double sreg[4])
{
    constexpr int NB = ND_NB;
    const int nb = min(NB, nP - kb);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int idx = tid + k * T;
        sreg[k] = 0.0;
        if (idx < NB * NB) {
            const int r = idx / NB, c = idx - r * NB;
            sreg[k] = (r < nb && c <= r) ? L[(size_t)(kb + c) * nF + kb + r] : (r == c ? 1.0 : 0.0);
        }
    }
}
static __device__ __forceinline__ void nd_diag_store(double *S, int tid, int T, const double sreg[4])
{
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int idx = tid + k * T;
        if (idx < ND_NB * ND_NB) S[idx] = sreg[k];
    }
}

// ---------------------------------------------------------------------------
// forward substitution, one level: y_P = L11⁻¹(b_P + children), update vector = children − L21 y_P
// vec: per slot, unknowns in pixel order (b on entry; the pivot entries become y)
// Only the PIVOT rows are updated inside the serial block loop; the ring rows (the bulk of a front) take all their
// blocks in one parallel pass afterwards, block by block in the same order — the same sums, the same bits as a loop that
// updates every row at every step, with a chain of nP/16 short steps instead of nP/16 passes over the whole front.
// VG (large fronts): the front's vector lives in global memory, in the front's slice of nd.scr (2·even(nFmax) doubles at
// blockIdx.x); the same sums in the same order.
// ---------------------------------------------------------------------------
template <bool VG>
static __device__ __forceinline__ void nd_fwd_body(const NdDev &nd, int t0, int par, double *vec_all, size_t vec_stride, int nFmax)
{
    ND_DYN_SMEM(sm);
    constexpr int NB = ND_NB;
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int t = t0 + blockIdx.x, slot = blockIdx.y;
    const NdFront f = nd.fronts[t];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + t;
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int *off = nd.off ? nd.off + nd.off_stride * slot : nullptr;
    const int nP = pos[f.npiv], nF = pos[f.npiv + f.nring], nR = nF - nP;
    const double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
    double *uv = nd.UV[par] + nd.UV_stride * slot + foff[4 * (size_t)t + 2];
    double *vec = vec_all + vec_stride * slot;
    const int nFe = (nF + 1) & ~1;
    double *v = VG ? nd.scr + nd.scr_stride * slot + (size_t)blockIdx.x * 2 * nd_even(nFmax) : sm;
    double *Sb = VG ? sm : sm + 2 * nFe, *ys = Sb + 2 * NB * NB;
    double sreg[4];

    if (nP > 0) nd_diag_fetch(L, nF, nP, 0, tid, T, sreg);
    for (int k = tid; k < f.npiv + f.nring; k += T) {
        const int a0 = pos[k], m = pos[k + 1] - a0;
        if (k < f.npiv) {
            const int q = nd.pixlist[f.pix0 + k];
            const int g0 = off ? off[q] : q;
            for (int al = 0; al < m; ++al) v[a0 + al] = vec[g0 + al];
        } else {
            for (int al = 0; al < m; ++al) v[a0 + al] = 0.0;
        }
    }
    nd_diag_store(Sb, tid, T, sreg);
    __syncthreads();
    for (int ci = 0; ci < 2; ++ci) {
        const int c = ci == 0 ? f.child0 : f.child1;
        if (c < 0) continue;
        const NdFront cf = nd.fronts[c];
        const int *cpos = nd.posg + nd.posg_stride * slot + cf.pix0 + c + cf.npiv;
        const int cnP = cpos[0];
        const double *cuv = nd.UV[par ^ 1] + nd.UV_stride * slot + foff[4 * (size_t)c + 2];
        for (int k = tid; k < cf.nring; k += T) {
            const int r0 = cpos[k] - cnP, m = cpos[k + 1] - cpos[k];
            const int R0 = pos[nd.cmap[cf.cmap0 + k]];
            for (int al = 0; al < m; ++al) v[R0 + al] += cuv[r0 + al];
        }
        __syncthreads();
    }
    for (int kb = 0, b = 0; kb < nP; kb += NB, ++b) {
        const int nb = min(NB, nP - kb), k1 = kb + nb;
        double *S = Sb + (b & 1) * NB * NB;
        if (k1 < nP) nd_diag_fetch(L, nF, nP, k1, tid, T, sreg);
        if (tid < NB) ys[tid] = tid < nb ? v[kb + tid] : 0.0;
        __syncthreads();
        if (warp == 0) nd_block_subst(S, ys, false, lane);
        __syncthreads();
        if (k1 < nP) nd_diag_store(Sb + ((b + 1) & 1) * NB * NB, tid, T, sreg);
        if (tid < nb) v[kb + tid] = ys[tid];
        for (int r = k1 + tid; r < nP; r += T) {
            const double *col = L + (size_t)kb * nF + r;
            double s0 = 0.0, s1 = 0.0;
            if (nb == NB) {         // all 16 loads of the row in flight together (one L2 round trip on the serial chain)
                double l[NB];
#pragma unroll
                for (int c = 0; c < NB; ++c) l[c] = col[(size_t)c * nF];
#pragma unroll
                for (int c = 0; c < NB; c += 2) {
                    s0 = fma(l[c], ys[c], s0);
                    s1 = fma(l[c + 1], ys[c + 1], s1);
                }
            } else {
                for (int c = 0; c < nb; c += 2) {
                    s0 = fma(col[(size_t)c * nF], ys[c], s0);
                    if (c + 1 < nb) s1 = fma(col[(size_t)(c + 1) * nF], ys[c + 1], s1);
                }
            }
            v[r] -= s0 + s1;
        }
        __syncthreads();
    }
    // ring rows: every block of pivot columns in turn (16 independent loads per block and row)
    for (int r = nP + tid; r < nF; r += T) {
        double acc = v[r];
        for (int kb = 0; kb < nP; kb += NB) {
            const int nb = min(NB, nP - kb);
            const double *col = L + (size_t)kb * nF + r;
            double s0 = 0.0, s1 = 0.0;
            if (nb == NB) {
                double l[NB];
#pragma unroll
                for (int c = 0; c < NB; ++c) l[c] = col[(size_t)c * nF];
#pragma unroll
                for (int c = 0; c < NB; c += 2) {
                    s0 = fma(l[c], v[kb + c], s0);
                    s1 = fma(l[c + 1], v[kb + c + 1], s1);
                }
            } else {
                for (int c = 0; c < nb; c += 2) {
                    s0 = fma(col[(size_t)c * nF], v[kb + c], s0);
                    if (c + 1 < nb) s1 = fma(col[(size_t)(c + 1) * nF], v[kb + c + 1], s1);
                }
            }
            acc -= s0 + s1;
        }
        v[r] = acc;
    }
    for (int k = tid; k < f.npiv; k += T) {
        const int a0 = pos[k], m = pos[k + 1] - a0;
        const int q = nd.pixlist[f.pix0 + k];
        const int g0 = off ? off[q] : q;
        for (int al = 0; al < m; ++al) vec[g0 + al] = v[a0 + al];
    }
    for (int r = tid; r < nR; r += T) uv[r] = v[nP + r];
}
__global__ void nd_fwd_kernel(NdDev nd, int t0, int par, double *vec_all, size_t vec_stride) { nd_fwd_body<false>(nd, t0, par, vec_all, vec_stride, 0); }
__global__ void nd_fwd_large_kernel(NdDev nd, int t0, int par, double *vec_all, size_t vec_stride, int nFmax) { nd_fwd_body<true>(nd, t0, par, vec_all, vec_stride, nFmax); }

// ---------------------------------------------------------------------------
// backward substitution, one level: x_P = L11⁻ᵀ(y_P − L21ᵀ x_ring); the ring's x comes from the ancestors.
// The ring part of every pivot column's dot product is formed up front, in parallel (a warp per column); the serial
// block loop adds the part over the pivot rows below the block.  VG: as nd_fwd_body.
// ---------------------------------------------------------------------------
template <bool VG>
static __device__ __forceinline__ void nd_bwd_body(const NdDev &nd, int t0, double *vec_all, size_t vec_stride, int nFmax)
{
    ND_DYN_SMEM(sm);
    constexpr int NB = ND_NB;
    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
    const int t = t0 + blockIdx.x, slot = blockIdx.y;
    const NdFront f = nd.fronts[t];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + t;
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int *off = nd.off ? nd.off + nd.off_stride * slot : nullptr;
    const int nP = pos[f.npiv], nF = pos[f.npiv + f.nring];
    const double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
    double *vec = vec_all + vec_stride * slot;
    const int nFe = (nF + 1) & ~1;
    double *v = VG ? nd.scr + nd.scr_stride * slot + (size_t)blockIdx.x * 2 * nd_even(nFmax) : sm, *tR = v + nFe;
    double *Sb = VG ? sm : sm + 2 * nFe, *ts = Sb + 2 * NB * NB;
    double sreg[4];
    const int nblk = (nP + NB - 1) / NB;

    if (nblk > 0) nd_diag_fetch(L, nF, nP, (nblk - 1) * NB, tid, T, sreg);
    for (int k = tid; k < f.npiv + f.nring; k += T) {
        const int a0 = pos[k], m = pos[k + 1] - a0;
        const int q = nd.pixlist[f.pix0 + k];
        const int g0 = off ? off[q] : q;
        for (int al = 0; al < m; ++al) v[a0 + al] = vec[g0 + al];
    }
    if (nblk > 0) nd_diag_store(Sb + ((nblk - 1) & 1) * NB * NB, tid, T, sreg);
    __syncthreads();
    for (int c = warp; c < nP; c += nwarps) {
        const double *col = L + (size_t)c * nF;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        for (int r = nP + lane; r < nF; r += 128) {
            const double l0 = col[r], l1 = r + 32 < nF ? col[r + 32] : 0.0, l2 = r + 64 < nF ? col[r + 64] : 0.0,
                         l3 = r + 96 < nF ? col[r + 96] : 0.0;
            s0 = fma(l0, v[r], s0);
            if (r + 32 < nF) s1 = fma(l1, v[r + 32], s1);
            if (r + 64 < nF) s2 = fma(l2, v[r + 64], s2);
            if (r + 96 < nF) s3 = fma(l3, v[r + 96], s3);
        }
        double s = (s0 + s1) + (s2 + s3);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) tR[c] = s;
    }
    __syncthreads();
    for (int blk = nblk - 1; blk >= 0; --blk) {
        const int kb = blk * NB, nb = min(NB, nP - kb), k1 = kb + nb;
        double *S = Sb + (blk & 1) * NB * NB;
        if (blk > 0) nd_diag_fetch(L, nF, nP, kb - NB, tid, T, sreg);
        for (int c = warp; c < NB; c += nwarps) {
            double s = 0.0;
            if (c < nb) {
                const double *col = L + (size_t)(kb + c) * nF;
                double s0 = 0.0, s1 = 0.0;
                for (int r = k1 + lane; r < nP; r += 128) {      // four loads in flight; the sums keep their order
                    const double l0 = col[r], l1 = r + 32 < nP ? col[r + 32] : 0.0, l2 = r + 64 < nP ? col[r + 64] : 0.0,
                                 l3 = r + 96 < nP ? col[r + 96] : 0.0;
                    s0 = fma(l0, v[r], s0);
                    if (r + 32 < nP) s1 = fma(l1, v[r + 32], s1);
                    if (r + 64 < nP) s0 = fma(l2, v[r + 64], s0);
                    if (r + 96 < nP) s1 = fma(l3, v[r + 96], s1);
                }
                s = s0 + s1;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            }
            if (lane == 0) ts[c] = c < nb ? v[kb + c] - (tR[kb + c] + s) : 0.0;
        }
        if (blk > 0) nd_diag_store(Sb + ((blk - 1) & 1) * NB * NB, tid, T, sreg);
        __syncthreads();
        if (warp == 0) nd_block_subst(S, ts, true, lane);
        __syncthreads();
        if (tid < nb) v[kb + tid] = ts[tid];
        __syncthreads();
    }
    for (int k = tid; k < f.npiv; k += T) {
        const int a0 = pos[k], m = pos[k + 1] - a0;
        const int q = nd.pixlist[f.pix0 + k];
        const int g0 = off ? off[q] : q;
        for (int al = 0; al < m; ++al) vec[g0 + al] = v[a0 + al];
    }
}
__global__ void nd_bwd_kernel(NdDev nd, int t0, double *vec_all, size_t vec_stride) { nd_bwd_body<false>(nd, t0, vec_all, vec_stride, 0); }
__global__ void nd_bwd_large_kernel(NdDev nd, int t0, double *vec_all, size_t vec_stride, int nFmax) { nd_bwd_body<true>(nd, t0, vec_all, vec_stride, nFmax); }


// ===========================================================================
// Small fronts (the bottom levels of the tree: thousands of fronts of 25-60 unknowns per image): ONE WARP per front,
// several fronts per CTA, the whole front in shared memory, no CTA barrier inside the factorisation.  The generic
// kernels above spend a 64-thread CTA, five CTA barriers per block step and a round trip through global memory on
// each of them (ncu, 148 images of 128×128: 70 % of the factorisation time in the four bottom levels).
// The CTA's shared-memory arena is packed greedily: the fronts of its warps are processed in as few rounds as fit
// (one, except when a multiplier-form image is flat nearly everywhere).
// ===========================================================================
constexpr int ND_SMALL_WARPS = 8;
constexpr int ND_SMALL_MAXF = 128;      // levels whose largest possible front is at most this (and whose typical front is at most
constexpr int ND_SMALL_TYPF = 64;       // this) may go to the small kernels — when there are enough fronts to fill the GPU with warps

// arena (doubles) of a level: room for the largest possible single front, and for ND_SMALL_WARPS typical ones
static inline int nd_small_arena(int nF_worst, int nP_worst, int nF_typ, bool factor)
{
    const long long one = factor ? (long long)nF_worst * nF_worst + nF_worst + 2 : (long long)nF_worst * nP_worst + nF_worst + 2;
    const long long typ = factor ? (long long)nF_typ * nF_typ + nF_typ + 2 : (long long)nF_typ * std::min(nP_worst, nF_typ) + nF_typ + 2;
    long long a = std::max(one, (long long)ND_SMALL_WARPS * typ);
    a = std::min(a, std::max(one, (long long)12 * 1024));      // ≤ 96 KB unless a single front needs more: ≥ 2 CTAs per SM
    return (int)((a + 1) & ~1LL);
}
static inline size_t nd_small_smem(int arena) { return (size_t)arena * sizeof(double) + 2 * ND_SMALL_WARPS * sizeof(int); }

// which warps of the CTA run in round `round`: warps [w0, w1) such that their needs fit the arena (greedy, in order).
// Every thread evaluates this from the same shared table, so all agree without further communication.
static __device__ __forceinline__ bool nd_small_round(const int *s_need, int nw, int arena, int round, int w, int &base)
{
    int w0 = 0;
    for (int r = 0;; ++r) {
        int w1 = w0, used = 0;
        while (w1 < nw && (w1 == w0 || used + s_need[w1] <= arena)) { used += s_need[w1]; ++w1; }
        if (r == round) {
            if (w < w0 || w >= w1) return false;
            base = 0;
            for (int k = w0; k < w; ++k) base += s_need[k];
            return true;
        }
        w0 = w1;
        if (w0 >= nw) return false;
    }
}
static __device__ __forceinline__ int nd_small_rounds(const int *s_need, int nw, int arena)
{
    int w0 = 0, rounds = 0;
    while (w0 < nw) {
        int w1 = w0, used = 0;
        while (w1 < nw && (w1 == w0 || used + s_need[w1] <= arena)) { used += s_need[w1]; ++w1; }
        w0 = w1; ++rounds;
    }
    return rounds;
}

static __device__ __forceinline__ double nd_warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
static __device__ __forceinline__ double nd_warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// grid (ceil(fronts of the level / ND_SMALL_WARPS), slots), block 32·ND_SMALL_WARPS
__global__ void __launch_bounds__(32 * ND_SMALL_WARPS) nd_factor_small_kernel(NdDev nd, int t0, int nfr, int par, double guard, int arena)
{
    ND_DYN_SMEM(sm);
    int *s_need = reinterpret_cast<int *>(sm + arena);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int slot = blockIdx.y;
    const int t = t0 + blockIdx.x * nw + warp;
    const bool live = t < t0 + nfr;
    const NdFront f = nd.fronts[live ? t : t0];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + (live ? t : t0);
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int nP = live ? pos[f.npiv] : 0, nF = live ? pos[f.npiv + f.nring] : 0, nR = nF - nP;
    if (lane == 0) s_need[warp] = live ? ((nF * nF + nF + 2) & ~1) : 0;
    __syncthreads();
    const int rounds = nd_small_rounds(s_need, nw, arena);
    const double *ast = nd.ast + nd.ast_stride * slot;
    const int MB = nd.mb, MB2 = MB * MB;
    int guarded = 0, bad = 0;
    for (int round = 0; round < rounds; ++round) {
        int base = 0;
        if (live && nd_small_round(s_need, nw, arena, round, warp, base)) {
            double *F = sm + base;                              // column-major nF×nF, lower triangle
            int *umap = reinterpret_cast<int *>(F + (size_t)nF * nF);
            double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
            double *U = nd.U[par] + nd.U_stride * slot + foff[4 * (size_t)t + 1];
            for (int k = lane; k < nF * nF; k += 32) F[k] = 0.0;
            __syncwarp();
            {
                const int ne = nd.nnb + 1;
                for (int idx = lane; idx < f.npiv * ne; idx += 32) {
                    const int kp = idx / ne, e = idx - kp * ne;
                    const int p = nd.pixlist[f.pix0 + kp];
                    const int a0 = pos[kp], mp = pos[kp + 1] - a0;
                    if (e == 0) {
                        const double *blk = ast + (size_t)p * nd.nh * MB2;
                        for (int al = 0; al < mp; ++al)
                            for (int be = al; be < mp; ++be) F[(a0 + al) * nF + a0 + be] = blk[be * MB + al];
                    } else {
                        const int kq = nd.nbr[f.nbr0 + kp * nd.nnb + (e - 1)];
                        if (kq <= kp) continue;
                        const int q = nd.pixlist[f.pix0 + kq];
                        const int b0 = pos[kq], mq = pos[kq + 1] - b0;
                        const int h = 1 + ((e - 1) >> 1);
                        const bool fwd = ((e - 1) & 1) == 0;
                        const double *blk = ast + ((size_t)(fwd ? p : q) * nd.nh + h) * MB2;
                        for (int al = 0; al < mp; ++al)
                            for (int be = 0; be < mq; ++be)
                                F[(a0 + al) * nF + b0 + be] = fwd ? blk[be * MB + al] : blk[al * MB + be];
                    }
                }
            }
            __syncwarp();
            for (int ci = 0; ci < 2; ++ci) {
                const int c = ci == 0 ? f.child0 : f.child1;
                if (c < 0) continue;
                const NdFront cf = nd.fronts[c];
                const int *cpos = nd.posg + nd.posg_stride * slot + cf.pix0 + c + cf.npiv;
                const int cnP = cpos[0], cnR = cpos[cf.nring] - cnP;
                for (int k = lane; k < cf.nring; k += 32) {
                    const int r0 = cpos[k] - cnP, m = cpos[k + 1] - cpos[k];
                    const int R0 = pos[nd.cmap[cf.cmap0 + k]];
                    for (int al = 0; al < m; ++al) umap[r0 + al] = R0 + al;
                }
                __syncwarp();
                const double *cU = nd.U[par ^ 1] + nd.U_stride * slot + foff[4 * (size_t)c + 1];
                for (int idx = lane; idx < cnR * cnR; idx += 32) {
                    const int r = idx % cnR, cc = idx / cnR;
                    if (r < cc) continue;
                    int R = umap[r], C = umap[cc];
                    if (R < C) { const int s = R; R = C; C = s; }
                    F[C * nF + R] += cU[idx];
                }
                __syncwarp();
            }
            // right-looking Cholesky of the first nP columns; the pivot rule sees the whole column (see nd_diag_block)
            for (int c = 0; c < nP; ++c) {
                double *col = F + c * nF;
                double d = col[c];
                if (guard > 0.0) {
                    double am = 0.0;
                    for (int r = c + 1 + lane; r < nF; r += 32) am = fmax(am, fabs(col[r]));
                    am = nd_warp_max(am);
                    const double floor_ = fmax(guard, am * am * 0.0625);
                    if (!(d >= floor_)) { d = floor_; if (lane == 0) ++guarded; }
                } else if (!(d > 0.0)) {
                    bad = 1; d = 1.0;
                }
                const double inv = rsqrt(d);
                __syncwarp();
                if (lane == 0) col[c] = d * inv;
                for (int r = c + 1 + lane; r < nF; r += 32) {
                    const double l = col[r] * inv;
                    col[r] = l;
                    if (!(fabs(l) <= ND_LMAX)) bad = 1;
                }
                __syncwarp();
                // rank-one update of the trailing lower triangle: each lane keeps the multipliers of its rows
                // (r = c+1+lane, +32, …) in registers and sweeps four columns at a time — loads, FMAs, stores grouped
                // so that the shared-memory round trips of the four columns overlap
                {
                    double lr[ND_SMALL_MAXF / 32];
#pragma unroll
                    for (int k = 0; k < ND_SMALL_MAXF / 32; ++k) {
                        const int r = c + 1 + lane + 32 * k;
                        lr[k] = r < nF ? col[r] : 0.0;
                    }
                    for (int c2 = c + 1; c2 < nF; c2 += 4) {
                        double lc[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) lc[j] = c2 + j < nF ? col[c2 + j] : 0.0;
#pragma unroll
                        for (int k = 0; k < ND_SMALL_MAXF / 32; ++k) {
                            const int r = c + 1 + lane + 32 * k;
                            if (r < c2 || r >= nF) continue;
                            double tv[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) tv[j] = (c2 + j <= r) ? F[(c2 + j) * nF + r] : 0.0;
#pragma unroll
                            for (int j = 0; j < 4; ++j) tv[j] = fma(-lr[k], lc[j], tv[j]);
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (c2 + j <= r) F[(c2 + j) * nF + r] = tv[j];
                        }
                    }
                }
                __syncwarp();
            }
            for (int idx = lane; idx < nF * nP; idx += 32) L[idx] = F[idx];
            for (int idx = lane; idx < nR * nR; idx += 32) {
                const int r = idx % nR, cc = idx / nR;
                if (r >= cc) U[idx] = F[(nP + cc) * nF + nP + r];
            }
        }
        __syncthreads();
    }
    if (guarded) atomicAdd(nd.info + 4 * slot, guarded);
    if (bad) atomicAdd(nd.info + 4 * slot + 1, 1);
}

__global__ void __launch_bounds__(32 * ND_SMALL_WARPS) nd_fwd_small_kernel(NdDev nd, int t0, int nfr, int par, double *vec_all, size_t vec_stride, int arena)
{
    ND_DYN_SMEM(sm);
    int *s_need = reinterpret_cast<int *>(sm + arena);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int slot = blockIdx.y;
    const int t = t0 + blockIdx.x * nw + warp;
    const bool live = t < t0 + nfr;
    const NdFront f = nd.fronts[live ? t : t0];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + (live ? t : t0);
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int *off = nd.off ? nd.off + nd.off_stride * slot : nullptr;
    const int nP = live ? pos[f.npiv] : 0, nF = live ? pos[f.npiv + f.nring] : 0, nR = nF - nP;
    if (lane == 0) s_need[warp] = live ? ((nF * nP + nF + 2) & ~1) : 0;
    __syncthreads();
    const int rounds = nd_small_rounds(s_need, nw, arena);
    double *vec = vec_all + vec_stride * slot;
    for (int round = 0; round < rounds; ++round) {
        int base = 0;
        if (live && nd_small_round(s_need, nw, arena, round, warp, base)) {
            double *Ls = sm + base, *v = Ls + (size_t)nF * nP;
            const double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
            double *uv = nd.UV[par] + nd.UV_stride * slot + foff[4 * (size_t)t + 2];
            for (int idx = lane; idx < nF * nP; idx += 32) Ls[idx] = L[idx];
            for (int k = lane; k < f.npiv + f.nring; k += 32) {
                const int a0 = pos[k], m = pos[k + 1] - a0;
                if (k < f.npiv) {
                    const int q = nd.pixlist[f.pix0 + k];
                    const int g0 = off ? off[q] : q;
                    for (int al = 0; al < m; ++al) v[a0 + al] = vec[g0 + al];
                } else {
                    for (int al = 0; al < m; ++al) v[a0 + al] = 0.0;
                }
            }
            __syncwarp();
            for (int ci = 0; ci < 2; ++ci) {
                const int c = ci == 0 ? f.child0 : f.child1;
                if (c < 0) continue;
                const NdFront cf = nd.fronts[c];
                const int *cpos = nd.posg + nd.posg_stride * slot + cf.pix0 + c + cf.npiv;
                const int cnP = cpos[0];
                const double *cuv = nd.UV[par ^ 1] + nd.UV_stride * slot + foff[4 * (size_t)c + 2];
                for (int k = lane; k < cf.nring; k += 32) {
                    const int r0 = cpos[k] - cnP, m = cpos[k + 1] - cpos[k];
                    const int R0 = pos[nd.cmap[cf.cmap0 + k]];
                    for (int al = 0; al < m; ++al) v[R0 + al] += cuv[r0 + al];
                }
                __syncwarp();
            }
            for (int c = 0; c < nP; ++c) {
                const double *col = Ls + c * nF;
                const double yc = v[c] / col[c];
                __syncwarp();
                if (lane == 0) v[c] = yc;
                for (int r = c + 1 + lane; r < nF; r += 32) v[r] = fma(-col[r], yc, v[r]);
                __syncwarp();
            }
            for (int k = lane; k < f.npiv; k += 32) {
                const int a0 = pos[k], m = pos[k + 1] - a0;
                const int q = nd.pixlist[f.pix0 + k];
                const int g0 = off ? off[q] : q;
                for (int al = 0; al < m; ++al) vec[g0 + al] = v[a0 + al];
            }
            for (int r = lane; r < nR; r += 32) uv[r] = v[nP + r];
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(32 * ND_SMALL_WARPS) nd_bwd_small_kernel(NdDev nd, int t0, int nfr, double *vec_all, size_t vec_stride, int arena)
{
    ND_DYN_SMEM(sm);
    int *s_need = reinterpret_cast<int *>(sm + arena);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int slot = blockIdx.y;
    const int t = t0 + blockIdx.x * nw + warp;
    const bool live = t < t0 + nfr;
    const NdFront f = nd.fronts[live ? t : t0];
    const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + (live ? t : t0);
    const long long *foff = nd.foff + nd.foff_stride * slot;
    const int *off = nd.off ? nd.off + nd.off_stride * slot : nullptr;
    const int nP = live ? pos[f.npiv] : 0, nF = live ? pos[f.npiv + f.nring] : 0;
    if (lane == 0) s_need[warp] = live ? ((nF * nP + nF + 2) & ~1) : 0;
    __syncthreads();
    const int rounds = nd_small_rounds(s_need, nw, arena);
    double *vec = vec_all + vec_stride * slot;
    for (int round = 0; round < rounds; ++round) {
        int base = 0;
        if (live && nd_small_round(s_need, nw, arena, round, warp, base)) {
            double *Ls = sm + base, *v = Ls + (size_t)nF * nP;
            const double *L = nd.L + nd.L_stride * slot + foff[4 * (size_t)t];
            for (int idx = lane; idx < nF * nP; idx += 32) Ls[idx] = L[idx];
            for (int k = lane; k < f.npiv + f.nring; k += 32) {
                const int a0 = pos[k], m = pos[k + 1] - a0;
                const int q = nd.pixlist[f.pix0 + k];
                const int g0 = off ? off[q] : q;
                for (int al = 0; al < m; ++al) v[a0 + al] = vec[g0 + al];
            }
            __syncwarp();
            for (int c = nP - 1; c >= 0; --c) {
                const double *col = Ls + c * nF;
                double s = 0.0;
                for (int r = c + 1 + lane; r < nF; r += 32) s = fma(col[r], v[r], s);
                s = nd_warp_sum(s);
                const double xc = (v[c] - s) / col[c];
                __syncwarp();
                if (lane == 0) v[c] = xc;
                __syncwarp();
            }
            for (int k = lane; k < f.npiv; k += 32) {
                const int a0 = pos[k], m = pos[k + 1] - a0;
                const int q = nd.pixlist[f.pix0 + k];
                const int g0 = off ? off[q] : q;
                for (int al = 0; al < m; ++al) vec[g0 + al] = v[a0 + al];
            }
        }
        __syncthreads();
    }
}


// how one level of the tree is launched (shared by gradient_nd.cuh and the emulation harness)
struct NdLevelPlan {
    bool small;                 // warp-per-front kernels
    int t0, nfr;                // fronts of the level
    int nFw;                    // largest possible front (mb unknowns on every pixel)
    int nRc;                    // largest possible ring of a child (unknowns): the extend-add map of the generic kernel
    int nb;                     // columns per block step of the generic factorisation (16; 8 for fronts beyond its panel)
    int threads_f, threads_s;   // generic kernels: CTA sizes of the factorisation / of the solves
    size_t smem_f, smem_s;      // dynamic shared memory of the factorisation / of the solves
    int arena_f, arena_s;       // small kernels: arena (doubles)
    bool large_f = false;       // generic factorisation with the panel in global memory (nd_factor_*large*)
    bool large_s = false;       // generic solves with the front vector in global memory (nd_fwd/bwd_large_kernel)
    bool lu = false;            // LU form (nd_lu_factor_*): two panels, every level on the generic factorisation
};
static inline NdLevelPlan nd_level_plan(const NdSymbolic &sym, int s, int mb, double typ_per_pixel, int max_warps_f = 16,
                                       int max_threads_s = 512)
{
    NdLevelPlan lp;
    lp.t0 = sym.step_start[s]; lp.nfr = sym.step_start[s + 1] - lp.t0;
    lp.nFw = mb * sym.step_max_front_pix[s];
    lp.nRc = s > 0 ? mb * sym.step_max_ring_pix[s - 1] : 0;
    lp.nb = ND_NB;
    const int nPw = mb * sym.step_max_piv_pix[s];
    const int nFt = std::min(lp.nFw, (int)(typ_per_pixel * sym.step_max_front_pix[s]) + 1);
    lp.small = lp.nFw <= ND_SMALL_MAXF && nFt <= ND_SMALL_TYPF;
    const int nt = (nFt + 31) / 32, ntiles = nt * (nt + 1) / 2;
    lp.threads_f = 32 * std::min(max_warps_f, std::max(2, ntiles));
    lp.threads_s = std::min(max_threads_s, std::max(64, (nFt + 31) & ~31));
    lp.arena_f = lp.arena_s = 0;
    if (lp.small) {
        lp.arena_f = nd_small_arena(lp.nFw, nPw, nFt, true);
        lp.arena_s = nd_small_arena(lp.nFw, nPw, nFt, false);
        lp.smem_f = nd_small_smem(lp.arena_f);
        lp.smem_s = nd_small_smem(lp.arena_s);
    } else {
        lp.smem_f = nd_factor_smem(lp.nFw, lp.nRc);
        lp.smem_s = nd_solve_smem(lp.nFw);
    }
    return lp;
}

// The same for a level whose sizes were MEASURED on the device (nd_level_sizes_kernel): the forms with many unknowns per
// pixel (sum-of-regularisers multipliers: 3-6) cannot afford worst-case shared memory.  Generic kernels only.
static inline NdLevelPlan nd_level_plan_sized(const NdSymbolic &sym, int s, int nF, int nRchild, size_t smem_optin,
                                             int max_warps_f = 16, int max_threads_s = 512)
{
    NdLevelPlan lp;
    lp.t0 = sym.step_start[s]; lp.nfr = sym.step_start[s + 1] - lp.t0;
    lp.nFw = std::max(nF, 1);
    lp.nRc = nRchild;
    lp.small = false;
    const int nt = (lp.nFw + 31) / 32, ntiles = nt * (nt + 1) / 2;
    lp.threads_f = 32 * std::min(max_warps_f, std::max(2, ntiles));
    lp.threads_s = std::min(max_threads_s, std::max(64, (lp.nFw + 31) & ~31));
    lp.arena_f = lp.arena_s = 0;
    lp.nb = nd_factor_smem(lp.nFw, lp.nRc, ND_NB) <= smem_optin ? ND_NB : 8;
    lp.smem_f = nd_factor_smem(lp.nFw, lp.nRc, lp.nb);
    lp.smem_s = nd_solve_smem(lp.nFw);
    return lp;
}

// shared memory of the generic kernels of a level, as they will be launched
static inline size_t nd_level_smem_f(const NdLevelPlan &lp) { return nd_factor_smem(lp.nFw, lp.nRc, lp.nb, lp.large_f, lp.lu); }
static inline size_t nd_level_smem_s(const NdLevelPlan &lp) { return nd_solve_smem(lp.nFw, lp.large_s); }

// Sends the generic kernels of a level to the large-front variants when their shared memory would exceed `limit` bytes
// (the opt-in maximum, or less under a test hook).  A front beyond the 8-column panel takes 16-column block steps there
// (half the steps, half the passes over the trailing matrix); a level sent by the hook alone keeps its block width, and
// so its bits.  false: the level needs the variants for a front beyond `smem_optin` but `allow` is not set — the caller
// lets a band solver try the shape first, as before the variants existed.
// A level in the LU form (before nd_level_large): 8-column block steps when the two 16-column panels do not fit in
// `smem_optin` (the largest front of a 512² image: 1536 unknowns, 393 KB at 16 columns, 203 KB at 8).
static inline void nd_level_lu(NdLevelPlan &lp, size_t smem_optin)
{
    lp.lu = true;
    if (nd_factor_smem(lp.nFw, lp.nRc, ND_NB, false, true) > smem_optin) lp.nb = 8;
}

static inline bool nd_level_large(NdLevelPlan &lp, size_t limit, size_t smem_optin, bool allow)
{
    const size_t f = nd_factor_smem(lp.nFw, lp.nRc, lp.nb, false, lp.lu), s = nd_solve_smem(lp.nFw);
    if (!allow && (f > smem_optin || s > smem_optin)) return false;
    lp.large_f = f > limit;
    lp.large_s = s > limit;
    if (lp.large_f && f > smem_optin) lp.nb = ND_NB;
    if (!lp.small) { lp.smem_f = nd_level_smem_f(lp); lp.smem_s = nd_level_smem_s(lp); }
    return true;
}

// scratch (doubles per image) of a level on the large-front variants with C CTAs per front: one panel per CTA, the
// vector and the ring sums per front
static inline size_t nd_level_scratch(const NdLevelPlan &lp, int C)
{
    const size_t f = lp.large_f ? (size_t)lp.nfr * C * (lp.lu ? 2 : 1) * lp.nb * nd_panel_pitch(lp.nFw) : 0;
    const size_t s = lp.large_s ? (size_t)lp.nfr * 2 * nd_even(lp.nFw) : 0;
    return std::max(f, s);
}

// largest front and largest ring (unknowns) of every level over the images of the wave → lvl[2s], lvl[2s+1] (zeroed by
// the caller).  grid (ceil(fronts / 256), slots)
__global__ void __launch_bounds__(256) nd_level_sizes_kernel(NdDev nd, int *lvl)
{
    const int slot = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nd.nfronts) {
        const NdFront f = nd.fronts[t];
        const int *pos = nd.posg + nd.posg_stride * slot + f.pix0 + t;
        const int nP = pos[f.npiv], nF = pos[f.npiv + f.nring];
        const int s = nd.nsteps - 1 - f.depth;
        atomicMax(lvl + 2 * s, nF);
        atomicMax(lvl + 2 * s + 1, nF - nP);
    }
}

}  // namespace bpltv
