// nd_sumregs.cuh — the scalar `sumregs_gradient_reg` system (/root/reference/src/SumRegsLearningFunction.jl:112-167) in the
// form nd_solver.cuh factorises (fp64, node space).
//
//     (I + Σ_k α_k G_kᵀ(B_k − C_k)G_k) p = ū − u,      g_k = pᵀ G_kᵀ(Act_k Den_k G_k u + γ Inact_k G_k u)        (:160-166)
//
// with the three difference operators (forward, backward, centred).  For SCALAR α_k the matrix is symmetric positive
// definite, one unknown per node, and couples nodes at most two pixels apart (G_kᵀ T G_k reaches ±2 rows / columns): the
// nested-dissection multifrontal Cholesky of the TV learning function takes it with coupling radius W = 2.  The PATCH
// variant, :195-262, scales the rows of each term by a different map: not symmetric, it takes the LU form of the same
// fronts (nd_lu_factor_body) on the stencil of nd3_stencil_map_kernel.
// The per-(pixel, operator) tensors and weights are lu3_classify's, the matrix-free residual is lu3_apply, the functional
// and the backward-error rule are those of lu3_solve (lu_band.cuh): the band LU remains the second implementation.
//
// Kernels: nd3_stencil / nd3_stencil_map (the matrix in pixel-stencil form + the right-hand side), nd3_residual (r − M p
// through the stencils and tensors, independent of the assembled matrix), nd3_axpy, nd3_finish (backward error,
// functional, sums).
#pragma once
#include "lu_band.cuh"
#include "nd_solver.cuh"

namespace bpltv {

constexpr int ND3_W = 2;
constexpr int ND3_NH = 13;      // nd_nh(2): the node itself + 12 forward offsets

// forward offset index h of nd_symbolic.h (W = 2) for (di, dj), dj > 0 or (dj == 0 and di > 0)
static __host__ __device__ __forceinline__ int nd3_h(int di, int dj) { return dj == 0 ? di : 3 + 5 * (dj - 1) + (di + 2); }

// Row v of I + Σ_k α_k G_kᵀ T_k G_k (13 stencil offsets, the summation order of lu3_assemble), written as the entries
// A[v + d, v] = A[v, v + d] of the forward offsets d; p ← r (the solve runs in place).  The slot's `ast` must be zero.
// grid (slots, chunks)
__global__ void __launch_bounds__(256) nd3_stencil_kernel(LuSlots ws, Lu3Params pr, double *ast_all, size_t ast_stride)
{
    const int slot = blockIdx.x;
    const int n = ws.n, N = ws.N;
    double *pix = ws.pix + ws.pix_stride * slot;
    double *ast = ast_all + ast_stride * slot;
    const int offs[13] = {-2 * n, -n - 1, -n, -n + 1, -2, -1, 0, 1, 2, n - 1, n, n + 1, 2 * n};   // distinct for n ≥ 4
    for (int v = blockIdx.y * blockDim.x + threadIdx.x; v < N; v += gridDim.y * blockDim.x) {
        const int i = v % n, j = v / n;
        double acc[13];
#pragma unroll
        for (int s = 0; s < 13; ++s) acc[s] = 0.0;
        acc[6] = 1.0;
        visit_node(i, j, n, [&](int q, int k, double c1, double c2) {
            if (k >= ws.nops) return;
            const double *tk = pix + (size_t)(6 * k) * N;
            const double a = pr.alpha[k];
            const double v1 = c1 * tk[q] + c2 * tk[(size_t)2 * N + q];                  // (c1 c2)·T
            const double v2 = c1 * tk[(size_t)N + q] + c2 * tk[(size_t)3 * N + q];
            visit_stencil(k, q % n, q / n, n, [&](int node, double e1, double e2) {
                const double val = a * (v1 * e1 + v2 * e2);
                const int d = node - v;
#pragma unroll
                for (int s = 0; s < 13; ++s)
                    if (offs[s] == d) { acc[s] += val; break; }
            });
        });
        double *row = ast + (size_t)v * ND3_NH;
        row[0] = acc[6];
        row[nd3_h(1, 0)] = acc[7];
        row[nd3_h(2, 0)] = acc[8];
        row[nd3_h(-1, 1)] = acc[9];
        row[nd3_h(0, 1)] = acc[10];
        row[nd3_h(1, 1)] = acc[11];
        row[nd3_h(0, 2)] = acc[12];
        pix[(size_t)LU_PL_P * N + v] = pix[(size_t)LU_PL_R * N + v];
    }
}

// Row v of I + Σ_k diag(α_k) G_kᵀ T_k G_k with the λ-maps α_k (rows scaled by α_k(v): not symmetric), in the LU form's
// stencil (nd_lu_factor_body: 2·ND3_NH − 1 entries per node) — the values and summation order of lu3_assemble:
//   [0] A[v, v],  [h] A[v + d_h, v],  [ND3_NH − 1 + h] A[v, v + d_h]
// Row v gives A[v, v + d_h] of its own node and A[v, v − d_h], the [h] entry of node v − d_h (written only for nodes
// inside the image, so every entry has one writer); p ← r.  The slot's `ast` must be zero.  grid (slots, chunks)
constexpr int ND3_NH2 = 2 * ND3_NH - 1;
template <typename Real>
__global__ void __launch_bounds__(256) nd3_stencil_map_kernel(LuSlots ws, Lu3Params pr, const Real *alpha_maps, double *ast_all,
                                                              size_t ast_stride)
{
    const int slot = blockIdx.x;
    const int n = ws.n, N = ws.N;
    double *pix = ws.pix + ws.pix_stride * slot;
    double *ast = ast_all + ast_stride * slot;
    const int offs[13] = {-2 * n, -n - 1, -n, -n + 1, -2, -1, 0, 1, 2, n - 1, n, n + 1, 2 * n};   // distinct for n ≥ 4
    const int di[6] = {1, 2, -1, 0, 1, 0}, dj[6] = {0, 0, 1, 1, 1, 2};     // forward offsets of offs[7..12]
    for (int v = blockIdx.y * blockDim.x + threadIdx.x; v < N; v += gridDim.y * blockDim.x) {
        const int i = v % n, j = v / n;
        double acc[13];
#pragma unroll
        for (int s = 0; s < 13; ++s) acc[s] = 0.0;
        acc[6] = 1.0;
        visit_node(i, j, n, [&](int q, int k, double c1, double c2) {
            if (k >= ws.nops) return;
            const double *tk = pix + (size_t)(6 * k) * N;
            const double a = lu3_alpha<Real>(alpha_maps, pr, N, k, v);
            const double v1 = c1 * tk[q] + c2 * tk[(size_t)2 * N + q];                  // (c1 c2)·T
            const double v2 = c1 * tk[(size_t)N + q] + c2 * tk[(size_t)3 * N + q];
            visit_stencil(k, q % n, q / n, n, [&](int node, double e1, double e2) {
                const double val = a * (v1 * e1 + v2 * e2);
                const int d = node - v;
#pragma unroll
                for (int s = 0; s < 13; ++s)
                    if (offs[s] == d) { acc[s] += val; break; }
            });
        });
        double *row = ast + (size_t)v * ND3_NH2;
        row[0] = acc[6];
#pragma unroll
        for (int s = 0; s < 6; ++s) {
            const int h = nd3_h(di[s], dj[s]);
            row[ND3_NH - 1 + h] = acc[7 + s];                       // A[v, v + d_h]
            const int ii = i - di[s], jj = j - dj[s];               // A[v, v − d_h] = A[w + d_h, w], w = v − d_h
            if (ii >= 0 && ii < n && jj >= 0 && jj < n) ast[(size_t)(ii + n * jj) * ND3_NH2 + h] = acc[5 - s];
        }
        pix[(size_t)LU_PL_P * N + v] = pix[(size_t)LU_PL_R * N + v];
    }
}

// work = r − M p (matrix-free; the λ-maps when given), relres = ‖work‖ / ‖r‖.  One CTA per image.
// rstate (2 doubles per slot, or nullptr): the stop of lu3_solve's refinement at step `it` (0: after the first solve) —
// after pr.refine steps, at rounding level, or when a step no longer gains a factor 4, rstate[1] is set and nd3_axpy
// leaves p alone from then on (the residual of the unchanged p is formed again, with the same bits).
template <typename Real>
__global__ void __launch_bounds__(1024) nd3_residual_kernel(LuSlots ws, Lu3Params pr, double *relres_img, int img0,
                                                            const Real *alpha_maps = nullptr, double *rstate = nullptr, int it = 0)
{
    __shared__ double red[40];
    const int slot = blockIdx.x, tid = threadIdx.x;
    const int n = ws.n, N = ws.N;
    double *pix = ws.pix + ws.pix_stride * slot;
    const double *r = pix + (size_t)LU_PL_R * N, *p = pix + (size_t)LU_PL_P * N;
    double *work = pix + (size_t)LU_PL_WORK * N;
    double bn2 = 0.0, rn2 = 0.0;
    for (int v = tid; v < N; v += blockDim.x) {
        const double res = r[v] - lu3_apply<Real>(pix, n, N, ws.nops, alpha_maps, pr, p, v);
        work[v] = res;
        rn2 = fma(res, res, rn2);
        bn2 = fma(r[v], r[v], bn2);
    }
    rn2 = lu_block_sum(rn2, red);
    bn2 = lu_block_sum(bn2, red);
    if (tid == 0) {
        const double rel = bn2 > 0.0 ? sqrt(rn2 / bn2) : 0.0;
        relres_img[img0 + slot] = rel;
        if (rstate) {
            double *rs = rstate + 2 * slot;       // [0] residual of the last step taken, [1] ≠ 0: stopped
            if (it == 0) { rs[0] = 1e300; rs[1] = 0.0; }
            if (rs[1] == 0.0) {
                if (it >= pr.refine || rel <= 1e-14 || !(rel <= 0.25 * rs[0])) rs[1] = 1.0;
                else rs[0] = rel;
            }
        }
    }
}

// p += work (not once the slot's refinement stopped: rstate as nd3_residual_kernel).  grid (slots, chunks)
__global__ void __launch_bounds__(256) nd3_axpy_kernel(LuSlots ws, const double *rstate = nullptr)
{
    const int slot = blockIdx.x, N = ws.N;
    if (rstate && rstate[2 * slot + 1] != 0.0) return;
    double *pix = ws.pix + ws.pix_stride * slot;
    double *p = pix + (size_t)LU_PL_P * N;
    const double *work = pix + (size_t)LU_PL_WORK * N;
    for (int v = blockIdx.y * blockDim.x + threadIdx.x; v < N; v += gridDim.y * blockDim.x) p[v] += work[v];
}

// Normwise backward error ‖r − Mp‖ / (‖M‖‖p‖ + ‖r‖) with the bound ‖M‖ ≤ 1 + 18·γ·max α (as lu3_solve) → relres_img; a
// factorisation that broke down or an error above `tol` poisons the result with NaN (→ BPLTV_ERR_NUMERIC).
// g_k = Σ_v p_v (G_kᵀ w_k)_v per operator (:166), summed per patch of the lm×ln grid (1×1 for the scalar parameter).
// With the λ-maps (:195-262), max α runs over the maps and relres_img keeps the relative residual ‖r − Mp‖/‖r‖ of
// nd3_residual_kernel, as lu3_solve reports it.  `work` must hold the residual of the final p.  One CTA per image.
template <typename Real = double>
__global__ void __launch_bounds__(1024) nd3_finish_kernel(LuSlots ws, Lu3Params pr, const int *nd_info, double tol, double *out_img,
                                                         double *relres_img, int img0, const Real *alpha_maps = nullptr)
{
    __shared__ double red[40];
    const int slot = blockIdx.x, tid = threadIdx.x;
    const int n = ws.n, N = ws.N;
    double *pix = ws.pix + ws.pix_stride * slot;
    const double *r = pix + (size_t)LU_PL_R * N, *p = pix + (size_t)LU_PL_P * N, *work = pix + (size_t)LU_PL_WORK * N;
    double *fk = pix + (size_t)LU_PL_F * N;
    double pn2 = 0.0, bn2 = 0.0, rn2 = 0.0;
    for (int v = tid; v < N; v += blockDim.x) {
        pn2 = fma(p[v], p[v], pn2);
        bn2 = fma(r[v], r[v], bn2);
        rn2 = fma(work[v], work[v], rn2);
    }
    pn2 = lu_block_sum(pn2, red);
    bn2 = lu_block_sum(bn2, red);
    rn2 = lu_block_sum(rn2, red);
    double amax = 0.0;
    if (alpha_maps) {
        for (int v = tid; v < N; v += blockDim.x)
            for (int k = 0; k < ws.nops; ++k) amax = fmax(amax, lu3_alpha<Real>(alpha_maps, pr, N, k, v));
        amax = lu_block_max(amax, red);
    } else {
        for (int k = 0; k < ws.nops; ++k) amax = fmax(amax, pr.alpha[k]);
    }
    const double berr = sqrt(rn2) / ((1.0 + 18.0 * pr.gamma * amax) * sqrt(pn2) + sqrt(bn2) + 1e-300);
    const bool failed = nd_info[4 * slot + 1] != 0 || !(berr <= tol);
    const int ng = pr.lm * pr.ln;
    for (int k = 0; k < ws.nops; ++k) {
        const double *w1 = pix + (size_t)(6 * k + 4) * N, *w2 = pix + (size_t)(6 * k + 5) * N;
        for (int v = tid; v < N; v += blockDim.x) {
            double s = 0.0;
            visit_node(v % n, v / n, n, [&](int q, int kk, double c1, double c2) {
                if (kk == k) s += c1 * w1[q] + c2 * w2[q];
            });
            fk[v] = p[v] * s;
        }
        __syncthreads();
        for (int g = 0; g < ng; ++g) {
            const int pi = g % pr.lm, pj = g / pr.lm;
            double acc = 0.0;
            for (int v = tid; v < N; v += blockDim.x) {
                const int i = v % n, j = v / n;
                const int qi = (int)(((long long)i * pr.lm) / n), qj = (int)(((long long)j * pr.ln) / n);
                if (qi == pi && qj == pj) acc += fk[v];
            }
            acc = lu_block_sum(acc, red);
            if (tid == 0) out_img[((size_t)(img0 + slot) * ws.nops + k) * ng + g] = failed ? nan("") : acc;
        }
        __syncthreads();
    }
    if (tid == 0 && !alpha_maps) relres_img[img0 + slot] = berr;
}


// ===========================================================================
// MULT3 — `sumregs_gradient` (non-regularised: scalar :264-327, patch :330-407) in multiplier space on the same solver
// ===========================================================================
// (diag(E) + B Bᵀ) ζ = B r,  p = r − Bᵀζ, the formulation of gradient_sumregs.cuh (one mode per sloped (pixel, operator),
// two per flat one, numbered pixel-major / operator-minor): 3-6 unknowns per pixel.  The modes of a pixel touch only the
// five nodes of its cross (q, q±1, q±n), so two pixels couple when their crosses share a node — |d|₁ ≤ 2, inside the
// coupling radius W = 2 of the tree.  The band Cholesky of gradient.cuh stays as the second implementation.
constexpr int ND3M_MB = 6;
constexpr int ND3M_PLANES = 18;   // [5k..5k+4] ea, eb, E, w1, w2 of operator k; 15 r = u − ū; 16 p; 17 functional scratch

struct Nd3mSlots {
    int n, N;
    double *pix; size_t pix_stride;
    int *off3; size_t off3_stride;      // 3N+1 per slot: first mode of (pixel q, operator k) at 3q+k
    int *poff; size_t poff_stride;      // N+1 per slot: first mode of pixel q (the solver's numbering)
    double *vec; size_t vec_stride;     // 3 vectors of 6N per slot: b, ζ, work
    int *info;                          // the solver's: 4 per slot
};
struct Nd3mVariant {
    int patch, lm, ln;
    double alpha[3], act_tol, eps_act, relres_tol;
};

static __device__ __forceinline__ double nd3m_beta(const double *pix, int N, int q, int k, int m, bool iso, double c1, double c2)
{
    if (iso) return m == 0 ? c1 : c2;
    return pix[(size_t)(5 * k) * N + q] * c1 + pix[(size_t)(5 * k + 1) * N + q] * c2;
}

// per (pixel, operator) modes + exclusive scan of the mode counts.  One CTA per image.
template <typename Real>
__global__ void __launch_bounds__(1024) nd3m_classify_kernel(Nd3mSlots ws, Nd3mVariant gv, const Real *u_all, const Real *ubar_all,
                                                            const Real *alpha_maps, int img0)
{
    __shared__ int s_warp[33];
    const int slot = blockIdx.x;
    const int n = ws.n, N = ws.N;
    const Real *u = u_all + (size_t)(img0 + slot) * N;
    const Real *ub = ubar_all + (size_t)(img0 + slot) * N;
    double *pix = ws.pix + ws.pix_stride * slot;
    int *off3 = ws.off3 + ws.off3_stride * slot, *poff = ws.poff + ws.poff_stride * slot;
    if (threadIdx.x < 4) ws.info[4 * slot + threadIdx.x] = 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    int base = 0;
    for (int q0 = 0; q0 < N; q0 += blockDim.x) {
        const int q = q0 + (int)threadIdx.x;
        int cnt = 0, ck[3] = {0, 0, 0};
        if (q < N) {
            const int i = q % n, j = q / n;
            pix[(size_t)15 * N + q] = (double)u[q] - (double)ub[q];          // u − ū (:322, :391)
            for (int k = 0; k < 3; ++k) {
                double g1, g2;
                op_apply<Real>(k, i, j, n, u, q, g1, g2);
                const double nrm = sqrt(g1 * g1 + g2 * g2);
                const double a = gv.patch ? (double)alpha_maps[(size_t)k * N + q] : gv.alpha[k];
                const bool iso = nrm < gv.act_tol;                           // act = |G_k u| < 1e-12 (:273)
                double *pk = pix + (size_t)(5 * k) * N;
                pk[q] = iso ? 1.0 : -g2 / nrm;
                pk[(size_t)N + q] = iso ? 0.0 : g1 / nrm;
                pk[(size_t)2 * N + q] = iso ? gv.eps_act : nrm / a;
                pk[(size_t)3 * N + q] = iso ? 0.0 : g1 / nrm;
                pk[(size_t)4 * N + q] = iso ? 0.0 : g2 / nrm;
                ck[k] = iso ? 2 : 1;
                cnt += ck[k];
            }
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int v = lane < nw ? s_warp[lane] : 0, iv = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, iv, o);
                if (lane >= o) iv += t;
            }
            s_warp[lane] = iv - v;
            if (lane == 31) s_warp[32] = iv;
        }
        __syncthreads();
        if (q < N) {
            const int a0 = base + s_warp[warp] + incl - cnt;
            poff[q] = a0;
            off3[3 * q] = a0; off3[3 * q + 1] = a0 + ck[0]; off3[3 * q + 2] = a0 + ck[0] + ck[1];
        }
        base += s_warp[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) { poff[N] = base; off3[3 * N] = base; }
}

// the modes of pixel q as rows over the nodes of its cross — c = 0: q, 1: q+1, 2: q−1, 3: q+n, 4: q−n — and their compliances
static __device__ void nd3m_pixel_modes(const double *pix, const int *off3, int n, int N, int q, double B[ND3M_MB][5],
                                        double Em[ND3M_MB], int &nm_out)
{
    const int i = q % n, j = q / n;
    int m = 0;
    for (int k = 0; k < 3; ++k) {
        const int nm = off3[3 * q + k + 1] - off3[3 * q + k];
        for (int mm = 0; mm < nm; ++mm) {
            for (int c = 0; c < 5; ++c) B[m][c] = 0.0;
            visit_stencil(k, i, j, n, [&](int node, double c1, double c2) {
                const int d = node - q;
                const int c = d == 0 ? 0 : (d == 1 ? 1 : (d == -1 ? 2 : (d == n ? 3 : 4)));
                B[m][c] = nd3m_beta(pix, N, q, k, mm, nm == 2, c1, c2);
            });
            Em[m] = pix[(size_t)(5 * k + 2) * N + q];
            ++m;
        }
    }
    nm_out = m;
}

// diag(E) + B Bᵀ in pixel-stencil form (MB = 6, NH = 13) and b = B r.  One thread per (pixel, forward offset); grid (slots, chunks)
__global__ void __launch_bounds__(256) nd3m_stencil_kernel(Nd3mSlots ws, double *ast_all, size_t ast_stride)
{
    const int slot = blockIdx.x;
    const int n = ws.n, N = ws.N;
    const double *pix = ws.pix + ws.pix_stride * slot;
    const int *off3 = ws.off3 + ws.off3_stride * slot;
    double *ast = ast_all + ast_stride * slot;
    double *bvec = ws.vec + ws.vec_stride * slot;
    const double *rc = pix + (size_t)15 * N;
    constexpr int MB = ND3M_MB;
    const int ex[5] = {0, 1, -1, 0, 0}, ey[5] = {0, 0, 0, 1, -1};
    for (long long idx = (long long)blockIdx.y * blockDim.x + threadIdx.x; idx < (long long)N * ND3_NH; idx += (long long)gridDim.y * blockDim.x) {
        const int p = (int)(idx / ND3_NH), h = (int)(idx - (long long)p * ND3_NH);
        const int i = p % n, j = p / n;
        double Bp[MB][5], Ep[MB];
        int mp;
        nd3m_pixel_modes(pix, off3, n, N, p, Bp, Ep, mp);
        double *blk = ast + ((size_t)p * ND3_NH + h) * MB * MB;
        if (h == 0) {
            for (int be = 0; be < MB; ++be)
                for (int al = 0; al < MB; ++al) {
                    double v = 0.0;
                    if (be < mp && al < mp) {
                        for (int c = 0; c < 5; ++c) v += Bp[be][c] * Bp[al][c];
                        if (be == al) v += Ep[be];
                    }
                    blk[be * MB + al] = v;
                }
            const int a0 = off3[3 * p];
            for (int m = 0; m < mp; ++m) {
                double s = 0.0;
                for (int c = 0; c < 5; ++c) {
                    const int ii = i + ex[c], jj = j + ey[c];
                    if (Bp[m][c] != 0.0 && ii >= 0 && ii < n && jj >= 0 && jj < n) s += Bp[m][c] * rc[ii + n * jj];
                }
                bvec[a0 + m] = s;
            }
            continue;
        }
        // forward offset h of nd_symbolic.h at W = 2 (nd_fwd_offset): (1,0) (2,0), then dj = 1, 2 with di = −2..2
        const int di = h <= 2 ? h : (h - 3) % 5 - 2, dj = h <= 2 ? 0 : 1 + (h - 3) / 5;
        const int ii = i + di, jj = j + dj;
        const bool in = ii >= 0 && ii < n && jj >= 0 && jj < n && (abs(di) + abs(dj) <= 2);
        double Bq[MB][5], Eq[MB];
        int mq = 0;
        if (in) nd3m_pixel_modes(pix, off3, n, N, ii + n * jj, Bq, Eq, mq);
        for (int be = 0; be < MB; ++be)
            for (int al = 0; al < MB; ++al) {
                double v = 0.0;
                if (in && be < mq && al < mp) {
                    // node p + e_c = q + e_c'  ⇔  e_c' = e_c − d
                    for (int c = 0; c < 5; ++c) {
                        const int fx = ex[c] - di, fy = ey[c] - dj;
                        if (abs(fx) + abs(fy) > 1) continue;
                        const int c2 = fx == 0 ? (fy == 0 ? 0 : (fy == 1 ? 3 : 4)) : (fx == 1 ? 1 : 2);
                        v += Bq[be][c2] * Bp[al][c];
                    }
                }
                blk[be * MB + al] = v;
            }
    }
}

// p = r − Bᵀζ; res = B p − E ζ (through the stencils) → work; relres = ‖res‖/‖b‖.  One CTA per image.
__global__ void __launch_bounds__(1024) nd3m_residual_kernel(Nd3mSlots ws, double *relres_img, int img0)
{
    __shared__ double red[40];
    const int slot = blockIdx.x, tid = threadIdx.x;
    const int n = ws.n, N = ws.N;
    double *pix = ws.pix + ws.pix_stride * slot;
    const double *rc = pix + (size_t)15 * N;
    double *p = pix + (size_t)16 * N;
    const int *off3 = ws.off3 + ws.off3_stride * slot;
    double *vec = ws.vec + ws.vec_stride * slot;
    const double *bvec = vec, *zeta = vec + (size_t)ND3M_MB * N;
    double *work = vec + (size_t)2 * ND3M_MB * N;
    const int Nd = off3[3 * N];
    double bn2 = 0.0;
    for (int a = tid; a < Nd; a += blockDim.x) bn2 = fma(bvec[a], bvec[a], bn2);
    bn2 = lu_block_sum(bn2, red);
    for (int v = tid; v < N; v += blockDim.x) {
        double s = 0.0;
        visit_node(v % n, v / n, n, [&](int q, int k, double c1, double c2) {
            const int a0 = off3[3 * q + k], nm = off3[3 * q + k + 1] - a0;
            for (int m = 0; m < nm; ++m) s += nd3m_beta(pix, N, q, k, m, nm == 2, c1, c2) * zeta[a0 + m];
        });
        p[v] = rc[v] - s;
    }
    __syncthreads();
    double rn2 = 0.0;
    for (int e = tid; e < 3 * N; e += blockDim.x) {
        const int q = e / 3, k = e - 3 * q;
        double d1, d2;
        op_apply<double>(k, q % n, q / n, n, p, q, d1, d2);
        const int a0 = off3[e], nm = off3[e + 1] - a0;
        const double E = pix[(size_t)(5 * k + 2) * N + q];
        for (int m = 0; m < nm; ++m) {
            const double r = nd3m_beta(pix, N, q, k, m, nm == 2, d1, d2) - E * zeta[a0 + m];
            work[a0 + m] = r;
            rn2 = fma(r, r, rn2);
        }
    }
    rn2 = lu_block_sum(rn2, red);
    if (tid == 0) relres_img[img0 + slot] = bn2 > 0.0 ? sqrt(rn2 / bn2) : 0.0;
}

// vec[dst] (+)= vec[src] over the image's modes.  grid (slots, chunks)
__global__ void __launch_bounds__(256) nd3m_axpy_kernel(Nd3mSlots ws, int dst, int src, int add)
{
    const int slot = blockIdx.x;
    const int Nd = ws.poff[ws.poff_stride * slot + ws.N];
    double *vec = ws.vec + ws.vec_stride * slot;
    double *y = vec + (size_t)dst * ND3M_MB * ws.N;
    const double *x = vec + (size_t)src * ND3M_MB * ws.N;
    for (int a = blockIdx.y * blockDim.x + threadIdx.x; a < Nd; a += gridDim.y * blockDim.x) y[a] = add ? y[a] + x[a] : x[a];
}

// functional per operator: scalar −Σ_q ⟨(G_k p)_q, w_kq⟩ (:326); patch −p_ν (G_kᵀ w_k)_ν summed over each patch (:395-405).
// out_img: 3·lm·ln per image, [operator][patch].  A broken factorisation or a residual above the tolerance poisons with NaN.
__global__ void __launch_bounds__(1024) nd3m_finish_kernel(Nd3mSlots ws, Nd3mVariant gv, const double *relres_img, double *out_img, int img0)
{
    __shared__ double red[40];
    const int slot = blockIdx.x, tid = threadIdx.x;
    const int n = ws.n, N = ws.N;
    double *pix = ws.pix + ws.pix_stride * slot;
    const double *p = pix + (size_t)16 * N;
    double *fk = pix + (size_t)17 * N;
    const int ng = gv.lm * gv.ln;
    const bool poisoned = ws.info[4 * slot + 1] != 0 || !(relres_img[img0 + slot] <= gv.relres_tol);
    for (int k = 0; k < 3; ++k) {
        const double *w1 = pix + (size_t)(5 * k + 3) * N, *w2 = pix + (size_t)(5 * k + 4) * N;
        for (int v = tid; v < N; v += blockDim.x) {
            const int i = v % n, j = v / n;
            double val;
            if (!gv.patch) {
                double d1, d2;
                op_apply<double>(k, i, j, n, p, v, d1, d2);
                val = -(d1 * w1[v] + d2 * w2[v]);
            } else {
                double s = 0.0;
                visit_node(i, j, n, [&](int q, int kk, double c1, double c2) {
                    if (kk == k) s += c1 * w1[q] + c2 * w2[q];
                });
                val = -p[v] * s;
            }
            fk[v] = val;
        }
        __syncthreads();
        for (int g = 0; g < ng; ++g) {
            const int pi = g % gv.lm, pj = g / gv.lm;
            double acc = 0.0;
            for (int v = tid; v < N; v += blockDim.x) {
                const int i = v % n, j = v / n;
                const int qi = (int)(((long long)i * gv.lm) / n), qj = (int)(((long long)j * gv.ln) / n);
                if (ng == 1 || (qi == pi && qj == pj)) acc += fk[v];
            }
            acc = lu_block_sum(acc, red);
            if (tid == 0) out_img[((size_t)(img0 + slot) * 3 + k) * ng + g] = poisoned ? nan("") : acc;
        }
        __syncthreads();
    }
}

}  // namespace bpltv
