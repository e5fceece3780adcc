// emu_nd_lu.cpp — TEST INFRASTRUCTURE: runs the patch sumregs_gradient_reg path of gradient_nd.cuh (run_gradient3_nd_reg
// with λ-maps: lu3_classify → nd3_stencil_map → LU of the nested-dissection fronts → forward sweep on L, backward sweep on
// Uᵀ, with the band LU's refinement stop → nd3_finish) for ONE image on the CPU thread emulation (emu_cuda.h).  Without
// maps it runs the scalar path on the Cholesky of the same fronts, for comparison.  Levels may be sent to the 8-column
// kernels (smem_limit), to the large-front variants (large_limit) and to cluster-shared fronts (csize), as the planner
// does on the device.  Built by tests/test_emu_nd_lu.py with g++ -std=c++20 -DBPLTV_EMU; never shipped.
#include "emu_cuda.h"

#include <climits>
#include <cmath>
#include <cstring>

#include "../../bpldenoising_b200/csrc/nd_sumregs.cuh"

using namespace bpltv;
using NdFactorKernelFn = void (*)(NdDev, int, int, double, int);

// the row v of the assembled LU-form stencil set to zero: a matrix the factorisation must report as broken down
static void emu_zero_row(std::vector<double> &ast, int n, int v)
{
    const int i = v % n, j = v / n;
    const int di[6] = {1, 2, -1, 0, 1, 0}, dj[6] = {0, 0, 1, 1, 1, 2};
    ast[(size_t)v * ND3_NH2] = 0.0;
    for (int s = 0; s < 6; ++s) {
        const int h = nd3_h(di[s], dj[s]);
        ast[(size_t)v * ND3_NH2 + ND3_NH - 1 + h] = 0.0;
        const int ii = i - di[s], jj = j - dj[s];
        if (ii >= 0 && ii < n && jj >= 0 && jj < n) ast[(size_t)(ii + n * jj) * ND3_NH2 + h] = 0.0;
    }
}

// alpha_maps: 3·n·n (LU form, patch sums over the lm×ln grid) or NULL (scalar alpha3, Cholesky form, `refine` steps).
// smem_limit: shared memory the 16-column LU panels may take (beyond it: 8 columns); large_limit: levels whose kernels
// would take more go to the large-front variants (< 0: none); csize: CTAs per front of ≥ 64 unknowns; zero_row ≥ 0: that
// row of the stencil is zeroed before the factorisation.
// stats_out (8 doubles or NULL): relres, breakdown flag, levels, levels on 8-column steps, levels on the large-front
// factorisation, levels on the large-front solves, backward-error test passed (LU form), largest front (pixels)
extern "C" int emu_nd_lu_gradient_reg(int n, const double *u, const double *ubar, const double *alpha3, const double *alpha_maps,
                                      int lm, int ln, double gamma, int refine, int leaf, int use_small, int csize,
                                      long long smem_limit, long long large_limit, int zero_row, double *out, double *stats_out,
                                      double *p_out)
{
    const int N = n * n, nops = 3;
    const bool lu = alpha_maps != nullptr;
    const int ng = lu ? lm * ln : 1;
    NdSymbolic sym;
    sym.build(n, ND3_W, leaf);
    const int nf = (int)sym.fronts.size(), nsteps = sym.nsteps();
    const size_t posg_len = sym.pixlist.size() + nf;

    std::vector<double> pix((size_t)LU_PLANES * N, 0.0), ast((size_t)(lu ? ND3_NH2 : ND3_NH) * N, 0.0);
    std::vector<int> posg(posg_len, 0);
    std::vector<long long> foff((size_t)4 * nf, 0), totals(4, 0);
    int info[4] = {0, 0, 0, 0};
    double rstate[2] = {0.0, 0.0};
    LuSlots ws;
    ws.ab = nullptr; ws.ab_stride = 0; ws.pix = pix.data(); ws.pix_stride = pix.size(); ws.info = info;
    ws.n = n; ws.N = N; ws.bw = 0; ws.bwx = 0; ws.LD = 0; ws.use_pin = 0; ws.nops = nops;
    Lu3Params pr;
    for (int k = 0; k < 3; ++k) pr.alpha[k] = alpha3 ? alpha3[k] : 0.0;
    pr.gamma = gamma; pr.lm = lu ? lm : 1; pr.ln = lu ? ln : 1; pr.refine = lu ? 3 : 0;

    NdDev nd;
    nd.n = n; nd.N = N; nd.W = ND3_W; nd.nnb = sym.nnb; nd.nh = nd_nh(ND3_W); nd.mb = 1; nd.nfronts = nf; nd.nsteps = nsteps;
    nd.fronts = sym.fronts.data(); nd.pixlist = sym.pixlist.data(); nd.nbr = sym.nbr.data(); nd.cmap = sym.cmap.data();
    nd.step_start = sym.step_start.data();
    nd.off = nullptr; nd.off_stride = 0;
    nd.posg = posg.data(); nd.posg_stride = 0; nd.foff = foff.data(); nd.foff_stride = 0; nd.totals = totals.data();
    nd.ast = ast.data(); nd.ast_stride = 0; nd.info = info;

    const int chunks = std::max(1, std::min(4, (N + 255) / 256));
    emu::launch(dim3(1, chunks), 256, [&] { lu3_classify_kernel<double>(ws, gamma, u, ubar, 0); });
    if (lu) emu::launch(dim3(1, chunks), 256, [&] { nd3_stencil_map_kernel<double>(ws, pr, alpha_maps, ast.data(), 0); });
    else emu::launch(dim3(1, chunks), 256, [&] { nd3_stencil_kernel(ws, pr, ast.data(), 0); });
    if (zero_row >= 0 && lu) emu_zero_row(ast, n, zero_row);
    emu::launch(dim3((nf + 7) / 8, 1), 256, [&] { nd_dims_kernel(nd); });
    emu::launch(dim3(1), 256, [&] { nd_scan_kernel(nd); });
    const size_t Ls = ((size_t)totals[0] + 1) & ~(size_t)1;
    std::vector<double> Lp((lu ? 2 : 1) * Ls + 2, 0.0), U0((size_t)totals[1] + 2, 0.0),
        U1((size_t)totals[1] + 2, 0.0), UV0((size_t)totals[2] + 2, 0.0), UV1((size_t)totals[2] + 2, 0.0);
    auto al16 = [](std::vector<double> &v) { double *p = v.data(); return (reinterpret_cast<std::uintptr_t>(p) & 15) ? p + 1 : p; };
    nd.L = al16(Lp); nd.U[0] = al16(U0); nd.U[1] = al16(U1); nd.UV[0] = al16(UV0); nd.UV[1] = al16(UV1);
    nd.L_stride = nd.U_stride = nd.UV_stride = 0;
    if (lu) nd.L_stride = 2 * Ls;          // one slot: L, then Uᵀ (nd_lu_factor_body)

    std::vector<NdLevelPlan> plan(nsteps);
    int levels8 = 0, nlarge_f = 0, nlarge_s = 0;
    size_t scr_len = 0;
    for (int s = 0; s < nsteps; ++s) {
        NdLevelPlan &lp = plan[s];
        lp = nd_level_plan(sym, s, 1, 1.0);
        if (!use_small && lp.small) {
            lp.small = false;
            lp.smem_f = nd_factor_smem(lp.nFw, lp.nRc);
            lp.smem_s = nd_solve_smem(lp.nFw);
        }
        if (lu) nd_level_lu(lp, (size_t)smem_limit);
        if (large_limit >= 0) nd_level_large(lp, (size_t)large_limit, SIZE_MAX, true);
        levels8 += lp.nb != ND_NB;
        nlarge_f += lp.large_f;
        nlarge_s += lp.large_s && !lp.small;
        NdLevelPlan g = lp;
        g.small = false;
        scr_len = std::max(scr_len, nd_level_scratch(g, csize > 1 && lp.nFw >= 64 ? csize : 1));
    }
    std::vector<double> scr(scr_len + 2, 0.0);
    nd.scr = al16(scr); nd.scr_stride = 0;

    for (int s = 0; s < nsteps; ++s) {
        const NdLevelPlan &lp = plan[s];
        if (lp.small && !lp.lu) {
            emu::launch(dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, 1), 32 * ND_SMALL_WARPS,
                        [&] { nd_factor_small_kernel(nd, lp.t0, lp.nfr, s & 1, 0.0, lp.arena_f); }, lp.smem_f / 8 + 2);
            continue;
        }
        const bool cl = csize > 1 && lp.nFw >= 64;
        const int C = cl ? csize : 1;
        emu::launch(dim3(lp.nfr * C, 1), lp.threads_f, [&] {
            const int t0 = lp.t0, par = s & 1, nF = lp.nFw;
            NdFactorKernelFn k = nullptr;
            if (lp.lu) {
                if (lp.large_f) k = lp.nb != ND_NB ? (cl ? nd_lu_factor8_large_cluster_kernel : nd_lu_factor8_large_kernel)
                                                   : (cl ? nd_lu_factor_large_cluster_kernel : nd_lu_factor_large_kernel);
                else k = lp.nb != ND_NB ? (cl ? nd_lu_factor8_cluster_kernel : nd_lu_factor8_kernel)
                                        : (cl ? nd_lu_factor_cluster_kernel : nd_lu_factor_kernel);
            } else {
                if (lp.large_f) k = cl ? nd_factor_large_cluster_kernel : nd_factor_large_kernel;
                else k = cl ? nd_factor_cluster_kernel : nd_factor_kernel;
            }
            k(nd, t0, par, 0.0, nF);
        }, nd_level_smem_f(lp) / 8 + 2, C);
    }
    NdDev ndb = nd;
    if (lu) ndb.L += Ls;
    auto solve = [&](double *v) {
        for (int s = 0; s < nsteps; ++s) {
            const NdLevelPlan &lp = plan[s];
            if (lp.small)
                emu::launch(dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, 1), 32 * ND_SMALL_WARPS,
                            [&] { nd_fwd_small_kernel(nd, lp.t0, lp.nfr, s & 1, v, 0, lp.arena_s); }, lp.smem_s / 8 + 2);
            else
                emu::launch(dim3(lp.nfr, 1), lp.threads_s, [&] {
                    if (lp.large_s) nd_fwd_large_kernel(nd, lp.t0, s & 1, v, 0, lp.nFw); else nd_fwd_kernel(nd, lp.t0, s & 1, v, 0);
                }, nd_level_smem_s(lp) / 8 + 2);
        }
        for (int s = nsteps - 1; s >= 0; --s) {
            const NdLevelPlan &lp = plan[s];
            if (lp.small)
                emu::launch(dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, 1), 32 * ND_SMALL_WARPS,
                            [&] { nd_bwd_small_kernel(ndb, lp.t0, lp.nfr, v, 0, lp.arena_s); }, lp.smem_s / 8 + 2);
            else
                emu::launch(dim3(lp.nfr, 1), lp.threads_s, [&] {
                    if (lp.large_s) nd_bwd_large_kernel(ndb, lp.t0, v, 0, lp.nFw); else nd_bwd_kernel(ndb, lp.t0, v, 0);
                }, nd_level_smem_s(lp) / 8 + 2);
        }
    };
    double relres = -1.0;
    double *p = pix.data() + (size_t)LU_PL_P * N, *work = pix.data() + (size_t)LU_PL_WORK * N;
    const int steps = lu ? pr.refine : refine;
    double *rs = lu ? rstate : nullptr;
    solve(p);
    emu::launch(dim3(1), 512, [&] { nd3_residual_kernel<double>(ws, pr, &relres, 0, alpha_maps, rs, 0); });
    for (int it = 0; it < steps; ++it) {
        solve(work);
        emu::launch(dim3(1, chunks), 256, [&] { nd3_axpy_kernel(ws, rs); });
        emu::launch(dim3(1), 512, [&] { nd3_residual_kernel<double>(ws, pr, &relres, 0, alpha_maps, rs, it + 1); });
    }
    std::vector<double> out_img((size_t)nops * ng, 0.0);
    double fin = relres;
    emu::launch(dim3(1), 512, [&] { nd3_finish_kernel<double>(ws, pr, info, lu ? 1e-11 : 1e300, out_img.data(), &fin, 0, alpha_maps); });
    std::memcpy(out, out_img.data(), out_img.size() * sizeof(double));
    if (p_out) std::memcpy(p_out, p, N * sizeof(double));
    if (stats_out) {
        stats_out[0] = lu ? relres : fin; stats_out[1] = info[1]; stats_out[2] = nsteps; stats_out[3] = levels8;
        stats_out[4] = nlarge_f; stats_out[5] = nlarge_s; stats_out[6] = std::isfinite(out_img[0]) ? 1 : 0;
        stats_out[7] = sym.max_front_pix;
    }
    return 0;
}
