// emu_nd_large.cpp — TEST INFRASTRUCTURE: runs the sum-of-regularisers paths of gradient_nd.cuh (scalar
// sumregs_gradient_reg in node space, run_gradient3_nd_reg; sumregs_gradient in multiplier space, run_gradient3_nd_mult)
// for ONE image on the CPU thread emulation (emu_cuda.h), as emu_nd3.cpp does, and in addition sends every level whose
// shared-memory front kernels would take more than `large_limit` bytes to the large-front variants of nd_solver.cuh
// (panel / front vector in global memory), as nd_level_large does on the device.  Built by tests/test_emu_nd_large.py
// with g++ -std=c++20 -DBPLTV_EMU; never shipped.
#include "emu_cuda.h"

#include <climits>
#include <cstring>

#include "../../bpldenoising_b200/csrc/nd_sumregs.cuh"

using namespace bpltv;

// the levels whose kernels would take more than large_limit bytes of shared memory (< 0: none) go to the large-front
// variants; returns the scratch they need (doubles), with C CTAs per front on the levels the cluster kernels take
static size_t emu_large_levels(std::vector<NdLevelPlan> &plan, long long large_limit, int csize, int &nlarge_f, int &nlarge_s)
{
    size_t scr = 0;
    nlarge_f = nlarge_s = 0;
    for (NdLevelPlan &lp : plan) {
        if (large_limit >= 0) nd_level_large(lp, (size_t)large_limit, SIZE_MAX, true);
        nlarge_f += lp.large_f && !lp.small;
        nlarge_s += lp.large_s && !lp.small;
        if (!lp.small) scr = std::max(scr, nd_level_scratch(lp, csize > 1 && lp.nFw >= 64 ? csize : 1));
    }
    return scr;
}

// one level of the generic factorisation, alone or shared by csize CTAs (fronts of ≥ 64 unknowns)
static void emu_factor_level(const NdDev &nd, const NdLevelPlan &lp, int s, double guard, int csize)
{
    const bool cl = csize > 1 && lp.nFw >= 64;
    const int C = cl ? csize : 1;
    emu::launch(dim3(lp.nfr * C, 1), lp.threads_f, [&] {
        const int t0 = lp.t0, par = s & 1, nF = lp.nFw;
        if (lp.large_f) {
            if (lp.nb != ND_NB) { if (cl) nd_factor8_large_cluster_kernel(nd, t0, par, guard, nF); else nd_factor8_large_kernel(nd, t0, par, guard, nF); }
            else { if (cl) nd_factor_large_cluster_kernel(nd, t0, par, guard, nF); else nd_factor_large_kernel(nd, t0, par, guard, nF); }
        } else {
            if (lp.nb != ND_NB) { if (cl) nd_factor8_cluster_kernel(nd, t0, par, guard, nF); else nd_factor8_kernel(nd, t0, par, guard, nF); }
            else { if (cl) nd_factor_cluster_kernel(nd, t0, par, guard, nF); else nd_factor_kernel(nd, t0, par, guard, nF); }
        }
    }, lp.smem_f / 8 + 2, C);
}

static void emu_fwd_level(const NdDev &nd, const NdLevelPlan &lp, int s, double *v)
{
    emu::launch(dim3(lp.nfr, 1), lp.threads_s, [&] {
        if (lp.large_s) nd_fwd_large_kernel(nd, lp.t0, s & 1, v, 0, lp.nFw); else nd_fwd_kernel(nd, lp.t0, s & 1, v, 0);
    }, lp.smem_s / 8 + 2);
}
static void emu_bwd_level(const NdDev &nd, const NdLevelPlan &lp, double *v)
{
    emu::launch(dim3(lp.nfr, 1), lp.threads_s, [&] {
        if (lp.large_s) nd_bwd_large_kernel(nd, lp.t0, v, 0, lp.nFw); else nd_bwd_kernel(nd, lp.t0, v, 0);
    }, lp.smem_s / 8 + 2);
}

// stats_out (8 doubles or NULL): backward error, vanished-pivot flag, L doubles, fronts, levels, largest front (pixels),
// levels on the large-front factorisation, levels on the large-front solves.  csize: CTAs per front (≥ 64 unknowns).
extern "C" int emu_nd_large_gradient_reg(int n, const double *u, const double *ubar, const double *alpha3, double gamma,
                                       int refine, int leaf, int use_small, int csize, long long large_limit, double *out,
                                       double *stats_out, double *p_out, double *ast_out)
{
    const int N = n * n, nops = 3;
    NdSymbolic sym;
    sym.build(n, ND3_W, leaf);
    const int nf = (int)sym.fronts.size(), nsteps = sym.nsteps();
    const size_t posg_len = sym.pixlist.size() + nf;

    std::vector<double> pix((size_t)LU_PLANES * N, 0.0), ast((size_t)ND3_NH * N, 0.0);
    std::vector<int> posg(posg_len, 0);
    std::vector<long long> foff((size_t)4 * nf, 0), totals(4, 0);
    int info[4] = {0, 0, 0, 0};
    LuSlots ws;
    ws.ab = nullptr; ws.ab_stride = 0; ws.pix = pix.data(); ws.pix_stride = pix.size(); ws.info = info;
    ws.n = n; ws.N = N; ws.bw = 0; ws.bwx = 0; ws.LD = 0; ws.use_pin = 0; ws.nops = nops;
    Lu3Params pr;
    for (int k = 0; k < 3; ++k) pr.alpha[k] = alpha3[k];
    pr.gamma = gamma; pr.lm = 1; pr.ln = 1; pr.refine = 0;

    NdDev nd;
    nd.n = n; nd.N = N; nd.W = ND3_W; nd.nnb = sym.nnb; nd.nh = nd_nh(ND3_W); nd.mb = 1; nd.nfronts = nf; nd.nsteps = nsteps;
    nd.fronts = sym.fronts.data(); nd.pixlist = sym.pixlist.data(); nd.nbr = sym.nbr.data(); nd.cmap = sym.cmap.data();
    nd.step_start = sym.step_start.data();
    nd.off = nullptr; nd.off_stride = 0;
    nd.posg = posg.data(); nd.posg_stride = 0; nd.foff = foff.data(); nd.foff_stride = 0; nd.totals = totals.data();
    nd.ast = ast.data(); nd.ast_stride = 0; nd.info = info;

    const int chunks = std::max(1, std::min(4, (N + 255) / 256));
    emu::launch(dim3(1, chunks), 256, [&] { lu3_classify_kernel<double>(ws, gamma, u, ubar, 0); });
    emu::launch(dim3(1, chunks), 256, [&] { nd3_stencil_kernel(ws, pr, ast.data(), 0); });
    if (ast_out) std::memcpy(ast_out, ast.data(), ast.size() * sizeof(double));
    emu::launch(dim3((nf + 7) / 8, 1), 256, [&] { nd_dims_kernel(nd); });
    emu::launch(dim3(1), 256, [&] { nd_scan_kernel(nd); });
    std::vector<double> Lp((size_t)totals[0] + 2, 0.0), U0((size_t)totals[1] + 2, 0.0), U1((size_t)totals[1] + 2, 0.0),
        UV0((size_t)totals[2] + 2, 0.0), UV1((size_t)totals[2] + 2, 0.0);
    auto al16 = [](std::vector<double> &v) { double *p = v.data(); return (reinterpret_cast<std::uintptr_t>(p) & 15) ? p + 1 : p; };
    nd.L = al16(Lp); nd.U[0] = al16(U0); nd.U[1] = al16(U1); nd.UV[0] = al16(UV0); nd.UV[1] = al16(UV1);
    nd.L_stride = nd.U_stride = nd.UV_stride = 0;

    std::vector<NdLevelPlan> plan(nsteps);
    for (int s = 0; s < nsteps; ++s) {
        plan[s] = nd_level_plan(sym, s, 1, 1.0);
        if (!use_small && plan[s].small) {
            plan[s].small = false;
            plan[s].smem_f = nd_factor_smem(plan[s].nFw, s > 0 ? sym.step_max_ring_pix[s - 1] : 0);
            plan[s].smem_s = nd_solve_smem(plan[s].nFw);
        }
    }
    int nlarge_f = 0, nlarge_s = 0;
    std::vector<double> scr(emu_large_levels(plan, large_limit, csize, nlarge_f, nlarge_s) + 2, 0.0);
    nd.scr = al16(scr); nd.scr_stride = 0;
    for (int s = 0; s < nsteps; ++s) {
        const NdLevelPlan &lp = plan[s];
        if (lp.small)
            emu::launch(dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, 1), 32 * ND_SMALL_WARPS,
                        [&] { nd_factor_small_kernel(nd, lp.t0, lp.nfr, s & 1, 0.0, lp.arena_f); }, lp.smem_f / 8 + 2);
        else
            emu_factor_level(nd, lp, s, 0.0, csize);
    }
    auto solve = [&](double *v) {
        for (int s = 0; s < nsteps; ++s) {
            const NdLevelPlan &lp = plan[s];
            if (lp.small)
                emu::launch(dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, 1), 32 * ND_SMALL_WARPS,
                            [&] { nd_fwd_small_kernel(nd, lp.t0, lp.nfr, s & 1, v, 0, lp.arena_s); }, lp.smem_s / 8 + 2);
            else
                emu_fwd_level(nd, lp, s, v);
        }
        for (int s = nsteps - 1; s >= 0; --s) {
            const NdLevelPlan &lp = plan[s];
            if (lp.small)
                emu::launch(dim3((lp.nfr + ND_SMALL_WARPS - 1) / ND_SMALL_WARPS, 1), 32 * ND_SMALL_WARPS,
                            [&] { nd_bwd_small_kernel(nd, lp.t0, lp.nfr, v, 0, lp.arena_s); }, lp.smem_s / 8 + 2);
            else
                emu_bwd_level(nd, lp, v);
        }
    };
    double relres = -1.0;
    double *p = pix.data() + (size_t)LU_PL_P * N, *work = pix.data() + (size_t)LU_PL_WORK * N;
    solve(p);
    emu::launch(dim3(1), 512, [&] { nd3_residual_kernel<double>(ws, pr, &relres, 0); });
    for (int it = 0; it < refine; ++it) {
        solve(work);
        emu::launch(dim3(1, chunks), 256, [&] { nd3_axpy_kernel(ws); });
        emu::launch(dim3(1), 512, [&] { nd3_residual_kernel<double>(ws, pr, &relres, 0); });
    }
    std::vector<double> out_img(nops, 0.0);
    emu::launch(dim3(1), 512, [&] { nd3_finish_kernel(ws, pr, info, 1e300, out_img.data(), &relres, 0); });
    std::memcpy(out, out_img.data(), nops * sizeof(double));
    if (p_out) std::memcpy(p_out, p, N * sizeof(double));
    if (stats_out) {
        stats_out[0] = relres; stats_out[1] = info[1]; stats_out[2] = (double)totals[0]; stats_out[3] = nf;
        stats_out[4] = nsteps; stats_out[5] = sym.max_front_pix; stats_out[6] = nlarge_f; stats_out[7] = nlarge_s;
    }
    return 0;
}


// sumregs_gradient (non-regularised) in multiplier space, the launch order of run_gradient3_nd_mult.  alpha_maps: 3·n·n or NULL.
// stats_out (8 doubles or NULL): relres, guarded pivots, breakdown flag, modes, largest front (unknowns), levels on 8-column
// steps, levels on the large-front factorisation, levels on the large-front solves
extern "C" int emu_nd_large_gradient_mult(int n, const double *u, const double *ubar, const double *alpha3, const double *alpha_maps,
                                        int lm, int ln, double act_tol, double eps_act, int refine, int leaf, int csize,
                                        long long smem_limit, long long large_limit, double *out, double *stats_out, double *p_out)
{
    const int N = n * n, mb = ND3M_MB, ng = lm * ln;
    NdSymbolic sym;
    sym.build(n, ND3_W, leaf);
    const int nf = (int)sym.fronts.size(), nsteps = sym.nsteps();
    const size_t posg_len = sym.pixlist.size() + nf;
    std::vector<double> pix((size_t)ND3M_PLANES * N, 0.0), ast((size_t)ND3_NH * mb * mb * N, 0.0), vec((size_t)3 * mb * N, 0.0);
    std::vector<int> off3((size_t)3 * N + 1, 0), poff(N + 2, 0), posg(posg_len, 0), lvl(128, 0);
    std::vector<long long> foff((size_t)4 * nf, 0), totals(4, 0);
    int info[4] = {0, 0, 0, 0};
    Nd3mSlots ws;
    ws.n = n; ws.N = N; ws.pix = pix.data(); ws.pix_stride = pix.size(); ws.off3 = off3.data(); ws.off3_stride = off3.size();
    ws.poff = poff.data(); ws.poff_stride = poff.size(); ws.vec = vec.data(); ws.vec_stride = vec.size(); ws.info = info;
    Nd3mVariant gv;
    gv.patch = alpha_maps != nullptr; gv.lm = lm; gv.ln = ln;
    for (int k = 0; k < 3; ++k) gv.alpha[k] = alpha3 ? alpha3[k] : 0.0;
    gv.act_tol = act_tol; gv.eps_act = eps_act; gv.relres_tol = 1e300;
    NdDev nd;
    nd.n = n; nd.N = N; nd.W = ND3_W; nd.nnb = sym.nnb; nd.nh = nd_nh(ND3_W); nd.mb = mb; nd.nfronts = nf; nd.nsteps = nsteps;
    nd.fronts = sym.fronts.data(); nd.pixlist = sym.pixlist.data(); nd.nbr = sym.nbr.data(); nd.cmap = sym.cmap.data();
    nd.step_start = sym.step_start.data();
    nd.off = poff.data(); nd.off_stride = 0;
    nd.posg = posg.data(); nd.posg_stride = 0; nd.foff = foff.data(); nd.foff_stride = 0; nd.totals = totals.data();
    nd.ast = ast.data(); nd.ast_stride = 0; nd.info = info;

    const int chunks = std::max(1, std::min(4, (N + 255) / 256));
    emu::launch(dim3(1), 512, [&] { nd3m_classify_kernel<double>(ws, gv, u, ubar, alpha_maps, 0); });
    emu::launch(dim3((nf + 7) / 8, 1), 256, [&] { nd_dims_kernel(nd); });
    emu::launch(dim3(1), 256, [&] { nd_scan_kernel(nd); });
    emu::launch(dim3((nf + 255) / 256, 1), 256, [&] { nd_level_sizes_kernel(nd, lvl.data()); });
    emu::launch(dim3(1, 8), 256, [&] { nd3m_stencil_kernel(ws, ast.data(), 0); });
    std::vector<double> Lp((size_t)totals[0] + 2, 0.0), U0((size_t)totals[1] + 2, 0.0), U1((size_t)totals[1] + 2, 0.0),
        UV0((size_t)totals[2] + 2, 0.0), UV1((size_t)totals[2] + 2, 0.0);
    auto al16 = [](std::vector<double> &v) { double *p = v.data(); return (reinterpret_cast<std::uintptr_t>(p) & 15) ? p + 1 : p; };
    nd.L = al16(Lp); nd.U[0] = al16(U0); nd.U[1] = al16(U1); nd.UV[0] = al16(UV0); nd.UV[1] = al16(UV1);
    nd.L_stride = nd.U_stride = nd.UV_stride = 0;
    std::vector<NdLevelPlan> plan(nsteps);
    int maxF = 0, levels8 = 0;
    for (int s = 0; s < nsteps; ++s) {
        // smem_limit: bytes of shared memory the plan may use for the 16-column panel (a small value sends fronts to the
        // 8-column kernels)
        plan[s] = nd_level_plan_sized(sym, s, lvl[2 * s], s > 0 ? lvl[2 * (s - 1) + 1] : 0, (size_t)smem_limit, 4, 128);
        maxF = std::max(maxF, lvl[2 * s]);
    }
    int nlarge_f = 0, nlarge_s = 0;
    std::vector<double> scr(emu_large_levels(plan, large_limit, csize, nlarge_f, nlarge_s) + 2, 0.0);
    nd.scr = al16(scr); nd.scr_stride = 0;
    for (int s = 0; s < nsteps; ++s) {
        if (plan[s].nb != ND_NB) ++levels8;
        emu_factor_level(nd, plan[s], s, 1e-13, csize);
    }
    auto solve = [&](double *v) {
        for (int s = 0; s < nsteps; ++s) emu_fwd_level(nd, plan[s], s, v);
        for (int s = nsteps - 1; s >= 0; --s) emu_bwd_level(nd, plan[s], v);
    };
    double relres = -1.0;
    double *zeta = vec.data() + (size_t)mb * N, *work = vec.data() + (size_t)2 * mb * N;
    emu::launch(dim3(1, chunks), 256, [&] { nd3m_axpy_kernel(ws, 1, 0, 0); });
    solve(zeta);
    emu::launch(dim3(1), 512, [&] { nd3m_residual_kernel(ws, &relres, 0); });
    for (int it = 0; it < refine; ++it) {
        solve(work);
        emu::launch(dim3(1, chunks), 256, [&] { nd3m_axpy_kernel(ws, 1, 2, 1); });
        emu::launch(dim3(1), 512, [&] { nd3m_residual_kernel(ws, &relres, 0); });
    }
    std::vector<double> out_img((size_t)3 * ng, 0.0);
    emu::launch(dim3(1), 512, [&] { nd3m_finish_kernel(ws, gv, &relres, out_img.data(), 0); });
    std::memcpy(out, out_img.data(), out_img.size() * sizeof(double));
    if (p_out) std::memcpy(p_out, pix.data() + (size_t)16 * N, N * sizeof(double));
    if (stats_out) {
        stats_out[0] = relres; stats_out[1] = info[0]; stats_out[2] = info[1]; stats_out[3] = off3[3 * N]; stats_out[4] = maxF;
        stats_out[5] = levels8; stats_out[6] = nlarge_f; stats_out[7] = nlarge_s;
    }
    return 0;
}

