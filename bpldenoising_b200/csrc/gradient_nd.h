// gradient_nd.h — interface of the nested-dissection adjoint solver's translation unit (gradient_nd.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace bpltv {

struct NdWork;      // plan, workspaces and pools of one device (gradient_nd.cuh)

// gradient (regularised = false) / gradient_reg (true) of /root/reference/src/TVLearningFunctionVec.jl:72-254 for a
// stack of O images on the device; u, ubar, alpha_map are device pointers of the context's precision (prec = 64 | 32)
struct NdProblem {
    const void *u, *ubar;
    int prec;
    int M, N, O;
    double alpha_s;
    const void *alpha_map;      // M·N map of the patch parameter, or nullptr
    int lm, ln;
    bool regularised;
    double gamma, act_tol, eps_act;
    double tol;                 // backward error above which the result is poisoned with NaN (≤ 0: never)
    int maxit;                  // refinement steps (≤ 0: default)
    bool large_fronts;          // fronts beyond shared memory take the large-front variants instead of returning -1
};

// sumregs_gradient_reg of /root/reference/src/SumRegsLearningFunction.jl for a stack of O images on the device (three
// difference operators, node space, coupling radius 2): scalar (:112-167, symmetric: Cholesky of the fronts) or patch
// (:195-262, alpha_maps: rows scaled by a different map per operator, LU of the fronts, refined and checked as the band
// LU does — tol and maxit are not used then)
struct Nd3Problem {
    const void *u, *ubar;
    int prec;
    int M, N, O;
    double alpha[3];
    double gamma;
    double tol;                 // backward error above which the result is poisoned with NaN (≤ 0: never)
    int maxit;                  // refinement steps (≤ 0: default)
    bool large_fronts;          // fronts beyond shared memory take the large-front variants instead of returning -1
    const void *alpha_maps = nullptr;     // 3 maps of M·N (patch) or nullptr (scalar: alpha[3])
    int lm = 1, ln = 1;                   // the patch grid
};

// sumregs_gradient (non-regularised; scalar :264-327, patch :330-407) in multiplier space: 3-6 unknowns per pixel,
// coupling radius 2.  alpha_maps: 3 maps of M·N (patch) or nullptr (scalar: alpha[3]).
struct Nd3mProblem {
    const void *u, *ubar, *alpha_maps;
    int prec;
    int M, N, O;
    double alpha[3];
    int lm, ln;
    double act_tol, eps_act;
    double tol;                 // relative residual above which the result is poisoned with NaN (≤ 0: never)
    int maxit;                  // refinement steps (≤ 0: default)
    bool large_fronts;          // fronts beyond shared memory take the large-front variants instead of returning -1
};

NdWork *nd_work_create();
void nd_work_destroy(NdWork *w);
const char *nd_work_error(const NdWork *w);
size_t nd_work_bytes_per_image(const NdWork *w);
const double *nd_work_relres_max(const NdWork *w);      // device pointer: worst backward error of the last call
// 0 ok; -1: the shape is not taken (fronts beyond shared memory and large_fronts not set) — use the band solver; other
// negatives: bpltv_status (BPLTV_ERR_ALLOC: the workspace of one image does not fit; the message names its size)
int nd_run_gradient(NdWork *w, const NdProblem &gp, int sm_count, size_t smem_optin, cudaStream_t st, double *d_grad_out,
                    long long *launches);
// d_grad_out: 3·lm·ln doubles, [operator][patch] (3 for the scalar parameter).  Use a workspace of its own (the plan is
// keyed by the coupling radius).
int nd_run_gradient3_reg(NdWork *w, const Nd3Problem &gp, int sm_count, size_t smem_optin, cudaStream_t st, double *d_grad_out,
                         long long *launches);

// d_grad_out: 3·lm·ln doubles, [operator][patch].  Shares the workspace of nd_run_gradient3_reg (same tree).
int nd_run_gradient3(NdWork *w, const Nd3mProblem &gp, int sm_count, size_t smem_optin, cudaStream_t st, double *d_grad_out,
                     long long *launches);

}  // namespace bpltv
