/* bpltv.h — C ABI of libbpltv.so: B200-native (sm_100a) TV-denoising solve and
 * λ-gradient for bilevel parameter learning.
 *
 * This is the drop-in boundary for ONE path of dvillacis/BPLDenoising: the
 * body of `tv_op_learning_function(x, data, Δ)` and of `denoise(data, x, op)`
 * (/root/reference/src/TVLearningFunctionVec.jl:14-27, :45-70), widened to its
 * direct callers: the λ-sweeps / validation solves of src/BPLDenoising.jl
 * (bpltv_sweep) and the sum-of-regularisers learning function of
 * src/SumRegsLearningFunction.jl (bpltv_sumregs_*).  Julia calls these entry
 * points with `ccall` (julia/BPLTV.jl; INTEGRATION.md); the trust-region
 * driver (/root/reference/src/TRBox.jl:192-273) is unchanged.
 *
 * Conventions
 *  - plain pointers and sizes only; every host array is caller-owned, is read
 *    or written during the call and never retained after return;
 *  - images are column-major M×N×O stacks of doubles (Julia `Array{Float64,3}`,
 *    /root/reference/src/TRBox.jl:28), row index fastest;
 *  - λ ("x", "α" in the reference) is an lm×ln column-major grid; lm=ln=1 is the
 *    scalar case (`x::Real`), anything else the patch case (`x::AbstractArray`,
 *    up-sampled block-constant to M×N like PatchOp, :57-60);
 *  - every function returns 0 on success or a negative bpltv_status; the text of
 *    the last error of the calling thread is `bpltv_last_error()`;
 *  - there is no CPU fallback: without a usable CUDA device `bpltv_create` fails.
 */
#ifndef BPLTV_H
#define BPLTV_H

#ifdef __cplusplus
extern "C" {
#endif

#define BPLTV_VERSION 100

typedef struct bpltv_ctx bpltv_ctx;

enum bpltv_status {
    BPLTV_OK = 0,
    BPLTV_ERR_ARG = -1,      /* bad argument (ArgumentError on the Julia side)   */
    BPLTV_ERR_CUDA = -2,     /* CUDA runtime / launch failure                    */
    BPLTV_ERR_NODEVICE = -3, /* no sm_100 device: the library refuses to run     */
    BPLTV_ERR_STATE = -4,    /* e.g. learn_eval before set_dataset               */
    BPLTV_ERR_NUMERIC = -5,  /* non-finite cost/gradient, solver breakdown       */
    BPLTV_ERR_ALLOC = -6
};

enum bpltv_arith {
    BPLTV_ARITH_STRICT = 0, /* one IEEE op per reference operator, no FMA: iterates
                               are bit-identical to the reference operation order */
    BPLTV_ARITH_FAST = 1    /* FMA, reciprocal step constants, rsqrt projection   */
};

enum bpltv_pdps_kernel {
    BPLTV_KERNEL_AUTO = 0,
    BPLTV_KERNEL_GENERIC = 1,  /* any size, one thread per pixel                  */
    BPLTV_KERNEL_MARCH = 2,    /* HBM-streaming column march, one iteration/launch */
    BPLTV_KERNEL_RESIDENT = 3, /* whole image on chip for all iterations           */
    BPLTV_KERNEL_TBLOCK = 4    /* temporally blocked streaming: T iterations per HBM
                                  pass, software-pipelined along the column march   */
};

/* Inner solver parameters = `denoising_default_params`
 * (/root/reference/src/TVLearningFunctionVec.jl:33-43) plus the switches of
 * docs/SEMANTICS.md.                                                            */
typedef struct bpltv_pdps_opts {
    double tau0;    /* τ₀ = 5                                        (:36) */
    double sigma0;  /* σ₀ = 0.99/5                                   (:37) */
    double rho;     /* ρ = 0                                         (:34) */
    double opnorm;  /* R_K = opnorm_estimate(FwdGradientOp) = √8 (S2)      */
    int accel;      /* accel = true                                  (:38) */
    int maxiter;    /* 5000 (:40); TVDenoise uses 10000 (BPLDenoising.jl:51) */
    int init_mode;  /* S3: 0 → x⁰ = 0 (default), 1 → x⁰ = f                 */
    int arith;      /* enum bpltv_arith                                     */
    int kernel;     /* enum bpltv_pdps_kernel                               */
    int tblock;     /* temporal blocking depth T of BPLTV_KERNEL_TBLOCK, 2..4
                       (0 = auto: 4; 2 for strict arithmetic in fp32 and for
                       strict fp64 stacks with few columns per CTA)             */
    int reserved[4];
} bpltv_pdps_opts;

/* Parameters of the upper-level evaluation (tv_op_learning_function, :14-27). */
typedef struct bpltv_eval_opts {
    bpltv_pdps_opts pdps;
    double delta_t;   /* Δt = 1e-6: Δ > Δt → gradient, else gradient_reg  (:14,:21) */
    double gamma;     /* γ = 1e8 Huber parameter of gradient_reg      (:142,:197) */
    double act_tol;   /* |∇u| < 1e-12 is "active" in gradient         (:109,:231) */
    double eps_act;   /* weight of the active rows: eps() scalar (:128),
                         sqrt(eps()) patch (:245); 0 → those defaults            */
    double solver_tol;   /* backward error of the adjoint solve (matrix-free residual after
                            refinement) above which the gradient is reported as
                            BPLTV_ERR_NUMERIC instead of returned; 1e-9; <= 0: never   */
    int solver_maxit;    /* steps of iterative refinement; 0 -> default (1)           */
    int solver;          /* 0 auto = 2; 2 nested-dissection multifrontal Cholesky (the
                            whole GPU per image); 1 the banded factorisations of round 1
                            (one SM per image), kept as a second implementation.  Sum of
                            regularisers: the symmetric variants (sumregs_gradient scalar
                            and patch, scalar sumregs_gradient_reg) follow this switch; the
                            row-scaled patch sumregs_gradient_reg takes the band LU, and
                            above 430² (where the band LU refuses) the LU of the
                            nested-dissection fronts; solver 1 keeps it on the band LU   */
    int force_branch;    /* 0: by Δ (reference); 1: gradient; 2: gradient_reg;
                            3: cost only (grad_out left zero; λ-sweeps, validation)  */
    int reserved0;
    double gamma_patch;  /* γ of the PATCH variant of sumregs_gradient_reg, 1e8
                            (SumRegsLearningFunction.jl:200; the scalar variant uses
                            `gamma` = 1e3, :117); 0 → `gamma`.  Unused by the TV path.  */
    int reserved[2];
} bpltv_eval_opts;

typedef struct bpltv_stats {
    double ms_upload, ms_pdps, ms_cost, ms_gradient, ms_download, ms_total;
    long long pdps_iterations;   /* of the last call                           */
    long long pixel_iterations;  /* M·N·O·iterations of the last call          */
    long long solver_iterations; /* reserved (0)                               */
    long long kernel_launches;   /* CUDA kernels launched by the last call     */
    double solver_max_relres;    /* worst residual of the adjoint solves over the images (host-pointer
                                    entry points).  Nested dissection (solver 0/2): the normwise
                                    backward error that solver_tol bounds (TV, scalar
                                    sumregs_gradient_reg) or the relative residual |r|/|b| of the
                                    multiplier system (sumregs_gradient).  Banded solvers (solver 1) and
                                    patch sumregs_gradient_reg (band LU or the fronts' LU): the relative
                                    residual |r|/|b| after the last refinement step — informational
                                    (with entries up to alpha*gamma it is not a backward error); both
                                    LUs apply their own backward-error test and poison the gradient
                                    with NaN                                                         */
    int pdps_kernel_used;        /* enum bpltv_pdps_kernel actually dispatched */
    int n_devices;
    int tblock_depth;            /* PDPS iterations per HBM pass of that kernel (1 unless TBLOCK) */
    int reserved[5];
} bpltv_stats;

void bpltv_default_pdps_opts(bpltv_pdps_opts *o);
void bpltv_default_eval_opts(bpltv_eval_opts *o);

/* Context: owns streams, device buffers and (after set_dataset) the resident
 * dataset on each listed device.  precision: 64 (reference arithmetic) or 32.
 * device_ids == NULL → device 0..ndev-1.  Images are sharded over the devices in
 * contiguous blocks along O (SURVEY §8e); partial costs/gradients are summed on
 * the host in device order (single process: no collective is needed).  A device
 * id may repeat, and each entry is its own shard: tests/test_gpu_sharded.py runs
 * the sharded path on one GPU with [0, 0].                                       */
int bpltv_create(const int *device_ids, int ndev, int precision, bpltv_ctx **out);
int bpltv_destroy(bpltv_ctx *ctx);

/* Replaces `ds = (ū, f)` of bilevel_learn (/root/reference/src/TRBox.jl:192;
 * data[1]=truth, data[2]=noisy: TVLearningFunctionVec.jl:15-16).  Uploaded once,
 * reused by every later learn_eval / denoise(noisy=NULL).                       */
int bpltv_set_dataset(bpltv_ctx *ctx, const double *truth, const double *noisy,
                      int M, int N, int O);

/* Replaces denoise(data, x, op) (TVLearningFunctionVec.jl:45-70) and
 * TVDenoise(data, parameter) (/root/reference/src/BPLDenoising.jl:41-82).
 * noisy == NULL → the resident dataset's noisy stack (M,N,O must then match).
 * u_out: M×N×O doubles.                                                         */
int bpltv_denoise(bpltv_ctx *ctx, const double *noisy, int M, int N, int O,
                  const double *lam, int lm, int ln, const bpltv_pdps_opts *opts,
                  double *u_out);

/* Replaces tv_op_learning_function(x, data, Δ; Δt) (TVLearningFunctionVec.jl:14-27)
 * on the resident dataset: u = denoise(f, x); cost = 0.5‖u-ū‖² (:20);
 * grad = Δ > Δt ? gradient : gradient_reg (:21-25), summed over images (:72-96,
 * :163-190).  u_out may be NULL; grad_out has lm×ln entries (same shape as x).  */
int bpltv_learn_eval(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                     const bpltv_eval_opts *opts, double *u_out, double *cost_out,
                     double *grad_out);

/* Gradient of a caller-supplied u (tests grade the adjoint solve on the oracle's
 * u, SURVEY §7.3-3): replaces gradient / gradient_reg (:72-96, :98-161, :163-254).
 * u: M×N×O doubles, same shape as the resident dataset.                          */
int bpltv_gradient(bpltv_ctx *ctx, const double *u, const double *lam, int lm, int ln,
                   int regularised, const bpltv_eval_opts *opts, double *grad_out);

/* λ-sweep on the resident dataset: replaces the loops `for i: u = denoise_function(data,
 * parameter_range[i]); costs[i] = cost_function(u, true_)` of generate_cost / generate_2d_cost
 * (/root/reference/src/BPLDenoising.jl:92-111, :136-158; the reference passes TVDenoise, i.e.
 * opts->maxiter = 10000, :51).  All L parameter sets × O images are solved as ONE batch of
 * independent problems.  lams: L consecutive lm×ln column-major grids (lm = ln = 1: scalars).
 * cost_out[l] = 0.5‖u_l - ū‖² over the whole stack (L2CostFunction, :84-86);
 * sqerr_out (may be NULL): O×L, ‖u_l[:,:,o] - ū[:,:,o]‖² per image (PSNR of validate_tv_parameter,
 * :381-415); u_out (may be NULL): M×N×O×L.                                                        */
int bpltv_sweep(bpltv_ctx *ctx, const double *lams, int L, int lm, int ln,
                const bpltv_pdps_opts *opts, double *cost_out, double *sqerr_out, double *u_out);

/* ---- sum-of-regularisers interface (/root/reference/src/SumRegsLearningFunction.jl) ----------
 * Three TV-type regularisers: forward, backward and centred differences (op₁, op₂, op₃, :9-11).
 * λ is a 3-vector (lm = ln = 1; `x::AbstractVector{Float64}`, :8) or an lm×ln×3 column-major array
 * (`x::AbstractArray{T,3}`, :22), each layer up-sampled like PatchOp.  Semantics of the un-vendored
 * operators and solver: docs/SEMANTICS.md S10-S13.                                             */

/* bpltv_default_eval_opts with the sum-of-regularisers constants: pdps.opnorm = √18 (S12),
 * Δt = 1e-3 (:8), γ = 1e3 (:117).                                                             */
void bpltv_default_sumregs_eval_opts(bpltv_eval_opts *o);

/* Replaces sumregs_denoise(data, x, op₁, op₂, op₃[, pOp]) (:38-85).  opts == NULL → the defaults
 * above.  noisy == NULL → the resident dataset's noisy stack.                                  */
int bpltv_sumregs_denoise(bpltv_ctx *ctx, const double *noisy, int M, int N, int O,
                          const double *lam, int lm, int ln, const bpltv_pdps_opts *opts,
                          double *u_out);

/* Replaces sumregs_learning_function(x, data, Δ; Δt=1e-3) (:8-36) on the resident dataset:
 * u = sumregs_denoise(f, x); cost = 0.5‖u-ū‖²; grad = Δ > Δt ? sumregs_gradient (:264-327, :330-407)
 * : sumregs_gradient_reg (:112-167), summed over images (:87-110, :169-193).  grad_out has the shape
 * of x: 3 (lm = ln = 1) or lm×ln×3 entries.  The patch variant of sumregs_gradient_reg (:195-262),
 * whose system is row-scaled by a different λ-map per operator and therefore not symmetric, is
 * solved by a banded LU in node space (γ = opts->gamma_patch) up to M = N ≤ 430 and by an LU of the
 * nested-dissection fronts beyond.  Every variant takes any square size: where the fronts of the
 * nested-dissection solver outgrow shared memory and the band solvers refuse the size too, its
 * large-front kernels (panels and front vector in global memory) take over; an
 * image whose workspace does not fit in device memory returns BPLTV_ERR_ALLOC, and
 * bpltv_last_error names the gigabytes one image needs.  opts == NULL → the
 * sum-of-regularisers defaults.                                                              */
int bpltv_sumregs_learn_eval(bpltv_ctx *ctx, const double *lam, int lm, int ln, double Delta,
                             const bpltv_eval_opts *opts, double *u_out, double *cost_out,
                             double *grad_out);

/* Gradient of a caller-supplied u (the tests grade the adjoint solve on the oracle's u).     */
int bpltv_sumregs_gradient(bpltv_ctx *ctx, const double *u, const double *lam, int lm, int ln,
                           int regularised, const bpltv_eval_opts *opts, double *grad_out);

/* Device-resident variants (single-device contexts only): pointers are device
 * memory of the context's precision (double or float), `stream` a cudaStream_t
 * (NULL → the context's stream).  All work is enqueued on `stream` and the call
 * returns without waiting for it, with these exceptions a caller overlapping
 * other streams should know: (1) the first call with a given shape / option set
 * allocates workspaces (cudaMalloc / cudaFree synchronise the device) and uploads
 * the step-size table (one stream synchronisation); later calls reuse both;
 * (2) the non-regularised gradient (Δ > Δt) synchronises `stream` once per wave of
 * ≤ 256 images, after the pixel classification, to size its factor pools (the
 * number of unknowns is data dependent; one 32-byte read per image).  The loss-only
 * and the regularised evaluations have no such point.
 * d_costgrad: 1 + lm·ln doubles = [cost, grad...] (what one NCCL all-reduce sums
 * across ranks, SURVEY §8e).  d_u_out may be NULL for learn_eval_device.        */
int bpltv_denoise_device(bpltv_ctx *ctx, const void *d_noisy, int M, int N, int O,
                         const double *lam, int lm, int ln, const bpltv_pdps_opts *opts,
                         void *d_u_out, void *stream);
int bpltv_set_dataset_device(bpltv_ctx *ctx, const void *d_truth, const void *d_noisy,
                             int M, int N, int O, void *stream);
int bpltv_learn_eval_device(bpltv_ctx *ctx, const double *lam, int lm, int ln,
                            double Delta, const bpltv_eval_opts *opts, void *d_u_out,
                            double *d_costgrad, void *stream);

/* One process per GPU (MPI / Distributed.jl / torchrun): the job's single collective lives in the library.  Every rank
 * owns a single-device context holding ITS shard of the images (contiguous blocks of ceil(O/nranks) images, the same
 * split bpltv_create uses across the devices of one process) and joins one NCCL communicator; from then on
 * bpltv_learn_eval, bpltv_learn_eval_device and bpltv_sumregs_learn_eval return the loss and the gradient of the WHOLE
 * job on every rank — the per-image sums of /root/reference/src/TVLearningFunctionVec.jl:72-83, :163-175 completed by
 * ONE ncclAllReduce (fp64 sum) of [cost, grad...] per evaluation on the context's stream; the denoised images stay
 * per rank.  NCCL is bound at run time (dlopen of $BPLTV_NCCL_LIB, else libnccl.so.2): no communicator, no dependency.
 *   rank 0:  bpltv_comm_unique_id(id);  ship the 128 bytes to the other ranks by any means;
 *   all:     bpltv_comm_init(ctx, nranks, rank, id)   (collective: returns when every rank has joined).          */
#define BPLTV_COMM_ID_BYTES 128
int bpltv_comm_unique_id(unsigned char *id_out);
int bpltv_comm_init(bpltv_ctx *ctx, int nranks, int rank, const unsigned char *id);
int bpltv_comm_destroy(bpltv_ctx *ctx);

int bpltv_get_stats(bpltv_ctx *ctx, bpltv_stats *out);
/* The developer switches (environment variables BPLTV_*, DESIGN.md) are read once, when the first context is
 * created; this re-reads them (the test-suite flips them between calls).  Not needed by a normal caller. */
void bpltv_reload_env(void);
/* Arithmetic self-test (test-suite entry point, not needed by a caller).  what = 0: the strict kernels form the
 * projection scale `α / sqrt(n²)` of the reference's PDPS step by a branch-free chain instead of the compiler's IEEE
 * sqrt / div expansions (csrc/common.cuh, BallScale); this runs `count` operand pairs of the context's precision
 * through both.  mode 0: the operand range of image data, 1: the chain's whole range, 2: structured significands
 * (rounding boundaries, perfect squares ± 1 ulp), 3: every `a` bit pattern in turn (exhaustive for a 32-bit context
 * from count = 2^30).  result[0] = pairs the chain took (the others go through the IEEE operations in the kernels as
 * well), result[1] = pairs whose bits differ (must be 0), result[2], result[3] = bit patterns of the first such
 * (a | 2^63, α). */
int bpltv_selftest(bpltv_ctx *ctx, int what, int mode, unsigned long long count, unsigned long long seed,
                   unsigned long long *result);
const char *bpltv_last_error(void);
int bpltv_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BPLTV_H */
