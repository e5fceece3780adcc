"""Host restatement of the reference's trust-region driver (SURVEY §8f row 2).

`bilevel_learn` follows /root/reference/src/TRBox.jl:192-273 statement by statement,
and the outer iterator's logging cadence and stop rule follow
/root/reference/src/BilevelVisualise.jl:185-256.  It exists so that an end-to-end
"bilevel learn wall time" can be measured where Julia is not installed; with Julia
present the reference's own driver calls the library unchanged (INTEGRATION.md).

The driver is scalar control flow around ≤ 21 learning-function evaluations; it does
no image arithmetic.  Quirks of the reference are kept, each marked QUIRK:

* scalar `dogleg_box`: the Newton step is `pn = B\\gx` without a minus sign (:63);
* `step_to_bound` returns the element-wise max of the two ratios, no minimum (:149-152);
* scalar `updateBFGS!` rebinds a local, so the caller's `B` stays 0.1 (:181-186, :237);
* array `updateBFGS!` pushes the pair as `(y, s)` into an operator whose `push!`
  expects `(s, y)` (:174-179);
* the step is accepted whenever ρ > 0 (:251), the radius shrinks once more when the
  predicted reduction is negative (:247-249), and the run stops only when a *logged*
  iteration sees Δ < tol (BilevelVisualise.jl:246-248).

The two third-party pieces (un-vendored packages, `/root/reference/Project.toml`) are restated from their published
algorithms, not bit for bit (nothing to check them against without Julia):
* `LinearOperators.LBFGSOperator(n)` — forward (Hessian) L-BFGS, memory 5, initial matrix (yᵀy / yᵀs)·I of the newest
  pair (`scaling = true`), pairs with yᵀs ≤ 1e-20 skipped: `LBFGSOperator` below (the same operator; the package keeps
  the compact vectors a_k, b_k, this class unrolls the recursion);
* `Krylov.cg_lanczos(B, b)` — the conjugate-gradient iterates with the package's default stopping rule
  ‖r‖ ≤ √eps + √eps·‖b‖ and ≤ 2n products: `cg_solve` below.
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass, field
from typing import Callable, List, Optional

import numpy as np

EPS = float(np.finfo(np.float64).eps)

# /root/reference/src/BPLDenoising.jl:306-323 (scalar) and :350-357 (patch)
DEFAULT_PARAMS = dict(verbose_iter=1, maxiter=20, tol=1e-5)
BILEVEL_PARAMS = dict(eta1=0.25, eta2=0.75, beta1=0.25, beta2=1.9, Delta0=0.1, alpha0=0.1)
# /root/reference/src/BPLDenoising.jl:423-430 (scalar sum-of-regularisers experiment)
SUMREGS_BILEVEL_PARAMS = dict(eta1=0.25, eta2=0.75, beta1=0.25, beta2=1.9, Delta0=0.01,
                              alpha0=np.array([0.001, 0.001, 0.001]))
# /root/reference/src/BPLDenoising.jl:455-462 (patch sum-of-regularisers experiment)
PATCH_SUMREGS_BILEVEL_PARAMS = dict(eta1=0.25, eta2=0.75, beta1=0.25, beta2=1.5, Delta0=0.1,
                                    alpha0=0.001 * np.ones((2, 2, 3)))
PATCH_BILEVEL_PARAMS = dict(eta1=0.25, eta2=0.75, beta1=0.25, beta2=1.9, Delta0=1e-4,
                            alpha0=1e-4 * np.ones((2, 2)))


@dataclass
class LogEntry:  # BilevelLogEntry, BilevelVisualise.jl:39-46
    iter: int
    time: float
    function_value: float
    gradient_norm: float
    radius: float
    residual: float


@dataclass
class LearnResult:
    x: object
    u: np.ndarray
    log: List[LogEntry] = field(default_factory=list)
    evaluations: int = 0
    seconds: float = 0.0


class LBFGSOperator:
    """Forward L-BFGS operator (approximates the Hessian), memory `mem`, scaled identity
    start.  Stand-in for LinearOperators.LBFGSOperator (TRBox.jl:50)."""

    def __init__(self, n: int, mem: int = 5):
        self.n, self.mem = n, mem
        self.s: List[np.ndarray] = []
        self.y: List[np.ndarray] = []

    def push(self, s: np.ndarray, y: np.ndarray):
        ys = float(y @ s)
        if ys <= 1e-20:
            return
        self.s.append(s.copy()); self.y.append(y.copy())
        if len(self.s) > self.mem:
            self.s.pop(0); self.y.pop(0)

    def mul(self, v: np.ndarray) -> np.ndarray:
        if not self.s:
            return v.copy()
        s_l, y_l = self.s[-1], self.y[-1]
        scale = float(y_l @ y_l) / float(y_l @ s_l)
        # unrolled BFGS recursion: B_{k+1} = B_k - (B_k s sᵀ B_k)/(sᵀ B_k s) + (y yᵀ)/(yᵀ s)
        bs: List[np.ndarray] = []
        for k, (s, y) in enumerate(zip(self.s, self.y)):
            b = scale * s
            for j in range(k):
                sj, yj, bj = self.s[j], self.y[j], bs[j]
                b = b - bj * float(bj @ s) / float(sj @ bj) + yj * float(yj @ s) / float(yj @ sj)
            bs.append(b)
        out = scale * v
        for s, y, b in zip(self.s, self.y, bs):
            out = out - b * float(b @ v) / float(s @ b) + y * float(y @ v) / float(y @ s)
        return out

    def dense(self) -> np.ndarray:
        return np.column_stack([self.mul(e) for e in np.eye(self.n)])


def cg_solve(mul: Callable[[np.ndarray], np.ndarray], b: np.ndarray) -> np.ndarray:
    """`pn, ks = Krylov.cg_lanczos(B, -gx[:])` (TRBox.jl:136).  CG-Lanczos produces the conjugate-gradient iterates (it is CG
    written on the Lanczos basis) and stops, with Krylov.jl's defaults, at ‖r_k‖ ≤ atol + rtol·‖b‖, atol = rtol = √eps, after
    at most 2n products — so the reference's Newton step is an INEXACT solve at the 1e-8 level, which an exact dense solve
    would not reproduce.  Here: plain CG from x₀ = 0 with that stopping rule (the same iterates in exact arithmetic)."""
    n = b.size
    tol = math.sqrt(EPS)
    x = np.zeros(n)
    r = b.astype(np.float64).copy()
    bnorm = float(np.linalg.norm(r))
    if bnorm == 0.0:
        return x
    eps_stop = tol + tol * bnorm
    pdir = r.copy()
    rr = float(r @ r)
    for _ in range(2 * n):
        if math.sqrt(rr) <= eps_stop:
            break
        Ap = mul(pdir)
        curv = float(pdir @ Ap)
        if curv <= 0.0:                      # cg_lanczos stops on non-positive curvature; L-BFGS operators are SPD
            break
        a = rr / curv
        x += a * pdir
        r -= a * Ap
        rr_new = float(r @ r)
        pdir = r + (rr_new / rr) * pdir
        rr = rr_new
    return x


# ---- auxiliary functions (TRBox.jl:59-186) ----------------------------------------
def get_bounds(x, Delta):  # :160-164
    lb = np.maximum(-Delta, EPS - np.asarray(x, dtype=np.float64))
    ub = Delta * np.ones(np.shape(x))
    return lb, ub


def in_bounds(lb, ub, x) -> bool:  # :155-157
    return bool(np.all(x >= lb) and np.all(x <= ub))


def step_to_bound(p, lb, ub):  # :149-152  QUIRK: element-wise max, no minimum
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.maximum(lb / p, ub / p)


def pred(B, p, gx) -> float:  # :166-172
    if isinstance(B, LBFGSOperator):
        pv, gv = np.ravel(p, order="F"), np.ravel(gx, order="F")
        return float(-pv @ gv - 0.5 * pv @ B.mul(pv))
    return float(-p * gx - 0.5 * p * B * p)


def dogleg_box(x, gx, B, Delta):
    lb, ub = get_bounds(x, Delta)
    if not isinstance(B, LBFGSOperator):  # scalar, :60-76
        pn = gx / B  # QUIRK: `pn = B\gx`, no minus sign (:63)
        if in_bounds(lb, Delta, pn):
            return float(pn)
        p = -(abs(gx) ** 2 / (gx * (B * gx))) * gx  # Cauchy step (:67)
        if not in_bounds(lb, Delta, p):
            d = p / abs(p)
            t = step_to_bound(d, lb, Delta)
            return float(d * t)
        t = step_to_bound(pn - p, lb, Delta)
        return float(p + t * (pn - p))
    # array, :99-114
    g = np.ravel(gx, order="F")
    pn = cg_solve(B.mul, -g).reshape(np.shape(gx), order="F")  # newton_step (:135-141)
    if in_bounds(lb, Delta, pn):
        return pn
    p = (-(np.linalg.norm(g) ** 2 / float(g @ B.mul(g))) * g).reshape(np.shape(gx), order="F")  # :143-146
    if not in_bounds(lb, Delta, p):
        d = p / np.linalg.norm(p)
        return d * step_to_bound(d, lb, Delta)
    return p + step_to_bound(pn - p, lb, Delta) * (pn - p)


def update_bfgs(B, y, s):  # :174-186
    if isinstance(B, LBFGSOperator):
        yv, sv = np.ravel(y, order="F"), np.ravel(s, order="F")
        if float(yv @ B.mul(yv)) > 0:
            B.push(yv, sv)  # QUIRK: push!(B, y, s) although the operator expects (s, y)
        return B
    return B  # QUIRK: the scalar update rebinds a local; the caller's B is unchanged


def bilevel_learn(ds, learning_function: Callable, xinit, params: Optional[dict] = None,
                  verbose: bool = False) -> LearnResult:
    """bilevel_learn(ds, learning_function; xinit, iterate, params) — TRBox.jl:192-273 with
    the iterator of BilevelVisualise.jl:185-256 inlined."""
    prm = dict(DEFAULT_PARAMS)
    scalar = np.ndim(xinit) == 0
    prm.update(BILEVEL_PARAMS if scalar else PATCH_BILEVEL_PARAMS)
    prm.update(params or {})
    eta1, eta2, beta1, beta2 = prm["eta1"], prm["eta2"], prm["beta1"], prm["beta2"]
    t0 = time.perf_counter()
    # init_rest (:34-52)
    x = float(xinit) if scalar else np.array(xinit, dtype=np.float64, order="F")
    Delta = float(prm["Delta0"])
    u, fx, gx = learning_function(x, ds, Delta)
    evals = 1
    B = 0.1 if scalar else LBFGSOperator(int(np.size(x)))
    residual = 0.0 * x
    log: List[LogEntry] = []
    for it in range(1, int(prm["maxiter"]) + 1):
        p = dogleg_box(x, gx, B, Delta)                       # :221
        xb = x + p                                           # :224
        ub_, fxb, gxb = learning_function(xb, ds, Delta)      # :227  ★ hot call
        evals += 1
        predf = pred(B, p, gx)                                # :229
        rho = (fx - fxb) / predf if predf != 0 else math.copysign(math.inf, fx - fxb)  # :230-233
        B = update_bfgs(B, np.asarray(gxb) - np.asarray(gx), p)  # :237
        if rho < eta1:                                        # :239-245
            Delta = beta1 * Delta
        elif rho > eta2:
            if np.linalg.norm(np.ravel(p)) > 0.8 * Delta:
                Delta = beta2 * Delta
        if predf < 0:                                         # :247-249
            Delta = beta1 * Delta
        if rho > 0:                                           # :251-257
            residual = x - xb
            x, u, fx, gx = xb, ub_, fxb, gxb
        # iterator: log cadence and stop rule (BilevelVisualise.jl:198-200, 246-248)
        verb = prm["verbose_iter"] != 0 and it % prm["verbose_iter"] == 0
        if verb or it <= 20 or (it <= 200 and it % 10 == 0):
            entry = LogEntry(it, time.perf_counter() - t0, float(fx), float(np.linalg.norm(np.ravel(gx))),
                             Delta, float(np.linalg.norm(np.ravel(residual))))
            log.append(entry)
            if verbose:
                print(f"{it}/{prm['maxiter']} x={np.linalg.norm(np.ravel(x)):e}, f={fx:.3e}, "
                      f"g={entry.gradient_norm:.4e}, Δ={Delta:.3e}, stop={entry.residual:.3e}")
            if Delta < prm["tol"]:
                break
    return LearnResult(x=x, u=u, log=log, evaluations=evals, seconds=time.perf_counter() - t0)


def scalar_bilevel_tv_learn(data, ctx=None, **kwargs) -> LearnResult:
    """scalar_bilevel_tv_learn (BPLDenoising.jl:325-344) without IO/visualisation: `data` is
    the (truth, noisy) pair the reference's `testdataset` + `num_samples` slicing yields."""
    from .learning import tv_op_learning_function

    prm = dict(BILEVEL_PARAMS); prm.update(kwargs)
    return bilevel_learn(data, lambda x, ds, D: tv_op_learning_function(x, ds, D, ctx=ctx),
                         prm.pop("alpha0"), prm)


def patch_bilevel_tv_learn(data, ctx=None, **kwargs) -> LearnResult:
    """patch_bilevel_tv_learn (BPLDenoising.jl:359-376) without IO/visualisation."""
    from .learning import tv_op_learning_function

    prm = dict(PATCH_BILEVEL_PARAMS); prm.update(kwargs)
    return bilevel_learn(data, lambda x, ds, D: tv_op_learning_function(x, ds, D, ctx=ctx),
                         prm.pop("alpha0"), prm)


def scalar_bilevel_sumregs_learn(data, ctx=None, **kwargs) -> LearnResult:
    """scalar_bilevel_sumregs_learn (BPLDenoising.jl:432-451) without IO/visualisation: the
    3-vector parameter takes the driver's array path (L-BFGS model, TRBox.jl:50, :99-114)."""
    from .learning import sumregs_learning_function

    prm = dict(SUMREGS_BILEVEL_PARAMS); prm.update(kwargs)
    return bilevel_learn(data, lambda x, ds, D: sumregs_learning_function(x, ds, D, ctx=ctx),
                         prm.pop("alpha0"), prm)


def patch_bilevel_sumregs_learn(data, ctx=None, **kwargs) -> LearnResult:
    """patch_bilevel_sumregs_learn (BPLDenoising.jl:464-481) without IO/visualisation.  Once the trust
    region shrinks below Δt = 1e-3 the learning function switches to the patch variant of
    sumregs_gradient_reg (SumRegsLearningFunction.jl:195-262), which libbpltv solves with its band LU up to 430²
    and with the LU of its nested-dissection fronts beyond."""
    from .learning import sumregs_learning_function

    prm = dict(PATCH_SUMREGS_BILEVEL_PARAMS); prm.update(kwargs)
    return bilevel_learn(data, lambda x, ds, D: sumregs_learning_function(x, ds, D, ctx=ctx),
                         prm.pop("alpha0"), prm)
