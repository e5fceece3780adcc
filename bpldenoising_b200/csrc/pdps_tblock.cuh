// pdps_tblock.cuh — kernel C: temporally blocked HBM-streaming PDPS ("pipelined march").
//
// One launch = T consecutive primal-dual iterations over the whole M×N×O stack for the
// HBM traffic of ONE: read {x, y1, y2, f}, write {x, y1, y2} = 7 words per pixel per
// launch (8 with a λ-map), i.e. 7/T words per pixel-iteration, plus a halo of T-1 columns
// per column range.
//
// Same decomposition as kernel A (pdps_march.cuh): the N·O image columns are cut into one
// contiguous range per CTA, a CTA spans the whole column height and marches along j.  The
// T iterations are software-pipelined along the march, entirely in registers.  Stage s
// (iteration k+s of the launch) trails the march front by 2s columns: at march step c it
//     P-phase: forms x^{s+1}, x̄^{s+1} of column p = c-2s,
//     D-phase: finishes y^{s+1} of column p-1 (which needed x̄^{s+1}(:,p)),
// reading the duals stage s-1 finished in the PREVIOUS step and the x it formed two steps
// ago.  Because every stage works on data of earlier steps, the T stages of one step are
// independent instruction streams (the dependent chain of one iteration — prox, shuffle,
// gradient, dual ascent, √ and ÷ of the projection — is what limits a single stage; the
// projections of all stages and rows of a thread are issued together for the same reason)
// and a step needs two CTA barriers whatever T is: one after the P-phase (x̄ of the first
// row of each warp → the warp above), one after the D-phase (the finished y1 of the last
// row of each warp → the warp below).  Only stage 0 reads state from memory, only stage
// T-1 writes it.  The march loop is unrolled by two with the carried state in two register
// sets that swap roles, so nothing is copied from step to step.
//
// Loads: with 16-byte vectors a column is a 16-byte multiple, and stage 0's input columns
// {x, y1, y2, f} arrive through a shared-memory ring filled by the TMA engine (1-D
// cp.async.bulk, one mbarrier per slot, TB_PF columns ahead of the march front), so no
// thread ever waits on an HBM load; later stages re-read f from the same ring.
//
// Range ends: a range [c0,c1) of an image starts marching at cs = c0-(T-1) and loads up to
// c1+T-1 (clipped to the image), recomputing the T-1 halo columns on each side; stage s is
// exact from column cs+s on (its left neighbour y2^s(cs+s-1) is unknown before that), which
// is exactly what stage T-1 needs at c0.  At the image's right edge each stage "flushes"
// the dual of column N-1 with Δy2 = 0, as kernel A does.  The pipeline fill and drain
// steps run the same code with per-stage activity flags (template STEADY = false).
//
// The arithmetic is common.cuh's primal_update / dual ascent / projection in the same order
// per pixel and iteration, so strict mode stays bit-identical to the oracle.
#pragma once
#ifdef BPLTV_EMU
#include <cstdint>
#include <cstdio>
#include <thread>
#endif
#include "common.cuh"

namespace bpltv {

// ---- 1-D bulk TMA + mbarrier (column prefetch ring), 32-bit shared addresses -------------
constexpr int TB_R = 4;              // ring slots of the x / y1 / y2 planes (power of two)
constexpr int TB_PF = TB_R - 1;      // columns in flight ahead of the march front
// ring slots of f: later stages read f of column c-2s (power of two ≥ TB_R + 2(T-1))
template <int T> struct TBRingF { static constexpr int value = (TB_R + 2 * (T - 1)) <= 8 ? 8 : 16; };

#ifdef BPLTV_EMU
// Thread emulation (tests/emu): shared-window addresses are plain pointers, a bulk copy is a memcpy by the issuing thread,
// and an mbarrier is a 64-bit word — low half: bytes the current phase still expects, high half: completed phases.
typedef std::uintptr_t tb_addr;
static inline tb_addr smem_u32(const void *p) { return reinterpret_cast<tb_addr>(p); }
static inline void mbar_init(tb_addr bar, unsigned) { __atomic_store_n(reinterpret_cast<unsigned long long *>(bar), 0ULL, __ATOMIC_RELEASE); }
static inline void mbar_fence_init() {}
static inline void mbar_expect_tx(tb_addr bar, unsigned bytes)
{
    __atomic_fetch_add(reinterpret_cast<unsigned long long *>(bar), (unsigned long long)bytes, __ATOMIC_RELAXED);
}
static inline void mbar_wait(tb_addr bar, unsigned parity)
{
    while (((__atomic_load_n(reinterpret_cast<unsigned long long *>(bar), __ATOMIC_ACQUIRE) >> 32) & 1ULL) == parity) std::this_thread::yield();
}
static inline void tma_load_1d(tb_addr dst, const void *src, unsigned bytes, tb_addr bar)
{
    if ((dst & 15) || (reinterpret_cast<std::uintptr_t>(src) & 15) || (bytes & 15)) { std::fprintf(stderr, "emu: misaligned bulk copy\n"); std::abort(); }
    std::memcpy(reinterpret_cast<void *>(dst), src, bytes);
    unsigned long long *b = reinterpret_cast<unsigned long long *>(bar);
    const unsigned long long before = __atomic_fetch_sub(b, (unsigned long long)bytes, __ATOMIC_ACQ_REL);
    if ((unsigned)(before & 0xffffffffULL) == bytes) __atomic_fetch_add(b, 1ULL << 32, __ATOMIC_RELEASE);   // the phase completes
}
template <typename Real, int VEC>
static inline void lds16(tb_addr addr, Real (&v)[VEC]) { std::memcpy(v, reinterpret_cast<const void *>(addr), sizeof(Real) * VEC); }
template <typename Real>
static inline Real lds1(tb_addr addr, Real) { Real v; std::memcpy(&v, reinterpret_cast<const void *>(addr), sizeof(Real)); return v; }
#else
typedef unsigned tb_addr;
static __device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
static __device__ __forceinline__ tb_addr smem_u32(const void *p) { return (tb_addr)__cvta_generic_to_shared(p); }
static __device__ __forceinline__ void mbar_init(tb_addr bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
static __device__ __forceinline__ void mbar_expect_tx(tb_addr bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
static __device__ __forceinline__ void mbar_wait(tb_addr bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra TB_DONE;\n"
        "bra TB_WAIT;\n"
        "TB_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// global → shared copy of `bytes` (multiple of 16, both addresses 16-byte aligned) by the TMA
// engine; completion is counted in bytes on the mbarrier `bar`
static __device__ __forceinline__ void tma_load_1d(tb_addr dst, const void *src, unsigned bytes, tb_addr bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// 16-byte shared-memory load of VEC Reals
static __device__ __forceinline__ void lds16(tb_addr addr, double (&v)[2])
{
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr));
}
static __device__ __forceinline__ void lds16(tb_addr addr, float (&v)[4])
{
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}
template <typename Real, int VEC>
static __device__ __forceinline__ void lds16(tb_addr, Real (&)[VEC]) {}  // never called (RING ⇒ 16-byte vectors)
static __device__ __forceinline__ double lds1(tb_addr addr, double)
{
    double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr)); return v;
}
static __device__ __forceinline__ float lds1(tb_addr addr, float)
{
    float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v;
}
#endif

// a > b as a 0/1 word.  Opaque to the front end on purpose: it turns a thread's OR of the ball tests `n² > α²` into
// a maximum of the n² (an fmax chain with NaN handling, about seven instructions per pixel against two here).
#ifdef BPLTV_EMU
template <typename Real>
static inline unsigned tb_gt(Real a, Real b) { return a > b ? 1u : 0u; }
#else
static __device__ __forceinline__ unsigned tb_gt(double a, double b)
{
    unsigned r; asm("{\n.reg .pred p;\nsetp.gt.f64 p, %1, %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(r) : "d"(a), "d"(b)); return r;
}
static __device__ __forceinline__ unsigned tb_gt(float a, float b)
{
    unsigned r; asm("{\n.reg .pred p;\nsetp.gt.f32 p, %1, %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(r) : "f"(a), "f"(b)); return r;
}
#endif

template <typename Real, int T>
struct TBlockArgs {
    const Real *x_in, *y1_in, *y2_in, *f;
    Real *x_out, *y1_out, *y2_out;
    const Real *alpha_map;            // M×N (shared by all images) or nullptr
    StepConsts<Real> sc[T];           // constants of the T iterations of this launch
    int M, N, O;
    long long total_cols;             // N·O
    Real alpha_s;
    BatchMap<Real> bm;
};

// What one pipeline stage keeps from step to step (registers).
template <typename Real, int VEC>
struct TBStage {
    Real xb[VEC], d1[VEC], y1[VEC], y2[VEC];  // carried column p: x̄, Δy1 and the stage's input duals
    Real xn[VEC], f[VEC];                      // x^{s+1}(:,p), f(:,p): stage s+1 reads them two steps later
    Real o1[VEC], o2[VEC];                     // y^{s+1}(:,p-1): stage s+1 reads them in the next step
};

// Per-segment constants of the march.
template <typename Real>
struct TBSeg {
    const Real *xin, *y1in, *y2in, *fin, *amap;
    Real *xout, *y1out, *y2out;
    int M, N, c0, c1, cs, cl, lane, warp;
    int r0;            // first row of this thread (clamped into the image for threads beyond it)
    bool st_ok;        // this thread owns rows (threads beyond the column compute a copy, store nothing)
    bool multi_warp;
    Real alpha_s;
    Real alpha2;       // RN(α²) of the scalar α (strict arithmetic): the ball's test, once per segment
    bool alpha_ok;     // BallScale's α range test of the scalar α
    // column prefetch ring (RING kernels), shared-window byte addresses of this thread's rows:
    // slot i of {x,y1,y2} at ring_t + i·3·colb (planes colb apart), slot j of f at fring_t + j·colb;
    // image column c of the segment is load number k0 + (c - cs)
    tb_addr ring_t, fring_t, ring0, fring0, bars;
    unsigned colb;
    int k0;
};

template <typename Real>
static __device__ __forceinline__ void tb_set_alpha(TBSeg<Real> &g, Real al)
{
    g.alpha_s = al;
    g.alpha2 = StrictOps<Real>::mul(al, al);
    g.alpha_ok = BallScale<Real>::fast_ok_alpha(al);
}

// thread 0: start the TMA copies of image column `col` (load number kk)
template <typename Real, int T>
static __device__ __forceinline__ void tb_issue(const TBSeg<Real> &g, int kk, int col)
{
    const tb_addr bar = g.bars + 8u * (unsigned)(kk & (TB_R - 1));
    const tb_addr sx = g.ring0 + (unsigned)(kk & (TB_R - 1)) * 3u * g.colb;
    const size_t off = (size_t)col * g.M;
    mbar_expect_tx(bar, 4 * g.colb);
    tma_load_1d(sx, g.xin + off, g.colb, bar);
    tma_load_1d(sx + g.colb, g.y1in + off, g.colb, bar);
    tma_load_1d(sx + 2 * g.colb, g.y2in + off, g.colb, bar);
    tma_load_1d(g.fring0 + (unsigned)(kk & (TBRingF<T>::value - 1)) * g.colb, g.fin + off, g.colb, bar);
}

// One march step.  Reads the state of the previous step from P (and, for x/f, the values
// stage s-1 left in C two steps ago), writes the new state to C.
template <typename Real, int VEC, int T, bool MAP, bool STRICT, bool RING, bool STEADY>
static __device__ __forceinline__ void tblock_step(const int c, const TBStage<Real, VEC> (&P)[T],
                                                   TBStage<Real, VEC> (&C)[T], const TBSeg<Real> &g,
                                                   const StepConsts<Real> (&scs)[T], Real (&s_dn)[T][33],
                                                   Real (&s_up)[T][34])
{
    typedef VecIO<Real, VEC> IO;
    typedef StrictOps<Real> A;
    constexpr int RF = TBRingF<T>::value;
    const int M = g.M, N = g.N, r0 = g.r0, lane = g.lane, warp = g.warp;
    bool do_primal[T], do_dual[T], do_flush[T];
    Real xb_c[T][VEC], y1_c[T][VEC], y2_c[T][VEC];

    // ---------------- P-phase: stages in descending order (stage s reads what stage s-1
    // left in C two steps ago before stage s-1 overwrites it) -------------------------
#pragma unroll
    for (int s = T - 1; s >= 0; --s) {
        const int p = c - 2 * s;
        const int pl = min(g.c1 + (T - 1 - s), N - 1);          // last primal column this stage needs
        do_primal[s] = STEADY || (p >= g.cs && p <= pl);         // CTA-uniform
        do_dual[s] = STEADY || (p - 1 >= g.cs && p <= pl);
        do_flush[s] = !STEADY && (p == N && pl == N - 1);
        if (!do_primal[s]) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) xb_c[s][v] = y1_c[s][v] = y2_c[s][v] = 0;
            continue;
        }
        Real x_c[VEC], f_c[VEC], up_c = 0;
        const int k = g.k0 + (p - g.cs);                          // load number of column p (RING)
        if (s == 0) {
            if (RING) {
                if (threadIdx.x == 0 && p + TB_PF <= g.cl) tb_issue<Real, T>(g, k + TB_PF, p + TB_PF);
                mbar_wait(g.bars + 8u * (unsigned)(k & (TB_R - 1)), ((unsigned)k / TB_R) & 1u);
                const tb_addr sx = g.ring_t + (unsigned)(k & (TB_R - 1)) * 3u * g.colb;
                lds16(sx, x_c);
                lds16(sx + g.colb, y1_c[0]);
                lds16(sx + 2 * g.colb, y2_c[0]);
                lds16(g.fring_t + (unsigned)(k & (RF - 1)) * g.colb, f_c);
                if (lane == 0 && r0 > 0) up_c = lds1(sx + g.colb - (unsigned)sizeof(Real), Real());  // y1 of the row above
            } else {
                const size_t off = (size_t)p * M + r0;
                IO::ld(g.xin + off, x_c);
                IO::ld(g.fin + off, f_c);
                IO::ld(g.y1in + off, y1_c[0]);
                IO::ld(g.y2in + off, y2_c[0]);
                if (lane == 0 && r0 > 0) up_c = __ldg(g.y1in + off - 1);
            }
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                x_c[v] = C[s - 1].xn[v];                                   // from two steps ago
                if (!RING) f_c[v] = C[s - 1].f[v];
                y1_c[s][v] = P[s - 1].o1[v]; y2_c[s][v] = P[s - 1].o2[v];  // from the previous step
            }
            if (RING) lds16(g.fring_t + (unsigned)(k & (RF - 1)) * g.colb, f_c);
            if (g.multi_warp && lane == 0 && warp > 0) up_c = s_up[s][warp];
        }
        Real up = __shfl_up_sync(0xffffffffu, y1_c[s][VEC - 1], 1);
        if (lane == 0) up = up_c;  // 0 at the top row
        Real xn_c[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            const Real y1up = (v == 0) ? up : y1_c[s][v - 1];
            xn_c[v] = primal_update<Real, STRICT>(x_c[v], f_c[v], y1up, y1_c[s][v], P[s].y2[v], y2_c[s][v], scs[s],
                                                  xb_c[s][v]);
        }
        if (s == T - 1) {
            if (g.st_ok && p >= g.c0 && p < g.c1) IO::st(g.xout + (size_t)p * M + r0, xn_c);
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) { C[s].xn[v] = xn_c[v]; if (!RING) C[s].f[v] = f_c[v]; }
        }
        if (g.multi_warp && lane == 0) s_dn[s][warp] = xb_c[s][0];
    }
    if (g.multi_warp) __syncthreads();

    // ---------------- D-phase ---------------------------------------------------------------
    // Δy1 of the new column; dual ascent v = y + σ∇x̄ of column p-1 for every active stage
    Real v1[T][VEC], v2[T][VEC], n2[T][VEC], al[T][VEC];
    unsigned out[T][VEC], outside = 0;      // out: n² > α² (strict arithmetic, scalar α)
    // scalar α: stages in descending order, so that stage s reads its input duals before stage s-1 forms the ones it
    // hands on (see the end of the step) and the two never need registers at the same time.  The λ-map kernels keep
    // the ascending order and the per-pixel α² and select of the projection: on them the scalar form measured slower.
#pragma unroll
    for (int i = 0; i < T; ++i) {
        const int s = MAP ? i : T - 1 - i;
        const int p = c - 2 * s;
        if (do_primal[s]) {
            Real dn = __shfl_down_sync(0xffffffffu, xb_c[s][0], 1);
            if (g.multi_warp && lane == 31) dn = s_dn[s][warp + 1];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const Real nxt = (v == VEC - 1) ? dn : xb_c[s][v + 1];
                const bool last_row = v == VEC - 1 && r0 + v == M - 1;   // M % VEC == 0
                C[s].d1[v] = last_row ? (Real)0 : (STRICT ? A::sub(nxt, xb_c[s][v]) : nxt - xb_c[s][v]);
            }
        }
#pragma unroll
        for (int v = 0; v < VEC; ++v) { v1[s][v] = v2[s][v] = n2[s][v] = 0; al[s][v] = g.alpha_s; out[s][v] = 0; }
        if (do_dual[s] || do_flush[s]) {
            if (MAP) IO::ld(g.amap + (size_t)(p - 1) * M + r0, al[s]);
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                Real d2 = (Real)0;
                if (STRICT) {
                    if (do_dual[s]) d2 = A::sub(xb_c[s][v], P[s].xb[v]);
                    v1[s][v] = A::add(P[s].y1[v], A::mul(scs[s].sigma, P[s].d1[v]));
                    v2[s][v] = A::add(P[s].y2[v], A::mul(scs[s].sigma, d2));
                    n2[s][v] = A::add(A::mul(v1[s][v], v1[s][v]), A::mul(v2[s][v], v2[s][v]));
                    if (MAP) {
                        outside |= n2[s][v] > A::mul(al[s][v], al[s][v]);
                    } else {
                        out[s][v] = tb_gt(n2[s][v], g.alpha2);
                        outside |= out[s][v];
                    }
                } else {
                    if (do_dual[s]) d2 = xb_c[s][v] - P[s].xb[v];
                    v1[s][v] = fma_(scs[s].sigma, P[s].d1[v], P[s].y1[v]);
                    v2[s][v] = fma_(scs[s].sigma, d2, P[s].y2[v]);
                    n2[s][v] = fma_(v1[s][v], v1[s][v], v2[s][v] * v2[s][v]);
                    outside |= n2[s][v] > al[s][v] * al[s][v];
                }
            }
        }
    }
    // projection onto the λ-ball, `if n² > α²` as in the reference: all of the thread's pixels
    // that left the ball are scaled in one block so that their √ and ÷ chains overlap (a
    // thread none of whose pixels left the ball skips it entirely)
    if (outside) {
        if (STRICT && MAP) {
            // α / sqrt(n²) with both operations correctly rounded, as branch-free chains (BallScale, common.cuh): the
            // T·VEC chains of the thread interleave; a pixel outside the chain's operand range (never on image data)
            // sends the thread's pixels through the IEEE operations instead
            Real sc[T][VEC];
            bool outm[T][VEC], ok = true;
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    outm[s][v] = n2[s][v] > A::mul(al[s][v], al[s][v]);
                    if (!outm[s][v]) n2[s][v] = (Real)1;
                    ok &= BallScale<Real>::fast_ok(n2[s][v], al[s][v]);
                }
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v) sc[s][v] = BallScale<Real>::eval(n2[s][v], al[s][v]);
            if (!ok) {
#pragma unroll
                for (int s = 0; s < T; ++s)
#pragma unroll
                    for (int v = 0; v < VEC; ++v) sc[s][v] = ball_scale_ieee<Real>(n2[s][v], al[s][v]);
            }
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v)
                    if (outm[s][v]) { v1[s][v] = A::mul(v1[s][v], sc[s][v]); v2[s][v] = A::mul(v2[s][v], sc[s][v]); }
        } else if (STRICT) {
            // α / sqrt(n²) with both operations correctly rounded, as branch-free chains (BallScale, common.cuh): the
            // T·VEC chains of the thread interleave; a pixel outside the chain's operand range (never on image data)
            // sends the thread's pixels through the IEEE operations instead.  The scalar α is checked once per segment.
            //   A pixel inside the ball goes through the chain with n² := α², and its factor RN(α / RN(√RN(α²))) is
            // exactly 1: RN(√RN(α²)) = α for every α > 0 whose square neither overflows nor underflows in binary
            // floating point (Boldo, "Stupid is as stupid does: taking the square root of the square of a floating-point
            // number", 2015), which the α range of fast_ok guarantees.  Multiplying by 1 is exact for every non-NaN
            // operand (±0, subnormals and ±inf included), so every pixel is scaled without a select of the factor or of
            // the products.  The IEEE path selects explicitly (its α need not be positive).
            Real sc[T][VEC];
            bool ok = g.alpha_ok;
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    if (!out[s][v]) n2[s][v] = g.alpha2;
                    ok &= BallScale<Real>::fast_ok_a(n2[s][v]);
                }
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v) sc[s][v] = BallScale<Real>::eval(n2[s][v], al[s][v]);
            if (!ok) {
#pragma unroll
                for (int s = 0; s < T; ++s)
#pragma unroll
                    for (int v = 0; v < VEC; ++v) {
                        const Real q = ball_scale_ieee<Real>(n2[s][v], al[s][v]);
                        sc[s][v] = n2[s][v] > g.alpha2 ? q : (Real)1;
                    }
            }
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    v1[s][v] = A::mul(v1[s][v], sc[s][v]);
                    v2[s][v] = A::mul(v2[s][v], sc[s][v]);
                }
        } else {
#pragma unroll
            for (int s = 0; s < T; ++s)
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    const bool out = n2[s][v] > al[s][v] * al[s][v];
                    const Real sc = al[s][v] * rsqrt_(out ? n2[s][v] : (Real)1);
                    if (out) { v1[s][v] *= sc; v2[s][v] *= sc; }
                }
        }
    }
#pragma unroll
    for (int s = 0; s < T; ++s) {
        const int p = c - 2 * s;
        if (do_dual[s] || do_flush[s]) {
            if (s == T - 1) {
                if (g.st_ok && p - 1 >= g.c0 && p - 1 < g.c1) {
                    IO::st(g.y1out + (size_t)(p - 1) * M + r0, v1[s]);
                    IO::st(g.y2out + (size_t)(p - 1) * M + r0, v2[s]);
                }
            } else {
#pragma unroll
                for (int v = 0; v < VEC; ++v) { C[s].o1[v] = v1[s][v]; C[s].o2[v] = v2[s][v]; }
                if (g.multi_warp && lane == 31) s_up[s + 1][warp + 1] = v1[s][VEC - 1];
            }
        }
        // carried column of this stage
        if (do_primal[s]) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) { C[s].xb[v] = xb_c[s][v]; C[s].y1[v] = y1_c[s][v]; C[s].y2[v] = y2_c[s][v]; }
        } else {  // fill / drain: the stage keeps what it had
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                C[s].xb[v] = P[s].xb[v]; C[s].d1[v] = P[s].d1[v]; C[s].y1[v] = P[s].y1[v]; C[s].y2[v] = P[s].y2[v];
            }
        }
    }
    if (g.multi_warp) __syncthreads();
}

// dynamic shared memory of a RING kernel for column height M
template <typename Real, int T>
static inline size_t tblock_ring_bytes(int M) { return (size_t)(3 * TB_R + TBRingF<T>::value) * M * sizeof(Real); }

// BATCH: the stack is a λ-sweep's virtual stack (BatchMap: per-image λ, shared f); kept out of the plain
// instantiation because its per-segment values cost registers the T = 2 kernel does not have to spare
template <typename Real, int VEC, int T, bool MAP, bool STRICT, bool RING, bool BATCH, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) pdps_tblock_kernel(const TBlockArgs<Real, T> a)
{
    typedef VecIO<Real, VEC> IO;
#ifdef BPLTV_EMU
    unsigned char *tb_smem = reinterpret_cast<unsigned char *>(emu::dyn_smem());
#else
    extern __shared__ __align__(128) unsigned char tb_smem[];
#endif
    __shared__ unsigned long long s_bars[TB_R];
    // slot [warp] of s_dn: x̄ of the warp's first row (read by the warp above it);
    // slot [warp+1] of s_up: the finished y1 of the warp's last row (read by the warp below)
    __shared__ Real s_dn[T][33];
    __shared__ Real s_up[T][34];

    const int M = a.M, N = a.N;
    TBSeg<Real> g;
    g.M = M; g.N = N; g.amap = a.alpha_map;
    tb_set_alpha(g, a.alpha_s);
    g.st_ok = (int)threadIdx.x * VEC < M;                 // M % VEC == 0 → all VEC rows valid together
    g.r0 = min((int)threadIdx.x * VEC, M - VEC);          // threads beyond the column shadow its last rows
    g.lane = threadIdx.x & 31; g.warp = threadIdx.x >> 5;
    g.multi_warp = blockDim.x > 32;
    g.colb = (unsigned)(M * sizeof(Real));
    g.ring0 = smem_u32(tb_smem);
    g.fring0 = g.ring0 + 3u * TB_R * g.colb;
    g.ring_t = g.ring0 + (unsigned)(g.r0 * sizeof(Real));
    g.fring_t = g.fring0 + (unsigned)(g.r0 * sizeof(Real));
    g.bars = smem_u32(s_bars);
    g.k0 = 0; g.cl = 0;
    if (RING) {
        if (threadIdx.x == 0) {
#pragma unroll
            for (int i = 0; i < TB_R; ++i) mbar_init(g.bars + 8u * i, 1);
            mbar_fence_init();
        }
        __syncthreads();
    }

    const long long per = (a.total_cols + gridDim.x - 1) / gridDim.x;
    long long gc = (long long)blockIdx.x * per;
    const long long g_end = min(a.total_cols, gc + per);

    while (gc < g_end) {
        const int o = (int)(gc / N);
        const int c0 = (int)(gc - (long long)o * N);
        const int c1 = (int)min((long long)N, (long long)c0 + (g_end - gc));  // exclusive
        gc += c1 - c0;
        const size_t img = (size_t)o * M * N;
        g.xin = a.x_in + img; g.y1in = a.y1_in + img; g.y2in = a.y2_in + img;
        if (BATCH) {
            g.fin = a.f + (size_t)a.bm.f_image(o) * M * N;
            if (MAP) g.amap = a.alpha_map + (size_t)a.bm.lam_set(o) * a.bm.map_stride;
            tb_set_alpha(g, a.bm.scalar(o, a.alpha_s));
        } else {
            g.fin = a.f + img;
        }
        g.xout = a.x_out + img; g.y1out = a.y1_out + img; g.y2out = a.y2_out + img;
        g.c0 = c0; g.c1 = c1;
        const int cs = max(0, c0 - (T - 1));                           // first marched column
        g.cs = cs;
        const int c_end = ((c1 == N) ? N : c1) + 2 * (T - 1);          // last march step
        const int c_lo = cs + 1 + 2 * (T - 1);                         // steady state: every stage forms
        const int c_hi = min(c1 + T - 1, N - 1);                       // and finishes a column per step
        g.cl = c_hi;                                                   // last column loaded

        TBStage<Real, VEC> A[T], B[T];
#pragma unroll
        for (int s = 0; s < T; ++s) {
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                A[s].xb[v] = A[s].d1[v] = A[s].y1[v] = A[s].y2[v] = A[s].xn[v] = A[s].f[v] = A[s].o1[v] = A[s].o2[v] = 0;
            B[s] = A[s];
        }
        if (cs > 0) IO::ld(g.y2in + (size_t)(cs - 1) * M + g.r0, A[0].y2);
        if (RING && threadIdx.x == 0) {
#pragma unroll
            for (int i = 0; i < TB_PF; ++i)
                if (cs + i <= c_hi) tb_issue<Real, T>(g, g.k0 + i, cs + i);
        }

        int c = cs;
        // fill (and everything, for ranges too short to reach the steady state)
        for (; c <= c_end && c < c_lo; ++c) {
            tblock_step<Real, VEC, T, MAP, STRICT, RING, false>(c, A, B, g, a.sc, s_dn, s_up);
#pragma unroll
            for (int s = 0; s < T; ++s) {
                // B holds the new state; A keeps the two-steps-ago x/f until the next step reads them
                TBStage<Real, VEC> t = A[s]; A[s] = B[s]; B[s] = t;
            }
        }
        // steady state, two steps per trip: the register sets swap roles
        for (; c + 1 <= c_hi; c += 2) {
            tblock_step<Real, VEC, T, MAP, STRICT, RING, true>(c, A, B, g, a.sc, s_dn, s_up);
            tblock_step<Real, VEC, T, MAP, STRICT, RING, true>(c + 1, B, A, g, a.sc, s_dn, s_up);
        }
        // drain
        for (; c <= c_end; ++c) {
            tblock_step<Real, VEC, T, MAP, STRICT, RING, false>(c, A, B, g, a.sc, s_dn, s_up);
#pragma unroll
            for (int s = 0; s < T; ++s) {
                TBStage<Real, VEC> t = A[s]; A[s] = B[s]; B[s] = t;
            }
        }
        g.k0 += c_hi - cs + 1;
    }
}

}  // namespace bpltv
