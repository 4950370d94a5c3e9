// Common device helpers for the gpso_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace gpso {

constexpr int KERNEL_MATERN12 = 0;
constexpr int KERNEL_MATERN32 = 1;
constexpr int KERNEL_MATERN52 = 2;
constexpr int KERNEL_SE = 3;
constexpr int KERNEL_RQ = 4;  // gpflow.kernels.RationalQuadratic: one more hyper-parameter, the shape alpha

constexpr int TB = 128;           // tile / panel edge: every dense matrix is padded to a multiple of TB
constexpr double R2_CLIP = 1e-36; // GPflow clips the scaled squared distance before the sqrt (Matern kernels)

// tf.maximum(r2, 1e-36) propagates NaN (a NaN input must reach the Cholesky and be reported, not be clipped away);
// fmax() would return the non-NaN operand
__device__ __forceinline__ double clip_r2(double r2) { return (r2 < R2_CLIP) ? R2_CLIP : r2; }

// ---- FP64 tensor op: D(8x8) = A(8x4) * B(4x8) + C.  SASS: DMMA.8x8x4 -------------------------------------------
// fragment layout (g = lane>>2, t = lane&3):  a = A[g][t],  b = B[t][g],  c0 = C[g][2t], c1 = C[g][2t+1]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// ---- cp.async (LDGSTS) 16-byte global->shared copies ------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// ---- exp(-s) for s >= 0 -----------------------------------------------------------------------------------------------
// Every covariance function on the path evaluates exp of a non-positive argument.  Branch-free Cody-Waite reduction
// (n = rint(-s log2 e) by the 1.5*2^52 trick, r = -s - n ln2 in two FMAs) and a degree-13 Horner polynomial; the result
// is scaled by adding n to the exponent field.  19 FP64-pipe operations against ~26 DFMA-equivalents of exp()
// (profiles/r01_fp64_probe.txt) and no per-call constant materialisation; max relative error 2.2e-16 on [0, 690]
// (the same as libm's exp against long double), exactly 1 at s = 0, 0 beyond s = 700 (true value < 1e-304), NaN -> NaN.
__device__ __forceinline__ double exp_neg(double s) {
    const double MAGIC = 6755399441055744.0;
    double t = fma(-s, 1.4426950408889634074, MAGIC);
    double nf = t - MAGIC;
    int n = __double2loint(t);
    double r = fma(-nf, 6.93147180369123816490e-01, -s);
    r = fma(-nf, 1.90821492927058770002e-10, r);
    double p = 1.0 / 6227020800.0;
    p = fma(p, r, 1.0 / 479001600.0);
    p = fma(p, r, 1.0 / 39916800.0);
    p = fma(p, r, 1.0 / 3628800.0);
    p = fma(p, r, 1.0 / 362880.0);
    p = fma(p, r, 1.0 / 40320.0);
    p = fma(p, r, 1.0 / 5040.0);
    p = fma(p, r, 1.0 / 720.0);
    p = fma(p, r, 1.0 / 120.0);
    p = fma(p, r, 1.0 / 24.0);
    p = fma(p, r, 1.0 / 6.0);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    double v = __longlong_as_double(__double_as_longlong(p) + ((long long)n << 52));
    v = (s > 700.0) ? 0.0 : v;
    return (s != s) ? s : v;
}

// ---- sqrt of a positive finite number ---------------------------------------------------------------------------------
// sqrt(x) = x / sqrt(x):  hardware seed y ~ 1/sqrt(x) (MUFU.RSQ64H, ~2^-22) and one third-order correction
// y(1 + e/2 + 3e^2/8), e = 1 - x y^2 (remaining error < 2^-64 before the final rounding; result within 1.5 ulp, measured
// 1.4e-16 in tools/microbench/diag_probe.cu).  7 FP64-pipe operations instead of the ~17 DFMA-equivalents of the IEEE
// sqrt() (profiles/r01_fp64_probe.txt).  The argument is always >= 1e-36 here (GPflow's clip).  NaN -> NaN.
__device__ __forceinline__ double sqrt_pos(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double t = x * y;          // ~ sqrt(x)
    const double e = fma(-t, y, 1.0);
    const double pl = fma(0.375, e, 0.5);
    const double q = t * e;
    return fma(q, pl, t);
}

// exp_neg's constants for the W-wide forms below (the first object in constant memory: its bank offsets stay put)
__constant__ double EXPNEG_C[16] = {
    1.4426950408889634074,        // 0: log2(e)
    6.93147180369123816490e-01,   // 1: ln2 high
    1.90821492927058770002e-10,   // 2: ln2 low
    1.0 / 6227020800.0, 1.0 / 479001600.0, 1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 362880.0, 1.0 / 40320.0, 1.0 / 5040.0,
    1.0 / 720.0, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0,  // 3..13: 1/13! .. 1/3!
    2.23606797749978969641,       // 14: sqrt(5)
    1.73205080756887729353,       // 15: sqrt(3)
};

// ---- log(1 + z) for z >= 0 --------------------------------------------------------------------------------------------
// The RationalQuadratic covariance is var * exp(-alpha log1p(z)), z = r2 / (2 alpha): an absolute error d of log1p costs
// k * alpha * d, unbounded in alpha, so log1p must be accurate RELATIVE to its result, also near z = 0.  Branch-free:
//   z < sqrt2 - 1:  f = z exactly (no rounding of 1 + z), e = 0
//   otherwise:      1 + z = u + c exactly (Fast2Sum of max(1, z) and min(1, z)), u = 2^e m, m in [sqrt(1/2), sqrt(2)), f = m - 1
// and log1p(f) by fdlibm's e_log.c kernel: s = f / (2 + f), R(s^2) degree-7 minimax (error < 2^-58.45),
//   log1p(z) = e ln2_hi - ((f^2/2 - (s (f^2/2 + R) + (e ln2_lo + c / u))) - f).
// The reciprocal 1/(2 + f) is the MUFU.RCP64H seed with a third-order correction (as sqrt_pos); c / u <= 2^-53 is a
// correction only where the result is >= log(sqrt 2), so the bare seed serves there.  Result within a few ulp relative
// (tests/rq_oracle.py emulates it); exactly 0 at z = 0; +inf -> +inf; NaN -> NaN.  22 FP64-pipe operations.
__constant__ double LOG1P_C[7] = {
    6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01,
    1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01,  // fdlibm Lg1 .. Lg7
};
constexpr double LOG1P_SPLIT = 0.41421356237309503;  // sqrt(2) - 1

__device__ __forceinline__ double rcp_pos(double x) {  // 1/x for x in [1, 3]: seed + third-order correction
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x, y, 1.0);
    return fma(y, fma(e, e, e), y);
}

__device__ __forceinline__ double log1p_pos(double z) {
    const bool big = z >= LOG1P_SPLIT;
    const double a = big ? fmax(z, 1.0) : 1.0;
    const double b = big ? fmin(z, 1.0) : z;
    const double u = a + b;
    const double c = b - (u - a);
    int hx = __double2hiint(u) + (0x3ff00000 - 0x3fe6a09e);
    const int e = big ? (hx >> 20) - 0x3ff : 0;
    hx = (hx & 0x000fffff) + 0x3fe6a09e;
    const double f = big ? __hiloint2double(hx, __double2loint(u)) - 1.0 : z;
    double cu;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(cu) : "d"(u));
    cu = big ? c * cu : 0.0;
    const double s = f * rcp_pos(2.0 + f);
    const double w = s * s;
    double R = LOG1P_C[6];
#pragma unroll
    for (int i = 5; i >= 0; i--) R = fma(R, w, LOG1P_C[i]);
    R *= w;
    const double hfsq = 0.5 * f * f;
    const double ed = (double)e;
    const double v = fma(ed, 6.93147180369123816490e-01, -((hfsq - fma(s, hfsq + R, fma(ed, 1.90821492927058770002e-10, cu))) - f));
    return (z > 1.7976931348623157e308) ? z : v;
}

// ---- z = r2 / (2 alpha) of the RationalQuadratic kernel ---------------------------------------------------------------
// z = (r2 * ia) * sc with ia = 0.5 / (alpha / sc), both factors formed once per thread (rq_scale): two multiplications per
// element instead of a division, within an ulp or two of GPflow's 0.5 * r2 / alpha.  sc = 1 while 0.5 / alpha is finite;
// below alpha = 2^-1000 (softplus(u_alpha) for u_alpha < -693, which L-BFGS-B line searches do probe) 0.5 / alpha alone would
// overflow and r2 = 0 would give 0 * inf = NaN, so alpha is scaled by 2^600 first: r2 = 0 gives z = 0 and z overflows to inf
// where GPflow's quotient does.  alpha = 0 gives ia = inf; the callers select k = var there.
__device__ __forceinline__ void rq_scale(double alpha, double& ia, double& sc) {
    const bool tiny = alpha < 0x1p-1000;
    sc = tiny ? 0x1p600 : 1.0;
    ia = 0.5 / (tiny ? alpha * 0x1p600 : alpha);
}
__device__ __forceinline__ double rq_z(double r2, double ia, double sc) { return (r2 * ia) * sc; }

// ---- covariance functions (gpflow.kernels.stationaries) ----------------------------------------------------------
// r2 = scaled squared distance (inputs already divided by the lengthscale), var = kernel variance, alpha = the
// RationalQuadratic shape (read by KERNEL_RQ only).  RQ: var * (1 + r2 / (2 alpha))^-alpha = var * exp(-alpha log1p(z));
// alpha = 0 (softplus underflow) gives var for every pair, as pow(x, -0) = 1 does in GPflow.
template <int KID>
__device__ __forceinline__ double cov_from_r2(double r2, double var, double alpha) {
    if (KID == KERNEL_RQ) {
        double ia, sc;
        rq_scale(alpha, ia, sc);
        const double E = alpha * log1p_pos(rq_z(r2, ia, sc));
        return var * exp_neg(alpha > 0.0 ? E : 0.0);
    } else if (KID == KERNEL_SE) {
        return var * exp_neg(0.5 * r2);
    } else {
        double r = sqrt_pos(clip_r2(r2));
        if (KID == KERNEL_MATERN52) {
            const double s5 = 2.23606797749978969641;
            double sr = s5 * r;
            // variance * (1 + sqrt5 r + 5/3 r^2) * exp(-sqrt5 r), GPflow's evaluation order
            return var * (1.0 + sr + (5.0 / 3.0) * (r * r)) * exp_neg(sr);
        } else if (KID == KERNEL_MATERN32) {
            const double s3 = 1.73205080756887729353;
            double sr = s3 * r;
            return var * (1.0 + sr) * exp_neg(sr);
        } else {
            return var * exp_neg(r);
        }
    }
}

// ---- W-wide variants for the hot cross-covariance loop ---------------------------------------------------------------
// The same operation sequences as exp_neg / sqrt_pos / cov_from_r2 (bit-identical results), written over W independent
// arguments so that the W dependent chains interleave in the instruction stream (the scalar forms compile to one serial
// chain per element, ~8 clk between dependent DFMAs), with the 64-bit polynomial coefficients read from the constant bank
// as DFMA operands instead of being rebuilt by two UMOV / IMAD.MOV per use (28 of 140 instructions per element before).

template <int W>
__device__ __forceinline__ void exp_neg_v(const double (&s)[W], double (&v)[W]) {
    const double MAGIC = 6755399441055744.0;
    double nf[W], r[W], p[W];
    int n[W];
#pragma unroll
    for (int i = 0; i < W; i++) {
        double t = fma(-s[i], EXPNEG_C[0], MAGIC);
        nf[i] = t - MAGIC;
        n[i] = __double2loint(t);
    }
#pragma unroll
    for (int i = 0; i < W; i++) r[i] = fma(-nf[i], EXPNEG_C[1], -s[i]);
#pragma unroll
    for (int i = 0; i < W; i++) r[i] = fma(-nf[i], EXPNEG_C[2], r[i]);
#pragma unroll
    for (int i = 0; i < W; i++) p[i] = fma(EXPNEG_C[3], r[i], EXPNEG_C[4]);
#pragma unroll
    for (int c = 5; c <= 13; c++) {
#pragma unroll
        for (int i = 0; i < W; i++) p[i] = fma(p[i], r[i], EXPNEG_C[c]);
    }
#pragma unroll
    for (int i = 0; i < W; i++) p[i] = fma(p[i], r[i], 0.5);
#pragma unroll
    for (int i = 0; i < W; i++) p[i] = fma(p[i], r[i], 1.0);
#pragma unroll
    for (int i = 0; i < W; i++) p[i] = fma(p[i], r[i], 1.0);
#pragma unroll
    for (int i = 0; i < W; i++) {
        double x = __longlong_as_double(__double_as_longlong(p[i]) + ((long long)n[i] << 52));
        x = (s[i] > 700.0) ? 0.0 : x;
        v[i] = (s[i] != s[i]) ? s[i] : x;
    }
}

template <int W>
__device__ __forceinline__ void sqrt_pos_v(const double (&x)[W], double (&out)[W]) {
    double y[W], t[W], e[W];
#pragma unroll
    for (int i = 0; i < W; i++) asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y[i]) : "d"(x[i]));
#pragma unroll
    for (int i = 0; i < W; i++) t[i] = x[i] * y[i];
#pragma unroll
    for (int i = 0; i < W; i++) e[i] = fma(-t[i], y[i], 1.0);
#pragma unroll
    for (int i = 0; i < W; i++) {
        const double pl = fma(0.375, e[i], 0.5);
        const double q = t[i] * e[i];
        out[i] = fma(q, pl, t[i]);
    }
}

// log1p_pos over W arguments, the same operation sequence stage by stage
template <int W>
__device__ __forceinline__ void log1p_pos_v(const double (&z)[W], double (&out)[W]) {
    double u[W], cu[W], f[W], ed[W], s[W], w[W], R[W];
#pragma unroll
    for (int i = 0; i < W; i++) {
        const bool big = z[i] >= LOG1P_SPLIT;
        const double a = big ? fmax(z[i], 1.0) : 1.0;
        const double b = big ? fmin(z[i], 1.0) : z[i];
        u[i] = a + b;
        const double c = b - (u[i] - a);
        int hx = __double2hiint(u[i]) + (0x3ff00000 - 0x3fe6a09e);
        ed[i] = (double)(big ? (hx >> 20) - 0x3ff : 0);
        hx = (hx & 0x000fffff) + 0x3fe6a09e;
        f[i] = big ? __hiloint2double(hx, __double2loint(u[i])) - 1.0 : z[i];
        double r;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(u[i]));
        cu[i] = big ? c * r : 0.0;
    }
#pragma unroll
    for (int i = 0; i < W; i++) s[i] = f[i] * rcp_pos(2.0 + f[i]);
#pragma unroll
    for (int i = 0; i < W; i++) {
        w[i] = s[i] * s[i];
        R[i] = LOG1P_C[6];
    }
#pragma unroll
    for (int c = 5; c >= 0; c--) {
#pragma unroll
        for (int i = 0; i < W; i++) R[i] = fma(R[i], w[i], LOG1P_C[c]);
    }
#pragma unroll
    for (int i = 0; i < W; i++) {
        R[i] *= w[i];
        const double hfsq = 0.5 * f[i] * f[i];
        const double v = fma(ed[i], 6.93147180369123816490e-01,
                             -((hfsq - fma(s[i], hfsq + R[i], fma(ed[i], 1.90821492927058770002e-10, cu[i]))) - f[i]));
        out[i] = (z[i] > 1.7976931348623157e308) ? z[i] : v;
    }
}

template <int KID, int W>
__device__ __forceinline__ void cov_from_r2_v(const double (&r2)[W], double var, double alpha, double (&k)[W]) {
    double s[W], e[W];
    if (KID == KERNEL_RQ) {
        double ia, sc;
        rq_scale(alpha, ia, sc);
#pragma unroll
        for (int i = 0; i < W; i++) s[i] = rq_z(r2[i], ia, sc);
        log1p_pos_v<W>(s, e);
#pragma unroll
        for (int i = 0; i < W; i++) s[i] = alpha > 0.0 ? alpha * e[i] : 0.0;
        exp_neg_v<W>(s, e);
#pragma unroll
        for (int i = 0; i < W; i++) k[i] = var * e[i];
    } else if (KID == KERNEL_SE) {
#pragma unroll
        for (int i = 0; i < W; i++) s[i] = 0.5 * r2[i];
        exp_neg_v<W>(s, e);
#pragma unroll
        for (int i = 0; i < W; i++) k[i] = var * e[i];
    } else {
        double c[W], r[W];
#pragma unroll
        for (int i = 0; i < W; i++) c[i] = clip_r2(r2[i]);
        sqrt_pos_v<W>(c, r);
        if (KID == KERNEL_MATERN52) {
#pragma unroll
            for (int i = 0; i < W; i++) s[i] = EXPNEG_C[14] * r[i];
            exp_neg_v<W>(s, e);
#pragma unroll
            for (int i = 0; i < W; i++) k[i] = var * (1.0 + s[i] + (5.0 / 3.0) * (r[i] * r[i])) * e[i];
        } else if (KID == KERNEL_MATERN32) {
#pragma unroll
            for (int i = 0; i < W; i++) s[i] = EXPNEG_C[15] * r[i];
            exp_neg_v<W>(s, e);
#pragma unroll
            for (int i = 0; i < W; i++) k[i] = var * (1.0 + s[i]) * e[i];
        } else {
            exp_neg_v<W>(r, e);
#pragma unroll
            for (int i = 0; i < W; i++) k[i] = var * e[i];
        }
    }
}

// covariance value and the radial factor g with  dK/d(ls_j) = g * Delta_j^2 / ls_j^3  (Delta in UNscaled units),
// i.e. for a scalar lengthscale dK/d(ls) = g * r2 / ls.  g = 0 where r2 was clipped (GPflow: zero gradient there).
// RQ also gives ka = dk/dalpha = k (z / (1 + z) - log1p(z)), 0 where k = 0; g = k / (1 + z).  alpha = 0: k = var, g = ka = 0 (the host
// zeroes the alpha entry there: its chain factor sigmoid(u) is 0).
template <int KID>
__device__ __forceinline__ void cov_and_radial(double r2, double var, double alpha, double& k, double& g, double& ka) {
    if (KID == KERNEL_RQ) {
        double ia, sc;
        rq_scale(alpha, ia, sc);
        const double z = rq_z(r2, ia, sc);
        const double l = log1p_pos(z);
        const bool live = alpha > 0.0;
        k = var * exp_neg(live ? alpha * l : 0.0);
        const double iu = 1.0 / (1.0 + z);
        g = live ? k * iu : 0.0;
        ka = (live && k != 0.0) ? k * (z * iu - l) : 0.0;  // k = 0 (z = inf): the limit 0, not 0 * (inf * 0 - inf)
    } else if (KID == KERNEL_SE) {
        k = var * exp_neg(0.5 * r2);
        g = k;
    } else {
        bool live = r2 > R2_CLIP;
        double r = sqrt_pos(clip_r2(r2));
        if (KID == KERNEL_MATERN52) {
            const double s5 = 2.23606797749978969641;
            double sr = s5 * r;
            double e = exp_neg(sr);
            k = var * (1.0 + sr + (5.0 / 3.0) * (r * r)) * e;
            g = live ? (5.0 / 3.0) * var * (1.0 + sr) * e : 0.0;
        } else if (KID == KERNEL_MATERN32) {
            const double s3 = 1.73205080756887729353;
            double sr = s3 * r;
            double e = exp_neg(sr);
            k = var * (1.0 + sr) * e;
            g = live ? 3.0 * var * e : 0.0;
        } else {
            k = var * exp_neg(r);
            g = live ? k / r : 0.0;
        }
    }
}

// ---- sum kernel (gpflow.kernels.Sum) -----------------------------------------------------------------------------------
// k = sum_c k_c in component order, each component one of the five families above with its own variance, alpha and
// lengthscales.  Component c reads its own scaled inputs Xs_c = X / ls_c, stored at Xs + c * d * Np ([C][d][Np]), and its
// lengthscales expanded to d entries at ls + c * d.  The table travels by value as the last kernel argument (constant bank):
// every thread reads the same family, so the switch below never diverges.
constexpr int KERNEL_SUM = 5;
constexpr int MAX_SUM = 4;
struct SumTable {
    int n;                 // components, 1..MAX_SUM (0 in the launches of the other kernels, which never read the table)
    int fam[MAX_SUM];      // KERNEL_MATERN12 .. KERNEL_RQ
    double var[MAX_SUM];   // component variances (a product: {var_prod, 1, 1, 1})
    double alpha[MAX_SUM]; // RationalQuadratic shape (read for KERNEL_RQ components only)
};

// The rows of a sum or product's components, read by the KERNEL_SUM_EMB / KERNEL_PRODUCT_EMB instantiations only (a sum or product
// with periodic components; appended last to the covariance kernels, a separate argument so that the table above keeps its
// layout): component c covers the rows [off[c], off[c] + rows[c]) of the scaled inputs and of the width-wide candidate rows
// (rows[c] = 2d for a periodic component's embedded rows, d otherwise); pmask has bit c set for a periodic component.
struct SumRows {
    int off[MAX_SUM], rows[MAX_SUM], width, pmask;
};

__device__ __forceinline__ double sum_term(const SumTable& t, int c, double r2) {
    const double v = t.var[c], a = t.alpha[c];
    switch (t.fam[c]) {
        case KERNEL_MATERN12: return cov_from_r2<KERNEL_MATERN12>(r2, v, a);
        case KERNEL_MATERN32: return cov_from_r2<KERNEL_MATERN32>(r2, v, a);
        case KERNEL_MATERN52: return cov_from_r2<KERNEL_MATERN52>(r2, v, a);
        case KERNEL_SE: return cov_from_r2<KERNEL_SE>(r2, v, a);
        default: return cov_from_r2<KERNEL_RQ>(r2, v, a);
    }
}

// ---- product kernel (gpflow.kernels.Product) ---------------------------------------------------------------------------
// k = prod_c k_c in factor order, with the sum kernel's layout and table.  The table's variances are {var_prod, 1, 1, 1}
// (var_prod = prod_c var_c, fp64 in factor order): k = cov(r2_0; var_prod) * prod_{c>=1} cov(r2_c; 1), so k(x, x) is exactly
// var_prod, small factor variances cannot underflow in fp32, and a one-factor product is its bare kernel's operations.
constexpr int KERNEL_PRODUCT = 6;
// A sum / product with periodic components (gpflow.kernels.Periodic terms): the covariance kernels' instantiations for it read each
// component's rows at the table's offsets (the rows of a periodic component are its embedded inputs, at unit lengthscale, and
// its family is its base's), and the candidates as rows of the table's width.  Internal ids: the C ABI's id 7 is the periodic kernel.
constexpr int KERNEL_SUM_EMB = 8;
constexpr int KERNEL_PRODUCT_EMB = 9;
// A sum with Linear terms (gpflow.kernels.Linear, k(x, x') = sum_r var_r x_r x'_r: not stationary, so k(x, x) depends on x): the
// row layout of KERNEL_SUM_EMB, its own instantiations of gram_kernel, crosscov_kernel and joint_syrk_kernel.  A Linear component
// has the family KERNEL_LINEAR (the C ABI's GPSO_KERNEL_LINEAR) in the table, and its rows are its (active) columns divided by the
// "lengthscale" 1 / sqrt(var_r), so that its covariance is the plain dot product of its rows (sum_r (x_r / l_r)(x'_r / l_r)) and
// k(x, x) the squared norm of x's.
constexpr int KERNEL_LINEAR = 10;
constexpr int KERNEL_SUM_LIN = 11;
__host__ __device__ constexpr bool embedded_composite(int kid) { return kid == KERNEL_SUM_EMB || kid == KERNEL_PRODUCT_EMB; }
__host__ __device__ constexpr bool product_kernel(int kid) { return kid == KERNEL_PRODUCT || kid == KERNEL_PRODUCT_EMB; }
__host__ __device__ constexpr bool composite_kernel(int kid) {
    return kid == KERNEL_SUM || kid == KERNEL_PRODUCT || embedded_composite(kid);
}
// the running combination of the component values: added for a sum, multiplied for a product
template <int KID>
__device__ __forceinline__ double combine(double acc, double t) { return product_kernel(KID) ? acc * t : acc + t; }

template <int W>
__device__ __forceinline__ void sum_term_v(const SumTable& t, int c, const double (&r2)[W], double (&k)[W]) {
    const double v = t.var[c], a = t.alpha[c];
    switch (t.fam[c]) {
        case KERNEL_MATERN12: cov_from_r2_v<KERNEL_MATERN12, W>(r2, v, a, k); break;
        case KERNEL_MATERN32: cov_from_r2_v<KERNEL_MATERN32, W>(r2, v, a, k); break;
        case KERNEL_MATERN52: cov_from_r2_v<KERNEL_MATERN52, W>(r2, v, a, k); break;
        case KERNEL_SE: cov_from_r2_v<KERNEL_SE, W>(r2, v, a, k); break;
        default: cov_from_r2_v<KERNEL_RQ, W>(r2, v, a, k); break;
    }
}

// cov_and_radial of factor c's family (the product gradient), warp-uniform like sum_term
__device__ __forceinline__ void sum_term_radial(const SumTable& t, int c, double r2, double& k, double& g, double& ka) {
    const double v = t.var[c], a = t.alpha[c];
    ka = 0.0;
    switch (t.fam[c]) {
        case KERNEL_MATERN12: cov_and_radial<KERNEL_MATERN12>(r2, v, a, k, g, ka); break;
        case KERNEL_MATERN32: cov_and_radial<KERNEL_MATERN32>(r2, v, a, k, g, ka); break;
        case KERNEL_MATERN52: cov_and_radial<KERNEL_MATERN52>(r2, v, a, k, g, ka); break;
        case KERNEL_SE: cov_and_radial<KERNEL_SE>(r2, v, a, k, g, ka); break;
        default: cov_and_radial<KERNEL_RQ>(r2, v, a, k, g, ka); break;
    }
}

// ---- deterministic block reductions -----------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// sum over a block of NT threads (NT multiple of 32, <= 1024); result valid in thread 0; fixed order
template <int NT>
__device__ __forceinline__ double block_sum(double v, double* scratch /* >= NT/32 doubles */) {
    v = warp_sum(v);
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) scratch[w] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < NT / 32; i++) s += scratch[i];
    }
    return s;
}

// arg-max record with numpy semantics: first NaN wins, otherwise largest value, lowest index on ties
struct Best {
    double val;
    long long idx;
};
__device__ __forceinline__ bool best_better(double av, long long ai, double bv, long long bi) {
    bool an = isnan(av), bn = isnan(bv);
    if (an || bn) {
        if (an && bn) return ai < bi;
        return an;
    }
    if (av > bv) return true;
    if (av < bv) return false;
    return ai < bi;
}

}  // namespace gpso
