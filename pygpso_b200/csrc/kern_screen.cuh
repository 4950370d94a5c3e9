// Screen-and-refine arg-max: a cheap low-precision pass over ALL candidates that only has to decide which candidates can
// possibly be the arg-max; the few survivors are then re-scored by the full-precision engine (kern_ozaki.cuh, S = 5..8
// digits), whose record is what the call returns.  The returned (index, mean, var, ucb) is therefore bit-identical to the
// unscreened path as long as the true winner survives, which the error bound E below guarantees with a wide margin and the
// caller verifies on the survivors (gpso_capi.cu: score_argmax; on any doubt it falls back to the full pass).
//
// Why it pays: the full-precision product kernel is bound by L2 -> SM operand traffic, not by the tensor pipe (105.9 GB per
// 87 040-candidate window at N = 4096, S = 6 = 8.97 ms at the 11.8 TB/s the L2 delivers; profiles/r01s4_ncu_summary.md).
// Bytes per candidate scale with S * (128 + NT) / NT per (row block, k-step): S = 2 digits and NT = 128-candidate tiles move
// 4.5x fewer bytes (and 7x fewer MMA operations: 3 digit pairs instead of 21).
//
//   crosscov_screen_kernel   candidates -> k* in FP32 (FFMA / MUFU pipes: these co-issue with the int8 tensor pipe, unlike
//                            DFMA which shares its datapath, profiles/r01s4_corun_probe.txt) -> S balanced 8-bit digits
//                            [ct][ks][q][NT x 32] + posterior mean (fp32 products, fp64 accumulation across super-steps)
//   ozaki_screen_kernel      the tcgen05 kind::i8 product of kern_ozaki.cuh for S <= 4 with NT = 128 candidates per tile, TWO
//                            accumulator buffers in TMEM when 2 * S * NT <= 512 columns (the issuer never waits for the
//                            epilogue), and an FP32 epilogue (I2F / FFMA / FADD only: nothing on the FP64 datapath)
//   screen_finalize_kernel   ucb_s = mean_s + varsigma * var_s per candidate -> scr_ucb[global index]; running maximum
//   screen_select_kernel     survivors = { c : ucb_s(c) is NaN  or  ucb_s(c) >= max_c ucb_s - 2E }  -> index list
//   gather_rows_kernel       survivor coordinates -> compact matrix for the refine pass
//   screen_check_kernel      max |ucb_refined - ucb_s| over the survivors (must stay below E / 4)
#pragma once
#include "kern_ozaki.cuh"

namespace gpso {

constexpr int SCR_NT = 128;  // candidates per tile of the screening product

// FULL: all S^2 digit pairs are kept (levels 0 .. 2S-2): the product of the S-digit operands is then exact and the only error
// left is the operand rounding -- at S = 2 that is 4 pairs instead of the 6 of the triangular 3-digit product, with 16 KB
// instead of 24 KB of operands per k-step.  (The triangular 2-digit product drops the pair (1,1), which is as large as the result.)
template <int S, int NT, bool FULL = false>
struct ScrCfg {
    static constexpr int A_BYTES = S * OZ_A_SLICE;
    static constexpr int B_SLICE = NT * 32;
    static constexpr int B_BYTES = S * B_SLICE;
    // k-steps (of 32) per ring stage: one bulk copy of A and one of B per stage (consecutive k-steps are contiguous in both
    // digit buffers) and ONE tcgen05.commit per stage -- every row block has a multiple of 4 k-steps.  The 2-digit full product
    // takes four (64 KB of operands per stage, three stages): 41.8 vs 43.4 ms per 2.1e6 candidates against two k-steps x six stages
    static constexpr int KPS = FULL ? 4 : 2;
    static constexpr int STAGE_BYTES = KPS * (A_BYTES + B_BYTES);
    // the ring is what hides the L2 latency: bytes in flight / latency is the operand bandwidth this CTA can draw (24 KB
    // chunks, 8 in flight reach 20 TB/s chip-wide, profiles/r01_i8_tcgen05_probe.txt).  192 KB leave room for one
    // cross-covariance block of the next window on the same SM.
    static constexpr int STAGES = (192 * 1024 / STAGE_BYTES) > 12 ? 12 : (192 * 1024 / STAGE_BYTES);
    static constexpr int RING_BYTES = STAGES * STAGE_BYTES;
    static constexpr int LEVELS = FULL ? 2 * S - 1 : S;           // digit-pair levels p + q kept
    static constexpr int ACC_COLS = LEVELS * NT;                  // TMEM columns of one accumulator buffer
    static constexpr int NBUF = (2 * ACC_COLS <= OZ_TMEM_COLS) ? 2 : 1;
    static constexpr int SMEM_BYTES = RING_BYTES + 1024 + 4 * NT * (int)sizeof(float);
    static_assert(ACC_COLS <= OZ_TMEM_COLS, "accumulator levels do not fit in TMEM");
    static_assert(NT == 64 || NT == 128 || NT == 256, "tile width");
};

struct ScrParams {
    const uint8_t* A;        // [nb][nks][S][4096]
    const uint8_t* B;        // [nct][nks][S][NT*32]
    const double* rowscale;  // [Np] 2^(e_i)
    float* part;             // [nb][ldp]  sum over the 128 rows of block I of (L^-1 k*)^2, fp32
    double gscale;
    int nb, nks, nct;
    long long ldp;
};

// ---- FP32 covariance (screening only) -----------------------------------------------------------------------------------
// Absolute error against the fp64 evaluation below 2e-6 * variance for every kernel family (tests/test_screen_model.py
// checks the same formulas in numpy float32; MUFU.EX2 / MUFU.RSQ add ~2 ulp each).  NaN propagates.
//
// RationalQuadratic: k = var * 2^(-alpha log2(1 + z)), z = r2 / (2 alpha).  An absolute error d of log2(1 + z) costs
// k * alpha * ln2 * d, unbounded in alpha, so log2(1 + z) must be accurate relative to its result:
//   z <  1/4:  z * P(z), P the degree-5 relative-minimax fit of log2(1 + z) / z (fit error 9e-9, 1.2e-7 after fp32 Horner)
//   z >= 1/4:  MUFU.LG2 of fl(1 + z): absolute error ~1.6e-7 plus the rounding of 1 + z, on a result >= log2(1.25) = 0.32
// i.e. a relative error rho < 8e-7, and since x e^-x <= 1/e the covariance error stays below var * rho / e for every alpha.
// tests/rq_oracle.py emulates this evaluation in numpy float32.
constexpr float RQ32_SPLIT = 0.25f;
__constant__ float RQ32_P[6] = {  // log2(e) times the fit of log1p(z) / z on [0, 1/4]
    1.4426950216293335f, -0.7213437557220459f, 0.48071789741516113f, -0.357472687959671f, 0.26215097308158875f, -0.1332305371761322f,
};

template <int KID>
__device__ __forceinline__ float cov32_from_r2(float r2, float var, float alpha) {
    if (KID == KERNEL_RQ) {
        const float z = r2 * __fdividef(0.5f, alpha);
        float p = RQ32_P[5];
#pragma unroll
        for (int i = 4; i >= 0; i--) p = fmaf(p, z, RQ32_P[i]);
        const float l2 = (z < RQ32_SPLIT) ? z * p : __log2f(1.0f + z);
        return var * exp2f(-alpha * l2);
    } else if (KID == KERNEL_SE) {
        return var * __expf(-0.5f * r2);
    } else {
        const float c = (r2 < 1e-36f) ? 1e-36f : r2;
        const float r = c * rsqrtf(c);
        if (KID == KERNEL_MATERN52) {
            const float s = 2.2360679775f * r;
            return var * (1.0f + s + 1.6666666667f * (r * r)) * __expf(-s);
        } else if (KID == KERNEL_MATERN32) {
            const float s = 1.7320508076f * r;
            return var * (1.0f + s) * __expf(-s);
        } else {
            return var * __expf(-r);
        }
    }
}

// ---- packed FP32 pairs (sm_100: add / mul / fma .f32x2 -> FADD2 / FMUL2 / FFMA2, one issue slot for two lanes of work) ---------
// The cross-covariance kernel is issue-bound (83 % of the issue slots busy, FMA pipe 50 %, profiles/r02_ncu_screen_kernels.csv):
// its two candidates per thread ride in the two halves of one 64-bit register.
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t f2_pack(float lo, float hi) {
    f32x2_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(f32x2_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2_t f2_sub(f32x2_t a, f32x2_t b) {
    f32x2_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2_t f2_add(f32x2_t a, f32x2_t b) {
    f32x2_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2_t f2_mul(f32x2_t a, f32x2_t b) {
    f32x2_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2_t f2_fma(f32x2_t a, f32x2_t b, f32x2_t c) {
    f32x2_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float scr_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float scr_rsqrt(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// cov32_from_r2 for the two halves of a packed pair (same formulas; exp(-s) = 2^(-s log2 e))
__device__ __forceinline__ float scr_lg2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

template <int KID>
__device__ __forceinline__ f32x2_t cov32x2_from_r2(f32x2_t r2, float var, float alpha) {
    const float L2E = 1.4426950408889634f;
    const f32x2_t var2 = f2_pack(var, var);
    float a, b;
    if (KID == KERNEL_RQ) {
        const float ia = __fdividef(0.5f, alpha);
        const f32x2_t z = f2_mul(r2, f2_pack(ia, ia));
        f32x2_t p = f2_pack(RQ32_P[5], RQ32_P[5]);
#pragma unroll
        for (int i = 4; i >= 0; i--) p = f2_fma(p, z, f2_pack(RQ32_P[i], RQ32_P[i]));
        p = f2_mul(p, z);
        const f32x2_t u = f2_add(z, f2_pack(1.0f, 1.0f));
        float za, zb, pa, pb, ua, ub;
        f2_unpack(z, za, zb);
        f2_unpack(p, pa, pb);
        f2_unpack(u, ua, ub);
        // z < 1/4 (and not NaN): the polynomial; otherwise the MUFU logarithm (NaN propagates through it)
        const f32x2_t l2 = f2_pack((za < RQ32_SPLIT) ? pa : scr_lg2(ua), (zb < RQ32_SPLIT) ? pb : scr_lg2(ub));
        f2_unpack(f2_mul(l2, f2_pack(-alpha, -alpha)), a, b);
        return f2_mul(var2, f2_pack(scr_ex2(a), scr_ex2(b)));
    } else if (KID == KERNEL_SE) {
        const f32x2_t t = f2_mul(r2, f2_pack(-0.5f * L2E, -0.5f * L2E));
        f2_unpack(t, a, b);
        return f2_mul(var2, f2_pack(scr_ex2(a), scr_ex2(b)));
    } else {
        f2_unpack(r2, a, b);
        a = (a < 1e-36f) ? 1e-36f : a;  // NaN propagates (a select, not fmaxf)
        b = (b < 1e-36f) ? 1e-36f : b;
        const f32x2_t c = f2_pack(a, b);
        const f32x2_t r = f2_mul(c, f2_pack(scr_rsqrt(a), scr_rsqrt(b)));
        if (KID == KERNEL_MATERN52) {
            const f32x2_t s = f2_mul(r, f2_pack(2.2360679775f, 2.2360679775f));
            const f32x2_t t = f2_mul(s, f2_pack(-L2E, -L2E));
            f2_unpack(t, a, b);
            const f32x2_t e = f2_pack(scr_ex2(a), scr_ex2(b));
            // 1 + s + 5/3 r^2
            const f32x2_t poly = f2_add(f2_fma(f2_mul(r, r), f2_pack(1.6666666667f, 1.6666666667f), s), f2_pack(1.0f, 1.0f));
            return f2_mul(f2_mul(var2, poly), e);
        } else if (KID == KERNEL_MATERN32) {
            const f32x2_t s = f2_mul(r, f2_pack(1.7320508076f, 1.7320508076f));
            const f32x2_t t = f2_mul(s, f2_pack(-L2E, -L2E));
            f2_unpack(t, a, b);
            const f32x2_t e = f2_pack(scr_ex2(a), scr_ex2(b));
            return f2_mul(f2_mul(var2, f2_add(s, f2_pack(1.0f, 1.0f))), e);
        } else {
            const f32x2_t t = f2_mul(r, f2_pack(-L2E, -L2E));
            f2_unpack(t, a, b);
            return f2_mul(var2, f2_pack(scr_ex2(a), scr_ex2(b)));
        }
    }
}

// balanced base-256 digits of an integer |X| < 2^(8S-2), S <= 4 (32-bit form of oz_digits)
template <int S>
__device__ __forceinline__ uint32_t scr_digits(float k, float scale) {
    const int X = __float2int_rn(k * scale);
    constexpr uint32_t C = (S >= 4) ? 0x00808080u : (S == 3) ? 0x00008080u : 0x00000080u;
    return ((uint32_t)X + C) ^ C;
}

// fp32 copies of the scaled training inputs and of alpha (once per factorisation)
__global__ void __launch_bounds__(256) screen_convert_kernel(const double* __restrict__ Xs, const double* __restrict__ alpha, int d,
                                                             int Np, float* __restrict__ Xs32, float* __restrict__ alpha32) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i < d * Np) Xs32[i] = (float)Xs[i];
    if (i < Np) alpha32[i] = (float)alpha[i];
}

// S = 0: posterior mean only (no digit tiles are formed or written): the first level of the bound-and-refine arg-max, which
// needs nothing but the mean of every candidate (gpso_capi.cu: bound_pass).
// One block = 64 candidates x all training points (super-steps of 128 training points), the register tiling of
// crosscov_slices_kernel in FP32: thread = 2 candidates (lane, lane + 32) x 16 consecutive training points (warp w owns
// points 16 w .. 16 w + 15 of the super-step).  The digit tiles are written in the NT-candidate layout of the screening
// product.  Candidates with a NaN or huge coordinate get a NaN mean (-> NaN screened UCB -> always refined).
template <int KID, int S, int NT>
__global__ void __launch_bounds__(256, 2) crosscov_screen_kernel(const double* __restrict__ Xc, long long Mw, int d,
                                                                 const double* __restrict__ ls, int n_ls,
                                                                 const float* __restrict__ Xs32, const float* __restrict__ alpha32,
                                                                 int N, int Np, float var, double c0, float bscale, int nks,
                                                                 uint8_t* __restrict__ B, double* __restrict__ mean, float rq_alpha,
                                                                 SumTable sum, SumRows srow) {
    // sum / product: the C components' scaled coordinates are dx = C d rows ([C][d] component-major), in Xs32 and in shared memory alike
    const int dx = embedded_composite(KID) ? srow.width : (composite_kernel(KID) ? sum.n * d : d);
    extern __shared__ __align__(16) float smf[];
    float* sC = smf;                       // [dx][64]
    float* sX = sC + dx * 64;              // [2][dx][128]
    float* sAl = sX + 2 * dx * OZ_XK;      // [2][128]
    double* sR = reinterpret_cast<double*>(sAl + 2 * OZ_XK);  // [8][64]
    __shared__ int sBad[64];
    const int tid = threadIdx.x, cl = tid & 31, kg = tid >> 5;
    const long long blk = blockIdx.x;      // 64-candidate group
    if (tid < 64) sBad[tid] = 0;
    __syncthreads();
    if constexpr (composite_kernel(KID)) {
        for (int e = tid; e < 64 * dx; e += 256) {
            const int cc = e / dx, qd = e - cc * dx, dim = qd % d;  // qd = q d + dim: component q's own lengthscales
            const long long cg = blk * 64 + cc;
            double x = 0.0;
            if (cg < Mw) {
                x = Xc[embedded_composite(KID) ? cg * dx + qd : cg * d + dim] / ls[qd];  // periodic components: rows of width dx
                if (!(fabs(x) <= 1.0e15)) sBad[cc] = 1;
            }
            sC[qd * 64 + cc] = (float)x;
        }
    } else {
        for (int e = tid; e < 64 * d; e += 256) {
            const int cc = e / d, dim = e - cc * d;
            const long long cg = blk * 64 + cc;
            double x = 0.0;
            if (cg < Mw) {
                x = Xc[cg * d + dim] / ls[n_ls > 1 ? dim : 0];
                if (!(fabs(x) <= 1.0e15)) sBad[cc] = 1;  // NaN, inf or beyond the fp32-safe range (benign race: all write 1)
            }
            sC[dim * 64 + cc] = (float)x;
        }
    }
    for (int e = tid; e < dx * (OZ_XK / 4); e += 256) {
        const int dim = e >> 5, q4 = (e & 31) * 4;
        cp_async16(sX + dim * OZ_XK + q4, Xs32 + (size_t)dim * Np + q4);
    }
    if (tid < OZ_XK / 4) cp_async16(sAl + tid * 4, alpha32 + tid * 4);
    cp_async_commit();
    const bool cvalid[2] = {blk * 64 + cl < Mw, blk * 64 + cl + 32 < Mw};
    double macc[2] = {0.0, 0.0};
    const int nss = Np / OZ_XK;
    // position of this block's candidates inside their NT-wide tile
    const long long ct = (blk * 64) / NT;
    const int rbase = (int)((blk * 64) % NT);
    for (int ss = 0; ss < nss; ss++) {
        cp_async_wait<0>();
        __syncthreads();
        const int b = ss & 1;
        if (ss + 1 < nss) {
            float* nx = sX + (b ^ 1) * dx * OZ_XK;
            for (int e = tid; e < dx * (OZ_XK / 4); e += 256) {
                const int dim = e >> 5, q4 = (e & 31) * 4;
                cp_async16(nx + dim * OZ_XK + q4, Xs32 + (size_t)dim * Np + (ss + 1) * OZ_XK + q4);
            }
            if (tid < OZ_XK / 4) cp_async16(sAl + (b ^ 1) * OZ_XK + tid * 4, alpha32 + (ss + 1) * OZ_XK + tid * 4);
            cp_async_commit();
        }
        const float* x = sX + b * dx * OZ_XK + kg * 16;
        // squared distances of this thread's two candidates (low / high half) to its 16 training points
        f32x2_t r2[16];
#pragma unroll
        for (int i = 0; i < 16; i++) r2[i] = 0ULL;
        f32x2_t kv[16];  // sum / product: the covariance, component values added (multiplied) in order in fp32
        if constexpr (composite_kernel(KID)) {
            for (int q = 0; q < sum.n; q++) {
                f32x2_t rq[16];
#pragma unroll
                for (int i = 0; i < 16; i++) rq[i] = 0ULL;
                const int r0 = embedded_composite(KID) ? srow.off[q] : q * d, r1 = embedded_composite(KID) ? r0 + srow.rows[q] : (q + 1) * d;
                for (int dim = r0; dim < r1; dim++) {
                    const f32x2_t xc = f2_pack(sC[dim * 64 + cl], sC[dim * 64 + cl + 32]);
                    const float4* xr = reinterpret_cast<const float4*>(x + dim * OZ_XK);
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const float4 xv = xr[i];
                        f32x2_t df;
                        df = f2_sub(f2_pack(xv.x, xv.x), xc); rq[4 * i] = f2_fma(df, df, rq[4 * i]);
                        df = f2_sub(f2_pack(xv.y, xv.y), xc); rq[4 * i + 1] = f2_fma(df, df, rq[4 * i + 1]);
                        df = f2_sub(f2_pack(xv.z, xv.z), xc); rq[4 * i + 2] = f2_fma(df, df, rq[4 * i + 2]);
                        df = f2_sub(f2_pack(xv.w, xv.w), xc); rq[4 * i + 3] = f2_fma(df, df, rq[4 * i + 3]);
                    }
                }
                const float v = (float)sum.var[q], al = (float)sum.alpha[q];
                const int fam = sum.fam[q];
#pragma unroll
                for (int g = 0; g < 16; g++) {
                    f32x2_t t;
                    switch (fam) {
                        case KERNEL_MATERN12: t = cov32x2_from_r2<KERNEL_MATERN12>(rq[g], v, al); break;
                        case KERNEL_MATERN32: t = cov32x2_from_r2<KERNEL_MATERN32>(rq[g], v, al); break;
                        case KERNEL_MATERN52: t = cov32x2_from_r2<KERNEL_MATERN52>(rq[g], v, al); break;
                        case KERNEL_SE: t = cov32x2_from_r2<KERNEL_SE>(rq[g], v, al); break;
                        default: t = cov32x2_from_r2<KERNEL_RQ>(rq[g], v, al); break;
                    }
                    kv[g] = (q == 0) ? t : (product_kernel(KID) ? f2_mul(kv[g], t) : f2_add(kv[g], t));
                }
            }
        } else {
            for (int dim = 0; dim < d; dim++) {
                const f32x2_t xc = f2_pack(sC[dim * 64 + cl], sC[dim * 64 + cl + 32]);
                const float4* xr = reinterpret_cast<const float4*>(x + dim * OZ_XK);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const float4 xv = xr[i];
                    f32x2_t df;
                    df = f2_sub(f2_pack(xv.x, xv.x), xc); r2[4 * i] = f2_fma(df, df, r2[4 * i]);
                    df = f2_sub(f2_pack(xv.y, xv.y), xc); r2[4 * i + 1] = f2_fma(df, df, r2[4 * i + 1]);
                    df = f2_sub(f2_pack(xv.z, xv.z), xc); r2[4 * i + 2] = f2_fma(df, df, r2[4 * i + 2]);
                    df = f2_sub(f2_pack(xv.w, xv.w), xc); r2[4 * i + 3] = f2_fma(df, df, r2[4 * i + 3]);
                }
            }
        }
        const int j0 = ss * OZ_XK + kg * 16;
        const int ks = ss * 4 + (kg >> 1), half = kg & 1;
        const float* al = sAl + b * OZ_XK + kg * 16;
        constexpr int SD = S > 0 ? S : 1;
        uint32_t out[2][SD][4];
#pragma unroll
        for (int a = 0; a < 2; a++)
#pragma unroll
            for (int p = 0; p < SD; p++) out[a][p][0] = out[a][p][1] = out[a][p][2] = out[a][p][3] = 0u;
        f32x2_t msum = 0ULL;
        const f32x2_t bs2 = f2_pack(bscale, bscale);
        // training points beyond N exist only in the last super-step (padding of the last 128-row block)
        const bool tail = j0 + 16 > N;
#pragma unroll
        for (int g = 0; g < 16; g++) {
            f32x2_t k2;
            if constexpr (composite_kernel(KID)) k2 = kv[g];
            else k2 = cov32x2_from_r2<KID>(r2[g], var, rq_alpha);
            float k0, k1;
            f2_unpack(k2, k0, k1);
            k0 = cvalid[0] ? k0 : 0.0f;
            k1 = cvalid[1] ? k1 : 0.0f;
            if (tail && j0 + g >= N) k0 = k1 = 0.0f;
            k2 = f2_pack(k0, k1);
            msum = f2_fma(k2, f2_pack(al[g], al[g]), msum);
            if (S > 0) {
                float q0, q1;
                f2_unpack(f2_mul(k2, bs2), q0, q1);
                constexpr uint32_t C = (SD >= 4) ? 0x00808080u : (SD == 3) ? 0x00008080u : 0x00000080u;
                const uint32_t z[2] = {((uint32_t)__float2int_rn(q0) + C) ^ C, ((uint32_t)__float2int_rn(q1) + C) ^ C};
#pragma unroll
                for (int a = 0; a < 2; a++)
#pragma unroll
                    for (int p = 0; p < SD; p++) {
                        // digit p (0 = most significant) = byte S-1-p of z -> byte (g & 3) of word g >> 2
                        const uint32_t sel = (0x3210u & ~(0xFu << (4 * (g & 3)))) | ((uint32_t)(4 + (SD - 1 - p)) << (4 * (g & 3)));
                        out[a][p][g >> 2] = __byte_perm(out[a][p][g >> 2], z[a], sel);
                    }
            }
        }
        {
            float m0, m1;
            f2_unpack(msum, m0, m1);
            macc[0] += (double)m0;
            macc[1] += (double)m1;
        }
        if (S > 0) {
#pragma unroll
            for (int a = 0; a < 2; a++) {
                const int r = rbase + cl + 32 * a;
                uint8_t* dst = B + ((size_t)ct * nks + ks) * SD * (NT * 32) + (r >> 3) * 256 + half * 128 + (r & 7) * 16;
#pragma unroll
                for (int p = 0; p < SD; p++)
                    *reinterpret_cast<uint4*>(dst + (size_t)p * (NT * 32)) = make_uint4(out[a][p][0], out[a][p][1], out[a][p][2], out[a][p][3]);
            }
        }
    }
    sR[kg * 64 + cl] = macc[0];
    sR[kg * 64 + cl + 32] = macc[1];
    __syncthreads();
    if (tid < 64) {
        const double* q = sR + tid;
        const double m = (((q[0] + q[64]) + (q[128] + q[192])) + ((q[256] + q[320]) + (q[384] + q[448]))) + c0;
        mean[blk * 64 + tid] = sBad[tid] ? __longlong_as_double(0x7ff8000000000000LL) : m;
    }
}

// ---- the screening product ------------------------------------------------------------------------------------------------
// Same roles as ozaki_kernel: warp 0 producer (cp.async.bulk + mbarrier tx), warp 1 single-thread tcgen05.mma issuer, warps
// 2..9 epilogue.  Work unit = candidate tile x pair of row blocks (I, nb-1-I) via OzItems<OZ_TRMM> (OzParams-compatible view).
template <int S, int NT, bool FULL>
__global__ void __launch_bounds__(OZ_THREADS, 1) ozaki_screen_kernel(ScrParams P) {
    using Cfg = ScrCfg<S, NT, FULL>;
    constexpr int LEVELS = Cfg::LEVELS;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int NBUF = Cfg::NBUF;
    extern __shared__ __align__(1024) uint8_t scr_smem_raw[];
    uint8_t* ring = scr_smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(scr_smem_raw + Cfg::RING_BYTES);
    uint64_t* full = bars;                      // [STAGES]
    uint64_t* empty = bars + STAGES;            // [STAGES]
    uint64_t* tmem_full = bars + 2 * STAGES;    // [2]
    uint64_t* tmem_empty = tmem_full + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    float* red = reinterpret_cast<float*>(scr_smem_raw + Cfg::RING_BYTES + 1024);  // [4][NT]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; i++) {
            oz_mbar_init(&full[i], 1);
            oz_mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 2; i++) {
            oz_mbar_init(&tmem_full[i], 1);
            oz_mbar_init(&tmem_empty[i], 8);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(oz_smem(tmem_slot)), "r"(OZ_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    oz_fence_before();
    __syncthreads();
    oz_fence_after();
    const uint32_t tbase = *tmem_slot;
    const int nks = P.nks;
    // the item iterator of the full-precision kernel (candidate tile x pair of row blocks) only reads nb / nct
    OzParams Q;
    Q.nb = P.nb;
    Q.nct = P.nct;
    Q.nks = P.nks;

    if (warp == 0) {
        if (lane == 0) {
            int st = 0;
            uint32_t ph = 0;
            const uint64_t keep = oz_policy_evict_last();
            OzItems<OZ_TRMM> items(Q);
            int I, ks0, n;
            long long ct;
            while (items.next(I, ct, ks0, n)) {
                const uint8_t* a = P.A + ((size_t)I * nks) * Cfg::A_BYTES;
                const uint8_t* b = P.B + ((size_t)ct * nks) * Cfg::B_BYTES;
                for (int ks = 0; ks < n; ks += Cfg::KPS) {
                    oz_mbar_wait(&empty[st], ph ^ 1);
                    uint8_t* dst = ring + (size_t)st * Cfg::STAGE_BYTES;
                    oz_mbar_expect_tx(&full[st], Cfg::STAGE_BYTES);
                    oz_bulk_g2s_hint(dst, a + (size_t)ks * Cfg::A_BYTES, Cfg::KPS * Cfg::A_BYTES, &full[st], keep);
                    oz_bulk_g2s(dst + Cfg::KPS * Cfg::A_BYTES, b + (size_t)ks * Cfg::B_BYTES, Cfg::KPS * Cfg::B_BYTES, &full[st]);
                    if (++st == STAGES) {
                        st = 0;
                        ph ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int st = 0, buf = 0;
            uint32_t ph = 0, acc_ph[2] = {0, 0};
            const uint32_t ring_addr = oz_smem(ring);
            constexpr int DPM = 256 / NT;  // B digits covered by one MMA (N <= 256)
            OzItems<OZ_TRMM> items(Q);
            int I, ks0, n;
            long long ct;
            while (items.next(I, ct, ks0, n)) {
                oz_mbar_wait(&tmem_empty[buf], acc_ph[buf] ^ 1);  // the epilogue has drained this accumulator buffer
                oz_fence_after();
                const uint32_t tacc = tbase + (uint32_t)(buf * Cfg::ACC_COLS);
                for (int ks = 0; ks < n; ks += Cfg::KPS) {
                    oz_mbar_wait(&full[st], ph);
                    oz_fence_after();
#pragma unroll
                    for (int kk = 0; kk < Cfg::KPS; kk++) {
                        const uint32_t sa = ring_addr + (uint32_t)st * Cfg::STAGE_BYTES + kk * Cfg::A_BYTES;
                        const uint32_t sb = ring_addr + (uint32_t)st * Cfg::STAGE_BYTES + Cfg::KPS * Cfg::A_BYTES + kk * Cfg::B_BYTES;
                        if (FULL && ks + kk == 0) {
                            // first k-step of an item, full product: digit by digit, because one MMA cannot start a level
                            // (p >= 1: its last B digit opens level p + S - 1) and accumulate into the others
#pragma unroll
                            for (int p = 0; p < S; p++) {
                                const uint64_t ad = oz_desc(sa + p * OZ_A_SLICE);
#pragma unroll
                                for (int q = 0; q < S; q++)
                                    oz_mma(tacc + (uint32_t)((p + q) * NT), ad, oz_desc(sb + q * Cfg::B_SLICE), oz_idesc(NT),
                                           (p == 0 || q == S - 1) ? 0u : 1u);
                            }
                        } else {
#pragma unroll
                            for (int p = 0; p < S; p++) {
                                const uint64_t ad = oz_desc(sa + p * OZ_A_SLICE);
                                constexpr int SQ = S;  // digits of B
                                const int nqs = FULL ? SQ : S - p;
#pragma unroll
                                for (int q0 = 0; q0 < (FULL ? SQ : S - p); q0 += DPM) {
                                    const int nq = (nqs - q0 < DPM) ? nqs - q0 : DPM;
                                    oz_mma(tacc + (uint32_t)((p + q0) * NT), ad, oz_desc(sb + q0 * Cfg::B_SLICE), oz_idesc(nq * NT),
                                           (ks + kk > 0 || p > 0) ? 1u : 0u);
                                }
                            }
                        }
                    }
                    oz_commit(&empty[st]);
                    if (++st == STAGES) {
                        st = 0;
                        ph ^= 1;
                    }
                }
                oz_commit(&tmem_full[buf]);
                acc_ph[buf] ^= 1;
                buf = (buf + 1 == NBUF) ? 0 : buf + 1;
            }
        }
    } else {
        // epilogue: TMEM lane group lg = warp & 3 (rows), column half hsel (NT / 2 candidates), chunks of 8 columns
        const int lg = warp & 3;
        const int hsel = (warp - 2) >> 2;
        const int et = threadIdx.x - 64;
        constexpr int NCH = NT / 16;  // 8-column chunks per warp
        int buf = 0;
        uint32_t acc_ph[2] = {0, 0};
        OzItems<OZ_TRMM> items(Q);
        int I, ks0, n;
        long long ct;
        while (items.next(I, ct, ks0, n)) {
            const int row = I * 128 + lg * 32 + lane;
            const float rs = (float)(P.rowscale[row] * P.gscale);
            oz_mbar_wait(&tmem_full[buf], acc_ph[buf]);
            oz_fence_after();
            acc_ph[buf] ^= 1;
            const uint32_t tacc = tbase + ((uint32_t)(lg * 32) << 16) + (uint32_t)(buf * Cfg::ACC_COLS + hsel * (NT / 2));
            float tot[NCH];
            // software-pipelined drain: the TMEM loads of chunk cc+1 are in flight while chunk cc is reduced, so the issuer
            // (which waits for the hand-over when there is only one accumulator buffer) gets the columns back after the read
            // time of the tile, not after read + arithmetic
            uint32_t r[2][LEVELS][8];
#pragma unroll
            for (int t = 0; t < LEVELS; t++) oz_tmem_ld8(tacc + (uint32_t)(t * NT), r[0][t]);
#pragma unroll
            for (int cc = 0; cc < NCH; cc++) {
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (cc + 1 < NCH) {
#pragma unroll
                    for (int t = 0; t < LEVELS; t++) oz_tmem_ld8(tacc + (uint32_t)(t * NT + (cc + 1) * 8), r[(cc + 1) & 1][t]);
                } else {
                    oz_fence_before();
                    __syncwarp();
                    if (lane == 0) oz_mbar_arrive(&tmem_empty[buf]);
                }
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    float w = (float)(int32_t)r[cc & 1][0][i];
#pragma unroll
                    for (int t = 1; t < LEVELS; t++) w = fmaf(w, 256.0f, (float)(int32_t)r[cc & 1][t][i]);
                    w *= rs;
                    v[i] = w * w;
                }
#pragma unroll
                for (int o = 16, nn = 4; o >= 4; o >>= 1, nn >>= 1) {
                    const bool up = (lane & o) != 0;
#pragma unroll
                    for (int i = 0; i < nn; i++) {
                        const float send = up ? v[i] : v[i + nn];
                        const float keepv = up ? v[i + nn] : v[i];
                        v[i] = keepv + __shfl_xor_sync(0xffffffffu, send, o);
                    }
                }
                const float t2 = v[0] + __shfl_xor_sync(0xffffffffu, v[0], 2);
                tot[cc] = t2 + __shfl_xor_sync(0xffffffffu, t2, 1);
            }
            buf = (buf + 1 == NBUF) ? 0 : buf + 1;
            const int idx = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if ((lane & 3) == 0) {
#pragma unroll
                for (int cc = 0; cc < NCH; cc++) red[lg * NT + hsel * (NT / 2) + cc * 8 + idx] = tot[cc];
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            if (et < NT) {
                const float s = (red[et] + red[NT + et]) + (red[2 * NT + et] + red[3 * NT + et]);
                P.part[(size_t)I * P.ldp + (size_t)ct * NT + et] = s;
            }
        }
    }
    oz_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(OZ_TMEM_COLS));
}

// ---- order-preserving key of a double for atomicMax on 64-bit words ---------------------------------------------------------
__host__ __device__ __forceinline__ unsigned long long scr_key(double v) {
    unsigned long long b;
#ifdef __CUDA_ARCH__
    b = (unsigned long long)__double_as_longlong(v);
#else
    memcpy(&b, &v, sizeof b);
#endif
    return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
__host__ __device__ __forceinline__ double scr_unkey(unsigned long long k) {
    const unsigned long long b = (k & 0x8000000000000000ULL) ? (k & 0x7fffffffffffffffULL) : ~k;
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double v;
    memcpy(&v, &b, sizeof v);
    return v;
#endif
}

// state[0] = key of the running maximum of the screened UCB (non-NaN candidates); state[1] = survivor counter;
// state[2] = bits of the largest |refined - screened| UCB difference seen by screen_check_kernel
__global__ void __launch_bounds__(256) screen_finalize_kernel(const float* __restrict__ part, const double* __restrict__ mean, int nb,
                                                              long long ldp, long long Mw, long long idx0, double variance,
                                                              double noise, double varsigma, double* __restrict__ scr_ucb,
                                                              unsigned long long* __restrict__ state) {
    const long long c = (long long)blockIdx.x * 256 + threadIdx.x;
    double u = -INFINITY;
    if (c < Mw) {
        double ss = 0.0;
        for (int I = 0; I < nb; I++) ss += (double)part[(size_t)I * ldp + c];
        const double v = (variance - ss) + noise;
        u = mean[c] + varsigma * v;
        scr_ucb[idx0 + c] = u;
    }
    unsigned long long key = (u == u) ? scr_key(u) : 0ULL;  // NaN does not take part in the maximum (it always survives)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    __shared__ unsigned long long sk[8];
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; i++) key = sk[i] > key ? sk[i] : key;
        atomicMax(state, key);
    }
}

// first level of the bound-and-refine arg-max: store the (fp32-evaluated) posterior mean per candidate, running maximum
__global__ void __launch_bounds__(256) bound_finalize_kernel(const double* __restrict__ mean, long long Mw, long long idx0,
                                                             double* __restrict__ scr_ucb, unsigned long long* __restrict__ state) {
    const long long c = (long long)blockIdx.x * 256 + threadIdx.x;
    double m = -INFINITY;
    if (c < Mw) {
        m = mean[c];
        scr_ucb[idx0 + c] = m;
    }
    unsigned long long key = (m == m) ? scr_key(m) : 0ULL;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    __shared__ unsigned long long sk[8];
    if ((threadIdx.x & 31) == 0) sk[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; i++) key = sk[i] > key ? sk[i] : key;
        atomicMax(state, key);
    }
}

__global__ void __launch_bounds__(256) screen_select_kernel(const double* __restrict__ scr_ucb, long long M, double two_e,
                                                            unsigned long long* __restrict__ state, long long* __restrict__ list,
                                                            unsigned int cap) {
    const long long c = (long long)blockIdx.x * 256 + threadIdx.x;
    if (c >= M) return;
    const double thr = scr_unkey(state[0]) - two_e;
    const double u = scr_ucb[c];
    if (!(u < thr)) {  // NaN or within 2E of the best screened value
        const unsigned long long pos = atomicAdd(state + 1, 1ULL);
        if (pos < cap) list[pos] = c;
    }
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const double* __restrict__ Xc, const long long* __restrict__ list, long long n,
                                                          int d, double* __restrict__ out) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= n * d) return;
    const long long r = e / d;
    out[e] = Xc[list[r] * d + (e - r * d)];
}

// refined (full-precision) UCB of the survivors of one refine window against their screened value (mean_only: the stored
// value is the screened MEAN, first level of the bound-and-refine arg-max)
__global__ void __launch_bounds__(256) screen_check_kernel(const double* __restrict__ mean, const double* __restrict__ var, long long Mw,
                                                           const long long* __restrict__ list, double varsigma,
                                                           const double* __restrict__ scr_ucb, unsigned long long* __restrict__ state,
                                                           int mean_only) {
    const long long c = (long long)blockIdx.x * 256 + threadIdx.x;
    if (c >= Mw) return;
    const double u = mean_only ? mean[c] : __dadd_rn(mean[c], __dmul_rn(varsigma, var[c]));
    const double us = scr_ucb[list[c]];
    const double diff = fabs(u - us);
    // NaN on either side: nothing to compare (a NaN screened value is refined unconditionally).  An infinite difference
    // (finite refined, infinite screened) is reported and fails the check.
    if (diff == diff) atomicMax(state + 2, (unsigned long long)__double_as_longlong(diff));
}

}  // namespace gpso
