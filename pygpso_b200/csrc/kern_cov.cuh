// Covariance-function kernels: input scaling, Gram build, cross-covariance window (+ posterior mean), and the
// log-marginal-likelihood gradient reduction.  All HBM access is coalesced along the training-point index j:
// the scaled inputs are stored dimension-major, Xs[dim][Np], so consecutive lanes read consecutive doubles.
#pragma once
#include "common.cuh"

namespace gpso {

// Xs[dim*Np + j] = X[j*d + dim] / ls[dim]   (GPflow divides by the lengthscale, Stationary.scale); pad j>=N with 0
__global__ void scale_inputs_kernel(const double* __restrict__ X, const double* __restrict__ ls, int n_ls, int N, int d,
                                    int Np, double* __restrict__ Xs) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= Np) return;
    for (int dim = 0; dim < d; dim++) {
        double l = ls[n_ls > 1 ? dim : 0];
        Xs[(size_t)dim * Np + j] = (j < N) ? X[(size_t)j * d + dim] / l : 0.0;
    }
}

// ---- Gram matrix K + noise*I, lower 64x64 tiles of the padded [Np,Np] matrix; padding = identity ----------------
constexpr int CT = 64;    // covariance tile edge
constexpr int CDCH = 32;  // dimensions staged in shared memory per pass

template <int KID>
__global__ void __launch_bounds__(256) gram_kernel(const double* __restrict__ Xs, int N, int d, int Np, double var,
                                                   double noise, double* __restrict__ K, double rq_alpha, SumTable sum, SumRows srow) {
    const int bj = blockIdx.x, bi = blockIdx.y;
    if (bj > bi) return;
    __shared__ double sXi[CDCH][CT];
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int j = bj * CT + tx;
    if constexpr (KID == KERNEL_SUM_LIN) {
        // a Linear component adds the dot product of its rows, the others their stationary value as KERNEL_SUM_EMB does
        double kv[16];
        for (int c = 0; c < sum.n; c++) {
            const bool lin = sum.fam[c] == KERNEL_LINEAR;
            const int rn = srow.rows[c];
            const double* Xc = Xs + (size_t)srow.off[c] * Np;
            double acc[16];
#pragma unroll
            for (int r = 0; r < 16; r++) acc[r] = 0.0;
            for (int d0 = 0; d0 < rn; d0 += CDCH) {
                int dc = min(CDCH, rn - d0);
                __syncthreads();
                for (int e = threadIdx.x; e < dc * CT; e += 256) sXi[e / CT][e % CT] = Xc[(size_t)(d0 + e / CT) * Np + bi * CT + e % CT];
                __syncthreads();
                for (int dd = 0; dd < dc; dd++) {
                    const double xj = Xc[(size_t)(d0 + dd) * Np + j];
                    if (lin) {
#pragma unroll
                        for (int r = 0; r < 16; r++) acc[r] = fma(sXi[dd][ty + 4 * r], xj, acc[r]);
                    } else {
#pragma unroll
                        for (int r = 0; r < 16; r++) {
                            const double df = sXi[dd][ty + 4 * r] - xj;
                            acc[r] = fma(df, df, acc[r]);
                        }
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const double t = lin ? acc[r] : sum_term(sum, c, acc[r]);
                kv[r] = (c == 0) ? t : kv[r] + t;
            }
        }
#pragma unroll
        for (int r = 0; r < 16; r++) {
            int i = bi * CT + ty + 4 * r;
            double v;
            if (i < N && j < N) {
                v = kv[r];
                if (i == j) v += noise;
            } else {
                v = (i == j) ? 1.0 : 0.0;
            }
            K[(size_t)i * Np + j] = v;
        }
        return;
    } else if constexpr (composite_kernel(KID)) {
        // the loop below once per component (its own scaled inputs), the component values added (multiplied) in order
        double kv[16];
        for (int c = 0; c < sum.n; c++) {
            const int rn = embedded_composite(KID) ? srow.rows[c] : d;
            const double* Xc = (embedded_composite(KID) ? Xs + (size_t)srow.off[c] * Np : Xs + (size_t)c * d * Np);
            double r2[16];
#pragma unroll
            for (int r = 0; r < 16; r++) r2[r] = 0.0;
            for (int d0 = 0; d0 < rn; d0 += CDCH) {
                int dc = min(CDCH, rn - d0);
                __syncthreads();
                for (int e = threadIdx.x; e < dc * CT; e += 256) sXi[e / CT][e % CT] = Xc[(size_t)(d0 + e / CT) * Np + bi * CT + e % CT];
                __syncthreads();
                for (int dd = 0; dd < dc; dd++) {
                    double xj = Xc[(size_t)(d0 + dd) * Np + j];
#pragma unroll
                    for (int r = 0; r < 16; r++) {
                        double df = sXi[dd][ty + 4 * r] - xj;
                        r2[r] = fma(df, df, r2[r]);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const double t = sum_term(sum, c, r2[r]);
                kv[r] = (c == 0) ? t : combine<KID>(kv[r], t);
            }
        }
#pragma unroll
        for (int r = 0; r < 16; r++) {
            int i = bi * CT + ty + 4 * r;
            double v;
            if (i < N && j < N) {
                v = kv[r];
                if (i == j) v += noise;
            } else {
                v = (i == j) ? 1.0 : 0.0;
            }
            K[(size_t)i * Np + j] = v;
        }
        return;
    }
    double r2[16];
#pragma unroll
    for (int r = 0; r < 16; r++) r2[r] = 0.0;
    for (int d0 = 0; d0 < d; d0 += CDCH) {
        int dc = min(CDCH, d - d0);
        __syncthreads();
        for (int e = threadIdx.x; e < dc * CT; e += 256) sXi[e / CT][e % CT] = Xs[(size_t)(d0 + e / CT) * Np + bi * CT + e % CT];
        __syncthreads();
        for (int dd = 0; dd < dc; dd++) {
            double xj = Xs[(size_t)(d0 + dd) * Np + j];
#pragma unroll
            for (int r = 0; r < 16; r++) {
                double df = sXi[dd][ty + 4 * r] - xj;
                r2[r] = fma(df, df, r2[r]);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 16; r++) {
        int i = bi * CT + ty + 4 * r;
        double v;
        if (i < N && j < N) {
            v = cov_from_r2<KID>(r2[r], var, rq_alpha);
            if (i == j) v += noise;
        } else {
            v = (i == j) ? 1.0 : 0.0;
        }
        K[(size_t)i * Np + j] = v;
    }
}

// ---- cross-covariance window -------------------------------------------------------------------------------------
// KsT[c][j] = k(x_j, xc_c) for the window's candidates c (row-major [Mw_pad, Np], j contiguous -> it is the "B"
// operand of the triangular product), zero for j >= N and for padding candidates c >= Mw; and the posterior mean
// mean[c] = sum_j KsT[c][j] * alpha[j] + c0.  One block = XG candidates x all training points: each scaled training
// coordinate is loaded once per block and reused for XG candidates.  Every candidate sees exactly the same sequence
// of operations (position-independent results: duplicated candidates give bit-identical outputs).
constexpr int XG = 8;

// crosscov_kernel of a sum with Linear terms (KERNEL_SUM_LIN): the rows of KERNEL_SUM_EMB, and the prior variance k(x_c, x_c) of every
// candidate c of the launch (grid XG-candidate blocks) after the means, at mean[gridDim.x XG + c]: the squared norm of a Linear
// component's rows, the variance of the others, added in fp64 in component order (joint_syrk_kernel forms the same sum).
__device__ __forceinline__ void crosscov_sum_lin(const double* __restrict__ Xc, long long Mw, const double* __restrict__ ls,
                                                 const double* __restrict__ Xs, const double* __restrict__ alpha, int N, int Np,
                                                 double c0, double* __restrict__ KsT, double* __restrict__ mean, const SumTable& sum,
                                                 const SumRows& srow, double* sm) {
    double* sC = sm;  // [XG][width]
    double* sR = sm + XG * srow.width;
    const long long cbase = (long long)blockIdx.x * XG;
    const int w = srow.width;
    for (int e = threadIdx.x; e < XG * w; e += 256) {
        const long long c = cbase + e / w;
        const int r = e % w;
        sC[e] = (c < Mw) ? Xc[c * w + r] / ls[r] : 0.0;
    }
    __syncthreads();
    double macc[XG];
#pragma unroll
    for (int c = 0; c < XG; c++) macc[c] = 0.0;
    for (int j = threadIdx.x; j < Np; j += 256) {
        double kv[XG];
        for (int q = 0; q < sum.n; q++) {
            const bool lin = sum.fam[q] == KERNEL_LINEAR;
            const int rn = srow.rows[q];
            const double* Xq = Xs + (size_t)srow.off[q] * Np;
            const double* sq = sC + srow.off[q];
            double acc[XG];
#pragma unroll
            for (int c = 0; c < XG; c++) acc[c] = 0.0;
            if (lin) {
                for (int dim = 0; dim < rn; dim++) {
                    const double xj = Xq[(size_t)dim * Np + j];
#pragma unroll
                    for (int c = 0; c < XG; c++) acc[c] = fma(xj, sq[c * w + dim], acc[c]);
                }
            } else {
                for (int dim = 0; dim < rn; dim++) {
                    const double xj = Xq[(size_t)dim * Np + j];
#pragma unroll
                    for (int c = 0; c < XG; c++) {
                        const double df = xj - sq[c * w + dim];
                        acc[c] = fma(df, df, acc[c]);
                    }
                }
#pragma unroll
                for (int c = 0; c < XG; c++) acc[c] = sum_term(sum, q, acc[c]);
            }
#pragma unroll
            for (int c = 0; c < XG; c++) kv[c] = (q == 0) ? acc[c] : kv[c] + acc[c];
        }
        const double a = alpha[j];
#pragma unroll
        for (int c = 0; c < XG; c++) {
            const double k = (j < N && cbase + c < Mw) ? kv[c] : 0.0;
            KsT[(size_t)(cbase + c) * Np + j] = k;
            macc[c] = fma(k, a, macc[c]);
        }
    }
#pragma unroll
    for (int c = 0; c < XG; c++) macc[c] = warp_sum(macc[c]);
    const int wp = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) {
#pragma unroll
        for (int c = 0; c < XG; c++) sR[wp * XG + c] = macc[c];
    }
    __syncthreads();
    if (threadIdx.x < XG) {
        double s = 0.0;
#pragma unroll
        for (int ww = 0; ww < 8; ww++) s += sR[ww * XG + threadIdx.x];
        mean[cbase + threadIdx.x] = s + c0;
    }
    if (threadIdx.x < XG) {
        double s = 0.0;
        for (int q = 0; q < sum.n; q++) {
            double t = sum.var[q];
            if (sum.fam[q] == KERNEL_LINEAR) {
                t = 0.0;
                for (int r = srow.off[q]; r < srow.off[q] + srow.rows[q]; r++) t = fma(sC[threadIdx.x * w + r], sC[threadIdx.x * w + r], t);
            }
            s = (q == 0) ? t : s + t;
        }
        mean[(long long)gridDim.x * XG + cbase + threadIdx.x] = s;
    }
}

template <int KID>
__global__ void __launch_bounds__(256) crosscov_kernel(const double* __restrict__ Xc, long long Mw, int d,
                                                       const double* __restrict__ ls, int n_ls,
                                                       const double* __restrict__ Xs, const double* __restrict__ alpha,
                                                       int N, int Np, double var, double c0, double* __restrict__ KsT,
                                                       double* __restrict__ mean, double rq_alpha, SumTable sum, SumRows srow) {
    extern __shared__ double sm[];  // [XG][d] scaled candidate coords (sum: [C][XG][d]), then [8 warps][XG] reduction scratch
    double* sC = sm;
    const int nsc = composite_kernel(KID) ? sum.n : 1;  // scaled copies of the candidates
    double* sR = sm + (embedded_composite(KID) ? XG * srow.width : nsc * XG * d);
    const long long cbase = (long long)blockIdx.x * XG;
    if constexpr (KID == KERNEL_SUM_LIN) {
        crosscov_sum_lin(Xc, Mw, ls, Xs, alpha, N, Np, c0, KsT, mean, sum, srow, sm);
        return;
    } else if constexpr (embedded_composite(KID)) {
        // [XG][width]: candidate row r divided by ls[r] (a periodic component's embedded rows by its unit lengthscale)
        const int w = srow.width;
        for (int e = threadIdx.x; e < XG * w; e += 256) {
            const long long c = cbase + e / w;
            const int r = e % w;
            sC[e] = (c < Mw) ? Xc[c * w + r] / ls[r] : 0.0;
        }
    } else if constexpr (composite_kernel(KID)) {
        // component q divides by its own lengthscales (expanded to d entries at ls + q d): the bare kernel's division
        for (int e = threadIdx.x; e < nsc * XG * d; e += 256) {
            const int q = e / (XG * d), f = e - q * XG * d;
            long long c = cbase + f / d;
            int dim = f % d;
            sC[e] = (c < Mw) ? Xc[c * d + dim] / ls[q * d + dim] : 0.0;
        }
    } else {
        for (int e = threadIdx.x; e < XG * d; e += 256) {
            long long c = cbase + e / d;
            int dim = e % d;
            sC[e] = (c < Mw) ? Xc[c * d + dim] / ls[n_ls > 1 ? dim : 0] : 0.0;
        }
    }
    __syncthreads();
    double macc[XG];
#pragma unroll
    for (int c = 0; c < XG; c++) macc[c] = 0.0;
    if constexpr (composite_kernel(KID)) {
        for (int j = threadIdx.x; j < Np; j += 256) {
            double kv[XG];
            for (int q = 0; q < sum.n; q++) {
                constexpr bool E = embedded_composite(KID);
                const int rn = E ? srow.rows[q] : d, cs = E ? srow.width : d;  // rows of component q, candidate stride
                const double* Xq = (E ? Xs + (size_t)srow.off[q] * Np : Xs + (size_t)q * d * Np);
                const double* sq = E ? sC + srow.off[q] : sC + q * XG * d;
                double r2[XG];
#pragma unroll
                for (int c = 0; c < XG; c++) r2[c] = 0.0;
                for (int dim = 0; dim < rn; dim++) {
                    double xj = Xq[(size_t)dim * Np + j];
#pragma unroll
                    for (int c = 0; c < XG; c++) {
                        double df = xj - sq[c * cs + dim];
                        r2[c] = fma(df, df, r2[c]);
                    }
                }
#pragma unroll
                for (int c = 0; c < XG; c++) {
                    const double t = sum_term(sum, q, r2[c]);
                    kv[c] = (q == 0) ? t : combine<KID>(kv[c], t);
                }
            }
            double a = alpha[j];
#pragma unroll
            for (int c = 0; c < XG; c++) {
                double k = (j < N && cbase + c < Mw) ? kv[c] : 0.0;
                KsT[(size_t)(cbase + c) * Np + j] = k;
                macc[c] = fma(k, a, macc[c]);
            }
        }
    } else {
        for (int j = threadIdx.x; j < Np; j += 256) {
            double r2[XG];
#pragma unroll
            for (int c = 0; c < XG; c++) r2[c] = 0.0;
            for (int dim = 0; dim < d; dim++) {
                double xj = Xs[(size_t)dim * Np + j];
#pragma unroll
                for (int c = 0; c < XG; c++) {
                    double df = xj - sC[c * d + dim];
                    r2[c] = fma(df, df, r2[c]);
                }
            }
            double a = alpha[j];  // zero for j >= N
#pragma unroll
            for (int c = 0; c < XG; c++) {
                double k = (j < N && cbase + c < Mw) ? cov_from_r2<KID>(r2[c], var, rq_alpha) : 0.0;
                KsT[(size_t)(cbase + c) * Np + j] = k;
                macc[c] = fma(k, a, macc[c]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < XG; c++) macc[c] = warp_sum(macc[c]);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) {
#pragma unroll
        for (int c = 0; c < XG; c++) sR[w * XG + c] = macc[c];
    }
    __syncthreads();
    if (threadIdx.x < XG) {
        double s = 0.0;
#pragma unroll
        for (int ww = 0; ww < 8; ww++) s += sR[ww * XG + threadIdx.x];
        mean[cbase + threadIdx.x] = s + c0;
    }
}

// ---- LML gradient: sum_ij W_ij dK_ij/dtheta with W = alpha alpha^T - K_y^-1, never materialising dK -------------
// One block per lower 64x64 tile (bi >= bj).  Strictly-lower tiles count twice (symmetry).  Partial sums per block:
//   part[blk][0] = sum W*k            (-> d/d variance after / variance)
//   part[blk][1] = sum_i W_ii         (-> d/d noise)
//   part[blk][2 + q] = sum W*g*r2     (scalar lengthscale, q = 0)  or  sum W*g*(xs_i - xs_j)_dim^2 for dim = dim0+q
//   part[blk][stride - 1] = sum W*dk/dalpha   (RationalQuadratic only: stride = 3 + n_ls)
constexpr int GRAD_DCH = 4;  // ARD dimensions reduced per launch

template <int KID, bool ARD>
__global__ void __launch_bounds__(256) lml_grad_kernel(const double* __restrict__ Xs, const double* __restrict__ alpha,
                                                       const double* __restrict__ Kinv, int N, int d, int Np, double var,
                                                       int dim0, int ndim, double* __restrict__ part, int part_stride,
                                                       double rq_alpha) {
    // triangular block index -> (bi, bj)
    int blk = blockIdx.x;
    int bi = (int)((sqrt(8.0 * blk + 1.0) - 1.0) * 0.5);
    while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
    while (bi * (bi + 1) / 2 > blk) bi--;
    int bj = blk - bi * (bi + 1) / 2;
    __shared__ double sXi[CDCH][CT];
    __shared__ double sRed[8];
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int j = bj * CT + tx;
    double r2[16];
    double gd[16][ARD ? GRAD_DCH : 1];
#pragma unroll
    for (int r = 0; r < 16; r++) {
        r2[r] = 0.0;
#pragma unroll
        for (int q = 0; q < (ARD ? GRAD_DCH : 1); q++) gd[r][q] = 0.0;
    }
    for (int d0 = 0; d0 < d; d0 += CDCH) {
        int dc = min(CDCH, d - d0);
        __syncthreads();
        for (int e = threadIdx.x; e < dc * CT; e += 256) sXi[e / CT][e % CT] = Xs[(size_t)(d0 + e / CT) * Np + bi * CT + e % CT];
        __syncthreads();
        for (int dd = 0; dd < dc; dd++) {
            double xj = Xs[(size_t)(d0 + dd) * Np + j];
            int q = d0 + dd - dim0;
#pragma unroll
            for (int r = 0; r < 16; r++) {
                double df = sXi[dd][ty + 4 * r] - xj;
                double sq = df * df;
                r2[r] += sq;
                if (ARD) {
#pragma unroll
                    for (int qq = 0; qq < GRAD_DCH; qq++)
                        if (qq == q) gd[r][qq] = sq;
                }
            }
        }
    }
    double s_k = 0.0, s_tr = 0.0, s_a = 0.0, s_l[ARD ? GRAD_DCH : 1];
#pragma unroll
    for (int q = 0; q < (ARD ? GRAD_DCH : 1); q++) s_l[q] = 0.0;
    const double aj = alpha[j];
    const double wsym = (bi == bj) ? 1.0 : 2.0;
#pragma unroll
    for (int r = 0; r < 16; r++) {
        int i = bi * CT + ty + 4 * r;
        // diagonal tiles: the tile holds both triangles of a symmetric quantity, take every element once
        if (i < N && j < N) {
            double kin = (j <= i) ? Kinv[(size_t)i * Np + j] : Kinv[(size_t)j * Np + i];
            double W = fma(alpha[i], aj, -kin) * wsym;
            double k, g, ka;
            cov_and_radial<KID>(r2[r], var, rq_alpha, k, g, ka);
            s_k = fma(W, k, s_k);
            if (KID == KERNEL_RQ) s_a = fma(W, ka, s_a);
            if (i == j) s_tr += W;
            double wg = W * g;
            if (ARD) {
#pragma unroll
                for (int q = 0; q < GRAD_DCH; q++) s_l[q] = fma(wg, gd[r][q], s_l[q]);
            } else {
                s_l[0] = fma(wg, fmax(r2[r], 0.0), s_l[0]);
            }
        }
    }
    double v;
    v = block_sum<256>(s_k, sRed);
    if (threadIdx.x == 0 && dim0 == 0) part[(size_t)blk * part_stride + 0] = v;
    v = block_sum<256>(s_tr, sRed);
    if (threadIdx.x == 0 && dim0 == 0) part[(size_t)blk * part_stride + 1] = v;
    if (KID == KERNEL_RQ) {
        v = block_sum<256>(s_a, sRed);
        if (threadIdx.x == 0 && dim0 == 0) part[(size_t)blk * part_stride + part_stride - 1] = v;
    }
#pragma unroll
    for (int q = 0; q < (ARD ? GRAD_DCH : 1); q++) {
        v = block_sum<256>(s_l[q], sRed);
        if (threadIdx.x == 0 && q < ndim) part[(size_t)blk * part_stride + 2 + dim0 + q] = v;
    }
}

// ---- LML gradient of a product kernel (k = prod_c k_c) -----------------------------------------------------------
// dK/dtheta_c = P_-c dk_c/dtheta_c with P_-c = prod_{j != c} k_j formed per pair from prefix and suffix products (never as
// K / k_c: k_c can be 0).  One launch for every entry: one block per lower 64x64 tile, the tile's scaled coordinates of all C
// factors (rows bi and columns bj, [C d][64] each) in shared memory, each pair's factor values formed once.  Partial sums:
//   part[blk][0] = sum W*K                                  (-> d/d var_c = s_K / var_c for every factor)
//   part[blk][1] = sum_i W_ii                               (-> d/d noise)
//   then per factor c in order, at off_c (off_0 = 2):
//   part[blk][off_c + q] = sum W*P_-c*g_c*(xs_i - xs_j)_q^2  (ARD: q < d)   or   sum W*P_-c*g_c*r2_c  (scalar lengthscale)
//   part[blk][off_c + n_ls_c] = sum W*P_-c*dk_c/dalpha      (RationalQuadratic factors only)
// Scalar entries reduce from registers.  An ARD factor's per-pair weight W*P_-c*g_c goes to shared memory ([64][64] per ARD
// factor), and a second pass gives warp w the dimensions e = w, w + 8, ... of all ARD factors, each summed over the tile's
// 4096 pairs in a fixed order: the distance work is at most twice the product's, whatever d.
__global__ void __launch_bounds__(256) lml_grad_product_kernel(const double* __restrict__ Xs, const double* __restrict__ alpha,
                                                               const double* __restrict__ Kinv, int N, int d, int Np, int ard_mask,
                                                               double* __restrict__ part, int part_stride, SumTable tab) {
    int blk = blockIdx.x;
    int bi = (int)((sqrt(8.0 * blk + 1.0) - 1.0) * 0.5);
    while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
    while (bi * (bi + 1) / 2 > blk) bi--;
    int bj = blk - bi * (bi + 1) / 2;
    const int n = tab.n, dx = n * d;
    extern __shared__ double smg[];
    double* sXi = smg;                // [dx][64] scaled coordinates of the tile's rows
    double* sXj = smg + dx * CT;      // [dx][64] ... and of its columns
    double* sW = sXj + dx * CT;       // [ARD factors][64 * 64] per-pair weights W P_-c g_c
    __shared__ double sRed[8];
    for (int e = threadIdx.x; e < dx * CT; e += 256) {
        const size_t row = (size_t)(e / CT) * Np;
        sXi[e] = Xs[row + bi * CT + e % CT];
        sXj[e] = Xs[row + bj * CT + e % CT];
    }
    __syncthreads();
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int j = bj * CT + tx;
    const double aj = alpha[j];
    const double wsym = (bi == bj) ? 1.0 : 2.0;
    double s_k = 0.0, s_tr = 0.0, s_l[MAX_SUM], s_a[MAX_SUM];
#pragma unroll
    for (int c = 0; c < MAX_SUM; c++) s_l[c] = s_a[c] = 0.0;
#pragma unroll 1
    for (int r = 0; r < 16; r++) {
        const int il = ty + 4 * r, i = bi * CT + il;
        const bool valid = i < N && j < N;
        // diagonal tiles: the tile holds both triangles of a symmetric quantity, take every element once
        double W = 0.0;
        if (valid) W = fma(alpha[i], aj, -((j <= i) ? Kinv[(size_t)i * Np + j] : Kinv[(size_t)j * Np + i])) * wsym;
        double r2[MAX_SUM], k[MAX_SUM], g[MAX_SUM], ka[MAX_SUM];
#pragma unroll
        for (int c = 0; c < MAX_SUM; c++) {
            r2[c] = 0.0;
            k[c] = 1.0;  // absent factors: the products below stay those of the n present ones
            g[c] = ka[c] = 0.0;
            if (c < n) {
                for (int q = c * d; q < (c + 1) * d; q++) {
                    const double df = sXi[q * CT + il] - sXj[q * CT + tx];
                    r2[c] = fma(df, df, r2[c]);
                }
                sum_term_radial(tab, c, r2[c], k[c], g[c], ka[c]);
            }
        }
        double pre[MAX_SUM], suf[MAX_SUM];
        pre[0] = 1.0;
#pragma unroll
        for (int c = 1; c < MAX_SUM; c++) pre[c] = pre[c - 1] * k[c - 1];
        suf[MAX_SUM - 1] = 1.0;
#pragma unroll
        for (int c = MAX_SUM - 2; c >= 0; c--) suf[c] = suf[c + 1] * k[c + 1];
        if (valid) {
            s_k = fma(W, pre[MAX_SUM - 1] * k[MAX_SUM - 1], s_k);
            if (i == j) s_tr += W;
        }
        int slot = 0;
#pragma unroll
        for (int c = 0; c < MAX_SUM; c++) {
            if (c < n) {
                const double pw = W * (pre[c] * suf[c]);
                if (ard_mask >> c & 1) {
                    sW[slot * CT * CT + il * CT + tx] = valid ? pw * g[c] : 0.0;
                    slot++;
                } else if (valid) {
                    s_l[c] = fma(pw * g[c], fmax(r2[c], 0.0), s_l[c]);
                }
                if (valid && tab.fam[c] == KERNEL_RQ) s_a[c] = fma(pw, ka[c], s_a[c]);
            }
        }
    }
    double v = block_sum<256>(s_k, sRed);
    if (threadIdx.x == 0) part[(size_t)blk * part_stride + 0] = v;
    v = block_sum<256>(s_tr, sRed);
    if (threadIdx.x == 0) part[(size_t)blk * part_stride + 1] = v;
    int off = 2;
#pragma unroll
    for (int c = 0; c < MAX_SUM; c++) {
        if (c >= n) break;
        const bool ard = ard_mask >> c & 1, rq = tab.fam[c] == KERNEL_RQ;
        if (!ard) {
            v = block_sum<256>(s_l[c], sRed);
            if (threadIdx.x == 0) part[(size_t)blk * part_stride + off] = v;
        }
        const int nl = ard ? d : 1;
        if (rq) {
            v = block_sum<256>(s_a[c], sRed);
            if (threadIdx.x == 0) part[(size_t)blk * part_stride + off + nl] = v;
        }
        off += nl + rq;
    }
    if (ard_mask == 0) return;
    __syncthreads();  // the weights of every pair are in sW
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int c = 0, slot = 0, o = 2; c < n; c++) {
        const bool ard = ard_mask >> c & 1;
        if (ard) {
            const double* ws = sW + slot * CT * CT;
            for (int q = w; q < d; q += 8) {
                const double* xi = sXi + (c * d + q) * CT;
                const double* xj = sXj + (c * d + q) * CT;
                double acc = 0.0;
                for (int p = lane; p < CT * CT; p += 32) {
                    const double df = xi[p >> 6] - xj[p & 63];
                    acc = fma(ws[p], df * df, acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) part[(size_t)blk * part_stride + o + q] = acc;
            }
            slot++;
        }
        o += (ard ? d : 1) + (tab.fam[c] == KERNEL_RQ);
    }
}

// The raw coordinates of a product's periodic factors: X[N][width], factor c's from column off[c] (without active dims every
// periodic factor reads all d columns of the inputs: width = d, off = 0).
struct RawCols {
    int off[MAX_SUM], width;
};

// A product on the rows of srow (periodic factors, or active dims): lml_grad_product_kernel with factor c's rows [srow.off[c],
// + srow.rows[c]) over its k_c dimensions -- k_c rows, or a periodic factor's 2 k_c embedded rows -- and X[N][xw] holding the raw
// coordinates the periodic factors read, factor c's k_c of them from column raw.off[c] (a separate kernel, so that the one above
// stays as it is).  A periodic factor always takes a weight slot (set in ard_mask) and writes, like lml_grad_periodic_kernel, per
// dimension j the lengthscale entry sum w ((De_j)^2 + (De_{k+j})^2) and the period entry sum w (x_j - x'_j) (e_{k+j} e'_j - e_j e'_{k+j}),
// 2 k_c entries before its alpha.
__global__ void __launch_bounds__(256) lml_grad_product_periodic_kernel(const double* __restrict__ Xs, const double* __restrict__ alpha,
                                                                        const double* __restrict__ Kinv, int N, int Np,
                                                                        int ard_mask, double* __restrict__ part, int part_stride,
                                                                        SumTable tab, const double* __restrict__ X, SumRows srow,
                                                                        RawCols raw) {
    int blk = blockIdx.x;
    int bi = (int)((sqrt(8.0 * blk + 1.0) - 1.0) * 0.5);
    while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
    while (bi * (bi + 1) / 2 > blk) bi--;
    int bj = blk - bi * (bi + 1) / 2;
    const int n = tab.n, dx = srow.width, xw = raw.width;
    extern __shared__ double smg[];
    double* sXi = smg;                // [dx][64] scaled coordinates of the tile's rows
    double* sXj = smg + dx * CT;      // [dx][64] ... and of its columns
    double* sRi = sXj + dx * CT;      // [xw][64] raw coordinates of the tile's rows, then of its columns
    double* sRj = sRi + xw * CT;
    double* sW = sRj + xw * CT;       // [ARD / periodic factors][64 * 64] per-pair weights W P_-c g_c
    __shared__ double sRed[8];
    for (int e = threadIdx.x; e < dx * CT; e += 256) {
        const size_t row = (size_t)(e / CT) * Np;
        sXi[e] = Xs[row + bi * CT + e % CT];
        sXj[e] = Xs[row + bj * CT + e % CT];
    }
    for (int e = threadIdx.x; e < xw * CT; e += 256) {
        const int q = e / CT, t = e % CT, ri = bi * CT + t, rj = bj * CT + t;
        sRi[e] = ri < N ? X[(size_t)ri * xw + q] : 0.0;
        sRj[e] = rj < N ? X[(size_t)rj * xw + q] : 0.0;
    }
    __syncthreads();
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int j = bj * CT + tx;
    const double aj = alpha[j];
    const double wsym = (bi == bj) ? 1.0 : 2.0;
    double s_k = 0.0, s_tr = 0.0, s_l[MAX_SUM], s_a[MAX_SUM];
#pragma unroll
    for (int c = 0; c < MAX_SUM; c++) s_l[c] = s_a[c] = 0.0;
#pragma unroll 1
    for (int r = 0; r < 16; r++) {
        const int il = ty + 4 * r, i = bi * CT + il;
        const bool valid = i < N && j < N;
        // diagonal tiles: the tile holds both triangles of a symmetric quantity, take every element once
        double W = 0.0;
        if (valid) W = fma(alpha[i], aj, -((j <= i) ? Kinv[(size_t)i * Np + j] : Kinv[(size_t)j * Np + i])) * wsym;
        double r2[MAX_SUM], k[MAX_SUM], g[MAX_SUM], ka[MAX_SUM];
#pragma unroll
        for (int c = 0; c < MAX_SUM; c++) {
            r2[c] = 0.0;
            k[c] = 1.0;  // absent factors: the products below stay those of the n present ones
            g[c] = ka[c] = 0.0;
            if (c < n) {
                const int r0 = srow.off[c], r1 = r0 + srow.rows[c];
                for (int q = r0; q < r1; q++) {
                    const double df = sXi[q * CT + il] - sXj[q * CT + tx];
                    r2[c] = fma(df, df, r2[c]);
                }
                sum_term_radial(tab, c, r2[c], k[c], g[c], ka[c]);
            }
        }
        double pre[MAX_SUM], suf[MAX_SUM];
        pre[0] = 1.0;
#pragma unroll
        for (int c = 1; c < MAX_SUM; c++) pre[c] = pre[c - 1] * k[c - 1];
        suf[MAX_SUM - 1] = 1.0;
#pragma unroll
        for (int c = MAX_SUM - 2; c >= 0; c--) suf[c] = suf[c + 1] * k[c + 1];
        if (valid) {
            s_k = fma(W, pre[MAX_SUM - 1] * k[MAX_SUM - 1], s_k);
            if (i == j) s_tr += W;
        }
        int slot = 0;
#pragma unroll
        for (int c = 0; c < MAX_SUM; c++) {
            if (c < n) {
                const double pw = W * (pre[c] * suf[c]);
                if (ard_mask >> c & 1) {
                    sW[slot * CT * CT + il * CT + tx] = valid ? pw * g[c] : 0.0;
                    slot++;
                } else if (valid) {
                    s_l[c] = fma(pw * g[c], fmax(r2[c], 0.0), s_l[c]);
                }
                if (valid && tab.fam[c] == KERNEL_RQ) s_a[c] = fma(pw, ka[c], s_a[c]);
            }
        }
    }
    double v = block_sum<256>(s_k, sRed);
    if (threadIdx.x == 0) part[(size_t)blk * part_stride + 0] = v;
    v = block_sum<256>(s_tr, sRed);
    if (threadIdx.x == 0) part[(size_t)blk * part_stride + 1] = v;
    int off = 2;
#pragma unroll
    for (int c = 0; c < MAX_SUM; c++) {
        if (c >= n) break;
        const bool ard = ard_mask >> c & 1, rq = tab.fam[c] == KERNEL_RQ;
        if (!ard) {
            v = block_sum<256>(s_l[c], sRed);
            if (threadIdx.x == 0) part[(size_t)blk * part_stride + off] = v;
        }
        const int nl = (srow.pmask >> c & 1) ? srow.rows[c] : (ard ? srow.rows[c] : 1);
        if (rq) {
            v = block_sum<256>(s_a[c], sRed);
            if (threadIdx.x == 0) part[(size_t)blk * part_stride + off + nl] = v;
        }
        off += nl + rq;
    }
    if (ard_mask == 0) return;
    __syncthreads();  // the weights of every pair are in sW
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int c = 0, slot = 0, o = 2; c < n; c++) {
        const bool ard = ard_mask >> c & 1, per = srow.pmask >> c & 1;
        const int k = per ? srow.rows[c] / 2 : srow.rows[c];  // the factor's dimensions
        if (per) {
            const double* ws = sW + slot * CT * CT;
            for (int q = w; q < k; q += 8) {
                const int r = srow.off[c] + q;
                const double *ci = sXi + r * CT, *cj = sXj + r * CT, *si = sXi + (r + k) * CT, *sj = sXj + (r + k) * CT;
                const double *xi = sRi + (raw.off[c] + q) * CT, *xj = sRj + (raw.off[c] + q) * CT;
                double acc_l = 0.0, acc_p = 0.0;
                for (int p = lane; p < CT * CT; p += 32) {
                    const int a = p >> 6, b = p & 63;
                    const double dc = ci[a] - cj[b], ds = si[a] - sj[b];
                    acc_l = fma(ws[p], fma(dc, dc, ds * ds), acc_l);
                    acc_p = fma(ws[p] * (xi[a] - xj[b]), fma(si[a], cj[b], -(ci[a] * sj[b])), acc_p);
                }
                acc_l = warp_sum(acc_l);
                acc_p = warp_sum(acc_p);
                if (lane == 0) {
                    part[(size_t)blk * part_stride + o + q] = acc_l;
                    part[(size_t)blk * part_stride + o + k + q] = acc_p;
                }
            }
            slot++;
        } else if (ard) {
            const double* ws = sW + slot * CT * CT;
            for (int q = w; q < k; q += 8) {
                const int r = srow.off[c] + q;
                const double* xi = sXi + r * CT;
                const double* xj = sXj + r * CT;
                double acc = 0.0;
                for (int p = lane; p < CT * CT; p += 32) {
                    const double df = xi[p >> 6] - xj[p & 63];
                    acc = fma(ws[p], df * df, acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) part[(size_t)blk * part_stride + o + q] = acc;
            }
            slot++;
        }
        o += (per ? 2 * k : (ard ? k : 1)) + (tab.fam[c] == KERNEL_RQ);
    }
}

// ---- periodic kernel (gpflow.kernels.Periodic with a SquaredExponential / RationalQuadratic base) ------------------------
// k(x, x') = base.K_r2(r2), r2 = sum_j sin^2(pi (x_j - x'_j) / p_j) / l_j^2, is the base kernel at unit lengthscale on the
// embedded rows  e_j(x) = cos(theta_j) / (2 l_j),  e_{d+j}(x) = sin(theta_j) / (2 l_j),  theta_j = 2 pi x_j / p_j
// (chord: |e(x) - e(x')|^2 = (2 - 2 cos(theta - theta')) / (4 l^2) = sin^2((theta - theta') / 2) / l^2).  The phase is one fp64
// sincospi(2 x / p) per coordinate; lp = [l expanded to d entries, p expanded to d entries].  out[i * s_row + r * s_dim] for rows
// i < rows, zero for padding rows rows <= i < rows_pad (dimension-major training inputs [2d][Np], or row-major candidates
// [M][2d]).  A NaN or infinite coordinate gives NaN rows.
__global__ void __launch_bounds__(256) periodic_embed_kernel(const double* __restrict__ X, long long rows, long long rows_pad, int d,
                                                             const double* __restrict__ lp, long long s_row, long long s_dim,
                                                             double* __restrict__ out) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= rows_pad * d) return;
    const long long i = e / d;
    const int j = (int)(e - i * d);
    double c = 0.0, s = 0.0;
    if (i < rows) {
        const double l2 = 2.0 * lp[j];
        sincospi(2.0 * X[e] / lp[d + j], &s, &c);
        c /= l2;
        s /= l2;
    }
    out[i * s_row + (long long)j * s_dim] = c;
    out[i * s_row + (long long)(d + j) * s_dim] = s;
}

// ---- the rows of a sum / product's components (KERNEL_SUM_EMB / KERNEL_PRODUCT_EMB) -------------------------------------
// One slot per active column of each component, in component order: slot s reads input column src[s].  A plain slot writes row
// r0[s]: the coordinate over l[s] (scale != 0: training inputs, a joint call's candidates) or the raw coordinate (scale == 0: a
// window's candidates, which the covariance kernels divide themselves).  A periodic slot writes the embedded pair to the rows r0[s]
// (cos) and r1[s] (sin) with periodic_embed_kernel's arithmetic, so that its rows are the same bits.
constexpr int STAGE_SLOTS = 64;  // the rows of all components may not exceed 64, so neither may their slots
struct RowMap {
    int n;
    int src[STAGE_SLOTS], r0[STAGE_SLOTS], r1[STAGE_SLOTS];  // r1 < 0: a plain slot
    double l[STAGE_SLOTS], p[STAGE_SLOTS];
};

// out[i * s_row + r * s_dim] for the rows i < rows of X[.][d], zero for padding rows rows <= i < rows_pad
__global__ void __launch_bounds__(256) stage_rows_kernel(const double* __restrict__ X, long long rows, long long rows_pad, int d,
                                                         RowMap m, int scale, long long s_row, long long s_dim,
                                                         double* __restrict__ out) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= rows_pad * m.n) return;
    const long long i = e / m.n;
    const int s = (int)(e - i * m.n);
    const double x = i < rows ? X[i * d + m.src[s]] : 0.0;
    if (m.r1[s] < 0) {
        out[i * s_row + (long long)m.r0[s] * s_dim] = i < rows ? (scale ? x / m.l[s] : x) : 0.0;
        return;
    }
    double c = 0.0, sn = 0.0;
    if (i < rows) {
        const double l2 = 2.0 * m.l[s];
        sincospi(2.0 * x / m.p[s], &sn, &c);
        c /= l2;
        sn /= l2;
    }
    out[i * s_row + (long long)m.r0[s] * s_dim] = c;
    out[i * s_row + (long long)m.r1[s] * s_dim] = sn;
}

// LML gradient of a periodic kernel: every entry in one launch.  One block per lower 64x64 tile, the tile's embedded rows
// (Xs[2d][Np]) and raw coordinates (the first d columns of X[N][xw]) of its rows and columns in shared memory.  Per pair W, the base covariance k and
// g = -2 dk/dr2 are formed once; W g goes to shared memory and a second pass gives warp w the dimensions j = w, w + 8, ...:
//   part[blk][0]         = sum W k                                                (-> d/d variance after / variance)
//   part[blk][1]         = sum_i W_ii                                             (-> d/d noise)
//   part[blk][2 + j]     = sum W g ((e_j - e'_j)^2 + (e_{d+j} - e'_{d+j})^2)       (dK/dl_j = g r2_j / l_j)
//   part[blk][2 + d + j] = sum W g (x_j - x'_j) (e_{d+j} e'_j - e_j e'_{d+j})       (dK/dp_j = 2 pi g delta_j sin(2 pi delta_j / p_j) / (4 l_j^2 p_j^2))
//   part[blk][2 + 2d]    = sum W dk/dalpha                                        (RationalQuadratic base only)
// Scalar lengthscales / periods are the sums of these entries over j (the host adds them).
template <int KID>
__global__ void __launch_bounds__(256) lml_grad_periodic_kernel(const double* __restrict__ Xs, const double* __restrict__ X,
                                                                const double* __restrict__ alpha, const double* __restrict__ Kinv,
                                                                int N, int d, int Np, double var, double rq_alpha,
                                                                double* __restrict__ part, int part_stride, int xw) {
    int blk = blockIdx.x;
    int bi = (int)((sqrt(8.0 * blk + 1.0) - 1.0) * 0.5);
    while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
    while (bi * (bi + 1) / 2 > blk) bi--;
    int bj = blk - bi * (bi + 1) / 2;
    const int dx = 2 * d;
    extern __shared__ double smg[];
    double* sXi = smg;               // [2d][64] embedded rows of the tile's rows
    double* sXj = sXi + dx * CT;     // [2d][64] ... and of its columns
    double* sRi = sXj + dx * CT;     // [d][64]  raw coordinates of the tile's rows
    double* sRj = sRi + d * CT;      // [d][64]  ... and of its columns
    double* sW = sRj + d * CT;       // [64 * 64] W g per pair
    __shared__ double sRed[8];
    for (int e = threadIdx.x; e < dx * CT; e += 256) {
        const size_t row = (size_t)(e / CT) * Np;
        sXi[e] = Xs[row + bi * CT + e % CT];
        sXj[e] = Xs[row + bj * CT + e % CT];
    }
    for (int e = threadIdx.x; e < d * CT; e += 256) {
        const int q = e / CT, t = e % CT, ri = bi * CT + t, rj = bj * CT + t;
        sRi[e] = ri < N ? X[(size_t)ri * xw + q] : 0.0;
        sRj[e] = rj < N ? X[(size_t)rj * xw + q] : 0.0;
    }
    __syncthreads();
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int j = bj * CT + tx;
    const double aj = alpha[j];
    const double wsym = (bi == bj) ? 1.0 : 2.0;
    double s_k = 0.0, s_tr = 0.0, s_a = 0.0;
#pragma unroll 1
    for (int r = 0; r < 16; r++) {
        const int il = ty + 4 * r, i = bi * CT + il;
        double wg = 0.0;
        if (i < N && j < N) {
            const double W = fma(alpha[i], aj, -((j <= i) ? Kinv[(size_t)i * Np + j] : Kinv[(size_t)j * Np + i])) * wsym;
            double r2 = 0.0;
            for (int q = 0; q < dx; q++) {
                const double df = sXi[q * CT + il] - sXj[q * CT + tx];
                r2 = fma(df, df, r2);
            }
            double k, g, ka;
            cov_and_radial<KID>(r2, var, rq_alpha, k, g, ka);
            s_k = fma(W, k, s_k);
            if (KID == KERNEL_RQ) s_a = fma(W, ka, s_a);
            if (i == j) s_tr += W;
            wg = W * g;
        }
        sW[il * CT + tx] = wg;
    }
    double v = block_sum<256>(s_k, sRed);
    if (threadIdx.x == 0) part[(size_t)blk * part_stride + 0] = v;
    v = block_sum<256>(s_tr, sRed);
    if (threadIdx.x == 0) part[(size_t)blk * part_stride + 1] = v;
    if (KID == KERNEL_RQ) {
        v = block_sum<256>(s_a, sRed);
        if (threadIdx.x == 0) part[(size_t)blk * part_stride + 2 + dx] = v;
    }
    __syncthreads();  // the weights of every pair are in sW
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int q = w; q < d; q += 8) {
        const double *ci = sXi + q * CT, *cj = sXj + q * CT, *si = sXi + (d + q) * CT, *sj = sXj + (d + q) * CT;
        const double *xi = sRi + q * CT, *xj = sRj + q * CT;
        double acc_l = 0.0, acc_p = 0.0;
        for (int p = lane; p < CT * CT; p += 32) {
            const int a = p >> 6, b = p & 63;
            const double dc = ci[a] - cj[b], ds = si[a] - sj[b];
            acc_l = fma(sW[p], fma(dc, dc, ds * ds), acc_l);
            acc_p = fma(sW[p] * (xi[a] - xj[b]), fma(si[a], cj[b], -(ci[a] * sj[b])), acc_p);
        }
        acc_l = warp_sum(acc_l);
        acc_p = warp_sum(acc_p);
        if (lane == 0) {
            part[(size_t)blk * part_stride + 2 + q] = acc_l;
            part[(size_t)blk * part_stride + 2 + d + q] = acc_p;
        }
    }
}

// LML gradient of a Linear component over its rows Xs[k][Np] (s_j = x_j / l_j, l_j = 1 / sqrt(var_j)): one block per lower 64x64 tile,
// the tile's rows and columns and the pair weights W in shared memory, then warp w sums the columns j = w, w + 8, ...:
//   part[blk][0] = 0, part[blk][1] = sum_i W_ii (-> d/d noise), part[blk][2 + j] = s_j^T W s_j over the tile
// dK/dvar_j = x_j x_j^T, so dLML/dvar_j = 0.5 l_j^2 s_j^T W s_j; a scalar variance takes the sum over j (the host does both).
__global__ void __launch_bounds__(256) lml_grad_linear_kernel(const double* __restrict__ Xs, const double* __restrict__ alpha,
                                                              const double* __restrict__ Kinv, int N, int k, int Np,
                                                              double* __restrict__ part, int part_stride) {
    int blk = blockIdx.x;
    int bi = (int)((sqrt(8.0 * blk + 1.0) - 1.0) * 0.5);
    while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
    while (bi * (bi + 1) / 2 > blk) bi--;
    int bj = blk - bi * (bi + 1) / 2;
    extern __shared__ double smg[];
    double* sXi = smg;             // [k][64] the tile's rows
    double* sXj = sXi + k * CT;    // [k][64] ... and its columns
    double* sW = sXj + k * CT;     // [64 * 64] W per pair
    __shared__ double sRed[8];
    for (int e = threadIdx.x; e < k * CT; e += 256) {
        const size_t row = (size_t)(e / CT) * Np;
        sXi[e] = Xs[row + bi * CT + e % CT];
        sXj[e] = Xs[row + bj * CT + e % CT];
    }
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int j = bj * CT + tx;
    const double aj = alpha[j];
    const double wsym = (bi == bj) ? 1.0 : 2.0;
    double s_tr = 0.0;
    for (int r = 0; r < 16; r++) {
        const int il = ty + 4 * r, i = bi * CT + il;
        double W = 0.0;
        // diagonal tiles: the tile holds both triangles of a symmetric quantity, take every element once
        if (i < N && j < N) {
            W = fma(alpha[i], aj, -((j <= i) ? Kinv[(size_t)i * Np + j] : Kinv[(size_t)j * Np + i])) * wsym;
            if (i == j) s_tr += W;
        }
        sW[il * CT + tx] = W;
    }
    const double v = block_sum<256>(s_tr, sRed);
    if (threadIdx.x == 0) {
        part[(size_t)blk * part_stride + 0] = 0.0;
        part[(size_t)blk * part_stride + 1] = v;
    }
    __syncthreads();  // the weights of every pair are in sW
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int q = w; q < k; q += 8) {
        const double* xi = sXi + q * CT;
        const double* xj = sXj + q * CT;
        double acc = 0.0;
        for (int p = lane; p < CT * CT; p += 32) acc = fma(sW[p] * xi[p >> 6], xj[p & 63], acc);
        acc = warp_sum(acc);
        if (lane == 0) part[(size_t)blk * part_stride + 2 + q] = acc;
    }
}

// out[q] = sum_blk part[blk][q], fixed order; one block per q
__global__ void __launch_bounds__(256) reduce_partials_kernel(const double* __restrict__ part, int nblk, int stride,
                                                              double* __restrict__ out) {
    __shared__ double sRed[8];
    int q = blockIdx.x;
    double s = 0.0;
    for (int b = threadIdx.x; b < nblk; b += 256) s += part[(size_t)b * stride + q];
    double v = block_sum<256>(s, sRed);
    if (threadIdx.x == 0) out[q] = v;
}

}  // namespace gpso
