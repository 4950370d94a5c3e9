// Joint posterior of M candidates (gpflow.models.GPR.predict_f(Xnew, full_cov=True) and predict_f_samples):
//
//   A = L^-1 K(X, X*)        cov = K(X*, X*) - A^T A        f = mean + chol(cov + jitter I) z
//
// Every stage is FP64 on the DMMA tile core of gemm_core.cuh, and every buffer is padded to Mp = M rounded up to 128:
//   joint_v_kernel       V^T[c][k] = (L^-1 k*(c))_k: the predict_trmm_kernel schedule (row block I of L^-1 times candidate
//                        tile ct, contraction over k < 128 (I+1)), the tile is stored transposed so that each candidate's
//                        row is contiguous -- the K-contiguous operand the next product wants
//   joint_syrk_kernel    lower tiles (a >= b) of Sigma = K** - V^T V (+ jitter on the diagonal), the prior covariance
//                        evaluated in the epilogue exactly as gram_kernel does (difference-first r2, cov_from_r2), identity on
//                        padding rows / columns, zeros above the diagonal
//   joint_mirror_kernel  cov[M][M] with both triangles from the lower one (exactly symmetric)
//   joint_tril_kernel    zeros the strict upper triangle of the diagonal tiles after the Cholesky (its tile updates write
//                        whole 128x128 tiles, the diagonal-block task whole 32-wide row segments)
//   joint_pad_kernel     Z[Sp][Mp] = z[S][M] with zero padding (the tile core loads whole slabs)
//   joint_sample_kernel  out[s][m] = mean[m] + sum_k Lc[m][k] Z[s][k]: row block I of Lc times sample tile, contraction over
//                        k < 128 (I+1) with the diagonal-block skip of the tile core
// The 128x128 product tiles of the store epilogues go through shared memory (odd pitch) so that the transposed global
// stores coalesce.  A candidate's row of V^T, and therefore its row and column of Sigma, is computed by the same operation
// sequence wherever it sits in the batch: duplicated candidates give bit-identical rows and columns.
#pragma once
#include "gemm_core.cuh"
#include "kern_dense.cuh"
#include "kern_predict.cuh"

namespace gpso {

constexpr int JST = TB + 1;  // row pitch of the staged 128x128 tile (odd: conflict-free column reads)

// acc -> stage[r][c] (r = tile row, c = tile column).  All 256 threads; the ring of the main loop is reused.
__device__ __forceinline__ void joint_stage_tile(const TileAcc& acc, double* stage) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
    __syncthreads();  // every warp is done reading the operand ring
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int r = wm * 64 + i * 8 + g, c = wn * 32 + j * 8 + 2 * t;
            stage[r * JST + c] = acc.v[i][j][0];
            stage[r * JST + c + 1] = acc.v[i][j][1];
        }
    __syncthreads();
}

struct JointVParams {
    const double* Linv;  // [Np, Np]
    const double* KsT;   // [nct*128, Np]
    double* VT;          // [nct*128, Np]
    int Np, nb, nct;
    int* counter;        // tile counter (zeroed before launch)
};

__global__ void __launch_bounds__(GTHREADS, 1) joint_v_kernel(JointVParams P) {
    extern __shared__ double smem[];
    __shared__ int s_tile;
    const int Np = P.Np, nb = P.nb, nct = P.nct;
    const int ntiles = nct * nb;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_tile = atomicAdd(P.counter, 1);
        __syncthreads();
        const int tile = s_tile;
        if (tile >= ntiles) break;
        int I, ct;
        predict_tile_of(tile, nb, nct, I, ct);
        TileOperands w;
        w.A = P.Linv + (size_t)I * TB * Np;
        w.B = P.KsT + (size_t)ct * TB * Np;
        w.lda = w.ldb = Np;
        w.kbeg = 0;
        w.kend = (I + 1) * TB;
        w.tri_off = I * TB;
        TileAcc acc;
        gemm_tile_mainloop(w, acc, smem);
        joint_stage_tile(acc, smem);
        // stage[r][c] = V[128 I + r][128 ct + c]  ->  VT[128 ct + c][128 I + r]
        double* dst = P.VT + (size_t)ct * TB * Np + (size_t)I * TB;
        for (int e = threadIdx.x; e < TB * TB; e += GTHREADS) {
            const int c = e >> 7, r = e & (TB - 1);
            dst[(size_t)c * Np + r] = smem[r * JST + c];
        }
    }
}

// grid = mb (mb + 1) / 2 lower tiles of the [Mp, Mp] matrix.  Xcs[dim][Mp]: scaled candidates (scale_inputs_kernel).
template <int KID>
__global__ void __launch_bounds__(GTHREADS, 1) joint_syrk_kernel(const double* __restrict__ VT, const double* __restrict__ Xcs, int M,
                                                                 int Mp, int Np, int d, double var, double jitter,
                                                                 double* __restrict__ Sigma) {
    extern __shared__ double smem[];
    int a, b;
    tri_index(blockIdx.x, a, b);
    TileOperands w;
    w.A = VT + (size_t)a * TB * Np;
    w.B = VT + (size_t)b * TB * Np;
    w.lda = w.ldb = Np;
    w.kbeg = 0;
    w.kend = Np;
    w.tri_off = TRI_DENSE;
    TileAcc acc;
    gemm_tile_mainloop(w, acc, smem);
    joint_stage_tile(acc, smem);
    for (int e = threadIdx.x; e < TB * TB; e += GTHREADS) {
        const int r = e >> 7, c = e & (TB - 1);
        const int gi = a * TB + r, gj = b * TB + c;
        double v;
        if (gi >= M || gj >= M) {
            v = (gi == gj) ? 1.0 : 0.0;
        } else if (gj > gi) {
            v = 0.0;
        } else {
            double r2 = 0.0;
            for (int dim = 0; dim < d; dim++) {
                const double df = Xcs[(size_t)dim * Mp + gi] - Xcs[(size_t)dim * Mp + gj];
                r2 = fma(df, df, r2);
            }
            v = cov_from_r2<KID>(r2, var) - smem[r * JST + c];
            if (gi == gj) v += jitter;
        }
        Sigma[(size_t)gi * Mp + gj] = v;
    }
}

// cov[i][j] (i, j < M) from the lower triangle of Sigma; grid (ceil(M/32), ceil(M/32)), block (32, 8)
__global__ void __launch_bounds__(256) joint_mirror_kernel(const double* __restrict__ Sigma, int M, int Mp, double* __restrict__ cov) {
    __shared__ double s[32][33];
    const int bx = blockIdx.x, by = blockIdx.y, tx = threadIdx.x, ty = threadIdx.y;
    if (by >= bx) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = by * 32 + ty + 8 * k, j = bx * 32 + tx;
            if (i < M && j < M) cov[(size_t)i * M + j] = (j <= i) ? Sigma[(size_t)i * Mp + j] : Sigma[(size_t)j * Mp + i];
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < 4; k++) s[ty + 8 * k][tx] = Sigma[(size_t)(bx * 32 + ty + 8 * k) * Mp + by * 32 + tx];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int i = by * 32 + ty + 8 * k, j = bx * 32 + tx;
        if (i < M && j < M) cov[(size_t)i * M + j] = s[tx][ty + 8 * k];
    }
}

// strict upper triangle of the diagonal tile blockIdx.x -> 0
__global__ void __launch_bounds__(256) joint_tril_kernel(double* __restrict__ L, int Mp) {
    double* tile = L + (size_t)blockIdx.x * TB * Mp + (size_t)blockIdx.x * TB;
    for (int e = threadIdx.x; e < TB * TB; e += 256) {
        const int r = e >> 7, c = e & (TB - 1);
        if (c > r) tile[(size_t)r * Mp + c] = 0.0;
    }
}

__global__ void __launch_bounds__(256) joint_pad_kernel(const double* __restrict__ z, int S, int M, int Sp, int Mp, double* __restrict__ Z) {
    const long long n = (long long)Sp * Mp;
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < n; e += (long long)gridDim.x * 256) {
        const int s = (int)(e / Mp), m = (int)(e % Mp);
        Z[e] = (s < S && m < M) ? z[(size_t)s * M + m] : 0.0;
    }
}

// grid = mb * nsb tiles, long contractions (large I) first
__global__ void __launch_bounds__(GTHREADS, 1) joint_sample_kernel(const double* __restrict__ Lc, const double* __restrict__ Z,
                                                                   const double* __restrict__ mean, int M, int Mp, int S, int mb,
                                                                   int nsb, double* __restrict__ out) {
    extern __shared__ double smem[];
    const int I = mb - 1 - (int)blockIdx.x / nsb, st = (int)blockIdx.x % nsb;
    TileOperands w;
    w.A = Lc + (size_t)I * TB * Mp;
    w.B = Z + (size_t)st * TB * Mp;
    w.lda = w.ldb = Mp;
    w.kbeg = 0;
    w.kend = (I + 1) * TB;
    w.tri_off = I * TB;
    TileAcc acc;
    gemm_tile_mainloop(w, acc, smem);
    joint_stage_tile(acc, smem);
    // stage[m][s] = (Lc Z^T)[128 I + m][128 st + s]  ->  out[128 st + s][128 I + m]
    for (int e = threadIdx.x; e < TB * TB; e += GTHREADS) {
        const int s = e >> 7, m = e & (TB - 1);
        const int gs = st * TB + s, gm = I * TB + m;
        if (gs < S && gm < M) out[(size_t)gs * M + gm] = mean[gm] + smem[m * JST + s];
    }
}

}  // namespace gpso
