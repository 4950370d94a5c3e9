// Posterior variance + UCB + arg-max over a window of candidates.
//
//   var_f(c) = variance - || L^-1 k*(c) ||^2 ,  k*(c) = K(X, x_c)      (gpflow.conditionals.base_conditional)
//
// For a window of Mw candidates the cross-covariance rows KsT[c][:] (written by crosscov_kernel) are multiplied by the
// lower-triangular L^-1 with the DMMA tile core: tile (I, ct) = rows [128 I, 128 I + 128) of L^-1 times candidates
// [128 ct, 128 ct + 128), contraction over k < 128 (I+1) only (block-triangular skip; inside the diagonal block the
// structural zeros are skipped at 8-row granularity).  The 128x128 product tile is never stored: the epilogue squares
// and sums it over its rows and writes ONE double per (row block, candidate):  part[I][c].  A persistent grid of one
// CTA per SM pulls tiles from an atomic counter in longest-first order so the triangular imbalance does not cost a
// tail.  Tiles are grouped so that the K* rows of PRED_GROUP candidate tiles stay resident in the 126 MB L2 while all
// of their row blocks are processed.
//
// The finalise kernel then forms var = (variance - sum_I part[I][c]) + noise (GPflow's order of operations),
// ucb = mean + varsigma * var with separate rounding of the product and the sum (numpy semantics, no FMA), and reduces
// the window to its first-maximum candidate.  Every candidate undergoes an identical operation sequence, so duplicated
// candidates produce bit-identical UCBs and the lowest-index tie-break reproduces np.argmax.
#pragma once
#include "gemm_core.cuh"

namespace gpso {

constexpr int PRED_GROUP = 8;  // candidate tiles per L2 group (8 * 128 candidates * Np * 8 B = 32 MB at Np = 4096)

struct PredictParams {
    const double* Linv;
    const double* KsT;   // [nct*128, Np]
    double* part;        // [nb, nct*128]
    int Np, nb, nct;
    int* counter;        // tile counter (zeroed before launch)
};

__device__ __forceinline__ void predict_tile_decode(int t, int nb, int nct, int& I, int& ct) {
    // groups of PRED_GROUP candidate tiles; inside a group: row blocks from the most expensive (I = nb-1) down
    int per_group = PRED_GROUP * nb;
    int grp = t / per_group;
    int r = t - grp * per_group;
    int gsize = min(PRED_GROUP, nct - grp * PRED_GROUP);  // last group may be short
    I = nb - 1 - r / gsize;
    ct = grp * PRED_GROUP + r % gsize;
}

// tile -> (row block I, candidate tile ct) over all nct * nb tiles, the short last group included: tiles of full groups first
__device__ __forceinline__ void predict_tile_of(int tile, int nb, int nct, int& I, int& ct) {
    int full_groups = nct / PRED_GROUP;
    int full_tiles = full_groups * PRED_GROUP * nb;
    if (tile < full_tiles) {
        predict_tile_decode(tile, nb, nct, I, ct);
    } else {
        int r = tile - full_tiles;
        int gsize = nct - full_groups * PRED_GROUP;
        I = nb - 1 - r / gsize;
        ct = full_groups * PRED_GROUP + r % gsize;
    }
}

__global__ void __launch_bounds__(GTHREADS, 1) predict_trmm_kernel(PredictParams P) {
    extern __shared__ double smem[];
    __shared__ int s_tile;
    __shared__ double s_red[2][GN];
    const int Np = P.Np, nb = P.nb, nct = P.nct;
    // total tiles: full groups contribute PRED_GROUP*nb, the last (short) group gsize*nb
    const int ntiles = nct * nb;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t4 = lane & 3;
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
        // column sums of squares over the warp's 64 rows
#pragma unroll
        for (int j = 0; j < 4; j++) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                s0 = fma(acc.v[i][j][0], acc.v[i][j][0], s0);
                s1 = fma(acc.v[i][j][1], acc.v[i][j][1], s1);
            }
            // reduce over g (lane bits 2..4)
#pragma unroll
            for (int o = 4; o <= 16; o <<= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (g == 0) {
                s_red[wm][wn * 32 + j * 8 + 2 * t4] = s0;
                s_red[wm][wn * 32 + j * 8 + 2 * t4 + 1] = s1;
            }
        }
        __syncthreads();
        if (threadIdx.x < GN) {
            P.part[(size_t)I * (nct * TB) + (size_t)ct * TB + threadIdx.x] = s_red[0][threadIdx.x] + s_red[1][threadIdx.x];
        }
    }
}

// ---- finalise: var, ucb, window arg-max ---------------------------------------------------------------------------
struct BestRec {
    double ucb, mean, var;
    long long idx;
};

// mode 0: write mean/var for candidates [0, Mw) of the window to out_mean/out_var (already offset to the window)
// mode 1: per-block best record -> blockbest[blockIdx.x] (mean/var are written too when out_mean is given)
// idx_map (optional): global index of window candidate c is idx_map[idx0 + c] instead of idx0 + c (refine pass of the
// screened arg-max: the window holds a gathered subset of the caller's candidates)
__global__ void __launch_bounds__(256) predict_finalize_kernel(const double* __restrict__ part, const double* __restrict__ mean,
                                                               int nb, int ldp, long long Mw, long long idx0, double variance,
                                                               double noise, double varsigma, int mode,
                                                               double* __restrict__ out_mean, double* __restrict__ out_var,
                                                               BestRec* __restrict__ blockbest,
                                                               const long long* __restrict__ idx_map) {
    long long c = (long long)blockIdx.x * 256 + threadIdx.x;
    double m = 0.0, v = 0.0, u = 0.0;
    bool valid = c < Mw;
    if (valid) {
        double ss = 0.0;
        for (int I = 0; I < nb; I++) ss += part[(size_t)I * ldp + c];
        m = mean[c];
        v = __dadd_rn(__dsub_rn(variance, ss), noise);
        u = __dadd_rn(m, __dmul_rn(varsigma, v));
    }
    if (out_mean != nullptr && valid) {
        out_mean[c] = m;
        out_var[c] = v;
    }
    if (mode == 0) return;
    // block arg-max, numpy semantics (first NaN wins; lowest index on ties)
    long long gi = valid ? (idx_map != nullptr ? idx_map[idx0 + c] : idx0 + c) : 0x7fffffffffffffffLL;
    double bu = valid ? u : -INFINITY, bm = m, bv = v;
    long long bi = gi;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ou = __shfl_xor_sync(0xffffffffu, bu, o);
        double om = __shfl_xor_sync(0xffffffffu, bm, o);
        double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (best_better(ou, oi, bu, bi)) {
            bu = ou; bm = om; bv = ov; bi = oi;
        }
    }
    __shared__ BestRec sb[8];
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sb[w] = BestRec{bu, bm, bv, bi};
    __syncthreads();
    if (threadIdx.x == 0) {
        BestRec b = sb[0];
        for (int i = 1; i < 8; i++)
            if (best_better(sb[i].ucb, sb[i].idx, b.ucb, b.idx)) b = sb[i];
        blockbest[blockIdx.x] = b;
    }
}

// predict_finalize_kernel for a kernel with Linear terms: the prior variance of candidate c is its own, mean[ldp + c] (written after the
// window's means by crosscov_kernel<KERNEL_SUM_LIN>), not one kernel variance; everything else as above
__global__ void __launch_bounds__(256) predict_finalize_kss_kernel(const double* __restrict__ part, const double* __restrict__ mean,
                                                                   int nb, int ldp, long long Mw, long long idx0, double noise,
                                                                   double varsigma, int mode, double* __restrict__ out_mean,
                                                                   double* __restrict__ out_var, BestRec* __restrict__ blockbest,
                                                                   const long long* __restrict__ idx_map) {
    long long c = (long long)blockIdx.x * 256 + threadIdx.x;
    double m = 0.0, v = 0.0, u = 0.0;
    bool valid = c < Mw;
    if (valid) {
        double ss = 0.0;
        for (int I = 0; I < nb; I++) ss += part[(size_t)I * ldp + c];
        m = mean[c];
        v = __dadd_rn(__dsub_rn(mean[ldp + c], ss), noise);
        u = __dadd_rn(m, __dmul_rn(varsigma, v));
    }
    if (out_mean != nullptr && valid) {
        out_mean[c] = m;
        out_var[c] = v;
    }
    if (mode == 0) return;
    long long gi = valid ? (idx_map != nullptr ? idx_map[idx0 + c] : idx0 + c) : 0x7fffffffffffffffLL;
    double bu = valid ? u : -INFINITY, bm = m, bv = v;
    long long bi = gi;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ou = __shfl_xor_sync(0xffffffffu, bu, o);
        double om = __shfl_xor_sync(0xffffffffu, bm, o);
        double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (best_better(ou, oi, bu, bi)) {
            bu = ou; bm = om; bv = ov; bi = oi;
        }
    }
    __shared__ BestRec sb[8];
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sb[w] = BestRec{bu, bm, bv, bi};
    __syncthreads();
    if (threadIdx.x == 0) {
        BestRec b = sb[0];
        for (int i = 1; i < 8; i++)
            if (best_better(sb[i].ucb, sb[i].idx, b.ucb, b.idx)) b = sb[i];
        blockbest[blockIdx.x] = b;
    }
}

// running[0] = best of (running[0] if !first) and blockbest[0..n)
__global__ void __launch_bounds__(256) best_merge_kernel(const BestRec* __restrict__ blockbest, int n, BestRec* __restrict__ running,
                                                         int first) {
    BestRec b;
    b.ucb = -INFINITY; b.mean = 0.0; b.var = 0.0; b.idx = 0x7fffffffffffffffLL;
    for (int i = threadIdx.x; i < n; i += 256) {
        BestRec o = blockbest[i];
        if (best_better(o.ucb, o.idx, b.ucb, b.idx)) b = o;
    }
    __shared__ BestRec sb[256];
    sb[threadIdx.x] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
        BestRec r = sb[0];
        for (int i = 1; i < 256; i++)
            if (best_better(sb[i].ucb, sb[i].idx, r.ucb, r.idx)) r = sb[i];
        if (!first) {
            BestRec o = running[0];
            if (best_better(o.ucb, o.idx, r.ucb, r.idx)) r = o;
        }
        running[0] = r;
    }
}

// ---- top-k --------------------------------------------------------------------------------------------------------------
// The k best candidates of one window in arg-max order (first NaN, then the larger UCB, the lowest index on ties): k passes of
// a block-wide arg-max that skips the winners of the earlier passes.  mean/var are the window's finalised values; the UCB is
// formed exactly as in predict_finalize_kernel, so record 0 equals the fused arg-max bit for bit.  Slots beyond the number
// of candidates keep idx = LLONG_MAX.
constexpr int TOPK_MAX = 64;

__global__ void __launch_bounds__(1024) topk_window_kernel(const double* __restrict__ mean, const double* __restrict__ var, long long Mw,
                                                           long long idx0, double varsigma, int k, BestRec* __restrict__ out) {
    __shared__ long long taken[TOPK_MAX];
    __shared__ BestRec sb[32];
    const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
    for (int pass = 0; pass < k; pass++) {
        double bu = -INFINITY, bm = 0.0, bv = 0.0;
        long long bi = 0x7fffffffffffffffLL;
        for (long long c = tid; c < Mw; c += 1024) {
            const long long gi = idx0 + c;
            bool skip = false;
            for (int t = 0; t < pass; t++) skip |= (taken[t] == gi);
            if (skip) continue;
            const double m = mean[c], v = var[c];
            const double u = __dadd_rn(m, __dmul_rn(varsigma, v));
            if (best_better(u, gi, bu, bi)) {
                bu = u; bm = m; bv = v; bi = gi;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ou = __shfl_xor_sync(0xffffffffu, bu, o);
            double om = __shfl_xor_sync(0xffffffffu, bm, o);
            double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (best_better(ou, oi, bu, bi)) {
                bu = ou; bm = om; bv = ov; bi = oi;
            }
        }
        if (l == 0) sb[w] = BestRec{bu, bm, bv, bi};
        __syncthreads();
        if (tid == 0) {
            BestRec b = sb[0];
            for (int i = 1; i < 32; i++)
                if (best_better(sb[i].ucb, sb[i].idx, b.ucb, b.idx)) b = sb[i];
            out[pass] = b;
            taken[pass] = b.idx;
        }
        __syncthreads();
    }
}

}  // namespace gpso
