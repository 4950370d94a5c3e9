// Posterior-variance product V = L^-1 K* on the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM),
// exact-integer ("Ozaki scheme") emulation of the fp64 product.
//
// Why: B200's FP64 pipe peaks at 37 TFLOP/s (DMMA == DFMA rate, profiles/r01_fp64_probe.txt) while its int8 tensor
// path sustains 4.5 POP/s (profiles/r01_i8_tcgen05_probe.txt).  Both operands are split into S signed 8-bit digits of a
// fixed-point representation,
//
//      L^-1[i,k] = 2^(e_i - (8S-2)) * sum_p a_p[i,k] 256^(S-1-p)        (per-row exponent e_i)
//      K*[k,c]   = 2^(f   - (8S-2)) * sum_q b_q[k,c] 256^(S-1-q)        (one exponent f: 0 <= k* <= kernel variance)
//
// (balanced digits in [-128,127], so slice products are zero-mean), and
//
//      V[i,c] = 2^(e_i + f - 2(8S-2) + 8(S-1)) * sum_{t<S} 256^(S-1-t) * C_t[i,c],    C_t = sum_{p+q=t} a_p b_q^T
//
// where every C_t is an EXACT int32 sum (|a b| <= 2^14, K <= 8192, <= 8 digit pairs per level).  The only rounding is
// the fixed-point conversion of the operands (8S-2 bits: 46 at S=6) and the neglected levels t >= S; S is chosen per fit
// from the row scales so that the error stays two orders below the parity tolerance (see gpso_capi.cu, pick_slices).
// Integer accumulation makes the result independent of summation order, tile position and GPU: duplicated candidates
// give bit-identical variances by construction.
//
// Data flow (nothing below is a general GEMM library; every layout is produced by our own kernels for this product):
//   linv_slices_kernel      L^-1 (fp64, lower)  -> A digit tiles  [I][ks][p][128 rows x 32 k]  canonical UMMA K-major,
//                                                   no-swizzle core matrices (8 rows x 16 B), once per factorisation
//   crosscov_slices_kernel  candidates -> k*(fp64, registers) -> B digit tiles [ct][ks][q][64 cand x 32 k] + posterior mean
//   ozaki_kernel<S, MODE>   warp-specialised persistent kernel, one CTA per SM (MODE: OZ_TRMM below; OZ_LAUUM / OZ_GEMM reuse the
//                           mainloop for K_y^-1 = L^-T L^-1 and the inverse factor of the fit path, see OzItems and the epilogue):
//        warp 0   producer : cp.async.bulk (UBLKCP) of one k-step (S*4 KB of A, S*2 KB of B) per stage, mbarrier tx
//        warp 1   issuer   : tcgen05.mma.cta_group::1.kind::i8, M=128, N up to 256: digit p of A against digits
//                            0..S-1-p of B stacked along N, accumulating level t=p+q into TMEM columns [64t, 64t+64)
//        warps 2-9 epilogue (two per TMEM lane group, 32 candidates each): tcgen05.ld, exact int64 recombination, one
//                            fp64 rounding, square, column sums over the
//                            128 rows -> part[I][c]   (same partial-sum interface as the DMMA kernel)
//   Work unit = candidate tile x PAIR of row blocks (I, nb-1-I): every unit costs nb+1 k-blocks, so a static
//   round-robin over the persistent CTAs is balanced and the 148 CTAs share ~10 candidate tiles of B and all of A in L2.
#pragma once
#include "common.cuh"

namespace gpso {

constexpr int OZ_NT = 64;                 // candidates per tile
constexpr int OZ_A_SLICE = 128 * 32;      // bytes of one A digit tile (128 rows x 32 k)
constexpr int OZ_B_SLICE = OZ_NT * 32;    // bytes of one B digit tile
constexpr int OZ_THREADS = 320;            // producer warp, issuer warp, 8 epilogue warps
constexpr int OZ_TMEM_COLS = 512;

template <int S>
struct OzCfg {
    static constexpr int STAGE_BYTES = S * (OZ_A_SLICE + OZ_B_SLICE);
    static constexpr int STAGES = (S <= 5) ? 6 : (S == 6) ? 5 : 4;
    static constexpr int RING_BYTES = STAGES * STAGE_BYTES;
    static constexpr int SMEM_BYTES = RING_BYTES + 1024 /* barriers + tmem slot */ + 4 * OZ_NT * (int)sizeof(double);
    // OZ_TRMM: two k-steps per ring stage (consecutive k-steps are contiguous in both digit buffers: one bulk copy of A and one of
    // B per stage) and ONE tcgen05.commit per stage -- a commit per 32-wide k-step cost ~40 clocks of tensor pipe each (8 % of the
    // screening product, profiles/README.md round 2).  Every row block has a multiple of 4 k-steps.
    static constexpr int KPS_TRMM = (S <= 6) ? 2 : 1;
    static constexpr int STAGE_BYTES_TRMM = KPS_TRMM * STAGE_BYTES;
    static constexpr int STAGES_TRMM = (S <= 6) ? 3 : STAGES;
    static constexpr int RING_BYTES_TRMM = STAGES_TRMM * STAGE_BYTES_TRMM;
    static constexpr int SMEM_BYTES_TRMM = RING_BYTES_TRMM + 1024 + 4 * OZ_NT * (int)sizeof(double);
};

struct OzParams {
    const uint8_t* A;        // [nb][nks][S][4096]
    const uint8_t* B;        // [nct][nks][S][2048]   (OZ_LAUUM: the A tiles again, read as 64-row halves)
    const double* rowscale;  // [Np] 2^(e_i)
    double* part;            // [nb][ldp]
    double gscale;           // 2^(f - 2(8S-2) + 8(S-1))
    int nb, nks, nct;
    long long ldp;
    // OZ_LAUUM / OZ_GEMM only
    const int* items;        // OZ_LAUUM: [rounds][gridDim.x]  (row block << 16 | 64-wide column tile), -1 = none
                             // OZ_GEMM:  [rounds][gridDim.x][4]  (row block, 64-row tile of B, first k-step, k-steps), I < 0 = none
    int rounds;
    double* out;             // [Np][Np] row-major output
    int Np;
    const double* colscale;  // OZ_GEMM: row scales of the B operand (its rows are the output columns)
    double* out_t;           // OZ_GEMM: optional second, transposed copy of the output (out_t[col][row])
    double sign;             // OZ_GEMM: +1 / -1
    int accumulate;          // OZ_GEMM: 1 = out += sign * product (Schur-complement update of the hybrid factorisation), 0 = store
};

// What one launch of the product kernel computes
//   OZ_TRMM   part[I][c] = sum over the 128 rows of block I of (L^-1 k*_c)^2      (posterior variance, predict path)
//   OZ_LAUUM  K_y^-1[i][j] = sum_{k >= i} L^-T[i][k] L^-T[j][k], j <= i            (fit path: the gradient's trace terms)
//   OZ_GEMM   out[i][j] = sign * sum_{k in item range} A[i][k] B[j][k]                 (fit path: the two products per level of
//             the recursive-doubling inverse factor; tiles, k-ranges and the tile -> CTA deal come from a host table)
constexpr int OZ_TRMM = 0;
constexpr int OZ_LAUUM = 1;
constexpr int OZ_GEMM = 2;

// Sequence of work items of one persistent CTA; producer, MMA issuer and epilogue warps each walk their own copy.
// An item = one 128 x 64 accumulator tile: row block I, column tile ct, k-steps [ks0, ks0 + n).
template <int MODE>
struct OzItems {
    const OzParams& P;
    long long u;
    int it, r;
    __device__ __forceinline__ OzItems(const OzParams& P_) : P(P_), u(blockIdx.x), it(0), r(0) {}
    __device__ __forceinline__ bool next(int& I, long long& ct, int& ks0, int& n) {
        if (MODE == OZ_TRMM) {
            // candidate tile x PAIR of row blocks (nb-1-j, j): every unit costs nb+1 k-blocks, static round-robin is balanced
            const int npairs = (P.nb + 1) >> 1;
            if (u >= (long long)P.nct * npairs) return false;
            ct = u / npairs;
            const int j = (int)(u - ct * npairs);
            const int items = (P.nb - 1 - j != j) ? 2 : 1;
            I = it == 0 ? P.nb - 1 - j : j;
            ks0 = 0;
            n = 4 * (I + 1);
            if (++it == items) {
                it = 0;
                u += gridDim.x;
            }
            return true;
        } else if (MODE == OZ_GEMM) {
            while (r < P.rounds) {
                const int4 it4 = reinterpret_cast<const int4*>(P.items)[(size_t)r * gridDim.x + blockIdx.x];
                r++;
                if (it4.x >= 0) {
                    I = it4.x;
                    ct = it4.y;
                    ks0 = it4.z;
                    n = it4.w;
                    return true;
                }
            }
            return false;
        } else {
            // the host dealt the tiles to the CTAs longest-first (gpso_capi.cu: build_lauum_items)
            while (r < P.rounds) {
                const int code = P.items[(size_t)r * gridDim.x + blockIdx.x];
                r++;
                if (code >= 0) {
                    I = code >> 16;
                    ct = code & 0xffff;
                    ks0 = 4 * I;
                    n = P.nks - ks0;
                    return true;
                }
            }
            return false;
        }
    }
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t oz_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void oz_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(oz_smem(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void oz_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\tOZ_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra OZ_DONE;\n\tbra OZ_WAIT;\n\tOZ_DONE:\n\t}\n" ::"r"(oz_smem(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void oz_mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(oz_smem(bar)) : "memory");
}
__device__ __forceinline__ void oz_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(oz_smem(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void oz_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(oz_smem(dst)),
                 "l"(src), "r"(bytes), "r"(oz_smem(bar))
                 : "memory");
}
// same copy with an L2 eviction-priority hint (createpolicy): the A digits of L^-1 are re-read by every candidate tile of
// every window and must survive the 2 GB of B digits that stream through L2 per window
__device__ __forceinline__ void oz_bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     oz_smem(dst)),
                 "l"(src), "r"(bytes), "r"(oz_smem(bar)), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ uint64_t oz_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void oz_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(oz_smem(bar)) : "memory");
}
__device__ __forceinline__ void oz_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void oz_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, no swizzle: core matrix = 8 rows x 16 B contiguous; LBO = 128 B between the
// two 16-byte K chunks of a K=32 instruction, SBO = 256 B between 8-row groups (validated by tools/microbench/i8_probe.cu)
__device__ __forceinline__ uint64_t oz_desc(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
}
// instruction descriptor: D = S32, A = B = signed int8, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t oz_idesc(int n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void oz_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void oz_tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void oz_tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}

// ---- fixed-point digits -------------------------------------------------------------------------------------------
// x * scale is rounded to an integer X with |X| < 2^(8S-2); its balanced base-256 digits d_p in [-128,127]
// (X = sum_p d_p 256^p) are the bytes of (X + 0x80..80) ^ 0x80..80 with the constant covering bytes 0..S-2: adding 128 to
// every lower byte turns the signed digit into an unsigned byte with the right carry, the xor maps it back to int8.
template <int S>
__device__ __forceinline__ unsigned long long oz_digits(double x, double scale) {
    long long X = __double2ll_rn(x * scale);
    constexpr unsigned long long C = (S >= 8 ? 0x0080808080808080ULL : (0x8080808080808080ULL >> (8 * (9 - S))));
    unsigned long long Y = (unsigned long long)X + C;
    return Y ^ C;
}
// byte `pos` (0..3) of word w <- byte `b` (0..7) of the digit word z
__device__ __forceinline__ uint32_t oz_put(uint32_t w, unsigned long long z, int b, int pos) {
    uint32_t src = (b < 4) ? (uint32_t)z : (uint32_t)(z >> 32);
    uint32_t sel = 0x3210u;
    sel = (sel & ~(0xFu << (4 * pos))) | ((uint32_t)(4 + (b & 3)) << (4 * pos));
    return __byte_perm(w, src, sel);
}

// ---- A digit tiles from L^-1 ----------------------------------------------------------------------------------------
// rowscale[i] = 2^(e_i) with max_k |Linv[i,k]| < 2^(e_i - 0) (one warp per row, k <= i only)
// UPPER: the matrix is L^-T (row i holds column i of L^-1, k >= i)
// rowl2 (optional): sum of squares of the row -- the error model of the screening pass wants |L^-1|_F^2 and the largest row norm
template <bool UPPER>
__global__ void __launch_bounds__(256) linv_rowscale_kernel(const double* __restrict__ Linv, int Np, double* __restrict__ rowscale,
                                                            double* __restrict__ rowmax, double* __restrict__ rowl2 = nullptr) {
    int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= Np) return;
    const double* r = Linv + (size_t)row * Np;
    double m = 0.0, s2 = 0.0;
    if (UPPER) {
        for (int k = row + lane; k < Np; k += 32) {
            m = fmax(m, fabs(r[k]));
            s2 = fma(r[k], r[k], s2);
        }
    } else {
        for (int k = lane; k <= row; k += 32) {
            m = fmax(m, fabs(r[k]));
            s2 = fma(r[k], r[k], s2);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) {
        int e = (m > 0.0 && isfinite(m)) ? ilogb(m) + 1 : 0;
        rowscale[row] = ldexp(1.0, e);
        rowmax[row] = m;
        if (rowl2 != nullptr) rowl2[row] = s2;
    }
}

template <int S, bool UPPER>
__global__ void __launch_bounds__(256) linv_slices_kernel(const double* __restrict__ Linv, const double* __restrict__ rowscale, int Np,
                                                          int nks, uint8_t* __restrict__ A) {
    const int ks = blockIdx.x, I = blockIdx.y;
    if (UPPER ? (ks < 4 * I) : (ks >= 4 * (I + 1))) return;  // the other side of the block diagonal: never read
    const int r = threadIdx.x & 127, half = threadIdx.x >> 7;
    const int row = I * 128 + r;
    const double scale = ldexp(1.0, 8 * S - 2) / rowscale[row];
    const double* src = Linv + (size_t)row * Np + ks * 32 + half * 16;
    uint32_t out[S][4];
#pragma unroll
    for (int p = 0; p < S; p++) out[p][0] = out[p][1] = out[p][2] = out[p][3] = 0u;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        unsigned long long z = oz_digits<S>(src[i], scale);
#pragma unroll
        for (int p = 0; p < S; p++) out[p][i >> 2] = oz_put(out[p][i >> 2], z, S - 1 - p, i & 3);  // slice 0 = most significant
    }
    uint8_t* dst = A + ((size_t)I * nks + ks) * S * OZ_A_SLICE + (r >> 3) * 256 + half * 128 + (r & 7) * 16;
#pragma unroll
    for (int p = 0; p < S; p++) *reinterpret_cast<uint4*>(dst + (size_t)p * OZ_A_SLICE) = make_uint4(out[p][0], out[p][1], out[p][2], out[p][3]);
}

// ---- operands of the recursive-doubling inverse (fit path, OZ_GEMM) -----------------------------------------------------
// At level s the diagonal blocks of s tiles of L^-1 are complete.  The products of the level read, per 128-row tile I with
// block [b0, b1) = [floor(I/s) s, min(b0+s, nb)) and pair start a = floor(I/2s) 2s:
//   OZR_LINVT  L^-T rows of the first half of a pair,  k in tiles [I, b1)   (upper part of the block: operand of X^T = L11^-T L21^T)
//   OZR_LINV   L^-1 rows of the second half of a pair, k in tiles [b0, I]   (lower part of the block: operand of Y = L22^-1 X)
//   OZR_XT     X^T rows of the first half of a pair,  k in tiles [a+s, min(a+2s, nb))
//   OZR_L      rows of the Cholesky factor, k in tiles [0, I)   (strictly below the diagonal tile: the L21 blocks)
// and of the hybrid factorisation (gpso_capi.cu: hybrid_node), for a node split after s tiles:
//   OZR_PANEL  rows I >= s, k in tiles [0, s)      (A21, later L21: operand of L21 = A21 L11^-T, of the Schur update and of X^T)
//   OZR_LOWER  rows I <  s, k in tiles [0, I]      (L11^-1: operand of L21 = A21 L11^-T)
// Each row is scaled by a power of two above its largest entry IN THAT RANGE, then cut into S balanced 8-bit digits.
constexpr int OZR_LINVT = 0, OZR_LINV = 1, OZR_XT = 2, OZR_L = 3, OZR_PANEL = 4, OZR_LOWER = 5;

__device__ __forceinline__ void ozr_tile_range(int kind, int I, int s, int nb, int& t0, int& t1) {
    const int b0 = (I / s) * s, b1 = min(b0 + s, nb), a = (I / (2 * s)) * (2 * s);
    if (kind == OZR_LINVT) {
        t0 = I, t1 = (I < a + s) ? b1 : I;          // only first-half rows are read (operand of X^T)
    } else if (kind == OZR_LINV) {
        t0 = b0, t1 = (I >= a + s) ? I + 1 : b0;    // only second-half rows are read (operand of Y)
    } else if (kind == OZR_XT) {
        t0 = a + s, t1 = (I < a + s) ? min(a + 2 * s, nb) : a + s;  // second-half rows: empty
    } else if (kind == OZR_PANEL) {
        t0 = 0, t1 = (I >= s) ? s : 0;
    } else if (kind == OZR_LOWER) {
        t0 = 0, t1 = (I < s) ? I + 1 : 0;
    } else {
        t0 = 0, t1 = I;
    }
}

__global__ void __launch_bounds__(256) range_rowscale_kernel(const double* __restrict__ M, int Np, int kind, int s, int nb,
                                                             double* __restrict__ rowscale) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= Np) return;
    int t0, t1;
    ozr_tile_range(kind, row >> 7, s, nb, t0, t1);
    const double* r = M + (size_t)row * Np;
    double m = 0.0;
    for (int k = t0 * 128 + lane; k < t1 * 128; k += 32) m = fmax(m, fabs(r[k]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) rowscale[row] = ldexp(1.0, (m > 0.0 && isfinite(m)) ? ilogb(m) + 1 : 0);
}

template <int S>
__global__ void __launch_bounds__(256) range_slices_kernel(const double* __restrict__ M, const double* __restrict__ rowscale, int Np,
                                                           int nks, int kind, int s, int nb, uint8_t* __restrict__ A) {
    const int ks = blockIdx.x, I = blockIdx.y;
    int t0, t1;
    ozr_tile_range(kind, I, s, nb, t0, t1);
    if (ks < 4 * t0 || ks >= 4 * t1) return;
    const int r = threadIdx.x & 127, half = threadIdx.x >> 7;
    const int row = I * 128 + r;
    const double scale = ldexp(1.0, 8 * S - 2) / rowscale[row];
    const double* src = M + (size_t)row * Np + ks * 32 + half * 16;
    uint32_t out[S][4];
#pragma unroll
    for (int p = 0; p < S; p++) out[p][0] = out[p][1] = out[p][2] = out[p][3] = 0u;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        unsigned long long z = oz_digits<S>(src[i], scale);
#pragma unroll
        for (int p = 0; p < S; p++) out[p][i >> 2] = oz_put(out[p][i >> 2], z, S - 1 - p, i & 3);
    }
    uint8_t* dst = A + ((size_t)I * nks + ks) * S * OZ_A_SLICE + (r >> 3) * 256 + half * 128 + (r & 7) * 16;
#pragma unroll
    for (int p = 0; p < S; p++) *reinterpret_cast<uint4*>(dst + (size_t)p * OZ_A_SLICE) = make_uint4(out[p][0], out[p][1], out[p][2], out[p][3]);
}

// ---- B digit tiles + posterior mean from the candidates -------------------------------------------------------------
// One block = one candidate tile (64 candidates) x all training points, in super-steps of OZ_XK = 128 training points.
// Register tile per thread: 2 candidates (cl and cl + 32, cl = lane) x 16 consecutive training points (warp w owns points
// 16 w .. 16 w + 15 of the super-step), so that every shared-memory load feeds 16 or 32 distance updates: the training
// coordinates are warp-wide broadcasts (LDS.128, one wavefront for two points), the candidate coordinates two conflict-free
// LDS.64 per dimension.  ~0.1 shared-memory wavefronts per covariance element instead of 0.35 -- this kernel runs beside the
// persistent tensor-core product kernel of the previous window, which keeps the shared-memory ports ~85 % busy with UMMA
// operand reads and bulk-copy writes (profiles/r01s4_overlap.md); and 32 independent covariance chains per thread keep the
// FP64 pipe fed with 8 warps.  Every candidate goes through the same operation sequence (position-independent results).
constexpr int OZ_XK = 128;  // training points per super-step of crosscov_slices_kernel
constexpr int XW = 4;       // covariance evaluations interleaved per thread (independent FP64 chains)

template <int KID, int S>
__global__ void __launch_bounds__(256, 2) crosscov_slices_kernel(const double* __restrict__ Xc, long long Mw, int d,
                                                              const double* __restrict__ ls, int n_ls,
                                                              const double* __restrict__ Xs, const double* __restrict__ alpha, int N,
                                                              int Np, double var, double c0, double bscale, int nks,
                                                              uint8_t* __restrict__ B, double* __restrict__ mean, double rq_alpha,
                                                              SumTable sum, SumRows srow) {
    // sum / product: the C components' scaled coordinates are dx = C d rows ([C][d] component-major), in Xs and in shared memory alike
    const int dx = embedded_composite(KID) ? srow.width : (composite_kernel(KID) ? sum.n * d : d);
    extern __shared__ double sm[];
    double* sC = sm;                      // [dx][64]      scaled candidate coordinates, dimension-major
    double* sX = sC + dx * OZ_NT;         // [2][dx][128]  scaled training coordinates of the current / next super-step
    double* sAl = sX + 2 * dx * OZ_XK;    // [2][128]
    double* sR = sAl + 2 * OZ_XK;         // [8][64]       per-warp partial means
    const int tid = threadIdx.x, cl = tid & 31, kg = tid >> 5;
    const long long ct = blockIdx.x;
    if constexpr (composite_kernel(KID)) {
        for (int e = tid; e < OZ_NT * dx; e += 256) {
            int cc = e / dx, qd = e - cc * dx, dim = qd % d;  // qd = q d + dim: component q divides by its own lengthscales
            long long cg = ct * OZ_NT + cc;
            // periodic components: candidate rows of the table's width, row qd divided by ls[qd]
            sC[qd * OZ_NT + cc] = (cg < Mw) ? Xc[embedded_composite(KID) ? cg * dx + qd : cg * d + dim] / ls[qd] : 0.0;
        }
    } else {
        for (int e = tid; e < OZ_NT * d; e += 256) {
            int cc = e / d, dim = e - cc * d;
            long long cg = ct * OZ_NT + cc;
            sC[dim * OZ_NT + cc] = (cg < Mw) ? Xc[cg * d + dim] / ls[n_ls > 1 ? dim : 0] : 0.0;
        }
    }
    for (int e = tid; e < dx * OZ_XK; e += 256) sX[e] = Xs[(size_t)(e >> 7) * Np + (e & 127)];
    if (tid < OZ_XK) sAl[tid] = alpha[tid];
    const bool cvalid[2] = {ct * OZ_NT + cl < Mw, ct * OZ_NT + cl + 32 < Mw};
    double macc[2] = {0.0, 0.0};
    const int nss = Np / OZ_XK;
    for (int ss = 0; ss < nss; ss++) {
        cp_async_wait<0>();
        __syncthreads();
        const int b = ss & 1;
        if (ss + 1 < nss) {
            // next slab of training coordinates / alpha: asynchronous 16-byte copies (LDGSTS), no registers and no
            // scoreboard stall in front of the FP64 work (13 % of the issue stalls when these were plain loads)
            double* nx = sX + (b ^ 1) * dx * OZ_XK;
            for (int e = tid; e < dx * (OZ_XK / 2); e += 256) {
                const int dim = e >> 6, pr = (e & 63) * 2;
                cp_async16(nx + dim * OZ_XK + pr, Xs + (size_t)dim * Np + (ss + 1) * OZ_XK + pr);
            }
            if (tid < OZ_XK / 2) cp_async16(sAl + (b ^ 1) * OZ_XK + tid * 2, alpha + (ss + 1) * OZ_XK + tid * 2);
            cp_async_commit();
        }
        const double* x = sX + b * dx * OZ_XK + kg * 16;
        if constexpr (composite_kernel(KID)) {
            // one candidate at a time (the component loop needs a second register tile): per component the distance loop
            // and covariance of the bare kernel, the component values added (multiplied) in order
            const int j0 = ss * OZ_XK + kg * 16;
            const int ks = ss * 4 + (kg >> 1), half = kg & 1;
            const double* al = sAl + b * OZ_XK + kg * 16;
#pragma unroll
            for (int a = 0; a < 2; a++) {
                double kv[16];
                for (int q = 0; q < sum.n; q++) {
                    double r2[16];
#pragma unroll
                    for (int i = 0; i < 16; i++) r2[i] = 0.0;
                    const int r0 = embedded_composite(KID) ? srow.off[q] : q * d, r1 = embedded_composite(KID) ? r0 + srow.rows[q] : (q + 1) * d;
                    for (int dim = r0; dim < r1; dim++) {
                        const double xa = sC[dim * OZ_NT + cl + 32 * a];
                        const double2* xr = reinterpret_cast<const double2*>(x + dim * OZ_XK);
#pragma unroll
                        for (int i = 0; i < 8; i++) {
                            const double2 xv = xr[i];
                            double df = xv.x - xa;
                            r2[2 * i] = fma(df, df, r2[2 * i]);
                            df = xv.y - xa;
                            r2[2 * i + 1] = fma(df, df, r2[2 * i + 1]);
                        }
                    }
#pragma unroll
                    for (int g = 0; g < 16; g += XW) {
                        double rr[XW], kk[XW];
#pragma unroll
                        for (int i = 0; i < XW; i++) rr[i] = r2[g + i];
                        sum_term_v<XW>(sum, q, rr, kk);
#pragma unroll
                        for (int i = 0; i < XW; i++) kv[g + i] = (q == 0) ? kk[i] : combine<KID>(kv[g + i], kk[i]);
                    }
                }
                uint32_t out[S][4];
#pragma unroll
                for (int p = 0; p < S; p++) out[p][0] = out[p][1] = out[p][2] = out[p][3] = 0u;
#pragma unroll
                for (int g = 0; g < 16; g++) {
                    const double k = (cvalid[a] && j0 + g < N) ? kv[g] : 0.0;
                    macc[a] = fma(k, al[g], macc[a]);
                    unsigned long long z = oz_digits<S>(k, bscale);
#pragma unroll
                    for (int p = 0; p < S; p++) out[p][g >> 2] = oz_put(out[p][g >> 2], z, S - 1 - p, g & 3);
                }
                const int c = cl + 32 * a;
                uint8_t* dst = B + ((size_t)ct * nks + ks) * S * OZ_B_SLICE + (c >> 3) * 256 + half * 128 + (c & 7) * 16;
#pragma unroll
                for (int p = 0; p < S; p++) *reinterpret_cast<uint4*>(dst + (size_t)p * OZ_B_SLICE) = make_uint4(out[p][0], out[p][1], out[p][2], out[p][3]);
            }
            continue;
        }
        double r2[2][16];
#pragma unroll
        for (int i = 0; i < 16; i++) r2[0][i] = r2[1][i] = 0.0;
        for (int dim = 0; dim < d; dim++) {
            const double xa = sC[dim * OZ_NT + cl];
            const double xb = sC[dim * OZ_NT + cl + 32];
            const double2* xr = reinterpret_cast<const double2*>(x + dim * OZ_XK);
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const double2 xv = xr[i];
                double df = xv.x - xa;
                r2[0][2 * i] = fma(df, df, r2[0][2 * i]);
                df = xv.y - xa;
                r2[0][2 * i + 1] = fma(df, df, r2[0][2 * i + 1]);
                df = xv.x - xb;
                r2[1][2 * i] = fma(df, df, r2[1][2 * i]);
                df = xv.y - xb;
                r2[1][2 * i + 1] = fma(df, df, r2[1][2 * i + 1]);
            }
        }
        const int j0 = ss * OZ_XK + kg * 16;
        const int ks = ss * 4 + (kg >> 1), half = kg & 1;
        const double* al = sAl + b * OZ_XK + kg * 16;
#pragma unroll
        for (int a = 0; a < 2; a++) {
            uint32_t out[S][4];
#pragma unroll
            for (int p = 0; p < S; p++) out[p][0] = out[p][1] = out[p][2] = out[p][3] = 0u;
#pragma unroll
            for (int g = 0; g < 16; g += XW) {
                double rr[XW], kk[XW];
#pragma unroll
                for (int i = 0; i < XW; i++) rr[i] = r2[a][g + i];
                cov_from_r2_v<KID, XW>(rr, var, rq_alpha, kk);
#pragma unroll
                for (int i = 0; i < XW; i++) {
                    const double k = (cvalid[a] && j0 + g + i < N) ? kk[i] : 0.0;
                    macc[a] = fma(k, al[g + i], macc[a]);
                    unsigned long long z = oz_digits<S>(k, bscale);
#pragma unroll
                    for (int p = 0; p < S; p++) out[p][(g + i) >> 2] = oz_put(out[p][(g + i) >> 2], z, S - 1 - p, (g + i) & 3);
                }
            }
            const int c = cl + 32 * a;
            uint8_t* dst = B + ((size_t)ct * nks + ks) * S * OZ_B_SLICE + (c >> 3) * 256 + half * 128 + (c & 7) * 16;
#pragma unroll
            for (int p = 0; p < S; p++) *reinterpret_cast<uint4*>(dst + (size_t)p * OZ_B_SLICE) = make_uint4(out[p][0], out[p][1], out[p][2], out[p][3]);
        }
    }
    sR[kg * OZ_NT + cl] = macc[0];
    sR[kg * OZ_NT + cl + 32] = macc[1];
    __syncthreads();
    if (tid < OZ_NT) {
        const double* q = sR + tid;
        mean[ct * OZ_NT + tid] = (((q[0] + q[OZ_NT]) + (q[2 * OZ_NT] + q[3 * OZ_NT])) +
                                  ((q[4 * OZ_NT] + q[5 * OZ_NT]) + (q[6 * OZ_NT] + q[7 * OZ_NT]))) + c0;
    }
}

// ---- the product kernel ---------------------------------------------------------------------------------------------
template <int S, int MODE>
__global__ void __launch_bounds__(OZ_THREADS, 1) ozaki_kernel(OzParams P) {
    using Cfg = OzCfg<S>;
    constexpr int KPS = (MODE == OZ_TRMM) ? Cfg::KPS_TRMM : 1;                           // k-steps per ring stage
    constexpr int STAGES = (MODE == OZ_TRMM) ? Cfg::STAGES_TRMM : Cfg::STAGES;
    constexpr int STAGE_BYTES = KPS * Cfg::STAGE_BYTES;
    constexpr int RING_BYTES = STAGES * STAGE_BYTES;
    extern __shared__ __align__(1024) uint8_t oz_smem_raw[];
    uint8_t* ring = oz_smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(oz_smem_raw + RING_BYTES);
    uint64_t* full = bars;                  // [STAGES] producer -> issuer (tx bytes)
    uint64_t* empty = bars + STAGES;        // [STAGES] issuer (tcgen05.commit) -> producer
    uint64_t* tmem_full = bars + 2 * STAGES;   // issuer -> epilogue
    uint64_t* tmem_empty = tmem_full + 1;      // epilogue (8 warps) -> issuer
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 1);
    double* red = reinterpret_cast<double*>(oz_smem_raw + RING_BYTES + 1024);  // [4][64]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; i++) {
            oz_mbar_init(&full[i], 1);
            oz_mbar_init(&empty[i], 1);
        }
        oz_mbar_init(tmem_full, 1);
        oz_mbar_init(tmem_empty, 8);
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

    if (warp == 0) {
        // ================= producer =================
        if (lane == 0) {
            int st = 0;
            uint32_t ph = 0;
            const uint64_t keep = oz_policy_evict_last();
            OzItems<MODE> items(P);
            int I, ks0, n;
            long long ct;
            while (items.next(I, ct, ks0, n)) {
                const uint8_t* a = P.A + ((size_t)I * nks + ks0) * S * OZ_A_SLICE;
                // OZ_TRMM: digit tiles of candidate tile ct; OZ_LAUUM: rows 64 (ct & 1) .. + 63 of row block ct >> 1
                // (OZ_GEMM: the same with another digit buffer)
                const uint8_t* b = MODE == OZ_TRMM ? P.B + ((size_t)ct * nks + ks0) * S * OZ_B_SLICE
                                                   : P.B + ((size_t)(ct >> 1) * nks + ks0) * S * OZ_A_SLICE + (ct & 1) * OZ_B_SLICE;
                for (int ks = 0; ks < n; ks += KPS) {
                    oz_mbar_wait(&empty[st], ph ^ 1);
                    uint8_t* dst = ring + (size_t)st * STAGE_BYTES;
                    oz_mbar_expect_tx(&full[st], STAGE_BYTES);
                    if (MODE == OZ_TRMM) {
                        // stage = [A of KPS k-steps][B of KPS k-steps]
                        oz_bulk_g2s_hint(dst, a + (size_t)ks * S * OZ_A_SLICE, KPS * S * OZ_A_SLICE, &full[st], keep);
                        oz_bulk_g2s(dst + KPS * S * OZ_A_SLICE, b + (size_t)ks * S * OZ_B_SLICE, KPS * S * OZ_B_SLICE, &full[st]);
                    } else {
                        oz_bulk_g2s(dst, a + (size_t)ks * S * OZ_A_SLICE, S * OZ_A_SLICE, &full[st]);
#pragma unroll
                        for (int q = 0; q < S; q++)
                            oz_bulk_g2s(dst + S * OZ_A_SLICE + q * OZ_B_SLICE, b + ((size_t)ks * S + q) * OZ_A_SLICE, OZ_B_SLICE, &full[st]);
                    }
                    if (++st == STAGES) {
                        st = 0;
                        ph ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            int st = 0;
            uint32_t ph = 0, acc_ph = 0;
            const uint32_t ring_addr = oz_smem(ring);
            OzItems<MODE> items(P);
            int I, ks0, n;
            long long ct;
            while (items.next(I, ct, ks0, n)) {
                oz_mbar_wait(tmem_empty, acc_ph ^ 1);  // epilogue has drained the accumulators of the previous item
                oz_fence_after();
                for (int ks = 0; ks < n; ks += KPS) {
                    oz_mbar_wait(&full[st], ph);
                    oz_fence_after();
#pragma unroll
                    for (int kk = 0; kk < KPS; kk++) {
                        const uint32_t sa = ring_addr + (uint32_t)st * STAGE_BYTES + kk * S * OZ_A_SLICE;
                        const uint32_t sb = ring_addr + (uint32_t)st * STAGE_BYTES + KPS * S * OZ_A_SLICE + kk * S * OZ_B_SLICE;
#pragma unroll
                        for (int p = 0; p < S; p++) {
                            // digit p of A against digits 0..S-1-p of B (stacked along N), level t = p+q -> columns 64 t
                            const uint64_t ad = oz_desc(sa + p * OZ_A_SLICE);
                            const int rem = S - p;
                            const int nch = (rem + 3) / 4;
                            const int take = (rem + nch - 1) / nch;
#pragma unroll
                            for (int q0 = 0; q0 < rem; q0 += take) {
                                const int nq = (rem - q0 < take) ? rem - q0 : take;
                                oz_mma(tbase + (uint32_t)((p + q0) * OZ_NT), ad, oz_desc(sb + q0 * OZ_B_SLICE), oz_idesc(nq * OZ_NT),
                                       (ks + kk > 0 || p > 0) ? 1u : 0u);
                            }
                        }
                    }
                    oz_commit(&empty[st]);  // frees the stage once these MMAs have read it
                    if (++st == STAGES) {
                        st = 0;
                        ph ^= 1;
                    }
                }
                oz_commit(tmem_full);  // accumulators of this item are complete
                acc_ph ^= 1;
            }
        }
    } else {
        // ================= epilogue (warps 2..9: TMEM lane group warp & 3, column half (warp - 2) >> 2) =================
        const int lg = warp & 3;
        const int hsel = (warp - 2) >> 2;
        const int et = threadIdx.x - 64;  // 0..255
        uint32_t acc_ph = 0;
        constexpr int H = S / 2;  // levels folded into the low word
        const double hi_mul = ldexp(1.0, 8 * H);
        OzItems<MODE> items(P);
        int I, ks0, n;
        long long ct;
        while (items.next(I, ct, ks0, n)) {
            const int row = I * 128 + lg * 32 + lane;
            const double rs = P.rowscale[row] * P.gscale * (MODE == OZ_GEMM ? P.sign : 1.0);
            oz_mbar_wait(tmem_full, acc_ph);
            oz_fence_after();
            acc_ph ^= 1;
            double tot[4];  // OZ_TRMM: this lane's share of the column sums: candidate hsel*32 + cc*8 + idx(lane)
#pragma unroll
            for (int cc = 0; cc < 4; cc++) {
                uint32_t r[S][8];
#pragma unroll
                for (int t = 0; t < S; t++)
                    oz_tmem_ld8(tbase + ((uint32_t)(lg * 32) << 16) + (uint32_t)(t * OZ_NT + hsel * 32 + cc * 8), r[t]);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (cc == 3) {
                    // all TMEM reads of this item are done: hand the accumulators back to the issuer
                    oz_fence_before();
                    __syncwarp();
                    if (lane == 0) oz_mbar_arrive(tmem_empty);
                }
                double v[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    long long whi = 0, wlo = 0;
#pragma unroll
                    for (int t = 0; t < S - H; t++) whi += (long long)(int32_t)r[t][i] << (8 * (S - H - 1 - t));
#pragma unroll
                    for (int t = S - H; t < S; t++) wlo += (long long)(int32_t)r[t][i] << (8 * (S - 1 - t));
                    double w = fma((double)whi, hi_mul, (double)wlo);
                    v[i] = w * rs;
                }
                if (MODE == OZ_LAUUM || MODE == OZ_GEMM) {
                    // out[row][col0 .. col0 + 7]: the exact integer sum, scaled by the two power-of-two row scales
                    const int col0 = (int)ct * OZ_NT + hsel * 32 + cc * 8;
                    const double* cs = MODE == OZ_GEMM ? P.colscale : P.rowscale;
                    const double4 c0 = *reinterpret_cast<const double4*>(cs + col0);
                    const double4 c1 = *reinterpret_cast<const double4*>(cs + col0 + 4);
                    const double o[8] = {v[0] * c0.x, v[1] * c0.y, v[2] * c0.z, v[3] * c0.w, v[4] * c1.x, v[5] * c1.y, v[6] * c1.z, v[7] * c1.w};
                    double2* dst = reinterpret_cast<double2*>(P.out + (size_t)row * P.Np + col0);
                    if (MODE == OZ_GEMM && P.accumulate) {
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const double2 c = dst[i];
                            dst[i] = make_double2(c.x + o[2 * i], c.y + o[2 * i + 1]);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; i++) dst[i] = make_double2(o[2 * i], o[2 * i + 1]);
                    }
                    if (MODE == OZ_GEMM && P.out_t != nullptr) {
                        // lanes hold consecutive rows: 256 contiguous bytes per column
#pragma unroll
                        for (int i = 0; i < 8; i++) P.out_t[(size_t)(col0 + i) * P.Np + row] = o[i];
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 8; i++) v[i] = v[i] * v[i];
                    // transposed butterfly: 8 values x 32 lanes -> four lanes hold each column sum; the same fixed tree
                    // over the 32 rows for every candidate (position-independent rounding)
#pragma unroll
                    for (int o = 16, nn = 4; o >= 4; o >>= 1, nn >>= 1) {
                        const bool up = (lane & o) != 0;
#pragma unroll
                        for (int i = 0; i < nn; i++) {
                            double send = up ? v[i] : v[i + nn];
                            double keep = up ? v[i + nn] : v[i];
                            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                        }
                    }
                    double t2 = v[0] + __shfl_xor_sync(0xffffffffu, v[0], 2);
                    tot[cc] = t2 + __shfl_xor_sync(0xffffffffu, t2, 1);
                }
            }
            if (MODE == OZ_TRMM) {
                // candidate index held by this lane within an 8-chunk: bit4 -> 4, bit3 -> 2, bit2 -> 1
                const int idx = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                asm volatile("bar.sync 1, 256;" ::: "memory");  // previous item's cross-warp reduction has been consumed
                if ((lane & 3) == 0) {
#pragma unroll
                    for (int cc = 0; cc < 4; cc++) red[lg * OZ_NT + hsel * 32 + cc * 8 + idx] = tot[cc];
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
                if (et < OZ_NT) {
                    double s = (red[et] + red[OZ_NT + et]) + (red[2 * OZ_NT + et] + red[3 * OZ_NT + et]);
                    P.part[(size_t)I * P.ldp + (size_t)ct * OZ_NT + et] = s;
                }
            }
        }
    }
    oz_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(OZ_TMEM_COLS));
}

}  // namespace gpso
