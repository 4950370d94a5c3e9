// gpso_b200 C ABI (see include/gpso_b200.h): handle, device memory, and the launch sequences of the three pipelines
//   fit     : scale -> Gram -> blocked Cholesky -> L^-1 (recursive doubling) -> K_y^-1 -> alpha -> LML + gradient
//   predict : per candidate window: cross-covariance (+mean) -> triangular product + column sum of squares -> finalise
//   explore : leaf generation on the device -> predict -> UCB arg-max
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -shared -Xcompiler -fPIC
#include "../../include/gpso_b200.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <functional>
#include <string>
#include <map>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "gemm_core.cuh"
#include "kern_cov.cuh"
#include "kern_dense.cuh"
#include "kern_leaves.cuh"
#include "kern_ozaki.cuh"
#include "kern_predict.cuh"
#include "kern_joint.cuh"
#include "kern_screen.cuh"
#include "kern_probe.cuh"
#include "kern_mean.cuh"

using namespace gpso;

static thread_local std::string g_last_error;

static int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define CU_TRY(call)                                                                                          \
    do {                                                                                                      \
        cudaError_t e__ = (call);                                                                             \
        if (e__ != cudaSuccess) {                                                                             \
            char buf__[512];                                                                                  \
            snprintf(buf__, sizeof buf__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return fail(e__ == cudaErrorMemoryAllocation ? GPSO_E_NOMEM : GPSO_E_CUDA, buf__);                \
        }                                                                                                     \
    } while (0)

#define GP_TRY(call)             \
    do {                         \
        int rc__ = (call);       \
        if (rc__ != 0) return rc__; \
    } while (0)

namespace {

constexpr int MAX_LS = LEAF_MAXD;  // maximum input dimension supported
constexpr double NOISE_FLOOR = 1.0e-6;
constexpr long long WINDOW_BYTES = 2LL << 30;  // rolling cross-covariance window budget (2 GiB)
constexpr int OZ_XCOV_SMEM_MAX = 172 * 1024;   // crosscov_slices_kernel dynamic shared memory at d = 64 (320 d + 768 doubles)
constexpr int OZ_MIN_NP = 256;                 // below this the int8 path is not worth its fixed costs (automatic mode); config C5
                                               // (N = 21..500, 265 720 candidates per call): 9.6 s wall with 512, 7.0 s with 256, 7.0 s with 128
constexpr int OZ_MAX_NP = 8192;                // int32 accumulators stay exact: pairs per level (<= S = 8) * 2^14 * Np <= 2^30 < 2^31
                                               // (16384 would reach exactly 2^31); larger problems stay on the FP64 DMMA engines
constexpr int OZ_KINV_S = 7;                   // digits per operand of the int8 K_y^-1 = L^-T L^-1 product (54-bit fixed point per row)
constexpr int OZ_KINV_MIN_NP = 512;            // automatic mode; measured down to N = 512 (LML+grad 0.553 -> 0.498 ms there, 1.13 -> 1.01 ms at 1024)
constexpr int OZ_INV_S = 8;                    // digits per operand of the int8 inverse-factor products (62-bit fixed point per row)
// Levels s < cap tiles of the inverse recursion stay in the persistent FP64 kernel, queued as soon as their inputs are (they
// run on the SMs the chain-bound factorisation leaves idle); the int8 engine takes the levels above.  Measured per LML+grad
// evaluation: N = 300 0.40 -> 0.31 ms, 600 0.54 -> 0.47, 1024 0.73 -> 0.68 (cap 8 = everything in the kernel up to 1024 rows);
// at 4096 rows the FP64 merges start to get in the chain's way (cap 4 / 8 / 16: 3.23 / 3.26 / 3.41 ms).
static inline int oz_inv_dmma_cap(int n_tiles) { return n_tiles >= 24 ? 4 : 8; }
constexpr int OZ_HYB_S = 7;                    // digits per operand of the hybrid factorisation's panel and Schur products: 54-bit fixed point per
                                               // row, the rounding of an fp64 product of the same operands (the K_y^-1 product uses the same)
constexpr int OZ_INV_MIN_NP = 512;             // automatic mode; measured down to N = 512 (0.498 -> 0.474 ms there, 2.05 -> 1.75 ms at 2048)
constexpr double OZ_TARGET = 0.02;             // accepted (estimated error) / (parity tolerance 1e-8 * variance)
// screen-and-refine arg-max (kern_screen.cuh)
constexpr int SCREEN_MIN_NP = 512;             // below this the full-precision pass is cheap: no screening (config C2, N = 512, 1e5
                                               // candidates: 1.92e8 -> 2.55e8 candidates/s with the screen, 323 survivors)
constexpr long long SCREEN_MIN_M = 65536;      // fewer candidates than this: no screening
constexpr double SCREEN_SAFETY = 4.0;          // error bound E = SAFETY * (model estimate); the refine pass must observe <= E / 4
constexpr unsigned SCREEN_LIST_CAP = 1u << 20; // survivor list capacity; more survivors than this or than M / 16 -> full pass
constexpr int SCREEN_S_MIN = 2, SCREEN_S_MAX = 4;
constexpr int SCREEN_MODE_BOUND = 5;           // gpso_set_screen_mode: mean-bound level first, then the automatic digit screen
constexpr int SCREEN_MODE_FULL2 = 6;           // gpso_set_screen_mode: forced 2-digit full product

// ---- device memory: blocks are recycled through a per-device pool ------------------------------------------------------------
// The optimiser opens a new handle for every fit (the reference builds a new GPflow model per update); a handle owns ~40
// buffers, and cudaMalloc / cudaFree cost 0.1-1 ms each and synchronise the device.  Released blocks therefore go to a free
// list (per device, rounded sizes: powers of two up to 1 MB, multiples of 2 MB above) and are handed out again to requests of
// nearly the same size.  Nothing is in flight on a block when it enters the list: gpso_destroy synchronises the device before
// the buffers go, and a buffer that grows does the same before it lets go of its old block.
namespace {
constexpr size_t POOL_MAX_CACHED = 24ULL << 30;  // bytes kept per device; beyond this released blocks are freed
constexpr int POOL_MAX_DEV = 64;
struct DevPool {
    std::mutex mu;
    std::multimap<size_t, void*> blocks[POOL_MAX_DEV];
    size_t cached[POOL_MAX_DEV] = {0};
    static size_t rounded(size_t bytes) {
        if (bytes <= (1u << 20)) {
            size_t r = 512;
            while (r < bytes) r <<= 1;
            return r;
        }
        const size_t g = 2u << 20;
        return (bytes + g - 1) / g * g;
    }
    void* take(int dev, size_t want, size_t* got) {  // want is a rounded size; blocks up to 25 % larger qualify
        if (dev < 0 || dev >= POOL_MAX_DEV) return nullptr;
        std::lock_guard<std::mutex> lock(mu);
        auto it = blocks[dev].lower_bound(want);
        if (it == blocks[dev].end() || it->first > want + want / 4) return nullptr;
        void* p = it->second;
        *got = it->first;
        cached[dev] -= it->first;
        blocks[dev].erase(it);
        return p;
    }
    bool give(int dev, void* p, size_t bytes) {
        if (dev < 0 || dev >= POOL_MAX_DEV) return false;
        std::lock_guard<std::mutex> lock(mu);
        if (cached[dev] + bytes > POOL_MAX_CACHED) return false;
        blocks[dev].emplace(bytes, p);
        cached[dev] += bytes;
        return true;
    }
    void flush(int dev) {  // out of memory: give everything back to the driver
        if (dev < 0 || dev >= POOL_MAX_DEV) return;
        std::lock_guard<std::mutex> lock(mu);
        for (auto& kv : blocks[dev]) cudaFree(kv.second);
        blocks[dev].clear();
        cached[dev] = 0;
    }
};
DevPool g_pool;
}  // namespace

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;    // bytes the owner may use
    size_t block = 0;  // size of the pool block behind p
    int dev = -1;
    int ensure(size_t bytes, bool zero = false) {
        if (bytes <= cap) return 0;
        if (p) {
            cudaDeviceSynchronize();  // kernels of this handle may still read the old block
            release();
        }
        cudaGetDevice(&dev);
        const size_t want = DevPool::rounded(bytes);
        p = g_pool.take(dev, want, &block);
        if (!p) {
            cudaError_t e = cudaMalloc(&p, want);
            if (e != cudaSuccess) {
                cudaGetLastError();
                g_pool.flush(dev);
                e = cudaMalloc(&p, want);
            }
            if (e != cudaSuccess) {
                p = nullptr;
                char b[256];
                snprintf(b, sizeof b, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
                return fail(GPSO_E_NOMEM, b);
            }
            block = want;
        }
        cap = bytes;
        if (zero) {
            // the handle's streams are non-blocking: a legacy-stream memset is not ordered with them, so finish it here
            cudaMemset(p, 0, bytes);
            cudaDeviceSynchronize();
        }
        return 0;
    }
    void release() {
        if (p && !g_pool.give(dev, p, block)) cudaFree(p);
        p = nullptr;
        cap = 0;
        block = 0;
    }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }  // every buffer of a handle goes with it (gpso_destroy synchronises the device first)
    template <class T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};

double softplus(double u) { return u > 0 ? u + log1p(exp(-u)) : log1p(exp(u)); }
double sigmoid(double u) { return 1.0 / (1.0 + exp(-u)); }

}  // namespace

struct gpso_handle {
    int device = 0, kernel_id = KERNEL_MATERN52, ard = 0, mean_id = GPSO_MEAN_CONSTANT;
    int N = 0, d = 0, Np = 0, nb = 0;
    int nsm = 0;
    size_t l2_persist_max = 0, l2_window_max = 0;  // device limits for the persisting-L2 access window of the A digits
    int l2_window = 1;                              // gpso_set_l2_window
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev_copy[2] = {nullptr, nullptr}, ev_used[2] = {nullptr, nullptr}, ev_t0 = nullptr, ev_t1 = nullptr;
    bool used_pending[2] = {false, false};
    // data + fitted state
    DevBuf X, y, Xs, ls, alpha;
    DevBuf meanA;  // GPSO_MEAN_LINEAR: A (d doubles)
    DevBuf K, Linv, LinvT, T, Kinv;
    DevBuf resid, a, logdet, scalars, gpart, gout, info, counter;
    DevBuf chol_state;      // state [next, err, counters] of the fit's persistent factorisation kernel (task lists: factor_plans)
    // predict workspaces
    DevBuf KsT, part, blockbest, running, cand[2], leaves, omean, ovar, topk;
    // joint posterior (kern_joint.cuh): scaled candidates, cross-covariance, mean, V^T, Sigma; for the samples the factor's
    // scratch (inverse diagonal blocks and their transposes, log-determinant, pivot status, scheduler state) and the padded
    // normals; host staging of candidates, normals and outputs.  Separate from the fit's buffers, which a joint call never touches.
    DevBuf jXcs, jKsT, jmean, jVT, jSigma, jLinv, jLinvT, jlogdet, jinfo, jstate, jcounter, jZ, jcand, jzin, jout;
    int jLinv_mp = 0;       // row pitch jLinv was cleared for (its zero sub-blocks above the diagonal are never written)
    // int8 tensor-core (tcgen05) variance product: digit tiles of L^-1 and of the cross-covariance window
    DevBuf ozA, ozBb[2], wmeanb[2], rowscale, rowmax, rowl2;
    // int8 tensor-core K_y^-1 = L^-T L^-1 (fit path): digit tiles of L^-T, its row scales, the tile -> CTA table
    DevBuf ozT, colscale, colmax, lauum_items, kinv_part;
    int lauum_items_nb = 0, lauum_rounds = 0;
    int kinv_mode = 0;      // 0 = automatic (int8 from OZ_KINV_MIN_NP), 1 = FP64 DMMA tiles, 2 = int8 tcgen05
    // int8 tensor-core inverse factor (recursive doubling, two products per level): digit tiles and row scales of the four
    // operands (L, L^-T block diagonal, L^-1 block diagonal, X^T) and the per-level tile -> CTA tables
    DevBuf ozL, ozLT, ozLI, ozXT, rsL, rsLT, rsLI, rsXT;
    struct InvLevel { int s; size_t xt_off; int xt_rounds; size_t y_off; int y_rounds; };
    int inverse_mode = 0;   // 0 = automatic (int8 from OZ_INV_MIN_NP), 1 = FP64 DMMA tile tasks, 2 = int8 tcgen05
    // persistent and hybrid factorisation (hybrid_node): task lists / item tables per sub-matrix size, built on first use
    struct FactorPlan { DevBuf tasks; int ntasks = 0, ncounters = 0; };
    struct InvPlan { DevBuf items; std::vector<InvLevel> levels; };
    struct ItemList { DevBuf items; int rounds = 0; };
    std::map<int, FactorPlan> factor_plans;    // key 2048 n + levels of the inverse done by the kernel (cap)
    std::map<int, InvPlan> inv_plans;          // key n
    std::map<long long, ItemList> hyb_items;   // key (kind, split, n)
    // gpso_set_factor_mode: 0 = one launch per step (reference schedule), 1 = persistent kernel, hybrid above HYB_LEAF_TILES
    // tiles (automatic), 2 = one persistent kernel for the whole matrix, 3 = hybrid with leaves of 2 tiles (tests); the hybrid
    // needs the int8 inverse engine in force, without it modes 1 and 3 are mode 2
    int factor_mode = 1;
    int hybrid_nodes = 0;   // inner nodes of the last factorisation (0 = one persistent kernel)
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_probe = nullptr;  // early verdict of a screening rung (screen_pass)
    cudaEvent_t ev_start = nullptr, ev_xcov[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    int overlap = 1;
    int predict_mode = 0;   // 0 = automatic, 1 = FP64 DMMA product, 2 = int8 tcgen05 product
    int oz_force_slices = 0;
    int oz_S = 0;           // digits per operand chosen at the last factorisation (0: DMMA path in force)
    double oz_est = 0.0;    // error estimate / tolerance for the chosen S
    long long window_override = 0;
    // screen-and-refine arg-max: fp32 copies of the scaled inputs / alpha, low-digit tiles of L^-1, per-candidate screened UCB,
    // {max key, survivor count, max |refined - screened|}, survivor index list and gathered survivor coordinates
    DevBuf Xs32, alpha32, ozAs, part32, scr_ucb, scr_state, surv_list, surv_X;
    int screen_mode = 1;        // 0 off, 1 automatic (digits adapt to the survivor fraction), 2..4 forced digits
    int screen_S_cur = 0;       // rung of SCREEN_LADDER the automatic mode starts from
    int screen_built_S = 0;     // digits of the tiles in ozAs (0: stale)
    bool screen_ready = false;  // fp32 copies and norms valid for the factor in force
    long long scr_rows = 0;     // scr_ucb[0, scr_rows) holds the values the last screening level of the last fused call wrote
    double alpha_l2 = 0.0, rho_max = 0.0, rho_l2sq = 0.0;
    double linv_frob2 = 0.0, linv_rowl2_max = 0.0;  // |L^-1|_F^2 (= tr K_y^-1) and the largest row norm of L^-1
    // last call: [0] path (0 unscreened, 1 screened, 2 fallback: too many survivors, 3 fallback: check failed), [1] digits,
    // [2] survivors, [3] E, [4] max |refined - screened| over the survivors, [5] best screened UCB, [6] screen windows,
    // [7] screening product ms, [8] refine windows, [9] E_var, [10] E_mean
    double scr_info[12] = {0};
    size_t scr_prod_marks = 0;
    // host copies of the hyper-parameters in force
    double ls_host[MAX_LS] = {0}, variance = 1.0, noise = 1.0, c0 = 0.0;  // c0: the mean constant, or b of the linear mean
    double A_host[MAX_LS] = {0};  // GPSO_MEAN_LINEAR: A, also in meanA on the device
    double rq_alpha = 1.0;  // RationalQuadratic shape (KERNEL_RQ only; the other kernels never read it)
    // KERNEL_SUM (gpso_create_sum): the component table the covariance kernels take (families, variances, alphas; n = 0 for the
    // other kernels) and the ARD flag of each component.  `variance` then holds the prior variance var_tot = sum_c var_c, the fp64
    // sum in component order, and ls_host the lengthscales of every component expanded to d entries ([C][d], as on the device).
    SumTable sum = {};
    SumRows srow = {};  // the components' rows (sum / product with periodic components)
    int sum_ard[MAX_SUM] = {0};
    // KERNEL_PRODUCT (gpso_create_product) shares that table and ARD flags.  `variance` holds var_prod = prod_c var_c (fp64,
    // factor order), the table's variances are {var_prod, 1, 1, 1}, and prod_var keeps the factor variances themselves.
    double prod_var[MAX_SUM] = {0};
    // GPSO_KERNEL_PERIODIC (gpso_create_periodic): kernel_id is the base family (SE or RQ), whose covariance kernels run at unit
    // lengthscale on the 2d embedded rows of kern_cov.cuh's periodic_embed_kernel.  ls_host keeps the base lengthscale(s) as
    // packed and per_p the period(s); the device buffer ls holds the unit lengthscale, plp the embedding's [l(d), p(d)] (from
    // plp_host), pX the embedded candidates of a window or of a joint call (row-major [M][2d]).
    bool periodic = false;
    int per_ard = 0;
    double per_p[MAX_LS] = {0}, plp_host[2 * MAX_LS] = {0}, unit_ls = 1.0;
    // A sum / product with periodic components (gpso_create_combination): sum_per[c] marks component c as periodic (its fam is
    // the base's) with the period ARD flag sum_per_ard[c] and its period(s) comp_p[c]; srow's off / rows / width give each
    // component's rows (ensure_shape).  ls then holds the unit lengthscale on a periodic component's rows, rmap its (l, p).
    int sum_per[MAX_SUM] = {0}, sum_per_ard[MAX_SUM] = {0};
    double comp_p[MAX_SUM][MAX_LS] = {{0}};
    DevBuf plp, pX;
    // gpso_set_active_dims: leaf c (component c; a periodic leaf's base) reads the map_n[c] input columns map_cols[map_off[c] ..];
    // nmap = 0 without a map.  A handle with a map always runs the row layout of a sum / product with periodic components: a bare
    // kernel becomes a one-component sum (bare_kid keeps its kernel id, restored when the map is cleared).  ls_host then holds
    // component c's lengthscales from ls_off(c), rmap describes the rows (stage_rows_kernel), Xg[N][raw.width] holds the
    // periodic leaves' raw active columns for the gradient.
    int nmap = 0, map_n[MAX_SUM] = {0}, map_off[MAX_SUM + 1] = {0};
    std::vector<int> map_cols;
    int bare_kid = -1, bare_ard = 0, bare_per_ard = 0;
    // GPSO_KERNEL_LINEAR: a Linear component has the family KERNEL_LINEAR (bit c of lin_mask); ls_host holds its variance(s) where a
    // stationary component's lengthscales go, and its rows are its (active) columns over 1 / sqrt(variance) (common.cuh).  A bare
    // Linear kernel is a one-component sum from the start (bare_lin), with or without a map.
    int lin_mask = 0;
    bool bare_lin = false;
    RowMap rmap = {};
    RawCols raw = {};
    DevBuf Xg;
    bool have_data = false, factorized = false;
    double factor_nlml = 0.0;
    double* host_rec = nullptr;  // pinned: results of an evaluation come back in one record without staging copies
    long long launches = 0;
    double last_ms[4] = {0, 0, 0, 0};
    // optional per-stage profiling: 4 events per window on the launch stream
    bool profile = false;
    std::vector<cudaEvent_t> prof_events;
    size_t prof_used = 0;
    // always on: one event pair around every variance-product launch (its summed duration is last_ms[2])
    std::vector<cudaEvent_t> prod_events;
    size_t prod_used = 0;
    long long last_windows = 0;
    // optional timeline of the window pipeline (gpso_set_profile(h, 2)): events on the streams the kernels run on, the
    // overlap stays in force; read back with gpso_debug_trace as (tag, window, ms since the first event) triples
    bool trace = false;
    std::vector<cudaEvent_t> trace_events;
    std::vector<int> trace_tags;
    size_t trace_used = 0;
    std::vector<double> trace_out;
    bool is_sum() const { return kernel_id == KERNEL_SUM; }
    bool is_product() const { return kernel_id == KERNEL_PRODUCT; }
    bool composite() const { return composite_kernel(kernel_id); }  // a sum or a product: the component table is in force
    // rows of the scaled inputs Xs per input dimension: C for a sum or a product, 2 for a periodic kernel
    bool emb() const { return composite() && (srow.pmask != 0 || nmap != 0 || lin_mask != 0); }
    bool has_lin() const { return lin_mask != 0; }
    bool comp_lin(int c) const { return lin_mask >> c & 1; }  // a sum / product with periodic components or a map
    bool embeds() const { return periodic || emb(); }           // the candidates are embedded before the covariance kernels
    // the covariance kernels' instantiation: a sum / product with periodic components has its own
    int cov_kid() const { return has_lin() ? KERNEL_SUM_LIN : emb() ? (is_product() ? KERNEL_PRODUCT_EMB : KERNEL_SUM_EMB) : kernel_id; }
    // rows of the scaled inputs Xs for input dimension dd: [C][d] for a sum or a product (2d for a periodic component), [2][d]
    // for a periodic kernel
    int rows_for(int dd) const {
        if (!composite()) return periodic ? 2 * dd : dd;
        int r = 0;
        for (int c = 0; c < sum.n; c++) r += sum_per[c] ? 2 * cdim(c, dd) : cdim(c, dd);
        return r;
    }
    int cdim(int c, int dd) const { return nmap ? map_n[c] : dd; }  // input columns component c reads
    int ls_off(int c) const { return nmap ? map_off[c] : c * d; }   // component c's lengthscales in ls_host
    int dx() const { return rows_for(d); }
    int cand_width() const { return emb() ? dx() : 2 * d; }  // columns of the embedded candidates (pX)
    int comp_np(int c) const { return sum_per[c] ? (sum_per_ard[c] ? cdim(c, d) : 1) : 0; }  // packed periods of component c
    int kd() const { return periodic ? 2 * d : d; }  // the input dimension the covariance kernels are launched with
    int n_ls() const { return composite() ? ls_off(sum.n) : (ard ? d : 1); }
    int kern_nls() const { return periodic ? 1 : n_ls(); }  // lengthscales the covariance kernels read from ls
    int n_per() const { return periodic ? (per_ard ? d : 1) : 0; }  // packed periods
    double comp_var(int c) const { return is_product() ? prod_var[c] : sum.var[c]; }  // component c's own variance
    int n_rq() const { return kernel_id == KERNEL_RQ ? 1 : 0; }  // alpha leads the packed vector (GPflow's sorted names)
    int comp_ls(int c) const { return sum_ard[c] ? cdim(c, d) : 1; }  // packed lengthscales of sum component c (Linear: variances)
    // [alpha], lengthscale(s), variance, [period(s)]; a Linear component: variance(s)
    int comp_params(int c) const { return (sum.fam[c] == KERNEL_RQ) + comp_ls(c) + (comp_lin(c) ? 0 : 1) + comp_np(c); }
    int n_kernel_params() const {
        if (!composite()) return n_rq() + n_ls() + 1 + n_per();
        int n = 0;
        for (int c = 0; c < sum.n; c++) n += comp_params(c);
        return n;
    }
    bool linear() const { return mean_id == GPSO_MEAN_LINEAR; }
    int n_mean() const { return mean_id == GPSO_MEAN_CONSTANT ? 1 : (linear() ? d + 1 : 0); }  // A (d entries) before b
    int n_params() const { return n_kernel_params() + 1 + n_mean(); }
};

// ---------------------------------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------------------------------
static int set_device(gpso_handle* h) {
    CU_TRY(cudaSetDevice(h->device));
    return 0;
}

static int check_launch(gpso_handle* h, const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        char b[256];
        snprintf(b, sizeof b, "launch of %s failed: %s", what, cudaGetErrorString(e));
        return fail(GPSO_E_CUDA, b);
    }
    h->launches++;
    return 0;
}

// Pivot status of a factorisation (LAPACK info: the 1-based row of the first non-positive pivot, < 0 when the tile scheduler
// gave up waiting) -> return code and message; `what` names the factorised matrix.
static int pivot_status(int info, const char* what) {
    if (info < 0) return fail(GPSO_E_CUDA, "Cholesky tile scheduler timed out waiting for a dependency");
    if (info > 0) {
        char b[128];
        snprintf(b, sizeof b, "%s is not positive definite (pivot %d)", what, info);
        return fail(info, b);
    }
    return 0;
}

// The set-aside is a device-wide setting and shrinks the L2 left to everything else (the factorisation kernels pass their
// tiles between SMs through L2: LML+grad at N = 4096 went from 3.8 to 4.6 ms with the set-aside left on), so it is only in
// force between a factorisation for scoring and the next fit evaluation.
static size_t g_l2_setaside[64] = {0};
static int l2_setaside(gpso_handle* h, size_t bytes) {
    const int dev = h->device & 63;
    if (g_l2_setaside[dev] == bytes) return 0;
    if (bytes == 0) CU_TRY(cudaCtxResetPersistingL2Cache());
    CU_TRY(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes));
    g_l2_setaside[dev] = bytes;
    return 0;
}

// The covariance families, in one list: AllKernels::with runs f with a kernel id as a compile-time constant (gpso_create accepts
// no other id), AllKernels::each runs it for every family and stops at the first error.
template <int... KIDS>
struct KernelIds {
    template <class F>
    static void with(int kid, F&& f) {
        (void)((kid == KIDS ? (f(std::integral_constant<int, KIDS>()), true) : false) || ...);
    }
    template <class F>
    static int each(F&& f) {
        int rc = 0;
        (void)(((rc = f(std::integral_constant<int, KIDS>())) == 0) && ...);
        return rc;
    }
};
static_assert(GPSO_KERNEL_SUM == KERNEL_SUM && GPSO_KERNEL_PRODUCT == KERNEL_PRODUCT && GPSO_MAX_SUM == MAX_SUM && GPSO_KERNEL_SE == KERNEL_SE &&
              GPSO_KERNEL_RQ == KERNEL_RQ,
              "sum and product kernel constants of the C ABI");
using AllKernels = KernelIds<KERNEL_MATERN12, KERNEL_MATERN32, KERNEL_MATERN52, KERNEL_SE, KERNEL_RQ>;
// The covariance kernels also have KERNEL_SUM and KERNEL_PRODUCT instantiations; the gradient of a sum runs the families' own
// kernel per component, a product's runs lml_grad_product_kernel.
using CovKernels = KernelIds<KERNEL_MATERN12, KERNEL_MATERN32, KERNEL_MATERN52, KERNEL_SE, KERNEL_RQ, KERNEL_SUM, KERNEL_PRODUCT,
                             KERNEL_SUM_EMB, KERNEL_PRODUCT_EMB>;

// gram_kernel, crosscov_kernel and joint_syrk_kernel also have the KERNEL_SUM_LIN instantiation (a sum with Linear terms); the
// other covariance kernels do not (such a handle never screens nor runs the int8 variance product)
using FullCovKernels = KernelIds<KERNEL_MATERN12, KERNEL_MATERN32, KERNEL_MATERN52, KERNEL_SE, KERNEL_RQ, KERNEL_SUM, KERNEL_PRODUCT,
                                 KERNEL_SUM_EMB, KERNEL_PRODUCT_EMB, KERNEL_SUM_LIN>;

static void launch_gram(gpso_handle* h, cudaStream_t st) {
    dim3 grid(h->Np / CT, h->Np / CT);
    FullCovKernels::with(h->cov_kid(), [&](auto kid) {
        gram_kernel<kid><<<grid, 256, 0, st>>>(h->Xs.as<double>(), h->N, h->kd(), h->Np, h->variance, h->noise, h->K.as<double>(),
                                               h->rq_alpha, h->sum, h->srow);
    });
}

static void launch_crosscov(gpso_handle* h, cudaStream_t st, const double* Xc, long long Mw, long long Mw_pad) {
    size_t sm = (size_t)(XG * h->dx() + 8 * XG) * sizeof(double);
    FullCovKernels::with(h->cov_kid(), [&](auto kid) {
        crosscov_kernel<kid><<<(unsigned)(Mw_pad / XG), 256, sm, st>>>(Xc, Mw, h->kd(), h->ls.as<double>(), h->kern_nls(), h->Xs.as<double>(),
                                                                      h->alpha.as<double>(), h->N, h->Np, h->variance, h->c0,
                                                                      h->KsT.as<double>(), h->wmeanb[0].as<double>(), h->rq_alpha,
                                                                      h->sum, h->srow);
    });
}

template <int S>
static int oz_configure() {
    CU_TRY(cudaFuncSetAttribute(ozaki_kernel<S, OZ_TRMM>, cudaFuncAttributeMaxDynamicSharedMemorySize, OzCfg<S>::SMEM_BYTES_TRMM));
    // full shared-memory carve-out for both kernels: the persistent product CTA (one per SM) must leave room for a
    // cross-covariance block of the next window on the same SM (they use different pipes and overlap)
    CU_TRY(cudaFuncSetAttribute(ozaki_kernel<S, OZ_TRMM>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return CovKernels::each([](auto kid) -> int {
        CU_TRY(cudaFuncSetAttribute(crosscov_slices_kernel<kid, S>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        CU_TRY(cudaFuncSetAttribute(crosscov_slices_kernel<kid, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_XCOV_SMEM_MAX));
        return 0;
    });
}

template <int S>
static int screen_configure() {
    CU_TRY(cudaFuncSetAttribute(ozaki_screen_kernel<S, SCR_NT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ScrCfg<S, SCR_NT, false>::SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(ozaki_screen_kernel<S, SCR_NT, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (S == 2) {
        CU_TRY(cudaFuncSetAttribute(ozaki_screen_kernel<2, SCR_NT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ScrCfg<2, SCR_NT, true>::SMEM_BYTES));
        CU_TRY(cudaFuncSetAttribute(ozaki_screen_kernel<2, SCR_NT, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    }
    return CovKernels::each([](auto kid) -> int {
        CU_TRY(cudaFuncSetAttribute(crosscov_screen_kernel<kid, S, SCR_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_XCOV_SMEM_MAX));
        CU_TRY(cudaFuncSetAttribute(crosscov_screen_kernel<kid, S, SCR_NT>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        return 0;
    });
}

static size_t screen_xcov_smem(int d) {
    return (size_t)(64 * d + 2 * d * OZ_XK + 2 * OZ_XK) * sizeof(float) + 8 * 64 * sizeof(double);
}

// S = 0: posterior mean only (bound pass)
template <int S>
static void launch_screen_crosscov(gpso_handle* h, cudaStream_t st, const double* Xc, long long Mw, long long ngroups, float bscale,
                                   uint8_t* B, double* wmean) {
    CovKernels::with(h->cov_kid(), [&](auto kid) {
        crosscov_screen_kernel<kid, S, SCR_NT><<<(unsigned)ngroups, 256, screen_xcov_smem(h->dx()), st>>>(
            Xc, Mw, h->kd(), h->ls.as<double>(), h->kern_nls(), h->Xs32.as<float>(), h->alpha32.as<float>(), h->N, h->Np, (float)h->variance,
            h->c0, bscale, h->Np / 32, B, wmean, (float)h->rq_alpha, h->sum, h->srow);
    });
}

template <int S, bool FULL = false>
static void launch_screen_product(gpso_handle* h, cudaStream_t st, long long nct, long long ldp, double gscale, const uint8_t* B) {
    ScrParams P;
    P.A = h->ozAs.as<uint8_t>();
    P.B = B;
    P.rowscale = h->rowscale.as<double>();
    P.part = h->part32.as<float>();
    P.gscale = gscale;
    P.nb = h->nb;
    P.nks = h->Np / 32;
    P.nct = (int)nct;
    P.ldp = ldp;
    const long long units = nct * ((h->nb + 1) / 2);
    const int grid = (int)std::min<long long>(h->nsm, units);
    ozaki_screen_kernel<S, SCR_NT, FULL><<<grid, OZ_THREADS, ScrCfg<S, SCR_NT, FULL>::SMEM_BYTES, st>>>(P);
}

template <int S>
static void launch_screen_slices(gpso_handle* h, cudaStream_t st) {
    dim3 grid(h->Np / 32, h->nb);
    linv_slices_kernel<S, false><<<grid, 256, 0, st>>>(h->Linv.as<double>(), h->rowscale.as<double>(), h->Np, h->Np / 32, h->ozAs.as<uint8_t>());
}

#define DISPATCH_SCREEN_S(S_, fn, ...)         \
    switch (S_) {                              \
        case 2: fn<2>(__VA_ARGS__); break;     \
        case 3: fn<3>(__VA_ARGS__); break;     \
        default: fn<4>(__VA_ARGS__); break;    \
    }

static size_t oz_xcov_smem(int d) { return (size_t)(OZ_NT * d + 2 * d * OZ_XK + 2 * OZ_XK + 8 * OZ_NT) * sizeof(double); }

template <int S>
static void launch_oz_crosscov(gpso_handle* h, cudaStream_t st, const double* Xc, long long Mw, long long nct, double bscale,
                               uint8_t* B, double* wmean) {
    CovKernels::with(h->cov_kid(), [&](auto kid) {
        crosscov_slices_kernel<kid, S><<<(unsigned)nct, 256, oz_xcov_smem(h->dx()), st>>>(
            Xc, Mw, h->kd(), h->ls.as<double>(), h->kern_nls(), h->Xs.as<double>(), h->alpha.as<double>(), h->N, h->Np, h->variance, h->c0,
            bscale, h->Np / 32, B, wmean, h->rq_alpha, h->sum, h->srow);
    });
}

template <int S>
static void launch_oz_trmm(gpso_handle* h, cudaStream_t st, long long nct, long long ldp, double gscale, const uint8_t* B) {
    OzParams P;
    P.A = h->ozA.as<uint8_t>();
    P.B = B;
    P.rowscale = h->rowscale.as<double>();
    P.part = h->part.as<double>();
    P.gscale = gscale;
    P.nb = h->nb;
    P.nks = h->Np / 32;
    P.nct = (int)nct;
    P.ldp = ldp;
    P.items = nullptr;
    P.rounds = 0;
    P.out = nullptr;
    P.Np = h->Np;
    long long units = nct * ((h->nb + 1) / 2);
    int grid = (int)std::min<long long>(h->nsm, units);
    ozaki_kernel<S, OZ_TRMM><<<grid, OZ_THREADS, OzCfg<S>::SMEM_BYTES_TRMM, st>>>(P);
}

template <int S>
static void launch_oz_slices(gpso_handle* h, cudaStream_t st) {
    dim3 grid(h->Np / 32, h->nb);
    linv_slices_kernel<S, false><<<grid, 256, 0, st>>>(h->Linv.as<double>(), h->rowscale.as<double>(), h->Np, h->Np / 32, h->ozA.as<uint8_t>());
}

#define DISPATCH_S(S_, fn, ...)                \
    switch (S_) {                              \
        case 5: fn<5>(__VA_ARGS__); break;     \
        case 6: fn<6>(__VA_ARGS__); break;     \
        case 7: fn<7>(__VA_ARGS__); break;     \
        default: fn<8>(__VA_ARGS__); break;    \
    }

// The partial sums of one covariance family on d scaled input rows (a sum kernel calls this once per component, with the
// component's own scaled inputs, dimensions, variance and alpha, into its own block of partial sums).
static void launch_grad(gpso_handle* h, cudaStream_t st, int nblk, int stride, int kernel_id, int ard, const double* Xs, int d, double var,
                        double rq_alpha, double* part) {
    AllKernels::with(kernel_id, [&](auto kid) {
        if (!ard) {
            lml_grad_kernel<kid, false><<<nblk, 256, 0, st>>>(Xs, h->alpha.as<double>(), h->Kinv.as<double>(), h->N,
                                                             d, h->Np, var, 0, 1, part, stride, rq_alpha);
            h->launches++;
        } else {
            for (int dim0 = 0; dim0 < d; dim0 += GRAD_DCH) {
                int nd = std::min(GRAD_DCH, d - dim0);
                lml_grad_kernel<kid, true><<<nblk, 256, 0, st>>>(Xs, h->alpha.as<double>(), h->Kinv.as<double>(),
                                                                h->N, d, h->Np, var, dim0, nd, part,
                                                                stride, rq_alpha);
                h->launches++;
            }
        }
    });
}

static size_t periodic_grad_smem(int d) { return (size_t)(6 * d * CT + CT * CT) * sizeof(double); }
static const int PERIODIC_GRAD_SMEM_MAX = (int)periodic_grad_smem(MAX_LS / 2);
static size_t linear_grad_smem(int k) { return (size_t)(2 * k * CT + CT * CT) * sizeof(double); }
static const int LINEAR_GRAD_SMEM_MAX = (int)linear_grad_smem(MAX_LS);

// Function attributes (dynamic shared-memory limits, carve-out preferences) belong to the device's primary context: set once per
// device and process, not per handle (the ~90 cudaFuncSetAttribute calls cost 0.3 s per gpso_create).
static bool g_configured[64] = {false};
static int configure_kernels_once(int device);

static int configure_kernels() {
    CU_TRY(cudaFuncSetAttribute(dense_gemm_kernel<MODE_CHOL_PANEL>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(dense_gemm_kernel<MODE_CHOL_TRAIL>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(dense_gemm_kernel<MODE_TRTRI_XT>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(dense_gemm_kernel<MODE_TRTRI_Y>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(dense_gemm_kernel<MODE_LAUUM>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(dense_gemm_kernel<MODE_LAUUM_PART>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(predict_trmm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(joint_v_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(joint_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(diag_factor_inverse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(factor_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(diag_transpose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DIAG_TRANSPOSE_SMEM));
    CU_TRY(cudaFuncSetAttribute(grow_leaves_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, leaf_smem_bytes(LEAF_MAXD)));
    CU_TRY(cudaFuncSetAttribute(ozaki_kernel<OZ_KINV_S, OZ_LAUUM>, cudaFuncAttributeMaxDynamicSharedMemorySize, OzCfg<OZ_KINV_S>::SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(ozaki_kernel<OZ_INV_S, OZ_GEMM>, cudaFuncAttributeMaxDynamicSharedMemorySize, OzCfg<OZ_INV_S>::SMEM_BYTES));
    CU_TRY(cudaFuncSetAttribute(ozaki_kernel<OZ_HYB_S, OZ_GEMM>, cudaFuncAttributeMaxDynamicSharedMemorySize, OzCfg<OZ_HYB_S>::SMEM_BYTES));
    // up to 64 scaled coordinate rows of the tile's rows and columns, and four ARD factors' pair weights
    CU_TRY(cudaFuncSetAttribute(lml_grad_product_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (2 * MAX_LS * CT + MAX_SUM * CT * CT) * (int)sizeof(double)));
    // with periodic factors also 2 x 32 raw coordinate rows: 224 KB, within the 227 KB of a block
    CU_TRY(cudaFuncSetAttribute(lml_grad_product_periodic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (2 * MAX_LS * CT + MAX_LS * CT + MAX_SUM * CT * CT) * (int)sizeof(double)));
    // a periodic kernel of up to 32 dimensions: 64 embedded and 32 raw coordinate rows of the tile's rows and columns, the pair weights
    CU_TRY(cudaFuncSetAttribute(lml_grad_periodic_kernel<KERNEL_SE>, cudaFuncAttributeMaxDynamicSharedMemorySize, PERIODIC_GRAD_SMEM_MAX));
    CU_TRY(cudaFuncSetAttribute(lml_grad_periodic_kernel<KERNEL_RQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, PERIODIC_GRAD_SMEM_MAX));
    CU_TRY(cudaFuncSetAttribute(joint_syrk_kernel<KERNEL_SUM_LIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    // a Linear component of up to 64 columns: its rows for the tile's rows and columns, the pair weights
    CU_TRY(cudaFuncSetAttribute(lml_grad_linear_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LINEAR_GRAD_SMEM_MAX));
    GP_TRY(CovKernels::each([](auto kid) -> int {
        CU_TRY(cudaFuncSetAttribute(joint_syrk_kernel<kid>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
        CU_TRY(cudaFuncSetAttribute(crosscov_screen_kernel<kid, 0, SCR_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_XCOV_SMEM_MAX));
        return 0;
    }));
    GP_TRY(screen_configure<2>());
    GP_TRY(screen_configure<3>());
    GP_TRY(screen_configure<4>());
    GP_TRY(oz_configure<5>());
    GP_TRY(oz_configure<6>());
    GP_TRY(oz_configure<7>());
    GP_TRY(oz_configure<8>());
    return 0;
}

static int configure_kernels_once(int device) {
    const int slot = device & 63;
    if (g_configured[slot]) return 0;
    GP_TRY(configure_kernels());
    g_configured[slot] = true;
    return 0;
}

// (re)allocate everything that depends on the problem shape
static int ensure_shape(gpso_handle* h, int N, int d) {
    int Np = ((N + TB - 1) / TB) * TB;
    size_t mat = (size_t)Np * Np * sizeof(double);
    GP_TRY(h->X.ensure((size_t)N * d * sizeof(double)));
    GP_TRY(h->y.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->Xs.ensure((size_t)h->rows_for(d) * Np * sizeof(double)));
    GP_TRY(h->ls.ensure(MAX_LS * sizeof(double)));
    if (h->periodic) GP_TRY(h->plp.ensure(2 * MAX_LS * sizeof(double)));
    if (h->composite()) {  // each component's rows: its d (active) columns, or 2d embedded rows for a periodic component
        int off = 0;
        for (int c = 0; c < h->sum.n; c++) {
            h->srow.off[c] = off;
            h->srow.rows[c] = h->sum_per[c] ? 2 * h->cdim(c, d) : h->cdim(c, d);
            off += h->srow.rows[c];
        }
        h->srow.width = off;
    }
    if (h->linear()) GP_TRY(h->meanA.ensure(MAX_LS * sizeof(double)));
    GP_TRY(h->alpha.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->resid.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->a.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->K.ensure(mat, true));
    GP_TRY(h->Linv.ensure(mat, true));
    GP_TRY(h->LinvT.ensure(mat, true));
    GP_TRY(h->logdet.ensure((size_t)(Np / TB) * sizeof(double)));
    GP_TRY(h->scalars.ensure(16 * sizeof(double)));
    GP_TRY(h->info.ensure(sizeof(int)));
    GP_TRY(h->counter.ensure(sizeof(int)));
    GP_TRY(h->running.ensure(sizeof(BestRec)));
    if (Np != h->Np) {
        // the factor kernels never write the structural zeros of L^-1 / L^-T inside diagonal blocks: clear both buffers
        // whenever the row pitch changes (a buffer that was large enough is reused with a different layout)
        CU_TRY(cudaStreamSynchronize(h->stream));
        CU_TRY(cudaMemsetAsync(h->Linv.p, 0, mat, h->stream));
        CU_TRY(cudaMemsetAsync(h->LinvT.p, 0, mat, h->stream));
        CU_TRY(cudaStreamSynchronize(h->stream));  // rare (shape change); callers may continue on another stream
    }
    h->N = N;
    h->d = d;
    h->Np = Np;
    h->nb = Np / TB;
    return 0;
}

// Xs[dim][Np] = X / ls; a sum: Xs_c = X / ls_c at Xs + c d Np, the division of the bare kernel (ls_c expanded to d entries);
// a periodic kernel: the embedded rows [cos rows; sin rows] = [2d][Np]; a sum / product with periodic components or a map: the
// rows of rmap, one launch
static int scale_inputs(gpso_handle* h, cudaStream_t st, const double* X, int rows, int Np, double* Xs) {
    if (h->periodic) {
        periodic_embed_kernel<<<(unsigned)(((long long)Np * h->d + 255) / 256), 256, 0, st>>>(X, rows, Np, h->d, h->plp.as<double>(), 1,
                                                                                              Np, Xs);
        return check_launch(h, "periodic_embed");
    }
    if (h->emb()) {
        stage_rows_kernel<<<(unsigned)(((long long)Np * h->rmap.n + 255) / 256), 256, 0, st>>>(X, rows, Np, h->d, h->rmap, 1, 1, Np, Xs);
        return check_launch(h, "stage_rows");
    }
    if (!h->composite()) {
        scale_inputs_kernel<<<(Np + 255) / 256, 256, 0, st>>>(X, h->ls.as<double>(), h->n_ls(), rows, h->d, Np, Xs);
        return check_launch(h, "scale_inputs");
    }
    for (int c = 0; c < h->sum.n; c++) {
        scale_inputs_kernel<<<(Np + 255) / 256, 256, 0, st>>>(X, h->ls.as<double>() + c * h->d, h->d, rows, h->d, Np,
                                                              Xs + (size_t)c * h->d * Np);
        GP_TRY(check_launch(h, "scale_inputs"));
    }
    return 0;
}

// a periodic kernel: the unit lengthscale of the base kernel on the embedded rows, and [l, p] (each expanded to d entries) for
// the embedding
static int upload_lengthscales(gpso_handle* h, cudaStream_t st) {
    if (h->periodic) {
        for (int k = 0; k < h->d; k++) {
            h->plp_host[k] = h->ls_host[h->ard ? k : 0];
            h->plp_host[h->d + k] = h->per_p[h->per_ard ? k : 0];
        }
        CU_TRY(cudaMemcpyAsync(h->ls.p, &h->unit_ls, sizeof(double), cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(h->plp.p, h->plp_host, sizeof(double) * 2 * h->d, cudaMemcpyHostToDevice, st));
        return 0;
    }
    if (h->emb()) {  // ls: [width], a periodic component's rows at unit lengthscale; rmap: one slot per active column
        double lsw[MAX_LS];
        RowMap& m = h->rmap;
        m.n = 0;
        for (int c = 0; c < h->sum.n; c++) {
            const int o = h->srow.off[c], k = h->cdim(c, h->d), lo = h->ls_off(c);
            for (int j = 0; j < k; j++, m.n++) {
                m.src[m.n] = h->nmap ? h->map_cols[h->map_off[c] + j] : j;
                m.r0[m.n] = o + j;
                m.r1[m.n] = h->sum_per[c] ? o + k + j : -1;
                // a Linear component's rows: its columns over 1 / sqrt(variance)
                const double l = h->comp_lin(c) ? 1.0 / sqrt(h->ls_host[lo + j]) : h->ls_host[lo + j];
                m.l[m.n] = l;
                m.p[m.n] = h->sum_per[c] ? h->comp_p[c][h->sum_per_ard[c] ? j : 0] : 0.0;
                lsw[o + j] = h->sum_per[c] ? 1.0 : l;
                if (h->sum_per[c]) lsw[o + k + j] = 1.0;
            }
        }
        CU_TRY(cudaMemcpyAsync(h->ls.p, lsw, sizeof(double) * h->dx(), cudaMemcpyHostToDevice, st));
        CU_TRY(cudaStreamSynchronize(st));  // lsw is on this stack frame
        return 0;
    }
    CU_TRY(cudaMemcpyAsync(h->ls.p, h->ls_host, sizeof(double) * h->n_ls(), cudaMemcpyHostToDevice, st));
    return 0;
}

// Linear mean: out[0..rows) += sgn * (x_i . A) for the rows x_i of X, one launch on st, the stream that produces out (the
// constant b is already in out as c0).  Nothing for the other mean functions.
static int add_linear_offset(gpso_handle* h, cudaStream_t st, const double* X, long long rows, double sgn, double* out) {
    if (!h->linear()) return 0;
    linear_offset_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(X, rows, h->d, h->meanA.as<double>(), sgn, out);
    return check_launch(h, "linear_offset");
}

// Task list of the persistent factorisation kernel (kern_dense.cuh): topological, with look-ahead.  Cholesky in blocks of
// W panels.  Per panel p of a block [p0, p1): DIAG(p) (the last update of its tile, narrow or wide, is fused in), the
// narrow updates of panel p-1 (they run beside DIAG(p)), wide updates of the previous block as cover for the time the
// diagonal block takes, PANEL(.,p), TRANSPOSE(p), cover for the panels.  Then the wide updates of block b: the columns of
// block b+1 first, the rest becomes the cover of the next block's chain (the queue is popped at about nsm / T_wide tasks per
// microsecond).  After the Cholesky: the recursive-doubling inverse, level by level, long tiles first; its tasks carry
// pair-level dependencies, so the levels overlap instead of being separated by launches.
namespace {
struct FactorTask {
    int w[TASK_WORDS];
    FactorTask(int op, int p, int i, int j, int s, int tile) {
        for (int k = 0; k < TASK_WORDS; k++) w[k] = 0;
        w[0] = op; w[1] = p; w[2] = i; w[3] = j; w[4] = s; w[5] = tile;
        w[6] = w[7] = w[8] = -1;
        w[12] = 0; w[13] = 0;
    }
    FactorTask& dep(int idx, int val) {
        for (int k = 0; k < 3; k++)
            if (w[6 + k] < 0) { w[6 + k] = idx; w[9 + k] = val; return *this; }
        return *this;  // more than three dependencies: a builder bug, caught by the host-side simulation in the tests
    }
    FactorTask& done(int idx, int val) { w[12] = idx; w[13] = val; return *this; }
};
}  // namespace

static int make_factor_tasks(int nb, int nsm, std::vector<int>& flat, int& ntasks, int& ncounters_out, int inv_cap = 1 << 30) {
    // panels per block of the two-level blocking.  Up to 47 panels (the leaves of the hybrid factorisation, every matrix up to
    // N = 4096) the factorisation is bound by its chains of dependent tile tasks, not by the DMMA pipe: unblocked updates (W = 1)
    // keep the off-diagonal chain PANEL -> UPDATE -> PANEL at 56 us per step (W = 2: 63 us); measured 3.28 vs 3.40 ms per LML+grad
    // evaluation at N = 4096, 1.38 vs 1.52 at 2048
    const int W = nb >= 48 ? 4 : 1;
    if (nb < 1 || nb > 255) return fail(GPSO_E_BADARG, "matrix too large for the tile scheduler (more than 255 panels)");
    const int LV = 8;  // levels of the inverse recursion: s = 1 .. 128
    auto T = [nb](int i, int j) { return i * nb + j; };          // tile counters
    const int TR_ALL = nb * nb;                                    // transposes completed
    auto XTD = [nb, LV](int l, int q) { return nb * nb + 1 + l * nb + q; };
    auto YD = [nb, LV](int l, int q) { return nb * nb + 1 + LV * nb + l * nb + q; };
    auto STRIP = [nb, LV](int j) { return nb * nb + 1 + 2 * LV * nb + j; };  // strips of the tile (j+1, j) completed
    auto PRE = [nb, LV](int p) { return nb * nb + 1 + 2 * LV * nb + nb + p; };    // early part of the last wide update of tile (p, p)
    auto TRC = [nb, LV](int p) { return nb * nb + 1 + 2 * LV * nb + 2 * nb + p; };  // transposes of the tiles 0 .. p done
    const int ncounters = nb * nb + 1 + 2 * LV * nb + 3 * nb;
    auto ops = [W](int j) { return chol_ops(j, W); };
    auto fin = [W](int j) { return chol_ops(j, W) + 1; };
    // "tile (i, j) is final": its own counter, or for the strip-solved tile below the diagonal the strip counter
    auto FINC = [&](int i, int j) { return i == j + 1 ? STRIP(j) : T(i, j); };
    auto FINV = [&](int i, int j) { return i == j + 1 ? PANEL_STRIPS : fin(j); };

    const double t_wide_us = 17.0 * W + 12.0;  // tile time of a wide update (DMMA at peak + tile write-back)
    const double pops_per_us = nsm / t_wide_us;
    std::vector<FactorTask> q, wide;
    size_t wpos = 0;
    auto cover = [&](double us) {
        if (us <= 0) return;
        const double want = pops_per_us * us;
        const size_t e = want >= (double)(wide.size() - wpos) ? wide.size() : wpos + (size_t)want;
        q.insert(q.end(), wide.begin() + wpos, wide.begin() + e);
        wpos = e;
    };
    auto wide_task = [&](int b, int i, int j) {
        const int p0 = b * W, p1 = std::min(nb, p0 + W), last = p1 - 1;
        return FactorTask(CT_UPD, p0, i, j, p1 - p0, 0).dep(FINC(i, last), FINV(i, last)).dep(FINC(j, last), FINV(j, last)).dep(T(i, j), b).done(T(i, j), b + 1);
    };
    // ---- inverse factor by recursive doubling, levels s < inv_cap (the int8 engine takes the levels above): level s merges
    // the inverses of the tile ranges [a, a+s) and [a+s, a+s+nv), a = 2 q s.  The tasks of a pair enter the queue as soon as
    // the Cholesky step that completes their inputs has been queued -- X^T = L11^-T L21^T after the last panel of the first
    // half, the merge L21^-1 = -L22^-1 X after the last tile of the pair -- so that they run on the SMs the chain-bound
    // factorisation leaves idle instead of after it.
    int nlevels = 0;
    for (int s = 1; s < nb && s < inv_cap; s *= 2) nlevels++;
    if (nlevels > LV) return fail(GPSO_E_BADARG, "matrix too large for the inverse recursion of the tile scheduler");
    std::vector<std::vector<int>> pair_off(nlevels);  // first tile index of pair q in the kernel's enumeration, per level
    for (int s = 1, l = 0; l < nlevels; s *= 2, l++) {
        int total = 0;
        for (int qq = 0; 2 * qq * s < nb; qq++) {
            pair_off[l].push_back(total);
            total += s * trtri_pair_vtiles(nb, s, qq);
        }
    }
    auto inverse_tasks_ready_after = [&](int p) {
        for (int s = 1, l = 0; l < nlevels; s *= 2, l++)
            for (int qq = 0; 2 * qq * s < nb; qq++) {
                const int nv = trtri_pair_vtiles(nb, s, qq), a = 2 * qq * s;
                if (nv == 0) continue;
                if (a + s + nv - 1 == p) {  // the pair is complete: merge
                    for (int v = nv - 1; v >= 0; v--)  // large v = long contraction first
                        for (int u = 0; u < s; u++) {
                            FactorTask t(CT_Y, 0, 0, 0, s, pair_off[l][qq] + u * nv + v);
                            t.dep(XTD(l, qq), s * nv);
                            if (nv == 1) {
                                t.dep(T(a + s, a + s), fin(a + s));
                            } else {
                                int s2 = 1, l2 = 0;
                                while (s2 * 2 < nv) { s2 *= 2; l2++; }
                                t.dep(YD(l2, (a + s) / (2 * s2)), s2 * (nv - s2));
                            }
                            q.push_back(t.done(YD(l, qq), 0));
                        }
                }
                if (a + s - 1 == p) {  // the first half and the rows of L21 up to its last column are complete: X^T
                    for (int u = 0; u < s; u++)  // small u = long contraction first
                        for (int v = 0; v < nv; v++) {
                            FactorTask t(CT_XT, 0, 0, 0, s, pair_off[l][qq] + u * nv + v);
                            t.dep(TRC(a + s - 1), 1);
                            if (s > 1) t.dep(YD(l - 1, 2 * qq), (s / 2) * (s / 2));
                            t.dep(FINC(a + s + v, a + s - 1), FINV(a + s + v, a + s - 1));
                            q.push_back(t.done(XTD(l, qq), 0));
                        }
                }
            }
    };
    const int nblk = (nb + W - 1) / W;
    for (int b = 0; b < nblk; b++) {
        const int p0 = b * W, p1 = std::min(nb, p0 + W);
        for (int p = p0; p < p1; p++) {
            // the first diagonal tile of a block still lacks the wide update of the previous block: all but the last panel of
            // it were applied by an ordinary task while the chain was busy with that panel (PRE, queued below), so that every
            // DIAG fuses exactly one panel (10 us on the chain instead of 10 W)
            const bool pre_done = W >= 2 && p > 0 && p % W == 0;
            const int nprev = p > 0 ? 1 : 0;
            FactorTask dg(CT_DIAG, p, p, p, nprev, 0);
            if (p > 0) dg.dep(T(p, p), ops(p) - 1).dep(FINC(p, p - 1), FINV(p, p - 1));
            if (pre_done) dg.dep(PRE(p), 1);
            q.push_back(dg.done(T(p, p), fin(p)));
            size_t narrow = 0;
            if (p > p0)
                for (int j = p; j < p1; j++)
                    for (int i = j; i < nb; i++)
                        if (!(i == p && j == p)) {
                            const int at = j / W + (p - 1) % W;  // updates tile (i,j) has received before this one
                            q.push_back(FactorTask(CT_UPD, p - 1, i, j, 1, 0).dep(FINC(i, p - 1), FINV(i, p - 1)).dep(FINC(j, p - 1), FINV(j, p - 1)).dep(T(i, j), at).done(T(i, j), at + 1));
                            narrow++;
                        }
            // the successors of DIAG(p) on the chain take their tickets BEFORE the filler updates and wait for it on their SMs:
            // the four strips of tile (p+1, p) (DIAG(p+1) waits for them) and PANEL(p+2, p) (the update of tile (p+2, p+1),
            // which the strips of the next step wait for); five idle SMs for one DIAG instead of a chain that waits for a free one
            auto panel_task = [&](int i) {
                return FactorTask(CT_PANEL, p, i, p, 0, 0).dep(T(p, p), fin(p)).dep(T(i, p), ops(p)).done(T(i, p), fin(p));
            };
            if (p + 1 < nb)
                for (int k = 0; k < PANEL_STRIPS; k++)
                    q.push_back(FactorTask(CT_PANEL, p, p + 1, p, k + 1, 0).dep(T(p, p), fin(p)).dep(T(p + 1, p), ops(p)).done(STRIP(p), 0));
            if (p + 2 < nb) q.push_back(panel_task(p + 2));
            cover((p > p0 ? 42.0 : 30.0 + 10.0 * nprev) - narrow * 30.0 / nsm);
            for (int i = p + 3; i < nb; i++) q.push_back(panel_task(i));
            if (W >= 2 && p == p1 - 2 && p1 - p0 == W && p1 < nb)
                q.push_back(FactorTask(CT_UPD, p0, p1, p1, W - 1, 0).dep(T(p1, p), fin(p)).dep(T(p1, p1), b).done(PRE(p1), 1));
            {
                FactorTask tr(CT_TRANSPOSE, p, p, p, 0, 0);
                tr.dep(T(p, p), fin(p));
                if (p > 0) tr.dep(TRC(p - 1), 1);
                q.push_back(tr.done(TRC(p), 1));
            }
            inverse_tasks_ready_after(p);
            cover(22.0);
        }
        cover(1e30);  // flush
        wide.clear();
        wpos = 0;
        const int next_end = std::min(nb, p1 + W);
        for (int j = p1; j < next_end; j++)
            for (int i = j; i < nb; i++)
                if (!(i == p1 && j == p1)) q.push_back(wide_task(b, i, j));  // tile (p1,p1): fused into DIAG(p1)
        for (int j = next_end; j < nb; j++)
            for (int i = j; i < nb; i++) wide.push_back(wide_task(b, i, j));
    }
    flat.clear();
    flat.reserve(q.size() * TASK_WORDS);
    for (const FactorTask& t : q) flat.insert(flat.end(), t.w, t.w + TASK_WORDS);
    ntasks = (int)q.size();
    ncounters_out = ncounters;
    return 0;
}

static int get_factor_plan(gpso_handle* h, int n, int inv_cap, gpso_handle::FactorPlan** out) {
    inv_cap = std::min(inv_cap, 1 << 10);
    gpso_handle::FactorPlan& plan = h->factor_plans[2048 * n + inv_cap];
    if (!plan.tasks.p) {
        std::vector<int> flat;
        GP_TRY(make_factor_tasks(n, h->nsm > 0 ? h->nsm : 148, flat, plan.ntasks, plan.ncounters, inv_cap));
        GP_TRY(plan.tasks.ensure(flat.size() * sizeof(int)));
        CU_TRY(cudaMemcpy(plan.tasks.p, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    *out = &plan;
    return 0;
}

// Operands of the dense kernels for the n-tile diagonal block that starts at tile t0 of matrices with row pitch Np (T may be
// null: only the FP64 inverse recursion uses it).
static DenseParams dense_block(double* K, double* Linv, double* LinvT, double* T, int Np, int t0, int n) {
    const size_t off = (size_t)t0 * TB * Np + (size_t)t0 * TB;
    DenseParams P{};
    P.K = K + off;
    P.Linv = Linv + off;
    P.LinvT = LinvT + off;
    P.T = T ? T + off : nullptr;
    P.Np = Np;
    P.nb = n;
    P.pivot_off = t0 * TB;
    return P;
}

// One launch of the persistent factorisation kernel over the task list of `plan` (rows >= N of the block are padding);
// `state` is its scheduler state, cleared here.
static int launch_factor(gpso_handle* h, cudaStream_t st, const DenseParams& P, int N, const gpso_handle::FactorPlan* plan,
                         DevBuf& state, double* logdet, int* info) {
    const size_t bytes = (size_t)(2 + plan->ncounters) * sizeof(int);
    GP_TRY(state.ensure(bytes));
    CU_TRY(cudaMemsetAsync(state.p, 0, bytes, st));
    const int grid = std::min(plan->ntasks, h->nsm > 0 ? h->nsm : 148);
    factor_persistent_kernel<<<grid, GTHREADS, DIAG_SMEM_BYTES, st>>>(P, N, plan->tasks.as<int>(), plan->ntasks, state.as<int>(), logdet,
                                                                       info);
    return check_launch(h, "factor_persistent");
}

// Host-only introspection (no GPU needed): the task list for a matrix of nb panels on nsm SMs, TASK_WORDS ints per task.
// Used by the CPU tests to check that the queue is a topological order of its own dependencies.
extern "C" int gpso_debug_factor_tasks_cap(int nb, int nsm, int inv_cap, int* out, int64_t capacity_words, int* ntasks, int* ncounters);
extern "C" int gpso_debug_factor_tasks(int nb, int nsm, int* out, int64_t capacity_words, int* ntasks, int* ncounters) {
    return gpso_debug_factor_tasks_cap(nb, nsm, 1 << 30, out, capacity_words, ntasks, ncounters);
}
extern "C" int gpso_debug_factor_tasks_cap(int nb, int nsm, int inv_cap, int* out, int64_t capacity_words, int* ntasks, int* ncounters) {
    if (!ntasks || !ncounters || inv_cap < 0) return fail(GPSO_E_BADARG, "gpso_debug_factor_tasks: bad argument");
    std::vector<int> flat;
    GP_TRY(make_factor_tasks(nb, nsm, flat, *ntasks, *ncounters, inv_cap));
    if (out) {
        if (capacity_words < (int64_t)flat.size()) return fail(GPSO_E_BADARG, "gpso_debug_factor_tasks: buffer too small");
        std::copy(flat.begin(), flat.end(), out);
    }
    return 0;
}

// Deal tiles (row block, 64-row tile of B, first k-step, k-steps) to G persistent CTAs, longest first, each to the CTA with the
// least work so far; appended to `all` as a [rounds][G][4] table (-1 = none).
static void deal_items(std::vector<std::array<int, 4>>& items, int G, std::vector<int>& all, size_t& off, int& rounds) {
    std::stable_sort(items.begin(), items.end(), [](const std::array<int, 4>& a, const std::array<int, 4>& b) { return a[3] > b[3]; });
    std::vector<std::vector<int>> per(G);
    std::vector<long long> load(G, 0);
    for (size_t i = 0; i < items.size(); i++) {
        int best = 0;
        for (int g = 1; g < G; g++)
            if (load[g] < load[best]) best = g;
        per[best].push_back((int)i);
        load[best] += items[i][3] + 6;
    }
    size_t r = 0;
    for (int g = 0; g < G; g++) r = std::max(r, per[g].size());
    off = all.size();
    rounds = (int)r;
    all.resize(off + r * G * 4, -1);
    for (int g = 0; g < G; g++)
        for (size_t k = 0; k < per[g].size(); k++)
            for (int c = 0; c < 4; c++) all[off + (k * G + g) * 4 + c] = items[per[g][k]][c];
}

// K_y^-1 = L^-T L^-1 on the int8 tensor cores (kern_ozaki.cuh, OZ_LAUUM).  The tiles (row block I, 64-wide column tile
// ct <= 2I+1) cost nks - 4I k-steps each (the contraction runs over k >= i only); they are dealt as above and stored as a
// [rounds][nsm] table of I << 16 | ct (-1 = none) the kernel walks by rounds.
static void make_lauum_items(int nb, int G, std::vector<int>& flat, int& rounds) {
    std::vector<std::array<int, 4>> items;
    for (int I = 0; I < nb; I++)
        for (int ct = 0; ct <= 2 * I + 1; ct++) items.push_back({I, ct, 0, 4 * (nb - I)});
    std::vector<int> all;
    size_t off = 0;
    deal_items(items, G, all, off, rounds);
    flat.resize(all.size() / 4);
    for (size_t k = 0; k < flat.size(); k++) flat[k] = all[4 * k] < 0 ? -1 : (all[4 * k] << 16 | all[4 * k + 1]);
}

static int build_lauum_items(gpso_handle* h) {
    const int nb = h->nb, G = h->nsm > 0 ? h->nsm : 148;
    if (h->lauum_items_nb == nb && h->lauum_items.p) return 0;
    std::vector<int> flat;
    int rounds = 0;
    make_lauum_items(nb, G, flat, rounds);
    GP_TRY(h->lauum_items.ensure(flat.size() * sizeof(int)));
    CU_TRY(cudaMemcpy(h->lauum_items.p, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice));
    h->lauum_items_nb = nb;
    h->lauum_rounds = (int)rounds;
    return 0;
}

static int kinv_int8(gpso_handle* h, cudaStream_t st) {
    constexpr int S = OZ_KINV_S;
    const int Np = h->Np, nb = h->nb, nks = Np / 32;
    GP_TRY(h->colscale.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->colmax.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->ozT.ensure((size_t)Np * Np * S));
    GP_TRY(build_lauum_items(h));
    linv_rowscale_kernel<true><<<(Np + 7) / 8, 256, 0, st>>>(h->LinvT.as<double>(), Np, h->colscale.as<double>(), h->colmax.as<double>());
    GP_TRY(check_launch(h, "linvT_rowscale"));
    linv_slices_kernel<S, true><<<dim3(nks, nb), 256, 0, st>>>(h->LinvT.as<double>(), h->colscale.as<double>(), Np, nks, h->ozT.as<uint8_t>());
    GP_TRY(check_launch(h, "linvT_slices"));
    OzParams P;
    P.A = h->ozT.as<uint8_t>();
    P.B = h->ozT.as<uint8_t>();
    P.rowscale = h->colscale.as<double>();
    P.part = nullptr;
    P.gscale = ldexp(1.0, -2 * (8 * S - 2) + 8 * (S - 1));
    P.nb = nb;
    P.nks = nks;
    P.nct = 2 * nb;
    P.ldp = 0;
    P.items = h->lauum_items.as<int>();
    P.rounds = h->lauum_rounds;
    P.out = h->Kinv.as<double>();
    P.Np = Np;
    const int grid = h->nsm > 0 ? h->nsm : 148;
    ozaki_kernel<S, OZ_LAUUM><<<grid, OZ_THREADS, OzCfg<S>::SMEM_BYTES, st>>>(P);
    GP_TRY(check_launch(h, "ozaki_lauum"));
    return 0;
}

// L^-1 by recursive doubling on the int8 tensor cores (kern_ozaki.cuh, OZ_GEMM).  Level s merges the finished inverses of
// the tile ranges [a, a+s) and [a+s, a+s+nv), a = 2 q s:   X^T = L11^-T L21^T,   L21^-1 = -(L22^-1 X)   (and its transpose into
// L^-T).  Every operand row is cut into 8 balanced 8-bit digits of a 62-bit fixed-point number relative to the row's
// largest entry in the range the level reads, so the operand rounding (2^-62 of the row scale) is below the fp64 rounding of
// those entries and the integer accumulation is exact.  Tiles (128 x 64) are dealt to the persistent CTAs longest-first.
namespace {
struct InvLevelInfo { int s; size_t xt_off; int xt_rounds; size_t y_off; int y_rounds; };
}
static void make_inverse_items(int nb, int G, std::vector<int>& all, std::vector<InvLevelInfo>& levels) {
    all.clear();
    levels.clear();
    for (int s = 1; s < nb; s *= 2) {
        std::vector<std::array<int, 4>> xt, y;
        for (int q = 0; 2 * q * s < nb; q++) {
            const int nv = trtri_pair_vtiles(nb, s, q), a = 2 * q * s;
            for (int u = 0; u < s; u++)
                for (int v = 0; v < nv; v++)
                    for (int hh = 0; hh < 2; hh++) {
                        xt.push_back({a + u, 2 * (a + s + v) + hh, 4 * (a + u), 4 * (s - u)});
                        y.push_back({a + s + v, 2 * (a + u) + hh, 4 * (a + s), 4 * (v + 1)});
                    }
        }
        InvLevelInfo lv;
        lv.s = s;
        deal_items(xt, G, all, lv.xt_off, lv.xt_rounds);
        deal_items(y, G, all, lv.y_off, lv.y_rounds);
        levels.push_back(lv);
    }
    if (all.empty()) all.resize(4, -1);
}

static int get_inverse_plan(gpso_handle* h, int n, gpso_handle::InvPlan** out) {
    gpso_handle::InvPlan& plan = h->inv_plans[n];
    if (!plan.items.p) {
        std::vector<int> all;
        std::vector<InvLevelInfo> levels;
        make_inverse_items(n, h->nsm > 0 ? h->nsm : 148, all, levels);
        for (const InvLevelInfo& lv : levels) plan.levels.push_back({lv.s, lv.xt_off, lv.xt_rounds, lv.y_off, lv.y_rounds});
        GP_TRY(plan.items.ensure(all.size() * sizeof(int)));
        CU_TRY(cudaMemcpy(plan.items.p, all.data(), all.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    *out = &plan;
    return 0;
}

static int ensure_inverse_buffers(gpso_handle* h) {
    const size_t dig = (size_t)h->Np * h->Np * OZ_INV_S;
    GP_TRY(h->ozL.ensure(dig));
    GP_TRY(h->ozLT.ensure(dig));
    GP_TRY(h->ozLI.ensure(dig));
    GP_TRY(h->ozXT.ensure(dig));
    GP_TRY(h->rsL.ensure((size_t)h->Np * sizeof(double)));
    GP_TRY(h->rsLT.ensure((size_t)h->Np * sizeof(double)));
    GP_TRY(h->rsLI.ensure((size_t)h->Np * sizeof(double)));
    GP_TRY(h->rsXT.ensure((size_t)h->Np * sizeof(double)));
    GP_TRY(h->T.ensure((size_t)h->Np * h->Np * sizeof(double), true));
    return 0;
}

// S digits per operand of the products below: OZ_INV_S for the inverse factor, OZ_HYB_S for the panel solve and Schur
// complement of the hybrid factorisation.
// Digits of the rows of the n-tile sub-matrix whose first element is M (row pitch Np), over the k-range `kind` selects.
template <int S>
static int oz_range_digits(gpso_handle* h, cudaStream_t st, const double* M, int n, int kind, int s, DevBuf& scales, DevBuf& out,
                           const char* what) {
    const int Np = h->Np, nks = Np / 32;
    range_rowscale_kernel<<<n * 16, 256, 0, st>>>(M, Np, kind, s, n, scales.as<double>());
    GP_TRY(check_launch(h, what));
    range_slices_kernel<S><<<dim3(4 * n, n), 256, 0, st>>>(M, scales.as<double>(), Np, nks, kind, s, n, out.as<uint8_t>());
    return check_launch(h, what);
}

// out[i][j] (+)= sign * sum_k A[i][k] B[j][k] over the tiles and k-ranges of an item table, on the int8 tensor cores
template <int S>
static int oz_range_product(gpso_handle* h, cudaStream_t st, const DevBuf& A, const DevBuf& rsA, const DevBuf& B, const DevBuf& rsB,
                            const int* items, int rounds, int n, double* out, double* out_t, double sign, bool accumulate,
                            const char* what) {
    OzParams P;
    P.A = A.as<uint8_t>();
    P.B = B.as<uint8_t>();
    P.rowscale = rsA.as<double>();
    P.colscale = rsB.as<double>();
    P.part = nullptr;
    P.gscale = ldexp(1.0, -2 * (8 * S - 2) + 8 * (S - 1));
    P.nb = n;
    P.nks = h->Np / 32;
    P.nct = 2 * n;
    P.ldp = 0;
    P.items = items;
    P.rounds = rounds;
    P.out = out;
    P.out_t = out_t;
    P.sign = sign;
    P.accumulate = accumulate ? 1 : 0;
    P.Np = h->Np;
    ozaki_kernel<S, OZ_GEMM><<<h->nsm > 0 ? h->nsm : 148, OZ_THREADS, OzCfg<S>::SMEM_BYTES, st>>>(P);
    return check_launch(h, what);
}

// Levels s_lo <= s < s_hi of the recursive-doubling inverse of the n-tile diagonal block that starts at tile t0 (the whole
// matrix: t0 = 0, n = nb, all levels).  A single level (the merge of a hybrid node) only needs the L21 rows of the factor.
static int inverse_int8(gpso_handle* h, cudaStream_t st, int t0, int n, int s_lo, int s_hi) {
    const int Np = h->Np;
    GP_TRY(ensure_inverse_buffers(h));
    gpso_handle::InvPlan* plan = nullptr;
    GP_TRY(get_inverse_plan(h, n, &plan));
    const size_t off = (size_t)t0 * 128 * Np + (size_t)t0 * 128;
    const double* L = h->K.as<double>() + off;
    double* Linv = h->Linv.as<double>() + off;
    double* LinvT = h->LinvT.as<double>() + off;
    double* T = h->T.as<double>() + off;
    const bool single = s_hi <= 2 * s_lo;
    GP_TRY(oz_range_digits<OZ_INV_S>(h, st, L, n, single ? OZR_PANEL : OZR_L, single ? s_lo : 1, h->rsL, h->ozL, "digits_L"));
    for (const gpso_handle::InvLevel& lv : plan->levels) {
        if (lv.xt_rounds == 0 || lv.s < s_lo || lv.s >= s_hi) continue;
        GP_TRY(oz_range_digits<OZ_INV_S>(h, st, LinvT, n, OZR_LINVT, lv.s, h->rsLT, h->ozLT, "digits_LinvT"));
        GP_TRY(oz_range_product<OZ_INV_S>(h, st, h->ozLT, h->rsLT, h->ozL, h->rsL, plan->items.as<int>() + lv.xt_off, lv.xt_rounds, n, T,
                                          nullptr, 1.0, false, "inverse_xt"));
        GP_TRY(oz_range_digits<OZ_INV_S>(h, st, T, n, OZR_XT, lv.s, h->rsXT, h->ozXT, "digits_XT"));
        GP_TRY(oz_range_digits<OZ_INV_S>(h, st, Linv, n, OZR_LINV, lv.s, h->rsLI, h->ozLI, "digits_Linv"));
        GP_TRY(oz_range_product<OZ_INV_S>(h, st, h->ozLI, h->rsLI, h->ozXT, h->rsXT, plan->items.as<int>() + lv.y_off, lv.y_rounds, n, Linv,
                                          LinvT, -1.0, false, "inverse_y"));
    }
    return 0;
}

// ---- hybrid factorisation: FP64 leaves, int8 tensor-core panels and Schur complements --------------------------------------
// The blocked Cholesky of factor_persistent_kernel is bound by its chain of dependent 128-tile steps up to N ~ 4096 and by
// the FP64 DMMA pipe above (0.55 of its peak at N = 8192).  The exact-integer products that already build L^-1 run at ~2.5x
// the FP64 peak in fp64-equivalent work, so a node of n tiles is split after s = the largest power of two below n:
//      [A11      ]      L11, L11^-1            the node's first half, recursively
//      [A21  A22 ]      L21 = A21 L11^-T       one int8 product (OZ_HYB_S = 7 digits per operand, 54-bit fixed point per row)
//                       A22 -= L21 L21^T       one int8 product, accumulated into the lower tiles of A22
//                       L22, L22^-1            the second half, recursively
//                       L21^-1 = -L22^-1 L21 L11^-1     the level-s merge of the recursive-doubling inverse (work the whole-matrix
//                                                      inverse did anyway)
// Leaves (<= HYB_LEAF_TILES tiles) are factorised by the persistent FP64 kernel on the sub-matrix in place; that kernel is
// bound by its chain of 128-tile steps (~70 us each), so smaller leaves do not shorten it, they only add product launches.
// Without the hybrid the whole matrix is one leaf.
constexpr int HYB_LEAF_TILES = 32;  // 4096 rows: measured 11.8 ms per LML+grad evaluation at N = 8192 against 13.5 with leaves of 2048 and 14.1
                                    // with one kernel; at N = 4096 one kernel (3.43 ms) beats two leaves of 2048 (3.89 ms)

// Tile table of one hybrid product for a node of n tiles split after s.  kind 0: L21 tile (I, J), I >= s > J, contraction over
// the tiles [0, J] of row block J of L11^-1;  kind 1: Schur tile (I, J), s <= J <= I, contraction over the s tiles of L21.
static void make_hybrid_items(int kind, int s, int n, int G, std::vector<int>& all, int& rounds) {
    std::vector<std::array<int, 4>> items;
    for (int I = s; I < n; I++) {
        if (kind == 0) {
            for (int J = 0; J < s; J++)
                for (int hh = 0; hh < 2; hh++) items.push_back({I, 2 * J + hh, 0, 4 * (J + 1)});
        } else {
            for (int J = s; J <= I; J++)
                for (int hh = 0; hh < 2; hh++) items.push_back({I, 2 * J + hh, 0, 4 * s});
        }
    }
    all.clear();
    size_t off = 0;
    deal_items(items, G, all, off, rounds);
}

static int get_hybrid_items(gpso_handle* h, int kind, int s, int n, gpso_handle::ItemList** out) {
    gpso_handle::ItemList& list = h->hyb_items[((long long)kind << 40) | ((long long)s << 20) | n];
    if (!list.items.p) {
        std::vector<int> all;
        make_hybrid_items(kind, s, n, h->nsm > 0 ? h->nsm : 148, all, list.rounds);
        GP_TRY(list.items.ensure(all.size() * sizeof(int)));
        CU_TRY(cudaMemcpy(list.items.p, all.data(), all.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    *out = &list;
    return 0;
}

// The hybrid factorisation of n tiles starting at tile t0 as a flat list of steps {op, t0, n, s} in execution order
// (tests/test_hybrid_plan.py replays it in numpy).  A node splits after s = the largest power of two below n.
constexpr int HYB_LEAF = 0, HYB_PANEL = 1, HYB_SCHUR = 2, HYB_MERGE = 3;
static void plan_hybrid(int t0, int n, int leaf, std::vector<std::array<int, 4>>& ops) {
    if (n <= leaf) {
        ops.push_back({HYB_LEAF, t0, n, 0});
        return;
    }
    int s = 1;
    while (2 * s < n) s *= 2;
    plan_hybrid(t0, s, leaf, ops);
    ops.push_back({HYB_PANEL, t0, n, s});
    ops.push_back({HYB_SCHUR, t0, n, s});
    plan_hybrid(t0 + s, n - s, leaf, ops);
    ops.push_back({HYB_MERGE, t0, n, s});
}

extern "C" int64_t gpso_debug_hybrid_plan(int nb, int leaf, int* out, int64_t capacity) {
    if (nb < 1 || leaf < 1) {
        fail(GPSO_E_BADARG, "gpso_debug_hybrid_plan: bad argument");
        return -1;
    }
    std::vector<std::array<int, 4>> ops;
    plan_hybrid(0, nb, leaf, ops);
    if (out)
        for (size_t i = 0; i < ops.size() && (int64_t)(4 * i + 3) < capacity; i++)
            for (int c = 0; c < 4; c++) out[4 * i + c] = ops[i][c];
    return (int64_t)ops.size();
}

extern "C" int64_t gpso_debug_hybrid_items(int kind, int s, int n, int nsm, int* out, int64_t capacity, int* rounds) {
    if (kind < 0 || kind > 1 || s < 1 || n <= s || nsm < 1 || !rounds) {
        fail(GPSO_E_BADARG, "gpso_debug_hybrid_items: bad argument");
        return -1;
    }
    std::vector<int> all;
    make_hybrid_items(kind, s, n, nsm, all, *rounds);
    if (out) std::copy(all.begin(), all.begin() + std::min<int64_t>(capacity, (int64_t)all.size()), out);
    return (int64_t)all.size();
}

// Cholesky factor and inverse of the n-tile diagonal block at tile t0, in place, by the persistent FP64 kernel.  inv8: the int8
// engine is in force for the inverse factor; it then takes the levels from oz_inv_dmma_cap up, the kernel the levels below.
static int hybrid_leaf(gpso_handle* h, cudaStream_t st, int t0, int n, bool inv8) {
    const int Np = h->Np;
    if (n > 1) GP_TRY(h->T.ensure((size_t)Np * Np * sizeof(double), true));
    const DenseParams P = dense_block(h->K.as<double>(), h->Linv.as<double>(), h->LinvT.as<double>(), h->T.as<double>(), Np, t0, n);
    const int Nsub = h->N - t0 * TB;
    double* logdet = h->logdet.as<double>() + t0;
    if (n == 1) {
        diag_factor_inverse_kernel<<<1, DIAG_THREADS, DIAG_SMEM_BYTES, st>>>(P.K, P.Linv, Np, 0, Nsub, logdet, h->info.as<int>(), P.pivot_off);
        GP_TRY(check_launch(h, "diag_factor_inverse"));
        diag_transpose_kernel<<<1, 256, DIAG_TRANSPOSE_SMEM, st>>>(P.Linv, P.LinvT, Np);
        return check_launch(h, "diag_transpose");
    }
    const int cap = inv8 ? oz_inv_dmma_cap(n) : (1 << 30);
    gpso_handle::FactorPlan* plan = nullptr;
    GP_TRY(get_factor_plan(h, n, cap, &plan));
    GP_TRY(launch_factor(h, st, P, Nsub, plan, h->chol_state, logdet, h->info.as<int>()));
    if (cap < n) GP_TRY(inverse_int8(h, st, t0, n, cap, n));
    return 0;
}

static int hybrid_node(gpso_handle* h, cudaStream_t st, int t0_root, int n_root, int leaf, bool inv8) {
    std::vector<std::array<int, 4>> ops;
    plan_hybrid(t0_root, n_root, leaf, ops);
    const int Np = h->Np;
    for (const std::array<int, 4>& op : ops) {
        const int t0 = op[1], n = op[2], s = op[3];
        const size_t off = (size_t)t0 * 128 * Np + (size_t)t0 * 128;
        double* A = h->K.as<double>() + off;
        gpso_handle::ItemList* items = nullptr;
        switch (op[0]) {
            case HYB_LEAF:
                GP_TRY(hybrid_leaf(h, st, t0, n, inv8));
                break;
            case HYB_PANEL:  // L21 = A21 L11^-T
                h->hybrid_nodes++;
                GP_TRY(ensure_inverse_buffers(h));  // the products of a node use the digit buffers of the int8 inverse
                GP_TRY(oz_range_digits<OZ_HYB_S>(h, st, A, n, OZR_PANEL, s, h->rsL, h->ozL, "digits_A21"));
                GP_TRY(oz_range_digits<OZ_HYB_S>(h, st, h->Linv.as<double>() + off, n, OZR_LOWER, s, h->rsLI, h->ozLI, "digits_Linv11"));
                GP_TRY(get_hybrid_items(h, 0, s, n, &items));
                GP_TRY(oz_range_product<OZ_HYB_S>(h, st, h->ozL, h->rsL, h->ozLI, h->rsLI, items->items.as<int>(), items->rounds, n, A, nullptr,
                                                  1.0, false, "hybrid_panel"));
                break;
            case HYB_SCHUR:  // A22 -= L21 L21^T (lower tiles)
                GP_TRY(oz_range_digits<OZ_HYB_S>(h, st, A, n, OZR_PANEL, s, h->rsL, h->ozL, "digits_L21"));
                GP_TRY(get_hybrid_items(h, 1, s, n, &items));
                GP_TRY(oz_range_product<OZ_HYB_S>(h, st, h->ozL, h->rsL, h->ozL, h->rsL, items->items.as<int>(), items->rounds, n, A, nullptr,
                                                  -1.0, true, "hybrid_schur"));
                break;
            default:         // L21^-1 = -L22^-1 L21 L11^-1: the level-s merge of the recursive-doubling inverse
                GP_TRY(inverse_int8(h, st, t0, n, s, 2 * s));
                break;
        }
    }
    return 0;
}

// The reference schedule (gpso_set_factor_mode 0): one launch per step of the blocked Cholesky, then the inverse factor by
// recursive doubling, level by level.
static int factor_stepwise(gpso_handle* h, cudaStream_t st, bool inv8) {
    const int Np = h->Np, nb = h->nb;
    DenseParams P = dense_block(h->K.as<double>(), h->Linv.as<double>(), h->LinvT.as<double>(), nullptr, Np, 0, nb);
    for (int p = 0; p < nb; p++) {
        diag_factor_inverse_kernel<<<1, DIAG_THREADS, DIAG_SMEM_BYTES, st>>>(P.K, P.Linv, Np, p, h->N, h->logdet.as<double>(),
                                                                             h->info.as<int>());
        GP_TRY(check_launch(h, "diag_factor_inverse"));
        int nt = nb - 1 - p;
        if (nt > 0) {
            P.p = p;
            dense_gemm_kernel<MODE_CHOL_PANEL><<<nt, GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
            GP_TRY(check_launch(h, "chol_panel"));
            dense_gemm_kernel<MODE_CHOL_TRAIL><<<nt*(nt + 1) / 2, GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
            GP_TRY(check_launch(h, "chol_trailing"));
        }
    }
    diag_transpose_kernel<<<nb, 256, DIAG_TRANSPOSE_SMEM, st>>>(P.Linv, P.LinvT, Np);
    GP_TRY(check_launch(h, "diag_transpose"));
    if (inv8) {
        GP_TRY(inverse_int8(h, st, 0, nb, 1, nb));
    } else if (nb > 1) {
        GP_TRY(h->T.ensure((size_t)Np * Np * sizeof(double), true));
        P.T = h->T.as<double>();
        for (int s = 1; s < nb; s *= 2) {
            int cnt = 0;
            for (int q = 0; 2 * q * s < nb; q++) cnt += s * trtri_pair_vtiles(nb, s, q);
            if (cnt == 0) continue;
            P.s = s;
            dense_gemm_kernel<MODE_TRTRI_XT><<<cnt, GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
            GP_TRY(check_launch(h, "trtri_xt"));
            dense_gemm_kernel<MODE_TRTRI_Y><<<cnt, GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
            GP_TRY(check_launch(h, "trtri_y"));
        }
    }
    return 0;
}

// Gram -> Cholesky -> inverse factor -> [K_y^-1] -> a, alpha -> scalars.  Uses h->ls_host/variance/noise/c0.
static int factor_pipeline(gpso_handle* h, cudaStream_t st, bool need_kinv) {
    const int Np = h->Np, nb = h->nb;
    GP_TRY(l2_setaside(h, 0));  // the whole L2 for the tile traffic of the factorisation (see set_l2_window)
    GP_TRY(upload_lengthscales(h, st));
    if (h->linear()) CU_TRY(cudaMemcpyAsync(h->meanA.p, h->A_host, sizeof(double) * h->d, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemsetAsync(h->info.p, 0, sizeof(int), st));
    GP_TRY(scale_inputs(h, st, h->X.as<double>(), h->N, Np, h->Xs.as<double>()));
    launch_gram(h, st);
    GP_TRY(check_launch(h, "gram"));

    const bool inv8 = nb > 1 && Np <= OZ_MAX_NP && (h->inverse_mode == 2 || (h->inverse_mode == 0 && Np >= OZ_INV_MIN_NP));
    h->hybrid_nodes = 0;
    if (h->factor_mode == 0) {
        GP_TRY(factor_stepwise(h, st, inv8));
    } else {
        const bool hybrid = inv8 && h->factor_mode != 2;
        GP_TRY(hybrid_node(h, st, 0, nb, hybrid ? (h->factor_mode == 3 ? 2 : HYB_LEAF_TILES) : nb, inv8));
    }
    DenseParams P = dense_block(h->K.as<double>(), h->Linv.as<double>(), h->LinvT.as<double>(), nullptr, Np, 0, nb);
    if (need_kinv) {
        GP_TRY(h->Kinv.ensure((size_t)Np * Np * sizeof(double), true));
        P.Kinv = h->Kinv.as<double>();
        const bool int8 = Np <= OZ_MAX_NP && (h->kinv_mode == 2 || (h->kinv_mode == 0 && Np >= OZ_KINV_MIN_NP));
        if (int8) {
            GP_TRY(kinv_int8(h, st));
        } else {
            if (nb >= 2 && nb <= 4) {
                // every 128-wide k-chunk of every tile on its own SM, then a fixed-order sum (kern_dense.cuh: lauum_reduce_kernel)
                int chunks = 0;
                for (int i = 0; i < nb; i++) chunks += (i + 1) * (nb - i);
                GP_TRY(h->kinv_part.ensure((size_t)chunks * 128 * 128 * sizeof(double)));
                P.part = h->kinv_part.as<double>();
                dense_gemm_kernel<MODE_LAUUM_PART><<<chunks, GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
                GP_TRY(check_launch(h, "lauum_part"));
                lauum_reduce_kernel<<<nb*(nb + 1) / 2, 256, 0, st>>>(P.part, nb, Np, P.Kinv);
                GP_TRY(check_launch(h, "lauum_reduce"));
            } else {
                dense_gemm_kernel<MODE_LAUUM><<<nb*(nb + 1) / 2, GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
                GP_TRY(check_launch(h, "lauum"));
            }
        }
    }
    residual_kernel<<<(Np + 255) / 256, 256, 0, st>>>(h->y.as<double>(), h->c0, h->N, Np, h->resid.as<double>());
    GP_TRY(check_launch(h, "residual"));
    GP_TRY(add_linear_offset(h, st, h->X.as<double>(), h->N, -1.0, h->resid.as<double>()));  // (y - b) - x . A
    tri_matvec_kernel<true><<<(Np + 7) / 8, 256, 0, st>>>(P.Linv, h->resid.as<double>(), Np, h->a.as<double>());
    GP_TRY(check_launch(h, "trimv_lower"));
    tri_matvec_kernel<false><<<(Np + 7) / 8, 256, 0, st>>>(P.LinvT, h->a.as<double>(), Np, h->alpha.as<double>());
    GP_TRY(check_launch(h, "trimv_upper"));
    lml_scalars_kernel<<<1, 256, 0, st>>>(h->a.as<double>(), h->alpha.as<double>(), h->logdet.as<double>(), h->N, nb,
                                          h->scalars.as<double>());
    GP_TRY(check_launch(h, "lml_scalars"));
    return 0;
}

static double nlml_from_scalars(const gpso_handle* h, const double* sc) {
    return 0.5 * sc[0] + 0.5 * h->N * log(2.0 * M_PI) + sc[1];
}

// Digits per operand for the int8 product.  Error model (kern_ozaki.cuh): the fixed-point rounding of both operands
// and the neglected digit-pair levels give  std(dV_i) ~ 3 * rho_i * beta * 2^(-8S) * sqrt(N)  (rho_i = row scale of
// L^-1, beta = scale of k*), hence  |d(sum V^2)| <~ 6 * sigma_f * beta * 2^(-8S) * sqrt(N) * max_i rho_i.  The parity
// tolerance of the posterior variance is 1e-8 * kernel variance; S is the smallest digit count whose estimate is below
// OZ_TARGET of it.
static double slices_error(const gpso_handle* h, double rho_max, double beta, int S) {  // the estimate / tolerance at S digits
    const double sigma_f = sqrt(h->variance);
    const double tol = 1.0e-8 * h->variance;
    return 6.0 * sigma_f * beta * ldexp(1.0, -8 * S) * sqrt((double)h->N) * rho_max / tol;
}

static int pick_slices(const gpso_handle* h, double rho_max, double beta) {
    for (int S = 5; S < 8; S++)
        if (slices_error(h, rho_max, beta, S) <= OZ_TARGET) return S;
    return 8;
}

static double oz_beta(const gpso_handle* h) {  // 2^f with kernel variance < 2^f: k* / 2^f in [0, 1)
    return ldexp(1.0, ilogb(h->variance) + 1);
}

// The A digits of L^-1 are re-read by every candidate tile of every window (69 GB of L2 -> SM traffic per 87k-candidate
// window at N = 4096) while 2 GB of B digits stream through the same L2.  An access-policy window on the product stream
// marks the A buffer as persisting (set-aside L2) so the stream cannot evict it: only the lower-triangle tiles are ever
// touched (half of the buffer), hitRatio scales the request down when even that exceeds the set-aside.
static int set_l2_window(gpso_handle* h, void* base, size_t bytes) {
    if (!h->l2_window || h->l2_persist_max == 0 || h->l2_window_max == 0 || !base) return 0;
    GP_TRY(l2_setaside(h, h->l2_persist_max));
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof attr);
    const size_t win = std::min(bytes, h->l2_window_max);
    const double touched = 0.5 * (double)win + 1.0;
    attr.accessPolicyWindow.base_ptr = base;
    attr.accessPolicyWindow.num_bytes = win;
    attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, 0.9 * (double)h->l2_persist_max / touched);
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    CU_TRY(cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    return 0;
}

// After L^-1 is known: decide whether the int8 tensor-core product is used for this fit and build its A digit tiles.
static int prepare_ozaki(gpso_handle* h, cudaStream_t st) {
    h->oz_S = 0;
    h->oz_est = 0.0;
    h->screen_ready = false;
    h->screen_built_S = 0;
    // a kernel with Linear terms: the FP64 DMMA product (the int8 slices are scaled by a bound on |k*| that it does not have)
    bool want = !h->has_lin() && (h->predict_mode == 2 || (h->predict_mode == 0 && h->Np >= OZ_MIN_NP));
    if (!want || h->Np > OZ_MAX_NP) return 0;
    const int Np = h->Np;
    GP_TRY(h->rowscale.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->rowmax.ensure((size_t)Np * sizeof(double)));
    GP_TRY(h->rowl2.ensure((size_t)Np * sizeof(double)));
    linv_rowscale_kernel<false><<<(Np + 7) / 8, 256, 0, st>>>(h->Linv.as<double>(), Np, h->rowscale.as<double>(), h->rowmax.as<double>(),
                                                              h->rowl2.as<double>());
    GP_TRY(check_launch(h, "linv_rowscale"));
    std::vector<double> rs(Np), rl2(Np);
    CU_TRY(cudaMemcpyAsync(rs.data(), h->rowscale.p, sizeof(double) * Np, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(rl2.data(), h->rowl2.p, sizeof(double) * Np, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    double rho_max = 0.0;
    for (int i = 0; i < h->N; i++) rho_max = std::max(rho_max, rs[i]);
    if (!(rho_max > 0.0) || !std::isfinite(rho_max)) return 0;  // degenerate factor: stay on the FP64 path
    const int S = h->oz_force_slices ? h->oz_force_slices : pick_slices(h, rho_max, oz_beta(h));
    const double est = slices_error(h, rho_max, oz_beta(h), S);
    GP_TRY(h->ozA.ensure((size_t)Np * Np * S));
    DISPATCH_S(S, launch_oz_slices, h, st);
    GP_TRY(check_launch(h, "linv_slices"));
    h->oz_S = S;
    h->oz_est = est;
    GP_TRY(set_l2_window(h, h->ozA.p, (size_t)Np * Np * S));
    // screening state of the factor in force: fp32 copies of the scaled inputs and alpha, |alpha|_2 and the largest row scale
    // (both enter the error bound); the low-digit tiles of L^-1 are built by the first screened call (their digit count adapts)
    h->rho_max = rho_max;
    h->rho_l2sq = 0.0;
    h->linv_frob2 = 0.0;
    h->linv_rowl2_max = 0.0;
    for (int i = 0; i < h->N; i++) {
        h->rho_l2sq += rs[i] * rs[i];
        h->linv_frob2 += rl2[i];
        h->linv_rowl2_max = std::max(h->linv_rowl2_max, sqrt(rl2[i]));
    }
    if (h->screen_mode != 0 && Np >= SCREEN_MIN_NP) {
        GP_TRY(h->Xs32.ensure((size_t)h->dx() * Np * sizeof(float)));
        GP_TRY(h->alpha32.ensure((size_t)Np * sizeof(float)));
        screen_convert_kernel<<<(h->dx() * Np + 255) / 256, 256, 0, st>>>(h->Xs.as<double>(), h->alpha.as<double>(), h->dx(), Np,
                                                                       h->Xs32.as<float>(), h->alpha32.as<float>());
        GP_TRY(check_launch(h, "screen_convert"));
        std::vector<double> al(Np);
        CU_TRY(cudaMemcpyAsync(al.data(), h->alpha.p, sizeof(double) * Np, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        double s2 = 0.0;
        for (int i = 0; i < h->N; i++) s2 += al[i] * al[i];
        h->alpha_l2 = sqrt(s2);
        h->screen_ready = std::isfinite(h->alpha_l2);
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// library
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int gpso_version(void) { return 1; }
extern "C" const char* gpso_last_error(void) { return g_last_error.c_str(); }
extern "C" int gpso_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(GPSO_E_NOGPU, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    return n;
}

static int init_handle(gpso_handle* h, int device, int kernel_id, int ard, int mean_id, const cudaDeviceProp& prop) {
    h->device = device;
    h->kernel_id = kernel_id;
    h->ard = ard ? 1 : 0;
    h->mean_id = mean_id;
    h->nsm = prop.multiProcessorCount;
    h->l2_persist_max = (size_t)std::max(0, prop.persistingL2CacheMaxSize);
    h->l2_window_max = (size_t)std::max(0, prop.accessPolicyMaxWindowSize);
    // h->stream carries the tensor-core product kernels: highest priority, so that its persistent CTAs are placed before
    // the (default-priority) cross-covariance blocks of the next window when both become eligible at the same time
    int prio_least = 0, prio_greatest = 0;
    CU_TRY(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
    CU_TRY(cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_greatest));
    CU_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
    CU_TRY(cudaEventCreateWithFlags(&h->ev_start, cudaEventDisableTiming));
    CU_TRY(cudaEventCreateWithFlags(&h->ev_probe, cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
        CU_TRY(cudaEventCreateWithFlags(&h->ev_copy[i], cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&h->ev_used[i], cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&h->ev_xcov[i], cudaEventDisableTiming));
        CU_TRY(cudaEventCreateWithFlags(&h->ev_free[i], cudaEventDisableTiming));
    }
    CU_TRY(cudaEventCreate(&h->ev_t0));
    CU_TRY(cudaEventCreate(&h->ev_t1));
    // room for the gradient record of gpso_neg_lml_grad: 4 + partial sums (up to MAX_LS + 3, a sum kernel's components up to
    // MAX_LS + 3 MAX_SUM together) + the linear mean's A (MAX_LS)
    CU_TRY(cudaHostAlloc((void**)&h->host_rec, (2 * MAX_LS + 16 + 3 * MAX_SUM) * sizeof(double), cudaHostAllocDefault));
    GP_TRY(configure_kernels_once(device));
    return 0;
}

extern "C" int gpso_destroy(gpso_handle* h);

static int create_handle(int device, int kernel_id, int ard, int mean_id, const SumTable& sum, const int* sum_ard, gpso_handle** out,
                         int pmask = 0);

extern "C" int gpso_create(int device, int kernel_id, int ard, int mean_id, gpso_handle** out) {
    if (!out) return fail(GPSO_E_BADARG, "gpso_create: out is null");
    *out = nullptr;
    // GPSO_KERNEL_SUM and GPSO_KERNEL_PRODUCT have components: gpso_create_sum, gpso_create_product
    if ((kernel_id < 0 || kernel_id > KERNEL_RQ) && kernel_id != GPSO_KERNEL_LINEAR) return fail(GPSO_E_BADARG, "gpso_create: unknown kernel id");
    if (mean_id < GPSO_MEAN_ZERO || mean_id > GPSO_MEAN_LINEAR) return fail(GPSO_E_BADARG, "gpso_create: unknown mean id");
    if (kernel_id == GPSO_KERNEL_LINEAR) {  // a one-component sum from the start: the row layout of a sum with Linear terms
        if (ard != 0 && ard != 1) return fail(GPSO_E_BADARG, "gpso_create: the Linear kernel's ard flag must be 0 or 1");
        SumTable tab = {};
        tab.n = 1;
        tab.fam[0] = KERNEL_LINEAR;
        tab.var[0] = tab.alpha[0] = 1.0;
        GP_TRY(create_handle(device, KERNEL_SUM, 0, mean_id, tab, &ard, out));
        (*out)->lin_mask = 1;
        (*out)->bare_lin = true;
        return 0;
    }
    return create_handle(device, kernel_id, ard, mean_id, SumTable{}, nullptr, out);
}

// The arguments of gpso_create_sum, gpso_create_product and gpso_create_combination: n components (1..MAX_SUM) of the five
// families, ARD flags 0 / 1; with base_ids (gpso_create_combination only) a component of id GPSO_KERNEL_PERIODIC is periodic with
// the base base_ids[c] (SE or RQ) and the period ARD flag period_ard[c].
static int component_table(const char* who, int n, const int* kernel_ids, const int* ard, int mean_id, gpso_handle** out,
                           SumTable& tab, const int* base_ids = nullptr, const int* period_ard = nullptr, int* pmask = nullptr,
                           int* lmask = nullptr) {
    const std::string w(who);
    if (!out) return fail(GPSO_E_BADARG, w + ": out is null");
    *out = nullptr;
    if (n < 1 || n > MAX_SUM) return fail(GPSO_E_BADARG, w + ": the number of components must be in 1..4");
    if (!kernel_ids || !ard) return fail(GPSO_E_BADARG, w + ": null argument");
    if (mean_id < GPSO_MEAN_ZERO || mean_id > GPSO_MEAN_LINEAR) return fail(GPSO_E_BADARG, w + ": unknown mean id");
    tab = {};
    tab.n = n;
    int pm = 0, lm = 0;
    for (int c = 0; c < n; c++) {
        const bool per = base_ids && kernel_ids[c] == GPSO_KERNEL_PERIODIC;
        const bool lin = lmask && kernel_ids[c] == GPSO_KERNEL_LINEAR;
        if (!per && !lin && (kernel_ids[c] < 0 || kernel_ids[c] > KERNEL_RQ)) return fail(GPSO_E_BADARG, w + ": unknown component kernel id");
        if (per && base_ids[c] != KERNEL_SE && base_ids[c] != KERNEL_RQ)
            return fail(GPSO_E_BADARG, w + ": a periodic component's base must be SquaredExponential or RationalQuadratic");
        if ((ard[c] != 0 && ard[c] != 1) || (per && period_ard[c] != 0 && period_ard[c] != 1))
            return fail(GPSO_E_BADARG, w + ": ard flags must be 0 or 1");
        tab.fam[c] = per ? base_ids[c] : kernel_ids[c];
        pm |= per ? 1 << c : 0;
        lm |= lin ? 1 << c : 0;
        tab.var[c] = 1.0;
        tab.alpha[c] = 1.0;
    }
    if (pmask) *pmask = pm;
    if (lmask) *lmask = lm;
    return 0;
}

extern "C" int gpso_create_sum(int device, int n, const int* kernel_ids, const int* ard, int mean_id, gpso_handle** out) {
    SumTable sum;
    GP_TRY(component_table("gpso_create_sum", n, kernel_ids, ard, mean_id, out, sum));
    return create_handle(device, KERNEL_SUM, 0, mean_id, sum, ard, out);
}

extern "C" int gpso_create_combination(int device, int kind, int n, const int* kernel_ids, const int* ard, const int* base_ids,
                                       const int* period_ard, int mean_id, gpso_handle** out) {
    if (kind != KERNEL_SUM && kind != KERNEL_PRODUCT) {
        if (out) *out = nullptr;
        return fail(GPSO_E_BADARG, "gpso_create_combination: kind must be GPSO_KERNEL_SUM or GPSO_KERNEL_PRODUCT");
    }
    if (!base_ids || !period_ard) {
        if (out) *out = nullptr;
        return fail(GPSO_E_BADARG, "gpso_create_combination: null argument");
    }
    if (kind == KERNEL_PRODUCT && kernel_ids && n >= 1 && n <= MAX_SUM)
        for (int c = 0; c < n; c++)
            if (kernel_ids[c] == GPSO_KERNEL_LINEAR) {
                if (out) *out = nullptr;
                return fail(GPSO_E_BADARG, "gpso_create_combination: a Linear kernel cannot be a factor of a product");
            }
    SumTable tab;
    int pmask = 0, lmask = 0;
    GP_TRY(component_table("gpso_create_combination", n, kernel_ids, ard, mean_id, out, tab, base_ids, period_ard, &pmask,
                           kind == KERNEL_SUM ? &lmask : nullptr));
    GP_TRY(create_handle(device, kind, 0, mean_id, tab, ard, out, pmask));
    (*out)->lin_mask = lmask;
    for (int c = 0; c < n; c++) (*out)->sum_per_ard[c] = (pmask >> c & 1) ? period_ard[c] : 0;
    return 0;
}

extern "C" int gpso_create_product(int device, int n, const int* kernel_ids, const int* ard, int mean_id, gpso_handle** out) {
    SumTable tab;
    GP_TRY(component_table("gpso_create_product", n, kernel_ids, ard, mean_id, out, tab));
    return create_handle(device, KERNEL_PRODUCT, 0, mean_id, tab, ard, out);
}

extern "C" int gpso_create_periodic(int device, int base_id, int ard, int period_ard, int mean_id, gpso_handle** out) {
    if (!out) return fail(GPSO_E_BADARG, "gpso_create_periodic: out is null");
    *out = nullptr;
    if (base_id != KERNEL_SE && base_id != KERNEL_RQ)
        return fail(GPSO_E_BADARG, "gpso_create_periodic: the base kernel must be SquaredExponential or RationalQuadratic");
    if ((ard != 0 && ard != 1) || (period_ard != 0 && period_ard != 1))
        return fail(GPSO_E_BADARG, "gpso_create_periodic: ard flags must be 0 or 1");
    if (mean_id < GPSO_MEAN_ZERO || mean_id > GPSO_MEAN_LINEAR) return fail(GPSO_E_BADARG, "gpso_create_periodic: unknown mean id");
    GP_TRY(create_handle(device, base_id, ard, mean_id, SumTable{}, nullptr, out));
    (*out)->periodic = true;
    (*out)->per_ard = period_ard;
    return 0;
}

static int create_handle(int device, int kernel_id, int ard, int mean_id, const SumTable& sum, const int* sum_ard, gpso_handle** out,
                         int pmask) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return fail(GPSO_E_NOGPU, "gpso_create: no CUDA device available");
    if (device < 0 || device >= n) return fail(GPSO_E_BADARG, "gpso_create: device index out of range");
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        char b[256];
        snprintf(b, sizeof b, "gpso_create: device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU", device, prop.name, prop.major,
                 prop.minor);
        return fail(GPSO_E_NOGPU, b);
    }
    CU_TRY(cudaSetDevice(device));
    gpso_handle* h = new gpso_handle();
    h->sum = sum;
    h->srow.pmask = pmask;
    for (int c = 0; c < sum.n; c++) {
        h->sum_ard[c] = sum_ard[c];
        h->sum_per[c] = pmask >> c & 1;
        h->prod_var[c] = sum.var[c];
    }
    int rc = init_handle(h, device, kernel_id, ard, mean_id, prop);
    if (rc != 0) {
        gpso_destroy(h);  // releases whatever was created before the failure (null streams / events are skipped)
        return rc;
    }
    *out = h;
    return 0;
}


extern "C" int gpso_destroy(gpso_handle* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    // a handle whose creation failed half-way arrives here too: every stream / event may still be null
    // the buffers go back to the pool, not to the driver: nothing may be in flight on them, whichever stream the caller used
    cudaDeviceSynchronize();
    auto drop = [](cudaEvent_t e) {
        if (e) cudaEventDestroy(e);
    };
    for (int i = 0; i < 2; i++) {
        drop(h->ev_copy[i]);
        drop(h->ev_used[i]);
        drop(h->ev_xcov[i]);
        drop(h->ev_free[i]);
    }
    drop(h->ev_start);
    drop(h->ev_probe);
    drop(h->ev_t0);
    drop(h->ev_t1);
    for (cudaEvent_t e : h->prof_events) drop(e);
    for (cudaEvent_t e : h->prod_events) drop(e);
    for (cudaEvent_t e : h->trace_events) drop(e);
    for (cudaStream_t st : {h->aux_stream, h->stream, h->copy_stream})
        if (st) cudaStreamDestroy(st);
    if (h->host_rec) cudaFreeHost(h->host_rec);
    delete h;  // ~DevBuf releases every device buffer of the handle
    cudaGetLastError();
    return 0;
}

extern "C" int gpso_set_data(gpso_handle* h, const double* X_host, const double* y_host, int N, int d) {
    if (!h || !X_host || !y_host) return fail(GPSO_E_BADARG, "gpso_set_data: null argument");
    if (N <= 0 || d <= 0) return fail(GPSO_E_BADARG, "gpso_set_data: N and d must be positive");
    if (d > MAX_LS) return fail(GPSO_E_BADARG, "gpso_set_data: input dimension above the supported maximum (64)");
    if (h->nmap) {
        if (h->nmap != h->sum.n) return fail(GPSO_E_BADARG, "gpso_set_data: the active dims map has a leaf count other than the kernel's");
        for (int col : h->map_cols)
            if (col >= d) return fail(GPSO_E_BADARG, "gpso_set_data: an active dim is not below the input dimension");
        if (h->rows_for(d) > MAX_LS)
            return fail(GPSO_E_BADARG, "gpso_set_data: the rows of all components (their active columns, twice for a periodic one) may not exceed 64");
    } else if (h->composite() && h->sum.n * d > MAX_LS)
        return fail(GPSO_E_BADARG, h->is_sum() ? "gpso_set_data: a sum kernel supports components x input dimension up to 64"
                                               : "gpso_set_data: a product kernel supports factors x input dimension up to 64");
    if (h->periodic && 2 * d > MAX_LS)
        return fail(GPSO_E_BADARG, "gpso_set_data: a periodic kernel embeds each input dimension in 2 rows: input dimension up to 32");
    if (h->emb() && h->rows_for(d) > MAX_LS)
        return fail(GPSO_E_BADARG, "gpso_set_data: the rows of all components (d each, 2d for a periodic component) may not exceed 64");
    GP_TRY(set_device(h));
    CU_TRY(cudaStreamSynchronize(h->stream));
    GP_TRY(ensure_shape(h, N, d));
    CU_TRY(cudaMemcpyAsync(h->X.p, X_host, sizeof(double) * (size_t)N * d, cudaMemcpyHostToDevice, h->stream));
    CU_TRY(cudaMemsetAsync(h->y.p, 0, sizeof(double) * h->Np, h->stream));
    CU_TRY(cudaMemcpyAsync(h->y.p, y_host, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, h->stream));
    // the raw coordinates the periodic components' gradient reads: X itself, or with a map their active columns, gathered
    h->raw = {};
    h->raw.width = d;
    std::vector<double> xg;
    if (h->nmap) {
        h->raw.width = 0;
        for (int c = 0; c < h->sum.n; c++)
            if (h->sum_per[c]) {
                h->raw.off[c] = h->raw.width;
                h->raw.width += h->map_n[c];
            }
        xg.resize((size_t)N * h->raw.width);
        for (int i = 0; i < N; i++)
            for (int c = 0; c < h->sum.n; c++)
                for (int j = 0; h->sum_per[c] && j < h->map_n[c]; j++)
                    xg[(size_t)i * h->raw.width + h->raw.off[c] + j] = X_host[(size_t)i * d + h->map_cols[h->map_off[c] + j]];
        if (!xg.empty()) {
            GP_TRY(h->Xg.ensure(xg.size() * sizeof(double)));
            CU_TRY(cudaMemcpyAsync(h->Xg.p, xg.data(), xg.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        }
    }
    CU_TRY(cudaStreamSynchronize(h->stream));
    h->have_data = true;
    h->factorized = false;
    return 0;
}

extern "C" int gpso_set_active_dims(gpso_handle* h, int n, const int* counts, const int* dims) {
    if (!h) return fail(GPSO_E_BADARG, "gpso_set_active_dims: null handle");
    if (n < 0 || n > MAX_SUM) return fail(GPSO_E_BADARG, "gpso_set_active_dims: the number of leaves must be in 0..4");
    if (n > 0 && (!counts || !dims)) return fail(GPSO_E_BADARG, "gpso_set_active_dims: null argument");
    int total = 0;
    for (int c = 0; c < n; c++) {
        if (counts[c] < 1 || counts[c] > MAX_LS) return fail(GPSO_E_BADARG, "gpso_set_active_dims: each leaf needs 1..64 columns");
        total += counts[c];
    }
    for (int i = 0; i < total; i++)
        if (dims[i] < 0) return fail(GPSO_E_BADARG, "gpso_set_active_dims: negative column index");
    GP_TRY(set_device(h));
    CU_TRY(cudaStreamSynchronize(h->stream));
    if (n == 0 && h->bare_kid >= 0) {  // back to the bare kernel the map turned into a one-component sum
        h->kernel_id = h->bare_kid;
        h->ard = h->bare_ard;
        h->periodic = h->sum_per[0] != 0;
        h->per_ard = h->bare_per_ard;
        h->sum = SumTable{};
        h->srow = SumRows{};
        h->sum_ard[0] = h->sum_per[0] = h->sum_per_ard[0] = 0;
        h->bare_kid = -1;
    } else if (n > 0 && !h->composite()) {  // a bare kernel: a one-component sum, which packs and computes as the bare kernel does
        h->bare_kid = h->kernel_id;
        h->bare_ard = h->ard;
        h->bare_per_ard = h->per_ard;
        h->sum = SumTable{};
        h->sum.n = 1;
        h->sum.fam[0] = h->kernel_id;
        h->sum.var[0] = h->sum.alpha[0] = 1.0;
        h->sum_ard[0] = h->ard;
        h->sum_per[0] = h->periodic ? 1 : 0;
        h->sum_per_ard[0] = h->periodic ? h->per_ard : 0;
        h->srow.pmask = h->sum_per[0];
        h->kernel_id = KERNEL_SUM;
        h->ard = h->per_ard = 0;
        h->periodic = false;
    }
    h->nmap = n;
    h->map_cols.assign(dims, dims + (n ? total : 0));
    for (int c = 0; c < MAX_SUM; c++) {
        h->map_n[c] = c < n ? counts[c] : 0;
        h->map_off[c + 1] = h->map_off[c] + h->map_n[c];
    }
    // the rows, the packed vector's length and the scaled inputs follow the map: the data has to be set again
    h->have_data = false;
    h->factorized = false;
    return 0;
}

static void load_mean(gpso_handle* h, const double* m) {  // the mean function's entries of the packed vector
    if (h->linear()) {
        for (int k = 0; k < h->d; k++) h->A_host[k] = m[k];
        h->c0 = m[h->d];
    } else {
        h->c0 = (h->mean_id == GPSO_MEAN_CONSTANT) ? m[0] : 0.0;
    }
}

static int load_theta(gpso_handle* h, const double* theta, int p, const char* who, bool allow_zero = false) {
    if (p != h->n_params()) {
        char b[256];
        snprintf(b, sizeof b, "%s: expected %d hyper-parameters, got %d", who, h->n_params(), p);
        return fail(GPSO_E_BADARG, b);
    }
    auto positive = [&](double v) { return v > 0.0 || (allow_zero && v == 0.0); };
    if (h->composite()) {
        // per component [alpha], lengthscale(s), variance; the prior variance is their variances' fp64 sum (a product: product)
        // in component order
        double var_tot = 0.0;
        for (int c = 0; c < h->sum.n; c++) {
            if (h->sum.fam[c] == KERNEL_RQ) {
                if (!positive(theta[0])) return fail(GPSO_E_BADARG, std::string(who) + ": alpha must be positive");
                h->sum.alpha[c] = *theta++;
            }
            const int nl = h->comp_ls(c);
            if (h->comp_lin(c)) {  // variance(s) only, held on the component's rows; the constant part of the prior variance is the others'
                for (int i = 0; i < nl; i++)
                    if (!positive(theta[i])) return fail(GPSO_E_BADARG, std::string(who) + ": variances must be positive");
                for (int k = 0; k < h->cdim(c, h->d); k++) h->ls_host[h->ls_off(c) + k] = theta[nl > 1 ? k : 0];
                h->sum.var[c] = theta[0];
                theta += nl;
                continue;
            }
            for (int i = 0; i < nl; i++)
                if (!positive(theta[i])) return fail(GPSO_E_BADARG, std::string(who) + ": lengthscale must be positive");
            for (int k = 0; k < h->cdim(c, h->d); k++) h->ls_host[h->ls_off(c) + k] = theta[nl > 1 ? k : 0];
            if (!positive(theta[nl])) return fail(GPSO_E_BADARG, std::string(who) + ": variances must be positive");
            if (h->is_product()) {
                h->prod_var[c] = theta[nl];
                var_tot = (c == 0) ? theta[nl] : var_tot * theta[nl];
            } else {
                h->sum.var[c] = theta[nl];
                var_tot = (var_tot == 0.0) ? theta[nl] : var_tot + theta[nl];
            }
            for (int i = 0; i < h->comp_np(c); i++) {  // a periodic component's period(s) follow its variance
                if (!positive(theta[nl + 1 + i])) return fail(GPSO_E_BADARG, std::string(who) + ": period must be positive");
                h->comp_p[c][i] = theta[nl + 1 + i];
            }
            theta += nl + 1 + h->comp_np(c);
        }
        h->variance = var_tot;
        if (h->is_product())  // the table: var_prod on the first factor, unit variance on the others
            for (int c = 0; c < h->sum.n; c++) h->sum.var[c] = (c == 0) ? var_tot : 1.0;
        h->noise = theta[0];
        if (!(h->noise > 0.0)) return fail(GPSO_E_BADARG, std::string(who) + ": variances must be positive");
        load_mean(h, theta + 1);
        return 0;
    }
    if (h->n_rq()) {
        if (!(theta[0] > 0.0) && !(allow_zero && theta[0] == 0.0))
            return fail(GPSO_E_BADARG, std::string(who) + ": alpha must be positive");
        h->rq_alpha = theta[0];
        theta++;
    }
    int nl = h->n_ls();
    for (int i = 0; i < nl; i++) {
        if (!(theta[i] > 0.0) && !(allow_zero && theta[i] == 0.0))
            return fail(GPSO_E_BADARG, std::string(who) + ": lengthscale must be positive");
        h->ls_host[i] = theta[i];
    }
    h->variance = theta[nl];
    const int np = h->n_per();  // a periodic kernel's period(s) follow the variance ('base_kernel' < 'period')
    for (int i = 0; i < np; i++) {
        if (!positive(theta[nl + 1 + i])) return fail(GPSO_E_BADARG, std::string(who) + ": period must be positive");
        h->per_p[i] = theta[nl + 1 + i];
    }
    h->noise = theta[nl + 1 + np];
    if (!(h->variance > 0.0 || (allow_zero && h->variance == 0.0)) || !(h->noise > 0.0))
        return fail(GPSO_E_BADARG, std::string(who) + ": variances must be positive");
    load_mean(h, theta + nl + 2 + np);
    return 0;
}

// Sum kernel: the gradient of a sum with respect to one component's parameters is that component's own gradient, so the
// family's lml_grad_kernel runs once per component (its scaled inputs Xs_c, variance and alpha) into the component's own block
// of partial sums, and each block is chained through the component's sigmoids.
// Product kernel: dK/dtheta_c = P_-c dk_c/dtheta_c, all factors' entries from one lml_grad_product_kernel launch and one
// reduction, whatever the ARD flags: [s_K, sum_i W_ii, then per factor its lengthscale entries and (RationalQuadratic) alpha];
// d/d var_c = s_K / var_c for every factor.  The noise and mean entries are taken once.
static int neg_lml_grad_composite(gpso_handle* h, const double* u, int p, double* f_host, double* grad_host) {
    const int K = h->n_kernel_params();
    std::vector<double> theta(p);
    for (int i = 0; i < K; i++) theta[i] = softplus(u[i]);
    theta[K] = NOISE_FLOOR + softplus(u[K]);
    for (int i = 0; i < h->n_mean(); i++) theta[K + 1 + i] = u[K + 1 + i];
    GP_TRY(load_theta(h, theta.data(), p, "gpso_neg_lml_grad", true));
    h->factorized = false;
    cudaStream_t st = h->stream;
    CU_TRY(cudaEventRecord(h->ev_t0, st));
    GP_TRY(factor_pipeline(h, st, true));
    const int nb64 = h->Np / CT;
    const int nblk = nb64 * (nb64 + 1) / 2;
    // where component c's entries sit in the reduced partial sums: its variance entry (s_K), lengthscales and alpha
    // a periodic component's entries are per dimension for its lengthscales and its periods: 2d entries before its alpha
    int ik[MAX_SUM], il[MAX_SUM], ia[MAX_SUM], stride[MAX_SUM], off[MAX_SUM + 1] = {0};
    if (h->is_product()) off[0] = 2;
    for (int c = 0; c < h->sum.n; c++) {
        // a Linear component: one entry per column, [0, sum_i W_ii, x_j^T W x_j (j < k)] (lml_grad_linear_kernel)
        const int nls = h->sum_per[c] ? 2 * h->cdim(c, h->d) : h->comp_lin(c) ? h->cdim(c, h->d) : h->comp_ls(c),
                  rq = h->sum.fam[c] == KERNEL_RQ;
        stride[c] = (h->is_product() ? 0 : 2) + nls + rq;
        ik[c] = h->is_product() ? 0 : off[c];
        il[c] = h->is_product() ? off[c] : off[c] + 2;
        ia[c] = il[c] + nls;
        off[c + 1] = off[c] + stride[c];
    }
    const int total = off[h->sum.n];
    const int nA = h->linear() ? h->d : 0;
    GP_TRY(h->gpart.ensure((size_t)nblk * total * sizeof(double)));
    GP_TRY(h->gout.ensure((size_t)(total + 4 + nA) * sizeof(double)));
    if (h->is_product()) {
        int ard_mask = 0, nard = 0;  // a periodic factor always takes a weight slot
        for (int c = 0; c < h->sum.n; c++) {
            const int slot = h->sum_ard[c] | h->sum_per[c];
            ard_mask |= slot << c;
            nard += slot;
        }
        const size_t smem = ((size_t)2 * h->dx() * CT + (h->emb() ? (size_t)2 * h->raw.width * CT : 0) + (size_t)nard * CT * CT) * sizeof(double);
        if (h->emb())
            lml_grad_product_periodic_kernel<<<nblk, 256, smem, st>>>(h->Xs.as<double>(), h->alpha.as<double>(), h->Kinv.as<double>(),
                                                                      h->N, h->Np, ard_mask, h->gpart.as<double>(), total, h->sum,
                                                                      h->nmap ? h->Xg.as<double>() : h->X.as<double>(), h->srow, h->raw);
        else
            lml_grad_product_kernel<<<nblk, 256, smem, st>>>(h->Xs.as<double>(), h->alpha.as<double>(), h->Kinv.as<double>(), h->N,
                                                             h->d, h->Np, ard_mask, h->gpart.as<double>(), total, h->sum);
        GP_TRY(check_launch(h, "lml_grad_product"));
        reduce_partials_kernel<<<total, 256, 0, st>>>(h->gpart.as<double>(), nblk, total, h->gout.as<double>());
        GP_TRY(check_launch(h, "reduce_partials"));
    } else {
        for (int c = 0; c < h->sum.n; c++) {
            double* part = h->gpart.as<double>() + (size_t)nblk * off[c];
            const double* Xs_c = h->Xs.as<double>() + (size_t)h->srow.off[c] * h->Np;
            const int k = h->cdim(c, h->d);
            if (h->comp_lin(c)) {
                lml_grad_linear_kernel<<<nblk, 256, linear_grad_smem(k), st>>>(Xs_c, h->alpha.as<double>(), h->Kinv.as<double>(), h->N, k,
                                                                               h->Np, part, stride[c]);
                h->launches++;
            } else if (h->sum_per[c]) {
                const double* Xr = h->nmap ? h->Xg.as<double>() + h->raw.off[c] : h->X.as<double>();
                KernelIds<KERNEL_SE, KERNEL_RQ>::with(h->sum.fam[c], [&](auto kid) {
                    lml_grad_periodic_kernel<kid><<<nblk, 256, periodic_grad_smem(k), st>>>(
                        Xs_c, Xr, h->alpha.as<double>(), h->Kinv.as<double>(), h->N, k, h->Np, h->sum.var[c], h->sum.alpha[c], part,
                        stride[c], h->raw.width);
                });
                h->launches++;
            } else {
                launch_grad(h, st, nblk, stride[c], h->sum.fam[c], h->sum_ard[c], Xs_c, k, h->sum.var[c], h->sum.alpha[c], part);
            }
            if (cudaGetLastError() != cudaSuccess) return fail(GPSO_E_CUDA, "launch of lml_grad failed");
            reduce_partials_kernel<<<stride[c], 256, 0, st>>>(part, nblk, stride[c], h->gout.as<double>() + off[c]);
            GP_TRY(check_launch(h, "reduce_partials"));
        }
    }
    if (nA) {
        linear_grad_kernel<<<nA, 256, 0, st>>>(h->X.as<double>(), h->alpha.as<double>(), h->N, h->d, h->gout.as<double>() + total);
        GP_TRY(check_launch(h, "linear_grad"));
    }
    CU_TRY(cudaEventRecord(h->ev_t1, st));
    double* rec = h->host_rec;
    CU_TRY(cudaMemcpyAsync(rec, h->scalars.p, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(rec + 3, h->info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(rec + 4, h->gout.p, sizeof(double) * (total + nA), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    const double* sc = rec;
    int info = 0;
    memcpy(&info, rec + 3, sizeof(int));
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1);
    h->last_ms[0] = ms;
    h->last_ms[1] = h->last_ms[2] = h->last_ms[3] = 0;
    GP_TRY(pivot_status(info, "Gram matrix"));
    *f_host = nlml_from_scalars(h, sc);
    const double* g = rec + 4;
    int pos = 0;
    for (int c = 0; c < h->sum.n; c++) {
        if (h->sum.fam[c] == KERNEL_RQ) {  // alpha == 0 only when softplus underflowed: the entry is 0, as for the variance
            grad_host[pos] = h->sum.alpha[c] > 0.0 ? -(0.5 * g[ia[c]]) * sigmoid(u[pos]) : 0.0;
            pos++;
        }
        const int nl = h->comp_ls(c), np = h->comp_np(c), d = h->cdim(c, h->d), lo = h->ls_off(c);
        if (h->comp_lin(c)) {  // dK/dvar_j = x_j x_j^T: d(-LML)/dvar_j = -0.5 x_j^T W x_j; a scalar variance takes the sum over j
            const double* Q = g + il[c];
            // the rows are x_j / l_j with l_j^2 = 1 / var_j: x_j^T W x_j = Q_j / var_j (var_j = 0 only where softplus underflowed,
            // with the chain factor sigmoid(u) 0 too: the entry is 0 there)
            double Qs = 0.0;
            for (int k = 0; k < d; k++) Qs += Q[k] / h->ls_host[lo + k];
            for (int i = 0; i < nl; i++) {
                const double v = h->ls_host[lo + i];
                grad_host[pos + i] = v > 0.0 ? -(0.5 * (nl > 1 ? Q[i] / v : Qs)) * sigmoid(u[pos + i]) : 0.0;
            }
            pos += nl;
            continue;
        }
        if (h->sum_per[c]) {  // per-dimension entries L(d), Q(d) as for a bare periodic kernel (gpso_neg_lml_grad)
            const double* L = g + il[c];
            const double* Q = g + il[c] + d;
            double Ls = 0.0, Qs = 0.0;
            for (int k = 0; k < d; k++) {
                Ls += L[k];
                Qs += Q[k];
            }
            for (int i = 0; i < nl; i++) grad_host[pos + i] = -(0.5 * (nl > 1 ? L[i] : Ls) / h->ls_host[lo + i]) * sigmoid(u[pos + i]);
            for (int i = 0; i < np; i++)
                grad_host[pos + nl + 1 + i] =
                    -(M_PI * (np > 1 ? Q[i] : Qs) / (h->comp_p[c][i] * h->comp_p[c][i])) * sigmoid(u[pos + nl + 1 + i]);
        } else {
            for (int i = 0; i < nl; i++) grad_host[pos + i] = -(0.5 * g[il[c] + i] / h->ls_host[lo + i]) * sigmoid(u[pos + i]);
        }
        pos += nl;
        const double var_c = h->comp_var(c);
        grad_host[pos] = var_c > 0.0 ? -(0.5 * g[ik[c]] / var_c) * sigmoid(u[pos]) : 0.0;
        pos += 1 + np;
    }
    grad_host[pos] = -(0.5 * g[1]) * sigmoid(u[pos]);  // sum_i W_ii, taken from the first component's block
    if (h->mean_id == GPSO_MEAN_CONSTANT) grad_host[pos + 1] = -sc[2];
    if (nA) {
        for (int k = 0; k < nA; k++) grad_host[pos + 1 + k] = -rec[4 + total + k];
        grad_host[pos + 1 + nA] = -sc[2];
    }
    return 0;
}

extern "C" int gpso_neg_lml_grad(gpso_handle* h, const double* u, int p, double* f_host, double* grad_host) {
    if (!h || !u || !f_host || !grad_host) return fail(GPSO_E_BADARG, "gpso_neg_lml_grad: null argument");
    if (!h->have_data) return fail(GPSO_E_STATE, "gpso_neg_lml_grad: call gpso_set_data first");
    if (p != h->n_params()) return fail(GPSO_E_BADARG, "gpso_neg_lml_grad: wrong number of hyper-parameters");
    GP_TRY(set_device(h));
    if (h->composite()) return neg_lml_grad_composite(h, u, p, f_host, grad_host);
    const int nl = h->n_ls(), na = h->n_rq(), np = h->n_per();
    std::vector<double> theta(p);
    for (int i = 0; i < na; i++) theta[i] = softplus(u[i]);  // alpha: positive, no floor
    grad_host += na;  // the shared layout after alpha
    u += na;
    for (int i = 0; i < nl; i++) theta[na + i] = softplus(u[i]);
    theta[na + nl] = softplus(u[nl]);
    for (int i = 0; i < np; i++) theta[na + nl + 1 + i] = softplus(u[nl + 1 + i]);  // period(s): positive, no floor
    theta[na + nl + 1 + np] = NOISE_FLOOR + softplus(u[nl + 1 + np]);
    for (int i = 0; i < h->n_mean(); i++) theta[na + nl + 2 + np + i] = u[nl + 2 + np + i];  // unconstrained
    // softplus(u) underflows to exactly 0 for u < -745 and L-BFGS-B line searches do probe such points: like GPflow, evaluate
    // them (kernel variance 0 -> K_y = noise * I; lengthscale 0 -> NaN objective) instead of rejecting the call
    GP_TRY(load_theta(h, theta.data(), p, "gpso_neg_lml_grad", true));
    h->factorized = false;
    cudaStream_t st = h->stream;
    CU_TRY(cudaEventRecord(h->ev_t0, st));
    GP_TRY(factor_pipeline(h, st, true));
    const int nb64 = h->Np / CT;
    const int nblk = nb64 * (nb64 + 1) / 2;
    // a periodic kernel's partial sums are per dimension for the lengthscales and the periods alike: [s_K, tr, L(d), Q(d), (alpha)]
    const int stride = 2 + (h->periodic ? 2 * h->d : nl) + na;
    const int nA = h->linear() ? h->d : 0;  // X^T alpha follows the reduced partial sums in gout
    GP_TRY(h->gpart.ensure((size_t)nblk * stride * sizeof(double)));
    GP_TRY(h->gout.ensure((size_t)(stride + 4 + nA) * sizeof(double)));
    if (h->periodic) {
        KernelIds<KERNEL_SE, KERNEL_RQ>::with(h->kernel_id, [&](auto kid) {
            lml_grad_periodic_kernel<kid><<<nblk, 256, periodic_grad_smem(h->d), st>>>(
                h->Xs.as<double>(), h->X.as<double>(), h->alpha.as<double>(), h->Kinv.as<double>(), h->N, h->d, h->Np, h->variance,
                h->rq_alpha, h->gpart.as<double>(), stride, h->d);
        });
        GP_TRY(check_launch(h, "lml_grad_periodic"));
    } else {
        launch_grad(h, st, nblk, stride, h->kernel_id, h->ard, h->Xs.as<double>(), h->d, h->variance, h->rq_alpha, h->gpart.as<double>());
        if (cudaGetLastError() != cudaSuccess) return fail(GPSO_E_CUDA, "launch of lml_grad failed");
    }
    reduce_partials_kernel<<<stride, 256, 0, st>>>(h->gpart.as<double>(), nblk, stride, h->gout.as<double>());
    GP_TRY(check_launch(h, "reduce_partials"));
    if (nA) {
        linear_grad_kernel<<<nA, 256, 0, st>>>(h->X.as<double>(), h->alpha.as<double>(), h->N, h->d, h->gout.as<double>() + stride);
        GP_TRY(check_launch(h, "linear_grad"));
    }
    CU_TRY(cudaEventRecord(h->ev_t1, st));
    // one pinned record [scalars(3) | info | gradient partial sums(stride) | X^T alpha(nA)]: three truly asynchronous copies, one wait
    double* rec = h->host_rec;
    CU_TRY(cudaMemcpyAsync(rec, h->scalars.p, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(rec + 3, h->info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(rec + 4, h->gout.p, sizeof(double) * (stride + nA), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    const double* sc = rec;
    const double* g = rec + 4;
    int info = 0;
    memcpy(&info, rec + 3, sizeof(int));
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1);
    h->last_ms[0] = ms;
    h->last_ms[1] = h->last_ms[2] = h->last_ms[3] = 0;
    GP_TRY(pivot_status(info, "Gram matrix"));
    *f_host = nlml_from_scalars(h, sc);
    // dLML/dtheta = 0.5 * sum W * dK/dtheta ; chain through softplus: dtheta/du = sigmoid(u)
    if (h->periodic) {
        // dK/dl_j = g r2_j / l_j and dK/dp_j = 2 pi g delta_j sin(2 pi delta_j / p_j) / (4 l_j^2) / p_j^2: dLML/dl_j = 0.5 L_j / l_j,
        // dLML/dp_j = pi Q_j / p_j^2; a scalar lengthscale or period takes the sum over the dimensions
        const double* L = g + 2;
        const double* Q = g + 2 + h->d;
        double Ls = 0.0, Qs = 0.0;
        for (int k = 0; k < h->d; k++) {
            Ls += L[k];
            Qs += Q[k];
        }
        for (int i = 0; i < nl; i++) grad_host[i] = -(0.5 * (nl > 1 ? L[i] : Ls) / h->ls_host[i]) * sigmoid(u[i]);
        for (int i = 0; i < np; i++)
            grad_host[nl + 1 + i] = -(M_PI * (np > 1 ? Q[i] : Qs) / (h->per_p[i] * h->per_p[i])) * sigmoid(u[nl + 1 + i]);
    } else {
        for (int i = 0; i < nl; i++) grad_host[i] = -(0.5 * g[2 + i] / h->ls_host[i]) * sigmoid(u[i]);
    }
    // variance == 0 only when softplus underflowed, where the chain factor sigmoid(u) is 0 too: the entry is 0, not 0/0
    grad_host[nl] = h->variance > 0.0 ? -(0.5 * g[0] / h->variance) * sigmoid(u[nl]) : 0.0;
    grad_host[nl + 1 + np] = -(0.5 * g[1]) * sigmoid(u[nl + 1 + np]);
    if (h->mean_id == GPSO_MEAN_CONSTANT) grad_host[nl + 2 + np] = -sc[2];
    if (nA) {  // d(-LML)/dA = -X^T alpha, d(-LML)/db = -sum(alpha)
        for (int k = 0; k < nA; k++) grad_host[nl + 2 + np + k] = -g[stride + k];
        grad_host[nl + 2 + np + nA] = -sc[2];
    }
    // alpha (slot stride - 1 of the partial sums); alpha == 0 only when softplus underflowed: the entry is 0, as for the variance
    if (na) grad_host[-1] = h->rq_alpha > 0.0 ? -(0.5 * g[stride - 1]) * sigmoid(u[-1]) : 0.0;
    return 0;
}

extern "C" int gpso_factorize(gpso_handle* h, const double* theta_host, int p) {
    if (!h || !theta_host) return fail(GPSO_E_BADARG, "gpso_factorize: null argument");
    if (!h->have_data) return fail(GPSO_E_STATE, "gpso_factorize: call gpso_set_data first");
    GP_TRY(set_device(h));
    GP_TRY(load_theta(h, theta_host, p, "gpso_factorize"));
    h->factorized = false;
    cudaStream_t st = h->stream;
    GP_TRY(factor_pipeline(h, st, false));
    double sc[3];
    int info = 0;
    CU_TRY(cudaMemcpyAsync(sc, h->scalars.p, sizeof sc, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(&info, h->info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    GP_TRY(pivot_status(info, "Gram matrix"));
    h->factor_nlml = nlml_from_scalars(h, sc);
    GP_TRY(prepare_ozaki(h, st));
    h->factorized = true;
    return 0;
}

extern "C" int gpso_factor_lml(gpso_handle* h, double* lml_host) {
    if (!h || !lml_host) return fail(GPSO_E_BADARG, "gpso_factor_lml: null argument");
    if (!h->factorized) return fail(GPSO_E_STATE, "gpso_factor_lml: call gpso_factorize first");
    *lml_host = -h->factor_nlml;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// predict
// ---------------------------------------------------------------------------------------------------------------------
static long long window_size(const gpso_handle* h, long long M) {
    long long group = (long long)PRED_GROUP * TB;
    long long per_cand = h->oz_S ? (long long)h->Np * h->oz_S : (long long)h->Np * 8;
    long long maxw = h->window_override > 0 ? h->window_override : WINDOW_BYTES / per_cand;
    maxw = std::max(group, (maxw / group) * group);
    long long need = ((M + TB - 1) / TB) * TB;
    return std::min(maxw, need);
}

static int prof_mark(gpso_handle* h, cudaStream_t st) {
    if (!h->profile) return 0;
    if (h->prof_used == h->prof_events.size()) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreate(&e));
        h->prof_events.push_back(e);
    }
    CU_TRY(cudaEventRecord(h->prof_events[h->prof_used++], st));
    return 0;
}

static int trace_mark(gpso_handle* h, cudaStream_t st, int tag, long long window) {
    if (!h->trace) return 0;
    if (h->trace_used == h->trace_events.size()) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreate(&e));
        h->trace_events.push_back(e);
        h->trace_tags.push_back(0);
        h->trace_tags.push_back(0);
    }
    h->trace_tags[2 * h->trace_used] = tag;
    h->trace_tags[2 * h->trace_used + 1] = (int)window;
    CU_TRY(cudaEventRecord(h->trace_events[h->trace_used++], st));
    return 0;
}

static int prod_mark(gpso_handle* h, cudaStream_t st) {
    if (h->prod_used == h->prod_events.size()) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreate(&e));
        h->prod_events.push_back(e);
    }
    CU_TRY(cudaEventRecord(h->prod_events[h->prod_used++], st));
    return 0;
}

// sums the per-window stage times recorded by prof_mark (call after the stream has been synchronised)
static void prof_collect(gpso_handle* h) {
    h->last_ms[1] = h->last_ms[2] = h->last_ms[3] = 0.0;
    double screen_ms = 0.0;
    for (size_t i = 0; i + 1 < h->prod_used; i += 2) {
        float t = 0;
        cudaEventElapsedTime(&t, h->prod_events[i], h->prod_events[i + 1]);
        h->last_ms[2] += t;
        if (i < h->scr_prod_marks) screen_ms += t;  // the launches of the screening pass come first
    }
    if (h->scr_prod_marks) h->scr_info[7] = screen_ms;
    h->scr_prod_marks = 0;
    h->prod_used = 0;
    if (h->trace) {
        h->trace_out.clear();
        for (size_t i = 0; i < h->trace_used; i++) {
            float t = 0;
            cudaEventElapsedTime(&t, h->trace_events[0], h->trace_events[i]);
            h->trace_out.push_back((double)h->trace_tags[2 * i]);
            h->trace_out.push_back((double)h->trace_tags[2 * i + 1]);
            h->trace_out.push_back((double)t);
        }
        h->trace_used = 0;
    }
    if (!h->profile) return;
    h->last_ms[2] = 0.0;
    for (size_t i = 0; i + 3 < h->prof_used; i += 4) {
        float a = 0, b = 0, c = 0;
        cudaEventElapsedTime(&a, h->prof_events[i], h->prof_events[i + 1]);
        cudaEventElapsedTime(&b, h->prof_events[i + 1], h->prof_events[i + 2]);
        cudaEventElapsedTime(&c, h->prof_events[i + 2], h->prof_events[i + 3]);
        h->last_ms[1] += a;
        h->last_ms[2] += b;
        h->last_ms[3] += c;
    }
    h->prof_used = 0;
}

// ---- the window pipeline ---------------------------------------------------------------------------------------------
// Candidates are processed in windows.  Per window:  [H2D copy]  ->  cross-covariance (+ mean)  ->  product  ->  finalise.
// With overlap the cross-covariance of window w+1 (stream `aux`) runs beside the product of window w (the handle's
// high-priority stream): digit tiles and means are double-buffered, events order the two streams.  Host-resident candidates
// are staged through two device buffers by a third (copy) stream.  The full-precision, screening and bound passes all run
// through window_pipeline; each supplies its list of windows, whether it overlaps, and the work of one window.
struct WindowSpan {
    long long off, n;  // first candidate, candidates
};

// A periodic kernel: the embedded rows of M candidates, row-major [M][2d] in pX (the layout the cross-covariance kernels stage).
// A sum / product with periodic components or a map: rows of cand_width() columns, each component's at its offset -- the
// embedded rows of a periodic component, the raw (active) coordinates of the others; one launch.
static int embed_candidates(gpso_handle* h, cudaStream_t st, const double* Xc, long long M) {
    if (h->periodic) {
        periodic_embed_kernel<<<(unsigned)((M * h->d + 255) / 256), 256, 0, st>>>(Xc, M, M, h->d, h->plp.as<double>(), 2 * h->d, 1,
                                                                                  h->pX.as<double>());
        return check_launch(h, "periodic_embed");
    }
    stage_rows_kernel<<<(unsigned)((M * h->rmap.n + 255) / 256), 256, 0, st>>>(Xc, M, M, h->d, h->rmap, 0, h->cand_width(), 1,
                                                                               h->pX.as<double>());
    return check_launch(h, "stage_rows");
}

static std::vector<WindowSpan> uniform_windows(long long M, long long W) {
    std::vector<WindowSpan> wins;
    for (long long off = 0; off < M; off += W) wins.push_back({off, std::min(W, M - off)});
    return wins;
}

struct Window {
    long long w, off, Mw;
    const double* src;  // the window's candidates on the device
    int b;              // digit-tile / mean buffer (0 without overlap)
    const double* xk;   // what the covariance kernels read: src, or a periodic kernel's embedded candidates
};

// The work of one window.  xcov runs on the stream it is given, everything else on the product stream.  A pass without a
// product stage (the bound pass) marks its cross-covariance only.  `after` runs once the window has released buffer b and may
// stop the pass: the windows queued so far still complete and are joined.
struct WindowStages {
    std::function<int(const Window&, cudaStream_t)> xcov, product, finalise;
    std::function<int(const Window&, cudaStream_t, bool*)> after;
};

// Queues the windows `wins` of the candidates (Xc_dev or Xc_host) behind the work already on `st`, the caller's stream, which
// continues after the last of them.  W bounds the windows (staging buffer size).  *done: windows queued.
static int window_pipeline(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, long long W,
                           const std::vector<WindowSpan>& wins, bool overlap, const WindowStages& body, long long* done = nullptr) {
    const bool host = Xc_host != nullptr;
    const int d = h->d;
    if (host) {
        GP_TRY(h->cand[0].ensure((size_t)W * d * sizeof(double)));
        GP_TRY(h->cand[1].ensure((size_t)W * d * sizeof(double)));
    }
    // one buffer: the embedding of window w + 1 follows the cross-covariance of window w on the same stream
    if (h->embeds()) GP_TRY(h->pX.ensure((size_t)W * h->cand_width() * sizeof(double)));
    cudaStream_t user_st = st;
    cudaStream_t xs = overlap ? h->aux_stream : st;  // stream of the cross-covariance kernels
    cudaStream_t cs = h->copy_stream;
    // everything enqueued so far on `st` (factorisation, leaf generation) precedes the first work on the side streams
    CU_TRY(cudaEventRecord(h->ev_start, st));
    if (overlap && st != h->stream) {  // products run on the handle's high-priority stream, joined back at the end
        st = h->stream;
        CU_TRY(cudaStreamWaitEvent(st, h->ev_start, 0));
    }
    if (xs != st) CU_TRY(cudaStreamWaitEvent(xs, h->ev_start, 0));
    if (host) CU_TRY(cudaStreamWaitEvent(cs, h->ev_start, 0));
    const bool marks = (bool)body.product;
    bool cand_busy[2] = {false, false}, buf_busy[2] = {false, false};
    long long w = 0;
    for (bool stop = false; w < (long long)wins.size() && !stop; w++) {
        const int cb = (int)(w & 1);  // candidate staging buffer
        Window win = {w, wins[(size_t)w].off, wins[(size_t)w].n, nullptr, overlap ? cb : 0, nullptr};
        h->last_windows++;
        // ---- 1. candidates of this window on the device
        if (host) {
            if (cand_busy[cb]) CU_TRY(cudaStreamWaitEvent(cs, h->ev_used[cb], 0));
            CU_TRY(cudaMemcpyAsync(h->cand[cb].p, Xc_host + win.off * d, (size_t)win.Mw * d * sizeof(double), cudaMemcpyHostToDevice, cs));
            CU_TRY(cudaEventRecord(h->ev_copy[cb], cs));
            CU_TRY(cudaStreamWaitEvent(xs, h->ev_copy[cb], 0));
            win.src = h->cand[cb].as<double>();
        } else {
            win.src = Xc_dev + win.off * d;
        }
        // ---- 2. cross-covariance (+ posterior mean)
        if (overlap && buf_busy[win.b]) CU_TRY(cudaStreamWaitEvent(xs, h->ev_free[win.b], 0));  // window w-2 has released buffer b
        GP_TRY(prof_mark(h, xs));
        GP_TRY(trace_mark(h, xs, 1, w));
        win.xk = win.src;
        if (h->embeds()) {
            GP_TRY(embed_candidates(h, xs, win.src, win.Mw));
            win.xk = h->pX.as<double>();
        }
        GP_TRY(body.xcov(win, xs));
        GP_TRY(trace_mark(h, xs, 2, w));
        if (host) {
            CU_TRY(cudaEventRecord(h->ev_used[cb], xs));
            cand_busy[cb] = true;
        }
        if (xs != st) {
            CU_TRY(cudaEventRecord(h->ev_xcov[win.b], xs));
            CU_TRY(cudaStreamWaitEvent(st, h->ev_xcov[win.b], 0));
        }
        // ---- 3. product, 4. finalise
        if (marks) {
            GP_TRY(prof_mark(h, st));
            GP_TRY(prod_mark(h, st));
            GP_TRY(trace_mark(h, st, 3, w));
            GP_TRY(body.product(win, st));
            GP_TRY(prod_mark(h, st));
            GP_TRY(trace_mark(h, st, 4, w));
            GP_TRY(prof_mark(h, st));
        }
        GP_TRY(body.finalise(win, st));
        if (marks) {
            GP_TRY(prof_mark(h, st));
            GP_TRY(trace_mark(h, st, 5, w));
        }
        if (overlap) {
            CU_TRY(cudaEventRecord(h->ev_free[win.b], st));
            buf_busy[win.b] = true;
        }
        if (body.after) GP_TRY(body.after(win, st, &stop));
    }
    if (done) *done = w;
    if (st != user_st) {  // the caller's stream continues after the last product / finalise
        CU_TRY(cudaEventRecord(h->ev_start, st));
        CU_TRY(cudaStreamWaitEvent(user_st, h->ev_start, 0));
    }
    return 0;
}

// What the full-precision pass produces
struct ScoreOutputs {
    enum Kind { VALUES, ARGMAX, TOPK } kind;
    double* mean = nullptr;              // VALUES: mean / var of every candidate, host or device memory like the candidates
    double* var = nullptr;
    const long long* idx_map = nullptr;  // ARGMAX, refine pass: global index of every (gathered) candidate; the refined UCB of
    bool check_mean = false;             // each is compared with its screened UCB (check_mean: the screened value is the mean)
    int k = 0;                           // TOPK: records per window
};

// The full-precision pass: the int8 tensor-core engine (oz_S digits) or the FP64 DMMA product
static int full_pass(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, long long M, double varsigma,
                     const ScoreOutputs& out) {
    const bool oz = h->oz_S != 0;
    const bool host = Xc_host != nullptr;
    const long long W = window_size(h, M);
    const long long nwin = (M + W - 1) / W;
    // overlap needs the second set of buffers; a single window or the profiling mode (per-stage events) runs in order
    const bool overlap = oz && h->overlap && !h->profile && nwin > 1;
    const int nbuf = overlap ? 2 : 1;
    GP_TRY(h->part.ensure((size_t)W * h->nb * sizeof(double)));
    GP_TRY(h->blockbest.ensure((size_t)((W + 255) / 256) * sizeof(BestRec)));
    for (int b = 0; b < nbuf; b++) {
        // Linear terms: the window's prior variances follow its (padded) means; W is a multiple of the padded window
        GP_TRY(h->wmeanb[b].ensure((size_t)W * (h->has_lin() ? 2 : 1) * sizeof(double)));
        if (oz) GP_TRY(h->ozBb[b].ensure((size_t)W * h->Np * h->oz_S));
    }
    if (!oz) GP_TRY(h->KsT.ensure((size_t)W * h->Np * sizeof(double)));
    const bool argmax = out.kind == ScoreOutputs::ARGMAX, topk = out.kind == ScoreOutputs::TOPK;
    const bool check = argmax && out.idx_map != nullptr;
    // the finalised mean / var of a window stay on the device: copied back to the host per window, read by the top-k pass
    // or compared with the screened values
    const bool staged = (out.kind == ScoreOutputs::VALUES && host) || topk || check;
    if (staged) {
        GP_TRY(h->omean.ensure((size_t)W * sizeof(double)));
        GP_TRY(h->ovar.ensure((size_t)W * sizeof(double)));
    }
    if (topk) GP_TRY(h->topk.ensure((size_t)nwin * out.k * sizeof(BestRec)));
    const int S = h->oz_S;
    const double beta = oz ? oz_beta(h) : 0.0;
    const double bscale = oz ? ldexp(1.0, 8 * S - 2) / beta : 0.0;
    const double gscale = oz ? beta * ldexp(1.0, -2 * (8 * S - 2) + 8 * (S - 1)) : 0.0;
    auto pad = [](long long Mw) { return ((Mw + TB - 1) / TB) * TB; };
    WindowStages body;
    body.xcov = [&](const Window& win, cudaStream_t xs) {
        if (oz) {
            DISPATCH_S(S, launch_oz_crosscov, h, xs, win.xk, win.Mw, pad(win.Mw) / OZ_NT, bscale, h->ozBb[win.b].as<uint8_t>(),
                       h->wmeanb[win.b].as<double>());
            GP_TRY(check_launch(h, "crosscov_slices"));
        } else {
            launch_crosscov(h, xs, win.xk, win.Mw, pad(win.Mw));
            GP_TRY(check_launch(h, "crosscov"));
        }
        return add_linear_offset(h, xs, win.src, win.Mw, 1.0, h->wmeanb[win.b].as<double>());
    };
    // part[I][c] = sum over the rows of block I of (L^-1 k*)^2
    body.product = [&](const Window& win, cudaStream_t ps) {
        const long long Mw_pad = pad(win.Mw);
        if (oz) {
            DISPATCH_S(S, launch_oz_trmm, h, ps, Mw_pad / OZ_NT, Mw_pad, gscale, h->ozBb[win.b].as<uint8_t>());
            return check_launch(h, "ozaki_trmm");
        }
        PredictParams P;
        P.Linv = h->Linv.as<double>();
        P.KsT = h->KsT.as<double>();
        P.part = h->part.as<double>();
        P.Np = h->Np;
        P.nb = h->nb;
        P.nct = (int)(Mw_pad / TB);
        P.counter = h->counter.as<int>();
        CU_TRY(cudaMemsetAsync(h->counter.p, 0, sizeof(int), ps));
        int grid = std::min(h->nsm, P.nct * P.nb);
        predict_trmm_kernel<<<grid, GTHREADS, GEMM_SMEM_BYTES, ps>>>(P);
        return check_launch(h, "predict_trmm");
    };
    // var, ucb, window arg-max merged into the running record / top-k records of the window / check of the survivors
    body.finalise = [&](const Window& win, cudaStream_t ps) {
        double* om = staged ? h->omean.as<double>() : out.mean ? out.mean + win.off : nullptr;
        double* ov = staged ? h->ovar.as<double>() : out.var ? out.var + win.off : nullptr;
        const int fb = (int)((win.Mw + 255) / 256);
        if (h->has_lin())
            predict_finalize_kss_kernel<<<fb, 256, 0, ps>>>(h->part.as<double>(), h->wmeanb[win.b].as<double>(), h->nb, (int)pad(win.Mw),
                                                            win.Mw, win.off, h->noise, varsigma, argmax ? 1 : 0, om, ov,
                                                            h->blockbest.as<BestRec>(), out.idx_map);
        else
            predict_finalize_kernel<<<fb, 256, 0, ps>>>(h->part.as<double>(), h->wmeanb[win.b].as<double>(), h->nb, (int)pad(win.Mw), win.Mw,
                                                        win.off, h->variance, h->noise, varsigma, argmax ? 1 : 0, om, ov,
                                                        h->blockbest.as<BestRec>(), out.idx_map);
        GP_TRY(check_launch(h, "predict_finalize"));
        if (check) {
            screen_check_kernel<<<fb, 256, 0, ps>>>(om, ov, win.Mw, out.idx_map + win.off, varsigma, h->scr_ucb.as<double>(),
                                                    h->scr_state.as<unsigned long long>(), out.check_mean ? 1 : 0);
            GP_TRY(check_launch(h, "screen_check"));
        }
        if (topk) {
            topk_window_kernel<<<1, 1024, 0, ps>>>(om, ov, win.Mw, win.off, varsigma, out.k, h->topk.as<BestRec>() + win.w * out.k);
            GP_TRY(check_launch(h, "topk_window"));
        }
        if (argmax) {
            best_merge_kernel<<<1, 256, 0, ps>>>(h->blockbest.as<BestRec>(), fb, h->running.as<BestRec>(), win.w == 0 ? 1 : 0);
            GP_TRY(check_launch(h, "best_merge"));
        }
        return 0;
    };
    if (out.kind == ScoreOutputs::VALUES && host)
        body.after = [&](const Window& win, cudaStream_t ps, bool*) {
            CU_TRY(cudaMemcpyAsync(out.mean + win.off, h->omean.p, (size_t)win.Mw * sizeof(double), cudaMemcpyDeviceToHost, ps));
            CU_TRY(cudaMemcpyAsync(out.var + win.off, h->ovar.p, (size_t)win.Mw * sizeof(double), cudaMemcpyDeviceToHost, ps));
            return 0;
        };
    return window_pipeline(h, st, Xc_dev, Xc_host, W, uniform_windows(M, W), overlap, body);
}

// per-call state of a scoring call: profiling and trace events and the window count start afresh
static int begin_scoring(gpso_handle* h) {
    h->prof_used = 0;
    h->prod_used = 0;
    h->trace_used = 0;
    h->last_windows = 0;
    return set_device(h);
}

static int predict_common_checks(gpso_handle* h, const void* a, long long M, const char* who) {
    if (!h || !a) return fail(GPSO_E_BADARG, std::string(who) + ": null argument");
    if (M <= 0) return fail(GPSO_E_BADARG, std::string(who) + ": M must be positive");
    if (!h->factorized) return fail(GPSO_E_STATE, std::string(who) + ": call gpso_factorize first");
    return begin_scoring(h);
}

static int fetch_best(gpso_handle* h, cudaStream_t st, double* result_host) {
    BestRec r;
    CU_TRY(cudaMemcpyAsync(h->host_rec, h->running.p, sizeof r, cudaMemcpyDeviceToHost, st));  // pinned: no staging copy
    CU_TRY(cudaStreamSynchronize(st));
    memcpy(&r, h->host_rec, sizeof r);
    prof_collect(h);
    result_host[0] = (double)r.idx;
    result_host[1] = r.mean;
    result_host[2] = r.var;
    result_host[3] = r.ucb;
    return 0;
}

// ---- screen-and-refine arg-max (kern_screen.cuh) ------------------------------------------------------------------------
// Error bound of the screened UCB against the full-precision one.  Variance: pick_slices' model of the digit rounding and of
// the neglected digit-pair levels at S digits (absolute: 6 sigma_f beta 2^-8S sqrt(N) max_i rho_i; measured deviations are
// ~30x below it, profiles/r01_engine_error_c3.txt), plus the fp32 covariance evaluation seen through
// d var = 2 dk^T K_y^-1 k*  with  |K_y^-1 k*|_2 <= sigma_f / sigma_n, plus the fp32 epilogue.  Mean: dk^T alpha with independent
// fp32 errors of the covariance values and of the 16-term fp32 partial sums.  Everything times SCREEN_SAFETY; the refine pass
// checks the bound on every survivor with another factor 4 of margin.
struct ScreenFit {  // what the error model needs to know about a fit
    int N;
    double variance, noise;
    double rho_max, rho_l2sq;        // largest power-of-two row scale of L^-1, sum of their squares
    double rowl2_max, frob2;         // largest row norm of L^-1, |L^-1|_F^2
    double alpha_l2;
};

static void screen_error_model(const ScreenFit& f, int S, int full, double varsigma, double* e_total, double* e_var_out,
                               double* e_mean_out) {
    const double sigma_f = sqrt(f.variance), beta = ldexp(1.0, ilogb(f.variance) + 1);
    const double sqrtN = sqrt((double)f.N);
    double est_var1, est_var2;
    if (full) {
        // all S^2 digit pairs: the product of the rounded operands is exact, what is left is the rounding itself,
        //   dv_i = sum_k dA_ik b_k + A_ik db_k,  dA_ik ~ U(+-u rho_i), db_k ~ U(+-u beta), u = 2^-(8S-1),  0 <= b_k <= variance:
        //   Var dv_i = u^2/3 (rho_i^2 |b|^2 + beta^2 |A_i|^2),  |b|^2 <= N variance^2
        const double u2_3 = ldexp(1.0, -2 * (8 * S - 1)) / 3.0;
        const double b2 = (double)f.N * f.variance * f.variance;
        est_var1 = 2.0 * sigma_f * sqrt(u2_3 * (f.rho_max * f.rho_max * b2 + beta * beta * f.rowl2_max * f.rowl2_max));  // 2 sum v_i dv_i
        est_var2 = u2_3 * (f.rho_l2sq * b2 + beta * beta * f.frob2);                                                      // sum dv_i^2
    } else {
        // triangular product (pairs p + q < S): per-row standard deviation c rho_i beta 2^-8S sqrt(N); operand rounding of A and
        // of B contribute 1.15 each (against the other operand at its bound), the neglected levels 1.3 sqrt(S-1): c = 3 for S <= 4
        const double unit = 3.0 * beta * ldexp(1.0, -8 * S) * sqrtN;
        est_var1 = 2.0 * sigma_f * unit * f.rho_max;   // first order:  2 sum_i v_i dv_i,  |v|_2 <= sigma_f
        est_var2 = unit * unit * f.rho_l2sq;           // second order: sum_i dv_i^2 (a bias; matters at 2 digits only)
    }
    // the fp32 covariance contract of kern_screen.cuh, for every kernel family and, for RationalQuadratic, every alpha.  The
    // rest of the model (pick_slices' digit scale, the mean bound of bound_pass, the int8 engines) relies only on
    // 0 <= k* <= variance, which RationalQuadratic satisfies too: no kernel-specific term anywhere else.
    const double eps_k32 = 2.0e-6 * f.variance;
    const double var_b = 2.0 * eps_k32 * sigma_f / sqrt(f.noise);
    const double var_epi = 1.0e-6 * f.variance;
    const double e_var = SCREEN_SAFETY * (est_var1 + est_var2 + var_b + var_epi);
    const double e_mean = SCREEN_SAFETY * (eps_k32 + 1.0e-6 * f.variance) * f.alpha_l2;
    *e_var_out = e_var;
    *e_mean_out = e_mean;
    *e_total = e_mean + fabs(varsigma) * e_var;
}

static void screen_error_bound(const gpso_handle* h, int S, bool full, double varsigma, double* e_total, double* e_var_out,
                               double* e_mean_out) {
    const ScreenFit f = {h->N, h->variance, h->noise, h->rho_max, h->rho_l2sq, h->linv_rowl2_max, h->linv_frob2, h->alpha_l2};
    screen_error_model(f, S, full ? 1 : 0, varsigma, e_total, e_var_out, e_mean_out);
}

// The ladder of screening variants, cheapest first: 2 digits with all four digit pairs (16 KB of operands per k-step, exact
// product of 14-bit operands), then the triangular products of 3 and 4 digits.  screen_S_cur is the rung the survivor
// feedback of earlier calls asked for.  A rung is tried when its variance bound is below the kernel variance (a screen with
// a looser bound cannot separate anything); how well it separates THESE candidates only the survivor count can tell.
struct ScreenVariant { int S; bool full; };
struct ScreenHint { int rung = 0; unsigned calls = 0; };
static ScreenHint g_screen_hint[65];  // per matrix size in tiles; performance state only (see score_argmax)
static const ScreenVariant SCREEN_LADDER[] = {{2, true}, {3, false}, {4, false}};
constexpr int SCREEN_RUNGS = 3;

// Host-only (no GPU needed): the error bound of the screening pass for a fit with N training points, the given kernel / noise
// variance, largest power-of-two row scale of L^-1, sum of the squared row scales and |alpha|_2.  out3 = {E, E_var, E_mean}.
// tests/test_screen_model.py checks it against a numpy emulation of the screening arithmetic.
extern "C" int gpso_debug_screen_bound(int N, double variance, double noise, const double* fit5, int digits, int full, double varsigma,
                                       double* out3) {
    if (!out3 || !fit5 || N <= 0 || digits < SCREEN_S_MIN || digits > SCREEN_S_MAX)
        return fail(GPSO_E_BADARG, "gpso_debug_screen_bound: bad argument");
    const ScreenFit f = {N, variance, noise, fit5[0], fit5[1], fit5[2], fit5[3], fit5[4]};
    screen_error_model(f, digits, full, varsigma, &out3[0], &out3[1], &out3[2]);
    return 0;
}

static bool screen_applicable(const gpso_handle* h, long long M) {
    if (h->screen_mode == 0 || !h->screen_ready || h->oz_S == 0 || h->profile) return false;
    if (h->Np < SCREEN_MIN_NP || M < SCREEN_MIN_M) return false;
    // the fp32 path needs the kernel variance and the lengthscales well inside the float range
    if (!(h->variance > 1e-30 && h->variance < 1e30)) return false;
    if (h->n_rq() && !(h->rq_alpha > 1e-30 && h->rq_alpha < 1e30)) return false;
    for (int c = 0; c < h->sum.n; c++)
        if (h->sum.fam[c] == KERNEL_RQ && !(h->sum.alpha[c] > 1e-30 && h->sum.alpha[c] < 1e30)) return false;
    for (int i = 0; i < h->n_ls(); i++)
        if (!(h->ls_host[i] > 1e-30 && h->ls_host[i] < 1e30)) return false;
    for (int i = 0; i < h->n_per(); i++)
        if (!(h->per_p[i] > 1e-30 && h->per_p[i] < 1e30)) return false;
    for (int c = 0; c < h->sum.n; c++)
        for (int i = 0; i < h->comp_np(c); i++)
            if (!(h->comp_p[c][i] > 1e-30 && h->comp_p[c][i] < 1e30)) return false;
    return true;
}

// Window list of a screening pass over M candidates with windows of at most W (a multiple of 1024).  With the stream overlap
// the cross-covariance of the FIRST window is the one stage nothing hides (1.6 ms of a 32 ms step when eight GPUs share the
// candidates): the pipeline ramps up through a quarter and a half window; the rest is split evenly (no short tail launch).
static void make_screen_windows(long long M, long long W, bool ramp, bool even, std::vector<WindowSpan>& wins) {
    wins.clear();
    long long off = 0;
    if (ramp && (M + W - 1) / W >= 3)
        for (long long part : {W / 4, W / 2}) {
            const long long r = part / 1024 * 1024;
            if (r >= 1024 && off + r < M) {
                wins.push_back({off, r});
                off += r;
            }
        }
    const long long rest = M - off, nrest = (rest + W - 1) / W;
    const long long each = (even && nrest > 0) ? std::min(W, ((rest + nrest - 1) / nrest + 1023) / 1024 * 1024) : W;
    for (; off < M; off += each) wins.push_back({off, std::min(each, M - off)});
}

extern "C" int64_t gpso_debug_screen_windows(int64_t M, int64_t W, int ramp, int even, int64_t* out, int64_t capacity) {
    if (M <= 0 || W < 1024 || W % 1024 != 0) {
        fail(GPSO_E_BADARG, "gpso_debug_screen_windows: need M > 0 and W a positive multiple of 1024");
        return -1;
    }
    std::vector<WindowSpan> wins;
    make_screen_windows(M, W, ramp != 0, even != 0, wins);
    if (out)
        for (size_t i = 0; i < wins.size() && (int64_t)(2 * i + 1) < capacity; i++) {
            out[2 * i] = wins[i].off;
            out[2 * i + 1] = wins[i].n;
        }
    return (int64_t)wins.size();
}

// The screening pass over all candidates: per window [H2D] -> fp32 cross-covariance digits (+ mean) -> low-digit tensor-core
// product -> screened UCB per candidate + running maximum.  Leaves scr_ucb[0..M) and scr_state[0] (key of the maximum) on the
// device.
static int screen_pass(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, long long M, int S, bool full,
                       double varsigma, double two_e, bool* hopeless) {
    *hopeless = false;
    const long long per_cand = (long long)h->Np * S;
    long long W = (WINDOW_BYTES / per_cand) / 1024 * 1024;
    if (h->window_override > 0) W = std::max<long long>(1024, h->window_override / 1024 * 1024);
    W = std::min(W, ((M + SCR_NT - 1) / SCR_NT) * SCR_NT);
    const long long nwin = (M + W - 1) / W;
    // side-stream overlap of the next window's cross-covariance; both kernels are power-bound, so it gains little
    // (profiles/r02c_screen_trace.json: 86.1 vs 88.4 ms per 2.1e6 candidates)
    const bool overlap = h->overlap && nwin > 1;
    const int nbuf = overlap ? 2 : 1;
    std::vector<WindowSpan> wins;
    make_screen_windows(M, W, overlap && h->window_override == 0, h->window_override == 0, wins);
    GP_TRY(h->part32.ensure((size_t)W * h->nb * sizeof(float)));
    GP_TRY(h->scr_ucb.ensure((size_t)M * sizeof(double)));
    GP_TRY(h->scr_state.ensure(4 * sizeof(unsigned long long)));
    for (int b = 0; b < nbuf; b++) {
        GP_TRY(h->wmeanb[b].ensure((size_t)W * sizeof(double)));
        GP_TRY(h->ozBb[b].ensure((size_t)W * per_cand));
    }
    if (h->screen_built_S != S) {
        // tiles above the block diagonal are neither built nor read: row block I of the product runs over k-steps
        // [0, 4 (I + 1)) (OzItems<OZ_TRMM>), exactly the tiles linv_slices_kernel<S, false> writes
        GP_TRY(h->ozAs.ensure((size_t)h->Np * h->Np * S));
        DISPATCH_SCREEN_S(S, launch_screen_slices, h, st);
        GP_TRY(check_launch(h, "screen_slices"));
        h->screen_built_S = S;
    }
    CU_TRY(cudaMemsetAsync(h->scr_state.p, 0, 4 * sizeof(unsigned long long), st));
    // during the screening pass the persisting-L2 window of the product stream covers the low-digit tiles of L^-1
    GP_TRY(set_l2_window(h, h->ozAs.p, (size_t)h->Np * h->Np * S));
    long long probe_rows = 0;
    unsigned long long* probe = reinterpret_cast<unsigned long long*>(h->host_rec + MAX_LS + 14);  // pinned, unused during the pass
    const double beta = oz_beta(h);
    const float bscale = (float)(ldexp(1.0, 8 * S - 2) / beta);
    // triangular product: levels t < S, the lowest kept level has weight 256^0; full product: levels t <= 2S-2
    const double gscale = full ? beta * ldexp(1.0, -2 * (8 * S - 2)) : beta * ldexp(1.0, -2 * (8 * S - 2) + 8 * (S - 1));
    auto pad = [](long long Mw) { return ((Mw + SCR_NT - 1) / SCR_NT) * SCR_NT; };
    WindowStages body;
    body.xcov = [&](const Window& win, cudaStream_t xs) {
        DISPATCH_SCREEN_S(S, launch_screen_crosscov, h, xs, win.xk, win.Mw, pad(win.Mw) / 64, bscale, h->ozBb[win.b].as<uint8_t>(),
                          h->wmeanb[win.b].as<double>());
        GP_TRY(check_launch(h, "crosscov_screen"));
        return add_linear_offset(h, xs, win.src, win.Mw, 1.0, h->wmeanb[win.b].as<double>());  // the refine pass adds the same
    };
    body.product = [&](const Window& win, cudaStream_t ps) {
        const long long Mw_pad = pad(win.Mw);
        if (full) {
            launch_screen_product<2, true>(h, ps, Mw_pad / SCR_NT, Mw_pad, gscale, h->ozBb[win.b].as<uint8_t>());
        } else {
            DISPATCH_SCREEN_S(S, launch_screen_product, h, ps, Mw_pad / SCR_NT, Mw_pad, gscale, h->ozBb[win.b].as<uint8_t>());
        }
        return check_launch(h, "ozaki_screen");
    };
    body.finalise = [&](const Window& win, cudaStream_t ps) {
        screen_finalize_kernel<<<(unsigned)((win.Mw + 255) / 256), 256, 0, ps>>>(h->part32.as<float>(), h->wmeanb[win.b].as<double>(), h->nb,
                                                                                 pad(win.Mw), win.Mw, win.off, h->variance, h->noise,
                                                                                 varsigma, h->scr_ucb.as<double>(),
                                                                                 h->scr_state.as<unsigned long long>());
        return check_launch(h, "screen_finalize");
    };
    body.after = [&](const Window& win, cudaStream_t ps, bool* stop) {
        if (win.w == 0 && wins.size() >= 4) {
            // early verdict on this variant: if more than 1/16 of the first window lies within 2E of the window's own best value
            // the screen cannot separate these candidates -- stop instead of paying for the other windows.  The count is
            // queued behind window 0 and read (pinned record) once window 1 has been queued, so the pipeline never drains.
            GP_TRY(h->surv_list.ensure(sizeof(long long)));
            screen_select_kernel<<<(unsigned)((win.Mw + 255) / 256), 256, 0, ps>>>(h->scr_ucb.as<double>(), win.Mw, two_e,
                                                                                   h->scr_state.as<unsigned long long>(),
                                                                                   h->surv_list.as<long long>(), 0u);
            GP_TRY(check_launch(h, "screen_select"));
            CU_TRY(cudaMemcpyAsync(probe, h->scr_state.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ps));
            CU_TRY(cudaMemsetAsync(h->scr_state.as<unsigned long long>() + 1, 0, sizeof(unsigned long long), ps));
            CU_TRY(cudaEventRecord(h->ev_probe, ps));
            probe_rows = win.Mw;
        }
        if (win.w == 1 && probe_rows > 0) {
            CU_TRY(cudaEventSynchronize(h->ev_probe));
            if ((long long)probe[1] * 16 > probe_rows) {
                *hopeless = true;
                h->scr_info[2] = (double)probe[1] * ((double)M / (double)probe_rows);  // extrapolated survivor count, for the record
                *stop = true;
            }
        }
        return 0;
    };
    long long done = 0;
    h->scr_rows = 0;
    GP_TRY(window_pipeline(h, st, Xc_dev, Xc_host, W, wins, overlap, body, &done));
    h->scr_info[6] = (double)done;
    for (long long w = 0; w < done; w++) h->scr_rows += wins[(size_t)w].n;  // after the early stop: the windows that ran
    return set_l2_window(h, h->ozA.p, (size_t)h->Np * h->Np * h->oz_S);  // back on the full-precision tiles (refine pass)
}

// ---- bound-and-refine, level 0 (screen mode 5) ---------------------------------------------------------------------------
// UCB = mean + varsigma * var with sigma_n^2 <= var <= sigma_f^2 + sigma_n^2 for EVERY candidate (the posterior variance of
// the latent function lies between 0 and the prior variance), so a candidate whose posterior mean is more than
// |varsigma| sigma_f^2 below the best mean cannot be the arg-max whatever its variance.  Only the mean is evaluated for all
// candidates (fp32 cross-covariance, error bound E_mean of screen_error_model); the survivors go straight to the
// full-precision engine.  Exact like the digit screen, and much cheaper when the means spread wider than |varsigma| sigma_f^2;
// when they do not (too many survivors) the caller continues with the digit screen over all candidates.  One stream.
static int bound_pass(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, long long M) {
    long long W = 1LL << 19;
    if (h->window_override > 0) W = std::max<long long>(1024, h->window_override / 1024 * 1024);
    W = std::min(W, ((M + SCR_NT - 1) / SCR_NT) * SCR_NT);
    GP_TRY(h->scr_ucb.ensure((size_t)M * sizeof(double)));
    GP_TRY(h->scr_state.ensure(4 * sizeof(unsigned long long)));
    GP_TRY(h->wmeanb[0].ensure((size_t)W * sizeof(double)));
    CU_TRY(cudaMemsetAsync(h->scr_state.p, 0, 4 * sizeof(unsigned long long), st));
    WindowStages body;
    body.xcov = [&](const Window& win, cudaStream_t xs) {
        launch_screen_crosscov<0>(h, xs, win.xk, win.Mw, ((win.Mw + SCR_NT - 1) / SCR_NT) * SCR_NT / 64, 0.0f, nullptr,
                                  h->wmeanb[0].as<double>());
        GP_TRY(check_launch(h, "crosscov_mean"));
        return add_linear_offset(h, xs, win.src, win.Mw, 1.0, h->wmeanb[0].as<double>());
    };
    body.finalise = [&](const Window& win, cudaStream_t ps) {
        bound_finalize_kernel<<<(unsigned)((win.Mw + 255) / 256), 256, 0, ps>>>(h->wmeanb[0].as<double>(), win.Mw, win.off,
                                                                                h->scr_ucb.as<double>(),
                                                                                h->scr_state.as<unsigned long long>());
        return check_launch(h, "bound_finalize");
    };
    long long done = 0;
    h->scr_rows = 0;
    GP_TRY(window_pipeline(h, st, Xc_dev, Xc_host, W, uniform_windows(M, W), false, body, &done));
    h->scr_info[6] = (double)done;
    h->scr_rows = std::min(M, done * W);
    return 0;
}

// survivors of a screening level (scr_ucb / scr_state on the device, slack = admissible distance below the best value) ->
// gathered, re-scored by the full-precision engine with the per-survivor check.  Returns 0 with *ok = true when the record in
// result_host can be trusted, *ok = false when the caller has to fall back (too many survivors, or the check failed).
static int refine_survivors(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, long long M, double varsigma,
                            double slack, double check_bound, bool mean_only, long long cap_in, double* result_host, bool* ok) {
    *ok = false;
    const unsigned cap = (unsigned)std::min<long long>(SCREEN_LIST_CAP, std::max<long long>(cap_in, 1024));
    GP_TRY(h->surv_list.ensure((size_t)cap * sizeof(long long)));
    screen_select_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(h->scr_ucb.as<double>(), M, slack, h->scr_state.as<unsigned long long>(),
                                                                     h->surv_list.as<long long>(), cap);
    GP_TRY(check_launch(h, "screen_select"));
    unsigned long long state[4] = {0, 0, 0, 0};
    CU_TRY(cudaMemcpyAsync(state, h->scr_state.p, sizeof state, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    const long long count = (long long)state[1];
    h->scr_info[2] = (double)count;
    h->scr_info[5] = scr_unkey(state[0]);
    if (count < 1 || count > (long long)cap) {
        h->scr_info[0] = 2.0;
        return 0;
    }
    const long long windows_before = h->last_windows;
    std::vector<double> gathered;
    const double* rdev = nullptr;
    const double* rhost = nullptr;
    if (Xc_host != nullptr) {
        std::vector<long long> list((size_t)count);
        CU_TRY(cudaMemcpyAsync(list.data(), h->surv_list.p, (size_t)count * sizeof(long long), cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        gathered.resize((size_t)count * h->d);
        for (long long i = 0; i < count; i++)
            memcpy(&gathered[(size_t)i * h->d], Xc_host + list[(size_t)i] * h->d, sizeof(double) * h->d);
        rhost = gathered.data();
    } else {
        GP_TRY(h->surv_X.ensure((size_t)count * h->d * sizeof(double)));
        gather_rows_kernel<<<(unsigned)((count * h->d + 255) / 256), 256, 0, st>>>(Xc_dev, h->surv_list.as<long long>(), count, h->d,
                                                                                h->surv_X.as<double>());
        GP_TRY(check_launch(h, "gather_rows"));
        rdev = h->surv_X.as<double>();
    }
    ScoreOutputs out = {ScoreOutputs::ARGMAX};
    out.idx_map = h->surv_list.as<long long>();
    out.check_mean = mean_only;
    GP_TRY(full_pass(h, st, rdev, rhost, count, varsigma, out));
    unsigned long long dbits = 0;
    CU_TRY(cudaMemcpyAsync(&dbits, h->scr_state.as<unsigned long long>() + 2, sizeof dbits, cudaMemcpyDeviceToHost, st));
    GP_TRY(fetch_best(h, st, result_host));  // synchronises st
    double dmax;
    memcpy(&dmax, &dbits, sizeof dmax);
    h->scr_info[4] = dmax;
    h->scr_info[8] = (double)(h->last_windows - windows_before);
    if (dmax <= 0.25 * check_bound) {
        *ok = true;
        return 0;
    }
    h->scr_info[0] = 3.0;  // the bound did not hold with the required margin: do not trust the screen
    return 0;
}

// Fused predict_y + UCB + arg-max of M candidates (device- or host-resident): screened when it pays, else the plain window
// pipeline.  The record returned is always produced by the full-precision engine.
static int score_argmax(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, long long M, double varsigma,
                        double* result_host) {
    for (int i = 0; i < 12; i++) h->scr_info[i] = 0.0;
    h->scr_prod_marks = 0;
    h->scr_rows = 0;
    // the screen keeps one double per candidate: when that does not fit beside the caller's data the call runs unscreened
    const bool room = screen_applicable(h, M) && h->scr_ucb.ensure((size_t)M * sizeof(double)) == 0;
    if (room) {
        double E = 0.0, e_var = 0.0, e_mean = 0.0;
        bool ok = false;
        if (h->screen_mode == SCREEN_MODE_BOUND) {
            // level 0: posterior mean of every candidate, variance bounded by the prior
            screen_error_bound(h, SCREEN_S_MAX, false, varsigma, &E, &e_var, &e_mean);
            GP_TRY(bound_pass(h, st, Xc_dev, Xc_host, M));
            const double width = fabs(varsigma) * h->variance * (1.0 + 2.0e-6);  // |varsigma| (v_max - v_min) with rounding slack
            h->scr_info[1] = 0.0;
            h->scr_info[3] = e_mean;
            h->scr_info[10] = e_mean;
            h->scr_info[11] = width;
            GP_TRY(refine_survivors(h, st, Xc_dev, Xc_host, M, varsigma, 2.0 * e_mean + width, e_mean, true, M / 64, result_host, &ok));
            if (ok) {
                h->scr_info[0] = 4.0;
                return 0;
            }
            // too many survivors (the means do not separate the candidates) or check failed: digit screen over all candidates
        }
        // forced variant, or the ladder from the rung the survivor feedback of earlier calls asked for: a rung that cannot
        // separate these candidates (too many survivors, seen after the first window or at the end) or whose bound fails the
        // check hands over to the next, more precise one; after the last rung the call runs the full pass
        const bool automatic = h->screen_mode == 1 || h->screen_mode == SCREEN_MODE_BOUND;
        // The optimiser builds a new model (a new handle) for every fit: the rung the previous handles ended on is kept per
        // matrix size for the process, so that a run whose candidates no cheap rung can separate does not walk the ladder again
        // after every fit.  Every 32nd call starts one rung lower again (the verdict may change as the data grow).  Only the
        // cost depends on this state; the record returned never does.
        ScreenHint& hint = g_screen_hint[std::min(h->nb, 64)];
        int first = 0;
        if (automatic) {
            first = std::max(std::max(0, h->screen_S_cur), hint.rung);
            if (first > 0 && (++hint.calls % 32u) == 0u) first--;
        }
        for (int rung = first; rung < (automatic ? SCREEN_RUNGS : 1); rung++) {
            ScreenVariant v = SCREEN_LADDER[std::min(rung, SCREEN_RUNGS - 1)];
            if (!automatic) {
                if (h->screen_mode == SCREEN_MODE_FULL2) v = {2, true};
                else v = {std::min(std::max(h->screen_mode, SCREEN_S_MIN), SCREEN_S_MAX), false};
            }
            if (v.S >= h->oz_S) break;  // nothing to gain
            const int S = v.S;
            screen_error_bound(h, S, v.full, varsigma, &E, &e_var, &e_mean);
            if (automatic && !(e_var <= 1.0 * h->variance)) continue;  // a looser bound than the prior variance separates nothing
            bool hopeless = false;
            h->prod_used = 0;
            GP_TRY(screen_pass(h, st, Xc_dev, Xc_host, M, S, v.full, varsigma, 2.0 * E, &hopeless));
            h->scr_prod_marks = h->prod_used;
            h->scr_info[1] = S;
            h->scr_info[3] = E;
            h->scr_info[9] = e_var;
            h->scr_info[10] = e_mean;
            h->scr_info[11] = v.full ? 1.0 : 0.0;
            if (hopeless) {
                h->scr_info[0] = 2.0;
                CU_TRY(cudaStreamSynchronize(st));
                prof_collect(h);
            } else {
                GP_TRY(refine_survivors(h, st, Xc_dev, Xc_host, M, varsigma, 2.0 * E, E, false, M / 16, result_host, &ok));
            }
            // feedback for later calls: start from the next rung when this one left more than M / 64 survivors or failed
            const long long count = (long long)h->scr_info[2];
            if (automatic) {
                const bool weak = hopeless || count * 64 > M || h->scr_info[0] == 3.0;
                h->screen_S_cur = weak ? rung + 1 : rung;
                hint.rung = h->screen_S_cur;
            }
            if (ok) {
                h->scr_info[0] = 1.0;
                return 0;
            }
        }
    }
    GP_TRY(full_pass(h, st, Xc_dev, Xc_host, M, varsigma, {ScoreOutputs::ARGMAX}));
    return fetch_best(h, st, result_host);
}

// Device time of a scoring call in last_ms[0]: `work` is queued on st between ev_t0 and ev_t1, `finish` waits for ev_t1 (after
// queueing the copies of the results behind it, where there are any).
template <class Work, class Finish>
static int timed_call(gpso_handle* h, cudaStream_t st, Work&& work, Finish&& finish) {
    CU_TRY(cudaEventRecord(h->ev_t0, st));
    GP_TRY(work());
    CU_TRY(cudaEventRecord(h->ev_t1, st));
    GP_TRY(finish());
    float ms = 0;
    cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1);
    h->last_ms[0] = ms;
    return 0;
}

static int wait_t1(gpso_handle* h) {
    CU_TRY(cudaEventSynchronize(h->ev_t1));
    return 0;
}

extern "C" int gpso_predict_y_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double* mean_dev, double* var_dev,
                                  void* stream) {
    GP_TRY(predict_common_checks(h, Xc_dev, M, "gpso_predict_y_dev"));
    if (!mean_dev || !var_dev) return fail(GPSO_E_BADARG, "gpso_predict_y_dev: null output");
    return full_pass(h, (cudaStream_t)stream, Xc_dev, nullptr, M, 0.0, {ScoreOutputs::VALUES, mean_dev, var_dev});
}

extern "C" int gpso_ucb_argmax_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double varsigma, double* result_host,
                                   void* stream) {
    GP_TRY(predict_common_checks(h, Xc_dev, M, "gpso_ucb_argmax_dev"));
    if (!result_host) return fail(GPSO_E_BADARG, "gpso_ucb_argmax_dev: null output");
    cudaStream_t st = (cudaStream_t)stream;
    return timed_call(h, st, [&] { return score_argmax(h, st, Xc_dev, nullptr, M, varsigma, result_host); }, [&] { return wait_t1(h); });
}

extern "C" int gpso_predict_y_host(gpso_handle* h, const double* Xc_host, int64_t M, double* mean_host, double* var_host) {
    GP_TRY(predict_common_checks(h, Xc_host, M, "gpso_predict_y_host"));
    if (!mean_host || !var_host) return fail(GPSO_E_BADARG, "gpso_predict_y_host: null output");
    cudaStream_t st = h->stream;
    return timed_call(
        h, st, [&] { return full_pass(h, st, nullptr, Xc_host, M, 0.0, {ScoreOutputs::VALUES, mean_host, var_host}); },
        [&] {
            CU_TRY(cudaStreamSynchronize(st));
            prof_collect(h);
            return 0;
        });
}

extern "C" int gpso_ucb_argmax_host(gpso_handle* h, const double* Xc_host, int64_t M, double varsigma, double* result_host) {
    GP_TRY(predict_common_checks(h, Xc_host, M, "gpso_ucb_argmax_host"));
    if (!result_host) return fail(GPSO_E_BADARG, "gpso_ucb_argmax_host: null output");
    cudaStream_t st = h->stream;
    return timed_call(h, st, [&] { return score_argmax(h, st, nullptr, Xc_host, M, varsigma, result_host); }, [&] { return wait_t1(h); });
}

// Top-k variant of the fused scoring call: the k candidates with the highest UCB in arg-max order (first NaN, larger UCB,
// lowest index on ties).  Per window a k-pass block arg-max on the device, the per-window lists are merged on the host.
static int topk_common(gpso_handle* h, cudaStream_t st, const double* Xc_dev, const double* Xc_host, int64_t M, double varsigma, int k,
                       double* result_host, int* found) {
    if (k < 1 || k > TOPK_MAX) return fail(GPSO_E_BADARG, "gpso_ucb_topk: k must be in 1..64");
    ScoreOutputs out = {ScoreOutputs::TOPK};
    out.k = k;
    std::vector<BestRec> rec;
    GP_TRY(timed_call(
        h, st, [&] { return full_pass(h, st, Xc_dev, Xc_host, M, varsigma, out); },
        [&] {
            rec.resize((size_t)h->last_windows * k);
            CU_TRY(cudaMemcpyAsync(rec.data(), h->topk.p, rec.size() * sizeof(BestRec), cudaMemcpyDeviceToHost, st));
            CU_TRY(cudaStreamSynchronize(st));
            prof_collect(h);
            return 0;
        }));
    std::vector<BestRec> live;
    for (const BestRec& r : rec)
        if (r.idx != 0x7fffffffffffffffLL) live.push_back(r);
    auto better = [](const BestRec& a, const BestRec& b) {
        const bool an = a.ucb != a.ucb, bn = b.ucb != b.ucb;
        if (an || bn) return an && bn ? a.idx < b.idx : an;
        if (a.ucb != b.ucb) return a.ucb > b.ucb;
        return a.idx < b.idx;
    };
    std::sort(live.begin(), live.end(), better);
    const int n = (int)std::min<size_t>(live.size(), (size_t)k);
    for (int i = 0; i < n; i++) {
        result_host[4 * i + 0] = (double)live[i].idx;
        result_host[4 * i + 1] = live[i].mean;
        result_host[4 * i + 2] = live[i].var;
        result_host[4 * i + 3] = live[i].ucb;
    }
    if (found) *found = n;
    return 0;
}

extern "C" int gpso_ucb_topk_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double varsigma, int k, double* result_host, int* found,
                                 void* stream) {
    GP_TRY(predict_common_checks(h, Xc_dev, M, "gpso_ucb_topk_dev"));
    if (!result_host) return fail(GPSO_E_BADARG, "gpso_ucb_topk_dev: null output");
    return topk_common(h, (cudaStream_t)stream, Xc_dev, nullptr, M, varsigma, k, result_host, found);
}

extern "C" int gpso_ucb_topk_host(gpso_handle* h, const double* Xc_host, int64_t M, double varsigma, int k, double* result_host, int* found) {
    GP_TRY(predict_common_checks(h, Xc_host, M, "gpso_ucb_topk_host"));
    if (!result_host) return fail(GPSO_E_BADARG, "gpso_ucb_topk_host: null output");
    return topk_common(h, h->stream, nullptr, Xc_host, M, varsigma, k, result_host, found);
}

// ---------------------------------------------------------------------------------------------------------------------
// joint posterior (kern_joint.cuh): a fixed number of launches per call, on one stream, into the handle's j* buffers
// ---------------------------------------------------------------------------------------------------------------------
static int joint_checks(gpso_handle* h, const void* xc, long long M, const void* out1, const void* out2, const char* who) {
    if (M < 1 || M > GPSO_MAX_JOINT) return fail(GPSO_E_BADARG, std::string(who) + ": M must be in 1..8192 (draw larger batches in parts)");
    if (!h || !xc || !out1 || !out2) return fail(GPSO_E_BADARG, std::string(who) + ": null argument");
    return 0;
}

static int joint_ready(gpso_handle* h, const char* who) {
    if (!h->factorized) return fail(GPSO_E_STATE, std::string(who) + ": call gpso_factorize first");
    return set_device(h);
}

static void launch_joint_crosscov(gpso_handle* h, cudaStream_t st, const double* Xc, int M, int Mp) {
    size_t sm = (size_t)(XG * h->dx() + 8 * XG) * sizeof(double);
    FullCovKernels::with(h->cov_kid(), [&](auto kid) {
        crosscov_kernel<kid><<<(unsigned)(Mp / XG), 256, sm, st>>>(Xc, M, h->kd(), h->ls.as<double>(), h->kern_nls(), h->Xs.as<double>(),
                                                                  h->alpha.as<double>(), h->N, h->Np, h->variance, h->c0,
                                                                  h->jKsT.as<double>(), h->jmean.as<double>(), h->rq_alpha, h->sum, h->srow);
    });
}

static void launch_joint_syrk(gpso_handle* h, cudaStream_t st, int M, int Mp, double jitter) {
    const int mb = Mp / TB;
    FullCovKernels::with(h->cov_kid(), [&](auto kid) {
        joint_syrk_kernel<kid><<<mb * (mb + 1) / 2, GTHREADS, GEMM_SMEM_BYTES, st>>>(h->jVT.as<double>(), h->jXcs.as<double>(), M, Mp,
                                                                                   h->Np, h->kd(), h->variance, jitter,
                                                                                   h->jSigma.as<double>(), h->rq_alpha, h->sum, h->srow);
    });
}

// scaled candidates -> cross-covariance + mean -> V^T = (L^-1 K*)^T -> lower triangle of K** - V^T V (+ jitter I) in jSigma
static int joint_sigma(gpso_handle* h, cudaStream_t st, const double* Xc, int M, double jitter) {
    const int Mp = (M + TB - 1) / TB * TB, Np = h->Np;
    GP_TRY(h->jXcs.ensure((size_t)h->dx() * Mp * sizeof(double)));
    GP_TRY(h->jKsT.ensure((size_t)Mp * Np * sizeof(double)));
    GP_TRY(h->jmean.ensure((size_t)Mp * (h->has_lin() ? 2 : 1) * sizeof(double)));  // Linear terms: the prior variances follow
    GP_TRY(h->jVT.ensure((size_t)Mp * Np * sizeof(double)));
    GP_TRY(h->jSigma.ensure((size_t)Mp * Mp * sizeof(double)));
    GP_TRY(h->jcounter.ensure(sizeof(int)));
    GP_TRY(scale_inputs(h, st, Xc, M, Mp, h->jXcs.as<double>()));
    const double* xk = Xc;
    if (h->embeds()) {
        GP_TRY(h->pX.ensure((size_t)M * h->cand_width() * sizeof(double)));
        GP_TRY(embed_candidates(h, st, Xc, M));
        xk = h->pX.as<double>();
    }
    launch_joint_crosscov(h, st, xk, M, Mp);
    GP_TRY(check_launch(h, "crosscov"));
    GP_TRY(add_linear_offset(h, st, Xc, M, 1.0, h->jmean.as<double>()));
    JointVParams P;
    P.Linv = h->Linv.as<double>();
    P.KsT = h->jKsT.as<double>();
    P.VT = h->jVT.as<double>();
    P.Np = Np;
    P.nb = h->nb;
    P.nct = Mp / TB;
    P.counter = h->jcounter.as<int>();
    CU_TRY(cudaMemsetAsync(h->jcounter.p, 0, sizeof(int), st));
    joint_v_kernel<<<std::min(h->nsm > 0 ? h->nsm : 148, P.nct * P.nb), GTHREADS, GEMM_SMEM_BYTES, st>>>(P);
    GP_TRY(check_launch(h, "joint_v"));
    launch_joint_syrk(h, st, M, Mp, jitter);
    return check_launch(h, "joint_syrk");
}

static int joint_cov(gpso_handle* h, cudaStream_t st, const double* Xc, int M, double* mean, double* cov, bool host) {
    GP_TRY(joint_sigma(h, st, Xc, M, 0.0));
    const int Mp = (M + TB - 1) / TB * TB;
    double* dst = cov;
    if (host) {
        GP_TRY(h->jout.ensure((size_t)M * M * sizeof(double)));
        dst = h->jout.as<double>();
    }
    joint_mirror_kernel<<<dim3((M + 31) / 32, (M + 31) / 32), dim3(32, 8), 0, st>>>(h->jSigma.as<double>(), M, Mp, dst);
    GP_TRY(check_launch(h, "joint_mirror"));
    const cudaMemcpyKind kind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    CU_TRY(cudaMemcpyAsync(mean, h->jmean.p, (size_t)M * sizeof(double), kind, st));
    if (host) CU_TRY(cudaMemcpyAsync(cov, dst, (size_t)M * M * sizeof(double), kind, st));
    return 0;
}

// Sigma = cov + jitter I -> Lc (in place, Cholesky tasks of the persistent kernel on the joint scratch) -> out = mean + Z Lc^T
static int joint_samples(gpso_handle* h, cudaStream_t st, const double* Xc, int M, int S, double jitter, const double* z, double* out) {
    GP_TRY(joint_sigma(h, st, Xc, M, jitter));
    const int Mp = (M + TB - 1) / TB * TB, mb = Mp / TB;
    const int Sp = (S + TB - 1) / TB * TB, nsb = Sp / TB;
    const size_t mat = (size_t)Mp * Mp * sizeof(double);
    gpso_handle::FactorPlan* plan = nullptr;
    GP_TRY(get_factor_plan(h, mb, 0, &plan));
    GP_TRY(h->jLinv.ensure(mat));
    GP_TRY(h->jLinvT.ensure(mat));
    GP_TRY(h->jlogdet.ensure((size_t)mb * sizeof(double)));
    GP_TRY(h->jinfo.ensure(sizeof(int)));
    GP_TRY(h->jZ.ensure((size_t)Sp * Mp * sizeof(double)));
    // the panel solves read whole diagonal blocks of the inverse, whose zero sub-blocks above the diagonal the diagonal task
    // never writes: cleared on every call (Mp^2 doubles, ~1 % of the factorisation's time at any size)
    CU_TRY(cudaMemsetAsync(h->jLinv.p, 0, mat, st));
    CU_TRY(cudaMemsetAsync(h->jinfo.p, 0, sizeof(int), st));
    const DenseParams P = dense_block(h->jSigma.as<double>(), h->jLinv.as<double>(), h->jLinvT.as<double>(), nullptr, Mp, 0, mb);
    GP_TRY(launch_factor(h, st, P, M, plan, h->jstate, h->jlogdet.as<double>(), h->jinfo.as<int>()));
    joint_tril_kernel<<<mb, 256, 0, st>>>(h->jSigma.as<double>(), Mp);
    GP_TRY(check_launch(h, "joint_tril"));
    const long long nz = (long long)Sp * Mp;
    joint_pad_kernel<<<(unsigned)std::min<long long>((nz + 255) / 256, 4096), 256, 0, st>>>(z, S, M, Sp, Mp, h->jZ.as<double>());
    GP_TRY(check_launch(h, "joint_pad"));
    joint_sample_kernel<<<mb * nsb, GTHREADS, GEMM_SMEM_BYTES, st>>>(h->jSigma.as<double>(), h->jZ.as<double>(), h->jmean.as<double>(), M,
                                                                     Mp, S, mb, nsb, out);
    return check_launch(h, "joint_sample");
}

// waits for the stream and reports the pivot status of the last joint_samples
static int joint_pivot_status(gpso_handle* h, cudaStream_t st) {
    int info = 0;
    CU_TRY(cudaMemcpyAsync(&info, h->jinfo.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return pivot_status(info, "posterior covariance + jitter");
}

static int joint_sample_checks(gpso_handle* h, const void* xc, long long M, int S, double jitter, const void* z, const void* out,
                               const char* who) {
    GP_TRY(joint_checks(h, xc, M, z, out, who));
    if (S < 1) return fail(GPSO_E_BADARG, std::string(who) + ": S must be positive");
    if (!(jitter >= 0.0)) return fail(GPSO_E_BADARG, std::string(who) + ": jitter must be a non-negative number");
    return joint_ready(h, who);
}

extern "C" int gpso_predict_f_cov_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double* mean_dev, double* cov_dev, void* stream) {
    GP_TRY(joint_checks(h, Xc_dev, M, mean_dev, cov_dev, "gpso_predict_f_cov_dev"));
    GP_TRY(joint_ready(h, "gpso_predict_f_cov_dev"));
    return joint_cov(h, (cudaStream_t)stream, Xc_dev, (int)M, mean_dev, cov_dev, false);
}

extern "C" int gpso_predict_f_cov_host(gpso_handle* h, const double* Xc_host, int64_t M, double* mean_host, double* cov_host) {
    GP_TRY(joint_checks(h, Xc_host, M, mean_host, cov_host, "gpso_predict_f_cov_host"));
    GP_TRY(joint_ready(h, "gpso_predict_f_cov_host"));
    cudaStream_t st = h->stream;
    GP_TRY(h->jcand.ensure((size_t)M * h->d * sizeof(double)));
    CU_TRY(cudaMemcpyAsync(h->jcand.p, Xc_host, (size_t)M * h->d * sizeof(double), cudaMemcpyHostToDevice, st));
    GP_TRY(joint_cov(h, st, h->jcand.as<double>(), (int)M, mean_host, cov_host, true));
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int gpso_predict_f_samples_dev(gpso_handle* h, const double* Xc_dev, int64_t M, int S, double jitter, const double* z_dev,
                                          double* out_dev, void* stream) {
    GP_TRY(joint_sample_checks(h, Xc_dev, M, S, jitter, z_dev, out_dev, "gpso_predict_f_samples_dev"));
    cudaStream_t st = (cudaStream_t)stream;
    GP_TRY(joint_samples(h, st, Xc_dev, (int)M, S, jitter, z_dev, out_dev));
    return joint_pivot_status(h, st);
}

extern "C" int gpso_predict_f_samples_host(gpso_handle* h, const double* Xc_host, int64_t M, int S, double jitter, const double* z_host,
                                           double* out_host) {
    GP_TRY(joint_sample_checks(h, Xc_host, M, S, jitter, z_host, out_host, "gpso_predict_f_samples_host"));
    cudaStream_t st = h->stream;
    const size_t zbytes = (size_t)S * M * sizeof(double);
    GP_TRY(h->jcand.ensure((size_t)M * h->d * sizeof(double)));
    GP_TRY(h->jzin.ensure(zbytes));
    GP_TRY(h->jout.ensure(zbytes));
    CU_TRY(cudaMemcpyAsync(h->jcand.p, Xc_host, (size_t)M * h->d * sizeof(double), cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemcpyAsync(h->jzin.p, z_host, zbytes, cudaMemcpyHostToDevice, st));
    GP_TRY(joint_samples(h, st, h->jcand.as<double>(), (int)M, S, jitter, h->jzin.as<double>(), h->jout.as<double>()));
    CU_TRY(cudaMemcpyAsync(out_host, h->jout.p, zbytes, cudaMemcpyDeviceToHost, st));
    return joint_pivot_status(h, st);
}

// ---------------------------------------------------------------------------------------------------------------------
// leaves
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int64_t gpso_grow_count(int depth) {
    if (depth < 0 || depth > 38) return -1;
    int64_t n = 0, w = 1;
    for (int l = 0; l < depth; l++) {
        n += w;
        w *= 3;
    }
    return n;
}

static int grow_launch(const double* bounds_host, int d, int depth, double* out_dev, cudaStream_t st, DevBuf& bdev) {
    if (!bounds_host || !out_dev) return fail(GPSO_E_BADARG, "gpso_grow_leaves: null argument");
    if (d <= 0 || d > LEAF_MAXD) return fail(GPSO_E_BADARG, "gpso_grow_leaves: dimension must be in 1..64");
    if (depth < 1 || depth > 20) return fail(GPSO_E_BADARG, "gpso_grow_leaves: depth must be in 1..20");
    for (int j = 0; j < d; j++)
        if (!(bounds_host[2 * j + 1] > bounds_host[2 * j])) return fail(GPSO_E_BADARG, "gpso_grow_leaves: need hi > lo per dimension");
    GP_TRY(bdev.ensure(sizeof(double) * 2 * LEAF_MAXD));
    CU_TRY(cudaMemcpyAsync(bdev.p, bounds_host, sizeof(double) * 2 * d, cudaMemcpyHostToDevice, st));
    long long rows = gpso_grow_count(depth);
    grow_leaves_kernel<<<(unsigned)((rows + 127) / 128), LEAF_THREADS, leaf_smem_bytes(d), st>>>(bdev.as<double>(), d, depth, rows, out_dev);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(GPSO_E_CUDA, std::string("launch of grow_leaves failed: ") + cudaGetErrorString(e));
    return 0;
}

extern "C" int gpso_grow_leaves_dev(int device, const double* bounds_host, int d, int depth, double* out_dev, void* stream) {
    CU_TRY(cudaSetDevice(device));
    GP_TRY(configure_kernels_once(device));
    DevBuf b;
    int rc = grow_launch(bounds_host, d, depth, out_dev, (cudaStream_t)stream, b);
    if (rc == 0) {
        cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);  // bounds buffer is freed below
        if (e != cudaSuccess) rc = fail(GPSO_E_CUDA, cudaGetErrorString(e));
    }
    b.release();
    return rc;
}

extern "C" int gpso_grow_leaves_host(int device, const double* bounds_host, int d, int depth, double* out_host) {
    if (!out_host) return fail(GPSO_E_BADARG, "gpso_grow_leaves_host: null output");
    CU_TRY(cudaSetDevice(device));
    GP_TRY(configure_kernels_once(device));
    long long rows = gpso_grow_count(depth);
    if (rows <= 0) return fail(GPSO_E_BADARG, "gpso_grow_leaves_host: bad depth");
    DevBuf out, b;
    GP_TRY(out.ensure((size_t)rows * d * sizeof(double)));
    int rc = grow_launch(bounds_host, d, depth, out.as<double>(), 0, b);
    if (rc == 0) {
        cudaError_t e = cudaMemcpy(out_host, out.p, (size_t)rows * d * sizeof(double), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(GPSO_E_CUDA, cudaGetErrorString(e));
    }
    out.release();
    b.release();
    return rc;
}

// Rows [row0, row1) of the grow(depth) batch of the box: generated on the device, scored, reduced to their arg-max.  The index
// returned is the row number inside the FULL batch, so the records of several ranks (each with its own row range) merge like
// those of gpso_ucb_argmax_* with a global offset.
extern "C" int gpso_grow_ucb_argmax_range(gpso_handle* h, const double* bounds_host, int d, int depth, double varsigma, int64_t row0,
                                          int64_t row1, double* result_host) {
    if (!h || !bounds_host || !result_host) return fail(GPSO_E_BADARG, "gpso_grow_ucb_argmax: null argument");
    if (!h->factorized) return fail(GPSO_E_STATE, "gpso_grow_ucb_argmax: call gpso_factorize first");
    GP_TRY(begin_scoring(h));
    if (d != h->d) return fail(GPSO_E_BADARG, "gpso_grow_ucb_argmax: dimension differs from the training data");
    const long long total = gpso_grow_count(depth);
    if (total <= 0) return fail(GPSO_E_BADARG, "gpso_grow_ucb_argmax: bad depth");
    if (row0 < 0 || row1 > total || row0 >= row1) return fail(GPSO_E_BADARG, "gpso_grow_ucb_argmax: empty or out-of-range row range");
    const long long rows = row1 - row0;
    GP_TRY(h->leaves.ensure((size_t)rows * d * sizeof(double) + sizeof(double) * 2 * LEAF_MAXD));
    // bounds live at the tail of the leaves buffer
    double* bdev = h->leaves.as<double>() + (size_t)rows * d;
    cudaStream_t st = h->stream;
    for (int j = 0; j < d; j++)
        if (!(bounds_host[2 * j + 1] > bounds_host[2 * j])) return fail(GPSO_E_BADARG, "gpso_grow_ucb_argmax: need hi > lo per dimension");
    if (depth < 1 || depth > 20) return fail(GPSO_E_BADARG, "gpso_grow_ucb_argmax: depth must be in 1..20");
    GP_TRY(timed_call(
        h, st,
        [&] {
            CU_TRY(cudaMemcpyAsync(bdev, bounds_host, sizeof(double) * 2 * d, cudaMemcpyHostToDevice, st));
            grow_leaves_kernel<<<(unsigned)((rows + 127) / 128), LEAF_THREADS, leaf_smem_bytes(d), st>>>(bdev, d, depth, rows,
                                                                                                         h->leaves.as<double>(), row0);
            GP_TRY(check_launch(h, "grow_leaves"));
            return score_argmax(h, st, h->leaves.as<double>(), nullptr, rows, varsigma, result_host);
        },
        [&] { return wait_t1(h); }));
    result_host[0] += (double)row0;
    return 0;
}

extern "C" int gpso_grow_ucb_argmax(gpso_handle* h, const double* bounds_host, int d, int depth, double varsigma,
                                    double* result_host) {
    return gpso_grow_ucb_argmax_range(h, bounds_host, d, depth, varsigma, 0, gpso_grow_count(depth), result_host);
}

// ---------------------------------------------------------------------------------------------------------------------
// multi-GPU state exchange: [ header (128 doubles) | Xs (d*Np) | alpha (Np) | Linv (Np*Np) | A (d, linear mean only)
//                              | component block (sum and product only) ]
// header: N, d, kernel variance, noise variance, mean constant (b of the linear mean), -LML, kernel id, ard, RationalQuadratic
// alpha (0 for the other kernels), mean id, lengthscales from slot 16.  A does not fit beside 64 lengthscales in the header.
// A sum kernel: slot 2 is the prior variance var_tot, Xs holds the C scaled copies (C*d*Np), the header's lengthscales are the
// components' expanded to d entries each, and the component block is [C, then per component: family, lengthscale count,
// variance, alpha, lengthscales].  A product kernel: the same, with slot 2 the prior variance var_prod and the factor variances
// in the component block.  A periodic kernel: the kernel id is its base family's, slot 10 is 1 and slot 11 the period's ARD
// flag, Xs holds the 2d embedded rows (2*d*Np) and the period(s) follow the lengthscale slots (STATE_PERIODS).
// A handle with an active dims map (gpso_set_active_dims): slot 12 is its leaf count, the lengthscale and period counts of the
// component block are those of the active columns, and the map block [leaf count, counts, columns] follows the component block.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int STATE_HEADER = 128;
constexpr int STATE_PERIODS = 16 + MAX_LS;  // a periodic kernel's period(s); slot 10 = 1 marks it, slot 11 = the period's ARD flag

// the family entry of a component in the state's component block: its family id, + 16 for a periodic component (its base's id),
// KERNEL_LINEAR (10) for a Linear component, whose lengthscale slots hold its variance(s)
static int comp_code(const gpso_handle* h, int c) { return h->sum.fam[c] + (h->sum_per[c] ? 16 : 0); }
// the block entries of component c: family, lengthscale count, variance, alpha, lengthscales, [period count, periods]
static int comp_block(const gpso_handle* h, int c, int d) {
    const int k = h->cdim(c, d);
    return 4 + (h->sum_ard[c] ? k : 1) + (h->sum_per[c] ? 1 + (h->sum_per_ard[c] ? k : 1) : 0);
}

static long long sum_block_size(const gpso_handle* h, int d) {
    if (!h->composite()) return 0;
    long long n = 1;
    for (int c = 0; c < h->sum.n; c++) n += comp_block(h, c, d);
    return n;
}

// slots 12..14 of the state header: leaf count, column count and a fingerprint of the map (exact in a double), so that a state with
// another map is refused before its layout is read
static void map_header(const gpso_handle* h, double* out3) {
    long long f = 0;
    const long long P = (1LL << 52) - 47;
    for (int c = 0; c < h->nmap; c++) f = (f * 131 + h->map_n[c]) % P;
    for (int col : h->map_cols) f = (f * 131 + col + 1) % P;
    out3[0] = h->nmap;
    out3[1] = h->nmap ? (double)h->map_cols.size() : 0.0;
    out3[2] = (double)f;
}

static long long map_block_size(const gpso_handle* h) { return h->nmap ? 1 + h->nmap + (long long)h->map_cols.size() : 0; }

static std::vector<double> map_block(const gpso_handle* h) {
    std::vector<double> m;
    if (!h->nmap) return m;
    m.push_back(h->nmap);
    for (int c = 0; c < h->nmap; c++) m.push_back(h->map_n[c]);
    for (int col : h->map_cols) m.push_back(col);
    return m;
}

extern "C" int gpso_state_bytes(gpso_handle* h, int N, int d, int64_t* bytes) {
    if (!h || !bytes || N <= 0 || d <= 0) return fail(GPSO_E_BADARG, "gpso_state_bytes: bad argument");
    long long Np = ((N + TB - 1) / TB) * TB;
    if (h->periodic && 2 * d > MAX_LS)
        return fail(GPSO_E_BADARG, "gpso_state_bytes: a periodic kernel embeds each input dimension in 2 rows: input dimension up to 32");
    const long long dx = h->rows_for(d);
    *bytes = (int64_t)sizeof(double) * (STATE_HEADER + dx * Np + Np + Np * Np + (h->linear() ? d : 0) + sum_block_size(h, d) +
                                        map_block_size(h));
    return 0;
}

extern "C" int gpso_export_state_dev(gpso_handle* h, void* dst_dev, int64_t bytes, void* stream) {
    if (!h || !dst_dev) return fail(GPSO_E_BADARG, "gpso_export_state_dev: null argument");
    if (!h->factorized) return fail(GPSO_E_STATE, "gpso_export_state_dev: call gpso_factorize first");
    GP_TRY(set_device(h));
    int64_t need = 0;
    gpso_state_bytes(h, h->N, h->d, &need);
    if (bytes < need) return fail(GPSO_E_BADARG, "gpso_export_state_dev: destination too small");
    cudaStream_t st = (cudaStream_t)stream;
    double hdr[STATE_HEADER] = {0};
    hdr[0] = h->N;
    hdr[1] = h->d;
    hdr[2] = h->variance;
    hdr[3] = h->noise;
    hdr[4] = h->c0;
    hdr[5] = h->factor_nlml;
    hdr[6] = h->bare_lin ? GPSO_KERNEL_LINEAR : h->kernel_id;
    hdr[7] = h->ard;
    if (h->n_rq()) hdr[8] = h->rq_alpha;
    hdr[9] = h->mean_id;
    for (int i = 0; i < h->n_ls(); i++) hdr[16 + i] = h->ls_host[i];
    if (h->periodic) {
        hdr[10] = 1.0;
        hdr[11] = h->per_ard;
        for (int i = 0; i < h->n_per(); i++) hdr[STATE_PERIODS + i] = h->per_p[i];
    }
    map_header(h, hdr + 12);
    double* dst = (double*)dst_dev;
    CU_TRY(cudaStreamSynchronize(h->stream));
    CU_TRY(cudaMemcpyAsync(dst, hdr, sizeof hdr, cudaMemcpyHostToDevice, st));
    size_t Np = h->Np;
    const size_t dx = h->dx();
    CU_TRY(cudaMemcpyAsync(dst + STATE_HEADER, h->Xs.p, sizeof(double) * dx * Np, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaMemcpyAsync(dst + STATE_HEADER + dx * Np, h->alpha.p, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaMemcpyAsync(dst + STATE_HEADER + dx * Np + Np, h->Linv.p, sizeof(double) * Np * Np, cudaMemcpyDeviceToDevice, st));
    if (h->linear())
        CU_TRY(cudaMemcpyAsync(dst + STATE_HEADER + dx * Np + Np + Np * Np, h->meanA.p, sizeof(double) * h->d, cudaMemcpyDeviceToDevice, st));
    std::vector<double> blk;
    if (h->composite()) {
        blk.push_back(h->sum.n);
        for (int c = 0; c < h->sum.n; c++) {
            const int nl = h->comp_ls(c);
            blk.insert(blk.end(), {(double)comp_code(h, c), (double)nl, h->comp_var(c), h->sum.alpha[c]});
            for (int i = 0; i < nl; i++) blk.push_back(h->ls_host[h->ls_off(c) + i]);
            if (h->sum_per[c]) {  // a periodic component: its period count and period(s)
                blk.push_back(h->comp_np(c));
                for (int i = 0; i < h->comp_np(c); i++) blk.push_back(h->comp_p[c][i]);
            }
        }
        const std::vector<double> mb = map_block(h);
        blk.insert(blk.end(), mb.begin(), mb.end());
        CU_TRY(cudaMemcpyAsync(dst + STATE_HEADER + dx * Np + Np + Np * Np + (h->linear() ? h->d : 0), blk.data(),
                               sizeof(double) * blk.size(), cudaMemcpyHostToDevice, st));
    }
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int gpso_import_state_dev(gpso_handle* h, const void* src_dev, int64_t bytes, int N, int d, void* stream) {
    if (!h || !src_dev) return fail(GPSO_E_BADARG, "gpso_import_state_dev: null argument");
    if (N <= 0 || d <= 0 || d > MAX_LS || (h && h->rows_for(d) > MAX_LS))
        return fail(GPSO_E_BADARG, "gpso_import_state_dev: bad shape");
    GP_TRY(set_device(h));
    cudaStream_t st = (cudaStream_t)stream;
    const double* src = (const double*)src_dev;
    double hdr[STATE_HEADER];
    if (bytes >= (int64_t)sizeof hdr) {  // the map decides the layout of the rest: compare it first
        double mh[3];
        map_header(h, mh);
        CU_TRY(cudaMemcpyAsync(hdr, src, sizeof hdr, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        if (hdr[12] != mh[0] || hdr[13] != mh[1] || hdr[14] != mh[2])
            return fail(GPSO_E_BADARG, "gpso_import_state_dev: active dims mismatch");
    }
    int64_t need = 0;
    gpso_state_bytes(h, N, d, &need);
    if (bytes < need) return fail(GPSO_E_BADARG, "gpso_import_state_dev: source too small");
    CU_TRY(cudaStreamSynchronize(h->stream));
    GP_TRY(ensure_shape(h, N, d));
    if ((int)hdr[0] != N || (int)hdr[1] != d) return fail(GPSO_E_BADARG, "gpso_import_state_dev: header shape mismatch");
    if ((int)hdr[6] != (h->bare_lin ? GPSO_KERNEL_LINEAR : h->kernel_id) || (int)hdr[7] != h->ard)
        return fail(GPSO_E_BADARG, "gpso_import_state_dev: kernel mismatch");
    if ((hdr[10] == 1.0) != h->periodic || (h->periodic && (int)hdr[11] != h->per_ard))
        return fail(GPSO_E_BADARG, "gpso_import_state_dev: periodic kernel mismatch");
    if (((int)hdr[9] == GPSO_MEAN_LINEAR) != h->linear())
        return fail(GPSO_E_BADARG, "gpso_import_state_dev: linear mean function on one side only");
    const size_t dx = h->dx();
    std::vector<double> blk(sum_block_size(h, d) + map_block_size(h));
    if (h->composite()) {
        // the component block: the same count, families and lengthscale counts (ARD flags) as this handle's, or no import
        CU_TRY(cudaMemcpyAsync(blk.data(), src + STATE_HEADER + dx * h->Np + h->Np + (size_t)h->Np * h->Np + (h->linear() ? d : 0),
                               sizeof(double) * blk.size(), cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        // a map: the same map as this handle's, or no import (the component block's counts depend on it, so it is compared first)
        const std::vector<double> mb = map_block(h);
        if (!std::equal(mb.begin(), mb.end(), blk.end() - mb.size()))
            return fail(GPSO_E_BADARG, "gpso_import_state_dev: active dims mismatch");
        bool same = (int)blk[0] == h->sum.n;
        for (int c = 0, q = 1; same && c < h->sum.n; q += comp_block(h, c, d), c++) {
            const int k = h->cdim(c, d);
            same = (int)blk[q] == comp_code(h, c) && (int)blk[q + 1] == (h->sum_ard[c] ? k : 1) &&
                   (!h->sum_per[c] || (int)blk[q + 4 + (h->sum_ard[c] ? k : 1)] == (h->sum_per_ard[c] ? k : 1));
        }
        if (!same)
            return fail(GPSO_E_BADARG, h->is_sum() ? "gpso_import_state_dev: sum kernel component mismatch"
                                                   : "gpso_import_state_dev: product kernel component mismatch");
        for (int c = 0, q = 1; c < h->sum.n; q += comp_block(h, c, d), c++) {
            const int k = h->cdim(c, d);
            for (int i = 0; h->sum_per[c] && i < (h->sum_per_ard[c] ? k : 1); i++) h->comp_p[c][i] = blk[q + 5 + (h->sum_ard[c] ? k : 1) + i];
            if (h->is_product())  // the table's variances are {var_prod, 1, 1, 1}, var_prod from slot 2
                h->prod_var[c] = blk[q + 2];
            else
                h->sum.var[c] = blk[q + 2];
            h->sum.alpha[c] = blk[q + 3];
        }
    }
    h->variance = hdr[2];
    if (h->is_product())
        for (int c = 0; c < h->sum.n; c++) h->sum.var[c] = (c == 0) ? h->variance : 1.0;
    h->noise = hdr[3];
    h->c0 = hdr[4];
    h->factor_nlml = hdr[5];
    if (h->n_rq()) h->rq_alpha = hdr[8];
    for (int i = 0; i < h->n_ls(); i++) h->ls_host[i] = hdr[16 + i];
    for (int i = 0; i < h->n_per(); i++) h->per_p[i] = hdr[STATE_PERIODS + i];
    size_t Np = h->Np;
    CU_TRY(cudaMemcpyAsync(h->Xs.p, src + STATE_HEADER, sizeof(double) * dx * Np, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaMemcpyAsync(h->alpha.p, src + STATE_HEADER + dx * Np, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
    CU_TRY(cudaMemcpyAsync(h->Linv.p, src + STATE_HEADER + dx * Np + Np, sizeof(double) * Np * Np, cudaMemcpyDeviceToDevice, st));
    if (h->linear()) {
        CU_TRY(cudaMemcpyAsync(h->meanA.p, src + STATE_HEADER + dx * Np + Np + Np * Np, sizeof(double) * d, cudaMemcpyDeviceToDevice, st));
        CU_TRY(cudaMemcpyAsync(h->A_host, h->meanA.p, sizeof(double) * d, cudaMemcpyDeviceToHost, st));
    }
    GP_TRY(upload_lengthscales(h, st));
    CU_TRY(cudaStreamSynchronize(st));
    GP_TRY(prepare_ozaki(h, st));  // the digit tiles are rebuilt locally from the imported L^-1 (bit-identical on every rank)
    CU_TRY(cudaStreamSynchronize(st));
    h->have_data = false;  // no raw training data on this rank: predict only
    h->factorized = true;
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// introspection
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int64_t gpso_launch_count(gpso_handle* h) { return h ? h->launches : 0; }

extern "C" int gpso_debug_fetch(gpso_handle* h, int which, double* out_host, int64_t count) {
    if (!h || !out_host) return fail(GPSO_E_BADARG, "gpso_debug_fetch: null argument");
    GP_TRY(set_device(h));
    CU_TRY(cudaStreamSynchronize(h->stream));
    const int N = h->N, Np = h->Np;
    if (which == 5) {  // screened value (UCB, or mean for the bound level) of the first `count` candidates of the last screened call
        // scr_ucb outlives the call that wrote it: refuse rows the last fused call did not screen (unscreened call, early stop)
        if (count < 0 || count > h->scr_rows)
            return fail(GPSO_E_STATE, "gpso_debug_fetch: the last fused call screened " + std::to_string(h->scr_rows) + " candidates, not " +
                                          std::to_string(count));
        CU_TRY(cudaMemcpy(out_host, h->scr_ucb.p, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost));
        return 0;
    }
    if (which == 3) {
        if (count < N) return fail(GPSO_E_BADARG, "gpso_debug_fetch: buffer too small");
        CU_TRY(cudaMemcpy(out_host, h->alpha.p, sizeof(double) * N, cudaMemcpyDeviceToHost));
        return 0;
    }
    const DevBuf* src = which == 1 ? &h->K : which == 2 ? &h->Linv : which == 4 ? &h->Kinv : nullptr;
    if (!src || !src->p) return fail(GPSO_E_BADARG, "gpso_debug_fetch: unknown or unavailable matrix");
    if (count < (int64_t)N * N) return fail(GPSO_E_BADARG, "gpso_debug_fetch: buffer too small");
    CU_TRY(cudaMemcpy2D(out_host, sizeof(double) * N, src->p, sizeof(double) * Np, sizeof(double) * N, N, cudaMemcpyDeviceToHost));
    for (int i = 0; i < N; i++)
        for (int j = i + 1; j < N; j++) out_host[(size_t)i * N + j] = 0.0;  // only the lower triangle is defined
    return 0;
}

extern "C" int gpso_last_timing(gpso_handle* h, double* out_ms4) {
    if (!h || !out_ms4) return fail(GPSO_E_BADARG, "gpso_last_timing: null argument");
    for (int i = 0; i < 4; i++) out_ms4[i] = h->last_ms[i];
    return 0;
}

extern "C" int gpso_set_profile(gpso_handle* h, int enabled) {
    if (!h) return fail(GPSO_E_BADARG, "gpso_set_profile: null handle");
    h->profile = enabled == 1;  // per-stage events, windows run in order
    h->trace = enabled == 2;    // timeline events on the side streams, overlap kept
    return 0;
}

extern "C" int64_t gpso_debug_trace(gpso_handle* h, double* out, int64_t capacity) {
    if (!h) return -1;
    int64_t n = (int64_t)h->trace_out.size();
    if (out)
        for (int64_t i = 0; i < n && i < capacity; i++) out[i] = h->trace_out[i];
    return n;
}

extern "C" int64_t gpso_last_windows(gpso_handle* h) { return h ? h->last_windows : 0; }

extern "C" int gpso_set_predict_mode(gpso_handle* h, int mode, int slices) {
    if (!h || mode < 0 || mode > 2) return fail(GPSO_E_BADARG, "gpso_set_predict_mode: mode must be 0 (auto), 1 (fp64 DMMA) or 2 (int8 tcgen05)");
    if (slices != 0 && (slices < 5 || slices > 8)) return fail(GPSO_E_BADARG, "gpso_set_predict_mode: slices must be 0 (auto) or 5..8");
    if (mode == 2 && h->has_lin())
        return fail(GPSO_E_BADARG, "gpso_set_predict_mode: a kernel with a Linear term has no bound on |k*| for the int8 engine: modes 0 and 1 only");
    h->predict_mode = mode;
    h->oz_force_slices = slices;
    h->factorized = false;  // takes effect at the next gpso_factorize
    return 0;
}

extern "C" int gpso_set_overlap(gpso_handle* h, int enabled) {
    if (!h) return fail(GPSO_E_BADARG, "gpso_set_overlap: null handle");
    h->overlap = enabled != 0;
    return 0;
}

extern "C" int gpso_set_factor_mode(gpso_handle* h, int mode) {
    if (!h || mode < 0 || mode > 3) return fail(GPSO_E_BADARG, "gpso_set_factor_mode: bad argument");
    h->factor_mode = mode;
    return 0;
}

extern "C" int gpso_trim_pool(int device, int64_t* cached_bytes_before) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n || device >= POOL_MAX_DEV)
        return fail(GPSO_E_BADARG, "gpso_trim_pool: device index out of range");
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaDeviceSynchronize());
    if (cached_bytes_before) {
        std::lock_guard<std::mutex> lock(g_pool.mu);
        *cached_bytes_before = (int64_t)g_pool.cached[device];
    }
    g_pool.flush(device);
    return 0;
}

extern "C" int gpso_factor_info(gpso_handle* h, int* out2) {
    if (!h || !out2) return fail(GPSO_E_BADARG, "gpso_factor_info: null argument");
    out2[0] = h->factor_mode == 0 ? 0 : (h->hybrid_nodes > 0 ? 2 : 1);
    out2[1] = h->hybrid_nodes;
    return 0;
}

// Host-only introspection (no GPU needed) of the tile -> CTA tables of the int8 fit-path products.  kind 0: K_y^-1 (one
// int per slot: row block << 16 | column tile, -1 empty; levels = 1, info = {rounds});  kind 1: inverse factor (four ints
// per slot: row block, 64-row tile of B, first k-step, k-steps; info = per level {s, xt_offset, xt_rounds, y_offset, y_rounds},
// offsets in ints).  Returns the number of ints of the table; copies min(capacity, that) ints.
extern "C" int64_t gpso_debug_product_items(int kind, int nb, int nsm, int* out, int64_t capacity, int* info, int info_capacity,
                                            int* levels_out) {
    if (nb < 1 || nb > 255 || nsm < 1) return fail(GPSO_E_BADARG, "gpso_debug_product_items: bad argument");
    std::vector<int> flat;
    std::vector<int> meta;
    if (kind == 0) {
        int rounds = 0;
        make_lauum_items(nb, nsm, flat, rounds);
        meta.push_back(rounds);
        if (levels_out) *levels_out = 1;
    } else if (kind == 1) {
        std::vector<InvLevelInfo> levels;
        make_inverse_items(nb, nsm, flat, levels);
        for (const InvLevelInfo& lv : levels) {
            meta.push_back(lv.s);
            meta.push_back((int)lv.xt_off);
            meta.push_back(lv.xt_rounds);
            meta.push_back((int)lv.y_off);
            meta.push_back(lv.y_rounds);
        }
        if (levels_out) *levels_out = (int)levels.size();
    } else {
        return fail(GPSO_E_BADARG, "gpso_debug_product_items: kind must be 0 or 1");
    }
    if (out)
        for (int64_t i = 0; i < (int64_t)flat.size() && i < capacity; i++) out[i] = flat[i];
    if (info)
        for (int i = 0; i < (int)meta.size() && i < info_capacity; i++) info[i] = meta[i];
    return (int64_t)flat.size();
}

extern "C" int gpso_set_kinv_mode(gpso_handle* h, int mode) {
    if (!h || mode < 0 || mode > 2) return fail(GPSO_E_BADARG, "gpso_set_kinv_mode: mode must be 0 (auto), 1 (fp64 DMMA) or 2 (int8 tcgen05)");
    h->kinv_mode = mode;
    return 0;
}

extern "C" int gpso_set_inverse_mode(gpso_handle* h, int mode) {
    if (!h || mode < 0 || mode > 2) return fail(GPSO_E_BADARG, "gpso_set_inverse_mode: mode must be 0 (auto), 1 (fp64 DMMA) or 2 (int8 tcgen05)");
    h->inverse_mode = mode;
    h->factorized = false;
    return 0;
}

extern "C" int gpso_set_l2_window(gpso_handle* h, int enabled) {
    if (!h) return fail(GPSO_E_BADARG, "gpso_set_l2_window: null handle");
    h->l2_window = enabled != 0;
    if (!enabled && h->stream) {
        cudaStreamAttrValue attr;
        memset(&attr, 0, sizeof attr);
        CU_TRY(cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &attr));
    }
    h->factorized = false;
    return 0;
}

extern "C" int gpso_predict_info(gpso_handle* h, double* out3) {
    if (!h || !out3) return fail(GPSO_E_BADARG, "gpso_predict_info: null argument");
    out3[0] = h->oz_S ? 2.0 : 1.0;
    out3[1] = (double)h->oz_S;
    out3[2] = h->oz_est;
    return 0;
}

extern "C" int gpso_set_screen_mode(gpso_handle* h, int mode) {
    if (!h || mode < 0 || mode > SCREEN_MODE_FULL2)
        return fail(GPSO_E_BADARG, "gpso_set_screen_mode: mode must be 0 (off), 1 (automatic), 2..4 (digits), 5 (mean bound first) or 6 (2 digits, all pairs)");
    if (mode >= 2 && h->has_lin())
        return fail(GPSO_E_BADARG, "gpso_set_screen_mode: a kernel with a Linear term is not screened (its prior variance differs per candidate): modes 0 and 1 only");
    h->screen_mode = mode;
    h->screen_S_cur = 0;
    if (h->nb > 0) g_screen_hint[std::min(h->nb, 64)] = ScreenHint();  // an explicit call restarts the ladder for this matrix size
    h->factorized = false;  // the fp32 copies are prepared by the next gpso_factorize
    return 0;
}

extern "C" int gpso_screen_info(gpso_handle* h, double* out12) {
    if (!h || !out12) return fail(GPSO_E_BADARG, "gpso_screen_info: null argument");
    for (int i = 0; i < 12; i++) out12[i] = h->scr_info[i];
    return 0;
}

// Pipe peaks of this GPU, measured now (best of 3 launches each, CUDA events on the default stream; ~0.2 s in total):
// out[0] int8 tensor TOP/s (tcgen05 kind::i8, M=128 N=256, one issuing thread per SM), out[1] FP64 TFLOP/s (DMMA.8x8x4),
// out[2] L2 -> shared-memory bulk-copy GB/s (24 KB chunks, 8 in flight per SM, 64 MB working set), out[3] number of SMs.
extern "C" int gpso_probe_peaks(int device, double* out4) {
    if (!out4) return fail(GPSO_E_BADARG, "gpso_probe_peaks: null argument");
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    const int nsm = prop.multiProcessorCount;
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    DevBuf sink, dout, src;
    GP_TRY(sink.ensure(64, true));
    auto best_of = [&](auto launch, double* best_ms) -> int {
        *best_ms = 1e30;
        for (int r = 0; r < 4; r++) {  // the first launch warms up
            CU_TRY(cudaEventRecord(e0, 0));
            launch();
            CU_TRY(cudaEventRecord(e1, 0));
            CU_TRY(cudaEventSynchronize(e1));
            if (cudaGetLastError() != cudaSuccess) return fail(GPSO_E_CUDA, "gpso_probe_peaks: probe launch failed");
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (r > 0) *best_ms = std::min(*best_ms, (double)ms);
        }
        return 0;
    };
    double ms = 0.0;
    // int8 tensor pipe
    const int iters8 = 200000;
    const int smem8 = 2 * (4096 + 256 * 32);
    CU_TRY(cudaFuncSetAttribute(probe_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem8));
    GP_TRY(best_of([&] { probe_i8_kernel<<<nsm, 128, smem8>>>(iters8, sink.as<int>()); }, &ms));
    out4[0] = 2.0 * 128 * 256 * 32 * (double)(iters8 / 2 * 2) * nsm / (ms * 1e-3) / 1e12;
    // FP64 pipe
    const int iters64 = 20000, blocks = nsm * 4;
    GP_TRY(dout.ensure((size_t)blocks * 256 * sizeof(double)));
    GP_TRY(best_of([&] { probe_dmma_kernel<<<blocks, 256>>>(dout.as<double>(), iters64, 1.0000001, 0.9999999); }, &ms));
    out4[1] = 2.0 * 8 * 8 * 4 * 16.0 * iters64 * (double)blocks * 8 / (ms * 1e-3) / 1e12;
    // L2 -> SMEM bulk copies
    const int chunk = 24576, per_cta = 4096;
    const size_t bytes = (size_t)64 << 20;
    GP_TRY(src.ensure(bytes, true));
    CU_TRY(cudaFuncSetAttribute(probe_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * chunk));
    GP_TRY(best_of([&] { probe_bulk_kernel<<<nsm, 128, 8 * chunk>>>(src.as<uint8_t>(), bytes / chunk, chunk, per_cta); }, &ms));
    out4[2] = (double)per_cta * nsm * chunk / (ms * 1e-3) / 1e9;
    out4[3] = nsm;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return 0;
}

extern "C" int gpso_set_window(gpso_handle* h, int64_t candidates) {
    if (!h || candidates < 0) return fail(GPSO_E_BADARG, "gpso_set_window: bad argument");
    h->window_override = candidates;
    return 0;
}
