/*
 * gpso_b200.h -- C ABI of the B200-native Gaussian-process surrogate hot path of pyGPSO.
 *
 * One opaque handle = one GPR surrogate on one GPU (training data, Cholesky factor L, inverse factor L^-1, alpha and
 * all workspaces live in that GPU's HBM for the life of the handle).  Plain C: pointers, sizes, status codes; no
 * C++ / torch types cross this boundary.  A handle is not thread-safe; use one per surrogate per GPU.
 *
 * The reference (jajcayn/pygpso, pure Python) has no FFI for this path; the seam is the Python attribute
 * GPSurrogate.gpflow_model (gpso/gp_surrogate.py:163).  Each entry point below names the reference call it replaces.
 *
 * Conventions
 *   - all matrices are row-major (C-contiguous) fp64, exactly like the numpy arrays the reference passes around;
 *   - "_host"  : the pointer is host memory (pageable or pinned); the call does its own H2D/D2H and returns when the
 *                outputs are valid;
 *     "_dev"   : device memory of the handle's GPU; the call is enqueued on `stream` (a cudaStream_t passed as void*,
 *                NULL = default stream) and is asynchronous unless stated;
 *   - return value: 0 = GPSO_OK; >0 = LAPACK-style info, the Gram matrix is not positive definite at column `info`
 *                (1-based); <0 = GPSO_E_* below.  No exception crosses the ABI; gpso_last_error() gives the text.
 *   - hyper-parameter vectors are packed in GPflow's trainable_variables order:
 *         [ lengthscale(s) (1, or d when ard) , kernel variance , likelihood (noise) variance , mean constant (if any) ]
 *     `u`     = unconstrained (softplus pre-image; noise variance has the 1e-6 floor of gpflow.likelihoods.Gaussian),
 *     `theta` = constrained values.
 */
#ifndef GPSO_B200_H
#define GPSO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gpso_handle gpso_handle;

enum {
    GPSO_OK = 0,
    GPSO_E_BADARG = -1,   /* null pointer, size <= 0, wrong length ...            */
    GPSO_E_CUDA = -2,     /* a CUDA runtime call failed (text in gpso_last_error) */
    GPSO_E_STATE = -3,    /* call order violated (e.g. predict before factorize)  */
    GPSO_E_NOGPU = -4,    /* no usable sm_100 device                              */
    GPSO_E_NOMEM = -5
};

/* gpflow.kernels.* accepted by GPRSurrogate(gp_kernel=...), gp_surrogate.py:393-402, default Matern52 (:424) */
enum { GPSO_KERNEL_MATERN12 = 0, GPSO_KERNEL_MATERN32 = 1, GPSO_KERNEL_MATERN52 = 2, GPSO_KERNEL_SE = 3 };
/* gpflow.mean_functions.*: None/Zero or Constant (:167, :427) */
enum { GPSO_MEAN_ZERO = 0, GPSO_MEAN_CONSTANT = 1 };

/* ---- library ------------------------------------------------------------------------------------------------- */
int gpso_version(void);                 /* ABI version, currently 1 */
const char* gpso_last_error(void);      /* thread-local text of the last failure */
int gpso_device_count(void);            /* number of CUDA devices, or GPSO_E_* */

/* ---- life cycle: replaces gpflow.models.GPR(...) construction, gp_surrogate.py:490-495 ----------------------- */
int gpso_create(int device, int kernel_id, int ard, int mean_id, gpso_handle** out);
int gpso_destroy(gpso_handle* h);

/* model.data = (x, y), gp_surrogate.py:498.  X_host[N,d], y_host[N] are copied to the device. */
int gpso_set_data(gpso_handle* h, const double* X_host, const double* y_host, int N, int d);

/* ---- fit: the closure scipy's L-BFGS-B calls, i.e. model.training_loss + TF autodiff, gp_surrogate.py:500-503 -- */
/* f = -log marginal likelihood at unconstrained u[p]; grad[p] = df/du.  Host in, host out, synchronous.            */
int gpso_neg_lml_grad(gpso_handle* h, const double* u_host, int p, double* f_host, double* grad_host);

/* Fix the hyper-parameters used by the predict calls: Gram -> Cholesky -> L^-1 -> alpha, cached on the device.
 * (GPflow re-factorises inside every predict_y call; here it is done once per parameter change.) */
int gpso_factorize(gpso_handle* h, const double* theta_host, int p);
/* -LML at the factorised theta (valid after gpso_factorize). */
int gpso_factor_lml(gpso_handle* h, double* lml_host);

/* ---- predict: model.predict_y(Xnew), gp_surrogate.py:298 (noise variance included) ---------------------------- */
int gpso_predict_y_host(gpso_handle* h, const double* Xc_host, int64_t M, double* mean_host, double* var_host);
int gpso_predict_y_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double* mean_dev, double* var_dev,
                       void* stream);

/* ---- joint posterior: model.predict_f(Xnew, full_cov=True) and model.predict_f_samples(Xnew, S) (GPflow 2 GPR) ---- */
/* Candidates per call of the joint entry points: the M x M covariance, its Cholesky factor and V = L^-1 K(X, X*) stay on the
 * device (~2.5 GB at M = N = 8192); more candidates are drawn in batches. */
#define GPSO_MAX_JOINT 8192
/* model.predict_f(Xnew, full_cov=True): mean[M], cov[M*M] row-major, both triangles written (exactly symmetric).
 * cov = K(X*, X*) - A^T A, A = L^-1 K(X, X*) (no noise variance).  Valid after gpso_factorize; 1 <= M <= GPSO_MAX_JOINT.
 * The fitted state of the handle is not modified; the FP64 L^-1 is used whatever gpso_set_predict_mode selected. */
int gpso_predict_f_cov_host(gpso_handle* h, const double* Xc_host, int64_t M, double* mean_host, double* cov_host);
int gpso_predict_f_cov_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double* mean_dev, double* cov_dev, void* stream);
/* model.predict_f_samples(Xnew, S): out[s*M + m] = mean[m] + sum_k Lc[m][k] * z[s*M + k],  Lc = chol(cov + jitter*I).
 * z[S,M] standard normals supplied by the caller; jitter >= 0.  Returns info > 0 (LAPACK pivot) when cov + jitter*I is
 * not positive definite.  The _dev form is synchronous on `stream` at return (it reads the pivot status). */
int gpso_predict_f_samples_host(gpso_handle* h, const double* Xc_host, int64_t M, int S, double jitter, const double* z_host,
                                double* out_host);
int gpso_predict_f_samples_dev(gpso_handle* h, const double* Xc_dev, int64_t M, int S, double jitter, const double* z_dev,
                               double* out_dev, void* stream);

/* ---- exploitation step: gp_eval_best_ucb(normed_coords), gp_surrogate.py:313-328 ------------------------------ */
/* ucb = mean + varsigma * var ; winner = FIRST index of the maximum (np.argmax; a NaN wins like in numpy).
 * result_host[4] = { (double)index, mean, var, ucb }.  The cross-covariance is never materialised beyond a
 * rolling window of candidates; mean/var of the non-winners are not written anywhere. */
int gpso_ucb_argmax_host(gpso_handle* h, const double* Xc_host, int64_t M, double varsigma, double* result_host);
/* Device-resident candidates.  Synchronous on `stream` at return (the 4 result doubles are copied back). */
int gpso_ucb_argmax_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double varsigma, double* result_host,
                        void* stream);
/* Top-k variant (the multi-GPU path gathers k records per rank): the k candidates with the highest UCB in the order
 * np.argsort(-ucb, kind="stable") would visit them (first NaN, larger UCB, lowest index on ties), 1 <= k <= 64.
 * result_host[4*i + 0..3] = (index, mean, var, ucb) of the i-th best; *found = min(k, M).  Record 0 equals
 * gpso_ucb_argmax_* bit for bit. */
int gpso_ucb_topk_host(gpso_handle* h, const double* Xc_host, int64_t M, double varsigma, int k, double* result_host, int* found);
int gpso_ucb_topk_dev(gpso_handle* h, const double* Xc_dev, int64_t M, double varsigma, int k, double* result_host, int* found,
                      void* stream);

/* ---- leaf-coordinate batching: LeafNode.grow(depth), param_space.py:175-200 (+ ternary_split :257-307) -------- */
/* bounds_host[d,2] = (lo,hi) per dimension of the leaf; out[(3^depth-1)/2, d] = centres in the reference's order
 * (level by level, parents in order, children l,c,r), bit-identical to the Python arithmetic (no FMA contraction). */
int64_t gpso_grow_count(int depth);
int gpso_grow_leaves_host(int device, const double* bounds_host, int d, int depth, double* out_host);
int gpso_grow_leaves_dev(int device, const double* bounds_host, int d, int depth, double* out_dev, void* stream);
/* child.grow(depth) fused with gp_eval_best_ucb: optimisation.py:379-381.  Leaves never leave the device. */
int gpso_grow_ucb_argmax(gpso_handle* h, const double* bounds_host, int d, int depth, double varsigma,
                         double* result_host);
/* The same for rows [row0, row1) of the batch only (a rank of a candidate-sharded run scores its own slice of the leaf batch,
 * reference call site gpso/optimisation.py:379-381); result_host[0] is the row number inside the FULL batch. */
int gpso_grow_ucb_argmax_range(gpso_handle* h, const double* bounds_host, int d, int depth, double varsigma, int64_t row0,
                               int64_t row1, double* result_host);

/* ---- multi-GPU: share one fit with the ranks that score candidate shards -------------------------------------- */
/* The fitted state (theta, scaled training inputs, alpha, L^-1) is exposed as ONE contiguous device buffer so the host
 * side can broadcast it with a single NCCL call (torch.distributed.broadcast) and import it on the other ranks. */
int gpso_state_bytes(gpso_handle* h, int N, int d, int64_t* bytes);   /* size for a given problem shape */
int gpso_export_state_dev(gpso_handle* h, void* dst_dev, int64_t bytes, void* stream);
int gpso_import_state_dev(gpso_handle* h, const void* src_dev, int64_t bytes, int N, int d, void* stream);

/* ---- introspection for benchmarks / tests ---------------------------------------------------------------------- */
/* kernel launches issued by this handle since creation (our own kernels only; memcpy/memset not counted) */
int64_t gpso_launch_count(gpso_handle* h);
/* copy device-side intermediates to the host for parity tests: which = 1 L (N*N, lower), 2 L^-1 (N*N, lower),
 * 3 alpha (N), 4 K_y^-1 (N*N, lower; valid after gpso_neg_lml_grad) */
int gpso_debug_fetch(gpso_handle* h, int which, double* out_host, int64_t count);
/* elapsed device time in ms of the last gpso_ucb_argmax_* / gpso_predict_y_* / gpso_neg_lml_grad call (CUDA events on
 * the launching stream): out[0]=total; with gpso_set_profile(h,1) also the per-stage sums over all windows:
 * out[1]=cross-covariance generation, out[2]=triangular product + reduction (the dominant kernel, one launch per
 * window), out[3]=finalise/argmax.  gpso_last_windows = number of windows (= launches of each stage) of that call. */
int gpso_last_timing(gpso_handle* h, double* out_ms4);
int gpso_set_profile(gpso_handle* h, int enabled);
int64_t gpso_last_windows(gpso_handle* h);
/* gpso_set_profile(h, 2): record a timeline of the window pipeline of the next scoring calls without giving up the stream
 * overlap.  gpso_debug_trace copies (tag, window, ms since the first event) triples of the last call to out (capacity in
 * doubles) and returns how many doubles the trace holds; tags: 1/2 cross-covariance start/end (side stream), 3/4
 * variance product start/end, 5 finalise + arg-max merge end (product stream). */
int64_t gpso_debug_trace(gpso_handle* h, double* out, int64_t capacity);
/* Engine of the variance product V = L^-1 k* inside predict_y / ucb_argmax (takes effect at the next gpso_factorize):
 *   mode 0 automatic (int8 when the padded N >= 256), 1 = FP64 DMMA (mma.sync m8n8k4.f64), 2 = exact-integer emulation
 *   of the fp64 product on the int8 tensor cores (tcgen05.mma kind::i8, accumulators in TMEM).
 *   slices: 8-bit digits per operand for mode 2, 5..8, or 0 = chosen per fit from the row scales of L^-1 so that the
 *   estimated error stays below 2% of the parity tolerance 1e-8 * kernel variance. */
int gpso_set_predict_mode(gpso_handle* h, int mode, int slices);
/* Engine of K_y^-1 = L^-T L^-1 inside gpso_neg_lml_grad (the gradient's trace terms need K_y^-1 element-wise):
 *   0 automatic (int8 when the padded N >= 512), 1 = FP64 DMMA tiles, 2 = exact-integer product of 7-digit (54-bit)
 *   fixed-point operands on the int8 tensor cores -- operand rounding 2^-54 relative to each row's largest entry, i.e.
 *   the size of the fp64 rounding of those entries; the integer accumulation itself is exact. */
int gpso_set_kinv_mode(gpso_handle* h, int mode);
/* Host-only (no GPU): the tile -> CTA tables of the int8 fit-path products for a matrix of nb panels on nsm SMs, for the
 * CPU tests.  kind 0 = K_y^-1 (one int per slot: row block << 16 | 64-wide column tile, -1 = empty; info = {rounds});
 * kind 1 = inverse factor (four ints per slot: row block, 64-row tile of the second operand, first k-step, k-steps;
 * info = per level {s, xt offset, xt rounds, y offset, y rounds}, offsets in ints).  Returns the table size in ints. */
int64_t gpso_debug_product_items(int kind, int nb, int nsm, int* out, int64_t capacity, int* info, int info_capacity,
                                 int* levels_out);
/* Engine of the recursive-doubling inverse factor L^-1 (both gpso_factorize and gpso_neg_lml_grad):
 *   0 automatic (int8 when the padded N >= 512), 1 = FP64 DMMA tile tasks inside the persistent factorisation kernel,
 *   2 = exact-integer products of 8-digit (62-bit) fixed-point operands on the int8 tensor cores, two per level. */
int gpso_set_inverse_mode(gpso_handle* h, int mode);
/* int8 engine only: keep the digit tiles of L^-1 in the persisting (set-aside) part of L2 through an access-policy
 * window on the handle's product stream (default on; takes effect at the next gpso_factorize) */
int gpso_set_l2_window(gpso_handle* h, int enabled);
/* out[0] = engine in force after the last gpso_factorize (1 or 2), out[1] = digits per operand (0 for engine 1),
 * out[2] = estimated error of the variance / parity tolerance for that choice */
int gpso_predict_info(gpso_handle* h, double* out3);
/* int8 engine only: overlap the cross-covariance of window w+1 (FP64 CUDA cores, side stream) with the tensor-core
 * product of window w (default on; results are bit-identical either way) */
int gpso_set_overlap(gpso_handle* h, int enabled);
/* schedule of the blocked Cholesky inside gpso_neg_lml_grad / gpso_factorize: 1 (default) = one persistent kernel, one CTA
 * per SM pulling DIAG / PANEL / UPDATE tile tasks from a dependency-ordered queue (look-ahead, no launch gaps); 0 = one
 * launch per step (diagonal block, panel, trailing update).  Same tile arithmetic; the schedules differ in summation order
 * only (wide K = 512 updates, one update fused into the diagonal block), i.e. at rounding level. */
int gpso_set_factor_mode(gpso_handle* h, int mode);
/* mode 1 is the default and means "automatic": matrices of more than 32 tiles (N > 4096) use the HYBRID factorisation -- the
 * matrix is split recursively at powers of two; the leaves (<= 4096 rows) go through the persistent FP64 kernel in place, the
 * panel L21 = A21 L11^-T and the Schur complement A22 -= L21 L21^T are exact-integer products on the int8 tensor cores
 * (8 digits per operand), and the inverse factor's level that merges the two halves follows immediately.  mode 2 = always one
 * persistent FP64 kernel (round-1 behaviour), mode 3 = hybrid down to leaves of 2 tiles (tests).
 * gpso_factor_info: out2 = {schedule of the last factorisation: 0 stepwise / 1 persistent / 2 hybrid, inner nodes of the hybrid}. */
int gpso_factor_info(gpso_handle* h, int* out2);
/* Host-only introspection (works without a GPU) of the hybrid factorisation of nb tiles with leaves of at most `leaf` tiles:
 * the steps in execution order, four ints each {op, first tile, tiles, split}: op 0 = leaf (persistent FP64 kernel + its
 * inverse), 1 = panel L21 = A21 L11^-T, 2 = Schur complement A22 -= L21 L21^T, 3 = merge of the two halves' inverses.  Returns
 * the number of steps (out may be NULL).  gpso_debug_hybrid_items: the tile -> CTA table of a panel (kind 0) or Schur (kind 1)
 * product of a node of n tiles split after s: [rounds][nsm][4] ints (row block, 64-row tile of B, first k-step, k-steps; row
 * block < 0 = empty slot); returns the number of ints. */
/* Host-only: the windows (first candidate, candidates) a screening pass cuts M candidates into, for windows of at most W
 * candidates; ramp = the quarter / half window ramp-up used with the stream overlap, even = equal windows instead of a short
 * tail.  Returns the number of windows (out may be NULL; 2 int64 per window). */
int64_t gpso_debug_screen_windows(int64_t M, int64_t W, int ramp, int even, int64_t* out, int64_t capacity);
int64_t gpso_debug_hybrid_plan(int nb, int leaf, int* out, int64_t capacity);
int64_t gpso_debug_hybrid_items(int kind, int s, int n, int nsm, int* out, int64_t capacity, int* rounds);
/* Device memory of destroyed handles is kept in a per-device pool (up to 24 GB) and handed to the next handle: the optimiser
 * creates one handle per fit, and cudaMalloc / cudaFree of a handle's ~40 buffers cost more than a small fit.  This call gives
 * the cached blocks of `device` back to the driver (cached_bytes_before, if not NULL, receives how much that was). */
int gpso_trim_pool(int device, int64_t* cached_bytes_before);
/* Host-only introspection (works without a GPU): the task list of the persistent factorisation kernel for a matrix of nb
 * 128-wide panels on nsm SMs, 16 ints per task (op, p, i, j, s, tile, 3 x dependency counter, 3 x value, counter to
 * signal, value / 0 = increment, 2 unused).  out may be NULL to query the sizes. */
int gpso_debug_factor_tasks(int nb, int nsm, int* out, int64_t capacity_words, int* ntasks, int* ncounters);
/* the same list with only the levels s < inv_cap (in tiles) of the inverse recursion in it -- what the library runs when the
 * int8 engine takes the levels above (inv_cap 8, or 4 from 24 tiles; 0 = Cholesky tasks only) */
int gpso_debug_factor_tasks_cap(int nb, int nsm, int inv_cap, int* out, int64_t capacity_words, int* ntasks, int* ncounters);
/* tuning knob: candidates per rolling window (0 = automatic) */
int gpso_set_window(gpso_handle* h, int64_t candidates);
/* Screen-and-refine form of the fused arg-max calls (gpso_ucb_argmax_*, gpso_grow_ucb_argmax; replaces the same reference call
 * sites, gpso/gp_surrogate.py:313-328): all candidates are first scored with `digits` 8-bit digits per operand and an fp32
 * cross-covariance, the candidates whose screened UCB is within 2E of the best one (E = modelled error bound, checked on the
 * survivors) are re-scored by the full-precision engine, and the record of that engine is returned -- bit-identical to the
 * unscreened call.  mode 0 = off, 1 = automatic (default; from N >= 512 and M >= 65536, digits adapt to the survivor
 * fraction), 2..4 = forced digit count, 5 = bound-and-refine: a first level evaluates only the posterior MEAN of every
 * candidate (the variance lies between the noise variance and prior + noise variance, so a candidate whose mean is more than
 * |varsigma| * kernel variance below the best mean cannot win) and hands its survivors to the full-precision engine; when the
 * means do not separate the candidates it continues with the automatic digit screen; 6 = forced 2-digit screen with all four
 * digit pairs (the first rung of the automatic ladder: 2 digits / all pairs, then 3 and 4 digits / triangular).  Takes effect
 * at the next gpso_factorize.  gpso_predict_y_* and gpso_ucb_topk_* never screen.  The rung the automatic ladder ended on
 * (or "no rung separates these candidates") is remembered per matrix size for the process, because the optimiser opens a new
 * handle for every fit; every 32nd call starts one rung lower again, and an explicit call of this function restarts the ladder
 * for the handle's matrix size.  That state only changes the cost of a call, never the record it returns. */
int gpso_set_screen_mode(gpso_handle* h, int mode);
/* last fused arg-max call: out[0] path (0 unscreened, 1 screened, 2 full pass: too many survivors, 3 full pass: bound check
 * failed, 4 mean-bound level + refine), out[1] screening digits (0 for path 4), out[2] survivors, out[3] error bound E, out[4] largest |refined - screened| UCB over
 * the survivors, out[5] best screened UCB, out[6] screening windows, out[7] summed duration (ms) of the screening product
 * launches, out[8] refine windows, out[9] E_var, out[10] E_mean, out[11] 1 when the screening product kept all digit pairs (path 1); mode
 * 5: admissible distance below the best mean (path 4) */
int gpso_screen_info(gpso_handle* h, double* out12);
/* 3-digit screening product as CTA pairs (tcgen05.mma.cta_group::2, the B digits of a k-step split between the two shared
 * memories of a TPC; needs an even number of 128-row blocks) or as single CTAs (default: the pair form moves 17 % fewer
 * bytes into shared memory and reads 30 % fewer from it, but measured 5.48 vs 5.37 ms per window at N = 4096 -- the kernel is
 * bound by the accumulator hand-over, not by operand traffic); bit-identical results */
int gpso_set_screen_pair(gpso_handle* h, int enabled);
/* Pipe peaks of GPU `device`, measured now (~0.2 s): out4 = {int8 tensor TOP/s (tcgen05 kind::i8 issue rate), FP64 TFLOP/s
 * (DMMA.8x8x4 issue rate), L2 -> shared-memory bulk-copy GB/s, number of SMs}.  bench.py divides by these. */
int gpso_probe_peaks(int device, double* out4);
/* Host-only (works without a GPU): the error bound E of the screening pass and its variance / mean parts,
 * out3 = {E, E_var, E_mean}, for N training points, kernel variance, noise variance and fit5 = {largest power-of-two row scale of
 * L^-1, sum of the squared row scales, largest row norm of L^-1, |L^-1|_F^2, |alpha|_2}, the screening digit count (2..4), whether
 * all digit pairs are kept (full product) and the UCB multiplier. */
int gpso_debug_screen_bound(int N, double variance, double noise, const double* fit5, int digits, int full, double varsigma,
                            double* out3);

#ifdef __cplusplus
}
#endif
#endif /* GPSO_B200_H */
