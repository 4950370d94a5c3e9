#!/usr/bin/env python
"""
Benchmark of the hot path: predict_y + UCB + arg-max over leaf candidates (BASELINE.json metric, config C3:
N=4096 training points, d=10, 1e7 candidates, Matern-5/2, fp64).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one full scoring pass over the candidate set (a `gp_eval_best_ucb` call at C3 size).  With N > 1 GPUs
the candidates are sharded contiguously over the ranks (total work fixed -> "scaling": "strong"); the fit state is
broadcast once with NCCL before the timed region (reported as broadcast_ms), and every step ends with the all-gather
of one 32-byte record per rank.  Prints ONE JSON line on rank 0 (keys described in DESIGN.md section "Measurement").

--impl reference times the CPU restatement of the reference's own path (oracle/gpr_oracle.py, GPflow op order incl.
the Cholesky inside every predict_y call) on the box's host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if "reference" in sys.argv:
    # the CPU arm uses every host core: torchrun exports OMP_NUM_THREADS=1 to its workers, which would pin OpenBLAS to one
    # thread (the reference arm of the scaling runs in round 1 was 2.3x slower than the stand-alone one for that reason)
    for _var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_var] = str(os.cpu_count() or 1)

import numpy as np
from scipy.special import erfcinv

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20240517
WORKLOADS = {
    # name: (N, d, M, description)
    "c3": (4096, 10, 10_000_000, "C3: UCB scoring, N=4096 train, d=10, 1e7 leaf candidates, Matern-5/2 fp64"),
    "c2": (512, 2, 100_000, "C2: predict_y+UCB microbench, N=512 train, d=2, 1e5 candidates, Matern-5/2 fp64"),
}
# pipe peaks are measured inside the run (backend.probe_peaks: tcgen05 kind::i8 issue rate, DMMA issue rate, L2 -> shared
# memory bulk copies); these round-1 figures of the same probes (profiles/r01_*_probe.txt) are only the fallback
FP64_PEAK_TFLOPS = 37.03
INT8_PEAK_TOPS = 4528.7
VARSIGMA = float(erfcinv(0.01))  # UCB multiplier of the reference (gp_surrogate.py:397)
CPU_SAMPLE = 8192         # candidates per CPU-baseline step (bounded sample of the same workload)
LOGICAL_SHARDS = 64       # the candidate matrix is generated in 64 seeded pieces, so it is the same for every GPU count


def synthetic_training(N, d):
    rng = np.random.default_rng(SEED)
    X = rng.random((N, d))
    y = np.sin(3.0 * X.sum(axis=1)) + 0.01 * rng.standard_normal(N)
    return X, y[:, None]


def fill_candidates(out, start, stop, M, d):
    """Rows [start, stop) of the M x d synthetic candidate matrix into ``out``.  Logical shard s (rows s*ceil(M/64) ...) comes
    from ``default_rng([SEED, s])`` (SURVEY.md 8d), whatever the number of ranks: every GPU count scores the same matrix."""
    per = -(-M // LOGICAL_SHARDS)
    for s in range(start // per, (stop - 1) // per + 1 if stop > start else 0):
        lo, hi = s * per, min(M, (s + 1) * per)
        block = np.random.default_rng([SEED, s]).random((hi - lo, d))
        a, b = max(lo, start), min(hi, stop)
        out[a - start:b - start] = block[a - lo:b - lo]


def pack_unconstrained(ls, variance, noise, c):
    """Unconstrained L-BFGS-B variables of (lengthscale, kernel variance, noise variance, constant mean): softplus^-1, with
    GPflow's 1e-6 floor under the noise variance (SURVEY.md appendix A.1)."""
    inv = lambda v: float(np.log(np.expm1(v)))
    return np.array([inv(ls), inv(variance), inv(noise - 1.0e-6), c])


def fixed_theta(d):
    return np.array([0.25 * np.sqrt(d), 1.0, 1.0e-3, 0.0])


def use_all_host_cores():
    """BLAS thread pools of this process at the number of host cores, whatever the launcher exported."""
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass


def make_config(desc, N, d, M, theta):
    """The workload description printed by both arms (identical dicts: the driver compares them)."""
    return {"workload": desc, "N": N, "d": d, "M": M, "kernel": "Matern52", "theta": [float(t) for t in theta],
            "varsigma": VARSIGMA, "candidates": "64 seeded logical shards, uniform in [0,1)^d", "dtype": "f64"}


def blas_threads():
    try:
        from threadpoolctl import threadpool_info

        infos = [i for i in threadpool_info() if i.get("user_api") == "blas"]
        if infos:
            return int(max(i["num_threads"] for i in infos)), infos[0].get("internal_api", "blas")
    except Exception:
        pass
    return os.cpu_count() or 1, "unknown"


def cpu_reference_step(X, y, theta, Xc, varsigma):
    """The reference path on the CPU: predict_y (Cholesky inside, Kmn materialised, two TRSMs) + UCB + argmax."""
    from oracle import gpr_oracle as go

    h = go.Hyper(theta[0], theta[1], theta[2], theta[3])
    mean, var = go.predict_y("Matern52", X, y, h, Xc, chunk=65536)
    return go.ucb_argmax(mean, var, varsigma)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU with nvidia-smi while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, smax, reasons = [], 0.0, set()
        for row in self.rows:
            try:
                sm.append(float(row[0]))
                smax = max(smax, float(row[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), row[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def bench_lml_grad(cuda, peaks, cpu=True, shapes=((4096, 10), (8192, 20)), evals=5):
    """LML + gradient evaluations per second through the C ABI (gpso_neg_lml_grad: Gram -> Cholesky -> L^-1 -> K_y^-1 ->
    fused gradient reduction), host in / host out, at the shapes of configs C3 and C4.  Algorithmic work: N^3 flops.
    Every shape is checked against the CPU oracle (LML and gradient) outside the timed loops."""
    out = []
    fp64_peak = peaks["fp64_tflops"]
    for N, d in shapes:
        X, y = synthetic_training(N, d)
        u = pack_unconstrained(0.25 * np.sqrt(d), 1.0, 1.0e-3, 0.0)
        sess = cuda.open_session("Matern52", 1, True)
        sess.set_data(X, y)
        f, g = sess.neg_lml_and_grad(u)  # warm-up (allocations)
        # three repetitions of `evals` calls, the median one is reported: a 16 ms timed region is at the mercy of one host hiccup
        reps = []
        for _ in range(3):
            t0 = time.perf_counter()
            dev_ms = 0.0
            for i in range(evals):
                f, g = sess.neg_lml_and_grad(u + 1e-3 * (i + 1))
                dev_ms += sess.last_timing_ms()[0]
            reps.append((time.perf_counter() - t0, dev_ms))
        wall, dev_ms = sorted(reps)[1]
        factor_info = sess.factor_info()
        # the same closure with ONE persistent FP64 kernel for the whole matrix (round-1 schedule; only differs above 4096 rows)
        one_ms = None
        if factor_info["schedule"] == "hybrid":
            sess.set_factor_mode(True, hybrid=False)
            sess.neg_lml_and_grad(u)
            one_ms = 0.0
            for i in range(evals):
                sess.neg_lml_and_grad(u + 1e-3 * (i + 1))
                one_ms += sess.last_timing_ms()[0]
            one_ms /= evals
        # the same closure with the step-by-step launches (gpso_set_factor_mode 0) beside the persistent tile scheduler
        sess.set_factor_mode(False)
        sess.neg_lml_and_grad(u)
        step_ms = 0.0
        for i in range(evals):
            sess.neg_lml_and_grad(u + 1e-3 * (i + 1))
            step_ms += sess.last_timing_ms()[0]
        sess.set_factor_mode(True)
        rec = {"N": N, "d": d, "evals_per_s": evals / wall, "device_ms_per_eval": dev_ms / evals,
               "wall_ms_per_eval_repetitions": [w / evals * 1e3 for w, _ in reps],
               "device_ms_per_eval_stepwise_launches": step_ms / evals,
               "device_ms_per_eval_one_fp64_kernel": one_ms,
               "factorisation": factor_info,
               "schedule": ("hybrid Cholesky: leaves of <= 4096 rows by the persistent FP64 DMMA kernel (task queue + per-tile "
                            "dependency counters, the panel tile on the chain in four row strips), panel solve and Schur complement "
                            "as exact-integer products on the int8 tensor cores; " if factor_info["schedule"] == "hybrid" else
                            "blocked Cholesky as ONE persistent kernel on FP64 DMMA (task queue + per-tile dependency counters, the "
                            "panel tile on the chain in four row strips); ") +
                           "L^-1 by recursive doubling and K_y^-1 = L^-T L^-1 as exact-integer products on the int8 tensor cores",
               "library_bar_ms": {4096: {"cusolver_dpotrf": 1.675, "cusolver_dpotri": 14.005},
                                  8192: {"cusolver_dpotrf": 7.753, "cusolver_dpotri": 61.528}}.get(N),
               "fp64_equivalent_tflops": (float(N) ** 3 / (dev_ms / evals * 1e-3)) / 1e12, "fp64_peak_tflops": fp64_peak,
               "ratio_to_fp64_peak": (float(N) ** 3 / (dev_ms / evals * 1e-3)) / 1e12 / fp64_peak,
               "ratio_note": "N^3/3 flops (Cholesky) run on the FP64 pipe (above 4096 rows: only the leaves), 2N^3/3 (L^-1, K_y^-1) as "
                             "int8 tensor-core products: the ratio to the FP64 pipe peak can exceed 1",
               "neg_lml": f}
        if cpu:
            from oracle import gpr_oracle as go  # CPU leg of the LML side measurement (checker + baseline)

            t0 = time.perf_counter()
            f_ref, g_ref = go.neg_lml_and_grad("Matern52", X, y, u + 1e-3 * evals, 1, True)
            rec["cpu_evals_per_s"] = 1.0 / (time.perf_counter() - t0)
            rec["lml_rel_err_vs_cpu"] = abs(f - f_ref) / max(abs(f_ref), N)        # bar: 1e-9
            rec["grad_rel_err_vs_cpu"] = float(np.max(np.abs(g - g_ref) / np.maximum(np.abs(g_ref), 1.0)))  # bar: 1e-6
        sess.close()
        out.append(rec)
    return out


def bench_restarts(cuda, world, rank, group=None, N=8192, d=20, restarts_per_rank=2, maxiter=3):
    """Config C4, bounded: multi-start L-BFGS-B restarts of the hyper-parameter fit sharded over the ranks (restart i on
    rank i mod W, all-gather of (-LML*, u*)).  Aggregate LML+grad evaluations per second = evaluations of all ranks / the
    slowest rank's wall time.  The full configuration (64 restarts x maxiter 50) is tools/c4_restarts.py."""
    import torch

    from pygpso_b200 import gpmodel
    from pygpso_b200.distributed import sharded_multistart_fit

    X, y = synthetic_training(N, d)
    model = gpmodel.GPR(data=(X, y), kernel=gpmodel.Matern52(lengthscales=0.25 * np.sqrt(d), variance=1.0),
                        mean_function=gpmodel.Constant(0.0), noise_variance=1.0e-3, backend=cuda)
    u0 = model._pack()
    model.neg_log_marginal_likelihood_and_grad(u0)  # allocations
    n0 = model.n_loss_evaluations
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier(group=group)
    t0 = time.perf_counter()
    u_best, f_best, rid, table = sharded_multistart_fit(model.neg_log_marginal_likelihood_and_grad, u0,
                                                        restarts_per_rank * world, group=group, maxiter=maxiter)
    wall = time.perf_counter() - t0
    evals = model.n_loss_evaluations - n0
    model.close()
    if world > 1:
        t = torch.tensor([wall, float(evals)], dtype=torch.float64, device="cuda")
        tmax = t.clone()
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX, group=group)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM, group=group)
        wall, evals = float(tmax[0].item()), int(t[1].item())
    return {"N": N, "d": d, "restarts": restarts_per_rank * world, "maxiter": maxiter, "evaluations": int(evals), "wall_s": wall,
            "evals_per_s": evals / wall, "best_restart": int(rid), "best_neg_lml": float(f_best),
            "note": "bounded sample of config C4 (64 restarts x maxiter 50): restarts_per_rank x W restarts, each rank runs its own "
                    "L-BFGS-B chains on its own GPU; weak scaling in the number of restarts"}


def run_reference(args, rank):
    """--impl reference: the CPU path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    use_all_host_cores()
    N, d, M, desc = WORKLOADS[args.workload]
    X, y = synthetic_training(N, d)
    theta = fixed_theta(d)
    sample = min(M, CPU_SAMPLE)
    Xc = np.empty((sample, d))
    fill_candidates(Xc, 0, sample, M, d)
    for _ in range(args.warmup):
        cpu_reference_step(X, y, theta, Xc, VARSIGMA)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        result = cpu_reference_step(X, y, theta, Xc, VARSIGMA)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_record(args.dump_outputs, result)
    cores, blas = blas_threads()
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": "predict_y+UCB candidates/sec", "value": value, "unit": "candidates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(desc, N, d, M, theta),
        "cpu_baseline": {"value": value, "unit": "candidates/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} of the {M} candidates per step (numpy/scipy restatement of GPflow's predict_y op "
                                   f"sequence incl. the per-call Cholesky; {blas} BLAS, {cores} threads; GPflow itself is not "
                                   "installable here)"},
        "e2e": {"value": value, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def verify_result(session, cuda, X, y, theta, xc_dev, m_local, varsigma, stream, result, screen_mode=1):
    """Independent confirmation of the selected candidate, outside the timed region (single GPU): (1) the whole candidate set
    once more on the FP64 DMMA engine (no int8 emulation, no screening) must select the same index with mean / variance / UCB
    within the parity tolerance; (2) the 64 best candidates of the full-precision int8 engine (gpso_ucb_topk_dev, never
    screened) are re-scored by the CPU oracle, whose arg-max among them must be the same candidate."""
    from oracle import gpr_oracle as go  # checker only

    out = {}
    session.set_screen_mode(0)
    session.set_predict_mode(1, 0)
    session.factorize(theta)
    t0 = time.perf_counter()
    dm = session.ucb_argmax_dev(xc_dev.data_ptr(), m_local, varsigma, stream)
    out["dmma_engine_full_pass_s"] = time.perf_counter() - t0
    out["dmma_engine_index"] = int(dm[0])
    out["dmma_same_index"] = bool(dm[0] == result[0])
    out["dmma_mean_rel"] = abs(dm[1] - result[1]) / max(abs(result[1]), float(np.abs(y).max()))
    out["dmma_var_rel"] = abs(dm[2] - result[2]) / max(abs(result[2]), float(theta[1]))
    session.set_predict_mode(0, 0)
    session.factorize(theta)
    top = session.ucb_topk_dev(xc_dev.data_ptr(), m_local, varsigma, 64, stream)
    out["topk_first_is_result"] = bool(int(top[0, 0]) == result[0] and top[0, 3] == result[3])
    idx = top[:, 0].astype(np.int64)
    rows = xc_dev[idx.tolist()].cpu().numpy()
    h = go.Hyper(theta[0], theta[1], theta[2], theta[3])
    mean, var = go.predict_y("Matern52", X, y, h, rows)
    k = int(go.ucb_argmax(mean, var, varsigma)[0])
    out["oracle_argmax_of_top64"] = int(idx[k])
    out["oracle_same_index"] = bool(int(idx[k]) == result[0])
    out["oracle_mean_rel"] = float(np.max(np.abs(mean[:, 0] - top[:, 1]) / np.maximum(np.abs(mean[:, 0]), np.abs(y).max())))
    out["oracle_var_rel"] = float(np.max(np.abs(var[:, 0] - top[:, 2]) / np.maximum(np.abs(var[:, 0]), theta[1])))
    out["oracle_var_pure_rel"] = float(np.max(np.abs(var[:, 0] - top[:, 2]) / np.abs(var[:, 0])))
    out["ok"] = bool(out["dmma_same_index"] and out["oracle_same_index"] and out["topk_first_is_result"]
                     and out["dmma_mean_rel"] <= 1e-8 and out["dmma_var_rel"] <= 1e-8
                     and out["oracle_mean_rel"] <= 1e-8 and out["oracle_var_rel"] <= 1e-8)
    session.set_screen_mode(screen_mode)
    session.factorize(theta)
    return out


def dump_record(out_dir, result):
    """The arg-max record a caller of the scoring path receives, one float64 array per field (the index is exact in float64
    up to 2^53 candidates)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, value in zip(("index", "mean", "var", "ucb"), result):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.array([value], dtype=np.float64))


def side_leg(fn, *a, **kw):
    """Run a side measurement; a failure there must not cost the headline line (the error text is reported instead)."""
    try:
        return fn(*a, **kw)
    except Exception as err:  # noqa: BLE001
        return {"error": f"{type(err).__name__}: {err}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--candidates", type=int, default=0, help="override the number of candidates (smoke runs only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-lml", action="store_true", help="skip the LML+grad evaluations/s side measurements")
    ap.add_argument("--no-verify", action="store_true", help="skip the independent confirmation of the selected candidate")
    ap.add_argument("--engine", default="auto", choices=["auto", "dmma", "int8"],
                    help="variance-product engine: FP64 DMMA or the exact-integer int8 tcgen05 emulation (auto picks int8 at this size)")
    ap.add_argument("--screen", type=int, default=1, help="screen-and-refine arg-max: 0 off, 1 automatic, 2..4 forced screening digits")
    ap.add_argument("--no-bound", action="store_true", help="skip the bound-and-refine side measurement (screen mode 5)")
    ap.add_argument("--no-overlap", action="store_true", help="int8 engine: run cross-covariance and product back to back")
    ap.add_argument("--slices", type=int, default=0, help="8-bit digits per operand for the int8 engine (0 = automatic)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the record the last timed step returned (index, mean, var, ucb) as DIR/<name>.npy in float64, "
                         "so that two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    from pygpso_b200 import backend, gpmodel
    from pygpso_b200.distributed import ShardedScorer, gather_records, pick_best, shard_bounds

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (pygpso_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    os.environ.setdefault("GPSO_DEVICE", str(local_rank))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    N, d, M, desc = WORKLOADS[args.workload]
    if args.candidates:
        M = args.candidates
    varsigma = VARSIGMA
    X, y = synthetic_training(N, d)
    theta = fixed_theta(d)
    cuda = backend.CudaBackend(device=local_rank)
    # pipe peaks of THIS GPU in THIS run (tcgen05 kind::i8 and DMMA issue rates, L2 -> shared-memory bulk copies)
    peaks = cuda.probe_peaks()

    # the model object of the public API (GPR == the reference's gpflow_model); rank 0 fits, the others import
    kernel = gpmodel.Matern52(lengthscales=theta[0], variance=theta[1])
    model = gpmodel.GPR(data=(X, y), kernel=kernel, mean_function=gpmodel.Constant(theta[3]), noise_variance=theta[2], backend=cuda)
    session = model._session
    session.set_predict_mode({"auto": 0, "dmma": 1, "int8": 2}[args.engine], args.slices)
    session.set_screen_mode(args.screen)
    session.set_overlap(not args.no_overlap)
    t0 = time.perf_counter()
    if rank == 0:
        model._ensure_factor()  # Gram -> Cholesky -> L^-1 -> alpha on rank 0 only
    factor_ms = (time.perf_counter() - t0) * 1e3
    broadcast_ms = None
    scorer = None
    if world > 1:
        scorer = ShardedScorer(session)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        scorer.broadcast_fit(N, d, src=0)  # one NCCL broadcast of (scaled X, alpha, L^-1, theta) per fit
        torch.cuda.synchronize()
        dist.barrier()
        broadcast_ms = (time.perf_counter() - t0) * 1e3
        model._factor_key = model._theta().tobytes()

    # this rank's shard of the candidates, in pinned host memory (for the end-to-end leg) and resident in HBM
    start, stop = shard_bounds(M, world, rank)
    m_local = stop - start
    host = torch.empty((max(m_local, 1), d), dtype=torch.float64, pin_memory=True)
    xc_host = host.numpy()[:m_local]
    fill_candidates(xc_host, start, stop, M, d)
    xc_dev = host[:m_local].to("cuda", non_blocking=False)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        rec = [-np.inf, -1.0, 0.0, 0.0]
        if m_local:
            idx, mean, var, ucb = session.ucb_argmax_dev(xc_dev.data_ptr(), m_local, varsigma, stream)
            rec = [ucb, float(start + idx), mean, var]
        return pick_best(gather_records(rec)) if world > 1 else (int(rec[1]), rec[2], rec[3], rec[0])

    def step_e2e():
        # public API with HOST buffers: H2D of the candidates + D2H of the result inside the call
        if world > 1:
            return scorer.ucb_argmax(xc_host, start, varsigma)
        return model.ucb_argmax(xc_host, varsigma)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident measurement -------------------------------------------------------------------------------
    for _ in range(args.warmup):
        result = step_device()
    sync_all()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = session.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms = np.zeros(4)
    windows = 0
    screen = {"paths": [], "survivors": [], "product_ms": 0.0, "windows": 0, "digits": 0, "error_bound": 0.0, "max_dev": 0.0}
    ev0.record()
    for _ in range(args.steps):
        result = step_device()
        stage_ms += session.last_timing_ms()
        windows += session.last_windows()
        info = session.screen_info()
        screen["paths"].append(info["path"])
        screen["survivors"].append(info["survivors"])
        screen["product_ms"] += info["screen_product_ms"]
        screen["windows"] += info["screen_windows"]
        screen["digits"] = info["digits"]
        screen["all_pairs"] = bool(info["all_pairs"])
        screen["error_bound"] = info["error_bound"]
        screen["max_dev"] = max(screen["max_dev"], info["max_observed_deviation"])
    ev1.record()
    sync_all()
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = session.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_record(args.dump_outputs, result)
    product_ms = stage_ms[2]  # summed duration of all variance-product launches (event pairs on their stream)
    engine = session.predict_info()
    screened = bool(screen["paths"]) and all(p == "screened" for p in screen["paths"])

    # ---- end-to-end measurement (host buffers through the public API) ------------------------------------------------
    for _ in range(min(args.warmup, 1)):
        step_e2e()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        result_e2e = step_e2e()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    if world > 1:
        dist.barrier()

    # ---- the dominant kernel without its neighbour: one screened step with the stream overlap off (in the timed steps the
    # cross-covariance kernel of the next window runs beside the product and slows it; both are power-bound) ---------------
    standalone = None
    if screened:
        session.set_overlap(False)
        step_device()
        step_device()
        sinfo = session.screen_info()
        standalone = {"product_ms_per_step": sinfo["screen_product_ms"], "windows": sinfo["screen_windows"]}
        session.set_overlap(not args.no_overlap)

    # ---- one step of the unscreened full-precision pass and its per-stage breakdown (outside the timed regions) ------
    full_pass = None
    stage_profile = None
    if screened:
        session.set_screen_mode(0)
        if rank == 0:
            session.factorize(theta)
        if world > 1:
            scorer.broadcast_fit(N, d, src=0)
        step_device()
        sync_all()
        t0 = time.perf_counter()
        full_result = step_device()
        sync_all()
        full_s = max_over_ranks(time.perf_counter() - t0)
        full_pass = {"value": M / full_s, "ms_per_step": full_s * 1e3, "same_record": bool(tuple(full_result) == tuple(result)),
                     "engine": session.predict_info()}
    session.set_profile(True)
    step_device()
    stage_profile = session.last_timing_ms()
    session.set_profile(False)
    if screened:
        session.set_screen_mode(args.screen)
        if rank == 0:
            session.factorize(theta)
        if world > 1:
            scorer.broadcast_fit(N, d, src=0)

    # ---- side measurement: bound-and-refine (gpso_set_screen_mode 5: posterior mean of every candidate first, variance only
    # for the candidates the mean cannot rule out) -- not the headline, reported beside it ------------------------------------
    bound = None
    if screened and not args.no_bound:
        session.set_screen_mode(5)
        if rank == 0:
            session.factorize(theta)
        if world > 1:
            scorer.broadcast_fit(N, d, src=0)
        step_device()
        sync_all()
        bev0, bev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        bev0.record()
        for _ in range(args.steps):
            bound_result = step_device()
        bev1.record()
        sync_all()
        bound_ms = max_over_ranks(bev0.elapsed_time(bev1)) / args.steps
        binfo = session.screen_info()
        bound = {"value": M / (bound_ms * 1e-3), "ms_per_step": bound_ms, "path": binfo["path"], "survivors": binfo["survivors"],
                 "same_record": bool(tuple(bound_result) == tuple(result)), "e_mean": binfo["e_mean"],
                 "max_observed_deviation": binfo["max_observed_deviation"],
                 "note": "opt-in mode, not the headline: only the posterior mean is evaluated for every candidate (fp32 "
                         "cross-covariance); var lies in [noise, prior + noise], so candidates whose mean is more than |varsigma| * "
                         "kernel variance below the best mean are ruled out exactly; the rest is scored by the full-precision engine"}
        session.set_screen_mode(args.screen)
        if rank == 0:
            session.factorize(theta)
        if world > 1:
            scorer.broadcast_fit(N, d, src=0)

    # ---- second half of the BASELINE metric at every GPU count: bounded config-C4 restart leg ---------------------------
    restarts = None
    if not args.no_lml:
        restarts = side_leg(bench_restarts, cuda, world, rank)

    if rank == 0:
        assert result_e2e[0] == result[0], "end-to-end and device-resident passes selected different candidates"
        value = M * args.steps / (dev_ms * 1e-3)
        e2e_value = M * args.steps / e2e_s
        flops64 = float(N) * N * m_local * args.steps  # algorithmic fp64 work: N^2 per candidate (SURVEY.md section 8d)
        clock_ratio = (clocks["sm_mhz"] / clocks["sm_max_mhz"]) if clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") else None
        Np = -(-N // 128) * 128
        nb = Np // 128
        ksteps = sum(4 * (i + 1) for i in range(nb))  # k-steps of 32 over the lower-triangular row blocks
        if screened:
            S = screen["digits"]
            all_pairs = screen.get("all_pairs", False)
            pairs = S * S if all_pairs else S * (S + 1) // 2  # all digit pairs, or the triangle p + q < S
            variant = f"{S},128,true" if all_pairs else f"{S},128"
            ops = pairs * flops64
            t_prod = screen["product_ms"] * 1e-3
            achieved = ops / t_prod / 1e12
            launches_dom = max(int(screen["windows"]), 1)
            # operand bytes the kernel pulls L2 -> shared memory: per (candidate tile of 128, row block, k-step) S digit
            # tiles of A (4 KB) and of B (4 KB)
            l2_bytes = (m_local * args.steps / 128.0) * ksteps * S * (4096 + 4096)
            roofline = {
                "bound": "tensor",
                "kernel": f"ozaki_screen_kernel<{variant}> (tcgen05.mma kind::i8 screening product: {S} 8-bit digits per operand, {pairs} "
                          "digit pairs, 128-candidate tiles, TMEM accumulators, fp32 epilogue); the survivors are re-scored by "
                          f"ozaki_kernel<{engine['slices']},OZ_TRMM>",
                "achieved": achieved, "peak": peaks["int8_tops"], "unit": "TFLOP/s", "frac": achieved / peaks["int8_tops"],
                "frac_at_clock": (achieved / (peaks["int8_tops"] * clock_ratio)) if clock_ratio else None,
                "op_kind": "int8 tensor op (2 per multiply-add); algorithmic = digit_pairs * N^2 per candidate",
                "digits": S, "digit_pairs": pairs, "all_digit_pairs": all_pairs,
                "traffic": None,
                "peak_source": "measured in this run: tcgen05.mma.cta_group::1.kind::i8 M=128 N=256 issue rate on all SMs "
                               "(gpso_probe_peaks); MEASURED_PEAKS.json has no int8 entry",
                "l2_operand": {"bytes_per_launch": l2_bytes / launches_dom, "achieved_gbs": l2_bytes / t_prod / 1e9,
                               "peak_gbs": peaks["l2_to_smem_gbs"], "frac": l2_bytes / t_prod / 1e9 / peaks["l2_to_smem_gbs"],
                               "note": "the product kernels are bound by L2 -> shared-memory operand traffic before the tensor "
                                       "pipe; peak = cp.async.bulk probe of this run (24 KB chunks, 8 in flight per SM)"},
                "fp64_equivalent": {"achieved_tflops": flops64 / t_prod / 1e12, "fp64_pipe_peak_tflops": peaks["fp64_tflops"],
                                    "ratio_to_fp64_peak": flops64 / t_prod / 1e12 / peaks["fp64_tflops"]},
                "launches": launches_dom, "avg_launch_ms": screen["product_ms"] / launches_dom,
                "algorithmic_ops_per_launch": ops / launches_dom,
                "product_share_of_step": screen["product_ms"] / dev_ms,
                "timing_note": "achieved / frac use the launch durations inside the timed steps, where the cross-covariance kernel of "
                               "the next window runs beside the product on a second stream (the step is power-bound: the pair takes "
                               "the sum of the two energies); `standalone` is the same kernel with the overlap off",
            }
            if standalone and standalone["windows"]:
                t_alone = standalone["product_ms_per_step"] * 1e-3
                ops_step = pairs * float(N) * N * m_local
                roofline["standalone"] = {"avg_launch_ms": standalone["product_ms_per_step"] / standalone["windows"],
                                          "achieved": ops_step / t_alone / 1e12, "frac": ops_step / t_alone / 1e12 / peaks["int8_tops"]}
        elif engine["engine"] == "int8-tcgen05":
            S = engine["slices"]
            pairs = S * (S + 1) // 2
            ops = pairs * flops64
            achieved = ops / (product_ms * 1e-3) / 1e12
            l2_bytes = (m_local * args.steps / 64.0) * ksteps * S * (4096 + 2048)
            roofline = {
                "bound": "tensor",
                "kernel": f"ozaki_kernel<{S},OZ_TRMM> (tcgen05.mma kind::i8, {S} 8-bit digits per operand, {pairs} digit pairs, "
                          "TMEM accumulators, exact int32 sums recombined to fp64 in the epilogue)",
                "achieved": achieved, "peak": peaks["int8_tops"], "unit": "TFLOP/s", "frac": achieved / peaks["int8_tops"],
                "frac_at_clock": (achieved / (peaks["int8_tops"] * clock_ratio)) if clock_ratio else None,
                "op_kind": "int8 tensor op (2 per multiply-add); algorithmic = digit_pairs * N^2 per candidate",
                "digits": S, "digit_pairs": pairs, "traffic": None,
                "peak_source": "measured in this run (gpso_probe_peaks): tcgen05 kind::i8 M=128 N=256 issue rate",
                "l2_operand": {"achieved_gbs": l2_bytes / (product_ms * 1e-3) / 1e9, "peak_gbs": peaks["l2_to_smem_gbs"],
                               "frac": l2_bytes / (product_ms * 1e-3) / 1e9 / peaks["l2_to_smem_gbs"]},
                "fp64_equivalent": {"achieved_tflops": flops64 / (product_ms * 1e-3) / 1e12, "fp64_pipe_peak_tflops": peaks["fp64_tflops"],
                                    "ratio_to_fp64_peak": flops64 / (product_ms * 1e-3) / 1e12 / peaks["fp64_tflops"]},
                "error_estimate_over_tolerance": engine["error_estimate_over_tol"],
                "launches": int(max(windows, 1)), "avg_launch_ms": product_ms / max(windows, 1),
                "algorithmic_ops_per_launch": ops / max(windows, 1), "product_share_of_step": product_ms / dev_ms,
            }
        else:
            achieved = flops64 / (product_ms * 1e-3) / 1e12
            roofline = {
                "bound": "tensor", "kernel": "predict_trmm_kernel (FP64 DMMA triangular product + column sum of squares)",
                "achieved": achieved, "peak": peaks["fp64_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["fp64_tflops"],
                "frac_at_clock": (achieved / (peaks["fp64_tflops"] * clock_ratio)) if clock_ratio else None, "traffic": None,
                "peak_source": "measured in this run (gpso_probe_peaks): DMMA.8x8x4 issue rate",
                "launches": int(max(windows, 1)), "avg_launch_ms": product_ms / max(windows, 1),
                "algorithmic_ops_per_launch": flops64 / max(windows, 1), "product_share_of_step": product_ms / dev_ms,
            }
        # DRAM traffic of the dominant kernel from an ncu --set full capture of the same configuration (per launch), if one
        # was committed for this workload / engine; never a number from another configuration
        prof_json = os.path.join(ROOT, "profiles", "product_kernel_traffic.json")
        if os.path.exists(prof_json):
            try:
                variant_key = f"screen{screen['digits']}{'f' if screen.get('all_pairs') else ''}" if screened else engine["engine"]
                entry = json.load(open(prof_json)).get(f"{args.workload}:{variant_key}")
                if entry:
                    # the capture is one full window; the launches of a step are not all full (ramp-up and tail windows):
                    # scaled to the average number of candidates per launch of this run
                    per_launch = m_local * args.steps / max(roofline.get("launches", 1), 1)
                    scale = per_launch / entry["candidates_per_launch"] if entry.get("candidates_per_launch") else 1.0
                    roofline["traffic"] = entry.get("dram_bytes_per_launch") * scale
                    roofline["traffic_source"] = entry.get("source") + f"; scaled by {scale:.3f} = candidates per launch of this run / of the capture"
            except Exception:
                pass
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
        except Exception:
            pass
        hbm_alg = (80.0 * M * args.steps / (dev_ms * 1e-3)) / 1e9
        roofline.update({
            "hbm_peak_gbs": hbm_peak, "hbm_peak_source": "MEASURED_PEAKS.json (driver-written)" if hbm_peak else None,
            "hbm_frac_algorithmic": (hbm_alg / hbm_peak) if hbm_peak else None,
            "hbm_algorithmic_gbs": (80.0 * M * args.steps / (dev_ms * 1e-3)) / 1e9,
            "hbm_note": "algorithmic HBM traffic is 80 B per candidate (coordinates in, fused arg-max out): the pass is compute-bound by "
                        "five orders of magnitude, the 70 %-of-HBM target of north_star cannot apply to a variance pass (SURVEY 7.2)",
            "stage_ms_one_step_full_precision_serialised": {"crosscov": stage_profile[1], "product": stage_profile[2],
                                                            "finalize": stage_profile[3]},
        })
        line = {
            "metric": "predict_y+UCB candidates/sec", "value": value, "unit": "candidates/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": make_config(desc, N, d, M, theta),
            "run": {"parallelism": f"candidates sharded over {world} GPU(s)", "engine": engine,
                    "l2": "inputs larger than L2: 80 B/candidate x M candidates in HBM plus two 2 GiB rolling windows of "
                          "cross-covariance digit tiles per GPU vs 126 MB L2"},
            "screen": {"mode": args.screen, "paths": sorted(set(screen["paths"])), "digits": screen["digits"], "all_digit_pairs": screen.get("all_pairs", False),
                       "survivors_per_step": screen["survivors"], "survivors_per_window": (float(np.mean(screen["survivors"])) /
                                                                                         max(screen["windows"] / max(args.steps, 1), 1)),
                       "error_bound": screen["error_bound"], "max_observed_deviation": screen["max_dev"],
                       "note": "every candidate is screened with few digits + fp32 cross-covariance; candidates within 2E of the best "
                               "screened UCB are re-scored by the full-precision engine, whose record is returned (bit-identical to the "
                               "unscreened call, see full_precision_pass.same_record)"},
            "full_precision_pass": full_pass,
            "bound_and_refine": bound,
            "e2e": {"value": e2e_value, "unit": "candidates/s", "h2d_bytes_per_step": int(M) * d * 8,
                    "d2h_bytes_per_step": 32 * world, "ms_per_step": e2e_s / args.steps * 1e3},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "peaks_measured_in_this_run": peaks,
            "roofline": roofline,
            "setup": {"factorize_ms": factor_ms, "broadcast_ms": broadcast_ms, "state_bytes": session.state_bytes(N, d)},
            "result": {"index": int(result[0]), "mean": result[1], "var": result[2], "ucb": result[3]},
            "lml_grad_restarts": restarts,
        }
        # ---- independent confirmation of the selected candidate (single-GPU runs) ----------------------------------------
        if world == 1 and not args.no_verify:
            line["result"]["verified"] = side_leg(verify_result, session, cuda, X, y, theta, xc_dev, m_local, varsigma, stream, result, args.screen)
        # ---- second half of the BASELINE metric: LML + gradient evaluations per second (the L-BFGS-B closure) ---------
        if world == 1 and not args.no_lml:
            line["lml_grad"] = side_leg(bench_lml_grad, cuda, peaks, cpu=not args.no_cpu_baseline)
        # ---- CPU baseline beside it (bounded sample, rank 0, single GPU runs only) -----------------------------------
        if world == 1 and not args.no_cpu_baseline:
            use_all_host_cores()
            sample = min(M, CPU_SAMPLE)
            xs = xc_host[:sample]
            cpu_reference_step(X, y, theta, xs[:256], varsigma)
            t0 = time.perf_counter()
            ref = cpu_reference_step(X, y, theta, xs, varsigma)
            cpu_s = time.perf_counter() - t0
            cores, blas = blas_threads()
            # the same sample through the CUDA path must select the same candidate
            got = session.ucb_argmax(xs, varsigma)
            line["cpu_baseline"] = {
                "value": sample / cpu_s, "unit": "candidates/s", "cores": cores, "kind": "port",
                "sample": f"first {sample} of the {M} candidates, one pass (numpy/scipy restatement of GPflow's predict_y op "
                          f"sequence incl. the per-call Cholesky; {blas} BLAS, {cores} threads)",
                "same_argmax_as_gpu": bool(got[0] == ref[0]),
            }
        print(json.dumps(line), flush=True)
    model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
