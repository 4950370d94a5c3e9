"""
Cost of the covariance function on the device: Matern-5/2 against RationalQuadratic (alpha = 0.5 and 2) on the same GPU, in
the same process, the arms alternating and each repeated --reps times.

    python tools/kernel_bench.py --out profiles/r04_rq_bench.json [--reps 3] [--candidates 10000000]

Per arm:
  * C3 scoring: bench.py's seeded training set (N = 4096, d = 10), its candidate matrix resident in HBM and its theta (plus
    alpha), device-resident gpso_ucb_argmax_dev, candidates/s between CUDA events; the screening rung and survivor count of
    the call (gpso_screen_info), and the per-stage split of one profiled call (gpso_set_profile(h, 1): this runs the
    unscreened window pipeline with events between the stages);
  * LML + gradient (the L-BFGS-B closure) at N = 4096, d = 10 and N = 8192, d = 20, ms per call;
  * predict_f(full_cov=True) at N = M = 4096, ms per call (gpso_predict_f_cov_dev).
The JSON also holds the GPU's name and power limit, the pipe peaks probed in the same run and, per figure, every repetition
and its spread (max / min).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from pygpso_b200 import backend  # noqa: E402

ARMS = [("Matern52", None), ("RationalQuadratic", 0.5), ("RationalQuadratic", 2.0)]


def arm_name(kernel, alpha):
    return kernel if alpha is None else f"{kernel}(alpha={alpha:g})"


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def theta_of(alpha, d):
    th = bench.fixed_theta(d)
    return th if alpha is None else np.concatenate([[alpha], th])


def open_fitted(cuda, kernel, alpha, X, y, factorize=True):
    s = cuda.open_session(kernel, 1, True)
    s.set_data(X, y)
    if factorize:
        s.factorize(theta_of(alpha, X.shape[1]))
    return s


def event_ms(torch, fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps


def spread(values):
    v = np.asarray(values, dtype=np.float64)
    return {"runs": [float(x) for x in v], "median": float(np.median(v)), "spread_max_over_min": float(v.max() / v.min())}


def main():
    import torch

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[1])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--candidates", type=int, default=10_000_000)
    ap.add_argument("--calls", type=int, default=3, help="timed scoring calls per repetition")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("kernel_bench.py measures the GPU: no CUDA device visible")

    cuda = backend.CudaBackend(device=0)
    peaks = cuda.probe_peaks()
    N, d, M = 4096, 10, args.candidates
    X, y = bench.synthetic_training(N, d)
    host = np.empty((M, d))
    bench.fill_candidates(host, 0, M, M, d)
    xc = torch.from_numpy(host).to("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    names = [arm_name(*a) for a in ARMS]
    res = {n: {"c3_candidates_per_s": [], "c3_records": [], "screen": None, "stages_ms": None,
               "lml_grad_ms": {"4096x10": [], "8192x20": []}, "predict_f_cov_ms_4096": []} for n in names}

    # C3 scoring: one fitted session per arm, the arms alternating within each repetition
    sessions = {n: open_fitted(cuda, k, a, X, y) for n, (k, a) in zip(names, ARMS)}
    for n, s in sessions.items():
        s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)   # warm-up: module load, screening rung feedback
        s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)
    for _ in range(args.reps):
        for n, s in sessions.items():
            rec = []
            ms = event_ms(torch, lambda: rec.append(s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)), args.calls)
            res[n]["c3_candidates_per_s"].append(M / (ms * 1e-3))
            res[n]["c3_records"].append(list(rec[-1]))
            info = s.screen_info()
            res[n]["screen"] = {"path": info["path"], "digits": info["digits"], "all_pairs": info["all_pairs"],
                                "survivors": info["survivors"], "screen_product_ms": info["screen_product_ms"]}
    for n, s in sessions.items():
        s.set_profile(1)
        s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)
        t = s.last_timing_ms()
        res[n]["stages_ms"] = {"unscreened_total": float(t[0]), "cross_covariance": float(t[1]), "variance_product": float(t[2]),
                               "finalise_argmax": float(t[3]), "windows": s.last_windows()}
        s.set_profile(0)
        s.close()
    del xc

    # LML + gradient
    for (Nl, dl) in ((4096, 10), (8192, 20)):
        Xl, yl = bench.synthetic_training(Nl, dl)
        sess = {n: open_fitted(cuda, k, a, Xl, yl, factorize=False) for n, (k, a) in zip(names, ARMS)}
        us = {n: np.concatenate([[] if a is None else [np.log(np.expm1(a))],
                                 bench.pack_unconstrained(*bench.fixed_theta(dl))]) for n, (k, a) in zip(names, ARMS)}
        for n, s in sess.items():
            s.neg_lml_and_grad(us[n])
        for _ in range(args.reps):
            for n, s in sess.items():
                t0 = time.perf_counter()
                for _ in range(5):
                    s.neg_lml_and_grad(us[n])
                res[n]["lml_grad_ms"][f"{Nl}x{dl}"].append((time.perf_counter() - t0) * 1e3 / 5)
        for s in sess.values():
            s.close()

    # joint posterior at N = M = 4096
    Mj = 4096
    xj = torch.from_numpy(np.ascontiguousarray(host[:Mj])).to("cuda")
    mean = torch.empty(Mj, dtype=torch.float64, device="cuda")
    cov = torch.empty((Mj, Mj), dtype=torch.float64, device="cuda")
    sess = {n: open_fitted(cuda, k, a, X, y) for n, (k, a) in zip(names, ARMS)}
    for n, s in sess.items():
        s.predict_f_cov_dev(xj.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream)
    for _ in range(args.reps):
        for n, s in sess.items():
            res[n]["predict_f_cov_ms_4096"].append(
                event_ms(torch, lambda: s.predict_f_cov_dev(xj.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream), 5))
    for s in sess.values():
        s.close()

    out = {"gpu": gpu_identity(), "probed_peaks": peaks, "reps": args.reps, "calls_per_rep": args.calls,
           "workload": f"bench.py C3 inputs: N={N}, d={d}, M={M}, theta={list(bench.fixed_theta(d))} (+ alpha first for RQ)",
           "arms": {}}
    for n in names:
        r = res[n]
        out["arms"][n] = {
            "c3_candidates_per_s": spread(r["c3_candidates_per_s"]), "c3_record_last": r["c3_records"][-1],
            "screen": r["screen"], "stages_ms_profiled_unscreened": r["stages_ms"],
            "lml_grad_ms": {k: spread(v) for k, v in r["lml_grad_ms"].items()},
            "predict_f_cov_ms_4096": spread(r["predict_f_cov_ms_4096"]),
        }
    base = out["arms"][names[0]]["c3_candidates_per_s"]["median"]
    out["c3_rate_vs_matern52"] = {n: out["arms"][n]["c3_candidates_per_s"]["median"] / base for n in names}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as handle:
        json.dump(out, handle, indent=1)
    print(json.dumps(out["c3_rate_vs_matern52"]))


if __name__ == "__main__":
    main()
