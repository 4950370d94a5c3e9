"""
Joint posterior on the device: gpso_predict_f_cov_dev and gpso_predict_f_samples_dev against a torch fp64 pipeline
(cuBLAS / cuSOLVER) on the same GPU, in the same process.

    python tools/joint_bench.py --out DIR [--shapes 300,512,64 4096,4096,1024 1024,8192,256] [--min-seconds 1]

Inputs are bench.py's seeded training set and candidate matrix (Matern-5/2, d = 10), at bench.py's fixed theta and at a theta
fitted by L-BFGS-B on the device with the noise variance at its 1e-6 floor (ill-conditioned K_y).  Per shape and theta: the
time of one covariance call and of one sampling call (CUDA events, warmed up, repeated for at least --min-seconds), the
algorithm's FLOPs per stage (V = L^-1 K*: N^2 M, SYRK: M^2 N, Cholesky of the covariance: M^3 / 3, samples: M^2 S), the
achieved FP64 rate over the DMMA peak measured in the same run, and the torch pipeline's time and its deviation from the
library's outputs.  Writes DIR/joint_bench.json with the GPU's name and power limit.
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
from pygpso_b200 import backend, gpmodel  # noqa: E402

D = 10
JITTER = gpmodel.SAMPLE_JITTER


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown"


def timed(fn, torch, min_seconds):
    """ms per call: two warm-up calls, then enough repetitions to cover min_seconds between two CUDA events."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    reps = max(3, int(np.ceil(min_seconds / max(time.perf_counter() - t0, 1e-6))))
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / reps, reps


def fitted_theta(cuda, X, y):
    th = bench.fixed_theta(X.shape[1])
    m = gpmodel.GPR((X, y), gpmodel.Matern52(lengthscales=th[0], variance=th[1]), gpmodel.Constant(th[3]), noise_variance=1.1e-6,
                    backend=cuda)
    m.likelihood.variance.trainable = False
    gpmodel.Scipy().minimize(m.training_loss, m.trainable_variables, options={"maxiter": 60})
    theta = m._theta()
    m.close()
    return theta


def matern52(torch, A, B, ls, var):
    r2 = ((A[:, None, :] - B[None, :, :]) / ls).pow(2).sum(-1)
    r = torch.sqrt(torch.clamp(r2, min=1e-36))
    s = np.sqrt(5.0) * r
    return var * (1.0 + s + (5.0 / 3.0) * r * r) * torch.exp(-s)


def run_case(cuda, torch, N, M, S, theta_name, theta, X, y, peak, min_seconds):
    dev = torch.device("cuda", cuda.device)
    st = torch.cuda.current_stream(dev)
    s = cuda.open_session("Matern52", 1, True)
    s.set_data(X, y)
    s.factorize(theta)
    xc_host = np.empty((M, D))
    bench.fill_candidates(xc_host, 0, M, M, D)
    xc = torch.from_numpy(xc_host).to(dev)
    mean = torch.empty(M, dtype=torch.float64, device=dev)
    cov = torch.empty((M, M), dtype=torch.float64, device=dev)
    z = torch.from_numpy(np.random.default_rng([bench.SEED, 99]).standard_normal((S, M))).to(dev)
    out = torch.empty((S, M), dtype=torch.float64, device=dev)
    sp = st.cuda_stream

    t_cov, reps_cov = timed(lambda: s.predict_f_cov_dev(xc.data_ptr(), M, mean.data_ptr(), cov.data_ptr(), sp), torch, min_seconds)
    t_smp, reps_smp = timed(lambda: s.predict_f_samples_dev(xc.data_ptr(), M, S, JITTER, z.data_ptr(), out.data_ptr(), sp), torch,
                            min_seconds)

    # torch fp64 baseline on the handle's own factor: A = L^-1 K*, cov = K** - A^T A, chol, matmul
    L = torch.from_numpy(s.debug_fetch(1)).to(dev).tril()
    alpha = torch.from_numpy(s.debug_fetch(3)).to(dev)
    Xt = torch.from_numpy(X).to(dev)
    ls, var, c = float(theta[0]), float(theta[1]), float(theta[3])
    eye = torch.eye(M, dtype=torch.float64, device=dev)
    res = {}

    def baseline():
        Kxs = matern52(torch, Xt, xc, ls, var)
        A = torch.linalg.solve_triangular(L, Kxs, upper=False)
        cv = matern52(torch, xc, xc, ls, var) - A.T @ A
        Lc = torch.linalg.cholesky(cv + JITTER * eye)
        mu = Kxs.T @ alpha + c
        res["cov"], res["f"] = cv, mu[None, :] + z @ Lc.T

    t_torch, reps_torch = timed(baseline, torch, min_seconds)
    s.predict_f_cov_dev(xc.data_ptr(), M, mean.data_ptr(), cov.data_ptr(), sp)
    s.predict_f_samples_dev(xc.data_ptr(), M, S, JITTER, z.data_ptr(), out.data_ptr(), sp)
    torch.cuda.synchronize()
    cov_dev = float(((cov - res["cov"]).abs() / torch.clamp(res["cov"].abs(), min=var)).max())
    f_dev = float((out - res["f"]).abs().max()) / np.sqrt(var)
    s.close()

    flops = {"V": float(N) * N * M, "syrk": float(M) * M * N, "cholesky": float(M) ** 3 / 3, "samples": float(M) * M * S}
    f_cov = flops["V"] + flops["syrk"]
    f_all = sum(flops.values())
    return {
        "N": N, "M": M, "S": S, "d": D, "theta_name": theta_name, "theta": [float(t) for t in theta],
        "flops": flops,
        "cov_call_ms": t_cov, "cov_call_reps": reps_cov,
        "samples_call_ms": t_smp, "samples_call_reps": reps_smp,
        "samples_minus_cov_ms": t_smp - t_cov,
        "cov_call_tflops": f_cov / t_cov * 1e-9, "samples_call_tflops": f_all / t_smp * 1e-9,
        "samples_call_fraction_of_fp64_peak": f_all / t_smp * 1e-9 / peak,
        "torch_pipeline_ms": t_torch, "torch_reps": reps_torch,
        "speedup_vs_torch": t_torch / t_smp,
        "cov_max_dev_over_max_ref_var": cov_dev, "cov_within_1e-8": cov_dev <= 1e-8,
        "samples_max_abs_dev_over_sigma_f": f_dev,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", nargs="*", default=["300,512,64", "4096,4096,1024", "1024,8192,256"])
    ap.add_argument("--min-seconds", type=float, default=1.0)
    args = ap.parse_args()
    import torch

    cuda = backend.default_backend()
    torch.cuda.set_device(cuda.device)
    peaks = cuda.probe_peaks()
    rows = []
    for shape in args.shapes:
        N, M, S = (int(v) for v in shape.split(","))
        X, y = bench.synthetic_training(N, D)
        for name, theta in (("fixed", bench.fixed_theta(D)), ("fitted_noise_floor", fitted_theta(cuda, X, y))):
            row = run_case(cuda, torch, N, M, S, name, theta, X, y, peaks["fp64_tflops"], args.min_seconds)
            print(json.dumps(row), flush=True)
            rows.append(row)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "joint_bench.json"), "w") as fh:
        json.dump({"gpu": gpu_identity(), "peaks": peaks, "torch": torch.__version__, "results": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
