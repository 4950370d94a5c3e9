"""
Cost of the sum kernel on the device: Matern52 against Sum([Matern52, SquaredExponential]) on the same GPU, in the same
process, the arms alternating and each repeated --reps times.

    python tools/sum_kernel_bench.py --out profiles/r06_sum_bench.json [--reps 3] [--candidates 10000000]

Per arm:
  * C3 scoring: bench.py's seeded training set (N = 4096, d = 10), its candidate matrix resident in HBM and its theta,
    device-resident gpso_ucb_argmax_dev, candidates/s between CUDA events, screened (automatic mode, the default) and
    unscreened (screen mode 0), with the path, digits and survivors of the screened call;
  * LML + gradient (the L-BFGS-B closure) at N = 4096, d = 10 and N = 8192, d = 20, ms per call;
  * predict_f(full_cov=True) at N = M = 4096, ms per call (gpso_predict_f_cov_dev);
  * launches per call of each figure (gpso_launch_count).
Both arms have bench.py's Matern52 term; the sum adds a SquaredExponential term with twice the lengthscale and a quarter of the
variance (both scalar lengthscales).  The JSON holds the GPU's name and power limit and, per figure, every repetition and its
spread (max / min).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from pygpso_b200 import backend  # noqa: E402
from tools.kernel_bench import event_ms, gpu_identity, spread  # noqa: E402

ARMS = ("Matern52", "Matern52+SE")


def se_term(d):
    ls, var = bench.fixed_theta(d)[:2]
    return np.array([2.0 * ls, 0.25 * var])


def theta_of(arm, d):
    th = bench.fixed_theta(d)
    return th if arm == "Matern52" else np.concatenate([th[:2], se_term(d), th[2:]])


def u_of(arm, d):
    u = bench.pack_unconstrained(*bench.fixed_theta(d))
    return u if arm == "Matern52" else np.concatenate([u[:2], np.log(np.expm1(se_term(d))), u[2:]])


def open_fitted(cuda, arm, X, y, factorize=True):
    if arm == "Matern52":
        s = cuda.open_session("Matern52", 1, True)
    else:
        s = cuda.open_session("Sum", 0, True, components=[("Matern52", 1), ("SquaredExponential", 1)])
    s.set_data(X, y)
    if factorize:
        s.factorize(theta_of(arm, X.shape[1]))
    return s


def main():
    import torch

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[1])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--candidates", type=int, default=10_000_000)
    ap.add_argument("--calls", type=int, default=3, help="timed scoring calls per repetition")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sum_kernel_bench.py measures the GPU: no CUDA device visible")

    cuda = backend.CudaBackend(device=0)
    N, d, M = 4096, 10, args.candidates
    X, y = bench.synthetic_training(N, d)
    host = np.empty((M, d))
    bench.fill_candidates(host, 0, M, M, d)
    xc = torch.from_numpy(host).to("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    res = {a: {"c3_screened_candidates_per_s": [], "c3_unscreened_candidates_per_s": [], "lml_grad_ms": {"4096x10": [], "8192x20": []},
               "predict_f_cov_ms_4096": [], "launches": {}, "records": {}} for a in ARMS}

    # C3 scoring, screened (default mode) and unscreened (mode 0): one fitted session per arm and mode, the arms alternating
    for mode, key in ((1, "c3_screened_candidates_per_s"), (0, "c3_unscreened_candidates_per_s")):
        sessions = {}
        for a in ARMS:
            s = open_fitted(cuda, a, X, y, factorize=False)
            s.set_screen_mode(mode)
            s.factorize(theta_of(a, d))
            sessions[a] = s
        for a, s in sessions.items():
            s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)   # warm-up: module load, screening rung feedback
            c0 = s.launch_count()
            s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)
            res[a]["launches"][key] = {"launches": s.launch_count() - c0, "windows": s.last_windows()}
        for _ in range(args.reps):
            for a, s in sessions.items():
                rec = []
                ms = event_ms(torch, lambda: rec.append(s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)), args.calls)
                res[a][key].append(M / (ms * 1e-3))
                info = s.screen_info()
                res[a]["records"][key] = list(rec[-1]) + [info["path"], info["digits"], info["survivors"]]
        for s in sessions.values():
            s.close()
    del xc

    # LML + gradient
    for (Nl, dl) in ((4096, 10), (8192, 20)):
        Xl, yl = bench.synthetic_training(Nl, dl)
        sess = {a: open_fitted(cuda, a, Xl, yl, factorize=False) for a in ARMS}
        for a, s in sess.items():
            s.neg_lml_and_grad(u_of(a, dl))
            c0 = s.launch_count()
            s.neg_lml_and_grad(u_of(a, dl))
            res[a]["launches"][f"lml_grad_{Nl}x{dl}"] = s.launch_count() - c0
        for _ in range(args.reps):
            for a, s in sess.items():
                u = u_of(a, dl)
                t0 = time.perf_counter()
                for _ in range(5):
                    s.neg_lml_and_grad(u)
                res[a]["lml_grad_ms"][f"{Nl}x{dl}"].append((time.perf_counter() - t0) * 1e3 / 5)
        for s in sess.values():
            s.close()

    # joint posterior at N = M = 4096
    Mj = 4096
    xj = torch.from_numpy(np.ascontiguousarray(host[:Mj])).to("cuda")
    mean = torch.empty(Mj, dtype=torch.float64, device="cuda")
    cov = torch.empty((Mj, Mj), dtype=torch.float64, device="cuda")
    sess = {a: open_fitted(cuda, a, X, y) for a in ARMS}
    for a, s in sess.items():
        s.predict_f_cov_dev(xj.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream)
        torch.cuda.synchronize()
        c0 = s.launch_count()
        s.predict_f_cov_dev(xj.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream)
        res[a]["launches"]["predict_f_cov_4096"] = s.launch_count() - c0
    for _ in range(args.reps):
        for a, s in sess.items():
            res[a]["predict_f_cov_ms_4096"].append(
                event_ms(torch, lambda: s.predict_f_cov_dev(xj.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream), 5))
    for s in sess.values():
        s.close()

    out = {"gpu": gpu_identity(), "reps": args.reps, "calls_per_rep": args.calls,
           "workload": f"bench.py C3 inputs: N={N}, d={d}, M={M}, Matern52, theta={bench.fixed_theta(d).tolist()}; "
                       f"Matern52+SE: SquaredExponential (lengthscale, variance) = {se_term(d).tolist()}", "arms": {}}
    for a in ARMS:
        r = res[a]
        out["arms"][a] = {
            "c3_screened_candidates_per_s": spread(r["c3_screened_candidates_per_s"]),
            "c3_unscreened_candidates_per_s": spread(r["c3_unscreened_candidates_per_s"]),
            "lml_grad_ms": {k: spread(v) for k, v in r["lml_grad_ms"].items()},
            "predict_f_cov_ms_4096": spread(r["predict_f_cov_ms_4096"]),
            "launches_per_call": r["launches"], "last_records": r["records"],
        }
    lin, con = out["arms"]["Matern52+SE"], out["arms"]["Matern52"]
    out["sum_over_bare"] = {
        "c3_screened_rate": lin["c3_screened_candidates_per_s"]["median"] / con["c3_screened_candidates_per_s"]["median"],
        "c3_unscreened_rate": lin["c3_unscreened_candidates_per_s"]["median"] / con["c3_unscreened_candidates_per_s"]["median"],
        "lml_grad_4096x10_time": lin["lml_grad_ms"]["4096x10"]["median"] / con["lml_grad_ms"]["4096x10"]["median"],
        "lml_grad_8192x20_time": lin["lml_grad_ms"]["8192x20"]["median"] / con["lml_grad_ms"]["8192x20"]["median"],
        "predict_f_cov_4096_time": lin["predict_f_cov_ms_4096"]["median"] / con["predict_f_cov_ms_4096"]["median"],
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as handle:
        json.dump(out, handle, indent=1)
    print(json.dumps(out["sum_over_bare"]))


if __name__ == "__main__":
    main()
