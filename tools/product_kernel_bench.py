"""
Cost of the product kernel on the device: Matern52, Matern52 + SquaredExponential (the sum) and Matern52 * SquaredExponential
(the product) on the same GPU, in the same process, the arms alternating and each repeated --reps times.

    python tools/product_kernel_bench.py --out profiles/r07_product_bench.json [--reps 3] [--candidates 10000000]

Per arm:
  * C3 scoring: bench.py's seeded training set (N = 4096, d = 10), its candidate matrix resident in HBM and its theta,
    device-resident gpso_ucb_argmax_dev, candidates/s between CUDA events, screened (automatic mode, the default) and
    unscreened (screen mode 0), with the path, digits and survivors of the screened call;
  * LML + gradient (the L-BFGS-B closure) at N = 4096, d = 10 with scalar lengthscales and at N = 8192, d = 20 with ARD
    lengthscales (every term), ms per call;
  * predict_f(full_cov=True) at N = M = 4096, ms per call (gpso_predict_f_cov_dev);
  * launches per call of each figure (gpso_launch_count).
Every arm has bench.py's Matern52 term.  The SquaredExponential term has twice its lengthscale, with a quarter of its variance in
the sum (the arm of profiles/r06_sum_bench.json) and unit variance in the product (so the product's prior variance is bench.py's).
The JSON holds the GPU's name and power limit and, per figure, every repetition and its spread (max / min).
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

ARMS = ("Matern52", "Matern52+SE", "Matern52*SE")
SE_VARIANCE = {"Matern52+SE": 0.25, "Matern52*SE": 1.0}


def theta_of(arm, d, ard=False):
    """Constrained packed vector: [ls (d entries with ARD), var] per term, then noise and the constant mean."""
    ls, var, noise, c = bench.fixed_theta(d)
    nl = d if ard else 1
    th = [ls] * nl + [var]
    if arm != "Matern52":
        th += [2.0 * ls] * nl + [SE_VARIANCE[arm]]
    return np.array(th + [noise, c])


def u_of(arm, d, ard=False):
    th = theta_of(arm, d, ard)
    u = np.log(np.expm1(th))
    u[-2] = np.log(np.expm1(th[-2] - 1.0e-6))   # GPflow's noise floor
    u[-1] = th[-1]
    return u


def open_fitted(cuda, arm, X, y, ard=False, factorize=True):
    nl = X.shape[1] if ard else 1
    if arm == "Matern52":
        s = cuda.open_session("Matern52", nl, True)
    else:
        s = cuda.open_session("Sum" if arm == "Matern52+SE" else "Product", 0, True,
                              components=[("Matern52", nl), ("SquaredExponential", nl)])
    s.set_data(X, y)
    if factorize:
        s.factorize(theta_of(arm, X.shape[1], ard))
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
        raise SystemExit("product_kernel_bench.py measures the GPU: no CUDA device visible")

    cuda = backend.CudaBackend(device=0)
    N, d, M = 4096, 10, args.candidates
    X, y = bench.synthetic_training(N, d)
    host = np.empty((M, d))
    bench.fill_candidates(host, 0, M, M, d)
    xc = torch.from_numpy(host).to("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    lml_shapes = ((4096, 10, False), (8192, 20, True))
    lml_key = lambda Nl, dl, ard: f"{Nl}x{dl}" + ("_ard" if ard else "")  # noqa: E731
    res = {a: {"c3_screened_candidates_per_s": [], "c3_unscreened_candidates_per_s": [],
               "lml_grad_ms": {lml_key(*s): [] for s in lml_shapes}, "predict_f_cov_ms_4096": [], "launches": {}, "records": {}}
           for a in ARMS}

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
    for (Nl, dl, ard) in lml_shapes:
        Xl, yl = bench.synthetic_training(Nl, dl)
        k = lml_key(Nl, dl, ard)
        sess = {a: open_fitted(cuda, a, Xl, yl, ard=ard, factorize=False) for a in ARMS}
        for a, s in sess.items():
            s.neg_lml_and_grad(u_of(a, dl, ard))
            c0 = s.launch_count()
            s.neg_lml_and_grad(u_of(a, dl, ard))
            res[a]["launches"][f"lml_grad_{k}"] = s.launch_count() - c0
        for _ in range(args.reps):
            for a, s in sess.items():
                u = u_of(a, dl, ard)
                t0 = time.perf_counter()
                for _ in range(5):
                    s.neg_lml_and_grad(u)
                res[a]["lml_grad_ms"][k].append((time.perf_counter() - t0) * 1e3 / 5)
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
                       f"SquaredExponential term: twice the lengthscale, variance {SE_VARIANCE}", "arms": {}}
    for a in ARMS:
        r = res[a]
        out["arms"][a] = {
            "c3_screened_candidates_per_s": spread(r["c3_screened_candidates_per_s"]),
            "c3_unscreened_candidates_per_s": spread(r["c3_unscreened_candidates_per_s"]),
            "lml_grad_ms": {k: spread(v) for k, v in r["lml_grad_ms"].items()},
            "predict_f_cov_ms_4096": spread(r["predict_f_cov_ms_4096"]),
            "launches_per_call": r["launches"], "last_records": r["records"],
        }

    def ratios(arm, base):
        x, b = out["arms"][arm], out["arms"][base]
        r = {"c3_screened_rate": x["c3_screened_candidates_per_s"]["median"] / b["c3_screened_candidates_per_s"]["median"],
             "c3_unscreened_rate": x["c3_unscreened_candidates_per_s"]["median"] / b["c3_unscreened_candidates_per_s"]["median"],
             "predict_f_cov_4096_time": x["predict_f_cov_ms_4096"]["median"] / b["predict_f_cov_ms_4096"]["median"]}
        for k in x["lml_grad_ms"]:
            r[f"lml_grad_{k}_time"] = x["lml_grad_ms"][k]["median"] / b["lml_grad_ms"][k]["median"]
        return r

    out["product_over_sum"] = ratios("Matern52*SE", "Matern52+SE")
    out["product_over_bare"] = ratios("Matern52*SE", "Matern52")
    out["sum_over_bare"] = ratios("Matern52+SE", "Matern52")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as handle:
        json.dump(out, handle, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "product_over_sum", "product_over_bare")}))


if __name__ == "__main__":
    main()
