"""
Cost of the periodic kernel on the device: Periodic(SquaredExponential) on d inputs beside SquaredExponential on d and on 2 d
inputs, on the same GPU, in the same process, the arms alternating and each repeated --reps times.

    python tools/periodic_kernel_bench.py --out profiles/r08_periodic_bench.json [--reps 3] [--candidates 10000000]

Per arm:
  * LML + gradient (the L-BFGS-B closure) at N = 300, 4096 and 8192 with scalar lengthscales (and period), ms per call;
  * C3 scoring: bench.py's seeded training set (N = 4096, d = 10; the SE at 2 d arm reads 20 columns of the same generator),
    its candidate matrix resident in HBM, device-resident gpso_ucb_argmax_dev in the default (screened) mode, candidates/s
    between CUDA events, with the path, digits and survivors of the call;
  * joint samples: predict_f_samples at N = 4096, M = 4096, S = 1024, ms per call (gpso_predict_f_samples_dev);
  * launches per call of each figure (gpso_launch_count).
Every arm uses bench.py's theta (lengthscale 0.25 sqrt(d), unit variance, noise 1e-3, zero constant); the periodic arm adds a
period of 0.7 in every dimension.  The output check runs the periodic arm against tests/periodic_oracle.py on the same seeded
inputs: the LML and gradient at N = 300 and predict_y of 512 candidates at N = 4096.  The JSON holds the GPU's name and power
limit and, per figure, every repetition and its spread (max / min).
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

ARMS = ("SE_d", "Periodic(SE)_d", "SE_2d")
PERIOD = 0.7


def dim_of(arm, d):
    return 2 * d if arm == "SE_2d" else d


def theta_of(arm, d):
    """Constrained packed vector: ls, var, (period), noise, constant mean."""
    ls, var, noise, c = bench.fixed_theta(d)
    return np.array([ls, var] + ([PERIOD] if arm == "Periodic(SE)_d" else []) + [noise, c])


def u_of(arm, d):
    th = theta_of(arm, d)
    u = th.copy()   # the constant mean is unconstrained
    u[:-2] = np.log(np.expm1(th[:-2]))
    u[-2] = np.log(np.expm1(th[-2] - 1.0e-6))   # GPflow's noise floor
    return u


def open_fitted(cuda, arm, X, y, factorize=True):
    if arm == "Periodic(SE)_d":
        s = cuda.open_session("Periodic", 1, True, components=[("SquaredExponential", 1)])
    else:
        s = cuda.open_session("SquaredExponential", 1, True)
    s.set_data(X, y)
    if factorize:
        s.factorize(theta_of(arm, X.shape[1]))
    return s


def oracle_check(cuda):
    from tests import periodic_oracle as pe

    d = 10
    X, y = bench.synthetic_training(300, d)
    ls, var, noise, c = bench.fixed_theta(d)
    h = pe.PeriodicHyper("SquaredExponential", ls, var, PERIOD, noise, mean=c)
    s = open_fitted(cuda, "Periodic(SE)_d", X, y, factorize=False)
    u = u_of("Periodic(SE)_d", d)
    f, g = s.neg_lml_and_grad(u)
    f_ref, g_ref = pe.neg_lml_and_grad("SquaredExponential", 1, 1, X, y, u, 1)
    s.close()
    X, y = bench.synthetic_training(4096, d)
    xc = np.empty((512, d))
    bench.fill_candidates(xc, 0, 512, 512, d)
    s = open_fitted(cuda, "Periodic(SE)_d", X, y)
    mean, var_ = s.predict_y(xc)
    s.close()
    m_ref, v_ref = pe.predict_y(h, X, y, xc)
    return {"lml_abs_err_over_max_lml_N": abs(f - f_ref) / max(abs(f_ref), 300),
            "grad_max_err_over_max_g_1": float(np.max(np.abs(g - g_ref) / np.maximum(np.abs(g_ref), 1.0))),
            "predict_mean_max_abs_err": float(np.max(np.abs(mean - m_ref[:, 0]))),
            "predict_var_max_abs_err": float(np.max(np.abs(var_ - v_ref[:, 0])))}


def main():
    import torch

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[1])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--candidates", type=int, default=10_000_000)
    ap.add_argument("--calls", type=int, default=3, help="timed scoring calls per repetition")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("periodic_kernel_bench.py measures the GPU: no CUDA device visible")

    cuda = backend.CudaBackend(device=0)
    N, d, M = 4096, 10, args.candidates
    stream = torch.cuda.current_stream().cuda_stream
    res = {a: {"lml_grad_ms": {}, "c3_screened_candidates_per_s": [], "joint_samples_ms_4096x4096x1024": [], "launches": {},
               "records": {}} for a in ARMS}

    # LML + gradient
    for Nl in (300, 4096, 8192):
        sess = {}
        for a in ARMS:
            Xl, yl = bench.synthetic_training(Nl, dim_of(a, d))
            sess[a] = open_fitted(cuda, a, Xl, yl, factorize=False)
            res[a]["lml_grad_ms"][str(Nl)] = []
        for a, s in sess.items():
            s.neg_lml_and_grad(u_of(a, d))
            c0 = s.launch_count()
            s.neg_lml_and_grad(u_of(a, d))
            res[a]["launches"][f"lml_grad_{Nl}"] = s.launch_count() - c0
        for _ in range(args.reps):
            for a, s in sess.items():
                u = u_of(a, d)
                t0 = time.perf_counter()
                for _ in range(5):
                    s.neg_lml_and_grad(u)
                res[a]["lml_grad_ms"][str(Nl)].append((time.perf_counter() - t0) * 1e3 / 5)
        for s in sess.values():
            s.close()

    # C3 scoring (default, screened mode) and the joint samples
    for a in ARMS:
        da = dim_of(a, d)
        X, y = bench.synthetic_training(N, da)
        host = np.empty((M, da))
        bench.fill_candidates(host, 0, M, M, da)
        res[a]["xc"] = torch.from_numpy(host).to("cuda")
        res[a]["session"] = open_fitted(cuda, a, X, y)
    for a in ARMS:
        s, xc = res[a]["session"], res[a]["xc"]
        s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)   # warm-up: module load, screening rung feedback
        c0 = s.launch_count()
        s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)
        res[a]["launches"]["c3_screened"] = {"launches": s.launch_count() - c0, "windows": s.last_windows()}
    for _ in range(args.reps):
        for a in ARMS:
            s, xc = res[a]["session"], res[a]["xc"]
            rec = []
            ms = event_ms(torch, lambda: rec.append(s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)), args.calls)
            res[a]["c3_screened_candidates_per_s"].append(M / (ms * 1e-3))
            info = s.screen_info()
            res[a]["records"]["c3_screened"] = list(rec[-1]) + [info["path"], info["digits"], info["survivors"]]
    Mj, Sj = 4096, 1024
    z = torch.from_numpy(np.random.default_rng(1).standard_normal((Sj, Mj))).to("cuda")
    out_s = torch.empty((Sj, Mj), dtype=torch.float64, device="cuda")
    for a in ARMS:
        s, xc = res[a]["session"], res[a]["xc"]
        s.predict_f_samples_dev(xc.data_ptr(), Mj, Sj, 1e-6, z.data_ptr(), out_s.data_ptr(), stream)
        c0 = s.launch_count()
        s.predict_f_samples_dev(xc.data_ptr(), Mj, Sj, 1e-6, z.data_ptr(), out_s.data_ptr(), stream)
        res[a]["launches"]["joint_samples"] = s.launch_count() - c0
    for _ in range(args.reps):
        for a in ARMS:
            s, xc = res[a]["session"], res[a]["xc"]
            res[a]["joint_samples_ms_4096x4096x1024"].append(
                event_ms(torch, lambda: s.predict_f_samples_dev(xc.data_ptr(), Mj, Sj, 1e-6, z.data_ptr(), out_s.data_ptr(), stream), 3))
    for a in ARMS:
        res[a].pop("session").close()
        del res[a]["xc"]

    out = {"gpu": gpu_identity(), "reps": args.reps, "calls_per_rep": args.calls,
           "workload": f"bench.py C3 inputs: N={N}, d={d} (SE_2d: {2 * d}), M={M}, theta={bench.fixed_theta(d).tolist()}, "
                       f"period {PERIOD}", "arms": {}, "oracle_check_periodic": oracle_check(cuda)}
    for a in ARMS:
        r = res[a]
        out["arms"][a] = {"lml_grad_ms": {k: spread(v) for k, v in r["lml_grad_ms"].items()},
                          "c3_screened_candidates_per_s": spread(r["c3_screened_candidates_per_s"]),
                          "joint_samples_ms_4096x4096x1024": spread(r["joint_samples_ms_4096x4096x1024"]),
                          "launches_per_call": r["launches"], "last_records": r["records"]}

    def ratios(arm, base):
        x, b = out["arms"][arm], out["arms"][base]
        r = {"c3_screened_rate": x["c3_screened_candidates_per_s"]["median"] / b["c3_screened_candidates_per_s"]["median"],
             "joint_samples_time": x["joint_samples_ms_4096x4096x1024"]["median"] / b["joint_samples_ms_4096x4096x1024"]["median"]}
        for k in x["lml_grad_ms"]:
            r[f"lml_grad_{k}_time"] = x["lml_grad_ms"][k]["median"] / b["lml_grad_ms"][k]["median"]
        return r

    out["periodic_over_se_d"] = ratios("Periodic(SE)_d", "SE_d")
    out["periodic_over_se_2d"] = ratios("Periodic(SE)_d", "SE_2d")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as handle:
        json.dump(out, handle, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "periodic_over_se_d", "periodic_over_se_2d", "oracle_check_periodic")}))


if __name__ == "__main__":
    main()
