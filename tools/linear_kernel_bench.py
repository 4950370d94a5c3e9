"""
Cost of the Linear kernel (gpflow.kernels.Linear) on the device: four arms on the same GPU, in the same process, the arms
alternating and each repeated --reps times.

    python tools/linear_kernel_bench.py --out profiles/r10_linear_kernel_bench.json [--reps 3] [--candidates 10000000]

Arms (d = 10, and d = 20 for the ARD LML): Matern52; Matern52 + Matern52; Linear + Matern52; bare Linear.  The arms with a Linear
term score on the FP64 engines and decline the screen; Linear + Matern52 against Matern52 + Matern52 in mode 0 is the cost of
the Linear term itself (the same two-component row layout, one fewer covariance evaluation per pair).
Per arm:
  * C3 scoring: bench.py's seeded training set (N = 4096, d = 10), its candidate matrix resident in HBM, device-resident
    gpso_ucb_argmax_dev, screened (default mode) and unscreened (mode 0), candidates/s between CUDA events;
  * LML + gradient (the L-BFGS-B closure) at N = 4096, d = 10 (scalar lengthscales) and N = 8192, d = 20 (ARD), ms per call;
  * predict_f_cov at N = M = 4096, ms per call (gpso_predict_f_cov_dev);
  * launches per call of each figure (gpso_launch_count).
Every stationary component takes bench.py's theta (lengthscale 0.25 sqrt(d), unit variance; noise 1e-3, zero constant mean); a
Linear term the variance 1 / d (one per column at d = 20), so that its prior variance on [0, 1]^d is of the order of the other
terms'.  The JSON holds the GPU's name and power limit and, per figure, every repetition and its spread.
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

# an arm: (kind, leaves); a leaf is "M52" or "Lin"
ARMS = {
    "M52": ("Bare", ["M52"]),
    "M52+M52": ("Sum", ["M52", "M52"]),
    "Lin+M52": ("Sum", ["Lin", "M52"]),
    "Lin": ("Bare", ["Lin"]),
}
PAIRS = (("Lin+M52", "M52+M52"), ("Lin", "M52"))


def open_arm(cuda, arm, d, ard):
    kind, leaves = ARMS[arm]
    nl = [d if ard else 1] * len(leaves)
    if kind == "Bare":
        s = cuda.open_session("Matern52" if leaves[0] == "M52" else "Linear", nl[0], True)
    else:
        s = cuda.open_session(kind, 0, True, components=[("Matern52" if leaf == "M52" else "Linear", n) for leaf, n in zip(leaves, nl)])
    ls, var, noise, c0 = bench.fixed_theta(d)
    theta = []
    for leaf, n in zip(leaves, nl):
        theta += [ls] * n + [var] if leaf == "M52" else [1.0 / d] * n
    theta = np.array(theta + [noise, c0])
    u = theta.copy()   # the constant mean is unconstrained
    u[:-2] = np.log(np.expm1(theta[:-2]))
    u[-2] = np.log(np.expm1(theta[-2] - 1.0e-6))   # GPflow's noise floor
    return s, theta, u


def main():
    import torch

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[1])
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--candidates", type=int, default=10_000_000)
    ap.add_argument("--calls", type=int, default=3, help="timed scoring calls per repetition")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("linear_kernel_bench.py measures the GPU: no CUDA device visible")

    cuda = backend.CudaBackend(device=0)
    N, d, M = 4096, 10, args.candidates
    stream = torch.cuda.current_stream().cuda_stream
    res = {a: {"lml_grad_ms": {}, "c3_screened_candidates_per_s": [], "c3_unscreened_candidates_per_s": [],
               "predict_f_cov_ms_4096x4096": [], "launches": {}, "records": {}} for a in ARMS}

    # LML + gradient: N = 4096 at d = 10 (scalar lengthscales), N = 8192 at d = 20 (ARD)
    for Nl, dl, ard in ((4096, 10, False), (8192, 20, True)):
        key = f"N{Nl}_d{dl}" + ("_ard" if ard else "")
        Xl, yl = bench.synthetic_training(Nl, dl)
        sess = {}
        for a in ARMS:
            s, _, u = open_arm(cuda, a, dl, ard)
            s.set_data(Xl, yl)
            sess[a] = (s, u)
            res[a]["lml_grad_ms"][key] = []
        for a, (s, u) in sess.items():
            s.neg_lml_and_grad(u)
            c0 = s.launch_count()
            s.neg_lml_and_grad(u)
            res[a]["launches"][f"lml_grad_{key}"] = s.launch_count() - c0
        for _ in range(args.reps):
            for a, (s, u) in sess.items():
                t0 = time.perf_counter()
                for _ in range(5):
                    s.neg_lml_and_grad(u)
                res[a]["lml_grad_ms"][key].append((time.perf_counter() - t0) * 1e3 / 5)
        for s, _ in sess.values():
            s.close()

    # C3 scoring, screened and unscreened, and the joint covariance
    X, y = bench.synthetic_training(N, d)
    host = np.empty((M, d))
    bench.fill_candidates(host, 0, M, M, d)
    xc = torch.from_numpy(host).to("cuda")
    sess = {}
    for a in ARMS:
        s, theta, _ = open_arm(cuda, a, d, False)
        s.set_data(X, y)
        s.factorize(theta)
        sess[a] = (s, theta)
    for mode, key in ((1, "c3_screened"), (0, "c3_unscreened")):
        for a, (s, theta) in sess.items():
            s.set_screen_mode(mode)
            s.factorize(theta)
            s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)   # warm-up: module load, screening rung feedback
            c0 = s.launch_count()
            s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)
            res[a]["launches"][key] = {"launches": s.launch_count() - c0, "windows": s.last_windows()}
        for _ in range(args.reps):
            for a, (s, _) in sess.items():
                rec = []
                ms = event_ms(torch, lambda: rec.append(s.ucb_argmax_dev(xc.data_ptr(), M, bench.VARSIGMA, stream)), args.calls)
                res[a][f"{key}_candidates_per_s"].append(M / (ms * 1e-3))
                info = s.screen_info()
                res[a]["records"][key] = list(rec[-1]) + [info["path"], info["digits"], info["survivors"]]
    Mj = 4096
    mean = torch.empty(Mj, dtype=torch.float64, device="cuda")
    cov = torch.empty((Mj, Mj), dtype=torch.float64, device="cuda")
    for a, (s, _) in sess.items():
        s.predict_f_cov_dev(xc.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream)
        c0 = s.launch_count()
        s.predict_f_cov_dev(xc.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream)
        res[a]["launches"]["predict_f_cov"] = s.launch_count() - c0
    for _ in range(args.reps):
        for a, (s, _) in sess.items():
            res[a]["predict_f_cov_ms_4096x4096"].append(
                event_ms(torch, lambda: s.predict_f_cov_dev(xc.data_ptr(), Mj, mean.data_ptr(), cov.data_ptr(), stream), 3))
    for s, _ in sess.values():
        s.close()

    out = {"gpu": gpu_identity(), "reps": args.reps, "calls_per_rep": args.calls,
           "workload": f"bench.py C3 inputs: N={N}, d={d}, M={M}, theta={bench.fixed_theta(d).tolist()} per Matern52 component, Linear variance 1/d",
           "arms": {}}
    for a in ARMS:
        r = res[a]
        out["arms"][a] = {"lml_grad_ms": {k: spread(v) for k, v in r["lml_grad_ms"].items()},
                          "c3_screened_candidates_per_s": spread(r["c3_screened_candidates_per_s"]),
                          "c3_unscreened_candidates_per_s": spread(r["c3_unscreened_candidates_per_s"]),
                          "predict_f_cov_ms_4096x4096": spread(r["predict_f_cov_ms_4096x4096"]),
                          "launches_per_call": r["launches"], "last_records": r["records"]}
    out["ratios"] = {}
    for arm, base in PAIRS:
        x, b = out["arms"][arm], out["arms"][base]
        r = {k: x[k]["median"] / b[k]["median"] for k in ("c3_screened_candidates_per_s", "c3_unscreened_candidates_per_s")}
        r["predict_f_cov_time"] = x["predict_f_cov_ms_4096x4096"]["median"] / b["predict_f_cov_ms_4096x4096"]["median"]
        for k in x["lml_grad_ms"]:
            r[f"lml_grad_{k}_time"] = x["lml_grad_ms"][k]["median"] / b["lml_grad_ms"][k]["median"]
        out["ratios"][f"{arm} / {base}"] = r
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as handle:
        json.dump(out, handle, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "ratios")}))


if __name__ == "__main__":
    main()
