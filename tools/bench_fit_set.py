"""Fit sets: one launch for every problem and copy against a fit and a launch per problem -> one JSON file.

    python tools/bench_fit_set.py [--out profiles/fit_set_r07.json] [--reps 5] [--copies 1000] [--sets 64,256]

Workload: K problems of configs.correlator(nexp) with ny drawn from 48 ... 80 per problem (so x grids and ny differ),
correlated data drawn around the truth, a prior per problem (scaled per problem), 1000 bootstrap copies each; the
K = 4 shape (nexp = 4, np = 8) and the C3 shape (nexp = 8, np = 16), for 64 and 256 problems.  Arms:
  (a)  lsqfit_b200.fit_set(...).bootstrapped_fits(copies): one whitening call, one central launch, the copies' means
       and one copies launch, end to end; (a_launch) the copies launch alone, set and means prebuilt;
  (b)  what users do without sets: per problem a nonlinear_fit plus bootstrapped_fits(copies) with the default kernel,
       end to end;
  (c)  (b) with every problem's fit (plan, whitening) prebuilt and its means given: the central and copies launches.
The arms alternate within each of --reps repetitions after a warm-up of each; times are host clocks around work that
ends in a device synchronise (min / median / max reported).  The card's name and power limit are read in the same run.
Fails without a GPU.
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


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def clock(torch, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), r


def stats(ms):
    return dict(min=min(ms), median=float(np.median(ms)), max=max(ms), all=ms)


def problems(nexp, K, seed=17):
    from lsqfit_b200 import configs
    rng = np.random.default_rng(seed)
    data, priors = [], []
    for k in range(K):
        cfg = configs.correlator(nexp, ny=int(rng.integers(48, 81)), dt=0.1 + 0.05 * rng.random())
        y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ rng.standard_normal(cfg["ny"])
        data.append((cfg["x"], y, cfg["ycov"]))
        priors.append((cfg["prior_mean"], cfg["prior_sdev"] * (1 + 0.2 * rng.random())))
    return data, priors


def shape(nexp, K, copies, reps, seed=17):
    import torch
    import lsqfit_b200 as lb
    from lsqfit_b200 import fitter
    fitter.PLAN_CACHE.capacity = 2 * K + 16          # arm (c) keeps every problem's plan alive at once
    data, priors = problems(nexp, K, seed)
    seeds = [seed + k for k in range(K)]

    def arm_a():
        fs = lb.fit_set(data, priors, fcn="multiexp")
        return fs, fs.bootstrapped_fits(copies, seeds=seeds)

    def arm_b():
        out = []
        for d, p, s in zip(data, priors, seeds):
            f = lb.nonlinear_fit(data=d, prior=p, fcn="multiexp")
            out.append(f.bootstrapped_fits(copies, seed=s))
        return out

    fits = [lb.nonlinear_fit(data=d, prior=p, fcn="multiexp") for d, p in zip(data, priors)]
    fmeans = [f.bootstrap_means(copies, s) for f, s in zip(fits, seeds)]
    fs, _ = arm_a()
    smeans = fs.bootstrap_means(copies, seeds=seeds)

    def arm_c():
        out = []
        for f, m in zip(fits, fmeans):
            plan = f._spec.plan(f.device)
            plan.fit_batch(f._spec.mean, f.p0, tol=f.tol, maxit=f.maxit)
            out.append(f._batch(m, f.pmean))
        return out

    def arm_a_launch():
        return fs._fit(smeans, fs.pmean, K * copies)

    arms = dict(a=arm_a, b=arm_b, c=arm_c, a_launch=arm_a_launch)
    for fn in arms.values():
        clock(torch, fn)                                    # warm-up
    ms = dict((k, []) for k in arms)
    for _ in range(reps):
        for k, fn in arms.items():
            ms[k].append(clock(torch, fn)[0])
    _, (fs_, bs) = clock(torch, arm_a)
    a = bs.arrays()
    conv = float(np.mean(a["status"] > 0))
    nys = [len(d[1]) for d in data]
    return dict(nexp=nexp, np=2 * nexp, problems=K, copies=copies, fits=K * copies, ny_min=min(nys), ny_max=max(nys),
                converged_fraction=conv, central_stopping=[int(v) for v in np.unique(fs_.stopping_criterion)],
                ms=dict((k, stats(v)) for k, v in ms.items()),
                speedup_median=dict(b_over_a=float(np.median(ms["b"]) / np.median(ms["a"])),
                                    c_over_a=float(np.median(ms["c"]) / np.median(ms["a"])),
                                    c_over_a_launch=float(np.median(ms["c"]) / np.median(ms["a_launch"]))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fit_set_r07.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--copies", type=int, default=1000)
    ap.add_argument("--sets", default="64,256")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_fit_set needs a CUDA device")
    res = dict(card=card(), reps=args.reps, shapes=[])
    for K in (int(v) for v in args.sets.split(",")):
        for nexp in (4, 8):
            r = shape(nexp, K, args.copies, args.reps)
            res["shapes"].append(r)
            print(json.dumps(dict((k, r[k]) for k in ("nexp", "problems", "fits", "speedup_median"))), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
