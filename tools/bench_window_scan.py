"""Fit-window scans: one launch for every window and copy against a fit and a launch per window -> one JSON file.

    python tools/bench_window_scan.py [--out profiles/window_scan_r05.json] [--reps 5] [--copies 1000] [--cpu 16]

Workload: configs.correlator(K) with 64 points, windows tmin = 1..16 x tmax in {40, 48, 56, 64} (1-based time
indices, inclusive: 64 windows), 1000 bootstrap copies each; K = 4 and the C3 shape K = 8.  Arms:
  (a)  fit.window_fits(masks).bootstrapped_fits(copies): one whitening call, one central launch, one copies launch,
       end to end; (a_launch) the copies launch alone, scan and means prebuilt;
  (b)  what users do without scans: per window a nonlinear_fit plus bootstrapped_fits(copies) with the default kernel,
       end to end;
  (c)  (b) with every window's fit (plan, whitening) prebuilt and the means given: the 64 launches only;
  (d)  the oracle (scipy trf on the host, one core) over --cpu (window, copy) pairs, as fits/s.
The arms alternate within each of --reps repetitions after a warm-up of each; times are host clocks around work that
ends in a device synchronise (min / median / max reported).  ns per evaluation: the window kernel against the
shared-memory-staged one-warp kernel on the same 64 x copies bootstrap fits of the full-range window (kernel time over
the batch's function evaluations, b200lm_last_stats).  The card's name and power limit are read in the same run.
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


def masks_of(ny):
    i = np.arange(1, ny + 1)
    return np.array([(i >= lo) & (i <= hi) for lo in range(1, 17) for hi in (40, 48, 56, 64)])


def shape(K, copies, reps, ncpu, seed=17):
    import torch
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs, fitter
    fitter.PLAN_CACHE.capacity = 512          # arm (c) keeps 64 windows' plans alive at once
    cfg = configs.correlator(K)
    ny = cfg["ny"]
    y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ np.random.default_rng(seed).standard_normal(ny)
    prior = (cfg["prior_mean"], cfg["prior_sdev"])
    fit = lb.nonlinear_fit(data=(cfg["x"], y, cfg["ycov"]), fcn="multiexp", prior=prior)
    masks = masks_of(ny)
    nwin = len(masks)
    means = fit.bootstrap_means(copies, seed)

    def arm_a():
        return fit.window_fits(masks).bootstrapped_fits(copies, means=means)

    def window_fit(m):
        return lb.nonlinear_fit(data=(cfg["x"][m], y[m], cfg["ycov"][np.ix_(m, m)]), fcn="multiexp", prior=prior,
                                p0=fit.pmean)

    def arm_b():
        return [window_fit(m).bootstrapped_fits(copies, means=means[:, torch.as_tensor(np.concatenate(
            [np.nonzero(m)[0], np.arange(ny, fit.yp_pdf.size)]), device=means.device)]) for m in masks]

    scan = fit.window_fits(masks)
    fits = [window_fit(m) for m in masks]
    sels = [torch.as_tensor(s, device=means.device) for s in scan.sels]
    wmeans = [means[:, s].contiguous() for s in sels]

    def arm_a_launch():
        return scan.bootstrapped_fits(copies, means=means)

    def arm_c():
        return [f._batch(wm, f.pmean) for f, wm in zip(fits, wmeans)]

    arms = dict(a=arm_a, a_launch=arm_a_launch, b=arm_b, c=arm_c)
    for fn in arms.values():
        clock(torch, fn)                      # warm-up
    ms = dict((k, []) for k in arms)
    for _ in range(reps):
        for k, fn in arms.items():
            ms[k].append(clock(torch, fn)[0])
    nfits = nwin * copies
    out = dict(K=K, np=cfg["np"], ny=ny, nwin=nwin, copies=copies, fits=nfits,
               nchiv=dict(min=int(scan.nchiv.min()), max=int(scan.nchiv.max())),
               default_kernel_warps_per_fit=None)
    fits[0]._batch(wmeans[0], fits[0].pmean)
    out["default_kernel_warps_per_fit"] = fits[0]._spec.plan().last_team()
    for k in arms:
        out["ms_" + k] = stats(ms[k])
        out["fits_per_s_" + k] = nfits / (1e-3 * float(np.median(ms[k])))
    # results of (a) and (c) agree? (different kernels sum in a different order: to rounding)
    a = scan.bootstrapped_fits(copies, means=means).arrays()
    c = arm_c()
    dx = max(float(np.max(np.abs(a["x"][w * copies:(w + 1) * copies] - c[w].arrays()["x"]) /
                          np.sqrt(np.diagonal(scan.cov[w]))[None, :])) for w in range(nwin))
    out["max_dx_a_vs_c_in_sdev"] = dx
    # ns per evaluation: the window kernel against the staged one-warp kernel, the full-range window, 64 x copies fits
    full = fit.window_fits(np.ones((1, ny), dtype=bool))
    big = fit.bootstrap_means(nfits, seed + 1)
    plan = fit._spec.plan()
    per_eval = dict(window=[], staged=[])
    for _ in range(reps + 1):
        t, _ = clock(torch, lambda: full.plan.fit_batch(big, full.pmean[0], tol=fit.tol, maxit=fit.maxit))
        per_eval["window"].append(1e6 * t / full.plan.last_stats()[0])
        plan.set_team(1)
        try:
            t, _ = clock(torch, lambda: plan.fit_batch(big, full.pmean[0], tol=fit.tol, maxit=fit.maxit))
            per_eval["staged"].append(1e6 * t / plan.last_stats()[0])
        finally:
            plan.set_team(0)
    out["ns_per_evaluation"] = dict((k, stats(v[1:])) for k, v in per_eval.items())    # first pair: warm-up
    # (d) the oracle on one host core
    if ncpu:
        from oracle.fit import nonlinear_fit as ofit
        rng = np.random.default_rng(seed)
        mh = means.cpu().numpy()
        t0 = time.perf_counter()
        for i in range(ncpu):
            w, j = int(rng.integers(nwin)), int(rng.integers(copies))
            m = masks[w]
            ofit("multiexp", cfg["x"][m], mh[j, :ny][m], cfg["ycov"][np.ix_(m, m)], prior_mean=mh[j, ny:],
                 prior_cov=np.diag(cfg["prior_sdev"] ** 2), p0=scan.pmean[w], svdcut=fit.svdcut, tol=fit.tol)
        out["oracle_fits_per_s_one_core"] = ncpu / (time.perf_counter() - t0)
        out["oracle_sample"] = ncpu
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "window_scan_r05.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--copies", type=int, default=1000)
    ap.add_argument("--cpu", type=int, default=16)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_window_scan: needs a CUDA device")
    res = dict(card=card(), results=[shape(K, a.copies, a.reps, a.cpu) for K in (4, 8)])
    res["card_after"] = card()
    for r in res["results"]:
        print(json.dumps(dict((k, v) for k, v in r.items() if not k.startswith("ms_")), default=float))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
