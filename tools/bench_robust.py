"""Cost of a robust loss in the batched kernels (fit_kernel<F, 6>, scipy's trf with loss= / f_scale=) -> one JSON file.

    python tools/bench_robust.py [--out profiles/robust_r10.json] [--reps 5] [--c4 1000000] [--c3 10000]
                                 [--single 100] [--cpu 200]

Workloads, each with soft_l1 and cauchy at f_scale = 2, and soft_l1 on copies with outliers planted in 3 % of the
copies' means (one data point moved by 30 sigma: rows on the far side of every loss's kink, clipped rows for cauchy):
* C4 shape (3-exponential correlator, 10^6 simulated copies, p0 = pexact), one warp per fit;
* C3 shape (8-exponential correlator, 10^4 bootstrap copies, p0 = prior mean).
For each: ms per batch (median and min-max of --reps repeats, alternating with the plain batch on the same copies,
CUDA events, after a warm-up of both), evaluations per fit and ns per evaluation, next to MODE 0 (no loss, one warp per
fit) on the same copies.  What users have without this kernel: the copies one at a time on the single-fit path
(nonlinear_fit(..., loss=...) with the copy's means and the parent's whitening, --single copies, ms per fit); and
scipy's robust trf (the oracle) on every host core over --cpu copies.  Registers, stack frame and spills of
fit_kernel<MultiExp<3|4|8>, 0 | 6> from cuobjdump -res-usage of the built library.  The card's name and power limit
are read in the same run.  Fails without a GPU.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CASES = (("soft_l1", 2.0, False), ("cauchy", 2.0, False), ("soft_l1", 2.0, True))


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def timed(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def summary(ms, B, out):
    ms = np.array(ms)
    nfev = float(out.nit.double().mean())
    return dict(ms_median=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()),
                fits_per_s=float(B / (np.median(ms) * 1e-3)), evals_per_fit=nfev,
                ns_per_eval=float(np.median(ms) * 1e6 / (B * nfev)), converged=float((out.status > 0).double().mean()))


def setup(lb, cfg, B, vary_prior):
    from lsqfit_b200 import configs
    ny, npar = cfg["ny"], cfg["np"]
    N = ny + npar
    full = np.zeros((N, N))
    full[:ny, :ny] = cfg["ycov"]
    full[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
    pdf = lb.PDF(np.concatenate([cfg["f"], cfg["prior_mean"]]), full, svdcut=cfg["svdcut"])
    means = configs.bootstrap_means(cfg, B, cfg["seed"], cov=pdf.cov[:ny, :ny], vary_prior=vary_prior)
    return pdf, means


def plant(cfg, means, seed=31):
    """one data point of 3 % of the copies moved by 30 sigma"""
    rng = np.random.default_rng(seed)
    B, ny = means.shape[0], cfg["ny"]
    rows = rng.choice(B, size=max(1, B * 3 // 100), replace=False)
    pts = rng.integers(0, ny, size=rows.size)
    out = means.copy()
    out[rows, pts] += 30.0 * np.sqrt(np.diag(cfg["ycov"]))[pts] * rng.choice([-1.0, 1.0], size=rows.size)
    return out


def shape(torch, lb, cfg, pdf, means, reps, team):
    dev = torch.device("cuda", 0)
    plan = lb.Plan("multiexp", cfg["np"], cfg["ny"], cfg["x"], pdf.i_invwgts, team=team)
    p0, B = cfg["p0"], means.shape[0]
    kw = dict(tol=cfg["tol"], maxit=cfg["maxit"])
    res = {}
    for loss, fs, outliers in CASES:
        md = torch.as_tensor(plant(cfg, means) if outliers else means).to(dev)
        plain = plan.fit_batch(md, p0, **kw)                          # warm-up of both
        rob = plan.fit_batch(md, p0, loss=loss, f_scale=fs, **kw)
        t_plain, t_rob = [], []
        for _ in range(reps):
            t_plain.append(timed(torch, lambda: plan.fit_batch(md, p0, out=plain, **kw)))
            t_rob.append(timed(torch, lambda: plan.fit_batch(md, p0, out=rob, loss=loss, f_scale=fs, **kw)))
        name = "%s_f%g%s" % (loss, fs, "_outliers" if outliers else "")
        res[name] = dict(mode0=dict(summary(t_plain, B, plain), warps_per_fit=team),
                         robust=dict(summary(t_rob, B, rob), warps_per_fit=plan.last_team()))
        res[name]["robust_over_mode0_time"] = res[name]["robust"]["ms_median"] / res[name]["mode0"]["ms_median"]
        print(name, json.dumps(res[name]))
        del md, plain, rob
    return res


def single_path(lb, cfg, pdf, means, n):
    """copies one at a time on the single-fit path (what batch drivers refused before): ms per fit"""
    import warnings
    ny = cfg["ny"]
    args = dict(fcn="multiexp", _yp_pdf=pdf, p0=cfg["p0"], tol=cfg["tol"], loss="soft_l1", f_scale=2.0)
    ms = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        lb.nonlinear_fit(data=(cfg["x"], means[0, :ny], None), prior=(means[0, ny:], cfg["prior_sdev"]), **args)
        for m in means[:n]:
            t0 = time.perf_counter()
            lb.nonlinear_fit(data=(cfg["x"], m[:ny], None), prior=(m[ny:], cfg["prior_sdev"]), **args)
            ms.append((time.perf_counter() - t0) * 1e3)
    ms = np.array(ms)
    return dict(copies=n, loss="soft_l1", f_scale=2.0, ms_per_fit_median=float(np.median(ms)),
                ms_per_fit_min=float(ms.min()), ms_per_fit_max=float(ms.max()),
                note="nonlinear_fit(..., loss=) per copy with the parent's whitening (_yp_pdf): single-fit path")


def scipy_rate(K, cfg, means, n):
    import test_robust_batch_gpu as T
    jobs = [(m, cfg["p0"], "soft_l1", 2.0) for m in means[:n]]
    t0 = time.perf_counter()
    T._pool(T._corr_init, (K,), T._corr_job, jobs)
    dt = time.perf_counter() - t0
    return dict(copies=n, cores=os.cpu_count(), seconds=dt, fits_per_s=n / dt, loss="soft_l1", f_scale=2.0,
                tol=list(T.TOL), note="scipy least_squares(loss=) through the oracle on a process pool; wall time with pool start-up")


def resources():
    """registers, stack frame and spills of fit_kernel<MultiExp<K>, 0 | 6> (cuobjdump -res-usage of the library)"""
    lib = os.path.join(ROOT, "lsqfit_b200", "libb200lm.so")
    r = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True)
    out, fn = {}, None
    for line in r.stdout.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        dm = fn and re.match(r"_ZN6b200lm10fit_kernelINS_8MultiExpILi(\d)EEELi(\d)EEEvNS_9FitParamsE$", fn)
        if dm and dm.group(1) in "348" and dm.group(2) in "06":
            vals = dict((k, int(v)) for k, v in re.findall(r"(REG|STACK|LOCAL):(\d+)", line))
            out["MultiExp<%s>, %s" % (dm.group(1), dm.group(2))] = vals
            fn = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "robust_r10.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c4", type=int, default=1000000)
    ap.add_argument("--c3", type=int, default=10000)
    ap.add_argument("--single", type=int, default=100)
    ap.add_argument("--cpu", type=int, default=200)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_robust: no CUDA device (this measurement needs the GPU)")
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    res = dict(card=card(), settings=vars(args), resources=resources())
    print(json.dumps(res["resources"]))
    for name, K, B, vary in (("c4", 3, args.c4, False), ("c3", 8, args.c3, True)):
        cfg = getattr(configs, name)(B=B)
        pdf, means = setup(lb, cfg, B, vary)
        res[name] = dict(B=B, shapes=shape(torch, lb, cfg, pdf, means, args.reps, 1))
        res[name]["single_fit_path"] = single_path(lb, cfg, pdf, means, args.single)
        print(name, "single", json.dumps(res[name]["single_fit_path"]))
        res[name]["cpu_scipy_robust_trf"] = scipy_rate(K, cfg, means, args.cpu)
        print(name, "scipy", json.dumps(res[name]["cpu_scipy_robust_trf"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
