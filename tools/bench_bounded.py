"""Cost of bound constraints in the batched kernels (fit_kernel<F, 3>, scipy's trf_bounds decisions) -> one JSON file.

    python tools/bench_bounded.py [--out profiles/bounded_r03.json] [--reps 5] [--c4 1000000] [--c3 10000] [--cpu 2000]

* C4 shape (3-exponential correlator, simulated copies, p0 = pexact): the bounded and the unbounded one-warp kernel on
  the SAME batch, alternating, CUDA events, after a warm-up of both; box: E_k >= 0 and the two highest energies within
  one standard deviation (of the unbounded copies) of pexact, so that a share of the copies ends on a bound.
* C3 shape (8-exponential correlator, bootstrap copies, p0 = prior mean): E_k >= 0 and a box on the amplitudes
  (a_k in [0, 1]); the bounded one-warp kernel next to the unbounded default kernel of the shape.
* CPU rate: scipy's bounded trf (the oracle, tests/../oracle) on every host core over --cpu C4 copies.
Reports fits/s, mean function evaluations per fit and the fraction of copies with an active bound, with the card's
name and power limit read in the same run.  Fails without a GPU.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def timed(torch, fn, reps):
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def active_fraction(x, lo, hi):
    on = (np.isfinite(lo) & (np.abs(x - lo) <= 1e-7 * np.maximum(1, np.abs(lo)))) | \
         (np.isfinite(hi) & (np.abs(x - hi) <= 1e-7 * np.maximum(1, np.abs(hi))))
    return float(np.mean(np.any(on, axis=1)))


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


def summary(ms, B, out):
    ms = np.array(ms)
    return dict(ms_median=float(np.median(ms)), ms_min=float(ms.min()), ms_max=float(ms.max()),
                fits_per_s=float(B / (np.median(ms) * 1e-3)), mean_nfev=float(out.nit.double().mean()),
                converged=float((out.status > 0).double().mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bounded_r03.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c4", type=int, default=1000000)
    ap.add_argument("--c3", type=int, default=10000)
    ap.add_argument("--cpu", type=int, default=2000)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_bounded: no CUDA device (this measurement needs the GPU)")
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    res = dict(card=card(), settings=dict(reps=args.reps, c4=args.c4, c3=args.c3, cpu=args.cpu))
    dev = torch.device("cuda", 0)

    # ---- C4 shape: bounded vs unbounded one-warp kernel, same batch, alternating
    cfg = configs.c4(B=args.c4)
    npar = cfg["np"]
    pdf, means = setup(lb, cfg, args.c4, vary_prior=False)
    md, p0 = torch.as_tensor(means).to(dev), cfg["p0"]
    plan = lb.Plan("multiexp", npar, cfg["ny"], cfg["x"], pdf.i_invwgts, team=1)
    free = plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], want_cov=False)
    sd = free.x[free.status > 0].std(dim=0).cpu().numpy()
    K = npar // 2
    lo, hi = np.full(npar, -np.inf), np.full(npar, np.inf)
    lo[K:] = 0.0
    for j in (npar - 2, npar - 1):
        lo[j], hi[j] = p0[j] - sd[j], p0[j] + sd[j]
    bnd = plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], want_cov=False, bounds=(lo, hi))
    t_free, t_bnd = [], []
    for _ in range(args.reps):
        t_free += timed(torch, lambda: plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], out=free), 1)
        t_bnd += timed(torch, lambda: plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], out=bnd,
                                                     bounds=(lo, hi)), 1)
    res["c4"] = dict(B=args.c4, box=dict(lb=lo.tolist(), ub=hi.tolist()), kernel="one warp per fit (team 1)",
                     unbounded=summary(t_free, args.c4, free), bounded=summary(t_bnd, args.c4, bnd),
                     active_fraction=active_fraction(bnd.x.cpu().numpy(), lo, hi))
    res["c4"]["bounded_over_unbounded_time"] = res["c4"]["bounded"]["ms_median"] / res["c4"]["unbounded"]["ms_median"]
    print(json.dumps(res["c4"], indent=1))
    c4_box, c4_means = (lo, hi), means[:args.cpu]
    del md, free, bnd, plan

    # ---- C3 shape: bounded one-warp kernel vs the unbounded default kernel
    cfg = configs.c3(B=args.c3)
    npar = cfg["np"]
    K = npar // 2
    pdf, means = setup(lb, cfg, args.c3, vary_prior=True)
    md, p0 = torch.as_tensor(means).to(dev), cfg["p0"]
    plan = lb.Plan("multiexp", npar, cfg["ny"], cfg["x"], pdf.i_invwgts)
    lo, hi = np.full(npar, -np.inf), np.full(npar, np.inf)
    lo[:K], hi[:K], lo[K:] = 0.0, 1.0, 0.0
    free = plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"])
    team = plan.last_team()
    bnd = plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], bounds=(lo, hi))
    t_free, t_bnd = [], []
    for _ in range(args.reps):
        t_free += timed(torch, lambda: plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], out=free), 1)
        t_bnd += timed(torch, lambda: plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], out=bnd,
                                                     bounds=(lo, hi)), 1)
    res["c3"] = dict(B=args.c3, box=dict(lb=lo.tolist(), ub=hi.tolist()),
                     unbounded=dict(summary(t_free, args.c3, free), warps_per_fit=team),
                     bounded=dict(summary(t_bnd, args.c3, bnd), warps_per_fit=plan.last_team()),
                     active_fraction=active_fraction(bnd.x.cpu().numpy(), lo, hi))
    print(json.dumps(res["c3"], indent=1))

    # ---- CPU rate of scipy's bounded trf on the C4 copies
    import test_bounded_batch_gpu as T
    cfg4 = configs.c4(B=args.cpu)
    jobs = [(m, cfg4["p0"], cfg4["tol"], c4_box[0], c4_box[1]) for m in c4_means]
    t0 = time.perf_counter()
    ref = T._pool(T._corr_init, (3,), T._corr_job, jobs)
    dt = time.perf_counter() - t0
    res["cpu_scipy_bounded_trf"] = dict(B=len(jobs), cores=os.cpu_count(), seconds=dt, fits_per_s=len(jobs) / dt,
                                        mean_nfev=float(np.mean([r["nit"] for r in ref])),
                                        note="wall time including the process pool's start-up")
    print(json.dumps(res["cpu_scipy_bounded_trf"], indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
