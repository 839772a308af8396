"""fit.p of every window of a fit-window scan, jointly: scan.p against a fit and fit.p per window -> one JSON file.

    python tools/bench_window_propagate.py [--out profiles/window_propagate_r06.json] [--reps 5]

Workload: configs.correlator(K) with 64 points.  The 64 windows of tools/bench_window_scan.py (tmin = 1..16 x tmax in
{40, 48, 56, 64}, 1-based inclusive) for K = 4 and the C3 shape K = 8, and one scan of 256 windows (tmin = 1..32 x
tmax in {36, 40, ..., 64}) for K = 4.  Arms:
  (a)  scan.p on a built scan (its cached result dropped before each call): the central batch again with J, the
       window propagation (DMMA GEMMs, whitening applied from the row tables, per-window svd corrections), and the
       copies of D and of the joint covariance to the host;
  (b)  what users do without it: per window a nonlinear_fit of the window's data plus fit.p and fit.D, then the joint
       covariance D C D^T of all windows in numpy.
The arms alternate within each of --reps repetitions after a warm-up of each; times are host clocks around work that
ends in a device synchronise (min / median / max reported).  The largest difference between the two arms' joint
covariances (normalised by sqrt(S_ii S_jj)) is recorded: the windows' fits run on different kernels, so they agree to
the fits' tolerance, not to rounding.  The card's name and power limit are read in the same run.  Fails without a GPU.
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


def masks_of(ny, tmins, tmaxs):
    i = np.arange(1, ny + 1)
    return np.array([(i >= lo) & (i <= hi) for lo in tmins for hi in tmaxs])


def shape(K, masks, reps, seed=17):
    import torch
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    cfg = configs.correlator(K)
    ny = cfg["ny"]
    y = cfg["f"] + np.linalg.cholesky(cfg["ycov"]) @ np.random.default_rng(seed).standard_normal(ny)
    prior = (cfg["prior_mean"], cfg["prior_sdev"])
    fit = lb.nonlinear_fit(data=(cfg["x"], y, cfg["ycov"]), fcn="multiexp", prior=prior)
    C = fit.yp_pdf.cov_in
    N = C.shape[0]
    nwin, npar = len(masks), cfg["np"]
    scan = fit.window_fits(masks)

    def arm_a():
        scan._p = None
        return scan.p[1]

    def arm_b():
        D = np.zeros((nwin, npar, N))
        own = []
        for w, m in enumerate(masks):
            f = lb.nonlinear_fit(data=(cfg["x"][m], y[m], cfg["ycov"][np.ix_(m, m)]), fcn="multiexp", prior=prior,
                                 p0=fit.pmean)
            own.append(f.p[1])
            D[w][:, scan.sels[w]] = f.D
        Dall = D.reshape(nwin * npar, N)
        S = (Dall @ C @ Dall.T).reshape(nwin, npar, nwin, npar)
        for w in range(nwin):
            S[w, :, w, :] = own[w]
        return S

    arms = dict(a=arm_a, b=arm_b)
    res = {}
    for k, fn in arms.items():
        res[k] = clock(torch, fn)[1]          # warm-up
    ms = dict((k, []) for k in arms)
    for _ in range(reps):
        for k, fn in arms.items():
            ms[k].append(clock(torch, fn)[0])
    n = nwin * npar
    s = np.sqrt(np.diagonal(res["b"].reshape(n, n)))
    diff = np.abs(res["a"] - res["b"]).reshape(n, n) / np.outer(s, s)
    out = dict(K=K, np=npar, ny=ny, N=N, nwin=nwin, nchiv=dict(min=int(scan.nchiv.min()), max=int(scan.nchiv.max())),
               joint_cov_doubles=n * n, max_normalised_diff_a_vs_b=float(diff.max()))
    for k in arms:
        out["ms_" + k] = stats(ms[k])
    out["speedup_b_over_a"] = float(np.median(ms["b"]) / np.median(ms["a"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "window_propagate_r06.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_window_propagate: needs a CUDA device")
    ny = 64
    m64 = masks_of(ny, range(1, 17), (40, 48, 56, 64))
    m256 = masks_of(ny, range(1, 33), range(36, 65, 4))
    assert len(m64) == 64 and len(m256) == 256
    res = dict(card=card(), results=[shape(4, m64, a.reps), shape(8, m64, a.reps), shape(4, m256, a.reps)])
    res["card_after"] = card()
    for r in res["results"]:
        print(json.dumps(dict((k, (v["median"] if k.startswith("ms_") else v)) for k, v in r.items()), default=float))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, default=float)


if __name__ == "__main__":
    main()
