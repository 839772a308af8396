"""Parameter distributions (fit_kernel<F, 5>: the model at q = T(p)) against the kernels without them -> one JSON file.

    python tools/bench_pdist.py [--out profiles/pdist_r09.json] [--reps 5] [--c4-copies 1000000] [--c3-copies 10000]

* C4 shape (3-exponential correlator, np 6, simulated copies, p0 = pexact): the untransformed one-warp kernel (MODE 0)
  against log(E) on every energy (MODE 5), both one warp per fit.  Evaluations per fit and batch time over the total
  number of evaluations ("ns per evaluation": a throughput figure of the whole GPU, not the latency of one).
* C3 shape (8 exponentials, np 16, 10^4 bootstrap copies, prior means varied): MODE 5 against the untransformed default
  kernel (a team of two warps per fit) and against the untransformed one-warp kernel.
* Against a plug-in: a body-form cuda_functor that takes exp of its own energy parameters (4 exponentials, plain keys)
  against the built-in multiexp with log(E) codes (MODE 5), 10^5 simulated copies.  Same model, same data, same prior.
The log(E) fits have the prior log E_k = log(E_k)(0.2 / E_k) (the linearised width of the plain prior E_k(0.2)), so the
two fits of a pair are close but not the same statistical model; the plug-in pair is the same model.
Every timed batch is a CUDA-event interval after a warm-up of every plan, the variants alternate, 5 repeats, medians with
min and max.  The card's name and power limit are read in the same run.  Fails without a GPU.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

TOL = (1e-8, 1e-10, 1e-10)
EXP_ENERGIES = """
const double t = x[0];
T s = b[0] * exp(-(exp(b[4]) * t));
s = s + b[1] * exp(-(exp(b[5]) * t));
s = s + b[2] * exp(-(exp(b[6]) * t));
s = s + b[3] * exp(-(exp(b[7]) * t));
return s;
"""


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


def log_problem(K):
    """(cfg, oracle PDF of the plain prior, oracle PDF of the log(E) prior, log-space prior mean and sdev)"""
    from oracle.whiten import PDF as OPDF
    from lsqfit_b200 import configs
    cfg = configs.correlator(K)
    ny = cfg["ny"]
    pm, ps = cfg["prior_mean"].copy(), cfg["prior_sdev"].copy()
    lpm, lps = pm.copy(), ps.copy()
    lpm[K:], lps[K:] = np.log(pm[K:]), ps[K:] / pm[K:]
    pdfs = []
    for s in (ps, lps):
        C = np.zeros((ny + 2 * K, ny + 2 * K))
        C[:ny, :ny] = cfg["ycov"]
        C[ny:, ny:] = np.diag(s ** 2)
        pdfs.append(OPDF(np.concatenate([cfg["f"], pm]), C, svdcut=1e-12))
    return cfg, pdfs[0], pdfs[1], lpm, lps


def to_log_means(means, cfg, lpm, lps):
    """the same draws with the prior columns of E moved to the log(E) prior: z = (m - pm) / ps -> lpm + lps z"""
    K, ny = cfg["K"], cfg["ny"]
    out = means.clone()
    pm, ps = cfg["prior_mean"], cfg["prior_sdev"]
    for k in range(K, 2 * K):
        z = (means[:, ny + k] - pm[k]) / ps[k]
        out[:, ny + k] = lpm[k] + lps[k] * z
    return out


def run(torch, variants, reps, n):
    """variants: name -> (plan, means, p0).  Warm-up, then `reps` alternating timed batches."""
    outs, ms, nfev = {}, dict((k, []) for k in variants), {}
    for k, (plan, m, p0) in variants.items():
        outs[k] = plan.fit_batch(m, p0, tol=TOL, maxit=1000).numpy()
    for _ in range(reps):
        for k, (plan, m, p0) in variants.items():
            ms[k].append(timed(torch, lambda: plan.fit_batch(m, p0, tol=TOL, maxit=1000)))
            nfev[k] = plan.last_stats()[0]
    res = {}
    for k, (plan, _, _) in variants.items():
        med = float(np.median(ms[k]))
        res[k] = dict(ms=[round(v, 3) for v in ms[k]], median_ms=round(med, 3), min_ms=round(min(ms[k]), 3),
                      max_ms=round(max(ms[k]), 3), fits_per_s=round(n / (med * 1e-3)),
                      evals_per_fit=round(nfev[k] / n, 3), ns_per_eval=round(med * 1e6 / nfev[k], 3),
                      last_team=plan.last_team(), converged=float(np.mean(outs[k]["status"] > 0)))
    return res, outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pdist_r09.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c4-copies", type=int, default=1000000)
    ap.add_argument("--c3-copies", type=int, default=10000)
    ap.add_argument("--plugin-copies", type=int, default=100000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_pdist: no CUDA device (there is no CPU fallback)")
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    res = dict(card=card(), reps=a.reps, tol=TOL)
    # ---- C4: MODE 0 against MODE 5, one warp per fit -------------------------------------------------------------
    cfg, opdf, lpdf, lpm, lps = log_problem(3)
    ny, npar, K = cfg["ny"], cfg["np"], 3
    code = np.array([0] * K + [1] * K, dtype=np.int32)
    means = torch.as_tensor(configs.bootstrap_means(cfg, a.c4_copies, 777, cov=opdf.cov[:ny, :ny],
                                                    vary_prior=False)).cuda()
    lmeans = to_log_means(means, cfg, lpm, lps)
    plain = lb.Plan("multiexp", npar, ny, cfg["x"], opdf.i_invwgts, team=1)
    trans = lb.Plan("multiexp", npar, ny, cfg["x"], lpdf.i_invwgts, pdist=(code, np.zeros(npar), np.ones(npar)))
    p0 = cfg["ptrue"].copy()
    lp0 = np.concatenate([p0[:K], np.log(p0[K:])])
    res["c4"], _ = run(torch, dict(mode0=(plain, means, p0), mode5_logE=(trans, lmeans, lp0)), a.reps, a.c4_copies)
    res["c4"]["copies"] = a.c4_copies
    res["c4"]["mode5_over_mode0_ns_per_eval"] = round(res["c4"]["mode5_logE"]["ns_per_eval"] /
                                                      res["c4"]["mode0"]["ns_per_eval"], 4)
    del means, lmeans, plain, trans
    torch.cuda.empty_cache()
    # ---- C3: MODE 5 against the default (team of two) and the one-warp kernel -------------------------------------
    cfg, opdf, lpdf, lpm, lps = log_problem(8)
    ny, npar, K = cfg["ny"], cfg["np"], 8
    code = np.array([0] * K + [1] * K, dtype=np.int32)
    means = torch.as_tensor(configs.bootstrap_means(cfg, a.c3_copies, 12345, cov=opdf.cov[:ny, :ny])).cuda()
    lmeans = to_log_means(means, cfg, lpm, lps)
    default = lb.Plan("multiexp", npar, ny, cfg["x"], opdf.i_invwgts)
    one = lb.Plan("multiexp", npar, ny, cfg["x"], opdf.i_invwgts, team=1)
    trans = lb.Plan("multiexp", npar, ny, cfg["x"], lpdf.i_invwgts, pdist=(code, np.zeros(npar), np.ones(npar)))
    p0, lp0 = cfg["prior_mean"].copy(), lpm.copy()
    res["c3"], _ = run(torch, dict(default=(default, means, p0), one_warp=(one, means, p0),
                                   mode5_logE=(trans, lmeans, lp0)), a.reps, a.c3_copies)
    res["c3"]["copies"] = a.c3_copies
    # ---- a plug-in that takes exp of its energies against MODE 5 ---------------------------------------------------
    with tempfile.TemporaryDirectory() as d:
        os.environ["B200LM_FUNCTOR_CACHE"] = d
        fcn = lb.cuda_functor("bench_pdist_expE", EXP_ENERGIES, 8)
    cfg, opdf, lpdf, lpm, lps = log_problem(4)
    ny, npar, K = cfg["ny"], cfg["np"], 4
    code = np.array([0] * K + [1] * K, dtype=np.int32)
    means = torch.as_tensor(configs.bootstrap_means(cfg, a.plugin_copies, 4245, cov=opdf.cov[:ny, :ny],
                                                    vary_prior=False)).cuda()
    lmeans = to_log_means(means, cfg, lpm, lps)
    plug = lb.Plan(fcn, npar, ny, cfg["x"], lpdf.i_invwgts, team=1)
    trans = lb.Plan("multiexp", npar, ny, cfg["x"], lpdf.i_invwgts, pdist=(code, np.zeros(npar), np.ones(npar)))
    lp0 = np.concatenate([cfg["ptrue"][:K], np.log(cfg["ptrue"][K:])])
    res["plugin"], outs = run(torch, dict(plugin_exp_body=(plug, lmeans, lp0), mode5_logE=(trans, lmeans, lp0)),
                              a.reps, a.plugin_copies)
    res["plugin"]["copies"] = a.plugin_copies
    sd = np.sqrt(np.einsum("bii->bi", outs["plugin_exp_body"]["cov"]))
    ok = (outs["plugin_exp_body"]["status"] > 0) & (outs["mode5_logE"]["status"] > 0)
    res["plugin"]["max_dx_over_sd"] = float(np.max(np.abs(outs["mode5_logE"]["x"] - outs["plugin_exp_body"]["x"])[ok]
                                                   / sd[ok]))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
