"""User-defined device models (lsqfit_b200.cuda_functor) against the built-in functor of the same model -> one JSON file.

    python tools/bench_user_functor.py [--out profiles/user_functor_r04.json] [--reps 5] [--copies 1000000]

* Fit rate on the C4 shape (3-exponential correlator, np 6, simulated copies, p0 = pexact, the one-warp kernel that
  the shape gets by default) for three functors of the same model, on the SAME batch, alternating, CUDA events, after
  a warm-up of each:
    builtin  MultiExp<3> of the library (hand-written gradient);
    functor  the same template re-exported by a functor-form plug-in (the same machine code: expected equal);
    body     the model as a body-form plug-in, differentiated by Dual<6> (ADFunctor).
* Plug-in compile time for a body of np 4 and one of np 16 (a fresh cache directory, wall clock of nvcc on this host).
The card's name and power limit are read in the same run.  Fails without a GPU.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MULTIEXP = "template <int NP> using Model = MultiExp<NP / 2>;"
MULTIEXP_BODY = """
const double t = x[0];
T f = b[0] * exp(-(b[3] * t));
f = f + b[1] * exp(-(b[4] * t));
f = f + b[2] * exp(-(b[5] * t));
return f;
"""
RAT43 = "return b[0] / pow(1.0 + exp(b[1] - b[2] * x[0]), 1.0 / b[3]);"
POLY16 = """
const double t = x[0];
T f = b[15];
for (int n = 14; n >= 0; --n) f = f * t + b[n];
return exp(-f);
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


def compile_times():
    from lsqfit_b200 import user_functor as uf
    out = {}
    with tempfile.TemporaryDirectory() as d:
        os.environ["B200LM_FUNCTOR_CACHE"] = d
        try:
            for label, src, n in (("np4_rat43_body", RAT43, 4), ("np16_exp_poly_body", POLY16, 16)):
                t0 = time.perf_counter()
                uf.build_plugin("bench_compile_%d" % n, src, n)
                out[label] = round(time.perf_counter() - t0, 2)
        finally:
            del os.environ["B200LM_FUNCTOR_CACHE"]
    out["host_cpus"] = os.cpu_count()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "user_functor_r04.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--copies", type=int, default=1000000)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_user_functor: no CUDA device (there is no CPU fallback)")
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs
    from parity_util import correlator_problem
    res = dict(card=card(), copies=a.copies, reps=a.reps)
    res["compile_s"] = compile_times()
    models = dict(builtin=lb.Functor("multiexp"),
                  functor=lb.cuda_functor("ut_multiexp", MULTIEXP, (6, 16), form="functor"),
                  body=lb.cuda_functor("bench_multiexp_body", MULTIEXP_BODY, 6))
    cfg, opdf = correlator_problem(3)
    ny, npar = cfg["ny"], cfg["np"]
    means = torch.as_tensor(configs.bootstrap_means(cfg, a.copies, 4245, cov=opdf.cov[:ny, :ny], vary_prior=False)).cuda()
    p0 = cfg["ptrue"].copy()
    plans = dict((k, lb.Plan(f, npar, ny, cfg["x"], opdf.i_invwgts)) for k, f in models.items())
    tol = (1e-8, 1e-10, 1e-10)
    outs = {}
    for k, p in plans.items():                                  # warm-up; keep the results
        outs[k] = p.fit_batch(means, p0, tol=tol, maxit=1000).numpy()
    ms = dict((k, []) for k in plans)
    nfev = {}
    for _ in range(a.reps):
        for k, p in plans.items():
            ms[k].append(timed(torch, lambda: p.fit_batch(means, p0, tol=tol, maxit=1000)))
            nfev[k] = p.last_stats()[0] / a.copies
    ref = outs["builtin"]
    sd = np.sqrt(np.einsum("bii->bi", ref["cov"]))
    res["c4"] = {}
    for k in plans:
        o = outs[k]
        res["c4"][k] = dict(ms=[round(v, 3) for v in ms[k]], median_ms=round(float(np.median(ms[k])), 3),
                            fits_per_s=round(a.copies / (float(np.median(ms[k])) * 1e-3)),
                            spread=round((max(ms[k]) - min(ms[k])) / float(np.median(ms[k])), 4),
                            nfev_per_fit=round(nfev[k], 3), last_team=plans[k].last_team(),
                            converged=float(np.mean(o["status"] > 0)),
                            bits_equal_builtin=bool(all(o[q].tobytes() == ref[q].tobytes() for q in
                                                        ("x", "chi2", "cov", "logdet", "nit", "status"))),
                            max_dx_over_sd_vs_builtin=float(np.max(np.abs(o["x"] - ref["x"]) / sd)))
    res["body_over_builtin_time"] = round(res["c4"]["body"]["median_ms"] / res["c4"]["builtin"]["median_ms"], 3)
    res["functor_over_builtin_time"] = round(res["c4"]["functor"]["median_ms"] / res["c4"]["builtin"]["median_ms"], 3)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
