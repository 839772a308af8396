#!/usr/bin/env python
"""Benchmark of the batched LM hot path (see DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json config 3): 8-exponential correlator, 64 correlated time slices,
16 diagonal priors, svdcut=1e-12, 10^4 bootstrap copies per GPU per step, p0 = prior mean,
tol=(1e-8,1e-10,1e-10), maxit=1000.  One "step" = one launch of the fit kernel over the
whole batch (plus, for N>1, the NCCL all-gather of the packed per-fit results).
Weak scaling: every rank fits its OWN 10^4 copies (a different seed per rank).

Prints ONE JSON line on rank 0 (stdout); NCCL's own log goes to stderr.
"""
import os
# The contract is ONE JSON line on stdout, and NCCL prints its banner / INFO lines to stdout unless told
# otherwise: its log is sent to stderr.  NCCL_DEBUG itself is left as the launcher set it (INFO by default
# for multi-rank runs, so that the rank count and the transport are visible in the captured log).
if int(os.environ.get("WORLD_SIZE", "1")) > 1 and os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
    os.environ["NCCL_DEBUG"] = "INFO"                      # communicator size and transport visible in the log
    os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
# NCCL prints its version banner to file descriptor 1 whatever NCCL_DEBUG_FILE says.  The real stdout is
# therefore put aside and fd 1 points at stderr for the whole run; emit() writes the one JSON line to the
# real stdout at the end.
import sys
sys.stdout.flush()
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (line + "\n").encode())
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fp64 LM fits/sec"
UNIT = "fits/s"
WORKLOAD = "C3: 8-exp correlator, 64 correlated time slices, 16 priors, 10k bootstrap fits per GPU"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=10000, help="fits per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=2000, help="fits timed on the host for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C1/C2/C4/C5 and saturated-batch figures")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (float64; above 60 MB in all, "
                         "a seeded sample of the fits)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no fit results")
    return args


DUMP_LIMIT = 60 * 1000 * 1000


def dump_outputs(path, arrays):
    """Writes every array as <path>/<name>.npy in float64 (nit and status are small integers, exact in float64).  Above
    DUMP_LIMIT bytes in all, every array keeps the same fraction of its rows (fits), chosen by a fixed seed from its
    shape alone: two builds run with the same arguments write the same rows and can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    arrays = dict((k, np.asarray(v, dtype=np.float64)) for k, v in arrays.items())
    frac = min(1.0, DUMP_LIMIT / float(sum(a.nbytes for a in arrays.values())))
    for name, a in sorted(arrays.items()):
        if frac < 1.0:
            rows = np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * frac), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(path, name + ".npy"), a)


def load_configs():
    """lsqfit_b200/configs.py loaded BY PATH: it is pure numpy, and importing it as part of the package
    would map libb200lm.so into the process -- the reference arm must not load any of the product."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_b200lm_configs", os.path.join(ROOT, "lsqfit_b200", "configs.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


# ------------------------------------------------------------------------------ CPU oracle leg
# The oracle restates lsqfit's scipy_least_squares plugin (src/lsqfit/_scipy.py:115-181).  ORACLE_XSCALE:
# "jac" = More' column scaling, the policy the device runs by default (GSL's default scaler, scipy
# x_scale='jac'); the reference plugin's own default is x_scale=1 -- both are timed and reported.
def _oracle_setup():
    configs = load_configs()
    from oracle.whiten import PDF as OPDF
    cfg = configs.c3()
    ny, npar = cfg["ny"], cfg["np"]
    N = ny + npar
    full = np.zeros((N, N))
    full[:ny, :ny] = cfg["ycov"]
    full[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
    mean0 = np.concatenate([cfg["f"], cfg["prior_mean"]])
    pdf = OPDF(mean0, full, svdcut=cfg["svdcut"])
    return configs, cfg, pdf


_G = {}


def _oracle_init():
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    os.environ["OMP_NUM_THREADS"] = "1"
    _G["configs"], _G["cfg"], _G["pdf"] = _oracle_setup()


def _oracle_fit(arg):
    from oracle.fit import nonlinear_fit
    mean, x_scale = arg
    cfg, pdf = _G["cfg"], _G["pdf"]
    ny = cfg["ny"]
    kw = {} if x_scale is None else dict(x_scale=x_scale)
    fit = nonlinear_fit("multiexp", cfg["x"], mean[:ny], prior_mean=mean[ny:], _yp_pdf=pdf,
                        p0=cfg["p0"], tol=cfg["tol"], maxit=cfg["maxit"], **kw)
    return fit.nit


def cpu_fits_per_sec(means, cores, x_scale):
    """The oracle on `cores` host processes; whitening shared (simulated_fit_iter style)."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    jobs = [(m, x_scale) for m in means]
    with ctx.Pool(cores, initializer=_oracle_init) as pool:
        pool.map(_oracle_fit, jobs[:cores])          # warm the workers
        t0 = time.perf_counter()
        nit = pool.map(_oracle_fit, jobs, chunksize=max(1, len(jobs) // (cores * 8)))
        dt = time.perf_counter() - t0
    return len(means) / dt, float(np.mean(nit))


def _ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the fit kernel per launch.  STATIC: taken from the
    committed `ncu --set full` capture of this kernel (newest profiles/traffic_r*.json), not measured in
    this run (DRAM counters need a profiler).  Returns (bytes or None, source)."""
    pdir = os.path.join(ROOT, "profiles")
    try:
        names = sorted(n for n in os.listdir(pdir) if n.startswith("traffic_r") and n.endswith(".json"))
    except OSError:
        names = []
    for name in reversed(names):
        try:
            t = json.load(open(os.path.join(pdir, name)))
            return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"]), "static: profiles/" + name
        except (OSError, ValueError, KeyError):
            continue
    return None, "no capture committed"


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
            except (ValueError, IndexError):
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=smax,
                    reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------ peaks
def fp64_peak():
    """(TFLOP/s, source).  MEASURED_PEAKS.json holds no FP64 figure, so the denominator is the
    FP64 FMA peak measured on this pool by profiles/fp64_peak.cu (committed as
    profiles/fp64_peak_r01.json); fallback = nominal 37 TFLOP/s."""
    for name in ("fp64_peak_r01.json",):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                d = json.load(open(p))
                return float(d["fp64_tflops"]), "measured (profiles/%s: %s)" % (name, d.get("how", ""))
            except Exception:
                pass
    return 37.0, "fallback: nominal B200 FP64 37 TFLOP/s (no measured FP64 peak available)"


# ------------------------------------------------------------------------------ reference arm
def run_reference(args, rank):
    """The reference's CPU path for this workload on all host cores.  lsqfit itself cannot be installed
    (gvar and GSL are absent, DESIGN.md section 1), so this times the oracle restatement of
    lsqfit.scipy_least_squares with the plugin's OWN defaults (x_scale = 1).  Nothing of the product is
    imported: no lsqfit_b200 package, no libb200lm.so, no CUDA."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    _oracle_init()
    configs, cfg, pdf = _G["configs"], _G["cfg"], _G["pdf"]
    per_step = max(cores * 25, 200)
    means = configs.bootstrap_means(cfg, per_step * (args.steps + args.warmup), cfg["seed"],
                                    cov=pdf.cov[:cfg["ny"], :cfg["ny"]])
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_oracle_init) as pool:
        k = 0
        for _ in range(args.warmup):
            pool.map(_oracle_fit, [(m, None) for m in means[k:k + per_step]])
            k += per_step
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_oracle_fit, [(m, None) for m in means[k:k + per_step]], chunksize=max(1, per_step // (cores * 8)))
            k += per_step
        dt = time.perf_counter() - t0
    v = per_step * args.steps / dt
    sample = ("%d fits per step (bounded sample of the 10k-copy batch), scipy least_squares(trf, x_scale=1: the plugin's "
              "default) oracle restatement of lsqfit.scipy_least_squares, whitening shared, %d processes on %s"
              % (per_step, cores, cpu_model()))
    line = dict(impl="reference", metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * dt / args.steps, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=WORKLOAD, fits_per_step=per_step),
                cpu_baseline=dict(value=v, unit=UNIT, cores=cores, kind="port", sample=sample),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                product_modules_loaded=sorted(m for m in sys.modules if m.split(".")[0] == "lsqfit_b200"))
    emit(json.dumps(line))


# ------------------------------------------------------------------------------ extras (not the headline)
def _timed(torch, fn, reps=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def extras_single_gpu(torch, lb, configs, dev, peak):
    """C1, C2, C5 and the saturated C3 batch on one GPU (BASELINE.json configs[0], [1], [4]); every entry
    is guarded so that a failure here can never cost the headline line."""
    ex = {}
    # ---- saturated C3 batch, one warp per fit (the kernel's throughput regime)
    try:
        cfg = configs.c3()
        ny, npar = cfg["ny"], cfg["np"]
        N = ny + npar
        full = np.zeros((N, N)); full[:ny, :ny] = cfg["ycov"]; full[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
        pdf = lb.PDF(np.concatenate([cfg["f"], cfg["prior_mean"]]), full, svdcut=cfg["svdcut"], device=dev.index)
        Bs = 160000
        md = torch.as_tensor(configs.bootstrap_means(cfg, Bs, cfg["seed"] + 7, cov=pdf.cov[:ny, :ny])).to(dev)
        p0 = torch.as_tensor(cfg["p0"]).to(dev)
        rows = {}
        for team in (1, 4, 32):
            plan = lb.Plan("multiexp", npar, ny, cfg["x"], pdf.i_invwgts, device=dev.index, team=team)
            out = plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], want_cov=True)
            ms, _ = _timed(torch, lambda: plan.fit_batch(md, p0, tol=cfg["tol"], maxit=cfg["maxit"], out=out), reps=2)
            nfev, njev, nfac = plan.last_stats()
            fl = njev * configs.eval_flops(ny, npar, cfg["K"])
            key = "wave_kernel" if team == 32 else "warps_per_fit_%d" % team
            rows[key] = dict(ms=ms, fits_per_s=Bs / ms * 1e3, tflops=fl / (ms * 1e-3) / 1e12,
                             frac=fl / (ms * 1e-3) / 1e12 / peak, kernel_used=plan.last_team())
            plan.close()
        ex["c3_saturated"] = dict(B=Bs, note="wave_kernel = lm_wave.cuh (b200lm_set_team(h, 32)): 32 fits per CTA in lock-step "
                                  "phases, one DMMA GEMM per chunk of 8 fits; its time includes the finalisation pass "
                                  "(covariances) of the one-warp kernel", **rows)
    except Exception as e:                                   # noqa: BLE001
        ex["c3_saturated"] = dict(error=repr(e))
    # ---- one fit with millions of uncorrelated points (examples/uncorrelated.py:30-41; BASELINE.md's first row):
    # the one-pass normal-equation kernel is HBM bound -- 24 B per row (x, y, 1/sigma) are read once
    try:
        from lsqfit_b200.dense import DenseFit
        hbm = None
        try:
            hbm = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
        except Exception:                                    # noqa: BLE001
            pass
        Nu = 2000000
        rng = np.random.default_rng(12)
        xu = np.linspace(0.2, 2.0, Nu)
        yu = 0.5 + 0.4 * np.exp(-0.7 * xu) + 1e-3 * rng.standard_normal(Nu)
        fit = None
        for _ in range(2):
            del fit
            fit = DenseFit((xu, yu, np.full(Nu, 1e-3)), (np.zeros(3), np.ones(3)), p0=[0.1, 0.1, 0.1], fcn="offset_exp",
                           tol=1e-10, device=dev.index)
        import ctypes as C
        from lsqfit_b200 import _cabi

        # SIX copies of the inputs (6 x 48 MB = 288 MB > the 126 MB L2), visited round-robin: every launch reads its
        # rows from HBM; time per launch = CUDA-event time of 30 back-to-back launches / 30
        NSET = 6
        hs, ys, ws = [], [], []
        for k in range(NSET):
            hk = _cabi.handle_t()
            _cabi.check(_cabi.lib.b200lm_create(fit.functor.family, fit.ny, fit.np, fit.functor.nx, 0, dev.index, C.byref(hk)))
            _cabi.check(_cabi.lib.b200lm_set_const(hk, fit.xrows.ctypes.data, fit.xrows.size), hk)
            hs.append(hk); ys.append(fit.d_y.clone()); ws.append(fit.wdiag.clone())
        outs = fit.nacc.clone()

        def nd_round(n=30):
            for i in range(n):
                k = i % NSET
                _cabi.check(_cabi.lib.b200lm_normal_diag(hs[k], fit.x.data_ptr(), ys[k].data_ptr(), ws[k].data_ptr(),
                                                         outs.data_ptr(), fit.la.stream()), hs[k])
        ts = []
        for _ in range(5):
            t1, _ = _timed(torch, nd_round, reps=1)
            ts.append(t1 / 30.0)
        ms_k = float(np.median(ts))
        for hk in hs:
            _cabi.lib.b200lm_destroy(hk)
        gbs = 24.0 * Nu / (ms_k * 1e-3) / 1e9
        ex["uncorrelated_2e6"] = dict(ny=Nu, np=3, fit_s=fit.times["fit"], nit=int(fit.nit), chi2_dof=float(fit.chi2 / fit.dof),
                                      fused_kernel=bool(fit.fused), normal_diag_ms=ms_k, algorithmic_bytes=24 * Nu,
                                      achieved_gbs=gbs, hbm_peak_gbs=hbm, frac=(gbs / hbm) if hbm else None,
                                      l2="six copies of the inputs (288 MB > L2) visited round-robin, 30 back-to-back launches per "
                                         "timing: every launch reads from HBM",
                                      note="reference: ~2 minutes for this fit (examples/uncorrelated.py:36).  ~50 FP64 "
                                           "instructions per 24-byte row put this kernel at the machine's ridge point "
                                           "(5.7 flop/B): neither the HBM nor the FP64 roofline can be approached alone "
                                           "(tools/micro/nd_bench.cu: 18.7 us with the rows in L2, 21.8 us from HBM)")
        del fit, ys, ws
    except Exception as e:                                   # noqa: BLE001
        ex["uncorrelated_2e6"] = dict(error=repr(e))
    # ---- C1: examples/simple.py, one fit: latency
    try:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "examples.json")))["examples"]["simple"]
        ny1 = len(g["ymean"]); yc = np.zeros((ny1, ny1)); i = 0
        for b in g["ycov_blocks"]:
            b = np.array(b); yc[i:i + len(b), i:i + len(b)] = b; i += len(b)
        f1 = lb.nonlinear_fit(data=(np.array(g["x"]), g["ymean"], yc), fcn="simple", prior=(g["prior_mean"], g["prior_sdev"]),
                              device=dev.index)
        plan1 = f1._spec.plan(dev.index)
        mean1 = np.concatenate([g["ymean"], g["prior_mean"]])
        md1, pd1 = torch.as_tensor(mean1).to(dev), torch.as_tensor(f1.p0).to(dev)
        t_dev, _ = _timed(torch, lambda: plan1.fit_batch(md1, pd1), reps=50)
        for _ in range(5):
            plan1.fit_batch_host(mean1[None, :], f1.p0)
        t0 = time.perf_counter()
        for _ in range(50):
            plan1.fit_batch_host(mean1[None, :], f1.p0)
        ex["c1_simple"] = dict(device_launch_us=1e3 * t_dev, host_call_us=1e6 * (time.perf_counter() - t0) / 50, nit=int(f1.nit),
                               chi2_dof=float(f1.chi2 / f1.dof), golden_chi2_dof="0.17 [5] (examples/simple.out:2)")
    except Exception as e:                                   # noqa: BLE001
        ex["c1_simple"] = dict(error=repr(e))
    # ---- C2: NIST StRD x 10^4 perturbed starts
    try:
        probs = json.load(open(os.path.join(ROOT, "tests", "golden", "nist.json")))["problems"]
        B2, rows, tot_fits, tot_ms = 10000, [], 0, 0.0
        for k, pr in enumerate(probs):
            x = np.array(pr["x"]); ny2, np2 = len(pr["y"]), len(pr["p0"])
            mean = np.concatenate([pr["y"], pr["prior_mean"]]); sd = np.concatenate([pr["ysdev"], pr["prior_sdev"]])
            plan = lb.Plan(pr["form"], np2, ny2, x, [(np.arange(ny2 + np2), 1.0 / sd)], device=dev.index)
            rng = np.random.default_rng(20240 + k)
            p0 = torch.as_tensor(np.array(pr["p0"])[None, :] * (1 + 0.1 * rng.uniform(-1, 1, size=(B2, np2)))).to(dev)
            md = torch.as_tensor(mean).to(dev)
            ms, out = _timed(torch, lambda: plan.fit_batch(md, p0, tol=1e-10, maxit=1000), reps=2)
            o = out.numpy()
            cert, csd = np.array(pr["certified"]), np.array(pr["certified_sdev"])
            good = (o["status"] > 0) & (np.max(np.abs(o["x"] - cert[None]) / csd[None], axis=1) < 1e-2)
            rows.append(dict(name=pr["name"], fits_per_s=B2 / ms * 1e3, converged=float((o["status"] > 0).mean()),
                             at_certified_minimum=float(good.mean()), mean_nit=float(o["nit"].mean())))
            tot_fits += B2; tot_ms += ms
            plan.close()
        ex["c2_nist_x10k"] = dict(problems=len(rows), fits_per_s_all=tot_fits / tot_ms * 1e3,
                                  fits_per_s_min=min(r["fits_per_s"] for r in rows), fits_per_s_max=max(r["fits_per_s"] for r in rows),
                                  at_certified_minimum_median=float(np.median([r["at_certified_minimum"] for r in rows])),
                                  per_problem=rows)
    except Exception as e:                                   # noqa: BLE001
        ex["c2_nist_x10k"] = dict(error=repr(e))
    # ---- C5: one large dense fit (5000 correlated points, 2000 parameters, svdcut)
    try:
        from lsqfit_b200.dense import DenseFit
        cfg5 = configs.c5()
        fit = None
        for _ in range(2):                                   # second pass = warm
            del fit
            fit = DenseFit((cfg5["t"], cfg5["ymean"], cfg5["ycov"]), (cfg5["prior_mean"], cfg5["prior_sdev"]),
                           svdcut=cfg5["svdcut"], tol=cfg5["tol"], maxit=cfg5["maxit"], device=dev.index)
        fit.propagate()
        ms_prop, _ = _timed(torch, fit.propagate, reps=2)
        ex["c5_dense"] = dict(ny=cfg5["ny"], np=cfg5["np"], svdn=int(fit.svdn), nit=int(fit.nit), whiten_s=fit.times["whiten"],
                              fit_s=fit.times["fit"], per_iteration_ms=1e3 * fit.times["fit"] / max(1, fit.nit),
                              propagate_ms=ms_prop, chi2_dof=float(fit.chi2 / fit.dof),
                              stopping_criterion=int(fit.stopping_criterion))
        del fit
    except Exception as e:                                   # noqa: BLE001
        ex["c5_dense"] = dict(error=repr(e))
    return ex


def c4_strong(torch, dist, lb, configs, lbdist, dev, rank, world, B=1000000, comm=None):
    """BASELINE config 4: 10^6 simulated fits of a 3-exp correlator SHARDED over the ranks (strong scaling):
    every rank generates its shard of the Philox stream on its own GPU, fits it, then one all-gather of the
    packed results and one all-reduce of the moments.  Timed on the device, max over ranks."""
    from lsqfit_b200 import bootstrap as bs
    cfg = configs.c4(B=B)
    ny, npar = cfg["ny"], cfg["np"]
    N = ny + npar
    full = np.zeros((N, N)); full[:ny, :ny] = cfg["ycov"]; full[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
    mean0 = np.concatenate([cfg["f"], cfg["prior_mean"]])
    pdf = lb.PDF(mean0, full, svdcut=cfg["svdcut"], device=dev.index)
    val, vec = np.linalg.eigh(pdf.cov)
    L = vec * np.sqrt(np.clip(val, 0, None)); L[ny:, :] = 0.0      # simulated fits: prior means fixed
    Ld, m0d, p0d = torch.as_tensor(L).to(dev), torch.as_tensor(mean0).to(dev), torch.as_tensor(cfg["p0"]).to(dev)
    # BENCH kernel choice for this job: the wave kernel (lm_wave.cuh) -- a million fits saturate every kernel, which is
    # its regime (measured on this shape: 21.3 M vs 18.4 M fits/s for one warp per fit; same parity bars,
    # tests/test_gpu_configs.py); B200LM_C4_TEAM overrides (0 = the default kernel of the shape)
    c4_team = int(os.environ.get("B200LM_C4_TEAM", "32"))
    plan = lb.Plan("multiexp", npar, ny, cfg["x"], pdf.i_invwgts, device=dev.index, team=c4_team or None)
    lo, hi = lbdist.shard_range(B, rank, world)

    def job():
        means = bs.bootstrap_means(m0d, Ld, hi - lo, cfg["seed"], first=lo, device=dev.index)
        out = plan.fit_batch(means, p0d, tol=cfg["tol"], maxit=cfg["maxit"], want_cov=False)
        packed = lbdist.pack_results(out.x, out.chi2, out.nit, out.status)
        allp = lbdist.gather_results(packed, B_total=B, comm=comm)
        m, c, n = lbdist.moments(out.x, out.status > 0, comm=comm)
        return allp, m, c, n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    job(); barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        allp, m, c, n = job()
    e1.record(); barrier()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    nfev = plan.last_stats()[0]
    tt = torch.tensor([float(nfev)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt)
    kernel_used = plan.last_team()
    plan.close()
    ms = float(t[0])
    bias = float(torch.max(torch.abs(m - p0d) / torch.sqrt(torch.diagonal(c)) * (n ** 0.5)))
    return dict(workload="C4: 3-exp correlator, 10^6 simulated fits sharded over the ranks (generate + fit + gather + moments)",
                B=B, n_gpus=world, ms=ms, fits_per_s=B / ms * 1e3, scaling="strong", converged=int(n),
                gathered_rows=int(allp.shape[0]), nfev_per_fit=float(tt[0]) / B, kernel_used=kernel_used,
                pmean_minus_pexact_in_sigma_of_mean=bias,
                note="the mean of the best-fit parameters is BIASED with respect to pexact at second order in the noise "
                     "(nonlinear model, prior pull); tests/test_gpu_parity.py::test_c4_bias_matches_oracle shows the CPU "
                     "oracle has the same bias on the same copies")


# ------------------------------------------------------------------------------ our arm
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import lsqfit_b200 as lb
    from lsqfit_b200 import configs, dist as lbdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")

    # CPU baseline first (rank 0, N=1 only), before CUDA is initialised in this process, so that
    # the worker processes are forked from a CUDA-free parent.
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        _oracle_init()
        ocfg, opdf = _G["cfg"], _G["pdf"]
        n = min(args.cpu_sample, args.batch)
        om = configs.bootstrap_means(ocfg, args.batch, ocfg["seed"], cov=opdf.cov[:ocfg["ny"], :ocfg["ny"]])[:n]
        v, mean_nit = cpu_fits_per_sec(om, cores, "jac")
        v1, mean_nit1 = cpu_fits_per_sec(om[:max(cores * 25, 200)], cores, None)
        cpu = dict(value=v, unit=UNIT, cores=cores, kind="port",
                   sample="first %d of the %d bootstrap copies of this workload; oracle = scipy least_squares(trf) "
                          "restatement of lsqfit.scipy_least_squares (numpy AD Jacobian, whitening shared) with the SAME "
                          "scaling policy as the device (More' / x_scale='jac'), %d processes, mean nfev %.1f, %s"
                          % (n, args.batch, cores, mean_nit, cpu_model()),
                   plugin_default_x_scale_1=dict(value=v1, mean_nfev=mean_nit1,
                                                 note="the reference plugin's own default scaling (what --impl reference times)"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = configs.c3(B=args.batch)
    ny, npar, B = cfg["ny"], cfg["np"], args.batch
    N = ny + npar
    full = np.zeros((N, N))
    full[:ny, :ny] = cfg["ycov"]
    full[ny:, ny:] = np.diag(cfg["prior_sdev"] ** 2)
    mean0 = np.concatenate([cfg["f"], cfg["prior_mean"]])
    pdf = lb.PDF(mean0, full, svdcut=cfg["svdcut"], device=local_rank)          # device whitening
    # Weak scaling: every rank fits its OWN batch (seed + rank).  B200LM_BENCH_SAME=1 gives every rank the same
    # batch instead (isolates the engine's scaling from the workload's straggler statistics).
    same = os.environ.get("B200LM_BENCH_SAME", "0") == "1"
    means_h = configs.bootstrap_means(cfg, B, cfg["seed"] + (0 if same else rank), cov=pdf.cov[:ny, :ny])
    plan = lb.Plan("multiexp", npar, ny, cfg["x"], pdf.i_invwgts, device=local_rank)
    means_d = torch.as_tensor(means_h).to(dev)
    p0_d = torch.as_tensor(cfg["p0"]).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)   # 256 MiB > 126 MB L2

    out = plan.fit_batch(means_d, p0_d, tol=cfg["tol"], maxit=cfg["maxit"])          # allocates outputs
    # data-path collectives through the library's own C ABI (b200lm_gather / b200lm_allreduce_sum, csrc/comm.cu);
    # torch.distributed only ships the NCCL id and runs the timing barriers
    nccl_comm, nccl_comm_note = None, None
    if world > 1:
        try:
            nccl_comm = lbdist.Comm(local_rank)
            nccl_comm_note = "b200lm_gather / b200lm_allreduce_sum (NCCL behind the C ABI)"
        except Exception as e:                               # noqa: BLE001
            nccl_comm_note = "torch.distributed (C-ABI communicator unavailable: %r)" % (e,)

    def step():
        plan.fit_batch(means_d, p0_d, tol=cfg["tol"], maxit=cfg["maxit"], out=out)
        if world > 1:
            packed = lbdist.pack_results(out.x, out.chi2, out.nit, out.status)
            return lbdist.gather_results(packed, comm=nccl_comm)
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        step()
    barrier()
    launches0 = plan.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    gathered = None
    for k in range(args.steps):
        flush.zero_()                       # L2 flush between timed iterations (not timed)
        ev[k][0].record()
        kev[k][0].record()
        plan.fit_batch(means_d, p0_d, tol=cfg["tol"], maxit=cfg["maxit"], out=out)
        kev[k][1].record()
        if world > 1:
            packed = lbdist.pack_results(out.x, out.chi2, out.nit, out.status)
            gathered = lbdist.gather_results(packed, comm=nccl_comm)
        ev[k][1].record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = plan.launch_count() - launches0
    t_ms = sum(a.elapsed_time(b) for a, b in ev)
    tk_ms = sum(a.elapsed_time(b) for a, b in kev)
    nfev, njev, nfac = plan.last_stats()
    tt = torch.tensor([t_ms, tk_ms], device=dev, dtype=torch.float64)
    ts = torch.tensor([float(nfev), float(njev), float(nfac), float(out.nit.max())], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        tsum = ts.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        nfev_all, njev_all, nfac_all = float(tsum[0]), float(tsum[1]), float(tsum[2])
    else:
        nfev_all, njev_all, nfac_all = float(nfev), float(njev), float(nfac)
    t_ms, tk_ms = float(tt[0]), float(tt[1])
    max_nit = int(ts[3])
    res = out.numpy()
    if args.dump_outputs and rank == 0:
        # what the last timed step returned, before the e2e and queued runs below reuse `out`
        dump_outputs(args.dump_outputs, dict(res, gathered=gathered.cpu().numpy()) if world > 1 else res)
    conv = float((res["status"] > 0).mean())
    warps_per_fit = plan.last_team()

    # ---- e2e: the public host-buffer call, pinned inputs, H2D + D2H inside the timed region
    means_pin = torch.as_tensor(means_h).pin_memory()
    outs = dict(x=torch.empty((B, npar), dtype=torch.float64).pin_memory().numpy(),
                chi2=torch.empty(B, dtype=torch.float64).pin_memory().numpy(),
                cov=torch.empty((B, npar, npar), dtype=torch.float64).pin_memory().numpy(),
                logdet=torch.empty(B, dtype=torch.float64).pin_memory().numpy(),
                nit=torch.empty(B, dtype=torch.int32).pin_memory().numpy(),
                status=torch.empty(B, dtype=torch.int32).pin_memory().numpy(), f=None, J=None)
    mp_np = means_pin.numpy()
    for _ in range(3):
        plan.fit_batch_host(mp_np, cfg["p0"], tol=cfg["tol"], maxit=cfg["maxit"], out=outs)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        plan.fit_batch_host(mp_np, cfg["p0"], tol=cfg["tol"], maxit=cfg["maxit"], out=outs)
    torch.cuda.synchronize()
    te = time.perf_counter() - t0
    te_t = torch.tensor([te], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te_t, op=dist.ReduceOp.MAX)
    te = float(te_t[0])
    h2d = B * N * 8 + npar * 8
    d2h = B * (npar + 2 + npar * npar) * 8 + B * 8

    # ---- extra (not the headline): the same steps QUEUED on two streams / two plans, so that the next
    # batch fills the SMs that idle during the long-fit tail of the previous one
    plan_b = lb.Plan("multiexp", npar, ny, cfg["x"], pdf.i_invwgts, device=local_rank)
    means_b = torch.as_tensor(configs.bootstrap_means(cfg, B, cfg["seed"] + 1000 + rank, cov=pdf.cov[:ny, :ny])).to(dev)
    out_b = plan_b.fit_batch(means_b, p0_d, tol=cfg["tol"], maxit=cfg["maxit"])
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    jobs = [(plan, means_d, out), (plan_b, means_b, out_b)]
    torch.cuda.synchronize()
    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    flush.zero_()
    torch.cuda.synchronize()
    q0.record()
    for k in range(args.steps):
        pl, mm, oo = jobs[k & 1]
        with torch.cuda.stream(streams[k & 1]):
            if k == 0 or k == 1:
                streams[k & 1].wait_event(q0)
            pl.fit_batch(mm, p0_d, tol=cfg["tol"], maxit=cfg["maxit"], out=oo)
    for st in streams:
        torch.cuda.current_stream(dev).wait_stream(st)
    q1.record()
    torch.cuda.synchronize()
    tq_ms = q0.elapsed_time(q1)
    plan_b.close()

    peak, peak_src = fp64_peak()
    extras = {}
    if not args.no_extras:
        try:
            extras["c4_strong"] = c4_strong(torch, dist, lb, configs, lbdist, dev, rank, world, comm=nccl_comm)
        except Exception as e:                               # noqa: BLE001
            extras["c4_strong"] = dict(error=repr(e))
        if world == 1:
            extras.update(extras_single_gpu(torch, lb, configs, dev, peak))

    comm = None
    if world > 1:
        comm = dict(backend=dist.get_backend(), nranks=dist.get_world_size(),
                    nccl_version=".".join(str(v) for v in torch.cuda.nccl.version()),
                    nccl_debug=os.environ.get("NCCL_DEBUG"), log="stderr (NCCL_DEBUG_FILE=/dev/stderr)",
                    collectives_per_step="1 all-gather of [B, np+3] fp64 rows; no host synchronisation",
                    data_path=nccl_comm_note)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the fit kernel is the only kernel of a step)
    F_eval = configs.eval_flops(ny, npar, cfg["K"])
    F_res = 2.0 * ny * ny + 2.0 * N + ny * cfg["K"] * 3.0       # residual-only trial evaluation
    flops_launch = (njev_all * F_eval + (nfev_all - njev_all) * F_res) / world     # per launch (per rank)
    achieved = flops_launch / (tk_ms / args.steps * 1e-3) / 1e12
    traffic, traffic_src = _ncu_traffic()
    kname = "fit_team_kernel<MultiExp<8>, %d>" % warps_per_fit if warps_per_fit > 1 else "fit_kernel<MultiExp<8>>"
    roofline = dict(bound="tensor", achieved=achieved, peak=peak, unit="TFLOP/s", frac=achieved / peak,
                    traffic=traffic, traffic_source=traffic_src, kernel=kname, warps_per_fit=warps_per_fit,
                    peak_source=peak_src, flops_per_launch=flops_launch,
                    flops_per_launch_survey_formula=nfev_all * F_eval / world,
                    nfev_per_fit=nfev_all / (B * world), njev_per_fit=njev_all / (B * world),
                    chol_per_fit=nfac_all / (B * world), max_nfev_of_a_fit=max_nit, kernel_ms=tk_ms / args.steps,
                    queue_order=int(plan.last_order()),
                    queue_order_note="1: the work queue hands out the fits with the largest start-point chi2 first "
                                     "(b200lm_set_order default policy for this shape); kernel_ms then spans the "
                                     "start-point pass (one evaluation per fit, NOT counted in the flops), the ranking "
                                     "kernel and the fit kernel",
                    note="FP64 pipe (DMMA/DFMA share one pipe; tcgen05 has no FP64 kind).  The step is bounded by the "
                         "latency of its slowest fits, not by throughput: see extras.c3_saturated for the saturated batch")

    queued = dict(value=B * args.steps / (tq_ms * 1e-3), unit=UNIT + " per GPU", streams=2, ms_per_step=tq_ms / args.steps,
                  note="same steps queued on two streams (two plans): throughput of a stream of 10k-fit batches; "
                       "not the headline, which times one batch at a time")
    line = dict(metric=METRIC, value=world * B * args.steps / (t_ms * 1e-3), unit=UNIT, n_gpus=world,
                steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=t_ms / args.steps,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=WORKLOAD, fits_per_gpu_per_step=B, ny=ny, np=npar, svdcut=cfg["svdcut"],
                            tol=list(cfg["tol"]), maxit=cfg["maxit"], l2="flushed between timed steps (256 MiB memset)",
                            per_rank_data="identical batch on every rank (B200LM_BENCH_SAME=1)" if same
                            else "a different batch on every rank (seed + rank)",
                            converged_frac=conv, svdn=int(pdf.nmod)),
                clocks=clocks,
                e2e=dict(value=world * B * args.steps / te, unit=UNIT, h2d_bytes_per_step=h2d,
                         d2h_bytes_per_step=d2h, ms_per_step=1e3 * te / args.steps,
                         api="lsqfit_b200.Plan.fit_batch_host -> b200lm_fit_batch_host (pinned host buffers)",
                         d2h_route="covariances: stored by the kernels straight into the pinned host buffer over PCIe "
                                   "(B200LM_NO_ZEROCOPY=1: device copy + D2H transfer); x, chi2, log det, nit, status: "
                                   "D2H copies after the launch"),
                gpu_launches=int(launches), roofline=roofline, cpu_baseline=cpu, queued=queued, comm=comm, extras=extras)
    emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
