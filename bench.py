#!/usr/bin/env python
"""bench.py -- continuation steps/sec on 2-D Swift-Hohenberg (SH2d-fronts 1024^2, fp64) + achieved HBM GB/s of the
fused JVP+Arnoldi kernel, per BASELINE.json.

Workload (BASELINE.json configs[2]: "SH2d-fronts 1024^2, PALC branch of 200 steps sharded 8xB200"): the localized-front branch
of examples/SH2d-fronts.jl from its start point over a fixed WINDOW of PALC arclength S = K * B * dsmax -- the same window for
every number of GPUs (strong scaling).  A bench "step" = one BATCH of B = 10 continuation steps at dsmax (the unit after
which the (lambda, ||u||) rows are exchanged, north_star); `value` = K * B / t in continuation steps per second, where a
continuation step = secant predictor + Newton-Krylov corrector (per Newton iteration 2 residuals and one MatrixFreeBLS solve =
one GMRES(100) with the DCT preconditioner on the right, fused JVP+Arnoldi kernels).  K = 20, B = 10 -> the 200-step branch.

N = 1: plain continuation over the window (exactly K * B steps).  N > 1 ("replicas only", SURVEY.md 8(e) / tier rule 5): PALC is a
sequential recurrence, so one branch does not shard; every rank runs an independent replica of the same job (replicated state,
nothing crosses NVLink), the rows (lambda, ||u||, itnewton, itlinear) are all_gathered per job -- and must agree bit for bit
across the GPUs, which the JSON reports -- `value` = N * K * B / max-over-ranks time, "scaling": "weak".  (A family of branches
nu_r = nu (1 + 0.002 r) was tried first: at nu_1 the same start-up already lands on a different, 30x cheaper branch, so the
ranks would not do comparable work.)
The alternative `--partition scout` cuts ONE branch window into chunks seeded by a cheap scout inside the timed region
(segments.py); measured on this branch it does not work -- a scout loose enough to be cheap leaves the snaking branch
(profiles/r02_scout_probe.txt, DESIGN.md section 6) -- so it is kept as an option, not the default.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--grid 1024] [--batch 10] [--impl reference] [--dump-outputs DIR]

Besides `e2e` (the plugin surfaces with host vectors) the line carries `e2e_native`: the same window through ONE C-ABI call from and
to host buffers (bk_palc_run, the PALC loop as host C++ inside the library), with a check that its rows equal the device-resident
run's bit for bit.

--impl reference : times the CPU restatement of the reference path -- oracle/c, C++17/OpenMP on all host cores (CSR SpMV with the
kron-assembled L1, MGS GMRES, DCT preconditioner; SURVEY.md 8(d)); Julia is absent from this image, see DESIGN.md -- on a
bounded sample of the same window.
"""
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

LX0, LY0 = 8 * np.pi, 4 * np.pi / np.sqrt(3)  # examples/SH2d-fronts.jl:10-11 (151 x 100 grid)


def domain(n):
    """The domain grows with the grid so that the mesh width stays that of the reference's own GPU example
    (examples/SH2d-fronts-cuda.jl:66-69: Nx = Ny = 512 on lx = 16 pi, ly = 2*2pi/sqrt(3)*2, i.e. the example's
    lengths x2): lengths = example lengths x n/256.  On the ORIGINAL lengths a 1024^2 grid has hy = 0.014 and the
    rounding floor of evaluating (I+Lap)^2 u in fp64 (~ eps/hy^4 ~ 4e-8, measured) sits ABOVE the example's Newton
    tolerances (1e-8 / 1e-9), for the reference's sparse-matrix path just as for the stencil."""
    s = max(1.0, n / 256.0)
    return LX0 * s, LY0 * s


PAR = (-0.1, 1.3)                            # (l, nu) examples/SH2d-fronts.jl:55
CONT = dict(dsmin=1e-4, dsmax=5e-3, ds=-1e-3, p_min=-1.0, p_max=0.0)  # examples/SH2d-fronts.jl:86
GMRES = dict(reltol=1e-5, restart=100, maxiter=100)  # examples/SH2d-fronts.jl:122 (reltol), config "GMRES(100)"
BRANCH = {"kind": "front"}  # "front": localized front of SH2d-fronts.jl:70-80; "hexagons": the example's own continuation (:88-92)
BLS = {"kind": "matrixfree"}  # MatrixFreeBLS (1 GMRES on the N+1 bordered system) or "bordering" (BorderingBLS: 2 GMRES + BEC)


def sol0(n):
    LX, LY = domain(n)
    X = -LX + 2 * LX / n * np.arange(n)
    Y = -LY + 2 * LY / n * np.arange(n)
    s = np.cos(X)[None, :] + np.cos(X / 2)[None, :] * np.cos(np.sqrt(3.0) * Y / 2)[:, None]
    s = s - s.min()
    s = s / s.max()
    return ((s - 0.25) * 1.7).reshape(-1)


def front_guess(u_hexa, n):
    LX, LY = domain(n)
    X = -LX + 2 * LX / n * np.arange(n)
    return 0.4 * u_hexa * np.tile(np.exp(-((X + LX) ** 2) / 25.0), n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            self.proc.wait()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of k2_fused<8,1> from the committed `ncu --set full` capture of
    the shipped kernel (profiles/r02_ncu_k2_fused.csv, falling back to the round-1 capture of k2_fused<7,1>)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_k2_fused.csv")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r01c_ncu_k2_fused.csv")
    try:
        import csv
        rows = list(csv.reader(open(p)))
        h = rows[0]
        vals = [float(r[h.index("dram__bytes_read.sum")]) + float(r[h.index("dram__bytes_write.sum")]) for r in rows[2:]]
        out = {"bytes_per_launch": 1e6 * sum(vals) / len(vals), "source": os.path.relpath(p, ROOT) + " (k2_fused, one ncu --set full capture)"}
        if p.endswith("r02_ncu_k2_fused.csv"):
            # the capture sits at Krylov index j = 14 of a 1024^2 solve: algorithmic 8N(j+2) + 16N = 151 MB; moved in addition: the
            # right-preconditioned input z (its own vector, +8N) and the stencil halo rows ((E+4)/E on z)
            out.update(j_at_capture=14, algorithmic_bytes_at_capture=8 * 1024 * 1024 * (14 + 2) + 16 * 1024 * 1024)
        return out
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------- GPU arm
def gpu_setup(bk, n, device, host_state=False):
    P = bk.palc
    ctx = bk.Context(bk.BK_SH2D, (n, n), domain(n), krylov_m=GMRES["restart"], device=device, params=PAR)
    ctx.precond_setup(bk.BK_PC_SH_DCT, 1.0)  # (L1 + I)^-1, examples/SH2d-fronts.jl:121
    ls = bk.GMRESB200(N=n * n, Pr=True, **GMRES)
    wrap = (lambda a: np.array(a)) if host_state else ctx.to_device
    opt = P.NewtonPar(tol=1e-8, max_iterations=20, linsolver=ls)  # examples/SH2d-fronts.jl:57
    prob = P.BifurcationProblemB200(ctx, wrap(sol0(n)), PAR, lens=0)
    hexa = P.newton(prob, prob.u0, PAR[0], opt, P.norminf)
    assert hexa.converged, hexa.residuals
    if BRANCH["kind"] == "hexagons":
        # the branch the example itself continues: continuation(prob, PALC(), optcont) with prob.u0 = vec(sol0)
        # (examples/SH2d-fronts.jl:88-92; the line that would substitute the deflated front is commented out, :87)
        pol = P.newton(prob, hexa.u, PAR[0], P.NewtonPar(tol=1e-9, max_iterations=30, linsolver=ls), P.norminf)
        assert pol.converged, pol.residuals
        return ctx, ls, pol.u
    uh = hexa.u if host_state else hexa.u.numpy()
    prob = P.BifurcationProblemB200(ctx, wrap(front_guess(uh, n)), PAR, lens=0)
    fr = P.newton(prob, prob.u0, PAR[0], P.NewtonPar(tol=1e-9, max_iterations=30, linsolver=ls), P.norminf)
    assert fr.converged, fr.residuals
    return ctx, ls, fr.u


def gpu_run(bk, ctx, ls, u_start, p_start, steps, warmup, torch, timing=True, u1=None, p1=None, flush=None):
    """Runs warmup+steps PALC steps; returns (rows, per-step ms list (CUDA events on the library's stream), stats delta)."""
    P = bk.palc
    cp = P.ContinuationPar(max_steps=warmup + steps, newton_options=P.NewtonPar(tol=1e-9, max_iterations=15, linsolver=ls),
                           **CONT)
    alg = P.PALC(bls=bk.MatrixFreeBLSB200(ls) if BLS["kind"] == "matrixfree" else bk.BorderingBLSB200(ls, check_precision=False))
    pars = list(PAR)
    pars[0] = p_start
    prob = P.BifurcationProblemB200(ctx, u_start, pars, lens=0)
    stream = torch.cuda.ExternalStream(ctx.lib.bk_stream(ctx.handle))
    starts, ends = [], []
    state = {"n": 0, "s0": None}

    def cb(st):
        # called at step 0 and after each accepted step: close the running step's event pair, flush L2, open the next
        k = state["n"]
        if k > 0:
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            ends.append(e)
        if k == warmup:
            ctx.sync()
            ctx.set_timing(timing)
            state["s0"] = ctx.stats()
            torch.cuda.profiler.start()  # cudaProfilerStart: lets `ncu --profile-from-start off` see only the timed region
        if flush is not None:
            with torch.cuda.stream(stream):
                flush.zero_()
        e2 = torch.cuda.Event(enable_timing=True)
        e2.record(stream)
        starts.append(e2)
        state["n"] += 1
        return True

    rows, st = P.continuation(prob, alg, cp, normC=P.norminf, u1=u1, p1=p1, callback=cb)
    ctx.sync()
    torch.cuda.profiler.stop()
    ctx.set_timing(False)
    s1 = ctx.stats()
    ms = [starts[i].elapsed_time(ends[i]) for i in range(len(ends))]
    delta = {k: s1[k] - state["s0"][k] for k in s1} if state["s0"] else {}
    return rows, ms[warmup:], delta, st


def best_blas_threads(n, cores):
    """BLAS-1 on 8 MB vectors does not scale to every core of a big host (thread wake-up dominates): calibrate the thread
    count that makes the oracle's inner loop (dot + axpy) fastest and use it -- 'all the host threads it can use'."""
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return cores, None
    x, y = np.random.default_rng(0).standard_normal(n), np.random.default_rng(1).standard_normal(n)
    best, best_t = cores, None
    for t in sorted({1, 2, 4, 8, 16, 32, 64, cores}):
        if t > cores:
            continue
        with threadpool_limits(limits=t, user_api="blas"):
            np.dot(x, y)
            t0 = time.perf_counter()
            for _ in range(40):
                h = np.dot(x, y)
                y -= 1e-9 * h * x
            dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = t, dt
    return best, threadpool_limits


def bordered_precond(P, N):
    """P on the first N entries, identity on the border component (vectors of the MatrixFreeBLS system have N+1 entries)."""
    return lambda r: P(r) if len(r) == N else np.concatenate([P(r[:N]), r[N:]])


def cpu_steps(n, u_start, p_start, nsteps, workers):
    """CPU restatement (oracle/) of the same PALC steps; returns (rows, seconds)."""
    from oracle import problems, krylov, bls as obls, palc as opalc, precond as oprecond
    nthr, limiter = best_blas_threads(n * n, workers)
    if limiter is not None:
        limiter(limits=nthr, user_api="blas")  # stays in force for the rest of the process
    cpu_steps.blas_threads = nthr
    sh = problems.SwiftHohenberg((n, n), domain(n), l=PAR[0], nu=PAR[1])
    Pinv = bordered_precond(oprecond.dct_precond((n, n), domain(n), 1.0, workers=workers), n * n)
    ols = krylov.GMRESIterativeSolvers(N=n * n, Pr=Pinv, **GMRES)
    prob = opalc.Problem(F=lambda u, l: sh.F(u, l), J=lambda u, l: (lambda v: sh.dF(u, v, l)), u0=u_start, p0=p_start)
    cp = opalc.ContinuationPar(max_steps=nsteps, newton_options=opalc.NewtonPar(tol=1e-9, max_iterations=15, linsolver=ols), **CONT)
    tmark = {}

    def cb(st):
        tmark.setdefault("t", []).append(time.perf_counter())
        return True

    t0 = time.perf_counter()
    obl = obls.MatrixFreeBLS(ols) if BLS["kind"] == "matrixfree" else obls.BorderingBLS(ols, check_precision=False)
    rows, st = opalc.continuation(prob, opalc.PALC(bls=obl), cp, normC=opalc.norminf, callback=cb)
    t1 = time.perf_counter()
    # the first callback fires at step 0, i.e. after the two start-up Newton solves, which the metric excludes
    # (src/Continuation.jl:370-393): steps/sec is counted over the continuation! loop only
    ts = tmark.get("t", [])
    if len(ts) >= 2:
        return rows, (ts[-1] - ts[0]), len(ts) - 1
    return rows, (t1 - t0), 1


class StepTimer:
    """CUDA-event timing of continuation steps on the library's stream.  `wrap(cb)` returns a continuation callback that
    closes the running step's event pair, flushes L2 (outside the pair) and opens the next pair, then calls `cb`."""

    def __init__(self, ctx, torch, flush):
        self.ctx, self.torch, self.flush = ctx, torch, flush
        self.stream = torch.cuda.ExternalStream(ctx.lib.bk_stream(ctx.handle))
        self.pairs, self.open = [], None

    def _event(self):
        e = self.torch.cuda.Event(enable_timing=True)
        e.record(self.stream)
        return e

    def start(self):
        """opens a pair now (used to time work that precedes a continuation loop's step 0: the start-up Newton solves of the scout)"""
        if self.flush is not None:
            with self.torch.cuda.stream(self.stream):
                self.flush.zero_()
        self.open = self._event()

    def stop(self):
        if self.open is not None:
            self.pairs.append((self.open, self._event()))
            self.open = None

    def wrap(self, cb):
        def f(st):
            self.stop()
            keep = cb(st) if cb is not None else True
            if keep is not False:  # a callback that ends the loop leaves no step to time
                self.start()
            return keep
        return f

    def total_ms(self):
        self.stop()
        self.ctx.sync()
        return float(sum(a.elapsed_time(b) for a, b in self.pairs))

    def step_ms(self):
        """device time of every closed pair, in order (call after total_ms): pair k = continuation step k + 1 with the rejected
        attempts before it"""
        return [float(a.elapsed_time(b)) for a, b in self.pairs]


def make_algs(bk, ctx, ls, n):
    """(fine alg, fine ContinuationPar factory, scout alg, scout ContinuationPar)"""
    P = bk.palc
    mkbls = lambda l: bk.MatrixFreeBLSB200(l) if BLS["kind"] == "matrixfree" else bk.BorderingBLSB200(l, check_precision=False)
    alg = P.PALC(bls=mkbls(ls))
    cp = lambda ds=None: P.ContinuationPar(max_steps=10**6, newton_options=P.NewtonPar(tol=1e-9, max_iterations=15, linsolver=ls),
                                          **dict(CONT, ds=CONT["ds"] if ds is None else ds))
    ls_s = bk.GMRESB200(N=n * n, Pr=True, **dict(GMRES, reltol=SCOUT["gmres_reltol"]))
    cps = P.ContinuationPar(max_steps=10**6, newton_options=P.NewtonPar(tol=SCOUT["newton_tol"], max_iterations=SCOUT["newton_maxit"], linsolver=ls_s),
                            **dict(CONT, dsmax=SCOUT["ds_factor"] * CONT["dsmax"], ds=SCOUT["ds_factor"] * CONT["ds"]))
    return alg, cp, P.PALC(bls=mkbls(ls_s)), cps


TIMING_EVERY = 8  # roofline sampling: the event records sit between PDL launches, so timing every solve would slow the step it measures


SCOUT = dict(ds_factor=4.0, newton_tol=1e-4, newton_maxit=8, gmres_reltol=1e-2)  # seed generator of the N > 1 partition (tools/scout_probe.py)


def window_job(bk, ctx, ls, n, u_start, s_total, rank, world, torch, flush, timing=True, wrap=None, nsteps=None, spec=None):
    """One rank's job.  world == 1 (also every rank of the default "replicas" mode): exactly `nsteps` continuation steps from
    u_start; world > 1: this rank's chunk of the arclength window s_total (--partition scout).  Returns (rows, ms, stats delta, info)."""
    P, S = bk.palc, bk.segments
    wrap = wrap or (lambda v: v)
    alg, cpf, alg_s, cps = make_algs(bk, ctx, ls, n)
    mkprob = lambda u, p: P.BifurcationProblemB200(ctx, u, [p] + list(PAR[1:]), lens=0)
    tm = StepTimer(ctx, torch, flush)
    ctx.sync()
    ctx.set_timing(TIMING_EVERY if timing else 0)  # CUDA-event pairs around the fused kernels of every TIMING_EVERY-th solve
    s0 = ctx.stats()
    torch.cuda.profiler.start()
    info = {"scout_ms": 0.0, "scout_points": 0, "chunk": None, "rejected": 0, "work_newton": 0, "work_linear": 0}
    # the loop's own bound (step <= max_steps) corrects one step past max_steps and discards it: stop at step `nsteps` instead,
    # so that the timed window holds exactly the steps the value counts
    last_step = lambda st: st.step < nsteps
    if spec is not None:
        # --partition speculative: ONE branch on all ranks, rank r correcting with the r-times-halved step (segments.continuation_speculative);
        # spec = (dist, device).  Rows equal the 1-GPU rows; the collectives are an all_gather of 4 doubles and a broadcast of the accepted
        # point per step, both inside the timed region.
        cp1 = cpf()
        cp1.max_steps = nsteps
        rows, st, sinfo = S.continuation_speculative(P, mkprob(u_start, PAR[0]), alg, cp1, P.norminf, spec[0], torch, spec[1], callback=tm.wrap(last_step))
        rows = rows[: nsteps + 1]
        info["speculative"] = sinfo
    elif world == 1:
        cp1 = cpf()
        cp1.max_steps = nsteps
        rows, st = P.continuation(mkprob(u_start, PAR[0]), alg, cp1, normC=P.norminf, callback=tm.wrap(last_step))
        rows = rows[: nsteps + 1]
    else:
        tm.start()  # the scout's two start-up Newton solves are part of the job
        sc = S.run_scout(P, mkprob(u_start, PAR[0]), alg_s, cps, P.norminf, s_total, lambda v: wrap(v.copy() if hasattr(v, "copy") else v),
                         margin=2.0 * SCOUT["ds_factor"] * CONT["dsmax"], wrap_callback=tm.wrap)
        info["scout_ms"] = tm.total_ms()
        tm.start()  # partition + the chunk's start-up belong to the job as well
        info["scout_points"] = len(sc.points)
        b = S.partition_by_cost(sc.cost, world)
        if rank < len(b) - 1:
            info["chunk"] = [float(sc.sigma[b[rank]]), float(sc.sigma[b[rank + 1]])]
            rows, st, trk = S.run_chunk(P, mkprob, alg, cpf(np.sign(CONT["ds"]) * CONT["dsmax"]), P.norminf, sc, b[rank], b[rank + 1], s_total,
                                        rank, rank == len(b) - 2, wrap_callback=tm.wrap)
        else:
            rows, st = [], None
    ms = tm.total_ms()
    ctx.sync()
    try:
        info["step_ms"] = tm.step_ms() if world == 1 else None
    except Exception:  # informational only: never let it touch the measurement
        info["step_ms"] = None
    torch.cuda.profiler.stop()
    ctx.set_timing(False)
    s1 = ctx.stats()
    if st is not None:
        info.update(rejected=int(st.nfail), work_newton=int(st.work_newton), work_linear=int(st.work_linear))
    info["state"] = st
    return rows, ms, {k: s1[k] - s0[k] for k in s1}, info


def config_dict(n, workload, K, B):
    """Identical in both arms (driver: same_config); everything run-specific goes under "details"."""
    return {"workload": workload, "grid": [n, n],
            "window": f"localized-front branch of examples/SH2d-fronts.jl from lambda = -0.1: {K} batches x {B} continuation steps",
            "batch": B, "newton_tol": 1e-9, "gmres": GMRES, "bls": BLS["kind"], "continuation": CONT,
            "l2": "GPU arm: 256 MiB L2 flush between continuation steps (outside the event pairs); the Krylov basis of a solve exceeds L2"}


DUMP_MAX_ENTRIES = 1 << 21  # per state vector (16 MiB in fp64): the dump stays below 64 MiB at any grid
ROW_KEYS = ("param", "x", "itnewton", "itlinear", "ds", "step", "n_unstable")


def dump_outputs(d, rows, st):
    """Writes what the timed continuation returns to its caller as d/<name>.npy (float64): `branch` = its rows (ROW_KEYS), and
    the state after its last step: `u`, `p` (solution), `tau_u`, `tau_p` (secant tangent).  A state vector longer than
    DUMP_MAX_ENTRIES is written as the same seeded sample of entries on every run, so two builds compare entry for entry."""
    os.makedirs(d, exist_ok=True)
    host = lambda v: v.numpy() if hasattr(v, "numpy") else np.asarray(v, dtype=np.float64)
    out = {"branch": np.array([[float(r[k]) for k in ROW_KEYS] for r in rows], dtype=np.float64).reshape(-1, len(ROW_KEYS)),
           "u": host(st.z_u), "p": np.array([st.z_p]), "tau_u": host(st.tau_u), "tau_p": np.array([st.tau_p])}
    n = len(out["u"])
    if n > DUMP_MAX_ENTRIES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ENTRIES, replace=False))
        out["u"], out["tau_u"] = out["u"][idx], out["tau_u"][idx]
    for k, v in out.items():
        np.save(os.path.join(d, k + ".npy"), np.ascontiguousarray(v, dtype=np.float64))


def cpp_opts(cb, max_steps, workers):
    return cb.make_opts(ds=CONT["ds"], dsmin=CONT["dsmin"], dsmax=CONT["dsmax"], p_min=CONT["p_min"], p_max=CONT["p_max"], max_steps=max_steps,
                        newton_tol=1e-9, newton_maxit=15, reltol=GMRES["reltol"], restart=GMRES["restart"], maxiter=GMRES["maxiter"],
                        pc_shift=1.0, nthreads=workers)


def main():
    global PAR
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="K: timed batches of --batch continuation steps")
    ap.add_argument("--warmup", type=int, default=3, help="W: untimed continuation steps before the timed window")
    ap.add_argument("--grid", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=10, help="B: continuation steps (at dsmax) per bench step")
    ap.add_argument("--impl", default="bk200")
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--ref-batches", type=int, default=4, help="reference arm: bounded sample = the first batches of the window")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--bls", default="matrixfree", choices=["matrixfree", "bordering"])
    ap.add_argument("--branch", default="front", choices=["front", "hexagons"])
    ap.add_argument("--partition", default="replicas", choices=["replicas", "scout", "speculative"],
                    help="N > 1: independent replicas (default), one window cut by a scout, or one branch with speculative step sizes (not measured on GPUs yet)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed window, write its branch rows and final state to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs")
    n, K, B = args.grid, args.steps, args.batch
    BLS["kind"] = args.bls
    BRANCH["kind"] = args.branch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    workload = f"SH2d-fronts {n}x{n} fp64 on (lx, ly) = {n / 256:g} x (8 pi, 4 pi/sqrt 3), PALC (secant) + {'MatrixFreeBLS' if args.bls == 'matrixfree' else 'BorderingBLS'} + GMRES({GMRES['restart']}) reltol {GMRES['reltol']:g}, Pr = DCT (L1+I)^-1"
    cores = os.cpu_count() or 1
    s_total = K * B * CONT["dsmax"]
    metric = "continuation steps/sec (SH2d PALC)"

    if args.impl == "reference":
        if rank != 0:
            return
        # CPU restatement of the reference path in C++/OpenMP on all host cores (oracle/c); bounded sample: the first
        # ref_batches batches of the same window, from the same start point (computed by the same CPU code)
        from oracle import cbaseline as cb
        t_setup = time.perf_counter()
        thr = cb.calibrated_threads(n * n)
        co = cpp_opts(cb, 1, thr)
        hexa, ok, _, _ = cb.newton((n, n), domain(n), PAR[0], PAR[1], sol0(n), 1e-8, 20, co)
        assert ok, "CPU Newton to the hexagons failed"
        fr, ok, _, _ = cb.newton((n, n), domain(n), PAR[0], PAR[1], front_guess(hexa, n), 1e-9, 30, co)
        assert ok, "CPU Newton to the front failed"
        t_setup = time.perf_counter() - t_setup
        nb = max(1, min(K, args.ref_batches))
        try:
            cb.reset_counters()
        except Exception:
            pass
        rows, secs, tstep, _, work = cb.palc((n, n), domain(n), PAR[1], fr, PAR[0], cpp_opts(cb, nb * B, thr))
        nst = len(rows) - 1
        v = nst / secs
        try:  # how close the CPU arm itself runs to its host's memory system (informational)
            b1, sp = cb.counters()
            triad = cb.triad_gbs(thr)
            host_roofline = {"bound": "host dram", "achieved": (b1 + sp) / secs * 1e-9, "peak": triad, "unit": "GB/s", "frac": (b1 + sp) / secs * 1e-9 / triad,
                             "note": "algorithmic bytes of the MGS / BLAS-1 sweeps (dot 16 N, axpy 24 N) and the CSR SpMVs (12 B per entry + vectors) of the sample, "
                                     "the preconditioner's FFT passes not counted, over the loop time; peak = STREAM triad on the same threads",
                             "blas1_gbytes": b1 * 1e-9, "spmv_gbytes": sp * 1e-9}
        except Exception as exc:
            host_roofline = {"error": repr(exc)}
        print(json.dumps({"metric": metric, "value": v, "unit": "steps/s", "n_gpus": args.gpus, "steps": K, "warmup": args.warmup,
                          "ms_per_step": 1e3 * B / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "impl": "reference",
                          "config": config_dict(n, workload, K, B),
                          "details": {"setup_s": round(t_setup, 1), "sample_steps": nst, "corrector_work": {"newton_its": work[0], "linear_its": work[1]}},
                          "cpu_baseline": {"value": v, "unit": "steps/s", "cores": thr, "kind": "port",
                                           "sample": f"the first {nst} continuation steps ({nb} of {K} batches) of the window from the converged front; "
                                                     f"C++17/OpenMP restatement (oracle/c: CSR SpMV with the kron-assembled L1, MGS GMRES, pair-FFT DCT Pr) on {thr} threads "
                                                     f"(fastest of the calibrated counts; the host offers {cb.load().bkcpu_max_threads()})",
                                           "host_roofline": host_roofline},
                          "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import __graft_entry__ as g
    bk = g.load_package()
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = local if world > 1 else 0
    torch.cuda.set_device(dev)
    replicas = world > 1 and args.partition == "replicas"
    ctx, ls, u_front = gpu_setup(bk, n, dev)
    jw = 1 if (replicas or world == 1) else world  # "world" seen by window_job
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=f"cuda:{dev}")  # > 126 MB L2

    # ---- warm-up: W untimed continuation steps from the start point (kernels, caches, allocator pools)
    if args.warmup > 0:
        gpu_run(bk, ctx, ls, u_front, PAR[0], args.warmup, 0, torch, timing=False, flush=flush)

    sampler = ClockSampler(dev)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    spec = (dist, f"cuda:{dev}") if (world > 1 and args.partition == "speculative") else None
    try:
        rows, my_ms, delta, info = window_job(bk, ctx, ls, n, u_front, s_total, rank, 1 if spec else jw, torch, flush, nsteps=K * B, spec=spec)
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
    finally:
        clocks = sampler.stop()
    if (jw == 1 or spec) and len(rows) != K * B + 1:
        raise RuntimeError(f"the branch ended after {len(rows) - 1} of the {K * B} continuation steps --steps {K} asks for")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, rows, info["state"])
    tt = torch.tensor([my_ms, float(len(rows)), info["scout_ms"], float(info["rejected"]), float(info["work_newton"]), float(info["work_linear"])],
                      dtype=torch.float64, device=f"cuda:{dev}")
    replica_dev = None
    if dist:
        allt = [torch.zeros_like(tt) for _ in range(world)]
        dist.all_gather(allt, tt)
        tmax = max(float(t[0]) for t in allt)
        per_rank = [{"ms": round(float(t[0]), 1), "steps": int(t[1]), "scout_ms": round(float(t[2]), 1), "rejected": int(t[3])} for t in allt]
        # the path's only collective: all_gather of the branch rows (lambda, ||u||, itnewton, itlinear)
        gathered = bk.segments.all_gather_rows(rows, 4 * K * B + 64, dist, torch, f"cuda:{dev}")
        branch = bk.segments.merge_chunks(gathered)  # replicas: the N branches one after the other
        if replicas:  # determinism across GPUs: every replica must produce the same rows
            g0 = gathered[0]
            replica_dev = float(max(np.nanmax(np.abs(np.nan_to_num(gr[:, :2]) - np.nan_to_num(g0[:, :2]))) for gr in gathered))
        wn, wl = int(sum(float(t[4]) for t in allt)), int(sum(float(t[5]) for t in allt))
    else:
        tmax, per_rank = my_ms, None
        branch = np.array([[r["param"], r["x"], r["itnewton"], r["itlinear"]] for r in rows])
        wn, wl = info["work_newton"], info["work_linear"]

    # ---- e2e: the same job through the plugin / C ABI with HOST buffers (pinned NumPy state; H2D/D2H inside every call)
    e2e = None
    if not args.no_e2e and spec is None:
        nthr, limiter = best_blas_threads(n * n, cores)
        if limiter is not None:
            limiter(limits=nthr, user_api="blas")
        ctx.pin_host = True
        bk.palc.V.host_alloc = ctx.pinned_empty
        uh = ctx.pinned_array(u_front.numpy())
        if dist:
            dist.barrier()
        rows_h, ms_h, d_h, info_h = window_job(bk, ctx, ls, n, uh, s_total, rank, jw, torch, flush, timing=False, wrap=ctx.pinned_array, nsteps=K * B)
        ctx.pin_host = False
        bk.palc.V.host_alloc = None
        th = torch.tensor([ms_h, float(d_h["h2d_bytes"]), float(d_h["d2h_bytes"]), float(info_h["work_newton"]), float(info_h["work_linear"]),
                           float(info_h["rejected"])], dtype=torch.float64, device=f"cuda:{dev}")
        if dist:
            allh = [torch.zeros_like(th) for _ in range(world)]
            dist.all_gather(allh, th)
            tmax_h = max(float(t[0]) for t in allh)
            h2d, d2h = sum(float(t[1]) for t in allh), sum(float(t[2]) for t in allh)
            wh = [int(sum(float(t[k]) for t in allh)) for k in (3, 4, 5)]
        else:
            tmax_h, h2d, d2h = ms_h, float(d_h["h2d_bytes"]), float(d_h["d2h_bytes"])
            wh = [info_h["work_newton"], info_h["work_linear"], info_h["rejected"]]
        e2e = {"value": (world if replicas else 1) * K * B / (tmax_h * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": int(h2d / K), "d2h_bytes_per_step": int(d2h / K),
               "corrector_work": {"newton_its": int(wh[0]), "linear_its": int(wh[1]), "rejected_steps": int(wh[2])},
               "note": "step acceptance in the snaking region is sensitive to rounding: the host-vector path (BLAS reductions) rejects a different set of steps than the device path, so its corrector work -- and its steps/s -- differ from run to run by up to 1.5x; the same window with pinned host NumPy state vectors: every residual / Jacobian / bordered solve crosses the C ABI with host pointers (H2D + D2H inside the timed region); bytes are per bench step (batch), all ranks"}
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return

    # ---- the same job through ONE C-ABI call from and to host buffers: bk_palc_run (include/bk200.h; the PALC loop as host C++
    # inside the library, same kernels in the same order as the plugin path above).  Rank 0's own run; replicas are identical.
    e2e_native = None
    if not args.no_e2e and world == 1:  # N = 1 only: at N > 1 the other ranks have left by now and rank 0 should not linger
        try:
            Pn = bk.palc
            alg_n, cpf_n, _, _ = make_algs(bk, ctx, ls, n)
            cpn = cpf_n()
            cpn.max_steps = K * B
            u_host = ctx.pinned_array(u_front.numpy())
            prob_n = Pn.BifurcationProblemB200(ctx, u_host, list(PAR), lens=0)
            ctx.sync()
            ctx.set_timing(0)
            sn0 = ctx.stats()
            st_n = torch.cuda.ExternalStream(ctx.lib.bk_stream(ctx.handle))
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(st_n)
            rows_n, info_n = Pn.continuation_native(prob_n, alg_n, cpn, normC=Pn.norminf)
            info_n["u"].numpy()  # the final state back on the host, inside the timed region
            ev1.record(st_n)
            ctx.sync()
            ms_n = float(ev0.elapsed_time(ev1))
            sn1 = ctx.stats()
            rows_n = rows_n[: K * B + 1]
            same = len(rows_n) == len(rows) and all(a["param"] == b["param"] and a["x"] == b["x"] and a["itlinear"] == b["itlinear"]
                                                    for a, b in zip(rows_n, rows))
            e2e_native = {"value": (world if replicas else 1) * K * B / (ms_n * 1e-3), "unit": "steps/s",
                          "h2d_bytes_per_step": int((sn1["h2d_bytes"] - sn0["h2d_bytes"]) / K), "d2h_bytes_per_step": int((sn1["d2h_bytes"] - sn0["d2h_bytes"] + 8 * 6 * len(rows_n)) / K),  # final state (counted by the library) + the rows
                          "abi_calls": 1, "rows_identical_to_the_device_resident_run": bool(same),
                          "corrector_work": {"newton_its": int(info_n["work_newton"]), "linear_its": int(info_n["work_linear"]), "rejected_steps": int(info_n["nfail"])},
                          "note": "bk_palc_run(ctx, opts, linsolver, u0 [host], ..., rows [host], u_final): one C-ABI call for the whole window; start vector uploaded "
                                  "once, rows and the final state returned to the host; CUDA events around the call on the library's stream; no L2 flush inside the call "
                                  "(the Krylov basis of a solve exceeds L2)"
                                  + ("; rank 0's run x the number of (identical, independent) replicas" if replicas else "")}
        except Exception as exc:  # an extra measurement: it must never cost the line
            e2e_native = {"error": repr(exc)}

    value = (world if replicas else 1) * K * B / (tmax * 1e-3)
    nst = len(branch)
    peak, peak_src = measured_peak()
    fused_ms, fused_b, fused_l = delta.get("total_fused_ms", 0.0), delta.get("total_fused_bytes", 0), delta.get("total_fused_launches", 0)
    ach = (fused_b / 1e9) / (fused_ms * 1e-3) if fused_ms > 0 else None
    pc_ms, pc_n = delta.get("total_precond_ms", 0.0), delta.get("total_precond_applies", 0)
    roofline = {"bound": "hbm", "kernel": "k2_fused<E,bordered> + k2_update<E> (fused JVP+Arnoldi step = 2 launches per Krylov iteration; TMA ring)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None, "peak_source": peak_src,
                "traffic": ncu_traffic(), "launches": int(fused_l), "avg_launch_us": (fused_ms * 1e3 / fused_l) if fused_l else None,
                "algorithmic_bytes_per_launch": (fused_b / fused_l) if fused_l else None,
                "share_of_step": (TIMING_EVERY * fused_ms / my_ms) if my_ms else None,
                "sampling": f"CUDA-event pairs around both kernels of every {TIMING_EVERY}th GMRES solve of the timed region",
                "preconditioner": {"applies": int(pc_n), "avg_us": (pc_ms * 1e3 / pc_n) if pc_n else None, "share_of_step": (TIMING_EVERY * pc_ms / my_ms) if my_ms else None,
                                   "algorithmic_bytes_per_apply": 3 * 16 * n * n}}

    out = {"metric": metric, "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
           "ms_per_step": tmax / max(1, K), "higher_is_better": True, "scaling": "weak" if (replicas or world == 1) else "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic",
           "config": config_dict(n, workload, K, B),
           "details": dict({
               "continuation_steps_taken": int(nst - (world if replicas else (1 if world == 1 else 0))), "mean_itnewton": float(np.mean(branch[1:, 2])) if nst > 1 else 0.0,
               "mean_itlinear_per_step": float(np.mean(branch[1:, 3])) if nst > 1 else 0.0,
               "corrector_work": {"newton_its": int(wn), "linear_its": int(wl)}, "rejected_steps": int(sum(p["rejected"] for p in per_rank)) if per_rank else int(info["rejected"]),
               "parallelism": ("1 GPU" if world == 1 else
                               (f"one branch on {world} GPUs with speculative step sizes (segments.continuation_speculative): rank r corrects with the r-times-halved "
                                f"step, all_gather of 4 doubles + broadcast of the accepted point per step; {info.get('speculative')}") if spec else
                               (f"replicas only: {world} independent replicas of the job, one per GPU; replicated state; all_gather of rows only; "
                                f"max |row difference| between replicas = {replica_dev:g}") if replicas else
                               (f"one window cut into {world} chunks of equal predicted cost; replicated scout inside the timed region "
                                f"(ds x{SCOUT['ds_factor']:g}, Newton tol {SCOUT['newton_tol']:g}, GMRES reltol {SCOUT['gmres_reltol']:g})")),
               "per_rank": per_rank, "scout_ms": info["scout_ms"], "scout_points": info["scout_points"],
               "lambda_range": [float(branch[:, 0].min()), float(branch[:, 0].max())] if nst else None}),
           "clocks": clocks, "gpu_launches": int(delta.get("kernel_launches", 0)), "roofline": roofline, "e2e": e2e, "e2e_native": e2e_native}

    # ---- the GPU arm on the reference arm's sample: `--impl reference` times the first ref_batches batches of the window (a bounded
    # sample, cheaper per step than the window's average: the Krylov counts grow along the branch), `value` the whole window
    try:
        sm = info.get("step_ms")
        nref = max(1, min(K, args.ref_batches)) * B
        if sm and len(sm) >= nref:
            out["details"]["per_batch_ms"] = [round(float(sum(sm[i * B:(i + 1) * B])), 1) for i in range(K)]
            out["details"]["on_reference_sample"] = {
                "steps": nref, "steps_per_s": (world if replicas else 1) * nref / (sum(sm[:nref]) * 1e-3),
                "note": f"this rank's device time over the first {nref} continuation steps of the window = the sample bench.py --impl reference times"}
    except Exception as exc:  # informational only
        out["details"]["on_reference_sample"] = {"error": repr(exc)}

    # ---- cpu_baseline: C++/OpenMP restatement on the host cores, bounded sample from the same start point
    if not args.no_cpu_baseline and world == 1:
        from oracle import cbaseline as cb
        thr = cb.calibrated_threads(n * n)
        rows_c, secs, tstep, _, work = cb.palc((n, n), domain(n), PAR[1], u_front.numpy(), PAR[0], cpp_opts(cb, args.cpu_steps, thr))
        nc = len(rows_c) - 1
        out["cpu_baseline"] = {"value": nc / secs, "unit": "steps/s", "cores": thr, "kind": "port",
                               "sample": f"the first {nc} continuation steps of the same window from the same start point; C++17/OpenMP restatement "
                                         f"(oracle/c: CSR SpMV with the kron-assembled L1, MGS GMRES, pair-FFT DCT Pr) on {thr} threads (calibrated; host offers {cb.load().bkcpu_max_threads()})"}
        m = min(len(rows_c), len(rows))
        out["cpu_baseline"]["max_abs_param_diff_vs_gpu"] = float(max(abs(rows_c[i]["param"] - rows[i]["param"]) for i in range(m)))
    print(json.dumps(out))
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
