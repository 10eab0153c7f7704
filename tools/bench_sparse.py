"""Sparse vs named operator on the B200: k_spmv (BK_SPARSE) against the SH2d stencil kernels at the config sizes.

  python tools/bench_sparse.py --out DIR [--reps 200]

Writes DIR/bench_sparse.json with
  - the card and its power limit (nvidia-smi, read in the same run);
  - bk_jvp on a BK_SPARSE context holding the SH2d Jacobian (oracle jac_sparse, 13 entries per row) vs bk_jvp on the BK_SH2D
    context, at 512^2 and 1024^2: CUDA-event device time per launch, median of `reps` warm launches; algorithmic bytes of the
    SpMV 12 nnz + 4 (N + 1) + 16 N and its GB/s, as a fraction of MEASURED_PEAKS.json hbm_gbs when that file exists;
  - GMRES at 1024^2, 100 Arnoldi iterations with Pr = SH_DCT (restart 100, unreachable tolerance): ms per iteration (wall clock of
    the synchronous solve / 100, median of 3), sparse vs named.
Needs a CUDA device: fails without one."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0 or not r.stdout.strip():
        raise SystemExit("bench_sparse: no GPU (nvidia-smi failed): " + r.stderr.strip())
    name, power = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}


def time_jvp(torch, ctx, x, y, reps):
    """median device time (ms) of one bk_jvp launch on device vectors, CUDA events around each launch on the library's stream"""
    stream = torch.cuda.ExternalStream(ctx.lib.bk_stream(ctx.handle))
    for _ in range(20):
        ctx.jvp(x, out=y, a0=0.0, a1=1.0)
    pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in pairs:
        a.record(stream)
        ctx.jvp(x, out=y, a0=0.0, a1=1.0)
        b.record(stream)
    ctx.sync()
    return statistics.median(a.elapsed_time(b) for a, b in pairs)


def time_gmres(bk, ctx, J, rhs, reps=3):
    ls = bk.GMRESB200(reltol=1e-30, restart=100, maxiter=100, Pr=True)
    ls(J, rhs, a0=2.0, a1=-1.0)  # warm
    out = []
    for _ in range(reps):
        ctx.sync()
        t = time.perf_counter()
        _, ok, it = ls(J, rhs, a0=2.0, a1=-1.0)
        ctx.sync()
        out.append((time.perf_counter() - t) * 1e3 / it)
    assert it == 100, it
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    info = gpu_info()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse: no CUDA device")
    import bench
    import __graft_entry__ as g
    from oracle import problems
    bk = g.load_package()
    peak_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peak_path))["hbm_gbs"]) if os.path.exists(peak_path) else None
    res = {"gpu": info, "reps": a.reps,
           "peak_reference": ({"hbm_gbs": peak, "source": "MEASURED_PEAKS.json hbm_gbs"} if peak else
                              {"hbm_gbs": 7700.0, "source": "B200 data-sheet HBM3e bandwidth (reference only, not a measured peak)"}),
           "spmv": [], "gmres": None}
    for n in (512, 1024):
        L = bench.domain(n)
        sh = problems.SwiftHohenberg((n, n), L, l=-0.1, nu=1.3)
        u = bench.sol0(n)
        A = sh.jac_sparse(u)
        N, nnz = A.shape[0], A.nnz
        sctx = bk.Context(bk.BK_SPARSE, (n, n), L, krylov_m=100)
        sctx.sparse_load(A)
        nctx = bk.Context(bk.BK_SH2D, (n, n), L, krylov_m=100, params=(-0.1, 1.3))
        nctx.jacobian(nctx.to_device(u))
        v = np.random.default_rng(0).standard_normal(N)
        row = {"n": n, "N": N, "nnz": nnz, "nnz_per_row": nnz / N}
        for key, c in (("sparse", sctx), ("named", nctx)):
            x, y = c.to_device(v), c.zeros()
            row[f"{key}_ms"] = time_jvp(torch, c, x, y, a.reps)
        byts = 12 * nnz + 4 * (N + 1) + 16 * N
        row["sparse_bytes"] = byts
        row["matrix_mb"] = (12 * nnz + 4 * (N + 1)) / 1e6
        row["sparse_gbs"] = byts / (row["sparse_ms"] * 1e-3) / 1e9
        row["sparse_over_named_time"] = row["sparse_ms"] / row["named_ms"]
        if peak:
            row["fraction_of_measured_peak"] = row["sparse_gbs"] / peak
        row["note"] = ("matrix larger than the 126 MB L2: every apply streams it from HBM" if row["matrix_mb"] > 126 else
                       "matrix smaller than the 126 MB L2: warm applies may be served partly from L2")
        res["spmv"].append(row)
        print(json.dumps(row), flush=True)
        if n == 1024:
            rhs = np.random.default_rng(1).standard_normal(N)
            g_ = {"n": n, "iterations": 100, "precond": "Pr = SH_DCT"}
            for key, c, J in (("sparse", sctx, bk.Jacobian(sctx)), ("named", nctx, bk.Jacobian(nctx))):
                c.precond_setup(bk.BK_PC_SH_DCT, 1.0)
                g_[f"{key}_ms_per_iter"] = time_gmres(bk, c, J, c.to_device(rhs))
            g_["sparse_over_named"] = g_["sparse_ms_per_iter"] / g_["named_ms_per_iter"]
            res["gmres"] = g_
            print(json.dumps(g_), flush=True)
        del sctx, nctx
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_sparse.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
