#!/usr/bin/env python
"""spgemm_bench.py -- what the product of two resident CSR handles costs (spmv_b200_csr_spgemm),
one JSON line per config on stdout (and in --out FILE).

  python tools/spgemm_bench.py [--configs c2sq,galerkin,rmat,ata] [--reps 3] [--cpu] [--out FILE]

  c2sq      C2 (3D 27-point stencil 128^3) squared: 1142^3 products, nnz(C) = 634^3
  galerkin  P^T (A P) on C2, P the 2x2x2 piecewise-constant aggregation (from_coo), P^T by
            transpose(): two products, 64^3 coarse rows
  rmat      R-MAT scale 16, 16 edges per vertex, squared (power-law: long rows in the global table)
  ata       A^T A of uniform random n = 10^6, 16 per row (A^T by transpose())

Per config:
  ms_median / ms    host clock around the synchronous product(s) after a device synchronise,
                    median and all of --reps runs after one warm-up run
  products, nnz     products a_p b_q (computed from the factors' row lengths) and entries of C
  gflops            2 * products / median time
  spmv_multiple     median time over one id-2 SpMV on A (CUDA events, median of 20)
  cpu               with --cpu: scipy's single-threaded A @ B on the same arrays (one run)
  parity            C x against the chain of SpMVs of the factors, id 2, within
                    1e-12 * (|F1| (|F2| ... |x|)) per row
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from coo_bench import power_limit  # noqa: E402

TOL = 1e-12


def products(A, B):
    """Products a_p b_q of A·B from downloaded arrays: sum over A's entries of B's row lengths."""
    _, ja, _ = A.download()
    irp_b = B.download()[0]
    return int(np.diff(irp_b)[ja].sum())


def to_scipy(h):
    import scipy.sparse
    irp, ja, as_ = h.download()
    return scipy.sparse.csr_matrix((as_, ja, irp), shape=(h.M, h.N))


def abs_handle(sp, h):
    irp, ja, as_ = h.download()
    return sp.CsrDevice.from_arrays(h.M, h.N, irp if h.NZ >= (1 << 31) - 64 else irp.astype(np.int32), ja,
                                    np.abs(as_))


def parity(sp, torch, C, factors):
    """C x against F1 (F2 (... x)) with kernel id 2, bound |F1| (|F2| (... |x|))."""
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.rand(C.N, dtype=torch.float64, device="cuda", generator=g) * 2 - 1
    y, b = x, x.abs()
    for F in reversed(factors):
        Fa = abs_handle(sp, F)
        y1 = torch.zeros(F.M, dtype=torch.float64, device="cuda")
        b1 = torch.zeros(F.M, dtype=torch.float64, device="cuda")
        F.spmv(y, y1, kernel=2)
        Fa.spmv(b, b1, kernel=2)
        Fa.close()
        y, b = y1, b1
    yc = torch.zeros(C.M, dtype=torch.float64, device="cuda")
    C.spmv(x, yc, kernel=2)
    err = (yc - y).abs()
    worst = float((err / torch.clamp(b, min=1e-300)).max()) / TOL if C.M else 0.0
    return {"ok": bool((err <= TOL * b).all()), "worst_ratio": worst, "tol": TOL, "kernel": 2}


def setup(sp, torch, name):
    """(A for the SpMV yardstick, the product as a function returning C and the handles it made,
    [(left, right)] factor pairs for the product count, factors for parity, the scipy product)."""
    if name in ("c2sq", "galerkin"):
        A = sp.CsrDevice.stencil27(128, 128, 128)
    elif name == "rmat":
        A = sp.CsrDevice.from_host(sp.gen_rmat(16, 16))
    elif name == "ata":
        A = sp.CsrDevice.from_host(sp.gen_uniform_random(1000000, 16))
    else:
        raise KeyError(name)
    if name == "galerkin":
        n, m = 128, 64
        i = np.arange(n**3)
        agg = i % n // 2 + m * (i // n % n // 2) + m * m * (i // (n * n) // 2)
        P = sp.CsrDevice.from_coo(n**3, m**3, torch.from_numpy(i).cuda(), torch.from_numpy(agg).cuda(),
                                  torch.ones(n**3, dtype=torch.float64, device="cuda"))
        Pt = P.transpose()

        def run():
            AP = A.matmul(P)
            return Pt.matmul(AP), [AP]

        def cpu(As, Ps, Pts):
            return Pts @ (As @ Ps)
        return A, run, [Pt, A, P], cpu, (A, P, Pt)
    if name == "ata":
        At = A.transpose()
        return A, lambda: (At.matmul(A), []), [At, A], lambda At_s, A_s: At_s @ A_s, (At, A)
    return A, lambda: (A.matmul(A), []), [A, A], lambda A_s, _: A_s @ A_s, (A, A)


def run_config(sp, torch, name, reps, cpu, devinfo, watts):
    A, run, factors, cpu_fn, cpu_args = setup(sp, torch, name)
    x = torch.rand(A.N, dtype=torch.float64, device="cuda")
    y = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    spmv_ms = statistics.median(A.time(x, y, kernel=2, warmup=3, reps=20))

    C, extra = run()  # warm-up
    for h in [C] + extra:
        h.close()
    times = []
    for i in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        C, extra = run()
        times.append((time.perf_counter() - t0) * 1e3)
        if i + 1 < reps:
            for h in [C] + extra:
                h.close()
    med = statistics.median(times)
    if name == "galerkin":
        nprod = products(A, cpu_args[1]) + products(cpu_args[2], extra[0])
    else:
        nprod = products(factors[0], factors[1])
    rec = {"config": name, "device": devinfo["name"], "power_limit_w": watts, "M": C.M, "N": C.N,
           "products": nprod, "nnz": C.NZ, "ms_median": med, "ms": times,
           "gflops": 2 * nprod / (med * 1e-3) / 1e9, "spmv_id2_ms": spmv_ms, "spmv_multiple": med / spmv_ms,
           "parity": parity(sp, torch, C, factors)}
    if cpu:
        mats = [to_scipy(h) for h in cpu_args]
        t0 = time.perf_counter()
        S = cpu_fn(*mats)
        rec["cpu"] = {"scipy_ms": (time.perf_counter() - t0) * 1e3, "scipy_nnz": int(S.nnz)}
        rec["cpu"]["gpu_speedup"] = rec["cpu"]["scipy_ms"] / med
    rec["parity_ok"] = rec["parity"]["ok"]
    for h in [C] + extra + list({id(h): h for h in factors + list(cpu_args)}.values()):
        h.close()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="c2sq,galerkin,rmat,ata", help="comma-separated subset")
    ap.add_argument("--reps", type=int, default=3, help="timed runs per config (after one warm-up)")
    ap.add_argument("--cpu", action="store_true", help="also time scipy's A @ B on the host")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    import spmv_scpa_b200 as sp
    devinfo = sp.device_info()
    watts = power_limit()
    for name in [c for c in args.configs.split(",") if c]:
        line = json.dumps(run_config(sp, torch, name, args.reps, args.cpu, devinfo, watts))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
