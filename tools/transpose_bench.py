#!/usr/bin/env python
"""transpose_bench.py -- what building Aᵀ on the GPU costs (spmv_b200_csr_transpose) and how fast
the transposed handle multiplies, one JSON line per config on stdout (and in --out FILE).

  python tools/transpose_bench.py [--configs c2,c4] [--c3] [--builds 3] [--out FILE]

  c2  3D 27-point stencil 128^3, generated in HBM (symmetric: Aᵀ must equal A bit for bit)
  c4  R-MAT scale 24, 16 edges per vertex (power-law rows and columns, duplicates kept)
  c3  uniform random n = 16 M, 32 per row (--c3: its host generation and host oracle take minutes)

Per config:
  build_ms    host clock around the synchronous transpose call, median (and all) of --builds builds
              after one warm-up build
  spmv        kernel id 2 on A and on Aᵀ: CsrDevice.time, 3 warm-ups + 20 launches, median and min;
              B_min / t (Aᵀ's B_min with rows and columns swapped) against the measured 6 559.7 GB/s
  route       Aᵀ's SELL-P plan (sell_info(build=True)) and row bins (plan_info())
  parity      Aᵀ x (id 2) against the oracle port's serial CSR on scipy's transpose of the host
              arrays, and Aᵀ's download against those arrays bit for bit
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import scipy.sparse  # noqa: E402

MEASURED_HBM_GBS = 6559.7  # torch copy_ read+write on the B200 pool (DESIGN.md section 3)
TOL = 1e-12


def roofline_bytes(n_rows, n_cols, nnz):
    return 12 * nnz + 4 * (n_rows + 1) + 8 * n_rows + 8 * n_cols


def power_limit():
    """Power limit of the visible GPU from a read-only nvidia-smi query (None if unavailable)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        want = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0].strip()
        for line in out:
            idx, watts = (s.strip() for s in line.split(","))
            if idx == want:
                return float(watts)
        return float(out[0].split(",")[1]) if out else None
    except Exception:
        return None


def host_arrays(sp, O, name):
    """(M, N, IRP, JA, AS) on the host, and a function creating the resident handle."""
    if name == "c2":
        M, N, IRP, JA, AS = O.gen_stencil27(128, 128, 128)
        return (M, N, IRP, JA, AS), lambda: sp.CsrDevice.stencil27(128, 128, 128)
    A = sp.gen_rmat(24, 16) if name == "c4" else sp.gen_uniform_random(16000000, 32, 42)
    return (A.M, A.N, A.IRP, A.JA, A.AS), lambda: sp.CsrDevice.from_host(A)


def spmv_times(torch, h, n_in):
    x = torch.from_numpy(np.random.default_rng(0).uniform(0, 1, n_in)).cuda()
    y = torch.zeros(h.M, dtype=torch.float64, device="cuda")
    ms = h.time(x, y, kernel=2, warmup=3, reps=20)
    med = statistics.median(ms)
    b = roofline_bytes(h.M, h.N, h.NZ)
    return {"ms_median": med, "ms_min": min(ms), "B_min_bytes": b, "gbs": b / (med * 1e6),
            "of_measured": b / (med * 1e6) / MEASURED_HBM_GBS}


def run_config(sp, O, torch, name, builds, devinfo, watts):
    (M, N, IRP, JA, AS), make = host_arrays(sp, O, name)
    A = make()
    A.transpose().close()                      # warm-up build
    times = []
    for _ in range(builds):
        t0 = time.perf_counter()
        T = A.transpose()
        times.append((time.perf_counter() - t0) * 1e3)
        if len(times) < builds:
            T.close()
    rec = {"config": name, "device": devinfo["name"], "power_limit_w": watts,
           "M": M, "N": N, "nnz": int(A.NZ),
           "build_ms_median": statistics.median(times), "build_ms": times,
           "spmv_A": spmv_times(torch, A, A.N), "spmv_AT": spmv_times(torch, T, T.N)}
    rec["build_over_spmv_A"] = rec["build_ms_median"] / rec["spmv_A"]["ms_median"]
    info = T.sell_info(build=True)
    rec["route_AT"] = {"sell": info, "plan_info": T.plan_info()}
    rec["route_A"] = {"sell": A.sell_info(build=True), "plan_info": A.plan_info()}

    # parity: oracle arrays from scipy's CSR transpose (a stable counting sort by column)
    S = scipy.sparse.csr_matrix((np.asarray(AS), np.asarray(JA), np.asarray(IRP)), shape=(M, N)).T.tocsr()
    t_irp, t_ja, t_as = S.indptr.astype(np.int32), S.indices.astype(np.int32), S.data
    irp, ja, as_ = T.download()
    rec["layout_bit_exact"] = bool(np.array_equal(irp, t_irp) and np.array_equal(ja, t_ja)
                                   and np.array_equal(as_.view(np.uint64), t_as.view(np.uint64)))
    if name == "c2":
        a_irp, a_ja, a_as = A.download()
        rec["AT_equals_A"] = bool(np.array_equal(irp, a_irp) and np.array_equal(ja, a_ja)
                                  and np.array_equal(as_.view(np.uint64), a_as.view(np.uint64)))
    del irp, ja, as_
    x = np.random.default_rng(1).uniform(-1, 1, T.N)
    y = torch.zeros(T.M, dtype=torch.float64, device="cuda")
    T.spmv(torch.from_numpy(x).cuda(), y, kernel=2)
    ok, worst = O.check_tolerance(y.cpu().numpy(), O.csr_spmv(T.M, t_irp, t_ja, t_as, x),
                                  O.csr_abs_bound(T.M, t_irp, t_ja, t_as, x), TOL)
    rec["parity"] = {"ok": ok, "worst_ratio": worst, "tol": TOL, "against": "oracle port serial CSR on scipy's Aᵀ"}
    T.close()
    A.close()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="c2,c4", help="comma-separated subset of c2,c4,c3")
    ap.add_argument("--c3", action="store_true", help="also run c3 (minutes of host generation)")
    ap.add_argument("--builds", type=int, default=3, help="timed builds per config (after one warm-up)")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    import spmv_scpa_b200 as sp
    from oracle import oracle as O
    O.port()
    devinfo = sp.device_info()
    watts = power_limit()
    names = [c for c in args.configs.split(",") if c]
    if args.c3 and "c3" not in names:
        names.append("c3")
    for name in names:
        rec = run_config(sp, O, torch, name, args.builds, devinfo, watts)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
