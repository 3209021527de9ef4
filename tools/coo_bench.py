#!/usr/bin/env python
"""coo_bench.py -- what building a resident CSR from COO triplets in device memory costs
(spmv_b200_csr_from_coo), against the host path, one JSON line per config on stdout (and in
--out FILE).

  python tools/coo_bench.py [--configs c2,c4] [--c3] [--reps 3] [--out FILE]

  c2  3D 27-point stencil 128^3 from the host generator (sorted columns, no duplicates)
  c4  R-MAT scale 24, 16 edges per vertex (power-law rows, duplicates)
  c3  uniform random n = 16 M, 32 per row (--c3: its host generation takes minutes)

The matrix's entries are put in device memory as int64 COO (torch's index type) in two orders:
shuffled (a seeded permutation), and sorted by (row, col) with the order of equal pairs kept.
Three builds per config, duplicates kept (flags 0):
  shuffled   from_coo on the shuffled COO (pack, radix sort, fill)
  sorted     from_coo on the sorted COO (the sort is skipped)
  host       the path without from_coo: sorted COO -> .cpu() -> host CSR (row counts, no sort
             needed) -> from_arrays; the cheapest form of the host path
Per build:
  ms_median / ms   host clock around the synchronous call (after a device synchronise), median and
                   all of --reps builds after one warm-up build
  entries_per_s    entries / median time
  peak_temp_bytes  the device temporaries of the build computed from the shapes (the formula of
                   csr_from_coo_here in csrc/spmv_b200.cu), CUB's scratch not included
  parity           kernel id 2 on the built handle against the oracle port's serial CSR on the host
                   generator's arrays (same entries per row), |dy| <= 1e-12 * sum |a x| per row
sorted_equals_host_path: the sorted build and the host build download bit for bit equal.
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

TOL = 1e-12


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


def index_bits(n):
    """Bits that can be non-zero in an index below n (at least 1, at most 31)."""
    b = 1
    while b < 31 and (1 << b) < n:
        b += 1
    return b


def peak_temp_bytes(M, N, n, unsorted, sum_runs):
    """Device temporaries of one from_coo build without CUB's scratch: the larger of the sort
    phase (two key and two index buffers) and the fill phase (keys, permutation, output positions
    when runs are summed, row counts)."""
    kb = 4 if index_bits(M) + index_bits(N) <= 32 else 8
    sort = (2 * kb + 8) * n if unsorted else 0
    fill = kb * n + (4 * n if unsorted else 0) + (4 * (n + 1) if sum_runs else 0) + 4 * (M + 1)
    return max(sort, fill)


def host_csr(sp, name):
    A = {"c2": lambda: sp.gen_stencil27(128, 128, 128), "c4": lambda: sp.gen_rmat(24, 16),
         "c3": lambda: sp.gen_uniform_random(16000000, 32, 42)}[name]()
    return A.M, A.N, A.IRP.copy(), A.JA.copy(), A.AS.copy()


def timed(torch, fn, reps):
    fn().close()  # warm-up build
    times, h = [], None
    for i in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h = fn()
        times.append((time.perf_counter() - t0) * 1e3)
        if i + 1 < reps:
            h.close()
    return h, times


def parity(O, torch, h, M, x, y_ref, bound):
    y = torch.full((M,), float("nan"), dtype=torch.float64, device="cuda")
    h.spmv(torch.from_numpy(x).cuda(), y, kernel=2)
    ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
    return {"ok": bool(ok), "worst_ratio": worst, "tol": TOL, "kernel": 2}


def run_config(sp, O, torch, name, reps, devinfo, watts):
    M, N, IRP, JA, AS = host_csr(sp, name)
    n = len(JA)
    x = np.random.default_rng(1).uniform(-1, 1, N)
    y_ref = O.csr_spmv(M, IRP, JA, AS, x)
    bound = O.csr_abs_bound(M, IRP, JA, AS, x)

    # device COO: in the generator's order, then sorted by (row, col) stably, then shuffled
    crow = torch.from_numpy(np.asarray(IRP, np.int64)).cuda()
    row = torch.repeat_interleave(crow.diff(), output_size=n)
    col = torch.from_numpy(np.asarray(JA, np.int64)).cuda()
    val = torch.from_numpy(AS).cuda()
    del crow
    o = torch.sort(row * N + col, stable=True).indices
    s_row, s_col, s_val = row[o], col[o], val[o]
    p = torch.randperm(n, generator=torch.Generator(device="cuda").manual_seed(7), device="cuda")
    r_row, r_col, r_val = row[p], col[p], val[p]
    del row, col, val, o, p
    torch.cuda.synchronize()

    def host_path():
        r, c, v = s_row.cpu().numpy(), s_col.cpu().numpy(), s_val.cpu().numpy()
        irp = np.zeros(M + 1, np.int64)
        irp[1:] = np.cumsum(np.bincount(r, minlength=M))
        return sp.CsrDevice.from_arrays(M, N, irp if n >= (1 << 31) - 64 else irp.astype(np.int32),
                                        c.astype(np.int32), v)

    builds = {"shuffled": (lambda: sp.CsrDevice.from_coo(M, N, r_row, r_col, r_val), True),
              "sorted": (lambda: sp.CsrDevice.from_coo(M, N, s_row, s_col, s_val), False),
              "host": (host_path, None)}
    rec = {"config": name, "device": devinfo["name"], "power_limit_w": watts, "M": M, "N": N, "nnz": n,
           "index_dtype": "int64", "sum_duplicates": False,
           "key_bits": index_bits(M) + index_bits(N)}
    handles = {}
    for key, (fn, unsorted) in builds.items():
        h, ms = timed(torch, fn, reps)
        med = statistics.median(ms)
        rec[key] = {"ms_median": med, "ms": ms, "entries_per_s": n / (med * 1e-3),
                    "peak_temp_bytes": None if unsorted is None else peak_temp_bytes(M, N, n, unsorted, False),
                    "parity": parity(O, torch, h, M, x, y_ref, bound)}
        handles[key] = h
    a, b = handles["sorted"].download(), handles["host"].download()
    rec["sorted_equals_host_path"] = bool(all(np.array_equal(u.view(np.uint8), w.view(np.uint8))
                                              for u, w in zip(a, b)))
    rec["host_over_shuffled"] = rec["host"]["ms_median"] / rec["shuffled"]["ms_median"]
    rec["parity_ok"] = all(rec[k]["parity"]["ok"] for k in builds)
    for h in handles.values():
        h.close()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--configs", default="c2,c4", help="comma-separated subset of c2,c4,c3")
    ap.add_argument("--c3", action="store_true", help="also run c3 (minutes of host generation)")
    ap.add_argument("--reps", type=int, default=3, help="timed builds per path (after one warm-up)")
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
        line = json.dumps(run_config(sp, O, torch, name, args.reps, devinfo, watts))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
