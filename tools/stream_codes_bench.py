"""A/B of the column codes of the staged CSR kernel on one GPU, in one process.

For C5 (the 512^3 27-point stencil on one GPU, 64-bit row offsets) and C2 (128^3), alternates the
knob csr_codes = 1 / 0 over several rounds of CUDA-event-timed launches of kernel 4 and reports
ms per launch, B_min GB/s and streamed GB/s, the CTAs each kernel body is launched with (from a
torch.profiler trace: the grid is SMs x the occupancy the body allows), the build time of the code
blocks, and whether y is bit-identical between the two settings.  Prints one JSON line per matrix and writes them all to
--out.  The device name and power limit are read in the same run.

    python tools/stream_codes_bench.py [--rounds 5] [--reps 20] [--wpb 4] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bench import roofline_bytes  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def streamed_bytes(H, codes_bytes):
    """Bytes one launch moves: values, columns (int32 or code blocks), one row offset per row (the
    tiles of consecutive rows read irp[row] and irp[row + 1]; 8 bytes from 2^31 - 64 entries on,
    as the library chooses, else 4), x and y."""
    idx = codes_bytes if codes_bytes else 4 * H.NZ
    off = 8 if H.NZ >= (1 << 31) - 64 else 4
    return 8 * H.NZ + idx + off * (H.M + 1) + 8 * H.M + 8 * H.N


def launch_grid(torch, H, x, y, wpb):
    """CTAs of the csr_stream_kernel launch of one SpMV, read from a torch.profiler trace."""
    with tempfile.TemporaryDirectory() as d:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            H.spmv(x, y, kernel=4, warps_per_block=wpb)
            torch.cuda.synchronize()
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    grids = [e["args"]["grid"][0] for e in events
             if e.get("cat") == "kernel" and "csr_stream_kernel" in e.get("name", "")]
    return grids[0] if grids else None


def measure(sp, torch, name, make, rounds, reps, wpb):
    H = make()
    x = torch.from_numpy(np.random.default_rng(0).uniform(-1, 1, H.N)).cuda()
    ys = {c: torch.empty(H.M, dtype=torch.float64, device="cuda") for c in (0, 1)}
    # int32 plan first, then the code blocks on their own, timed
    sp.set_knob("csr_codes", 0)
    H.spmv(x, ys[0], kernel=4, warps_per_block=wpb)
    torch.cuda.synchronize()
    sp.set_knob("csr_codes", 1)
    t0 = time.perf_counter()
    H.spmv(x, ys[1], kernel=4, warps_per_block=wpb)
    torch.cuda.synchronize()
    first_coded_ms = (time.perf_counter() - t0) * 1e3
    info = H.codes_info()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid = {}
    for c in (0, 1):
        sp.set_knob("csr_codes", c)
        grid[c] = launch_grid(torch, H, x, ys[c], wpb)
    ms = {0: [], 1: []}
    for _ in range(rounds):
        for c in (1, 0):
            sp.set_knob("csr_codes", c)
            ms[c] += H.time(x, ys[c], kernel=4, warps_per_block=wpb, warmup=3, reps=reps)
    for c in (0, 1):
        sp.set_knob("csr_codes", c)
        H.spmv(x, ys[c], kernel=4, warps_per_block=wpb)
    torch.cuda.synchronize()
    sp.set_knob("csr_codes", 1)
    same = bool(torch.equal(ys[0].view(torch.int64), ys[1].view(torch.int64)))
    b_min = roofline_bytes(H.M, H.N, H.NZ)
    rec = {"matrix": name, "rows": H.M, "nnz": H.NZ, "wpb": wpb, "codes": info, "y_bit_identical": same,
           "B_min_bytes": b_min, "build_plus_first_launch_ms": first_coded_ms}
    for c, label in ((0, "int32"), (1, "coded")):
        mean, mn = statistics.mean(ms[c]), min(ms[c])
        sb = streamed_bytes(H, info["bytes"] if c else 0)
        rec[label] = {"ms_mean": mean, "ms_min": mn, "launches": len(ms[c]), "grid_ctas": grid[c],
                      "ctas_per_sm": grid[c] / sms if grid[c] else None,
                      "B_min_GBps": b_min / (mean * 1e6), "streamed_bytes": sb,
                      "streamed_GBps": sb / (mean * 1e6)}
    rec["build_ms"] = first_coded_ms - rec["coded"]["ms_mean"]
    rec["speedup_mean"] = rec["int32"]["ms_mean"] / rec["coded"]["ms_mean"]
    H.close()
    sp.release_all()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--wpb", type=int, default=4)
    ap.add_argument("--only", choices=("c5", "c2"), default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import spmv_scpa_b200 as sp
    if not torch.cuda.is_available():
        raise SystemExit("stream_codes_bench: needs a CUDA device")
    device = card()
    cases = [("c5: 27-point 512^3, one GPU", lambda: sp.CsrDevice.stencil27(512, 512, 512)),
             ("c2: 27-point 128^3", lambda: sp.CsrDevice.stencil27(128, 128, 128))]
    if args.only:
        cases = [c for c in cases if c[0].startswith(args.only)]
    lines = []
    for name, make in cases:
        rec = measure(sp, torch, name, make, args.rounds, args.reps, args.wpb)
        rec["device"] = device
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
