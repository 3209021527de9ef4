#!/usr/bin/env python
"""bench.py -- FP64 SpMV (CSR, HLL) throughput on B200 against the HBM roofline.

Contract (one JSON line on stdout, printed by rank 0):
  python bench.py --gpus N --steps K --warmup W [--impl reference]
                  [--workload c5|c2w|c1|c2|c3|c4] [--format csr|hll] [--kernel ID] [--wpb W]
                  [--dump-outputs DIR]

  metric   GFLOP/s = 2*nnz / t  (BASELINE.json), with achieved HBM GB/s on the
           minimum-traffic byte count B_min = 12 nnz + 4 (M+1) + 8 M + 8 N.
  workload default, EVERY N (1, 2, 4, 8): BASELINE configs[4], the 3D 27-point stencil 512^3
           (n = 134 217 728, nnz = 3 609 741 304; 46 GB and 64-bit row offsets on one GPU) split
           into N z-slabs, iterated x_{k+1} = A x_k with a one-plane halo per neighbour per step:
           STRONG scaling.  --workload c2w is round 1's weak-scaling proxy (one 128^3 slab per
           GPU); c1..c4 time one single-GPU config (N = 1 only).
  step     one SpMV pass over the whole (distributed) matrix.
  value    whole-job GFLOP/s with inputs resident in HBM over exactly K timed steps, cut into
           --regions (1) regions, every region bracketed by barrier + synchronize on both
           sides, timed with CUDA events on the stepping stream, max over ranks.
  outputs  --dump-outputs DIR: y of the last timed step as DIR/y.npy, float64, at most 2^21 rows
           (dump_rows()).  c5/c2w: the iterate after the last region, x_{w+k} = A^(w+k) x_0 with
           w = config.warmup_steps_per_region and k = region_steps[-1], gathered over ranks.
           --impl reference: y of the headline variant's last pass.
           Inputs are generated from fixed seeds, so equal arguments give equal inputs.
  e2e      same metric through the host-buffer C ABI call (spmv_b200_csr_spmv_host): HOST x
           slice in, HOST y slice out, copies inside the timed region.  Headline = PAGEABLE
           caller buffers (what the reference's compute_benchmark_csr hands over); "pinned" =
           page-locked buffers as a sub-key.
  configs  (N = 1 default run) one sub-record per single-GPU BASELINE config -- C1 (L2-flushed),
           C2, C3, C4 -- with GFLOP/s, roofline fraction, parity against the oracle and the
           reference's CPU paths on that very matrix; each times K steps per format.
  roofline dominant kernel: B_min / mean CUDA-event launch time vs the measured
           HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline / --impl reference: the reference's own CPU code (oracle/_ref, compiled from
           the original project's src/) on the machine's host cores.  --impl reference times
           exactly K passes of every variant and reports the median pass.
  side legs  K does not govern these; each reports its own count: the e2e legs (min(K, 20)
           calls, at least 3), the stand-alone kernel of c5/c2w before and after the run (20
           reps, 8 above 10^9 entries) and the cpu_baseline sub-records of the B200 line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# libgomp reads these when it is first loaded: idle OpenMP workers must sleep, not spin
# (BASELINE.md section 3: the reference's OpenMP rows collapse otherwise on shared cores)
os.environ.setdefault("OMP_WAIT_POLICY", "passive")
os.environ.setdefault("OMP_PROC_BIND", "close")

import numpy as np  # noqa: E402

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


def ncu_traffic(workload, kernel_symbol):
    """Per-launch dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the
    committed ncu summary (profiles/traffic.json, written by tools/summarize_profile.py), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            allt = json.load(f)
        keys = sorted(k for k in allt if k.endswith("_" + workload))
        for k in reversed(keys):
            for name, v in allt[k].items():
                if name.startswith(kernel_symbol):
                    return v
    except Exception:
        pass
    return None


def roofline_bytes(n_rows, n_cols, nnz):
    return 12 * nnz + 4 * (n_rows + 1) + 8 * n_rows + 8 * n_cols


DUMP_MAX_ROWS = 1 << 21     # 16 MB of float64 per dumped vector


def dump_rows(n):
    """Rows of an n-row result that --dump-outputs writes: all of them up to DUMP_MAX_ROWS, else the
    same seeded sample in every run and every build, in ascending order."""
    if n <= DUMP_MAX_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ROWS, replace=False))


def dump_outputs(directory, arrays):
    """arrays: name -> float64 vector; written as <directory>/<name>.npy."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, np.float64))


DESCR = {
    "c1": "2D 5-point Poisson 1000x1000",
    "c2": "3D 27-point stencil 128^3",
    "c3": "uniform random n=16M, 32 nnz/row",
    "c4": "R-MAT scale 24, degree 16",
    "c5": "3D 27-point stencil 512^3",
    "c2w": "3D 27-point stencil 128x128x128N, one 128^3 slab per GPU",
    "tiny": "3D 27-point stencil 32^3 (self-test)",
}


def host_matrix(sp, workload):
    return {"c1": lambda: sp.gen_poisson2d(1000, 1000), "c2": lambda: sp.gen_stencil27(128, 128, 128),
            "c3": lambda: sp.gen_uniform_random(16000000, 32, 42), "c4": lambda: sp.gen_rmat(24, 16),
            "tiny": lambda: sp.gen_stencil27(32, 32, 32)}[workload]()


def _host_cores_now():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


_HOST_CORES = _host_cores_now()   # taken at start-up: NCCL narrows the calling thread's mask during init


def host_cores():
    return _HOST_CORES


# ------------------------------------------------------------------ clocks --
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        rows = [l for (t, l) in self.lines if t0 - 0.1 <= t <= t1 + 0.15] or [l for _, l in self.lines]
        for l in rows:
            f = [s.strip() for s in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                               f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------- reference (CPU) --
def cpu_reference_run(O, A_arrays, x, steps, warmup, threads=None, hll=True, serial_steps=None, ys=None):
    """Times the reference's own CPU CSR SpMV on this box.  Returns the best variant (GFLOP/s) and
    every variant measured.  oracle/_ref when present ("reference"), else the oracle port ("port").
    Every OpenMP variant times `steps` passes, the serial one `serial_steps` (default min(steps, 2));
    each variant reports its count as "steps".  ys: a dict that receives each variant's last y."""
    M, N, IRP, JA, AS = A_arrays
    nnz = len(JA)
    nthreads = threads or O.max_threads()
    variants = {}
    if O.ref_available():
        kind = "reference"
        R = O.RefCsr(M, N, IRP, JA, AS)

        def run(name):
            if name == "serial":
                return O.ref_csr_serial(R, x)
            sched = "guided" if name == "omp_guided" else "nnz"
            return O.ref_csr_omp(R, x, nthreads, sched)[:2]

        names = ["serial", "omp_guided", "omp_nnz"]
    else:
        kind = "port"
        IRPc, JAc, ASc = (np.ascontiguousarray(IRP, np.int32), np.ascontiguousarray(JA, np.int32),
                          np.ascontiguousarray(AS, np.float64))

        def run(name):
            return O.csr_spmv_timed(M, IRPc, JAc, ASc, x, 1 if name == "serial" else nthreads)

        names = ["serial", "omp_guided"]
    for name in names:
        n_w, n_s = ((min(warmup, 1), min(steps, 2) if serial_steps is None else serial_steps) if name == "serial"
                    else (warmup, steps))
        for _ in range(n_w):
            run(name)
        ms = []
        for _ in range(n_s):
            t, y = run(name)
            ms.append(t)
        if ys is not None:
            ys[name] = y
        variants[name] = {"ms_per_step": statistics.median(ms),
                          "gflops": 2.0 * nnz / (statistics.median(ms) * 1e6),
                          "cores": 1 if name == "serial" else nthreads, "steps": n_s}
    best = max(variants, key=lambda k: variants[k]["gflops"])
    if hll and kind == "reference" and nnz <= 100_000_000:
        # the reference's HLL CPU paths too (row-major hacks, its own packer); reported beside
        # the CSR ones, never the headline: the B200 arm's value is CSR
        try:
            ser, omp = [], []
            for _ in range(max(1, min(steps, 3))):
                s_ms, o_ms, _ = O.ref_hll_bench(R, x, nthreads)
                ser.append(s_ms)
                omp.append(o_ms)
            for name, ms, cores in (("hll_serial", statistics.median(ser), 1),
                                    ("hll_omp_guided", statistics.median(omp), nthreads)):
                variants[name] = {"ms_per_step": ms, "gflops": 2.0 * nnz / (ms * 1e6), "cores": cores}
        except Exception as e:  # a missing HLL row must not cost the CSR baseline
            variants["hll_error"] = repr(e)[:120]
    return kind, best, variants, nthreads


def reference_sample(O, workload, gpus):
    """The matrix the CPU arm times: the config itself when it is small, else a bounded sample of
    it.  Built by the ORACLE-side generators (oracle/oracle.c) -- this arm maps no product library."""
    if workload == "c5":
        planes = 32
        M, N, IRP, JA, AS = O.gen_stencil27_rows(512, 512, 512, 0, planes * 512 * 512)
        return (M, N, IRP, JA, AS), (f"rows of the first {planes} of 512 planes ({len(JA) / 1e6:.0f} M of "
                                     f"3 610 M entries; the whole matrix does not fit an int-indexed sparse_csr)")
    if workload == "c2w":
        M, N, IRP, JA, AS = O.gen_stencil27(128, 128, 128 * gpus)
        return (M, N, IRP, JA, AS), f"full 128x128x{128 * gpus} stencil"
    if workload == "c3":
        rows = 4_000_000
        M, N, IRP, JA, AS = O.gen_uniform_rows(16_000_000, 32, 42, 0, rows)
        return (M, N, IRP, JA, AS), f"first {rows} of 16 M rows (128 M of 512 M entries), x full length"
    if workload == "c4":
        M, N, IRP, JA, AS = O.gen_rmat(22, 16)
        return (M, N, IRP, JA, AS), "R-MAT scale 22 (same parameters, a quarter of scale 24's entries)"
    if workload == "c1":
        return O.gen_poisson2d(1000, 1000), "full matrix"
    if workload == "tiny":
        return O.gen_stencil27(32, 32, 32), "full matrix"
    return O.gen_stencil27(128, 128, 128), "full matrix"


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # torchrun exports OMP_NUM_THREADS=1 to every rank; this arm is the reference's OpenMP code on
    # ALL host cores, and libgomp reads the variable once, when it is first loaded (below)
    cores = host_cores()
    os.environ["OMP_NUM_THREADS"] = str(cores)
    from oracle import oracle as O
    t0 = time.time()
    arrays, sample = reference_sample(O, args.workload, args.gpus)
    M, N, IRP, JA, AS = arrays
    x = np.random.default_rng(0).uniform(0, 1, N)
    steps = max(1, args.steps)
    ys = {}
    kind, best, variants, nthreads = cpu_reference_run(O, arrays, x, steps, max(min(args.warmup, 2), 1),
                                                       threads=max(O.max_threads(), 1), hll=False,
                                                       serial_steps=steps, ys=ys)
    v = variants[best]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"y": ys[best][dump_rows(M)]})
    line = {
        "impl": "reference", "metric": "fp64_spmv_gflops", "value": v["gflops"], "unit": "GFLOP/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": v["ms_per_step"],
        "higher_is_better": True, "scaling": "strong" if args.workload == "c5" else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "gpu_launches": 0,
        "config": {"workload": f"{args.workload}: {DESCR[args.workload]}", "format": "csr", "rows": M,
                   "nnz": len(JA), "variant": best, "B_min_bytes": roofline_bytes(M, N, len(JA)),
                   "note": "GFLOP/s of the sample; SpMV throughput of the stencil does not depend on "
                           "how many planes are timed"},
        "cpu_baseline": {"value": v["gflops"], "unit": "GFLOP/s", "cores": v["cores"], "kind": kind,
                         "sample": f"{sample}, {steps} SpMV passes per variant, median",
                         "variants": variants, "host_threads": nthreads, "host_cores": cores,
                         "build": O.ref_kind() if kind == "reference" else "port"},
        "e2e": {"value": v["gflops"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------- single-GPU configs (C1..C4) --
KERNEL_SYMBOL = {("csr", 0): "csr_vec_kernel<1,", ("csr", 1): "csr_vec_kernel<32,",
                 ("csr", 2): "csr_stream_kernel", ("csr", 3): "csr_block_row_kernel",
                 ("csr", 4): "csr_stream_kernel", ("hll", 0): "hll_warp_kernel<1",
                 ("hll", 1): "hll_warp_kernel<1", ("hll", 2): "hll_warp_kernel<1",
                 ("hll", 3): "hll_stream_kernel"}


# what ids 2 of each format resolve to on the BASELINE configs (profiles/r2_*_ncu_summary.md)
DOMINANT_KERNEL = {("c1", "csr"): "csr_pipe_kernel", ("c1", "hll"): "hll_pipe_kernel",
                   ("c3", "csr"): "sell_kernel", ("c3", "hll"): "sell_kernel", ("c4", "csr"): "sell_kernel"}


def single_config(sp, O, torch, workload, steps, warmup, wpb, with_cpu=True, with_e2e=True, kernels=None,
                  keep_y=None):
    """One BASELINE single-GPU config: parity gate, then device-timed CSR and HLL, the e2e entry
    points and the reference's CPU paths on the same matrix.  keep_y: a format; the dump_rows()
    of the y its last timed step computed go to rec["y"]."""
    t_start = time.time()
    A = host_matrix(sp, workload)
    nnz, M, N = A.NZ, A.M, A.N
    bmin = roofline_bytes(M, N, nnz)
    peak, peak_src = measured_peak()
    x_host = np.random.default_rng(0).uniform(0, 1, N)
    hcsr = sp.CsrDevice.from_host(A)
    hhll = hcsr.to_hll() if workload != "c4" else None      # HLL padding explodes on power-law rows
    x = torch.from_numpy(x_host).cuda()
    y = torch.zeros(M, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()
    ck, hk = (kernels or {}).get("csr", 2), (kernels or {}).get("hll", 2)
    fmt = {"csr": (hcsr, ck, sp.CSR_KERNEL_NAMES[ck]), "hll": (hhll, hk, sp.HLL_KERNEL_NAMES[hk])}
    small = bmin <= 256e6  # fits (or nearly fits) the 126 MB L2
    import ctypes

    # parity gate on this very input before anything is timed: the reference's own serial CSR
    # (oracle/_ref) where it exists, else the port
    if O.ref_available():
        _, y_ref = O.ref_csr_serial(O.RefCsr(M, N, A.IRP, A.JA, A.AS), x_host)
        oracle_kind = "reference serial CSR (oracle/_ref)"
    else:
        y_ref = O.csr_spmv(M, A.IRP, A.JA, A.AS, x_host)
        oracle_kind = "oracle port"
    bound = O.csr_abs_bound(M, A.IRP, A.JA, A.AS, x_host)
    parity = {"oracle": oracle_kind}
    for name, (h, k, _) in fmt.items():
        if h is None:
            continue
        y.fill_(float("nan"))
        h.spmv(x, y, kernel=k, warps_per_block=wpb)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, 1e-12)
        parity[name] = {"ok": ok, "worst_ratio": worst}
        if not ok:
            raise SystemExit(f"{workload}: parity failed for {name} kernel {k}: worst ratio {worst}")

    results = {}
    for name, (h, k, kname) in fmt.items():
        if h is None:
            continue
        for _ in range(warmup):
            h.spmv(x, y, kernel=k, warps_per_block=wpb)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        c0 = sp.counters()["launches"]
        torch.cuda.synchronize()
        s_all, e_all = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_all.record(stream)
        for a, b in ev:
            if small:  # matrix fits L2: evict it before every timed launch (outside the events)
                sp._lib.b200.spmv_b200_flush_l2(ctypes.c_void_p(stream.cuda_stream))
            a.record(stream)
            h.spmv(x, y, kernel=k, warps_per_block=wpb)
            b.record(stream)
        e_all.record(stream)
        torch.cuda.synchronize()
        if name == keep_y:
            y_last = y.cpu().numpy()[dump_rows(M)]
        per = [a.elapsed_time(b) for a, b in ev]
        total_ms = sum(per) if small else s_all.elapsed_time(e_all)
        ms_step, kern_ms = total_ms / steps, statistics.mean(per)
        launches = sp.counters()["launches"] - c0
        rec = {"kernel": kname, "kernel_id": k, "ms_per_step": ms_step, "gflops": 2.0 * nnz / (ms_step * 1e6),
               "gbs": bmin / (ms_step * 1e6), "launches_per_step": launches // steps,
               "roofline": {"bound": "hbm", "achieved": bmin / (kern_ms * 1e6), "peak": peak, "unit": "GB/s",
                            "frac": bmin / (kern_ms * 1e6) / peak, "frac_of_8TBs": bmin / (kern_ms * 1e6) / 8000.0,
                            "traffic": ncu_traffic(workload, DOMINANT_KERNEL.get((workload, name), KERNEL_SYMBOL[(name, k)])),
                            "peak_source": peak_src, "kernel_ms_mean": kern_ms, "kernel_ms_min": min(per),
                            "algorithmic_bytes": bmin}}
        if name == "csr":
            rec["sell"] = hcsr.sell_info()
        elif hhll is not None:
            rec["sell"] = hhll.sell_info()
        results[name] = rec

    # e2e through the reference-facing entry points: host x in, host y out, matrix resident after
    # the first call (cache policy "trust": what INTEGRATION.md tells an integrator to set)
    e2e = {}
    if with_e2e:
        L = sp._lib.b200
        dp = ctypes.POINTER(ctypes.c_double)
        sp.set_timing(0, 0)       # one pass per call: no separately timed launches inside the region
        sp.set_cache_policy("trust")
        # (host-side HLL packing of a 512 M-entry matrix is minutes of CPU work: CSR entry only there)
        Hc = sp.csr_to_hll(A, True) if hhll is not None and nnz <= 100_000_000 else None
        entry = {"csr": (L.csr_spmv_cuda_halfwarp_row_text if ck == 4 else L.csr_spmv_cuda_halfwarp_row, A),
                 "hll": (L.hll_spmv_cuda_warp_block, Hc)}
        L.set_csr_warps_per_block(wpb)
        L.set_hll_warps_per_block(wpb)
        n_e2e = max(3, min(steps, 20))
        for name, (fn, mat) in entry.items():
            if mat is None:
                continue
            for mem in ("pageable", "pinned"):
                if mem == "pinned":
                    xh, yh = sp.pinned_empty(N), sp.pinned_empty(M)
                else:
                    xh, yh = sp.aligned_array(N), sp.aligned_array(M)
                xh[:] = x_host
                xp, yp = xh.ctypes.data_as(dp), yh.ctypes.data_as(dp)
                for _ in range(2):
                    if fn(mat.ptr, xp, yp, None) <= 0:
                        raise SystemExit("e2e entry point failed: " + sp._lib.last_error())
                c0 = sp.counters()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(n_e2e):
                    fn(mat.ptr, xp, yp, None)
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t0) / n_e2e
                c1 = sp.counters()
                ok, worst = O.check_tolerance(yh, y_ref, bound, 1e-12)
                if not ok:
                    raise SystemExit(f"{workload}: e2e parity failed for {name}/{mem}: {worst}")
                e2e.setdefault(name, {})[mem] = {
                    "value": 2.0 * nnz / (dt * 1e9), "unit": "GFLOP/s", "ms_per_step": dt * 1e3, "steps": n_e2e,
                    "h2d_bytes_per_step": (c1["h2d_bytes"] - c0["h2d_bytes"]) // n_e2e,
                    "d2h_bytes_per_step": (c1["d2h_bytes"] - c0["d2h_bytes"]) // n_e2e}
                if mem == "pinned":
                    sp.pinned_free(xh)
                    sp.pinned_free(yh)
        if nnz <= 100_000_000:
            # the default policy re-hashes the caller's arrays on every call: what an UNMODIFIED
            # reference driver gets
            sp.set_cache_policy("hash")
            xh, yh = sp.aligned_array(N), sp.aligned_array(M)
            xh[:] = x_host
            fn, mat = entry["csr"]
            fn(mat.ptr, xh.ctypes.data_as(dp), yh.ctypes.data_as(dp), None)
            t0 = time.perf_counter()
            for _ in range(3):
                fn(mat.ptr, xh.ctypes.data_as(dp), yh.ctypes.data_as(dp), None)
            dt = (time.perf_counter() - t0) / 3
            e2e["csr"]["pageable_hash_policy"] = {"value": 2.0 * nnz / (dt * 1e9), "unit": "GFLOP/s",
                                                  "ms_per_step": dt * 1e3}
        sp.set_cache_policy("hash")
        sp.set_timing(1, 3)
        sp.release_all()
        del Hc

    cpu = None
    if with_cpu:
        big = nnz > 100_000_000
        kind, best, variants, nthreads = cpu_reference_run(
            O, (M, N, A.IRP, A.JA, A.AS), x_host, steps=2 if big else 5, warmup=1)
        cpu = {"value": variants[best]["gflops"], "unit": "GFLOP/s", "cores": variants[best]["cores"],
               "kind": kind, "variant": best,
               "sample": f"full {workload} matrix, {2 if big else 5} SpMV passes per variant (serial + OpenMP), median",
               "variants": variants, "host_threads": nthreads}
    for h in (hhll, hcsr):
        if h is not None:
            h.close()
    rec = {"workload": f"{workload}: {DESCR[workload]}", "rows": M, "cols": N, "nnz": nnz, "B_min_bytes": bmin,
           "l2_policy": ("L2 flushed (512 MB memset) before every timed launch; ms_per_step = mean launch interval"
                         if small else "inputs larger than L2"),
           "parity": parity, "formats": results, "e2e": e2e, "cpu_baseline": cpu,
           "wall_s": time.time() - t_start}
    if keep_y is not None:
        rec["y"] = y_last
    del A
    progress(f"config {workload} done in {rec['wall_s']:.1f} s")
    return rec


def reference_gpu_rows(workload="c2"):
    """The reference's own CUDA kernels rebuilt for sm_100a, on this GPU, in a separate process
    (both libraries export csr_spmv_cuda_*).  None when oracle/_ref/libspmv_ref_cuda.so is absent."""
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libspmv_ref_cuda.so")):
        return None
    try:
        r = subprocess.run([sys.executable, "-m", "oracle.oracle", "refcuda", workload], cwd=ROOT,
                           capture_output=True, text=True, timeout=600)
        line = [l for l in r.stdout.splitlines() if l.startswith("{")]
        return json.loads(line[-1]) if line else {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as e:
        return {"error": repr(e)[:200]}


def run_single(args):
    """--workload c1|c2|c3|c4 at N = 1: that config as the headline line."""
    import torch
    import spmv_scpa_b200 as sp
    from oracle import oracle as O
    torch.cuda.set_device(0)
    sampler = ClockSampler(0)
    sampler.start()
    time.sleep(0.25)
    t0 = time.time()
    kernels = {"csr": args.kernel if args.kernel is not None and args.format == "csr" else 2,
               "hll": args.kernel if args.kernel is not None and args.format == "hll" else 2}
    rec = single_config(sp, O, torch, args.workload, args.steps, args.warmup, args.wpb,
                        with_cpu=not args.no_cpu, kernels=kernels,
                        keep_y=args.format if args.dump_outputs else None)
    clocks = sampler.stop(t0, time.time())
    head = rec["formats"][args.format]
    e2e = rec["e2e"].get(args.format, {})
    line = {
        "metric": "fp64_spmv_gflops", "value": head["gflops"], "unit": "GFLOP/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": rec["workload"], "format": args.format, "kernel": head["kernel"],
                   "warps_per_block": args.wpb, "rows": rec["rows"], "cols": rec["cols"], "nnz": rec["nnz"],
                   "B_min_bytes": rec["B_min_bytes"], "l2_policy": rec["l2_policy"], "parity": rec["parity"],
                   "e2e_matrix": "resident after the first call (cache policy 'trust')"},
        "hbm_gbs": head["gbs"], "roofline": head["roofline"], "cpu_baseline": rec["cpu_baseline"],
        "e2e": dict(e2e.get("pageable", {}), pinned=e2e.get("pinned"), hash_policy=e2e.get("pageable_hash_policy")),
        "gpu_launches": head["launches_per_step"] * args.steps, "clocks": clocks,
        "formats": rec["formats"], "e2e_formats": rec["e2e"], "device": sp.device_info()["name"],
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"y": rec["y"]})
    emit(line)
    return 0


_T_START = time.time()


def progress(msg):
    """Phase marker on stderr (stdout carries the one JSON line)."""
    sys.stderr.write(f"[bench +{time.time() - _T_START:6.1f}s] {msg}\n")
    sys.stderr.flush()


def emit(line):
    out = getattr(sys, "_bench_real_stdout", None) or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(DESCR),
                    help="c5 (default) = 512^3 stencil over --gpus z-slabs, strong scaling; c2w = one 128^3 slab "
                         "per GPU, weak scaling; c1..c4 = one single-GPU config")
    ap.add_argument("--format", default="csr", choices=["csr", "hll"])
    ap.add_argument("--kernel", type=int, default=None)
    ap.add_argument("--wpb", type=int, default=4)
    ap.add_argument("--regions", type=int, default=1,
                    help="c5/c2w: the K timed steps are cut into this many regions, each after a reset of x")
    ap.add_argument("--configs", default="auto", choices=["auto", "all", "none"],
                    help="single-GPU BASELINE configs as sub-records of the N=1 line (auto: at N=1)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/y.npy (float64; all rows, or the "
                         "same seeded sample of 2^21 rows when there are more)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)
    # ONE line on stdout: libraries that print there (NCCL's version banner ...) are sent to stderr
    # while the run lasts; emit() writes the JSON line to the real stdout
    sys.stdout.flush()
    sys._bench_real_stdout = os.fdopen(os.dup(1), "w")   # on `sys`: bench_dist imports this file as a module
    os.dup2(2, 1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload in ("c5", "c2w") or args.gpus > 1 or world > 1:
        if args.workload not in ("c5", "c2w"):
            raise SystemExit(f"--workload {args.workload} is a single-GPU config; use c5 or c2w with --gpus > 1")
        if "RANK" not in os.environ:  # plain `python bench.py`: a 1-rank group
            os.environ.update(RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1",
                              MASTER_PORT=os.environ.get("MASTER_PORT", "29531"))
        import bench_dist
        return bench_dist.run(args)
    return run_single(args)


if __name__ == "__main__":
    sys.exit(main())
