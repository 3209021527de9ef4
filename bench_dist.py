"""bench.py's distributed leg (one rank per GPU, launched by torchrun; also the N = 1 default).
Part of the benchmark harness, not of the product package: it is allowed to use oracle/ as checker.

Workload c5 (default): BASELINE configs[4], the 512^3 27-point stencil cut into `world` z-slabs
generated directly in HBM, iterated x_{k+1} = A x_k with a one-plane halo per neighbour per step:
strong scaling.  Workload c2w: one 128^3 slab per GPU (round 1's weak-scaling proxy).

Every step runs inside libspmv_b200 (csrc/dist.cu: plan, push epilogue, epoch flags, CUDA graph);
torch.distributed only moves the connection blobs, provides the barriers and reduces the timings.
"""
import json
import os
import statistics
import time

import numpy as np

import spmv_scpa_b200 as sp
from spmv_scpa_b200 import dist as D


def x0_slice(g0, g1):
    """x_0[g] in (0,1), a pure function of the global index (so every rank can
    regenerate any part of it)."""
    g = np.arange(g0, g1, dtype=np.uint64)
    z = g + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z = z ^ (z >> np.uint64(31))
    return ((z >> np.uint64(11)).astype(np.float64) + 0.5) / 9007199254740992.0


def slab_geometry(workload, rank, world):
    if workload == "c5":
        nx = ny = nz = 512
    else:
        nx = ny = 128
        nz = 128 * world
    z = [nz * r // world for r in range(world + 1)]
    return nx, ny, nz, z


def gather_lists(dist, torch, device, values):
    """every rank's list of floats -> list of lists (same length on all ranks)"""
    mine = torch.tensor(values, dtype=torch.float64, device=device)
    out = [torch.zeros_like(mine) for _ in range(dist.get_world_size())]
    dist.all_gather(out, mine)
    return [t.cpu().tolist() for t in out]


def run(args):
    import torch
    import torch.distributed as dist
    from bench import (ClockSampler, DESCR, dump_outputs, dump_rows, emit, host_cores, measured_peak, ncu_traffic,
                       progress, roofline_bytes, reference_gpu_rows, single_config, cpu_reference_run)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    from oracle import oracle as O

    nx, ny, nz, z = slab_geometry(args.workload, rank, world)
    plane = nx * ny
    table = [D.stencil27_shard_desc(nx, ny, nz, z[r], z[r + 1]) for r in range(world)]
    mode = os.environ.get("SPMV_B200_EXCHANGE", "auto")
    plan = D.Plan(rank, table, mode=mode)
    r0, r1, c0, c1 = plan.r0, plan.r1, plan.c0, plan.c1
    kernel = args.kernel if args.kernel is not None else 4

    t_build = time.time()
    shard = sp.CsrDevice.stencil27(nx, ny, nz, z[rank], z[rank + 1], col_offset=c0, n_local=c1 - c0, cuts=plan.cuts)
    torch.cuda.synchronize()
    t_build = time.time() - t_build
    bmin_local = roofline_bytes(shard.M, shard.N, shard.NZ)

    # ---- stand-alone kernel on this rank's shard BEFORE any peer mapping exists ----
    xs = torch.from_numpy(x0_slice(c0, c1)).to(device)
    ys = torch.zeros(shard.M, dtype=torch.float64, device=device)
    reps_alone = 20 if shard.NZ < 1_000_000_000 else 8
    torch.cuda.synchronize()
    dist.barrier()
    pre = shard.time(xs, ys, kernel=kernel, warps_per_block=args.wpb, warmup=5, reps=reps_alone)

    it = D.DistSpMV(dist, shard, plan, kernel=kernel, wpb=args.wpb, device=device)
    x0_own = xs[r0 - c0:r1 - c0].contiguous()

    # ---- parity of step 1 on this rank's rows against the oracle (bounded: own slab) ----
    it.set_x(x0_own)
    it.iterate(1)
    y1 = it.result_own()
    M_own = r1 - r0
    # checked rows: the whole slab when it is small, else its first and last two planes
    # (the rows that depend on the halo) plus two planes from the middle
    if M_own <= 4 * 128 * 128 * 128:
        spans = [(0, M_own)]
    else:
        mid = (M_own // plane // 2) * plane
        spans = [(0, 2 * plane), (mid, mid + 2 * plane), (M_own - 2 * plane, M_own)]
    xl = x0_slice(c0, c1)  # local view of x0 over [c0, c1), columns shifted like the shard's
    ok, worst = True, 0.0
    for a, b in spans:
        Mp, _, IRPp, JAp, ASp = O.gen_stencil27_rows(nx, ny, nz, r0 + a, r0 + b)
        ja_local = (JAp.astype(np.int64) - c0).astype(np.int32)
        y_ref = O.csr_spmv(Mp, IRPp, ja_local, ASp, xl)
        bound = O.csr_abs_bound(Mp, IRPp, ja_local, ASp, xl)
        ok_i, worst_i = O.check_tolerance(y1[a:b], y_ref, bound, 1e-12)
        ok, worst = ok and ok_i, max(worst, worst_i)
    flag = torch.tensor([0 if ok else 1], device=device)
    dist.all_reduce(flag)
    if int(flag.item()) != 0:
        raise SystemExit(f"rank {rank}: multi-GPU parity failed after step 1 (worst ratio {worst})")

    nnz_t = torch.tensor([shard.NZ], dtype=torch.int64, device=device)
    dist.all_reduce(nnz_t)
    nnz_total = int(nnz_t.item())
    n_total = nx * ny * nz
    bmin_total = roofline_bytes(n_total, n_total, nnz_total)

    # ---- timed regions ----
    # The K timed steps are cut into R regions of K/R steps.  Every region: x reset to x_0 (the
    # iteration multiplies magnitudes by up to 52 per step, so a region starts from bounded values),
    # W warm-up steps queued on the rank's stream, a stream-ordered rendezvous (one-word all-reduce
    # the stepping stream waits for: ranks leave the host barrier milliseconds apart, and in push
    # mode a rank may run one step ahead per hop), then its steps between two CUDA events on that
    # stream.  ms of a region = max over ranks.
    sampler = None
    if rank == 0:
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.25)
    t_region0 = time.time()
    warm = max(args.warmup, world + 4)
    warm += warm % 2
    sync_word = torch.zeros(1, device=device)
    launches0 = sp.counters()["launches"]
    n_regions = max(1, min(args.regions, args.steps))
    region_steps = [args.steps * (i + 1) // n_regions - args.steps * i // n_regions for i in range(n_regions)]
    region_ms_mine = []
    for k in region_steps:
        it.set_x(x0_own)                       # sync + barrier inside
        it.iterate(warm)
        with torch.cuda.stream(it.stream):
            dist.all_reduce(sync_word)
        region_ms_mine.append(it.time(k, 1)[0])
        torch.cuda.synchronize()
        dist.barrier()
    launches = sp.counters()["launches"] - launches0
    clocks = sampler.stop(t_region0, time.time()) if sampler else None
    if rank == 0:
        progress(f"{args.workload}: {len(region_ms_mine)} timed regions done")
    by_rank = gather_lists(dist, torch, device, region_ms_mine)          # [rank][region]
    region_ms = [max(by_rank[r][i] for r in range(world)) for i in range(len(region_ms_mine))]
    total_ms = sum(region_ms)
    x_last = it.result_own()                   # x after the last region's warm-up and timed steps: rows [r0, r1)
    finite = bool(np.isfinite(x_last).all())
    y_dump = None
    if args.dump_outputs:
        rows = dump_rows(n_total)
        parts = [None] * world
        dist.all_gather_object(parts, x_last[rows[(rows >= r0) & (rows < r1)] - r0])
        y_dump = np.concatenate(parts)         # slabs are in rank order
    del x_last
    launches_per_step = len(plan.segments) + (2 if it.mode == "push" and world > 1 else 0)

    # ---- stand-alone kernel again, after the peers are mapped and the job has run ----
    torch.cuda.synchronize()
    dist.barrier()
    post = shard.time(xs, ys, kernel=kernel, warps_per_block=args.wpb, warmup=5, reps=reps_alone)
    alone = gather_lists(dist, torch, device, [statistics.mean(pre), min(pre), statistics.mean(post), min(post)])
    kern_ms = statistics.mean(post)

    # ---- e2e: host x slice in, host y slice out, every step (spmv_b200_csr_spmv_host) ----
    n_e2e = max(3, min(args.steps, 20))
    e2e_ms = {}
    for mem in ("pageable", "pinned"):
        if mem == "pinned":
            xh, yh = sp.pinned_empty(shard.N), sp.pinned_empty(shard.M)
        else:
            xh, yh = sp.aligned_array(shard.N), sp.aligned_array(shard.M)
        xh[:] = xl
        for _ in range(2):
            shard.spmv_host(xh, yh, kernel=kernel, warps_per_block=args.wpb)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            shard.spmv_host(xh, yh, kernel=kernel, warps_per_block=args.wpb)
        torch.cuda.synchronize()
        dist.barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / n_e2e], dtype=torch.float64, device=device)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e_ms[mem] = float(dt.item()) * 1e3
        # y of the host call == step 1 of the distributed run (same x_0, same rows)
        for a, b in spans:
            if not np.allclose(yh[a:b], y1[a:b], rtol=1e-12, atol=1e-12 * float(np.abs(y1[a:b]).max())):
                raise SystemExit(f"rank {rank}: e2e ({mem}) result differs from the resident path")
        if mem == "pinned":
            sp.pinned_free(xh)
            sp.pinned_free(yh)
    sp.release_all()

    line = None
    if rank == 0:
        peak, peak_src = measured_peak()
        ms_step = total_ms / args.steps
        strong = args.workload == "c5"
        wl = (f"c5: 3D 27-point stencil 512^3, {world} z-slab(s)" if strong
              else f"c2w: 3D 27-point stencil 128x128x{nz}, one 128^3 slab per GPU")

        def e2e_rec(mem):
            return {"value": 2.0 * nnz_total / (e2e_ms[mem] * 1e6), "unit": "GFLOP/s", "ms_per_step": e2e_ms[mem],
                    "steps": n_e2e, "h2d_bytes_per_step": 8 * sum(t.c1 - t.c0 for t in table),
                    "d2h_bytes_per_step": 8 * n_total}

        line = {
            "metric": "fp64_spmv_gflops", "value": 2.0 * nnz_total / (ms_step * 1e6), "unit": "GFLOP/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl, "format": "csr", "kernel": sp.CSR_KERNEL_NAMES[kernel],
                       "warps_per_block": args.wpb, "rows": n_total, "nnz": nnz_total, "B_min_bytes": bmin_total,
                       "iteration": "x_{k+1} = A x_k, halo exchange of one plane per neighbour per step",
                       "exchange": it.mode, "cuda_graph": it.has_graph,
                       "halo_bytes_per_rank_per_step": plan.halo_bytes(),
                       "l2_policy": "inputs larger than L2 (>= 0.7 GB streamed per GPU per step)",
                       "timing": f"{args.steps} steps in {len(region_ms)} region(s) of {region_steps} steps, each after a "
                                 f"reset of x and {warm} warm-up steps; CUDA events on the stepping stream; max over ranks",
                       "warmup_steps_per_region": warm,
                       "shard_build_s": t_build, "finite": finite,
                       "e2e_path": "per rank: host x[c0,c1) in, host y slice out through spmv_b200_csr_spmv_host "
                                   "(x upload, row-chunk kernels, y download pipelined on 3 streams)"},
            "hbm_gbs": bmin_total / (ms_step * 1e6),
            "regions_ms": region_ms,
            "region_steps": region_steps,
            "region_ms_by_rank": {"min": [min(r) for r in by_rank], "median": [statistics.median(r) for r in by_rank],
                                  "max": [max(r) for r in by_rank]},
            "roofline": {"bound": "hbm", "achieved": bmin_local / (kern_ms * 1e6), "peak": peak, "unit": "GB/s",
                         "frac": bmin_local / (kern_ms * 1e6) / peak,
                         "frac_of_8TBs": bmin_local / (kern_ms * 1e6) / 8000.0,
                         "traffic": ncu_traffic(args.workload if world == 1 else f"{args.workload}n{world}",
                                                "csr_stream_kernel"),
                         "peak_source": peak_src, "kernel_ms_mean": kern_ms, "algorithmic_bytes": bmin_local,
                         "from_step": bmin_total / world / (ms_step * 1e6) / peak,
                         "note": "rank 0 shard, all rows, no exchange, measured after the timed regions; "
                                 "from_step = B_min per GPU / ms_per_step"},
            "standalone_kernel_ms_by_rank": {"before_peer_mapping_mean": [a[0] for a in alone],
                                             "before_peer_mapping_min": [a[1] for a in alone],
                                             "after_run_mean": [a[2] for a in alone],
                                             "after_run_min": [a[3] for a in alone], "reps": reps_alone},
            "cpu_baseline": None,
            "e2e": dict(e2e_rec("pageable"), pinned=e2e_rec("pinned")),
            "gpu_launches": launches_per_step * args.steps,
            "library_launch_count": launches,
            "clocks": clocks,
            "parity": {"step1_vs_oracle": True, "worst_ratio_rank0": worst,
                       "rows_checked": "whole slab" if len(spans) == 1 else "first, middle and last two planes of every slab"},
            "device": sp.device_info()["name"],
        }
    it.close()
    shard.close()
    del xs, ys
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    dist.barrier()

    if rank == 0:
        progress("stand-alone kernel, parity and e2e done")
    # ---- N = 1 extras: CPU baseline (bounded sample), the single-GPU BASELINE configs, and the
    #      reference's own CUDA kernels on this GPU ----
    if rank == 0 and world == 1:
        if not args.no_cpu:
            planes = 16
            arrays = O.gen_stencil27_rows(nx, ny, nz, 0, planes * plane)
            xc = np.random.default_rng(0).uniform(0, 1, arrays[1])
            kind, best, variants, nthreads = cpu_reference_run(O, arrays, xc, steps=3, warmup=1, hll=False)
            line["cpu_baseline"] = {
                "value": variants[best]["gflops"], "unit": "GFLOP/s", "cores": variants[best]["cores"], "kind": kind,
                "variant": best, "host_cores": host_cores(),
                "sample": f"rows of the first {planes} of {nz} planes of the same stencil ({len(arrays[3]) / 1e6:.0f} M "
                          f"entries), 3 SpMV passes per OpenMP variant, median",
                "variants": variants, "host_threads": nthreads}
            del arrays
        want = args.configs == "all" or (args.configs == "auto" and args.workload == "c5")
        if want:
            line["configs"] = {}
            for wl in ("c2", "c1", "c3", "c4"):
                try:
                    line["configs"][wl] = single_config(sp, O, torch, wl, steps=args.steps, warmup=args.warmup,
                                                        wpb=args.wpb, with_cpu=not args.no_cpu)
                except SystemExit as e:     # a failed parity gate is reported, never hidden
                    line["configs"][wl] = {"error": str(e)}
                torch.cuda.empty_cache()
            ref_gpu = reference_gpu_rows("c2")
            if line["cpu_baseline"] is not None:
                line["cpu_baseline"]["reference_gpu_sm100a"] = {
                    "what": "the reference's own kernels (src/cuda_csr.cu, src/cuda_hll.cu) rebuilt for sm_100a, "
                            "on this GPU, C2 (128^3 stencil), one launch per call as the reference times it",
                    "rows": ref_gpu}
    if rank == 0:
        if y_dump is not None:
            dump_outputs(args.dump_outputs, {"y": y_dump})
        emit(line)
    dist.barrier()
    dist.destroy_process_group()
    return 0
