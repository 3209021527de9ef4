"""bench.py prints ONE JSON line with the keys the driver reads (reference arm on CPU here,
the B200 arm under -m gpu)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True,
                       text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines          # ONE line on stdout, whatever the libraries print
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--workload", "tiny", "--steps", "3", "--warmup", "1")
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["unit"] == "GFLOP/s" and d["dtype"] == "f64"
    assert d["vs_baseline"] is None and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_times_every_step(tmp_path):
    """--steps K times exactly K passes of every variant (no cap), and --dump-outputs writes y of
    the headline variant: A x for x as bench.py draws it."""
    d = run_bench("--impl", "reference", "--workload", "tiny", "--steps", "12", "--warmup", "1",
                  "--dump-outputs", str(tmp_path))
    assert d["steps"] == 12
    variants = d["cpu_baseline"]["variants"]
    assert {"serial", "omp_guided"} <= set(variants)
    assert all(v["steps"] == 12 for v in variants.values())
    from oracle import oracle as O
    M, N, IRP, JA, AS = O.gen_stencil27(32, 32, 32)
    x = np.random.default_rng(0).uniform(0, 1, N)
    y = np.load(tmp_path / "y.npy")
    assert y.dtype == np.float64 and y.shape == (M,)
    assert O.check_tolerance(y, O.csr_spmv(M, IRP, JA, AS, x), O.csr_abs_bound(M, IRP, JA, AS, x), 1e-12)[0]


@pytest.mark.gpu
def test_b200_arm_line(tmp_path):
    d = run_bench("--workload", "tiny", "--steps", "5", "--warmup", "3", "--dump-outputs", str(tmp_path))
    assert BASE_KEYS | {"roofline", "gpu_launches", "clocks"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["value"] > 0
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and rf["peak"] > 1000
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert d["gpu_launches"] >= d["steps"]
    e = d["e2e"]                            # headline: pageable caller buffers; pinned as a sub-key
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 8 * d["config"]["cols"] and e["d2h_bytes_per_step"] == 8 * d["config"]["rows"]
    assert e["value"] < d["value"]            # the host round trip cannot be free
    assert e["pinned"]["value"] > 0 and e["pinned"]["h2d_bytes_per_step"] == 8 * d["config"]["cols"]
    assert d["cpu_baseline"]["value"] > 0
    assert d["config"]["parity"]["csr"]["ok"] and d["config"]["parity"]["hll"]["ok"]
    assert "sm_mhz" in d["clocks"] and isinstance(d["clocks"]["reasons"], list)
    # --dump-outputs: y = A x of the last timed step, every row (32^3 < 2^21), x as bench.py draws it
    from oracle import oracle as O
    M, N, IRP, JA, AS = O.gen_stencil27(32, 32, 32)
    x = np.random.default_rng(0).uniform(0, 1, N)
    y = np.load(tmp_path / "y.npy")
    assert y.dtype == np.float64 and y.shape == (M,)
    assert O.check_tolerance(y, O.csr_spmv(M, IRP, JA, AS, x), O.csr_abs_bound(M, IRP, JA, AS, x), 1e-12)[0]


@pytest.mark.gpu
def test_b200_default_path_line(tmp_path):
    """The default path (bench_dist, one rank = one GPU) on the small slab workload: strong/weak
    flag, K timed steps cut into regions, stand-alone kernel before and after, both e2e variants."""
    d = run_bench("--workload", "c2w", "--steps", "4", "--warmup", "3", "--regions", "3", "--configs", "none",
                  "--no-cpu", "--dump-outputs", str(tmp_path))
    assert BASE_KEYS | {"roofline", "gpu_launches", "clocks", "regions_ms"} <= set(d)
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and len(d["regions_ms"]) == 3
    assert d["config"]["nnz"] == 55742968 and d["config"]["cuda_graph"] is True and d["config"]["finite"]
    assert d["region_steps"] == [1, 1, 2]
    assert abs(d["ms_per_step"] * 4 - sum(d["regions_ms"])) < 1e-9
    assert 0.3 < d["roofline"]["frac"] < 1.2
    assert d["e2e"]["value"] > 0 and d["e2e"]["pinned"]["value"] >= 0.5 * d["e2e"]["value"]
    assert d["parity"]["step1_vs_oracle"] is True
    assert len(d["standalone_kernel_ms_by_rank"]["after_run_mean"]) == 1
    # --dump-outputs: x after the last region = A^(w+2) x_0 (w warm-up steps after the reset, then its
    # 2 timed steps), every row (128^3 = 2^21)
    from bench_dist import x0_slice
    from oracle import oracle as O
    M, N, IRP, JA, AS = O.gen_stencil27(128, 128, 128)
    steps = d["config"]["warmup_steps_per_region"] + 2
    x = x0_slice(0, N)
    for _ in range(steps):
        bound = O.csr_abs_bound(M, IRP, JA, AS, np.abs(x))
        x = O.csr_spmv(M, IRP, JA, AS, x)
    y = np.load(tmp_path / "y.npy")
    assert y.dtype == np.float64 and y.shape == (M,)
    assert O.check_tolerance(y, x, steps * bound, 1e-12)[0]


def test_reference_arm_under_torchrun_env():
    """N>1: rank 0 alone prints the line, the other ranks exit 0 without work; torchrun's
    OMP_NUM_THREADS=1 must not make the reference's OpenMP code run on one core."""
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29555",
               OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--workload", "tiny", "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
    env["RANK"] = "0"
    env["LOCAL_RANK"] = "0"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--workload", "tiny", "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
    cores = len(os.sched_getaffinity(0))
    assert d["cpu_baseline"]["host_cores"] == cores
    if cores > 1:
        assert d["cpu_baseline"]["variants"]["omp_guided"]["cores"] == cores
        assert d["cpu_baseline"]["cores"] >= 1


def test_reference_arm_maps_no_product_library():
    """The CPU arm is the reference's code only: neither libspmv_b200 nor libspmv_host may be
    mapped into its process (round-1 verdict: the arm generated its matrix with the product)."""
    code = ("import sys, runpy\n"
            "sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'tiny', '--steps', '2', '--warmup', '1']\n"
            "try:\n    runpy.run_path(%r, run_name='__main__')\nexcept SystemExit:\n    pass\n"
            "print('MAPS', sorted({l.split()[-1] for l in open('/proc/self/maps') if '.so' in l and %r in l}))\n"
            ) % (os.path.join(ROOT, "bench.py"), ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-1500:]
    maps = [l for l in r.stdout.splitlines() if l.startswith("MAPS")][0]
    assert "libspmv_b200" not in maps and "libspmv_host" not in maps, maps
    assert "oracle" in maps
