"""GPU tests of the resident-matrix API (include/spmv_b200.h): device layouts,
device-side generators and converters, row-range launches, the fused push
epilogue, and full-size (BASELINE configs[1]) parity + size-independent
properties."""
import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN_CASES, golden, golden_mtx

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


@pytest.mark.parametrize("case", GOLDEN_CASES)
def test_hll_device_layout_bit_exact(sp, O, torch, case):
    """What sits in HBM is the reference's device convention (src/cuda_hll.cu:173-195):
    column-major, stride 32, pads = previous column / 0 -- from either host layout and
    from the on-GPU CSR->HLL conversion."""
    g = golden(case)
    A = sp.io_load_csr(golden_mtx(case))
    want_hoff, want_ja, want_as = O.hll_device_layout(A.M, g["IRP"], g["JA"], g["AS"])
    built = [sp.HllDevice.from_host(sp.csr_to_hll(A, False)), sp.HllDevice.from_host(sp.csr_to_hll(A, True)),
             sp.CsrDevice.from_host(A).to_hll()]
    for h in built:
        hoff, ja, as_ = h.download()
        assert np.array_equal(hoff, want_hoff)
        assert np.array_equal(ja, want_ja)
        assert np.array_equal(as_.view(np.uint64), want_as.view(np.uint64))
        h.close()


def test_device_stencil_generator_matches_host(sp, torch):
    for (nx, ny, nz, z0, z1) in [(7, 5, 6, 0, 6), (9, 4, 8, 2, 5), (1, 1, 3, 0, 3), (5, 1, 1, 0, 1),
                                 (2, 2, 2, 0, 2), (16, 16, 9, 8, 9)]:
        plane = nx * ny
        want = sp.gen_stencil27_rows(nx, ny, nz, z0 * plane, z1 * plane)
        h = sp.CsrDevice.stencil27(nx, ny, nz, z0, z1)
        irp, ja, as_ = h.download()
        assert np.array_equal(irp, want.IRP.astype(np.int64))
        assert np.array_equal(ja, want.JA)
        assert np.array_equal(as_, want.AS)
        h.close()
    # column offset (shard with a halo): indices shift, nothing else
    nx, ny, nz = 6, 5, 7
    plane = nx * ny
    want = sp.gen_stencil27_rows(nx, ny, nz, 2 * plane, 5 * plane)
    h = sp.CsrDevice.stencil27(nx, ny, nz, 2, 5, col_offset=plane, n_local=5 * plane)
    _, ja, _ = h.download()
    assert np.array_equal(ja, want.JA - plane)
    h.close()


def test_row_range_launch_and_push(sp, O, torch):
    """spmv_rows on declared cut points == the same rows of a full spmv; the push epilogue
    mirrors the chosen rows into a second buffer (stand-in for a peer GPU's halo)."""
    A = sp.gen_stencil27(12, 10, 9)
    plane = 120
    cuts = [plane, A.M - plane]
    h = sp.CsrDevice.from_arrays(A.M, A.N, A.IRP, A.JA, A.AS, cuts=cuts)
    x = dev(torch, np.random.default_rng(0).uniform(-1, 1, A.N))
    y_full = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    for kernel in (2, 4, 0, 1):
        h.spmv(x, y_full, kernel=kernel)
        y = torch.full((A.M,), float("nan"), dtype=torch.float64, device="cuda")
        halo_lo = torch.zeros(plane, dtype=torch.float64, device="cuda")
        halo_hi = torch.zeros(plane, dtype=torch.float64, device="cuda")
        h.spmv(x, y, kernel=kernel, rows=(0, plane), push=[(0, plane, halo_lo.data_ptr())])
        h.spmv(x, y, kernel=kernel, rows=(A.M - plane, A.M),
               push=[(A.M - plane, A.M, halo_hi.data_ptr())])
        h.spmv(x, y, kernel=kernel, rows=(plane, A.M - plane))
        torch.cuda.synchronize()
        assert torch.equal(y, y_full)
        assert torch.equal(halo_lo, y_full[:plane]) and torch.equal(halo_hi, y_full[-plane:])
    with pytest.raises(RuntimeError, match="cut points"):
        h.spmv(x, y_full, rows=(5, 17))
    h.close()


def test_wide_offsets_path(sp, O, torch):
    """64-bit row offsets (shards beyond 2^31 entries) exercised on a small matrix."""
    A = sp.gen_ragged(4000, 200)
    irp64 = A.IRP.astype(np.int64)
    x = np.random.default_rng(1).uniform(-1, 1, A.N)
    y_ref = O.csr_spmv(A.M, A.IRP, A.JA, A.AS, x)
    bound = O.csr_abs_bound(A.M, A.IRP, A.JA, A.AS, x)
    sp.set_knob("force_wide", 1)
    try:
        h = sp.CsrDevice.from_arrays(A.M, A.N, irp64, A.JA, A.AS)
        hh = h.to_hll()
    finally:
        sp.set_knob("force_wide", 0)
    xd = dev(torch, x)
    y = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    for kernel in range(5):
        y.fill_(float("nan"))
        h.spmv(xd, y, kernel=kernel)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (kernel, worst)
    y.fill_(float("nan"))
    hh.spmv(xd, y, kernel=2)
    ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
    assert ok, ("hll from wide csr", worst)
    irp, ja, as_ = h.download()
    assert np.array_equal(irp, irp64) and np.array_equal(ja, A.JA)
    h.close()
    hh.close()


@pytest.fixture(scope="module")
def c2(sp):
    """BASELINE configs[1]: 3D 27-point stencil 128^3."""
    return sp.gen_stencil27(128, 128, 128)


def test_c2_full_size_parity(sp, O, torch, c2):
    A = c2
    assert (A.M, A.NZ) == (2097152, 55742968)
    x = np.random.default_rng(2).uniform(0, 1, A.N)
    y_ref = O.csr_spmv(A.M, A.IRP, A.JA, A.AS, x)
    if O.ref_available():
        _, y_refref = O.ref_csr_serial(O.RefCsr(A.M, A.N, A.IRP, A.JA, A.AS), x)
    bound = O.csr_abs_bound(A.M, A.IRP, A.JA, A.AS, x)
    h = sp.CsrDevice.from_host(A)
    hh = h.to_hll()
    xd = dev(torch, x)
    y = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    for kernel in (0, 1, 2, 4):
        y.fill_(float("nan"))
        h.spmv(xd, y, kernel=kernel, warps_per_block=8)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, ("csr", kernel, worst)
        if O.ref_available():
            ok, worst = O.check_tolerance(y.cpu().numpy(), y_refref, bound, TOL)
            assert ok, ("csr vs reference binary", kernel, worst)
    for kernel in (1, 2, 3):
        y.fill_(float("nan"))
        hh.spmv(xd, y, kernel=kernel, warps_per_block=4)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, ("hll", kernel, worst)
    # size-independent properties
    ones = torch.ones(A.N, dtype=torch.float64, device="cuda")
    h.spmv(ones, y, kernel=2)
    # interior rows of diag 26 / 26 neighbours -1 sum to 0; every row sum is 26 - (nnz_row - 1)
    rowsum = 27.0 - np.diff(A.IRP)
    assert np.array_equal(y.cpu().numpy(), rowsum)
    # linearity: A(2x + e) == 2 A x + A e, within tolerance
    y1 = torch.zeros_like(y)
    h.spmv(xd, y1, kernel=4)
    y2 = torch.zeros_like(y)
    h.spmv(2 * xd + ones, y2, kernel=4)
    resid = (y2 - (2 * y1 + y)).abs().cpu().numpy()
    assert (resid <= 4e-12 * (2 * bound + 52)).all()
    # CSR and HLL agree bit-for-bit in structure: same x, same y within tolerance
    y3 = torch.zeros_like(y)
    hh.spmv(xd, y3, kernel=2)
    ok, _ = O.check_tolerance(y3.cpu().numpy(), y1.cpu().numpy(), bound, 2 * TOL)
    assert ok
    h.close()
    hh.close()


def test_shard_with_column_offset_from_host_arrays(sp, O, torch):
    """A row slab uploaded with col_offset (how a rank holds its part of A): indices are stored
    relative to the local x slice [c0, c1), the result equals the same rows of the full product."""
    nx, ny, nz = 10, 9, 12
    plane = nx * ny
    full = sp.gen_stencil27(nx, ny, nz)
    x = np.random.default_rng(4).uniform(-1, 1, full.N)
    y_full = O.csr_spmv(full.M, full.IRP, full.JA, full.AS, x)
    bound = O.csr_abs_bound(full.M, full.IRP, full.JA, full.AS, x)
    z0, z1 = 4, 9
    r0, r1 = z0 * plane, z1 * plane
    c0, c1 = (z0 - 1) * plane, (z1 + 1) * plane
    part = sp.gen_stencil27_rows(nx, ny, nz, r0, r1)          # global column indices
    for wide in (0, 1):
        sp.set_knob("force_wide", wide)
        try:
            h = sp.CsrDevice.from_arrays(part.M, c1 - c0, part.IRP, part.JA, part.AS, col_offset=c0,
                                         cuts=[plane, part.M - plane])
        finally:
            sp.set_knob("force_wide", 0)
        _, ja_dev, _ = h.download()
        assert np.array_equal(ja_dev, part.JA - c0)
        xl = dev(torch, x[c0:c1])
        y = torch.full((part.M,), float("nan"), dtype=torch.float64, device="cuda")
        for kernel in (2, 4, 0, 1, 3):
            y.fill_(float("nan"))
            h.spmv(xl, y, kernel=kernel)
            ok, worst = O.check_tolerance(y.cpu().numpy(), y_full[r0:r1], bound[r0:r1], TOL)
            assert ok, (wide, kernel, worst)
        h.close()


# ----------------------------------------------------------------- SELL-P ------
def _sell_case(sp, name):
    if name == "ragged":
        return sp.gen_ragged(5000, 300)
    if name == "rmat":
        return sp.gen_rmat(13, 16)
    if name == "uniform":
        return sp.gen_uniform_random(20000, 32)
    return sp.gen_stencil27(20, 18, 11)


@pytest.mark.parametrize("name", ["ragged", "rmat", "uniform", "stencil"])
def test_sell_layout_bit_exact_and_parity(sp, O, torch, name):
    """Column-panelled, window-sorted slices (csrc/sell_kernels.cuh): what sits in HBM equals the
    oracle's independent restatement of the layout rule, for several panel counts / windows /
    long-row thresholds, from the CSR source; y is within the north-star tolerance from both the
    CSR and the HLL source."""
    A = _sell_case(sp, name)
    IRP, JA, AS = A.IRP.copy(), A.JA.copy(), A.AS.copy()
    x = np.random.default_rng(5).uniform(-1, 1, A.N)
    y_ref = O.csr_spmv(A.M, IRP, JA, AS, x)
    bound = O.csr_abs_bound(A.M, IRP, JA, AS, x)
    xd = dev(torch, x)
    y = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    try:
        sp.set_knob("sell", 1)
        for K, sigma, max_row in ((1, 64, 4096), (3, 256, 100), (4, 16384, 4096), (7, 32, 40)):
            sp.set_knob("sell_panels", K)
            sp.set_knob("sell_sigma", sigma)
            sp.set_knob("sell_max_row", max_row)
            h = sp.CsrDevice.from_host(A)
            info = h.sell_info(build=True)
            assert info["state"] == 1 and info["panels"] == K and info["sigma"] == sigma
            if A.M <= 6000:        # the numpy restatement is a per-row Python loop
                soff, perm, ja, as_ = h.sell_download()
                w_soff, w_perm, w_ja, w_as = O.sellp_layout(A.M, A.N, IRP, JA, AS, K, sigma, max_row)
                assert np.array_equal(soff, w_soff)
                assert np.array_equal(perm, w_perm)
                assert np.array_equal(ja, w_ja)
                assert np.array_equal(as_.view(np.uint64), w_as.view(np.uint64))
            assert info["long_rows"] == int((np.diff(IRP) > max_row).sum())
            for kernel in (2, 4):
                for wpb in (2, 8):
                    y.fill_(float("nan"))
                    h.spmv(xd, y, kernel=kernel, warps_per_block=wpb)
                    ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
                    assert ok, (name, "csr", K, sigma, max_row, kernel, wpb, worst)
            assert h.launches(2) >= K
            if max_row == 4096:
                hh = h.to_hll()
                y.fill_(float("nan"))
                hh.spmv(xd, y, kernel=2, warps_per_block=4)
                assert hh.sell_info()["state"] == 1 and hh.sell_info()["panels"] == K
                ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
                assert ok, (name, "hll", K, sigma, worst)
                hh.close()
            h.close()
    finally:
        for k, v in (("sell", -1), ("sell_panels", 0), ("sell_sigma", 16384), ("sell_max_row", 4096)):
            sp.set_knob(k, v)


@pytest.mark.parametrize("name", ["ragged", "rmat"])
def test_sell_virtual_rows_bit_exact_and_parity(sp, O, torch, name):
    """Ragged matrices: rows cut into virtual rows of `chunk` entries (no warp walks more than
    `chunk` steps; hub rows spread over many lanes; partial sums combined in piece order).  Layout
    bit-exact against the oracle's restatement, y within tolerance, and run-to-run identical."""
    A = _sell_case(sp, name)
    IRP, JA, AS = A.IRP.copy(), A.JA.copy(), A.AS.copy()
    x = np.random.default_rng(5).uniform(-1, 1, A.N)
    y_ref = O.csr_spmv(A.M, IRP, JA, AS, x)
    bound = O.csr_abs_bound(A.M, IRP, JA, AS, x)
    xd = dev(torch, x)
    y = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    try:
        sp.set_knob("sell", 1)        # "ragged" has 78 % of its rows in one length bin: force the route
        for chunk, sigma in ((64, 16384), (8, 256), (200, 32)):
            sp.set_knob("sell_chunk", chunk)
            sp.set_knob("sell_sigma", sigma)
            h = sp.CsrDevice.from_host(A)
            info = h.sell_info(build=True)
            assert info["state"] == 1 and info["panels"] == 1 and info["chunk"] == chunk
            lens = np.diff(IRP)
            assert info["split_rows"] == int((lens > chunk).sum())
            assert info["pieces"] == int(np.ceil(lens[lens > chunk] / chunk).sum())
            assert info["long_rows"] == 0
            if A.M <= 6000:
                soff, dest, ja, as_ = h.sell_download()
                w_soff, w_dest, w_ja, w_as, _, _ = O.sellv_layout(A.M, IRP, JA, AS, sigma, chunk)
                assert np.array_equal(soff, w_soff) and np.array_equal(dest, w_dest)
                assert np.array_equal(ja, w_ja) and np.array_equal(as_.view(np.uint64), w_as.view(np.uint64))
            outs = []
            for kernel, wpb in ((2, 4), (4, 8), (2, 4)):
                y.fill_(float("nan"))
                h.spmv(xd, y, kernel=kernel, warps_per_block=wpb)
                outs.append(y.cpu().numpy().copy())
                ok, worst = O.check_tolerance(outs[-1], y_ref, bound, TOL)
                assert ok, (name, chunk, sigma, kernel, worst)
            assert np.array_equal(outs[0], outs[2])       # deterministic: no atomics anywhere
            h.close()
    finally:
        sp.set_knob("sell", -1)
        sp.set_knob("sell_chunk", 256)
        sp.set_knob("sell_sigma", 16384)


def test_sell_auto_routing(sp, O, torch):
    """Who goes through SELL-P without a knob: ragged / power-law CSR (one panel while x fits
    the L2); regular rows stay on the staged kernel; and the host half of the plan (row order and
    slice offsets) is a pure function of the per-panel row counts."""
    R = sp.CsrDevice.from_host(sp.gen_rmat(14, 16))
    S = sp.CsrDevice.from_host(sp.gen_stencil27(24, 24, 24))
    x = torch.ones(R.N, dtype=torch.float64, device="cuda")
    y = torch.zeros(R.M, dtype=torch.float64, device="cuda")
    R.spmv(x, y, kernel=2)
    assert R.sell_info()["state"] == 1 and R.sell_info()["panels"] == 1
    xs = torch.ones(S.N, dtype=torch.float64, device="cuda")
    ys = torch.zeros(S.M, dtype=torch.float64, device="cuda")
    S.spmv(xs, ys, kernel=2)
    assert S.sell_info()["state"] == 0
    assert S.sell_info()["gather_span_ppm"] < 300000 and R.sell_info()["gather_span_ppm"] > 500000
    R.close()
    S.close()


# ------------------------------------------------------- fused iteration step ------
@pytest.mark.parametrize("name", ["stencil", "poisson", "rmat_sell"])
def test_fused_axpby_dot(sp, O, torch, name):
    """y = alpha A x + beta z and dot = sum y*w in ONE pass over the matrix
    (spmv_b200_{csr,hll}_spmv_fused): equals the unfused sequence, and the dot product is
    bit-reproducible from run to run (fixed reduction order)."""
    A = {"stencil": lambda: sp.gen_stencil27(30, 28, 26), "poisson": lambda: sp.gen_poisson2d(300, 200),
         "rmat_sell": lambda: sp.gen_rmat(13, 8)}[name]()
    rng = np.random.default_rng(6)
    x, z, w = (rng.uniform(-1, 1, n) for n in (A.N, A.M, A.M))
    alpha, beta = 0.75, -1.25
    IRP, JA, AS = A.IRP.copy(), A.JA.copy(), A.AS.copy()
    ax = O.csr_spmv(A.M, IRP, JA, AS, x)
    bound = O.csr_abs_bound(A.M, IRP, JA, AS, x)
    want = alpha * ax + beta * z
    lim = abs(alpha) * bound + abs(beta * z) * 4 * np.finfo(float).eps / 1e-12
    try:
        if name == "rmat_sell":
            sp.set_knob("sell_chunk", 1 << 20)       # no row is split into pieces: fused is allowed
        h = sp.CsrDevice.from_host(A)
        handles = [("csr", h, (2, 4))]
        if name != "rmat_sell":
            handles.append(("hll", h.to_hll(), (2,)))
        xd, zd, wd = dev(torch, x), dev(torch, z), dev(torch, w)
        for fmt, hd, kernels in handles:
            for kernel in kernels:
                y = torch.full((A.M,), float("nan"), dtype=torch.float64, device="cuda")
                dot = torch.zeros(1, dtype=torch.float64, device="cuda")
                hd.spmv_fused(xd, y, alpha, beta, zd, wd, dot, kernel=kernel)
                yh = y.cpu().numpy()
                ok, worst = O.check_tolerance(yh, want, lim, TOL)
                assert ok, (fmt, kernel, worst)
                d0 = float(dot.item())
                assert abs(d0 - float(yh @ w)) <= 1e-10 * float(np.abs(yh * w).sum())
                hd.spmv_fused(xd, y, alpha, beta, zd, wd, dot, kernel=kernel)
                assert float(dot.item()) == d0                       # bit-reproducible
                # ||y||^2 with w = y, no z
                hd.spmv_fused(xd, y, 1.0, 0.0, None, y, dot, kernel=kernel)
                yh = y.cpu().numpy()
                assert abs(float(dot.item()) - float(yh @ yh)) <= 1e-10 * float(yh @ yh)
                ok, worst = O.check_tolerance(yh, ax, bound, TOL)
                assert ok, (fmt, kernel, "plain", worst)
        for _, hd, _ in handles:
            hd.close()
    finally:
        sp.set_knob("sell_chunk", 256)


def test_hll_pipelined_narrow_hacks(sp, O, torch):
    """HLL id 2 on narrow hacks: persistent warps, each with its own ring of bulk-copied hacks
    (hll_pipe_kernel).  Same y as the reference serial CSR with empty hacks, hacks of different
    widths, fewer hacks than warps, hack ranges (the host-buffer pipeline's launches), the fused
    epilogue; matrices with a wider hack stay on the warp-per-hack kernel."""
    rng = np.random.default_rng(21)
    cases = []
    for M in (32 * 211 + 13, 32 * 9000 + 5, 40):
        N = 5000
        lens = rng.integers(0, 9, M)
        lens[32 * 40:32 * 44] = 0                             # four empty hacks
        lens[32 * 100:32 * 101] = 1
        IRP = np.zeros(M + 1, np.int32)
        IRP[1:] = np.cumsum(lens)
        JA = np.concatenate([np.sort(rng.choice(N, l, replace=False)) for l in lens] + [np.zeros(0, np.int64)]).astype(np.int32)
        AS = rng.uniform(-1, 1, JA.size)
        cases.append((f"narrow{M}", sp.csr_from_arrays("narrow", M, N, IRP, JA, AS)))
    cases += [("poisson", sp.gen_poisson2d(640, 333)), ("stencil27", sp.gen_stencil27(14, 13, 12))]
    try:
        for name, A in cases:
            irp, ja, as_ = A.IRP.copy(), A.JA.copy(), A.AS.copy()
            x = rng.uniform(-1, 1, A.N)
            y_ref = O.csr_spmv(A.M, irp, ja, as_, x)
            bound = O.csr_abs_bound(A.M, irp, ja, as_, x)
            xd = dev(torch, x)
            got = {}
            for pipe in (0, 1, -1):
                sp.set_knob("hll_pipe", pipe)
                for h in (sp.CsrDevice.from_host(A).to_hll(), sp.HllDevice.from_host(sp.csr_to_hll(A, True))):
                    y = torch.full((A.M,), float("nan"), dtype=torch.float64, device="cuda")
                    h.spmv(xd, y, kernel=2, warps_per_block=4)
                    got[pipe] = y.cpu().numpy()
                    ok, worst = O.check_tolerance(got[pipe], y_ref, bound, TOL)
                    assert ok, (name, pipe, worst)
                    yh = np.full(A.M, np.nan)
                    h.spmv_host(x, yh, kernel=2)              # launches on hack ranges
                    ok, worst = O.check_tolerance(yh, y_ref, bound, TOL)
                    assert ok, (name, pipe, "host", worst)
                    dot = torch.zeros(1, dtype=torch.float64, device="cuda")
                    h.spmv_fused(xd, y, 2.0, 0.0, None, y, dot, kernel=2)
                    assert np.array_equal(y.cpu().numpy(), 2.0 * got[pipe])
                    h.close()
            # lane = row and the same summation order in both kernels: bit-identical
            assert np.array_equal(got[0], got[1])
    finally:
        sp.set_knob("hll_pipe", -1)


def test_csr_pipelined_short_rows(sp, O, torch):
    """CSR ids 2 / 4 on short rows (<= 8 entries): persistent warps with private rings of bulk-copied
    row groups (csr_pipe_kernel).  Same y as the reference serial CSR with empty rows, a ragged last
    group, row-range launches on cut handles, 64-bit row offsets and the host-buffer pass."""
    rng = np.random.default_rng(22)
    cases = []
    for M in (32 * 211 + 13, 32 * 9000 + 5, 7):
        N = 5000
        lens = rng.integers(0, 9, M)
        lens[32 * 40:32 * 44] = 0
        IRP = np.zeros(M + 1, np.int32)
        IRP[1:] = np.cumsum(lens)
        JA = np.concatenate([np.sort(rng.choice(N, l, replace=False)) for l in lens] + [np.zeros(0, np.int64)]).astype(np.int32)
        cases.append((M, N, IRP, JA, rng.uniform(-1, 1, JA.size)))
    P = sp.gen_poisson2d(640, 333)
    cases.append((P.M, P.N, P.IRP.copy(), P.JA.copy(), P.AS.copy()))
    try:
        for M, N, IRP, JA, AS in cases:
            x = rng.uniform(-1, 1, N)
            y_ref = O.csr_spmv(M, IRP, JA, AS, x)
            bound = O.csr_abs_bound(M, IRP, JA, AS, x)
            xd = dev(torch, x)
            cut = (M // 3) // 32 * 32 + 5
            for pipe in (1, -1, 0):
                sp.set_knob("csr_pipe", pipe)
                for wide in (0, 1):
                    sp.set_knob("force_wide", wide)
                    h = sp.CsrDevice.from_arrays(M, N, IRP.astype(np.int64) if wide else IRP, JA, AS,
                                                 cuts=(cut,) if M > 100 else ())
                    sp.set_knob("force_wide", 0)
                    for kernel in (2, 4):
                        y = torch.full((M,), float("nan"), dtype=torch.float64, device="cuda")
                        h.spmv(xd, y, kernel=kernel)
                        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
                        assert ok, (M, pipe, wide, kernel, worst)
                    if M > 100:                               # the two segments one after the other
                        y = torch.full((M,), float("nan"), dtype=torch.float64, device="cuda")
                        h.spmv(xd, y, kernel=2, rows=(cut, M))
                        assert torch.isnan(y[:cut]).all()
                        h.spmv(xd, y, kernel=2, rows=(0, cut))
                        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
                        assert ok, (M, pipe, wide, "ranges", worst)
                    yh = np.full(M, np.nan)
                    h.spmv_host(x, yh, kernel=2)
                    ok, worst = O.check_tolerance(yh, y_ref, bound, TOL)
                    assert ok, (M, pipe, wide, "host", worst)
                    h.close()
    finally:
        sp.set_knob("csr_pipe", -1)
        sp.set_knob("force_wide", 0)


@pytest.mark.parametrize("name", ["stencil", "poisson", "rmat", "ragged", "uniform_panels", "wide"])
def test_spmm_matches_k_spmvs(sp, O, torch, name):
    """Y = A X for 2 and 4 right-hand sides in one pass (spmv_b200_csr_spmm, SURVEY 8(f)3): every
    column equals the reference serial CSR product with that column, on every route -- rows straight
    from CSR, virtual rows with split pieces, column panels with accumulation, 64-bit offsets."""
    make = {"stencil": lambda: sp.gen_stencil27(20, 18, 16), "poisson": lambda: sp.gen_poisson2d(150, 90),
            "rmat": lambda: sp.gen_rmat(14, 12), "ragged": lambda: sp.gen_ragged(6000, 700),
            "uniform_panels": lambda: sp.gen_uniform_random(30000, 24), "wide": lambda: sp.gen_ragged(3000, 90)}
    A = make[name]()
    IRP, JA, AS = A.IRP.copy(), A.JA.copy(), A.AS.copy()
    rng = np.random.default_rng(31)
    try:
        if name == "uniform_panels":
            sp.set_knob("sell_panels", 3)
        if name == "wide":
            sp.set_knob("force_wide", 1)
            h = sp.CsrDevice.from_arrays(A.M, A.N, IRP.astype(np.int64), JA, AS)
            sp.set_knob("force_wide", 0)
        else:
            h = sp.CsrDevice.from_host(A)
        for k in (2, 4):
            Xh = rng.uniform(-1, 1, (A.N, k))
            X = torch.from_numpy(Xh).cuda()
            Y = torch.full((A.M, k), float("nan"), dtype=torch.float64, device="cuda")
            h.spmm(X, Y)
            Yh = Y.cpu().numpy()
            for j in range(k):
                xj = np.ascontiguousarray(Xh[:, j])
                ok, worst = O.check_tolerance(np.ascontiguousarray(Yh[:, j]), O.csr_spmv(A.M, IRP, JA, AS, xj),
                                              O.csr_abs_bound(A.M, IRP, JA, AS, xj), TOL)
                assert ok, (name, k, j, worst)
            h.spmm(X, Y)                                   # run to run identical (no atomics anywhere)
            assert np.array_equal(Y.cpu().numpy(), Yh)
        with pytest.raises(RuntimeError):
            h.spmm(torch.zeros((A.N, 3), dtype=torch.float64, device="cuda"),
                   torch.zeros((A.M, 3), dtype=torch.float64, device="cuda"))
        h.close()
    finally:
        sp.set_knob("sell_panels", 0)
        sp.set_knob("force_wide", 0)


def test_spmm_builds_its_own_panels_when_x_outgrows_the_l2(sp, O, torch):
    """Column panels are sized for the x they keep in the L2; k right-hand sides make x k times as
    large, so SpMM on a scattered matrix with a large x runs on a slice plan of its own (more
    panels, accumulation across them) -- the C3 case at a tenth of its size."""
    A = sp.gen_uniform_random(14_000_000, 4)
    IRP, JA, AS = A.IRP.copy(), A.JA.copy(), A.AS.copy()
    h = sp.CsrDevice.from_host(A)
    assert h.sell_info(build=True)["panels"] == 2                 # x = 112 MB: two panels for SpMV
    rng = np.random.default_rng(33)
    for k in (2, 4):
        Xh = rng.uniform(-1, 1, (A.N, k))
        X = torch.from_numpy(Xh).cuda()
        Y = torch.full((A.M, k), float("nan"), dtype=torch.float64, device="cuda")
        h.spmm(X, Y)
        Yh = Y.cpu().numpy()
        for j in (0, k - 1):
            xj = np.ascontiguousarray(Xh[:, j])
            ok, worst = O.check_tolerance(np.ascontiguousarray(Yh[:, j]), O.csr_spmv(A.M, IRP, JA, AS, xj),
                                          O.csr_abs_bound(A.M, IRP, JA, AS, xj), TOL)
            assert ok, (k, j, worst)
    h.close()


def test_handle_host_spmv(sp, O, torch):
    """spmv_b200_{csr,hll}_spmv_host on resident handles, including a generated-in-HBM stencil
    (no host copy of the matrix: the chunk plan comes from device reductions), pinned and
    pageable buffers."""
    nx, ny, nz = 48, 48, 64
    h = sp.CsrDevice.stencil27(nx, ny, nz)
    hh = h.to_hll()
    A = sp.gen_stencil27(nx, ny, nz)
    x = np.random.default_rng(7).uniform(-1, 1, A.N)
    y_ref = O.csr_spmv(A.M, A.IRP, A.JA, A.AS, x)
    bound = O.csr_abs_bound(A.M, A.IRP, A.JA, A.AS, x)
    xp, yp = sp.pinned_empty(A.N), sp.pinned_empty(A.M)
    xp[:] = x
    for xb, yb in ((xp, yp), (x.copy(), np.zeros(A.M))):
        for hd, kernels in ((h, (4, 2, 1)), (hh, (2, 3))):
            for kernel in kernels:
                yb[:] = np.nan
                ms = hd.spmv_host(xb, yb, kernel=kernel)
                assert ms > 0
                ok, worst = O.check_tolerance(yb, y_ref, bound, TOL)
                assert ok, (type(hd).__name__, kernel, worst)
    sp.pinned_free(xp)
    sp.pinned_free(yp)
    h.close()
    hh.close()
    sp.release_all()


# --------------------------------------- full-size parity: BASELINE configs[2], [3] ------
def _full_size(sp, O, torch, A, kernels_csr, hll, label):
    x = np.random.default_rng(2).uniform(0, 1, A.N)
    IRP, JA, AS = A.IRP, A.JA, A.AS
    if O.ref_available():          # the reference's own serial CSR (oracle/_ref)
        _, y_ref = O.ref_csr_serial(O.RefCsr(A.M, A.N, IRP, JA, AS), x)
    else:
        y_ref = O.csr_spmv(A.M, IRP, JA, AS, x)
    bound = O.csr_abs_bound(A.M, IRP, JA, AS, x)
    h = sp.CsrDevice.from_host(A)
    xd = dev(torch, x)
    y = torch.zeros(A.M, dtype=torch.float64, device="cuda")
    for kernel in kernels_csr:
        y.fill_(float("nan"))
        h.spmv(xd, y, kernel=kernel, warps_per_block=8)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (label, "csr", kernel, worst)
    # size-independent property: row sums (x = 1) equal the sums of the stored values
    ones = torch.ones(A.N, dtype=torch.float64, device="cuda")
    h.spmv(ones, y, kernel=2)
    cs = np.concatenate([[0.0], np.cumsum(AS)])
    rowsum = cs[IRP[1:]] - cs[IRP[:-1]]
    absum = O.csr_abs_bound(A.M, IRP, JA, AS, np.ones(A.N))
    assert (np.abs(y.cpu().numpy() - rowsum) <= 1e-9 * np.maximum(absum, 1.0)).all()
    if hll:
        hh = h.to_hll()
        y.fill_(float("nan"))
        hh.spmv(xd, y, kernel=2, warps_per_block=8)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (label, "hll", worst)
        hh.close()
    info = h.sell_info()
    h.close()
    return info


def test_c3_full_size_parity(sp, O, torch):
    """BASELINE configs[2]: uniform random n = 16 M, 32 per row (512 M entries), CSR ids 2 / 4 and
    HLL id 2 against the reference's serial CSR.  x (128 MB) does not fit the L2: the library must
    have chosen column panels on its own."""
    A = sp.gen_uniform_random(16000000, 32, 42)
    assert (A.M, A.NZ) == (16000000, 512000000)
    info = _full_size(sp, O, torch, A, (2, 4), True, "c3")
    assert info["state"] == 1 and info["panels"] > 1


def test_c4_full_size_parity(sp, O, torch):
    """BASELINE configs[3]: R-MAT scale 24, 16 edges per vertex (268 M entries, duplicates kept),
    CSR ids 2 / 4 against the reference's serial CSR."""
    A = sp.gen_rmat(24, 16)
    assert (A.M, A.NZ) == (1 << 24, 1 << 28)
    info = _full_size(sp, O, torch, A, (2, 4), False, "c4")
    assert info["state"] == 1


def test_bad_column_indices_are_refused(sp, torch):
    """A shard whose stored columns fall outside its x slice would gather out of bounds: creation
    fails with -ERANGE instead (round-1 advisor finding)."""
    A = sp.gen_poisson2d(30, 30)
    with pytest.raises(RuntimeError, match="column indices span"):
        sp.CsrDevice.from_arrays(A.M, A.N - 5, A.IRP, A.JA, A.AS)          # x slice too short
    with pytest.raises(RuntimeError, match="column indices span"):
        sp.CsrDevice.from_arrays(A.M, A.N, A.IRP, A.JA, A.AS, col_offset=7)  # negative local columns
    sp.CsrDevice.from_arrays(A.M, A.N, A.IRP, A.JA, A.AS).close()
