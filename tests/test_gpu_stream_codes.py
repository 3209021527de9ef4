"""GPU tests of the column codes of the staged CSR kernel (csr_stream_kernel with CODES).

A coded plan streams one byte per entry and a per-tile dictionary of column offsets in place of the
int32 column indices.  The decoded column is the stored one and the summation order is unchanged,
so every y must be bit-identical to the int32 path (knob csr_codes = 0), on every route that
launches the row-tile configurations: plain, push-shaped and fused epilogues, both offset widths,
handles built by transpose() and from_coo(), and the 2-GPU iterated SpMV."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-12
WPBS = (2, 4, 8)   # stream configurations 10, 12 and 13 for rows of >= 12 entries


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture
def knobs(sp):
    """Sets knobs for one test and puts every one it touched back to its default."""
    defaults = {"csr_codes": 1, "force_wide": 0, "sell": -1}
    touched = set()

    def set_(key, value):
        touched.add(key)
        sp.set_knob(key, value)
    yield set_
    for key in touched:
        sp.set_knob(key, defaults[key])


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


def oracle_check(O, H, x, y):
    irp, ja, as_ = H.download()
    irp32 = irp.astype(np.int32)
    y_ref = O.csr_spmv(H.M, irp32, ja, as_, x)
    bound = O.csr_abs_bound(H.M, irp32, ja, as_, x)
    ok, worst = O.check_tolerance(y, y_ref, bound, TOL)
    assert ok, worst


def run_both(knobs, torch, f):
    """f() once with int32 columns and once with codes; returns both results as numpy."""
    out = []
    for codes in (0, 1):
        knobs("csr_codes", codes)
        r = f()
        torch.cuda.synchronize()
        out.append(r)
    return out


def assert_same(a, b):
    assert np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))


def check_handle(O, torch, knobs, H, x, kernels=(2, 4), expect_state=1):
    xd = dev(torch, x)
    for kernel in kernels:
        for wpb in WPBS:
            y = torch.empty(H.M, dtype=torch.float64, device="cuda")

            def f():
                y.fill_(float("nan"))
                H.spmv(xd, y, kernel=kernel, warps_per_block=wpb)
                return y.cpu().numpy()
            y_int, y_code = run_both(knobs, torch, f)
            assert_same(y_int, y_code)
            oracle_check(O, H, x, y_code)
    info = H.codes_info()
    assert info["state"] == expect_state, info
    return info


@pytest.mark.parametrize("wide", [0, 1])
def test_stencil_bit_identical(sp, O, torch, knobs, wide):
    knobs("force_wide", wide)
    H = sp.CsrDevice.stencil27(40, 36, 30)
    x = np.random.default_rng(1).uniform(-1, 1, H.N)
    info = check_handle(O, torch, knobs, H, x)
    assert 0 < info["max_dict"] <= 27 and info["tiles"] > 0
    # one plan per configuration of WPBS, each one byte per entry plus the dictionaries
    plans = len(WPBS)
    assert plans * H.NZ <= info["bytes"] <= plans * H.NZ + info["tiles"] * (16 + 27 * 4 + 16)
    del H
    sp.release_all()


def test_shard_plain_and_push(sp, O, torch, knobs):
    """A shard cut into three segments, each run alone, with and without a push epilogue into a
    buffer on the same GPU."""
    A = sp.gen_stencil27(24, 20, 36)
    M = A.M
    cuts = (M // 3, 2 * M // 3)
    H = sp.CsrDevice.from_arrays(M, A.N, A.IRP.copy(), A.JA.copy(), A.AS.copy(), cuts=cuts)
    x = np.random.default_rng(2).uniform(-1, 1, A.N)
    xd = dev(torch, x)
    bounds = (0,) + cuts + (M,)
    for kernel in (2, 4):
        y = torch.empty(M, dtype=torch.float64, device="cuda")
        halo = torch.empty(M, dtype=torch.float64, device="cuda")

        def f():
            y.fill_(float("nan"))
            halo.fill_(float("nan"))
            for s in range(3):
                r0, r1 = bounds[s], bounds[s + 1]
                if s == 1:   # push the first 100 rows of the middle segment
                    H.spmv(xd, y, kernel=kernel, rows=(r0, r1), push=[(r0, r0 + 100, halo.data_ptr())])
                else:
                    H.spmv(xd, y, kernel=kernel, rows=(r0, r1))
            return y.cpu().numpy(), halo[:100].cpu().numpy()
        (y_int, h_int), (y_code, h_code) = run_both(knobs, torch, f)
        assert_same(y_int, y_code)
        assert_same(h_int, h_code)
        assert_same(h_code, y_code[bounds[1]:bounds[1] + 100])
        oracle_check(O, H, x, y_code)
    assert H.codes_info()["state"] == 1
    del H
    sp.release_all()


def test_fused_step(sp, O, torch, knobs):
    H = sp.CsrDevice.stencil27(32, 32, 32)
    rng = np.random.default_rng(3)
    x, z, w = (rng.uniform(-1, 1, H.M) for _ in range(3))
    xd, zd, wd = dev(torch, x), dev(torch, z), dev(torch, w)
    for kernel in (2, 4):
        y = torch.empty(H.M, dtype=torch.float64, device="cuda")
        dot = torch.empty(1, dtype=torch.float64, device="cuda")

        def f():
            y.fill_(float("nan"))
            H.spmv_fused(xd, y, alpha=0.5, beta=-2.0, z=zd, w=wd, dot=dot, kernel=kernel)
            return y.cpu().numpy(), dot.cpu().numpy()
        (y_int, d_int), (y_code, d_code) = run_both(knobs, torch, f)
        assert_same(y_int, y_code)
        # the dot adds per-warp partials whose grouping follows the launch grid, and the two kernel
        # bodies may fit a different number of CTAs on an SM: equal within rounding, not bitwise
        assert abs(d_code[0] - d_int[0]) <= 1e-12 * np.dot(np.abs(y_code), np.abs(w))
        irp, ja, as_ = H.download()
        ax = O.csr_spmv(H.M, irp.astype(np.int32), ja, as_, x)
        want = 0.5 * ax - 2.0 * z
        bound = O.csr_abs_bound(H.M, irp.astype(np.int32), ja, as_, x) + 2.0 * np.abs(z)
        ok, worst = O.check_tolerance(y_code, want, bound, TOL)
        assert ok, worst
        assert abs(d_code[0] - np.dot(want, w)) <= 1e-10 * np.dot(np.abs(want), np.abs(w))
    assert H.codes_info()["state"] == 1
    del H
    sp.release_all()


def test_transpose_and_coo(sp, O, torch, knobs):
    A = sp.CsrDevice.stencil27(30, 28, 26)
    T = A.transpose()
    x = np.random.default_rng(4).uniform(-1, 1, A.N)
    check_handle(O, torch, knobs, T, x)
    irp, ja, as_ = A.download()
    rows = np.repeat(np.arange(A.M, dtype=np.int64), np.diff(irp))
    perm = np.random.default_rng(5).permutation(len(ja))   # triplets in any order
    C = sp.CsrDevice.from_coo(A.M, A.N, torch.from_numpy(rows[perm]).cuda(),
                              torch.from_numpy(ja[perm].astype(np.int64)).cuda(), dev(torch, as_[perm]))
    check_handle(O, torch, knobs, C, x)
    del A, T, C
    sp.release_all()


def csr_of_rows(rows, rng):
    """CSR arrays (int32 offsets) of a list of sorted column arrays, random values."""
    IRP = np.zeros(len(rows) + 1, np.int64)
    IRP[1:] = np.cumsum([len(r) for r in rows])
    JA = np.concatenate(rows).astype(np.int32)
    return IRP.astype(np.int32), JA, rng.uniform(-1, 1, len(JA))


def band_rows(M, offsets):
    """Row i holds the columns i + d, d in `offsets`, that fall inside [0, M)."""
    offsets = np.sort(np.asarray(offsets))
    return [(i + offsets)[(i + offsets >= 0) & (i + offsets < M)] for i in range(M)]


def test_wide_dictionaries_and_long_rows(sp, O, torch, knobs):
    """Dictionaries of 28 to 256 offsets (a band of 200 irregular diagonals), and a coded plan
    whose tiles include rows longer than a stage: those go to the long-row kernels, their tiles
    carry no code block."""
    rng = np.random.default_rng(8)
    M = 30000
    diags = rng.choice(np.arange(-4000, 4001), size=200, replace=False)
    rows = band_rows(M, diags)
    for r in (5000, 17000, 25000):   # 9 000-entry rows: beyond every stage (CAP <= 8 192)
        rows[r] = np.arange(r - 4500, r + 4500)
    IRP, JA, AS = csr_of_rows(rows, rng)
    H = sp.CsrDevice.from_arrays(M, M, IRP, JA, AS)
    x = rng.uniform(-1, 1, M)
    info = check_handle(O, torch, knobs, H, x)
    assert 28 <= info["max_dict"] <= 200, info
    del H
    sp.release_all()


def test_one_wide_tile_keeps_int32(sp, O, torch, knobs):
    """A banded matrix (16 diagonals) with one run of 300 rows whose columns are scattered: only
    the tiles over those rows exceed 256 offsets, and the whole plan keeps its int32 columns."""
    rng = np.random.default_rng(9)
    M = 20000
    rows = band_rows(M, np.arange(-8, 8))
    for r in range(9000, 9300):
        rows[r] = np.sort(rng.choice(M, size=16, replace=False))
    IRP, JA, AS = csr_of_rows(rows, rng)
    H = sp.CsrDevice.from_arrays(M, M, IRP, JA, AS)
    x = rng.uniform(-1, 1, M)
    info = check_handle(O, torch, knobs, H, x, expect_state=-1)
    assert info["tiles"] == 0 and info["bytes"] == 0
    del H
    sp.release_all()


def test_scattered_columns_keep_int32(sp, O, torch, knobs):
    """Regular rows whose columns are scattered over the whole (L2-sized) x: a tile has far more
    than 256 distinct offsets, so the plan keeps its int32 columns."""
    rng = np.random.default_rng(6)
    M, L = 20000, 16
    IRP = np.arange(0, (M + 1) * L, L, dtype=np.int32)
    JA = np.sort(rng.integers(0, M, size=(M, L)), axis=1).astype(np.int32).ravel()
    AS = rng.uniform(-1, 1, M * L)
    H = sp.CsrDevice.from_arrays(M, M, IRP, JA, AS)
    x = rng.uniform(-1, 1, M)
    info = check_handle(O, torch, knobs, H, x, expect_state=-1)
    assert info["tiles"] == 0 and info["bytes"] == 0
    del H
    sp.release_all()


def test_two_gpu_iterated(sp, O, torch, knobs):
    """The 2-GPU iterated SpMV of a stencil: boundary segments push, interior ones store, both
    coded; the graph-captured steps run the plans built by the eager ones."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from spmv_scpa_b200 import dist as D
    nx, ny, nz = 24, 22, 30
    x0 = np.random.default_rng(7).uniform(-1, 1, nx * ny * nz)
    out = []
    for codes in (0, 1):
        knobs("csr_codes", codes)
        g = D.DistGroup.stencil27(nx, ny, nz, 2)
        g.set_x(x0)
        g.iterate(4)
        out.append(g.get_x().copy())
        assert g.mode() == "push"
        g.close()
    assert_same(out[0], out[1])
    S = sp.gen_stencil27(nx, ny, nz)
    x, bound = x0.copy(), None
    for _ in range(4):
        bound = O.csr_abs_bound(S.M, S.IRP, S.JA, S.AS, np.abs(x))
        x = O.csr_spmv(S.M, S.IRP, S.JA, S.AS, x)
    ok, worst = O.check_tolerance(out[1], x, bound * 4, TOL)
    assert ok, worst
    sp.release_all()


def test_build_and_destroy_returns_memory(sp, torch, knobs):
    x = torch.ones(64 * 64 * 48, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)

    def once():
        H = sp.CsrDevice.stencil27(64, 64, 48)
        H.spmv(x, y, kernel=4)
        torch.cuda.synchronize()
        assert H.codes_info()["state"] == 1
        del H
    once()   # first use: module loading, cached workspaces
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(20):
        once()
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info()[0]
    assert abs(free0 - free1) <= 2 << 20, (free0, free1)
    sp.release_all()
