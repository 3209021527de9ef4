"""GPU tests of spmv_b200_csr_transpose / CsrDevice.transpose(): Aᵀ of a resident CSR built in HBM.

The layout is exact -- a stable sort of A's entries by column, duplicates and explicit zeros kept,
values copied -- so it is compared bit for bit with two independent host oracles.  Products on
Aᵀ are compared with the oracle port's serial CSR on the oracle's transposed arrays."""
import numpy as np
import pytest
import scipy.sparse

from conftest import GOLDEN_CASES, golden, random_csr

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


def oracle_transpose(M, N, IRP, JA, AS):
    """(t_IRP int64, t_JA int32, t_AS) of Aᵀ: a stable sort of the entries by column."""
    IRP = np.asarray(IRP, np.int64)
    JA = np.asarray(JA, np.int32)
    AS = np.asarray(AS, np.float64)
    row_of = np.repeat(np.arange(M, dtype=np.int32), np.diff(IRP))
    o = np.argsort(JA, kind="stable")
    t_irp = np.zeros(N + 1, np.int64)
    t_irp[1:] = np.cumsum(np.bincount(JA, minlength=N))
    return t_irp, row_of[o], AS[o]


def scipy_transpose(M, N, IRP, JA, AS):
    T = scipy.sparse.csr_matrix((np.asarray(AS, np.float64), np.asarray(JA), np.asarray(IRP)),
                                shape=(M, N)).T.tocsr()
    return T.indptr.astype(np.int64), T.indices.astype(np.int32), T.data


def assert_layout(T, want):
    irp, ja, as_ = T.download()
    assert np.array_equal(irp, want[0])
    assert np.array_equal(ja, want[1])
    assert np.array_equal(as_.view(np.uint64), np.asarray(want[2], np.float64).view(np.uint64))


def check_spmv(O, torch, T, t, x, kernels=(0, 1, 2, 3, 4), label=""):
    """T.spmv with each CSR kernel id against the oracle port on the oracle's arrays t."""
    irp32 = t[0].astype(np.int32)
    y_ref = O.csr_spmv(T.M, irp32, t[1], t[2], x)
    bound = O.csr_abs_bound(T.M, irp32, t[1], t[2], x)
    xd = dev(torch, x)
    y = torch.zeros(T.M, dtype=torch.float64, device="cuda")
    for kernel in kernels:
        y.fill_(float("nan"))
        T.spmv(xd, y, kernel=kernel)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (label, "csr", kernel, worst)
    return y_ref, bound


def _case(sp, name):
    """(M, N, IRP, JA, AS) of a named test matrix."""
    rng = np.random.default_rng(41)
    if name in GOLDEN_CASES:
        g = golden(name)
        return int(g["M"]), int(g["N"]), g["IRP"], g["JA"], g["AS"]
    if name == "random":                       # unsorted rows, duplicates, empty rows
        return (700, 900) + random_csr(rng, 700, 900, 40)
    if name == "empty_cols":                   # most columns empty: empty rows of Aᵀ
        IRP, JA, AS = random_csr(rng, 60, 2000, 12)
        return (60, 2000, IRP, JA, AS)
    if name == "one_row":
        return (1, 500) + random_csr(rng, 1, 500, 300, empty_frac=0.0)
    if name == "one_col":
        IRP, JA, AS = random_csr(rng, 500, 1, 3)
        return (500, 1, IRP, JA, AS)
    A = {"ragged": lambda: sp.gen_ragged(3000, 400), "rmat": lambda: sp.gen_rmat(12, 16),
         "uniform": lambda: sp.gen_uniform_random(5000, 16)}[name]()
    return A.M, A.N, A.IRP.copy(), A.JA.copy(), A.AS.copy()


LAYOUT_CASES = GOLDEN_CASES + ["random", "empty_cols", "one_row", "one_col", "ragged", "rmat", "uniform"]


@pytest.mark.parametrize("case", LAYOUT_CASES)
def test_transpose_layout_and_parity(sp, O, torch, have_ref, case):
    """download() of Aᵀ equals the stable-sort oracle (and scipy's .T.tocsr(), which the oracle
    must agree with); every CSR kernel id and every HLL id on Aᵀ matches the serial CSR product."""
    M, N, IRP, JA, AS = _case(sp, case)
    want = oracle_transpose(M, N, IRP, JA, AS)
    other = scipy_transpose(M, N, IRP, JA, AS)
    for a, b in zip(want, other):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b, a.dtype).view(np.uint8))
    A = sp.CsrDevice.from_arrays(M, N, np.asarray(IRP, np.int32), JA, AS)
    T = A.transpose()
    assert (T.M, T.N, T.NZ) == (A.N, A.M, A.NZ)
    assert_layout(T, want)
    x = np.random.default_rng(3).uniform(-1, 1, T.N)
    y_ref, bound = check_spmv(O, torch, T, want, x, label=case)
    if have_ref:
        _, y_refref = O.ref_csr_serial(O.RefCsr(T.M, T.N, want[0].astype(np.int32), want[1], want[2]), x)
        ok, worst = O.check_tolerance(y_ref, y_refref, bound, TOL)
        assert ok, (case, "oracle port vs reference", worst)
    H = T.to_hll()
    y = torch.zeros(T.M, dtype=torch.float64, device="cuda")
    for kernel in range(4):
        y.fill_(float("nan"))
        H.spmv(dev(torch, x), y, kernel=kernel)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (case, "hll", kernel, worst)
    H.close()
    T.close()
    A.close()


def test_transpose_routes(sp, O, torch):
    """Aᵀ is planned from its own row profile: the R-MAT hub column becomes a long row split into
    virtual-row pieces; a scattered matrix runs column panels; the 5-point stencil takes the
    short-row ring; fused step and SpMM on Aᵀ match the unfused product and the oracle."""
    rng = np.random.default_rng(43)
    # virtual rows with split pieces, chosen without a knob
    R = sp.gen_rmat(14, 16)
    t = oracle_transpose(R.M, R.N, R.IRP, R.JA, R.AS)
    A = sp.CsrDevice.from_host(R)
    T = A.transpose()
    check_spmv(O, torch, T, t, rng.uniform(-1, 1, T.N), kernels=(2, 4), label="rmat")
    info = T.sell_info()
    assert info["state"] == 1 and info["chunk"] > 0 and info["split_rows"] > 0
    assert info["split_rows"] == int((np.diff(t[0]) > info["chunk"]).sum())
    T.close()
    A.close()

    # column panels (knob), SpMM with 2 and 4 right-hand sides across them
    U = sp.gen_uniform_random(30000, 24)
    t = oracle_transpose(U.M, U.N, U.IRP, U.JA, U.AS)
    A = sp.CsrDevice.from_host(U)
    try:
        sp.set_knob("sell_panels", 3)
        T = A.transpose()
        check_spmv(O, torch, T, t, rng.uniform(-1, 1, T.N), kernels=(2, 4), label="panels")
        assert T.sell_info()["state"] == 1 and T.sell_info()["panels"] == 3
        irp32 = t[0].astype(np.int32)
        for k in (2, 4):
            Xh = rng.uniform(-1, 1, (T.N, k))
            Y = torch.full((T.M, k), float("nan"), dtype=torch.float64, device="cuda")
            T.spmm(torch.from_numpy(Xh).cuda(), Y)
            Yh = Y.cpu().numpy()
            y1 = torch.zeros(T.M, dtype=torch.float64, device="cuda")
            for j in range(k):
                xj = np.ascontiguousarray(Xh[:, j])
                ok, worst = O.check_tolerance(np.ascontiguousarray(Yh[:, j]), O.csr_spmv(T.M, irp32, t[1], t[2], xj),
                                              O.csr_abs_bound(T.M, irp32, t[1], t[2], xj), TOL)
                assert ok, ("spmm", k, j, worst)
                T.spmv(dev(torch, xj), y1, kernel=2)
                ok, worst = O.check_tolerance(np.ascontiguousarray(Yh[:, j]), y1.cpu().numpy(),
                                              O.csr_abs_bound(T.M, irp32, t[1], t[2], xj), 2 * TOL)
                assert ok, ("spmm vs spmv", k, j, worst)
        T.close()
    finally:
        sp.set_knob("sell_panels", 0)
    A.close()

    # short rows: the per-warp ring (forced, and the automatic choice)
    P = sp.gen_poisson2d(640, 333)
    t = oracle_transpose(P.M, P.N, P.IRP, P.JA, P.AS)
    A = sp.CsrDevice.from_host(P)
    try:
        for pipe in (1, -1):
            sp.set_knob("csr_pipe", pipe)
            T = A.transpose()
            check_spmv(O, torch, T, t, rng.uniform(-1, 1, T.N), kernels=(2, 4), label=("pipe", pipe))
            T.close()
    finally:
        sp.set_knob("csr_pipe", -1)
    A.close()

    # fused step on the transpose of a non-symmetric matrix
    M, N = 3000, 2000
    IRP, JA, AS = random_csr(rng, M, N, 12)
    t = oracle_transpose(M, N, IRP, JA, AS)
    A = sp.CsrDevice.from_arrays(M, N, IRP, JA, AS)
    T = A.transpose()
    x, z, w = rng.uniform(-1, 1, T.N), rng.uniform(-1, 1, T.M), rng.uniform(-1, 1, T.M)
    ax, bound = check_spmv(O, torch, T, t, x, kernels=(2,), label="fused")
    alpha, beta = 0.5, -2.0
    lim = abs(alpha) * bound + abs(beta * z) * 4 * np.finfo(float).eps / TOL
    xd, zd, wd = dev(torch, x), dev(torch, z), dev(torch, w)
    for kernel in (2, 4):
        y_plain = torch.zeros(T.M, dtype=torch.float64, device="cuda")
        T.spmv(xd, y_plain, kernel=kernel)
        y = torch.full((T.M,), float("nan"), dtype=torch.float64, device="cuda")
        dot = torch.zeros(1, dtype=torch.float64, device="cuda")
        T.spmv_fused(xd, y, alpha, beta, zd, wd, dot, kernel=kernel)
        yh = y.cpu().numpy()
        ok, worst = O.check_tolerance(yh, alpha * ax + beta * z, lim, TOL)
        assert ok, ("fused", kernel, worst)
        ok, worst = O.check_tolerance(yh, alpha * y_plain.cpu().numpy() + beta * z, lim, TOL)
        assert ok, ("fused vs unfused", kernel, worst)
        assert abs(float(dot.item()) - float(yh @ w)) <= 1e-10 * float(np.abs(yh * w).sum())
    T.close()
    A.close()


def test_transpose_of_symmetric_input_is_itself(sp, torch):
    """The device-generated 27-point stencil and the 5-point stencil equal their transposes bit for
    bit."""
    for A in (sp.CsrDevice.stencil27(14, 12, 11), sp.CsrDevice.from_host(sp.gen_poisson2d(90, 70))):
        T = A.transpose()
        assert (T.M, T.N, T.NZ) == (A.M, A.N, A.NZ)
        for a, b in zip(A.download(), T.download()):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
        T.close()
        A.close()


def test_transpose_twice(sp, torch):
    """transpose(transpose(A)) is A with every row stably sorted by column; for column-sorted
    generators that is A bit for bit."""
    rng = np.random.default_rng(44)
    M, N = 800, 600
    IRP, JA, AS = random_csr(rng, M, N, 30)
    row_of = np.repeat(np.arange(M), np.diff(IRP))
    o = np.lexsort((JA, row_of))
    A = sp.CsrDevice.from_arrays(M, N, IRP, JA, AS)
    T = A.transpose()
    TT = T.transpose()
    assert (TT.M, TT.N) == (M, N)
    assert_layout(TT, (IRP.astype(np.int64), JA[o], AS[o]))
    for H in (A, T, TT):
        H.close()
    for host in (sp.gen_uniform_random(4000, 9), sp.gen_ragged(2000, 100)):
        A = sp.CsrDevice.from_host(host)
        T = A.transpose()
        TT = T.transpose()
        for a, b in zip(A.download(), TT.download()):
            assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
        for H in (A, T, TT):
            H.close()


def test_transpose_wide_offsets(sp, O, torch):
    """64-bit row offsets on either side: every combination of a narrow or wide input handle with
    a narrow or wide result."""
    R = sp.gen_ragged(4000, 200)
    IRP, JA, AS = R.IRP.copy(), R.JA.copy(), R.AS.copy()
    t = oracle_transpose(R.M, R.N, IRP, JA, AS)
    x = np.random.default_rng(45).uniform(-1, 1, R.M)
    try:
        for wide_in in (0, 1):
            sp.set_knob("force_wide", wide_in)
            A = sp.CsrDevice.from_arrays(R.M, R.N, IRP.astype(np.int64) if wide_in else IRP, JA, AS)
            for wide_out in (0, 1):
                sp.set_knob("force_wide", wide_out)
                T = A.transpose()
                sp.set_knob("force_wide", 0)
                assert_layout(T, t)
                check_spmv(O, torch, T, t, x, label=("wide", wide_in, wide_out))
                T.close()
            A.close()
    finally:
        sp.set_knob("force_wide", 0)


def test_transpose_of_a_shard(sp, O, torch):
    """A handle created with col_offset and cuts transposes its local block: n_local rows, the
    shard's rows as columns, no cuts."""
    nx, ny, nz = 10, 9, 12
    plane = nx * ny
    z0, z1 = 4, 9
    r0, r1 = z0 * plane, z1 * plane
    c0, c1 = (z0 - 1) * plane, (z1 + 1) * plane
    part = sp.gen_stencil27_rows(nx, ny, nz, r0, r1)
    local_ja = part.JA - c0
    t = oracle_transpose(part.M, c1 - c0, part.IRP, local_ja, part.AS)
    for h in (sp.CsrDevice.from_arrays(part.M, c1 - c0, part.IRP, part.JA, part.AS, col_offset=c0,
                                       cuts=[plane, part.M - plane]),
              sp.CsrDevice.stencil27(nx, ny, nz, z0, z1, col_offset=c0, n_local=c1 - c0,
                                     cuts=[plane, part.M - plane])):
        T = h.transpose()
        assert (T.M, T.N, T.NZ) == (c1 - c0, part.M, part.NZ)
        assert_layout(T, t)
        x = np.random.default_rng(46).uniform(-1, 1, T.N)
        check_spmv(O, torch, T, t, x, label="shard")
        y = torch.zeros(T.M, dtype=torch.float64, device="cuda")
        with pytest.raises(RuntimeError, match="cut points"):
            T.spmv(dev(torch, x), y, rows=(plane, T.M - plane))
        T.close()
        h.close()


def test_transpose_leaves_a_alone_and_is_deterministic(sp, O, torch):
    """A is unchanged and still multiplies correctly; two transposes are bit-identical; Aᵀ
    outlives A."""
    rng = np.random.default_rng(47)
    M, N = 5000, 3000
    IRP, JA, AS = random_csr(rng, M, N, 60)
    t = oracle_transpose(M, N, IRP, JA, AS)
    A = sp.CsrDevice.from_arrays(M, N, IRP, JA, AS)
    before = A.download()
    T1, T2 = A.transpose(), A.transpose()
    for a, b in zip(before, A.download()):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    x = rng.uniform(-1, 1, N)
    y_ref = O.csr_spmv(M, IRP, JA, AS, x)
    bound = O.csr_abs_bound(M, IRP, JA, AS, x)
    y = torch.zeros(M, dtype=torch.float64, device="cuda")
    A.spmv(dev(torch, x), y, kernel=2)
    ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
    assert ok, worst
    for a, b in zip(T1.download(), T2.download()):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    A.close()
    T2.close()
    assert_layout(T1, t)
    check_spmv(O, torch, T1, t, rng.uniform(-1, 1, T1.N), kernels=(2, 4), label="after destroy")
    T1.close()


def test_transpose_null_handle(sp, torch):
    A = sp.CsrDevice.from_host(sp.gen_poisson2d(10, 10))
    A.close()
    with pytest.raises(RuntimeError, match="null CSR handle"):
        A.transpose()


def test_c4_transpose_full_size(sp, O, torch):
    """BASELINE configs[3] transposed: R-MAT scale 24, 16 edges per vertex (268 M entries,
    duplicates kept).  Layout against scipy, CSR ids 2 / 4 against the oracle port."""
    R = sp.gen_rmat(24, 16)
    assert (R.M, R.NZ) == (1 << 24, 1 << 28)
    t = scipy_transpose(R.M, R.N, R.IRP, R.JA, R.AS)
    A = sp.CsrDevice.from_host(R)
    T = A.transpose()
    A.close()
    assert_layout(T, t)
    irp32 = t[0].astype(np.int32)
    x = np.random.default_rng(2).uniform(0, 1, T.N)
    if O.ref_available():
        _, y_ref = O.ref_csr_serial(O.RefCsr(T.M, T.N, irp32, t[1], t[2]), x)
    else:
        y_ref = O.csr_spmv(T.M, irp32, t[1], t[2], x)
    bound = O.csr_abs_bound(T.M, irp32, t[1], t[2], x)
    xd = dev(torch, x)
    y = torch.zeros(T.M, dtype=torch.float64, device="cuda")
    for kernel in (2, 4):
        y.fill_(float("nan"))
        T.spmv(xd, y, kernel=kernel, warps_per_block=8)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, ("c4ᵀ", kernel, worst)
    assert T.sell_info()["state"] == 1
    T.close()
