"""Tests of spmv_b200_csr_from_coo / CsrDevice.from_coo / CsrDevice.from_torch: resident CSR built
in HBM from COO triplets already in device memory.

The layout is exact -- a stable sort of the entries by (row, col); with sum_duplicates, each run of
equal (row, col) added left to right in input order starting from its first value -- so it is
compared bit for bit with a numpy oracle.  The oracle itself is cross-checked against scipy's
coo_matrix(...).tocsr() without a GPU.  Products on the built handles are compared with the oracle
port's serial CSR on the oracle's arrays."""
import numpy as np
import pytest
import scipy.sparse

from conftest import GOLDEN_CASES, golden, random_csr

gpu = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


def oracle_coo(M, N, row, col, val, sum_dup):
    """(IRP int64, JA int32, AS) of the CSR built from COO triplets: np.lexsort (stable) by
    (row, col); with sum_dup each run of equal (row, col) becomes one entry, its values added left
    to right from the first one."""
    row = np.asarray(row, np.int64)
    col = np.asarray(col, np.int64)
    val = np.asarray(val, np.float64)
    o = np.lexsort((col, row))
    r, c, v = row[o], col[o], val[o]
    if sum_dup and len(o):
        head = np.ones(len(o), bool)
        head[1:] = (r[1:] != r[:-1]) | (c[1:] != c[:-1])
        start = np.flatnonzero(head)
        lens = np.diff(np.append(start, len(o)))
        acc = v[start].copy()
        act = np.arange(len(start))
        for j in range(1, int(lens.max())):
            act = act[lens[act] > j]
            acc[act] += v[start[act] + j]
        r, c, v = r[start], c[start], acc
    irp = np.zeros(M + 1, np.int64)
    irp[1:] = np.cumsum(np.bincount(r, minlength=M))
    return irp, c.astype(np.int32), v


def assert_layout(H, want):
    irp, ja, as_ = H.download()
    assert np.array_equal(irp, want[0])
    assert np.array_equal(ja, want[1])
    assert np.array_equal(as_.view(np.uint64), np.asarray(want[2], np.float64).view(np.uint64))


def same_bytes(A, B):
    for a, b in zip(A.download(), B.download()):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def check_spmv(O, torch, H, t, x, kernels=(0, 1, 2, 3, 4), hll=True, label=""):
    """H.spmv with each CSR kernel id (and each HLL id through to_hll()) against the oracle port on
    the oracle's arrays t."""
    irp32 = t[0].astype(np.int32)
    y_ref = O.csr_spmv(H.M, irp32, t[1], t[2], x)
    bound = O.csr_abs_bound(H.M, irp32, t[1], t[2], x)
    xd = dev(torch, x)
    y = torch.zeros(H.M, dtype=torch.float64, device="cuda")
    for kernel in kernels:
        y.fill_(float("nan"))
        H.spmv(xd, y, kernel=kernel)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (label, "csr", kernel, worst)
    if hll:
        Hh = H.to_hll()
        for kernel in range(4):
            y.fill_(float("nan"))
            Hh.spmv(xd, y, kernel=kernel)
            ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
            assert ok, (label, "hll", kernel, worst)
        Hh.close()


def csr_to_coo(IRP, JA, AS):
    IRP = np.asarray(IRP, np.int64)
    row = np.repeat(np.arange(len(IRP) - 1, dtype=np.int64), np.diff(IRP))
    return row, np.asarray(JA, np.int64), np.asarray(AS, np.float64)


def shuffled(rng, row, col, val):
    p = rng.permutation(len(row))
    return row[p], col[p], val[p]


def random_coo(rng, M, N, n, rows=None, cols=None):
    """n entries over a subset of `rows` x `cols` (all by default): many duplicates when the subset
    is small; values include explicit zeros and -0.0."""
    rs = np.arange(M) if rows is None else rng.choice(M, rows, replace=False)
    cs = np.arange(N) if cols is None else rng.choice(N, cols, replace=False)
    row = rs[rng.integers(0, len(rs), n)].astype(np.int64)
    col = cs[rng.integers(0, len(cs), n)].astype(np.int64)
    val = rng.uniform(-1, 1, n)
    val[rng.random(n) < 0.05] = 0.0
    val[rng.random(n) < 0.05] = -0.0
    return row, col, val


def _case(sp, name):
    """(M, N, row, col, val) of a named COO input."""
    rng = np.random.default_rng(51)
    if name in GOLDEN_CASES:
        g = golden(name)
        return (int(g["M"]), int(g["N"])) + shuffled(rng, *csr_to_coo(g["IRP"], g["JA"], g["AS"]))
    if name == "dups":                       # many repeated (row, col), zeros and -0.0
        return (300, 200) + random_coo(rng, 300, 200, 20000, rows=40, cols=30)
    if name == "empty_rows_cols":            # entries in 50 rows and 40 columns only
        return (1000, 3000) + random_coo(rng, 1000, 3000, 4000, rows=50, cols=40)
    if name == "one_row":
        return (1, 500) + random_coo(rng, 1, 500, 900)
    if name == "one_col":
        return (500, 1) + random_coo(rng, 500, 1, 900)
    if name == "one_by_one":                 # every entry a duplicate of the first
        return (1, 1) + random_coo(rng, 1, 1, 50)
    if name == "no_entries":
        return (7, 5, np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0))
    if name == "wide":                       # rectangular, 32-bit keys
        return (100, 100000) + random_coo(rng, 100, 100000, 30000)
    if name == "tall":
        return (200000, 30) + random_coo(rng, 200000, 30, 30000)
    if name == "wide_keys":                  # 17 + 17 key bits: 64-bit keys
        return (100000, 80000) + random_coo(rng, 100000, 80000, 60000, rows=3000, cols=2000)
    A = {"ragged": lambda: sp.gen_ragged(3000, 400), "rmat": lambda: sp.gen_rmat(12, 16),
         "uniform": lambda: sp.gen_uniform_random(5000, 16)}[name]()
    return (A.M, A.N) + shuffled(rng, *csr_to_coo(A.IRP, A.JA, A.AS))


LAYOUT_CASES = GOLDEN_CASES + ["dups", "empty_rows_cols", "one_row", "one_col", "one_by_one", "no_entries",
                               "wide", "tall", "wide_keys", "ragged", "rmat", "uniform"]


def build(sp, torch, M, N, row, col, val, sum_dup=False, idx=np.int64, stream=None):
    return sp.CsrDevice.from_coo(M, N, torch.from_numpy(np.asarray(row, idx)).cuda(),
                                 torch.from_numpy(np.asarray(col, idx)).cuda(), dev(torch, val),
                                 sum_duplicates=sum_dup, stream=stream)


@gpu
@pytest.mark.parametrize("case", LAYOUT_CASES)
def test_from_coo_layout_and_parity(sp, O, torch, case):
    """download() equals the oracle bit for bit in both modes and with both index widths; every
    CSR kernel id and every HLL id on the result matches the serial CSR product."""
    M, N, row, col, val = _case(sp, case)
    for sum_dup in (False, True):
        want = oracle_coo(M, N, row, col, val, sum_dup)
        for idx in (np.int32, np.int64):
            H = build(sp, torch, M, N, row, col, val, sum_dup, idx)
            assert (H.M, H.N, H.NZ) == (M, N, len(want[1]))
            assert_layout(H, want)
            if idx == np.int64:
                x = np.random.default_rng(3).uniform(-1, 1, N)
                check_spmv(O, torch, H, want, x, label=(case, sum_dup))
            H.close()


@pytest.mark.parametrize("dups", [False, True])
def test_oracle_matches_scipy(dups):
    """CPU only: the oracle against scipy's coo_matrix(...).tocsr() -- bit for bit without
    duplicates (either mode), within 1e-12 of the summed magnitudes where runs are added."""
    rng = np.random.default_rng(52)
    M, N = 400, 300
    if dups:
        row, col, val = random_coo(rng, M, N, 30000, rows=60, cols=50)
    else:
        k = rng.choice(M * N, 20000, replace=False)
        row, col = k // N, k % N
        val = rng.uniform(-1, 1, len(k))
    S = scipy.sparse.coo_matrix((val, (row, col)), shape=(M, N)).tocsr()
    S.sort_indices()
    got = oracle_coo(M, N, row, col, val, True)
    assert np.array_equal(got[0], S.indptr.astype(np.int64))
    assert np.array_equal(got[1], S.indices.astype(np.int32))
    if dups:
        mag = scipy.sparse.coo_matrix((np.abs(val), (row, col)), shape=(M, N)).tocsr()
        mag.sort_indices()
        assert np.all(np.abs(got[2] - S.data) <= 1e-12 * mag.data)
    else:
        assert np.array_equal(got[2].view(np.uint64), S.data.view(np.uint64))
        keep = oracle_coo(M, N, row, col, val, False)
        for a, b in zip(keep, got):
            assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


@gpu
def test_equals_host_path(sp, torch):
    """A host CSR with sorted columns fed in its own order (duplicates adjacent, kept) builds the
    same bytes as from_arrays; so does the same matrix without duplicates fed shuffled."""
    rng = np.random.default_rng(53)
    M, N = 2000, 1500
    IRP, JA, AS = random_csr(rng, M, N, 30, sort=True)
    A = sp.CsrDevice.from_arrays(M, N, IRP, JA, AS)
    H = build(sp, torch, M, N, *csr_to_coo(IRP, JA, AS))
    same_bytes(H, A)
    H.close()
    A.close()
    row, col, val = csr_to_coo(IRP, JA, AS)
    first = np.ones(len(row), bool)
    first[1:] = (row[1:] != row[:-1]) | (col[1:] != col[:-1])
    row, col, val = row[first], col[first], val[first]
    IRP = np.zeros(M + 1, np.int32)
    IRP[1:] = np.cumsum(np.bincount(row, minlength=M))
    A = sp.CsrDevice.from_arrays(M, N, IRP, col.astype(np.int32), val)
    H = build(sp, torch, M, N, *shuffled(rng, row, col, val))
    same_bytes(H, A)
    H.close()
    A.close()


@gpu
def test_equals_transpose(sp, torch):
    """Unsorted CSR with duplicates: from_coo(row=JA, col=row of each entry) equals
    from_arrays(...).transpose() bit for bit."""
    rng = np.random.default_rng(54)
    M, N = 900, 1200
    IRP, JA, AS = random_csr(rng, M, N, 40)
    A = sp.CsrDevice.from_arrays(M, N, IRP, JA, AS)
    T = A.transpose()
    row_of, _, _ = csr_to_coo(IRP, JA, AS)
    for idx in (np.int32, np.int64):
        H = build(sp, torch, N, M, JA, row_of, AS, idx=idx)
        same_bytes(H, T)
        H.close()
    T.close()
    A.close()


@gpu
def test_sorted_input_skips_the_sort(sp, torch):
    """Input already in (row, col) order builds the same bytes as the same entries shuffled, with
    fewer launches."""
    rng = np.random.default_rng(55)
    U = sp.gen_uniform_random(20000, 12)
    row, col, val = csr_to_coo(U.IRP, U.JA, U.AS)
    o = np.lexsort((col, row))
    first = np.ones(len(o), bool)
    first[1:] = (row[o][1:] != row[o][:-1]) | (col[o][1:] != col[o][:-1])
    row, col, val = row[o][first], col[o][first], val[o][first]
    args = [torch.from_numpy(row).cuda(), torch.from_numpy(col).cuda(), dev(torch, val)]
    r, c, v = shuffled(rng, row, col, val)
    sargs = [torch.from_numpy(r).cuda(), torch.from_numpy(c).cuda(), dev(torch, v)]
    for sum_dup in (False, True):
        l0 = sp.counters()["launches"]
        S = sp.CsrDevice.from_coo(U.M, U.N, *args, sum_duplicates=sum_dup)
        l1 = sp.counters()["launches"]
        H = sp.CsrDevice.from_coo(U.M, U.N, *sargs, sum_duplicates=sum_dup)
        l2 = sp.counters()["launches"]
        same_bytes(S, H)
        assert l1 - l0 < l2 - l1, (l1 - l0, l2 - l1)
        S.close()
        H.close()


@gpu
def test_long_run_is_summed_in_order(sp, torch):
    """One (row, col) repeated 2^17 times among other entries is added left to right exactly as
    the oracle adds it."""
    rng = np.random.default_rng(56)
    M, N = 5000, 4000
    row, col, val = random_coo(rng, M, N, 200000)
    run = 1 << 17
    pos = np.sort(rng.choice(len(row) + run, run, replace=False))
    mask = np.zeros(len(row) + run, bool)
    mask[pos] = True
    R, Cc, V = (np.empty(len(mask), np.int64), np.empty(len(mask), np.int64), np.empty(len(mask)))
    R[mask], Cc[mask], V[mask] = 1234, 777, rng.uniform(-1, 1, run) * 10.0 ** rng.integers(-8, 8, run)
    R[~mask], Cc[~mask], V[~mask] = row, col, val
    want = oracle_coo(M, N, R, Cc, V, True)
    H = build(sp, torch, M, N, R, Cc, V, True)
    assert_layout(H, want)
    H.close()


@gpu
def test_deterministic_and_independent_of_inputs(sp, O, torch):
    """Two builds are bit-identical; the handle outlives the caller's tensors, which are deleted
    and their memory overwritten after the build."""
    rng = np.random.default_rng(57)
    M, N = 3000, 2500
    row, col, val = random_coo(rng, M, N, 300000, rows=800, cols=600)
    for sum_dup in (False, True):
        want = oracle_coo(M, N, row, col, val, sum_dup)
        r, c, v = torch.from_numpy(row).cuda(), torch.from_numpy(col).cuda(), dev(torch, val)
        A = sp.CsrDevice.from_coo(M, N, r, c, v, sum_duplicates=sum_dup)
        B = sp.CsrDevice.from_coo(M, N, r, c, v, sum_duplicates=sum_dup)
        same_bytes(A, B)
        B.close()
        del r, c, v
        junk = [torch.full((len(row),), -7, dtype=torch.int64, device="cuda") for _ in range(2)]
        junk.append(torch.full((len(row),), float("nan"), dtype=torch.float64, device="cuda"))
        torch.cuda.synchronize()
        assert_layout(A, want)
        check_spmv(O, torch, A, want, rng.uniform(-1, 1, N), kernels=(2, 4), hll=False, label="after del")
        del junk
        A.close()


@gpu
def test_stream_ordering(sp, torch):
    """Inputs written on a side stream, built with stream= that stream and no host sync between:
    the build sees the written values."""
    rng = np.random.default_rng(58)
    M, N = 4000, 3000
    row, col, val = random_coo(rng, M, N, 500000)
    want = oracle_coo(M, N, row, col, val, True)
    src = [torch.from_numpy(row).cuda(), torch.from_numpy(col).cuda(), dev(torch, val)]
    dst = [torch.full_like(src[0], -1), torch.full_like(src[1], -1), torch.full_like(src[2], float("nan"))]
    big = torch.rand(4096, 4096, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            big = big @ big / 4096.0  # keeps the side stream busy before the writes
        for d, s in zip(dst, src):
            d.copy_(s)
    H = sp.CsrDevice.from_coo(M, N, *dst, sum_duplicates=True, stream=side)
    assert_layout(H, want)
    H.close()


@gpu
def test_wide_offsets(sp, O, torch):
    """force_wide gives 64-bit row offsets with the same layout and parity."""
    M, N, row, col, val = _case(sp, "dups")
    x = np.random.default_rng(59).uniform(-1, 1, N)
    try:
        sp.set_knob("force_wide", 1)
        for sum_dup in (False, True):
            want = oracle_coo(M, N, row, col, val, sum_dup)
            H = build(sp, torch, M, N, row, col, val, sum_dup)
            assert_layout(H, want)
            check_spmv(O, torch, H, want, x, label=("wide", sum_dup))
            H.close()
    finally:
        sp.set_knob("force_wide", 0)


@gpu
def test_from_torch(sp, torch, monkeypatch):
    """sparse_coo (coalesced and not) and sparse_csr (int32 and int64 indices) tensors build the
    same handle as from_coo on the same triplets; bad tensors raise before any C call."""
    rng = np.random.default_rng(60)
    M, N = 600, 500
    row, col, val = random_coo(rng, M, N, 20000, rows=200, cols=150)
    idx = torch.from_numpy(np.stack([row, col])).cuda()
    t = torch.sparse_coo_tensor(idx, dev(torch, val), (M, N))
    assert not t.is_coalesced()
    tc = t.coalesce()
    for sum_dup in (False, True):
        for tt in (t, tc):
            H = sp.CsrDevice.from_torch(tt, sum_duplicates=sum_dup)
            ix = tt._indices()
            R = sp.CsrDevice.from_coo(M, N, ix[0].contiguous(), ix[1].contiguous(), tt._values().contiguous(),
                                      sum_duplicates=sum_dup)
            same_bytes(H, R)
            H.close()
            R.close()
        H = sp.CsrDevice.from_torch(t, sum_duplicates=sum_dup)
        assert_layout(H, oracle_coo(M, N, row, col, val, sum_dup))
        H.close()
    IRP, JA, AS = random_csr(rng, M, N, 30)
    r_of, _, _ = csr_to_coo(IRP, JA, AS)
    for dt in (torch.int32, torch.int64):
        tcsr = torch.sparse_csr_tensor(torch.from_numpy(IRP).to(dt), torch.from_numpy(JA).to(dt),
                                       torch.from_numpy(AS), (M, N)).cuda()
        H = sp.CsrDevice.from_torch(tcsr)
        R = sp.CsrDevice.from_coo(M, N, torch.from_numpy(r_of).to(dt).cuda(), torch.from_numpy(JA).to(dt).cuda(),
                                  dev(torch, AS))
        same_bytes(H, R)
        assert_layout(H, oracle_coo(M, N, r_of, JA, AS, False))
        H.close()
        R.close()

    def no_c_call(*a):
        raise AssertionError("spmv_b200_csr_from_coo was called")

    monkeypatch.setattr(sp._lib.b200, "spmv_b200_csr_from_coo", no_c_call)
    bad = [tc.float(), tc.cpu(), tc.to_dense(),
           torch.sparse_coo_tensor(torch.zeros(3, 4, dtype=torch.int64), torch.ones(4, dtype=torch.float64),
                                   (2, 3, 3)).cuda(),
           torch.sparse_coo_tensor(torch.zeros(2, 4, dtype=torch.int64), torch.ones(4, 3, dtype=torch.float64),
                                   (3, 3, 3)).cuda(),
           torch.sparse_csr_tensor(torch.zeros(2, 3, dtype=torch.int64), torch.zeros(2, 0, dtype=torch.int64),
                                   torch.zeros(2, 0, dtype=torch.float64), (2, 2, 4)).cuda(),
           "not a tensor"]
    for b in bad:
        with pytest.raises((TypeError, ValueError)):
            sp.CsrDevice.from_torch(b)
    r, c, v = idx[0].contiguous(), idx[1].contiguous(), dev(torch, val)
    for args in ((r.int(), c, v), (r, c, v.float()), (r.cpu(), c, v), (r, c[:-1], v), (r, c, v[::2])):
        with pytest.raises((TypeError, ValueError)):
            sp.CsrDevice.from_coo(M, N, *args)


def _raw(sp, M, N, n, row, col, idx_bytes, val, flags=0):
    """spmv_b200_csr_from_coo through ctypes on the legacy default stream: (handle, last error)."""
    def ptr(a):
        if a is None:
            return None
        return a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data
    h = sp._lib.b200.spmv_b200_csr_from_coo(M, N, n, ptr(row), ptr(col), idx_bytes, ptr(val), flags, None)
    return h, sp._lib.last_error()


@gpu
def test_errors(sp, torch):
    """Every -EINVAL case, -ENOTSUP, messages naming the first bad entry, a host buffer rejected
    before any launch, and no device memory left behind by failing or repeated builds."""
    n = 1000
    r = torch.arange(n, dtype=torch.int64, device="cuda") % 50
    c = torch.arange(n, dtype=torch.int64, device="cuda") % 40
    v = torch.ones(n, dtype=torch.float64, device="cuda")
    lim = (1 << 31) - 64
    cases = [((-1, 40, n), "bad shape"), ((50, -1, n), "bad shape"), ((50, 40, -1), "bad shape"),
             ((lim, 40, n), "bad shape"), ((50, lim, n), "bad shape")]
    for (M, N, nn), msg in cases:
        h, err = _raw(sp, M, N, nn, r, c, 8, v)
        assert not h and msg in err, (M, N, nn, err)
    h, err = _raw(sp, 50, 40, n, r, c, 2, v)
    assert not h and "index width" in err
    h, err = _raw(sp, 50, 40, n, r, c, 8, v, flags=2)
    assert not h and "unknown flag" in err
    for args in ((None, c, v), (r, None, v), (r, c, None)):
        h, err = _raw(sp, 50, 40, n, args[0], args[1], 8, args[2])
        assert not h and "null array" in err
    h, err = _raw(sp, 50, 40, lim, r, c, 8, v)
    assert not h and "not supported" in err
    # a host buffer is rejected on the host, before any launch
    host = np.zeros(n, np.int64)
    l0 = sp.counters()["launches"]
    for args in ((host, c, v), (r, host, v), (r, c, np.zeros(n))):
        h, err = _raw(sp, 50, 40, n, args[0], args[1], 8, args[2])
        assert not h and "not device or managed memory" in err, err
    assert sp.counters()["launches"] == l0
    # out-of-range entries: the message names the first one
    for k, (rr, cc) in {5: (50, 0), 17: (0, 40), 321: (-1, 3), 999: (4, -2)}.items():
        rb, cbuf = r.clone(), c.clone()
        rb[k], cbuf[k] = rr, cc
        rb[k + 1:] = -5  # later bad entries do not change the message
        for idx in (torch.int32, torch.int64):
            with pytest.raises(RuntimeError, match=f"entry {k} has row {rr} and column {cc}"):
                sp.CsrDevice.from_coo(50, 40, rb.to(idx), cbuf.to(idx), v)
    # no device memory left behind by 20 failing builds or 20 build / close cycles
    big = 10_000_000
    br = torch.randint(0, 1000, (big,), dtype=torch.int64, device="cuda")
    bc = torch.randint(0, 1000, (big,), dtype=torch.int64, device="cuda")
    bv = torch.rand(big, dtype=torch.float64, device="cuda")
    for sum_dup in (False, True):  # first use of every kernel of this shape (lazy module loading)
        sp.CsrDevice.from_coo(1000, 1000, br, bc, bv, sum_duplicates=sum_dup).close()
    br[-1] = 1000
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(20):
        with pytest.raises(RuntimeError, match=f"entry {big - 1} has row 1000"):
            sp.CsrDevice.from_coo(1000, 1000, br, bc, bv, sum_duplicates=True)
    assert abs(torch.cuda.mem_get_info()[0] - free0) <= 2 << 20
    br[-1] = 7
    torch.cuda.synchronize()
    for i in range(20):
        sp.CsrDevice.from_coo(1000, 1000, br, bc, bv, sum_duplicates=bool(i & 1)).close()
    assert abs(torch.cuda.mem_get_info()[0] - free0) <= 2 << 20


@gpu
def test_c4_full_size(sp, O, torch):
    """BASELINE configs[3] as shuffled int64 COO: R-MAT scale 24, 16 edges per vertex (268 M
    entries, duplicates), in both modes.  Layout against the oracle, CSR ids 2 / 4 against the
    oracle port."""
    R = sp.gen_rmat(24, 16)
    assert (R.M, R.NZ) == (1 << 24, 1 << 28)
    M, N = R.M, R.N
    p = np.random.default_rng(61).permutation(R.NZ)
    key = (np.repeat(np.arange(M, dtype=np.int64), np.diff(R.IRP)) << 24 | R.JA)[p]  # 24 + 24 bits
    val = R.AS[p]
    del p, R
    rd, cd, vd = (torch.from_numpy(key >> 24).cuda(), torch.from_numpy(key & 0xFFFFFF).cuda(), dev(torch, val))
    # the oracle's stable (row, col) order: any sort by key, then input order within equal keys
    o = np.argsort(key)
    ks = key[o]
    del key
    head = np.ones(len(ks), bool)
    head[1:] = ks[1:] != ks[:-1]
    gid = np.cumsum(head) - 1
    o = np.sort(gid << 28 | o) & ((1 << 28) - 1)
    del gid
    v = val[o]
    del o, val
    x = np.random.default_rng(2).uniform(0, 1, N)
    for sum_dup in (False, True):
        if sum_dup:
            start = np.flatnonzero(head)
            lens = np.diff(np.append(start, len(ks)))
            acc = v[start].copy()
            act = np.flatnonzero(lens > 1)
            for j in range(1, int(lens.max())):
                act = act[lens[act] > j]
                acc[act] += v[start[act] + j]
            kk, vv = ks[start], acc
            del start, lens, act
        else:
            kk, vv = ks, v
        irp = np.zeros(M + 1, np.int64)
        irp[1:] = np.cumsum(np.bincount(kk >> 24, minlength=M))
        want = (irp, (kk & 0xFFFFFF).astype(np.int32), vv)
        del kk, vv
        H = sp.CsrDevice.from_coo(M, N, rd, cd, vd, sum_duplicates=sum_dup)
        assert_layout(H, want)
        check_spmv(O, torch, H, want, x, kernels=(2, 4), hll=False, label=("c4", sum_dup))
        H.close()
        del want
