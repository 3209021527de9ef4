"""Tests of spmv_b200_csr_spgemm / CsrDevice.matmul(): C = A·B of two resident CSR handles built in HBM.

The result is defined exactly -- each row's columns once in increasing order, and each value the
left-to-right FP64 sum of its products taken in (A entry, B entry) stored order -- so it is compared
bit for bit with a numpy restatement of that definition.  The restatement is checked against
scipy on the CPU.  Products on C are compared with the oracle port's serial CSR."""
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


def products(M, IRP_A, JA_A, AS_A, IRP_B, JA_B, AS_B):
    """(row, col, value) of every product a_p·b_q of A·B in the defined order: p over A's row in
    stored order, then q over B's row ja_A[p] in stored order."""
    IRP_A, IRP_B = np.asarray(IRP_A, np.int64), np.asarray(IRP_B, np.int64)
    JA_A, JA_B = np.asarray(JA_A, np.int64), np.asarray(JA_B, np.int32)
    AS_A, AS_B = np.asarray(AS_A, np.float64), np.asarray(AS_B, np.float64)
    reps = np.diff(IRP_B)[JA_A]
    n = int(reps.sum())
    p = np.repeat(np.arange(len(JA_A)), reps)
    q = np.repeat(IRP_B[JA_A] - (np.cumsum(reps) - reps), reps) + np.arange(n)
    row = np.repeat(np.arange(M, dtype=np.int64), np.diff(IRP_A))[p]
    with np.errstate(invalid="ignore", over="ignore"):
        val = AS_A[p] * AS_B[q]
    return row, JA_B[q], val


def oracle_spgemm(M, N, IRP_A, JA_A, AS_A, IRP_B, JA_B, AS_B):
    """(IRP int64, JA int32, AS) of C = A·B (N: columns of B): the products stably sorted by
    (row, col), each run summed strictly left to right starting from its first product."""
    row, col, val = products(M, IRP_A, JA_A, AS_A, IRP_B, JA_B, AS_B)
    key = row * max(N, 1) + col
    o = np.argsort(key, kind="stable")
    key, val = key[o], val[o]
    n = len(key)
    heads = np.flatnonzero(np.r_[True, key[1:] != key[:-1]]) if n else np.zeros(0, np.int64)
    lens = np.diff(np.r_[heads, n])
    by_len = np.argsort(-lens, kind="stable")  # runs still going at rank r: a prefix of by_len
    h, neg_len = heads[by_len], -lens[by_len]
    acc = val[h].copy()
    with np.errstate(invalid="ignore", over="ignore"):
        for r in range(1, int(-neg_len[0]) if n else 0):  # rank within the run, across all runs
            k = int(np.searchsorted(neg_len, -r, side="left"))  # runs longer than r
            acc[:k] = acc[:k] + val[h[:k] + r]
    out = np.empty_like(acc)
    out[by_len] = acc
    ukey = key[heads]
    irp = np.zeros(M + 1, np.int64)
    irp[1:] = np.cumsum(np.bincount(ukey // max(N, 1), minlength=M))
    return irp, (ukey % max(N, 1)).astype(np.int32), out


def transposed(M, N, IRP, JA, AS):
    """(IRP int32, JA, AS) of Aᵀ (stable by column)."""
    JA = np.asarray(JA, np.int32)
    row_of = np.repeat(np.arange(M, dtype=np.int32), np.diff(np.asarray(IRP, np.int64)))
    o = np.argsort(JA, kind="stable")
    irp = np.zeros(N + 1, np.int32)
    irp[1:] = np.cumsum(np.bincount(JA, minlength=N))
    return irp, row_of[o], np.asarray(AS, np.float64)[o]


def same_values(a, b):
    """Bit-equal, except that any NaN matches any NaN (the GPU's NaN bits differ from numpy's)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def assert_layout(C, want):
    irp, ja, as_ = C.download()
    assert np.array_equal(irp, want[0])
    assert np.array_equal(ja, want[1])
    assert same_values(as_, want[2])


def check_routes(O, torch, C, c, x, label=""):
    """Every CSR kernel id and every HLL id on C against the oracle port on the restated arrays."""
    irp32 = c[0].astype(np.int32)
    y_ref = O.csr_spmv(C.M, irp32, c[1], c[2], x)
    bound = O.csr_abs_bound(C.M, irp32, c[1], c[2], x)
    xd = dev(torch, x)
    y = torch.zeros(C.M, dtype=torch.float64, device="cuda")
    for kernel in range(5):
        y.fill_(float("nan"))
        C.spmv(xd, y, kernel=kernel)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (label, "csr", kernel, worst)
    H = C.to_hll()
    for kernel in range(4):
        y.fill_(float("nan"))
        H.spmv(xd, y, kernel=kernel)
        ok, worst = O.check_tolerance(y.cpu().numpy(), y_ref, bound, TOL)
        assert ok, (label, "hll", kernel, worst)
    H.close()


def _host(A):
    return A.M, A.N, A.IRP.copy(), A.JA.copy(), A.AS.copy()


def _pair(sp, name):
    """((M, K, IRP, JA, AS) of A, (K, N, IRP, JA, AS) of B) of a named product."""
    rng = np.random.default_rng(51)
    if name.startswith("square:"):
        g = golden(name[7:])
        a = (int(g["M"]), int(g["N"]), g["IRP"], g["JA"], g["AS"])
        return a, a
    if name.startswith("aat:") or name.startswith("ata:"):
        g = golden(name[4:])
        a = (int(g["M"]), int(g["N"]), g["IRP"], g["JA"], g["AS"])
        t = (a[1], a[0]) + transposed(*a)
        return (a, t) if name.startswith("aat:") else (t, a)
    if name == "random":        # M, K, N all different; unsorted rows, duplicates, empty rows
        return (300, 410) + random_csr(rng, 300, 410, 30), (410, 520) + random_csr(rng, 410, 520, 25)
    if name == "empty_a":
        return (40, 30) + random_csr(rng, 40, 30, 0), (30, 20) + random_csr(rng, 30, 20, 6)
    if name == "empty_b":
        return (40, 30) + random_csr(rng, 40, 30, 6), (30, 20) + random_csr(rng, 30, 20, 0)
    if name == "nz0":           # A's entries reference only B's empty rows
        IRP_B, JA_B, AS_B = random_csr(rng, 30, 20, 6, empty_frac=0.0)
        lens = np.diff(IRP_B)
        lens[:10] = 0
        IRP_B = np.r_[0, np.cumsum(lens)].astype(np.int32)
        JA_B, AS_B = JA_B[:IRP_B[-1]], AS_B[:IRP_B[-1]]
        IRP_A, JA_A, AS_A = random_csr(rng, 40, 10, 5)
        return (40, 30, IRP_A, JA_A, AS_A), (30, 20, IRP_B, JA_B, AS_B)
    if name == "outer":         # one column times one row: every row of C dense
        col = (500, 1) + random_csr(rng, 500, 1, 3)
        row = (1, 400) + random_csr(rng, 1, 400, 300, empty_frac=0.0)
        return col, row
    if name == "inner":         # one row times one column: a 1 x 1 result of 300 products
        row = (1, 600) + random_csr(rng, 1, 600, 300, empty_frac=0.0)
        col = (600, 1) + random_csr(rng, 600, 1, 3)
        return row, col
    if name == "rmat":
        R = _host(sp.gen_rmat(12, 16))
        return R, R
    if name == "ragged_uniform":
        Rg = _host(sp.gen_ragged(3000, 400))
        return Rg, _host(sp.gen_uniform_random(Rg[1], 16))
    raise KeyError(name)


def _square(name):
    g = golden(name)
    return int(g["M"]) == int(g["N"])


PAIR_CASES = ([f"square:{n}" for n in GOLDEN_CASES if _square(n)] +
              [f"{k}:{n}" for n in GOLDEN_CASES if not _square(n) for k in ("aat", "ata")] +
              ["random", "empty_a", "empty_b", "nz0", "outer", "inner", "rmat", "ragged_uniform"])


def _upload(sp, m):
    M, N, IRP, JA, AS = m
    return sp.CsrDevice.from_arrays(M, N, np.asarray(IRP, np.int32), JA, AS)


@pytest.mark.parametrize("dups", [False, True])
def test_restatement_matches_scipy(dups):
    """The numpy restatement agrees with scipy's A @ B: the same pattern once scipy's dropped zeros
    are accounted for, values within 1e-12 * sum |a||b| of each entry."""
    rng = np.random.default_rng(52)
    for M, K, N, la, lb in ((50, 60, 70, 12, 9), (300, 200, 100, 40, 30), (1, 80, 5, 80, 5)):
        IRP_A, JA_A, AS_A = random_csr(rng, M, K, la, sort=not dups)
        IRP_B, JA_B, AS_B = random_csr(rng, K, N, lb, sort=not dups)
        irp, ja, as_ = oracle_spgemm(M, N, IRP_A, JA_A, AS_A, IRP_B, JA_B, AS_B)
        assert np.all(np.diff(irp) >= 0) and irp[-1] == len(ja)
        row = np.repeat(np.arange(M), np.diff(irp))
        assert np.all((np.diff(row) > 0) | (np.diff(ja) > 0))  # each row strictly increasing
        A = scipy.sparse.csr_matrix((AS_A, JA_A, IRP_A), shape=(M, K))
        B = scipy.sparse.csr_matrix((AS_B, JA_B, IRP_B), shape=(K, N))
        S = (A @ B).tocsr()
        S.sort_indices()
        keep = as_ != 0
        assert np.array_equal(np.repeat(np.arange(M), np.diff(S.indptr)), row[keep])
        assert np.array_equal(S.indices, ja[keep])
        r, c, v = products(M, IRP_A, JA_A, np.abs(AS_A), IRP_B, JA_B, np.abs(AS_B))
        mag = scipy.sparse.csr_matrix((v, (r, c)), shape=(M, N))
        mag.sum_duplicates()
        mag.sort_indices()
        assert np.all(np.abs(S.data - as_[keep]) <= 1e-12 * mag.data[keep])


def test_matmul_rejects_before_any_c_call(sp, monkeypatch):
    """A B that is not a CsrDevice raises TypeError, a shape mismatch ValueError, both before the
    library is called."""
    def no_c_call(*a):
        raise AssertionError("spmv_b200_csr_spgemm was called")

    monkeypatch.setattr(sp._lib.b200, "spmv_b200_csr_spgemm", no_c_call)

    def fake(M, N):
        h = sp.CsrDevice.__new__(sp.CsrDevice)
        h._h, h.M, h.N, h.NZ = None, M, N, 0
        return h

    A = fake(5, 7)
    for bad in ("B", np.eye(7), None, scipy.sparse.eye(7, format="csr")):
        with pytest.raises(TypeError):
            A.matmul(bad)
    for B in (fake(6, 3), fake(8, 7), fake(5, 5)):
        with pytest.raises(ValueError, match="7 columns"):
            A.matmul(B)


@gpu
@pytest.mark.parametrize("case", PAIR_CASES)
def test_layout_and_routes(sp, O, torch, case):
    """download() of C equals the restatement bit for bit; every CSR and HLL id on C matches the
    serial CSR product."""
    a, b = _pair(sp, case)
    want = oracle_spgemm(a[0], b[1], a[2], a[3], a[4], b[2], b[3], b[4])
    A, B = _upload(sp, a), _upload(sp, b)
    C = A.matmul(B)
    assert (C.M, C.N, C.NZ) == (a[0], b[1], len(want[1]))
    assert_layout(C, want)
    check_routes(O, torch, C, want, np.random.default_rng(3).uniform(-1, 1, C.N), label=case)
    for h in (C, A, B):
        h.close()


def _every_path():
    """A whose rows have 0, 1 and 2^k - 1, 2^k, 2^k + 1 products (k = 1..17), and B with 2^18 + 7
    columns whose rows (one of each length 2^m, m = 0..17, and one empty row) repeat no column, so
    the table bound min(P_i, B.N) is P_i: both sides of every table size and of the shared /
    global switch."""
    rng = np.random.default_rng(53)
    NB = (1 << 18) + 7
    lens = [1 << m for m in range(18)] + [0]
    IRP_B = np.r_[0, np.cumsum(lens)].astype(np.int32)
    JA_B = np.concatenate([rng.choice(NB, n, replace=False) for n in lens]).astype(np.int32)
    AS_B = rng.uniform(-1, 1, len(JA_B))
    targets = sorted({0, 1} | {(1 << k) + d for k in range(1, 18) for d in (-1, 0, 1)})
    rows = []
    for t in targets:
        ent = [m for m in range(18) if t >> m & 1] or [18]  # t = 0: the empty row of B
        rows.append(rng.permutation(ent))
    rows.insert(5, np.zeros(0, np.int64))  # an empty row of A
    IRP_A = np.r_[0, np.cumsum([len(r) for r in rows])].astype(np.int32)
    JA_A = np.concatenate(rows).astype(np.int32)
    AS_A = rng.uniform(-1, 1, len(JA_A))
    return (len(rows), 19, IRP_A, JA_A, AS_A), (19, NB, IRP_B, JA_B, AS_B), targets


@gpu
def test_every_table_size(sp, O, torch):
    a, b, targets = _every_path()
    cs = np.r_[0, np.cumsum(np.diff(np.asarray(b[2], np.int64))[a[3]])]
    per_row = cs[a[2][1:]] - cs[a[2][:-1]]
    assert sorted(set(per_row.tolist())) == targets
    want = oracle_spgemm(a[0], b[1], a[2], a[3], a[4], b[2], b[3], b[4])
    A, B = _upload(sp, a), _upload(sp, b)
    C = A.matmul(B)
    assert_layout(C, want)
    check_routes(O, torch, C, want, np.random.default_rng(4).uniform(-1, 1, C.N), label="every path")
    for h in (C, A, B):
        h.close()


@gpu
def test_summation_order_and_special_values(sp, torch):
    """A column repeated 40 times in one row of B (two warp steps) with values whose sum depends on
    the order, referenced several times by A; explicit zeros, cancellation to exactly 0, a lone
    -0.0, NaN and Inf."""
    rng = np.random.default_rng(54)
    cyc = [1.0, 1e16, -1e16, 3.0, -1e16, 1e16, 0.5, 2.0**-30]
    r0_col = np.full(40, 5)
    r0_val = np.array([cyc[i % len(cyc)] for i in range(40)])
    extra = rng.integers(6, 12, 13)
    pos = np.sort(rng.choice(53, 13, replace=False))
    col0 = np.insert(r0_col, pos - np.arange(13), extra)
    val0 = np.insert(r0_val, pos - np.arange(13), rng.uniform(-1, 1, 13) * 1e15)
    rows_b = [(col0, val0),
              ([2, 3], [0.0, 1.0]),                         # explicit zero; +1 for a cancellation
              ([3], [-1.0]),                                # the -1 of the cancellation
              ([4], [-0.0]),                                # a lone -0.0
              ([6, 7, 8], [np.nan, np.inf, 1.0])]           # NaN and Inf
    IRP_B = np.r_[0, np.cumsum([len(c) for c, _ in rows_b])].astype(np.int32)
    JA_B = np.concatenate([np.asarray(c) for c, _ in rows_b]).astype(np.int32)
    AS_B = np.concatenate([np.asarray(v, np.float64) for _, v in rows_b])
    rows_a = [([0, 0, 0], [1.0, -1.0, 3.0]), ([0, 1, 0], [1.0, 2.0, 1e-3]), ([1, 2], [1.0, 1.0]),
              ([3], [1.0]), ([3], [-1.0]), ([4], [2.0]), ([1], [np.inf]), ([3, 0, 4, 0], [0.0, 1.0, 1.0, -2.0]),
              ([], [])]
    IRP_A = np.r_[0, np.cumsum([len(c) for c, _ in rows_a])].astype(np.int32)
    JA_A = np.concatenate([np.asarray(c, np.int32) for c, _ in rows_a]).astype(np.int32)
    AS_A = np.concatenate([np.asarray(v, np.float64) for _, v in rows_a])
    M, N = len(rows_a), 12
    want = oracle_spgemm(M, N, IRP_A, JA_A, AS_A, IRP_B, JA_B, AS_B)
    A = sp.CsrDevice.from_arrays(M, 5, IRP_A, JA_A, AS_A)
    B = sp.CsrDevice.from_arrays(5, N, IRP_B, JA_B, AS_B)
    C = A.matmul(B)
    assert_layout(C, want)
    irp, ja, as_ = C.download()

    def at(i, j):
        k = np.flatnonzero(ja[irp[i]:irp[i + 1]] == j)
        assert len(k) == 1, (i, j)
        return as_[irp[i] + k[0]]

    assert at(2, 2) == 0.0 and at(2, 3) == 0.0 and not np.signbit(at(2, 3))   # kept zeros
    assert at(3, 4) == 0.0 and np.signbit(at(3, 4))                          # lone -0.0 stays
    assert at(4, 4) == 0.0 and not np.signbit(at(4, 4))                      # (-1)·(-0.0)
    assert np.isnan(at(5, 6)) and at(5, 7) == np.inf and at(5, 8) == 2.0
    assert np.isnan(at(6, 2)) and at(6, 3) == np.inf                         # inf·0, inf·1
    assert irp[M] - irp[M - 1] == 0
    for h in (C, A, B):
        h.close()


@gpu
def test_c2_squared_full_size(sp, torch):
    """C2 (128^3 27-point stencil) squared: the 125-point stencil, nnz(C) = 634^3 exactly, and
    C·x agrees with A·(A·x) within 1e-12 (|A|·(|A|·|x|))_i per row."""
    n = 128
    A = sp.CsrDevice.stencil27(n, n, n)
    C = A.matmul(A)
    assert (C.M, C.N, C.NZ) == (n**3, n**3, 634**3)
    irp, ja, as_ = A.download()
    Aabs = sp.CsrDevice.from_arrays(A.M, A.N, irp.astype(np.int32), ja, np.abs(as_))
    del irp, ja, as_
    x = torch.rand(A.N, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(5)) * 2 - 1
    t, y, yc, b1, b2 = (torch.zeros(A.M, dtype=torch.float64, device="cuda") for _ in range(5))
    A.spmv(x, t, kernel=2)
    A.spmv(t, y, kernel=2)
    C.spmv(x, yc, kernel=2)
    Aabs.spmv(x.abs(), b1, kernel=2)
    Aabs.spmv(b1, b2, kernel=2)
    assert bool(((yc - y).abs() <= TOL * b2).all())
    for h in (C, Aabs, A):
        h.close()


@gpu
def test_galerkin_full_size(sp, torch):
    """Pᵀ·(A·P) on C2 with P the 2x2x2 piecewise-constant aggregation built by from_coo equals
    scipy's product bit for bit (small integers: every summation order is exact)."""
    n, m = 128, 64
    A = sp.CsrDevice.stencil27(n, n, n)
    i = np.arange(n**3)
    x, y, z = i % n, i // n % n, i // (n * n)
    agg = x // 2 + m * (y // 2) + m * m * (z // 2)
    P = sp.CsrDevice.from_coo(n**3, m**3, torch.from_numpy(i).cuda(), torch.from_numpy(agg).cuda(),
                              torch.ones(n**3, dtype=torch.float64, device="cuda"))
    AP = A.matmul(P)
    Pt = P.transpose()
    Ac = Pt.matmul(AP)
    assert (Ac.M, Ac.N) == (m**3, m**3)
    irp, ja, as_ = A.download()
    As = scipy.sparse.csr_matrix((as_, ja, irp), shape=(n**3, n**3))
    Ps = scipy.sparse.csr_matrix((np.ones(n**3), agg, np.arange(n**3 + 1)), shape=(n**3, m**3))
    ref = (Ps.T.tocsr() @ (As @ Ps)).tocsr()
    ref.sort_indices()
    got = Ac.download()
    assert np.all(got[2] != 0)  # no zero sums, so scipy drops nothing
    assert np.array_equal(got[0], ref.indptr.astype(np.int64))
    assert np.array_equal(got[1], ref.indices.astype(np.int32))
    assert np.array_equal(got[2].view(np.uint64), ref.data.view(np.uint64))
    for h in (Ac, Pt, AP, P, A):
        h.close()


@gpu
def test_wide_offsets(sp, O, torch):
    """Every combination of 32- and 64-bit row offsets for A and B, with narrow and wide results."""
    R = _host(sp.gen_ragged(2000, 150))
    rng = np.random.default_rng(55)
    b = (R[1], 900) + random_csr(rng, R[1], 900, 20)
    want = oracle_spgemm(R[0], 900, R[2], R[3], R[4], b[2], b[3], b[4])
    x = rng.uniform(-1, 1, 900)
    try:
        for wide_a in (0, 1):
            for wide_b in (0, 1):
                hs = []
                for wide, (M, N, IRP, JA, AS) in ((wide_a, R), (wide_b, b)):
                    sp.set_knob("force_wide", wide)
                    hs.append(sp.CsrDevice.from_arrays(M, N, np.asarray(IRP, np.int64 if wide else np.int32),
                                                       JA, AS))
                for wide_out in (0, 1):
                    sp.set_knob("force_wide", wide_out)
                    C = hs[0].matmul(hs[1])
                    sp.set_knob("force_wide", 0)
                    assert_layout(C, want)
                    check_routes(O, torch, C, want, x, label=("wide", wide_a, wide_b, wide_out))
                    C.close()
                for h in hs:
                    h.close()
    finally:
        sp.set_knob("force_wide", 0)


@gpu
def test_shard_multiplies_its_local_block(sp, O, torch):
    """A shard created with col_offset and cuts multiplies its local block: its n_local columns
    against B's rows; C has col_offset 0 and no cuts."""
    nx, ny, nz = 10, 9, 12
    plane = nx * ny
    z0, z1 = 4, 9
    r0, r1 = z0 * plane, z1 * plane
    c0, c1 = (z0 - 1) * plane, (z1 + 1) * plane
    part = sp.gen_stencil27_rows(nx, ny, nz, r0, r1)
    rng = np.random.default_rng(56)
    b = (c1 - c0, 333) + random_csr(rng, c1 - c0, 333, 9)
    want = oracle_spgemm(part.M, 333, part.IRP, part.JA - c0, part.AS, b[2], b[3], b[4])
    B = _upload(sp, b)
    for h in (sp.CsrDevice.from_arrays(part.M, c1 - c0, part.IRP, part.JA, part.AS, col_offset=c0,
                                       cuts=[plane, part.M - plane]),
              sp.CsrDevice.stencil27(nx, ny, nz, z0, z1, col_offset=c0, n_local=c1 - c0,
                                     cuts=[plane, part.M - plane])):
        C = h.matmul(B)
        assert (C.M, C.N) == (part.M, 333)
        assert_layout(C, want)
        check_routes(O, torch, C, want, rng.uniform(-1, 1, 333), label="shard")
        y = torch.zeros(C.M, dtype=torch.float64, device="cuda")
        with pytest.raises(RuntimeError, match="cut points"):
            C.spmv(dev(torch, np.zeros(333)), y, rows=(plane, C.M - plane))
        C.close()
        h.close()
    B.close()


@gpu
def test_more_than_2_31_products(sp, torch):
    """2^20 x 1 ones times a 1 x 1 matrix of 2100 duplicate entries 1.0: 2.2e9 products counted in
    64 bits, one entry of value 2100.0 per row."""
    M = 1 << 20
    A = sp.CsrDevice.from_arrays(M, 1, np.arange(M + 1, dtype=np.int32), np.zeros(M, np.int32), np.ones(M))
    B = sp.CsrDevice.from_arrays(1, 1, np.array([0, 2100], np.int32), np.zeros(2100, np.int32), np.ones(2100))
    C = A.matmul(B)
    assert (C.M, C.N, C.NZ) == (M, 1, M)
    irp, ja, as_ = C.download()
    assert np.array_equal(irp, np.arange(M + 1)) and not ja.any() and np.all(as_ == 2100.0)
    for h in (C, A, B):
        h.close()


def _raw(sp, A, B):
    """spmv_b200_csr_spgemm through ctypes: (handle, last error)."""
    h = sp._lib.b200.spmv_b200_csr_spgemm(A, B)
    return h, sp._lib.last_error()


@gpu
def test_errors(sp, torch):
    """A null handle and a shape mismatch give -EINVAL; a C of 2^31 - 64 or more entries gives
    -ENOTSUP, found before C is allocated."""
    rng = np.random.default_rng(57)
    A = _upload(sp, (30, 20) + random_csr(rng, 30, 20, 5))
    B = _upload(sp, (21, 10) + random_csr(rng, 21, 10, 5))
    h, err = _raw(sp, A._h, B._h)
    assert not h and "20" in err and "21" in err, err
    for a, b in ((None, B._h), (A._h, None), (None, None)):
        h, err = _raw(sp, a, b)
        assert not h and "null" in err, err
    A.close()
    B.close()
    M = 1 << 22
    A = sp.CsrDevice.from_arrays(M, 1, np.arange(M + 1, dtype=np.int32), np.zeros(M, np.int32), np.ones(M))
    B = sp.CsrDevice.from_arrays(1, 600, np.array([0, 600], np.int32), np.arange(600, dtype=np.int32),
                                 np.ones(600))
    small = sp.CsrDevice.from_arrays(2, 1, np.array([0, 1, 1], np.int32), np.zeros(1, np.int32), np.ones(1))
    small.matmul(B).close()  # first use of the kernels of this shape (lazy module loading)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    h, err = _raw(sp, A._h, B._h)
    assert not h and "not supported" in err, err
    with pytest.raises(RuntimeError, match="not supported"):
        A.matmul(B)
    assert abs(torch.cuda.mem_get_info()[0] - free0) <= 2 << 20
    for hh in (small, A, B):
        hh.close()


@gpu
def test_inputs_unchanged_and_deterministic(sp, O, torch):
    """A and B download unchanged after the call; two products are bit-identical; C outlives A and B."""
    rng = np.random.default_rng(58)
    a = (3000, 2500) + random_csr(rng, 3000, 2500, 60)
    b = (2500, 4000) + random_csr(rng, 2500, 4000, 50)
    want = oracle_spgemm(a[0], b[1], a[2], a[3], a[4], b[2], b[3], b[4])
    A, B = _upload(sp, a), _upload(sp, b)
    before = A.download() + B.download()
    C1, C2 = A.matmul(B), A.matmul(B)
    for u, w in zip(before, A.download() + B.download()):
        assert np.array_equal(u.view(np.uint8), w.view(np.uint8))
    for u, w in zip(C1.download(), C2.download()):
        assert np.array_equal(u.view(np.uint8), w.view(np.uint8))
    A.close()
    B.close()
    C2.close()
    assert_layout(C1, want)
    check_routes(O, torch, C1, want, rng.uniform(-1, 1, C1.N), label="after destroy")
    C1.close()
