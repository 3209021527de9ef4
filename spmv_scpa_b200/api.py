"""Python mirror of the reference's operator interface for the SpMV path.

Same names and argument meaning as the reference's C API (include/csr.h:29-49,
include/hll.h:54-70, include/vector.h:11-18 of the reference), so the parity
tests read like the reference's own call sequence (src/main.c:78-102,
:258-359):

    A  = io_load_csr("m.mtx")
    Hc = csr_to_hll(A, True)
    x  = vec_fill_random(A.N)
    ms, gflops, y = bench_csr_cuda_halfwarp_row(A, x, warps_per_block=4)

Everything here forwards to the in-tree C libraries (see _lib.py); errors keep
the reference's convention (negative errno) and surface as OSError.  The
device-resident API (CsrDevice / HllDevice) wraps include/spmv_b200.h and takes
torch CUDA tensors for x and y -- torch only supplies device memory and
streams.
"""
import ctypes as C
import os

import numpy as np

from . import _lib as L
from . import structs as S

CSR_KERNEL_NAMES = ("thread_row", "warp_row", "adaptive", "block_row", "stream_tma")
HOST_PIN = {}  # addresses page-locked through host_register()
HLL_KERNEL_NAMES = ("thread_row_rm", "thread_row", "warp_hack_vec", "stream_tma")


def _as_np(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,))


def _check_ptr(addr, what):
    if addr is None or addr == 0:
        raise MemoryError(f"{what} returned NULL")
    if S.is_err_ptr(addr):
        err = -S.ptr_err(addr)
        raise OSError(err, f"{what}: {os.strerror(err)}")
    return addr


# ------------------------------------------------------------------ host CSR --
class CsrMatrix:
    """A `sparse_csr *` (include/csr.h).  Arrays are numpy views, no copies."""

    def __init__(self, addr, owner="host", keep=None):
        self._addr = addr
        self._owner = owner  # "host": csr_free() on release; "numpy": arrays kept alive here
        self._keep = keep
        self.struct = S.sparse_csr.from_address(addr) if owner == "host" else keep[0]

    @property
    def ptr(self):
        return C.cast(C.c_void_p(self._addr), C.POINTER(S.sparse_csr))

    name = property(lambda self: self.struct.name.decode())
    M = property(lambda self: self.struct.M)
    N = property(lambda self: self.struct.N)
    NZ = property(lambda self: self.struct.NZ)
    IRP = property(lambda self: _as_np(self.struct.IRP, self.M + 1, np.int32))
    JA = property(lambda self: _as_np(self.struct.JA, self.NZ, np.int32))
    AS = property(lambda self: _as_np(self.struct.AS, self.NZ, np.float64))

    def free(self):
        if self._addr and self._owner == "host":
            L.host.csr_free(self._addr)
        self._addr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def io_load_csr(path):
    """Matrix Market -> CSR (reference src/csr.c:31-171). OSError(errno) on failure."""
    addr = L.host.io_load_csr(os.fsencode(path))
    return CsrMatrix(_check_ptr(addr, f"io_load_csr({path})"))


def csr_from_arrays(name, M, N, IRP, JA, AS):
    """init_csr() over caller arrays (reference include/csr.h:15-24); arrays are kept alive."""
    IRP = np.ascontiguousarray(IRP, dtype=np.int32)
    JA = np.ascontiguousarray(JA, dtype=np.int32)
    AS = np.ascontiguousarray(AS, dtype=np.float64)
    assert IRP.shape == (M + 1,) and JA.shape == AS.shape == (int(IRP[-1]),)
    st = S.sparse_csr()
    st.name = name.encode()[:S.MAX_NAME - 1]
    st.M, st.N, st.NZ = M, N, int(IRP[-1])
    st.IRP = IRP.ctypes.data_as(C.POINTER(C.c_int))
    st.JA = JA.ctypes.data_as(C.POINTER(C.c_int))
    st.AS = AS.ctypes.data_as(C.POINTER(C.c_double))
    return CsrMatrix(C.addressof(st), owner="numpy", keep=(st, IRP, JA, AS))


def _gen(fn, *args):
    addr = fn(*args)
    if not addr:
        raise MemoryError(f"{fn.__name__}{args} failed (too large for int32 indices or out of memory)")
    return CsrMatrix(addr)


def gen_poisson2d(nx, ny):
    return _gen(L.host.gen_poisson2d, nx, ny)


def gen_stencil27(nx, ny, nz):
    return _gen(L.host.gen_stencil27, nx, ny, nz)


def gen_stencil27_rows(nx, ny, nz, row0, row1):
    return _gen(L.host.gen_stencil27_rows, nx, ny, nz, row0, row1)


def gen_uniform_random(n, k, seed=42):
    return _gen(L.host.gen_uniform_random, n, k, seed)


def gen_rmat(scale, edge_factor=16, a=0.57, b=0.19, c=0.19, seed=42):
    return _gen(L.host.gen_rmat, scale, edge_factor, a, b, c, seed)


def gen_ragged(n, max_len, seed=7):
    return _gen(L.host.gen_ragged, n, max_len, seed)


def gen_write_mtx(A, path):
    rc = L.host.gen_write_mtx(A.ptr, os.fsencode(path))
    if rc:
        raise OSError(-rc, f"gen_write_mtx({path})")


# ------------------------------------------------------------------ host HLL --
class HllMatrix:
    """A `sparse_hll *` (include/hll.h)."""

    def __init__(self, addr, is_col_major):
        self._addr = addr
        self.is_col_major = bool(is_col_major)
        self.struct = S.sparse_hll.from_address(addr)

    @property
    def ptr(self):
        return C.cast(C.c_void_p(self._addr), C.POINTER(S.sparse_hll))

    name = property(lambda self: self.struct.name.decode())
    M = property(lambda self: self.struct.M)
    N = property(lambda self: self.struct.N)
    NZ = property(lambda self: self.struct.NZ)
    hack_size = property(lambda self: self.struct.hack_size)
    num_blocks = property(lambda self: self.struct.num_blocks)

    def block(self, b):
        """(M, N, NZ, max_NZ, JA view, AS view) of hack b."""
        blk = self.struct.blocks[b]
        n = blk.M * blk.max_NZ
        return blk.M, blk.N, blk.NZ, blk.max_NZ, _as_np(blk.JA, n, np.int32), _as_np(
            blk.AS, n, np.float64)

    def flat(self):
        """rows[nb], width[nb], nz[nb], off[nb+1], JA[slots], AS[slots] (hack after hack)."""
        nb = self.num_blocks
        rows = np.zeros(nb, np.int32)
        width = np.zeros(nb, np.int32)
        nz = np.zeros(nb, np.int32)
        off = np.zeros(nb + 1, np.int64)
        ja, as_ = [], []
        for b in range(nb):
            m, _, z, w, j, a = self.block(b)
            rows[b], width[b], nz[b] = m, w, z
            off[b + 1] = off[b] + m * w
            ja.append(j)
            as_.append(a)
        JA = np.concatenate(ja) if ja else np.zeros(0, np.int32)
        AS = np.concatenate(as_) if as_ else np.zeros(0, np.float64)
        return rows, width, nz, off, JA, AS

    def free(self):
        if self._addr:
            L.host.hll_free(self._addr)
        self._addr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def csr_to_hll(A, is_col_major):
    """CSR -> HLL, hack = 32 (reference src/hll.c:19-95)."""
    addr = L.host.csr_to_hll(A.ptr, bool(is_col_major))
    return HllMatrix(_check_ptr(addr, "csr_to_hll"), is_col_major)


# -------------------------------------------------------------------- vectors --
def vec_fill_random(n):
    """x[i] = rand()/RAND_MAX from the C library, like reference src/vector.c:36-41.
    (The C generator keeps its state across calls; only the first call of a
    process reproduces the reference's x.)"""
    v = L.host.vec_create(n)
    if not v.data:
        raise MemoryError("vec_create")
    L.host.vec_fill_random(C.byref(v))
    out = _as_np(v.data, n, np.float64).copy()
    L.host.vec_put(C.byref(v))
    return out


def aligned_array(n, dtype=np.float64):
    """64-byte aligned numpy array (the reference's OpenMP path asserts alignment)."""
    item = np.dtype(dtype).itemsize
    raw = np.zeros(n * item + 64, dtype=np.uint8)
    shift = (-raw.ctypes.data) % 64
    return raw[shift:shift + n * item].view(dtype)


def validation_vec_result(expected, res):
    """0 iff ||expected-res||_2 <= 0.1 (reference src/utils.c:39-60)."""
    e = np.ascontiguousarray(expected, np.float64)
    r = np.ascontiguousarray(res, np.float64)
    ve = S.vec(len(e), e.ctypes.data_as(C.POINTER(C.c_double)))
    vr = S.vec(len(r), r.ctypes.data_as(C.POINTER(C.c_double)))
    return L.host.validation_vec_result(ve, vr)


# ------------------------------------------------- reference-style GPU benches --
def _take_y(bench):
    n = bench.data.len
    y = _as_np(bench.data.data, n, np.float64).copy()
    L.host.vec_put(C.byref(bench.data))
    return y


def _run_cuda_bench(fname, mat, x, warps_per_block):
    x = np.ascontiguousarray(x, np.float64)
    assert x.shape == (mat.N,), f"x must have N={mat.N} entries"
    out = S.bench_cuda()
    out.warps_per_block = warps_per_block
    rc = getattr(L.host, fname)(mat.ptr, x.ctypes.data_as(C.POINTER(C.c_double)), C.byref(out))
    if rc:
        raise OSError(-rc, f"{fname} failed")
    y = _take_y(out.bench)
    if out.bench.duration_ms <= 0.0:
        raise RuntimeError(f"{fname}: GPU path failed: {L.last_error()}")
    return out.bench.duration_ms, out.bench.gflops, y


def _make_bench(fname):
    def f(mat, x, warps_per_block=4):
        return _run_cuda_bench(fname, mat, x, warps_per_block)

    f.__name__ = fname
    f.__doc__ = f"{fname}(A|H, x, warps_per_block) -> (duration_ms, gflops, y); see include/csr.h / hll.h"
    return f


for _n in L.CSR_BENCH_FUNCS + L.HLL_BENCH_FUNCS:
    globals()[_n] = _make_bench(_n)


def bench_csr_serial(A, x):
    x = np.ascontiguousarray(x, np.float64)
    out = S.bench()
    rc = L.host.bench_csr_serial(A.ptr, x.ctypes.data_as(C.POINTER(C.c_double)), C.byref(out))
    if rc:
        raise OSError(-rc, "bench_csr_serial")
    return out.duration_ms, out.gflops, _take_y(out)


def set_timing(warmup, reps):
    L.b200.spmv_b200_set_timing(warmup, reps)


def release_all():
    L.b200.spmv_b200_release_all()


CACHE_POLICIES = {"off": 0, "hash": 1, "trust": 2}


def set_cache_policy(policy):
    """Matrix cache of the reference-style entry points: "off" (upload per call, like the
    reference), "hash" (default: full content hash per call), "trust" (pointers + shape; call
    invalidate() after editing a matrix in place)."""
    rc = L.b200.spmv_b200_set_cache_policy(CACHE_POLICIES.get(policy, policy))
    if rc:
        raise ValueError(L.last_error())


def invalidate(mat=None):
    """Forget the device copy of one host matrix (CsrMatrix / HllMatrix), or of all."""
    L.b200.spmv_b200_invalidate(None if mat is None else C.c_void_p(mat._addr))


def pinned_empty(n, dtype=np.float64):
    """numpy array in page-locked memory from spmv_b200_host_alloc (freed with pinned_free)."""
    nbytes = n * np.dtype(dtype).itemsize
    p = L.b200.spmv_b200_host_alloc(nbytes)
    if not p:
        raise MemoryError(L.last_error())
    arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_ubyte)), shape=(max(nbytes, 1),))[:nbytes].view(dtype)
    HOST_PIN[arr.ctypes.data] = p
    return arr


def pinned_free(arr):
    p = HOST_PIN.pop(arr.ctypes.data, None)
    if p:
        L.b200.spmv_b200_host_free(p)


def counters():
    a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
    L.b200.spmv_b200_counters(C.byref(a), C.byref(b), C.byref(c))
    return {"launches": a.value, "h2d_bytes": b.value, "d2h_bytes": c.value}


def set_knob(key, value):
    rc = L.b200.spmv_b200_set_knob(key.encode(), int(value))
    if rc:
        raise ValueError(L.last_error())


def device_info():
    d = S.devinfo()
    rc = L.b200.spmv_b200_device_info(C.byref(d))
    if rc:
        raise RuntimeError(L.last_error())
    return {
        "name": d.name.decode(),
        "cc": (d.cc_major, d.cc_minor),
        "sm_count": d.sm_count,
        "l2_mb": d.l2_bytes_mb,
        "hbm_bytes": d.hbm_bytes,
        "max_smem_per_block": d.max_smem_per_block,
    }


# --------------------------------------------------------- device-resident API --
def _stream_ptr(stream):
    import torch
    if stream is None:
        stream = torch.cuda.current_stream()
    return C.c_void_p(stream.cuda_stream)


def _dev_ptr(t, n, what):
    import torch
    assert isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64 and t.is_contiguous(), \
        f"{what} must be a contiguous float64 CUDA tensor"
    assert t.numel() >= n, f"{what} has {t.numel()} entries, needs {n}"
    return C.c_void_p(t.data_ptr())


class CsrDevice:
    """A CSR matrix resident in HBM (spmv_b200_csr, include/spmv_b200.h)."""

    def __init__(self, handle):
        if not handle:
            raise RuntimeError(f"CSR handle creation failed: {L.last_error()}")
        self._h = C.c_void_p(handle)
        self.M = L.b200.spmv_b200_csr_rows(self._h)
        self.N = L.b200.spmv_b200_csr_cols(self._h)
        self.NZ = L.b200.spmv_b200_csr_nnz(self._h)

    @classmethod
    def from_host(cls, A):
        return cls(L.b200.spmv_b200_csr_create(A.ptr))

    @classmethod
    def from_arrays(cls, M, n_local, IRP, JA, AS, col_offset=0, cuts=()):
        IRP = np.ascontiguousarray(IRP)
        assert IRP.dtype in (np.int32, np.int64)
        JA = np.ascontiguousarray(JA, np.int32)
        AS = np.ascontiguousarray(AS, np.float64)
        cuts_a = np.ascontiguousarray(cuts, np.int64)
        return cls(L.b200.spmv_b200_csr_create_ex(
            M, n_local, int(IRP[-1]), IRP.ctypes.data_as(C.c_void_p), IRP.dtype.itemsize,
            JA.ctypes.data_as(L.c_ip), AS.ctypes.data_as(L.c_dp), col_offset,
            cuts_a.ctypes.data_as(L.c_i64p), len(cuts_a)))

    @classmethod
    def stencil27(cls, nx, ny, nz, z0=0, z1=None, col_offset=0, n_local=None, cuts=()):
        z1 = nz if z1 is None else z1
        n_local = nx * ny * nz if n_local is None else n_local
        cuts_a = np.ascontiguousarray(cuts, np.int64)
        return cls(L.b200.spmv_b200_csr_gen_stencil27(nx, ny, nz, z0, z1, col_offset, n_local,
                                                      cuts_a.ctypes.data_as(L.c_i64p), len(cuts_a)))

    @classmethod
    def from_coo(cls, M, N, row, col, val, sum_duplicates=False, stream=None):
        """CSR built on the GPU from COO triplets already in device memory
        (spmv_b200_csr_from_coo).  `row` and `col`: contiguous 1-D CUDA tensors of equal length,
        both int32 or both int64; `val`: contiguous float64 CUDA tensor of the same length.  Row r
        lists its entries in increasing column order; entries with equal (row, col) keep their
        input order, or with `sum_duplicates` become one entry holding their left-to-right sum.
        Ordered after earlier work on `stream` (default: torch's current stream); synchronous.
        The tensors are not retained."""
        import torch
        for name, t in (("row", row), ("col", col), ("val", val)):
            if not isinstance(t, torch.Tensor):
                raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
            if not t.is_cuda or t.layout != torch.strided or t.dim() != 1 or not t.is_contiguous():
                raise ValueError(f"{name} must be a contiguous 1-D CUDA tensor")
        if row.dtype != col.dtype or row.dtype not in (torch.int32, torch.int64):
            raise TypeError(f"row and col must both be int32 or both int64, got {row.dtype} and {col.dtype}")
        if val.dtype != torch.float64:
            raise TypeError(f"val must be float64, got {val.dtype}")
        n = row.numel()
        if col.numel() != n or val.numel() != n:
            raise ValueError(f"row, col and val have {n}, {col.numel()} and {val.numel()} entries")
        return cls(L.b200.spmv_b200_csr_from_coo(
            int(M), int(N), n, row.data_ptr(), col.data_ptr(), row.element_size(), val.data_ptr(),
            int(bool(sum_duplicates)), _stream_ptr(stream)))

    @classmethod
    def from_torch(cls, t, sum_duplicates=False, stream=None):
        """CSR built on the GPU from a 2-D float64 CUDA tensor in torch.sparse_coo (coalesced or
        not) or torch.sparse_csr layout; see from_coo.  A CSR tensor's row offsets are expanded
        to row indices on the device first."""
        import torch
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"expected a torch.Tensor, got {type(t).__name__}")
        if t.layout not in (torch.sparse_coo, torch.sparse_csr):
            raise TypeError(f"layout {t.layout} is not torch.sparse_coo or torch.sparse_csr")
        if t.dtype != torch.float64:
            raise TypeError(f"dtype {t.dtype} is not torch.float64")
        if not t.is_cuda:
            raise ValueError(f"tensor is on {t.device}, not on a CUDA device")
        if t.dim() != 2 or t.sparse_dim() != 2 or t.dense_dim() != 0:
            raise ValueError(f"need a 2-D sparse matrix without batch or dense dimensions, got shape "
                             f"{tuple(t.shape)} with {t.sparse_dim()} sparse and {t.dense_dim()} dense dimensions")
        M, N = t.shape
        if t.layout == torch.sparse_coo:
            idx = t._indices()
            return cls.from_coo(M, N, idx[0].contiguous(), idx[1].contiguous(), t._values().contiguous(),
                                sum_duplicates, stream)
        crow, col = t.crow_indices(), t.col_indices()
        with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream()):
            row = torch.repeat_interleave(crow.diff(), output_size=col.numel())
        return cls.from_coo(M, N, row, col.contiguous(), t.values().contiguous(), sum_duplicates, stream)

    def _check(self, rc):
        if rc:
            raise RuntimeError(f"libspmv_b200: {L.last_error()} (rc={rc})")

    def spmv(self, x, y, kernel=2, warps_per_block=4, stream=None, rows=None, push=None):
        """y = A x on the current (or given) torch stream.  `rows=(r0,r1)` restricts to a
        row range declared with `cuts` at creation; `push=[(r0,r1,dst_ptr),...]` adds the
        fused peer-store epilogue."""
        xp, yp = _dev_ptr(x, self.N, "x"), _dev_ptr(y, self.M, "y")
        st = _stream_ptr(stream)
        if rows is None and push is None:
            self._check(L.b200.spmv_b200_csr_spmv(self._h, kernel, warps_per_block, xp, yp, st))
        elif push is None:
            self._check(L.b200.spmv_b200_csr_spmv_rows(self._h, kernel, warps_per_block, rows[0],
                                                       rows[1], xp, yp, st))
        else:
            r0, r1 = rows if rows is not None else (0, self.M)
            n = len(push)
            a0 = (C.c_int64 * max(n, 1))(*[p[0] for p in push])
            a1 = (C.c_int64 * max(n, 1))(*[p[1] for p in push])
            dst = (C.c_void_p * max(n, 1))(*[p[2] for p in push])
            self._check(L.b200.spmv_b200_csr_spmv_rows_push(self._h, kernel, warps_per_block, r0,
                                                            r1, xp, yp, n, a0, a1, dst, st))
        return y

    def spmv_fused(self, x, y, alpha=1.0, beta=0.0, z=None, w=None, dot=None, kernel=4,
                   warps_per_block=4, stream=None):
        """y = alpha*A x + beta*z and (if `dot`, a 1-element CUDA tensor, is given) dot[0] = sum y*w
        in one pass over the matrix (spmv_b200_csr_spmv_fused)."""
        zp = _dev_ptr(z, self.M, "z") if z is not None else None
        wp = _dev_ptr(w, self.M, "w") if w is not None else None
        dp = _dev_ptr(dot, 1, "dot") if dot is not None else None
        self._check(L.b200.spmv_b200_csr_spmv_fused(self._h, kernel, warps_per_block, _dev_ptr(x, self.N, "x"),
                                                    _dev_ptr(y, self.M, "y"), alpha, beta, zp, wp, dp,
                                                    _stream_ptr(stream)))
        return y

    def spmm(self, X, Y, stream=None):
        """Y[M, k] = A X[N, k] for k = 2 or 4 right-hand sides, both row-major CUDA tensors
        (spmv_b200_csr_spmm): one pass over the matrix."""
        k = int(X.shape[1])
        assert X.is_contiguous() and Y.is_contiguous() and tuple(Y.shape) == (self.M, k) and X.shape[0] >= self.N
        self._check(L.b200.spmv_b200_csr_spmm(self._h, k, _dev_ptr(X, self.N * k, "X"), _dev_ptr(Y, self.M * k, "Y"),
                                              _stream_ptr(stream)))
        return Y

    def spmv_host(self, x, y, kernel=4, warps_per_block=4):
        """Host x (numpy, N) in, host y (numpy, M) out: upload, kernels and download pipelined
        (spmv_b200_csr_spmv_host).  Returns the span of the kernels in ms."""
        assert x.dtype == np.float64 and y.dtype == np.float64 and x.size >= self.N and y.size >= self.M
        ms = C.c_double()
        self._check(L.b200.spmv_b200_csr_spmv_host(self._h, kernel, warps_per_block, x.ctypes.data_as(C.c_void_p),
                                                   y.ctypes.data_as(C.c_void_p), C.byref(ms)))
        return ms.value

    def sell_info(self, build=False):
        out = (C.c_int64 * 11)()
        self._check(L.b200.spmv_b200_csr_sell_info(self._h, int(build), out, 11))
        keys = ("state", "panels", "sigma", "slices", "slots", "nnz_in_slices", "long_rows", "gather_span_ppm",
                "chunk", "split_rows", "pieces")
        return dict(zip(keys, list(out)))

    def codes_info(self):
        """Column codes of the staged row-tile plans built so far (spmv_b200_csr_codes_info):
        state (0 none built, 1 coded, -1 a plan keeps int32 columns), coded tiles, the largest
        dictionary of a tile and the bytes of the code blocks."""
        out = (C.c_int64 * 4)()
        self._check(L.b200.spmv_b200_csr_codes_info(self._h, out, 4))
        return dict(zip(("state", "tiles", "max_dict", "bytes"), list(out)))

    def sell_download(self):
        info = self.sell_info()
        assert info["state"] == 1, "no SELL-P plan on this handle"
        K, S_, slots = info["panels"], info["slices"], info["slots"]
        soff = np.zeros(K * (S_ + 1), np.int64)
        perm = np.zeros(K * S_ * 32, np.int32)
        ja = np.zeros(slots, np.int32)
        as_ = np.zeros(slots, np.float64)
        self._check(L.b200.spmv_b200_csr_sell_download(self._h, soff.ctypes.data_as(L.c_i64p),
                                                       perm.ctypes.data_as(L.c_ip), ja.ctypes.data_as(L.c_ip),
                                                       as_.ctypes.data_as(L.c_dp)))
        return soff.reshape(K, S_ + 1), perm.reshape(K, S_ * 32), ja, as_

    def time(self, x, y, kernel=2, warps_per_block=4, warmup=3, reps=20, flush_l2=False, stream=None):
        """Per-launch milliseconds (CUDA events on the launching stream)."""
        ms = (C.c_double * reps)()
        self._check(L.b200.spmv_b200_csr_time(self._h, kernel, warps_per_block,
                                              _dev_ptr(x, self.N, "x"), _dev_ptr(y, self.M, "y"),
                                              warmup, reps, int(flush_l2), ms, _stream_ptr(stream)))
        return list(ms)

    def launches(self, kernel):
        return L.b200.spmv_b200_csr_launches(self._h, kernel)

    def plan_info(self):
        out = (C.c_int64 * 10)()
        self._check(L.b200.spmv_b200_csr_plan_info(self._h, out, 10))
        return list(out)

    def download(self):
        irp = np.zeros(self.M + 1, np.int64)
        ja = np.zeros(self.NZ, np.int32)
        as_ = np.zeros(self.NZ, np.float64)
        self._check(L.b200.spmv_b200_csr_download(self._h, irp.ctypes.data_as(L.c_i64p),
                                                  ja.ctypes.data_as(L.c_ip), as_.ctypes.data_as(L.c_dp)))
        return irp, ja, as_

    def to_hll(self):
        return HllDevice(L.b200.spmv_b200_hll_from_csr(self._h))

    def transpose(self):
        """Aᵀ as a new resident CSR built on the GPU (spmv_b200_csr_transpose): row j lists column j
        of A in increasing row order, duplicates kept.  A shard gives the transpose of its local
        block.  Both handles are independent."""
        return CsrDevice(L.b200.spmv_b200_csr_transpose(self._h))

    def matmul(self, B):
        """C = A·B as a new resident CSR built on the GPU (spmv_b200_csr_spgemm): M rows, B.N
        columns, each row's columns once in increasing order, explicit zeros kept.  C[i][j] is the
        left-to-right sum, in FP64 without fused multiply-adds, of the products a_p·b_q landing in
        column j, taken for p in A's row i and q in B's row ja_A[p], both in stored order.  A shard
        multiplies its local block.  All three handles are independent."""
        if not isinstance(B, CsrDevice):
            raise TypeError(f"B must be a CsrDevice, got {type(B).__name__}")
        if self.N != B.M:
            raise ValueError(f"A has {self.N} columns but B has {B.M} rows")
        return CsrDevice(L.b200.spmv_b200_csr_spgemm(self._h, B._h))

    def close(self):
        if self._h:
            L.b200.spmv_b200_csr_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HllDevice:
    """An HLL matrix resident in HBM (spmv_b200_hll)."""

    def __init__(self, handle):
        if not handle:
            raise RuntimeError(f"HLL handle creation failed: {L.last_error()}")
        self._h = C.c_void_p(handle)
        self.M = L.b200.spmv_b200_hll_rows(self._h)
        self.N = L.b200.spmv_b200_hll_cols(self._h)
        self.NZ = L.b200.spmv_b200_hll_nnz(self._h)
        self.num_hacks = L.b200.spmv_b200_hll_num_hacks(self._h)
        self.slots = L.b200.spmv_b200_hll_slots(self._h)

    @classmethod
    def from_host(cls, H):
        return cls(L.b200.spmv_b200_hll_create(H.ptr, int(H.is_col_major)))

    def _check(self, rc):
        if rc:
            raise RuntimeError(f"libspmv_b200: {L.last_error()} (rc={rc})")

    def spmv(self, x, y, kernel=2, warps_per_block=4, stream=None):
        self._check(L.b200.spmv_b200_hll_spmv(self._h, kernel, warps_per_block,
                                              _dev_ptr(x, self.N, "x"), _dev_ptr(y, self.M, "y"),
                                              _stream_ptr(stream)))
        return y

    def spmv_fused(self, x, y, alpha=1.0, beta=0.0, z=None, w=None, dot=None, kernel=2,
                   warps_per_block=4, stream=None):
        zp = _dev_ptr(z, self.M, "z") if z is not None else None
        wp = _dev_ptr(w, self.M, "w") if w is not None else None
        dp = _dev_ptr(dot, 1, "dot") if dot is not None else None
        self._check(L.b200.spmv_b200_hll_spmv_fused(self._h, kernel, warps_per_block, _dev_ptr(x, self.N, "x"),
                                                    _dev_ptr(y, self.M, "y"), alpha, beta, zp, wp, dp,
                                                    _stream_ptr(stream)))
        return y

    def spmv_host(self, x, y, kernel=2, warps_per_block=4):
        assert x.dtype == np.float64 and y.dtype == np.float64 and x.size >= self.N and y.size >= self.M
        ms = C.c_double()
        self._check(L.b200.spmv_b200_hll_spmv_host(self._h, kernel, warps_per_block, x.ctypes.data_as(C.c_void_p),
                                                   y.ctypes.data_as(C.c_void_p), C.byref(ms)))
        return ms.value

    def sell_info(self, build=False):
        out = (C.c_int64 * 8)()
        self._check(L.b200.spmv_b200_hll_sell_info(self._h, int(build), out, 8))
        keys = ("state", "panels", "sigma", "slices", "slots", "nnz_in_slices", "long_rows", "gather_span_ppm")
        return dict(zip(keys, list(out)))

    def time(self, x, y, kernel=2, warps_per_block=4, warmup=3, reps=20, flush_l2=False, stream=None):
        ms = (C.c_double * reps)()
        self._check(L.b200.spmv_b200_hll_time(self._h, kernel, warps_per_block,
                                              _dev_ptr(x, self.N, "x"), _dev_ptr(y, self.M, "y"),
                                              warmup, reps, int(flush_l2), ms, _stream_ptr(stream)))
        return list(ms)

    def launches(self, kernel):
        return L.b200.spmv_b200_hll_launches(self._h, kernel)

    def download(self):
        hoff = np.zeros(self.num_hacks + 1, np.int64)
        ja = np.zeros(self.slots, np.int32)
        as_ = np.zeros(self.slots, np.float64)
        self._check(L.b200.spmv_b200_hll_download(self._h, hoff.ctypes.data_as(L.c_i64p),
                                                  ja.ctypes.data_as(L.c_ip), as_.ctypes.data_as(L.c_dp)))
        return hoff, ja, as_

    def close(self):
        if self._h:
            L.b200.spmv_b200_hll_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def roofline_bytes(n_rows, n_cols, nnz):
    """Minimum-traffic bytes of one FP64 CSR/HLL SpMV (BASELINE.json north_star):
    12*nnz + 4*(n_rows+1) + 8*n_rows + 8*n_cols."""
    return 12 * nnz + 4 * (n_rows + 1) + 8 * n_rows + 8 * n_cols
