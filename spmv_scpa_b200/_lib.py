"""Loads the two in-tree shared objects and declares their C signatures.

libspmv_b200.so  CUDA kernels + C ABI (include/cuda_csr.h, cuda_hll.h,
                 cuda_timer.h, spmv_b200.h)
libspmv_host.so  C host layer (include/csr.h, hll.h, vector.h, utils.h,
                 logger.h, mmio.h, spmv_gen.h)

There is no fallback: if a library is missing this module raises and tells the
user to build (`python -c "import __graft_entry__ as g; g.build()"` or `make`).
"""
import ctypes as C
import os

from . import structs as S

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "lib")


class BuildMissing(ImportError):
    pass


def _load(name):
    path = os.path.join(LIB_DIR, name)
    if not os.path.exists(path):
        raise BuildMissing(
            f"{path} not found: build the extension first (make -C {os.path.dirname(_HERE)} "
            "or __graft_entry__.build()); spmv_scpa_b200 has no CPU or pure-Python fallback")
    return C.CDLL(path, mode=C.RTLD_GLOBAL)


b200 = _load("libspmv_b200.so")
host = _load("libspmv_host.so")

_p = C.POINTER
c_i64 = C.c_int64
c_i64p = _p(C.c_int64)
c_ip = _p(C.c_int)
c_dp = _p(C.c_double)
vp = C.c_void_p


def _sig(lib, name, restype, *argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = list(argtypes)
    return fn


# ---- reference boundary (include/cuda_csr.h, include/cuda_hll.h) ------------
CSR_ENTRY_POINTS = (
    "csr_spmv_cuda_thread_row",
    "csr_spmv_cuda_warp_row",
    "csr_spmv_cuda_halfwarp_row",
    "csr_spmv_cuda_block_row",
    "csr_spmv_cuda_halfwarp_row_text",
)
HLL_ENTRY_POINTS = (
    "hll_spmv_cuda_threads_row_major",
    "hll_spmv_cuda_threads_col_major",
    "hll_spmv_cuda_warp_block",
    "hll_spmv_cuda_halfwarp_row",
)
_sig(b200, "set_csr_warps_per_block", None, C.c_int)
_sig(b200, "set_hll_warps_per_block", None, C.c_int)
for _n in CSR_ENTRY_POINTS:
    _sig(b200, _n, C.c_double, _p(S.sparse_csr), c_dp, c_dp, vp)
for _n in HLL_ENTRY_POINTS:
    _sig(b200, _n, C.c_double, _p(S.sparse_hll), c_dp, c_dp, vp)

# ---- include/cuda_timer.h ----------------------------------------------------
_sig(b200, "timer_init", C.c_int, _p(S.cuda_timer))
_sig(b200, "timer_start", None, _p(S.cuda_timer), vp)
_sig(b200, "timer_stop", C.c_double, _p(S.cuda_timer), vp)
_sig(b200, "timer_destroy", None, _p(S.cuda_timer))

# ---- include/spmv_b200.h -----------------------------------------------------
_sig(b200, "spmv_b200_last_error", C.c_char_p)
_sig(b200, "spmv_b200_version", C.c_char_p)
_sig(b200, "spmv_b200_device_count", C.c_int)
_sig(b200, "spmv_b200_set_device", C.c_int, C.c_int)
_sig(b200, "spmv_b200_device_info", C.c_int, _p(S.devinfo))
_sig(b200, "spmv_b200_dmalloc", vp, C.c_size_t)
_sig(b200, "spmv_b200_dfree", C.c_int, vp)
_sig(b200, "spmv_b200_h2d", C.c_int, vp, vp, C.c_size_t, vp)
_sig(b200, "spmv_b200_d2h", C.c_int, vp, vp, C.c_size_t, vp)
_sig(b200, "spmv_b200_dmemset", C.c_int, vp, C.c_int, C.c_size_t, vp)
_sig(b200, "spmv_b200_stream_sync", C.c_int, vp)
_sig(b200, "spmv_b200_host_alloc", vp, C.c_size_t)
_sig(b200, "spmv_b200_host_free", C.c_int, vp)
_sig(b200, "spmv_b200_flush_l2", C.c_int, vp)

_sig(b200, "spmv_b200_csr_create", vp, _p(S.sparse_csr))
_sig(b200, "spmv_b200_csr_create_ex", vp, c_i64, c_i64, c_i64, vp, C.c_int, c_ip, c_dp, c_i64,
     c_i64p, C.c_int)
_sig(b200, "spmv_b200_csr_gen_stencil27", vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_i64,
     c_i64, c_i64p, C.c_int)
_sig(b200, "spmv_b200_csr_transpose", vp, vp)
_sig(b200, "spmv_b200_csr_spgemm", vp, vp, vp)
_sig(b200, "spmv_b200_csr_from_coo", vp, c_i64, c_i64, c_i64, vp, vp, C.c_int, vp, C.c_int, vp)
_sig(b200, "spmv_b200_csr_rows", c_i64, vp)
_sig(b200, "spmv_b200_csr_cols", c_i64, vp)
_sig(b200, "spmv_b200_csr_nnz", c_i64, vp)
_sig(b200, "spmv_b200_csr_download", C.c_int, vp, c_i64p, c_ip, c_dp)
_sig(b200, "spmv_b200_csr_plan_info", C.c_int, vp, c_i64p, C.c_int)
_sig(b200, "spmv_b200_csr_spmv", C.c_int, vp, C.c_int, C.c_int, vp, vp, vp)
_sig(b200, "spmv_b200_csr_spmv_rows", C.c_int, vp, C.c_int, C.c_int, c_i64, c_i64, vp, vp, vp)
_sig(b200, "spmv_b200_csr_spmv_rows_push", C.c_int, vp, C.c_int, C.c_int, c_i64, c_i64, vp, vp,
     C.c_int, c_i64p, c_i64p, _p(vp), vp)
_sig(b200, "spmv_b200_csr_launches", C.c_int, vp, C.c_int)
_sig(b200, "spmv_b200_csr_time", C.c_int, vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int,
     c_dp, vp)
_sig(b200, "spmv_b200_csr_destroy", None, vp)

_sig(b200, "spmv_b200_hll_create", vp, _p(S.sparse_hll), C.c_int)
_sig(b200, "spmv_b200_hll_from_csr", vp, vp)
_sig(b200, "spmv_b200_hll_rows", c_i64, vp)
_sig(b200, "spmv_b200_hll_cols", c_i64, vp)
_sig(b200, "spmv_b200_hll_nnz", c_i64, vp)
_sig(b200, "spmv_b200_hll_num_hacks", c_i64, vp)
_sig(b200, "spmv_b200_hll_slots", c_i64, vp)
_sig(b200, "spmv_b200_hll_download", C.c_int, vp, c_i64p, c_ip, c_dp)
_sig(b200, "spmv_b200_hll_spmv", C.c_int, vp, C.c_int, C.c_int, vp, vp, vp)
_sig(b200, "spmv_b200_hll_launches", C.c_int, vp, C.c_int)
_sig(b200, "spmv_b200_hll_time", C.c_int, vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int,
     c_dp, vp)
_sig(b200, "spmv_b200_hll_destroy", None, vp)

_sig(b200, "spmv_b200_release_all", None)
_sig(b200, "spmv_b200_set_timing", None, C.c_int, C.c_int)
_sig(b200, "spmv_b200_counters", None, c_i64p, c_i64p, c_i64p)
_sig(b200, "spmv_b200_set_knob", C.c_int, C.c_char_p, C.c_int)
_sig(b200, "spmv_b200_host_register", C.c_int, vp, C.c_size_t)
_sig(b200, "spmv_b200_host_copy", C.c_int, vp, vp, C.c_size_t)
_sig(b200, "spmv_b200_host_unregister", C.c_int, vp)
_sig(b200, "spmv_b200_set_cache_policy", C.c_int, C.c_int)
_sig(b200, "spmv_b200_invalidate", None, vp)
_sig(b200, "spmv_b200_csr_spmm", C.c_int, vp, C.c_int, vp, vp, vp)
_sig(b200, "spmv_b200_csr_spmv_fused", C.c_int, vp, C.c_int, C.c_int, vp, vp, C.c_double, C.c_double,
     vp, vp, vp, vp)
_sig(b200, "spmv_b200_hll_spmv_fused", C.c_int, vp, C.c_int, C.c_int, vp, vp, C.c_double, C.c_double,
     vp, vp, vp, vp)
_sig(b200, "spmv_b200_csr_spmv_host", C.c_int, vp, C.c_int, C.c_int, vp, vp, c_dp)
_sig(b200, "spmv_b200_hll_spmv_host", C.c_int, vp, C.c_int, C.c_int, vp, vp, c_dp)
_sig(b200, "spmv_b200_csr_sell_info", C.c_int, vp, C.c_int, c_i64p, C.c_int)
_sig(b200, "spmv_b200_csr_codes_info", C.c_int, vp, c_i64p, C.c_int)
_sig(b200, "spmv_b200_hll_sell_info", C.c_int, vp, C.c_int, c_i64p, C.c_int)
_sig(b200, "spmv_b200_sell_plan", C.c_int, c_ip, c_i64, C.c_int, C.c_int, c_ip, c_i64p)
_sig(b200, "spmv_b200_sell_plan_vrows", C.c_int, c_i64p, c_i64, C.c_int, C.c_int, c_i64p, c_ip, c_i64p)
_sig(b200, "spmv_b200_csr_sell_download", C.c_int, vp, c_i64p, c_ip, c_ip, c_dp)

_sig(b200, "spmv_b200_ipc_export", C.c_int, vp, _p(C.c_ubyte))
_sig(b200, "spmv_b200_ipc_open", C.c_int, _p(C.c_ubyte), _p(vp))
_sig(b200, "spmv_b200_ipc_close", C.c_int, vp)
_sig(b200, "spmv_b200_enable_peer", C.c_int, C.c_int)
_sig(b200, "spmv_b200_signal_peers", C.c_int, vp, C.c_int, _p(vp), vp)
_sig(b200, "spmv_b200_wait_peers", C.c_int, vp, C.c_int, _p(vp), C.c_uint64, vp, vp)

# multi-GPU iterated SpMV
_sig(b200, "spmv_b200_partition_rows", C.c_int, c_i64, vp, C.c_int, C.c_int, C.c_int, c_i64p)
_sig(b200, "spmv_b200_shard_scan", C.c_int, c_i64, c_i64, vp, C.c_int, c_ip, _p(S.shard_desc))
_sig(b200, "spmv_b200_stencil27_shard_desc", C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
     _p(S.shard_desc))
_sig(b200, "spmv_b200_dist_make_plan", C.c_int, C.c_int, C.c_int, _p(S.shard_desc), C.c_int,
     _p(S.dist_plan))
_sig(b200, "spmv_b200_dist_create", vp, _p(S.dist_plan), _p(S.shard_desc), vp, C.c_int, C.c_int)
_sig(b200, "spmv_b200_dist_export", C.c_int, vp, _p(C.c_ubyte))
_sig(b200, "spmv_b200_dist_connect", C.c_int, vp, _p(C.c_ubyte))
_sig(b200, "spmv_b200_dist_set_x", C.c_int, vp, vp)
_sig(b200, "spmv_b200_dist_iterate", C.c_int, vp, C.c_int)
_sig(b200, "spmv_b200_dist_time", C.c_int, vp, C.c_int, C.c_int, c_dp)
_sig(b200, "spmv_b200_dist_sync", C.c_int, vp)
_sig(b200, "spmv_b200_dist_x", vp, vp)
_sig(b200, "spmv_b200_dist_xlocal", vp, vp)
_sig(b200, "spmv_b200_dist_get_x", C.c_int, vp, c_dp)
_sig(b200, "spmv_b200_dist_stream", vp, vp)
_sig(b200, "spmv_b200_dist_steps", c_i64, vp)
_sig(b200, "spmv_b200_dist_mode", C.c_int, vp)
_sig(b200, "spmv_b200_dist_has_graph", C.c_int, vp)
_sig(b200, "spmv_b200_dist_destroy", None, vp)
_sig(b200, "spmv_b200_dist_group_create", vp, _p(S.sparse_csr), C.c_int, C.c_int, C.c_int, C.c_int)
_sig(b200, "spmv_b200_dist_group_stencil27", vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
     C.c_int)
_sig(b200, "spmv_b200_dist_group_size", C.c_int, vp)
_sig(b200, "spmv_b200_dist_group_rank", vp, vp, C.c_int)
_sig(b200, "spmv_b200_dist_group_set_x", C.c_int, vp, c_dp)
_sig(b200, "spmv_b200_dist_group_iterate", C.c_int, vp, C.c_int, c_dp)
_sig(b200, "spmv_b200_dist_group_get_x", C.c_int, vp, c_dp)
_sig(b200, "spmv_b200_dist_group_destroy", None, vp)

# ---- host layer --------------------------------------------------------------
_sig(host, "io_load_csr", vp, C.c_char_p)
_sig(host, "csr_free", None, vp)
_sig(host, "csr_to_hll", vp, _p(S.sparse_csr), C.c_bool)
_sig(host, "hll_free", None, vp)
_sig(host, "vec_create", S.vec, C.c_size_t)
_sig(host, "vec_put", None, _p(S.vec))
_sig(host, "vec_fill", None, _p(S.vec), C.c_double)
_sig(host, "vec_fill_random", None, _p(S.vec))
_sig(host, "aligned_malloc", vp, C.c_size_t)
_sig(host, "validation_vec_result", C.c_int, S.vec, S.vec)
_sig(host, "logger_init", C.c_int, C.c_char_p)
_sig(host, "logger_close", None)
_sig(host, "bench_csr_serial", C.c_int, _p(S.sparse_csr), c_dp, _p(S.bench))
_sig(host, "bench_hll_serial", C.c_int, _p(S.sparse_hll), c_dp, _p(S.bench))
_sig(host, "bench_csr_omp_guided", C.c_int, _p(S.sparse_csr), c_dp, _p(S.bench_omp))
_sig(host, "bench_csr_omp_nnz_balancing", C.c_int, _p(S.sparse_csr), c_dp, _p(S.bench_omp))
_sig(host, "bench_hll_omp", C.c_int, _p(S.sparse_hll), c_dp, _p(S.bench_omp))
CSR_BENCH_FUNCS = ("bench_csr_cuda_thread_row", "bench_csr_cuda_warp_row",
                   "bench_csr_cuda_halfwarp_row", "bench_csr_cuda_block_row",
                   "bench_csr_cuda_halfwarp_row_text")
HLL_BENCH_FUNCS = ("bench_hll_cuda_threads_row_major", "bench_hll_cuda_threads_col_major",
                   "bench_hll_cuda_warp_block", "bench_hll_cuda_halfwarp_row")
for _n in CSR_BENCH_FUNCS:
    _sig(host, _n, C.c_int, _p(S.sparse_csr), c_dp, _p(S.bench_cuda))
for _n in HLL_BENCH_FUNCS:
    _sig(host, _n, C.c_int, _p(S.sparse_hll), c_dp, _p(S.bench_cuda))
_sig(host, "log_csr_serial_benchmark", None, _p(S.sparse_csr), S.bench)
_sig(host, "log_hll_serial_benchmark", None, _p(S.sparse_hll), S.bench)
_sig(host, "log_csr_omp_benchmark", None, _p(S.sparse_csr), S.bench_omp)
_sig(host, "log_hll_omp_benchmark", None, _p(S.sparse_hll), S.bench_omp)
_sig(host, "log_csr_cuda_benchmark", None, _p(S.sparse_csr), S.bench_cuda, C.c_int)
_sig(host, "log_hll_cuda_benchmark", None, _p(S.sparse_hll), S.bench_cuda, C.c_int)

_sig(host, "gen_poisson2d", vp, C.c_int, C.c_int)
_sig(host, "gen_stencil27", vp, C.c_int, C.c_int, C.c_int)
_sig(host, "gen_stencil27_rows", vp, C.c_int, C.c_int, C.c_int, c_i64, c_i64)
_sig(host, "gen_uniform_random", vp, C.c_int, C.c_int, C.c_uint64)
_sig(host, "gen_rmat", vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_uint64)
_sig(host, "gen_ragged", vp, C.c_int, C.c_int, C.c_uint64)
_sig(host, "gen_write_mtx", C.c_int, _p(S.sparse_csr), C.c_char_p)
_sig(host, "gen_mix64", C.c_uint64, C.c_uint64)


def last_error():
    return b200.spmv_b200_last_error().decode(errors="replace")
