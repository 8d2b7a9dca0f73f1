"""ctypes bindings to the in-tree native libraries.

``libtd_b200.so``  : sm_100a kernels + CUDA-VMM symmetric heap (needs a CUDA driver to *run*, not to load).
``libtd_host.so``  : CPU emulation runtime.

The libraries are built on first use by :mod:`triton_dist._build` (seconds; cached by content hash).  On a box
with a GPU the CUDA library is mandatory: ops raise instead of silently falling back to eager PyTorch.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

_LIBDIR = Path(__file__).resolve().parent / "lib"
_lock = threading.Lock()
_cuda = None
_host = None

c_void_p, c_int, c_uint, c_ll, c_ull, c_char_p = C.c_void_p, C.c_int, C.c_uint, C.c_longlong, C.c_ulonglong, C.c_char_p


class NativeError(RuntimeError):
    pass


def _ensure_built(which: str) -> Path:
    name = {"cuda": "libtd_b200.so", "host": "libtd_host.so"}[which]
    if which == "cuda":
        from . import _build as _b
        tmo = _b.debug_wait_timeout_ns()
        if tmo is not None:           # hang-detection variant (TD_DEBUG_WAITS=<ms>): built on first use, the default library is untouched
            name = f"libtd_b200_dbg{tmo // 1000000}.so"
    path = _LIBDIR / name
    if os.environ.get("TD_NO_AUTOBUILD") == "1" and path.exists():
        return path
    from . import _build
    return _build.build_cuda() if which == "cuda" else _build.build_host()


class GemmArgs(C.Structure):
    """Mirror of ``TdGemmArgs`` in csrc/gemm_sm100.cu (all fields 8 bytes)."""
    _fields_ = [(n, t) for n, t in [
        ("mode", c_ll), ("is_bf16", c_ll), ("bn", c_ll), ("cta_group", c_ll), ("group_m", c_ll),
        ("n_comm_ctas", c_ll), ("use_tma_store", c_ll), ("num_sms", c_ll),
        ("M", c_ll), ("N", c_ll), ("K", c_ll), ("m_rot", c_ll),
        ("A", c_void_p), ("a_rows", c_ll), ("lda", c_ll), ("a_nbuf", c_ll), ("a_buf_stride_bytes", c_ll),
        ("B", c_void_p), ("ldb", c_ll),
        ("C", c_void_p), ("c_rows", c_ll), ("ldc", c_ll), ("c_phase", c_void_p), ("c_nbuf", c_ll),
        ("c_buf_stride_bytes", c_ll), ("tile_expert", c_void_p), ("num_experts", c_ll),
        ("prof_buf", c_void_p), ("prof_cap", c_ll), ("prof_slots", c_ll),
        ("sfa", c_void_p), ("sfb", c_void_p), ("sfa_chunks", c_ll), ("sfb_chunks", c_ll),
        ("rank", c_ll), ("world", c_ll), ("symm_base", c_ull), ("symm_stride", c_ull), ("mc_base", c_ull),
        ("phase", c_void_p),
        ("ag_rows_per_rank", c_ll), ("ag_copy_local", c_ll), ("ag_skip_wait", c_ll),
        ("ag_a_local", c_void_p), ("ag_ws", c_void_p), ("ag_ws_buf_bytes", c_ll), ("ag_flags", c_void_p),
        ("ag_ready", c_void_p),
        ("rs_rows_per_rank", c_ll), ("rs_stage", c_void_p), ("rs_stage_buf_bytes", c_ll), ("rs_flags", c_void_p),
        ("rs_out", c_void_p), ("rs_ldo", c_ll),
        ("a_gather", c_void_p), ("a_gather_div", c_ll), ("a_gather_pad", c_ll), ("a_src_rows", c_ll), ("c_scatter", c_void_p),
        ("expert_stride_rows", c_ll),
        ("sk_ws", c_void_p), ("sk_ws_bytes", c_ll), ("sk_flags", c_void_p), ("sk_flag_count", c_ll), ("sk_max_parts", c_ll),
        ("rs_skip_wait", c_ll), ("rs_fp32", c_ll), ("ag_kslices", c_ll),
        ("row_scale", c_void_p), ("mrs_counter", c_void_p), ("mrs_total_padded", c_void_p), ("mrs_T", c_ll), ("mrs_topk", c_ll),
        ("mrs_allreduce", c_ll), ("mrs_chunk_n", c_ll),
        ("epd_send_off", c_void_p), ("epd_send_ids", c_void_p), ("epd_dest_off", c_void_p), ("epd_x", c_void_p),
        ("epd_topk", c_ll), ("epd_epr", c_ll), ("epd_cpd", c_ll), ("epd_rows_cap", c_ll), ("epd_meta", c_void_p), ("c_route", c_void_p),
        ("segk_off", c_void_p), ("segk_n", c_ll), ("scale_a", c_void_p), ("scale_b", c_void_p),
        ("ag_scale_ws", c_void_p), ("ag_sfa_local", c_void_p), ("ag_sfa_buf_chunks", c_ll),
    ]]


def _sig(lib, name, restype, argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = argtypes
    return fn


def cuda_lib():
    """Load (building if needed) the CUDA library.  Safe on CPU-only boxes (no libcuda link dependency)."""
    global _cuda
    with _lock:
        if _cuda is None:
            import torch  # noqa: F401  (loads libcudart.so.12 into the process first)
            lib = C.CDLL(str(_ensure_built("cuda")), mode=C.RTLD_GLOBAL)
            _sig(lib, "td_last_error", c_char_p, [])
            _sig(lib, "td_gemm_launch", c_int, [C.POINTER(GemmArgs), c_void_p])
            _sig(lib, "td_heap_create", c_void_p, [c_int, c_int, c_int, c_ull])
            _sig(lib, "td_heap_export_fd", c_int, [c_void_p])
            _sig(lib, "td_heap_map", c_int, [c_void_p, C.POINTER(c_int)])
            for n in ("td_heap_base", "td_heap_stride", "td_heap_bytes", "td_heap_mc_base"):
                _sig(lib, n, c_ull, [c_void_p])
            _sig(lib, "td_multicast_supported", c_int, [c_int])
            _sig(lib, "td_heap_mc_create", c_int, [c_void_p])
            _sig(lib, "td_heap_mc_import", c_int, [c_void_p, c_int])
            _sig(lib, "td_heap_mc_add_device", c_int, [c_void_p])
            _sig(lib, "td_heap_mc_bind_and_map", c_int, [c_void_p])
            _sig(lib, "td_heap_destroy", c_int, [c_void_p])
            _sig(lib, "td_stream_write_value32", c_int, [c_void_p, c_ull, c_uint])
            _sig(lib, "td_stream_wait_value32", c_int, [c_void_p, c_ull, c_uint, c_int])
            _sig(lib, "td_memcpy_async", c_int, [c_void_p, c_void_p, c_ull, c_void_p])
            _sig(lib, "td_device_info", c_int, [c_int, C.POINTER(c_int)])
            _sig(lib, "td_can_access_peer", c_int, [c_int, c_int])
            _sig(lib, "td_p2p_native_atomics", c_int, [c_int, c_int])
            _register_optional(lib)
            _cuda = lib
    return _cuda


_OPTIONAL = []  # (name, restype, argtypes) registered by kernel modules added later


def register(name, restype, argtypes):
    """Declare the signature of another exported launcher (called by the op modules at import time)."""
    _OPTIONAL.append((name, restype, argtypes))
    if _cuda is not None and hasattr(_cuda, name):
        _sig(_cuda, name, restype, argtypes)


def _register_optional(lib):
    for name, restype, argtypes in _OPTIONAL:
        if hasattr(lib, name):
            _sig(lib, name, restype, argtypes)


def host_lib():
    global _host
    with _lock:
        if _host is None:
            lib = C.CDLL(str(_ensure_built("host")))
            _sig(lib, "tdh_last_error", c_char_p, [])
            _sig(lib, "tdh_heap_create", c_void_p, [c_char_p, c_int, c_int, c_ull])
            _sig(lib, "tdh_heap_map", c_int, [c_void_p])
            _sig(lib, "tdh_heap_unlink", c_int, [c_void_p])
            for n in ("tdh_heap_base", "tdh_heap_stride", "tdh_heap_bytes"):
                _sig(lib, n, c_ull, [c_void_p])
            _sig(lib, "tdh_heap_destroy", c_int, [c_void_p])
            _sig(lib, "tdh_notify32", None, [c_void_p, c_uint, c_int])
            _sig(lib, "tdh_notify64", None, [c_void_p, c_ull, c_int])
            _sig(lib, "tdh_ld_acquire32", c_uint, [c_void_p])
            _sig(lib, "tdh_ld_acquire64", c_ull, [c_void_p])
            _sig(lib, "tdh_atomic_add32", c_uint, [c_void_p, c_uint])
            _sig(lib, "tdh_atomic_cas32", c_uint, [c_void_p, c_uint, c_uint])
            _sig(lib, "tdh_wait32", c_int, [c_void_p, c_uint, c_int, c_ll])
            _sig(lib, "tdh_wait32_n", c_int, [c_void_p, c_int, c_uint, c_int, c_ll])
            _sig(lib, "tdh_fence", None, [])
            _sig(lib, "tdh_barrier_all", c_int, [c_void_p, c_ull, c_uint, c_ll])
            _sig(lib, "tdh_memcpy", None, [c_void_p, c_void_p, c_ull])
            _host = lib
    return _host


_native_calls = 0


def native_calls() -> int:
    """Number of successful native launcher calls so far (every kernel launch goes through :func:`check`)."""
    return _native_calls


def check(rc: int, what: str = "native call"):
    global _native_calls
    _native_calls += 1
    if rc != 0:
        msg = cuda_lib().td_last_error().decode(errors="replace") if _cuda is not None else ""
        raise NativeError(f"{what} failed: {msg}")


def loaded_libraries():
    """Which native libraries this process has actually loaded (used by tests and bench.py)."""
    out = []
    if _cuda is not None:
        out.append(getattr(_cuda, "_name", str(_LIBDIR / "libtd_b200.so")))
    if _host is not None:
        out.append(str(_LIBDIR / "libtd_host.so"))
    return out
