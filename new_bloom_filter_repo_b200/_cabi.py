"""
ctypes binding of librbf_b200.so (include/rbf_b200.h).  No PyTorch, no CPU fallback:
if the library or a B200 is missing, this module raises -- it never computes on the host.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("RBF_B200_LIB") or os.path.join(_HERE, "librbf_b200.so")

_lib = None
_ctx = None
_lock = threading.RLock()       # re-entrant: ctx() loads the library under the same lock


class RbfError(RuntimeError):
    pass


class Seeds(C.Structure):
    _fields_ = [("h1", C.c_uint64), ("h2", C.c_uint64), ("act", C.c_uint64)]


class MaskInfo(C.Structure):
    _fields_ = [("n", C.c_uint64), ("ones", C.c_uint64), ("resid", C.c_uint64), ("l", C.c_uint64),
                ("wlen", C.c_uint64), ("act_T", C.c_uint64), ("p", C.c_double), ("k", C.c_double),
                ("floor_k", C.c_uint32), ("raw", C.c_uint32)]


ABI_VERSION = 2
IVC_SEEDS = (0x12345678, 0x87654321, 999)    # improved_video_compressor.py:62-63,94
BC_SEEDS = (0, 1, 999)                       # bloom_compress.py:163-164,195

EXPORTS = [
    "rbf_abi_version", "rbf_last_global_error", "rbf_ctx_create", "rbf_ctx_destroy", "rbf_last_error",
    "rbf_device_info", "rbf_set_option", "rbf_get_counter", "rbf_reset_counters", "rbf_sync",
    "rbf_timer_start", "rbf_timer_stop_ms",
    "rbf_xxh64", "rbf_hash_decimal", "rbf_hash_decimal_century", "rbf_probe_index",
    "rbf_activation_threshold", "rbf_optimal_params",
    "rbf_malloc", "rbf_free", "rbf_malloc_host", "rbf_free_host", "rbf_memcpy_h2d", "rbf_memcpy_d2h", "rbf_memset",
    "rbf_filter_create", "rbf_filter_destroy", "rbf_filter_add_indices", "rbf_filter_check_indices",
    "rbf_filter_add_strings", "rbf_filter_check_strings", "rbf_filter_get_bits", "rbf_filter_set_bits",
    "rbf_compress_mask", "rbf_decompress_mask",
    "rbf_stream_create", "rbf_stream_create_images", "rbf_stream_destroy", "rbf_stream_set_option", "rbf_stream_upload", "rbf_stream_frame_ptr", "rbf_stream_encode",
    "rbf_stream_encode_host", "rbf_stream_fetch", "rbf_stream_fetch_batch", "rbf_stream_decode_verify", "rbf_stream_decode", "rbf_stream_bitmap_region", "rbf_stream_stage_ms",
    "rbf_stream_gather_changed", "rbf_stream_apply_diff", "rbf_stream_download", "rbf_median_blur5", "rbf_stream_median5",
    "rbf_nccl_unique_id", "rbf_nccl_init", "rbf_nccl_allgather", "rbf_stream_allgather_bitmaps", "rbf_nccl_destroy",
    "rbf_peer_export", "rbf_peer_open", "rbf_peer_close", "rbf_peer_gather_init", "rbf_peer_gather_half", "rbf_peer_gather_shutdown",
]


def _sig(L):
    vp, u64, u32, i32, dbl = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_double
    P = C.POINTER
    L.rbf_abi_version.restype = i32
    L.rbf_last_global_error.restype = C.c_char_p
    L.rbf_ctx_create.argtypes = [i32, P(vp)]
    L.rbf_ctx_destroy.argtypes = [vp]
    L.rbf_ctx_destroy.restype = None
    L.rbf_last_error.argtypes = [vp]
    L.rbf_last_error.restype = C.c_char_p
    L.rbf_device_info.argtypes = [vp, C.c_char_p, i32, P(i32), P(i32), P(i32), P(u64)]
    L.rbf_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.rbf_get_counter.argtypes = [vp, C.c_char_p]
    L.rbf_get_counter.restype = C.c_int64
    L.rbf_reset_counters.argtypes = [vp]
    L.rbf_sync.argtypes = [vp]
    L.rbf_timer_start.argtypes = [vp]
    L.rbf_timer_stop_ms.argtypes = [vp, P(dbl)]
    L.rbf_xxh64.argtypes = [vp, u64, u64]
    L.rbf_xxh64.restype = u64
    L.rbf_hash_decimal.argtypes = [u32, u64]
    L.rbf_hash_decimal.restype = u64
    L.rbf_hash_decimal_century.argtypes = [u32, u64]
    L.rbf_hash_decimal_century.restype = u64
    L.rbf_probe_index.argtypes = [u64, u64, u32, u32]
    L.rbf_probe_index.restype = u32
    L.rbf_activation_threshold.argtypes = [dbl]
    L.rbf_activation_threshold.restype = u64
    L.rbf_optimal_params.argtypes = [u64, u64, P(dbl), P(dbl), P(u64)]
    L.rbf_malloc.argtypes = [vp, C.c_size_t, P(vp)]
    L.rbf_free.argtypes = [vp, vp]
    L.rbf_malloc_host.argtypes = [vp, C.c_size_t, P(vp)]
    L.rbf_free_host.argtypes = [vp, vp]
    L.rbf_memcpy_h2d.argtypes = [vp, vp, vp, C.c_size_t]
    L.rbf_memcpy_d2h.argtypes = [vp, vp, vp, C.c_size_t]
    L.rbf_memset.argtypes = [vp, vp, i32, C.c_size_t]
    L.rbf_filter_create.argtypes = [vp, u64, dbl, P(Seeds), P(vp)]
    L.rbf_filter_destroy.argtypes = [vp]
    L.rbf_filter_destroy.restype = None
    L.rbf_filter_add_indices.argtypes = [vp, vp, u32]
    L.rbf_filter_check_indices.argtypes = [vp, vp, u32, vp]
    L.rbf_filter_add_strings.argtypes = [vp, vp, vp, u32, i32]
    L.rbf_filter_check_strings.argtypes = [vp, vp, vp, u32, i32, vp]
    L.rbf_filter_get_bits.argtypes = [vp, vp]
    L.rbf_filter_set_bits.argtypes = [vp, vp]
    L.rbf_compress_mask.argtypes = [vp, vp, u64, P(Seeds), dbl, u64, P(MaskInfo), vp, vp]
    L.rbf_decompress_mask.argtypes = [vp, vp, u64, vp, u64, u64, dbl, P(Seeds), vp, P(u64)]
    L.rbf_stream_create.argtypes = [vp, u32, u32, u32, u32, u32, u32, P(vp)]
    L.rbf_stream_create_images.argtypes = [vp, u32, u32, u32, u32, u32, P(vp)]
    L.rbf_stream_destroy.argtypes = [vp]
    L.rbf_stream_destroy.restype = None
    L.rbf_stream_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.rbf_stream_upload.argtypes = [vp, u32, u32, vp]
    L.rbf_stream_frame_ptr.argtypes = [vp, u32, P(vp)]
    L.rbf_stream_encode.argtypes = [vp, vp, vp, u32, dbl, P(Seeds), vp, vp, vp]
    L.rbf_stream_encode_host.argtypes = [vp, vp, u32, dbl, P(Seeds), vp, vp, u64, vp, u64]
    L.rbf_stream_fetch.argtypes = [vp, u32, vp, vp, vp]
    L.rbf_stream_fetch_batch.argtypes = [vp, u32, u32, vp, u64, vp, u64, vp, u64]
    L.rbf_stream_decode_verify.argtypes = [vp, u32, vp]
    L.rbf_stream_decode.argtypes = [vp, u32, vp, vp, vp, P(Seeds), vp, u64, vp, u64, vp, u64, vp]
    L.rbf_stream_bitmap_region.argtypes = [vp, P(vp), P(u64)]
    L.rbf_stream_stage_ms.argtypes = [vp, vp]
    L.rbf_stream_gather_changed.argtypes = [vp, u32, vp, u64, vp]
    L.rbf_stream_apply_diff.argtypes = [vp, u32, u32, vp, vp, u64, P(u64)]
    L.rbf_stream_download.argtypes = [vp, u32, vp]
    L.rbf_median_blur5.argtypes = [vp, vp, u32, u32, u32, vp]
    L.rbf_stream_median5.argtypes = [vp, u32, vp]
    L.rbf_nccl_unique_id.argtypes = [vp]
    L.rbf_nccl_init.argtypes = [vp, vp, i32, i32]
    L.rbf_nccl_allgather.argtypes = [vp, vp, vp, u64]
    L.rbf_stream_allgather_bitmaps.argtypes = [vp, u32, u64, vp, vp]
    L.rbf_nccl_destroy.argtypes = [vp]
    L.rbf_peer_export.argtypes = [vp, vp, vp]
    L.rbf_peer_open.argtypes = [vp, vp, P(vp)]
    L.rbf_peer_close.argtypes = [vp, vp]
    L.rbf_peer_gather_init.argtypes = [vp, i32, i32, P(vp), P(vp)]
    L.rbf_peer_gather_half.argtypes = [vp, P(u32)]
    L.rbf_peer_gather_shutdown.argtypes = [vp]


def lib():
    """The loaded C-ABI library.  Raises RbfError if it has not been built (python __graft_entry__.py)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(SO_PATH):
                    raise RbfError("librbf_b200.so is not built (run `python -m new_bloom_filter_repo_b200.build`); "
                                   "this package has no CPU fallback")
                L = C.CDLL(SO_PATH)
                _sig(L)
                if L.rbf_abi_version() != ABI_VERSION:
                    raise RbfError("ABI version mismatch")
                _lib = L
    return _lib


def check(rc: int, ctx=None):
    if rc != 0:
        L = lib()
        msg = (L.rbf_last_error(ctx) if ctx else L.rbf_last_global_error()) or b""
        raise RbfError("rbf_b200 error %d: %s" % (rc, msg.decode("utf-8", "replace")))


def ctx():
    """Process-wide context on cuda:LOCAL_RANK (or RBF_DEVICE).  Raises when there is no B200."""
    global _ctx
    if _ctx is None:
        lib()                                             # load outside the critical section too (first call may be ctx())
        with _lock:
            if _ctx is None:
                dev = int(os.environ.get("RBF_DEVICE", os.environ.get("LOCAL_RANK", "0")))
                h = C.c_void_p()
                check(lib().rbf_ctx_create(dev, C.byref(h)))
                _ctx = h
                for key in ("query_variant", "insert_variant", "k1_variant", "encode_ranges", "pipe_k1_ctas_per_sm"):      # experiment knobs, e.g. RBF_QUERY_VARIANT=4
                    val = os.environ.get("RBF_" + key.upper())
                    if val is not None:
                        check(lib().rbf_set_option(h, key.encode(), int(val)), h)
    return _ctx


def device_info():
    name = C.create_string_buffer(256)
    sm, maj, mn, mem = C.c_int(), C.c_int(), C.c_int(), C.c_uint64()
    check(lib().rbf_device_info(ctx(), name, 256, C.byref(sm), C.byref(maj), C.byref(mn), C.byref(mem)), ctx())
    return {"name": name.value.decode(), "sm_count": sm.value, "cc": (maj.value, mn.value), "total_mem": mem.value}


def seeds_struct(seeds) -> Seeds:
    return Seeds(int(seeds[0]) & (2 ** 64 - 1), int(seeds[1]) & (2 ** 64 - 1), int(seeds[2]) & (2 ** 64 - 1))


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


# ---- exact host-side scalar helpers (run on the CPU inside the C library; used for parameters only)
def xxh64(data: bytes, seed: int = 0) -> int:
    return lib().rbf_xxh64(data, len(data), seed & (2 ** 64 - 1))


def activation_threshold(p_act: float) -> int:
    return lib().rbf_activation_threshold(float(p_act))


def optimal_params(n: int, ones: int):
    p, k, l = C.c_double(), C.c_double(), C.c_uint64()
    coded = lib().rbf_optimal_params(int(n), int(ones), C.byref(p), C.byref(k), C.byref(l))
    return bool(coded), p.value, k.value, int(l.value)
