"""ctypes loader for libjjschnorr_b200.so (the CUDA library; C ABI in include/jjschnorr_b200.h).

There is no fallback of any kind: if the shared library is missing, or no sm_100a device is usable,
every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("JJS_B200_LIB", os.path.join(_DIR, "libjjschnorr_b200.so"))  # override: A/B builds of the same ABI

EXPORTS = [
    "jjs_init", "jjs_destroy", "jjs_last_error", "jjs_device_count", "jjs_launch_count",
    "jjs_verify_single", "jjs_verify_double", "jjs_verify_vargen", "jjs_verify_aggregate",
    "jjs_verify_single_device", "jjs_verify_double_device", "jjs_verify_vargen_device",
    "jjs_challenge_only", "jjs_sign_batch", "jjs_profile_enable", "jjs_profile_collect", "jjs_subgroup_check", "jjs_fb_table_check", "jjs_verify_aggregate_device", "jjs_sign_aggregate_batch", "jjs_verify_ext", "jjs_points_to_ext", "jjs_multisig_combine",
    "jjs_verify_batch", "jjs_status_bitmap_device", "jjs_verify_batch_double", "jjs_verify_batch_vargen", "jjs_verify_batch_aggregate",
    "jjs_verify_mixed",
    "jjs_keyset_create", "jjs_keyset_destroy", "jjs_verify_keyed", "jjs_verify_keyed_device", "jjs_keyset_table_check",
    "jjs_keyset_create_limited", "jjs_keyset_info",
    "jjs_init_limited", "jjs_memory_info",
    "jjs_verify_all", "jjs_verify_all_device", "jjs_verify_all_mixed", "jjs_verify_all_mixed_device",
    "jjs_verify_grouped", "jjs_verify_grouped_device",
]


class Part(C.Structure):
    """struct jjs_part of include/jjschnorr_b200.h"""
    _fields_ = [("kind", C.c_int), ("pk", C.c_void_p), ("offsets", C.c_void_p), ("sig", C.c_void_p), ("msg32", C.c_void_p), ("n", C.c_size_t),
                ("status", C.c_void_p), ("c32", C.c_void_p), ("aggpk32", C.c_void_p), ("accept_bitmap", C.c_void_p)]


_lib = None


class NativeLibraryMissing(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryMissing(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  jubjub_schnorr_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz = C.c_void_p, C.c_size_t
    L.jjs_init.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.jjs_init.restype = C.c_int
    L.jjs_init_limited.argtypes = [C.POINTER(C.c_int), C.c_int, sz, C.POINTER(vp)]
    L.jjs_init_limited.restype = C.c_int
    L.jjs_memory_info.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
    L.jjs_memory_info.restype = C.c_int
    L.jjs_destroy.argtypes = [vp]
    L.jjs_destroy.restype = None
    L.jjs_last_error.argtypes = [vp]
    L.jjs_last_error.restype = C.c_char_p
    L.jjs_device_count.argtypes = [vp]
    L.jjs_device_count.restype = C.c_int
    L.jjs_launch_count.argtypes = [vp]
    L.jjs_launch_count.restype = C.c_uint64
    for name in ("jjs_verify_single", "jjs_verify_double", "jjs_verify_vargen"):
        f = getattr(L, name)
        f.argtypes = [vp, vp, vp, vp, sz, vp, vp]
        f.restype = C.c_int
    L.jjs_verify_batch.argtypes = [vp, vp, vp, vp, sz, vp]
    L.jjs_verify_batch.restype = C.c_int
    for name in ("jjs_verify_batch_double", "jjs_verify_batch_vargen"):
        f = getattr(L, name)
        f.argtypes = [vp, vp, vp, vp, sz, vp]
        f.restype = C.c_int
    L.jjs_verify_batch_aggregate.argtypes = [vp, vp, vp, vp, vp, sz, vp]
    L.jjs_verify_batch_aggregate.restype = C.c_int
    L.jjs_verify_mixed.argtypes = [vp, C.POINTER(Part), sz]
    L.jjs_verify_mixed.restype = C.c_int
    L.jjs_status_bitmap_device.argtypes = [vp, C.c_int, vp, sz, vp, vp]
    L.jjs_status_bitmap_device.restype = C.c_int
    L.jjs_verify_aggregate.argtypes = [vp, vp, vp, vp, vp, sz, vp, vp, vp]
    L.jjs_verify_aggregate.restype = C.c_int
    for name in ("jjs_verify_single_device", "jjs_verify_double_device", "jjs_verify_vargen_device"):
        f = getattr(L, name)
        f.argtypes = [vp, C.c_int, vp, vp, vp, sz, vp, vp, vp]
        f.restype = C.c_int
    L.jjs_challenge_only.argtypes = [vp, C.c_int, vp, vp, vp, sz, vp]
    L.jjs_challenge_only.restype = C.c_int
    L.jjs_sign_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, sz, vp, vp]
    L.jjs_sign_batch.restype = C.c_int
    L.jjs_profile_enable.argtypes = [vp, C.c_int]
    L.jjs_profile_enable.restype = None
    L.jjs_profile_collect.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.jjs_profile_collect.restype = C.c_int
    L.jjs_subgroup_check.argtypes = [vp, vp, sz, C.c_int, vp]
    L.jjs_subgroup_check.restype = C.c_int
    L.jjs_fb_table_check.argtypes = [vp, C.c_int, vp, sz, vp]
    L.jjs_fb_table_check.restype = C.c_int
    L.jjs_verify_aggregate_device.argtypes = [vp, C.c_int, vp, vp, vp, vp, vp, sz, vp, vp, vp, vp]
    L.jjs_verify_aggregate_device.restype = C.c_int
    L.jjs_sign_aggregate_batch.argtypes = [vp, vp, vp, vp, vp, sz, vp, vp]
    L.jjs_sign_aggregate_batch.restype = C.c_int
    L.jjs_verify_ext.argtypes = [vp, C.c_int, vp, vp, vp, sz, vp, vp]
    L.jjs_verify_ext.restype = C.c_int
    L.jjs_points_to_ext.argtypes = [vp, vp, vp, sz, vp]
    L.jjs_points_to_ext.restype = C.c_int
    L.jjs_multisig_combine.argtypes = [vp, vp, vp, vp, vp, vp, vp, sz, vp, vp, vp, vp]
    L.jjs_multisig_combine.restype = C.c_int
    L.jjs_keyset_create.argtypes = [vp, C.c_int, vp, sz, vp, C.POINTER(C.c_int)]
    L.jjs_keyset_create.restype = C.c_int
    L.jjs_keyset_destroy.argtypes = [vp, C.c_int]
    L.jjs_keyset_destroy.restype = C.c_int
    L.jjs_verify_keyed.argtypes = [vp, C.c_int, vp, vp, vp, sz, vp, vp, vp]
    L.jjs_verify_keyed.restype = C.c_int
    L.jjs_verify_keyed_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, sz, vp, vp, vp]
    L.jjs_verify_keyed_device.restype = C.c_int
    L.jjs_keyset_table_check.argtypes = [vp, C.c_int, vp, sz, vp]
    L.jjs_keyset_table_check.restype = C.c_int
    L.jjs_keyset_create_limited.argtypes = [vp, C.c_int, vp, sz, sz, vp, C.POINTER(C.c_int)]
    L.jjs_keyset_create_limited.restype = C.c_int
    L.jjs_keyset_info.argtypes = [vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_uint64)]
    L.jjs_keyset_info.restype = C.c_int
    L.jjs_verify_all.argtypes = [vp, C.c_int, vp, vp, vp, sz, vp, C.POINTER(C.c_int)]
    L.jjs_verify_all.restype = C.c_int
    L.jjs_verify_all_device.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, sz, vp, vp, vp]
    L.jjs_verify_all_device.restype = C.c_int
    L.jjs_verify_all_mixed.argtypes = [vp, C.POINTER(Part), sz, vp, C.POINTER(C.c_int)]
    L.jjs_verify_all_mixed.restype = C.c_int
    L.jjs_verify_all_mixed_device.argtypes = [vp, C.c_int, C.POINTER(Part), sz, vp, vp, vp, vp]
    L.jjs_verify_all_mixed_device.restype = C.c_int
    L.jjs_verify_grouped.argtypes = [vp, C.POINTER(Part), sz, vp, C.POINTER(C.c_uint64)]
    L.jjs_verify_grouped.restype = C.c_int
    L.jjs_verify_grouped_device.argtypes = [vp, C.c_int, C.POINTER(Part), sz, vp, vp, vp, vp]
    L.jjs_verify_grouped_device.restype = C.c_int
    _lib = L
    return L
