"""ctypes binding of include/rsd.h.  Loading never touches the GPU (the CUDA context is created
lazily by the first compute call, in the calling process — the reference's callers fork,
IRMethods.py:411,489,512).  A missing librsd.so is a hard error: there is no fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(HERE, "librsd.so")

RSD_OK, RSD_EINVAL, RSD_ENODEV, RSD_ECUDA, RSD_ENOMEM, RSD_ECOSTS, RSD_ERANGE = range(7)
MODE_AUTO, MODE_I16X2, MODE_I32, MODE_F64 = 0, 1, 2, 3
MODE_NAMES = {1: "i16x2", 2: "i32", 3: "f64"}
OP_INSERT, OP_DELETE, OP_UPDATE = 0, 1, 2


class RsdError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"librsd error {code}: {msg}")
        self.code = code


u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)
intp = C.POINTER(C.c_int)
vp = C.c_void_p
i64 = C.c_int64
ci = C.c_int
u32 = C.c_uint32

# name -> (restype, argtypes); mirrors include/rsd.h one to one (tests/test_abi.py checks both ways)
SIGNATURES = {
    "rsd_abi_version": (ci, []),
    "rsd_last_error": (C.c_char_p, []),
    "rsd_device_count": (ci, []),
    "rsd_create": (ci, [ci, C.POINTER(vp)]),
    "rsd_destroy": (ci, [vp]),
    "rsd_host_alloc": (ci, [C.POINTER(vp), i64]),
    "rsd_host_free": (ci, [vp]),
    "rsd_set_costs": (ci, [vp, C.c_double, C.c_double, f64p]),
    "rsd_classify": (ci, [vp, u32, i64, i64, ci, intp, intp]),
    "rsd_pack_words": (i64, [i32p, i64, ci]),
    "rsd_pack": (ci, [u8p, i64p, i64, ci, u32p, i64p, i32p, u32p]),
    "rsd_distance_batch": (ci, [vp, u32p, i64p, i32p, i64, u32p, i64p, i32p, i64, i64, i64, i64, ci, u32, ci, f64p, intp]),
    "rsd_distance_batch_codes": (ci, [vp, u8p, i32p, u8p, i32p, i64, i64, i64, ci, u32, ci, f64p, intp]),
    "rsd_distance_batch_dev": (ci, [vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, ci, u32, ci, vp, intp, vp]),
    "rsd_matrix": (ci, [vp, u8p, C.c_int32, u8p, C.c_int32, f64p, u8p]),
    "rsd_script_batch": (ci, [vp, u32p, i64p, i32p, i64, u32p, i64p, i32p, i64, i64, ci, u32, ci, i64,
                              u8p, i32p, i32p, i32p, f64p, intp]),
    "rsd_patch_batch": (ci, [vp, u8p, i32p, i32p, i32p, i64,
                             u32p, i64p, i32p, i64, u32p, i64p, i32p, i64, u32p, i64p, i32p, i64,
                             i64, ci, i64, u8p, i32p, i32p]),
    "rsd_script_patch_check_batch": (ci, [vp, u32p, i64p, i32p, i64, u32p, i64p, i32p, i64, i64, ci, u32, ci, i64,
                                          u8p, i32p, i32p, i32p, f64p, u8p, intp]),
    "rsd_db_load": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32, i64]),
    "rsd_db_free": (ci, [vp]),
    "rsd_db_append": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32]),
    "rsd_db_layout": (ci, [vp, i64p, i64p, i64p, u32p]),
    "rsd_db_search_topk": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32, ci, ci, i64p, f64p, f64p, intp]),
    "rsd_db_search_topk_dev": (ci, [vp, vp, vp, vp, i64, i64, ci, u32, ci, ci, vp, vp, intp, vp]),
    "rsd_db_search_range": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32, C.c_double, ci, i64, i64p, i64p, f64p, intp]),
    "rsd_db_similarity": (ci, [vp, u8p, C.c_int32, ci, ci, i64p, f64p, f64p]),
    "rsd_db_similarity_batch": (ci, [vp, u8p, i64p, i64, ci, ci, i64p, f64p, f64p]),
    "rsd_db_idf_table": (ci, [vp, f64p, f64p]),
    "rsd_db_vector_similarity_batch": (ci, [vp, u8p, i64p, i64, ci, ci, ci, i64p, f64p, f64p]),
    "rsd_topk_merge": (ci, [i64p, f64p, ci, i64, ci, i64p, f64p]),
    "rsd_multi_create": (ci, [intp, ci, C.POINTER(vp)]),
    "rsd_multi_destroy": (ci, [vp]),
    "rsd_multi_device_count": (ci, [vp]),
    "rsd_multi_set_costs": (ci, [vp, C.c_double, C.c_double, f64p]),
    "rsd_multi_db_load": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32]),
    "rsd_multi_db_free": (ci, [vp]),
    "rsd_multi_db_append": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32]),
    "rsd_multi_db_search_topk": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32, ci, ci, i64p, f64p, f64p, intp]),
    "rsd_multi_db_similarity": (ci, [vp, u8p, i64p, i64, ci, ci, i64p, f64p, f64p]),
    "rsd_multi_db_idf_table": (ci, [vp, f64p, f64p]),
    "rsd_multi_db_vector_similarity": (ci, [vp, u8p, i64p, i64, ci, ci, ci, i64p, f64p, f64p]),
    "rsd_multi_db_search_range": (ci, [vp, u32p, i64p, i32p, i64, i64, ci, u32, C.c_double, ci, i64, i64p, i64p, f64p, intp]),
    "rsd_multi_launch_count": (i64, [vp]),
    "rsd_long_pair": (ci, [vp, u8p, i64, u8p, i64, ci, ci, i64, u8p, i32p, i32p, i64p, f64p, intp]),
    "rsd_long_pairs": (ci, [vp, ci, C.POINTER(vp), i64p, C.POINTER(vp), i64p, ci, ci, i64p,
                            C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i64p, f64p, intp]),
    "rsd_long_forward_ms": (C.c_double, [vp]),
    "rsd_launch_count": (i64, [vp]),
    "rsd_last_kernel_ms": (C.c_double, [vp]),
    "rsd_set_timing": (ci, [vp, ci]),
    "rsd_ubench": (ci, [vp, ci, f64p]),
}

_lib = None


def library_path() -> str:
    return _SO


def load_library():
    """dlopen librsd.so and set the prototypes.  Raises RsdError when the extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise RsdError(RSD_ENODEV, f"{_SO} not found: build it with `python __graft_entry__.py build` "
                                   "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(_SO)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.rsd_abi_version() != 1:
        raise RsdError(RSD_EINVAL, "librsd ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise RsdError(rc, load_library().rsd_last_error().decode("utf-8", "replace"))


def ptr(arr, typ):
    return arr.ctypes.data_as(C.POINTER(typ))
