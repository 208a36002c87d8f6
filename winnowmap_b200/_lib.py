import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libwinnowmap_b200.so")
_lib = None

u8p = C.POINTER(C.c_uint8)
i8p = C.POINTER(C.c_int8)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)
i64p = C.POINTER(C.c_int64)
u64p = C.POINTER(C.c_uint64)


class ExtZ(C.Structure):
    """wm_extz_t (include/winnowmap_b200.h), field order of ksw_extz_t (reference src/ksw2.h:23-32)."""
    _fields_ = [(n, C.c_int32) for n in ("max", "zdropped", "max_q", "max_t", "mqe", "mqe_t", "mte", "mte_q", "score",
                                          "reach_end", "n_cigar", "reserved")]


def lib_path():
    return _SO


def lib():
    """The C-ABI library.  Fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise RuntimeError(f"{_SO} is missing: build it with `python -m winnowmap_b200.build` "
                               "(winnowmap_b200 has no CPU fallback)")
        # the orchestration threads start many short OpenMP regions; spinning idle workers starve the CUDA driver threads
        os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
        L = C.CDLL(_SO)
        L.wm_version.restype = C.c_char_p
        L.wm_device_count.restype = C.c_int
        L.wm_set_device.argtypes = [C.c_int]
        L.wm_ksw_extd2_batch.argtypes = [C.c_int, u8p, i64p, u8p, i64p, i8p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         i32p, i32p, i32p, i32p, C.POINTER(ExtZ), u32p, i64p]
        L.wm_bloom_build.restype = C.c_void_p
        L.wm_bloom_build.argtypes = [u64p, C.c_int64]
        L.wm_bloom_bits.restype = C.c_uint64
        L.wm_bloom_bits.argtypes = [C.c_void_p]
        L.wm_bloom_table.restype = C.c_void_p
        L.wm_bloom_table.argtypes = [C.c_void_p]
        L.wm_bloom_destroy.argtypes = [C.c_void_p]
        L.wm_sketch_batch.argtypes = [C.c_void_p, C.c_int, C.c_char_p, i64p, u32p, C.c_int, C.c_int,
                                      C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
        L.wm_radix_sort_128x_batch.argtypes = [C.c_int, u64p, i64p]
        L.wm_radix_sort_128x_batch_timed.argtypes = [C.c_int, u64p, i64p, C.POINTER(C.c_float)]
        L.wm_chain_dp_batch.argtypes = [C.c_int, u64p, i64p] + [C.c_int] * 8 + [C.c_float, i32p, u64p, u64p, i64p]
        _lib = L
    return _lib
