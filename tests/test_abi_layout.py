"""The structs that cross the drop-in boundary (wm_mapopt_t / wm_reg1_t / wm_extra_t / wm_idxopt_t, include/winnowmap_b200.h)
against the reference's own mm_* structs (src/minimap.h:80-176): sizeof and the offset of every addressable field, the
reference side compiled from the reference's header by oracle/ref_harness.cpp (recorded under tests/golden/ref/)."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as ol  # noqa: E402


def _ref_layout():
    R = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_harness.so"))
    b = np.zeros(256, np.int64)
    R.ref_abi_layout.argtypes = [C.c_void_p, C.c_int]
    return b[:R.ref_abi_layout(b.ctypes.data, 256)]


def test_struct_layouts_equal_the_reference(request):
    from winnowmap_b200 import lib
    from winnowmap_b200.mapper import IdxOpt, MapOpt
    g = ol.RefGolden(request)
    L = lib()
    a = np.zeros(256, np.int64)
    L.wm_abi_layout.argtypes = [C.c_void_p, C.c_int]
    na = L.wm_abi_layout(a.ctypes.data, 256)
    assert na > 90
    g.check(_ref_layout, a[:na], a[:na].tolist())
    g.done()
    # the ctypes mirrors the Python callers use
    assert C.sizeof(MapOpt) == a[0] and C.sizeof(IdxOpt) == a[3]
    for i, (name, _) in enumerate(MapOpt._fields_):
        assert getattr(MapOpt, name).offset == a[4 + i], name
