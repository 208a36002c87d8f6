"""ctypes bindings for the CPU oracle (oracle/libwm_oracle.so, a restatement) and for the
real reference (oracle/_ref/libref_harness.so), and the recorded answers of the reference
(RefGolden) that the tests compare with where the reference is not built.  TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "ref")
# WM_RECORD_REF_GOLDEN=1 (with oracle/_ref built): the tests call the reference and rewrite tests/golden/ref/
RECORD = os.environ.get("WM_RECORD_REF_GOLDEN") == "1"
_u8p = C.POINTER(C.c_uint8)
_i8p = C.POINTER(C.c_int8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_i32p = C.POINTER(C.c_int)


def _ptr(a, t):
    return a.ctypes.data_as(t)


def build_oracle():
    so = os.path.join(ORACLE_DIR, "libwm_oracle.so")
    src = os.path.join(ORACLE_DIR, "wm_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "libwm_oracle.so"], stdout=subprocess.DEVNULL)
    return so


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        L = C.CDLL(build_oracle())
        L.wmo_bloom_init.restype = C.c_void_p
        L.wmo_bloom_init.argtypes = [C.c_uint64]
        L.wmo_bloom_insert.argtypes = [C.c_void_p, C.c_uint64]
        L.wmo_bloom_contains.argtypes = [C.c_void_p, C.c_uint64]
        L.wmo_bloom_bits.restype = C.c_uint64
        L.wmo_bloom_bits.argtypes = [C.c_void_p]
        L.wmo_bloom_table.restype = C.c_void_p
        L.wmo_bloom_table.argtypes = [C.c_void_p]
        L.wmo_bloom_salts.argtypes = [C.c_void_p, _u32p]
        L.wmo_bloom_nsalt.argtypes = [C.c_void_p]
        L.wmo_bloom_free.argtypes = [C.c_void_p]
        L.wmo_sketch.restype = C.c_long
        L.wmo_sketch.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, _u64p, C.c_long]
        L.wmo_encode_kmer.restype = C.c_uint64
        L.wmo_encode_kmer.argtypes = [C.c_char_p, C.c_int]
        L.wmo_radix_sort_128x.argtypes = [_u64p, C.c_long]
        L.wmo_radix_sort_64.argtypes = [_u64p, C.c_long]
        L.wmo_idx_build.restype = C.c_void_p
        L.wmo_idx_build.argtypes = [_u64p, C.c_long]
        L.wmo_idx_free.argtypes = [C.c_void_p]
        L.wmo_collect_seed_hits.restype = C.c_long
        L.wmo_collect_seed_hits.argtypes = [C.c_void_p, C.c_int, _u64p, C.c_long, C.c_int, _u64p, C.c_long, _i32p, _u64p, _i32p]
        L.wmo_chain_dp.argtypes = [C.c_int] * 8 + [C.c_float, C.c_long, _u64p, _u64p, _u64p, C.POINTER(C.c_long)]
        L.wmo_ksw_extd2.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p] + [C.c_int] * 8 + [_i32p, _u32p, C.c_int]
        L.wmo_ksw_extz2.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p] + [C.c_int] * 6 + [_i32p, _u32p, C.c_int]
        L.wmo_ksw_exts2.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p] + [C.c_int] * 7 + [_u8p, _i32p, _u32p, C.c_int]
        L.wmo_ksw_ll.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p, C.c_int, C.c_int, _i32p, _i32p]
        L.wmo_counters_get.argtypes = [_u64p]
        _oracle = L
    return _oracle


def have_ref():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libref_harness.so"))


def _feed(h, v):
    if isinstance(v, np.ndarray):
        h.update(f"a{v.dtype.str}{v.shape}".encode())
        h.update(np.ascontiguousarray(v).tobytes())
    elif isinstance(v, (tuple, list)):
        h.update(b"(%d" % len(v))
        for x in v:
            _feed(h, x)
        h.update(b")")
    elif isinstance(v, bytes):
        h.update(b"b%d:" % len(v) + v)
    else:
        h.update(repr(v.item() if isinstance(v, np.generic) else v).encode())


def digest(v):
    """64-bit fingerprint of a result (arrays with dtype and shape, ints, bools, bytes, nested tuples / lists)."""
    h = hashlib.sha256()
    _feed(h, v)
    return h.hexdigest()[:16]


class RefGolden:
    """What the reference returned for the calls of one test, recorded in call order as digests of the results in
    tests/golden/ref/<module>.json (the results themselves -- sorted arrays, sketches, CIGARs -- are too large to store).

    check(ref_fn, got) compares `got` with the reference's answer: the recorded one, or -- with WM_RECORD_REF_GOLDEN=1
    and oracle/_ref built from the reference -- ref_fn(), whose digest is then recorded (the file is written after
    every call).  ref_fn is not called otherwise, so it may use objects that only exist when recording."""
    _files = {}

    def __init__(self, request):
        self.path = os.path.join(REF_GOLDEN_DIR, request.module.__name__ + ".json")
        self.key = request.node.name
        if self.path not in RefGolden._files:
            RefGolden._files[self.path] = json.load(open(self.path)) if os.path.exists(self.path) else {}
        self.table = RefGolden._files[self.path]
        if RECORD:
            assert have_ref(), "WM_RECORD_REF_GOLDEN=1 needs oracle/_ref (oracle/build_ref.sh)"
            self.table[self.key] = []
        assert self.key in self.table, f"no recorded reference results for {self.key} in {self.path}"
        self.want, self.i = self.table[self.key], 0

    def expect(self, ref_fn):
        """The digest of the reference's answer to the next call."""
        if RECORD:
            self.want.append(digest(ref_fn()))
            os.makedirs(REF_GOLDEN_DIR, exist_ok=True)
            with open(self.path, "w") as f:
                json.dump(self.table, f, indent=0, sort_keys=True)
        assert self.i < len(self.want), f"{self.key}: more calls than the {len(self.want)} recorded"
        self.i += 1
        return self.want[self.i - 1]

    def check(self, ref_fn, got, msg=""):
        want = self.expect(ref_fn)
        assert digest(got) == want, (f"{self.key}: call {self.i - 1} differs from the reference", msg)

    def done(self):
        assert self.i == len(self.want), f"{self.key}: {self.i} calls, {len(self.want)} recorded"


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libref_harness.so"))
        L.ref_ksw_extd2.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p] + [C.c_int] * 8 + [_i32p, _u32p, C.c_int]
        L.ref_ksw_extz2.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p] + [C.c_int] * 6 + [_i32p, _u32p, C.c_int]
        L.ref_ksw_exts2.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p] + [C.c_int] * 7 + [_u8p, _i32p, _u32p, C.c_int]
        L.ref_ksw_ll.argtypes = [C.c_int, _u8p, C.c_int, _u8p, _i8p, C.c_int, C.c_int, _i32p, _i32p]
        L.ref_radix_sort_128x.argtypes = [_u64p, C.c_long]
        L.ref_radix_sort_64.argtypes = [_u64p, C.c_long]
        L.ref_sketch_ctx.restype = C.c_void_p
        L.ref_sketch_ctx.argtypes = [C.c_int, _u64p]
        L.ref_bloom_size.restype = C.c_uint64
        L.ref_bloom_size.argtypes = [C.c_void_p]
        L.ref_bloom_table.argtypes = [C.c_void_p, _u8p]
        L.ref_bloom_contains.argtypes = [C.c_void_p, C.c_uint64]
        L.ref_sketch_free.argtypes = [C.c_void_p]
        L.ref_sketch.restype = C.c_long
        L.ref_sketch.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, _u64p, C.c_long]
        L.ref_chain_dp.argtypes = [C.c_int] * 8 + [C.c_float, C.c_long, _u64p, _u64p, _u64p, C.POINTER(C.c_long)]
        _ref = L
    return _ref


def simple_mat(a=2, b=4, sc_ambi=1):
    """src/align.c:9-22 (ksw_gen_simple_mat, m = 5)."""
    m = np.full((5, 5), -abs(b), dtype=np.int8)
    for i in range(4):
        m[i, i] = abs(a)
    m[4, :] = -abs(sc_ambi)
    m[:, 4] = -abs(sc_ambi)
    return np.ascontiguousarray(m.reshape(-1))


def _extd2(fn, q, t, mat, go, ge, go2, ge2, w, zdrop, end_bonus, flag):
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    ez = np.zeros(11, dtype=np.int32)
    cap = len(q) + len(t) + 8
    cig = np.zeros(cap, dtype=np.uint32)
    n = fn(len(q), _ptr(q, _u8p), len(t), _ptr(t, _u8p), _ptr(mat, _i8p), go, ge, go2, ge2, w, zdrop, end_bonus, flag,
           _ptr(ez, _i32p), _ptr(cig, _u32p), cap)
    return ez, cig[:n].copy()


def _extz2(fn, q, t, mat, go, ge, w, zdrop, end_bonus, flag):
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    ez = np.zeros(11, dtype=np.int32)
    cap = len(q) + len(t) + 8
    cig = np.zeros(cap, dtype=np.uint32)
    n = fn(len(q), _ptr(q, _u8p), len(t), _ptr(t, _u8p), _ptr(mat, _i8p), go, ge, w, zdrop, end_bonus, flag,
           _ptr(ez, _i32p), _ptr(cig, _u32p), cap)
    return ez, cig[:n].copy()


def _exts2(fn, q, t, mat, go, ge, go2, noncan, zdrop, junc_bonus, flag, junc=None):
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    ez = np.zeros(11, dtype=np.int32)
    cap = len(q) + len(t) + 8
    cig = np.zeros(cap, dtype=np.uint32)
    if junc is not None:
        junc = np.ascontiguousarray(junc, dtype=np.uint8)
    n = fn(len(q), _ptr(q, _u8p), len(t), _ptr(t, _u8p), _ptr(mat, _i8p), go, ge, go2, noncan, zdrop, junc_bonus, flag,
           _ptr(junc, _u8p) if junc is not None else None, _ptr(ez, _i32p), _ptr(cig, _u32p), cap)
    return ez, cig[:n].copy()


def oracle_exts2(*a, **k):
    return _exts2(oracle().wmo_ksw_exts2, *a, **k)


def ref_exts2(*a, **k):
    return _exts2(ref().ref_ksw_exts2, *a, **k)


def oracle_extz2(*a):
    return _extz2(oracle().wmo_ksw_extz2, *a)


def ref_extz2(*a):
    return _extz2(ref().ref_ksw_extz2, *a)


def oracle_extd2(*a):
    return _extd2(oracle().wmo_ksw_extd2, *a)


def ref_extd2(*a):
    return _extd2(ref().ref_ksw_extd2, *a)


def _ll(fn, q, t, mat, go, ge):
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    qe, te = C.c_int(), C.c_int()
    sc = fn(len(q), _ptr(q, _u8p), len(t), _ptr(t, _u8p), _ptr(mat, _i8p), go, ge, C.byref(qe), C.byref(te))
    return sc, qe.value, te.value


def oracle_ll(*a):
    return _ll(oracle().wmo_ksw_ll, *a)


def ref_ll(*a):
    return _ll(ref().ref_ksw_ll, *a)


def _sort(fn, arr, stride):
    a = np.ascontiguousarray(arr, dtype=np.uint64).copy()
    fn(_ptr(a, _u64p), len(a) // stride)
    return a


def oracle_sort128(xy):
    return _sort(oracle().wmo_radix_sort_128x, xy.reshape(-1), 2).reshape(-1, 2)


def ref_sort128(xy):
    return _sort(ref().ref_radix_sort_128x, xy.reshape(-1), 2).reshape(-1, 2)


def oracle_sort64(a):
    return _sort(oracle().wmo_radix_sort_64, a, 1)


def ref_sort64(a):
    return _sort(ref().ref_radix_sort_64, a, 1)


class OracleBloom:
    def __init__(self, kmers):
        self.L = oracle()
        kmers = np.asarray(kmers, dtype=np.uint64)
        self.h = self.L.wmo_bloom_init(len(kmers))
        for k in kmers:
            self.L.wmo_bloom_insert(self.h, int(k))

    def bits(self):
        return self.L.wmo_bloom_bits(self.h)

    def table(self):
        n = self.bits() // 8
        return np.ctypeslib.as_array(C.cast(self.L.wmo_bloom_table(self.h), _u8p), shape=(n,)).copy()

    def salts(self):
        s = (C.c_uint32 * 2)()
        self.L.wmo_bloom_salts(self.h, s)
        return [s[0], s[1]][: self.L.wmo_bloom_nsalt(self.h)]

    def contains(self, k):
        return bool(self.L.wmo_bloom_contains(self.h, int(k)))

    def __del__(self):
        try:
            self.L.wmo_bloom_free(self.h)
        except Exception:
            pass


def oracle_sketch(seq: bytes, w, k, rid, bloom: OracleBloom):
    cap = len(seq) // 4 + 64
    out = np.zeros(cap * 2, dtype=np.uint64)
    n = oracle().wmo_sketch(seq, len(seq), w, k, rid, bloom.h if bloom else None, _ptr(out, _u64p), cap)
    assert n <= cap
    return out[: 2 * n].reshape(-1, 2).copy()


class RefSketch:
    def __init__(self, kmers):
        self.L = ref()
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        self.h = self.L.ref_sketch_ctx(len(kmers), _ptr(kmers, _u64p))

    def bits(self):
        return self.L.ref_bloom_size(self.h)

    def table(self):
        t = np.zeros(self.bits() // 8, dtype=np.uint8)
        self.L.ref_bloom_table(self.h, _ptr(t, _u8p))
        return t

    def contains(self, k):
        return bool(self.L.ref_bloom_contains(self.h, int(k)))

    def sketch(self, seq: bytes, w, k, rid):
        cap = len(seq) // 4 + 64
        out = np.zeros(cap * 2, dtype=np.uint64)
        n = self.L.ref_sketch(self.h, seq, len(seq), w, k, rid, _ptr(out, _u64p), cap)
        assert n <= cap
        return out[: 2 * n].reshape(-1, 2).copy()

    def __del__(self):
        try:
            self.L.ref_sketch_free(self.h)
        except Exception:
            pass


def _chain(fn, a_xy, max_dist_x, min_dist_x, max_dist_y, bw, max_skip=25, max_iter=5000, min_cnt=3, min_sc=40, gap_scale=1.0):
    a = np.ascontiguousarray(a_xy, dtype=np.uint64).reshape(-1).copy()
    n = len(a) // 2
    u = np.zeros(max(n, 1), dtype=np.uint64)
    b = np.zeros(max(2 * n, 2), dtype=np.uint64)
    nb = C.c_long()
    n_u = fn(max_dist_x, min_dist_x, max_dist_y, bw, max_skip, max_iter, min_cnt, min_sc, C.c_float(gap_scale), n,
             _ptr(a, _u64p), _ptr(u, _u64p), _ptr(b, _u64p), C.byref(nb))
    return u[:n_u].copy(), b[: 2 * nb.value].reshape(-1, 2).copy()


def oracle_chain(a_xy, *args, **kw):
    return _chain(oracle().wmo_chain_dp, a_xy, *args, **kw)


def ref_chain(a_xy, *args, **kw):
    return _chain(ref().ref_chain_dp, a_xy, *args, **kw)


class OracleIndex:
    def __init__(self, mz_xy):
        self.L = oracle()
        m = np.ascontiguousarray(mz_xy, dtype=np.uint64).reshape(-1)
        self.h = self.L.wmo_idx_build(_ptr(m, _u64p), len(m) // 2)

    def seed_hits(self, mv_xy, qlen, max_occ=5000):
        mv = np.ascontiguousarray(mv_xy, dtype=np.uint64).reshape(-1)
        n_mv = len(mv) // 2
        cap = 1 << 16
        while True:
            a = np.zeros(2 * cap, dtype=np.uint64)
            mp = np.zeros(max(n_mv, 1), dtype=np.uint64)
            rep, nmp = C.c_int(), C.c_int()
            n = self.L.wmo_collect_seed_hits(self.h, max_occ, _ptr(mv, _u64p), n_mv, qlen, _ptr(a, _u64p), cap,
                                             C.byref(rep), _ptr(mp, _u64p), C.byref(nmp))
            if n <= cap:
                return a[: 2 * n].reshape(-1, 2).copy(), rep.value, mp[: nmp.value].copy()
            cap = n

    def __del__(self):
        try:
            self.L.wmo_idx_free(self.h)
        except Exception:
            pass
