"""numpy-facing wrappers over the kernel-level C-ABI entry points."""
import ctypes as C

import numpy as np

from ._lib import ExtZ, i8p, i32p, i64p, lib, u8p, u32p, u64p

EZ_FIELDS = ("max", "zdropped", "max_q", "max_t", "mqe", "mqe_t", "mte", "mte_q", "score", "reach_end", "n_cigar")


def _p(a, t):
    return a.ctypes.data_as(t)


def _concat(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    if len(seqs):
        off[1:] = np.cumsum([len(s) for s in seqs])
    buf = np.concatenate([np.asarray(s, dtype=np.uint8) for s in seqs]) if len(seqs) and off[-1] else np.zeros(0, np.uint8)
    return np.ascontiguousarray(buf), off


def ksw_extd2_batch(queries, targets, mat, q, e, q2, e2, w, zdrop, end_bonus, flag, cigar_cap=None):
    """Batched ksw_extd2 (reference src/ksw2_extd2_sse.c:26).  Returns (ez[n,11] int32, [cigar arrays])."""
    n = len(queries)
    qb, qoff = _concat(queries)
    tb, toff = _concat(targets)
    as32 = lambda v: np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.int32), (n,)))
    w, zdrop, end_bonus, flag = as32(w), as32(zdrop), as32(end_bonus), as32(flag)
    if cigar_cap is None:
        cap = np.array([len(a) + len(b) + 2 for a, b in zip(queries, targets)], dtype=np.int64)
    else:
        cap = np.broadcast_to(np.asarray(cigar_cap, dtype=np.int64), (n,))
    coff = np.zeros(n + 1, dtype=np.int64)
    coff[1:] = np.cumsum(cap)
    ez = (ExtZ * max(n, 1))()
    cig = np.zeros(max(int(coff[-1]), 1), dtype=np.uint32)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    if len(qb) == 0:
        qb = np.zeros(1, np.uint8)
    if len(tb) == 0:
        tb = np.zeros(1, np.uint8)
    lib().wm_ksw_extd2_batch(n, _p(qb, u8p), _p(qoff, i64p), _p(tb, u8p), _p(toff, i64p), _p(mat, i8p), q, e, q2, e2,
                             _p(w, i32p), _p(zdrop, i32p), _p(end_bonus, i32p), _p(flag, i32p), ez, _p(cig, u32p), _p(coff, i64p))
    out = np.array([[getattr(ez[i], f) for f in EZ_FIELDS] for i in range(n)], dtype=np.int32).reshape(n, len(EZ_FIELDS))
    cigs = [cig[coff[i]: coff[i] + min(out[i, 10], cap[i])].copy() for i in range(n)]
    return out, cigs


def ksw_exts2_batch(queries, targets, mat, q, e, q2, noncan, junc_bonus, zdrop, flag, juncs=None):
    """Batched ksw_exts2 (reference src/ksw2_exts2_sse.c:26), the splice-aware extension.  juncs: per-target annotation bytes
    (arrays as long as the targets) or None.  Returns (ez[n,11] int32, [cigar arrays])."""
    n = len(queries)
    qb, qoff = _concat(queries)
    tb, toff = _concat(targets)
    as32 = lambda v: np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.int32), (n,)))
    zdrop, flag = as32(zdrop), as32(flag)
    cap = np.array([len(a) + len(b) + 2 for a, b in zip(queries, targets)], dtype=np.int64)
    coff = np.zeros(n + 1, dtype=np.int64)
    coff[1:] = np.cumsum(cap)
    ez = (ExtZ * max(n, 1))()
    cig = np.zeros(max(int(coff[-1]), 1), dtype=np.uint32)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    jb = None
    if juncs is not None:
        jb, _ = _concat([j if j is not None else np.zeros(len(t), np.uint8) for j, t in zip(juncs, targets)])
        if len(jb) == 0:
            jb = np.zeros(1, np.uint8)
    if len(qb) == 0:
        qb = np.zeros(1, np.uint8)
    if len(tb) == 0:
        tb = np.zeros(1, np.uint8)
    L = lib()
    L.wm_ksw_exts2_batch.argtypes = [C.c_int, u8p, i64p, u8p, i64p, u8p, i8p] + [C.c_int] * 5 + [i32p, i32p, C.c_void_p, u32p, i64p]
    L.wm_ksw_exts2_batch(n, _p(qb, u8p), _p(qoff, i64p), _p(tb, u8p), _p(toff, i64p), _p(jb, u8p) if jb is not None else None, _p(mat, i8p),
                         q, e, q2, noncan, junc_bonus, _p(zdrop, i32p), _p(flag, i32p), C.cast(ez, C.c_void_p), _p(cig, u32p), _p(coff, i64p))
    out = np.array([[getattr(ez[i], f) for f in EZ_FIELDS] for i in range(n)], dtype=np.int32).reshape(n, len(EZ_FIELDS))
    cigs = [cig[coff[i]: coff[i] + min(out[i, 10], cap[i])].copy() for i in range(n)]
    return out, cigs


def ksw_ll_batch(queries, targets, mat, gapo, gape):
    """Batched ksw_ll_qinit + ksw_ll_i16 (reference src/ksw2_ll_sse.c:32,80).  Returns (n,3) int32: score, query end, target end."""
    n = len(queries)
    qb, qoff = _concat(queries)
    tb, toff = _concat(targets)
    if len(qb) == 0:
        qb = np.zeros(1, np.uint8)
    if len(tb) == 0:
        tb = np.zeros(1, np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    sc, qe, te = (np.zeros(max(n, 1), np.int32) for _ in range(3))
    L = lib()
    L.wm_ksw_ll_batch.argtypes = [C.c_int, u8p, i64p, u8p, i64p, i8p, C.c_int, C.c_int, i32p, i32p, i32p]
    L.wm_ksw_ll_batch(n, _p(qb, u8p), _p(qoff, i64p), _p(tb, u8p), _p(toff, i64p), _p(mat, i8p), gapo, gape, _p(sc, i32p), _p(qe, i32p), _p(te, i32p))
    return np.stack([sc, qe, te], axis=1)[:n]


_libc = C.CDLL(None)
_libc.free.argtypes = [C.c_void_p]


class Bloom:
    """Down-weighted k-mer filter (reference: bloom_filter built at src/index.c:404-432)."""

    def __init__(self, canon_kmers):
        k = np.ascontiguousarray(canon_kmers, dtype=np.uint64)
        self._k = k
        self.h = lib().wm_bloom_build(_p(k, u64p) if len(k) else None, len(k))

    def bits(self):
        return lib().wm_bloom_bits(self.h)

    def table(self):
        n = self.bits() // 8
        return np.ctypeslib.as_array(C.cast(lib().wm_bloom_table(self.h), u8p), shape=(n,)).copy()

    def __del__(self):
        try:
            lib().wm_bloom_destroy(self.h)
        except Exception:
            pass


def sketch_batch(bloom, seqs, w, k, rids=None):
    """Batched mm_sketch (reference src/sketch.c:128).  seqs: list of bytes.  Returns list of (n,2) uint64."""
    n = len(seqs)
    off = np.zeros(n + 1, dtype=np.int64)
    if n:
        off[1:] = np.cumsum([len(s) for s in seqs])
    buf = b"".join(seqs) + b"\0"
    rid = np.ascontiguousarray(rids if rids is not None else np.zeros(n), dtype=np.uint32)
    out, out_off = C.c_void_p(), C.c_void_p()
    rc = lib().wm_sketch_batch(bloom.h, n, buf, _p(off, i64p), _p(rid, u32p), w, k, C.byref(out), C.byref(out_off))
    if rc != 0:
        raise ValueError("wm_sketch_batch failed")
    o = np.ctypeslib.as_array(C.cast(out_off, i64p), shape=(n + 1,)).copy()
    tot = int(o[-1])
    xy = np.ctypeslib.as_array(C.cast(out, u64p), shape=(max(tot, 1) * 2,)).copy()[: tot * 2].reshape(-1, 2)
    _libc.free(out)
    _libc.free(out_off)
    return [xy[o[i]: o[i + 1]].copy() for i in range(n)]


def radix_sort_128x_batch(arrays, timed=False):
    """radix_sort_128x (reference src/misc.c:156) on each (n,2) uint64 array, tie order included.
    timed=True: returns (sorted arrays, device milliseconds of the sort alone, copies left out)."""
    n = len(arrays)
    off = np.zeros(n + 1, dtype=np.int64)
    if n:
        off[1:] = np.cumsum([len(a) for a in arrays])
    flat = np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=np.uint64).reshape(-1, 2) for a in arrays] + [np.zeros((1, 2), np.uint64)]))
    ms = C.c_float(0.0)
    if timed:
        lib().wm_radix_sort_128x_batch_timed(n, _p(flat, u64p), _p(off, i64p), C.byref(ms))
    else:
        lib().wm_radix_sort_128x_batch(n, _p(flat, u64p), _p(off, i64p))
    out = [flat[off[i]: off[i + 1]].copy() for i in range(n)]
    return (out, ms.value) if timed else out


def chain_dp_batch(arrays, max_dist_x, min_dist_x, max_dist_y, bw, max_skip=25, max_iter=5000, min_cnt=3, min_sc=40, gap_scale=1.0):
    """Batched mm_chain_dp (reference src/chain.c:22).  Returns list of (u, b)."""
    n = len(arrays)
    off = np.zeros(n + 1, dtype=np.int64)
    if n:
        off[1:] = np.cumsum([len(a) for a in arrays])
    flat = np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=np.uint64).reshape(-1, 2) for a in arrays] + [np.zeros((1, 2), np.uint64)]))
    tot = int(off[-1])
    n_u = np.zeros(max(n, 1), dtype=np.int32)
    n_b = np.zeros(max(n, 1), dtype=np.int64)
    u = np.zeros(max(tot, 1), dtype=np.uint64)
    b = np.zeros((max(tot, 1), 2), dtype=np.uint64)
    lib().wm_chain_dp_batch(n, _p(flat, u64p), _p(off, i64p), max_dist_x, min_dist_x, max_dist_y, bw, max_skip, max_iter, min_cnt, min_sc,
                            C.c_float(gap_scale), _p(n_u, i32p), _p(u, u64p), _p(b, u64p), _p(n_b, i64p))
    return [(u[off[i]: off[i] + n_u[i]].copy(), b[off[i]: off[i] + n_b[i]].copy()) for i in range(n)]
