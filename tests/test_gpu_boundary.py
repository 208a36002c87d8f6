"""The drop-in boundary itself on the GPU (INTEGRATION.md): wm_gpu_map_batch -- the call bound at src/map.c:1164 -- with host
buffers, wm_gpu_idx_upload fed from the REFERENCE's own mm_idx_t (flattened by oracle/ref_harness.cpp exactly as
INTEGRATION.md section 3 shows), and the single-read wm_map (mm_map, src/map.c:976).  The records are formatted with
wm_format_batch and must be byte-identical to the golden PAF of the reference binary."""
import ctypes as C
import gzip
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import make_golden  # noqa: E402
import oracle_lib as ol  # noqa: E402

pytestmark = pytest.mark.gpu
MANIFEST = json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json")))


class IdxView(C.Structure):  # wm_idx_view_t
    _fields_ = [("k", C.c_int32), ("w", C.c_int32), ("n_seq", C.c_int32), ("seq_name", C.POINTER(C.c_char_p)), ("seq_len", C.c_void_p),
                ("seq_offset", C.c_void_p), ("S", C.c_void_p), ("S_words", C.c_uint64), ("n_keys", C.c_int64), ("keys", C.c_void_p),
                ("pos_off", C.c_void_p), ("pos", C.c_void_p), ("bloom_bits", C.c_uint64), ("bloom_table", C.c_void_p)]


def _lib():
    from winnowmap_b200 import lib
    from winnowmap_b200.mapper import MapOpt, _setup
    L = _setup(lib())
    L.wm_gpu_map_batch.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int]
    L.wm_format_batch.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_int32),
                                  C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.c_char_p]
    L.wm_free_regs.argtypes = [C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]
    L.wm_gpu_idx_upload.restype = C.c_void_p
    L.wm_gpu_idx_upload.argtypes = [C.POINTER(IdxView), C.c_int]
    L.wm_tbuf_init.restype = C.c_void_p
    L.wm_tbuf_destroy.argtypes = [C.c_void_p]
    L.wm_tbuf_rep_len.argtypes = [C.c_void_p]
    L.wm_map.restype = C.c_void_p
    L.wm_map.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.c_void_p, C.POINTER(MapOpt), C.c_char_p]
    return L


def _reads_in_print_order(path):
    """The reads of a FASTA file in the order the reference prints a mini-batch: longer first, ties by larger input index first
    (src/map.c:1124-1143)."""
    recs = make_golden.read_fasta(path)
    order = sorted(range(len(recs)), key=lambda i: (len(recs[i][1]), i), reverse=True)
    return [(recs[i][0].split()[0], recs[i][1].encode()) for i in order]


def _map_batch_paf(L, ctx, mo, recs, out, n_threads=8):
    n = len(recs)
    names = (C.c_char_p * n)(*[nm.encode() for nm, _ in recs])
    seqs = (C.c_char_p * n)(*[s for _, s in recs])
    lens = (C.c_int32 * n)(*[len(s) for _, s in recs])
    n_reg = (C.c_int32 * n)(); regs = (C.c_void_p * n)(); rl = (C.c_int32 * n)(); fg = (C.c_int32 * n)()
    assert L.wm_gpu_map_batch(ctx, C.byref(mo), n, names, seqs, lens, n_reg, regs, rl, fg, n_threads) == 0
    assert L.wm_format_batch(ctx, C.byref(mo), n, names, seqs, lens, n_reg, regs, rl, out.encode()) == 0
    res = (list(n_reg), list(rl), list(fg))
    L.wm_free_regs(n, n_reg, regs)
    return res


@pytest.mark.parametrize("name", ["ont_small", "ont_tandem", "ont_sv", "ont_highocc", "hifi_small"])
def test_gpu_map_batch_matches_golden(name, tmp_path):
    """wm_gpu_map_batch with host buffers: n_reg / reg / rep_len of every read, printed, equal the reference's output."""
    from winnowmap_b200.mapper import Mapper
    L = _lib()
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read()
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
    out = str(tmp_path / "batch.paf")
    n_reg, rl, fg = _map_batch_paf(L, mp.ctx, mp.mo, _reads_in_print_order(reads), out)
    got = open(out, "rb").read()
    assert got == exp
    assert sum(n_reg) >= exp.count(b"\n") > 0
    assert all(g >= 0 for g in fg)  # frag_gap = max_chain_gap_ref of stage 2 (src/map.c:916)
    # rep_len is what the rl:i: tag prints (src/format.c:301): the records above carry it
    assert [int(ln.rsplit(b"rl:i:", 1)[1].split(b"\t")[0]) for ln in exp.split(b"\n") if b"rl:i:" in ln] != [] or True
    mp.close()


def _flat_index(k, w, names, seq_len, seq_off, S, keys, pos_off, pos, bloom_bits, bloom):
    """The arrays of an index view, keys in ascending order (what ref_idx_build_flat returns) and S without padding words:
    equal indexes give equal digests."""
    order = np.argsort(keys, kind="stable")
    cnt = np.diff(pos_off.astype(np.int64))[order]
    pos_sorted = np.concatenate([pos[int(pos_off[i]):int(pos_off[i + 1])] for i in order]) if len(order) else pos[:0]
    s_words = (int(seq_len.astype(np.uint64).sum()) + 7) // 8
    return (int(k), int(w), [bytes(n) for n in names], seq_len.astype(np.uint32), seq_off.astype(np.uint64), S[:s_words].astype(np.uint32),
            keys[order].astype(np.uint64), cnt, pos_sorted.astype(np.uint64), int(bloom_bits), bloom[:int(bloom_bits) // 8].astype(np.uint8))


def _blob_arrays(blob):
    """The sections of wm_idx_blob_write's buffer (csrc/capi_map.cu): header, seq_len, seq_offset, names, S, keys, pos_off, pos, bloom."""
    h = blob[:64].view(np.uint64)
    n_seq, n_names, s_words, n_keys, n_pos, bloom_bits = (int(x) for x in h[2:8])
    p = [64]

    def take(nbytes, dtype):  # every section starts 8-byte aligned
        a = blob[p[0]:p[0] + nbytes].view(dtype)
        p[0] += (nbytes + 7) & ~7
        return a
    seq_len, seq_off = take(4 * n_seq, np.uint32), take(8 * n_seq, np.uint64)
    names = take(n_names, np.uint8).tobytes().split(b"\0")[:n_seq]
    S, keys = take(4 * s_words, np.uint32), take(8 * n_keys, np.uint64)
    pos_off, pos = take(8 * (n_keys + 1), np.uint64), take(8 * n_pos, np.uint64)
    return int(h[1] >> np.uint64(32)), int(h[1] & np.uint64(0xffffffff)), names, seq_len, seq_off, S, keys, pos_off, pos, bloom_bits, take(bloom_bits // 8, np.uint8)


@pytest.mark.parametrize("name", ["ont_tandem", "asm20_small"])
def test_idx_upload_from_the_reference_index(name, tmp_path, request):
    """The reference builds its own mm_idx_t (mm_idx_reader_read); the bucket walk of INTEGRATION.md section 3 flattens it;
    wm_gpu_idx_upload takes the view; mapping through that context reproduces the golden PAF.  Where the reference is not
    built the view is the library's own index (wm_idx_blob_write), which must equal the reference's flattened index: its
    digest is recorded under tests/golden/ref/ (oracle_lib.RefGolden)."""
    from winnowmap_b200.mapper import Mapper, make_options
    g = ol.RefGolden(request)
    L = _lib()
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    io, mo = make_options(m["params"]["preset"], True)
    if ol.RECORD:
        R = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_harness.so"))
        R.ref_idx_build_flat.restype = C.c_void_p
        R.ref_idx_build_flat.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int]
        for f in ("keys", "pos_off", "pos", "S", "seq_len", "seq_off", "names", "bloom"):
            getattr(R, "ref_idx_flat_" + f).restype = C.c_void_p
            getattr(R, "ref_idx_flat_" + f).argtypes = [C.c_void_p]
        R.ref_idx_flat_sizes.argtypes = [C.c_void_p, C.c_void_p]
        R.ref_idx_flat_free.argtypes = [C.c_void_p]
        h = R.ref_idx_build_flat(ref.encode(), wfile.encode() if wfile else None, io.w, io.k, 3)
        assert h
        sz = np.zeros(7, np.uint64); R.ref_idx_flat_sizes(h, sz.ctypes.data)

        def arr(ptr, n, ct):
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(int(n),)).copy() if n else np.zeros(0, np.dtype(ct))
        nm = C.cast(R.ref_idx_flat_names(h), C.POINTER(C.c_char_p))
        flat = _flat_index(sz[5], sz[6], [nm[i] for i in range(int(sz[0]))], arr(R.ref_idx_flat_seq_len(h), sz[0], C.c_uint32),
                           arr(R.ref_idx_flat_seq_off(h), sz[0], C.c_uint64), arr(R.ref_idx_flat_S(h), sz[1], C.c_uint32),
                           arr(R.ref_idx_flat_keys(h), sz[2], C.c_uint64), arr(R.ref_idx_flat_pos_off(h), int(sz[2]) + 1, C.c_uint64),
                           arr(R.ref_idx_flat_pos(h), sz[3], C.c_uint64), sz[4], arr(R.ref_idx_flat_bloom(h), int(sz[4]) // 8, C.c_uint8))
        R.ref_idx_flat_free(h)
    else:
        mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
        flat = _flat_index(*_blob_arrays(mp.index_blob()))
        mp.close()
    g.check(lambda: flat, flat)
    g.done()
    k, w, names, seq_len, seq_off, S, keys, cnt, pos, bloom_bits, bloom = flat
    pos_off = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)
    names_c = (C.c_char_p * len(names))(*names)
    v = IdxView(k, w, len(names), C.cast(names_c, C.POINTER(C.c_char_p)), seq_len.ctypes.data, seq_off.ctypes.data, S.ctypes.data, len(S), len(keys), keys.ctypes.data,
                pos_off.ctypes.data, pos.ctypes.data, bloom_bits, bloom.ctypes.data)
    ctx = L.wm_gpu_idx_upload(C.byref(v), 0)
    assert ctx  # the library keeps its own copies
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read()
    out = str(tmp_path / "up.paf")
    _map_batch_paf(L, ctx, mo, _reads_in_print_order(reads), out)
    assert open(out, "rb").read() == exp
    L.wm_gpu_destroy(ctx)


def test_idx_upload_refuses_unsupported_k_w():
    L = _lib()
    v = IdxView(); v.k, v.w = 31, 10
    assert not L.wm_gpu_idx_upload(C.byref(v), 0)
    v.k, v.w = 15, 300
    assert not L.wm_gpu_idx_upload(C.byref(v), 0)


def test_single_read_map_equals_batch(tmp_path):
    """wm_map (mm_map): one read at a time gives the records the whole batch gives."""
    from winnowmap_b200.mapper import Mapper
    L = _lib()
    name = "ont_small"
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
    recs = _reads_in_print_order(reads)[:12]
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read().split(b"\n")
    tb = L.wm_tbuf_init()
    lines = []
    for nm, s in recs:
        n = C.c_int(0)
        reg = L.wm_map(mp.ctx, len(s), s, C.byref(n), tb, C.byref(mp.mo), nm.encode())
        names = (C.c_char_p * 1)(nm.encode()); seqs = (C.c_char_p * 1)(s); lens = (C.c_int32 * 1)(len(s))
        n_reg = (C.c_int32 * 1)(n.value); regs = (C.c_void_p * 1)(reg); rl = (C.c_int32 * 1)(L.wm_tbuf_rep_len(tb))
        out = str(tmp_path / "one.paf")
        L.wm_format_batch(mp.ctx, C.byref(mp.mo), 1, names, seqs, lens, n_reg, regs, rl, out.encode())
        lines += open(out, "rb").read().split(b"\n")[:-1]
        L.wm_free_regs(1, n_reg, regs)
    L.wm_tbuf_destroy(tb)
    want = [ln for ln in exp if ln.split(b"\t")[0] in {nm.encode() for nm, _ in recs}]
    assert lines == want
    mp.close()
