"""CPU check of the DP kernels' arithmetic: the product's fill sweep (csrc/ksw_extd2_v2.cuh: 16x2 SIMD, tagged maxima, block
rounding, stale score cells) and traceback / Z-drop walk (csrc/ksw_extd2_common.cuh) are compiled for the host on a
software warp (tests/hostsim/cuda_emul.h, kernel_emul.cpp) and compared with the oracle, bit for bit.  The same code
runs on the device in tests/test_gpu_extd2.py; this tier catches arithmetic regressions where there is no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as ol
from test_oracle_vs_ref import FLAGS, rand_pair

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emul():
    d = os.path.join(ROOT, "tests", "hostsim")
    subprocess.check_call([os.path.join(d, "build.sh")], stderr=subprocess.DEVNULL)
    L = C.CDLL(os.path.join(d, "libwm_hostsim.so"))
    L.wmt_emul_extd2.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p] + [C.c_int] * 9 + [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    return L


def _run(L, q, t, mat, prm, w, zdrop, eb, flag, global_state):
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    mat = np.ascontiguousarray(mat, dtype=np.int8)
    cap = len(q) + len(t) + 2
    ez = np.zeros(12, np.int32); cig = np.zeros(cap, np.uint32); zd = np.zeros(5, np.int32)
    rc = L.wmt_emul_extd2(q.ctypes.data, len(q), t.ctypes.data, len(t), mat.ctypes.data, *prm, w, zdrop, eb, flag, int(global_state),
                          ez.ctypes.data, cig.ctypes.data, cap, zd.ctypes.data)
    assert rc == 0
    return ez, cig[:max(0, ez[10])], zd


def _check(L, q, t, mat, prm, w, zdrop, eb, flag, global_state):
    ez, cig, _ = _run(L, q, t, mat, prm, w, zdrop, eb, flag, global_state)
    e0, c0 = ol.oracle_extd2(q, t, mat, *prm, w, zdrop, eb, flag)
    assert np.array_equal(e0[:11], ez[:11]), (len(q), len(t), w, hex(flag), global_state, e0, ez)
    assert np.array_equal(c0, cig), (len(q), len(t), w, hex(flag), global_state)


@pytest.mark.parametrize("seed", range(2))
def test_fill_and_traceback_match_oracle(emul, seed):
    rng = np.random.default_rng(4100 + seed)
    mat = ol.simple_mat()
    for it in range(36):
        tlen = int(rng.choice([1, 5, 16, 17, 33, 64, 100, 130, 250, 300, 480]))
        q, t = rand_pair(rng, tlen, err=float(rng.choice([0.02, 0.1, 0.3])), drift=int(rng.choice([0, 0, 30, 120])), n_runs=int(rng.integers(0, 3)))
        if len(q) > 640:
            q = q[:640]
        w = int(rng.choice([5, 20, 50, 100, 751])); zdrop = int(rng.choice([400, 200, 50, -1])); eb = int(rng.choice([-1, 0, 10]))
        flag = FLAGS[int(rng.integers(0, len(FLAGS)))]
        _check(emul, q, t, mat, (4, 2, 24, 1), w, zdrop, eb, flag, global_state=bool(it & 1))


def test_single_affine_sweep_matches_oracle(emul):
    """csrc/ksw_extz2.cuh (ksw_extz2_sse: unsigned-offset state, mixed signed / unsigned maxima) on the software warp against the
    oracle's restatement, which tests/test_oracle_vs_ref.py pins to the reference's function."""
    emul.wmt_emul_extz2.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    rng = np.random.default_rng(4300)
    for it in range(48):
        tlen = int(rng.choice([1, 5, 16, 17, 33, 64, 100, 130, 250, 300, 480, 900]))
        q, t = rand_pair(rng, tlen, err=float(rng.choice([0.02, 0.1, 0.3])), drift=int(rng.choice([0, 0, 30, 120])), n_runs=int(rng.integers(0, 3)))
        w = int(rng.choice([5, 20, 50, 100, 751, -1])); zdrop = int(rng.choice([400, 200, 50, -1])); eb = int(rng.choice([-1, 0, 10]))
        flag = FLAGS[int(rng.integers(0, len(FLAGS)))] | (0x10 if it % 5 == 0 else 0)
        a, b, go, ge = [(2, 4, 4, 2), (1, 4, 6, 2), (1, 9, 16, 2), (5, 4, 40, 20), (3, 6, 50, 13)][it % 5]
        mat = np.ascontiguousarray(ol.simple_mat(a, b, 1), dtype=np.int8)
        qq = np.ascontiguousarray(q, dtype=np.uint8); tt = np.ascontiguousarray(t, dtype=np.uint8)
        cap = len(qq) + len(tt) + 2
        ez = np.zeros(12, np.int32); cig = np.zeros(cap, np.uint32); zd = np.zeros(5, np.int32)
        assert emul.wmt_emul_extz2(qq.ctypes.data, len(qq), tt.ctypes.data, len(tt), mat.ctypes.data, go, ge, w, zdrop, eb, flag,
                                   ez.ctypes.data, cig.ctypes.data, cap, zd.ctypes.data) == 0
        e0, c0 = ol.oracle_extz2(qq, tt, mat, go, ge, w, zdrop, eb, flag)
        assert np.array_equal(e0[:11], ez[:11]), (it, len(qq), len(tt), w, hex(flag), (a, b, go, ge), e0, ez)
        assert np.array_equal(c0, cig[:max(0, ez[10])]), (it, len(qq), len(tt), w, hex(flag))


def _splice_cases(rng, n):
    """(q, t, flag, zdrop, scoring, junc) cases of the splice-aware extension, shared by the emulation test and the GPU test."""
    from test_oracle_vs_ref import spliced_pair
    out = []
    for it in range(n):
        if it % 5 == 4:
            q, t = rand_pair(rng, int(rng.choice([1, 5, 17, 33, 100, 300])), err=0.1, drift=int(rng.choice([0, 30])), n_runs=int(rng.integers(0, 2)))
        else:
            q, t = spliced_pair(rng, int(rng.integers(1, 6)), err=float(rng.choice([0.0, 0.05, 0.2])), rev_sites=bool(it & 1), n_runs=int(rng.integers(0, 2)))
        if it % 7 == 3:
            q, t = q[::-1].copy(), t[::-1].copy()
        flag = FLAGS[int(rng.integers(0, len(FLAGS)))] | (0x10 if rng.random() < 0.3 else 0) | (0x04 if rng.random() < 0.15 else 0)
        flag |= [0x100, 0x200, 0x300, 0][int(rng.integers(0, 4))] | (0x400 if rng.random() < 0.7 else 0)
        if it % 7 == 3:
            flag |= 0x80 | 0x02
        zdrop = int(rng.choice([200, 100, 30, -1]))
        sc = [(1, 2, 2, 1, 32, 9, 9), (1, 4, 6, 1, 24, 9, 5), (2, 4, 4, 2, 24, 5, 3), (1, 2, 2, 1, 3, 9, 9), (1, 2, 2, 1, 60, 0, 0)][it % 5]
        junc = None
        if rng.random() < 0.4:
            junc = np.where(rng.random(len(t)) < 0.05, rng.integers(1, 16, size=len(t)), 0).astype(np.uint8)
        out.append((np.ascontiguousarray(q, dtype=np.uint8), np.ascontiguousarray(t, dtype=np.uint8), flag, zdrop, sc, junc))
    return out


def test_splice_sweep_matches_oracle(emul):
    """csrc/ksw_exts2.cuh (ksw_exts2_sse: long-deletion state with donor / acceptor costs, N_SKIP traceback) on the software warp
    against the oracle's restatement, which tests/test_oracle_vs_ref.py pins to the reference's function."""
    emul.wmt_emul_exts2.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 7 + [C.c_void_p, C.c_void_p, C.c_int]
    n_intron = 0
    for it, (qq, tt, flag, zdrop, (a, b, go, ge, go2, noncan, jb), junc) in enumerate(_splice_cases(np.random.default_rng(4400), 60)):
        mat = np.ascontiguousarray(ol.simple_mat(a, b, 1), dtype=np.int8)
        cap = len(qq) + len(tt) + 2
        ez = np.zeros(12, np.int32); cig = np.zeros(cap, np.uint32)
        assert emul.wmt_emul_exts2(qq.ctypes.data, len(qq), tt.ctypes.data, len(tt), junc.ctypes.data if junc is not None else None, mat.ctypes.data,
                                   go, ge, go2, noncan, jb, zdrop, flag, ez.ctypes.data, cig.ctypes.data, cap) == 0
        e0, c0 = ol.oracle_exts2(qq, tt, mat, go, ge, go2, noncan, zdrop, jb, flag, junc=junc)
        assert np.array_equal(e0[:11], ez[:11]), (it, len(qq), len(tt), hex(flag), (a, b, go, ge, go2), e0, ez)
        assert np.array_equal(c0, cig[:max(0, ez[10])]), (it, len(qq), len(tt), hex(flag))
        n_intron += int((c0 & 0xf == 3).any())
    assert n_intron > 5


def test_other_scorings_and_a_long_target(emul):
    rng = np.random.default_rng(4200)
    for a, b, q_, e_, q2, e2 in [(1, 4, 6, 2, 26, 1), (2, 4, 24, 1, 4, 2)]:  # asm-like scoring; gap pair given in swapped order
        mat = ol.simple_mat(a, b, 1)
        for i in range(6):
            q, t = rand_pair(rng, int(rng.integers(20, 400)), err=0.05, drift=int(rng.choice([0, 50])))
            _check(emul, q[:640], t, mat, (q_, e_, q2, e2), 200, 200, -1, FLAGS[i % 4], global_state=False)
    q, t = rand_pair(rng, 1300, err=0.08, drift=100)  # beyond the shared-memory slice: global state rows only
    _check(emul, q, t, ol.simple_mat(), (4, 2, 24, 1), 751, 400, -1, 0x40, global_state=True)


def test_zdrop_walk_matches_the_host_walk(emul):
    """The device-side mm_test_zdrop walk (flag 0x10000) against a direct restatement of src/align.c:32-70."""
    rng = np.random.default_rng(4300)
    mat = ol.simple_mat()
    for _ in range(10):
        q, t = rand_pair(rng, int(rng.integers(100, 400)), err=0.12, drift=int(rng.choice([0, 80])), n_runs=2)
        q = q[:640]
        ez, cig, zd = _run(emul, q, t, mat, (4, 2, 24, 1), 751, 400, -1, 0x08 | 0x10000, False)
        score, mx, max_i, max_j, i, j, best, pos = 0, -(1 << 31), -1, -1, 0, 0, 0, [-1, -1, -1, -1]

        def upd(sc, ii, jj):
            nonlocal mx, max_i, max_j, best, pos
            if sc < mx:
                li, lj = ii - max_i, jj - max_j
                z = mx - sc - abs(li - lj) * 2
                if z > best:
                    best, pos = z, [max_i, ii, max_j, jj]
            else:
                mx, max_i, max_j = sc, ii, jj
        for c in cig:
            op, ln = int(c) & 0xf, int(c) >> 4
            if op == 0:
                for k in range(ln):
                    score += int(mat[int(t[i + k]) * 5 + int(q[j + k])])
                    upd(score, i + k, j + k)
                i += ln; j += ln
            else:
                score -= 4 + 2 * ln
                if op == 1:
                    j += ln
                else:
                    i += ln
                upd(score, i, j)
        assert list(zd) == [best] + pos


def _tandem_anchors(rng, n_q, n_copies, unit, span=15):
    """Anchors of a read crossing a tandem array: every query minimizer hits every copy of the unit."""
    q0 = np.sort(rng.choice(np.arange(50, 50 + n_q * 11), size=n_q, replace=False)).astype(np.int64)
    x, y = [], []
    for c in range(n_copies):
        x.append(1000 + c * unit + (q0 % unit))
        y.append(q0)
    x = np.concatenate(x).astype(np.uint64); y = np.concatenate(y).astype(np.uint64)
    xy = np.stack([x, np.uint64(span) << np.uint64(32) | y], axis=1)
    return ol.oracle_sort128(xy)  # the reference's order: tests/test_oracle_vs_ref.py::test_sorts_match_reference_including_ties


@pytest.mark.parametrize("dense", [0, 1, 2, 3, 4])
def test_chain_forward_pass_formulations(emul, dense):
    """The warp formulations of the chaining forward pass (csrc/chain_dev.cuh: 32 predecessors per step; dense
    candidates; sliding window in a shared-memory ring of 64 / 1024 slots with closed-form window starts; tiles of 32 anchors with per-anchor mark bitsets and the locked deep path) against a scalar restatement of src/chain.c:45-90: identical f / p / v for every anchor."""
    from test_oracle_vs_ref import make_anchors
    sig = [C.c_void_p, C.c_int] + [C.c_int] * 6 + [C.c_float]
    emul.wmt_emul_chain_fill.argtypes = sig + [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    emul.wmt_chain_fill_scalar.argtypes = sig + [C.c_void_p, C.c_void_p, C.c_void_p]
    rng = np.random.default_rng(4400)
    arrays = [make_anchors(rng, n, repeats=bool(i & 1)) for i, n in enumerate([1, 2, 33, 100, 700, 2500])]
    arrays += [_tandem_anchors(rng, 40, 30, 171), _tandem_anchors(rng, 90, 25, 64)]
    for a in arrays:
        a = np.ascontiguousarray(a, dtype=np.uint64)
        n = len(a)
        for prm in [(5000, 1000, 5000, 500, 25, 5000), (16000, 1000, 16000, 2000, 25, 5000), (5000, 50, 5000, 500, 3, 20), (5000, 500, 5000, 500, 25, 300)]:
            out = [np.full(n, -7, np.int32) for _ in range(6)]
            emul.wmt_chain_fill_scalar(a.ctypes.data, n, *prm, 1.0, out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data)
            emul.wmt_emul_chain_fill(a.ctypes.data, n, *prm, 1.0, dense, out[3].ctypes.data, out[4].ctypes.data, out[5].ctypes.data)
            for k, nm in enumerate("fpv"):
                assert np.array_equal(out[k], out[3 + k]), (n, prm, nm, int(np.argmax(out[k] != out[3 + k])))


def test_warp_radix_sort_reproduces_the_unstable_tie_order(emul):
    """csrc/rsort.cuh on the software warp against the reference's in-place MSD radix sort (src/ksort.h:98-151): equal keys
    must end up in the reference's order (the payload column shows it)."""
    emul.wmt_emul_sort128.argtypes = [C.c_void_p, C.c_int]
    rng = np.random.default_rng(4500)
    for n in [0, 1, 2, 63, 64, 65, 200, 1000, 5000, 20000]:
        for key_bits in [3, 12, 28, 64]:
            hi = (1 << key_bits) - 1
            x = rng.integers(0, hi, size=n, dtype=np.uint64, endpoint=True)
            if key_bits == 64 and n:
                x[::3] = x[0]
            a = np.stack([x, np.arange(n, dtype=np.uint64)], axis=1)
            got = np.ascontiguousarray(a).copy()
            emul.wmt_emul_sort128(got.ctypes.data, n)
            assert np.array_equal(ol.oracle_sort128(a), got), (n, key_bits)


@pytest.mark.parametrize("dense", [0, 1, 2, 3, 4])
def test_chaining_end_to_end_matches_oracle(emul, dense):
    """Forward pass + backtracking of csrc/chain_dev.cuh on the software warp against the oracle's mm_chain_dp: chains
    (score, count) and chained anchors, including the unstable re-sort of the chains."""
    from test_oracle_vs_ref import make_anchors
    emul.wmt_emul_chain.argtypes = [C.c_void_p, C.c_int] + [C.c_int] * 8 + [C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    rng = np.random.default_rng(4600)
    arrays = [make_anchors(rng, n, repeats=bool(i & 1)) for i, n in enumerate([1, 3, 10, 40, 100, 700, 3000])]
    arrays.append(_tandem_anchors(rng, 50, 30, 171))
    for a in arrays:
        for prm in [(5000, 1000, 5000, 500, 25, 5000), (16000, 1000, 16000, 2000, 25, 5000), (5000, 50, 5000, 500, 3, 20)]:
            ue, be = ol.oracle_chain(a, prm[0], prm[1], prm[2], prm[3], max_skip=prm[4], max_iter=prm[5])
            buf = np.ascontiguousarray(a, dtype=np.uint64).copy()
            n = len(buf)
            u = np.zeros(n + 1, np.uint64); n_u = C.c_int32(); n_b = C.c_int64()
            emul.wmt_emul_chain(buf.ctypes.data, n, *prm, 3, 40, 1.0, dense, u.ctypes.data, C.addressof(n_u), C.addressof(n_b))
            assert np.array_equal(ue, u[:n_u.value]), (n, prm, len(ue), n_u.value)
            assert np.array_equal(be, buf[:n_b.value]), (n, prm)


@pytest.mark.parametrize("seed,n,k", [(1, 20000, 15), (2, 20000, 19), (3, 7777, 28), (4, 100, 5), (5, 33, 1), (6, 50000, 16)])
def test_packed_read_pool_matches_bytewise_restatement(emul, seed, n, k):
    """csrc/pkseq.cuh compiled for the host: ASCII -> 2-bit + ambiguity mask, every k-mer as one 64-bit window (forward and
    reverse-complement words of src/sketch.c:162-163), masked copies (src/map.c:795-801) and the DP gather of both strands /
    both directions / the 4-bit reference (src/align.c:874-876), each against a byte-per-base restatement."""
    emul.wmt_pk_selftest.argtypes = [C.c_uint64, C.c_int64, C.c_int]
    assert emul.wmt_pk_selftest(seed, n, k) == 0
