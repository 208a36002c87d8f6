"""Pins the CPU oracle (oracle/wm_oracle.c, a restatement) against the REAL reference
functions (oracle/_ref/libref_harness.so, built from the reference's sources by oracle/build_ref.sh).
The reference's answers on these seeded inputs are recorded under tests/golden/ref/ (oracle_lib.RefGolden),
so the comparison runs without the reference."""
import numpy as np
import pytest

import oracle_lib as ol


def rand_pair(rng, tlen, err=0.1, drift=0, n_runs=0):
    t = rng.integers(0, 4, size=tlen, dtype=np.uint8)
    q = []
    for c in t:
        r = rng.random()
        if r < err * 0.4:
            q.append((c + rng.integers(1, 4)) & 3)
        elif r < err * 0.7:
            continue
        elif r < err:
            q.append(c)
            q.append(rng.integers(0, 4))
        else:
            q.append(c)
    q = np.array(q, dtype=np.uint8)
    if drift:
        pos = int(rng.integers(0, max(1, len(q) - 1)))
        if rng.random() < 0.5:
            q = np.concatenate([q[:pos], rng.integers(0, 4, size=drift, dtype=np.uint8), q[pos:]])
        else:
            q = np.concatenate([q[:pos], q[pos + drift:]])
    for _ in range(n_runs):
        if len(q) > 20:
            p = int(rng.integers(0, len(q) - 10))
            q[p:p + int(rng.integers(1, 10))] = 4
    if len(q) == 0:
        q = np.array([0], dtype=np.uint8)
    return q, t


FLAGS = [0, 0x08, 0x40, 0x40 | 0x02 | 0x80]


@pytest.mark.parametrize("seed", range(6))
def test_extd2_matches_reference(seed, request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(100 + seed)
    mat = ol.simple_mat()
    n = 0
    for it in range(60):
        tlen = int(rng.choice([1, 5, 17, 33, 100, 250, 300, 700, 1500]))
        w = int(rng.choice([5, 20, 50, 100, 751, 3001]))
        drift = int(rng.choice([0, 0, 30, 120, 400]))
        q, t = rand_pair(rng, tlen, err=float(rng.choice([0.02, 0.1, 0.3])), drift=drift, n_runs=int(rng.integers(0, 3)))
        flag = FLAGS[int(rng.integers(0, len(FLAGS)))]
        zdrop = int(rng.choice([400, 200, 50, -1]))
        end_bonus = int(rng.choice([-1, 0, 10]))
        params = (4, 2, 24, 1) if rng.random() < 0.8 else (6, 2, 26, 1)
        e2, c2 = ol.oracle_extd2(q, t, mat, *params, w, zdrop, end_bonus, flag)
        g.check(lambda: ol.ref_extd2(q, t, mat, *params, w, zdrop, end_bonus, flag), (e2, c2), (it, tlen, len(q), w, flag, zdrop, e2))
        n += 1
    assert n == 60
    g.done()


@pytest.mark.parametrize("seed", range(4))
def test_extz2_matches_reference(seed, request):
    """The single-affine restatement (oracle wmo_ksw_extz2) against the reference's ksw_extz2_sse (src/ksw2_extz2_sse.c:23), over the
    extd2 matrix plus scoring sets that push the unsigned-offset encoding (large gap costs, asm-like matrices)."""
    g = ol.RefGolden(request)
    rng = np.random.default_rng(300 + seed)
    n = 0
    for it in range(70):
        tlen = int(rng.choice([1, 5, 17, 33, 100, 250, 300, 700, 1500]))
        w = int(rng.choice([5, 20, 50, 100, 751, 3001, -1]))
        drift = int(rng.choice([0, 0, 30, 120, 400]))
        q, t = rand_pair(rng, tlen, err=float(rng.choice([0.02, 0.1, 0.3])), drift=drift, n_runs=int(rng.integers(0, 3)))
        flag = FLAGS[int(rng.integers(0, len(FLAGS)))] | (0x10 if rng.random() < 0.3 else 0)
        zdrop = int(rng.choice([400, 200, 50, -1]))
        end_bonus = int(rng.choice([-1, 0, 10]))
        a, b, go, ge = [(2, 4, 4, 2), (2, 4, 4, 2), (1, 4, 6, 2), (1, 9, 16, 2), (2, 8, 12, 2), (5, 4, 40, 20), (3, 6, 50, 13)][int(rng.integers(0, 7))]
        mat = ol.simple_mat(a, b, 1)
        e2, c2 = ol.oracle_extz2(q, t, mat, go, ge, w, zdrop, end_bonus, flag)
        g.check(lambda: ol.ref_extz2(q, t, mat, go, ge, w, zdrop, end_bonus, flag), (e2, c2), (it, tlen, len(q), w, flag, zdrop, (a, b, go, ge), e2))
        n += 1
    assert n == 70
    g.done()


def spliced_pair(rng, n_exons, err=0.05, rev_sites=False, n_runs=0):
    """(query, target): exons joined in the query, introns with GT..AG (or CT..AC) ends in the target; some sites left non-canonical."""
    q, t = [], []
    for i in range(n_exons):
        ex = rng.integers(0, 4, size=int(rng.integers(8, 120)), dtype=np.uint8)
        t.append(ex)
        qq, _ = rand_pair(rng, 1, err=0.0)
        ex_q = np.array([(c if rng.random() > err else (c + 1) & 3) for c in ex], dtype=np.uint8)
        q.append(ex_q)
        if i + 1 < n_exons:
            intron = rng.integers(0, 4, size=int(rng.integers(30, 400)), dtype=np.uint8)
            if rng.random() < 0.8:
                intron[:3] = [1, 3, 0] if rev_sites else [2, 3, 0]      # GTA / CTA
                intron[-3:] = [1, 0, 1] if rev_sites else [1, 0, 2]     # CAC / CAG
            t.append(intron)
    q = np.concatenate(q); t = np.concatenate(t)
    for _ in range(n_runs):
        if len(t) > 20:
            p0 = int(rng.integers(0, len(t) - 10)); t[p0:p0 + int(rng.integers(1, 6))] = 4
    return q, t


@pytest.mark.parametrize("seed", range(3))
def test_exts2_matches_reference(seed, request):
    """The splice-aware restatement (oracle wmo_ksw_exts2) against the reference's ksw_exts2_sse (src/ksw2_exts2_sse.c:26): the
    splice presets' scoring (src/options.c:116-128), both strands' signals, flank bonus, junction annotation, both gap
    alignments, reversed CIGAR, extension-only, approximate maximum, generic scoring."""
    g = ol.RefGolden(request)
    rng = np.random.default_rng(900 + seed)
    n = 0
    for it in range(90):
        rev_sites = bool(it & 1)
        if it % 5 == 4:
            q, t = rand_pair(rng, int(rng.choice([1, 5, 17, 33, 100, 300])), err=0.1, drift=int(rng.choice([0, 30])), n_runs=int(rng.integers(0, 2)))
        else:
            q, t = spliced_pair(rng, int(rng.integers(1, 6)), err=float(rng.choice([0.0, 0.05, 0.2])), rev_sites=rev_sites, n_runs=int(rng.integers(0, 2)))
        if it % 7 == 3:  # reversed inputs, as the left extension passes them (src/align.c:696-697)
            q, t = q[::-1].copy(), t[::-1].copy()
        flag = FLAGS[int(rng.integers(0, len(FLAGS)))] | (0x10 if rng.random() < 0.3 else 0) | (0x04 if rng.random() < 0.15 else 0)
        flag |= [0x100, 0x200, 0x300, 0][int(rng.integers(0, 4))] | (0x400 if rng.random() < 0.7 else 0)
        if it % 7 == 3:
            flag |= 0x80 | 0x02
        zdrop = int(rng.choice([200, 100, 30, -1]))
        a, b, go, ge, go2, noncan, jb = [(1, 2, 2, 1, 32, 9, 9), (1, 4, 6, 1, 24, 9, 5), (2, 4, 4, 2, 24, 5, 3), (1, 2, 2, 1, 3, 9, 9), (1, 2, 2, 1, 60, 0, 0)][int(rng.integers(0, 5))]
        mat = ol.simple_mat(a, b, 1)
        junc = None
        if rng.random() < 0.4:
            junc = np.where(rng.random(len(t)) < 0.05, rng.integers(1, 16, size=len(t)), 0).astype(np.uint8)
        e2, c2 = ol.oracle_exts2(q, t, mat, go, ge, go2, noncan, zdrop, jb, flag, junc=junc)
        g.check(lambda: ol.ref_exts2(q, t, mat, go, ge, go2, noncan, zdrop, jb, flag, junc=junc), (e2, c2),
                (it, len(t), len(q), hex(flag), zdrop, (a, b, go, ge, go2), e2))
        n += (c2 & 0xf == 3).any()
    assert n > 10  # introns were found
    g.done()


def test_extd2_swapped_gap_and_asm_scoring(request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(7)
    for a, b, q, e, q2, e2 in [(1, 4, 6, 2, 26, 1), (1, 9, 16, 2, 41, 1), (2, 4, 24, 1, 4, 2)]:
        mat = ol.simple_mat(a, b, 1)
        for it in range(15):
            qq, tt = rand_pair(rng, int(rng.integers(20, 600)), err=0.05, drift=int(rng.choice([0, 50])))
            flag = FLAGS[it % 4]
            r2 = ol.oracle_extd2(qq, tt, mat, q, e, q2, e2, 200, 200, -1, flag)
            g.check(lambda: ol.ref_extd2(qq, tt, mat, q, e, q2, e2, 200, 200, -1, flag), r2, (a, b, q, e, q2, e2, it))
    g.done()


@pytest.mark.parametrize("seed", range(3))
def test_ll_matches_reference(seed, request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(300 + seed)
    mat = ol.simple_mat()
    for it in range(80):
        tlen = int(rng.choice([1, 7, 8, 9, 40, 200, 600]))
        if rng.random() < 0.5:
            q, t = rand_pair(rng, tlen, err=0.15, n_runs=int(rng.integers(0, 2)))
        else:
            t = rng.integers(0, 5, size=tlen, dtype=np.uint8)
            q = rng.integers(0, 5, size=int(rng.integers(1, 300)), dtype=np.uint8)
        g.check(lambda: ol.ref_ll(q, t, mat, 4, 2), ol.oracle_ll(q, t, mat, 4, 2), (it, len(q), tlen))
    g.done()


def test_sorts_match_reference_including_ties(request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(5)
    for n in [0, 1, 2, 63, 64, 65, 200, 1000, 5000, 70000]:
        for key_bits in [3, 8, 12, 20, 40, 64]:
            hi = (1 << key_bits) - 1
            x = rng.integers(0, hi, size=n, dtype=np.uint64, endpoint=True)
            if key_bits == 64 and n:
                x[:: 3] = x[0]  # heavy ties
            y = np.arange(n, dtype=np.uint64)
            xy = np.stack([x, y], axis=1)
            g.check(lambda: ol.ref_sort128(xy), ol.oracle_sort128(xy), (n, key_bits))
            g.check(lambda: ol.ref_sort64(x), ol.oracle_sort64(x), (n, key_bits))
    g.done()


def test_bloom_and_sketch_match_reference(request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(11)
    for n_k, k in [(0, 15), (255, 15), (5000, 15), (300, 19)]:
        kmers = rng.integers(0, 1 << (2 * k), size=n_k, dtype=np.uint64)
        ob, rb = ol.OracleBloom(kmers), ol.RefSketch(kmers) if ol.RECORD else None
        g.check(lambda: rb.bits(), ob.bits(), (n_k, k))
        g.check(lambda: rb.table(), ob.table(), (n_k, k))
        probe = rng.integers(0, 1 << (2 * k), size=20000, dtype=np.uint64)
        g.check(lambda: [rb.contains(p) for p in probe[:3000]], [ob.contains(p) for p in probe[:3000]], (n_k, k))
        # sequences: random, with N runs, with short-period repeats (weight ties), down-weighted k-mers planted
        seqs = []
        s = rng.integers(0, 4, size=30000, dtype=np.uint8)
        seqs.append(bytes(b"ACGT"[c] for c in s))
        s2 = bytearray(seqs[0][:8000])
        for p in range(500, 7000, 900):
            s2[p:p + int(rng.integers(1, 80))] = b"N" * 200
        seqs.append(bytes(s2[:8000]))
        unit = bytes(b"ACGT"[c] for c in rng.integers(0, 4, size=7, dtype=np.uint8))
        seqs.append(seqs[0][:300] + unit * 60 + seqs[0][300:900] + b"A" * 120 + seqs[0][900:1500] + (b"AC" * 70) + seqs[0][1500:2000])
        if n_k:
            # plant listed k-mers so that the down-weighting branch is exercised
            planted = bytearray(seqs[0][:5000])
            for j in range(40):
                km = int(kmers[j])
                st = "".join("ACGT"[(km >> (2 * (k - 1 - i))) & 3] for i in range(k)).encode()
                p = 100 + j * 110
                planted[p:p + k] = st
            seqs.append(bytes(planted))
        seqs.append(b"ACGTACGTAC")  # shorter than k
        for w in (50, 10):
            for si, sq in enumerate(seqs):
                b = ol.oracle_sketch(sq, w, k, 3, ob)
                g.check(lambda: rb.sketch(sq, w, k, 3), b, (n_k, k, w, si, len(b)))
    g.done()


def test_sketch_even_k_symmetric_kmers(request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(12)
    ob, rb = ol.OracleBloom([]), ol.RefSketch(np.zeros(0, dtype=np.uint64)) if ol.RECORD else None
    s = bytes(b"ACGT"[c] for c in rng.integers(0, 4, size=5000, dtype=np.uint8))
    s = s[:1000] + b"ACGTACGTACGTACGTAATT" * 5 + s[1000:]
    for k in (6, 16):
        g.check(lambda: rb.sketch(s, 20, k, 0), ol.oracle_sketch(s, 20, k, 0, ob), k)
    g.done()


def make_anchors(rng, n, span=15, repeats=False):
    """Synthetic sorted anchors shaped like collect_seed_hits output."""
    rpos = np.sort(rng.integers(100, 60000, size=n)).astype(np.uint64)
    if repeats:
        rpos = (rpos // 7) * 7
    q = (rpos.astype(np.int64) + rng.integers(-40, 40, size=n)).clip(20, None).astype(np.uint64)
    rev = (rng.random(n) < 0.3).astype(np.uint64)
    x = rev << np.uint64(63) | rpos
    y = np.uint64(span) << np.uint64(32) | q
    xy = np.stack([x, y], axis=1)
    return ol.oracle_sort128(xy)  # the reference's order: test_sorts_match_reference_including_ties


@pytest.mark.parametrize("seed", range(4))
def test_chain_matches_reference(seed, request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(400 + seed)
    for n in [0, 1, 3, 10, 100, 700, 3000]:
        a = make_anchors(rng, n, repeats=bool(seed & 1))
        for (mx, mn, my, bw) in [(5000, 1000, 5000, 500), (16000, 1000, 16000, 2000)]:
            u2, b2 = ol.oracle_chain(a, mx, mn, my, bw)
            g.check(lambda: ol.ref_chain(a, mx, mn, my, bw), (u2, b2), (n, mx, len(u2)))
        # small max_iter exercises the Winnowmap window rule (chain.c:52-55)
        u2, b2 = ol.oracle_chain(a, 5000, 50, 5000, 500, max_iter=20, max_skip=3)
        g.check(lambda: ol.ref_chain(a, 5000, 50, 5000, 500, max_iter=20, max_skip=3), (u2, b2), (n, len(u2)))
    g.done()
