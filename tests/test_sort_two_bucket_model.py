"""The derivation behind csrc/seed.cu:wm_gs_two_bucket_pass, checked on the CPU against the reference's own sort.

A radix pass of the reference (rs_sort, src/ksort.h:116-146) whose keys fall into exactly TWO buckets is replaced in the walker kernels by
a closed form: the misplaced elements of the lower bucket's region swap, in order, with the misplaced ones of the upper region, and the
upper region shifts its own elements one slot to the right up to the last misplaced one.  Here the whole sort is restated in Python --
serial cycle-leader walk for the other passes, the closed form for the two-bucket ones -- and compared with ref_radix_sort_128x
(oracle/_ref, the reference's compiled code; its results on these seeded inputs are recorded under tests/golden/ref/).  The CUDA
implementation itself is checked on the GPU (tests/test_gpu_stages.py).

The second test checks the general form of the same observation (DESIGN.md section 8, not built as a kernel yet): the j-th element to
arrive in a bucket ejects that bucket's j-th misplaced element, so the serial part of ANY pass is a token walk over the destination
digits of the misplaced elements with one arrival counter per bucket; where each element lands follows from its arrival index."""
import numpy as np

import oracle_lib as ol


def _walk(a, beg, end, s):
    cnt = [0] * 256
    for i in range(beg, end):
        cnt[(int(a[i, 0]) >> s) & 255] += 1
    b, e, acc = [0] * 256, [0] * 256, beg
    for k in range(256):
        b[k] = acc; acc += cnt[k]; e[k] = acc
    w = b[:]
    k = 0
    while k < 256:  # src/ksort.h:126-138
        if w[k] != e[k]:
            l = (int(a[w[k], 0]) >> s) & 255
            if l != k:
                tmp = a[w[k]].copy()
                while True:
                    swap = tmp; tmp = a[w[l]].copy(); a[w[l]] = swap; w[l] += 1
                    l = (int(tmp[0]) >> s) & 255
                    if l == k:
                        break
                a[w[k]] = tmp; w[k] += 1
            else:
                w[k] += 1
        else:
            k += 1
    return b, e


def _closed_form(a, beg, end, s):
    d = (a[beg:end, 0] >> np.uint64(s)) & np.uint64(255)
    lo, hi = (int(v) for v in np.unique(d))
    n, mid = end - beg, int((d == lo).sum())
    orig, is_lo = a[beg:end].copy(), d == lo
    P = np.nonzero(~is_lo[:mid])[0]           # lower region, holding upper-bucket elements
    Q = np.nonzero(is_lo[mid:])[0] + mid      # upper region, holding lower-bucket elements
    m = len(P)
    assert len(Q) == m
    new = orig.copy()
    new[P] = orig[Q]
    c = 0
    for t in range(mid, n):
        if c == m:
            break
        new[t] = orig[P[c]] if (t == mid or is_lo[t - 1]) else orig[t - 1]
        c += int(is_lo[t])
    a[beg:end] = new
    b = [beg if k <= lo else (beg + mid if k <= hi else end) for k in range(256)]
    e = [beg if k < lo else (beg + mid if k < hi else end) for k in range(256)]
    return b, e


def _insertion(a, beg, end):  # src/ksort.h:104-115
    for i in range(beg + 1, end):
        if a[i, 0] < a[i - 1, 0]:
            tmp, j = a[i].copy(), i
            while j > beg and tmp[0] < a[j - 1, 0]:
                a[j] = a[j - 1]; j -= 1
            a[j] = tmp


def _rs(a, beg, end, s, used):
    d = (a[beg:end, 0] >> np.uint64(s)) & np.uint64(255)
    if len(np.unique(d)) == 2:
        b, e = _closed_form(a, beg, end, s); used[0] += 1
    else:
        b, e = _walk(a, beg, end, s)
    if s:
        for k in range(256):
            if e[k] - b[k] > 64:
                _rs(a, b[k], e[k], s - 8, used)
            elif e[k] - b[k] > 1:
                _insertion(a, b[k], e[k])


def test_two_bucket_closed_form_equals_the_reference_walk(request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(5)
    used = [0]
    for it in range(14):
        n = int(rng.choice([70, 200, 1000, 2500]))
        pos = rng.integers(65536 * 3 - 300, 65536 * 3 - 300 + int(rng.choice([300, 5000, 70000])), size=n).astype(np.uint64)
        if it % 4 == 0:  # few distinct positions: heavy ties
            pos = pos[rng.integers(0, max(2, n // 30), size=n)]
        strand = (rng.random(n) < [0.0, 0.01, 0.5][it % 3]).astype(np.uint64)
        x = (strand << np.uint64(63)) | (np.uint64(it % 2) << np.uint64(32)) | pos
        a = np.ascontiguousarray(np.stack([x, np.arange(n, dtype=np.uint64)], axis=1))
        got = a.copy()
        if n <= 64:
            _insertion(got, 0, n)
        else:
            _rs(got, 0, n, 56, used)
        g.check(lambda: ol.ref_sort128(a), got, (it, n))
    assert used[0] >= 10
    g.done()


def _token_pass(a, beg, end, s, steps):
    orig = a[beg:end].copy()
    d = ((orig[:, 0] >> np.uint64(s)) & np.uint64(255)).astype(np.int64)
    cnt = np.bincount(d, minlength=256)
    B = np.zeros(257, np.int64); B[1:] = np.cumsum(cnt)
    own = np.repeat(np.arange(256), cnt)                 # the bucket every slot belongs to
    mis = np.nonzero(d != own)[0]
    E = [mis[own[mis] == k] for k in range(256)]         # misplaced slots of every bucket, ascending
    D = [d[E[k]] for k in range(256)]                    # ... and where their elements want to go
    arrivals, A, land = [0] * 256, [0] * 256, {}
    for k in range(256):                                 # the serial part: digits and counters only
        A[k] = arrivals[k]                               # elements of k ejected by arrivals before its own turn
        for c in range(A[k], len(E[k])):                 # the others open a cycle each (src/ksort.h:129-136)
            cur, t = (k, c), int(D[k][c])
            while True:
                steps[0] += 1
                j = arrivals[t]; arrivals[t] += 1
                land[int(E[cur[0]][cur[1]])] = (0, t, j)  # lands at the start of run j of bucket t
                cur, t2 = (t, j), int(D[t][j])
                if t2 == k:
                    land[int(E[t][j])] = (1, k, c)        # closes the cycle: lands where it was opened
                    break
                t = t2
    new = orig.copy()                                    # the parallel part: pure index arithmetic
    for t in range(256):
        for r in range(A[t]):                            # the bucket's own elements of run r move one slot to the right
            start = int(B[t]) if r == 0 else int(E[t][r - 1]) + 1
            new[start + 1:int(E[t][r]) + 1] = orig[start:int(E[t][r])]
    for src, (closing, t, j) in land.items():
        if closing:
            new[int(E[t][j])] = orig[src]
        else:
            new[int(B[t]) if j == 0 else int(E[t][j - 1]) + 1] = orig[src]
    a[beg:end] = new
    return [beg + int(B[k]) for k in range(256)], [beg + int(B[k + 1]) for k in range(256)]


def _rs_token(a, beg, end, s, steps):
    b, e = _token_pass(a, beg, end, s, steps)
    if s:
        for k in range(256):
            if e[k] - b[k] > 64:
                _rs_token(a, b[k], e[k], s - 8, steps)
            elif e[k] - b[k] > 1:
                _insertion(a, b[k], e[k])


def test_token_walk_formulation_equals_the_reference_sort(request):
    g = ol.RefGolden(request)
    rng = np.random.default_rng(11)
    for it in range(10):
        n = int(rng.choice([100, 400, 1500, 4000]))
        pos = rng.integers(1000, 1000 + int(rng.choice([300, 5000, 70000, 900000])), size=n).astype(np.uint64)
        if it % 3 == 0:
            pos = pos[rng.integers(0, max(2, n // 25), size=n)]
        strand = (rng.random(n) < [0.0, 0.02, 0.5][it % 3]).astype(np.uint64)
        x = (strand << np.uint64(63)) | (np.uint64(rng.integers(0, 3)) << np.uint64(32)) | pos
        a = np.ascontiguousarray(np.stack([x, np.arange(n, dtype=np.uint64)], axis=1))
        got, steps = a.copy(), [0]
        _rs_token(got, 0, n, 56, steps)
        g.check(lambda: ol.ref_sort128(a), got, (it, n))
        assert steps[0] <= 2 * n  # serial steps of the whole sort: about 1.3 per element, against 2-3 walker steps per element today
    g.done()
