"""The token-walk radix pass of csrc/seed.cu:wm_anchor_sort_giant_kernel (wm_gs_token_pass).

A pass with three or more non-empty buckets is done in three parts: the misplaced slots are compacted (ascending, hence grouped by the
bucket that owns the slot) with the destination digit of their element; one thread walks the cycles over those digits only, with one
arrival pointer per bucket; and every element's destination follows from index arithmetic.  The CPU test restates the kernel's
flat-index form and compares it pass by pass with the serial walk of src/ksort.h:126-138 (_walk, whose sorts are pinned to the
reference's answers in test_sort_two_bucket_model.py) and its step count with the model there (_token_pass).  The GPU test runs the
kernel through the C ABI against the CPU oracle, on both sides of the shared-memory cap of the digit list and with the old walker."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
from test_sort_two_bucket_model import _token_pass, _walk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _flat_token_pass(a, beg, end, s):
    """The kernel's pass on a[beg:end] (in place).  Returns (B, E, steps)."""
    n = end - beg
    orig = a[beg:end].copy()
    d = ((orig[:, 0] >> np.uint64(s)) & np.uint64(255)).astype(np.int64)
    cnt = np.bincount(d, minlength=256)
    B = np.zeros(257, np.int64); B[1:] = np.cumsum(cnt)
    own = np.searchsorted(B[1:], np.arange(n), side="right")  # the bucket owning every slot (smallest k with E[k] > i)
    # compaction: M (slots), D (digits) and the per-bucket offsets moff of the misplaced list
    M = np.nonzero(d != own)[0]
    D = d[M]
    moff = np.zeros(257, np.int64); moff[1:] = np.cumsum(np.bincount(own[M], minlength=256))
    # the walk (one thread): ptr[] per bucket, land[] written only
    ptr, A, land, steps = moff[:256].copy(), np.zeros(256, np.int64), np.zeros(len(M), np.int64), 0
    for k in range(256):
        f = int(ptr[k]); A[k] = f - moff[k]
        while f < moff[k + 1]:
            opener, cur, t = f, f, int(D[f]); f += 1
            while True:
                p = int(ptr[t]); ptr[t] = p + 1; steps += 1
                land[cur] = p
                t2 = int(D[p])
                if t2 == k:
                    land[p] = ~opener
                    break
                cur, t = p, t2
        ptr[k] = f
    # destinations of the misplaced elements
    dest = np.empty(len(M), np.int64)
    for g in range(len(M)):
        L = int(land[g])
        if L < 0:
            dest[g] = M[~L]                                   # closes a cycle: where the cycle was opened
        else:
            t = int(np.searchsorted(moff[1:], L, side="right"))  # bucket of arrival index L
            dest[g] = B[t] if L == moff[t] else M[L - 1] + 1  # the start of run L - moff[t] of bucket t
    # placement: everything else moves one slot right if its run is ejected before its bucket's turn
    g = np.cumsum(d != own) - (d != own)                      # exclusive rank of every slot among the misplaced
    out = np.empty_like(orig)
    for i in range(n):
        if d[i] != own[i]:
            out[dest[g[i]]] = orig[i]
        else:
            out[i + 1 if g[i] - moff[own[i]] < A[own[i]] else i] = orig[i]
    a[beg:end] = out
    return [beg + int(B[k]) for k in range(256)], [beg + int(B[k + 1]) for k in range(256)], steps


def _array(rng, n, n_buckets, ties, shift):
    digits = rng.choice(256, size=n_buckets, replace=False).astype(np.uint64)
    x = digits[rng.integers(0, n_buckets, size=n)] << np.uint64(shift)
    x |= rng.integers(0, 1 << 20, size=n).astype(np.uint64) if not ties else rng.integers(0, 3, size=n).astype(np.uint64)
    return np.ascontiguousarray(np.stack([x, np.arange(n, dtype=np.uint64)], axis=1))


@pytest.mark.parametrize("n_buckets", [3, 4, 17, 100, 256])
@pytest.mark.parametrize("ties", [False, True])
def test_flat_token_pass_equals_the_serial_walk(n_buckets, ties):
    rng = np.random.default_rng(1000 * n_buckets + ties)
    for it in range(4):
        n = int(rng.choice([n_buckets + 5, 300, 3000]))
        s = 8 * int(rng.integers(3, 8))
        a = _array(rng, n, n_buckets, ties, s)
        if it == 1:  # a prefix already in place: buckets with no misplaced elements
            a[: n // 2] = a[np.argsort(a[: n // 2, 0] >> np.uint64(s), kind="stable")]
        if it == 3:  # the whole array in place except for a few elements
            a = a[np.argsort(a[:, 0] >> np.uint64(s), kind="stable")]
            sw = rng.integers(0, n, size=(3, 2))
            for i, j in sw:
                a[[i, j]] = a[[j, i]]
        want, got, model = a.copy(), a.copy(), a.copy()
        bw, ew = _walk(want, 0, n, s)
        bg, eg, steps = _flat_token_pass(got, 0, n, s)
        model_steps = [0]
        _token_pass(model, 0, n, s, model_steps)
        assert np.array_equal(want, got), (n_buckets, ties, it)
        assert (bw, ew) == (bg, eg)
        assert steps == model_steps[0]
        assert steps <= n


def test_flat_token_sort_on_tandem_arrays_matches_the_oracle():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_sort import tandem_array
    rng = np.random.default_rng(7)
    for frac in (0.0, 0.02, 0.5):
        a = tandem_array(rng, 3000, strand_frac=frac)
        got = a.copy()

        def rs(beg, end, s):
            b, e, _ = _flat_token_pass(got, beg, end, s)
            if s:
                for k in range(256):
                    if e[k] - b[k] > 64:
                        rs(b[k], e[k], s - 8)
                    elif e[k] - b[k] > 1:
                        got[b[k]:e[k]] = ol.oracle_sort128(got[b[k]:e[k]])
        rs(0, len(a), 56)
        assert np.array_equal(ol.oracle_sort128(a), got), frac


def _gpu_arrays():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_sort import tandem_array
    rng = np.random.default_rng(23)
    arrays = []
    for n in (2049, 2500, 9000, 40000, 150000, 520000):
        for frac in (0.0, 0.02, 0.5):
            arrays.append(tandem_array(rng, n + 750, strand_frac=frac)[:n])
    for n, nb in ((3000, 3), (5000, 256), (60000, 200), (200000, 256)):  # few misplaced (staged digits) to most misplaced (byte FIFOs)
        x = rng.integers(0, nb, size=n).astype(np.uint64) << np.uint64(24) | rng.integers(0, 40, size=n).astype(np.uint64)
        arrays.append(np.stack([x, rng.integers(0, 1 << 40, size=n).astype(np.uint64)], axis=1))
    return arrays


@pytest.mark.gpu
def test_token_walk_sort_matches_oracle():
    from winnowmap_b200 import kernels
    arrays = _gpu_arrays()
    got = kernels.radix_sort_128x_batch(arrays)
    for a, g in zip(arrays, got):
        assert np.array_equal(ol.oracle_sort128(a), g), len(a)


_OLD_WALKER = """
import sys, numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
import oracle_lib as ol
from test_sort_token_walk import _gpu_arrays
from winnowmap_b200 import kernels
arrays = _gpu_arrays()
for a, g in zip(arrays, kernels.radix_sort_128x_batch(arrays)):
    assert np.array_equal(ol.oracle_sort128(a), g), len(a)
print("ok")
"""


@pytest.mark.gpu
def test_old_walker_still_matches_oracle():
    env = dict(os.environ, WM_SORT_TOKEN_MIN="0")
    code = _OLD_WALKER.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-2000:]
