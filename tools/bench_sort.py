#!/usr/bin/env python
"""Tuning aid (GPU box): the tie-exact anchor sort on arrays shaped like the anchors of a read inside a tandem array
(concatenated ascending runs, many equal keys).  Prints the wall time of one call and the device time of the sort alone (CUDA
events, copies left out).  Run under ncu to see the kernel times:
   ncu --metrics gpu__time_duration.sum --csv --log-file x.csv python tools/bench_sort.py --n 30000 --arrays 200"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def tandem_array(rng, n, unit=171, n_kmers=4, strand_frac=0.0):
    copies = 750
    runs = max(1, n // copies)
    offs = rng.integers(0, unit, size=n_kmers)
    base = int(rng.integers(1 << 20, 1 << 27))
    x, y = [], []
    for m in range(runs):
        o = int(offs[m % n_kmers])
        x.append(base + np.arange(copies, dtype=np.int64) * unit + o)
        y.append(np.full(copies, 100 + m * 43, dtype=np.int64))
    x = np.concatenate(x).astype(np.uint64); y = np.concatenate(y).astype(np.uint64)
    if strand_frac > 0:  # hits on the other strand: bit 63 of x (two buckets in the first pass)
        x = x | (rng.random(len(x)) < strand_frac).astype(np.uint64) << np.uint64(63)
    return np.stack([x, np.uint64(15) << np.uint64(32) | y], axis=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=30000)
    ap.add_argument("--arrays", type=int, default=200)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--strand-frac", type=float, default=0.0)
    ap.add_argument("--repeat", type=int, default=5, help="device-timed runs of the whole batch")
    a = ap.parse_args()
    from winnowmap_b200 import kernels
    rng = np.random.default_rng(5)
    arrays = [tandem_array(rng, a.n, strand_frac=a.strand_frac) for _ in range(a.arrays)]
    kernels.radix_sort_128x_batch(arrays[:2])
    t0 = time.time()
    out = kernels.radix_sort_128x_batch(arrays)
    dt = time.time() - t0
    print(f"{a.arrays} arrays x {len(arrays[0])} anchors: {dt * 1e3:.1f} ms wall (incl. copies)")
    dev = [kernels.radix_sort_128x_batch(arrays, timed=True)[1] for _ in range(a.repeat)]
    print(f"{a.arrays} arrays x {len(arrays[0])} anchors: device ms of the sort (copies left out) median {np.median(dev):.2f} "
          f"min {min(dev):.2f} max {max(dev):.2f} over {a.repeat} runs")
    if a.check:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as ol
        for i in range(min(6, a.arrays)):
            assert np.array_equal(ol.oracle_sort128(arrays[i]), out[i]), i
        print("matches the oracle")


if __name__ == "__main__":
    main()
