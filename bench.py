#!/usr/bin/env python
"""bench.py -- mapped bases/sec of the seed-chain-align path on B200 (BASELINE.json metric).

Workload: BASELINE.json configs[4] (the configuration the metric and north_star's target are quoted on), scaled in
reference LENGTH only so that a default run ends within minutes on a fresh box: a tandem-repeat-enriched synthetic
reference (SURVEY.md 8d: every 1 Mbp an array of copies of a unit from a fixed family of 4 base units, 171 / 340 /
2000 / 5000 bp, ~15 % of the genome; seed 1005), WM_BENCH_REF_LEN bases (default 500 Mbp instead of 3 Gbp: the
3 Gbp reference takes the REFERENCE implementation ~10 minutes to index, and every driver run of either arm pays
that once; the read distribution, the repeat structure and every option are those of the config), ONT-like reads
N50 = 30 kb at 5 % error, `-x map-ont -W <top-0.02 % 15-mers> -c`.  WM_BENCH_REF_LEN=3000000000 runs the full size.

One "step" = one pass of the hot path (stage-1 MCAS waves + stage-2 remap: sketch, seed lookup, anchor sort,
chaining, extension DP with traceback, host glue) over --reads fresh reads (~26.5 Mbase; working set -- read pool,
anchors, backtrack matrices, multi-GB index -- far larger than L2).  Steps are submitted to the library in groups of
at most WM_BENCH_GROUP steps (default 32) and the library cuts each submission into chunks of WM_CHUNK_BASES bases
(pinned here to 32 Mbase), so device and host footprints do not grow with --steps.

  value : bases/s with the raw reads of all K steps already resident in one HBM pool (wm_bench_upload); CUDA events
          bracket the whole pass (ASCII -> 2-bit codes is inside: it is part of the path)
  e2e   : bases/s through wm_gpu_map_batch -- the call INTEGRATION.md binds at src/map.c:1164 -- with host buffers
          (staging + H2D of the reads, D2H of every chain, DP result and CIGAR inside the timed region)
  roofline : the dominant kernel of the run (the DP fill kernel or the chaining forward pass, whichever ran longer;
          the other one is reported under roofline_other): algorithmic bytes (SURVEY.md 8d) over the time during which a
          kernel of that class was running (CUDA events around every launch, union of the intervals), vs the measured HBM peak
  cpu_baseline : the real reference (oracle/_ref/winnowmap, SSE4.1, all host threads) on a bounded sample (N = 1 only)
  parity_checked : the records produced by the two timed passes (resident and host-buffer) for the reads of the CPU
          sample, formatted as PAF, are byte-identical to the reference's output on the same reads

--impl reference times the reference binary itself on the same workload in ONE invocation (one index build): the
reads of all W + K steps go into one file, the mini-batch size (-K) is a group of steps, and the timed interval is
taken from the reference's own per-mini-batch stderr stamps.
Under torchrun (N > 1) every rank maps its own K steps (reads shard with no data-path collective): weak scaling.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")  # before anything loads libgomp: idle workers must not spin (see _lib.py)
os.environ.setdefault("WM_CHUNK_BASES", "32000000")  # fixed chunk size: footprint independent of --steps

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

# per user: on a shared machine another user's cache directory is not writable
CACHE = os.environ.get("WM_BENCH_CACHE", os.path.join(tempfile.gettempdir(), f"wm_bench_cache_{os.getuid()}"))
REF_LEN = int(os.environ.get("WM_BENCH_REF_LEN", 500_000_000))
GROUP = max(1, int(os.environ.get("WM_BENCH_GROUP", 32)))
N50, ERR, K = 30000, 0.05, 15
CONTIGS = None  # set by load_workload(); read by the forked read generators


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def workload_name():
    full = REF_LEN >= 3_000_000_000
    return (f"BASELINE configs[4]{'' if full else ' at reduced reference length'}: {REF_LEN / 1e6:.0f} Mbp tandem-repeat-enriched synthetic ref "
            f"(4 unit families, ~15 % of the genome), ONT reads N50=30kb 5% err, -x map-ont -W top-0.02% k=15 -c")


def make_workload():
    """Reference FASTA + -W list on disk (cached); only one process per node does this."""
    import gen_data
    os.makedirs(CACHE, exist_ok=True)
    ref = os.path.join(CACHE, f"tr_ref_{REF_LEN}.fa")
    wf = os.path.join(CACHE, f"tr_rep_{REF_LEN}_k{K}.txt")
    if os.path.exists(ref) and os.path.exists(wf):
        return ref, wf
    t0 = time.time()
    rng = np.random.default_rng(1005)  # seed 1000 + cfg
    contigs = gen_data.make_ref(rng, REF_LEN, max(1, round(REF_LEN / 250_000_000)), True)  # one contig per 250 Mbp (SURVEY.md 8d)
    gen_data.write_fasta(ref + ".tmp", contigs)
    n, thr = gen_data.write_top_kmers(wf + ".tmp", contigs, K, 0.9998)
    os.replace(wf + ".tmp", wf)
    os.replace(ref + ".tmp", ref)  # last: its presence says both files are complete
    log(f"workload generated in {time.time() - t0:.1f}s; -W list: {n} k-mers above count {thr}")
    return ref, wf


def load_workload(rank):
    """(ref_path, w_path); the contigs end up in CONTIGS.  Rank 0 generates, the others wait for the files."""
    global CONTIGS
    ref = os.path.join(CACHE, f"tr_ref_{REF_LEN}.fa")
    wf = os.path.join(CACHE, f"tr_rep_{REF_LEN}_k{K}.txt")
    if rank == 0:
        make_workload()
    else:
        t0 = time.time()
        while not (os.path.exists(ref) and os.path.exists(wf)):
            if time.time() - t0 > 3600:
                raise RuntimeError("timed out waiting for rank 0 to generate the workload")
            time.sleep(1.0)
    raw = np.fromfile(ref, dtype=np.uint8)  # one line per contig (gen_data.write_fasta)
    nl = np.flatnonzero(raw == 10)
    CONTIGS = []
    for i in range(0, len(nl), 2):
        h0 = 0 if i == 0 else nl[i - 1] + 1
        CONTIGS.append((raw[h0 + 1:nl[i]].tobytes().decode(), raw[nl[i] + 1:nl[i + 1]]))
    return ref, wf


def _gen_step(args):
    import gen_data
    n_reads, seed = args
    recs = gen_data.make_reads(np.random.default_rng(seed), CONTIGS, n_reads, N50, ERR, min_len=1000)
    return [(f"s{seed}_{nm}", s.tobytes()) for nm, s in recs]


def gen_steps(n_steps, n_reads, seed0):
    """n_steps batches of n_reads reads (name, bytes), deterministic per (seed0, step); forked workers share CONTIGS."""
    import multiprocessing as mp
    jobs = [(n_reads, seed0 + s) for s in range(n_steps)]
    nproc = max(1, min(len(jobs), (os.cpu_count() or 2) // 2, 32))
    if nproc == 1:
        return [_gen_step(j) for j in jobs]
    with mp.get_context("fork").Pool(nproc) as pool:
        return pool.map(_gen_step, jobs)


def write_reads(path, recs):
    with open(path, "wb") as f:
        for nm, s in recs:
            f.write(b">" + nm.encode() + b"\n" + s + b"\n")


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML is polled in-process
    every 20 ms (an nvidia-smi subprocess takes longer than a short timed region); nvidia-smi is the fallback."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index=0, uuid=None):
        super().__init__(daemon=True)
        self.index, self.uuid, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, uuid, [], set(), False, None
        self.source = None

    def _nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = None
        if self.uuid:
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid if isinstance(self.uuid, bytes) else self.uuid.encode())
            except Exception:
                h = None
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        self.source = "nvml"
        while not self.stop_flag:
            self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
            try:
                r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            for nm, bit in self.REASONS.items():
                if r & bit:
                    self.reasons.add(nm)
            time.sleep(0.02)

    def _smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self.source = "nvidia-smi"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)

    def run(self):
        try:
            self._nvml()
        except Exception:
            if not self.stop_flag:
                self._smi()

    def result(self):
        self.stop_flag = True
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s),
                "source": self.source}


def run_reference(refbin, ref, wf, reads_fa, threads, out_path=None, mini_batch=None):
    """One invocation of the reference.  Returns (t_index, [(stamp, n_seq) per mini-batch]) from its own stderr stamps
    (main.c:401 "loaded/built the index", map.c:1220 "mapped N sequences"); stdout goes to out_path (or is discarded)."""
    cmd = [refbin, "-t", str(threads), "-c", "-x", "map-ont", "-W", wf]
    if mini_batch:
        cmd += ["-K", str(int(mini_batch))]
    cmd += [ref, reads_fa]
    out = open(out_path, "wb") if out_path else subprocess.DEVNULL
    try:
        p = subprocess.run(cmd, stdout=out, stderr=subprocess.PIPE, text=True)
    finally:
        if out_path:
            out.close()
    t_idx, stamps = None, []
    for ln in p.stderr.splitlines():
        if ln.startswith("[M::main::") and "loaded/built the index" in ln:
            t_idx = float(ln.split("::")[2].split("*")[0])
        if ln.startswith("[M::worker_pipeline::") and "mapped" in ln:
            stamps.append((float(ln.split("::")[2].split("*")[0]), int(ln.rsplit("mapped", 1)[1].split()[0])))
    if p.returncode != 0 or t_idx is None or not stamps:
        raise RuntimeError("reference run failed: " + p.stderr[-400:])
    return t_idx, stamps


# wm_reg1_t (include/winnowmap_b200.h): 15 int32, the bit-field word (mapq:8 split:2 rev:1 inv:1 sam_pri:1 ...), hash, div, ->p
REG1 = np.dtype([(f, "<i4") for f in ("id", "cnt", "rid", "score", "qs", "qe", "rs", "re", "parent", "subsc", "as", "mlen", "blen", "n_sub",
                                      "score0")] + [("bits", "<u4"), ("hash", "<u4"), ("div", "<f4"), ("p", "<u8")])
# reads of the last step dumped: a seeded sample of at most this many bases (all of a default step) -- about 0.45 byte of
# output per base on the bench workload, so the files stay well under DUMP_LIMIT
DUMP_BASES = 32_000_000
DUMP_LIMIT = 64 << 20


def dump_outputs(L, ctx, step_reads, first, out_dir):
    """The records the timed (resident) pass returned for the reads of its last step -- a fixed sample of them, drawn from the
    inputs alone -- as float64 arrays out_dir/<name>.npy: per read (read_*), per record (reg_*) and the CIGARs of the records,
    concatenated (cigar, len << 4 | op; reg_n_cigar says where each record's ops end)."""
    order = np.random.default_rng(0).permutation(len(step_reads))
    n_keep = int(np.searchsorted(np.cumsum([len(step_reads[i][1]) for i in order]), DUMP_BASES, side="right"))
    keep = np.sort(order[:max(1, n_keep)])
    L.wm_sizeof_reg1.restype = C.c_int
    assert L.wm_sizeof_reg1() == REG1.itemsize
    L.wm_bench_records.restype = C.c_int64
    L.wm_bench_records.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    out = {k: [] for k in ["read_index", "read_n_reg", "read_rep_len", "reg_read"] + [f"reg_{f}" for f in REG1.names[:15]] +
           ["reg_mapq", "reg_split", "reg_rev", "reg_inv", "reg_sam_pri", "reg_hash", "reg_div", "reg_dp_score", "reg_dp_max",
            "reg_dp_max2", "reg_n_ambi", "reg_trans_strand", "reg_n_cigar", "cigar"]}
    n_reg, rep_len = np.zeros(1, np.int32), np.zeros(1, np.int32)
    for i in keep:
        n = L.wm_bench_records(ctx, first + int(i), 1, n_reg.ctypes.data, rep_len.ctypes.data, None, 0)
        regs = np.zeros(n, REG1)
        L.wm_bench_records(ctx, first + int(i), 1, n_reg.ctypes.data, rep_len.ctypes.data, regs.ctypes.data, n)
        out["read_index"].append(i); out["read_n_reg"].append(n_reg[0]); out["read_rep_len"].append(rep_len[0])
        for r in regs:
            out["reg_read"].append(i)
            for f in REG1.names[:15]:
                out[f"reg_{f}"].append(r[f])
            b = int(r["bits"])
            for f, sh, w in (("mapq", 0, 8), ("split", 8, 2), ("rev", 10, 1), ("inv", 11, 1), ("sam_pri", 12, 1)):
                out[f"reg_{f}"].append((b >> sh) & ((1 << w) - 1))
            out["reg_hash"].append(r["hash"]); out["reg_div"].append(r["div"])
            # wm_extra_t: capacity, dp_score, dp_max, dp_max2, n_ambi:30 | trans_strand:2, n_cigar, cigar[]
            ex = np.frombuffer(C.string_at(int(r["p"]), 24), np.int32) if r["p"] else np.zeros(6, np.int32)
            for f, v in zip(("dp_score", "dp_max", "dp_max2"), ex[1:4]):
                out[f"reg_{f}"].append(v)
            amb = int(ex[4]) & 0xffffffff
            out["reg_n_ambi"].append(amb & 0x3fffffff); out["reg_trans_strand"].append(amb >> 30); out["reg_n_cigar"].append(ex[5])
            if ex[5] > 0:
                out["cigar"].append(np.frombuffer(C.string_at(int(r["p"]) + 24, 4 * int(ex[5])), np.uint32))
    out["cigar"] = np.concatenate(out["cigar"]) if out["cigar"] else np.zeros(0)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in out.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT}")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    log(f"dumped {len(keep)} of {len(step_reads)} reads of the last step, {len(arrays['reg_read'])} records, {total / 1e6:.1f} MB to {out_dir}")


def paf_by_read(path):
    """read name -> list of its lines, in file order (the reference prints a mini-batch sorted by length, we print in input order)."""
    d = {}
    with open(path, "rb") as f:
        for ln in f:
            d.setdefault(ln.split(b"\t", 1)[0], []).append(ln)
    return d


def reference_arm(a, cores, refbin):
    """--impl reference: the reference's own CPU implementation, one invocation, timed from its mini-batch stamps."""
    ref, wf = load_workload(0)
    per_step = a.cpu_reads_per_step
    steps = gen_steps(a.warmup + a.steps, per_step, 7_000_000)
    recs = [r for s in steps for r in s]
    lens = [len(s) for _, s in recs]
    # mini-batch = a group of steps (the reference cuts a batch when its bases reach -K): large enough to keep all threads busy
    g = max(1, min(GROUP, a.warmup if a.warmup > 0 else a.steps))
    mb = max(1, int(np.mean(lens) * per_step * g))
    with tempfile.TemporaryDirectory(prefix="wm_bench_") as td:
        fa = os.path.join(td, "reads.fa")
        write_reads(fa, recs)
        t_idx, stamps = run_reference(refbin, ref, wf, fa, cores, None, mb)
    # the timed interval starts at the stamp of the mini-batch that holds the last warm-up read
    n_warm = a.warmup * per_step
    done, t_start, bases, n_timed = 0, t_idx, 0, 0
    for t, n in stamps:
        if done + n <= n_warm or done < n_warm:
            t_start = t  # this batch still holds warm-up reads: excluded
        else:
            bases += sum(lens[done:done + n]); n_timed += n
        done += n
    t_end = stamps[-1][0]
    if n_timed == 0 or t_end <= t_start:
        raise RuntimeError("reference run: no timed mini-batch")
    dt = t_end - t_start
    val = bases / dt
    eq_steps = n_timed / per_step
    print(json.dumps({"impl": "reference", "metric": "mapped bases/sec", "value": val, "unit": "bases/s", "n_gpus": a.gpus, "steps": a.steps,
                      "warmup": a.warmup, "ms_per_step": 1e3 * dt / eq_steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "int8", "data": "synthetic",
                      "config": {"workload": workload_name(), "reads_per_step": per_step, "host_threads": cores,
                                 "note": f"one invocation, index build ({t_idx:.0f}s) excluded; mini-batches of {g} steps (-K {mb}); timed: "
                                         f"{n_timed} reads ({bases / 1e6:.0f} Mbase) after {done - n_timed} warm-up reads"},
                      "cpu_baseline": {"value": val, "unit": "bases/s", "cores": cores, "kind": "reference",
                                       "sample": f"{n_timed} reads ({bases / 1e6:.0f} Mbase) in {dt:.1f}s, winnowmap -t {cores}, mapping phase only"},
                      "e2e": {"value": val, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--reads", type=int, default=int(os.environ.get("WM_BENCH_READS", 1000)))
    ap.add_argument("--cpu-reads", type=int, default=int(os.environ.get("WM_BENCH_CPU_READS", 8000)), help="reads of the cpu_baseline / parity sample")
    ap.add_argument("--cpu-reads-per-step", type=int, default=int(os.environ.get("WM_BENCH_CPU_READS_PER_STEP", 500)),
                    help="--impl reference: reads per step (a bounded sample of the step)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of the timed pass's last step to DIR/<name>.npy (float64)")
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    cores = os.cpu_count() or 1
    refbin = os.path.join(ROOT, "oracle", "_ref", "winnowmap")

    if a.impl == "reference":
        if rank == 0:
            reference_arm(a, cores, refbin)
        return

    # ---- inputs first (forked generators must not inherit a CUDA context) ----
    t0 = time.time()
    ref, wf = load_workload(rank)
    seed0 = 2_005_000 + 100_000 * rank  # seeds 2000 + cfg, per rank and step
    steps = gen_steps(a.warmup + a.steps, a.reads, seed0)
    warm = [r for s in steps[:a.warmup] for r in s]
    timed = [r for s in steps[a.warmup:] for r in s]
    log(f"rank {rank}: workload + {len(warm) + len(timed)} reads ready in {time.time() - t0:.1f}s")

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from winnowmap_b200 import lib
    from winnowmap_b200.mapper import MapOpt, Mapper
    L = lib()
    L.wm_prof_get.argtypes = [C.POINTER(C.c_double)]
    L.wm_prof_get_copies.argtypes = [C.POINTER(C.c_double)]
    L.wm_gpu_map_batch.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int]
    L.wm_format_batch.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_int32),
                                  C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.c_char_p]
    L.wm_bench_upload.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.POINTER(C.c_int32)]
    L.wm_bench_map_resident.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.wm_bench_write.argtypes = [C.c_void_p, C.POINTER(MapOpt), C.c_int, C.c_char_p]
    L.wm_free_regs.argtypes = [C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]

    t0 = time.time()
    # one worker per physical core at N=1; with several ranks per node the ranks share the node's hardware threads
    n_thr = max(1, min(int(os.environ.get("WM_HOST_THREADS", 64)), (cores // 2) // max(1, world)))
    if "WM_THREADS_PER_RANK" in os.environ:
        n_thr = max(1, int(os.environ["WM_THREADS_PER_RANK"]))
    if world == 1:
        mp = Mapper(ref, wf, preset="map-ont", cigar=True, device=local, n_threads=n_thr)
    else:
        # one-time index fan-out: rank 0 builds, one NCCL broadcast (GPU to GPU over NVLink), the others adopt the blob
        from winnowmap_b200 import multi
        import torch
        if rank == 0:
            mp = Mapper(ref, wf, preset="map-ont", cigar=True, device=local, n_threads=n_thr)
            blob = mp.index_blob()
        else:
            blob = None
        tb = time.time()
        blob = multi.broadcast_blob(blob, 0, rank, device=torch.device("cuda", local))
        if rank != 0:
            mp = Mapper(None, None, preset="map-ont", cigar=True, device=local, n_threads=n_thr, blob=blob)
        log(f"rank {rank}: index blob {blob.nbytes / 1e6:.0f} MB broadcast+adopted in {time.time() - tb:.2f}s")
        del blob
    t_index = time.time() - t0
    log(f"rank {rank}: index ready in {t_index:.1f}s ({mp.stats()['n_keys']:.0f} keys, {mp.stats()['n_pos']:.0f} positions)")

    def pack(recs):
        n = len(recs)
        names = (C.c_char_p * n)(*[nm.encode() for nm, _ in recs])
        seqs = (C.c_char_p * n)(*[s for _, s in recs])
        lens = (C.c_int32 * n)(*[len(s) for _, s in recs])
        return n, names, seqs, lens

    group_reads = max(GROUP * a.reads, 1)

    def map_host(recs, keep_first=0, out_path=None):
        """recs through wm_gpu_map_batch in groups of GROUP steps; wall time of the calls; optionally formats the first keep_first reads."""
        dt, d2h = 0.0, 0
        for g0 in range(0, len(recs), group_reads):
            sub = recs[g0:g0 + group_reads]
            n, names, seqs, lens = pack(sub)
            n_reg = (C.c_int32 * n)(); regs = (C.c_void_p * n)(); rl = (C.c_int32 * n)(); fg = (C.c_int32 * n)()
            t = time.perf_counter()
            L.wm_gpu_map_batch(mp.ctx, C.byref(mp.mo), n, names, seqs, lens, n_reg, regs, rl, fg, n_thr)
            L.wm_device_synchronize()
            dt += time.perf_counter() - t
            if g0 == 0 and keep_first > 0 and out_path:
                m = min(keep_first, n)
                L.wm_format_batch(mp.ctx, C.byref(mp.mo), m, names, seqs, lens, n_reg, regs, rl, out_path.encode())
            d2h += sum(n_reg) * 80
            L.wm_free_regs(n, n_reg, regs)
        return dt, d2h

    def upload(recs):
        n, names, seqs, lens = pack(recs)
        L.wm_bench_upload(mp.ctx, n, names, seqs, lens)  # raw reads -> one HBM pool (not timed)
        L.wm_device_synchronize()

    def map_uploaded():
        ms = C.c_double()
        L.wm_bench_map_resident(mp.ctx, C.byref(mp.mo), n_thr, group_reads, C.byref(ms))  # CUDA events bracketing the whole pass
        return ms.value / 1e3

    def barrier():
        L.wm_device_synchronize()
        if dist is not None:
            dist.barrier()

    # warm-up in the shape of the timed passes: the W steps, device-resident and through the host API.  Every orchestration
    # lane must have sized its workspaces for a full chunk before the timed region, so when W steps hold fewer than about
    # one chunk per lane the same W steps are submitted several times over in one submission (no extra reads are made).
    if warm:
        lanes = int(os.environ.get("WM_LANES", max(2, min(8, n_thr))))
        warm_bases = sum(len(s) for _, s in warm)
        n_rep = max(1, -(-int(1.25 * lanes * int(os.environ["WM_CHUNK_BASES"])) // max(1, warm_bases)))
        warm_sub = warm * n_rep
        upload(warm_sub)
        map_uploaded()
        map_host(warm_sub)
        del warm_sub
    L.wm_prof_enable(1); L.wm_prof_reset()
    L.wm_dump_timers() if os.environ.get("WM_TIMING") else None
    mp.reset_stats() if hasattr(mp, "reset_stats") else None
    phys, uuid = local, None  # NVML numbers the physical devices: honour CUDA_VISIBLE_DEVICES
    vis = [x.strip() for x in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if x.strip()]
    if local < len(vis):
        if vis[local].isdigit():
            phys = int(vis[local])
        elif vis[local].startswith("GPU-"):
            uuid = vis[local]
    bases = sum(len(s) for _, s in timed)
    upload(timed)
    sampler = ClockSampler(phys, uuid); sampler.start()
    barrier()
    t_steps = map_uploaded()
    barrier()
    clocks = sampler.result()
    if os.environ.get("WM_BENCH_VALUE_TWICE"):  # tuning aid: the same resident pass once more (not reported in the JSON line)
        t2 = map_uploaded()
        log(f"resident pass again: {bases / t2 / 1e6:.1f} Mbase/s (first: {bases / t_steps / 1e6:.1f})")
    if os.environ.get("WM_TIMING"):
        log(f"timers over {a.steps} timed steps:")
        L.wm_dump_timers()
    prof = (C.c_double * 13)(); L.wm_prof_get(prof)
    L.wm_prof_enable(0)
    st = mp.stats()
    tmpd = tempfile.mkdtemp(prefix="wm_bench_")
    n_par = min(a.cpu_reads, len(timed))
    paf_res, paf_host = os.path.join(tmpd, "resident.paf"), os.path.join(tmpd, "host.paf")
    L.wm_bench_write(mp.ctx, C.byref(mp.mo), n_par, paf_res.encode())  # the records of the timed pass itself
    # end to end through the host-buffer API: the same K steps, host buffers in, alignment records out
    L.wm_prof_reset()  # zeroes the library's host<->device byte counters
    barrier()
    e2e_t, d2h_b = map_host(timed, n_par, paf_host)
    barrier()
    cp = (C.c_double * 2)(); L.wm_prof_get_copies(cp)
    mem = (C.c_double * 2)()
    L.wm_device_mem.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.wm_device_mem(mem, C.cast(C.addressof(mem) + 8, C.POINTER(C.c_double)))
    hbm_used_gb = (mem[1] - mem[0]) / 1e9  # the pools are never trimmed while mapping: the footprint's high-water mark
    h2d_step, d2h_step = int(cp[0] / a.steps), int(cp[1] / a.steps)
    e2e_b = bases
    if dist is not None:
        import torch
        t = torch.tensor([t_steps, e2e_t], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        b = torch.tensor([float(bases), float(e2e_b)], device="cuda"); dist.all_reduce(b, op=dist.ReduceOp.SUM)
        t_steps, e2e_t = t.tolist(); bases, e2e_b = b.tolist()
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if a.dump_outputs:
        dump_outputs(L, mp.ctx, timed[len(timed) - a.reads:], len(timed) - a.reads, a.dump_outputs)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)

    def roof(kind):
        ms_sum, ms_uni, n_l, alg, units, units2 = [prof[1 + 6 * kind + i] for i in range(6)]
        k_ms = ms_uni if ms_uni > 0 else ms_sum
        ach = alg / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
        r = {"bound": "hbm", "kernel": ["wm_extd2_fill_kernel", "wm_chain_fill_kernel"][kind], "achieved": ach, "peak": peak, "unit": "GB/s",
             "frac": ach / peak, "traffic": None, "of": "measured" if peaks else "fallback", "launches": int(n_l), "kernel_ms": k_ms,
             "kernel_ms_sum_over_launches": ms_sum, "algorithmic_bytes": alg}
        if kind == 0:
            # the contract's `bound` is "hbm" | "tensor"; this kernel is neither: alone on the GPU it is integer-issue bound
            r["limiter"] = ("integer ALU issue, not HBM: ncu --set full of the kernel alone shows ALU pipe 66 %, issue slots 68 %, DRAM 6 % of "
                            "peak at 333 G cells/s (profiles/r02_ncu_wm_extd2_fill_kernel_summary.txt); in the bench its launches share the SMs "
                            "with the other lanes' kernels")
            # DRAM traffic: one ncu --set full capture of this kernel (profiles/r02_ncu_wm_extd2_fill_kernel_summary.txt) moved 16.8 GB for a
            # launch of 14.1 GB algorithmic bytes; that ratio applied to this run's average launch
            # (kept out of `traffic`, which stays null: it is a property of that capture, not a measurement of this run)
            r["traffic_per_algorithmic_byte_ncu"] = 1.19
            r.update({"block_cells": units, "jobs": int(units2), "block_cells_per_s": units / (k_ms * 1e-3) if k_ms > 0 else 0.0})
        else:
            r.update({"anchors": units, "anchors_per_s": units / (k_ms * 1e-3) if k_ms > 0 else 0.0})
        return r
    r_fill, r_chain = roof(0), roof(1)
    dom, other = (r_fill, r_chain) if r_fill["kernel_ms"] >= r_chain["kernel_ms"] else (r_chain, r_fill)

    cpu, parity, parity_note = None, False, ""
    try:  # the reference beside it (N = 1 only), bounded sample, all host threads; its output is the parity oracle
        if world > 1:
            raise RuntimeError("reported by the N=1 run only")
        if os.environ.get("WM_BENCH_NO_CPU"):
            raise RuntimeError("WM_BENCH_NO_CPU set (profiling run)")
        sample = (timed + warm)[:a.cpu_reads]
        fa = os.path.join(tmpd, "cpu.fa"); write_reads(fa, sample)
        ref_paf = os.path.join(tmpd, "ref.paf")
        t_idx, stamps = run_reference(refbin, ref, wf, fa, cores, ref_paf)
        dt = stamps[-1][0] - t_idx
        nb = sum(len(s) for _, s in sample)
        cpu = {"value": nb / dt, "unit": "bases/s", "cores": cores, "kind": "reference",
               "sample": f"{len(sample)} reads ({nb / 1e6:.1f} Mbase) of the timed + warm-up steps in {dt:.1f}s, winnowmap -t {cores}, mapping phase only "
                         f"(index build {t_idx:.0f}s excluded)"}
        want = paf_by_read(ref_paf)
        names = [nm.encode() for nm, _ in timed[:n_par]]
        bad = 0
        for got_path in (paf_res, paf_host):
            got = paf_by_read(got_path)
            bad += sum(1 for nm in names if got.get(nm, []) != want.get(nm, []))
        parity = bad == 0 and n_par > 0
        parity_note = f"{n_par} reads x 2 passes (resident, host-buffer) vs oracle/_ref/winnowmap: {bad} reads differ"
    except Exception as e:  # noqa: BLE001
        if cpu is None:
            cpu = {"value": None, "unit": "bases/s", "cores": cores, "kind": "reference", "sample": f"unavailable: {e}"}
        parity_note = parity_note or f"not checked: {e}"
    try:
        import shutil
        shutil.rmtree(tmpd, ignore_errors=True)
    except Exception:
        pass
    print(json.dumps({
        "metric": "mapped bases/sec", "value": bases / t_steps, "unit": "bases/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * t_steps / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
        "config": {"workload": workload_name() + f"; {a.reads} fresh reads per step per GPU, working set >> L2", "reads_per_step": a.reads,
                   "host_threads": n_thr, "lanes": int(os.environ.get("WM_LANES", max(2, min(8, n_thr)))),
                   "chunk_bases": int(os.environ["WM_CHUNK_BASES"]), "steps_per_submission": GROUP, "index_build_s": t_index,
                   "hbm_used_gb": round(hbm_used_gb, 1)},
        "e2e": {"value": e2e_b / e2e_t, "unit": "bases/s", "h2d_bytes_per_step": h2d_step, "d2h_bytes_per_step": d2h_step},
        "gpu_launches": int(prof[0]),
        "roofline": dom, "roofline_other": other,
        "cpu_baseline": cpu, "parity_checked": parity, "parity": parity_note, "clocks": clocks,
        "breakdown_s": {"seed_chain": st["t_seed"], "dp_rounds": st["t_dp"], "host_glue": st["t_host"]},
    }))


if __name__ == "__main__":
    main()
