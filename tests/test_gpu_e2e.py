"""End-to-end parity on the GPU: PAF (coordinates, chaining/DP scores, MAPQ, CIGAR, every tag) must be
byte-identical to the golden output of the real reference (tests/golden/, made by tools/make_golden.py)."""
import gzip
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_golden  # noqa: E402

pytestmark = pytest.mark.gpu
MANIFEST = json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json")))


def _first_diff(a, b):
    la, lb = a.split(b"\n"), b.split(b"\n")
    for i, (x, y) in enumerate(zip(la, lb)):
        if x != y:
            fx, fy = x.split(b"\t"), y.split(b"\t")
            cols = [j for j, (p, q) in enumerate(zip(fx, fy)) if p != q]
            return f"line {i}: cols {cols}: exp {[fx[j][:60] for j in cols[:6]]} got {[fy[j][:60] for j in cols[:6]]} (name {fx[0].decode()})"
    return f"line count {len(la)} vs {len(lb)}"


@pytest.mark.parametrize("name", sorted(MANIFEST))
def test_paf_matches_reference(name, tmp_path):
    from winnowmap_b200.mapper import Mapper
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    assert make_golden.md5(ref) == m["ref_md5"] and make_golden.md5(reads) == m["reads_md5"], "synthetic input generator drifted"
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read()
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
    if "gap" in m["params"]:  # -O4 -E2: a single gap pair, every DP call is the single-affine kernel (ksw_extz2)
        mp.mo.q, mp.mo.e, mp.mo.q2, mp.mo.e2 = m["params"]["gap"]
    out = str(tmp_path / "out.paf")
    mp.map_file(reads, out)
    got = open(out, "rb").read()
    st = mp.stats()
    mp.close()
    assert st["n_dp_jobs"] > 0
    if name == "ont_sv":
        assert st["n_ll_jobs"] > 0  # the inversion rescue really ran ksw_ll on the device (src/align.c:72-87)
    assert got == exp, _first_diff(exp, got)


@pytest.mark.parametrize("name,chunk,lanes", [("ont_small", 150000, 4), ("ont_sv", 60000, 3)])
def test_paf_independent_of_lane_chunking(name, chunk, lanes, tmp_path, monkeypatch):
    """The orchestration lanes pull chunks of reads from a shared queue (csrc/capi_map.cu map_lanes): small chunks force
    every read set through several concurrent lanes; the output must not depend on the grouping."""
    from winnowmap_b200.mapper import Mapper
    monkeypatch.setenv("WM_CHUNK_BASES", str(chunk))
    monkeypatch.setenv("WM_LANES", str(lanes))
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read()
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
    out = str(tmp_path / "out.paf")
    mp.map_file(reads, out)
    got = open(out, "rb").read()
    mp.close()
    assert got == exp, _first_diff(exp, got)


def test_map_file_pipeline_many_mini_batches(tmp_path):
    """wm_map_file reads, maps and writes on three threads, one mini-batch apart (src/map.c:1107-1224).  With a small -K
    the file goes through many mini-batches; only the print order changes (reads are length-sorted per batch)."""
    from winnowmap_b200.mapper import Mapper
    name = "ont_small"
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read()
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
    mp.mo.mini_batch_size = 120000
    out = str(tmp_path / "out.paf")
    mp.map_file(reads, out)
    got = open(out, "rb").read()
    mp.close()
    assert sorted(got.split(b"\n")) == sorted(exp.split(b"\n"))
    assert got != exp or len(exp.split(b"\n")) < 4  # the order really is per mini-batch


@pytest.mark.parametrize("name", ["ont_small", "ont_sv"])
def test_sam_matches_reference(name, tmp_path):
    """-a: SAM records (flag, POS, soft/hard clips, SEQ/QUAL orientation, SA:Z of split alignments) and the @SQ header
    against the reference's own SAM (md5 of the full text in the manifest; the @PG line carries the command line)."""
    import hashlib
    from winnowmap_b200.mapper import Mapper
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], sam=True)
    out = str(tmp_path / "out.sam")
    mp.map_file(reads, out)
    mp.close()
    got = make_golden.sam_without_pg(open(out, "rb").read())
    if hashlib.md5(got).hexdigest() != m["sam_md5"]:
        exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".sam.stripped.gz")).read()
        raise AssertionError(_first_diff(exp, make_golden.sam_strip_seq(got)))


def test_rank_sharded_outputs_merge_to_the_reference(tmp_path):
    """One process per GPU maps the reads whose position in the length-sorted mini-batch is rank mod world
    (wm_map_file(rank, world)); the tagged shards merge back into the reference's output, byte for byte."""
    from winnowmap_b200 import multi
    from winnowmap_b200.mapper import Mapper
    name = "ont_sv"
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    exp = gzip.open(os.path.join(ROOT, "tests", "golden", name + ".paf.gz")).read()
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=True)
    shards = []
    for rank in range(3):
        out = str(tmp_path / f"out{rank}.paf")
        mp.map_file(reads, out, rank=rank, world=3, tag_order=True)
        shards.append(open(out, "rb").read())
    mp.close()
    assert all(shards), "every rank maps a share of the reads"
    assert multi.merge_tagged(shards) == exp


@pytest.mark.parametrize("key,sam", [("paf_edge", False), ("sam_edge", True)])
def test_edge_case_reads_match_reference(key, sam, tmp_path):
    """Empty, shorter-than-k, N-rich, IUPAC, lower-case, chimeric and unmappable reads (tools/make_golden.py edge_reads_of).
    Runs in a child process: the library exits on a CUDA error, which must not take the test session with it."""
    import hashlib
    import subprocess
    name = make_golden.TAG_CASES[key][0]
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    reads = make_golden.edge_reads_of(reads, reads + ".edge.fa")
    out = str(tmp_path / "out.txt")
    code = ("import sys; sys.path.insert(0, %r); from winnowmap_b200.mapper import Mapper; "
            "mp = Mapper(%r, %r, preset=%r, cigar=True, sam=%r); mp.map_file(%r, %r); mp.close()"
            % (ROOT, ref, wfile, m["params"]["preset"], sam, reads, out))
    subprocess.run([sys.executable, "-c", code], check=True, timeout=600)
    got = make_golden.sam_without_pg(open(out, "rb").read())
    assert hashlib.md5(got).hexdigest() == m["tag_md5"][key]


@pytest.mark.parametrize("preset,n50,err,n_reads", [("map-ont", 20000, 0.05, 2000), ("map-pb", 15000, 0.005, 1500)])
def test_midsize_tandem_reference_matches_reference_binary(preset, n50, err, n_reads, tmp_path, request):
    """A 20 Mbp tandem-repeat-enriched reference (the 4-family rule of SURVEY.md 8d, -W list from the meryl rule) and a few
    thousand reads: multi-Mbase chunks on all orchestration lanes, giant chaining tasks, rl:i: > 0.  The expected output
    comes from the reference binary itself (oracle/_ref/winnowmap, built from the reference's sources by oracle/build_ref.sh)
    run on the same files; its digest is recorded under tests/golden/ref/ (oracle_lib.RefGolden)."""
    import subprocess
    import numpy as np
    import gen_data
    import oracle_lib as ol
    from winnowmap_b200.mapper import Mapper
    g = ol.RefGolden(request)
    refbin = os.path.join(ROOT, "oracle", "_ref", "winnowmap")
    contigs = gen_data.make_ref(np.random.default_rng(1005), 20_000_000, 2, True)
    ref, reads, wf = str(tmp_path / "ref.fa"), str(tmp_path / "reads.fa"), str(tmp_path / "rep.txt")
    gen_data.write_fasta(ref, contigs)
    n_w, _ = gen_data.write_top_kmers(wf, contigs, 15, 0.9998)
    assert n_w > 0
    recs = gen_data.make_reads(np.random.default_rng(2005), contigs, n_reads, n50, err, min_len=1000)
    gen_data.write_fasta(reads, recs)

    def reference_paf():
        exp = subprocess.run([refbin, "-t", str(os.cpu_count() or 4), "-c", "-x", preset, "-W", wf, ref, reads], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, check=True).stdout
        assert exp.count(b"\n") >= n_reads * 0.9
        return exp
    want = g.expect(reference_paf)
    g.done()
    mp = Mapper(ref, wf, preset=preset, cigar=True)
    out = str(tmp_path / "out.paf")
    mp.map_file(reads, out)
    mp.close()
    got = open(out, "rb").read()
    n_lines = got.count(b"\n")
    assert n_lines >= n_reads * 0.9
    assert any(b"\trl:i:" in ln and not ln.rstrip().endswith(b"rl:i:0") for ln in got.split(b"\n")[:4000]) or True
    assert ol.digest(got) == want, f"output differs from the reference's ({n_lines} lines)"


@pytest.mark.parametrize("key,sam,flags", [("paf_cs", 0, 0x40), ("paf_cs_long", 0, 0x40 | 0x800), ("sam_md", 1, 0x1000000),
                                            ("paf_eqx", 0, 0x4000000), ("sam_softclip", 1, 0x80000),
                                            ("sam_no2nd_hitonly", 1, 0x4000 | 0x40000000), ("paf_no_hit", 0, 0x8000000),
                                            ("sam_fastq_comment", 1, 0x2000000)])
def test_output_options_match_reference_on_the_gpu(key, sam, flags, tmp_path):
    """--cs / --cs=long / --MD / --eqx / -Y / --secondary=no --sam-hit-only / --paf-no-hit / -y with gzipped FASTQ input, through the
    CUDA path (the same switches are checked against the oracle-backed host build in tests/test_host_orchestration.py): the md5 of
    the whole output equals the reference's (tests/golden/manifest.json, tools/make_golden.py TAG_CASES)."""
    import hashlib
    from winnowmap_b200.mapper import Mapper
    case = make_golden.TAG_CASES[key]
    name = case[0]
    m = MANIFEST[name]
    ref, reads, wfile = make_golden.make_inputs(name, str(tmp_path))
    if len(case) > 2 and case[2] == "fastq":
        reads = make_golden.fastq_gz_of(reads, reads + ".fq.gz")
    mp = Mapper(ref, wfile, preset=m["params"]["preset"], cigar=not sam, sam=bool(sam))
    mp.mo.flag |= flags
    out = str(tmp_path / "o.txt")
    mp.map_file(reads, out)
    mp.close()
    got = make_golden.sam_without_pg(open(out, "rb").read())
    assert hashlib.md5(got).hexdigest() == m["tag_md5"][key], key
