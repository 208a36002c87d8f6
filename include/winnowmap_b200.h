/*
 * winnowmap_b200.h -- C ABI of the B200-native seed-chain-align path of Winnowmap v2.03.
 *
 * Plain pointers and sizes only (no torch / CUDA types).  Every entry point cites the
 * reference interface it replaces (paths relative to the reference repository root).
 * All functions return 0 on success; on a CUDA failure they print a message to stderr
 * and exit(1), mirroring the reference's fatal-error convention (src/misc.c:123-151).
 * There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef WINNOWMAP_B200_H
#define WINNOWMAP_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- flags, identical values to src/ksw2.h:8-17 ---- */
#define WM_KSW_EZ_SCORE_ONLY  0x01
#define WM_KSW_EZ_RIGHT       0x02
#define WM_KSW_EZ_GENERIC_SC  0x04
#define WM_KSW_EZ_APPROX_MAX  0x08
#define WM_KSW_EZ_APPROX_DROP 0x10
#define WM_KSW_EZ_EXTZ_ONLY   0x40
#define WM_KSW_EZ_REV_CIGAR   0x80
#define WM_KSW_NEG_INF (-0x40000000)

/* (x,y) pair, same layout as mm128_t (src/minimap.h:55) */
typedef struct { uint64_t x, y; } wm128_t;

/* result of one extension DP; same fields as ksw_extz_t (src/ksw2.h:23-32) without the
 * heap pointer: the CIGAR of task i lives at cigar[cigar_off[i] .. +n_cigar) */
typedef struct {
	int32_t max, zdropped;
	int32_t max_q, max_t;
	int32_t mqe, mqe_t;
	int32_t mte, mte_q;
	int32_t score;
	int32_t reach_end;
	int32_t n_cigar;
	int32_t reserved;
} wm_extz_t;

/* library / device */
const char *wm_version(void);
int wm_device_count(void);                 /* number of visible CUDA devices (0 if none) */
int wm_set_device(int device);

/* ------------------------------------------------------------------------------------
 * Kernel-level batch entry points (used by the parity tests and by bench.py to time one
 * stage in isolation).  Host buffers in, host buffers out.
 * ---------------------------------------------------------------------------------- */

/* Batched ksw_extd2_sse (src/ksw2_extd2_sse.c:26; prototype src/ksw2.h:60-61), m = 5,
 * scoring matrix `mat` (25 entries, src/align.c:9-22).  Sequences are 0..4 codes.
 * qoff/toff: n+1 offsets into qseq/tseq.  w/zdrop/end_bonus/flag: per task.
 * cigar_off: n+1 offsets (capacity per task); a task whose CIGAR does not fit reports the
 * needed length in n_cigar and writes nothing beyond its capacity. */
int wm_ksw_extd2_batch(int n, const uint8_t *qseq, const int64_t *qoff, const uint8_t *tseq, const int64_t *toff,
                       const int8_t *mat, int q, int e, int q2, int e2,
                       const int32_t *w, const int32_t *zdrop, const int32_t *end_bonus, const int32_t *flag,
                       wm_extz_t *ez, uint32_t *cigar, const int64_t *cigar_off);

/* Batched ksw_exts2_sse (src/ksw2_exts2_sse.c:26; prototype src/ksw2.h:63-64), the splice-aware extension mm_align_pair
 * calls when MM_F_SPLICE is set (src/align.c:326-327): m = 5, no band, no end bonus.  flag: the KSW_EZ_* bits of
 * src/ksw2.h:7-17, including SPLICE_FOR 0x100 / SPLICE_REV 0x200 / SPLICE_FLANK 0x400.  junc: one annotation byte per
 * target base (mm_idx_bed_junc, src/index.c:780), same offsets as tseq, or NULL.  The kernel is complete and parity-
 * tested; the mapper itself still refuses -x splice (the splice branches of mm_align1 are not built). */
int wm_ksw_exts2_batch(int n, const uint8_t *qseq, const int64_t *qoff, const uint8_t *tseq, const int64_t *toff, const uint8_t *junc,
                       const int8_t *mat, int q, int e, int q2, int noncan, int junc_bonus,
                       const int32_t *zdrop, const int32_t *flag, wm_extz_t *ez, uint32_t *cigar, const int64_t *cigar_off);

/* Batched ksw_ll_qinit + ksw_ll_i16 (src/ksw2_ll_sse.c:32,80): score, query end, target end. */
int wm_ksw_ll_batch(int n, const uint8_t *qseq, const int64_t *qoff, const uint8_t *tseq, const int64_t *toff,
                    const int8_t *mat, int gapo, int gape, int32_t *score, int32_t *qe, int32_t *te);

/* Down-weighted k-mer filter: replaces the bloom_filter built in mm_idx_gen
 * (src/index.c:404-432; ext/bloom/bloom_filter.hpp).  `canon_kmers` are the values of
 * encodeKmer() (src/index.c:362-376) for each line of the -W file. */
typedef struct wm_bloom_s wm_bloom_t;
wm_bloom_t *wm_bloom_build(const uint64_t *canon_kmers, int64_t n);
uint64_t wm_bloom_bits(const wm_bloom_t *b);
const uint8_t *wm_bloom_table(const wm_bloom_t *b);
void wm_bloom_destroy(wm_bloom_t *b);

/* Batched mm_sketch (src/sketch.c:128; prototype src/mmpriv.h:57), is_hpc = 0.
 * seq: concatenated ASCII sequences, off: n+1 offsets, rid: per sequence.
 * Output: minimizers of sequence i at out[out_off[i] .. out_off[i+1]); *out / *out_off are
 * malloc()ed by the callee and owned by the caller (free()). */
int wm_sketch_batch(const wm_bloom_t *bloom, int n, const char *seq, const int64_t *off, const uint32_t *rid,
                    int w, int k, wm128_t **out, int64_t **out_off);

/* radix_sort_128x (src/misc.c:156; src/ksort.h:116-151) on n_arr independent arrays:
 * array i is a[off[i] .. off[i+1]); sorted in place with the reference's tie order. */
int wm_radix_sort_128x_batch(int n_arr, wm128_t *a, const int64_t *off);
/* The same, also returning in *ms the device time of the sort alone (CUDA events; the copies are left out). */
int wm_radix_sort_128x_batch_timed(int n_arr, wm128_t *a, const int64_t *off, float *ms);

/* Batched mm_chain_dp (src/chain.c:22; prototype src/mmpriv.h:67) for n_segs = 1,
 * is_cdna = 0.  Anchors of task i: a[off[i] .. off[i+1]) (sorted as by collect_seed_hits).
 * Outputs: n_u[i]; u at u[off[i] .. +n_u[i]); chained anchors at b[off[i] .. +n_b[i]). */
int wm_chain_dp_batch(int n_tasks, const wm128_t *a, const int64_t *off,
                      int max_dist_x, int min_dist_x, int max_dist_y, int bw, int max_skip, int max_iter,
                      int min_cnt, int min_sc, float gap_scale,
                      int32_t *n_u, uint64_t *u, wm128_t *b, int64_t *n_b);

/* ------------------------------------------------------------------------------------
 * Drop-in boundary: what the reference's batch driver binds (INTEGRATION.md).
 * ---------------------------------------------------------------------------------- */

/* Flattened view of an mm_idx_t (src/minimap.h:66-77, src/index.c:33-38): the caller walks
 * its buckets once and hands over plain arrays.  keys[i] (minimizer hash, i.e. mm128_t.x>>8)
 * owns the occurrence list pos[pos_off[i] .. pos_off[i+1]) sorted ascending exactly as
 * mm_idx_get() (src/index.c:88-105) would return it. */
typedef struct {
	int32_t k, w, n_seq;
	const char *const *seq_name;   /* n_seq names (mm_idx_seq_t.name) */
	const uint32_t *seq_len;       /* mm_idx_seq_t.len */
	const uint64_t *seq_offset;    /* mm_idx_seq_t.offset into S */
	const uint32_t *S;             /* 4-bit packed reference (mm_idx_t.S) */
	uint64_t S_words;              /* number of uint32 words in S */
	int64_t n_keys;
	const uint64_t *keys;
	const uint64_t *pos_off;       /* n_keys + 1 */
	const uint64_t *pos;
	uint64_t bloom_bits;           /* bloom_filter::size() */
	const uint8_t *bloom_table;    /* bloom_filter::table() */
} wm_idx_view_t;


/* ---- structs that cross the boundary: field-for-field the reference's public structs ---- */
#ifndef __cplusplus
#include <stdbool.h>
#endif
typedef struct { /* mm_extra_t, src/minimap.h:80-86 */
	uint32_t capacity;
	int32_t dp_score, dp_max, dp_max2;
	uint32_t n_ambi:30, trans_strand:2;
	uint32_t n_cigar;
	uint32_t cigar[];
} wm_extra_t;

typedef struct { /* mm_reg1_t, src/minimap.h:88-103 */
	int32_t id, cnt, rid, score;
	int32_t qs, qe, rs, re;
	int32_t parent, subsc;
	int32_t as;
	int32_t mlen, blen;
	int32_t n_sub;
	int32_t score0;
	uint32_t mapq:8, split:2, rev:1, inv:1, sam_pri:1, proper_frag:1, pe_thru:1, seg_split:1, seg_id:8, split_inv:1, is_alt:1, dummy:6;
	uint32_t hash;
	float div;
	wm_extra_t *p;
} wm_reg1_t;

typedef struct { /* mm_idxopt_t, src/minimap.h:106-110 */
	short k, w, flag, bucket_bits;
	int mini_batch_size;
	uint64_t batch_size;
} wm_idxopt_t;

typedef struct { /* mm_mapopt_t, src/minimap.h:112-176 */
	int64_t flag;
	int seed;
	int sdust_thres;
	int max_qlen;
	int bw;
	int max_gap, max_gap_ref;
	int min_gap_ref;
	int max_frag_len;
	int max_chain_skip, max_chain_iter;
	int min_cnt;
	int min_chain_score;
	float chain_gap_scale;
	bool SVaware;
	int SVawareMinReadLength;
	int suffixSampleOffset;
	int min_mapq;
	float min_qcov;
	int minPrefixLength;
	int maxPrefixLength;
	float prefixIncrementFactor;
	int stage2_bw;
	int stage2_zdrop_inv;
	int stage2_max_gap;
	int stage2_extension_inc;
	float mask_level;
	int mask_len;
	float pri_ratio;
	int best_n;
	int max_join_long, max_join_short;
	int min_join_flank_sc;
	float min_join_flank_ratio;
	float alt_drop;
	int a, b, q, e, q2, e2;
	int sc_ambi;
	int noncan;
	int junc_bonus;
	int zdrop, zdrop_inv;
	int end_bonus;
	int min_dp_max;
	int min_ksw_len;
	int anchor_ext_len, anchor_ext_shift;
	float max_clip_ratio;
	int pe_ori, pe_bonus;
	float mid_occ_frac;
	int32_t min_mid_occ;
	int32_t mid_occ;
	int32_t max_occ;
	int mini_batch_size;
	int64_t max_sw_mat;
	const char *kmer_freq_filename;
	const char *split_prefix;
} wm_mapopt_t;


/* mm_set_opt / mm_check_opt (src/options.c:89,133): same presets, same return codes */
int wm_set_opt(const char *preset, wm_idxopt_t *io, wm_mapopt_t *mo);
int wm_check_opt(const wm_idxopt_t *io, const wm_mapopt_t *mo);
int wm_sizeof_mapopt(void);
int wm_sizeof_reg1(void);
/* sizeof(wm_mapopt_t / wm_reg1_t / wm_extra_t / wm_idxopt_t) followed by the offset of every addressable field, in
 * declaration order: a reference-side binding (and tests/test_abi_layout.py) compares it with the mm_* structs once at
 * start-up.  Returns the number of values (only the first `cap` are written). */
int wm_abi_layout(int64_t *out, int cap);

typedef struct wm_gpu_ctx_s wm_gpu_ctx;

/* Upload the flattened index to CUDA device `device` (one context per GPU: a multi-GPU front end runs one process per
 * device, or calls this once per device).  Returns NULL on an unsupported (k, w).  Call site in the reference: after
 * main.c:403 (INTEGRATION.md section 3 shows the bucket walk that fills the view). */
wm_gpu_ctx *wm_gpu_idx_upload(const wm_idx_view_t *idx, int device);
void wm_gpu_destroy(wm_gpu_ctx *ctx);

/* Index construction from FASTA (mm_idx_gen, src/index.c:378-449; reader loop main.c:384): the reference
 * sequences are sketched by the same CUDA kernel as the reads, the -W list goes into the down-weight filter. */
wm_gpu_ctx *wm_index_build(const char *ref_fn, const char *kmer_freq_fn, int k, int w, int device);

/* One-time index fan-out (SURVEY.md 8e): the flattened index as one relocatable blob.  Rank 0 builds it, it travels
 * GPU-to-GPU in a single NCCL broadcast, every other rank re-creates its context with wm_idx_blob_load. */
int64_t wm_idx_blob_size(const wm_gpu_ctx *ctx);
int wm_idx_blob_write(const wm_gpu_ctx *ctx, uint8_t *buf);
wm_gpu_ctx *wm_idx_blob_load(const uint8_t *buf, int64_t size, int device);

/* Replaces kt_for(p->n_threads, worker_for, in, n_frag) (src/map.c:1162-1165; worker_for :1008-1048): one call per
 * mini-batch, blocking; fills n_reg[i], reg[i] (malloc()ed array whose ->p are malloc()ed, freed by the caller as
 * at src/map.c:1210-1211), rep_len[i] and frag_gap[i] (src/map.c:1025-1034).  n_threads = host threads for the glue. */
int wm_gpu_map_batch(wm_gpu_ctx *ctx, const wm_mapopt_t *opt, int n_seq, const char *const *names, const char *const *seqs,
                     const int32_t *lens, int32_t *n_reg, wm_reg1_t **reg, int32_t *rep_len, int32_t *frag_gap, int n_threads);

/* mm_tbuf_init / mm_tbuf_destroy / mm_map (src/minimap.h:329-351, src/map.c:18-38, :976-984): one read through the same path
 * (internally a batch of one).  The returned array and every ->p are malloc()ed and freed by the caller, as with mm_map.
 * The buffer carries what mm_tbuf_s carries for the caller: rep_len and frag_gap of the last call. */
typedef struct wm_tbuf_s wm_tbuf_t;
wm_tbuf_t *wm_tbuf_init(void);
void wm_tbuf_destroy(wm_tbuf_t *b);
int wm_tbuf_rep_len(const wm_tbuf_t *b);
int wm_tbuf_frag_gap(const wm_tbuf_t *b);
wm_reg1_t *wm_map(wm_gpu_ctx *ctx, int l_seq, const char *seq, int *n_regs, wm_tbuf_t *b, const wm_mapopt_t *opt, const char *name);

/* mm_map_file (src/map.c:1273) into out_fn ("-" = stdout): PAF (mm_write_paf3, src/format.c:308), or SAM when
 * opt->flag has MM_F_OUT_SAM (mm_write_sam3, src/format.c:391, single-segment reads; header as mm_write_sam_hdr,
 * src/format.c:118, written by rank 0 when tag_order == 0).  rank/world shard the reads of every mini-batch
 * round-robin over processes (one process per GPU); tag_order prefixes "<batch>\t<pos>\t" for merging. */
int wm_map_file(wm_gpu_ctx *ctx, const wm_mapopt_t *opt, const char *reads_fn, const char *out_fn, int n_threads, int rank, int world,
                int tag_order, int64_t max_batch_bases);
/* the command line recorded in the @PG header line of SAM output (the reference prints its own argv, src/format.c:130-135) */
void wm_set_sam_cl(wm_gpu_ctx *ctx, const char *cl);
/* mm_gen_cs / mm_gen_MD (src/minimap.h:389-390): the cs / MD string of one hit of read `seq` (ASCII) into *buf, which is
 * realloc()ed when *max_len is too small; returns the length.  The reference sequence comes from the context's index. */
int wm_gen_cs(const wm_gpu_ctx *ctx, char **buf, int *max_len, const wm_reg1_t *r, const char *seq, int no_iden);
int wm_gen_MD(const wm_gpu_ctx *ctx, char **buf, int *max_len, const wm_reg1_t *r, const char *seq);
/* mm_idx_getseq (0..4 codes of [st,en) of sequence rid; src/index.c:161-171), mm_idx_name2id (:131-140, -1 if absent) and
 * the sequence table (mm_idx_t::n_seq / seq[].name / seq[].len, src/minimap.h:59-77) of the index held by the context */
int wm_idx_getseq(const wm_gpu_ctx *ctx, uint32_t rid, uint32_t st, uint32_t en, uint8_t *seq);
int wm_idx_name2id(const wm_gpu_ctx *ctx, const char *name);
int wm_idx_n_seq(const wm_gpu_ctx *ctx);
const char *wm_idx_seq_name(const wm_gpu_ctx *ctx, int rid);
uint32_t wm_idx_seq_len(const wm_gpu_ctx *ctx, int rid);

/* frees what wm_gpu_map_batch returned (the reference's output step does this itself, src/map.c:1210-1211) */
void wm_free_regs(int n, const int32_t *n_reg, wm_reg1_t **reg);
/* the records wm_gpu_map_batch returned, as PAF (or SAM when opt->flag has MM_F_OUT_SAM) lines in input order: the writer
 * wm_map_file uses, i.e. what the output step of the reference prints for these reads (src/map.c:1189-1206) */
int wm_format_batch(const wm_gpu_ctx *ctx, const wm_mapopt_t *opt, int n_seq, const char *const *names, const char *const *seqs, const int32_t *lens,
                    const int32_t *n_reg, wm_reg1_t *const *reg, const int32_t *rep_len, const char *out_fn);
/* bench: upload a batch (not timed), then map it with the reads resident in HBM; *ms = CUDA-event time of the pass.  The
 * reads are submitted group_reads at a time (<= 0: all at once).  The records of the pass stay in the context until the next pass; wm_bench_write formats those of the first n_first reads. */
int wm_bench_upload(wm_gpu_ctx *ctx, int n_seq, const char *const *names, const char *const *seqs, const int32_t *lens);
int wm_bench_map_resident(wm_gpu_ctx *ctx, const wm_mapopt_t *opt, int n_threads, int group_reads, double *ms);
int wm_bench_write(wm_gpu_ctx *ctx, const wm_mapopt_t *opt, int n_first, const char *out_fn);
/* bench: n_reg[i] and rep_len[i] of reads first .. first + n - 1 of the last resident pass, and their records in input order into
 * regs (at most cap of them; each ->p stays owned by the context until the next pass).  Returns the number of records. */
int64_t wm_bench_records(const wm_gpu_ctx *ctx, int first, int n, int32_t *n_reg, int32_t *rep_len, wm_reg1_t *regs, int64_t cap);

/* bench instrumentation (csrc/prof.cu): launch counter and CUDA-event timing of the two dominant kernel classes */
void wm_prof_enable(int on);
void wm_prof_reset(void);
/* out[0] = kernel launches; then six values per class (DP fill at out[1], chaining forward pass at out[7]): sum of launch
 * ms, ms during which at least one kernel of the class ran (launches of concurrent lanes overlap), launches, algorithmic
 * bytes (SURVEY.md 8d), units (block cells / anchors), DP jobs */
void wm_prof_get(double *out13);
void wm_prof_get_copies(double *out2); /* bytes copied host-to-device / device-to-host by the mapping path since wm_prof_reset */
int wm_device_synchronize(void);
int wm_device_mem(double *free_bytes, double *total_bytes); /* cudaMemGetInfo of the current device */
void wm_dump_timers(void); /* prints and resets the orchestration wall-clock accumulators (stderr) */

void wm_get_stats(wm_gpu_ctx *ctx, double *out, int n);
void wm_reset_stats(wm_gpu_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
