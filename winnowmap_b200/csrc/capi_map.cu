// C-ABI of the drop-in boundary (include/winnowmap_b200.h): index upload / construction, batch mapping
// (the replacement of kt_for(worker_for), reference src/map.c:1162-1165) and the file-level driver that mirrors
// mm_map_file (src/map.c:1244-1276) for PAF output.
#include <stddef.h>
#include <string.h>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "wm_common.cuh"
#include "sketch.cuh"
#include "index_dev.cuh"
#include "gpu_backend.h"
#include "host_io.h"
#include "host_index.h"
#include "host_timers.h"

using namespace wmh;


struct wm_gpu_ctx_s {
	wm_host_idx hidx;
	Backend *be;
	int device;
	MapStats stats;
	double t_index, t_map;
	int64_t n_keys, n_pos;
	std::vector<wm_read> resident; // bench: reads already uploaded by wm_bench_upload ...
	char *d_resident = 0;          // ... their bases, one device pool (wm_read::dev_off)
	std::vector<std::vector<wm_reg1_t>> res_regs; std::vector<int> res_rl; // records of the last wm_bench_map_resident pass (wm_bench_write)
	std::string sam_cl;            // command line recorded in the @PG line of SAM output (wm_set_sam_cl)
	std::vector<Backend*> lanes;   // lanes[0] == be; further lanes share the index and own a stream + workspaces
	// host copy of the flattened index, kept for the one-time fan-out to the other GPUs (wm_idx_blob_*)
	std::vector<uint64_t> keys, pos_off, pos;
	std::vector<uint8_t> bloom;
	uint64_t bloom_bits;
};

static void free_reg_vectors(std::vector<std::vector<wm_reg1_t>> &regs);
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static void require_device(const char *who)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
		fprintf(stderr, "[ERROR] %s: no CUDA device visible; winnowmap-b200 has no CPU fallback\n", who);
		exit(1);
	}
}

// Orchestration lanes: the reads of a call are cut into chunks that L lanes pull from a shared counter and run through
// map_batch concurrently, each lane on its own host thread and CUDA stream, so that one lane's host glue overlaps the
// other lanes' kernels.  Results do not depend on the grouping (reads never interact, src/map.c:1008-1048).
static int n_lanes_wanted(int n_threads)
{ // eight lanes unless WM_LANES says otherwise: a lane mostly waits for the GPU, so lanes pay even with one host thread each
  // (measured with 8 host threads on the tandem-repeat workload: 2 lanes 53, 8 lanes 69 Mbase/s)
	const char *e = getenv("WM_LANES");
	int n = e ? atoi(e) : 8;
	if (!e && n > n_threads) n = n_threads < 2 ? 2 : n_threads;
	return n < 1 ? 1 : n > 16 ? 16 : n;
}

static void ensure_lanes(wm_gpu_ctx_s *c, int n_threads)
{
	if (!c->lanes.empty()) return;
	const int L = n_lanes_wanted(n_threads);
	c->lanes.push_back(c->be);
	const size_t budget = gpu_backend_get_budget(c->be) / (size_t)L;
	for (int i = 1; i < L; ++i) c->lanes.push_back(gpu_backend_clone(c->be, L));
	for (int i = 0; i < L; ++i) { gpu_backend_set_budget(c->lanes[i], budget); c->lanes[i]->set_resident_pool(c->d_resident); }
}

static void map_lanes(wm_gpu_ctx_s *c, const wm_mapopt_t *opt, const std::vector<const wm_read*> &reads, std::vector<std::vector<wm_reg1_t>> &regs,
                      std::vector<int> &rl, std::vector<int> &fg, int n_threads, bool resident)
{
	(void)resident;
	ensure_lanes(c, n_threads);
	const int n = (int)reads.size();
	regs.assign(n, std::vector<wm_reg1_t>()); rl.assign(n, 0); fg.assign(n, 0);
	if (n == 0) return;
	// The reads are cut into chunks of about chunk_bases bases (in input order) that the lanes pull from a shared counter:
	// a lane that finishes early takes the next chunk, and lanes drift out of phase so that one lane's host glue
	// overlaps the other lanes' kernels.
	std::vector<int> cb(1, 0);
	{
		// large chunks amortise the per-wave latencies of a batch; two chunks per lane leave room for the lanes to drift apart
		const char *e = getenv("WM_CHUNK_BASES");
		int64_t total = 0, acc = 0;
		for (int i = 0; i < n; ++i) total += (int64_t)reads[i]->seq.size();
		int64_t chunk_bases = total / (2 * (int64_t)c->lanes.size()) + 1;
		if (chunk_bases < 4000000) chunk_bases = 4000000;
		if (chunk_bases > 32000000) chunk_bases = 32000000;
		if (e && atoll(e) > 0) chunk_bases = atoll(e);
		// whole rounds: the latency of a chunk grows much more slowly than its size (it is set by the serial giant tasks of
		// its waves), so a lone chunk left over after the last full round costs almost a whole round.  The chunk size is
		// therefore adjusted (up to +35 %) so that the chunks fill a whole number of rounds of the lanes.
		const int64_t n_lanes = (int64_t)c->lanes.size();
		int64_t rounds = (int64_t)((double)total / (double)(n_lanes * chunk_bases) + 0.35);
		if (rounds < 1) rounds = 1;
		if (total > n_lanes * chunk_bases * 13 / 20) chunk_bases = (total + n_lanes * rounds - 1) / (n_lanes * rounds);
		else if (total / n_lanes >= 2000000) chunk_bases = (total + n_lanes - 1) / n_lanes; // less than a round: one chunk per lane
		for (int i = 0; i < n; ++i) {
			acc += (int64_t)reads[i]->seq.size();
			if (acc >= chunk_bases || i == n - 1) { cb.push_back(i + 1); acc = 0; }
		}
	}
	const int n_chunks = (int)cb.size() - 1;
	int L = (int)c->lanes.size();
	if (L > n_chunks) L = n_chunks;
	if (L == 1 && n_chunks == 1) {
		map_batch(c->lanes[0], &c->hidx, opt, reads, regs, rl, fg, n_threads, &c->stats);
		wm_dbuf_async = false; // the caller's thread may go on to the one-shot kernel entry points, which allocate synchronously
		return;
	}
	std::vector<MapStats> st(L);
	std::vector<double> lane_end(L, 0.0);
	std::vector<std::thread> th;
	std::atomic<int> next(0);
	const int thr = n_threads / L > 0 ? n_threads / L : 1;
	for (int l = 0; l < L; ++l) {
		memset(&st[l], 0, sizeof(MapStats));
		th.emplace_back([&, l]() {
			for (;;) {
				const int j = next.fetch_add(1);
				if (j >= n_chunks) break;
				std::vector<const wm_read*> sub(reads.begin() + cb[j], reads.begin() + cb[j + 1]);
				std::vector<std::vector<wm_reg1_t>> r2; std::vector<int> rl2, fg2;
				const double tb0 = wmh::Timers::now();
				map_batch(c->lanes[l], &c->hidx, opt, sub, r2, rl2, fg2, thr, &st[l]);
				wmh::g_timers.add("lane.map_batch", wmh::Timers::now() - tb0);
				for (size_t k = 0; k < sub.size(); ++k) { const int i = cb[j] + (int)k; regs[i].swap(r2[k]); rl[i] = rl2[k]; fg[i] = fg2[k]; }
			}
			lane_end[l] = wmh::Timers::now();
		});
	}
	for (auto &t : th) t.join();
	{ // what the lanes that finished early waited for the last one (tuning aid)
		const double t_end = wmh::Timers::now();
		for (int l = 0; l < L; ++l) wmh::g_timers.add("lane.idle_tail", t_end - lane_end[l]);
	}
	for (int l = 0; l < L; ++l) {
		MapStats &a = c->stats; const MapStats &b = st[l];
		a.n_reads += b.n_reads, a.n_bases += b.n_bases, a.n_minimaps += b.n_minimaps, a.n_chained += b.n_chained, a.n_dp_jobs += b.n_dp_jobs;
		a.n_ll_jobs += b.n_ll_jobs, a.n_rounds += b.n_rounds, a.t_seed += b.t_seed, a.t_dp += b.t_dp, a.t_host += b.t_host;
	}
}

// the sketch kernels size their shared arrays for the reference's own limits (assert at src/sketch.c:140)
static bool kw_ok(const char *who, int k, int w)
{
	if (w > 0 && w < 256 && k > 0 && k <= 28) return true;
	fprintf(stderr, "[ERROR] %s: k = %d, w = %d outside the supported range (0 < w < 256, 0 < k <= 28; src/sketch.c:140)\n", who, k, w);
	return false;
}

extern "C" wm_gpu_ctx_s *wm_gpu_idx_upload(const wm_idx_view_t *v, int device)
{
	require_device("wm_gpu_idx_upload");
	if (!kw_ok("wm_gpu_idx_upload", v->k, v->w)) return 0;
	wm_gpu_ctx_s *c = new wm_gpu_ctx_s();
	memset(&c->stats, 0, sizeof(c->stats));
	c->device = device; c->t_index = c->t_map = 0;
	c->hidx.k = v->k, c->hidx.w = v->w;
	for (int i = 0; i < v->n_seq; ++i) {
		c->hidx.name.push_back(v->seq_name && v->seq_name[i] ? v->seq_name[i] : std::to_string(i));
		c->hidx.len.push_back(v->seq_len[i]);
		c->hidx.offset.push_back(v->seq_offset[i]);
	}
	c->hidx.S.assign(v->S, v->S + v->S_words);
	c->n_keys = v->n_keys, c->n_pos = (int64_t)v->pos_off[v->n_keys];
	c->keys.assign(v->keys, v->keys + v->n_keys);
	c->pos_off.assign(v->pos_off, v->pos_off + v->n_keys + 1);
	c->pos.assign(v->pos, v->pos + v->pos_off[v->n_keys]);
	c->bloom.assign(v->bloom_table, v->bloom_table + v->bloom_bits / 8);
	c->bloom_bits = v->bloom_bits;
	c->be = gpu_backend_create(&c->hidx, v->keys, v->n_keys, v->pos_off, v->pos, v->bloom_bits, v->bloom_table, device);
	return c;
}

extern "C" void wm_gpu_destroy(wm_gpu_ctx_s *c)
{
	if (!c) return;
	for (size_t i = 1; i < c->lanes.size(); ++i) gpu_backend_destroy(c->lanes[i]); // clones first: they borrow the owner's index
	gpu_backend_destroy(c->be);
	if (c->d_resident) cudaFree(c->d_resident);
	gpu_backend_trim_pool(c->device);
	free_reg_vectors(c->res_regs);
	delete c;
}

// Index construction from a FASTA file (mm_idx_gen, src/index.c:378-449): same minimizers as the reference
// because the reference sequences go through the same sketch kernel as the reads.
extern "C" wm_gpu_ctx_s *wm_index_build(const char *ref_fn, const char *kmer_freq_fn, int k, int w, int device)
{
	require_device("wm_index_build");
	if (!kw_ok("wm_index_build", k, w)) return 0;
	WM_CUDA_CHECK(cudaSetDevice(device));
	const double t0 = now_s();
	SeqReader rd;
	if (!rd.open(ref_fn)) { fprintf(stderr, "ERROR: failed to open file '%s'\n", ref_fn); return 0; }
	wm_gpu_ctx_s *c = new wm_gpu_ctx_s();
	memset(&c->stats, 0, sizeof(c->stats));
	c->device = device; c->t_index = c->t_map = 0;
	wm_host_idx &H = c->hidx;
	H.k = k, H.w = w;
	std::vector<uint64_t> kmers;
	if (read_kmer_list(kmer_freq_fn, k, kmers) < 0) abort();
	wm_bloom_s *bloom = wm_bloom_build(kmers.empty() ? 0 : kmers.data(), (int64_t)kmers.size());
	uint8_t *d_table = wm_dev_alloc<uint8_t>(wm_bloom_bits(bloom) / 8 + 16);
	WM_CUDA_CHECK(cudaMemcpy(d_table, wm_bloom_table(bloom), wm_bloom_bits(bloom) / 8, cudaMemcpyHostToDevice));
	wm_bloom_dev bf; wm_bloom_dev_from_table(&bf, d_table, wm_bloom_bits(bloom));
	// read the reference, pack it 4 bits per base (mm_seq4_set, src/mmpriv.h:29) and sketch it in groups; the minimizers stay
	// on the device: they are sorted and cut into the CSR there (index_dev.cu)
	std::vector<std::pair<wm128_dev*, int64_t>> parts; int64_t n_mz_total = 0;
	wm_sketch_ws ws;
	std::vector<wm_sk_task> tasks; std::string group; uint64_t sum_len = 0;
	wm_dbuf d_ascii, d_pk, d_nm;
	auto flush = [&]() {
		if (tasks.empty()) return;
		char *da = (char*)d_ascii.need(group.size() + 16);
		wm_pkseq pks; // the group as a packed pool (pkseq.cuh)
		pks.pk = (uint32_t*)d_pk.need(sizeof(uint32_t) * wm_pk_words((int64_t)group.size()));
		pks.nm = (uint32_t*)d_nm.need(sizeof(uint32_t) * wm_nm_words((int64_t)group.size()));
		WM_CUDA_CHECK(cudaMemcpy(da, group.data(), group.size(), cudaMemcpyHostToDevice));
		wm_pack_ascii(da, (int64_t)group.size(), (uint32_t*)pks.pk, (uint32_t*)pks.nm, 0);
		int64_t n_mz = 0;
		wm_sketch_run(&ws, bf, pks, tasks.data(), (int)tasks.size(), w, k, &n_mz, 0);
		WM_CUDA_CHECK(cudaDeviceSynchronize());
		if (n_mz > 0) {
			wm128_dev *part = wm_dev_alloc<wm128_dev>(n_mz);
			WM_CUDA_CHECK(cudaMemcpy(part, ws.mz.p, sizeof(wm128_dev) * n_mz, cudaMemcpyDeviceToDevice));
			parts.push_back(std::make_pair(part, n_mz)); n_mz_total += n_mz;
		}
		tasks.clear(); group.clear();
	};
	wm_read r;
	while (rd.next(r)) {
		const uint32_t rid = (uint32_t)H.name.size();
		H.name.push_back(r.name); H.len.push_back((uint32_t)r.seq.size()); H.offset.push_back(sum_len);
		const uint64_t need_words = (sum_len + r.seq.size() + 7) / 8;
		if (H.S.size() < need_words) H.S.resize(need_words, 0);
		pack_seq4(H.S.data(), sum_len, r.seq.data(), r.seq.size());
		sum_len += r.seq.size();
		if (!r.seq.empty()) {
			wm_sk_task t; t.seq_off = (int64_t)group.size(); t.len = (int32_t)r.seq.size(); t.rid = rid;
			tasks.push_back(t); group += r.seq;
		}
		if (group.size() >= ((size_t)1 << 30)) flush();
	}
	flush();
	ws.release(); d_ascii.release(); d_pk.release(); d_nm.release(); cudaFree(d_table);
	// one array in position order, then sort + CSR on the device
	wm128_dev *d_all = wm_dev_alloc<wm128_dev>(n_mz_total + 1);
	{
		int64_t o = 0;
		for (auto &pp : parts) { WM_CUDA_CHECK(cudaMemcpy(d_all + o, pp.first, sizeof(wm128_dev) * pp.second, cudaMemcpyDeviceToDevice)); o += pp.second; cudaFree(pp.first); }
	}
	uint64_t *d_keys = 0, *d_poff = 0, *d_pos = 0; int64_t n_keys = 0;
	wm_index_build_dev(d_all, n_mz_total, k, &d_keys, &d_poff, &d_pos, &n_keys, 0);
	c->n_keys = n_keys, c->n_pos = n_mz_total;
	c->be = gpu_backend_create_dev(&H, d_keys, n_keys, d_poff, d_pos, wm_bloom_bits(bloom), wm_bloom_table(bloom), device);
	c->bloom_bits = wm_bloom_bits(bloom);
	c->bloom.assign(wm_bloom_table(bloom), wm_bloom_table(bloom) + c->bloom_bits / 8);
	wm_bloom_destroy(bloom);
	c->t_index = now_s() - t0;
	return c;
}

extern "C" int wm_set_opt(const char *preset, wm_idxopt_t *io, wm_mapopt_t *mo) { return set_opt(preset, io, mo); }
extern "C" int wm_check_opt(const wm_idxopt_t *io, const wm_mapopt_t *mo) { return check_opt(io, mo); }
extern "C" int wm_sizeof_mapopt(void) { return (int)sizeof(wm_mapopt_t); }
extern "C" int wm_sizeof_reg1(void) { return (int)sizeof(wm_reg1_t); }
extern "C" int wm_abi_layout(int64_t *out, int cap)
{
	int n = 0;
#define PUT(v) do { if (n < cap) out[n] = (int64_t)(v); ++n; } while (0)
	PUT(sizeof(wm_mapopt_t)); PUT(sizeof(wm_reg1_t)); PUT(sizeof(wm_extra_t)); PUT(sizeof(wm_idxopt_t));
#define MO(f) PUT(offsetof(wm_mapopt_t, f))
	MO(flag); MO(seed); MO(sdust_thres); MO(max_qlen); MO(bw); MO(max_gap); MO(max_gap_ref); MO(min_gap_ref); MO(max_frag_len); MO(max_chain_skip);
	MO(max_chain_iter); MO(min_cnt); MO(min_chain_score); MO(chain_gap_scale); MO(SVaware); MO(SVawareMinReadLength); MO(suffixSampleOffset);
	MO(min_mapq); MO(min_qcov); MO(minPrefixLength); MO(maxPrefixLength); MO(prefixIncrementFactor); MO(stage2_bw); MO(stage2_zdrop_inv);
	MO(stage2_max_gap); MO(stage2_extension_inc); MO(mask_level); MO(mask_len); MO(pri_ratio); MO(best_n); MO(max_join_long); MO(max_join_short);
	MO(min_join_flank_sc); MO(min_join_flank_ratio); MO(alt_drop); MO(a); MO(b); MO(q); MO(e); MO(q2); MO(e2); MO(sc_ambi); MO(noncan); MO(junc_bonus);
	MO(zdrop); MO(zdrop_inv); MO(end_bonus); MO(min_dp_max); MO(min_ksw_len); MO(anchor_ext_len); MO(anchor_ext_shift); MO(max_clip_ratio);
	MO(pe_ori); MO(pe_bonus); MO(mid_occ_frac); MO(min_mid_occ); MO(mid_occ); MO(max_occ); MO(mini_batch_size); MO(max_sw_mat);
	MO(kmer_freq_filename); MO(split_prefix);
#define RG(f) PUT(offsetof(wm_reg1_t, f))
	RG(id); RG(cnt); RG(rid); RG(score); RG(qs); RG(qe); RG(rs); RG(re); RG(parent); RG(subsc); RG(as); RG(mlen); RG(blen); RG(n_sub); RG(score0); RG(hash); RG(div); RG(p);
#define EX(f) PUT(offsetof(wm_extra_t, f))
	EX(capacity); EX(dp_score); EX(dp_max); EX(dp_max2); EX(n_cigar); EX(cigar);
#define IO(f) PUT(offsetof(wm_idxopt_t, f))
	IO(k); IO(w); IO(flag); IO(bucket_bits); IO(mini_batch_size); IO(batch_size);
#undef PUT
#undef MO
#undef RG
#undef EX
#undef IO
	return n;
}

// The GPU replacement of kt_for(n_threads, worker_for, ...) (src/map.c:1164): fills n_reg/reg/rep_len/frag_gap of
// every sequence exactly as worker_for does (:1025-1034).  reg[i] and each reg[i][j].p are malloc()ed; the caller
// frees them (src/minimap.h:355-356).
extern "C" int wm_gpu_map_batch(wm_gpu_ctx_s *c, const wm_mapopt_t *opt, int n_seq, const char *const *names, const char *const *seqs,
                                const int32_t *lens, int32_t *n_reg, wm_reg1_t **reg, int32_t *rep_len, int32_t *frag_gap, int n_threads)
{
	require_device("wm_gpu_map_batch");
	std::vector<wm_read> store(n_seq);
	std::vector<const wm_read*> reads(n_seq);
	#pragma omp parallel for schedule(dynamic, 16) num_threads(n_threads > 0 ? n_threads : 1)
	for (int i = 0; i < n_seq; ++i) {
		store[i].name = names && names[i] ? names[i] : "";
		store[i].seq.assign(seqs[i], lens[i]);
		reads[i] = &store[i];
	}
	std::vector<std::vector<wm_reg1_t>> regs; std::vector<int> rl, fg;
	map_lanes(c, opt, reads, regs, rl, fg, n_threads, false);
	for (int i = 0; i < n_seq; ++i) {
		n_reg[i] = (int32_t)regs[i].size();
		reg[i] = 0;
		if (n_reg[i] > 0) {
			reg[i] = (wm_reg1_t*)malloc(sizeof(wm_reg1_t) * n_reg[i]);
			memcpy(reg[i], regs[i].data(), sizeof(wm_reg1_t) * n_reg[i]);
		}
		rep_len[i] = rl[i], frag_gap[i] = fg[i];
	}
	return 0;
}

// mm_tbuf_t / mm_map (src/map.c:18-38, :976-984): the per-thread buffer only carries rep_len and frag_gap of the last call here
// (device workspaces belong to the context's lanes).  One read = a batch of one through the same path as wm_gpu_map_batch.
struct wm_tbuf_s { int rep_len, frag_gap; };
extern "C" wm_tbuf_s *wm_tbuf_init(void) { return (wm_tbuf_s*)calloc(1, sizeof(wm_tbuf_s)); }
extern "C" void wm_tbuf_destroy(wm_tbuf_s *b) { free(b); }
extern "C" int wm_tbuf_rep_len(const wm_tbuf_s *b) { return b->rep_len; }
extern "C" int wm_tbuf_frag_gap(const wm_tbuf_s *b) { return b->frag_gap; }
extern "C" wm_reg1_t *wm_map(wm_gpu_ctx_s *c, int l_seq, const char *seq, int *n_regs, wm_tbuf_s *b, const wm_mapopt_t *opt, const char *name)
{
	int32_t n_reg = 0, rl = 0, fg = 0, len = l_seq;
	wm_reg1_t *reg = 0;
	const char *nm = name ? name : "";
	wm_gpu_map_batch(c, opt, 1, &nm, &seq, &len, &n_reg, &reg, &rl, &fg, 1);
	if (b) b->rep_len = rl, b->frag_gap = fg;
	*n_regs = n_reg;
	return reg;
}

// mm_map_file for PAF output.  Reads are taken in the reference's mini-batches (src/bseq.c:80-119), sorted by
// length descending inside a batch (src/map.c:1124-1143) and printed in that order (:1173-1208).  With world > 1
// this process maps and prints only the reads whose position in the sorted batch is rank mod world; every output
// line is preceded by "<batch>\t<position>\t" when tag_order != 0 so that the shards can be merged back.
extern "C" int wm_map_file(wm_gpu_ctx_s *c, const wm_mapopt_t *opt, const char *reads_fn, const char *out_fn, int n_threads, int rank, int world,
                           int tag_order, int64_t max_batch_bases)
{
	require_device("wm_map_file");
	SeqReader rd;
	if (!rd.open(reads_fn)) { fprintf(stderr, "ERROR: failed to open file '%s': %s\n", reads_fn, strerror(errno)); return -1; }
	FILE *out = out_fn && strcmp(out_fn, "-") ? fopen(out_fn, "wb") : stdout;
	if (!out) return -1;
	const double t0 = now_s();
	const int64_t chunk = opt->mini_batch_size;
	if ((opt->flag & WM_F_OUT_SAM) && rank == 0 && !tag_order) { // mm_write_sam_hdr (src/main.c:391-393)
		std::string hdr;
		write_sam_hdr(hdr, &c->hidx, "2.03", c->sam_cl.c_str());
		fwrite(hdr.data(), 1, hdr.size(), out);
	}
	// The three steps of the reference's pipeline (src/map.c:1107-1224: read, map, write) run on three threads with
	// one mini-batch of slack between them: the next batch is parsed and the previous one formatted while the GPU maps.
	struct FileBatch {
		int64_t no;
		std::vector<wm_read> reads;
		std::vector<const wm_read*> mine; std::vector<int> mine_pos;          // this rank's reads, in output order
		std::vector<std::vector<wm_reg1_t>> regs; std::vector<int> rl;        // aligned with `mine`
	};
	struct Slot { // a one-element hand-over queue
		std::mutex mu; std::condition_variable cv; FileBatch *item = 0; bool closed = false;
		void put(FileBatch *b) { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return item == 0; }); item = b; cv.notify_all(); }
		void close() { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return item == 0; }); closed = true; cv.notify_all(); }
		FileBatch *get() { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return item != 0 || closed; }); FileBatch *b = item; item = 0; cv.notify_all(); return b; }
	} q_in, q_out;
	std::thread reader([&]() {
		int64_t batch_no = 0;
		for (;;) {
			FileBatch *b = new FileBatch();
			int64_t size = 0;
			wm_read r;
			const bool with_qual = (opt->flag & WM_F_OUT_SAM) && !(opt->flag & WM_F_NO_QUAL); // src/map.c:1112
			while (rd.next(r)) {
				size += (int64_t)r.seq.size();
				if (!with_qual) r.qual.clear();
				b->reads.push_back(r);
				if (size >= chunk) break;
			}
			if (b->reads.empty()) { delete b; break; }
			b->no = batch_no++;
			q_in.put(b);
		}
		q_in.close();
	});
	std::thread writer([&]() {
		std::vector<std::string> lines;
		for (;;) {
			FileBatch *b = q_out.get();
			if (!b) break;
			const int n = (int)b->mine.size();
			lines.assign(n, std::string());
			#pragma omp parallel num_threads(n_threads > 8 ? 8 : (n_threads > 0 ? n_threads : 1))
			{
				std::string line; char tag[64];
				#pragma omp for schedule(dynamic, 16)
				for (int i = 0; i < n; ++i) {
					const wm_read *t = b->mine[i];
					std::string &dst = lines[i];
					const bool sam = (opt->flag & WM_F_OUT_SAM) != 0;
					auto emit = [&](int j) { // hit j of the read, or the empty record (j < 0), src/map.c:1189-1206
						if (sam) write_sam(line, &c->hidx, t, j, (int)b->regs[i].size(), b->regs[i].data(), opt->flag, b->rl[i], "");
						else write_paf(line, &c->hidx, t, j >= 0 ? &b->regs[i][j] : 0, opt->flag, b->rl[i]);
						if (tag_order) { snprintf(tag, sizeof(tag), "%lld\t%d\t", (long long)b->no, b->mine_pos[i]); dst += tag; }
						dst += line; dst += '\n';
					};
					if (!b->regs[i].empty()) {
						for (size_t j = 0; j < b->regs[i].size(); ++j) {
							const wm_reg1_t *rr = &b->regs[i][j];
							if ((opt->flag & WM_F_NO_PRINT_2ND) && rr->id != rr->parent) continue;
							emit((int)j);
						}
					} else if ((opt->flag & WM_F_PAF_NO_HIT) || (sam && !(opt->flag & WM_F_SAM_HIT_ONLY))) emit(-1);
					for (auto &rr : b->regs[i]) free(rr.p);
				}
			}
			for (int i = 0; i < n; ++i) fwrite(lines[i].data(), 1, lines[i].size(), out);
			delete b;
		}
	});
	for (;;) {
		FileBatch *b = q_in.get();
		if (!b) break;
		// longer reads first; ties by larger input index first (std::greater on (len, index), src/map.c:1129)
		std::vector<std::pair<int, int>> ord;
		for (size_t i = 0; i < b->reads.size(); ++i) ord.emplace_back((int)b->reads[i].seq.size(), (int)i);
		std::sort(ord.begin(), ord.end(), std::greater<std::pair<int, int>>());
		for (size_t p = 0; p < ord.size(); ++p)
			if ((int)(p % (size_t)world) == rank) { b->mine.push_back(&b->reads[ord[p].second]); b->mine_pos.push_back((int)p); }
		b->regs.resize(b->mine.size()); b->rl.assign(b->mine.size(), 0);
		// internal sub-batches bound device memory; results do not depend on how reads are grouped
		size_t s0 = 0;
		while (s0 < b->mine.size()) {
			size_t s1 = s0; int64_t nb = 0;
			while (s1 < b->mine.size() && (s1 == s0 || nb + (int64_t)b->mine[s1]->seq.size() <= max_batch_bases)) nb += (int64_t)b->mine[s1]->seq.size(), ++s1;
			std::vector<const wm_read*> sub(b->mine.begin() + s0, b->mine.begin() + s1);
			std::vector<std::vector<wm_reg1_t>> regs; std::vector<int> rl, fg;
			map_lanes(c, opt, sub, regs, rl, fg, n_threads, false);
			for (size_t i = 0; i < sub.size(); ++i) { b->regs[s0 + i].swap(regs[i]); b->rl[s0 + i] = rl[i]; }
			s0 = s1;
		}
		q_out.put(b);
	}
	q_out.close();
	reader.join(); writer.join();
	if (out != stdout) fclose(out); else fflush(out);
	c->t_map += now_s() - t0;
	return 0;
}

extern "C" void wm_set_sam_cl(wm_gpu_ctx_s *c, const char *cl) { c->sam_cl = cl ? cl : ""; }

// mm_gen_cs / mm_gen_MD (src/minimap.h:389-390, src/format.c:245-266): *buf is (re)allocated with realloc() when it is too
// small, *max_len is its capacity; the string is NUL terminated; returns its length
static int gen_cs_or_md_c(const wm_gpu_ctx_s *c, char **buf, int *max_len, const wm_reg1_t *r, const char *seq, int is_MD, int no_iden)
{
	std::string s;
	gen_cs_or_MD(s, &c->hidx, r, seq, is_MD, no_iden);
	if ((int)s.size() + 1 > *max_len) {
		int m = (int)s.size() + 1;
		m += m >> 1; // kroundup-like slack
		*buf = (char*)realloc(*buf, (size_t)m);
		*max_len = m;
	}
	memcpy(*buf, s.data(), s.size());
	(*buf)[s.size()] = 0;
	return (int)s.size();
}
// mm_idx_getseq / mm_idx_name2id (src/index.c:161-171, :131-140) and the sequence table of the index (mm_idx_seq_t)
extern "C" int wm_idx_getseq(const wm_gpu_ctx_s *c, uint32_t rid, uint32_t st, uint32_t en, uint8_t *seq) { return c->hidx.getseq(rid, st, en, seq); }
extern "C" int wm_idx_name2id(const wm_gpu_ctx_s *c, const char *name)
{
	for (size_t i = 0; i < c->hidx.name.size(); ++i) if (c->hidx.name[i] == name) return (int)i;
	return -1;
}
extern "C" int wm_idx_n_seq(const wm_gpu_ctx_s *c) { return (int)c->hidx.name.size(); }
extern "C" const char *wm_idx_seq_name(const wm_gpu_ctx_s *c, int rid) { return rid >= 0 && (size_t)rid < c->hidx.name.size() ? c->hidx.name[rid].c_str() : 0; }
extern "C" uint32_t wm_idx_seq_len(const wm_gpu_ctx_s *c, int rid) { return rid >= 0 && (size_t)rid < c->hidx.len.size() ? c->hidx.len[rid] : 0; }

extern "C" int wm_gen_cs(const wm_gpu_ctx_s *c, char **buf, int *max_len, const wm_reg1_t *r, const char *seq, int no_iden)
{ return gen_cs_or_md_c(c, buf, max_len, r, seq, 0, no_iden); }
extern "C" int wm_gen_MD(const wm_gpu_ctx_s *c, char **buf, int *max_len, const wm_reg1_t *r, const char *seq)
{ return gen_cs_or_md_c(c, buf, max_len, r, seq, 1, 0); }

extern "C" void wm_get_stats(wm_gpu_ctx_s *c, double *o, int n)
{
	const MapStats &s = c->stats;
	double v[] = { (double)s.n_reads, (double)s.n_bases, (double)s.n_minimaps, (double)s.n_chained, (double)s.n_dp_jobs, (double)s.n_ll_jobs,
	               (double)s.n_rounds, s.t_seed, s.t_dp, s.t_host, c->t_index, c->t_map, (double)c->n_keys, (double)c->n_pos };
	for (int i = 0; i < n && i < (int)(sizeof(v) / sizeof(v[0])); ++i) o[i] = v[i];
}
extern "C" void wm_reset_stats(wm_gpu_ctx_s *c) { memset(&c->stats, 0, sizeof(c->stats)); c->t_map = 0; }

// ---- bench instrumentation ----
extern "C" void wm_prof_enable(int on) { g_wm_prof.enabled = on; }
extern "C" void wm_prof_reset(void) { int e = g_wm_prof.enabled; memset(&g_wm_prof, 0, sizeof(g_wm_prof)); g_wm_prof.enabled = e; wm_prof_region_begin(); }
extern "C" void wm_prof_get(double *o)
{ // o[0]: kernel launches; then per kernel class (0 = DP fill at o[1..6], 1 = chaining forward pass at o[7..12]):
  // sum of launch ms, union of launch intervals ms, launches, algorithmic bytes, units (block cells / anchors), units2 (DP jobs)
	wm_prof_collect();
	o[0] = (double)g_wm_prof.n_launches;
	for (int k = 0; k < WM_PK_N; ++k) {
		const wm_prof_kind &K = g_wm_prof.k[k];
		double *q = o + 1 + 6 * k;
		q[0] = K.ms, q[1] = K.union_ms, q[2] = (double)K.launches, q[3] = K.alg_bytes, q[4] = K.units, q[5] = K.units2;
	}
}
// host<->device traffic of the mapping path since wm_prof_reset: o[0] = host-to-device bytes, o[1] = device-to-host bytes
extern "C" void wm_prof_get_copies(double *o) { o[0] = (double)g_wm_prof.h2d_bytes; o[1] = (double)g_wm_prof.d2h_bytes; }
extern "C" int wm_device_synchronize(void) { WM_CUDA_CHECK(cudaDeviceSynchronize()); return 0; }
// free / total bytes of the current device (bench: with the stream-ordered pool never trimmed while mapping, total - free after a
// pass is the high-water mark of the library's footprint)
extern "C" int wm_device_mem(double *free_bytes, double *total_bytes)
{
	size_t f = 0, t = 0;
	WM_CUDA_CHECK(cudaMemGetInfo(&f, &t));
	*free_bytes = (double)f, *total_bytes = (double)t;
	return 0;
}

extern "C" void wm_free_regs(int n, const int32_t *n_reg, wm_reg1_t **reg)
{ // what the reference's output step does after printing (src/map.c:1210-1211)
	for (int i = 0; i < n; ++i) {
		for (int j = 0; j < n_reg[i]; ++j) free(reg[i][j].p);
		free(reg[i]);
	}
}

// bench: put a batch of reads into HBM (ASCII -> codes, both strands) outside the timed region ...
extern "C" int wm_bench_upload(wm_gpu_ctx_s *c, int n_seq, const char *const *names, const char *const *seqs, const int32_t *lens)
{
	c->resident.assign(n_seq, wm_read());
	int64_t tot = 0;
	for (int i = 0; i < n_seq; ++i) {
		c->resident[i].name = names && names[i] ? names[i] : "";
		c->resident[i].seq.assign(seqs[i], lens[i]);
		c->resident[i].dev_off = tot;
		tot += lens[i];
	}
	WM_CUDA_CHECK(cudaDeviceSynchronize());
	if (c->d_resident) { WM_CUDA_CHECK(cudaFree(c->d_resident)); c->d_resident = 0; }
	WM_CUDA_CHECK(cudaMalloc((void**)&c->d_resident, (size_t)tot + 16));
	{
		std::vector<char> stage((size_t)tot + 1);
		for (int i = 0; i < n_seq; ++i) memcpy(stage.data() + c->resident[i].dev_off, seqs[i], lens[i]);
		WM_CUDA_CHECK(cudaMemcpy(c->d_resident, stage.data(), (size_t)tot, cudaMemcpyHostToDevice));
	}
	for (auto *be : c->lanes) be->set_resident_pool(c->d_resident);
	WM_CUDA_CHECK(cudaDeviceSynchronize());
	return 0;
}

// ... and map them with the device copies already resident; *ms = device time between two events that bracket the
// whole step (recorded on the legacy default stream, which orders against the backend's blocking stream).
static void free_reg_vectors(std::vector<std::vector<wm_reg1_t>> &regs)
{
	for (auto &v : regs) for (auto &r : v) free(r.p);
	regs.clear();
}

extern "C" int wm_bench_map_resident(wm_gpu_ctx_s *c, const wm_mapopt_t *opt, int n_threads, int group_reads, double *ms)
{ // the resident reads are submitted in groups of group_reads reads (<= 0: all at once); two events bracket the whole pass
	static cudaEvent_t e0 = 0, e1 = 0;
	if (!e0) { WM_CUDA_CHECK(cudaEventCreate(&e0)); WM_CUDA_CHECK(cudaEventCreate(&e1)); }
	const int n = (int)c->resident.size();
	free_reg_vectors(c->res_regs);
	c->res_regs.resize(n); c->res_rl.assign(n, 0);
	if (group_reads <= 0) group_reads = n > 0 ? n : 1;
	WM_CUDA_CHECK(cudaEventRecord(e0, 0));
	for (int g0 = 0; g0 < n; g0 += group_reads) {
		const int g1 = std::min(n, g0 + group_reads);
		std::vector<const wm_read*> reads(g1 - g0);
		for (int i = g0; i < g1; ++i) reads[i - g0] = &c->resident[i];
		std::vector<std::vector<wm_reg1_t>> regs; std::vector<int> rl, fg;
		map_lanes(c, opt, reads, regs, rl, fg, n_threads, true);
		for (int i = g0; i < g1; ++i) { c->res_regs[i].swap(regs[i - g0]); c->res_rl[i] = rl[i - g0]; }
	}
	WM_CUDA_CHECK(cudaEventRecord(e1, 0));
	WM_CUDA_CHECK(cudaEventSynchronize(e1));
	float f = 0.f;
	WM_CUDA_CHECK(cudaEventElapsedTime(&f, e0, e1));
	*ms = f;
	return 0;
}

// One read's output lines (PAF, or SAM when opt->flag says so), as the output step of the reference prints them (src/map.c:1189-1206)
static void format_read(std::string &dst, const wm_host_idx *mi, const wm_mapopt_t *opt, const wm_read *t, int n_reg, const wm_reg1_t *regs, int rep_len)
{
	std::string line;
	const bool sam = (opt->flag & WM_F_OUT_SAM) != 0;
	auto emit = [&](int j) {
		if (sam) write_sam(line, mi, t, j, n_reg, regs, opt->flag, rep_len, "");
		else write_paf(line, mi, t, j >= 0 ? &regs[j] : 0, opt->flag, rep_len);
		dst += line; dst += '\n';
	};
	if (n_reg > 0) {
		for (int j = 0; j < n_reg; ++j) {
			if ((opt->flag & WM_F_NO_PRINT_2ND) && regs[j].id != regs[j].parent) continue;
			emit(j);
		}
	} else if ((opt->flag & WM_F_PAF_NO_HIT) || (sam && !(opt->flag & WM_F_SAM_HIT_ONLY))) emit(-1);
}

// bench: the records of the last resident pass, formatted for the first n_first reads in input order (parity check of the timed path)
extern "C" int wm_bench_write(wm_gpu_ctx_s *c, const wm_mapopt_t *opt, int n_first, const char *out_fn)
{
	FILE *out = fopen(out_fn, "wb");
	if (!out) return -1;
	const int n = std::min<int>(n_first, (int)c->res_regs.size());
	std::string buf;
	for (int i = 0; i < n; ++i) {
		buf.clear();
		format_read(buf, &c->hidx, opt, &c->resident[i], (int)c->res_regs[i].size(), c->res_regs[i].data(), c->res_rl[i]);
		fwrite(buf.data(), 1, buf.size(), out);
	}
	fclose(out);
	return n;
}

// bench: the records of the last resident pass themselves, for reads [first, first + n) (output comparison of two builds)
extern "C" int64_t wm_bench_records(const wm_gpu_ctx_s *c, int first, int n, int32_t *n_reg, int32_t *rep_len, wm_reg1_t *regs, int64_t cap)
{
	int64_t k = 0;
	for (int i = first; i < first + n; ++i) {
		const bool have = i >= 0 && i < (int)c->res_regs.size();
		n_reg[i - first] = have ? (int32_t)c->res_regs[i].size() : 0;
		rep_len[i - first] = have ? c->res_rl[i] : 0;
		if (have)
			for (const wm_reg1_t &r : c->res_regs[i]) { if (k < cap) regs[k] = r; ++k; }
	}
	return k;
}

// The records wm_gpu_map_batch returned, formatted in input order with the writer wm_map_file uses (mm_write_paf3 / mm_write_sam3)
extern "C" int wm_format_batch(const wm_gpu_ctx_s *c, const wm_mapopt_t *opt, int n_seq, const char *const *names, const char *const *seqs, const int32_t *lens,
                               const int32_t *n_reg, wm_reg1_t *const *reg, const int32_t *rep_len, const char *out_fn)
{
	FILE *out = fopen(out_fn, "wb");
	if (!out) return -1;
	std::string buf;
	wm_read t;
	for (int i = 0; i < n_seq; ++i) {
		t.name = names && names[i] ? names[i] : "";
		t.seq.assign(seqs[i], lens[i]);
		buf.clear();
		format_read(buf, &c->hidx, opt, &t, n_reg[i], reg[i], rep_len[i]);
		fwrite(buf.data(), 1, buf.size(), out);
	}
	fclose(out);
	return 0;
}

extern "C" void wm_dump_timers(void) { wmh::g_timers.dump(stderr); wmh::g_timers.reset(); }

// ---- one-time index fan-out: the flattened index as one relocatable blob ----
// Rank 0 builds the index, the blob travels GPU-to-GPU with one NCCL broadcast (torch.distributed in bench.py) and
// every other rank re-creates its context from it.  Layout: 8 x uint64 header, then the arrays, each 8-byte aligned.
static inline size_t pad8(size_t x) { return (x + 7) & ~(size_t)7; }

// the host copies of keys / pos_off / pos exist only when the index came through wm_gpu_idx_upload; an index built on the
// device (wm_index_build) is fetched when the blob is first asked for
static void fetch_index_arrays(wm_gpu_ctx_s *c)
{
	if (!c->keys.empty() || c->n_keys == 0) return;
	const uint64_t *dk, *dpo, *dp;
	gpu_backend_index_arrays(c->be, &dk, &dpo, &dp);
	c->keys.resize(c->n_keys); c->pos_off.resize(c->n_keys + 1); c->pos.resize(c->n_pos);
	WM_CUDA_CHECK(cudaMemcpy(c->keys.data(), dk, sizeof(uint64_t) * c->n_keys, cudaMemcpyDeviceToHost));
	WM_CUDA_CHECK(cudaMemcpy(c->pos_off.data(), dpo, sizeof(uint64_t) * (c->n_keys + 1), cudaMemcpyDeviceToHost));
	WM_CUDA_CHECK(cudaMemcpy(c->pos.data(), dp, sizeof(uint64_t) * c->n_pos, cudaMemcpyDeviceToHost));
}

extern "C" int64_t wm_idx_blob_size(const wm_gpu_ctx_s *c_)
{
	wm_gpu_ctx_s *c = const_cast<wm_gpu_ctx_s*>(c_);
	fetch_index_arrays(c);
	const wm_host_idx &H = c->hidx;
	size_t names = 0;
	for (auto &s : H.name) names += s.size() + 1;
	return (int64_t)(8 * 8 + pad8(H.len.size() * 4) + H.offset.size() * 8 + pad8(names) + pad8(H.S.size() * 4) + c->keys.size() * 8 +
	                 c->pos_off.size() * 8 + c->pos.size() * 8 + pad8(c->bloom.size()));
}

extern "C" int wm_idx_blob_write(const wm_gpu_ctx_s *c_, uint8_t *buf)
{
	wm_gpu_ctx_s *c = const_cast<wm_gpu_ctx_s*>(c_);
	fetch_index_arrays(c);
	const wm_host_idx &H = c->hidx;
	size_t names = 0;
	for (auto &s : H.name) names += s.size() + 1;
	uint64_t *h = (uint64_t*)buf;
	h[0] = 0x31584449424d57ULL; /* "WMBIDX1" */ h[1] = (uint64_t)H.k << 32 | (uint32_t)H.w; h[2] = H.len.size(); h[3] = names;
	h[4] = H.S.size(); h[5] = c->keys.size(); h[6] = c->pos.size(); h[7] = c->bloom_bits;
	uint8_t *p = buf + 64;
	memcpy(p, H.len.data(), H.len.size() * 4); p += pad8(H.len.size() * 4);
	memcpy(p, H.offset.data(), H.offset.size() * 8); p += H.offset.size() * 8;
	{ uint8_t *q = p; for (auto &s : H.name) { memcpy(q, s.c_str(), s.size() + 1); q += s.size() + 1; } p += pad8(names); }
	memcpy(p, H.S.data(), H.S.size() * 4); p += pad8(H.S.size() * 4);
	memcpy(p, c->keys.data(), c->keys.size() * 8); p += c->keys.size() * 8;
	memcpy(p, c->pos_off.data(), c->pos_off.size() * 8); p += c->pos_off.size() * 8;
	memcpy(p, c->pos.data(), c->pos.size() * 8); p += c->pos.size() * 8;
	memcpy(p, c->bloom.data(), c->bloom.size());
	return 0;
}

extern "C" wm_gpu_ctx_s *wm_idx_blob_load(const uint8_t *buf, int64_t size, int device)
{
	require_device("wm_idx_blob_load");
	const uint64_t *h = (const uint64_t*)buf;
	if (size < 64 || h[0] != 0x31584449424d57ULL) { fprintf(stderr, "[ERROR] wm_idx_blob_load: bad blob\n"); return 0; }
	const size_t n_seq = h[2], names = h[3], s_words = h[4], n_keys = h[5], n_pos = h[6], bloom_bytes = (size_t)(h[7] / 8);
	{ // every section length comes from the header: the total must be exactly the buffer (a truncated or foreign broadcast is refused)
		const unsigned __int128 need = (unsigned __int128)64 + pad8(n_seq * 4) + (unsigned __int128)n_seq * 8 + pad8(names) + pad8(s_words * 4) +
			(unsigned __int128)n_keys * 8 + ((unsigned __int128)n_keys + 1) * 8 + (unsigned __int128)n_pos * 8 + pad8(bloom_bytes);
		if (need != (unsigned __int128)size) { fprintf(stderr, "[ERROR] wm_idx_blob_load: blob of %lld bytes does not match its header\n", (long long)size); return 0; }
	}
	const uint8_t *p = buf + 64;
	const uint32_t *len = (const uint32_t*)p; p += pad8(n_seq * 4);
	const uint64_t *off = (const uint64_t*)p; p += n_seq * 8;
	const char *nm = (const char*)p, *nm_end = nm + names; p += pad8(names);
	const uint32_t *S = (const uint32_t*)p; p += pad8(s_words * 4);
	const uint64_t *keys = (const uint64_t*)p; p += n_keys * 8;
	const uint64_t *pos_off = (const uint64_t*)p; p += (n_keys + 1) * 8;
	const uint64_t *pos = (const uint64_t*)p; p += n_pos * 8;
	if (pos_off[n_keys] != n_pos) { fprintf(stderr, "[ERROR] wm_idx_blob_load: occurrence table does not match its header\n"); return 0; }
	std::vector<const char*> name_ptr(n_seq);
	for (size_t i = 0; i < n_seq; ++i) {
		const void *z = nm < nm_end ? memchr(nm, 0, (size_t)(nm_end - nm)) : 0;
		if (!z) { fprintf(stderr, "[ERROR] wm_idx_blob_load: sequence name table is truncated\n"); return 0; }
		name_ptr[i] = nm; nm = (const char*)z + 1;
	}
	wm_idx_view_t v;
	v.k = (int32_t)(h[1] >> 32), v.w = (int32_t)(uint32_t)h[1], v.n_seq = (int32_t)n_seq;
	v.seq_name = name_ptr.data(), v.seq_len = len, v.seq_offset = off, v.S = S, v.S_words = s_words;
	v.n_keys = (int64_t)n_keys, v.keys = keys, v.pos_off = pos_off, v.pos = pos, v.bloom_bits = h[7], v.bloom_table = p;
	return wm_gpu_idx_upload(&v, device);
}
