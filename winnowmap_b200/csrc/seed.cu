// Seed lookup and anchor generation on sm_100a: mm_idx_get (reference src/index.c:88-105),
// collect_matches (src/map.c:97-130) and collect_seed_hits (src/map.c:222-254) for a batch of
// sketched query windows, followed by the tie-exact anchor sort (rsort.cuh).
//
// Index layout in HBM (replicated per GPU): sorted unique minimizer hashes `keys`, CSR offsets
// `pos_off` into the occurrence array `pos` (each list ascending, as src/index.c:239 leaves it) and an
// open-addressing hash table key -> key index for O(1) probes.  The bucket/khash structure of the
// reference is an implementation detail; the contract "hash -> (sorted list, n)" is what is kept.
#include <vector>
#include <algorithm>
#include "wm_common.cuh"
#include "scan.cuh"
#include "sketch.cuh"
#include "rsort.cuh"
#include "seed.cuh"

#define WM_HT_EMPTY 0xffffffffffffffffULL

__device__ __forceinline__ uint64_t wm_ht_mix(uint64_t k)
{
	k ^= k >> 31; k *= 0x9E3779B97F4A7C15ULL; k ^= k >> 29;
	return k;
}

__global__ void wm_ht_fill_kernel(const uint64_t *__restrict__ keys, int64_t n_keys, uint64_t *ht_key, uint32_t *ht_val, uint64_t mask)
{
	int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n_keys) return;
	const uint64_t key = keys[i];
	uint64_t slot = wm_ht_mix(key) & mask;
	for (;;) {
		unsigned long long old = atomicCAS((unsigned long long*)&ht_key[slot], (unsigned long long)WM_HT_EMPTY, (unsigned long long)key);
		if (old == WM_HT_EMPTY || old == key) { ht_val[slot] = (uint32_t)i; return; }
		slot = (slot + 1) & mask;
	}
}

// mm_idx_get: returns the number of occurrences and the offset of the list in pos[]
__device__ __forceinline__ int wm_idx_get(const wm_idx_dev &ix, uint64_t minier, uint64_t *off)
{
	uint64_t slot = wm_ht_mix(minier) & ix.ht_mask;
	for (;;) {
		const uint64_t k = ix.ht_key[slot];
		if (k == minier) {
			const uint32_t i = ix.ht_val[slot];
			const uint64_t o = ix.pos_off[i];
			*off = o;
			return (int)(ix.pos_off[i + 1] - o);
		}
		if (k == WM_HT_EMPTY) { *off = 0; return 0; }
		slot = (slot + 1) & ix.ht_mask;
	}
}

// pass 1: one thread per query minimizer
__global__ void wm_seed_lookup_kernel(wm_idx_dev ix, const wm128_dev *__restrict__ mz, const int64_t *__restrict__ mz_off, int n_tasks, int64_t n_mz,
                                      int max_occ, int32_t *__restrict__ n_occ, int32_t *__restrict__ cnt, uint64_t *__restrict__ list_off,
                                      uint8_t *__restrict__ tandem, int32_t *__restrict__ mz_task)
{
	const int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (m >= n_mz) return;
	int lo = 0, hi = n_tasks; // task of this minimizer: last t with mz_off[t] <= m
	while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (mz_off[mid] <= m) lo = mid; else hi = mid; }
	const uint64_t h = mz[m].x >> 8;
	uint64_t off;
	const int t = wm_idx_get(ix, h, &off);
	n_occ[m] = t;
	cnt[m] = t >= max_occ ? 0 : t; // src/map.c:111
	list_off[m] = off;
	int td = 0; // src/map.c:121-122
	if (m > mz_off[lo] && mz[m - 1].x >> 8 == h) td = 1;
	if (m < mz_off[lo + 1] - 1 && mz[m + 1].x >> 8 == h) td = 1;
	tandem[m] = (uint8_t)td;
	mz_task[m] = lo;
}

// pass 2: one thread per anchor (src/map.c:233-249; skip_seed() is a no-op without -D/-X/--for-only/--rev-only)
__global__ void wm_seed_expand_kernel(wm_idx_dev ix, const wm128_dev *__restrict__ mz, int64_t n_mz, const int64_t *__restrict__ a_off,
                                      const uint64_t *__restrict__ list_off, const uint8_t *__restrict__ tandem, const int32_t *__restrict__ mz_task,
                                      const int32_t *__restrict__ qlen, int64_t n_a, wm128_dev *__restrict__ a)
{
	const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n_a) return;
	int64_t lo = 0, hi = n_mz; // last m with a_off[m] <= j
	while (hi - lo > 1) { int64_t mid = (lo + hi) >> 1; if (a_off[mid] <= j) lo = mid; else hi = mid; }
	const wm128_dev p = mz[lo];
	const uint64_t r = ix.pos[list_off[lo] + (uint64_t)(j - a_off[lo])];
	const uint32_t q_pos = (uint32_t)p.y, q_span = (uint32_t)(p.x & 0xff);
	const int32_t rpos = (uint32_t)r >> 1;
	wm128_dev o;
	if ((r & 1) == (q_pos & 1)) { // forward strand
		o.x = (r & 0xffffffff00000000ULL) | (uint32_t)rpos;
		o.y = (uint64_t)q_span << 32 | q_pos >> 1;
	} else { // reverse strand
		o.x = 1ULL << 63 | (r & 0xffffffff00000000ULL) | (uint32_t)rpos;
		o.y = (uint64_t)q_span << 32 | (uint32_t)(qlen[mz_task[lo]] - ((q_pos >> 1) + 1 - q_span) - 1);
	}
	o.y |= (uint64_t)(p.y >> 32) << 48; // MM_SEED_SEG_SHIFT
	if (tandem[lo]) o.y |= 1ULL << 42;   // MM_SEED_TANDEM
	a[j] = o;
}

// pass 3: one thread per task: rep_len (src/map.c:106-127), kept-minimizer count, anchor offsets
__global__ void wm_seed_task_kernel(const wm128_dev *__restrict__ mz, const int64_t *__restrict__ mz_off, const int64_t *__restrict__ a_off,
                                    const int32_t *__restrict__ n_occ, int max_occ, int n_tasks, int32_t *__restrict__ rep_len,
                                    int32_t *__restrict__ n_mini_pos, int64_t *__restrict__ task_a_off, uint32_t *__restrict__ mini_pos)
{
	const int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t > n_tasks) return;
	if (t == n_tasks) { task_a_off[t] = a_off[mz_off[t]]; return; }
	int rep_st = 0, rep_en = 0, rl = 0, nk = 0;
	for (int64_t m = mz_off[t]; m < mz_off[t + 1]; ++m) {
		const uint32_t q_pos = (uint32_t)mz[m].y, q_span = (uint32_t)(mz[m].x & 0xff);
		if (n_occ[m] >= max_occ) {
			int en = (int)(q_pos >> 1) + 1, st = en - (int)q_span;
			if (st > rep_en) { rl += rep_en - rep_st; rep_st = st, rep_en = en; }
			else rep_en = en;
			mini_pos[m] = q_pos >> 1;
		} else { ++nk; mini_pos[m] = (q_pos >> 1) | 0x80000000u; }
	}
	rl += rep_en - rep_st;
	rep_len[t] = rl, n_mini_pos[t] = nk;
	task_a_off[t] = a_off[mz_off[t]];
}

// tie-exact radix_sort_128x of each task's anchors (src/map.c:252)
__global__ void wm_anchor_sort_small_kernel(wm128_dev *__restrict__ a, const int64_t *__restrict__ off, int n_arr, const int32_t *__restrict__ ids)
{
	int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= n_arr) return;
	if (ids) t = ids[t];
	const int64_t n = off[t + 1] - off[t];
	if (n <= WM_RS_MIN_SIZE) wm_rs_insertsort(a + off[t], a + off[t] + n);
}

// One warp per array of more than 64 anchors.  Arrays of up to smem_cap anchors are staged in shared
// memory, where the serial cycle-leader walk of lane 0 runs at shared-memory instead of L2 latency.
__global__ void __launch_bounds__(32)
wm_anchor_sort_big_kernel(wm128_dev *__restrict__ a, const int64_t *__restrict__ off, const int32_t *__restrict__ big_ids, int n_big,
                          wm_rs_range *__restrict__ wl_all, int smem_cap)
{
	extern __shared__ __align__(16) unsigned char wm_sort_smem[];
	__shared__ wm_rs_warp_ws W;
	__shared__ __align__(8) uint64_t mbar;
	const int lane = threadIdx.x;
	uint32_t phase = 0;
	if (lane == 0) wm_mbar_init(&mbar, 1);
	__syncwarp();
	for (int i = blockIdx.x; i < n_big; i += gridDim.x) {
		const int t = big_ids[i];
		const int64_t base = off[t];
		const int n = (int)(off[t + 1] - base);
		wm_rs_range *wl = wl_all + (base >> 6) + t;
		wm128_dev *g = a + base;
		if (n <= smem_cap) {
			// the array into its shared-memory stage and back with bulk-asynchronous copies (16-byte elements: always aligned)
			wm128_dev *s = (wm128_dev*)wm_sort_smem;
			const uint32_t bytes = (uint32_t)n * (uint32_t)sizeof(wm128_dev);
			if (lane == 0) { wm_mbar_expect_tx(&mbar, bytes); wm_bulk_g2s(s, g, bytes, &mbar); }
			wm_mbar_wait(&mbar, phase); phase ^= 1;
			wm_radix_sort_warp(s, n, &W, wl, lane);
			__syncwarp();
			if (lane == 0) { wm_bulk_s2g(g, s, bytes); wm_bulk_s2g_wait(); } // (the stage is reused by the next array)
			__syncwarp();
		} else wm_radix_sort_warp(g, n, &W, wl, lane);
	}
}

// ---- giant arrays (a read inside a tandem array: 10^5..10^6 anchors) ----
// The permutation walk of a radix pass (ksort.h:126-138) is a serial chain: the element in hand decides the bucket, the
// bucket's write position gives the next element in hand.  One observation makes it fast: every position of the array
// is written exactly once, when its bucket's write pointer passes it, so until then it still holds its ORIGINAL element
// -- the upcoming elements of every bucket can be prefetched.  One CTA per array: thread 0 walks, three feeder warps keep
// a FIFO of the next WM_GS_F original elements of each of the 256 buckets in shared memory, the walker never waits for
// global memory.  Sub-buckets that need another big pass go back on the array's work list; the smaller ones are sorted
// by the four warps in parallel (staged in shared memory, rsort.cuh); the <= 64-element ones by one thread each.
#define WM_GS_THREADS 128
// WM_GS_F: FIFO depth per bucket (power of two); WM_GS_STAGE: sub-ranges up to this many elements are sorted by one warp in
// shared memory.  Two instantiations: <16, 2048> (142 KB of shared memory, one CTA per SM) for the giant arrays and
// <8, 512> (46 KB, four CTAs per SM) for the medium ones, of which there are thousands per wave.
template <int WM_GS_F, int WM_GS_STAGE>
struct wm_gs_sm {
	int B[256], E[256];            // bucket bounds of the current pass
	int b[256];                    // write pointers (walker)
	int filled[256];               // originals loaded so far, per bucket (feeders)
	int hist[256];
	int moff[257];                 // token pass: offsets of every bucket's misplaced slots in the list
	int A[256];                    // token pass: arrivals in every bucket before its own turn
	int wtot[4];                   // per-warp totals of wm_gs_block_excl
	int n_big, n_small, next_small, walk_done;
	wm_rs_warp_ws W[4];
	wm_rs_range swl[4][40];        // per-warp work list of phase 2 (disjoint sub-ranges of > 64 elements of a <= 2048-element range)
	uint64_t mbar[4];              // per-warp mbarriers of the bulk copies that stage a sub-range
	uint32_t mbar_phase[4];
	union alignas(16) { // (bulk copies land in `stage`: 16-byte aligned)
		wm128_dev fifo[256][WM_GS_F];
		wm128_dev stage[4][WM_GS_STAGE];
	} u;
};

// a FIFO entry, read in place of a plain load so that the compiler keeps it after the (volatile) poll of `filled` without a
// "memory" clobber in the walker's loop (which made it re-derive the shared-memory base, an S2UR, on every step)
__device__ __forceinline__ wm128_dev wm_gs_fifo_read(const wm128_dev *p)
{
	wm128_dev r; uint32_t x0, x1, y0, y1;
	asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(x0), "=r"(x1), "=r"(y0), "=r"(y1) : "r"((uint32_t)__cvta_generic_to_shared(p)));
	r.x = (uint64_t)x1 << 32 | x0, r.y = (uint64_t)y1 << 32 | y0;
	return r;
}

// ---- a pass with exactly two non-empty buckets, in closed form ----
// The walk of ksort.h:126-138 over two buckets A (lower digit, region [beg, mid)) and B ([mid, end)) does this: let
// p_1 < .. < p_m be the positions of A's region that hold B-elements and q_1 < .. < q_m those of B's region that hold
// A-elements.  Cycle j picks up the element at p_j, drops it at B's write pointer and pushes the B-elements it finds there
// one slot to the right until it kicks out the A-element at q_j, which lands at p_j.  Hence, with q_0 = mid - 1:
//   A's region: position p_j receives the element of q_j, everything else stays;
//   B's region: position q_{j-1} + 1 receives the element of p_j, the positions up to q_j the element of their left
//               neighbour; everything after q_m stays.
// Both are prefix sums over "is misplaced" flags -- no serial walk.  The strand byte of an anchor array always splits it two
// ways, and the 64 kb byte of the position often does.  tmp / idx: scratch of the array (elements / int32), same indexing as a.
__device__ __forceinline__ int wm_gs_block_excl(bool flag, int *warp_tot, int tid, int *total)
{ // exclusive rank of `flag` among the CTA's 128 threads (4 warps); *total = number of flags set
	const unsigned w = __ballot_sync(0xffffffffu, flag);
	const int lane = tid & 31, wid = tid >> 5;
	if (lane == 0) warp_tot[wid] = __popc(w);
	__syncthreads();
	const int t0 = warp_tot[0], t1 = warp_tot[1], t2 = warp_tot[2], t3 = warp_tot[3];
	__syncthreads();
	*total = t0 + t1 + t2 + t3;
	return __popc(w & ((1u << lane) - 1u)) + (wid > 0 ? t0 : 0) + (wid > 1 ? t1 : 0) + (wid > 2 ? t2 : 0);
}

__device__ void wm_gs_two_bucket_pass(wm128_dev *a, wm128_dev *tmp, int32_t *idx, int beg, int mid, int end, int s, int lo, int *warp_tot, int tid)
{
	int carry = 0, tot;
	for (int base = beg; base < mid; base += WM_GS_THREADS) { // the list p_j (idx[beg ..))
		const int t = base + tid;
		const bool flag = t < mid && (int)(a[t].x >> s & 255) != lo;
		const int r = carry + wm_gs_block_excl(flag, warp_tot, tid, &tot);
		if (flag) idx[beg + r] = t;
		carry += tot;
	}
	const int m = carry;
	__syncthreads();
	carry = 0;
	for (int base = mid; base < end; base += WM_GS_THREADS) { // the list q_j (idx[mid ..)) and B's region
		const int t = base + tid;
		wm128_dev e; e.x = e.y = 0;
		if (t < end) e = a[t];
		const bool flag = t < end && (int)(e.x >> s & 255) == lo;
		const int c = carry + wm_gs_block_excl(flag, warp_tot, tid, &tot); // A-elements in [mid, t)
		if (flag) idx[mid + c] = t;
		if (t < end) {
			wm128_dev v = e;
			if (c < m) {
				wm128_dev left; left.x = left.y = 0;
				if (t > mid) left = a[t - 1];
				v = (t == mid || (int)(left.x >> s & 255) == lo) ? a[idx[beg + c]] : left;
			}
			tmp[t] = v;
		}
		carry += tot;
	}
	__syncthreads();
	carry = 0;
	for (int base = beg; base < mid; base += WM_GS_THREADS) { // A's region
		const int t = base + tid;
		wm128_dev e; e.x = e.y = 0;
		if (t < mid) e = a[t];
		const bool flag = t < mid && (int)(e.x >> s & 255) != lo;
		const int j = carry + wm_gs_block_excl(flag, warp_tot, tid, &tot);
		if (t < mid) tmp[t] = flag ? a[idx[mid + j]] : e;
		carry += tot;
	}
	__syncthreads();
	for (int t = beg + tid; t < end; t += WM_GS_THREADS) a[t] = tmp[t];
	__syncthreads();
}

// ---- a pass with three or more non-empty buckets: a token walk over destination digits ----
// The j-th element to arrive in a bucket ejects that bucket's j-th misplaced element (a slot of its region holding another bucket's
// element).  So the serial part of the walk needs only the destination digits D of the misplaced elements, listed in slot order
// (hence grouped by the bucket that owns the slot: bucket k's at list indices [moff[k], moff[k+1])), and one arrival pointer per
// bucket.  Bucket k's turn opens a cycle at each of its list entries not yet ejected; the element in hand arrives at index
// p = ptr[t]++ of its bucket t's list and the element listed there is next in hand, until one whose digit is k closes the cycle.
// No 16-byte element moves during the walk: land[] records, per list index, an arrival index p or ~opener, and the elements are
// then placed by all threads with index arithmetic:
//   - an arrival at index p of bucket t lands at the start of run p - moff[t] of t (B[t], or one past the previous misplaced slot);
//   - the element closing a cycle lands in the slot where the cycle was opened;
//   - an element already in its region moves one slot to the right if its run r has r < A[t] (the arrivals in t before t's turn
//     emptied those runs' misplaced slots), and stays otherwise.
// tests/test_sort_token_walk.py restates this in the same flat form and checks it against the serial walk.
// Scratch: the list's slots M in tmp (as int32), land[] in idx.  D is staged in shared memory (the FIFO / stage union) when the list
// fits there; otherwise it stays in idx as int32 (land[] overwrites it after use) and the three feeder warps stream it to the walker
// through per-bucket byte FIFOs -- the walker consumes every bucket's list in order, as it consumes the element FIFOs.
__device__ __forceinline__ int wm_gs_owner(const int *E, int i)
{ // smallest k with E[k] > i (E non-decreasing, E[255] > i): the bucket whose region holds slot i
	int k = 0;
	#pragma unroll
	for (int w = 128; w > 0; w >>= 1) if (E[k + w - 1] <= i) k += w;
	return k;
}

__device__ __forceinline__ int wm_gs_byte_read(const unsigned char *p)
{ // (volatile: stays ahead of the store of the arrival pointer that frees the FIFO entry)
	uint32_t r;
	asm volatile("ld.shared.u8 %0, [%1];" : "=r"(r) : "r"((uint32_t)__cvta_generic_to_shared(p)));
	return (int)r;
}

template <bool WM_GS_DBG, typename sm_t>
__device__ void wm_gs_token_pass(sm_t *S, wm128_dev *a, wm128_dev *tmp, int32_t *idx, int beg, int end, int s, int tid,
                                 unsigned long long &n_steps, unsigned long long &n_wait, bool &byte_fifo)
{
	constexpr int DCAP = (int)sizeof(S->u); // digits that fit in shared memory
	constexpr int FB = DCAP / 256;          // byte FIFO depth per bucket
	int *M = (int*)(tmp + beg);
	int32_t *land = idx + beg;
	unsigned char *Ds = (unsigned char*)&S->u;
	const int lane = tid & 31, wid = tid >> 5;
	// 1. the list: slots, digits, and its length per bucket
	for (int k = tid; k < 256; k += WM_GS_THREADS) S->hist[k] = 0;
	__syncthreads();
	int carry = 0, tot;
	for (int base = beg; base < end; base += WM_GS_THREADS) {
		const int i = base + tid;
		int own = 0, d = 0;
		if (i < end) { own = wm_gs_owner(S->E, i); d = (int)(a[i].x >> s & 255); }
		const bool flag = i < end && d != own;
		const int g = carry + wm_gs_block_excl(flag, S->wtot, tid, &tot);
		const unsigned peers = __match_any_sync(0xffffffffu, flag ? own : 256 + lane);
		if (flag) {
			M[g] = i, land[g] = d;
			if (g < DCAP) Ds[g] = (unsigned char)d;
			if (lane == __ffs(peers) - 1) atomicAdd(&S->hist[own], __popc(peers));
		}
		carry += tot;
	}
	const int m = carry;
	const bool staged = m <= DCAP;
	byte_fifo = !staged;
	__syncthreads();
	if (wid == 0) { // list offsets; the arrival pointers b[] and the feeders' marks filled[] start there
		int cnt[8], sum = 0;
		#pragma unroll
		for (int k = 0; k < 8; ++k) { cnt[k] = S->hist[lane * 8 + k]; sum += cnt[k]; }
		int incl = sum;
		#pragma unroll
		for (int o = 1; o < 32; o <<= 1) { int t2 = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t2; }
		int acc = incl - sum;
		#pragma unroll
		for (int k = 0; k < 8; ++k) { S->moff[lane * 8 + k] = acc; S->b[lane * 8 + k] = acc; S->filled[lane * 8 + k] = acc; acc += cnt[k]; }
		if (lane == 31) S->moff[256] = acc;
		if (lane == 0) S->walk_done = 0;
	}
	__syncthreads();
	// 2. the walk
	if (tid == 0) {
		int *ptr = S->b; const int *moff = S->moff;
		if (staged) {
			for (int k = 0; k < 256; ++k) {
				int f = ptr[k]; // (no arrivals in k during its own turn: ptr[k] stays)
				const int fe = moff[k + 1];
				S->A[k] = f - moff[k];
				for (; f < fe; ++f) {
					int cur = f, t = Ds[f];
					for (;;) {
						const int p = ptr[t];
						ptr[t] = p + 1;
						land[cur] = p;
						const int t2 = Ds[p];
						if (WM_GS_DBG) ++n_steps;
						if (t2 == k) { land[p] = ~f; break; }
						cur = p, t = t2;
					}
				}
			}
		} else {
			volatile int *filled = S->filled;
			for (int k = 0; k < 256; ++k) {
				int f = ptr[k];
				const int fe = moff[k + 1];
				S->A[k] = f - moff[k];
				while (f < fe) {
					const int opener = f;
					while (filled[k] <= f) { if (WM_GS_DBG) ++n_wait; }
					int t = wm_gs_byte_read(&Ds[k * FB + (f & (FB - 1))]);
					*(volatile int*)&ptr[k] = ++f;
					int cur = opener;
					for (;;) {
						const int p = ptr[t];
						while (filled[t] <= p) { if (WM_GS_DBG) ++n_wait; }
						const int t2 = wm_gs_byte_read(&Ds[t * FB + (p & (FB - 1))]);
						*(volatile int*)&ptr[t] = p + 1;
						land[cur] = p;
						if (WM_GS_DBG) ++n_steps;
						if (t2 == k) { land[p] = ~opener; break; }
						cur = p, t = t2;
					}
				}
			}
		}
		__threadfence_block();
		*(volatile int*)&S->walk_done = 1;
	} else if (!staged && wid > 0) { // feeders: 96 threads, buckets tid - 32, + 96, + 192
		volatile int *bv = S->b; volatile int *done = &S->walk_done;
		for (;;) {
			bool any = false, fed = false;
			for (int k = tid - 32; k < 256; k += WM_GS_THREADS - 32) {
				const int fl = S->filled[k], ek = S->moff[k + 1];
				if (fl >= ek) continue;
				any = true;
				const int want = ek - fl < 16 ? ek - fl : 16;
				if (FB - (fl - bv[k]) >= want) {
					int r[16];
					#pragma unroll
					for (int q = 0; q < 16; ++q) if (q < want) r[q] = land[fl + q];
					#pragma unroll
					for (int q = 0; q < 16; ++q) if (q < want) Ds[k * FB + ((fl + q) & (FB - 1))] = (unsigned char)r[q];
					__threadfence_block();
					*(volatile int*)&S->filled[k] = fl + want;
					fed = true;
				}
			}
			if (!any || *done) break;
			if (!fed) __nanosleep(256);
		}
	}
	__syncthreads();
	// 3. where every listed element lands (M is read here for the last time)
	for (int f = tid; f < m; f += WM_GS_THREADS) {
		const int L = land[f];
		int dst;
		if (L < 0) dst = M[~L];
		else { const int t = wm_gs_owner(S->moff + 1, L); dst = L == S->moff[t] ? S->B[t] : M[L - 1] + 1; }
		land[f] = dst;
	}
	__syncthreads();
	// 4. placement into tmp, and back
	carry = 0;
	for (int base = beg; base < end; base += WM_GS_THREADS) {
		const int i = base + tid;
		wm128_dev e; e.x = e.y = 0;
		int own = 0;
		if (i < end) { e = a[i]; own = wm_gs_owner(S->E, i); }
		const bool flag = i < end && (int)(e.x >> s & 255) != own;
		const int g = carry + wm_gs_block_excl(flag, S->wtot, tid, &tot);
		if (i < end) tmp[flag ? land[g] : (g - S->moff[own] < S->A[own] ? i + 1 : i)] = e;
		carry += tot;
	}
	__syncthreads();
	for (int t = beg + tid; t < end; t += WM_GS_THREADS) a[t] = tmp[t];
	__syncthreads();
}

template <int WM_GS_F, int WM_GS_STAGE, bool WM_GS_DBG>
__global__ void __launch_bounds__(WM_GS_THREADS)
wm_anchor_sort_giant_kernel(wm128_dev *__restrict__ a_all, const int64_t *__restrict__ off, const int32_t *__restrict__ ids, int n_arr,
                            wm_rs_range *__restrict__ wl_all, unsigned long long *dbg, wm128_dev *__restrict__ tmp_all, int32_t *__restrict__ idx_all,
                            const int64_t *__restrict__ scr_off, int two_min, int token_min)
{
	// tmp_all / idx_all: scratch of the closed-form and token passes (one element + one int32 per anchor); array ai's slice starts at
	// scr_off[ai] and is indexed like the array.  two_min / token_min: ranges of at least this many elements take the closed form when
	// their pass has two non-empty buckets / the token walk when it has more (0: never)
	// dbg (tuning aid, WM_SORT_DEBUG=1): clocks spent by thread 0 in [0] histograms, [1] the walk (any pass kind), [2] sub-bucket
	// dispatch + tiny sorts, [3] phase 2, [4] walker steps, [5] walker waits (polls of an empty FIFO), [6] elements in closed-form
	// passes, [7] token-walk steps, [8] elements in token passes, [9] token passes fed through byte FIFOs
	long long t_dbg = dbg ? clock64() : 0;
	unsigned long long n_steps_dbg = 0, n_wait_dbg = 0, n_tok_dbg = 0;
#define WM_GS_LAP(i) do { if (dbg && tid == 0) { const long long t2 = clock64(); atomicAdd(dbg + (i), (unsigned long long)(t2 - t_dbg)); t_dbg = t2; } } while (0)
	extern __shared__ __align__(16) unsigned char wm_gs_smem[];
	typedef wm_gs_sm<WM_GS_F, WM_GS_STAGE> sm_t;
	sm_t *S = (sm_t*)wm_gs_smem;
	if (threadIdx.x < 4) { wm_mbar_init(&S->mbar[threadIdx.x], 1); S->mbar_phase[threadIdx.x] = 0; }
	__syncthreads();
	const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
	for (int ai = blockIdx.x; ai < n_arr; ai += gridDim.x) {
		const int task = ids[ai];
		const int64_t base = off[task];
		const int n = (int)(off[task + 1] - base);
		wm128_dev *a = a_all + base;
		wm128_dev *tmp = scr_off ? tmp_all + scr_off[ai] : 0;
		int32_t *idx = scr_off ? idx_all + scr_off[ai] : 0;
		asm volatile("" : "+l"(a)); // keep the pointer in registers: the walker's loop was re-deriving it from the parameter bank (an LDC per step)
		// work lists in global memory (the array's slice of wl_all: n / 64 + 1 entries): big ranges grow from the front,
		// small ones from the back
		wm_rs_range *wl = wl_all + (base >> 6) + task;
		const int wl_cap = (n >> 6) + 1;
		if (tid == 0) { S->n_big = 0, S->n_small = 0; wm_rs_range r; r.beg = 0, r.end = n, r.s = 56; wl[0] = r; S->n_big = 1; }
		__syncthreads();
		// ---- phase 1: big passes, one at a time ----
		for (;;) {
			if (S->n_big == 0) break;
			__syncthreads();
			wm_rs_range R = wl[S->n_big - 1];
			__syncthreads();
			if (tid == 0) --S->n_big;
			int beg = R.beg, end = R.end, s = R.s;
			bool single; int n_nz = 0, lo_digit = 0;
			for (;;) { // histogram of byte s >> 3; identity passes (one bucket holds everything) are skipped (ksort.h:121-125)
				for (int k = tid; k < 256; k += WM_GS_THREADS) S->hist[k] = 0;
				__syncthreads();
				for (int i = beg + tid; i < end; i += WM_GS_THREADS) atomicAdd(&S->hist[a[i].x >> s & 255], 1);
				__syncthreads();
				single = false; n_nz = 0; lo_digit = -1;
				for (int k = 0; k < 256; ++k) { // (uniform: every thread scans the same table)
					const int h = S->hist[k];
					if (h == end - beg) single = true;
					if (h > 0) { ++n_nz; if (lo_digit < 0) lo_digit = k; }
				}
				if (!single || s == 0) break;
				s = s > 8 ? s - 8 : 0;
				__syncthreads();
			}
			WM_GS_LAP(0);
			if (single) { __syncthreads(); continue; } // all keys equal down to the last byte: nothing moves
			if (wid == 0) { // bucket bounds: exclusive prefix over 256 counts
				int cnt[8], sum = 0;
				#pragma unroll
				for (int k = 0; k < 8; ++k) { cnt[k] = S->hist[lane * 8 + k]; sum += cnt[k]; }
				int incl = sum;
				#pragma unroll
				for (int o = 1; o < 32; o <<= 1) { int t2 = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t2; }
				int acc = beg + incl - sum;
				#pragma unroll
				for (int k = 0; k < 8; ++k) { S->B[lane * 8 + k] = acc; S->b[lane * 8 + k] = acc; S->filled[lane * 8 + k] = acc; acc += cnt[k]; S->E[lane * 8 + k] = acc; }
				if (lane == 0) S->walk_done = 0;
			}
			__syncthreads();
			if (n_nz == 2 && two_min > 0 && end - beg >= two_min) { // two buckets: the pass in closed form, by all threads
				wm_gs_two_bucket_pass(a, tmp, idx, beg, S->E[lo_digit], end, s, lo_digit, S->hist, tid);
				if (WM_GS_DBG && tid == 0) atomicAdd(dbg + 6, (unsigned long long)(end - beg));
			} else if (n_nz > 2 && token_min > 0 && end - beg >= token_min) { // the token walk, placement by all threads
				bool byte_fifo;
				wm_gs_token_pass<WM_GS_DBG>(S, a, tmp, idx, beg, end, s, tid, n_tok_dbg, n_wait_dbg, byte_fifo);
				if (WM_GS_DBG && tid == 0) { atomicAdd(dbg + 8, (unsigned long long)(end - beg)); if (byte_fifo) atomicAdd(dbg + 9, 1ULL); }
			} else
			if (tid == 0) { // the walker (ksort.h:126-138); b[] are its pointers, filled[] the feeders'
				volatile int *filled = S->filled; int *b = S->b; const int *E = S->E;
				for (int k = 0; k < 256;) {
					const int bk = b[k];
					if (bk != E[k]) {
						while (filled[k] <= bk) { if (WM_GS_DBG) ++n_wait_dbg; }
						wm128_dev tmp = wm_gs_fifo_read(&S->u.fifo[k][bk & (WM_GS_F - 1)]);
						if (WM_GS_DBG) ++n_steps_dbg;
						int l = (int)(tmp.x >> s & 255);
						if (l != k) {
							do {
								const int bl = b[l];
								while (filled[l] <= bl) { if (WM_GS_DBG) ++n_wait_dbg; }
								if (WM_GS_DBG) ++n_steps_dbg;
								const wm128_dev nxt = wm_gs_fifo_read(&S->u.fifo[l][bl & (WM_GS_F - 1)]);
								a[bl] = tmp;
								*(volatile int*)&b[l] = bl + 1;
								tmp = nxt;
								l = (int)(tmp.x >> s & 255);
							} while (l != k);
							a[bk] = tmp;
						}
						*(volatile int*)&b[k] = bk + 1;
					} else ++k;
				}
				__threadfence_block();
				*(volatile int*)&S->walk_done = 1;
			} else if (wid > 0) { // feeders: 96 threads, buckets tid - 32, + 96, + 192
				volatile int *bv = S->b; volatile int *done = &S->walk_done;
				for (;;) {
					bool any = false, fed = false;
					for (int k = tid - 32; k < 256; k += WM_GS_THREADS - 32) {
						const int fl = S->filled[k], Ek = S->E[k];
						if (fl >= Ek) continue;
						any = true;
						const int pending = fl - bv[k];   // loaded, not yet taken by the walker
						int room = WM_GS_F - pending;
						if (room > Ek - fl) room = Ek - fl;
						if (room > 8) room = 8;
						if (room > WM_GS_F) room = WM_GS_F;
						if (room >= WM_GS_F / 4 || (room > 0 && (room == Ek - fl || pending < WM_GS_F / 4))) { // refill in batches unless the FIFO runs low
							wm128_dev r[8];
							#pragma unroll
							for (int m = 0; m < 8; ++m) if (m < room) r[m] = a[fl + m];
							#pragma unroll
							for (int m = 0; m < 8; ++m) if (m < room) S->u.fifo[k][(fl + m) & (WM_GS_F - 1)] = r[m];
							__threadfence_block();
							*(volatile int*)&S->filled[k] = fl + room;
							fed = true;
						}
					}
					if (!any || *done) break;
					// nothing to load right now: do not hammer shared memory with polls (the walker's own loads queue behind them;
					// measured: 300 clocks per step with spinning feeders)
					if (!fed) __nanosleep(256);
				}
			}
			__syncthreads();
			WM_GS_LAP(1);
			// sub-buckets (ksort.h:140-145)
			if (s > 0) {
				const int ns = s > 8 ? s - 8 : 0;
				for (int k = tid; k < 256; k += WM_GS_THREADS) {
					const int cb = S->B[k], ce = S->E[k], sz = ce - cb;
					if (sz > WM_GS_STAGE) { const int q = atomicAdd(&S->n_big, 1); wm_rs_range r; r.beg = cb, r.end = ce, r.s = ns; wl[q] = r; }
					else if (sz > WM_RS_MIN_SIZE) { const int q = atomicAdd(&S->n_small, 1); wm_rs_range r; r.beg = cb, r.end = ce, r.s = ns; wl[wl_cap - 1 - q] = r; }
					else if (sz > 1) wm_rs_insertsort(a + cb, a + ce);
				}
			}
			__syncthreads();
		}
		WM_GS_LAP(2);
		// ---- phase 2: the small ranges, one warp each, staged in shared memory ----
		if (tid == 0) S->next_small = 0;
		__syncthreads();
		{
			wm128_dev *st = S->u.stage[wid];
			uint32_t ph2 = S->mbar_phase[wid]; // the warp's barrier survives from array to array: remember its phase
			for (;;) {
				int q = 0;
				if (lane == 0) q = atomicAdd(&S->next_small, 1);
				q = __shfl_sync(0xffffffffu, q, 0);
				if (q >= S->n_small) break;
				const wm_rs_range R = wl[wl_cap - 1 - q];
				const int m = R.end - R.beg;
				const uint32_t bytes = (uint32_t)m * (uint32_t)sizeof(wm128_dev);
				if (lane == 0) { wm_mbar_expect_tx(&S->mbar[wid], bytes); wm_bulk_g2s(st, a + R.beg, bytes, &S->mbar[wid]); }
				wm_mbar_wait(&S->mbar[wid], ph2); ph2 ^= 1;
				wm_radix_sort_warp_from(st, m, R.s, &S->W[wid], S->swl[wid], lane);
				__syncwarp();
				if (lane == 0) { wm_bulk_s2g(a + R.beg, st, bytes); wm_bulk_s2g_wait(); }
				__syncwarp();
			}
			if (lane == 0) S->mbar_phase[wid] = ph2;
		}
		__syncthreads();
		WM_GS_LAP(3);
	}
	if (dbg && tid == 0) { atomicAdd(dbg + 4, n_steps_dbg); atomicAdd(dbg + 5, n_wait_dbg); atomicAdd(dbg + 7, n_tok_dbg); }
#undef WM_GS_LAP
}

// sort n_arr arrays (device); h_off is the host copy of the offsets
void wm_anchor_sort_run(wm_seed_ws *ws, wm128_dev *d_a, const int64_t *d_off, const int64_t *h_off, int n_arr, cudaStream_t st, const int32_t *only, int n_only)
{ // only != null: just the arrays only[0 .. n_only) of the n_arr
	if (n_arr <= 0 || (only && n_only <= 0)) return;
	std::vector<int32_t> big, small_ids;
	if (only) {
		for (int q = 0; q < n_only; ++q) { const int i = only[q]; if (h_off[i + 1] - h_off[i] > WM_RS_MIN_SIZE) big.push_back(i); else if (h_off[i + 1] - h_off[i] > 1) small_ids.push_back(i); }
	} else for (int i = 0; i < n_arr; ++i) if (h_off[i + 1] - h_off[i] > WM_RS_MIN_SIZE) big.push_back(i);
	if (getenv("WM_DP_STATS")) {
		int64_t mx = 0, n_2k = 0, n_10k = 0;
		for (int i = 0; i < n_arr; ++i) { int64_t n = h_off[i + 1] - h_off[i]; mx = n > mx ? n : mx; n_2k += n > 2560; n_10k += n > 10240; }
		fprintf(stderr, "[sort-stats] arrays=%d big=%d >2560:%ld >10240:%ld max=%ld total=%ld\n", n_arr, (int)big.size(), (long)n_2k, (long)n_10k, (long)mx, (long)h_off[n_arr]);
	}
	if (!only) { wm_count_launch(); wm_anchor_sort_small_kernel<<<(n_arr + 127) / 128, 128, 0, st>>>(d_a, d_off, n_arr, 0); }
	else if (!small_ids.empty()) {
		int32_t *d_small = (int32_t*)ws->small_ids.need(sizeof(int32_t) * small_ids.size());
		WM_CUDA_CHECK(wm_memcpy_async(d_small, small_ids.data(), sizeof(int32_t) * small_ids.size(), cudaMemcpyHostToDevice, st));
		wm_count_launch(); wm_anchor_sort_small_kernel<<<(unsigned)((small_ids.size() + 127) / 128), 128, 0, st>>>(d_a, d_off, (int)small_ids.size(), d_small);
		wm_stream_sync(st); // small_ids is a local
	}
	WM_CUDA_CHECK(cudaGetLastError());
	if (!big.empty()) {
		// three launches by size class: the shared-memory stage of the array sets the occupancy
		static int cap_m_env = -1; // WM_SORT_GIANT_MIN: arrays above this many anchors go to the <16, 2048> instantiation (default: none --
		// measured on the tandem workload: everything on the light <8, 512> instantiation, four CTAs per SM, is 10 % faster end to end)
		if (cap_m_env < 0) { const char *e = getenv("WM_SORT_GIANT_MIN"); cap_m_env = e && atoi(e) >= 2048 ? atoi(e) : (1 << 30); } // (above 13312 only with the walker kernels: the single-warp kernel stages the array in 208 KB)
		static int giant = -1, medium_coop = -1; // WM_SORT_GIANT=0 / WM_SORT_MEDIUM=0: the single-warp kernels (kept for comparison)
		if (giant < 0) { const char *e = getenv("WM_SORT_GIANT"); giant = (e && *e == '0') ? 0 : 1; e = getenv("WM_SORT_MEDIUM"); medium_coop = (e && *e == '0') ? 0 : 1; }
		const int cap_s = 2048, cap_m = medium_coop || cap_m_env < 13312 ? cap_m_env : 13312; // 32 KB and up to 208 KB of anchors
		WM_CUDA_CHECK(cudaFuncSetAttribute(wm_anchor_sort_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (cap_m < 13312 ? cap_m : 13312) * (int)sizeof(wm128_dev)));
		std::stable_sort(big.begin(), big.end(), [&](int x, int y) { return h_off[x + 1] - h_off[x] > h_off[y + 1] - h_off[y]; });
		size_t n_l = 0, n_m = 0;
		while (n_l < big.size() && h_off[big[n_l] + 1] - h_off[big[n_l]] > cap_m) ++n_l;
		while (n_l + n_m < big.size() && h_off[big[n_l + n_m] + 1] - h_off[big[n_l + n_m]] > cap_s) ++n_m;
		const size_t n_s = big.size() - n_l - n_m;
		// scratch of the closed-form and token passes of the walker kernels: one element + one int32 per anchor of the arrays they sort,
		// array big[q] (q < n_l + n_m) at scratch offset scr[q]
		static int two_min = -1; // WM_SORT_TWO_MIN: ranges of at least this many anchors take the closed form (0: always walk)
		if (two_min < 0) { const char *e = getenv("WM_SORT_TWO_MIN"); two_min = e ? atoi(e) : 512; }
		static int token_min = -1; // WM_SORT_TOKEN_MIN: ranges of at least this many anchors take the token walk (0: always the element walker)
		if (token_min < 0) { const char *e = getenv("WM_SORT_TOKEN_MIN"); token_min = e ? atoi(e) : 512; }
		const size_t n_w = n_l + n_m;
		std::vector<int64_t> scr(n_w + 1, 0);
		for (size_t q = 0; q < n_w; ++q) scr[q + 1] = scr[q] + (h_off[big[q] + 1] - h_off[big[q]]);
		const bool use_scr = (two_min > 0 || token_min > 0) && n_w > 0;
		// device copies: scratch offsets (int64, first for alignment), then the array ids
		int64_t *d_scr = (int64_t*)ws->big_ids.need(sizeof(int64_t) * (n_w + 1) + sizeof(int32_t) * big.size());
		int32_t *d_big = (int32_t*)(d_scr + n_w + 1);
		wm_rs_range *d_wl = (wm_rs_range*)ws->rs_stacks.need(sizeof(wm_rs_range) * (size_t)((h_off[n_arr] >> 6) + n_arr + 2));
		WM_CUDA_CHECK(wm_memcpy_async(d_big, big.data(), sizeof(int32_t) * big.size(), cudaMemcpyHostToDevice, st));
		wm128_dev *d_tmp = 0; int32_t *d_idx = 0;
		if (use_scr) {
			WM_CUDA_CHECK(wm_memcpy_async(d_scr, scr.data(), sizeof(int64_t) * (n_w + 1), cudaMemcpyHostToDevice, st));
			d_tmp = (wm128_dev*)ws->sort_tmp.need(sizeof(wm128_dev) * (size_t)(scr[n_w] + 1));
			d_idx = (int32_t*)ws->sort_idx.need(sizeof(int32_t) * (size_t)(scr[n_w] + 1));
		}
		const int64_t *d_scr_l = use_scr ? d_scr : 0, *d_scr_m = use_scr ? d_scr + n_l : 0;
		const char *dbg_fmt = "[sort-debug] arrays=%d clocks: hist %llu walk %llu dispatch %llu phase2 %llu | walker steps %llu wait polls %llu | "
		                      "elements in closed-form passes %llu | token-walk steps %llu elements in token passes %llu byte-FIFO passes %llu\n";
		if (n_l) {
			wm_count_launch();
			if (giant) {
				typedef wm_gs_sm<16, 2048> sm_t;
				static bool attr_set = false;
				if (!attr_set) {
					WM_CUDA_CHECK(cudaFuncSetAttribute(wm_anchor_sort_giant_kernel<16, 2048, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(sm_t)));
					WM_CUDA_CHECK(cudaFuncSetAttribute(wm_anchor_sort_giant_kernel<16, 2048, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(sm_t)));
					attr_set = true;
				}
				unsigned long long *dbg = 0;
				if (getenv("WM_SORT_DEBUG")) { WM_CUDA_CHECK(cudaMalloc((void**)&dbg, 128)); WM_CUDA_CHECK(cudaMemset(dbg, 0, 128)); }
				static int giant_ctas = -1; // WM_SORT_GIANT_CTAS
				if (giant_ctas < 0) { const char *e = getenv("WM_SORT_GIANT_CTAS"); giant_ctas = e && atoi(e) > 0 ? atoi(e) : 148; }
				const unsigned g_l = (unsigned)(n_l < (size_t)giant_ctas ? n_l : (size_t)giant_ctas);
				if (dbg) wm_anchor_sort_giant_kernel<16, 2048, true><<<g_l, WM_GS_THREADS, sizeof(sm_t), st>>>(d_a, d_off, d_big, (int)n_l, d_wl, dbg, d_tmp, d_idx, d_scr_l, two_min, token_min);
				else wm_anchor_sort_giant_kernel<16, 2048, false><<<g_l, WM_GS_THREADS, sizeof(sm_t), st>>>(d_a, d_off, d_big, (int)n_l, d_wl, 0, d_tmp, d_idx, d_scr_l, two_min, token_min);
				if (dbg) {
					unsigned long long h[16];
					WM_CUDA_CHECK(cudaStreamSynchronize(st));
					WM_CUDA_CHECK(cudaMemcpy(h, dbg, 128, cudaMemcpyDeviceToHost));
					fprintf(stderr, dbg_fmt, (int)n_l, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], h[9]);
					cudaFree(dbg);
				}
			} else wm_anchor_sort_big_kernel<<<(unsigned)n_l, 32, 0, st>>>(d_a, d_off, d_big, (int)n_l, d_wl, 0);
		}
		if (n_m) {
			wm_count_launch();
			if (medium_coop) { // thousands of arrays per wave: the light instantiation, four CTAs per SM
				typedef wm_gs_sm<8, 512> sm_t;
				static bool attr_set = false;
				if (!attr_set) {
					WM_CUDA_CHECK(cudaFuncSetAttribute(wm_anchor_sort_giant_kernel<8, 512, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(sm_t)));
					WM_CUDA_CHECK(cudaFuncSetAttribute(wm_anchor_sort_giant_kernel<8, 512, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(sm_t)));
					attr_set = true;
				}
				unsigned long long *dbg = 0;
				if (getenv("WM_SORT_DEBUG")) { WM_CUDA_CHECK(cudaMalloc((void**)&dbg, 128)); WM_CUDA_CHECK(cudaMemset(dbg, 0, 128)); }
				static int med_ctas = -1; // WM_SORT_MEDIUM_CTAS: resident CTAs of the medium class (47 KB of shared memory each)
				if (med_ctas < 0) { const char *e = getenv("WM_SORT_MEDIUM_CTAS"); med_ctas = e && atoi(e) > 0 ? atoi(e) : 592; }
				const unsigned g_m = (unsigned)(n_m < (size_t)med_ctas ? n_m : (size_t)med_ctas);
				if (dbg) {
					wm_anchor_sort_giant_kernel<8, 512, true><<<g_m, WM_GS_THREADS, sizeof(sm_t), st>>>(d_a, d_off, d_big + n_l, (int)n_m, d_wl, dbg, d_tmp, d_idx, d_scr_m, two_min, token_min);
					unsigned long long h[16];
					WM_CUDA_CHECK(cudaStreamSynchronize(st));
					WM_CUDA_CHECK(cudaMemcpy(h, dbg, 128, cudaMemcpyDeviceToHost));
					fprintf(stderr, dbg_fmt, (int)n_m, h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], h[9]);
					cudaFree(dbg);
				} else wm_anchor_sort_giant_kernel<8, 512, false><<<g_m, WM_GS_THREADS, sizeof(sm_t), st>>>(d_a, d_off, d_big + n_l, (int)n_m, d_wl, 0, d_tmp, d_idx, d_scr_m, two_min, token_min);
			} else wm_anchor_sort_big_kernel<<<(unsigned)n_m, 32, cap_m * sizeof(wm128_dev), st>>>(d_a, d_off, d_big + n_l, (int)n_m, d_wl, cap_m);
		}
		if (n_s) { wm_count_launch(); wm_anchor_sort_big_kernel<<<(unsigned)n_s, 32, cap_s * sizeof(wm128_dev), st>>>(d_a, d_off, d_big + n_l + n_m, (int)n_s, d_wl, cap_s); }
		WM_CUDA_CHECK(cudaGetLastError());
	}
}

// Collect sorted anchors for all sketched tasks.  Inputs are the outputs of wm_sketch_run.
// On return: ws->a (anchors), ws->task_a_off (device, n_tasks+1), ws->rep_len, ws->n_mini_pos, ws->mini_pos;
// h_task_a_off (host, n_tasks+1) receives the anchor offsets.
void wm_seed_run(wm_seed_ws *ws, const wm_idx_dev &ix, const wm128_dev *d_mz, const int64_t *d_mz_off, int64_t n_mz, int n_tasks,
                 const int32_t *d_qlen, int max_occ, int64_t *h_task_a_off, cudaStream_t st)
{
	for (int i = 0; i <= n_tasks; ++i) h_task_a_off[i] = 0;
	int64_t *d_task_a_off = (int64_t*)ws->task_a_off.need(sizeof(int64_t) * (n_tasks + 1));
	int32_t *d_rep = (int32_t*)ws->rep_len.need(sizeof(int32_t) * (n_tasks + 1));
	int32_t *d_nmp = (int32_t*)ws->n_mini_pos.need(sizeof(int32_t) * (n_tasks + 1));
	WM_CUDA_CHECK(cudaMemsetAsync(d_task_a_off, 0, sizeof(int64_t) * (n_tasks + 1), st));
	WM_CUDA_CHECK(cudaMemsetAsync(d_rep, 0, sizeof(int32_t) * (n_tasks + 1), st));
	WM_CUDA_CHECK(cudaMemsetAsync(d_nmp, 0, sizeof(int32_t) * (n_tasks + 1), st));
	ws->n_a = 0;
	if (n_tasks <= 0) return;
	int32_t *d_nocc = (int32_t*)ws->n_occ.need(sizeof(int32_t) * (n_mz + 1));
	int32_t *d_cnt = (int32_t*)ws->cnt.need(sizeof(int32_t) * (n_mz + 1));
	uint64_t *d_loff = (uint64_t*)ws->list_off.need(sizeof(uint64_t) * (n_mz + 1));
	uint8_t *d_td = (uint8_t*)ws->tandem.need(n_mz + 1);
	int32_t *d_mtask = (int32_t*)ws->mz_task.need(sizeof(int32_t) * (n_mz + 1));
	int64_t *d_aoff = (int64_t*)ws->a_off.need(sizeof(int64_t) * (n_mz + 2));
	int64_t *d_tmp = (int64_t*)ws->scan_tmp.need(sizeof(int64_t) * wm_scan_tmp_elems(n_mz));
	uint32_t *d_mpos = (uint32_t*)ws->mini_pos.need(sizeof(uint32_t) * (n_mz + 1));
	if (n_mz > 0) {
		wm_count_launch(); wm_seed_lookup_kernel<<<(unsigned)((n_mz + 127) / 128), 128, 0, st>>>(ix, d_mz, d_mz_off, n_tasks, n_mz, max_occ, d_nocc, d_cnt, d_loff, d_td, d_mtask);
		WM_CUDA_CHECK(cudaGetLastError());
	}
	wm_exclusive_scan(d_cnt, n_mz, d_aoff, d_tmp, st);
	int64_t n_a = 0;
	WM_CUDA_CHECK(wm_memcpy_async(&n_a, d_aoff + n_mz, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
	wm_stream_sync(st);
	ws->n_a = n_a;
	wm128_dev *d_a = (wm128_dev*)ws->a.need(sizeof(wm128_dev) * (n_a + 1));
	if (n_a > 0) {
		wm_count_launch(); wm_seed_expand_kernel<<<(unsigned)((n_a + 127) / 128), 128, 0, st>>>(ix, d_mz, n_mz, d_aoff, d_loff, d_td, d_mtask, d_qlen, n_a, d_a);
		WM_CUDA_CHECK(cudaGetLastError());
	}
	wm_count_launch(); wm_seed_task_kernel<<<(n_tasks + 1 + 127) / 128, 128, 0, st>>>(d_mz, d_mz_off, d_aoff, d_nocc, max_occ, n_tasks, d_rep, d_nmp, d_task_a_off, d_mpos);
	WM_CUDA_CHECK(cudaGetLastError());
	WM_CUDA_CHECK(wm_memcpy_async(h_task_a_off, d_task_a_off, sizeof(int64_t) * (n_tasks + 1), cudaMemcpyDeviceToHost, st));
	wm_stream_sync(st);
	wm_anchor_sort_run(ws, d_a, d_task_a_off, h_task_a_off, n_tasks, st);
}

// ---- index upload ----
void wm_idx_dev_build_ht(wm_idx_dev *ix, cudaStream_t st)
{
	uint64_t cap = 1024;
	while (cap < (uint64_t)ix->n_keys * 2) cap <<= 1;
	uint64_t *hk = wm_dev_alloc<uint64_t>(cap);
	uint32_t *hv = wm_dev_alloc<uint32_t>(cap);
	WM_CUDA_CHECK(cudaMemsetAsync(hk, 0xff, cap * 8, st));
	if (ix->n_keys > 0) {
		wm_count_launch(); wm_ht_fill_kernel<<<(unsigned)((ix->n_keys + 255) / 256), 256, 0, st>>>(ix->keys, ix->n_keys, hk, hv, cap - 1);
		WM_CUDA_CHECK(cudaGetLastError());
	}
	ix->ht_key = hk, ix->ht_val = hv, ix->ht_mask = cap - 1;
}

// ---- C ABI: standalone tie-exact sort (for the parity tests and tools/bench_sort.py) ----
extern "C" int wm_radix_sort_128x_batch_timed(int n_arr, wm128_dev *a, const int64_t *off, float *ms)
{
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
		fprintf(stderr, "[ERROR] wm_radix_sort_128x_batch: no CUDA device visible; winnowmap-b200 has no CPU fallback\n");
		exit(1);
	}
	if (n_arr <= 0) return 0;
	const int64_t n = off[n_arr];
	wm128_dev *d_a = wm_dev_alloc<wm128_dev>(n + 1);
	int64_t *d_off = wm_dev_alloc<int64_t>(n_arr + 1);
	WM_CUDA_CHECK(cudaMemcpy(d_a, a, sizeof(wm128_dev) * n, cudaMemcpyHostToDevice));
	WM_CUDA_CHECK(cudaMemcpy(d_off, off, sizeof(int64_t) * (n_arr + 1), cudaMemcpyHostToDevice));
	wm_seed_ws ws;
	cudaEvent_t ev[2];
	if (ms) { WM_CUDA_CHECK(cudaEventCreate(&ev[0])); WM_CUDA_CHECK(cudaEventCreate(&ev[1])); WM_CUDA_CHECK(cudaEventRecord(ev[0], 0)); }
	wm_anchor_sort_run(&ws, d_a, d_off, off, n_arr, 0);
	if (ms) WM_CUDA_CHECK(cudaEventRecord(ev[1], 0));
	WM_CUDA_CHECK(cudaDeviceSynchronize());
	if (ms) { WM_CUDA_CHECK(cudaEventElapsedTime(ms, ev[0], ev[1])); cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]); }
	WM_CUDA_CHECK(cudaMemcpy(a, d_a, sizeof(wm128_dev) * n, cudaMemcpyDeviceToHost));
	ws.release();
	cudaFree(d_a); cudaFree(d_off);
	return 0;
}

extern "C" int wm_radix_sort_128x_batch(int n_arr, wm128_dev *a, const int64_t *off)
{
	return wm_radix_sort_128x_batch_timed(n_arr, a, off, 0);
}
