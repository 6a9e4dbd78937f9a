// fqsk_kernels.cuh -- the kernels of the k-mer statistics engine (sm_100a).  Host orchestration lives in fqsk.cu.
//
// Kernel inventory (DESIGN.md section 4):
//   k_mt_extend        mt19937 block recurrence, one CTA per chunk, state in shared memory (utils.h:257, 298)
//   k_mt_jump          mt19937 jump-ahead: the states j chunks ahead, so that G CTAs extend one stream side by side
//   k_prep             per read: duplicate flag, A/C/G/T totals, number of coded bases  (dna.cpp:1521-1533, 2047-2057)
//   (segment pipeline: k_lookup / k_partial / k_local / k_walk / k_rough / k_fold live in fqsk_pipeline.cuh)
//   k_locate_heads/k_apply_keys/k_commit_keys   InsertKmersToHT for s-/b-mers with ordered PRNG draws   (dna.cpp:2420-2446, ht_kmer.h:420-438)
//   k_siv_increment    InsertKmersToHT for p-mers                                        (dna.cpp:2401-2418)
//   k_find / k_count / k_siv_*   table-level batch mirrors                               (ht_kmer.h:441-510, bit_vec.h:53-123)
#pragma once
#include <cstddef>
#include "fqsk_dev.cuh"
#include "fqsk_sort.cuh"
#include "../../include/fqsk.h"

namespace fqsk {

struct U64x4 {
	unsigned long long v[4];
	__host__ __device__ U64x4 operator+(const U64x4 &o) const { U64x4 r; for (int i = 0; i < 4; ++i) r.v[i] = v[i] + o.v[i]; return r; }
};

// ------------------------------------------------------------------------------------------------------------------
// mt19937: extend a stream by n_blocks x 624 tempered outputs.  state[0..623] in HBM between launches.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mt_twist(uint32_t a, uint32_t b, uint32_t far) {
	uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
	return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}
// Double-buffered: the three phases of a block read the previous state from one array and write the new one into the other, so
// only the 3 true dependencies between the phases need a barrier (an in-place version needs 7 per block),
// and every thread tempers and stores the word it has just produced.  One CTA is bound by the recurrence's dependency distance
// (227 words): ~2 G outputs/s.  Late in a file the b-mer counters consume ~6 M draws per 51 000-read block, so long extensions
// run as G chunks side by side: CTA j starts from the state j chunks ahead (states[j], from k_mt_jump) and writes its own
// n_blocks x 624 outputs; the last CTA leaves the state the next launch continues from.  gridDim.x == 1: the plain sequential form.
__global__ void __launch_bounds__(256) k_mt_extend(uint32_t *state, const uint32_t *states, uint32_t *ring, unsigned long long mask, unsigned long long pos, uint32_t n_blocks) {
	__shared__ uint32_t st[2][624];
	const int t = threadIdx.x;
	const uint32_t *src = gridDim.x > 1 ? states + 624u * blockIdx.x : state;
	pos += (unsigned long long) blockIdx.x * n_blocks * 624ull;
	for (int i = t; i < 624; i += 256) st[0][i] = src[i];
	__syncthreads();
	int cur = 0;
	for (uint32_t blk = 0; blk < n_blocks; ++blk) {
		const uint32_t *o = st[cur];
		uint32_t *nw = st[cur ^ 1];
		const unsigned long long base = pos + (unsigned long long) blk * 624;
		auto emit = [&](int i, uint32_t v) {
			nw[i] = v;
			uint32_t y = v;
			y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
			ring[(base + i) & mask] = y;
		};
		if (t < 227) emit(t, mt_twist(o[t], o[t + 1], o[t + 397]));                                   // i in [0, 227): old i, i+1, i+397
		__syncthreads();
		if (t < 227) emit(t + 227, mt_twist(o[t + 227], o[t + 228], nw[t]));                          // i in [227, 454): old i, i+1, NEW i-227
		__syncthreads();
		if (t < 170) { const int i = t + 454; emit(i, mt_twist(o[i], i == 623 ? nw[0] : o[i + 1], nw[i - 227])); }   // i in [454, 624)
		__syncthreads();
		cur ^= 1;
	}
	if (blockIdx.x == gridDim.x - 1) for (int i = t; i < 624; i += 256) state[i] = st[cur][i];
}

// mt19937 jump-ahead (fqsk_mtjump.h): CTA j writes states[j] = the generator's state j chunks ahead of `state`, as the GF(2)
// combination XOR_{i : g_i = 1} x[i + t] of the next 19937 + 623 raw words, g = x^(j chunk) mod the characteristic polynomial
// (polys[j - 1]).  CTA 0 copies the state itself.  Dynamic shared memory: (624 + 33 * 624) words.
static const uint32_t MT_JUMP_WORDS = 624 + 33 * 624;
__global__ void __launch_bounds__(640) k_mt_jump(const uint32_t *state, const uint32_t *polys, uint32_t *states) {
	extern __shared__ uint32_t X[];
	const int t = threadIdx.x;
	const uint32_t j = blockIdx.x;
	if (j == 0) { if (t < 624) states[t] = state[t]; return; }
	if (t < 624) X[t] = state[t];
	__syncthreads();
	for (uint32_t blk = 0; blk < 33; ++blk) {      // 33 x 624 = 20 592 >= 19 937 + 623 new words
		const uint32_t *o = X + blk * 624;
		uint32_t *nw = X + (blk + 1) * 624;
		if (t < 227) nw[t] = mt_twist(o[t], o[t + 1], o[t + 397]);
		__syncthreads();
		if (t < 227) nw[t + 227] = mt_twist(o[t + 227], o[t + 228], nw[t]);
		__syncthreads();
		if (t < 170) { const int i = t + 454; nw[i] = mt_twist(o[i], i == 623 ? nw[0] : o[i + 1], nw[i - 227]); }
		__syncthreads();
	}
	if (t >= 624) return;
	const uint32_t *g = polys + (size_t) (j - 1) * 624;
	uint32_t acc0 = 0, acc1 = 0;
	for (uint32_t w = 0; w < 624; ++w) {
		uint32_t bits = __ldg(g + w);
		const uint32_t *xb = X + w * 32 + t;
		while (bits) {
			const uint32_t i = __ffs(bits) - 1; bits &= bits - 1;
			acc0 ^= xb[i];
			if (bits) { const uint32_t i2 = __ffs(bits) - 1; bits &= bits - 1; acc1 ^= xb[i2]; }
		}
	}
	states[624u * j + t] = acc0 ^ acc1;
}

// ------------------------------------------------------------------------------------------------------------------
// engine-wide device view
// ------------------------------------------------------------------------------------------------------------------
struct EngineDev {
	HtDev hb, hs;
	SivDev siv;
	CIncP cib, cis;                 // cinc_b / cinc_s; the local incrementers have the same parameters (dna.cpp:162-165)
	uint32_t p, s, b, prefix_len, sorted;
	uint32_t gate_missing;          // siv_pmer->avg_filling_factor() >= 7.0 (dna.cpp:376), constant inside a segment
	const uint32_t *draws[4];       // ring buffers of the streams cinc_b, cinc_s, cinc_lb, cinc_ls
	unsigned long long dmask[4], dpos[4], avail[4];   // ring size - 1, absolute consumed position, outputs available beyond it
	int *flags;                     // [0] draw window overflow, [1] unsupported path, [2] changed, [3] scratch
};

struct Carry {             // state a segment hands to the next one without a host round trip (k_seg_tail)
	uint32_t prev_len;     // read_prev.size(), 0 after ResetReadPrev (application.cpp:624)
	uint32_t pprev_valid;
	unsigned long long pprev_dir;   // pmer_can_prev (dna.cpp:167, 655): prefix p-mer of the last read, left-aligned
};

struct SyncIn {             // inputs of a sync that only the device knows when the sync is enqueued right behind its segment
	uint32_t ok;            // the segment settled on its first pass (k_seg_tail); 0 = every sync kernel is a no-op
	uint32_t n_b, n_s, n_p; // rows to apply (dna.cpp:2401-2446)
	unsigned long long dpos_b, dpos_s;   // absolute positions of the cinc_b / cinc_s streams after the segment's lookups
	uint32_t draws_b;       // out: mt19937 outputs consumed by the b-mer inserts of this sync
	uint32_t ok_pre;        // walk-level verdict (k_pre_verdict): the pushes are final, so the grouping half of the b-mer sync may run
	                        // next to the rough searches and merges; `ok` (k_seg_tail) additionally needs the merges to have settled
};

struct SegTotals {        // written by k_scan_reads, read by the host once per segment
	unsigned long long n_rec; U64x4 letters;
};

// The small device words of an engine's host-side control, in one allocation.  The host reads all of them with one look
// (k_publish) into a page-locked mirror of the same type; a copy of a single field lands in that field's mirror.
// "Per prep instance": indexed by the parity of fqsk_announce_device's double buffering (seg_par).
struct EngineStatus {
	int flags[8];                        // PipeDev::flags of the segment's passes; also the flags of the table-level inserts
	uint32_t n_miss, n_rscript, pool_used;   // list lengths of the segment (PipeDev)
	uint32_t n_rec[2];                   // coded positions of the segment (k_scan_reads), per prep instance
	struct { uint32_t ev[2], draws[2]; } hot;   // hot mode, per thread-local stream (cinc_lb, cinc_ls): queued events, draws consumed
	uint32_t row_tot[4];                 // rows b, s, p and the hidden p-mer updates of the segment (k_scan_u32x4)
	unsigned long long draws[2];         // draws of the segment's merges, streams b / s (k_scan_draws)
	SegTotals totals[2];                 // per prep instance (k_scan_reads)
	Carry carry;                         // written by k_seg_tail
	SyncIn syncin;                       // the sync enqueued behind its segment
	SyncIn syncin2;                      // a plain ordered insert (apply_indexed)
	int sflags[8];                       // ordered insert: [0] window short [2] flag corrected [6] hot k-mer [7] group too large
	int sfast;                           // the s-mer fast path saw a counter above thr
	int stash_full;                      // a table's stash ran full (HtDev::err, sticky)
	int wait_err;                        // sharded sync: a peer did not post in time (k_wait_seq / k_wait_applied)
	int rank_flags[8];                   // flags of k_delta_rank when it only counts (hot_rank): nothing reads them
	unsigned long long items[4];         // HtDev::n_items: [0, 1] b-mer table main / stash, [2, 3] s-mer table
	unsigned long long siv_fresh;        // p-mer fields that became non-zero (k_siv_increment)
	unsigned long long dump_n;           // entries a table dump wrote
	unsigned long long scratch[2];       // totals of the table-level k_find scan; the record checksum
	struct { uint32_t used; int overflow; } pe_pool;   // paired end: candidate pool of k_pe_decide (`used` also counts k_pair_heads)
	uint32_t pe_scan[4];                 // paired end: totals of the work-item scan
	unsigned long long pair_items;       // paired end: items in the pair table
};
static_assert(sizeof(Carry) == 16 && sizeof(SyncIn) == 40 && sizeof(SegTotals) == 40, "status block members");
static_assert(sizeof(EngineStatus) % 4 == 0, "k_publish copies the status block word by word");
static_assert(offsetof(EngineStatus, items) % 8 == 0 && offsetof(EngineStatus, siv_fresh) % 8 == 0 && offsetof(EngineStatus, dump_n) % 8 == 0 &&
              offsetof(EngineStatus, scratch) % 8 == 0 && offsetof(EngineStatus, pair_items) % 8 == 0, "64-bit atomics need 8-byte alignment");

struct SegDev {
	const uint8_t *dna; const unsigned long long *off; const uint32_t *len; uint32_t n_reads;
	const uint8_t *prev_read;                         // last read of the previous segment of this block (read_prev, dna.cpp:1550)
	const struct Carry *carry;                        // its length and pmer_can_prev, kept on the device between segments
	uint8_t *dup; uint32_t *n_coded; U64x4 *letters;  // k_prep outputs
	const unsigned long long *rec_off; const U64x4 *sl_prefix; U64x4 sl_base;
	fqsk_base_rec *recs;
	unsigned long long *push_b, *push_s, *push_p;     // per-read regions: b at 2*off, s at off, p at 2*off + 2*r
	uint32_t *cnt_b, *cnt_s, *cnt_p, *hidden;
	U64x4 *draw_cnt; const U64x4 *draw_guess;
	const uint32_t *base_b, *base_s;                  // push-index base of every read in the delta's numbering
	DeltaDev delta_b, delta_s;
	uint32_t *sorted_flag; unsigned long long *sorted_dif;
	// paired-end: the "reads" of the segment are work ITEMS (mate 1, mate 2 or its forward part, its reversed part), each with its
	// own first coded position, position bias and flags; all null for single-end segments
	const uint32_t *first_a, *bias_a, *dup_prev; const uint8_t *iflags;
	// 2-bit packed symbols of every read (N -> A, in a sorted prefix N -> T: dna.cpp:532-536 / 560-565 / 684), written by k_prep:
	// read r starts at word (off[r] >> 5) + 2 r and has one word of slack.  The registers of a position are two 64-bit loads.
	unsigned long long *pk;
};
__device__ __forceinline__ unsigned long long *pk_of(const SegDev &S, uint32_t r) { return S.pk + (S.off[r] >> 5) + 2ull * r; }
enum : uint8_t {
	IF_SKIP = 1,          // empty slot (a mate 2 coded in one piece has no reversed part)
	IF_NO_DUPCHECK = 2,   // only first-of-pair reads are compared with read_prev (dna.cpp:1523)
	IF_SEEDED = 4,        // registers seeded from a minimizer (dna.cpp:1579-1594, 1616-1631): no cor_pos from Ns in the preload
	IF_NO_LETTERS = 8,    // right part of a split mate 2: update_s_letters runs once, after the left part (dna.cpp:1635)
	IF_LETTERS_PREV = 16, // left part of a split mate 2: its own symbols plus those of the previous item beyond the shared b-mer
	IF_REVCOMP = 32,      // text = reverse complement of the source range (dna.cpp:1598-1602)
	IF_SORTED = 64,       // paired end in sorted order: first mate, coded by CompressSorted (dna.cpp:1793-1796); the second mate is not
};
__device__ __forceinline__ uint32_t item_first(const SegDev &S, uint32_t dflt, uint32_t r) { return S.first_a ? S.first_a[r] : dflt; }
__device__ __forceinline__ uint32_t item_flags(const SegDev &S, uint32_t r) { return S.iflags ? S.iflags[r] : 0u; }
// is read / item r coded by CompressSorted?  single-end sorted order: every read; paired-end sorted order: the first mates only
__device__ __forceinline__ bool item_sorted(const SegDev &S, uint32_t sorted_mode, uint32_t r) { return sorted_mode && (!S.iflags || (S.iflags[r] & IF_SORTED)); }

__device__ __forceinline__ uint32_t dna_code(uint8_t ch) {  // dna.cpp:18-23
	return ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'G' ? 2u : ch == 'T' ? 3u : 4u;
}

// the status words a segment starts from zero: k_prep clears them for the first evaluation of a segment, k_seg_reset for a retry.
// n_rec and totals are not among them: k_scan_reads may have written them ahead of the segment (fqsk_announce_device).
__device__ __forceinline__ void seg_reset_words(EngineStatus *st, uint32_t t) {
	if (t < 8) { st->flags[t] = 0; st->sflags[t] = 0; }
	if (t < 2) { st->hot.ev[t] = 0; st->hot.draws[t] = 0; }
	if (t == 8) { st->n_miss = 0; st->n_rscript = 0; st->pool_used = 0; }
	if (t == 9) st->sfast = 0;
	if (t == 10) st->siv_fresh = 0;
}
// pv_*: read_prev of the segment's first read when it is not the engine's own copy (fqsk_announce_device: the last read of the segment in flight)
__global__ void __launch_bounds__(128) k_prep(SegDev S, uint32_t first_len_bytes, uint32_t b, uint32_t sorted, EngineStatus *status,
                                              const uint8_t *pv_dna, const unsigned long long *pv_off, const uint32_t *pv_len) { pdl_enter();   // one warp per read
	if (status && blockIdx.x == 0 && threadIdx.x < 32) seg_reset_words(status, threadIdx.x);
	uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (r >= S.n_reads) return;
	const uint8_t *p = S.dna + S.off[r];
	uint32_t n = S.len[r];
	const uint32_t ifl = item_flags(S, r);
	first_len_bytes = item_first(S, first_len_bytes, r);
	sorted = item_sorted(S, sorted, r);
	const uint8_t *q; uint32_t qn;
	uint32_t pr = S.dup_prev ? S.dup_prev[r] : (r ? r - 1 : 0xFFFFFFFFu);     // the read this one is compared with (read_prev)
	if (pr == 0xFFFFFFFFu) { if (pv_off) { q = pv_dna + *pv_off; qn = *pv_len; } else { q = S.prev_read; qn = S.carry->prev_len; } } else { q = S.dna + S.off[pr]; qn = S.len[pr]; }
	bool same = qn == n && !(ifl & IF_NO_DUPCHECK);
	if (ifl & IF_SKIP) { same = true; n = 0; }
	uint32_t cnt[4] = {0, 0, 0, 0};
	unsigned long long *pkr = pk_of(S, r);
	for (uint32_t i0 = 0; i0 < n; i0 += 32) {
		const uint32_t i = i0 + lane;
		uint32_t c2 = 0;
		if (i < n) {
			uint8_t ch = p[i];
			if (same && q[i] != ch) same = false;
			uint32_t c = dna_code(ch);
			if (c < 4) { ++cnt[c]; ++cnt[3 - c]; }
			c2 = c < 4 ? c : ((sorted && i < first_len_bytes) ? 3u : 0u);
		}
		const unsigned b1 = __ballot_sync(0xffffffffu, c2 & 2u), b0 = __ballot_sync(0xffffffffu, c2 & 1u);
		if (lane == 0) pkr[i0 >> 5] = pk_from_ballots(b1, b0);
	}
	if (lane == 0) pkr[(n + 31) >> 5] = 0;     // the word of slack pk_window reads
	same = __all_sync(0xffffffffu, same);
	if (ifl & IF_LETTERS_PREV) {      // symbol + complement are counted (dna.cpp:2047-2057), so the reversed text counts like the original
		const uint8_t *pp = S.dna + S.off[r - 1];
		const uint32_t pn = S.len[r - 1];
		for (uint32_t i = b + lane; i < pn; i += 32) { uint32_t c = dna_code(pp[i]); if (c < 4) { ++cnt[c]; ++cnt[3 - c]; } }
	}
	for (int k = 0; k < 4; ++k) for (int o = 16; o; o >>= 1) cnt[k] += __shfl_xor_sync(0xffffffffu, cnt[k], o);
	if (lane == 0) {
		S.dup[r] = same;
		U64x4 L; for (int k = 0; k < 4; ++k) L.v[k] = (same || (ifl & IF_NO_LETTERS)) ? 0 : cnt[k];
		S.letters[r] = L;
		S.n_coded[r] = (!same && n > first_len_bytes) ? n - first_len_bytes : 0;
	}
}

// ------------------------------------------------------------------------------------------------------------------
// CHT_kmer::find (ht_kmer.h:504-510): full context -> one sector; front-truncated context -> 4^m completions in odometer
// order merged with the PRNG-aware addition (ht_kmer.h:266-327).  Lookups are issued 4 at a time for memory parallelism.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool any4(const uint32_t c[4]) { return (c[0] | c[1] | c[2] | c[3]) != 0; }

__device__ __forceinline__ KReg partial_trial(const KReg &r, uint32_t k, uint32_t m, uint32_t n) {
	uint32_t rev = 0;
	for (uint32_t j = 0; j < m; ++j) rev |= ((n >> (2 * j)) & 3u) << (2 * (m - 1 - j));
	KReg t;
	t.dir = (r.dir >> (2 * m)) | ((uint64_t) rev << (64 - 2 * m));
	t.rc = r.rc + ((uint64_t) (((1u << (2 * m)) - 1u) - n) << (64 - 2 * k));
	return t;
}

__device__ bool ht_find(const HtDev &t, const CIncP &ci, const KReg &r, uint32_t cur, uint32_t c[4], DrawCursor &dc) {
	c[0] = c[1] = c[2] = c[3] = 0;
	if (cur >= t.k) {
		bool d = kr_is_dir(r, t.k);
		ht_ctx_counts(t, d ? r.dir : r.rc, d, c);
		return any4(c);
	}
	uint32_t m = t.k - cur, trials = 1u << (2 * m);
	for (uint32_t n0 = 0; n0 < trials; n0 += 4) {
		HtKey key[4]; Bucket bk[4]; bool isd[4];
#pragma unroll
		for (int u = 0; u < 4; ++u) {
			KReg tr = partial_trial(r, t.k, m, n0 + u);
			isd[u] = kr_is_dir(tr, t.k);
			key[u] = ht_key(t, isd[u] ? tr.dir : tr.rc);
			bk[u] = ht_load_bucket(t, key[u]);
		}
#pragma unroll
		for (int u = 0; u < 4; ++u) {
			uint32_t loc[4] = {0, 0, 0, 0};
			ht_ctx_counts_from(t, key[u], isd[u], bk[u], loc);
			for (int i = 0; i < 4; ++i) if (loc[i]) c[i] = ci_plus(ci, c[i], loc[i], dc);
		}
	}
	return any4(c);
}

// ------------------------------------------------------------------------------------------------------------------
// per-read register state shared by the pipeline kernels
// ------------------------------------------------------------------------------------------------------------------
struct ReadState {
	KReg pc, sc, bc, pu, su, bu;
	uint32_t n;          // symbols pushed since the registers were reset
	uint32_t cor_pos, n_run;
};

__device__ __forceinline__ void rs_push_all(ReadState &R, const EngineDev &E, uint64_t s) {
	kr_push(R.pc, E.p, R.n, s); kr_push(R.sc, E.s, R.n, s); kr_push(R.bc, E.b, R.n, s);
	kr_push(R.pu, E.p, R.n, s); kr_push(R.su, E.s, R.n, s); kr_push(R.bu, E.b, R.n, s);
	++R.n;
}
__device__ __forceinline__ uint32_t cur_of(uint32_t k, uint32_t n) { return n < k ? n : k; }

__global__ void k_compare_u64(const unsigned long long *a, const unsigned long long *b, uint64_t n, int *changed) { pdl_enter();
	uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n && a[i] != b[i]) *changed = 1;
}
__global__ void k_compare_u32(const uint32_t *a, const uint32_t *b, uint64_t n, int *changed) { pdl_enter();
	uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n && a[i] != b[i]) *changed = 1;
}
__global__ void k_iota(uint32_t *a, uint32_t n) { pdl_enter(); uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) a[i] = i; }

// ------------------------------------------------------------------------------------------------------------------
// sync step for one hash table: InsertKmersToHT (dna.cpp:2420-2446) == for every pushed k-mer, in push order,
// CHT_kmer::insert(x, cinc) (ht_kmer.h:420-438).
// ------------------------------------------------------------------------------------------------------------------
// Input: the row sorted by k-mer (stable, so equal k-mers stay in push order) with the push index of every occurrence.
// k_locate_heads: one find-or-create per DISTINCT k-mer; it also sizes the group, reads the counter before the sync (c0) and
// writes the draw flag of every member in push order (pre-count c0 + r > thr, the counter cannot move otherwise below top).
// Groups that cannot reach the top of the counter (c0 + m < top) are final with those flags; the others are marked unsafe
// and go through the verifying passes (k_apply_keys with verify = 1) -- only there can a flag be wrong.
__global__ void k_locate_heads(HtDev t, CIncP ci, const unsigned long long *skeys, const uint32_t *sidx, uint32_t n, unsigned long long *slot_of, uint32_t *c0_of,
                               uint8_t *flag, int *flags) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	unsigned long long key = skeys[i];
	if (i > 0 && skeys[i - 1] == key) return;   // not a group head
	bool created;
	uint64_t s = ht_locate(t, key, created);
	uint32_t c0 = created ? 0u : ht_slot_get(t, s);
	uint32_t m = 0;
	for (uint32_t q = i; q < n && skeys[q] == key; ++q, ++m) flag[sidx[q]] = (c0 + m > ci.thr) ? 1 : 0;
	bool unsafe = c0 + m >= t.top;
	if (unsafe) flags[3] = 1;
	if (m > ci.thr + 1) flags[6] = 1;           // the thread-local table of the reference drew from its own stream for this k-mer
	slot_of[i] = s | (unsafe ? (1ull << 63) : 0ull);
	c0_of[i] = c0;
}
// k_apply_keys: one thread per group walks its occurrences in push order and applies Increment() with the scanned draw
// indices.  verify == 0: only safe groups, the final counter is written straight to the table (blind write: the item's key
// bits are known).  verify == 1: only unsafe groups; flags are checked against the counters seen (a counter reaching the
// top stops drawing, ht_kmer.h:435), a mismatch is corrected and reported (flags[2]); nothing is written until the host has
// seen a pass without corrections (commit == 1).
__global__ void k_apply_keys(HtDev t, CIncP ci, const unsigned long long *skeys, const uint32_t *sidx, uint32_t n, const unsigned long long *slot_of, const uint32_t *c0_of,
                             uint8_t *flag, const uint32_t *draw_off, const uint32_t *draws, unsigned long long dmask, unsigned long long dpos, unsigned long long avail,
                             int verify, int commit, int *flags) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	unsigned long long key = skeys[i];
	if (i > 0 && skeys[i - 1] == key) return;
	unsigned long long so = slot_of[i];
	const bool unsafe = (so >> 63) != 0;
	if (unsafe != (verify != 0)) return;
	uint32_t c = c0_of[i];
	for (uint32_t q = i; q < n && skeys[q] == key; ++q) {
		uint32_t j = sidx[q];
		if (verify) {
			uint8_t want = (c < t.top && c > ci.thr) ? 1 : 0;
			if (flag[j] != want) { flag[j] = want; flags[2] = 1; if (c <= ci.thr) ++c; continue; }
		}
		if (c >= t.top) continue;                  // ht_kmer.h:435: cnt < counter_max
		if (c <= ci.thr) { ++c; continue; }
		uint32_t di = draw_off[j];
		if (di >= avail) { flags[0] = 1; continue; }
		if (draws[(dpos + di) & dmask] % (ci.mult * (c - ci.thr)) == 0) ++c;
	}
	if (verify && !commit) return;
	// blind write of the item: [occupied | rem | ends | counter] resp. [(k-mer + 1) | counter]
	uint64_t slot = so & ~(1ull << 63), nm = 8ull << t.B;
	HtKey hk = ht_key(t, key);
	if (slot < nm) t.main[slot] = hk.q | c; else t.stash[slot - nm] = ((hk.kal + 1) << t.cbits) | c;
}

// ------------------------------------------------------------------------------------------------------------------
// bucket-grouped ordered insert (large rows).  Input: the row partitioned by table BUCKET (stable: push order survives inside a
// bucket's run; fqsk_sort.cuh) with the push index of every element.  One thread per run:
//   k_bucket_flags  reads the bucket's sector once and walks the run in push order with a tiny model of the counters it will
//                   touch: the draw flag of every occurrence is (counter before it > thr) -- exact as long as no counter can
//                   reach the top inside the row, which the kernel checks (flags[3]) -- read-only;
//   (k_scan_u8: flags in push order -> absolute draw indices)
//   k_bucket_apply  walks the run again with the draws, creates missing items in the free slots of the same sector (stash when
//                   the bucket is full) and writes the sector back once: one 32-byte read + one 32-byte write per touched
//                   bucket instead of find-or-create + read-modify-write per k-mer through the sorted-by-k-mer path.
// Runs with more than BUCKET_RUN_KEYS distinct k-mers, or rows in which a counter may saturate, are left to that path
// (flags[3] / flags[7]: nothing has been written yet when the host sees them).
// ------------------------------------------------------------------------------------------------------------------
static const int BUCKET_RUN_KEYS = 12;
struct BucketRun {
	unsigned long long key[BUCKET_RUN_KEYS];
	uint32_t cnt[BUCKET_RUN_KEYS], c0[BUCKET_RUN_KEYS], m[BUCKET_RUN_KEYS];      // running counter, counter before the row, occurrences in the row
	int8_t slot[BUCKET_RUN_KEYS];      // item of the bucket (0..7), -1: not in the bucket yet, -2: lives in the stash
	int n;
};
__device__ __forceinline__ uint64_t ht_bucket_of(const HtDev &t, unsigned long long x) { return ht_mix(t, ht_kernel(t, x)) >> t.rem_bits; }
// entry of k-mer x in the run's model; created from the table's present contents on first sight.  -1: model full
__device__ __forceinline__ int bucket_run_entry(const HtDev &t, BucketRun &R, const uint32_t it[8], unsigned long long x) {
	for (int j = 0; j < R.n; ++j) if (R.key[j] == x) return j;
	if (R.n >= BUCKET_RUN_KEYS) return -1;
	const HtKey hk = ht_key(t, x);
	const int j = R.n++;
	R.key[j] = x; R.m[j] = 0; R.cnt[j] = 0; R.c0[j] = 0; R.slot[j] = -1;
	bool full = true;
#pragma unroll
	for (int i = 0; i < 8; ++i) {
		if (it[i] == 0) { full = false; break; }
		if ((it[i] & ~t.top) == hk.q) { R.cnt[j] = R.c0[j] = it[i] & t.top; R.slot[j] = (int8_t) i; return j; }
	}
	if (full) {      // the k-mer may live in the stash
		const uint64_t smask = (1ull << t.stash_log2) - 1;
		for (uint64_t p = ht_stash_pos(t, hk.h), guard = 0; guard <= smask; p = (p + 1) & smask, ++guard) {
			const unsigned long long s = t.stash[p];
			if (s == 0) break;
			if ((s >> t.cbits) == hk.kal + 1) { R.cnt[j] = R.c0[j] = (uint32_t) (s & t.top); R.slot[j] = -2; break; }
		}
	}
	return j;
}
__global__ void __launch_bounds__(256) k_bucket_flags(HtDev t, CIncP ci, const unsigned long long *skeys, const uint32_t *sidx, uint32_t n, uint8_t *flag, int *flags) { pdl_enter();
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const unsigned long long x0 = skeys[i];
	const uint64_t bucket = ht_bucket_of(t, x0);
	if (i > 0 && ht_bucket_of(t, skeys[i - 1]) == bucket) return;      // not the head of a run
	const uint4 *bp = reinterpret_cast<const uint4 *>(t.main + bucket * 8);
	const uint4 lo = __ldg(bp), hi = __ldg(bp + 1);
	const uint32_t it[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
	BucketRun R; R.n = 0;
	for (uint32_t q = i; q < n; ++q) {
		const unsigned long long x = skeys[q];
		if (q > i && ht_bucket_of(t, x) != bucket) break;
		const int j = bucket_run_entry(t, R, it, x);
		if (j < 0) { flags[7] = 1; return; }
		const uint32_t c = R.cnt[j];
		flag[sidx[q]] = c > ci.thr ? 1 : 0;
		if (c <= ci.thr) R.cnt[j] = c + 1;      // above thr the counter stays above thr: all the flags need to know
		++R.m[j];
	}
	for (int j = 0; j < R.n; ++j) {
		if (R.c0[j] + R.m[j] >= t.top) flags[3] = 1;       // a counter could reach the top inside the row: the flags above may be wrong
		if (R.m[j] > ci.thr + 1) flags[6] = 1;             // the thread-local table of the reference drew from its own stream for this k-mer
	}
}
__global__ void __launch_bounds__(256) k_bucket_apply(HtDev t, CIncP ci, const unsigned long long *skeys, const uint32_t *sidx, uint32_t n, const uint32_t *draw_off,
                                                     const uint32_t *draws, unsigned long long dmask, unsigned long long dpos, unsigned long long avail, int *flags) { pdl_enter();
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	if (flags[3] | flags[7]) return;      // the row goes through the sorted-by-k-mer path: nothing may be written here
	const unsigned long long x0 = skeys[i];
	const uint64_t bucket = ht_bucket_of(t, x0);
	if (i > 0 && ht_bucket_of(t, skeys[i - 1]) == bucket) return;
	uint4 *bp = reinterpret_cast<uint4 *>(t.main + bucket * 8);
	const uint4 lo = bp[0], hi = bp[1];
	uint32_t it[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
	BucketRun R; R.n = 0;
	for (uint32_t q = i; q < n; ++q) {
		const unsigned long long x = skeys[q];
		if (q > i && ht_bucket_of(t, x) != bucket) break;
		const int j = bucket_run_entry(t, R, it, x);
		if (j < 0) return;      // cannot happen: k_bucket_flags saw the same run
		uint32_t c = R.cnt[j];
		++R.m[j];
		if (c >= t.top) continue;                  // ht_kmer.h:435: cnt < counter_max
		if (c <= ci.thr) { R.cnt[j] = c + 1; continue; }
		const uint32_t di = draw_off[sidx[q]];
		if (di >= avail) { flags[0] = 1; continue; }
		if (draws[(dpos + di) & dmask] % (ci.mult * (c - ci.thr)) == 0) R.cnt[j] = c + 1;
	}
	// write the counters back: existing items in place, new k-mers into the free slots of the sector, the rest into the stash
	uint32_t made_main = 0, made_stash = 0;
	const bool was_empty = it[0] == 0;
	for (int j = 0; j < R.n; ++j) {
		const HtKey hk = ht_key(t, R.key[j]);
		if (R.slot[j] >= 0) { it[R.slot[j]] = hk.q | R.cnt[j]; continue; }
		if (R.slot[j] == -1) {
			int f = -1;
#pragma unroll
			for (int s = 0; s < 8; ++s) if (f < 0 && it[s] == 0) f = s;
			if (f >= 0) { it[f] = hk.q | R.cnt[j]; ++made_main; continue; }
		}
		// stash: find-or-create (another bucket's thread may claim slots next to ours)
		const uint64_t smask = (1ull << t.stash_log2) - 1;
		const unsigned long long item = ((hk.kal + 1) << t.cbits) | (unsigned long long) R.cnt[j];
		uint64_t probes = 0;
		for (uint64_t p = ht_stash_pos(t, hk.h);; p = (p + 1) & smask) {
			if (++probes > smask) { if (t.err) *t.err = 1; break; }      // stash full: the host fails the call
			unsigned long long s = *((volatile unsigned long long *) (t.stash + p));
			if (s == 0) {
				const unsigned long long old = atomicCAS(t.stash + p, 0ull, item);
				if (old == 0) { ++made_stash; break; }
				s = old;
			}
			if ((s >> t.cbits) == hk.kal + 1) { t.stash[p] = item; break; }
		}
	}
	bp[0] = make_uint4(it[0], it[1], it[2], it[3]);
	bp[1] = make_uint4(it[4], it[5], it[6], it[7]);
	if (made_main) atomicAdd(t.n_items, (unsigned long long) made_main);
	if (made_stash) atomicAdd(t.n_items + 1, (unsigned long long) made_stash);
	if (t.occ && was_empty && it[0] != 0) atomicOr(t.occ + (bucket >> 5), 1u << (bucket & 31));
}

// ------------------------------------------------------------------------------------------------------------------
// sort-free ordered insert: the segment's delta table already holds every push as (k-mer, push time) with all entries of
// one k-mer in one probe run, so an occurrence gets its group size m and its exact push-order rank from that run.
//   k_sync_rank   per occurrence: m, rank, own / leader entry; the leader (rank 0) does the ONE find-or-create of the group
//   k_sync_flags  per occurrence: cold group (c0 + m <= thr + 1: all increments deterministic) -> leader records c0 + m;
//                 hot group -> draw flag in push order (pre-count c0 + rank > thr)
//   (exclusive scan of the flags = absolute draw indices in push order)
//   (k_scan_flags, fqsk_pipeline.cuh, also leaves every hot occurrence's draw index / flag at its delta entry)
//   k_sync_apply  per hot leader: members in time order, Increment() with the scanned draws; verifies the flags against the
//                 counters it sees (they differ only when a counter saturates inside the batch) and reports a change
// ------------------------------------------------------------------------------------------------------------------
struct SyncDev {
	DeltaDev D;
	const SyncIn *in; const uint32_t *n_dev; const unsigned long long *dpos_dev; uint32_t *total_draws;
	unsigned long long *lead_tslot; uint32_t *lead_c0, *lead_m, *draw_at, *j_at, *final_at; uint8_t *flag_at;   // per delta slot
	uint32_t *own, *lead, *rank; uint8_t *flag; const uint32_t *draw_off;                                       // per occurrence
	int *flags;   // [2] changed, [0] draw window short, [7] a hot group is too large for the in-thread path
};
static const uint32_t SYNC_GROUP_CAP = 48;

__global__ void k_sync_rank(HtDev t, SyncDev Y, const unsigned long long *row, const uint32_t *rt) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (!Y.in->ok_pre || j >= *Y.n_dev) return;
	const unsigned long long x = row[j];
	const uint32_t tm = rt[j];
	uint32_t m = 0, rank = 0, own = 0xFFFFFFFFu, lead = 0xFFFFFFFFu, lead_t = 0xFFFFFFFFu;
	for (uint64_t slot = delta_slot_of_key(x, Y.D.k, Y.D.t, Y.D.mask);; slot = (slot + 1) & Y.D.mask) {
		uint32_t et = Y.D.times[slot];
		if (et == DELTA_EMPTY) break;
		if (Y.D.keys[slot] != x) continue;
		++m;
		if (et < tm) ++rank;
		if (et == tm) own = (uint32_t) slot;
		if (et < lead_t) { lead_t = et; lead = (uint32_t) slot; }
	}
	Y.own[j] = own; Y.lead[j] = lead; Y.rank[j] = rank;
	Y.j_at[own] = j;
	if (rank == 0) {
		bool created;
		// a new slot is claimed as a zero-count item (== the reference's fresh slot): this kernel may run next to kernels that still
		// read the table for the segment (k_rough), and a zero counter adds nothing to any lookup
		uint64_t ts = ht_locate(t, x, created, 0u);
		Y.lead_tslot[own] = ts | (created ? (1ull << 63) : 0ull);
		Y.lead_c0[own] = created ? 0u : ht_slot_get(t, ts);
		Y.lead_m[own] = m;
	}
}
__global__ void k_sync_flags(HtDev t, CIncP ci, SyncDev Y) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (!Y.in->ok_pre || j >= *Y.n_dev) return;
	const uint32_t L = Y.lead[j], c0 = Y.lead_c0[L], m = Y.lead_m[L], rank = Y.rank[j];
	uint8_t f = 0;
	if (rank == 0 && m > ci.thr + 1) Y.flags[6] = 1;   // the thread-local table of the reference drew from its own stream for this k-mer
	if (c0 + m <= ci.thr + 1) { if (rank == 0) Y.final_at[L] = c0 + m; }    // cold group
	else {
		f = (c0 + rank > ci.thr) ? 1 : 0;
		if (rank == 0 && m > SYNC_GROUP_CAP) Y.flags[7] = 1;
	}
	Y.flag[j] = f;
}
__global__ void k_sync_apply(HtDev t, CIncP ci, SyncDev Y, const unsigned long long *row,
                             const uint32_t *draws, unsigned long long dmask, unsigned long long safe_abs) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (!Y.in->ok || j >= *Y.n_dev) return;
	if (Y.rank[j] != 0) return;
	const unsigned long long dpos = *Y.dpos_dev;
	const unsigned long long avail = safe_abs > dpos ? safe_abs - dpos : 0;
	const uint32_t L = Y.own[j];
	const uint32_t c0 = Y.lead_c0[L], m = Y.lead_m[L];
	const unsigned long long tslot = Y.lead_tslot[L] & ~(1ull << 63);
	// The leader writes the group's final counter right away (no separate commit launch).  If the row turns out not to be settled
	// -- a flag was corrected, the draw window was short, a group is too large -- the host runs this kernel again (it always
	// starts from the stored pre-sync counter c0, so rewriting is idempotent) or restores c0 with k_sync_unclaim and falls back.
	if (c0 + m <= ci.thr + 1) { ht_slot_set(t, tslot, c0 + m); return; }    // cold group: every increment is deterministic
	if (m > SYNC_GROUP_CAP) return;
	// members of the group in time order
	const unsigned long long x = row[j];
	uint32_t mt[SYNC_GROUP_CAP], ms[SYNC_GROUP_CAP];
	uint32_t k = 0;
	for (uint64_t slot = delta_slot_of_key(x, Y.D.k, Y.D.t, Y.D.mask);; slot = (slot + 1) & Y.D.mask) {
		uint32_t et = Y.D.times[slot];
		if (et == DELTA_EMPTY) break;
		if (Y.D.keys[slot] != x) continue;
		uint32_t q = k++;
		while (q > 0 && mt[q - 1] > et) { mt[q] = mt[q - 1]; ms[q] = ms[q - 1]; --q; }
		mt[q] = et; ms[q] = (uint32_t) slot;
	}
	uint32_t c = c0;
	for (uint32_t q = 0; q < k; ++q) {
		const uint32_t ds = ms[q];
		uint8_t fl = Y.flag_at[ds];
		uint8_t want;
		if (c >= t.top) want = 0;                       // ht_kmer.h:435: cnt < counter_max
		else if (c <= ci.thr) want = 0;
		else want = 1;
		if (fl != want) { Y.flag[Y.j_at[ds]] = want; Y.flags[2] = 1; if (c < t.top && c <= ci.thr) ++c; continue; }
		if (c >= t.top) continue;
		if (c <= ci.thr) { ++c; continue; }
		uint32_t di = Y.draw_at[ds];
		if (di >= avail) { Y.flags[0] = 1; continue; }
		if (draws[(dpos + di) & dmask] % (ci.mult * (c - ci.thr)) == 0) ++c;
	}
	Y.final_at[L] = c;
	ht_slot_set(t, tslot, c);
}
// fallback preparation: slots claimed by k_sync_rank (counter 1) become zero-count items, i.e. the reference's fresh slot
__global__ void k_sync_unclaim(HtDev t, SyncDev Y, uint32_t use_pre) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (!(use_pre ? Y.in->ok_pre : Y.in->ok) || j >= *Y.n_dev) return;
	if (Y.rank[j] != 0) return;
	// created slots stay as zero-count items (== the reference's fresh slot); existing ones get their pre-sync counter back
	// (k_sync_apply writes final counters without waiting for the verdict of the whole row)
	unsigned long long ts = Y.lead_tslot[Y.own[j]];
	ht_slot_set(t, ts & ~(1ull << 63), (ts >> 63) ? 0u : Y.lead_c0[Y.own[j]]);
}
// index of a plain row (table-level API): entry time = push index
__global__ void k_row_index_build(unsigned long long *keys, uint32_t *times, uint32_t mask, uint32_t k, uint32_t t, const unsigned long long *row, uint32_t n, uint32_t *rt) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	unsigned long long x = row[j];
	rt[j] = j;
	for (uint64_t slot = delta_slot_of_key(x, k, t, mask);; slot = (slot + 1) & mask)
		if (atomicCAS(times + slot, DELTA_EMPTY, j) == DELTA_EMPTY) { keys[slot] = x; return; }
}

// Fast path of the sync step: every occurrence does find-or-create and one atomic +1.  That equals the reference's ordered
// Increment()s exactly when no counter leaves the deterministic range (pre-count <= thr for every occurrence, utils.h:317-318);
// any occurrence that sees a pre-count above thr raises flags[2] and the host undoes the pass (k_insert_undo: the adds are
// plain arithmetic on the item, so subtracting them restores every bit) and runs the ordered path instead.
__global__ void k_insert_fast(HtDev t, CIncP ci, const unsigned long long *kmers, uint32_t n, uint8_t *added, int *refuted, const SyncIn *in = nullptr) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (in) { if (!in->ok) return; n = in->n_s; }
	if (j >= n) return;
	bool created;
	uint64_t s = ht_locate(t, kmers[j], created);
	added[j] = created ? 2 : 0;     // 2: this occurrence claimed the slot (counter 1 == Increment(0)), 1: it added one, 0: nothing
	if (created) return;
	// +1 unless the counter field is full (a carry would corrupt the key bits other lookups are comparing right now)
	uint64_t nm = 8ull << t.B;
	if (s < nm) {
		uint32_t *p = t.main + s;
		uint32_t old = *((volatile uint32_t *) p);
		for (;;) {
			if ((old & t.top) > ci.thr) { *refuted = 1; if ((old & t.top) >= t.top) return; }
			uint32_t seen = atomicCAS(p, old, old + 1);
			if (seen == old) { added[j] = 1; return; }
			old = seen;
		}
	} else {
		unsigned long long *p = t.stash + (s - nm);
		unsigned long long old = *((volatile unsigned long long *) p);
		for (;;) {
			if ((uint32_t) (old & t.top) > ci.thr) { *refuted = 1; if ((uint32_t) (old & t.top) >= t.top) return; }
			unsigned long long seen = atomicCAS(p, old, old + 1);
			if (seen == old) { added[j] = 1; return; }
			old = seen;
		}
	}
}
__global__ void k_insert_undo(HtDev t, const unsigned long long *kmers, uint32_t n, const uint8_t *added) { pdl_enter();
	uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	bool created;
	uint64_t s = ht_locate(t, kmers[j], created);   // every key exists now
	uint64_t nm = 8ull << t.B;
	if (!added[j]) return;      // met a full counter: nothing to take back
	// an add, or the claim of a new slot (counter 1 -> zero-count item == the reference's fresh slot)
	if (s < nm) atomicSub(t.main + s, 1u); else atomicAdd(t.stash + (s - nm), ~0ull);
}

__global__ void k_siv_increment(SivDev s, const unsigned long long *idx, uint64_t n, unsigned long long *n_new, const SyncIn *in = nullptr) { pdl_enter();
	uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (in) n = in->ok ? in->n_p : 0;
	uint32_t fresh = 0;
	if (i < n) fresh = siv_increment(s, idx[i]);
	unsigned mask = __ballot_sync(0xffffffffu, fresh);
	if ((threadIdx.x & 31) == 0 && mask) atomicAdd(n_new, (unsigned long long) __popc(mask));
}

// ------------------------------------------------------------------------------------------------------------------
// sharded sync (reference -t N: X_to_add[src][dst] + three barriers, dna.cpp:2393-2488).  The exchange matrix is written
// straight into the owners' inboxes with NVLink peer stores: k_owner_keys tags every pending k-mer with its owner and
// counts, a stable 3-bit radix sort groups the row by owner without disturbing push order, k_route_scatter copies group j
// into slot [table][src = this rank] of rank j's inbox and posts its length there.  The owners then apply the slots in
// source order with their own PRNG streams.
// ------------------------------------------------------------------------------------------------------------------
struct InboxDev {
	unsigned long long *base[8];     // every rank's inbox (peer mapping; [rank] = own)
	unsigned long long cap;          // entries per (table, source) slot
	uint32_t world, rank;
};
static const uint32_t INBOX_HDR = 128;   // u64 words: [0, 48) posted slot lengths [6 tables][8 sources]; [48, 56) routed and [56, 64) applied sync numbers per source;
                                         // [64, 68) global p-mer statistics of the sync under way, two instances (k_post_applied)
FQSK_HD unsigned long long *inbox_slot(unsigned long long *base, unsigned long long cap, uint32_t world, uint32_t table, uint32_t src) {
	return base + INBOX_HDR + ((unsigned long long) table * world + src) * cap;
}
// kind 0: p-mers (aligned index, owner by its top 12 bits), 1: s-/b-mers (normalised k-mer)
__global__ void k_owner_keys(const unsigned long long *row, uint32_t n, uint32_t kind, uint32_t pshift, uint32_t world, uint8_t *keys, uint32_t *hist) { pdl_enter();
	__shared__ uint32_t sh[8];
	if (threadIdx.x < 8) sh[threadIdx.x] = 0;
	__syncthreads();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) {
		unsigned long long x = row[i];
		uint32_t o = kind == 0 ? (uint32_t) ((x >> pshift) % world) : ht_owner(world, x);
		keys[i] = (uint8_t) o;
		atomicAdd(sh + o, 1u);
	}
	__syncthreads();
	if (threadIdx.x < 8 && sh[threadIdx.x]) atomicAdd(hist + threadIdx.x, sh[threadIdx.x]);
}
__global__ void k_route_scatter(const unsigned long long *sorted, uint32_t n, const uint32_t *hist, InboxDev I, uint32_t table, int *flags) { pdl_enter();
	uint32_t off[9];
	off[0] = 0;
	for (uint32_t o = 0; o < 8; ++o) off[o + 1] = off[o] + (o < I.world ? hist[o] : 0);
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < I.world) {
		if (hist[i] > I.cap) flags[4] = 1;
		I.base[i][table * 8 + I.rank] = hist[i];      // posted length of slot [table][src = rank] at owner i
	}
	if (i >= n) return;
	uint32_t o = 0;
	while (i >= off[o + 1]) ++o;
	if (hist[o] > I.cap) return;
	inbox_slot(I.base[o], I.cap, I.world, table, I.rank)[i - off[o]] = sorted[i];
}

// The three k-mer rows of a sync in two launches (blockIdx.y = table 0 p / 1 s / 2 b): k_route_count leaves the owner histogram of
// every chunk of 2048 pending k-mers, k_route_move gives every k-mer its place inside its owner's group -- chunks in order, a warp's
// 256 consecutive k-mers in order, lanes in order: push order survives (the owners insert in source order, dna.cpp:2421-2446) --
// and stores it straight into slot [table][src = this rank] of the owner's inbox (NVLink peer stores); the CTA of chunk 0 posts the
// slot lengths.  Replaces k_owner_keys + three radix launches + k_route_scatter per table.
static const uint32_t ROUTE_CHUNK = 2048;
struct RouteRows { const unsigned long long *row[3]; uint32_t n[3]; uint32_t pshift; };
__device__ __forceinline__ uint32_t route_owner(uint32_t table, unsigned long long x, uint32_t pshift, uint32_t world) {
	return table == 0 ? (uint32_t) ((x >> pshift) % world) : ht_owner(world, x);
}
__global__ void __launch_bounds__(256) k_route_count(RouteRows R, uint32_t world, uint32_t chunks_max, uint32_t *chunk_hist) { pdl_enter();      // chunk_hist[table][chunk][8]
	const uint32_t table = blockIdx.y, c = blockIdx.x, n = R.n[table];
	if ((unsigned long long) c * ROUTE_CHUNK >= n) return;
	__shared__ uint32_t sh[8];
	if (threadIdx.x < 8) sh[threadIdx.x] = 0;
	__syncthreads();
	const unsigned long long *row = R.row[table];
	uint32_t mine[8] = {0, 0, 0, 0, 0, 0, 0, 0};
	for (uint32_t q = 0; q < ROUTE_CHUNK / 256; ++q) {
		const uint32_t i = c * ROUTE_CHUNK + q * 256 + threadIdx.x;
		if (i < n) { const uint32_t o = route_owner(table, row[i], R.pshift, world); for (uint32_t k = 0; k < 8; ++k) mine[k] += (o == k); }
	}
	for (uint32_t k = 0; k < 8; ++k) {
		uint32_t v = mine[k];
		for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
		if ((threadIdx.x & 31) == 0 && v) atomicAdd(sh + k, v);
	}
	__syncthreads();
	if (threadIdx.x < 8) chunk_hist[((size_t) table * chunks_max + c) * 8 + threadIdx.x] = sh[threadIdx.x];
}
__global__ void __launch_bounds__(256) k_route_move(RouteRows R, uint32_t chunks_max, const uint32_t *chunk_hist, InboxDev I, int *flags) { pdl_enter();
	const uint32_t table = blockIdx.y, c = blockIdx.x, n = R.n[table], t = threadIdx.x, lane = t & 31, w = t >> 5;
	const uint32_t n_chunks = (n + ROUTE_CHUNK - 1) / ROUTE_CHUNK;
	__shared__ uint32_t base[8], total[8], wcnt[8][8];      // group position of the chunk's first k-mer per owner; row totals; per-warp counts
	if (c > 0 && c >= n_chunks) return;
	if (t < 8) {
		uint32_t b = 0, tot = 0;
		for (uint32_t q = 0; q < n_chunks; ++q) { const uint32_t v = chunk_hist[((size_t) table * chunks_max + q) * 8 + t]; if (q < c) b += v; tot += v; }
		base[t] = b; total[t] = tot;
	}
	for (uint32_t q = t; q < 64; q += 256) (&wcnt[0][0])[q] = 0;
	__syncthreads();
	if (c == 0 && t < I.world) {
		if (total[t] > I.cap) flags[4] = 1;
		I.base[t][table * 8 + I.rank] = total[t];      // posted length of slot [table][src = rank] at owner t
	}
	if ((unsigned long long) c * ROUTE_CHUNK >= n) return;
	const unsigned long long *row = R.row[table];
	// a warp owns 256 consecutive k-mers of the chunk and visits them in 8 rounds of 32
	unsigned long long x[8]; uint32_t own[8];
	const uint32_t wbase = c * ROUTE_CHUNK + w * 256;
#pragma unroll
	for (uint32_t r = 0; r < 8; ++r) {
		const uint32_t i = wbase + r * 32 + lane;
		x[r] = i < n ? row[i] : 0ull;
		own[r] = i < n ? route_owner(table, x[r], R.pshift, I.world) : 0xFFu;
	}
	uint32_t cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
	for (uint32_t r = 0; r < 8; ++r) for (uint32_t k = 0; k < 8; ++k) cnt[k] += __popc(__ballot_sync(0xffffffffu, own[r] == k));
	if (lane < 8) { uint32_t v = 0; for (uint32_t k = 0; k < 8; ++k) if (k == lane) v = cnt[k]; wcnt[w][lane] = v; }
	__syncthreads();
	uint32_t pos[8];      // running position inside the owner's group for this warp
	for (uint32_t k = 0; k < 8; ++k) { uint32_t b = base[k]; for (uint32_t q = 0; q < w; ++q) b += wcnt[q][k]; pos[k] = b; }
#pragma unroll
	for (uint32_t r = 0; r < 8; ++r) {
		const uint32_t o = own[r];
		uint32_t my = 0;
		for (uint32_t k = 0; k < 8; ++k) {
			const unsigned m = __ballot_sync(0xffffffffu, o == k);
			if (o == k) my = pos[k] + __popc(m & ((1u << lane) - 1u));
			pos[k] += __popc(m);
		}
		if (o < 8 && total[o] <= I.cap) inbox_slot(I.base[o], I.cap, I.world, table, I.rank)[my] = x[r];
	}
}

// First barrier of the reference's sync (application.cpp:645-648: "every worker has filled its X_to_add rows") without the host: each
// source posts the number of the sync into word [48 + src] of every owner's inbox header once its rows have landed there (a kernel of
// its own behind the scatter kernels: their peer stores are complete when it starts); an owner waits for all its sources on the
// device, in front of the copy that reads the posted lengths.  Bounded wait (~20 s): a rank that died must not hang the others.
static const uint32_t INBOX_SEQ = 48;
__global__ void k_post_seq(InboxDev I, unsigned long long seq) { pdl_enter();
	const uint32_t i = threadIdx.x;
	if (i >= I.world) return;
	__threadfence_system();
	*reinterpret_cast<volatile unsigned long long *>(I.base[i] + INBOX_SEQ + I.rank) = seq;
	__threadfence_system();
}
__global__ void k_wait_seq(const unsigned long long *inbox, uint32_t world, unsigned long long seq, int *err) { pdl_enter();
	const uint32_t i = threadIdx.x;
	if (i >= world) return;
	const long long t0 = clock64();
	while (*reinterpret_cast<const volatile unsigned long long *>(inbox + INBOX_SEQ + i) < seq) {
		if (clock64() - t0 > 40000000000ll) { *err = 1; break; }      // ~20 s
		__nanosleep(200);
	}
	__threadfence_system();
}

// Second barrier of the reference's sync (application.cpp:651-654: "every owner has inserted") and the global p-mer statistics
// (TSmallIntVector's atomics, bit_vec.h:212-220) without the host or a collective library: every rank adds its (fresh fields, updates)
// into the accumulators of ALL ranks (NVLink atomics) and then posts the sync's number in their headers; a rank that has seen all N
// numbers holds the complete sums.  Two accumulator instances alternate: a rank clears the next sync's instance before it posts this
// sync's number, and nobody adds to that instance before having seen that number.
static const uint32_t INBOX_APPLIED = 56, INBOX_ACC = 64, INBOX_GROW = 72;
// Growth requests travel the same way: a rank whose shard of the s-mer / b-mer / pair table is past half full after its inserts adds 1 to
// field 0 / 1 / 2 (16 bits each) of word INBOX_GROW + instance in every rank's header; every rank then reads the same word and all shards
// of a requested table double together (fqsk_sync_finish -> FQSK_RESHARD).  lim: items in the buckets / in the stash of the b-mer table,
// of the s-mer table, items of the pair table above which this rank asks (~0: the table cannot double any more).
struct GrowLim { unsigned long long v[5]; };
__global__ void k_post_applied(InboxDev I, unsigned long long seq, const unsigned long long *fresh_dev, unsigned long long updates,
                               const unsigned long long *counters, const unsigned long long *pair_items, GrowLim lim) { pdl_enter();
	const uint32_t t = threadIdx.x, par = (uint32_t) (seq & 1);
	if (t == 0) { unsigned long long *own = I.base[I.rank] + INBOX_ACC + 2 * (par ^ 1); own[0] = 0; own[1] = 0; I.base[I.rank][INBOX_GROW + (par ^ 1)] = 0; }
	__threadfence_system();
	__syncthreads();
	if (t < I.world) {
		unsigned long long req = 0;
		if (counters[2] > lim.v[2] || counters[3] > lim.v[3]) req |= 1ull;
		if (counters[0] > lim.v[0] || counters[1] > lim.v[1]) req |= 1ull << 16;
		if (pair_items && *pair_items > lim.v[4]) req |= 1ull << 32;
		atomicAdd_system(I.base[t] + INBOX_ACC + 2 * par, *fresh_dev);
		atomicAdd_system(I.base[t] + INBOX_ACC + 2 * par + 1, updates);
		if (req) atomicAdd_system(I.base[t] + INBOX_GROW + par, req);
	}
	__threadfence_system();
	__syncthreads();
	if (t < I.world) { *reinterpret_cast<volatile unsigned long long *>(I.base[t] + INBOX_APPLIED + I.rank) = seq; __threadfence_system(); }
}
__global__ void k_wait_applied(const unsigned long long *inbox, uint32_t world, unsigned long long seq, int *err) { pdl_enter();
	const uint32_t i = threadIdx.x;
	if (i >= world) return;
	const long long t0 = clock64();
	while (*reinterpret_cast<const volatile unsigned long long *>(inbox + INBOX_APPLIED + i) < seq) {
		if (clock64() - t0 > 40000000000ll) { *err = 1; break; }      // ~20 s
		__nanosleep(200);
	}
	__threadfence_system();
}

// checksum of a record stream (fqsk_recs_checksum): position-dependent term per record, summed mod 2^64
__global__ void __launch_bounds__(256) k_recs_checksum(const fqsk_base_rec *recs, unsigned long long n, unsigned long long *out) { pdl_enter();
	unsigned long long acc = 0;
	for (unsigned long long i = (unsigned long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long) gridDim.x * blockDim.x) {
		const uint32_t *w = reinterpret_cast<const uint32_t *>(recs + i);
		const unsigned long long a = w[0] | ((unsigned long long) w[1] << 32), b = w[2] | ((unsigned long long) w[3] << 32), c = w[4] | ((unsigned long long) w[5] << 32), d = w[6];
		acc += fmix64(a ^ fmix64(b ^ fmix64(c ^ fmix64(d + i))));
	}
	for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
	if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// ------------------------------------------------------------------------------------------------------------------
// table-level batch mirrors
// ------------------------------------------------------------------------------------------------------------------
__global__ void k_find(HtDev t, CIncP ci, const unsigned long long *dir, const unsigned long long *rc, const uint32_t *cur, uint32_t n,
                       uint32_t *counts, const uint32_t *draws, unsigned long long dmask, unsigned long long dpos, unsigned long long avail, const unsigned long long *guess, uint32_t *used, int *flags) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	DrawCursor dc; dc.ring = draws; dc.mask = dmask; dc.pos0 = dpos; dc.avail = avail; dc.base = guess ? guess[i] : 0; dc.used = 0; dc.overflow = flags;
	KReg r{dir[i], rc[i]};
	uint32_t c[4];
	ht_find(t, ci, r, cur[i], c, dc);
	for (int q = 0; q < 4; ++q) counts[4 * i + q] = c[q];
	used[i] = dc.used;
}
__global__ void k_count(HtDev t, const unsigned long long *kmers, uint32_t n, uint32_t *out) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) out[i] = ht_count(t, kmers[i]);
}
__global__ void k_siv_test(SivDev s, const unsigned long long *idx, uint32_t n, uint32_t *out) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) out[i] = siv_test(s, idx[i]);
}
__global__ void k_siv_counts(SivDev s, const unsigned long long *idx, uint32_t n, uint32_t *out) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) { uint32_t c[4]; siv_counts(s, idx[i], c, false); for (int q = 0; q < 4; ++q) out[4 * i + q] = c[q]; }
}
__global__ void k_siv_prefix(SivDev s, const unsigned long long *idx, const uint32_t *bits, uint32_t n, unsigned long long *out) { pdl_enter();
	uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) out[i] = siv_prefix_sum(s, idx[i], bits[i]);
}

// ------------------------------------------------------------------------------------------------------------------
// dumps (parity check 1) and table growth
// ------------------------------------------------------------------------------------------------------------------
struct MixInv { uint64_t inv1, inv2; };
__device__ __forceinline__ uint64_t ht_unmix(const HtDev &t, const MixInv &mi, uint64_t x) {
	x ^= x >> t.mix_sh;                 // mix_sh >= W/2 -> the xor-shift is an involution
	x = (x * mi.inv2) & t.maskW;
	x ^= x >> t.mix_sh;
	x = (x * mi.inv1) & t.maskW;
	return x;
}
__global__ void k_dump_ht(HtDev t, MixInv mi, unsigned long long *keys, unsigned long long *vals, unsigned long long cap, unsigned long long *n_out) { pdl_enter();
	uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
	uint64_t nm = 8ull << t.B, ns = 1ull << t.stash_log2;
	if (i >= nm + ns) return;
	uint64_t x, cnt;
	if (i < nm) {
		uint32_t it = t.main[i];
		if (!it) return;
		uint64_t rem = (it & 0x7fffffffu) >> (8 + t.cbits);
		uint64_t h = ((i >> 3) << t.rem_bits) | rem;
		uint64_t kernel = ht_unmix(t, mi, h);
		uint64_t ends = (it >> t.cbits) & 0xFF;
		x = ((ends >> 4) << 60) | (kernel << (64 - 2 * t.k + 4)) | ((ends & 0xF) << (64 - 2 * t.k));
		cnt = it & t.top;
	} else {
		unsigned long long it = t.stash[i - nm];
		if (!it) return;
		x = ((it >> t.cbits) - 1) << (64 - 2 * t.k);
		cnt = it & t.top;
	}
	unsigned long long o = atomicAdd(n_out, 1ull);
	if (o < cap) { keys[o] = x; vals[o] = cnt; }
}
__global__ void k_dump_siv(SivDev s, unsigned long long *keys, unsigned long long *vals, unsigned long long cap, unsigned long long *n_out) { pdl_enter();
	uint64_t w = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
	uint64_t tops = s.world > 1 ? (4096 + s.world - 1) / s.world : 4096;      // this rank's shard: ceil(4096 / world) top values
	uint64_t nw = s.world > 1 ? (tops << s.top_shift) >> 4 : (1ull << s.key_bits) >> 4;
	if (w >= nw) return;
	uint32_t d = s.w[w];
	if (!d) return;
	for (uint32_t r = 0; r < 16; ++r) {
		uint32_t f = (d >> (2 * r)) & 3;
		if (!f) continue;
		uint64_t li = w * 16 + r, gi = li;
		if (s.world > 1) gi = (((li >> s.top_shift) * s.world + s.rank) << s.top_shift) | (li & ((1ull << s.top_shift) - 1ull));
		unsigned long long o = atomicAdd(n_out, 1ull);
		if (o < cap) { keys[o] = gi; vals[o] = f; }
	}
}
// re-insert dumped (k-mer, counter) pairs into a fresh, larger table
__global__ void k_reinsert(HtDev t, const unsigned long long *keys, const unsigned long long *vals, uint64_t n) { pdl_enter();
	uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	bool created;
	uint64_t s = ht_locate(t, keys[i], created);
	ht_slot_set(t, s, (uint32_t) vals[i]);
}

}  // namespace fqsk
