// fqsk_pipeline.cuh -- the position-parallel segment pipeline (DESIGN.md section 5).
//
// The reference walks a read base by base and, per base, walks a cascade of table lookups (dna.cpp:457-502, 674-877).
// Three facts of that algorithm make it parallel without changing a bit of its output:
//   (1) the corrected registers equal the uncorrected ones except in the b-1 positions after a repair
//       (dna.cpp:363-365, 442-446, 697-705), and the uncorrected ones are a pure function of the read;
//   (2) repairs, pushes and the level of a position depend only on lookups of FULL contexts, which draw no random numbers
//       (ht_kmer.h:189-196); PRNG-dependent values (merges of front-truncated and of rough lookups, ht_kmer.h:321-323,
//       dna.cpp:285-287, 323-325) only reach the emitted counts;
//   (3) rough results never feed back into the registers (dna.cpp:707-735 vs 854-875).
// So:  k_lookup    one thread per (read, position): the whole cascade for the uncorrected registers, global tables only
//      k_partial   one warp per front-truncated lookup: 4^m completions across lanes -> ordered merge script
//      k_local     one thread per position the global tables could not answer: the segment delta (thread-local tables)
//      k_walk      one thread per read: registers, repairs, cor_pos, pushes; table traffic only inside repair windows
//      k_rough     one warp per rough request: 4(k-1) neighbours across lanes -> ordered merge script
//      k_fold      one thread per script: approximate-counter merges with the read-ordered mt19937 draw indices
#pragma once
#include "fqsk_kernels.cuh"
#include "../../include/fqsk_ctx.h"

namespace fqsk {

// per-position flags kept beside the provisional record
enum : uint8_t {
	PF_MISS_B = 1,        // b-mer context consulted and absent from the global table -> thread-local b table is next (dna.cpp:485)
	PF_MISS_S = 2,        // s-mer context consulted and absent from the global table -> thread-local s table is next (dna.cpp:495)
	PF_PARTIAL_B = 4,     // front-truncated b lookup (ordered merge script pending)
	PF_PARTIAL_S = 8,     // front-truncated s lookup
	PF_GLOBAL_S_HIT = 16, // the global s-mer lookup succeeded (its counts are stored in the miss entry)
};

struct Script {              // ordered list of per-trial count vectors to be merged with CCounterIncrementer::Increment(a, b)
	uint32_t rec;            // record index of the position
	uint8_t kind;            // 0 partial b, 1 partial s, 2 rough b, 3 rough s
	uint8_t valid;
	uint16_t n;              // entries (inline up to 8, the rest in the overflow pool)
	uint32_t overflow;       // first overflow entry
	uint16_t c2[4];          // s-mer counts for the `mixed` rule when a partial b merge ends with two saturated counters (dna.cpp:470-478)
	uint16_t e[8][4];
	uint32_t draws;          // mt19937 outputs this script's merge consumes (k_fold pass 0; confirmed by pass 1)
};
static const uint32_t SCRIPT_INLINE = 8;

struct MissEntry {           // a position whose uncorrected cascade needs the thread-local tables
	uint32_t rec, time;      // record index; lookup time = 2 * position id (byte offset of the base inside the packed DNA)
	uint32_t read;           // owning read (marked dirty when the thread-local answer changes)
	KReg breg;               // uncorrected b register with the placeholder (s register is derived from it)
	uint32_t cb;             // symbols held by the b register
	uint8_t flags;           // PF_*
	uint8_t glevel;          // level of the global-only cascade (SMER or NONE)
	uint16_t gs[4];          // its counts (global s-mer hit)
};


struct PipeDev {
	// geometry
	uint32_t n_rec, start;          // coded positions of the segment; first coded position of a read
	const unsigned long long *rec_off;
	// provisional / final records and per-position flags
	fqsk_base_rec *prov;            // find_counts result for the UNCORRECTED registers (k_lookup / k_partial / k_local)
	fqsk_base_rec *recs; uint8_t *pflags;   // final records (k_walk, then k_rough / k_fold)
	// scripts: partial ones are addressed densely (read * slots + slot); rough ones are appended
	Script *pscripts; uint32_t pslots; uint32_t pfirst_n; // slot = (i + 1) - pfirst_n
	Script *rscripts; uint32_t *n_rscript; uint32_t rscript_cap;   // rough scripts, allocated by k_rough
	uint8_t *rkind; KReg *rreg; uint32_t *rslot;                   // per position: rough request kind (0/2/3/4), its register, its script
	uint8_t *dirty;                                                // per read: must be walked again
	unsigned short *pool; uint32_t *pool_used; uint32_t pool_cap;   // overflow entries (4 x u16 each)
	MissEntry *miss; uint32_t *n_miss; uint32_t miss_cap;
	uint8_t *miss_fold;             // hot mode: 1 / 2 = this entry's thread-local merge (b / s) is done by the ordered evaluator
	unsigned long long *ev_key[2]; uint32_t *ev_val[2]; uint32_t *ev_n; uint32_t ev_cap;   // hot mode: time-ordered events of the cinc_lb / cinc_ls streams
	uint32_t *hot_draws;            // hot mode: draws consumed from cinc_lb, cinc_ls
	// per-read draw counts of the merge scripts (stream b, stream s) and their exclusive scans
	uint32_t *rdraws_b, *rdraws_s; const unsigned long long *doff_b, *doff_s;
	const uint32_t *n_rec_dev;      // number of coded positions, device copy (grids are sized from host-side upper bounds)
	// pushes
	uint32_t *time_b, *time_s;      // per-read regions parallel to push_b / push_s
	int *flags;                     // [0] draw overflow [1] unsupported [2] changed [3] window consulted the local tables
	                                // [4] capacity overflow (pool / miss / rough lists) [5] internal: draw in a no-draw path [6] k_local hit
	                                // [7] k_fold: a read's draw count differs from the scanned one
};

__device__ __forceinline__ uint32_t sym_at(bool sorted, const EngineDev &E, const uint8_t *p, uint32_t j) {
	uint32_t c = dna_code(p[j]);
	if (c == 4) c = (sorted && j < E.p) ? 3u : 0u;   // dna.cpp:532-536 / 560-565 / 684
	return c;
}
// uncorrected b register (with placeholder) in front of position i; cb = min(b, i + 1): symbols i - cb + 1 .. i - 1 of the packed
// read, then the placeholder (dir: A, rc: T at position 0, the complements mirrored behind it)
__device__ __forceinline__ KReg breg_from_words(uint64_t hi, uint64_t lo, uint32_t a, uint32_t cb) {
	KReg r;
	r.dir = pk_window(hi, lo, a, cb - 1);
	r.rc = (3ull << 62) | (cb > 1 ? rc_kmer(r.dir, cb - 1) >> 2 : 0ull);
	return r;
}
__device__ __forceinline__ KReg build_breg(const unsigned long long *pkr, uint32_t i, uint32_t cb) {
	const uint32_t a = i + 1 - cb;
	return breg_from_words(pkr[a >> 5], pkr[(a >> 5) + 1], a, cb);
}
// suffix register of length c (c <= cb) taken from a register holding cb symbols
__device__ __forceinline__ KReg suffix_reg(const KReg &r, uint32_t cb, uint32_t c) {
	KReg o;
	o.dir = r.dir << (2 * (cb - c));
	o.rc = r.rc & (~0ull << (64 - 2 * c));
	return o;
}
__device__ __forceinline__ uint32_t find_read(const unsigned long long *rec_off, uint32_t n_reads, uint32_t g, uint32_t n_rec) {
	// last r with rec_off[r] <= g.  Reads of a segment mostly have the same length, so interpolation lands on the read or next to
	// it (2 dependent loads instead of log2(n) -- this search sits at the head of every position's latency chain); the bracket
	// found by a few galloping steps is finished by bisection for ragged input.
	uint32_t r = (uint32_t) (((unsigned long long) g * n_reads) / (n_rec ? n_rec : 1));
	if (r >= n_reads) r = n_reads - 1;
	uint32_t lo, hi;
	if (rec_off[r] <= g) {
		uint32_t step = 1; lo = r; hi = r + 1;
		while (hi < n_reads && rec_off[hi] <= g) { lo = hi; hi = hi + step < n_reads ? hi + step : n_reads; step <<= 1; }
	} else {
		uint32_t step = 1; hi = r; lo = r >= 1 ? r - 1 : 0;
		while (lo > 0 && rec_off[lo] > g) { hi = lo; lo = lo >= step ? lo - step : 0; step <<= 1; }
	}
	while (hi - lo > 1) { uint32_t m = (lo + hi) >> 1; if (rec_off[m] <= g) lo = m; else hi = m; }
	return lo;
}
__device__ __forceinline__ void put_rec(fqsk_base_rec *rec, uint32_t pos, const uint32_t c[4], uint32_t lev) {
	fqsk_base_rec o;
	o.pos = pos; o.counts[0] = c[0]; o.counts[1] = c[1]; o.counts[2] = c[2]; o.counts[3] = c[3];
	o.cor_pos = 0; o.level = (uint8_t) lev; o.rough = 0; o.pad = 0;
	*rec = o;
}

// ------------------------------------------------------------------------------------------------------------------
// k_lookup: the find_counts cascade (dna.cpp:457-502) for the uncorrected registers of every coded position, global
// tables only.  Front-truncated table lookups are left to k_partial (flagged here).
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lookup(EngineDev E, SegDev S, PipeDev P) { pdl_enter();
	uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t n_rec = *P.n_rec_dev;
	if (g >= n_rec) return;
	uint32_t r = find_read(S.rec_off, S.n_reads, g, n_rec);
	uint32_t i = item_first(S, P.start, r) + (g - (uint32_t) S.rec_off[r]);
	const uint8_t *p = S.dna + S.off[r];
	const uint32_t n = i + 1;
	const uint32_t cb = n < E.b ? n : E.b, cs = n < E.s ? n : E.s, cp = n < E.p ? n : E.p;
	const uint32_t b_margin = E.b - E.s - 1, s_margin = E.s - E.p + 1;
	uint32_t c[4] = {0, 0, 0, 0};
	uint32_t lev = FQSK_LEVEL_NONE;
	uint8_t fl = 0;
	KReg br = build_breg(pk_of(S, r), i, cb);
	if (cb + b_margin >= E.b) {
		if (cb == E.b) {
			bool d = kr_is_dir(br, E.b);
			ht_ctx_counts(E.hb, d ? br.dir : br.rc, d, c);
			KReg sr = suffix_reg(br, cb, cs);
			if (any4(c)) {
				int sat = (c[0] == E.hb.top) + (c[1] == E.hb.top) + (c[2] == E.hb.top) + (c[3] == E.hb.top);
				lev = FQSK_LEVEL_BMER;
				if (sat > 1) {
					uint32_t c2[4] = {0, 0, 0, 0};
					bool d2 = kr_is_dir(sr, E.s);
					ht_ctx_counts(E.hs, d2 ? sr.dir : sr.rc, d2, c2);
					for (int q = 0; q < 4; ++q) c[q] += c2[q];
					lev = FQSK_LEVEL_MIXED;
				}
			} else {
				fl |= PF_MISS_B;
				bool d2 = kr_is_dir(sr, E.s);
				ht_ctx_counts(E.hs, d2 ? sr.dir : sr.rc, d2, c);
				if (any4(c)) { lev = FQSK_LEVEL_SMER; fl |= PF_GLOBAL_S_HIT; } else fl |= PF_MISS_S;
			}
		} else return;                 // front-truncated b lookup: k_partial owns this position (it runs next to this kernel)
	} else if (cs + s_margin >= E.s) {
		if (cs == E.s) {
			KReg sr = suffix_reg(br, cb, cs);
			bool d2 = kr_is_dir(sr, E.s);
			ht_ctx_counts(E.hs, d2 ? sr.dir : sr.rc, d2, c);
			if (any4(c)) { lev = FQSK_LEVEL_SMER; fl |= PF_GLOBAL_S_HIT; } else fl |= PF_MISS_S;
		} else return;                 // front-truncated s lookup: k_partial
	} else {
		KReg pr = suffix_reg(br, cb, cp);      // find_counts_p (dna.cpp:210-226)
		if (cp < E.p) {
			for (uint64_t j = 0; j < 4; ++j) { KReg t = pr; kr_set_last(t, cp, j); c[j] = (uint32_t) siv_prefix_sum(E.siv, t.rc >> (64 - 2 * cp), 2 * cp); }
		} else siv_counts(E.siv, pr.dir >> (64 - 2 * E.p), c, false);
		if (any4(c)) lev = FQSK_LEVEL_PMER;
	}
	put_rec(P.prov + g, i, c, lev);
	P.pflags[g] = fl;
	if ((fl & (PF_MISS_B | PF_MISS_S)) && !(fl & (PF_PARTIAL_B | PF_PARTIAL_S))) {
		// warp-aggregated append: misses come in runs (an uncovered stretch, the b positions after an error), one atomic per warp
		const unsigned am = __activemask();
		const uint32_t lane = threadIdx.x & 31, leader = (uint32_t) __ffs(am) - 1;
		uint32_t m = 0;
		if (lane == leader) m = atomicAdd(P.n_miss, (uint32_t) __popc(am));
		m = __shfl_sync(am, m, leader) + __popc(am & ((1u << lane) - 1u));
		if (m >= P.miss_cap) P.flags[4] = 1;
		if (m < P.miss_cap) {
			MissEntry e;
			e.rec = g; e.time = 2 * ((uint32_t) S.off[r] + i); e.read = r; e.breg = br; e.cb = cb; e.flags = fl; e.glevel = (uint8_t) lev;
			for (int q = 0; q < 4; ++q) e.gs[q] = (uint16_t) c[q];
			P.miss[m] = e;
			if (fl & PF_MISS_B) delta_note(S.delta_b, br, cb);
			if (fl & PF_MISS_S) delta_note(S.delta_s, suffix_reg(br, cb, cs), cs);
		}
	}
}

// ------------------------------------------------------------------------------------------------------------------
// k_partial: one warp per front-truncated position.  Lanes evaluate the 4^m completions (ht_kmer.h:276-310) 32 at a time;
// non-empty trials are appended, in trial order, to the position's merge script (ht_kmer.h:312-324 is replayed by k_fold).
// Then the warp finishes the cascade for that position: s-mer fallback and miss bookkeeping.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void script_append(PipeDev &P, Script &sc, uint32_t &n, uint32_t &ovf, const uint32_t loc[4], bool have, uint32_t remaining_upper) {
	// warp-collective: lanes with have==true append in lane order
	unsigned m = __ballot_sync(0xffffffffu, have);
	if (!m) return;
	uint32_t lane = threadIdx.x & 31;
	uint32_t pos = n + __popc(m & ((1u << lane) - 1));
	uint32_t total = n + __popc(m);
	if (total > SCRIPT_INLINE && ovf == 0xFFFFFFFFu) {
		// first spill: reserve room for everything that can still come
		uint32_t o = 0;
		if (lane == 0) o = atomicAdd(P.pool_used, remaining_upper);
		ovf = __shfl_sync(0xffffffffu, o, 0);
		if (ovf + remaining_upper > P.pool_cap) { if (lane == 0) P.flags[4] = 1; ovf = 0xFFFFFFFEu; }
	}
	if (have) {
		if (pos < SCRIPT_INLINE) { for (int q = 0; q < 4; ++q) sc.e[pos][q] = (uint16_t) loc[q]; }
		else if (ovf < 0xFFFFFFFEu) { unsigned short *d = P.pool + 4ull * (ovf + (pos - SCRIPT_INLINE)); for (int q = 0; q < 4; ++q) d[q] = (unsigned short) loc[q]; }
	}
	n = total;
}

__global__ void __launch_bounds__(128) k_partial(EngineDev E, SegDev S, PipeDev P) { pdl_enter();
	// one warp per (read, partial slot); slot -> n = pfirst_n + slot symbols in the registers (placeholder included)
	uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	uint32_t lane = threadIdx.x & 31;
	uint32_t r = w / P.pslots, slot = w % P.pslots;
	if (r >= S.n_reads) return;
	Script *scp = P.pscripts + (size_t) r * P.pslots + slot;
	if (lane == 0) scp->valid = 0;
	if (S.dup[r]) return;
	uint32_t n = P.pfirst_n + slot, i = n - 1;
	const uint32_t first_r = item_first(S, P.start, r);
	if (i < first_r || i >= S.len[r]) return;
	uint32_t g = (uint32_t) S.rec_off[r] + (i - first_r);
	const uint32_t cb = n < E.b ? n : E.b, cs = n < E.s ? n : E.s;
	// which positions are front-truncated table lookups is a function of the position alone (dna.cpp:461-466, 493): the same
	// thresholds as in k_lookup, which leaves exactly these positions to this kernel
	uint8_t fl = 0;
	if (cb + (E.b - E.s - 1) >= E.b) { if (cb < E.b) fl = PF_PARTIAL_B; }
	else if (cs + (E.s - E.p + 1) >= E.s) { if (cs < E.s) fl = PF_PARTIAL_S; }
	if (!fl) return;
	KReg br = build_breg(pk_of(S, r), i, cb);
	const bool is_b = (fl & PF_PARTIAL_B) != 0;
	const HtDev &t = is_b ? E.hb : E.hs;
	KReg reg = is_b ? br : suffix_reg(br, cb, cs);
	uint32_t cur = is_b ? cb : cs;
	uint32_t m = t.k - cur, trials = 1u << (2 * m);
	// the script lives in registers of lane 0 .. written through a shared staging copy
	__shared__ Script stage[4];
	Script &sc = stage[threadIdx.x >> 5];
	uint32_t n_ent = 0, ovf = 0xFFFFFFFFu;
	bool found = false;
	for (uint32_t n0 = 0; n0 < trials; n0 += 32) {
		uint32_t tn = n0 + lane;
		uint32_t loc[4] = {0, 0, 0, 0};
		if (tn < trials) {
			KReg tr = partial_trial(reg, t.k, m, tn);
			bool d = kr_is_dir(tr, t.k);
			ht_ctx_counts(t, d ? tr.dir : tr.rc, d, loc);
		}
		bool have = any4(loc);
		script_append(P, sc, n_ent, ovf, loc, have, trials - n0);
		found |= __any_sync(0xffffffffu, have);
	}
	__syncwarp();
	// rest of the cascade (lane 0): s-mer fallback after a partial-b miss (cs == s there), miss entry for the local tables
	if (lane == 0) {
		uint32_t c[4] = {0, 0, 0, 0};
		uint32_t lev = FQSK_LEVEL_NONE;
		uint8_t nf = fl;
		uint16_t c2[4] = {0, 0, 0, 0};
		if (is_b) {
			KReg sr = suffix_reg(br, cb, cs);
			bool d2 = kr_is_dir(sr, E.s);
			uint32_t cc[4] = {0, 0, 0, 0};
			ht_ctx_counts(E.hs, d2 ? sr.dir : sr.rc, d2, cc);     // needed for `mixed` (hit) or as the s fallback (miss)
			if (found) { lev = FQSK_LEVEL_BMER; for (int q = 0; q < 4; ++q) c2[q] = (uint16_t) cc[q]; }
			else {
				nf |= PF_MISS_B;
				for (int q = 0; q < 4; ++q) c[q] = cc[q];
				if (any4(cc)) { lev = FQSK_LEVEL_SMER; nf |= PF_GLOBAL_S_HIT; } else nf |= PF_MISS_S;
			}
		} else {
			if (found) lev = FQSK_LEVEL_SMER; else nf |= PF_MISS_S;
		}
		sc.rec = g; sc.kind = is_b ? 0 : 1; sc.valid = found ? 1 : 0; sc.n = (uint16_t) n_ent; sc.overflow = ovf;
		for (int q = 0; q < 4; ++q) sc.c2[q] = c2[q];
		*scp = sc;
		put_rec(P.prov + g, i, c, lev);
		P.pflags[g] = nf;
		if (nf & (PF_MISS_B | PF_MISS_S)) {
			uint32_t mi = atomicAdd(P.n_miss, 1u);
			if (mi >= P.miss_cap) P.flags[4] = 1;
			if (mi < P.miss_cap) {
				MissEntry e;
				e.rec = g; e.time = 2 * ((uint32_t) S.off[r] + i); e.read = r; e.breg = br; e.cb = cb; e.flags = nf; e.glevel = (uint8_t) lev;
				for (int q = 0; q < 4; ++q) e.gs[q] = (uint16_t) c[q];
				P.miss[mi] = e;
				if (nf & PF_MISS_B) delta_note(S.delta_b, br, cb);
				if (nf & PF_MISS_S) delta_note(S.delta_s, suffix_reg(br, cb, cs), cs);
			}
		}
	}
}

// ------------------------------------------------------------------------------------------------------------------
// k_local: thread-local table lookups (dna.cpp:485, 495) for the positions listed by k_lookup / k_partial, against the
// delta of the previous iteration.  Idempotent: always starts from the stored global-only result.
// Merges that would draw from the thread-local PRNG streams are reported as unsupported.
// ------------------------------------------------------------------------------------------------------------------
// phase 1 (always): evaluate the entries; phase 0 (hot mode only): find the front-truncated entries whose thread-local merge
// has to go through the ordered evaluator and queue them as events of their PRNG stream.
__global__ void __launch_bounds__(128) k_local(EngineDev E, SegDev S, PipeDev P, int phase) { pdl_enter();
	if (S.delta_b.n == 0 && S.delta_s.n == 0) return;
	uint32_t n_miss = *P.n_miss;
	if (n_miss > P.miss_cap) n_miss = P.miss_cap;
	for (uint32_t m = blockIdx.x * blockDim.x + threadIdx.x; m < n_miss; m += gridDim.x * blockDim.x) {
		MissEntry e = P.miss[m];
		const uint32_t cs = e.cb < E.s ? e.cb : E.s;
		if (phase == 0) {
			uint8_t fold = 0;
			uint32_t lc[4];
			int nf = 0;
			if ((e.flags & PF_MISS_B) && e.cb < E.b) { delta_find(S.delta_b, E.cib, e.breg, e.cb, e.time, lc, P.flags + 1, &nf); if (nf) fold = 1; }
			if (!fold && (e.flags & PF_MISS_S) && cs < E.s) {
				bool b_hit = false;
				if (e.flags & PF_MISS_B) { int dummy = 0; b_hit = delta_find(S.delta_b, E.cib, e.breg, e.cb, e.time, lc, P.flags + 1, &dummy); }
				if (!b_hit) { KReg sr = suffix_reg(e.breg, e.cb, cs); nf = 0; delta_find(S.delta_s, E.cis, sr, cs, e.time, lc, P.flags + 1, &nf); if (nf) fold = 2; }
			}
			P.miss_fold[m] = fold;
			if (fold) {
				uint32_t st = fold - 1;
				uint32_t q = atomicAdd(P.ev_n + st, 1u);
				if (q >= P.ev_cap) P.flags[4] = 1;
				else { P.ev_key[st][q] = (unsigned long long) e.time << 1; P.ev_val[st][q] = m | 0x80000000u; }
			}
			continue;
		}
		if (P.miss_fold[m]) continue;      // written by the ordered evaluator
		uint32_t c[4] = {e.gs[0], e.gs[1], e.gs[2], e.gs[3]};
		uint32_t lev = e.glevel;
		bool hit = false;
		if (e.flags & PF_MISS_B) {
			uint32_t lc[4];
			if (delta_find(S.delta_b, E.cib, e.breg, e.cb, e.time, lc, P.flags + 1)) { for (int q = 0; q < 4; ++q) c[q] = lc[q]; lev = FQSK_LEVEL_BMER; hit = true; }
		}
		if (!hit && (e.flags & PF_MISS_S)) {
			KReg sr = suffix_reg(e.breg, e.cb, cs);
			uint32_t lc[4];
			if (delta_find(S.delta_s, E.cis, sr, cs, e.time, lc, P.flags + 1)) { for (int q = 0; q < 4; ++q) c[q] = lc[q]; lev = FQSK_LEVEL_SMER; hit = true; }
		}
		fqsk_base_rec *rec = P.prov + e.rec;
		if (rec->level != lev || rec->counts[0] != c[0] || rec->counts[1] != c[1] || rec->counts[2] != c[2] || rec->counts[3] != c[3]) {
			rec->counts[0] = c[0]; rec->counts[1] = c[1]; rec->counts[2] = c[2]; rec->counts[3] = c[3];
			rec->level = (uint8_t) lev;
			P.dirty[e.read] = 1;      // the walk of this read consumed a different answer
			P.flags[6] = 1;
		}
	}
}

// ------------------------------------------------------------------------------------------------------------------
// hot mode (a k-mer is pushed more than thr + 1 times inside the segment and looked up there): the thread-local counters
// leave the deterministic range, so the reference's cinc_lb / cinc_ls draws -- one per thread-local insert above thr
// (ht_kmer.h:433-436) and the draws of thread-local front-truncated merges (ht_kmer.h:321-323), in program order -- are
// replayed by an ordered evaluator: k_delta_rank finds every entry's push-order rank and queues the inserts that draw,
// k_local(phase 0) queues the merges, the events are sorted by time and k_hot_eval walks them sequentially (one thread per
// stream).  Rare by construction: only segments that raised the flag are redone this way.
// ------------------------------------------------------------------------------------------------------------------
__global__ void k_delta_rank(DeltaDev D, PipeDev P, uint32_t stream) { pdl_enter();
	const uint64_t slots = (uint64_t) D.mask + 1;
	for (uint64_t sidx = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; sidx < slots; sidx += (uint64_t) gridDim.x * blockDim.x) {
		const uint32_t tm = D.times[sidx];
		if (tm == DELTA_EMPTY) continue;
		const unsigned long long x = D.keys[sidx];
		uint32_t rank = 0, prev = 0xFFFFFFFFu, prev_t = 0;
		for (uint64_t slot = delta_slot_of_key(x, D.k, D.t, D.mask);; slot = (slot + 1) & D.mask) {
			uint32_t et = D.times[slot];
			if (et == DELTA_EMPTY) break;
			if (et >= tm || D.keys[slot] != x) continue;
			++rank;
			if (prev == 0xFFFFFFFFu || et > prev_t) { prev_t = et; prev = (uint32_t) slot; }
		}
		D.rank_at[sidx] = rank; D.prev_at[sidx] = prev; D.cnt_at[sidx] = 0;
		if (rank >= D.exact_limit) {
			uint32_t q = atomicAdd(P.ev_n + stream, 1u);
			if (q >= P.ev_cap) P.flags[4] = 1;
			else { P.ev_key[stream][q] = ((unsigned long long) tm << 1) | 1ull; P.ev_val[stream][q] = (uint32_t) sidx; }
		}
	}
}

struct DeltaCollect {    // matches of a front-truncated context: (trial index, next symbol, latest entry)
	static const uint32_t CAP = 128;
	uint32_t key[CAP], tm[CAP], slot[CAP]; uint32_t n, m, lsh; bool overflow;
	FQSK_DEV void operator()(uint64_t Y, uint32_t t, uint32_t s) {
		uint32_t trial = 0;
		for (uint32_t j = 0; j < m; ++j) trial |= (uint32_t) ((Y >> (62 - 2 * j)) & 3) << (2 * j);    // front symbol 0 is the fastest digit (ht_kmer.h:291-310)
		uint32_t kk = (trial << 2) | (uint32_t) ((Y >> lsh) & 3);
		for (uint32_t q = 0; q < n; ++q) if (key[q] == kk) { if (t > tm[q]) { tm[q] = t; slot[q] = s; } return; }
		if (n >= CAP) { overflow = true; return; }
		key[n] = kk; tm[n] = t; slot[n] = s; ++n;
	}
};

// More than DeltaCollect::CAP distinct completions of one context (low-complexity reads: most of the 4^(m+1) possible ones pushed inside one
// segment): the matches go into a table indexed directly by (trial, next symbol) -- at most 4^6 entries, tagged with the number of the
// lookup so that it never has to be cleared -- and are read back in index order, which IS the merge order (ht_kmer.h:291-324).
struct DeltaTable {
	uint32_t *ep, *tm, *slot; uint32_t epoch, m, lsh;
	FQSK_DEV void operator()(uint64_t Y, uint32_t t, uint32_t s) {
		uint32_t trial = 0;
		for (uint32_t j = 0; j < m; ++j) trial |= (uint32_t) ((Y >> (62 - 2 * j)) & 3) << (2 * j);
		const uint32_t kk = (trial << 2) | (uint32_t) ((Y >> lsh) & 3);
		if (ep[kk] != epoch) { ep[kk] = epoch; tm[kk] = t; slot[kk] = s; }
		else if (t > tm[kk]) { tm[kk] = t; slot[kk] = s; }
	}
};
static const uint32_t HOT_TAB_ENTRIES = 4096;      // 4^(m + 1), m <= 5 (b - s - 1 at the reference's largest k-mer lengths; s - p + 1 <= 4)

__global__ void k_hot_eval(EngineDev E, SegDev S, PipeDev P, const unsigned long long *ek0, const uint32_t *ev0, uint32_t n0,
                           const unsigned long long *ek1, const uint32_t *ev1, uint32_t n1, uint32_t *tab) { pdl_enter();      // tab: 2 streams x 3 arrays x HOT_TAB_ENTRIES, zeroed by the caller
	if ((threadIdx.x & 31) != 0) return;
	const uint32_t st = threadIdx.x >> 5;     // 0: b / cinc_lb, 1: s / cinc_ls
	if (st > 1) return;
	const DeltaDev &D = st ? S.delta_s : S.delta_b;
	const CIncP ci = st ? E.cis : E.cib;
	const uint32_t top = st ? E.hs.top : E.hb.top;
	const unsigned long long *ek = st ? ek1 : ek0;
	const uint32_t *ev = st ? ev1 : ev0;
	const uint32_t n = st ? n1 : n0;
	DrawCursor dc;
	dc.ring = E.draws[2 + st]; dc.mask = E.dmask[2 + st]; dc.pos0 = E.dpos[2 + st]; dc.avail = E.avail[2 + st]; dc.base = 0; dc.used = 0; dc.overflow = E.flags + 0;
	uint32_t tab_epoch = 0;
	for (uint32_t i = 0; i < n; ++i) {
		const uint32_t v = ev[i];
		if (ek[i] & 1ull) {
			// a thread-local insert whose counter is above thr: one draw unless the counter is full (ht_kmer.h:433-436)
			const uint32_t rank = D.rank_at[v];
			uint32_t c = rank == D.exact_limit ? D.exact_limit : D.cnt_at[D.prev_at[v]];
			if (c < top && dc.next() % (ci.mult * (c - ci.thr)) == 0) ++c;
			D.cnt_at[v] = c;
			continue;
		}
		// a thread-local front-truncated lookup: completions in odometer order, merged with the approximate addition
		const uint32_t mi = v & 0x7fffffffu;
		const MissEntry e = P.miss[mi];
		const uint32_t cs = e.cb < E.s ? e.cb : E.s;
		const KReg reg = st ? suffix_reg(e.breg, e.cb, cs) : e.breg;
		const uint32_t cur = st ? cs : e.cb;
		DeltaCollect M; M.n = 0; M.m = D.k - cur; M.lsh = 64 - 2 * D.k; M.overflow = false;
		delta_scan(D, reg, cur, e.time, M);
		uint32_t c[4] = {0, 0, 0, 0};
		if (M.overflow) {
			if (M.m > 5) { P.flags[1] = 1; continue; }      // cannot happen: the margins of the front-truncated lookups are at most 5 symbols
			DeltaTable T;
			T.ep = tab + (size_t) st * 3 * HOT_TAB_ENTRIES; T.tm = T.ep + HOT_TAB_ENTRIES; T.slot = T.tm + HOT_TAB_ENTRIES;
			T.epoch = ++tab_epoch; T.m = M.m; T.lsh = M.lsh;
			delta_scan(D, reg, cur, e.time, T);
			const uint32_t n_keys = 4u << (2 * M.m);
			for (uint32_t kk = 0; kk < n_keys; ++kk) {
				if (T.ep[kk] != T.epoch) continue;
				const uint32_t loc = delta_count_at(D, T.slot[kk]);
				if (loc) c[kk & 3] = ci_plus(ci, c[kk & 3], loc, dc);
			}
		} else {
			for (uint32_t a = 1; a < M.n; ++a) {   // insertion sort by (trial, symbol)
				uint32_t kk = M.key[a], tt = M.tm[a], ss = M.slot[a]; uint32_t b = a;
				while (b > 0 && M.key[b - 1] > kk) { M.key[b] = M.key[b - 1]; M.tm[b] = M.tm[b - 1]; M.slot[b] = M.slot[b - 1]; --b; }
				M.key[b] = kk; M.tm[b] = tt; M.slot[b] = ss;
			}
			for (uint32_t a = 0; a < M.n; ++a) {
				uint32_t sym = M.key[a] & 3, loc = delta_count_at(D, M.slot[a]);
				if (loc) c[sym] = ci_plus(ci, c[sym], loc, dc);
			}
		}
		const uint32_t lev = st ? FQSK_LEVEL_SMER : FQSK_LEVEL_BMER;
		fqsk_base_rec *rec = P.prov + e.rec;
		if (rec->level != lev || rec->counts[0] != c[0] || rec->counts[1] != c[1] || rec->counts[2] != c[2] || rec->counts[3] != c[3]) {
			rec->counts[0] = c[0]; rec->counts[1] = c[1]; rec->counts[2] = c[2]; rec->counts[3] = c[3];
			rec->level = (uint8_t) lev;
			P.dirty[e.read] = 1;
			P.flags[6] = 1;
		}
	}
	P.hot_draws[st] = dc.used;
}

// ------------------------------------------------------------------------------------------------------------------
// k_sorted_dif: compress_prefix_sorted's (flag, dif) of every read that goes through CompressSorted (dna.cpp:589-605):
//   flag = 4 when the p-mer prefix equals the previous read's, else the prefix's field in the p-mer array;
//   dif  = how many p-mers strictly between the two prefixes hold that same field value.
// The reference counts with a linear scan over up to 4^p fields; here one CTA per read counts 16 fields per word, 4 words per load.
// (In a sorted file the ranges of consecutive reads are disjoint: over a whole input the array is read about once.)
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t siv_word_count_eq(uint32_t w, uint32_t flag) {      // fields of the word equal to flag
	const uint32_t x = w ^ (flag * 0x55555555u);
	return __popc(~(x | (x >> 1)) & 0x55555555u);
}
__global__ void __launch_bounds__(256) k_sorted_dif(EngineDev E, SegDev S) { pdl_enter();
	const uint32_t r = blockIdx.x, t = threadIdx.x;
	if (r >= S.n_reads) return;
	const bool sorted = item_sorted(S, E.sorted, r);
	if (S.dup[r] || !sorted) { if (t == 0) { S.sorted_flag[r] = 0; S.sorted_dif[r] = 0; } return; }
	const uint8_t *p = S.dna + S.off[r];
	unsigned long long cur_dir = 0;
	for (uint32_t i = 0; i < E.p; ++i) cur_dir |= (unsigned long long) sym_at(true, E, p, i) << (62 - 2 * i);
	unsigned long long prev_dir; bool prev_valid;
	const uint32_t back = S.iflags ? 3u : 1u;      // the previous read coded by CompressSorted: paired end -> the first mate of the previous pair
	if (r < back) { prev_dir = S.carry->pprev_dir; prev_valid = S.carry->pprev_valid != 0; }
	else {
		const uint8_t *q = S.dna + S.off[r - back];
		prev_dir = 0;
		for (uint32_t i = 0; i < E.p; ++i) { uint32_t sy = dna_code(q[i]); if (sy == 4) sy = 3; prev_dir |= (unsigned long long) sy << (62 - 2 * i); }
		prev_valid = true;
	}
	const uint64_t cur_al = cur_dir >> (64 - 2 * E.p);
	const uint64_t prev_al = prev_valid ? prev_dir >> (64 - 2 * E.p) : 0;
	const uint32_t flag = cur_dir == prev_dir ? 4u : siv_test(E.siv, cur_al);
	unsigned long long cnt = 0;
	const uint64_t lo = prev_al + 1, hi = cur_al;      // fields [lo, hi)
	if (flag < 4 && lo < hi && E.siv.world > 1) {
		// sharded p-mer array: consecutive runs of 2^top_shift fields belong to the ranks in turn (dna.cpp:845), a word (16 fields) never
		// spans two runs (top_shift >= 4, checked at create): every word is read from its owner's shard (NVLink peer mapping), one per thread
		const uint64_t w0 = lo >> 4, w1 = (hi - 1) >> 4;
		for (uint64_t wd = w0 + t; wd <= w1; wd += 256) {
			const uint32_t a = wd == w0 ? (uint32_t) (lo & 15) : 0u, b = wd == w1 ? (uint32_t) ((hi - 1) & 15) + 1u : 16u;      // fields [a, b) of this word
			uint64_t idx = wd << 4;
			const uint32_t *w = siv_shard(E.siv, idx);
			const uint32_t x = __ldg(w + (idx >> 4)) ^ (flag * 0x55555555u);
			uint32_t z = ~(x | (x >> 1)) & 0x55555555u;
			z &= (b == 16 ? 0xFFFFFFFFu : ((1u << (2 * b)) - 1u)) & ~((1u << (2 * a)) - 1u);
			cnt += (uint32_t) __popc(z);
		}
	} else if (flag < 4 && lo < hi) {
		const uint32_t *w = E.siv.w;                   // one array
		const uint64_t w0 = lo >> 4, w1 = (hi - 1) >> 4;      // first and last word touched
		auto masked = [&](uint64_t wd) {               // fields of word wd inside [lo, hi) that equal flag
			const uint32_t a = wd == w0 ? (uint32_t) (lo & 15) : 0u, b = wd == w1 ? (uint32_t) ((hi - 1) & 15) + 1u : 16u;      // fields [a, b) of this word
			const uint32_t x = __ldg(w + wd) ^ (flag * 0x55555555u);
			uint32_t z = ~(x | (x >> 1)) & 0x55555555u;
			z &= (b == 16 ? 0xFFFFFFFFu : ((1u << (2 * b)) - 1u)) & ~((1u << (2 * a)) - 1u);
			return (uint32_t) __popc(z);
		};
		if (w1 - w0 < 8) { if (t <= w1 - w0) cnt = masked(w0 + t); }
		else {
			if (t == 0) cnt += masked(w0);
			if (t == 1) cnt += masked(w1);
			// whole words (w0, w1): a head up to the next 16-byte boundary, uint4 loads, a tail
			const uint64_t a0 = w0 + 1, a1 = w1;       // [a0, a1)
			const uint64_t v0 = (a0 + 3) & ~3ull, v1 = a1 & ~3ull;
			if (v0 >= v1) { for (uint64_t wd = a0 + t; wd < a1; wd += 256) cnt += siv_word_count_eq(__ldg(w + wd), flag); }
			else {
				if (a0 + t < v0) cnt += siv_word_count_eq(__ldg(w + a0 + t), flag);
				if (v1 + t < a1) cnt += siv_word_count_eq(__ldg(w + v1 + t), flag);
				const uint4 *w4 = reinterpret_cast<const uint4 *>(w);
				uint64_t q = (v0 >> 2) + t;
				const uint64_t q1 = v1 >> 2;
				for (; q + 256 < q1; q += 512) {
					const uint4 x = __ldg(w4 + q), y = __ldg(w4 + q + 256);
					cnt += siv_word_count_eq(x.x, flag) + siv_word_count_eq(x.y, flag) + siv_word_count_eq(x.z, flag) + siv_word_count_eq(x.w, flag)
					     + siv_word_count_eq(y.x, flag) + siv_word_count_eq(y.y, flag) + siv_word_count_eq(y.z, flag) + siv_word_count_eq(y.w, flag);
				}
				for (; q < q1; q += 256) { const uint4 x = __ldg(w4 + q); cnt += siv_word_count_eq(x.x, flag) + siv_word_count_eq(x.y, flag) + siv_word_count_eq(x.z, flag) + siv_word_count_eq(x.w, flag); }
			}
		}
	}
	__shared__ unsigned long long part[8];
	for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
	if ((t & 31) == 0) part[t >> 5] = cnt;
	__syncthreads();
	if (t == 0) {
		unsigned long long tot = 0;
		for (int q = 0; q < 8; ++q) tot += part[q];
		S.sorted_flag[r] = flag; S.sorted_dif[r] = tot;
	}
}

// ------------------------------------------------------------------------------------------------------------------
// k_walk: one WARP per read, "speculative chunks with commit-prefix".
// The corrected registers of the reference are the registers of a CORRECTED READ: the original symbols with the patches
// made by repair_kmers_existing / repair_kmers_missing (dna.cpp:363-365, 442-446); a bmer_unc hit (dna.cpp:697-705) drops
// the patches that are still inside the b-mer window.  The warp keeps the last 64 corrected and original symbols in two
// shared-memory rings.  Each iteration the 32 lanes evaluate 32 consecutive positions in parallel from the rings as they
// are (registers, find_counts -- from the provisional record when corrected == uncorrected, from the tables otherwise --,
// pushes, repair decision).  The first lane whose position changes the rings (a repair or a bmer_unc revert) is the
// commit point: lanes up to it write their records and pushes, its event is applied to the ring, and the next chunk starts
// right behind it.  Everything a lane needs besides the rings (cor_pos, push counters) is constant up to the commit point,
// so committed lanes are exactly the reference's sequential steps.
// it == 0: every read; it > 0: only reads marked dirty, and any difference to the previous walk's pushes raises flags[2].
// ------------------------------------------------------------------------------------------------------------------
struct LaneRegs { KReg b; uint32_t cb; };

__device__ __forceinline__ KReg ring_breg(const uint8_t *ring, uint32_t i, uint32_t cb) {
	KReg r{0, 0};
	for (uint32_t t = 0; t + 1 < cb; ++t) {
		uint64_t sy = ring[(i + 1 - cb + t) & 63];
		r.dir |= sy << (62 - 2 * t);
		r.rc |= (3 - sy) << (64 - 2 * cb + 2 * t);
	}
	r.rc |= 3ull << 62;
	return r;
}

__global__ void __launch_bounds__(128) k_walk(EngineDev E, SegDev S, PipeDev P, uint32_t it) { pdl_enter();
	const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (r >= S.n_reads) return;
	if (it > 0) { if (!P.dirty[r]) return; }
	__syncwarp();
	if (lane == 0) P.dirty[r] = 0;
	const bool sorted = item_sorted(S, E.sorted, r);      // this read goes through CompressSorted (dna.cpp:1716-1754)
	if (S.dup[r]) { if (lane == 0) { S.cnt_b[r] = S.cnt_s[r] = S.cnt_p[r] = S.hidden[r] = 0; } return; }
	__shared__ uint8_t ringC_all[4][64], ringU_all[4][64];
	uint8_t *ringC = ringC_all[threadIdx.x >> 5], *ringU = ringU_all[threadIdx.x >> 5];
	const bool check = it > 0;
	bool changed = false, window_local = false;
	const uint8_t *p = S.dna + S.off[r];
	const uint32_t size = S.len[r];
	const uint32_t tbase = (uint32_t) S.off[r];
	unsigned long long *out_b = S.push_b + 2 * S.off[r];
	unsigned long long *out_s = S.push_s + S.off[r];
	unsigned long long *out_p = S.push_p + 2 * S.off[r] + 2ull * r;
	uint32_t *tim_b = P.time_b + 2 * S.off[r], *tim_s = P.time_s + S.off[r];
	const uint32_t g0 = (uint32_t) S.rec_off[r];
	uint32_t nb = 0, ns = 0, np = 0, hidden = 0;
	unsigned long long sl[4];
	for (int i = 0; i < 4; ++i) sl[i] = S.sl_base.v[i] + S.sl_prefix[r].v[i];
	int *unsupported = E.flags + 1;
	DrawCursor nodraw; nodraw.ring = nullptr; nodraw.mask = 0; nodraw.pos0 = 0; nodraw.avail = 0; nodraw.base = 0; nodraw.used = 0; nodraw.overflow = E.flags + 5;

	const uint32_t start = item_first(S, sorted ? E.p : E.prefix_len, r);
	const uint32_t bias = S.bias_a ? S.bias_a[r] : 0;      // record positions and cor_pos are in the frame of the whole mate (dna.cpp:1596)
	const bool seeded = (item_flags(S, r) & IF_SEEDED) != 0;
	uint32_t cor_pos = 0;
	// prefix: symbols enter the registers with N -> A (direct, cor_pos = position of the last N, dna.cpp:532-536) or N -> T (sorted, 560-565)
	{
		uint32_t npos = 0;
		for (uint32_t j = lane; j < start; j += 32) if (dna_code(p[j]) == 4) npos = j + 1;
		for (int o = 16; o; o >>= 1) { uint32_t y = __shfl_xor_sync(0xffffffffu, npos, o); npos = npos > y ? npos : y; }
		if (!sorted && npos && !seeded) cor_pos = npos - 1;
	}
	if (sorted) {      // flag / dif of compress_prefix_sorted come from k_sorted_dif; here only the two p-mer pushes of the prefix (dna.cpp:655-660)
		if (lane == 0) {
			unsigned long long cur_dir = 0, cur_rc = 0;
			for (uint32_t i = 0; i < E.p; ++i) cur_dir |= (unsigned long long) sym_at(sorted, E, p, i) << (62 - 2 * i);
			for (uint32_t i = 0; i < E.p; ++i) cur_rc |= (unsigned long long) (3 - sym_at(sorted, E, p, E.p - 1 - i)) << (62 - 2 * i);
			out_p[0] = cur_dir >> (64 - 2 * E.p); out_p[1] = cur_rc >> (64 - 2 * E.p);
		}
		np = 2;
	}
	// rings: positions [0, start + 32) that exist
	for (uint32_t j = lane; j < 64; j += 32) { ringC[j] = 0; ringU[j] = 0; }
	__syncwarp();
	uint32_t filled = 0;            // positions [.., filled) are in the rings
	uint32_t i0 = start;
	while (i0 < size) {
		// bring the rings up to position i0 + 31 (never more than 64 behind)
		uint32_t want = i0 + 32 < size ? i0 + 32 : size;
		uint32_t from = filled > (i0 >= 31 ? i0 - 31 : 0) ? filled : (i0 >= 31 ? i0 - 31 : 0);
		for (uint32_t j = from + lane; j < want; j += 32) { uint8_t sy = (uint8_t) sym_at(sorted, E, p, j); ringU[j & 63] = sy; ringC[j & 63] = sy; }
		filled = want;
		__syncwarp();
		const uint32_t i = i0 + lane;
		const bool valid = i < size;
		// the 64 ring symbols around the chunk as two packed words each (positions i0 - 32 .. i0 - 1 and i0 .. i0 + 31; positions that
		// do not exist are never inside a register): a lane's register is a funnel shift instead of 2 x 24 shared-memory loads
		uint64_t wU0, wU1, wC0, wC1;
		{
			const bool have_a = i0 + lane >= 32;
			const uint32_t sa = have_a ? ringU[(i0 + lane - 32) & 63] : 0, sb = ringU[(i0 + lane) & 63];
			const uint32_t ca = have_a ? ringC[(i0 + lane - 32) & 63] : 0, cbb = ringC[(i0 + lane) & 63];
			wU0 = pk_from_ballots(__ballot_sync(0xffffffffu, sa & 2u), __ballot_sync(0xffffffffu, sa & 1u));
			wU1 = pk_from_ballots(__ballot_sync(0xffffffffu, sb & 2u), __ballot_sync(0xffffffffu, sb & 1u));
			wC0 = pk_from_ballots(__ballot_sync(0xffffffffu, ca & 2u), __ballot_sync(0xffffffffu, ca & 1u));
			wC1 = pk_from_ballots(__ballot_sync(0xffffffffu, cbb & 2u), __ballot_sync(0xffffffffu, cbb & 1u));
		}
		// ---- per-lane evaluation of position i
		uint32_t lev = FQSK_LEVEL_NONE, c[4] = {0, 0, 0, 0};
		uint32_t sym = 4, cb = 0, cs = 0, cp = 0, lane_cor = cor_pos;
		bool ev_revert = false, ev_patch = false, repaired = false, lane_wl = false, lane_fmiss = false;
		int lane_unsup = 0;   // discarded (speculative) lanes must not raise global flags
		uint32_t patch_pos = 0, patch_sym = 0, new_cor = cor_pos;
		KReg bc{0, 0}, bu{0, 0};
		uint8_t rk = 0;
		bool push_b0 = false, push_s0 = false, push_p0 = false;
		uint32_t hid = 0;
		unsigned long long key_b0 = 0, key_s0 = 0, key_p0 = 0, key_p1 = 0, key_b1 = 0;
		if (valid) {
			const uint32_t n = i + 1;
			cb = n < E.b ? n : E.b; cs = n < E.s ? n : E.s; cp = n < E.p ? n : E.p;
			sym = dna_code(p[i]);
			const uint64_t ks = sym == 4 ? 0 : sym;
			const uint32_t a = 32 + lane + 1 - cb;                        // symbols i - cb + 1 .. i - 1 out of the 64 packed ones i0 - 32 .. i0 + 31
			bu = a < 32 ? breg_from_words(wU0, wU1, a, cb) : breg_from_words(wU1, 0ull, a, cb);
			bc = a < 32 ? breg_from_words(wC0, wC1, a, cb) : breg_from_words(wC1, 0ull, a, cb);
			const fqsk_base_rec pv = P.prov[g0 + (i - start)];
			if (bc.dir == bu.dir) {
				lev = pv.level; c[0] = pv.counts[0]; c[1] = pv.counts[1]; c[2] = pv.counts[2]; c[3] = pv.counts[3];
			} else {
				// repair window: cascade with the corrected registers (only reachable with a full b register)
				KReg sc = suffix_reg(bc, cb, cs);
				bool done = false;
				if (ht_find(E.hb, E.cib, bc, cb, c, nodraw)) {
					int sat = (c[0] == E.hb.top) + (c[1] == E.hb.top) + (c[2] == E.hb.top) + (c[3] == E.hb.top);
					if (sat > 1) { uint32_t c2[4]; ht_find(E.hs, E.cis, sc, cs, c2, nodraw); for (int q = 0; q < 4; ++q) c[q] += c2[q]; lev = FQSK_LEVEL_MIXED; }
					else lev = FQSK_LEVEL_BMER;
					done = true;
				} else {
					lane_wl = true;   // the thread-local table is consulted here: this read is re-walked when the delta exists / changes
					if (!delta_note(S.delta_b, bc, cb)) lane_fmiss = true;
					if (delta_find(S.delta_b, E.cib, bc, cb, 2 * (tbase + i), c, &lane_unsup)) { lev = FQSK_LEVEL_BMER; done = true; }
					if (!done && ht_find(E.hb, E.cib, bu, cb, c, nodraw)) { lev = FQSK_LEVEL_BMER_UNC; done = true; }
				}
				if (!done) {
					if (ht_find(E.hs, E.cis, sc, cs, c, nodraw)) lev = FQSK_LEVEL_SMER;
					else {
						if (!delta_note(S.delta_s, sc, cs)) lane_fmiss = true;
						if (delta_find(S.delta_s, E.cis, sc, cs, 2 * (tbase + i), c, &lane_unsup)) lev = FQSK_LEVEL_SMER;
					}
				}
				if (lev == FQSK_LEVEL_BMER_UNC) { bc = bu; ev_revert = true; lane_cor = 0; new_cor = 0; lev = FQSK_LEVEL_BMER; }   // dna.cpp:697-705
			}
			KReg sc = suffix_reg(bc, cb, cs), pc = suffix_reg(bc, cb, cp);
			if (lev == FQSK_LEVEL_NONE) {   // dna.cpp:709-735, deferred to k_rough
				if (cb == E.b) rk = 2; else if (cs == E.s) rk = 3; else if (cp == E.p) rk = 4;
			}
			KReg rq = rk == 2 ? bc : rk == 3 ? sc : pc;
			// the symbol becomes known (dna.cpp:810-816)
			kr_set_last(bc, cb, ks); kr_set_last(sc, cs, ks); kr_set_last(pc, cp, ks);
			if (sym < 4) {   // dna.cpp:818-852
				bool p_insert = true;
				if (cb == E.b) {
					push_b0 = true; key_b0 = kr_norm(bc, E.b);
					if ((lev == FQSK_LEVEL_SMER || lev == FQSK_LEVEL_BMER || lev == FQSK_LEVEL_MIXED) && c[sym] >= 3) p_insert = false;
				}
				if (cs == E.s) { push_s0 = true; key_s0 = kr_norm(sc, E.s); }
				if (cp == E.p && (i + bias) - lane_cor >= E.p - 1) {
					if (p_insert) { push_p0 = true; key_p0 = pc.dir >> (64 - 2 * E.p); key_p1 = pc.rc >> (64 - 2 * E.p); }
					else hid = 2;
				}
			}
			if (cb == E.b) {   // dna.cpp:854-875
				if (lev == FQSK_LEVEL_BMER || lev == FQSK_LEVEL_MIXED) {
					uint32_t best = 0;
					for (uint32_t q = 1; q < 4; ++q) if (c[q] > c[best] || (c[q] == c[best] && sl[q] > sl[best])) best = q;
					bool ok = true;
					if (sym != 4) ok = best != sym && c[sym] == 0 && c[best] > 3;
					if (ok) { kr_set_last(bc, cb, best); ev_patch = true; patch_pos = i; patch_sym = best; new_cor = i + bias; repaired = true; }
				} else if ((lev == FQSK_LEVEL_NONE || lev == FQSK_LEVEL_PMER) && E.gate_missing) {
					int best_c = 4, best_count = 0, best_j = 0;
					for (int j = 1; j < 6; ++j) {
						uint32_t cnts[4];
						uint64_t orig = kr_sym(bc, cb - 1 - j);
#pragma unroll
						for (uint64_t q = 0; q < 4; ++q) {
							cnts[q] = 0;
							if (q == orig) continue;
							KReg t = bc;
							kr_set(t, cb, q, cb - 1 - j);
							cnts[q] = ht_count(E.hb, kr_norm(t, E.b));
						}
						for (int q = 0; q < 4; ++q) {
							if ((uint64_t) q == orig) continue;
							int cnt = (int) cnts[q];
							if (cnt >= best_count && cnt >= 2) { best_c = q; best_count = cnt; best_j = j; }
						}
					}
					if (best_j) {
						kr_set(bc, cb, best_c, cb - 1 - best_j);
						ev_patch = true; patch_pos = i - (uint32_t) best_j; patch_sym = (uint32_t) best_c;
						uint32_t np2 = i + bias - (uint32_t) best_j;
						new_cor = lane_cor > np2 ? lane_cor : np2;
						repaired = true;
					}
				}
				if (repaired) key_b1 = kr_norm(bc, E.b);
			}
			(void) rq;
		}
		// ---- commit point (all 32 lanes participate in the collectives)
		const bool ev = valid && (ev_revert || ev_patch);
		const unsigned evm = __ballot_sync(0xffffffffu, ev);
		const unsigned vm = __ballot_sync(0xffffffffu, valid);
		const uint32_t last_valid = 31 - __clz(vm);
		const uint32_t f = evm ? (uint32_t) (__ffs(evm) - 1) : last_valid;
		const bool commit = valid && lane <= f;
		const unsigned below = (1u << lane) - 1u;
		const unsigned mb0 = __ballot_sync(0xffffffffu, commit && push_b0), mb1 = __ballot_sync(0xffffffffu, commit && repaired);
		const unsigned ms0 = __ballot_sync(0xffffffffu, commit && push_s0), mp0 = __ballot_sync(0xffffffffu, commit && push_p0);
		if (commit) {
			if (lane_unsup) *unsupported = 1;
			window_local |= lane_wl;
			if (lane_fmiss && S.delta_b.n) P.flags[2] = 1;   // the filtered delta was built without this context: one more pass (the bit is set now)
			const uint32_t g = g0 + (i - start);
			fqsk_base_rec o;
			o.pos = i + bias; o.counts[0] = c[0]; o.counts[1] = c[1]; o.counts[2] = c[2]; o.counts[3] = c[3];
			o.cor_pos = lane_cor; o.level = (uint8_t) lev; o.rough = 0; o.pad = 0;
			P.recs[g] = o;
			P.rkind[g] = check ? (uint8_t) (rk | 0x80u) : rk;      // 0x80: written by a re-walk (the rough searches that started after walk 0 redo it)
			if (rk) {
				// register before the symbol became known: rebuild from the (possibly reverted) corrected view
				KReg bq = ev_revert ? ring_breg(ringU, i, cb) : ring_breg(ringC, i, cb);
				P.rreg[g] = rk == 2 ? bq : rk == 3 ? suffix_reg(bq, cb, cs) : suffix_reg(bq, cb, cp);
			}
			// pushes: positions of earlier lanes first; inside a position: b, [repaired b]
			uint32_t ib = nb + __popc(mb0 & below) + __popc(mb1 & below);
			// push time = 2 * position (+1 for the repaired b-mer, which the reference pushes second: dna.cpp:822-826 vs 858-873)
			const uint32_t tpos = 2 * (tbase + i);
			if (push_b0) { if (check) changed |= (out_b[ib] != key_b0) | (tim_b[ib] != tpos); out_b[ib] = key_b0; tim_b[ib] = tpos; ++ib; }
			if (repaired) { if (check) changed |= (out_b[ib] != key_b1) | (tim_b[ib] != tpos + 1); out_b[ib] = key_b1; tim_b[ib] = tpos + 1; }
			uint32_t is = ns + __popc(ms0 & below);
			if (push_s0) { if (check) changed |= (out_s[is] != key_s0) | (tim_s[is] != tpos); out_s[is] = key_s0; tim_s[is] = tpos; }
			uint32_t ip = np + 2 * __popc(mp0 & below);
			if (push_p0) { out_p[ip] = key_p0; out_p[ip + 1] = key_p1; }
		}
		nb += __popc(mb0) + __popc(mb1); ns += __popc(ms0); np += 2 * __popc(mp0);
		{
			uint32_t hsum = commit ? hid : 0;
			for (int o = 16; o; o >>= 1) hsum += __shfl_xor_sync(0xffffffffu, hsum, o);
			hidden += hsum;
		}
		// ---- apply the event of lane f to the corrected ring and continue right behind it
		if (evm) {
			const uint32_t e_rev = __shfl_sync(0xffffffffu, (uint32_t) ev_revert, f);
			const uint32_t e_pat = __shfl_sync(0xffffffffu, (uint32_t) ev_patch, f);
			const uint32_t e_pos = __shfl_sync(0xffffffffu, patch_pos, f), e_sym = __shfl_sync(0xffffffffu, patch_sym, f);
			cor_pos = __shfl_sync(0xffffffffu, new_cor, f);
			const uint32_t i_f = i0 + f;
			__syncwarp();
			if (e_rev) {   // corrected registers := uncorrected ones: drop every patch inside the b window of position i_f
				uint32_t lo = i_f + 1 >= E.b ? i_f + 1 - E.b : 0;
				for (uint32_t j = lo + lane; j <= i_f; j += 32) ringC[j & 63] = ringU[j & 63];
			}
			__syncwarp();
			if (e_pat && lane == 0) ringC[e_pos & 63] = (uint8_t) e_sym;
			__syncwarp();
			i0 = i_f + 1;
		} else {
			i0 += 32;
		}
		__syncwarp();      // the next iteration refills ring slots that lanes of this one may still be reading (commit block)
	}
	changed = __any_sync(0xffffffffu, changed);
	window_local = __any_sync(0xffffffffu, window_local);
	if (lane == 0) {
		if (check && (changed || S.cnt_b[r] != nb || S.cnt_s[r] != ns)) P.flags[2] = 1;
		S.cnt_b[r] = nb; S.cnt_s[r] = ns; S.cnt_p[r] = np; S.hidden[r] = hidden;
		if (window_local) { P.dirty[r] = 1; if (it == 0) P.flags[3] = 1; }
	}
}

__global__ void k_compact2(SegDev S, PipeDev P, const uint32_t *off_b, const uint32_t *off_s, const uint32_t *off_p,
                           unsigned long long *row_b, unsigned long long *row_s, unsigned long long *row_p, uint32_t *rt_b, uint32_t *rt_s) { pdl_enter();
	uint32_t r = blockIdx.x;
	if (r >= S.n_reads) return;
	const unsigned long long *sb = S.push_b + 2 * S.off[r], *ss = S.push_s + S.off[r], *sp = S.push_p + 2 * S.off[r] + 2ull * r;
	const uint32_t *tb = P.time_b + 2 * S.off[r], *ts = P.time_s + S.off[r];
	for (uint32_t i = threadIdx.x; i < S.cnt_b[r]; i += blockDim.x) { row_b[off_b[r] + i] = sb[i]; rt_b[off_b[r] + i] = tb[i]; }
	for (uint32_t i = threadIdx.x; i < S.cnt_s[r]; i += blockDim.x) { row_s[off_s[r] + i] = ss[i]; rt_s[off_s[r] + i] = ts[i]; }
	for (uint32_t i = threadIdx.x; i < S.cnt_p[r]; i += blockDim.x) row_p[off_p[r] + i] = sp[i];
}
// delta build straight from the per-read push regions: one warp per read, one entry per push, placed by the canonical
// inner core of its k-mer
__global__ void __launch_bounds__(128) k_delta_build(SegDev S, PipeDev P, unsigned long long *kb, uint32_t *tb, uint32_t mask_b, uint32_t k_b, uint32_t t_b,
                                                     unsigned long long *ks, uint32_t *ts, uint32_t mask_s, uint32_t k_s, uint32_t t_s) { pdl_enter();
	uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (r >= S.n_reads) return;
	const unsigned long long *sb = S.push_b + 2 * S.off[r], *ss = S.push_s + S.off[r];
	const uint32_t *qb = P.time_b + 2 * S.off[r], *qs = P.time_s + S.off[r];
	const uint32_t *fb = S.delta_b.filter, *fs = S.delta_s.filter;
	for (uint32_t j = lane; j < S.cnt_b[r]; j += 32) {
		unsigned long long x = sb[j];
		if (fb) { const uint32_t q = delta_fbit_of_key(x, k_b, t_b, S.delta_b.fmask); if (!((__ldg(fb + (q >> 5)) >> (q & 31)) & 1u)) continue; }
		for (uint64_t slot = delta_slot_of_key(x, k_b, t_b, mask_b);; slot = (slot + 1) & mask_b)
			if (atomicCAS(tb + slot, DELTA_EMPTY, qb[j]) == DELTA_EMPTY) { kb[slot] = x; break; }
	}
	for (uint32_t j = lane; j < S.cnt_s[r]; j += 32) {
		unsigned long long x = ss[j];
		if (fs) { const uint32_t q = delta_fbit_of_key(x, k_s, t_s, S.delta_s.fmask); if (!((__ldg(fs + (q >> 5)) >> (q & 31)) & 1u)) continue; }
		for (uint64_t slot = delta_slot_of_key(x, k_s, t_s, mask_s);; slot = (slot + 1) & mask_s)
			if (atomicCAS(ts + slot, DELTA_EMPTY, qs[j]) == DELTA_EMPTY) { ks[slot] = x; break; }
	}
}

// the same for small segments, one thread per slot of the push regions: a segment of a few hundred reads has too few warps to
// hide the latency of a warp-per-read loop, but tens of thousands of pushes
__global__ void __launch_bounds__(256) k_delta_build_flat(SegDev S, PipeDev P, uint32_t slots_total, unsigned long long *kb, uint32_t *tb, uint32_t mask_b, uint32_t k_b, uint32_t t_b,
                                                          unsigned long long *ks, uint32_t *ts, uint32_t mask_s, uint32_t k_s, uint32_t t_s) { pdl_enter();
	const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;      // slot of the b regions, then of the s regions: [0, 2T) [2T, 3T), T = bytes of the segment
	if (g >= 3 * slots_total) return;
	const bool is_b = g < 2 * slots_total;
	const uint32_t j = is_b ? g : g - 2 * slots_total;
	const uint32_t at = is_b ? j >> 1 : j;                           // byte offset whose read owns the slot (regions: b at 2 * off, s at off)
	uint32_t lo = 0, hi = S.n_reads;                                 // last read with off <= at
	while (hi - lo > 1) { uint32_t m = (lo + hi) >> 1; if ((uint32_t) S.off[m] <= at) lo = m; else hi = m; }
	const uint32_t r = lo;
	if (is_b) {
		const uint32_t i = j - 2 * (uint32_t) S.off[r];
		if (i >= S.cnt_b[r]) return;
		const unsigned long long x = S.push_b[j];
		const uint32_t tm = P.time_b[j];
		for (uint64_t slot = delta_slot_of_key(x, k_b, t_b, mask_b);; slot = (slot + 1) & mask_b)
			if (atomicCAS(tb + slot, DELTA_EMPTY, tm) == DELTA_EMPTY) { kb[slot] = x; break; }
	} else {
		const uint32_t i = j - (uint32_t) S.off[r];
		if (i >= S.cnt_s[r]) return;
		const unsigned long long x = S.push_s[j];
		const uint32_t tm = P.time_s[j];
		for (uint64_t slot = delta_slot_of_key(x, k_s, t_s, mask_s);; slot = (slot + 1) & mask_s)
			if (atomicCAS(ts + slot, DELTA_EMPTY, tm) == DELTA_EMPTY) { ks[slot] = x; break; }
	}
}

// ------------------------------------------------------------------------------------------------------------------
// k_rough: one warp per request.  find_counts_rough_{s,b} (dna.cpp:257-330): 4(k-1) single-substitution neighbours across the
// lanes, non-empty ones appended in trial order to a merge script; find_counts_rough_p (dna.cpp:229-254) is a plain sum.
// ------------------------------------------------------------------------------------------------------------------
// only_marked = 0: every flagged position.  The first pass of a small segment starts this right behind walk 0, on a side stream next
// to the thread-local pass (delta, k_local, walk 1); positions the re-walk wrote carry the 0x80 marker and are done again afterwards
// with only_marked = 1 (their first scripts stay behind unreferenced).  Nothing here writes records: k_fold does.
// DEEP = false: one survivor per lane and round (sparse tables: a third of the trials survive the occupancy bits, one round; 55 registers);
// DEEP = true: up to four sector reads per lane in flight (dense tables: every trial survives, the kernel lives on memory-level parallelism)
template <bool DEEP>
__global__ void __launch_bounds__(128, 8) k_rough(EngineDev E, PipeDev P, uint32_t only_marked) { pdl_enter();   // E.hb / E.hs carry occ_read while the tables are sparse (HtDev::occ)
	const uint32_t lane = threadIdx.x & 31;
	const uint32_t n_rec = *P.n_rec_dev;
	const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
	__shared__ Script stage[4];
	__shared__ uint64_t surv_h_all[4][128];      // per warp: bucket hash of the trials that can hit, in trial order
	__shared__ uint8_t surv_m_all[4][128];       //           trial number | orientation << 7
	Script &sc = stage[threadIdx.x >> 5];
	uint64_t *surv_h = surv_h_all[threadIdx.x >> 5];
	uint8_t *surv_m = surv_m_all[threadIdx.x >> 5];
	const uint32_t RCHUNK = 4;      // positions per warp iteration: small, so that a tiny segment still spreads over every SM
	for (uint32_t g0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * RCHUNK; g0 < n_rec; g0 += warps * RCHUNK) {
		// each warp owns RCHUNK consecutive positions: find the flagged ones, then work on them one at a time with all lanes
		uint32_t mine = (lane < RCHUNK && g0 + lane < n_rec) ? P.rkind[g0 + lane] : 0;
		mine = only_marked ? ((mine & 0x80u) ? (mine & 0x7Fu) : 0u) : (mine & 0x7Fu);
		if (mine < 2 || mine > 4) mine = 0;      // (a value torn by a concurrent re-walk is redone by the marked pass)
		KReg myreg{0, 0};
		if (mine) myreg = P.rreg[g0 + lane];       // all registers of the chunk in one round trip, handed out by shuffles below
		unsigned todo = __ballot_sync(0xffffffffu, mine != 0);
		while (todo) {
			uint32_t q = __ffs(todo) - 1;
			todo &= todo - 1;
			const uint32_t g = g0 + q;
			const uint32_t kind = __shfl_sync(0xffffffffu, mine, q);
			KReg reg;
			reg.dir = __shfl_sync(0xffffffffu, myreg.dir, q); reg.rc = __shfl_sync(0xffffffffu, myreg.rc, q);
			if (kind == 4) {
				uint32_t c[4] = {0, 0, 0, 0};
				uint32_t trials = 4 * (E.p - 1);
				for (uint32_t t = lane; t < trials; t += 32) {
					KReg tr = reg;
					kr_set(tr, E.p, t & 3, t >> 2);
					siv_counts(E.siv, tr.dir >> (64 - 2 * E.p), c, true);
				}
				for (int qq = 0; qq < 4; ++qq) for (int o = 16; o; o >>= 1) c[qq] += __shfl_xor_sync(0xffffffffu, c[qq], o);
				if (lane == 0) {
					uint32_t slot = 0xFFFFFFFFu;
					if (any4(c)) {      // at most 3 * 4 (p - 1) per symbol: fits the script's u16 entries
						slot = atomicAdd(P.n_rscript, 1u);
						if (slot >= P.rscript_cap) { P.flags[4] = 1; slot = 0xFFFFFFFFu; }
						else {
							sc.rec = g; sc.kind = 4; sc.valid = 1; sc.n = 1; sc.overflow = 0xFFFFFFFFu; sc.draws = 0;
							for (int qq = 0; qq < 4; ++qq) { sc.c2[qq] = 0; sc.e[0][qq] = (uint16_t) c[qq]; }
							P.rscripts[slot] = sc;
						}
					}
					P.rslot[g] = slot;
				}
				__syncwarp();
				continue;
			}
			const HtDev &t = kind == 2 ? E.hb : E.hs;
			const uint32_t trials = 4 * (t.k - 1);      // <= 128
			uint32_t n_ent = 0, ovf = 0xFFFFFFFFu;
			// Phase 1: every trial's bucket hash (the expensive part: two 64-bit multiplies) is computed ONCE; while the table is sparse the
			// bucket-occupancy bit (L2-resident) decides which trials can hit at all.  The survivors -- about a third of the 4(k-1) trials in
			// the first blocks of a file -- are compacted, in trial order, into the warp's list in shared memory.
			// Phase 2: one survivor per lane: its sector is read and compared; non-empty results are appended to the script in list order =
			// trial order (dna.cpp:283-287, 321-325).  (Before: three rounds of 32 trials, every hash computed twice: issue bound.)
			uint32_t n_surv = 0;
			for (uint32_t u = 0; u * 32 < trials; ++u) {
				const uint32_t tn = u * 32 + lane;
				// a trial that puts the original symbol back is the context itself, which the global table has just failed to
				// answer (the level is `none`): known empty, no read
				bool keep = tn < trials && (tn & 3) != kr_sym(reg, tn >> 2);
				uint64_t hsh = 0; bool isd = false;
				if (keep) {
					KReg tr = reg;
					kr_set(tr, t.k, tn & 3, tn >> 2);
					isd = kr_is_dir(tr, t.k);
					hsh = ht_mix(t, ht_kernel(t, isd ? tr.dir : tr.rc));
					if (t.occ_read) { const uint64_t bucket = hsh >> t.rem_bits; keep = ((__ldg(t.occ_read + (bucket >> 5)) >> (bucket & 31)) & 1u) != 0; }
				}
				const unsigned m = __ballot_sync(0xffffffffu, keep);
				if (keep) { const uint32_t at = n_surv + __popc(m & ((1u << lane) - 1u)); surv_h[at] = hsh; surv_m[at] = (uint8_t) (tn | (isd ? 0x80u : 0u)); }
				n_surv += __popc(m);
			}
			__syncwarp();
			if (!DEEP) {
				for (uint32_t s0 = 0; s0 < n_surv; s0 += 32) {
					uint32_t loc[4] = {0, 0, 0, 0};
					if (s0 + lane < n_surv) {
						const uint32_t meta = surv_m[s0 + lane], tn = meta & 0x7Fu;
						const bool isd = (meta & 0x80u) != 0;
						KReg tr = reg;
						kr_set(tr, t.k, tn & 3, tn >> 2);
						const uint64_t x = isd ? tr.dir : tr.rc;
						HtKey key;
						key.h = surv_h[s0 + lane];
						key.bucket = key.h >> t.rem_bits;
						key.q = 0x80000000u | ((uint32_t) (key.h & ((1ull << t.rem_bits) - 1)) << (8 + t.cbits)) | (ht_ends(t, x) << t.cbits);
						key.kal = x >> (64 - 2 * t.k);
						key.owner = ht_owner(t.world, x);
						const uint4 *bp = reinterpret_cast<const uint4 *>(t.peer_main[key.owner] + key.bucket * 8);
						Bucket bk; bk.lo = __ldg(bp); bk.hi = __ldg(bp + 1);
						ht_ctx_counts_from(t, key, isd, bk, loc);
					}
					script_append(P, sc, n_ent, ovf, loc, any4(loc), n_surv - s0);
				}
			} else {
				// up to four survivors per lane: all their sector reads are issued before the first one is consumed (dense tables let every
				// trial through: 4(k-1) reads per request, and the kernel lives on memory-level parallelism)
				for (uint32_t s0 = 0; s0 < n_surv; s0 += 128) {
					Bucket bk[4];
	#pragma unroll
					for (int u = 0; u < 4; ++u) {
						const uint32_t i = s0 + u * 32 + lane;
						if (i < n_surv) {
							const uint32_t meta = surv_m[i], tn = meta & 0x7Fu;
							KReg tr = reg;
							kr_set(tr, t.k, tn & 3, tn >> 2);
							const uint32_t owner = ht_owner(t.world, (meta & 0x80u) ? tr.dir : tr.rc);
							const uint4 *bp = reinterpret_cast<const uint4 *>(t.peer_main[owner] + (surv_h[i] >> t.rem_bits) * 8);
							bk[u].lo = __ldg(bp); bk[u].hi = __ldg(bp + 1);
						}
					}
	#pragma unroll
					for (int u = 0; u < 4; ++u) {
						if (s0 + u * 32 >= n_surv) break;
						const uint32_t i = s0 + u * 32 + lane;
						uint32_t loc[4] = {0, 0, 0, 0};
						if (i < n_surv) {
							const uint32_t meta = surv_m[i], tn = meta & 0x7Fu;
							const bool isd = (meta & 0x80u) != 0;
							KReg tr = reg;
							kr_set(tr, t.k, tn & 3, tn >> 2);
							const uint64_t x = isd ? tr.dir : tr.rc;
							HtKey key;
							key.h = surv_h[i];
							key.bucket = key.h >> t.rem_bits;
							key.q = 0x80000000u | ((uint32_t) (key.h & ((1ull << t.rem_bits) - 1)) << (8 + t.cbits)) | (ht_ends(t, x) << t.cbits);
							key.kal = x >> (64 - 2 * t.k);
							key.owner = ht_owner(t.world, x);
							ht_ctx_counts_from(t, key, isd, bk[u], loc);
						}
						script_append(P, sc, n_ent, ovf, loc, any4(loc), n_surv - (s0 + u * 32));
					}
				}
			}
			__syncwarp();
			if (lane == 0) {
				uint32_t slot = 0xFFFFFFFFu;
				if (n_ent) {
					slot = atomicAdd(P.n_rscript, 1u);
					if (slot >= P.rscript_cap) { P.flags[4] = 1; slot = 0xFFFFFFFFu; }
					else {
						sc.rec = g; sc.kind = (uint8_t) kind; sc.valid = 1; sc.n = (uint16_t) n_ent; sc.overflow = ovf;
						for (int qq = 0; qq < 4; ++qq) sc.c2[qq] = 0;
						P.rscripts[slot] = sc;
					}
				}
				P.rslot[g] = slot;
			}
			__syncwarp();
		}
	}
}

// ------------------------------------------------------------------------------------------------------------------
// k_fold: one thread per read replays the ordered approximate-counter merges of that read's scripts (front-truncated
// lookups first, then the rough searches, each in position order = the reference's program order per PRNG stream) with
// their exact positions in the mt19937 streams.  pass 0 counts the draws of the read (offset-independent unless a counter
// saturates); after a scan over reads pass 1 evaluates with the true offsets, writes the final counts and re-reports the
// totals so the host can confirm the offsets.
// ------------------------------------------------------------------------------------------------------------------
// write: 0 = count the draws only, 1 = write the record, 2 = write it if the merge consumed no draw (its result then does not depend
// on where the read's scripts sit in the mt19937 stream: final without the scan over reads)
__device__ void fold_script(const EngineDev &E, const PipeDev &P, const Script &sc, DrawCursor &dc, int write) {
	const bool is_b = (sc.kind == 0 || sc.kind == 2);
	const bool rough = sc.kind >= 2;
	const CIncP ci = is_b ? E.cib : E.cis;
	uint32_t c[4] = {0, 0, 0, 0};
	if (sc.kind == 4) {      // find_counts_rough_p (dna.cpp:229-254): a plain sum, already formed by k_rough
		if (!write) return;
		for (int q = 0; q < 4; ++q) c[q] = sc.e[0][q];
		fqsk_base_rec *rec = P.recs + sc.rec;
		rec->counts[0] = c[0]; rec->counts[1] = c[1]; rec->counts[2] = c[2]; rec->counts[3] = c[3];
		rec->level = FQSK_LEVEL_PMER; rec->rough = 1;
		return;
	}
	for (uint32_t n = 0; n < sc.n; ++n) {
		uint32_t loc[4];
		if (n < SCRIPT_INLINE) { for (int q = 0; q < 4; ++q) loc[q] = sc.e[n][q]; }
		else { const unsigned short *d = P.pool + 4ull * (sc.overflow + (n - SCRIPT_INLINE)); for (int q = 0; q < 4; ++q) loc[q] = d[q]; }
		for (int q = 0; q < 4; ++q) if (rough || loc[q]) c[q] = ci_plus(ci, c[q], loc[q], dc);
	}
	if (!write || (write == 2 && dc.used)) return;
	fqsk_base_rec *rec = P.recs + sc.rec;
	uint32_t lev = rec->level;
	if (rough) { if (!any4(c)) return; lev = FQSK_LEVEL_PMER; rec->rough = 1; }
	else if (sc.kind == 0) {      // a found front-truncated b lookup is level bmer (never inside a repair window: the register is not full), or mixed;
		                          // written afresh, so that a merge evaluated again with other draws cannot inherit `mixed` from its first evaluation
		int sat = (c[0] == ci.top) + (c[1] == ci.top) + (c[2] == ci.top) + (c[3] == ci.top);
		lev = FQSK_LEVEL_BMER;
		if (sat > 1) { for (int q = 0; q < 4; ++q) c[q] += sc.c2[q]; lev = FQSK_LEVEL_MIXED; }
	}
	rec->counts[0] = c[0]; rec->counts[1] = c[1]; rec->counts[2] = c[2]; rec->counts[3] = c[3];
	rec->level = (uint8_t) lev;
}

__device__ __forceinline__ uint32_t warp_excl_sum(uint32_t v, uint32_t lane, uint32_t &total) {
	uint32_t x = v;
	for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
	total = __shfl_sync(0xffffffffu, x, 31);
	return x - v;
}

// One warp per read, one LANE per script: the scripts of a read are visited in program order (front-truncated lookups by
// position, then rough searches by position) 32 at a time.  pass 0 folds every script from offset 0 to count its draws;
// pass 1 gives every script its exact offset (read offset from the scan over reads + the counts of the scripts before it)
// and writes the final counts.  A count that differs from the stored one (a counter saturated) raises flags[7]: the host
// scans and runs pass 1 again.
__global__ void __launch_bounds__(128) k_fold(EngineDev E, SegDev S, PipeDev P, int pass) { pdl_enter();
	const uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
	if (r >= S.n_reads) return;
	if (pass && P.rdraws_b[r] == 0 && P.rdraws_s[r] == 0) return;      // no draws in this read: pass 0 has written its records
	uint32_t used[2] = {0, 0};          // draws of the scripts visited so far, per stream (b, s), as assumed by the offsets
	uint32_t now[2] = {0, 0};           // ... as consumed by this pass
	bool mismatch = false;
	const unsigned long long base[2] = {pass ? P.doff_b[r] : 0ull, pass ? P.doff_s[r] : 0ull};
	auto batch = [&](Script *sp) {      // warp-collective; sp == nullptr for idle lanes
		uint32_t st = 0, stored = 0;
		if (sp) { st = (sp->kind == 0 || sp->kind == 2) ? 0 : 1; stored = pass ? sp->draws : 0; }
		uint32_t tot0, tot1;
		uint32_t ex0 = warp_excl_sum(sp && st == 0 ? stored : 0, lane, tot0);
		uint32_t ex1 = warp_excl_sum(sp && st == 1 ? stored : 0, lane, tot1);
		uint32_t cnt = 0;
		if (sp) {
			DrawCursor dc;
			dc.ring = E.draws[st]; dc.mask = E.dmask[st]; dc.pos0 = E.dpos[st]; dc.avail = E.avail[st]; dc.used = 0; dc.overflow = E.flags + 0;
			dc.base = base[st] + used[st] + (st ? ex1 : ex0);
			fold_script(E, P, *sp, dc, pass != 0 ? 1 : 2);
			cnt = dc.used;
			if (pass == 0) sp->draws = cnt;
			else if (cnt != stored) { sp->draws = cnt; mismatch = true; }
		}
		uint32_t c0 = sp && st == 0 ? cnt : 0, c1 = sp && st == 1 ? cnt : 0;
		for (int o = 16; o; o >>= 1) { c0 += __shfl_xor_sync(0xffffffffu, c0, o); c1 += __shfl_xor_sync(0xffffffffu, c1, o); }
		now[0] += c0; now[1] += c1;
		if (pass == 0) { used[0] += c0; used[1] += c1; } else { used[0] += tot0; used[1] += tot1; }
	};
	if (!S.dup[r]) {
		// front-truncated lookups: slots are in position order
		Script *ps = P.pscripts + (size_t) r * P.pslots;
		for (uint32_t s0 = 0; s0 < P.pslots; s0 += 32) {
			Script *sp = (s0 + lane < P.pslots && ps[s0 + lane].valid) ? ps + s0 + lane : nullptr;
			if (__any_sync(0xffffffffu, sp != nullptr)) batch(sp);
		}
		// rough searches of this read, in position order.  The kind / script-slot loads of 8 chunks are issued together: a segment of
		// a few hundred reads has one warp per read and nothing to hide the latency of chunk-by-chunk dependent loads behind.
		const uint32_t g0 = (uint32_t) S.rec_off[r], g1 = (uint32_t) S.rec_off[r + 1];
		for (uint32_t gs = g0; gs < g1; gs += 256) {
			uint32_t kk[8], slot[8];
#pragma unroll
			for (int c = 0; c < 8; ++c) { const uint32_t g = gs + c * 32 + lane; kk[c] = g < g1 ? (P.rkind[g] & 0x7Fu) : 0; }
#pragma unroll
			for (int c = 0; c < 8; ++c) { const uint32_t g = gs + c * 32 + lane; slot[c] = kk[c] >= 2 ? P.rslot[g] : 0xFFFFFFFFu; }
#pragma unroll
			for (int c = 0; c < 8; ++c) {
				if (gs + c * 32 >= g1) break;
				if (__any_sync(0xffffffffu, slot[c] != 0xFFFFFFFFu)) batch(slot[c] != 0xFFFFFFFFu ? P.rscripts + slot[c] : nullptr);
			}
		}
	}
	mismatch = __any_sync(0xffffffffu, mismatch);
	if (lane) return;
	if (pass == 0 || mismatch) { P.rdraws_b[r] = now[0]; P.rdraws_s[r] = now[1]; }
	if (pass && mismatch) P.flags[7] = 1;
}

// Block-wide exclusive scan helper: every thread owns ITEMS consecutive elements (serial), warp shuffles + one smem round
// combine the per-thread sums; `carry` threads the running total through the chunks of a long array.
template <typename T, int NQ, int ITEMS>
__device__ __forceinline__ void block_scan_chunk(T (&v)[NQ][ITEMS], T (&ex)[NQ][ITEMS], T (*sh)[32], T *carry) {
	const uint32_t t = threadIdx.x, lane = t & 31, w = t >> 5;
	T tsum[NQ], inc[NQ];
	for (int q = 0; q < NQ; ++q) {
		T run = 0;
		for (int e = 0; e < ITEMS; ++e) { ex[q][e] = run; run += v[q][e]; }
		tsum[q] = run;
		T x = run;
		for (int o = 1; o < 32; o <<= 1) { T y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
		inc[q] = x;
		if (lane == 31) sh[q][w] = x;
	}
	__syncthreads();
	if (w == 0) {
		for (int q = 0; q < NQ; ++q) {
			T x = sh[q][lane];
			for (int o = 1; o < 32; o <<= 1) { T y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
			sh[q][lane] = x;
		}
	}
	__syncthreads();
	for (int q = 0; q < NQ; ++q) {
		T base = carry[q] + (w ? sh[q][w - 1] : 0) + inc[q] - tsum[q];
		for (int e = 0; e < ITEMS; ++e) ex[q][e] += base;
	}
	__syncthreads();
	if (t < NQ) carry[t] += sh[t][31];
	__syncthreads();
}

// Scans over per-read arrays, one CTA per chunk of 1024 * ITEMS reads (a single CTA is bound by what one SM can pull from
// HBM: 0.28 ms for 51 000 reads).  Every CTA scans its chunk, publishes the chunk totals tagged with the launch epoch and adds
// up the totals of the CTAs before it (cta_chain_prefix).  Grids are small (<= 2 CTAs per SM), so all CTAs are co-resident and
// waiting for lower-numbered ones cannot deadlock.
struct ScanChain { unsigned long long *vals; uint32_t *flags; uint32_t epoch; };     // vals[cta][8], flags[cta]
static const uint32_t SCAN_CHAIN_MAX = 256;

template <int NQ>
__device__ __forceinline__ void cta_chain_prefix(const ScanChain &C, const unsigned long long *mine /* shared, [NQ] */, unsigned long long (&pre)[NQ], unsigned long long (*sh)[32]) {
	const uint32_t b = blockIdx.x, t = threadIdx.x, lane = t & 31, w = t >> 5, nw = blockDim.x >> 5;
	if (gridDim.x == 1) { for (int q = 0; q < NQ; ++q) pre[q] = 0; return; }      // small segments: one chunk, nothing to chain
	if (t == 0) {
		for (int q = 0; q < NQ; ++q) C.vals[b * 8 + q] = mine[q];
		__threadfence();
		atomicExch(C.flags + b, C.epoch);
	}
	unsigned long long acc[NQ];
	for (int q = 0; q < NQ; ++q) acc[q] = 0;
	for (uint32_t c = t; c < b; c += blockDim.x) {
		while (*((volatile uint32_t *) (C.flags + c)) != C.epoch) { }
		__threadfence();
		for (int q = 0; q < NQ; ++q) acc[q] += *((volatile unsigned long long *) (C.vals + c * 8 + q));
	}
	for (int q = 0; q < NQ; ++q) {
		for (int o = 16; o; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
		if (lane == 0) sh[q][w] = acc[q];
	}
	__syncthreads();
	for (int q = 0; q < NQ; ++q) { unsigned long long x = 0; for (uint32_t i = 0; i < nw; ++i) x += sh[q][i]; pre[q] = x; }
	__syncthreads();
}

__global__ void __launch_bounds__(1024) k_scan_reads(SegDev S, unsigned long long *rec_off, U64x4 *sl_prefix, SegTotals *tot, uint32_t *n_rec_dev, ScanChain C) { pdl_enter();
	const int IT = 4;
	__shared__ unsigned long long sh[5][32];
	__shared__ unsigned long long carry[5];
	const uint32_t t = threadIdx.x;
	if (t < 5) carry[t] = 0;
	if (t < 32) for (int q = 0; q < 5; ++q) sh[q][t] = 0;       // CTAs of fewer than 32 warps (small segments)
	__syncthreads();
	const uint32_t base = blockIdx.x * blockDim.x * IT;
	unsigned long long v[5][IT], ex[5][IT];
	for (int e = 0; e < IT; ++e) {
		uint32_t r = base + t * IT + e;
		if (r < S.n_reads) { v[0][e] = S.n_coded[r]; U64x4 L = S.letters[r]; v[1][e] = L.v[0]; v[2][e] = L.v[1]; v[3][e] = L.v[2]; v[4][e] = L.v[3]; }
		else { v[0][e] = v[1][e] = v[2][e] = v[3][e] = v[4][e] = 0; }
	}
	block_scan_chunk<unsigned long long, 5, IT>(v, ex, sh, carry);      // carry = totals of this chunk
	unsigned long long pre[5];
	cta_chain_prefix<5>(C, carry, pre, sh);
	for (int e = 0; e < IT; ++e) {
		uint32_t r = base + t * IT + e;
		if (r < S.n_reads) { rec_off[r] = pre[0] + ex[0][e]; U64x4 o; o.v[0] = pre[1] + ex[1][e]; o.v[1] = pre[2] + ex[2][e]; o.v[2] = pre[3] + ex[3][e]; o.v[3] = pre[4] + ex[4][e]; sl_prefix[r] = o; }
	}
	if (t == 0 && blockIdx.x == gridDim.x - 1) {
		rec_off[S.n_reads] = pre[0] + carry[0];
		U64x4 o; o.v[0] = pre[1] + carry[1]; o.v[1] = pre[2] + carry[2]; o.v[2] = pre[3] + carry[3]; o.v[3] = pre[4] + carry[4];
		sl_prefix[S.n_reads] = o;
		tot->n_rec = pre[0] + carry[0]; tot->letters = o;
		*n_rec_dev = (uint32_t) (pre[0] + carry[0]);
	}
}

// up to 4 u32 arrays -> exclusive scans (u32) + totals
static const uint32_t SCAN_U32_CHUNK = 1024 * 8, SCAN_READS_CHUNK = 1024 * 4;
__global__ void __launch_bounds__(1024) k_scan_u32x4(uint32_t n, const uint32_t *a0, uint32_t *o0, const uint32_t *a1, uint32_t *o1,
                                                     const uint32_t *a2, uint32_t *o2, const uint32_t *a3, uint32_t *o3, uint32_t *totals, uint32_t *zero_me, ScanChain C) { pdl_enter();
	const int IT = 8;
	__shared__ unsigned long long sh[4][32];
	__shared__ unsigned long long carry[4];
	const uint32_t t = threadIdx.x;
	const uint32_t *in[4] = {a0, a1, a2, a3};
	uint32_t *out[4] = {o0, o1, o2, o3};
	if (t < 4) carry[t] = 0;
	if (t < 32) for (int q = 0; q < 4; ++q) sh[q][t] = 0;       // CTAs of fewer than 32 warps (small segments)
	__syncthreads();
	const uint32_t base = blockIdx.x * blockDim.x * IT;
	unsigned long long v[4][IT], ex[4][IT];
	for (int q = 0; q < 4; ++q) for (int e = 0; e < IT; ++e) { uint32_t r = base + t * IT + e; v[q][e] = (in[q] && r < n) ? in[q][r] : 0; }
	block_scan_chunk<unsigned long long, 4, IT>(v, ex, sh, carry);
	unsigned long long pre[4];
	cta_chain_prefix<4>(C, carry, pre, sh);
	for (int q = 0; q < 4; ++q) if (out[q]) for (int e = 0; e < IT; ++e) { uint32_t r = base + t * IT + e; if (r < n) out[q][r] = (uint32_t) (pre[q] + ex[q][e]); }
	if (blockIdx.x == gridDim.x - 1) {
		if (t < 4) { if (out[t]) out[t][n] = (uint32_t) (pre[t] + carry[t]); totals[t] = (uint32_t) (pre[t] + carry[t]); }
		if (t == 0 && zero_me) *zero_me = 0;
	}
}

// per-read draw counts (u32) -> exclusive scans (u64) + totals
__global__ void __launch_bounds__(1024) k_scan_draws(uint32_t n, const uint32_t *a0, unsigned long long *o0, const uint32_t *a1, unsigned long long *o1, unsigned long long *totals,
                                                     int *flags, ScanChain C) { pdl_enter();
	const int IT = 8;
	__shared__ unsigned long long sh[2][32];
	__shared__ unsigned long long carry[2];
	const uint32_t t = threadIdx.x;
	const uint32_t *in[2] = {a0, a1};
	unsigned long long *out[2] = {o0, o1};
	if (t < 2) carry[t] = 0;
	if (t < 32) for (int q = 0; q < 2; ++q) sh[q][t] = 0;       // CTAs of fewer than 32 warps (small segments)
	__syncthreads();
	const uint32_t base = blockIdx.x * blockDim.x * IT;
	unsigned long long v[2][IT], ex[2][IT];
	for (int q = 0; q < 2; ++q) for (int e = 0; e < IT; ++e) { uint32_t r = base + t * IT + e; v[q][e] = r < n ? in[q][r] : 0; }
	block_scan_chunk<unsigned long long, 2, IT>(v, ex, sh, carry);
	unsigned long long pre[2];
	cta_chain_prefix<2>(C, carry, pre, sh);
	for (int q = 0; q < 2; ++q) for (int e = 0; e < IT; ++e) { uint32_t r = base + t * IT + e; if (r < n) out[q][r] = pre[q] + ex[q][e]; }
	if (blockIdx.x == gridDim.x - 1) {
		if (t < 2) { out[t][n] = pre[t] + carry[t]; totals[t] = pre[t] + carry[t]; }
		if (t == 0 && flags) { flags[0] = 0; flags[7] = 0; }      // draw window short / offsets moved: k_fold pass 1 reports them afresh
	}
}

// draw flags (u8, push order) -> exclusive scan = draw index of every occurrence; n lives on the device.  Chained scan: every
// CTA scans 4096 flags, publishes its sum tagged with the launch epoch and adds up the sums of the CTAs before it.  The grid
// comes from a host-side bound and is small enough to be co-resident (rows that take this path are at most SYNC_INDEXED_MAX
// long), so waiting on lower-numbered CTAs cannot deadlock.
static const uint32_t SCANF_TILE = 4096;
__global__ void __launch_bounds__(256) k_scan_flags(const SyncIn *in, const uint32_t *n_dev, const uint8_t *flag, uint32_t *out, uint32_t *total,
                                                    unsigned long long *partials, uint32_t epoch, SyncDev Y, CIncP ci) { pdl_enter();
	const uint32_t n = in->ok_pre ? *n_dev : 0;
	const uint32_t b = blockIdx.x, t = threadIdx.x, lane = t & 31, w = t >> 5;
	const uint32_t base = b * SCANF_TILE;
	if (base >= n) { if (b == 0 && t == 0) { out[0] = 0; *total = 0; } return; }
	__shared__ uint32_t wsum[8];
	__shared__ uint32_t bprefix;
	const uint32_t r0 = base + t * 16;
	uint32_t v[16];
	if (r0 + 16 <= n) {
		const uint4 q = *reinterpret_cast<const uint4 *>(flag + r0);     // flag arrays are 16-byte aligned, r0 is a multiple of 16
		const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
		for (int e = 0; e < 16; ++e) v[e] = (wd[e >> 2] >> (8 * (e & 3))) & 0xFF;
	} else {
#pragma unroll
		for (int e = 0; e < 16; ++e) v[e] = r0 + e < n ? flag[r0 + e] : 0;
	}
	uint32_t run = 0;
#pragma unroll
	for (int e = 0; e < 16; ++e) { uint32_t x = v[e]; v[e] = run; run += x; }
	uint32_t inc = run;
	for (int o = 1; o < 32; o <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
	if (lane == 31) wsum[w] = inc;
	__syncthreads();
	uint32_t woff = 0, bsum = 0;
#pragma unroll
	for (int q = 0; q < 8; ++q) { if (q < (int) w) woff += wsum[q]; bsum += wsum[q]; }
	if (t == 0) {
		__threadfence();
		atomicExch(partials + b, ((unsigned long long) epoch << 32) | bsum);
	}
	// prefix of the CTAs before this one
	uint32_t pre = 0;
	for (uint32_t q = t; q < b; q += 256) {
		unsigned long long x;
		do { x = *((volatile unsigned long long *) (partials + q)); } while ((uint32_t) (x >> 32) != epoch);
		pre += (uint32_t) x;
	}
	for (int o = 16; o; o >>= 1) pre += __shfl_xor_sync(0xffffffffu, pre, o);
	__syncthreads();
	if (lane == 0) wsum[w] = pre;
	__syncthreads();
	if (t == 0) { uint32_t x = 0; for (int q = 0; q < 8; ++q) x += wsum[q]; bprefix = x; }
	__syncthreads();
	const uint32_t off = bprefix + woff + inc - run;
	if (r0 + 16 <= n) {
		uint4 *o4 = reinterpret_cast<uint4 *>(out + r0);
#pragma unroll
		for (int e = 0; e < 4; ++e) o4[e] = make_uint4(off + v[4 * e], off + v[4 * e + 1], off + v[4 * e + 2], off + v[4 * e + 3]);
	} else {
		for (int e = 0; e < 16; ++e) if (r0 + e < n) out[r0 + e] = off + v[e];
	}
	if (base + SCANF_TILE >= n && t == 0) { out[n] = bprefix + bsum; *total = bprefix + bsum; }
	// former k_sync_scatter: every occurrence of a hot group leaves its draw index and flag at its own delta entry, where the
	// group's leader reads them in time order (k_sync_apply)
	for (int e = 0; e < 16; ++e) {
		const uint32_t j = r0 + e;
		if (j >= n) break;
		const uint32_t L = Y.lead[j];
		if (Y.lead_c0[L] + Y.lead_m[L] <= ci.thr + 1) continue;
		const uint32_t own = Y.own[j];
		Y.draw_at[own] = off + v[e];
		Y.flag_at[own] = flag[j];
	}
}

// ------------------------------------------------------------------------------------------------------------------
// k_ctx_codes (SURVEY 8 row f1): the context ids of the DNA stream on the device.  One thread per coded base turns the final record
// into the 16-byte fqsk_ctx_rec of include/fqsk_ctx.h: cor_zone, the counts quantised at the four resolutions of
// determine_ctx_codes, let_max, the rank of the true symbol and the recent-rank history (the ranks of the 8 bases before it,
// recomputed from their records: they are neighbours in memory), dna.cpp:737-774, code_ctx.cpp:257-338.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool ctx_base(const SegDev &S, const PipeDev &P, const EngineDev &E, uint32_t r, uint32_t g, uint32_t first, const uint8_t *p, uint32_t lb, const unsigned long long sl[4],
                                         uint32_t &rsym, uint32_t &sym_out, uint32_t &n_run_out, fqsk_base_rec &rec) {
	// coded with counts? (dna.cpp:737) + the rank; i = position inside the item's text
	const uint32_t i = first + (g - (uint32_t) S.rec_off[r]);
	rec = P.recs[g];
	const uint32_t sym = dna_code(p[i]);
	uint32_t n_run = 0;      // N_run_len: Ns right before i, counted from the first position this call walked (sorted prefix included)
	for (uint32_t j = i; j > lb && dna_code(p[j - 1]) == 4 && n_run < 2; --j) ++n_run;
	sym_out = sym; n_run_out = n_run;
	const bool coded = rec.level != FQSK_LEVEL_NONE && n_run < 2;
	uint64_t s64[4] = {sl[0], sl[1], sl[2], sl[3]};
	rsym = coded ? fqsk_ctx_rank(rec.counts, s64, sym) : 4u;
	return coded;
}
__global__ void __launch_bounds__(256) k_ctx_codes(EngineDev E, SegDev S, PipeDev P, fqsk_ctx_rec *out) { pdl_enter();
	const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t n_rec = *P.n_rec_dev;
	if (g >= n_rec) return;
	const uint32_t r = find_read(S.rec_off, S.n_reads, g, n_rec);
	const bool sorted = item_sorted(S, E.sorted, r);
	const uint32_t first = item_first(S, sorted ? E.p : E.prefix_len, r);
	const uint32_t g0 = (uint32_t) S.rec_off[r];
	const uint8_t *p = S.dna + S.off[r];
	const uint32_t lb = sorted ? 0u : first;
	unsigned long long sl[4];
	for (int q = 0; q < 4; ++q) sl[q] = S.sl_base.v[q] + S.sl_prefix[r].v[q];
	// ctx_r_sym (dna.cpp:664-671, 774, 800): bit j = the base j + 1 positions back was coded with counts and ranked first
	uint32_t r_hist = 0;
	for (uint32_t j = 1; j <= 8 && g >= g0 + j; ++j) {
		uint32_t rs, sy, nr; fqsk_base_rec pr;
		if (ctx_base(S, P, E, r, g - j, first, p, lb, sl, rs, sy, nr, pr) && rs == 0) r_hist |= 1u << (j - 1);
	}
	uint32_t rs, sym, n_run; fqsk_base_rec rec;
	ctx_base(S, P, E, r, g, first, p, lb, sl, rs, sym, n_run, rec);
	const uint32_t fl = item_flags(S, r);
	const uint32_t bias = S.bias_a ? S.bias_a[r] : 0;
	const uint32_t i = rec.pos;                              // the coder's loop index (frame of the whole mate)
	uint32_t pos = i, read_len = S.len[r] + bias;
	if (fl & IF_REVCOMP) { pos = S.len[r] - (i - bias) - 1; read_len = 0xFFFFFFFFu; }      // dna.cpp:750-752
	uint64_t s64[4] = {sl[0], sl[1], sl[2], sl[3]};
	out[g] = fqsk_ctx_make(rec.counts, rec.level, rec.rough, rec.cor_pos, i, pos, read_len, sym, n_run, r_hist, s64, E.p, E.s, E.b);
}

// the host's look at the device: the status block into its page-locked mirror, then -- after a system-wide fence -- the sequence
// number the host is spinning on
__global__ void __launch_bounds__(128) k_publish(const EngineStatus *status, EngineStatus *out, unsigned long long *seq, unsigned long long want) { pdl_enter();
	const uint32_t *src = reinterpret_cast<const uint32_t *>(status);
	uint32_t *dst = reinterpret_cast<uint32_t *>(out);
	for (uint32_t i = threadIdx.x; i < sizeof(EngineStatus) / 4; i += blockDim.x) dst[i] = src[i];
	__threadfence_system();
	__syncthreads();
	if (threadIdx.x == 0) { *reinterpret_cast<volatile unsigned long long *>(seq) = want; __threadfence_system(); }
}
// a segment evaluated again (retry): the reset k_prep did for the first evaluation
__global__ void k_seg_reset(EngineStatus *status) { pdl_enter();
	seg_reset_words(status, threadIdx.x);
}
// Verdict of a segment's first pass for the sync that is enqueued behind it without a host look + the state the next segment
// inherits (read_prev, dna.cpp:1550-1551; in sorted order pmer_can_prev, dna.cpp:655), in one launch.  The pass settled when no
// flag asks for another iteration, a retry or the ordered thread-local evaluator.
__global__ void __launch_bounds__(256) k_seg_tail(const int *flags, const uint32_t *tot4, const unsigned long long *draws2, unsigned long long consumed_b, unsigned long long consumed_s,
                                                  uint32_t row_cap, SyncIn *in, SegDev S, uint32_t last, uint8_t *prev_read, Carry *carry, uint32_t sorted, uint32_t p,
                                                  uint32_t have_prefix, uint32_t force_fail) { pdl_enter();
	if (threadIdx.x == 0) {
		bool ok = !(flags[0] | flags[1] | flags[2] | flags[4] | flags[5] | flags[7]) && !force_fail;      // force_fail: fault injection (tests)
		if (tot4[0] > row_cap || tot4[1] > row_cap) ok = false;
		in->n_b = tot4[0]; in->n_s = tot4[1]; in->n_p = tot4[2];
		in->dpos_b = consumed_b + draws2[0]; in->dpos_s = consumed_s + draws2[1];
		in->ok = ok ? 1u : 0u;
		if (!have_prefix) { in->ok_pre = ok ? 1u : 0u; in->draws_b = 0; }     // otherwise k_pre_verdict has set ok_pre and the early flag scan has
		                                                                      // already left the row's draw total in draws_b
	}
	if (S.n_reads == 0) return;
	const uint8_t *q = S.dna + S.off[last];      // paired-end: only first-of-pair reads replace read_prev (dna.cpp:1550-1551)
	const uint32_t n = S.len[last];
	for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) prev_read[i] = q[i];
	if (threadIdx.x == 32) {
		carry->prev_len = n;
		if (sorted) {
			unsigned long long d = 0;
			for (uint32_t i = 0; i < p; ++i) { uint32_t sy = dna_code(q[i]); if (sy == 4) sy = 3; d |= (unsigned long long) sy << (62 - 2 * i); }
			carry->pprev_dir = d; carry->pprev_valid = 1;
		}
	}
}
// Walk-level verdict, available as soon as the pushes are compacted: no flag asks for another walk, a retry or the ordered
// thread-local evaluator, and the rows fit the indexed ordered insert.  The pushes are final then (what can still fail -- the
// merges of k_fold -- only touches records and draw counts), so k_sync_rank / k_sync_flags / k_scan_flags may run.
__global__ void k_pre_verdict(const int *flags, const uint32_t *tot4, uint32_t row_cap, SyncIn *in) { pdl_enter();
	if (threadIdx.x || blockIdx.x) return;
	bool ok = !(flags[1] | flags[2] | flags[4] | flags[5]);
	if (tot4[0] > row_cap || tot4[1] > row_cap) ok = false;
	in->n_b = tot4[0]; in->n_s = tot4[1]; in->n_p = tot4[2];
	in->draws_b = 0;
	in->ok = 0;
	in->ok_pre = ok ? 1u : 0u;
}
__global__ void k_set_syncin(SyncIn *in, uint32_t n_b, uint32_t n_s, uint32_t n_p, unsigned long long dpos_b, unsigned long long dpos_s) { pdl_enter();
	if (threadIdx.x || blockIdx.x) return;
	in->ok = 1; in->ok_pre = 1; in->n_b = n_b; in->n_s = n_s; in->n_p = n_p; in->dpos_b = dpos_b; in->dpos_s = dpos_s; in->draws_b = 0;
}

}  // namespace fqsk
