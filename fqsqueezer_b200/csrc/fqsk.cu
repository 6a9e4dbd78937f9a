// fqsk.cu -- host orchestration + C-ABI (include/fqsk.h) of the B200 k-mer statistics engine.
//
// The reference (refresh-bio/fqsqueezer 1.1) runs its k-mer engine sequentially, read after read, with three kinds of
// order-dependent state inside a sync segment: the thread-local delta tables, the mt19937 streams behind the approximate
// counters, and the running A/C/G/T totals.  Here a segment is replayed for all reads in parallel against
//   (a) the frozen global tables in HBM,
//   (b) a delta built from the PREVIOUS iteration's pushes (sorted by k-mer, then push index), and
//   (c) per-read draw offsets obtained by an exclusive scan of the PREVIOUS iteration's per-read draw counts,
// and iterated until pushes and draw counts reproduce themselves: at that fixed point every read has seen exactly the state
// the sequential reference would have shown it, so records, pushes and PRNG positions are bit-exact (DESIGN.md section 5).
// There is no CPU fallback anywhere in this file.
#include <algorithm>
#include <atomic>
#include <cctype>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "fqsk_pipeline.cuh"
#include "fqsk_front.cuh"
#include "fqsk_pe.cuh"
#include "fqsk_mtjump.h"
#include <mutex>

using namespace fqsk;

static thread_local std::string g_create_error;

namespace {

static std::atomic<bool> g_trace_alloc{false};      // FQSK_F_TRACE_ALLOC of any live handle

struct DevBuf {
	void *p = nullptr;
	size_t cap = 0;
	cudaError_t ensure(size_t bytes, int line = __builtin_LINE()) {
		if (bytes <= cap) return cudaSuccess;
		if (g_trace_alloc.load(std::memory_order_relaxed)) fprintf(stderr, "[fqsk alloc] line %d: %zu -> %zu bytes\n", line, cap, bytes);
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		size_t want = bytes + bytes / 2 + 256;
		cudaError_t e = cudaMalloc(&p, want);
		if (e == cudaSuccess) cap = want;
		return e;
	}
	cudaError_t ensure_keep(size_t bytes, cudaStream_t st) {   // grows without losing the contents
		if (bytes <= cap) return cudaSuccess;
		size_t want = bytes + bytes / 2 + 256;
		void *np = nullptr;
		cudaError_t e = cudaMalloc(&np, want);
		if (e != cudaSuccess) return e;
		if (p) { cudaMemcpyAsync(np, p, cap, cudaMemcpyDeviceToDevice, st); cudaStreamSynchronize(st); cudaFree(p); }
		p = np; cap = want;
		return cudaSuccess;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
	template <typename T> T *as() const { return (T *) p; }
};

struct Stream {            // one mt19937 stream (utils.h:257, seeded 5481 at utils.h:298): tempered outputs in an HBM ring buffer,
	uint32_t *buf = nullptr;   // generated ahead of use on a side CUDA stream
	uint32_t *state = nullptr;
	uint64_t cap = 0, generated = 0, consumed = 0;   // cap is a power of two; absolute positions
	uint64_t safe = 0;         // outputs below this position are known to be complete for the main stream (it waited for them)
	cudaEvent_t ev = nullptr;  // completion of the latest generation launch
	bool ev_pending = false;   // the main stream has not waited for `ev` yet
	uint32_t *jstates = nullptr;   // parallel extension: the states MT_PAR chunks ahead (k_mt_jump)
};
const uint32_t MT_PAR = 32, MT_CHUNK_BLOCKS = 420;      // long extensions: 32 CTAs x 420 blocks x 624 outputs = 8.4 M outputs per launch

struct Table {
	HtDev d{};
	MixInv inv{};
	CIncP ci{};
};

enum { ST_B = 0, ST_S = 1, ST_LB = 2, ST_LS = 3 };

struct SegCtx {            // everything the passes of one segment share (host side)
	SegDev S{}; PipeDev P{}; EngineDev E{};
	uint32_t n = 0, first = 0, it = 0, pass = 0, slots_b = 0, slots_s = 0, t_b = 0, t_s = 0;
	uint64_t dna_bytes_actual = 0;
	bool redo_walk = true, redo_tail = true;
};

struct LookBuf {           // page-locked, device-accessible: what the host reads back of the device
	EngineStatus st;       // mirror of the status block: k_publish fills all of it, a copy of one field lands in that field
	alignas(64) unsigned long long seq;   // sequence number of the last published look (k_publish stores it after st); on a cache
	                                      // line of its own: the host spins on it while k_publish writes st
	uint32_t insert_draws;    // draw total of an ordered insert row (draw_off[n]): not a status word
};

}  // namespace

struct fqsk_handle {
	fqsk_params P{};
	cudaStream_t st = nullptr, st_mt = nullptr;
	std::string err;
	Table tb, ts;
	SivDev siv{};
	Stream rng[4];
	EngineStatus *status = nullptr;      // the small device words of host-side control, read by the host in ONE look
	fqsk_stats S{};
	unsigned long long sl_base[4] = {0, 0, 0, 0};   // s_letters (dna.h:92, dna.cpp:2047-2057)
	uint64_t hidden_p = 0;                           // no_pmer_hidden_updates (dna.cpp:850, 2417)
	// previous read / previous prefix p-mer carried across segments
	DevBuf prev_read;
	// segment buffers
	DevBuf dna, off, len, dup, n_coded, letters, rec_off, sl_prefix, recs, push_b, push_s, push_p, cnt_b, cnt_s, cnt_p, hidden,
	       draw_cnt, draw_cnt_prev, draw_scan, off_b[2], off_s[2], off_p, row_b[2], row_s[2], row_p, dk_b, di_b, dk_s, di_s, iota, cub_tmp,
	       flag8, draw_off, final_cnt, slot_of, dump_k, dump_v, q0, q1, q2, q3, q4, sflag, sdif, hid_scan,
	       prov, pflags, pscripts, rscripts, rreqs, pool, miss, draws_b16, draws_s16, doff_b, doff_s, time_b, time_s, rt_b[2], rt_s[2],
	       sidx_b, sidx_s, stime_b, stime_s, sort_k, sort_v, rkind, rreg, rslot, dirty, rdraws_b, rdraws_s, totals,
	       y_tslot, y_c0, y_m, y_draw, y_j, y_final, y_flag_at, y_own, y_lead, y_rank, y_flag, y_doff, idx_k, idx_t, idx_rt,
	       miss_fold, hr_b[3], hr_s[3], evk[2], evv[2], evk_s[2], evv_s[2];
	unsigned long long look_seq = 0;         // sequence number of the last published look (k_publish)
	bool look_fresh = false;                 // look->st holds the status block as of the end of everything enqueued so far
	SegCtx ctx;                              // the segment being evaluated
	bool unsettled = false;                  // its first pass is enqueued, nobody has looked at the outcome yet
	bool miss_fold_dirty = true; void *miss_fold_seen = nullptr;
	uint32_t world = 1, rank = 0;            // reference worker `rank` of `world` (one per GPU)
	bool dev_finish = false;             // fqsk_sync_device: the apply step ends with the device-side second barrier
	unsigned long long sync_seq = 0;      // number of the sharded sync under way (posted to the owners' inbox headers)
	unsigned long long *inbox = nullptr; uint64_t inbox_cap = 0;      // this rank's inbox: header + [3 tables][world sources][inbox_cap]
	unsigned long long *peer_inbox[8] = {nullptr};
	void *peer_ptrs[8][8] = {{nullptr}};     // IPC mappings to close
	uint32_t attached = 0;                   // bit i: rank i's shard is mapped
	DevBuf route_keys, route_keys2, route_sorted, route_hist, route_perm, route_chunks;
	DevBuf hot_tab;      // k_hot_eval: direct-indexed match table of a front-truncated thread-local lookup with many completions
	uint64_t sync_fresh = 0, sync_updates = 0; bool routed = false, applied = false;
	// coordinated doubling of sharded tables: grow_local = what this rank's shards ask for after a sync (bit 0 s-mers, 1 b-mers, 2 pairs),
	// grow_all = the OR over all ranks (every shard of a table has the same geometry: all grow or none), grow_pending = fqsk_sync_finish has
	// returned FQSK_RESHARD and the doubling itself happens in the fqsk_shard_export that follows
	uint32_t grow_local = 0, grow_all = 0; bool grow_pending = false;
	uint32_t crowd_shift = 0;                // FQSK_F_TEST_CROWD: 6 -- tables double at 1/64 of the usual load (growth on small fixtures)
	uint64_t siv_local_filled = 0;           // non-zero fields of THIS rank's p-mer shard (S.siv_no_filled is the global statistic)
	DevBuf scan_vals; uint32_t scan_epoch2 = 0;
	DevBuf scan_part; uint32_t scan_epoch = 0;   // published CTA sums of k_scan_flags, tagged with the launch epoch
	DevBuf scan8_part; uint32_t scan8_epoch = 0; // ... of k_scan_u8
	DevBuf rdx_hist, rdx_k, rdx_v;               // radix partition (fqsk_sort.cuh): tile histograms + digit totals, ping-pong buffers
	bool hot = false;                        // the current segment is being redone with the ordered thread-local evaluator
	bool hot_seen[2] = {false, false};       // [0] s, [1] b: the last sync saw a k-mer pushed more than thr + 1 times in its row
	DeltaDev seg_delta_b{}, seg_delta_s{};   // the converged segment's delta tables (valid while `pending`)
	uint32_t miss_cap = 0, rreq_cap = 0, pool_cap = 1u << 18;
	bool fast_ok[2] = {true, true};     // [0] s-mers, [1] b-mers: the atomic fast path has not been refuted yet
	bool delta_b_valid = false, delta_s_valid = false;   // dk_b/sidx_b (dk_s/sidx_s) hold the pending row sorted by k-mer
	uint32_t iota_n = 0;
	// pending rows (device), valid after fqsk_segment until fqsk_sync
	bool pending = false;
	int cur = 0;                          // which of row_b/row_s/off_b/off_s holds the converged iteration
	uint32_t pend_b = 0, pend_s = 0, pend_p = 0;
	uint64_t n_recs = 0;
	uint32_t seg_reads = 0;
	// paired-end (fqsk_pe.cuh): the global pair table, the segment's sorted triples, the per-pair decisions and the work items
	PairDev pair{}; uint64_t pair_items = 0;
	DevBuf pe_uk, pe_uv, pe_uc;              // sharded sync: distinct (key, value, weight) rows of the segment before routing
	DevBuf pe_tk, pe_tv, pe_q, pe_sk, pe_sv, pe_sidx, pe_t1, pe_t2, pe_pool, pe_info, it_src, it_len, it_bytes, it_first, it_bias, it_dupprev,
	       it_flags, it_off32, it_off64, it_dna;
	uint32_t pe_pool_cap = 1u << 20, pe_pairs = 0, pe_nt = 0, seg_reads_in = 0;
	// the sync enqueued behind its segment (sync_spec_enqueue / sync_spec_finish)
	unsigned long long items_main[2] = {0, 0};   // items in the buckets of the b / s table as of the last look (sparse -> k_rough tests occupancy bits)
	cudaStream_t st_side[3] = {nullptr, nullptr, nullptr}; cudaEvent_t ev_side[3] = {nullptr, nullptr, nullptr}, ev_fork = nullptr, ev_aux = nullptr;   // p-mer / s-mer updates of a small sync
	bool spec_enqueued = false; SyncDev spec_Y{}; uint32_t spec_g = 0;
	uint32_t dbg_fail_every = 0, dbg_retry_every = 0, dbg_seg = 0;   // fault injection for tests (FQSK_F_TEST_HOOKS + fqsk_params.test_hooks): see fqsk_create
	bool dbg_retry_armed = false;
	bool spec_prefix = false;                // the grouping half of the pending segment's b-mer sync was enqueued with the segment (seg_pass)
	bool seg_extra_pass = false;             // the last segment needed more than its first pass: records were rewritten after the pass
	// fqsk_submit / fqsk_collect: double-buffered records, copies on their own stream
	DevBuf pk;                                       // 2-bit packed reads of the segment (k_prep)
	// fqsk_announce_device: k_prep / k_scan_reads of the NEXT segment run on a side stream while the segment in flight is still being evaluated;
	// their outputs (dup, n_coded, letters, rec_off, sl_prefix, packed reads, totals) therefore exist twice, a segment uses instance seg_par
	DevBuf f_dup, f_n_coded, f_letters, f_rec_off, f_sl_prefix, f_pk;
	int seg_par = 0;
	struct Front { bool valid = false; const uint8_t *dna = nullptr; uint64_t bytes = 0; const unsigned long long *off = nullptr; const uint32_t *len = nullptr; uint32_t n = 0; int par = 0; } front;
	cudaStream_t st_front = nullptr; cudaEvent_t ev_front = nullptr;
	// fqsk_submit: the reads of segment n + 1 go to the device (their own buffer, the front stream) and are prepared there while segment n is
	// still in flight; block_fresh: fqsk_block_start has cleared read_prev and no segment has run since (nothing may be prepared ahead)
	DevBuf dna2; cudaEvent_t ev_up = nullptr; bool block_fresh = false;
	DevBuf dfilter; bool delta_filtered = false;     // filter bits of the segment's delta (large segments), see seg_setup
	DevBuf recs_alt; int rec_par = 0;
	DevBuf ctxrec[2];                                // fqsk_submit_ctx: the 16-byte context records of the segment in flight, per parity
	cudaStream_t st_copy = nullptr; cudaEvent_t ev_recs = nullptr, ev_copied[2] = {nullptr, nullptr}, ev_meta = nullptr; bool meta_pending = false;
	uint8_t *h_stage2 = nullptr; size_t h_stage2_cap = 0;       // second pinned staging buffer (H2D of segment n + 1 while n is still needed)
	uint8_t *h_meta[2] = {nullptr, nullptr}; size_t h_meta_cap[2] = {0, 0};   // pinned per-ticket copies of dup / rec_off (item arrays in paired-end mode)
	struct Ticket { bool open = false, done = false; fqsk_ctx_rec *ctx = nullptr; fqsk_base_rec *recs = nullptr; uint64_t bound = 0, n_recs = 0; uint8_t *dup = nullptr; uint64_t *rec_off = nullptr; uint32_t n_reads = 0; int par = 0; uint64_t id = 0; } tk[2];
	bool tk_open = false; int tk_cur = 0; uint64_t tk_next = 1;
	int tk_info = -1;                        // ticket (parity) whose per-read extras (sorted prefix, pair decisions) fqsk_sorted_prefix / fqsk_pair_info serve; -1: the last blocking segment
	// pinned staging
	uint8_t *h_stage = nullptr; size_t h_stage_cap = 0;
	LookBuf *look = nullptr;              // the host's page-locked mirror of `status` (look)
	// profiling
	bool prof = false;
	bool trace_launch = false;      // FQSK_F_TRACE_LAUNCH
	bool serial = false;            // FQSK_F_SERIAL: no side streams
	double ph_ms[FQSK_PH_COUNT] = {0};
	struct Ev { cudaEvent_t a, b; int ph; };
	std::vector<Ev> evs;
	std::vector<cudaEvent_t> ev_pool;
	cudaEvent_t t0 = nullptr, t1 = nullptr;
};

namespace {

inline bool mode_pe(uint32_t m) { return m == FQSK_MODE_PE_ORIGINAL || m == FQSK_MODE_PE_SORTED; }
inline bool mode_sorted(uint32_t m) { return m == FQSK_MODE_SE_SORTED || m == FQSK_MODE_PE_SORTED; }

int fail(fqsk_handle *h, int code, const char *fmt, ...) {
	char b[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(b, sizeof b, fmt, ap);
	va_end(ap);
	if (h) h->err = b; else g_create_error = b;
	return code;
}
#define CK(call)                                                                                            \
	do {                                                                                                    \
		cudaError_t e_ = (call);                                                                            \
		if (e_ != cudaSuccess) return fail(h, e_ == cudaErrorMemoryAllocation ? FQSK_E_NOMEM : FQSK_E_CUDA, \
			"%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));                             \
	} while (0)
#define CKR(expr) do { int r_ = (expr); if (r_ != FQSK_OK) return r_; } while (0)
#define LAUNCHED(h) do { ++(h)->S.kernel_launches; if ((h)->trace_launch) trace_launch_sync(__LINE__); } while (0)
// FQSK_F_TRACE_LAUNCH: every launch is followed by a device synchronisation and a line on stderr -- the last line printed names the
// kernel that hangs or faults (debugging aid; serialises the side streams)
inline void trace_launch_sync(int line) {
	fprintf(stderr, "[fqsk launch] fqsk.cu:%d ...", line); fflush(stderr);
	cudaError_t e = cudaDeviceSynchronize();
	fprintf(stderr, " %s\n", e == cudaSuccess ? "ok" : cudaGetErrorString(e)); fflush(stderr);
}


// Every kernel of the engine starts with pdl_enter() (griddepcontrol.launch_dependents + griddepcontrol.wait) and is launched with
// programmatic stream serialization: the next kernel of the stream is scheduled while the last wave of this one is still running
// and waits, before touching memory, until this one has completed and flushed.  Semantics are those of plain stream order; what is
// saved is the launch latency between the ~25 small dependent kernels of a sync segment.
// fqsk_timeline (measurement aid): while a timeline is open every launch is bracketed by two timing events on ITS stream, so that the
// fork / join structure of a segment can be read off a run that keeps its side streams (an event between two kernels costs the
// programmatic overlap of that pair: read the structure, not the last microsecond)
struct TimelineEntry { const void *fn; cudaStream_t st; cudaEvent_t a, b; };
static std::vector<TimelineEntry> *g_timeline = nullptr;

template <typename... KArgs, typename... Args>
inline cudaError_t pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args &&...args) {
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
	cudaLaunchAttribute at[1];
	at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
	at[0].val.programmaticStreamSerializationAllowed = 1;
	cfg.attrs = at; cfg.numAttrs = 1;
	if (g_timeline) {
		TimelineEntry e{(const void *) kern, st, nullptr, nullptr};
		cudaEventCreate(&e.a); cudaEventCreate(&e.b);
		cudaEventRecord(e.a, st);
		cudaError_t rc = cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
		cudaEventRecord(e.b, st);
		g_timeline->push_back(e);
		return rc;
	}
	return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

inline uint32_t nblk(uint64_t n, uint32_t t) { return (uint32_t) ((n + t - 1) / t); }

struct Phase {   // optional CUDA-event bracket on the engine's stream
	fqsk_handle *h; int ph; cudaEvent_t a = nullptr;
	Phase(fqsk_handle *h_, int ph_) : h(h_), ph(ph_) {
		if (!h->prof) return;
		a = take(); cudaEventRecord(a, h->st);
	}
	~Phase() {
		if (!h->prof) return;
		cudaEvent_t b = take(); cudaEventRecord(b, h->st);
		h->evs.push_back({a, b, ph});
	}
	cudaEvent_t take() {
		if (!h->ev_pool.empty()) { cudaEvent_t e = h->ev_pool.back(); h->ev_pool.pop_back(); return e; }
		cudaEvent_t e; cudaEventCreate(&e); return e;
	}
};
void resolve_phases(fqsk_handle *h) {   // call after a stream synchronize
	for (auto &e : h->evs) {
		float ms = 0;
		if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) h->ph_ms[e.ph] += ms;
		h->ev_pool.push_back(e.a); h->ev_pool.push_back(e.b);
	}
	h->evs.clear();
}

uint64_t mod_inverse(uint64_t x) { uint64_t inv = x; for (int i = 0; i < 6; ++i) inv *= 2 - x * inv; return inv; }

// Allocations other ranks map through CUDA IPC get a size that is a multiple of 2 MiB: smaller cudaMalloc blocks are sub-allocated from a
// shared 2 MiB page, and an IPC handle then exports (and a close unmaps) the whole page with whatever else lives in it.
inline size_t ipc_size(const fqsk_handle *h, size_t bytes) { return h->world > 1 ? (bytes + ((size_t) 2 << 20) - 1) & ~(((size_t) 2 << 20) - 1) : bytes; }

int table_alloc(fqsk_handle *h, Table &t, uint32_t k, uint32_t cbits, uint32_t B, unsigned long long *counters) {
	HtDev &d = t.d;
	d.k = k; d.cbits = cbits; d.W = 2 * k - 8; d.top = (1u << cbits) - 1;
	uint32_t bmin = d.W + cbits > 23 ? d.W + cbits - 23 : 1;   // rem + 8 end bits + counter + the occupied bit fit 32 bits
	if (B < bmin) B = bmin;
	if (B >= d.W) B = d.W - 1;
	if (B > 30) return fail(h, FQSK_E_INVAL, "table with k=%u needs 2^%u buckets (more than 2^30 is not supported)", k, B);
	d.B = B; d.rem_bits = d.W - B;
	if (d.rem_bits + 8 + cbits > 31) return fail(h, FQSK_E_INVAL, "k=%u, %u counter bits do not fit a 32-bit item with 2^%u buckets", k, cbits, B);
	d.maskW = d.W >= 64 ? ~0ull : ((1ull << d.W) - 1);
	d.mix_sh = (d.W + 1) / 2;
	d.stash_log2 = B + 3 >= 5 + 12 ? B + 3 - 5 : 12;
	d.n_items = counters;
	d.err = &h->status->stash_full;
	t.inv.inv1 = mod_inverse(MIX_C1); t.inv.inv2 = mod_inverse(MIX_C2);
	size_t mb = (size_t) 32 << B, sb = (size_t) 8 << d.stash_log2;
	CK(cudaMalloc(&d.main, ipc_size(h, mb)));
	CK(cudaMalloc(&d.stash, ipc_size(h, sb)));
	{
		const size_t ob = std::max<size_t>(((size_t) 1 << B) / 8, 4);
		CK(cudaMalloc(&d.occ, ob));
		CK(cudaMemsetAsync(d.occ, 0, ob, h->st));
		d.occ_read = nullptr;
	}
	CK(cudaMemsetAsync(d.main, 0, mb, h->st));
	CK(cudaMemsetAsync(d.stash, 0, sb, h->st));
	CK(cudaMemsetAsync(counters, 0, 16, h->st));
	d.world = h->world; d.rank = h->rank;
	for (uint32_t i = 0; i < FQSK_MAX_WORLD; ++i) { d.peer_main[i] = nullptr; d.peer_stash[i] = nullptr; }
	d.peer_main[h->rank] = d.main; d.peer_stash[h->rank] = d.stash;
	return FQSK_OK;
}

// jump polynomials x^(j chunk) mod phi, j = 1 .. MT_PAR - 1: computed once per process on the host (~0.3 s), one copy per device
int mt_jump_polys(fqsk_handle *h, const uint32_t **out) {
	static std::mutex mu;
	static std::vector<uint32_t> host;
	static bool tried = false, ok = false;
	static uint32_t *dev[64] = {nullptr};
	std::lock_guard<std::mutex> lk(mu);
	if (!tried) { tried = true; ok = fqsk_mtjump::jump_polys((uint64_t) MT_CHUNK_BLOCKS * 624, (int) MT_PAR - 1, host); }
	if (!ok) return fail(h, FQSK_E_CUDA, "internal error: the characteristic polynomial of mt19937 was not recovered");
	const int d = h->P.device;
	if (d < 0 || d >= 64) return fail(h, FQSK_E_INVAL, "device ordinal %d", d);
	if (!dev[d]) {
		CK(cudaMalloc(&dev[d], host.size() * 4));
		CK(cudaMemcpy(dev[d], host.data(), host.size() * 4, cudaMemcpyHostToDevice));
		CK(cudaFuncSetAttribute(k_mt_jump, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (MT_JUMP_WORDS * 4)));
	}
	*out = dev[d];
	return FQSK_OK;
}

inline uint64_t stream_avail_of(const Stream &s) { return s.generated - s.consumed; }   // generated (maybe still in flight) ahead of the consumer
int stream_init(fqsk_handle *h, Stream &s, uint64_t cap) {
	uint32_t st[624];
	st[0] = 5481u;
	for (int i = 1; i < 624; ++i) st[i] = 1812433253u * (st[i - 1] ^ (st[i - 1] >> 30)) + (uint32_t) i;
	CK(cudaMalloc(&s.state, 624 * 4));
	CK(cudaMemcpy(s.state, st, 624 * 4, cudaMemcpyHostToDevice));
	CK(cudaMalloc(&s.buf, cap * 4));
	CK(cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming));
	s.cap = cap; s.generated = s.consumed = 0; s.safe = 0; s.ev_pending = false;
	return FQSK_OK;
}
// enqueue generation up to absolute position `upto` (rounded up to 624-blocks) on the side stream
int stream_generate(fqsk_handle *h, Stream &s, uint64_t upto) {
	if (upto <= s.generated) return FQSK_OK;
	uint64_t blocks = (upto - s.generated + 623) / 624;
	if (s.generated + blocks * 624 - s.consumed > s.cap) {
		// the ring must never overwrite unconsumed outputs: enlarge it (rare: a single call needing more than the ring holds)
		uint64_t live = s.generated - s.consumed;
		uint64_t ncap = s.cap;
		while (s.generated + blocks * 624 - s.consumed > ncap) ncap <<= 1;
		CK(cudaStreamSynchronize(h->st_mt)); CK(cudaStreamSynchronize(h->st));
		uint32_t *nb = nullptr;
		CK(cudaMalloc(&nb, ncap * 4));
		for (uint64_t done = 0; done < live;) {   // copy the live window, re-based to the new mask
			uint64_t from = (s.consumed + done) & (s.cap - 1), to = (s.consumed + done) & (ncap - 1);
			uint64_t len = std::min(std::min(live - done, s.cap - from), ncap - to);
			CK(cudaMemcpy(nb + to, s.buf + from, len * 4, cudaMemcpyDeviceToDevice));
			done += len;
		}
		cudaFree(s.buf);
		s.buf = nb; s.cap = ncap;
	}
	Phase ph(h, FQSK_PH_MT);
	// long extensions run as MT_PAR chunks side by side (jump-ahead, fqsk_mtjump.h); the rest sequentially
	while (blocks >= (uint64_t) MT_PAR * MT_CHUNK_BLOCKS && (s.generated + (uint64_t) MT_PAR * MT_CHUNK_BLOCKS * 624 - s.consumed <= s.cap)) {
		const uint32_t *polys = nullptr;
		CKR(mt_jump_polys(h, &polys));
		if (!s.jstates) CK(cudaMalloc(&s.jstates, (size_t) MT_PAR * 624 * 4));
		k_mt_jump<<<MT_PAR, 640, MT_JUMP_WORDS * 4, h->st_mt>>>(s.state, polys, s.jstates);
		k_mt_extend<<<MT_PAR, 256, 0, h->st_mt>>>(s.state, s.jstates, s.buf, s.cap - 1, s.generated, MT_CHUNK_BLOCKS);
		LAUNCHED(h); LAUNCHED(h);
		s.generated += (uint64_t) MT_PAR * MT_CHUNK_BLOCKS * 624; blocks -= (uint64_t) MT_PAR * MT_CHUNK_BLOCKS;
	}
	while (blocks) {
		uint32_t nb = (uint32_t) std::min<uint64_t>(blocks, 1u << 20);
		k_mt_extend<<<1, 256, 0, h->st_mt>>>(s.state, (const uint32_t *) nullptr, s.buf, s.cap - 1, s.generated, nb);
		LAUNCHED(h);
		s.generated += (uint64_t) nb * 624; blocks -= nb;
	}
	CK(cudaGetLastError());
	CK(cudaEventRecord(s.ev, h->st_mt));
	s.ev_pending = true;
	return FQSK_OK;
}
// make outputs [consumed, consumed + need) available to kernels launched on the main stream after this call
int stream_ensure(fqsk_handle *h, Stream &s, uint64_t need) {
	if (s.consumed + need > s.generated) CKR(stream_generate(h, s, s.consumed + need + (need < (1u << 20) ? (1u << 20) : need / 2)));
	// wait for the generator only when the requested range reaches into outputs the main stream has not waited for yet
	if (s.consumed + need > s.safe && s.ev_pending) { CK(cudaStreamWaitEvent(h->st, s.ev, 0)); s.ev_pending = false; s.safe = s.generated; }
	else if (!s.ev_pending) s.safe = s.generated;
	return FQSK_OK;
}
// keep the generator ahead of the consumer without blocking anybody
int stream_prefetch(fqsk_handle *h, Stream &s, uint64_t ahead) {
	if (stream_avail_of(s) * 2 < ahead) return stream_generate(h, s, s.consumed + ahead);
	return FQSK_OK;
}
// The b-mer stream of a long job: late in a file the ordered inserts of one reads_block consume 5-7 M draws and ask for a window as long
// as their row before they know how many they need.  Whole parallel launches (MT_PAR chunks side by side, 8.4 M outputs, ~0.25 ms) keep
// at least `low_water` outputs ahead of the consumer, so that neither the one-CTA path (2 G outputs/s) nor a wait is ever on the sync's
// critical path (measured before: every other steady-state block waited 0.8 ms for a window generated on demand).
int stream_keep_ahead(fqsk_handle *h, Stream &s, uint64_t low_water) {
	const uint64_t launch = (uint64_t) MT_PAR * MT_CHUNK_BLOCKS * 624;
	while (stream_avail_of(s) < low_water && s.generated + launch - s.consumed <= s.cap) CKR(stream_generate(h, s, s.generated + launch));
	return FQSK_OK;
}
inline const uint32_t *stream_ptr(const Stream &s) { return s.buf; }
inline uint64_t stream_avail(const Stream &s) { return (s.safe > s.consumed ? s.safe : s.consumed) - s.consumed; }

// published chunk totals of the multi-CTA scans (k_scan_reads / k_scan_u32x4 / k_scan_draws), tagged with a per-launch epoch
int scan_chain(fqsk_handle *h, ScanChain &C, int which = 0) {      // which = 1: a scan that may run next to another one (side stream)
	const size_t one = (size_t) SCAN_CHAIN_MAX * 8 * 8 + (size_t) SCAN_CHAIN_MAX * 4 + 64;
	if (!h->scan_vals.p) {
		CK(h->scan_vals.ensure(3 * one));
		CK(cudaMemsetAsync(h->scan_vals.p, 0, h->scan_vals.cap, h->st));
		CK(cudaStreamSynchronize(h->st));
	}
	C.vals = (unsigned long long *) (h->scan_vals.as<uint8_t>() + (size_t) which * one);      // which = 0: engine stream, 1: compaction side stream, 2: front stream
	C.flags = (uint32_t *) (C.vals + (size_t) SCAN_CHAIN_MAX * 8); C.epoch = ++h->scan_epoch2;
	return FQSK_OK;
}
int ensure_iota(fqsk_handle *h, uint32_t n) {
	if (n <= h->iota_n) return FQSK_OK;
	uint32_t want = n + n / 2 + 1024;
	CK(h->iota.ensure((size_t) want * 4));
	CK(pdl(k_iota, nblk(want, 256), 256, h->st, h->iota.as<uint32_t>(), want));
	LAUNCHED(h);
	h->iota_n = want;
	return FQSK_OK;
}

// rows of a sync are at most this long when the caller announced its largest segment: buffers sized once, not as segments grow
inline size_t row_reserve(const fqsk_handle *h, size_t n) {
	const size_t r = h->P.reserve_bytes ? 2 * (size_t) h->P.reserve_bytes + 2 * (size_t) h->P.reserve_reads + 64 : 0;
	return n > r ? n : r;
}

// flags (u8) -> exclusive scan (u32), out[n] = total: the engine's own chained scan (fqsk_sort.cuh)
int scan_flags_u8(fqsk_handle *h, const uint8_t *flag, uint32_t *out, uint32_t n) {
	const uint32_t g = std::max<uint32_t>(nblk(n, SCAN8_TILE), 1);
	const size_t need = (size_t) std::max<uint32_t>(g, nblk((uint32_t) row_reserve(h, n), SCAN8_TILE)) * 8 + 64;
	if (h->scan8_part.cap < need) { CK(h->scan8_part.ensure(need)); CK(cudaMemsetAsync(h->scan8_part.p, 0, h->scan8_part.cap, h->st)); }
	CK(pdl(k_scan_u8, g, 256, h->st, flag, n, out, h->scan8_part.as<unsigned long long>(), ++h->scan8_epoch)); LAUNCHED(h);
	return FQSK_OK;
}

// One stable LSD pass of the engine's radix partition (fqsk_sort.cuh): hist -> row scan -> scatter
template <int NBITS, class Op>
int rdx_pass(fqsk_handle *h, cudaStream_t st, const unsigned long long *kin, const uint32_t *vin, unsigned long long *kout, uint32_t *vout, uint32_t n, Op op) {
	const uint32_t tiles = nblk(n, RDX_TILE);
	uint32_t *hist = h->rdx_hist.as<uint32_t>(), *totals = hist + ((size_t) tiles << NBITS);
	CK(pdl(k_rdx_hist<NBITS, Op>, tiles, RDX_THREADS, st, kin, n, tiles, hist, op)); LAUNCHED(h);
	CK(pdl(k_rdx_rowscan, 1u << NBITS, 256, st, hist, tiles, totals)); LAUNCHED(h);
	CK(pdl(k_rdx_scatter<NBITS, Op>, tiles, RDX_THREADS, st, kin, vin, kout, vout, n, tiles, (const uint32_t *) hist, (const uint32_t *) totals, op)); LAUNCHED(h);
	return FQSK_OK;
}
int rdx_scratch(fqsk_handle *h, uint32_t n, bool need_tmp) {
	const size_t nr = row_reserve(h, n);
	CK(h->rdx_hist.ensure((((size_t) nblk((uint32_t) nr, RDX_TILE) + 1) << 9) * 4 + 4096));
	if (need_tmp) { CK(h->rdx_k.ensure(nr * 8)); CK(h->rdx_v.ensure(nr * 4)); }
	return FQSK_OK;
}
// stable sort of (key, value) pairs by the key bits [b0, b1); vin == nullptr: the values are the element indices.  kin is not modified.
int sort_pairs_u64_u32(fqsk_handle *h, const unsigned long long *kin, unsigned long long *kout, const uint32_t *vin, uint32_t *vout, uint32_t n, int b0, int b1, cudaStream_t st = nullptr) {
	if (!st) st = h->st;
	if (!n) return FQSK_OK;
	const int passes = std::max(1, (b1 - b0 + 7) / 8);
	CKR(rdx_scratch(h, n, passes > 1));
	const unsigned long long *ks = kin; const uint32_t *vs = vin;
	for (int p = 0; p < passes; ++p) {
		const bool to_out = ((passes - 1 - p) & 1) == 0;
		unsigned long long *kd = to_out ? kout : h->rdx_k.as<unsigned long long>();
		uint32_t *vd = to_out ? vout : h->rdx_v.as<uint32_t>();
		const int lo = b0 + 8 * p, bits = std::min(8, b1 - lo);
		CKR((rdx_pass<8, BitsOp>(h, st, ks, vs, kd, vd, n, BitsOp{(uint32_t) lo, (1u << bits) - 1u})));
		ks = kd; vs = vd;
	}
	return FQSK_OK;
}
// the same by the table bucket of the k-mers (B bits, 9 per pass)
int sort_by_bucket(fqsk_handle *h, const Table &t, const unsigned long long *kin, unsigned long long *kout, uint32_t *vout, uint32_t n) {
	const int passes = ((int) t.d.B + 8) / 9;
	CKR(rdx_scratch(h, n, passes > 1));
	const unsigned long long *ks = kin; const uint32_t *vs = nullptr;
	for (int p = 0; p < passes; ++p) {
		const bool to_out = ((passes - 1 - p) & 1) == 0;
		unsigned long long *kd = to_out ? kout : h->rdx_k.as<unsigned long long>();
		uint32_t *vd = to_out ? vout : h->rdx_v.as<uint32_t>();
		const int lo = 9 * p, bits = std::min(9, (int) t.d.B - lo);
		CKR((rdx_pass<9, BucketOp>(h, h->st, ks, vs, kd, vd, n, BucketOp{t.d, (uint32_t) lo, (1u << bits) - 1u})));
		ks = kd; vs = vd;
	}
	return FQSK_OK;
}

const char *const STASH_FULL = "a k-mer table ran full inside one sync (more new k-mers than it can take before it grows): create the engine with a larger expected_kmers / *_log2_buckets";
int read_flags(fqsk_handle *h, int *out, int n) {
	EngineStatus &seen = h->look->st;
	CK(cudaMemcpyAsync(seen.flags, h->status->flags, n * sizeof(int), cudaMemcpyDeviceToHost, h->st));
	CK(cudaMemcpyAsync(&seen.stash_full, &h->status->stash_full, sizeof(int), cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	memcpy(out, seen.flags, n * sizeof(int));
	resolve_phases(h);
	if (seen.stash_full) return fail(h, FQSK_E_CAPACITY, "%s", STASH_FULL);
	return FQSK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// dump / growth
// ---------------------------------------------------------------------------------------------------------------
int table_dump_device(fqsk_handle *h, Table &t, uint64_t *n_out) {   // into h->dump_k / dump_v (unsorted)
	uint64_t total = (8ull << t.d.B) + (1ull << t.d.stash_log2);
	unsigned long long items[2];
	CK(cudaMemcpyAsync(items, t.d.n_items, 16, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	uint64_t n = items[0] + items[1];
	CK(h->dump_k.ensure((n + 1) * 8));
	CK(h->dump_v.ensure((n + 1) * 8));
	CK(cudaMemsetAsync(&h->status->dump_n, 0, 8, h->st));
	CK(pdl(k_dump_ht, nblk(total, 256), 256, h->st, t.d, t.inv, h->dump_k.as<unsigned long long>(), h->dump_v.as<unsigned long long>(), n, &h->status->dump_n));
	LAUNCHED(h);
	unsigned long long got = 0;
	CK(cudaMemcpyAsync(&got, &h->status->dump_n, 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (got != n) return fail(h, FQSK_E_CUDA, "table dump found %llu items, counters say %llu", got, (unsigned long long) n);
	*n_out = n;
	return FQSK_OK;
}

int table_double(fqsk_handle *h, Table &t) {      // one doubling: dump, allocate 2^(B + 1) buckets, re-insert
	uint64_t n = 0;
	unsigned long long items[2];
	CKR(table_dump_device(h, t, &n));
	unsigned long long *counters = t.d.n_items;
	CK(cudaFree(t.d.main)); CK(cudaFree(t.d.stash)); CK(cudaFree(t.d.occ));
	t.d.main = nullptr; t.d.stash = nullptr; t.d.occ = nullptr;
	uint32_t k = t.d.k, cb = t.d.cbits, B = t.d.B + 1;
	CKR(table_alloc(h, t, k, cb, B, counters));
	if (n) { CK(pdl(k_reinsert, nblk(n, 256), 256, h->st, t.d, h->dump_k.as<unsigned long long>(), h->dump_v.as<unsigned long long>(), n)); LAUNCHED(h); }
	CK(cudaMemcpyAsync(items, t.d.n_items, 16, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (items[0] + items[1] != n) return fail(h, FQSK_E_CUDA, "table growth lost items (%llu -> %llu)", (unsigned long long) n, items[0] + items[1]);
	++h->S.n_table_growths;
	return FQSK_OK;
}
inline bool table_can_double(const Table &t) { return t.d.B + 1 < t.d.W && t.d.B + 1 <= 30 && t.d.W - (t.d.B + 1) >= 1; }
inline unsigned long long crowd_main(const fqsk_handle *h, const Table &t) { return (4ull << t.d.B) >> h->crowd_shift; }      // half of the 8 << B slots (FQSK_F_TEST_CROWD: 1/64 of that)
inline unsigned long long crowd_stash(const Table &t) { return (1ull << t.d.stash_log2) / 2; }
inline bool table_crowded(const fqsk_handle *h, const Table &t, unsigned long long main_items, unsigned long long stash_items) { return main_items > crowd_main(h, t) || stash_items > crowd_stash(t); }

int table_grow_if_needed(fqsk_handle *h, Table &t) {      // unsharded engines; shards double together (fqsk_sync_finish -> FQSK_RESHARD)
	unsigned long long items[2];
	CK(cudaMemcpyAsync(items, t.d.n_items, 16, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (h->world > 1 && table_crowded(h, t, items[0], items[1]))      // (reached through the table-level mirrors only: fqsk_ht_insert)
		return fail(h, FQSK_E_CAPACITY, "a table shard is more than half full: shards double together, at a sync (FQSK_RESHARD), not inside a table-level call");
	while (table_crowded(h, t, items[0], items[1]) && table_can_double(t)) {
		CKR(table_double(h, t));
		CK(cudaMemcpyAsync(items, t.d.n_items, 16, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
	}
	return FQSK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// ordered insert of a row of k-mers into one table (CHT_kmer::insert in push order with one PRNG stream).
// Input: the row sorted by k-mer (stable) + the push index of every sorted occurrence.
// ---------------------------------------------------------------------------------------------------------------
int apply_sorted(fqsk_handle *h, Table &t, Stream &rng, const unsigned long long *skeys, const uint32_t *sidx, uint32_t n) {
	if (!n) return FQSK_OK;
	h->look_fresh = false;
	{
		const size_t nr = row_reserve(h, n);
		CK(h->slot_of.ensure(nr * 8));
		CK(h->flag8.ensure(nr + 4)); CK(h->draw_off.ensure((nr + 1) * 4)); CK(h->final_cnt.ensure(nr * 4));
	}
	const uint32_t g = nblk(n, 256);
	uint8_t *flag = h->flag8.as<uint8_t>();
	uint32_t *doff = h->draw_off.as<uint32_t>(), *c0_of = h->final_cnt.as<uint32_t>();
	unsigned long long *slot_of = h->slot_of.as<unsigned long long>();
	{
		Phase ph(h, FQSK_PH_SYNC_LOCATE);
		CK(cudaMemsetAsync(h->status->flags, 0, 8 * sizeof(int), h->st));
		CK(cudaMemsetAsync(flag + n, 0, 4, h->st));
		CK(pdl(k_locate_heads, g, 256, h->st, t.d, t.ci, skeys, sidx, n, slot_of, c0_of, flag, h->status->flags)); LAUNCHED(h);
	}
	Phase ph(h, FQSK_PH_SYNC_APPLY);
	uint32_t total_draws = 0;
	bool safe_done = false;
	for (int it = 0;; ++it) {
		if (it > 64) return fail(h, FQSK_E_NO_CONVERGE, "sync insert: draw flags did not settle");
		CKR(scan_flags_u8(h, flag, doff, n));
		CKR(stream_ensure(h, rng, 0));
		CK(cudaMemsetAsync(h->status->flags, 0, 3 * sizeof(int), h->st));      // [0] draw window short, [2] corrected a flag; [3] unsafe seen / [6] hot seen stay
		if (!safe_done) { CK(pdl(k_apply_keys, g, 256, h->st, t.d, t.ci, skeys, sidx, n, slot_of, c0_of, flag, doff, rng.buf, rng.cap - 1, rng.consumed, stream_avail(rng), 0, 0, h->status->flags)); LAUNCHED(h); }
		LookBuf *L = h->look;
		CK(cudaMemcpyAsync(L->st.flags, h->status->flags, sizeof L->st.flags, cudaMemcpyDeviceToHost, h->st));
		CK(cudaMemcpyAsync(&L->insert_draws, doff + n, 4, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		resolve_phases(h);
		int fl[8]; memcpy(fl, L->st.flags, sizeof fl);
		total_draws = L->insert_draws;
		if (fl[6]) h->hot_seen[&t == &h->tb ? 1 : 0] = true;
		if (fl[0]) { CKR(stream_ensure(h, rng, (uint64_t) total_draws + (1u << 16))); continue; }   // safe groups rewrite the same values
		if (!fl[3]) break;                    // no group can saturate: done with one pass
		// unsafe groups: verify their flags until a pass makes no correction, then commit them; safe groups are committed again
		// by the final pass only if the indices moved (a correction shifts every later draw index)
		bool moved = false;
		for (int vit = 0;; ++vit) {
			if (vit > 64) return fail(h, FQSK_E_NO_CONVERGE, "sync insert: draw flags did not settle");
			CK(cudaMemsetAsync(h->status->flags, 0, 3 * sizeof(int), h->st));
			CK(pdl(k_apply_keys, g, 256, h->st, t.d, t.ci, skeys, sidx, n, slot_of, c0_of, flag, doff, rng.buf, rng.cap - 1, rng.consumed, stream_avail(rng), 1, 0, h->status->flags)); LAUNCHED(h);
			CKR(read_flags(h, fl, 8));
			if (fl[0]) { CKR(stream_ensure(h, rng, 2 * stream_avail(rng) + (1u << 16))); continue; }
			if (!fl[2]) break;
			moved = true;
			CKR(scan_flags_u8(h, flag, doff, n));
		}
		CK(cudaMemcpyAsync(&L->insert_draws, doff + n, 4, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		total_draws = L->insert_draws;
		CKR(stream_ensure(h, rng, (uint64_t) total_draws));
		if (moved) { CK(pdl(k_apply_keys, g, 256, h->st, t.d, t.ci, skeys, sidx, n, slot_of, c0_of, flag, doff, rng.buf, rng.cap - 1, rng.consumed, stream_avail(rng), 0, 0, h->status->flags)); LAUNCHED(h); }
		CK(pdl(k_apply_keys, g, 256, h->st, t.d, t.ci, skeys, sidx, n, slot_of, c0_of, flag, doff, rng.buf, rng.cap - 1, rng.consumed, stream_avail(rng), 1, 1, h->status->flags)); LAUNCHED(h);
		CKR(read_flags(h, fl, 8));
		if (fl[0] || fl[2]) return fail(h, FQSK_E_CUDA, "internal error: unsafe-group commit pass was not clean");
		break;
	}
	rng.consumed += total_draws;
	return FQSK_OK;
}

// sort a row by k-mer (stable): out keys + push indices
int sort_row(fqsk_handle *h, const unsigned long long *row, uint32_t n, uint32_t k, DevBuf &keys_out, DevBuf &idx_out) {
	if (!n) return FQSK_OK;
	Phase ph(h, FQSK_PH_SORT);
	CK(keys_out.ensure(row_reserve(h, n) * 8)); CK(idx_out.ensure(row_reserve(h, n) * 4));
	CKR(sort_pairs_u64_u32(h, row, keys_out.as<unsigned long long>(), nullptr, idx_out.as<uint32_t>(), n, 64 - 2 * (int) k, 64));
	return FQSK_OK;
}

const uint32_t SYNC_INDEXED_MAX = 400000;
const uint64_t SPEC_MAX_BYTES = 420000;   // segments up to this many DNA bytes get their sync enqueued without a host look in between
const uint32_t FORK_MAX_READS = 8192;  // segments below this size run independent kernels of their chain on side streams
const int RC_RETRY = 1;   // internal: a capacity was too small, grow and redo the segment

// Ordered insert of a large row, grouped by table bucket (k_bucket_flags / k_bucket_apply): one stable partition by the bucket bits,
// one read-only walk for the draw flags, their scan, one walk that applies the row sector by sector.  *done = false: a counter may
// saturate inside the row or a bucket's run holds too many distinct k-mers -- nothing was written, the caller takes the general path.
int apply_bucketed(fqsk_handle *h, Table &t, Stream &rng, const unsigned long long *row, uint32_t n, bool *done) {
	*done = false;
	const size_t nr = row_reserve(h, n);
	CK(h->sort_k.ensure(nr * 8)); CK(h->sort_v.ensure(nr * 4)); CK(h->flag8.ensure(nr + 16)); CK(h->draw_off.ensure((nr + 1) * 4));
	{ Phase ph(h, FQSK_PH_SORT); CKR(sort_by_bucket(h, t, row, h->sort_k.as<unsigned long long>(), h->sort_v.as<uint32_t>(), n)); }
	const unsigned long long *sk = h->sort_k.as<unsigned long long>(); const uint32_t *sv = h->sort_v.as<uint32_t>();
	uint8_t *flag = h->flag8.as<uint8_t>(); uint32_t *doff = h->draw_off.as<uint32_t>();
	const uint32_t g = nblk(n, 256);
	{
		Phase ph(h, FQSK_PH_SYNC_LOCATE);
		CK(cudaMemsetAsync(h->status->flags, 0, 8 * sizeof(int), h->st));
		CK(pdl(k_bucket_flags, g, 256, h->st, t.d, t.ci, sk, sv, n, flag, h->status->flags)); LAUNCHED(h);
		CKR(scan_flags_u8(h, flag, doff, n));
	}
	Phase ph(h, FQSK_PH_SYNC_APPLY);
	CKR(stream_ensure(h, rng, n));      // every occurrence draws at most once
	CK(pdl(k_bucket_apply, g, 256, h->st, t.d, t.ci, sk, sv, n, (const uint32_t *) doff, (const uint32_t *) rng.buf, (unsigned long long) (rng.cap - 1), (unsigned long long) rng.consumed,
	       (unsigned long long) stream_avail(rng), h->status->flags)); LAUNCHED(h);
	LookBuf *L = h->look;
	CK(cudaMemcpyAsync(L->st.flags, h->status->flags, sizeof L->st.flags, cudaMemcpyDeviceToHost, h->st));
	CK(cudaMemcpyAsync(&L->insert_draws, doff + n, 4, cudaMemcpyDeviceToHost, h->st));
	CK(cudaMemcpyAsync(&L->st.stash_full, &h->status->stash_full, sizeof(int), cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	resolve_phases(h);
	int fl[8]; memcpy(fl, L->st.flags, sizeof fl);
	if (L->st.stash_full) return fail(h, FQSK_E_CAPACITY, "%s", STASH_FULL);
	if (fl[3] || fl[7]) return FQSK_OK;
	if (fl[0]) return fail(h, FQSK_E_CUDA, "internal error: the draw window of a bucket-grouped insert was too short");
	if (fl[6]) h->hot_seen[&t == &h->tb ? 1 : 0] = true;
	rng.consumed += L->insert_draws;
	h->look_fresh = false;
	*done = true;
	return FQSK_OK;
}

int apply_inserts(fqsk_handle *h, Table &t, Stream &rng, const unsigned long long *d_kmers, uint32_t n, bool *fast_ok = nullptr) {
	if (!n) return FQSK_OK;
	if (n >= 0x80000000u) return fail(h, FQSK_E_INVAL, "more than 2^31 k-mers in one sync row");
	h->look_fresh = false;
	if (fast_ok && *fast_ok) {
		Phase ph(h, FQSK_PH_SYNC_APPLY);
		CK(cudaMemsetAsync(h->status->flags, 0, 8 * sizeof(int), h->st));
		CK(h->y_flag.ensure((size_t) n + 4));
		CK(pdl(k_insert_fast, nblk(n, 256), 256, h->st, t.d, t.ci, d_kmers, n, h->y_flag.as<uint8_t>(), &h->status->flags[2], (const SyncIn *) nullptr)); LAUNCHED(h);
		int fl[8];
		CKR(read_flags(h, fl, 8));
		if (!fl[2]) return FQSK_OK;
		// some counter left the deterministic range: undo (claimed slots stay as zero-count items == the reference's fresh slot) and
		// take the ordered path from now on for this table (once counters are above thr they stay there)
		CK(pdl(k_insert_undo, nblk(n, 256), 256, h->st, t.d, d_kmers, n, h->y_flag.as<uint8_t>())); LAUNCHED(h);
		// this row goes through the ordered path; the next row tries the fast path again
	}
	if (h->world == 1) {      // (a sharded table's buckets are this rank's own as well, but the exchange rows take the indexed path)
		bool done = false;
		CKR(apply_bucketed(h, t, rng, d_kmers, n, &done));
		if (done) return FQSK_OK;
	}
	CKR(sort_row(h, d_kmers, n, t.d.k, h->sort_k, h->sort_v));
	return apply_sorted(h, t, rng, h->sort_k.as<unsigned long long>(), h->sort_v.as<uint32_t>(), n);
}

// ordered insert of a row using a (k-mer, time) index whose probe runs group equal k-mers (the segment's delta table, or an
// index built from the row).  Row length and stream position are read from a SyncIn block on the device, so the same launch
// sequence serves a sync that is enqueued right behind its segment (no host look in between) and the plain call below.
int indexed_setup(fqsk_handle *h, const DeltaDev &D, uint32_t n_bound, SyncIn *in, bool is_b, SyncDev &Y) {
	const size_t slots = std::max<size_t>((size_t) D.mask + 1, (size_t) 1 << 21);    // generous floors: no reallocation while segments grow
	const size_t nb = std::max<size_t>(n_bound, 2 * SPEC_MAX_BYTES + 2) + 64;
	CK(h->y_tslot.ensure(slots * 8)); CK(h->y_c0.ensure(slots * 4)); CK(h->y_m.ensure(slots * 4)); CK(h->y_draw.ensure(slots * 4));
	CK(h->y_j.ensure(slots * 4)); CK(h->y_final.ensure(slots * 4)); CK(h->y_flag_at.ensure(slots));
	CK(h->y_own.ensure(nb * 4)); CK(h->y_lead.ensure(nb * 4)); CK(h->y_rank.ensure(nb * 4));
	CK(h->y_flag.ensure(nb + 64)); CK(h->y_doff.ensure((nb + 1) * 4));
	if (!h->scan_part.p) { CK(h->scan_part.ensure(4096 * 8)); CK(cudaMemsetAsync(h->scan_part.p, 0, h->scan_part.cap, h->st)); }
	if (nblk(nb, SCANF_TILE) > 1024) return fail(h, FQSK_E_INVAL, "row too long for the indexed ordered insert");
	Y = SyncDev{};
	Y.D = D;
	Y.in = in; Y.n_dev = is_b ? &in->n_b : &in->n_s; Y.dpos_dev = is_b ? &in->dpos_b : &in->dpos_s; Y.total_draws = &in->draws_b;
	Y.lead_tslot = h->y_tslot.as<unsigned long long>(); Y.lead_c0 = h->y_c0.as<uint32_t>(); Y.lead_m = h->y_m.as<uint32_t>();
	Y.draw_at = h->y_draw.as<uint32_t>(); Y.j_at = h->y_j.as<uint32_t>(); Y.final_at = h->y_final.as<uint32_t>(); Y.flag_at = h->y_flag_at.as<uint8_t>();
	Y.own = h->y_own.as<uint32_t>(); Y.lead = h->y_lead.as<uint32_t>(); Y.rank = h->y_rank.as<uint32_t>();
	Y.flag = h->y_flag.as<uint8_t>(); Y.draw_off = h->y_doff.as<uint32_t>(); Y.flags = h->status->sflags;
	return FQSK_OK;
}
inline unsigned long long stream_safe_abs(const Stream &s) { return s.safe > s.consumed ? s.safe : s.consumed; }
int indexed_head(fqsk_handle *h, Table &t, const SyncDev &Y, const unsigned long long *row, const uint32_t *rt, uint32_t g, bool reset = true, cudaStream_t st = nullptr) {
	if (!st) st = h->st;
	Phase ph(h, FQSK_PH_SYNC_LOCATE);
	if (reset) CK(cudaMemsetAsync(h->status->sflags, 0, 8 * sizeof(int), st));
	CK(pdl(k_sync_rank, g, 256, st, t.d, Y, row, rt)); LAUNCHED(h);
	CK(pdl(k_sync_flags, g, 256, st, t.d, t.ci, Y)); LAUNCHED(h);
	return FQSK_OK;
}
// scan of the draw flags (+ scatter of draw index / flag to the delta entries)
int indexed_scan(fqsk_handle *h, Table &t, const SyncDev &Y, uint32_t n_bound, cudaStream_t st = nullptr) {
	if (!st) st = h->st;
	CK(pdl(k_scan_flags, nblk(n_bound, SCANF_TILE), 256, st, Y.in, Y.n_dev, (const uint8_t *) Y.flag, h->y_doff.as<uint32_t>(), Y.total_draws, h->scan_part.as<unsigned long long>(), ++h->scan_epoch, Y, t.ci)); LAUNCHED(h);
	return FQSK_OK;
}
// the leaders evaluate and write their groups
int indexed_apply(fqsk_handle *h, Table &t, Stream &rng, const SyncDev &Y, const unsigned long long *row, uint32_t g, bool reset = true) {
	if (reset) CK(cudaMemsetAsync(h->status->sflags, 0, 4 * sizeof(int), h->st));      // [0] draw window short, [2] corrected a flag; [6] hot seen / [7] group too large stay
	CK(pdl(k_sync_apply, g, 256, h->st, t.d, t.ci, Y, row, (const uint32_t *) rng.buf, (unsigned long long) (rng.cap - 1), stream_safe_abs(rng))); LAUNCHED(h);
	return FQSK_OK;
}
int indexed_tail(fqsk_handle *h, Table &t, Stream &rng, const SyncDev &Y, const unsigned long long *row, uint32_t g, uint32_t n_bound, bool reset = true) {
	CKR(indexed_scan(h, t, Y, n_bound));
	return indexed_apply(h, t, rng, Y, row, g, reset);
}
// one look at the device: the whole status block
int look(fqsk_handle *h) {
	LookBuf *L = h->look;
	struct WaitTimer { fqsk_handle *h; std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
	                   ~WaitTimer() { ++h->S.n_looks; h->S.look_wait_ns += (uint64_t) std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count(); } } wait_timer{h};
	if (h->prof) {
		CK(cudaMemcpyAsync(&L->st, h->status, sizeof(EngineStatus), cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		resolve_phases(h);
		h->look_fresh = true;
		if (L->st.stash_full) return fail(h, FQSK_E_CAPACITY, "%s", STASH_FULL);
		return FQSK_OK;
	}
	// One small kernel stores the status block into the page-locked look buffer (device-accessible under UVA) and then a sequence
	// number; the host spins on that number.  A copy and a stream synchronisation through the driver cost 10-20 us of wake-up
	// latency per look -- once per sync segment, i.e. ~5 % of a small segment -- and jitter with the host load.
	volatile unsigned long long *seq = &L->seq;
	const unsigned long long want = ++h->look_seq;
	CK(pdl(k_publish, 1, 128, h->st, (const EngineStatus *) h->status, &L->st, &L->seq, want)); LAUNCHED(h);
	for (uint64_t spins = 0; *seq != want; ++spins) {
		if ((spins & 0xFFFF) == 0xFFFF) {      // a failed launch or a faulting kernel would never publish
			cudaError_t e = cudaStreamQuery(h->st);
			if (e != cudaSuccess && e != cudaErrorNotReady) return fail(h, FQSK_E_CUDA, "look: %s", cudaGetErrorString(e));
			if (e == cudaSuccess && *seq != want) return fail(h, FQSK_E_CUDA, "look: the status block was not published");
		}
	}
	std::atomic_thread_fence(std::memory_order_acquire);
	h->look_fresh = true;
	if (L->st.stash_full) return fail(h, FQSK_E_CAPACITY, "%s", STASH_FULL);
	return FQSK_OK;
}

int apply_indexed(fqsk_handle *h, Table &t, Stream &rng, const DeltaDev &D, const unsigned long long *row, const uint32_t *rt, uint32_t n) {
	if (!n) return FQSK_OK;
	const bool is_b = &t == &h->tb;
	SyncIn *in = &h->status->syncin2;
	CK(pdl(k_set_syncin, 1, 32, h->st, in, is_b ? n : 0, is_b ? 0 : n, 0, is_b ? rng.consumed : 0, is_b ? 0 : rng.consumed)); LAUNCHED(h);
	SyncDev Y;
	CKR(indexed_setup(h, D, n, in, is_b, Y));
	const uint32_t g = nblk(n, 256);
	CKR(indexed_head(h, t, Y, row, rt, g));
	Phase ph(h, FQSK_PH_SYNC_APPLY);
	uint32_t total_draws = 0;
	for (int it = 0;; ++it) {
		if (it > 64) return fail(h, FQSK_E_NO_CONVERGE, "sync insert: draw flags did not settle");
		CKR(stream_ensure(h, rng, 0));     // wait for the generator if it is still running
		CKR(indexed_tail(h, t, rng, Y, row, g, n));
		CKR(look(h));
		const int *fl = h->look->st.sflags;
		total_draws = h->look->st.syncin2.draws_b;
		if (fl[6]) h->hot_seen[is_b ? 1 : 0] = true;
		if (fl[7]) {   // a hot k-mer occurs more than SYNC_GROUP_CAP times in this row: sorted path for the whole row
			CK(pdl(k_sync_unclaim, g, 256, h->st, t.d, Y, 0u)); LAUNCHED(h);
			return apply_inserts(h, t, rng, row, n, nullptr);
		}
		if (fl[0]) { CKR(stream_ensure(h, rng, (uint64_t) total_draws + (1u << 16))); continue; }
		if (!fl[2]) break;
	}
	rng.consumed += total_draws;
	return FQSK_OK;
}

// build an index for a plain row (no segment behind it) and insert it
int apply_row(fqsk_handle *h, Table &t, Stream &rng, const unsigned long long *row, uint32_t n) {
	if (!n) return FQSK_OK;
	if (n > (1u << 21)) return apply_inserts(h, t, rng, row, n);     // long rows: one radix sort is cheaper (and k_scan_flags stays co-resident)
	uint32_t slots = 1024;
	while (slots < 2 * n) slots <<= 1;
	CK(h->idx_k.ensure((size_t) slots * 8)); CK(h->idx_t.ensure((size_t) slots * 4)); CK(h->idx_rt.ensure((size_t) n * 4));
	CK(cudaMemsetAsync(h->idx_t.p, 0xFF, (size_t) slots * 4, h->st));
	CK(pdl(k_row_index_build, nblk(n, 256), 256, h->st, h->idx_k.as<unsigned long long>(), h->idx_t.as<uint32_t>(), slots - 1, t.d.k, 1, row, n, h->idx_rt.as<uint32_t>())); LAUNCHED(h);
	DeltaDev D{h->idx_k.as<unsigned long long>(), h->idx_t.as<uint32_t>(), slots - 1, n, t.d.k, 1, t.ci.thr + 1};
	return apply_indexed(h, t, rng, D, row, h->idx_rt.as<uint32_t>(), n);
}

EngineDev make_engine_dev(fqsk_handle *h) {
	EngineDev E{};
	E.hb = h->tb.d; E.hs = h->ts.d; E.siv = h->siv; E.cib = h->tb.ci; E.cis = h->ts.ci;
	E.p = h->P.pmer_len; E.s = h->P.smer_len; E.b = h->P.bmer_len; E.prefix_len = h->P.prefix_len;
	E.sorted = mode_sorted(h->P.mode);
	double aff = h->S.siv_no_filled ? (double) h->S.siv_no_updates / (double) h->S.siv_no_filled : 0.0;   // bit_vec.h:204-210
	E.gate_missing = aff >= 7.0;
	for (int i = 0; i < 4; ++i) { E.draws[i] = h->rng[i].buf; E.dmask[i] = h->rng[i].cap - 1; E.dpos[i] = h->rng[i].consumed; E.avail[i] = stream_avail(h->rng[i]); }
	E.flags = h->status->flags;
	return E;
}

// ---------------------------------------------------------------------------------------------------------------
// one sync segment, reads resident on the device (DESIGN.md section 5).  All counts stay on the device; kernels are
// launched from host-side upper bounds.  seg_setup + seg_pass enqueue the first pass of the fixed launch schedule; the host
// does not look at the device until somebody needs the outcome (seg_settle): the sync that follows a small segment is
// enqueued behind it unseen, predicated on the device-side verdict of the pass (k_seg_tail).
// ---------------------------------------------------------------------------------------------------------------
// side streams of the fork / join points (created on first use): [0] compaction + early grouping, p-mer updates; [1] k_partial, s-mer
// inserts; [2] the rough searches that start behind walk 0
int ensure_side(fqsk_handle *h) {
	if (h->st_side[0]) return FQSK_OK;
	// the chain of small dependent kernels is what a segment waits for: its streams get the highest priority, the long bandwidth-bound
	// rough search that runs next to it the lowest (measured next to an unprioritised k_rough: k_delta_build_flat 67 us instead of 13)
	int lo = 0, hi = 0;
	CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
	for (int i = 0; i < 3; ++i) { CK(cudaStreamCreateWithPriority(&h->st_side[i], cudaStreamNonBlocking, i == 2 ? lo : hi)); CK(cudaEventCreateWithFlags(&h->ev_side[i], cudaEventDisableTiming)); }
	CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&h->ev_aux, cudaEventDisableTiming));
	return FQSK_OK;
}

struct PrepBufs { DevBuf *dup, *n_coded, *letters, *rec_off, *sl_prefix, *pk; };
inline PrepBufs prep_bufs(fqsk_handle *h, int par) {
	return par ? PrepBufs{&h->f_dup, &h->f_n_coded, &h->f_letters, &h->f_rec_off, &h->f_sl_prefix, &h->f_pk} : PrepBufs{&h->dup, &h->n_coded, &h->letters, &h->rec_off, &h->sl_prefix, &h->pk};
}

int seg_setup(fqsk_handle *h, bool reset_done = false) {      // reset_done: k_prep has just cleared the status words (first evaluation of the segment)
	SegCtx &C = h->ctx;
	SegDev &S = C.S;
	const uint32_t n = C.n;
	const uint64_t dna_bytes = std::max<uint64_t>(C.dna_bytes_actual, h->P.reserve_bytes);   // scratch sized once for the largest segment
	const size_t n1 = (size_t) std::max<uint32_t>(n, h->P.reserve_reads) + 1;
	const uint32_t rec_bound = (uint32_t) C.dna_bytes_actual;          // coded positions <= DNA bytes
	const size_t r1 = (size_t) dna_bytes + 1;
	const uint32_t pslots = h->P.bmer_len - h->P.pmer_len + 1;
	CK(h->prov.ensure(r1 * sizeof(fqsk_base_rec))); CK((h->rec_par ? h->recs_alt : h->recs).ensure(r1 * sizeof(fqsk_base_rec))); CK(h->pflags.ensure(r1));
	CK(h->rkind.ensure(r1)); CK(h->rreg.ensure(r1 * sizeof(KReg))); CK(h->rslot.ensure(r1 * 4)); CK(h->dirty.ensure(n1));
	CK(h->pscripts.ensure(n1 * pslots * sizeof(Script)));
	CK(h->rscripts.ensure(((size_t) h->rreq_cap + 1) * sizeof(Script)));
	CK(h->pool.ensure(((size_t) h->pool_cap + 1) * 8)); CK(h->miss.ensure(((size_t) h->miss_cap + 1) * sizeof(MissEntry)));
	CK(h->miss_fold.ensure((size_t) h->miss_cap + 1));
	if (h->hot || h->miss_fold_dirty || h->miss_fold.p != h->miss_fold_seen) {   // only the ordered evaluator (hot mode) ever marks entries
		CK(cudaMemsetAsync(h->miss_fold.p, 0, h->miss_fold.cap, h->st));
		h->miss_fold_dirty = h->hot; h->miss_fold_seen = h->miss_fold.p;
	}
	CK(h->rdraws_b.ensure(n1 * 4)); CK(h->rdraws_s.ensure(n1 * 4)); CK(h->doff_b.ensure(n1 * 8)); CK(h->doff_s.ensure(n1 * 8));
	CK(h->time_b.ensure((2 * dna_bytes + 2) * 4)); CK(h->time_s.ensure((dna_bytes + 1) * 4));
	CK(h->rt_b[0].ensure((2 * dna_bytes + 2) * 4)); CK(h->rt_s[0].ensure((dna_bytes + 1) * 4));

	PipeDev &P = C.P;
	P = PipeDev{};
	P.n_rec = rec_bound; P.start = C.first; P.rec_off = S.rec_off;
	P.prov = h->prov.as<fqsk_base_rec>(); P.recs = (h->rec_par ? h->recs_alt : h->recs).as<fqsk_base_rec>(); P.pflags = h->pflags.as<uint8_t>();
	P.pscripts = h->pscripts.as<Script>(); P.pslots = pslots; P.pfirst_n = h->P.pmer_len - 1;
	P.rscripts = h->rscripts.as<Script>(); P.n_rscript = &h->status->n_rscript; P.rscript_cap = h->rreq_cap;
	P.rkind = h->rkind.as<uint8_t>(); P.rreg = h->rreg.as<KReg>(); P.rslot = h->rslot.as<uint32_t>(); P.dirty = h->dirty.as<uint8_t>();
	P.pool = h->pool.as<unsigned short>(); P.pool_used = &h->status->pool_used; P.pool_cap = h->pool_cap;
	P.miss = h->miss.as<MissEntry>(); P.n_miss = &h->status->n_miss; P.miss_cap = h->miss_cap; P.miss_fold = h->miss_fold.as<uint8_t>();
	P.ev_n = h->status->hot.ev; P.hot_draws = h->status->hot.draws; P.ev_cap = 0;
	P.rdraws_b = h->rdraws_b.as<uint32_t>(); P.rdraws_s = h->rdraws_s.as<uint32_t>();
	P.doff_b = h->doff_b.as<unsigned long long>(); P.doff_s = h->doff_s.as<unsigned long long>();
	P.time_b = h->time_b.as<uint32_t>(); P.time_s = h->time_s.as<uint32_t>();
	P.flags = h->status->flags; P.n_rec_dev = &h->status->n_rec[h->seg_par];
	S.recs = P.recs;

	C.E = make_engine_dev(h);
	C.t_b = std::max<uint32_t>(h->P.bmer_len - h->P.smer_len - 1, 1); C.t_s = std::max<uint32_t>(h->P.smer_len - h->P.pmer_len + 1, 1);
	{
		// Large segments: the thread-local delta holds only the pushes a lookup can ask for (DeltaDev::filter).  Scattering all
		// 13 M pushes of a 51 000-read segment into a 600 MB table cost 1.06 ms and 2.1 GB of DRAM traffic, although only the
		// ~10 % of positions the global tables cannot answer ever look there.  Small segments keep the full delta: their sync
		// groups equal k-mers through it (apply_indexed / sync_spec_enqueue); so does the ordered thread-local evaluator (hot mode).
		const bool use_filter = !h->hot && h->world == 1 && C.dna_bytes_actual >= (1u << 20);
		const uint32_t FBITS = 1u << 26;
		uint32_t *fb = nullptr, *fs = nullptr;
		if (use_filter) {
			CK(h->dfilter.ensure((size_t) 2 * FBITS / 8));
			CK(cudaMemsetAsync(h->dfilter.p, 0, (size_t) 2 * FBITS / 8, h->st));
			fb = h->dfilter.as<uint32_t>(); fs = fb + FBITS / 32;
		}
		h->delta_filtered = use_filter;
		S.delta_b = DeltaDev{nullptr, nullptr, 0, 0, h->P.bmer_len, C.t_b, h->tb.ci.thr + 1, nullptr, nullptr, nullptr, fb, FBITS - 1};
		S.delta_s = DeltaDev{nullptr, nullptr, 0, 0, h->P.smer_len, C.t_s, h->ts.ci.thr + 1, nullptr, nullptr, nullptr, fs, FBITS - 1};
	}
	// one launch clears every status word the segment and a sync enqueued behind it start from: flags[8] | n_miss, n_rscript, pool_used
	// (n_rec_dev stays: k_scan_reads wrote it) | hot-mode counters | fresh p-mer fields | s fast-path verdict | ordered-insert flags
	if (!reset_done) { CK(pdl(k_seg_reset, 1, 32, h->st, h->status)); LAUNCHED(h); }
	// sorted order: (flag, dif) of compress_prefix_sorted per read, against the p-mer array as it is before this segment's sync
	if (mode_sorted(h->P.mode)) { CK(pdl(k_sorted_dif, n, 256, h->st, C.E, S)); LAUNCHED(h); }
	// full and front-truncated lookups touch disjoint positions: k_partial runs on a side stream next to k_lookup (not when profiling)
	// k_partial is bound by the latency of its dependent probes (38 % of the warps active on a 51 000-read segment), k_lookup by DRAM: next to
	// each other at every segment size
	const bool fork = !h->serial;
	if (fork) CKR(ensure_side(h));
	cudaStream_t st_pt = fork ? h->st_side[1] : h->st;
	if (fork) { CK(cudaEventRecord(h->ev_fork, h->st)); CK(cudaStreamWaitEvent(st_pt, h->ev_fork, 0)); }
	{ Phase ph(h, FQSK_PH_LOOKUP); CK(pdl(k_lookup, nblk(rec_bound, 256), 256, h->st, C.E, S, P)); LAUNCHED(h); }
	{ Phase ph(h, FQSK_PH_PARTIAL); CK(pdl(k_partial, nblk((uint64_t) n * pslots * 32, 128), 128, st_pt, C.E, S, P)); LAUNCHED(h); }
	if (fork) { CK(cudaEventRecord(h->ev_side[1], st_pt)); CK(cudaStreamWaitEvent(h->st, h->ev_side[1], 0)); }
	h->delta_b_valid = h->delta_s_valid = false;
	C.slots_b = 1024; C.slots_s = 1024;
	while (C.slots_b < 4 * C.dna_bytes_actual) C.slots_b <<= 1;      // at most 2 b pushes per base, half-full table
	while (C.slots_s < 2 * C.dna_bytes_actual) C.slots_s <<= 1;
	{
		size_t rb = 1024, rs = 1024;
		while (rb < 4 * dna_bytes) rb <<= 1;
		while (rs < 2 * dna_bytes) rs <<= 1;
		CK(h->dk_b.ensure(rb * 8)); CK(h->stime_b.ensure((rb + rs) * 4)); CK(h->dk_s.ensure(rs * 8));     // both time arrays in one allocation: one fill
	}
	{ Phase ph(h, FQSK_PH_WALK); CK(pdl(k_walk, nblk((uint64_t) n * 32, 128), 128, h->st, C.E, S, P, 0)); LAUNCHED(h); ++h->S.n_replays; }
	C.it = 0; C.pass = 0; C.redo_walk = true; C.redo_tail = true;
	return FQSK_OK;
}

int seg_build_delta(fqsk_handle *h, bool force_full = false) {
	SegCtx &C = h->ctx;
	SegDev &S = C.S; PipeDev &P = C.P;
	if (force_full) { S.delta_b.filter = nullptr; S.delta_s.filter = nullptr; }
	uint32_t *const fb = S.delta_b.filter, *const fs = S.delta_s.filter;
	const uint32_t fmask = S.delta_b.fmask;
	const uint32_t n = C.n, slots_b = C.slots_b, slots_s = C.slots_s;
	Phase ph(h, FQSK_PH_SORT);
	CK(h->dk_b.ensure((size_t) slots_b * 8)); CK(h->stime_b.ensure(((size_t) slots_b + slots_s) * 4));
	CK(h->dk_s.ensure((size_t) slots_s * 8));
	uint32_t *stime_s = h->stime_b.as<uint32_t>() + slots_b;
	CK(cudaMemsetAsync(h->stime_b.p, 0xFF, ((size_t) slots_b + slots_s) * 4, h->st));
	if (n < 8192 && C.dna_bytes_actual < (1u << 22))
		CK(pdl(k_delta_build_flat, nblk(3 * C.dna_bytes_actual, 256), 256, h->st, S, P, (uint32_t) C.dna_bytes_actual, h->dk_b.as<unsigned long long>(), h->stime_b.as<uint32_t>(), slots_b - 1,
		       h->P.bmer_len, C.t_b, h->dk_s.as<unsigned long long>(), stime_s, slots_s - 1, h->P.smer_len, C.t_s));
	else
	CK(pdl(k_delta_build, nblk((uint64_t) n * 32, 128), 128, h->st, S, P, h->dk_b.as<unsigned long long>(), h->stime_b.as<uint32_t>(), slots_b - 1, h->P.bmer_len, C.t_b,
	                                                             h->dk_s.as<unsigned long long>(), stime_s, slots_s - 1, h->P.smer_len, C.t_s));
	LAUNCHED(h);
	S.delta_b = DeltaDev{h->dk_b.as<unsigned long long>(), h->stime_b.as<uint32_t>(), slots_b - 1, 1, h->P.bmer_len, C.t_b, h->tb.ci.thr + 1, nullptr, nullptr, nullptr, fb, fmask};
	S.delta_s = DeltaDev{h->dk_s.as<unsigned long long>(), stime_s, slots_s - 1, 1, h->P.smer_len, C.t_s, h->ts.ci.thr + 1, nullptr, nullptr, nullptr, fs, fmask};
	if (!h->hot) return FQSK_OK;
	// hot mode: ranks, queued events (inserts above thr + thread-local merges), time order, sequential evaluation
	Phase ph2(h, FQSK_PH_LOCAL);
	for (int q = 0; q < 3; ++q) { CK(h->hr_b[q].ensure((size_t) slots_b * 4)); CK(h->hr_s[q].ensure((size_t) slots_s * 4)); }
	const uint32_t ev_cap = (uint32_t) std::min<uint64_t>(2 * C.dna_bytes_actual + 1024, 1u << 30);
	for (int q = 0; q < 2; ++q) { CK(h->evk[q].ensure((size_t) ev_cap * 8)); CK(h->evv[q].ensure((size_t) ev_cap * 4)); CK(h->evk_s[q].ensure((size_t) ev_cap * 8)); CK(h->evv_s[q].ensure((size_t) ev_cap * 4)); }
	S.delta_b.rank_at = h->hr_b[0].as<uint32_t>(); S.delta_b.prev_at = h->hr_b[1].as<uint32_t>(); S.delta_b.cnt_at = h->hr_b[2].as<uint32_t>();
	S.delta_s.rank_at = h->hr_s[0].as<uint32_t>(); S.delta_s.prev_at = h->hr_s[1].as<uint32_t>(); S.delta_s.cnt_at = h->hr_s[2].as<uint32_t>();
	for (int q = 0; q < 2; ++q) { P.ev_key[q] = h->evk[q].as<unsigned long long>(); P.ev_val[q] = h->evv[q].as<uint32_t>(); }
	P.ev_n = h->status->hot.ev; P.ev_cap = ev_cap; P.hot_draws = h->status->hot.draws;
	CK(cudaMemsetAsync(&h->status->hot, 0, sizeof h->status->hot, h->st));
	CK(pdl(k_delta_rank, 148 * 8, 256, h->st, S.delta_b, P, 0)); LAUNCHED(h);
	CK(pdl(k_delta_rank, 148 * 8, 256, h->st, S.delta_s, P, 1)); LAUNCHED(h);
	CK(pdl(k_local, std::min<uint32_t>(nblk(std::max<uint32_t>(h->miss_cap, 1), 128), 148 * 16), 128, h->st, C.E, S, P, 0)); LAUNCHED(h);
	EngineStatus &seen = h->look->st;
	CK(cudaMemcpyAsync(&seen, h->status, sizeof seen, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (seen.flags[4]) return fail(h, FQSK_E_NOMEM, "hot-mode event list overflow");     // cannot happen with the bound above
	uint32_t en[2] = {seen.hot.ev[0], seen.hot.ev[1]};
	for (int q = 0; q < 2; ++q) if (en[q]) {
		CKR(sort_pairs_u64_u32(h, h->evk[q].as<unsigned long long>(), h->evk_s[q].as<unsigned long long>(), h->evv[q].as<uint32_t>(), h->evv_s[q].as<uint32_t>(), en[q], 0, 34));      // by time
	}
	CKR(stream_ensure(h, h->rng[ST_LB], (uint64_t) en[0] * 8 + 1024)); CKR(stream_ensure(h, h->rng[ST_LS], (uint64_t) en[1] * 8 + 1024));
	C.E = make_engine_dev(h);
	CK(h->hot_tab.ensure((size_t) 2 * 3 * HOT_TAB_ENTRIES * 4)); CK(cudaMemsetAsync(h->hot_tab.p, 0, (size_t) 2 * 3 * HOT_TAB_ENTRIES * 4, h->st));
	CK(pdl(k_hot_eval, 1, 64, h->st, C.E, S, P, h->evk_s[0].as<unsigned long long>(), h->evv_s[0].as<uint32_t>(), en[0], h->evk_s[1].as<unsigned long long>(), h->evv_s[1].as<uint32_t>(), en[1], h->hot_tab.as<uint32_t>())); LAUNCHED(h);
	return FQSK_OK;
}

// Fixed launch schedule of one pass: the thread-local pass (delta, k_local, walk `it` on the reads it touched), compaction,
// rough searches, ordered merges.  If the look shows that the walk changed pushes (rare) the thread-local pass and everything
// after it is repeated; if only the merge offsets moved, only the merges.
int seg_pass(fqsk_handle *h, bool with_prefix = false) {
	SegCtx &C = h->ctx;
	SegDev &S = C.S; PipeDev &P = C.P; EngineDev &E = C.E;
	const uint32_t n = C.n, rec_bound = (uint32_t) C.dna_bytes_actual;
	const uint32_t max_it = h->P.max_iterations ? h->P.max_iterations : 16;
	uint32_t *d_tot4 = h->status->row_tot;
	unsigned long long *d_draw2 = h->status->draws;
	if (++C.pass > 64) return fail(h, FQSK_E_NO_CONVERGE, "segment did not settle");
	// sparse tables (the first blocks of a file): k_rough tests the bucket-occupancy bit before reading a neighbour's bucket
	EngineDev Er = E;
	if (h->world == 1 && h->items_main[0] < (1ull << h->tb.d.B)) Er.hb.occ_read = Er.hb.occ;
	if (h->world == 1 && h->items_main[1] < (1ull << h->ts.d.B)) Er.hs.occ_read = Er.hs.occ;
	const uint32_t rough_grid = std::max<uint32_t>(148, std::min<uint32_t>(nblk(rec_bound, 16), 148 * 32));
	const bool rough_deep = !Er.hb.occ_read;      // the b-mer table is past one item per bucket: (nearly) every trial reads its sector
	// First pass of a small segment: the rough searches -- the longest kernel of the chain -- start right behind walk 0 on a side stream,
	// next to the thread-local pass (delta, k_local, walk 1).  The few positions walk 1 writes again carry a marker and are searched
	// again below; k_rough writes scripts only (k_fold writes the records), so the two passes never race on a record.
	const bool spec_rough = !h->serial && !h->hot && n < FORK_MAX_READS && C.pass == 1 && C.redo_walk && C.redo_tail;
	// compaction of the pushes (+ the pre-verdict of the early grouping) on side stream 0
	auto enqueue_compaction = [&](cudaStream_t st_c) -> int {
		Phase ph(h, FQSK_PH_COMPACT);
		ScanChain sc; CKR(scan_chain(h, sc, 1));
		CK(pdl(k_scan_u32x4, n <= 2048 ? 1u : nblk(n, SCAN_U32_CHUNK), n <= 2048 ? 256 : 1024, st_c, n, h->cnt_b.as<uint32_t>(), h->off_b[0].as<uint32_t>(), h->cnt_s.as<uint32_t>(), h->off_s[0].as<uint32_t>(),
		                                     h->cnt_p.as<uint32_t>(), h->off_p.as<uint32_t>(), h->hidden.as<uint32_t>(), (uint32_t *) nullptr, d_tot4, (uint32_t *) nullptr, sc));
		LAUNCHED(h);
		CK(pdl(k_compact2, n, 64, st_c, S, P, h->off_b[0].as<uint32_t>(), h->off_s[0].as<uint32_t>(), h->off_p.as<uint32_t>(),
		                               h->row_b[0].as<unsigned long long>(), h->row_s[0].as<unsigned long long>(), h->row_p.as<unsigned long long>(),
		                               h->rt_b[0].as<uint32_t>(), h->rt_s[0].as<uint32_t>()));
		LAUNCHED(h);
		return FQSK_OK;
	};
	// grouping half of the b-mer sync (find-or-create per distinct k-mer, ranks, draw flags and their scan) behind the compaction, on the
	// same side stream: it runs while k_rough / k_fold work on the records.  Predicated on the walk-level verdict; if the pass then fails
	// to settle, the claimed slots are released again (sync_end: k_sync_unclaim).  Needs the segment's delta table (seg_build_delta).
	// Only behind the last walk of the pass: a slot claimed for a k-mer that a later walk no longer pushes could never be given back (the
	// tables have no deletion); behind walk 1 the verdict knows whether the pushes are final.
	auto enqueue_grouping = [&](cudaStream_t st_c) -> int {
		const uint32_t bound_b = (uint32_t) (2 * C.dna_bytes_actual + 2);
		CK(pdl(k_pre_verdict, 1, 32, st_c, (const int *) h->status->flags, (const uint32_t *) d_tot4, SYNC_INDEXED_MAX, &h->status->syncin)); LAUNCHED(h);
		CKR(indexed_setup(h, S.delta_b, bound_b, &h->status->syncin, true, h->spec_Y));
		h->spec_g = nblk(bound_b, 256);
		CKR(indexed_head(h, h->tb, h->spec_Y, h->row_b[0].as<unsigned long long>(), h->rt_b[0].as<uint32_t>(), h->spec_g, false, st_c));
		CKR(indexed_scan(h, h->tb, h->spec_Y, bound_b, st_c));
		return FQSK_OK;
	};
	if (spec_rough) {
		// Walk 1 only re-walks the reads whose thread-local answers differ and almost never changes a push; when it does, flags[2] fails
		// the pass and everything here is done again.  So all three consumers of walk 0 start behind it: the rough searches (side stream
		// 2), the compaction of the pushes (side stream 0) and the thread-local pass (this stream).
		CKR(ensure_side(h));
		CK(cudaEventRecord(h->ev_fork, h->st));
		CK(cudaStreamWaitEvent(h->st_side[2], h->ev_fork, 0)); CK(cudaStreamWaitEvent(h->st_side[0], h->ev_fork, 0));
		CK(pdl(rough_deep ? k_rough<true> : k_rough<false>, rough_grid, 128, h->st_side[2], Er, P, 0u)); LAUNCHED(h);
		CK(cudaEventRecord(h->ev_side[2], h->st_side[2]));
		CKR(enqueue_compaction(h->st_side[0]));
	}
	if (C.redo_walk) {
		if (++C.it >= max_it) return fail(h, FQSK_E_NO_CONVERGE, "segment did not reach its fixed point in %u iterations", max_it);
		if (C.pass > 1) CK(cudaMemsetAsync(&h->status->flags[2], 0, sizeof(int), h->st));     // first pass: still clear from k_seg_reset
		CKR(seg_build_delta(h));
		{ Phase ph(h, FQSK_PH_LOCAL); CK(pdl(k_local, std::min<uint32_t>(nblk(std::max<uint32_t>(h->miss_cap, 1), 128), 148 * 16), 128, h->st, E, S, P, 1)); LAUNCHED(h); }
		{ Phase ph(h, FQSK_PH_WALK); CK(pdl(k_walk, nblk((uint64_t) n * 32, 128), 128, h->st, E, S, P, C.it)); LAUNCHED(h); ++h->S.n_replays; }
		if (spec_rough && with_prefix) {      // the rows were compacted behind walk 0; the grouping waits for walk 1 (and its flags)
			CK(cudaEventRecord(h->ev_aux, h->st)); CK(cudaStreamWaitEvent(h->st_side[0], h->ev_aux, 0));
			CKR(enqueue_grouping(h->st_side[0]));
		}
	}
	if (C.redo_tail) {
		// The compaction of the pushes (rows of the sync) and the rough searches + merges (records) only meet again at the verdict:
		// the two small compaction kernels run on a side stream next to k_rough / k_fold.  Profiling keeps one stream.
		const bool fork = !h->serial && n < FORK_MAX_READS;
		if (fork) CKR(ensure_side(h));
		cudaStream_t st_c = fork ? h->st_side[0] : h->st;
		if (C.pass > 1) CK(cudaMemsetAsync(&h->status->n_rscript, 0, 4, h->st));      // rough scripts are rebuilt (first pass: still clear from k_seg_reset)
		if (!spec_rough) {
			if (fork) { CK(cudaEventRecord(h->ev_fork, h->st)); CK(cudaStreamWaitEvent(st_c, h->ev_fork, 0)); }
			CKR(enqueue_compaction(st_c));
			if (with_prefix) CKR(enqueue_grouping(st_c));
		}
		if (fork) CK(cudaEventRecord(h->ev_side[0], st_c));
		{ Phase ph(h, FQSK_PH_ROUGH);
			if (spec_rough) CK(cudaStreamWaitEvent(h->st, h->ev_side[2], 0));      // join; then only the positions walk 1 wrote
			CK(pdl(rough_deep ? k_rough<true> : k_rough<false>, rough_grid, 128, h->st, Er, P, spec_rough ? 1u : 0u)); LAUNCHED(h); }
		{ Phase ph(h, FQSK_PH_FOLD); CK(pdl(k_fold, nblk((uint64_t) n * 32, 128), 128, h->st, E, S, P, 0)); LAUNCHED(h); }
	}
	{
		Phase ph(h, FQSK_PH_FOLD);
		ScanChain sc; CKR(scan_chain(h, sc));
		CK(pdl(k_scan_draws, n <= 2048 ? 1u : nblk(n, SCAN_U32_CHUNK), n <= 2048 ? 256 : 1024, h->st, n, P.rdraws_b, h->doff_b.as<unsigned long long>(), P.rdraws_s, h->doff_s.as<unsigned long long>(), d_draw2, h->status->flags, sc)); LAUNCHED(h);   // + clears flags[0], flags[7]
		CK(pdl(k_fold, nblk((uint64_t) n * 32, 128), 128, h->st, E, S, P, 1)); LAUNCHED(h);
	}
	if (C.redo_tail && !h->serial && n < FORK_MAX_READS) CK(cudaStreamWaitEvent(h->st, h->ev_side[0], 0));      // join: the rows are compacted
	return FQSK_OK;
}

// Look at the enqueued pass (unless the caller has just done so) and iterate until the segment is settled; then take the
// totals over to the host side.  Returns RC_RETRY when the whole segment has to be set up again.
int seg_finish(fqsk_handle *h, bool have_look) {
	SegCtx &C = h->ctx;
	const EngineStatus &seen = h->look->st;
	for (;;) {
		if (!have_look) CKR(look(h));
		have_look = false;
		const int *fl = seen.flags;
		if (h->dbg_retry_armed) { h->dbg_retry_armed = false; h->seg_extra_pass = true; return RC_RETRY; }     // fault injection (tests)
		if (fl[4]) {
			if (seen.n_miss > h->miss_cap) h->miss_cap = seen.n_miss + seen.n_miss / 4 + 1024;
			if (seen.n_rscript > h->rreq_cap) h->rreq_cap = seen.n_rscript + seen.n_rscript / 4 + 1024;
			if (seen.pool_used > h->pool_cap) h->pool_cap = seen.pool_used + seen.pool_used / 2 + 1024;
			h->seg_extra_pass = true;
			return RC_RETRY;
		}
		if (fl[5]) return fail(h, FQSK_E_CUDA, "internal error: a draw was requested on a path that must not draw");
		if (fl[1]) {
			// a thread-local counter left the deterministic range: redo the segment with the ordered evaluator
			if (!h->hot) { h->hot = true; ++h->S.n_hot_segments; h->seg_extra_pass = true; return RC_RETRY; }
			return fail(h, FQSK_E_CUDA, "internal error: the ordered thread-local evaluator met a lookup it cannot represent");
		}
		if (fl[2] || fl[0] || fl[7]) h->seg_extra_pass = true;
		if (fl[2]) { C.redo_walk = true; C.redo_tail = true; CKR(seg_pass(h)); continue; }      // walk `it` changed pushes: one more thread-local pass
		C.redo_walk = false;
		if (fl[0]) {   // the pre-generated draw window was too short: extend and evaluate the merges again
			CKR(stream_ensure(h, h->rng[ST_B], seen.draws[0] + (1u << 16))); CKR(stream_ensure(h, h->rng[ST_S], seen.draws[1] + (1u << 12)));
			C.E = make_engine_dev(h);
			C.redo_tail = false;
			CKR(seg_pass(h));
			continue;
		}
		if (fl[7]) { C.redo_tail = false; CKR(seg_pass(h)); continue; }                     // a counter saturated inside a merge: offsets moved, merge again
		break;
	}
	h->seg_delta_b = C.S.delta_b; h->seg_delta_s = C.S.delta_s;
	h->cur = 0;
	{
		const SegTotals &tt = seen.totals[h->seg_par];
		h->pend_b = seen.row_tot[0]; h->pend_s = seen.row_tot[1]; h->pend_p = seen.row_tot[2];
		h->hidden_p += seen.row_tot[3];
		for (int i = 0; i < 4; ++i) h->sl_base[i] += tt.letters.v[i];
		h->n_recs = tt.n_rec;
		h->rng[ST_B].consumed += seen.draws[0]; h->rng[ST_S].consumed += seen.draws[1];
		if (h->hot) { h->rng[ST_LB].consumed += seen.hot.draws[0]; h->rng[ST_LS].consumed += seen.hot.draws[1]; }
	}
	for (int i = 0; i < 4; ++i) h->S.draws[i] = h->rng[i].consumed;
	h->unsettled = false;
	return FQSK_OK;
}

// make the outcome of the last fqsk_segment* call final on the host side (records, pending rows, stream positions)
int seg_settle(fqsk_handle *h, bool have_look = false) {
	if (!h->unsettled) return FQSK_OK;
	for (int attempt = 0;; ++attempt) {
		if (attempt > 8) return fail(h, FQSK_E_NOMEM, "segment buffers kept overflowing");
		int rc = seg_finish(h, have_look);
		have_look = false;
		if (rc == RC_RETRY) {
			// the segment is evaluated again from the tables: slots the early grouping (seg_pass with_prefix) claimed must not be seen
			if (h->spec_prefix) { CK(pdl(k_sync_unclaim, h->spec_g, 256, h->st, h->tb.d, h->spec_Y, 1u)); LAUNCHED(h); h->spec_prefix = false; }
			CKR(seg_setup(h)); CKR(seg_pass(h)); continue;
		}
		return rc;
	}
}

// ---------------------------------------------------------------------------------------------------------------
// paired-end front end (fqsk_pe.cuh): pair table, decisions, work items
// ---------------------------------------------------------------------------------------------------------------
int pair_alloc(fqsk_handle *h, PairDev &t, uint64_t slots) {
	t = PairDev{};
	t.b = h->P.bmer_len; t.vm = (1ull << (2 * t.b)) - 1; t.top = ~0ull >> (2 * t.b); t.mask = slots - 1;
	CK(cudaMalloc(&t.keys, ipc_size(h, slots * 8))); CK(cudaMalloc(&t.vcs, ipc_size(h, slots * 8)));
	CK(cudaMemsetAsync(t.keys, 0xFF, slots * 8, h->st)); CK(cudaMemsetAsync(t.vcs, 0xFF, slots * 8, h->st));
	t.world = h->world;
	for (uint32_t i = 0; i < 8; ++i) { t.peer_keys[i] = nullptr; t.peer_vcs[i] = nullptr; }
	t.peer_keys[h->rank] = t.keys; t.peer_vcs[h->rank] = t.vcs;
	return FQSK_OK;
}
int pair_resize(fqsk_handle *h, uint64_t slots) {
	PairDev nt;
	CKR(pair_alloc(h, nt, slots));
	CK(pdl(k_pair_rehash, 148 * 8, 256, h->st, h->pair, nt)); LAUNCHED(h);
	CK(cudaStreamSynchronize(h->st));
	cudaFree(h->pair.keys); cudaFree(h->pair.vcs);
	h->pair = nt;
	++h->S.n_table_growths;
	return FQSK_OK;
}
int pair_reserve(fqsk_handle *h, uint64_t incoming) {     // keep the table at most half full (contents, not layout, are the contract)
	uint64_t slots = h->pair.mask + 1;
	if ((h->pair_items + incoming) * 2 <= slots) return FQSK_OK;
	if (h->world > 1) {
		// shards double together, after the sync that crowded one of them (fqsk_sync_finish -> FQSK_RESHARD): this sync's rows still go into
		// the table as it is -- linear probing works at any load below 1 -- unless it would pass 7/8
		if ((h->pair_items + incoming) * 8 > slots * 7) return fail(h, FQSK_E_CAPACITY, "one sync brings %llu pairs to a pair-table shard of %llu slots holding %llu: create the engines with a larger pair_log2_slots",
		                                                            (unsigned long long) incoming, (unsigned long long) slots, (unsigned long long) h->pair_items);
		return FQSK_OK;
	}
	while ((h->pair_items + incoming) * 2 > slots) slots <<= 1;
	return pair_resize(h, slots);
}
PeSeg pe_seg(fqsk_handle *h) { return PeSeg{h->pe_sk.as<unsigned long long>(), h->pe_sv.as<unsigned long long>(), h->pe_sidx.as<uint32_t>(), h->pe_nt}; }

// Turns the n_pairs pairs of a segment into 3 * n_pairs work items (texts in it_dna, descriptors in it_*).
int pe_front(fqsk_handle *h, const uint8_t *d_dna, uint64_t dna_bytes, const unsigned long long *d_off, const uint32_t *d_len, uint32_t np, uint64_t *item_bytes_bound) {
	const uint32_t nt = 14 * np, ni = 3 * np, b = h->P.bmer_len;
	const uint32_t first1 = h->P.mode == FQSK_MODE_PE_SORTED ? h->P.pmer_len : h->P.prefix_len;      // mate 1: CompressSorted codes from p_len (dna.cpp:1793-1796)
	*item_bytes_bound = dna_bytes + (uint64_t) np * (b + (uint64_t) first1 + h->P.prefix_len) + 64;
	CK(h->pe_tk.ensure((size_t) nt * 8)); CK(h->pe_tv.ensure((size_t) nt * 8)); CK(h->pe_q.ensure((size_t) np * 32));
	CK(h->pe_sk.ensure((size_t) nt * 8)); CK(h->pe_sv.ensure((size_t) nt * 8)); CK(h->pe_sidx.ensure((size_t) nt * 4));
	CK(h->pe_t1.ensure((size_t) nt * 8)); CK(h->pe_t2.ensure((size_t) nt * 8)); CK(h->pe_info.ensure((size_t) np * 12));
	CK(h->it_src.ensure((size_t) ni * 8)); CK(h->it_len.ensure((size_t) ni * 4 + 4)); CK(h->it_bytes.ensure((size_t) ni * 4)); CK(h->it_first.ensure((size_t) ni * 4));
	CK(h->it_bias.ensure((size_t) ni * 4)); CK(h->it_dupprev.ensure((size_t) ni * 4)); CK(h->it_flags.ensure(ni));
	CK(h->it_off32.ensure((size_t) ni * 4 + 4)); CK(h->it_off64.ensure((size_t) ni * 8 + 8)); CK(h->it_dna.ensure(*item_bytes_bound));
	unsigned long long *tk = h->pe_tk.as<unsigned long long>(), *tv = h->pe_tv.as<unsigned long long>(), *q = h->pe_q.as<unsigned long long>();
	CK(pdl(k_pe_minim, nblk((uint64_t) np * 32, 128), 128, h->st, d_dna, d_off, d_len, np, b, tk, tv, q)); LAUNCHED(h);
	// stable two-pass sort of the triples by (key, value): value first, then key
	uint32_t *i1 = (uint32_t *) h->pe_t2.as<uint32_t>();
	CKR(sort_pairs_u64_u32(h, tv, h->pe_t1.as<unsigned long long>(), nullptr, i1, nt, 0, 2 * (int) b));
	CK(pdl(k_pe_gather, nblk(nt, 256), 256, h->st, tk, i1, h->pe_t1.as<unsigned long long>(), nt)); LAUNCHED(h);
	CKR(sort_pairs_u64_u32(h, h->pe_t1.as<unsigned long long>(), h->pe_sk.as<unsigned long long>(), i1, h->pe_sidx.as<uint32_t>(), nt, 0, 2 * (int) b + 1));
	CK(pdl(k_pe_gather, nblk(nt, 256), 256, h->st, tv, h->pe_sidx.as<uint32_t>(), h->pe_sv.as<unsigned long long>(), nt)); LAUNCHED(h);
	h->pe_nt = nt; h->pe_pairs = np;
	PeItems I{h->it_src.as<unsigned long long>(), h->it_len.as<uint32_t>(), h->it_bytes.as<uint32_t>(), h->it_first.as<uint32_t>(), h->it_bias.as<uint32_t>(),
	          h->it_dupprev.as<uint32_t>(), h->it_flags.as<uint8_t>()};
	for (int attempt = 0;; ++attempt) {
		if (attempt > 12) return fail(h, FQSK_E_NOMEM, "pair candidate pool kept overflowing");
		if (h->pe_pool_cap < 64 * np) h->pe_pool_cap = 64 * np;
		CK(h->pe_pool.ensure((size_t) h->pe_pool_cap * 8));
		CK(cudaMemsetAsync(&h->status->pe_pool, 0, sizeof h->status->pe_pool, h->st));
		CK(pdl(k_pe_decide, nblk((uint64_t) np * 32, 128), 128, h->st, h->pair, pe_seg(h), q, d_dna, d_off, d_len, np, h->P.prefix_len, first1, h->pe_pool.as<unsigned long long>(),
		                                                             &h->status->pe_pool.used, h->pe_pool_cap, &h->status->pe_pool.overflow, h->pe_info.as<uint32_t>(), I)); LAUNCHED(h);
		CK(cudaMemcpyAsync(&h->look->st.pe_pool, &h->status->pe_pool, sizeof h->status->pe_pool, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		if (!h->look->st.pe_pool.overflow) break;
		h->pe_pool_cap = h->pe_pool_cap < (1u << 29) ? h->pe_pool_cap * 4 : h->pe_pool_cap;
	}
	ScanChain sc; CKR(scan_chain(h, sc));
	CK(pdl(k_scan_u32x4, std::max<uint32_t>(nblk(ni, SCAN_U32_CHUNK), 1), 1024, h->st, ni, h->it_bytes.as<uint32_t>(), h->it_off32.as<uint32_t>(), (const uint32_t *) nullptr, (uint32_t *) nullptr, (const uint32_t *) nullptr, (uint32_t *) nullptr, (const uint32_t *) nullptr, (uint32_t *) nullptr, h->status->pe_scan, (uint32_t *) nullptr, sc)); LAUNCHED(h);
	CK(pdl(k_pe_fill, nblk((uint64_t) (ni + 1) * 32, 128), 128, h->st, d_dna, I, h->it_off32.as<uint32_t>(), ni, h->it_dna.as<uint8_t>(), h->it_off64.as<unsigned long long>())); LAUNCHED(h);
	return FQSK_OK;
}

// sync: the segment's triples into the global pair table (dna.cpp:2448-2468)
int pe_sync(fqsk_handle *h) {
	if (!h->pe_nt) return FQSK_OK;
	CKR(pair_reserve(h, h->pe_nt));
	CK(pdl(k_pair_insert, nblk(h->pe_nt, 256), 256, h->st, h->pair, pe_seg(h), &h->status->pair_items)); LAUNCHED(h);
	CK(cudaMemcpyAsync(&h->look->st.pair_items, &h->status->pair_items, 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	h->pair_items = h->look->st.pair_items;
	h->pe_nt = 0;
	return FQSK_OK;
}

int run_segment(fqsk_handle *h, const uint8_t *d_dna, uint64_t dna_bytes_actual, const unsigned long long *d_off, const uint32_t *d_len, uint32_t n) {
	if (h->pending) return fail(h, FQSK_E_INVAL, "fqsk_segment called twice without fqsk_sync (the reference syncs after every segment, application.cpp:643-662)");
	const bool pe = mode_pe(h->P.mode);
	const uint32_t n_in = n;
	const uint64_t bytes_in = dna_bytes_actual;
	h->seg_reads_in = n_in; h->pe_nt = 0; h->pe_pairs = 0;
	h->block_fresh = false;
	if (pe && (n & 1)) return fail(h, FQSK_E_INVAL, "paired-end segment with an odd number of reads");
	if (pe && n) {   // pairs -> work items: mate 1, mate 2 (whole or right of the shared minimizer), reversed left part
		uint64_t bound = 0;
		CKR(pe_front(h, d_dna, dna_bytes_actual, d_off, d_len, n / 2, &bound));
		d_dna = h->it_dna.as<uint8_t>(); d_off = h->it_off64.as<unsigned long long>(); d_len = h->it_len.as<uint32_t>();
		n = 3 * (n / 2); dna_bytes_actual = bound;
	}
	const uint64_t dna_bytes = std::max<uint64_t>(dna_bytes_actual, pe ? (uint64_t) h->P.reserve_bytes + h->P.reserve_bytes / 4 : h->P.reserve_bytes);
	if (h->world > 1 && h->grow_pending) return fail(h, FQSK_E_INVAL, "sharded engine: the last sync returned FQSK_RESHARD -- barrier, fqsk_shard_export, exchange, fqsk_shard_attach come first");
	if (h->world > 1 && h->attached != (1u << h->world) - 1) return fail(h, FQSK_E_INVAL, "sharded engine: not every peer shard is attached (fqsk_shard_attach)");
	const uint32_t first = mode_sorted(h->P.mode) ? h->P.pmer_len : h->P.prefix_len;
	h->seg_reads = n; h->n_recs = 0; h->pend_b = h->pend_s = h->pend_p = 0;
	h->hot = false; h->seg_extra_pass = false; h->spec_prefix = false;
	++h->S.n_segments;
	if (n == 0) { h->pending = true; return FQSK_OK; }
	if (dna_bytes >= (1ull << 30)) return fail(h, FQSK_E_INVAL, "segment larger than 1 GiB of DNA");   // push times are 2 * byte offset (+1) in 32 bits
	const size_t n1 = (size_t) std::max<uint32_t>(n, pe ? h->P.reserve_reads / 2 * 3 : h->P.reserve_reads) + 1;
	// announced (fqsk_announce_device)?  Then k_prep / k_scan_reads have run, or are running, on the front stream into the other instance
	const bool fronted = h->front.valid && !pe && h->front.dna == d_dna && h->front.bytes == dna_bytes_actual && h->front.off == d_off && h->front.len == d_len && h->front.n == n;
	if (h->front.valid && !fronted) CK(cudaStreamSynchronize(h->st_front));      // a hint that was not followed: let it drain, its outputs are dropped
	h->front.valid = false;
	if (fronted) h->seg_par = h->front.par;
	const PrepBufs PB = prep_bufs(h, h->seg_par);
	CK(PB.dup->ensure(n1)); CK(PB.n_coded->ensure(n1 * 4)); CK(PB.letters->ensure(n1 * 32)); CK(PB.rec_off->ensure(n1 * 8)); CK(PB.sl_prefix->ensure(n1 * 32));
	CK(h->push_b.ensure((2 * dna_bytes + 2) * 8)); CK(h->push_s.ensure((dna_bytes + 1) * 8)); CK(h->push_p.ensure((2 * dna_bytes + 2 * n1) * 8));
	CK(h->cnt_b.ensure(n1 * 4)); CK(h->cnt_s.ensure(n1 * 4)); CK(h->cnt_p.ensure(n1 * 4)); CK(h->hidden.ensure(n1 * 4));
	CK(h->off_b[0].ensure(n1 * 4)); CK(h->off_s[0].ensure(n1 * 4));
	CK(h->row_b[0].ensure((2 * dna_bytes + 2) * 8)); CK(h->row_s[0].ensure((dna_bytes + 1) * 8));
	CK(h->off_p.ensure(n1 * 4)); CK(h->row_p.ensure((2 * dna_bytes + 2 * n1) * 8));
	CK(h->sflag.ensure(n1 * 4)); CK(h->sdif.ensure(n1 * 8)); CK(h->totals.ensure(256));

	SegCtx &C = h->ctx;
	C.n = n; C.dna_bytes_actual = dna_bytes_actual; C.first = first;
	SegDev &S = C.S;
	S = SegDev{};
	S.dna = d_dna; S.off = d_off; S.len = d_len; S.n_reads = n;
	if (pe) { S.first_a = h->it_first.as<uint32_t>(); S.bias_a = h->it_bias.as<uint32_t>(); S.dup_prev = h->it_dupprev.as<uint32_t>(); S.iflags = h->it_flags.as<uint8_t>(); }
	CK(h->prev_read.ensure_keep((size_t) dna_bytes_actual + 64, h->st));     // a read is never longer than its segment
	S.prev_read = h->prev_read.as<uint8_t>(); S.carry = &h->status->carry;
	S.dup = PB.dup->as<uint8_t>(); S.n_coded = PB.n_coded->as<uint32_t>(); S.letters = PB.letters->as<U64x4>();
	S.rec_off = PB.rec_off->as<unsigned long long>(); S.sl_prefix = PB.sl_prefix->as<U64x4>();
	for (int i = 0; i < 4; ++i) S.sl_base.v[i] = h->sl_base[i];
	S.push_b = h->push_b.as<unsigned long long>(); S.push_s = h->push_s.as<unsigned long long>(); S.push_p = h->push_p.as<unsigned long long>();
	S.cnt_b = h->cnt_b.as<uint32_t>(); S.cnt_s = h->cnt_s.as<uint32_t>(); S.cnt_p = h->cnt_p.as<uint32_t>(); S.hidden = h->hidden.as<uint32_t>();
	S.sorted_flag = h->sflag.as<uint32_t>(); S.sorted_dif = h->sdif.as<unsigned long long>();
	CK(PB.pk->ensure((dna_bytes / 32 + 2 * n1 + 8) * 8));
	S.pk = PB.pk->as<unsigned long long>();
	if (n > SCAN_CHAIN_MAX * SCAN_READS_CHUNK) return fail(h, FQSK_E_INVAL, "more than %u reads in one segment", SCAN_CHAIN_MAX * SCAN_READS_CHUNK);
	if (fronted) CK(cudaStreamWaitEvent(h->st, h->ev_front, 0));      // prep + scan of this segment: done ahead, next to the previous segment
	else {
		Phase ph(h, FQSK_PH_PREP);
		CK(pdl(k_prep, nblk((uint64_t) n * 32, 128), 128, h->st, S, first, h->P.bmer_len, (uint32_t) mode_sorted(h->P.mode), h->status,
		       (const uint8_t *) nullptr, (const unsigned long long *) nullptr, (const uint32_t *) nullptr)); LAUNCHED(h);      // + the segment's status words cleared
		ScanChain sc; CKR(scan_chain(h, sc));
		CK(pdl(k_scan_reads, n <= 1024 ? 1u : nblk(n, SCAN_READS_CHUNK), n <= 1024 ? 256 : 1024, h->st, S, PB.rec_off->as<unsigned long long>(), PB.sl_prefix->as<U64x4>(),
		       &h->status->totals[h->seg_par], &h->status->n_rec[h->seg_par], sc)); LAUNCHED(h);
	}
	const uint32_t rec_bound = (uint32_t) dna_bytes;   // capacities follow the reserve as well
	if (h->miss_cap < std::min<uint32_t>(rec_bound, 1u << 20)) h->miss_cap = std::min<uint32_t>(rec_bound, 1u << 20);
	if (h->miss_cap < rec_bound / 4) h->miss_cap = rec_bound / 4 + 1024;
	if (h->rreq_cap < std::min<uint32_t>(rec_bound, 1u << 20)) h->rreq_cap = std::min<uint32_t>(rec_bound, 1u << 20);
	if (h->rreq_cap < rec_bound / 8) h->rreq_cap = rec_bound / 8 + 1024;
	// draw windows: the merges of the segment and, for a sync enqueued unseen, the ordered inserts of its b-mers
	CKR(stream_ensure(h, h->rng[ST_B], (1u << 16) + (dna_bytes_actual <= SPEC_MAX_BYTES ? 2 * dna_bytes_actual : 0))); CKR(stream_ensure(h, h->rng[ST_S], 1u << 12));
	CKR(seg_setup(h, !fronted));      // (an announced segment's k_prep ran before the previous look: it must not clear the status words)
	if (h->delta_filtered) ++h->S.n_filtered_segments;
	const bool prefix = h->world == 1 && h->fast_ok[0] && dna_bytes_actual <= SPEC_MAX_BYTES;     // the sync of this segment will be enqueued unseen
	CKR(seg_pass(h, prefix));
	h->spec_prefix = prefix;
	// verdict of the first pass for a sync enqueued unseen, and the state the next segment inherits (both are inputs only)
	// one launch: verdict of the first pass + the state the next segment inherits (read_prev, pmer_can_prev)
	CK(pdl(k_seg_tail, 1, 256, h->st, (const int *) h->status->flags, (const uint32_t *) h->status->row_tot, (const unsigned long long *) h->status->draws,
	       h->rng[ST_B].consumed, h->rng[ST_S].consumed, SYNC_INDEXED_MAX, &h->status->syncin,
	       S, pe ? n - 3 : n - 1, h->prev_read.as<uint8_t>(), &h->status->carry, (uint32_t) mode_sorted(h->P.mode), h->P.pmer_len, (uint32_t) prefix,
	       (uint32_t) ((h->dbg_fail_every && h->dbg_seg % h->dbg_fail_every == 0) || (h->dbg_retry_every && h->dbg_seg % h->dbg_retry_every == 1)))); LAUNCHED(h);
	h->dbg_retry_armed = h->dbg_retry_every && h->dbg_seg % h->dbg_retry_every == 1;     // a retry always comes with a failed verdict (as flags[4] would give)
	++h->dbg_seg;
	h->unsettled = true;
	h->pending = true;
	h->S.n_reads += n_in; h->S.n_bases += bytes_in;
	return FQSK_OK;
}

// The reference's thread-local tables draw from cinc_lb / cinc_ls on every insert whose counter is above thr, looked up or
// not (ht_kmer.h:433-436 via dna.cpp:826, 837, 862, 872).  When a sync row shows such a k-mer and the segment was not
// evaluated in hot mode, the ordered evaluator runs in accounting mode to advance the stream position exactly.
// first half of hot_account without the look: counts, per stream, the pushes of the segment that would draw from the thread-local
// incrementer (rank >= thr + 1) into hot.ev[stream]; the caller has cleared the counters and reads them with its next look
int hot_rank(fqsk_handle *h, int stream) {
	DeltaDev D = stream ? h->seg_delta_s : h->seg_delta_b;
	if (!D.keys || h->delta_filtered) return FQSK_OK;      // (a filtered delta exists on unsharded engines only; they account through hot_seen)
	const size_t slots = (size_t) D.mask + 1;
	DevBuf *hr = stream ? h->hr_s : h->hr_b;
	for (int q = 0; q < 3; ++q) CK(hr[q].ensure(slots * 4));
	D.rank_at = hr[0].as<uint32_t>(); D.prev_at = hr[1].as<uint32_t>(); D.cnt_at = hr[2].as<uint32_t>();
	PipeDev P{};
	P.ev_n = h->status->hot.ev; P.ev_cap = 0; P.hot_draws = h->status->hot.draws; P.flags = h->status->rank_flags;      // count only: ev_cap 0 stores nothing but sets the overflow flag
	CK(pdl(k_delta_rank, 148 * 8, 256, h->st, D, P, (uint32_t) stream)); LAUNCHED(h);
	return FQSK_OK;
}
int hot_account(fqsk_handle *h, int stream) {
	if (h->delta_filtered) {    // the accounting needs every push of the segment: build the unfiltered delta (rare: repeats inside one segment)
		CKR(seg_build_delta(h, true));
		h->seg_delta_b = h->ctx.S.delta_b; h->seg_delta_s = h->ctx.S.delta_s;
		h->delta_filtered = false;
	}
	DeltaDev D = stream ? h->seg_delta_s : h->seg_delta_b;
	if (!D.keys) return FQSK_OK;
	const size_t slots = (size_t) D.mask + 1;
	DevBuf *hr = stream ? h->hr_s : h->hr_b;
	for (int q = 0; q < 3; ++q) CK(hr[q].ensure(slots * 4));
	D.rank_at = hr[0].as<uint32_t>(); D.prev_at = hr[1].as<uint32_t>(); D.cnt_at = hr[2].as<uint32_t>();
	const uint32_t ev_cap = (uint32_t) std::min<size_t>(slots, 1u << 30);
	CK(h->evk[stream].ensure((size_t) ev_cap * 8)); CK(h->evv[stream].ensure((size_t) ev_cap * 4));
	CK(h->evk_s[stream].ensure((size_t) ev_cap * 8)); CK(h->evv_s[stream].ensure((size_t) ev_cap * 4));
	PipeDev P{};
	for (int q = 0; q < 2; ++q) { P.ev_key[q] = h->evk[q].as<unsigned long long>(); P.ev_val[q] = h->evv[q].as<uint32_t>(); }
	P.ev_n = h->status->hot.ev; P.ev_cap = ev_cap; P.hot_draws = h->status->hot.draws; P.flags = h->status->flags;
	CK(cudaMemsetAsync(&h->status->hot, 0, sizeof h->status->hot, h->st));
	CK(cudaMemsetAsync(h->status->flags, 0, 8 * sizeof(int), h->st));
	CK(pdl(k_delta_rank, 148 * 8, 256, h->st, D, P, (uint32_t) stream)); LAUNCHED(h);
	EngineStatus &seen = h->look->st;
	CK(cudaMemcpyAsync(&seen, h->status, sizeof seen, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	uint32_t en = seen.hot.ev[stream];
	if (!en) return FQSK_OK;
	CKR(sort_pairs_u64_u32(h, h->evk[stream].as<unsigned long long>(), h->evk_s[stream].as<unsigned long long>(), h->evv[stream].as<uint32_t>(), h->evv_s[stream].as<uint32_t>(), en, 0, 34));      // by time
	Stream &rng = h->rng[stream ? ST_LS : ST_LB];
	CKR(stream_ensure(h, rng, (uint64_t) en + 1024));
	EngineDev E = make_engine_dev(h);
	SegDev S{};
	S.delta_b = stream ? DeltaDev{} : D; S.delta_s = stream ? D : DeltaDev{};
	CK(h->hot_tab.ensure((size_t) 2 * 3 * HOT_TAB_ENTRIES * 4)); CK(cudaMemsetAsync(h->hot_tab.p, 0, (size_t) 2 * 3 * HOT_TAB_ENTRIES * 4, h->st));
	CK(pdl(k_hot_eval, 1, 64, h->st, E, S, P, h->evk_s[0].as<unsigned long long>(), h->evv_s[0].as<uint32_t>(), stream ? 0 : en,
	                               h->evk_s[1].as<unsigned long long>(), h->evv_s[1].as<uint32_t>(), stream ? en : 0, h->hot_tab.as<uint32_t>()));
	LAUNCHED(h);
	CK(cudaMemcpyAsync(&seen, h->status, sizeof seen, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (seen.flags[0]) return fail(h, FQSK_E_CUDA, "internal error: thread-local draw window too short");
	rng.consumed += seen.hot.draws[stream];
	return FQSK_OK;
}

}  // namespace

// =================================================================================================================
// C-ABI
// =================================================================================================================
extern "C" {

const char *fqsk_last_error(fqsk_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

static int prealloc_for_reserve(fqsk_handle *h);

int fqsk_create(const fqsk_params *p, fqsk_handle **out) {
	fqsk_handle *h = nullptr;
	if (!p || !out) return fail(h, FQSK_E_INVAL, "null argument");
	*out = nullptr;
	if (p->abi_version != FQSK_ABI_VERSION) return fail(h, FQSK_E_INVAL, "ABI version %u, library is %u", p->abi_version, FQSK_ABI_VERSION);
	const uint32_t world = p->world_size ? p->world_size : 1;
	if (world > FQSK_MAX_WORLD || p->rank >= world) return fail(h, FQSK_E_INVAL, "need rank < world_size <= %u", FQSK_MAX_WORLD);
	if (p->n_workers != world) return fail(h, FQSK_E_INVAL, "n_workers must equal world_size: one reference worker thread (-t) per GPU");
	if (world > 1 && (p->mode == FQSK_MODE_SE_SORTED || p->mode == FQSK_MODE_PE_SORTED) && p->pmer_len < 8) return fail(h, FQSK_E_UNSUPPORTED, "sharded operation in sorted order needs pmer_len >= 8 (a 16-field word of the p-mer array must lie inside one owner's run)");
	if (!(p->pmer_len >= 5 && p->pmer_len < p->smer_len && p->smer_len < p->bmer_len && p->bmer_len <= 31)) return fail(h, FQSK_E_INVAL, "need 5 <= p < s < b <= 31");
	if (p->pmer_len > 18) return fail(h, FQSK_E_INVAL, "pmer_len > 18 not supported");
	if (p->test_hooks && !(p->flags & FQSK_F_TEST_HOOKS)) return fail(h, FQSK_E_INVAL, "test_hooks without FQSK_F_TEST_HOOKS");
	if (p->mode > FQSK_MODE_PE_SORTED) return fail(h, FQSK_E_INVAL, "mode %u: not a dna_mode_t (params.h:18)", p->mode);
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(h, FQSK_E_NO_DEVICE, "no CUDA device: this library has no CPU path");
	if (p->device < 0 || p->device >= ndev) return fail(h, FQSK_E_INVAL, "device %d out of range (%d devices)", p->device, ndev);
	{
		cudaError_t e = cudaSetDevice(p->device);
		if (e != cudaSuccess) return fail(h, FQSK_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
	}
	h = new fqsk_handle();
	h->P = *p;
	h->world = world; h->rank = p->rank;
	h->prof = (p->flags & FQSK_F_PROFILE) != 0;
	h->trace_launch = (p->flags & FQSK_F_TRACE_LAUNCH) != 0;
	h->serial = h->prof || h->trace_launch || (p->flags & FQSK_F_SERIAL) != 0;      // phase brackets measure what they say on one stream
	// Fault injection (tests only; needs FQSK_F_TEST_HOOKS in the parameters, nothing is read from the environment): every N-th
	// segment has its first-pass verdict forced to "not settled" after the early grouping has run (exercises k_sync_unclaim + the
	// plain sync), resp. is evaluated a second time from scratch as after a capacity overflow (exercises the release of claimed
	// slots before the tables are read again).
	if (p->flags & FQSK_F_TEST_HOOKS) { h->dbg_fail_every = p->test_hooks & 0xFFFFu; h->dbg_retry_every = p->test_hooks >> 16; }
	if ((p->flags & FQSK_F_TEST_HOOKS) && (p->flags & FQSK_F_TEST_CROWD)) h->crowd_shift = 6;
	if (p->flags & FQSK_F_TRACE_ALLOC) g_trace_alloc.store(true);
	int rc = [&]() -> int {
		int prio_lo = 0, prio_hi = 0;
		CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
		CK(cudaStreamCreateWithPriority(&h->st, cudaStreamNonBlocking, prio_hi));         // see ensure_side
		CK(cudaStreamCreateWithPriority(&h->st_mt, cudaStreamNonBlocking, prio_hi));      // the mt19937 generator: 32 CTAs that work ahead; at a lower priority the full grids of
		                                                                                  // a large segment starved it and the ordered b-mer insert waited 0.8 ms for its draws
		CK(cudaMalloc(&h->status, sizeof(EngineStatus))); CK(cudaMemset(h->status, 0, sizeof(EngineStatus)));
		CK(cudaMallocHost(&h->look, sizeof(LookBuf)));
		memset(h->look, 0, sizeof(LookBuf));
		uint64_t expect = p->expected_kmers ? p->expected_kmers : (1ull << 22);
		uint32_t Bauto = 1;
		while ((4ull << Bauto) < expect && Bauto < 30) ++Bauto;    // <= 50 % of 8 << B slots
		CKR(table_alloc(h, h->tb, p->bmer_len, p->bmer_counter_bits ? p->bmer_counter_bits : 6, p->bmer_log2_buckets ? p->bmer_log2_buckets : Bauto, &h->status->items[0]));
		CKR(table_alloc(h, h->ts, p->smer_len, p->smer_counter_bits ? p->smer_counter_bits : 12, p->smer_log2_buckets ? p->smer_log2_buckets : Bauto, &h->status->items[2]));
		h->tb.ci = CIncP{7, 2, h->tb.d.top};                                  // cinc_b.Reset(7, 2, 63)            dna.cpp:162
		h->ts.ci = CIncP{h->ts.d.top / 2, 1, h->ts.d.top};                    // cinc_s.Reset(4095 / 2, 1, 4095)   dna.cpp:163
		if (h->tb.ci.thr > h->tb.ci.top) h->tb.ci.thr = h->tb.ci.top;
		h->siv.key_bits = 2 * p->pmer_len;                                    // application.cpp:88
		h->siv.world = world; h->siv.rank = p->rank; h->siv.top_shift = h->siv.key_bits - 12;
		size_t sb = world > 1 ? ((((size_t) 4096 + world - 1) / world) << h->siv.top_shift) / 4 : ((size_t) 1 << h->siv.key_bits) / 4;
		CK(cudaMalloc(&h->siv.w, ipc_size(h, sb)));
		CK(cudaMemsetAsync(h->siv.w, 0, sb, h->st));
		for (uint32_t i = 0; i < FQSK_MAX_WORLD; ++i) h->siv.peer_w[i] = nullptr;
		h->siv.peer_w[p->rank] = h->siv.w;
		if (world > 1) {
			// inbox: [64-word header: posted slot lengths][3 tables][world sources][cap k-mers]; a source never sends more than its own rows
			const uint64_t rb = p->reserve_bytes ? p->reserve_bytes : (1u << 23), rr = p->reserve_reads ? p->reserve_reads : (1u << 16);
			h->inbox_cap = 2 * rb + 2 * rr + 1024;
			size_t ib = (INBOX_HDR + 6ull * world * h->inbox_cap) * 8;      // tables 0-2: p / s / b rows; 3-5: key / value / weight planes of the pair rows
			CK(cudaMalloc(&h->inbox, ipc_size(h, ib)));
			CK(cudaMemsetAsync(h->inbox, 0, INBOX_HDR * 8, h->st));
			h->peer_inbox[p->rank] = h->inbox;
			h->attached = 1u << p->rank;
		}
		for (int i = 0; i < 4; ++i) CKR(stream_init(h, h->rng[i], i == ST_B ? (1ull << 25) : i == ST_S ? (1ull << 21) : (1ull << 16)));
		CKR(stream_generate(h, h->rng[ST_B], h->P.expected_kmers >= (1ull << 26) ? (1u << 23) + 4096 : (1u << 22))); CKR(stream_generate(h, h->rng[ST_S], 1u << 18));      // large jobs: the parallel generator (and its polynomials) from the start
		CK(h->prev_read.ensure(1 << 16));
		if (mode_pe(p->mode)) {          // CHT_pair_kmers(bmer_len, ...), application.cpp:91
			CKR(pair_alloc(h, h->pair, 1ull << (p->pair_log2_slots ? std::min<uint32_t>(std::max<uint32_t>(p->pair_log2_slots, 10), 34) : (world > 1 ? 22u : 16u))));
		}
		CK(cudaStreamSynchronize(h->st));
		CKR(prealloc_for_reserve(h));
		return FQSK_OK;
	}();
	if (rc != FQSK_OK) { g_create_error = h->err; fqsk_destroy(h); return rc; }
	*out = h;
	return FQSK_OK;
}

void fqsk_destroy(fqsk_handle *h) {
	if (!h) return;
	cudaSetDevice(h->P.device);
	if (h->st) cudaStreamSynchronize(h->st);
	for (Table *t : {&h->tb, &h->ts}) { if (t->d.main) cudaFree(t->d.main); if (t->d.stash) cudaFree(t->d.stash); if (t->d.occ) cudaFree(t->d.occ); }
	if (h->siv.w) cudaFree(h->siv.w);
	for (uint32_t i = 0; i < FQSK_MAX_WORLD; ++i) for (int q = 0; q < 8; ++q) if (h->peer_ptrs[i][q]) cudaIpcCloseMemHandle(h->peer_ptrs[i][q]);
	if (h->inbox) cudaFree(h->inbox);
	if (h->pair.keys) cudaFree(h->pair.keys);
	if (h->pair.vcs) cudaFree(h->pair.vcs);
	if (h->st_mt) cudaStreamSynchronize(h->st_mt);
	for (auto &s : h->rng) { if (s.buf) cudaFree(s.buf); if (s.state) cudaFree(s.state); if (s.jstates) cudaFree(s.jstates); if (s.ev) cudaEventDestroy(s.ev); }
	if (h->status) cudaFree(h->status);
	DevBuf *bufs[] = {&h->prev_read, &h->dna, &h->dna2, &h->off, &h->len, &h->dup, &h->n_coded, &h->letters, &h->rec_off, &h->sl_prefix, &h->recs, &h->push_b, &h->push_s,
	                  &h->push_p, &h->cnt_b, &h->cnt_s, &h->cnt_p, &h->hidden, &h->draw_cnt, &h->draw_cnt_prev, &h->draw_scan, &h->off_b[0], &h->off_b[1], &h->off_s[0],
	                  &h->off_s[1], &h->off_p, &h->row_b[0], &h->row_b[1], &h->row_s[0], &h->row_s[1], &h->row_p, &h->dk_b, &h->di_b, &h->dk_s, &h->di_s, &h->iota,
	                  &h->cub_tmp, &h->flag8, &h->draw_off, &h->final_cnt, &h->slot_of, &h->dump_k, &h->dump_v, &h->q0, &h->q1,
	                  &h->q2, &h->q3, &h->q4, &h->sflag, &h->sdif, &h->hid_scan, &h->prov, &h->pflags, &h->pscripts, &h->rscripts, &h->rreqs, &h->pool, &h->miss,
	                  &h->draws_b16, &h->draws_s16, &h->doff_b, &h->doff_s, &h->time_b, &h->time_s, &h->rt_b[0], &h->rt_b[1], &h->rt_s[0], &h->rt_s[1],
	                  &h->sidx_b, &h->sidx_s, &h->stime_b, &h->stime_s, &h->sort_k, &h->sort_v, &h->rkind, &h->rreg, &h->rslot, &h->dirty, &h->rdraws_b, &h->rdraws_s, &h->totals,
	                  &h->y_tslot, &h->y_c0, &h->y_m, &h->y_draw, &h->y_j, &h->y_final, &h->y_flag_at, &h->y_own, &h->y_lead, &h->y_rank, &h->y_flag, &h->y_doff,
	                  &h->idx_k, &h->idx_t, &h->idx_rt, &h->miss_fold, &h->hr_b[0], &h->hr_b[1], &h->hr_b[2], &h->hr_s[0], &h->hr_s[1], &h->hr_s[2],
	                  &h->evk[0], &h->evk[1], &h->evv[0], &h->evv[1], &h->evk_s[0], &h->evk_s[1], &h->evv_s[0], &h->evv_s[1], &h->ctxrec[0], &h->ctxrec[1], &h->scan_part, &h->scan8_part, &h->rdx_hist, &h->rdx_k, &h->rdx_v, &h->scan_vals, &h->recs_alt, &h->dfilter, &h->pk,
	                  &h->route_keys, &h->route_keys2, &h->route_sorted, &h->route_hist, &h->route_perm, &h->route_chunks, &h->hot_tab, &h->f_dup, &h->f_n_coded, &h->f_letters, &h->f_rec_off, &h->f_sl_prefix, &h->f_pk,
	                  &h->pe_uk, &h->pe_uv, &h->pe_uc, &h->pe_tk, &h->pe_tv, &h->pe_q, &h->pe_sk, &h->pe_sv, &h->pe_sidx, &h->pe_t1, &h->pe_t2, &h->pe_pool, &h->pe_info, &h->it_src, &h->it_len,
	                  &h->it_bytes, &h->it_first, &h->it_bias, &h->it_dupprev, &h->it_flags, &h->it_off32, &h->it_off64, &h->it_dna};

	for (DevBuf *b : bufs) b->release();
	if (h->h_stage) cudaFreeHost(h->h_stage);
	if (h->h_stage2) cudaFreeHost(h->h_stage2);
	for (int i = 0; i < 2; ++i) { if (h->h_meta[i]) cudaFreeHost(h->h_meta[i]); if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]); }
	if (h->ev_recs) cudaEventDestroy(h->ev_recs);
	if (h->ev_meta) cudaEventDestroy(h->ev_meta);
	for (int i = 0; i < 3; ++i) { if (h->st_side[i]) { cudaStreamSynchronize(h->st_side[i]); cudaStreamDestroy(h->st_side[i]); } if (h->ev_side[i]) cudaEventDestroy(h->ev_side[i]); }
	if (h->ev_fork) cudaEventDestroy(h->ev_fork);
	if (h->ev_aux) cudaEventDestroy(h->ev_aux);
	if (h->st_front) { cudaStreamSynchronize(h->st_front); cudaStreamDestroy(h->st_front); }
	if (h->ev_front) cudaEventDestroy(h->ev_front);
	if (h->ev_up) cudaEventDestroy(h->ev_up);
	if (h->st_copy) { cudaStreamSynchronize(h->st_copy); cudaStreamDestroy(h->st_copy); }
	if (h->look) cudaFreeHost(h->look);
	for (auto &e : h->evs) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
	for (auto e : h->ev_pool) cudaEventDestroy(e);
	if (h->t0) { cudaEventDestroy(h->t0); cudaEventDestroy(h->t1); }
	if (h->st) cudaStreamDestroy(h->st);
	if (h->st_mt) cudaStreamDestroy(h->st_mt);
	delete h;
}

// With a reserve hint everything a sync of the largest announced segment needs is allocated up front: cudaMalloc inside a run
// costs anything from 0.1 to 600 ms depending on the state of the driver (measured: blocks 84-97 of the config-2 job, where the
// radix-sort path, its scratch and the delta filter were first used, took 256-603 ms instead of 10 in some runs).
static int prealloc_for_reserve(fqsk_handle *h) {
	if (!h->P.reserve_bytes) return FQSK_OK;
	const size_t nr = row_reserve(h, 0);
	CK(h->sort_k.ensure(nr * 8)); CK(h->sort_v.ensure(nr * 4));
	CKR(rdx_scratch(h, (uint32_t) nr, true));
	{ const size_t need = (size_t) nblk((uint32_t) nr, SCAN8_TILE) * 8 + 64; CK(h->scan8_part.ensure(need)); CK(cudaMemsetAsync(h->scan8_part.p, 0, h->scan8_part.cap, h->st)); }
	CK(h->slot_of.ensure(nr * 8)); CK(h->flag8.ensure(nr + 4)); CK(h->draw_off.ensure((nr + 1) * 4)); CK(h->final_cnt.ensure(nr * 4));
	CK(h->q4.ensure(nr + 4)); CK(h->y_flag.ensure(nr + 64));
	if (h->world == 1 && h->P.reserve_bytes >= (1u << 20)) { CK(h->dfilter.ensure((size_t) 2 * (1u << 26) / 8)); }
	if (mode_pe(h->P.mode)) CK(h->pe_pool.ensure((size_t) std::max<uint32_t>(h->pe_pool_cap, 64 * (h->P.reserve_reads / 2 + 1)) * 8));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}

struct ApiTimer { fqsk_handle *h; std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
                  ~ApiTimer() { if (h) h->S.api_ns += (uint64_t) std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count(); } };
int fqsk_block_start(fqsk_handle *h) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	CK(cudaMemsetAsync(&h->status->carry.prev_len, 0, 4, h->st));   // read_prev.clear(), application.cpp:624
	h->block_fresh = true;
	return FQSK_OK;
}

int fqsk_segment_device(fqsk_handle *h, const uint8_t *d_dna, uint64_t dna_bytes, const uint64_t *d_off, const uint32_t *d_len, uint32_t n_reads, uint64_t *n_recs) {
	if (!h) return FQSK_E_INVAL;
	ApiTimer api_timer{h};
	CK(cudaSetDevice(h->P.device));
	h->tk_info = -1;
	if (h->meta_pending) { CK(cudaStreamWaitEvent(h->st, h->ev_meta, 0)); h->meta_pending = false; }
	CKR(run_segment(h, d_dna, dna_bytes, (const unsigned long long *) d_off, d_len, n_reads));
	if (n_recs) { CKR(seg_settle(h)); *n_recs = h->n_recs; }    // pass NULL to leave the look to fqsk_sync / fqsk_device_recs
	return FQSK_OK;
}

// The caller names the segment its NEXT fqsk_segment_device call will bring while the current one is still in flight (between that
// call and its fqsk_sync): duplicate flags, letter totals, packed reads and record offsets of the announced reads are functions of the
// reads alone (read_prev of its first read = the last read of the segment in flight, dna.cpp:1521-1533), so k_prep / k_scan_reads run
// now, on a side stream, instead of at the head of the next segment's dependent chain.  A hint: ignored where it does not apply.
static int ensure_front(fqsk_handle *h) {
	if (h->st_front) return FQSK_OK;
	int lo = 0, hi = 0;
	CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
	CK(cudaStreamCreateWithPriority(&h->st_front, cudaStreamNonBlocking, lo));      // works ahead: yields to the chain of the segment in flight
	CK(cudaEventCreateWithFlags(&h->ev_front, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&h->ev_up, cudaEventDisableTiming));
	return FQSK_OK;
}
static int announce_impl(fqsk_handle *h, const uint8_t *d_dna, uint64_t dna_bytes, const uint64_t *d_off, const uint32_t *d_len, uint32_t n_reads);
int fqsk_announce_device(fqsk_handle *h, const uint8_t *d_dna, uint64_t dna_bytes, const uint64_t *d_off, const uint32_t *d_len, uint32_t n_reads) {
	if (!h) return FQSK_E_INVAL;
	ApiTimer api_timer{h};
	CK(cudaSetDevice(h->P.device));
	return announce_impl(h, d_dna, dna_bytes, d_off, d_len, n_reads);
}
// (the arrays may still be on their way: when they are filled by a copy on the front stream -- fqsk_submit -- the kernels below follow it in stream order)
static int announce_impl(fqsk_handle *h, const uint8_t *d_dna, uint64_t dna_bytes, const uint64_t *d_off, const uint32_t *d_len, uint32_t n_reads) {
	if (h->front.valid) { CK(cudaStreamSynchronize(h->st_front)); h->front.valid = false; }
	const SegCtx &C = h->ctx;
	if (mode_pe(h->P.mode) || h->serial || !n_reads || !d_dna || !d_off || !d_len || !h->pending || !h->seg_reads || !C.n) return FQSK_OK;
	if (n_reads > SCAN_CHAIN_MAX * SCAN_READS_CHUNK || dna_bytes >= (1ull << 30)) return FQSK_OK;
	const uint64_t bytes_r = std::max<uint64_t>(dna_bytes, h->P.reserve_bytes);
	const size_t n1 = (size_t) std::max<uint32_t>(n_reads, h->P.reserve_reads) + 1;
	const int par = h->seg_par ^ 1;
	const PrepBufs PB = prep_bufs(h, par);
	const size_t need[6] = {n1, n1 * 4, n1 * 32, n1 * 8, n1 * 32, (bytes_r / 32 + 2 * n1 + 8) * 8};
	DevBuf *bufs[6] = {PB.dup, PB.n_coded, PB.letters, PB.rec_off, PB.sl_prefix, PB.pk};
	for (int i = 0; i < 6; ++i) CK(bufs[i]->ensure(need[i]));
	CKR(ensure_front(h));
	SegDev S{};
	S.dna = d_dna; S.off = (const unsigned long long *) d_off; S.len = d_len; S.n_reads = n_reads;
	S.carry = &h->status->carry; S.prev_read = h->prev_read.as<uint8_t>();      // (not read: read_prev comes from the segment in flight, below)
	S.dup = PB.dup->as<uint8_t>(); S.n_coded = PB.n_coded->as<uint32_t>(); S.letters = PB.letters->as<U64x4>();
	S.rec_off = PB.rec_off->as<unsigned long long>(); S.sl_prefix = PB.sl_prefix->as<U64x4>(); S.pk = PB.pk->as<unsigned long long>();
	const uint32_t first = mode_sorted(h->P.mode) ? h->P.pmer_len : h->P.prefix_len;
	const uint32_t last = C.n - 1;      // read_prev of the announced segment's first read: the last read of the segment in flight
	CK(pdl(k_prep, nblk((uint64_t) n_reads * 32, 128), 128, h->st_front, S, first, h->P.bmer_len, (uint32_t) mode_sorted(h->P.mode), (EngineStatus *) nullptr,
	       C.S.dna, C.S.off + last, C.S.len + last)); LAUNCHED(h);
	ScanChain sc; CKR(scan_chain(h, sc, 2));
	CK(pdl(k_scan_reads, n_reads <= 1024 ? 1u : nblk(n_reads, SCAN_READS_CHUNK), n_reads <= 1024 ? 256 : 1024, h->st_front, S, PB.rec_off->as<unsigned long long>(), PB.sl_prefix->as<U64x4>(),
	       &h->status->totals[par], &h->status->n_rec[par], sc)); LAUNCHED(h);
	CK(cudaEventRecord(h->ev_front, h->st_front));
	h->front.valid = true; h->front.dna = d_dna; h->front.bytes = dna_bytes; h->front.off = (const unsigned long long *) d_off; h->front.len = d_len; h->front.n = n_reads; h->front.par = par;
	return FQSK_OK;
}

int fqsk_device_recs(fqsk_handle *h, const fqsk_base_rec **d_recs, uint64_t *n_recs) {
	if (!h || !d_recs) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	CKR(seg_settle(h));
	*d_recs = (h->rec_par ? h->recs_alt : h->recs).as<fqsk_base_rec>();
	if (n_recs) *n_recs = h->n_recs;
	return FQSK_OK;
}

int fqsk_recs_checksum(fqsk_handle *h, uint64_t *sum, uint64_t *n_recs) {
	if (!h || !sum) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	CKR(seg_settle(h));
	unsigned long long *d_sum = &h->status->scratch[0];
	CK(cudaMemsetAsync(d_sum, 0, 8, h->st));
	if (h->n_recs) { CK(pdl(k_recs_checksum, std::min<uint32_t>(nblk(h->n_recs, 256), 148 * 8), 256, h->st, (const fqsk_base_rec *) (h->rec_par ? h->recs_alt : h->recs).as<fqsk_base_rec>(), (unsigned long long) h->n_recs, d_sum)); LAUNCHED(h); }
	CK(cudaMemcpyAsync(&h->look->st.scratch[0], d_sum, 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	*sum = h->look->st.scratch[0];
	if (n_recs) *n_recs = h->n_recs;
	return FQSK_OK;
}

int fqsk_sorted_prefix(fqsk_handle *h, uint32_t *flag, uint64_t *dif, uint32_t n_reads) {
	if (!h || !flag || !dif) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->tk_info >= 0) {      // the segment of the ticket collected last: served from its page-locked copies
		const auto &T = h->tk[h->tk_info];
		if (n_reads > T.n_reads) return fail(h, FQSK_E_INVAL, "the collected segment had %u reads", T.n_reads);
		const bool pe = mode_pe(h->P.mode);
		const uint32_t ni = pe ? T.n_reads / 2 * 3 : T.n_reads;
		const size_t o_off = ((size_t) ni + 8) & ~(size_t) 7, o_flag = o_off + ((size_t) ni + 1) * 8, o_dif = o_flag + ((((size_t) ni + 1) * 4 + 7) & ~(size_t) 7);
		const uint32_t *f = (const uint32_t *) (h->h_meta[h->tk_info] + o_flag);
		const unsigned long long *d = (const unsigned long long *) (h->h_meta[h->tk_info] + o_dif);
		for (uint32_t i = 0; i < n_reads; ++i) {
			const uint32_t it = pe ? 3 * (i / 2) : i;
			flag[i] = (pe && (i & 1)) ? 0u : f[it]; dif[i] = (pe && (i & 1)) ? 0ull : d[it];
		}
		return FQSK_OK;
	}
	if (n_reads > h->seg_reads) return fail(h, FQSK_E_INVAL, "last segment had %u reads", h->seg_reads);
	if (!n_reads) return FQSK_OK;
	CKR(seg_settle(h));
	if (mode_pe(h->P.mode)) {      // per read: the first mate of pair i is item 3i; second mates have no sorted prefix (zeros)
		if (n_reads > h->seg_reads_in) return fail(h, FQSK_E_INVAL, "last segment had %u reads", h->seg_reads_in);
		const uint32_t ni = (n_reads + 1) / 2 * 3;
		std::vector<uint32_t> f(ni); std::vector<unsigned long long> d(ni);
		CK(cudaMemcpyAsync(f.data(), h->sflag.p, (size_t) ni * 4, cudaMemcpyDeviceToHost, h->st));
		CK(cudaMemcpyAsync(d.data(), h->sdif.p, (size_t) ni * 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		for (uint32_t i = 0; i < n_reads; ++i) { flag[i] = (i & 1) ? 0u : f[3 * (i / 2)]; dif[i] = (i & 1) ? 0ull : d[3 * (i / 2)]; }
		return FQSK_OK;
	}
	CK(cudaMemcpyAsync(flag, h->sflag.p, (size_t) n_reads * 4, cudaMemcpyDeviceToHost, h->st));
	CK(cudaMemcpyAsync(dif, h->sdif.p, (size_t) n_reads * 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}

int fqsk_pair_info(fqsk_handle *h, uint32_t *info, uint32_t n_pairs) {
	if (!h || (!info && n_pairs)) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (!mode_pe(h->P.mode)) return fail(h, FQSK_E_INVAL, "not a paired-end engine");
	if (h->tk_info >= 0) {      // the segment of the ticket collected last
		const auto &T = h->tk[h->tk_info];
		if (n_pairs > T.n_reads / 2) return fail(h, FQSK_E_INVAL, "the collected segment had %u pairs", T.n_reads / 2);
		const uint32_t ni = T.n_reads / 2 * 3;
		const size_t o_off = ((size_t) ni + 8) & ~(size_t) 7, o_flag = o_off + ((size_t) ni + 1) * 8, o_dif = o_flag + ((((size_t) ni + 1) * 4 + 7) & ~(size_t) 7), o_pair = o_dif + (size_t) ni * 8;
		if (n_pairs) memcpy(info, h->h_meta[h->tk_info] + o_pair, (size_t) n_pairs * 12);
		return FQSK_OK;
	}
	if (n_pairs > h->pe_pairs) return fail(h, FQSK_E_INVAL, "last segment had %u pairs", h->pe_pairs);
	if (!n_pairs) return FQSK_OK;
	CK(cudaMemcpyAsync(info, h->pe_info.p, (size_t) n_pairs * 12, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}

// pack the DNA bytes of the segment (plus the few bytes the reference also reads when a read is shorter than the directly coded
// prefix, dna.cpp:518-521) into pinned memory -- [dna bytes | off u64 | len u32] -- and enqueue the copy to the device.
// *rec_bound = upper bound of the records the segment produces (exact unless it holds duplicates).
static int stage_segment(fqsk_handle *h, uint8_t *&stage, size_t &stage_cap, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads,
                         uint64_t *total_out, uint64_t *rec_bound) {
	const uint32_t first = mode_sorted(h->P.mode) ? h->P.pmer_len : h->P.prefix_len;      // paired end, sorted order: only first mates need p symbols, padding the second ones is harmless
	uint64_t total = 0, bound = 0;
	const bool pe_sorted = h->P.mode == FQSK_MODE_PE_SORTED;      // second mates are coded from prefix_len (CompressDirect), first mates from p_len
	for (uint32_t i = 0; i < n_reads; ++i) {
		total += std::max(reads[i].dna_len, first);
		const uint32_t coded_from = (pe_sorted && (i & 1)) ? h->P.prefix_len : first;
		if (reads[i].dna_len > coded_from) bound += reads[i].dna_len - coded_from;
	}
	size_t need = total + 64 + (size_t) n_reads * 12 + 64;
	if (need > stage_cap) {
		if (stage) cudaFreeHost(stage);
		stage = nullptr; stage_cap = 0;
		size_t want = std::max<size_t>(need + need / 4, (size_t) h->P.reserve_bytes + (size_t) h->P.reserve_reads * 16 + 4096);
		CK(cudaMallocHost(&stage, want));
		stage_cap = want;
	}
	size_t off_pos = (total + 63) & ~(size_t) 63;
	unsigned long long *h_off = (unsigned long long *) (stage + off_pos);
	uint32_t *h_len = (uint32_t *) (stage + off_pos + (size_t) n_reads * 8);
	uint64_t at = 0;
	for (uint32_t i = 0; i < n_reads; ++i) {
		uint32_t plen = std::max(reads[i].dna_len, first);
		uint64_t o = reads[i].dna_off;
		if (o > slab_size || reads[i].dna_len > slab_size - o) return fail(h, FQSK_E_INVAL, "read %u (offset %llu, %u symbols) does not lie inside the slab of %llu bytes", i, (unsigned long long) o, reads[i].dna_len, (unsigned long long) slab_size);
		uint64_t avail = std::min<uint64_t>(plen, slab_size - o);
		memcpy(stage + at, slab + o, avail);
		if (avail < plen) memset(stage + at + avail, 0, plen - avail);
		h_off[i] = at; h_len[i] = reads[i].dna_len;
		at += plen;
	}
	*total_out = total; *rec_bound = bound;
	return FQSK_OK;
}
// one H2D copy: the device buffer mirrors the staging layout [dna | off u64 | len u32]
struct Uploaded { const uint8_t *dna; const unsigned long long *off; const uint32_t *len; };
static int upload_segment(fqsk_handle *h, const uint8_t *stage, uint64_t total, uint32_t n_reads, Uploaded &U, DevBuf *buf = nullptr, cudaStream_t st = nullptr) {
	if (!buf) buf = &h->dna;
	if (!st) st = h->st;
	const size_t off_pos = (total + 63) & ~(size_t) 63;
	const size_t bytes = off_pos + (size_t) n_reads * 12;
	CK(buf->ensure(std::max<size_t>(bytes, (size_t) h->P.reserve_bytes + (size_t) h->P.reserve_reads * 12 + 128) + 64));
	if (n_reads) CK(cudaMemcpyAsync(buf->p, stage, bytes, cudaMemcpyHostToDevice, st));
	U.dna = buf->as<uint8_t>();
	U.off = (const unsigned long long *) (buf->as<uint8_t>() + off_pos);
	U.len = (const uint32_t *) (buf->as<uint8_t>() + off_pos + (size_t) n_reads * 8);
	return FQSK_OK;
}

int fqsk_segment(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads,
                 fqsk_base_rec *recs, uint64_t rec_cap, uint64_t *n_recs, uint8_t *dup, uint64_t *rec_off) {
	if (!h || (!slab && n_reads) || (!reads && n_reads)) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->tk_open) return fail(h, FQSK_E_INVAL, "a submitted segment is in flight: fqsk_collect it first");
	h->tk_info = -1;
	uint64_t total = 0, bound = 0;
	CKR(stage_segment(h, h->h_stage, h->h_stage_cap, slab, slab_size, reads, n_reads, &total, &bound));
	Uploaded U;
	CKR(upload_segment(h, h->h_stage, total, n_reads, U));
	CKR(run_segment(h, U.dna, total, U.off, U.len, n_reads));
	CKR(seg_settle(h));
	if (h->n_recs > rec_cap) return fail(h, FQSK_E_CAPACITY, "record buffer holds %llu, segment produced %llu", (unsigned long long) rec_cap, (unsigned long long) h->n_recs);
	if (h->n_recs && recs) CK(cudaMemcpyAsync(recs, (h->rec_par ? h->recs_alt : h->recs).p, h->n_recs * sizeof(fqsk_base_rec), cudaMemcpyDeviceToHost, h->st));
	if (mode_pe(h->P.mode)) {
		// per-read views of the per-item arrays: mate 1 = item 3i, mate 2 = items 3i+1 (+ 3i+2, contiguous records)
		const uint32_t ni = n_reads / 2 * 3;
		std::vector<uint8_t> idup(ni + 1);
		std::vector<unsigned long long> ioff(ni + 1);
		if (ni) {
			CK(cudaMemcpyAsync(idup.data(), prep_bufs(h, h->seg_par).dup->p, ni, cudaMemcpyDeviceToHost, h->st));
			CK(cudaMemcpyAsync(ioff.data(), prep_bufs(h, h->seg_par).rec_off->p, ((size_t) ni + 1) * 8, cudaMemcpyDeviceToHost, h->st));
		}
		CK(cudaStreamSynchronize(h->st));
		for (uint32_t i = 0; i < n_reads / 2; ++i) {
			if (dup) { dup[2 * i] = idup[3 * i]; dup[2 * i + 1] = 0; }
			if (rec_off) { rec_off[2 * i] = ioff[3 * i]; rec_off[2 * i + 1] = ioff[3 * i + 1]; }
		}
		if (rec_off) rec_off[n_reads] = ni ? ioff[ni] : 0;
		if (n_recs) *n_recs = h->n_recs;
		return FQSK_OK;
	}
	if (n_reads && dup) CK(cudaMemcpyAsync(dup, prep_bufs(h, h->seg_par).dup->p, n_reads, cudaMemcpyDeviceToHost, h->st));
	if (n_reads && rec_off) CK(cudaMemcpyAsync(rec_off, prep_bufs(h, h->seg_par).rec_off->p, ((size_t) n_reads + 1) * 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (n_recs) *n_recs = h->n_recs;
	return FQSK_OK;
}

// The sync of a small segment, enqueued right behind the segment's first pass without a host look in between: every kernel is
// predicated on the device-side verdict of that pass and takes row lengths and stream positions from the device (SyncIn).
// One look then settles the segment AND the sync.  *applied = false: the caller runs the plain path (nothing was changed).
static int sync_spec_enqueue(fqsk_handle *h) {
	SegCtx &C = h->ctx;
	SyncIn *in = &h->status->syncin;
	const uint32_t bound_b = (uint32_t) (2 * C.dna_bytes_actual + 2), bound_s = (uint32_t) (C.dna_bytes_actual + 1);
	const uint64_t bound_p = 2 * C.dna_bytes_actual + 2ull * C.n;
	// The three table updates are independent (p-mer array, s-mer table, b-mer table; separate status words): the p-mer and
	// s-mer kernels run on two side streams next to the b-mer chain and join before the look.  With the phase brackets on
	// (profiling) everything stays on the engine's stream so that the brackets measure what they say.
	const bool fork = !h->serial;
	if (fork) CKR(ensure_side(h));
	cudaStream_t st_p = fork ? h->st_side[0] : h->st, st_s = fork ? h->st_side[1] : h->st;
	CK(h->q4.ensure(row_reserve(h, bound_s) + 4));
	if (fork) { CK(cudaEventRecord(h->ev_fork, h->st)); CK(cudaStreamWaitEvent(st_p, h->ev_fork, 0)); CK(cudaStreamWaitEvent(st_s, h->ev_fork, 0)); }
	{   // siv_fresh, sfast and the ordered-insert flags are still clear from k_seg_reset
		Phase ph(h, FQSK_PH_SYNC_SIV);
		CK(pdl(k_siv_increment, nblk(bound_p, 256), 256, st_p, h->siv, h->row_p.as<unsigned long long>(), 0, &h->status->siv_fresh, (const SyncIn *) in)); LAUNCHED(h);
	}
	{
		Phase ph(h, FQSK_PH_SYNC_APPLY);
		CK(pdl(k_insert_fast, nblk(bound_s, 256), 256, st_s, h->ts.d, h->ts.ci, h->row_s[0].as<unsigned long long>(), 0, h->q4.as<uint8_t>(), &h->status->sfast, (const SyncIn *) in)); LAUNCHED(h);
	}
	if (fork) { CK(cudaEventRecord(h->ev_side[0], st_p)); CK(cudaEventRecord(h->ev_side[1], st_s)); }
	SyncDev &Y = h->spec_Y;
	const unsigned long long *row_b = h->row_b[0].as<unsigned long long>();
	if (!h->spec_prefix) {
		CKR(indexed_setup(h, C.S.delta_b, bound_b, in, true, Y));
		h->spec_g = nblk(bound_b, 256);
		CKR(indexed_head(h, h->tb, Y, row_b, h->rt_b[0].as<uint32_t>(), h->spec_g, false));
	}
	const uint32_t g = h->spec_g;
	{
		Phase ph(h, FQSK_PH_SYNC_APPLY);
		CKR(stream_ensure(h, h->rng[ST_B], 0));
		if (!h->spec_prefix) CKR(indexed_scan(h, h->tb, Y, bound_b));
		CKR(indexed_apply(h, h->tb, h->rng[ST_B], Y, row_b, g, false));
	}
	if (fork) { CK(cudaStreamWaitEvent(h->st, h->ev_side[0], 0)); CK(cudaStreamWaitEvent(h->st, h->ev_side[1], 0)); }
	h->spec_enqueued = true;
	return FQSK_OK;
}
static int sync_spec_finish(fqsk_handle *h, bool *applied, unsigned long long items[4], unsigned long long *siv_fresh) {
	*applied = false;
	h->spec_enqueued = false;
	SyncDev &Y = h->spec_Y;
	const uint32_t g = h->spec_g;
	const unsigned long long *row_b = h->row_b[0].as<unsigned long long>();
	CKR(look(h));
	const EngineStatus &seen = h->look->st;
	const SyncIn li = seen.syncin;
	int fl[8]; memcpy(fl, seen.sflags, sizeof fl);
	const int s_refuted = seen.sfast;
	memcpy(items, seen.items, sizeof seen.items); *siv_fresh = seen.siv_fresh;
	CKR(seg_settle(h, true));      // the same look carries the segment's flags and totals
	if (!li.ok) {                  // the first pass was not the last one (or the rows are large): nothing was applied ...
		if (h->spec_prefix) { CK(pdl(k_sync_unclaim, g, 256, h->st, h->tb.d, Y, 1u)); LAUNCHED(h); }    // ... except slots claimed by the early grouping
		h->spec_prefix = false;
		return FQSK_OK;
	}
	h->spec_prefix = false;
	*applied = true;
	bool relook = false;
	if (fl[6]) h->hot_seen[1] = true;
	if (fl[7] || fl[0] || fl[2]) {
		// a counter saturated inside the batch, the draw window was short or a group is too large: nothing was committed; release
		// the claimed slots and take the plain ordered path for this row
		CK(pdl(k_sync_unclaim, g, 256, h->st, h->tb.d, Y, 0u)); LAUNCHED(h);
		CKR(apply_indexed(h, h->tb, h->rng[ST_B], h->seg_delta_b, row_b, h->rt_b[0].as<uint32_t>(), h->pend_b));
		relook = true;
	} else h->rng[ST_B].consumed += li.draws_b;
	if (s_refuted) {
		CK(pdl(k_insert_undo, nblk(h->pend_s, 256), 256, h->st, h->ts.d, h->row_s[0].as<unsigned long long>(), h->pend_s, h->q4.as<uint8_t>())); LAUNCHED(h);
		CKR(apply_inserts(h, h->ts, h->rng[ST_S], h->row_s[0].as<unsigned long long>(), h->pend_s));
		relook = true;
	}
	if (relook) {      // (siv_fresh is from the first look: the p-mers were applied once)
		CK(cudaMemcpyAsync(h->look->st.items, h->status->items, sizeof seen.items, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		memcpy(items, seen.items, sizeof seen.items);
	}
	return FQSK_OK;
}

// fqsk_sync in two halves: sync_begin enqueues what can be enqueued without looking at the device (the predicated sync of a small
// segment), sync_end looks, settles the segment and finishes the sync.  fqsk_submit calls the first half right behind the segment
// and the second half when the caller comes back for the records.
static int sync_begin(fqsk_handle *h) {
	if (h->pending && h->seg_reads && h->unsettled && !h->spec_enqueued && h->fast_ok[0] && h->ctx.dna_bytes_actual <= SPEC_MAX_BYTES) CKR(sync_spec_enqueue(h));
	return FQSK_OK;
}
static int sync_end(fqsk_handle *h) {
	++h->S.n_syncs;
	if (h->pending && h->seg_reads) {
		h->hot_seen[0] = h->hot_seen[1] = false;
		unsigned long long items[4] = {0, 0, 0, 0}, siv_fresh = 0;
		bool applied = false;
		if (h->spec_enqueued) CKR(sync_spec_finish(h, &applied, items, &siv_fresh));
		CKR(seg_settle(h));
		if (h->spec_prefix) {      // the segment was looked at before its sync was enqueued: release what the early grouping claimed
			CK(pdl(k_sync_unclaim, h->spec_g, 256, h->st, h->tb.d, h->spec_Y, 1u)); LAUNCHED(h);
			h->spec_prefix = false;
		}
		if (mode_pe(h->P.mode)) CKR(pe_sync(h));
		if (!applied) {
			// The three tables are independent (see sync_spec_enqueue): p-mer and s-mer updates run on side streams next to the ordered
			// b-mer insert, which is a chain of sort / locate / apply launches with host looks in between.  Joined before the last look.
			const bool fork = !h->serial && h->fast_ok[0] && h->pend_s;
			if (fork) CKR(ensure_side(h));
			cudaStream_t st_p = fork ? h->st_side[0] : h->st, st_s = fork ? h->st_side[1] : h->st;
			// p-mers (dna.cpp:2401-2418): order-independent saturating increments; the fresh-field count is read with the next look
			CK(cudaMemsetAsync(&h->status->siv_fresh, 0, 8, h->st));
			if (fork) { CK(cudaEventRecord(h->ev_fork, h->st)); CK(cudaStreamWaitEvent(st_p, h->ev_fork, 0)); CK(cudaStreamWaitEvent(st_s, h->ev_fork, 0)); }
			if (h->pend_p) {
				Phase ph(h, FQSK_PH_SYNC_SIV);
				CK(pdl(k_siv_increment, nblk(h->pend_p, 256), 256, st_p, h->siv, h->row_p.as<unsigned long long>(), h->pend_p, &h->status->siv_fresh, (const SyncIn *) nullptr));
				LAUNCHED(h);
			}
			// s-mers and b-mers (dna.cpp:2425-2446) live in different tables and use different PRNG streams, so their rows are
			// independent of each other.  The s-mers go through the self-checking atomic path (counters stay far below thr = 2047);
			// b-mers: small rows through the sort-free grouping over the segment's delta table, large rows through one radix sort.
			bool s_fast_pending = false;
			h->look_fresh = false;
			if (h->fast_ok[0] && h->pend_s) {
				Phase ph(h, FQSK_PH_SYNC_APPLY);
				CK(h->q4.ensure(row_reserve(h, h->pend_s) + 4));
				CK(cudaMemsetAsync(&h->status->sfast, 0, sizeof(int), st_s));
				CK(pdl(k_insert_fast, nblk(h->pend_s, 256), 256, st_s, h->ts.d, h->ts.ci, h->row_s[0].as<unsigned long long>(), h->pend_s, h->q4.as<uint8_t>(), &h->status->sfast, (const SyncIn *) nullptr)); LAUNCHED(h);
				s_fast_pending = true;
			}
			else if (h->pend_s <= SYNC_INDEXED_MAX && !h->delta_filtered) CKR(apply_indexed(h, h->ts, h->rng[ST_S], h->seg_delta_s, h->row_s[0].as<unsigned long long>(), h->rt_s[0].as<uint32_t>(), h->pend_s));
			else CKR(apply_inserts(h, h->ts, h->rng[ST_S], h->row_s[0].as<unsigned long long>(), h->pend_s));
			h->look_fresh = false;
			if (h->pend_b <= SYNC_INDEXED_MAX && !h->delta_filtered) CKR(apply_indexed(h, h->tb, h->rng[ST_B], h->seg_delta_b, h->row_b[0].as<unsigned long long>(), h->rt_b[0].as<uint32_t>(), h->pend_b));
			else CKR(apply_inserts(h, h->tb, h->rng[ST_B], h->row_b[0].as<unsigned long long>(), h->pend_b));
			if (fork) {   // join: the looks of the b-mer path did not cover the side streams
				CK(cudaEventRecord(h->ev_side[0], st_p)); CK(cudaEventRecord(h->ev_side[1], st_s));
				CK(cudaStreamWaitEvent(h->st, h->ev_side[0], 0)); CK(cudaStreamWaitEvent(h->st, h->ev_side[1], 0));
				h->look_fresh = false;
			}
			if (!h->look_fresh) CKR(look(h));
			const EngineStatus &seen = h->look->st;
			memcpy(items, seen.items, sizeof items); siv_fresh = seen.siv_fresh;
			if (s_fast_pending && seen.sfast) {
				// some s-mer counter left the deterministic range: undo (claimed slots stay as zero-count items == the reference's fresh
				// slot) and insert the row in order
				CK(pdl(k_insert_undo, nblk(h->pend_s, 256), 256, h->st, h->ts.d, h->row_s[0].as<unsigned long long>(), h->pend_s, h->q4.as<uint8_t>())); LAUNCHED(h);
				CKR(apply_inserts(h, h->ts, h->rng[ST_S], h->row_s[0].as<unsigned long long>(), h->pend_s));
				CK(cudaMemcpyAsync(h->look->st.items, h->status->items, sizeof items, cudaMemcpyDeviceToHost, h->st));
				CK(cudaStreamSynchronize(h->st));
				items[2] = seen.items[2]; items[3] = seen.items[3];
			}
		}
		if (!h->hot) {   // hot segments already advanced the thread-local streams
			if (h->hot_seen[0]) CKR(hot_account(h, 1));
			if (h->hot_seen[1]) CKR(hot_account(h, 0));
		}
		h->hot_seen[0] = h->hot_seen[1] = false;
		h->S.siv_no_filled += siv_fresh;
		h->S.siv_no_updates += h->pend_p + h->hidden_p;
		h->hidden_p = 0;
		h->items_main[0] = items[0]; h->items_main[1] = items[2];
		for (int k = 0; k < 2; ++k) {
			Table &t = k ? h->tb : h->ts;
			if (table_crowded(h, t, items[2 - 2 * k], items[3 - 2 * k])) CKR(table_grow_if_needed(h, t));
		}
	} else {
		CKR(seg_settle(h));
		h->S.siv_no_updates += h->hidden_p;
		h->hidden_p = 0;
	}
	for (int i = 0; i < 4; ++i) h->S.draws[i] = h->rng[i].consumed;
	CKR(stream_keep_ahead(h, h->rng[ST_B], 12u << 20)); CKR(stream_prefetch(h, h->rng[ST_S], 1u << 18));
	h->pending = false; h->pend_b = h->pend_s = h->pend_p = 0; h->seg_reads = 0;
	resolve_phases(h);
	return FQSK_OK;
}

int fqsk_sync(fqsk_handle *h) {
	if (!h) return FQSK_E_INVAL;
	ApiTimer api_timer{h};
	CK(cudaSetDevice(h->P.device));
	if (h->world > 1) return fail(h, FQSK_E_INVAL, "sharded engine: use fqsk_sync_route / fqsk_sync_apply / fqsk_sync_finish");
	if (h->tk_open) return fail(h, FQSK_E_INVAL, "a submitted segment is in flight: fqsk_collect it first (fqsk_submit includes the sync)");
	CKR(sync_begin(h));
	return sync_end(h);
}

// ---- asynchronous, double-buffered segment + sync ---------------------------------------------------------------------
static fqsk_base_rec *dev_recs(fqsk_handle *h, int par) { return (par ? h->recs_alt : h->recs).as<fqsk_base_rec>(); }

// k_ctx_codes over the records of the segment being evaluated (h->ctx) into the context-record buffer of parity `par`
static int enqueue_ctx_codes(fqsk_handle *h, int par) {
	const SegCtx &C = h->ctx;
	const uint32_t bound = (uint32_t) C.dna_bytes_actual;
	if (!C.n || !bound) return FQSK_OK;
	CK(h->ctxrec[par].ensure(((size_t) std::max<uint64_t>(bound, (uint64_t) h->P.reserve_bytes + h->P.reserve_bytes / 4) + 1) * sizeof(fqsk_ctx_rec)));
	CK(pdl(k_ctx_codes, nblk(bound, 256), 256, h->st, C.E, C.S, C.P, h->ctxrec[par].as<fqsk_ctx_rec>())); LAUNCHED(h);
	return FQSK_OK;
}

// compute side of the ticket in flight: the sync (its look also settles the segment); if the segment needed more than its
// first pass the records were rewritten after the copy was enqueued, so they are copied again (the copy stream is in order)
static int submit_finish_compute(fqsk_handle *h) {
	if (!h->tk_open) return FQSK_OK;
	auto &T = h->tk[h->tk_cur];
	if (!T.open || T.done) return FQSK_OK;
	CKR(sync_end(h));
	T.n_recs = h->n_recs;
	if (T.n_recs > T.bound) return fail(h, FQSK_E_CAPACITY, "segment produced %llu records, more than its reads allow (%llu)", (unsigned long long) T.n_recs, (unsigned long long) T.bound);
	if (h->seg_extra_pass && T.n_recs && (T.recs || T.ctx)) {
		if (T.ctx) CKR(enqueue_ctx_codes(h, T.par));      // the records were rewritten: build the context records again
		CK(cudaEventRecord(h->ev_recs, h->st)); CK(cudaStreamWaitEvent(h->st_copy, h->ev_recs, 0));
		if (T.ctx) CK(cudaMemcpyAsync(T.ctx, h->ctxrec[T.par].p, T.n_recs * sizeof(fqsk_ctx_rec), cudaMemcpyDeviceToHost, h->st_copy));
		else CK(cudaMemcpyAsync(T.recs, dev_recs(h, T.par), T.n_recs * sizeof(fqsk_base_rec), cudaMemcpyDeviceToHost, h->st_copy));
		CK(cudaEventRecord(h->ev_copied[T.par], h->st_copy));
	}
	T.done = true;
	return FQSK_OK;
}

static int submit_impl(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads,
                       fqsk_base_rec *recs, fqsk_ctx_rec *ctx, uint64_t rec_cap, uint8_t *dup, uint64_t *rec_off, uint64_t *ticket);
int fqsk_submit(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads,
                fqsk_base_rec *recs, uint64_t rec_cap, uint8_t *dup, uint64_t *rec_off, uint64_t *ticket) {
	return submit_impl(h, slab, slab_size, reads, n_reads, recs, nullptr, rec_cap, dup, rec_off, ticket);
}
int fqsk_submit_ctx(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads,
                    fqsk_ctx_rec *ctx, uint64_t rec_cap, uint8_t *dup, uint64_t *rec_off, uint64_t *ticket) {
	if (h && !ctx && n_reads) return FQSK_E_INVAL;
	if (h) for (uint32_t i = 0; reads && i < n_reads; ++i) if (reads[i].dna_len >= FQSK_CTX_MAX_READ) return fail(h, FQSK_E_UNSUPPORTED, "read %u has %u symbols: context records cover reads shorter than %u", i, reads[i].dna_len, FQSK_CTX_MAX_READ);
	return submit_impl(h, slab, slab_size, reads, n_reads, nullptr, ctx, rec_cap, dup, rec_off, ticket);
}
static int submit_impl(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads,
                       fqsk_base_rec *recs, fqsk_ctx_rec *ctx, uint64_t rec_cap, uint8_t *dup, uint64_t *rec_off, uint64_t *ticket) {
	if (!h || !ticket || (!slab && n_reads) || (!reads && n_reads)) return FQSK_E_INVAL;
	ApiTimer api_timer{h};
	CK(cudaSetDevice(h->P.device));
	if (h->world > 1) return fail(h, FQSK_E_UNSUPPORTED, "fqsk_submit: not available on a sharded engine");
	if (!h->st_copy) {
		CK(cudaStreamCreateWithFlags(&h->st_copy, cudaStreamNonBlocking));
		CK(cudaEventCreateWithFlags(&h->ev_recs, cudaEventDisableTiming));
		CK(cudaEventCreateWithFlags(&h->ev_meta, cudaEventDisableTiming));
		for (int i = 0; i < 2; ++i) CK(cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming));
	}
	const int par = h->tk_open ? h->tk_cur ^ 1 : h->rec_par ^ 1;
	if (h->tk[par].open) return fail(h, FQSK_E_INVAL, "two segments are already in flight: fqsk_collect the older one first");
	// host work first (the GPU is still busy with the previous segment): stage the reads in the pinned buffer of this parity
	uint64_t total = 0, bound = 0;
	uint8_t *&stage = par ? h->h_stage2 : h->h_stage;
	size_t &stage_cap = par ? h->h_stage2_cap : h->h_stage_cap;
	CKR(stage_segment(h, stage, stage_cap, slab, slab_size, reads, n_reads, &total, &bound));
	if (bound > rec_cap) return fail(h, FQSK_E_CAPACITY, "record buffer holds %llu, the segment can produce %llu", (unsigned long long) rec_cap, (unsigned long long) bound);
	// Still ahead of the look at the previous segment: the reads travel to the device on the front stream, into the input buffer of this
	// parity (the segment in flight reads the other one; the previous user of this one was settled two submits ago), and what depends on
	// the reads alone -- duplicate flags, letter totals, packed reads, record offsets -- is computed behind the copy, next to the segment in
	// flight (announce_impl: the same preparation fqsk_announce_device gives a device-resident caller).  Neither the copy nor k_prep /
	// k_scan_reads then sits between the look at segment n and the first kernel of segment n + 1.  Not across a block start (read_prev
	// was cleared), not with FQSK_F_SERIAL (one stream).
	Uploaded U;
	const bool ahead = !h->serial;
	if (ahead) {
		CKR(ensure_front(h));
		CKR(upload_segment(h, stage, total, n_reads, U, par ? &h->dna2 : &h->dna, h->st_front));
		CK(cudaEventRecord(h->ev_up, h->st_front));
		if (!h->block_fresh && n_reads) CKR(announce_impl(h, U.dna, total, (const uint64_t *) U.off, U.len, n_reads));
	}
	CKR(submit_finish_compute(h));                                  // previous segment: settle + sync
	CK(cudaStreamWaitEvent(h->st, h->ev_copied[par], 0));             // the device records of this parity have left for the host
	h->rec_par = par;
	if (h->meta_pending) { CK(cudaStreamWaitEvent(h->st, h->ev_meta, 0)); h->meta_pending = false; }      // the previous segment's per-read results have left the buffers this one rewrites
	if (ahead) CK(cudaStreamWaitEvent(h->st, h->ev_up, 0));
	else CKR(upload_segment(h, stage, total, n_reads, U, par ? &h->dna2 : &h->dna));
	CKR(run_segment(h, U.dna, total, U.off, U.len, n_reads));
	const uint32_t ni = mode_pe(h->P.mode) ? n_reads / 2 * 3 : n_reads;
	size_t o_off = 0, o_flag = 0, o_dif = 0, o_pair = 0;
	if (ni) {
		// layout: [dup: ni bytes, padded to 8][rec_off: (ni + 1) u64][sorted flag: ni u32, padded][sorted dif: ni u64][pair decisions: 3 u32 per pair]
		o_off = ((size_t) ni + 8) & ~(size_t) 7; o_flag = o_off + ((size_t) ni + 1) * 8; o_dif = o_flag + ((((size_t) ni + 1) * 4 + 7) & ~(size_t) 7); o_pair = o_dif + (size_t) ni * 8;
		const size_t need = o_pair + (size_t) (n_reads / 2 + 1) * 12;
		if (need > h->h_meta_cap[par]) {
			if (h->h_meta[par]) cudaFreeHost(h->h_meta[par]);
			h->h_meta[par] = nullptr; h->h_meta_cap[par] = 0;
			const size_t want = std::max<size_t>(need + need / 4, (size_t) h->P.reserve_reads * 14 + 64);
			CK(cudaMallocHost(&h->h_meta[par], want));
			h->h_meta_cap[par] = want;
		}
	}
	if (bound && ctx && n_reads) CKR(enqueue_ctx_codes(h, par));      // the context ids of the segment's records, on the device
	if (n_reads) {
		// Everything the host gets back leaves on the copy stream while the sync and the next segment run: first the per-read results --
		// duplicate flags and record offsets (final after k_prep / k_scan_reads), what compress_prefix_sorted / CompressPE code per read /
		// pair (functions of the reads and of the tables as they were when the segment started: the first pass is final) --, then the records.
		// (On the engine's stream the small copies sat between the segment and its sync: four stream-ordered copies on the critical path.)
		CK(cudaEventRecord(h->ev_recs, h->st)); CK(cudaStreamWaitEvent(h->st_copy, h->ev_recs, 0));
		if (ni) {
			CK(cudaMemcpyAsync(h->h_meta[par], prep_bufs(h, h->seg_par).dup->p, ni, cudaMemcpyDeviceToHost, h->st_copy));
			CK(cudaMemcpyAsync(h->h_meta[par] + o_off, prep_bufs(h, h->seg_par).rec_off->p, ((size_t) ni + 1) * 8, cudaMemcpyDeviceToHost, h->st_copy));
			if (mode_sorted(h->P.mode)) {
				CK(cudaMemcpyAsync(h->h_meta[par] + o_flag, h->sflag.p, (size_t) ni * 4, cudaMemcpyDeviceToHost, h->st_copy));
				CK(cudaMemcpyAsync(h->h_meta[par] + o_dif, h->sdif.p, (size_t) ni * 8, cudaMemcpyDeviceToHost, h->st_copy));
			}
			if (mode_pe(h->P.mode) && n_reads >= 2) CK(cudaMemcpyAsync(h->h_meta[par] + o_pair, h->pe_info.p, (size_t) (n_reads / 2) * 12, cudaMemcpyDeviceToHost, h->st_copy));
			CK(cudaEventRecord(h->ev_meta, h->st_copy)); h->meta_pending = true;
		}
		if (bound && (recs || ctx)) {
			if (ctx) CK(cudaMemcpyAsync(ctx, h->ctxrec[par].p, bound * sizeof(fqsk_ctx_rec), cudaMemcpyDeviceToHost, h->st_copy));
			else CK(cudaMemcpyAsync(recs, dev_recs(h, par), bound * sizeof(fqsk_base_rec), cudaMemcpyDeviceToHost, h->st_copy));
		}
		CK(cudaEventRecord(h->ev_copied[par], h->st_copy));
	}
	CKR(sync_begin(h));
	auto &T = h->tk[par];
	T = fqsk_handle::Ticket{};
	T.open = true; T.done = false; T.recs = recs; T.ctx = ctx; T.bound = bound; T.dup = dup; T.rec_off = rec_off; T.n_reads = n_reads; T.par = par; T.id = h->tk_next++;
	h->tk_open = true; h->tk_cur = par;
	*ticket = T.id;
	return FQSK_OK;
}

int fqsk_collect(fqsk_handle *h, uint64_t ticket, uint64_t *n_recs) {
	if (!h) return FQSK_E_INVAL;
	ApiTimer api_timer{h};
	CK(cudaSetDevice(h->P.device));
	int par = -1;
	for (int i = 0; i < 2; ++i) if (h->tk[i].open && h->tk[i].id == ticket) par = i;
	if (par < 0) return fail(h, FQSK_E_INVAL, "no such ticket in flight");
	auto &T = h->tk[par];
	if (!T.done) {
		if (par != h->tk_cur) return fail(h, FQSK_E_CUDA, "internal error: an older ticket was left unfinished");
		CKR(submit_finish_compute(h));
	}
	if (T.n_reads) CK(cudaEventSynchronize(h->ev_copied[par]));
	const uint32_t n = T.n_reads;
	if (n) {
		const bool pe = mode_pe(h->P.mode);
		const uint32_t ni = pe ? n / 2 * 3 : n;
		const uint8_t *idup = h->h_meta[par];
		const unsigned long long *ioff = (const unsigned long long *) (h->h_meta[par] + (((size_t) ni + 8) & ~(size_t) 7));      // layout: fqsk_submit
		if (pe) {
			for (uint32_t i = 0; i < n / 2; ++i) {
				if (T.dup) { T.dup[2 * i] = idup[3 * i]; T.dup[2 * i + 1] = 0; }
				if (T.rec_off) { T.rec_off[2 * i] = ioff[3 * i]; T.rec_off[2 * i + 1] = ioff[3 * i + 1]; }
			}
			if (T.rec_off) T.rec_off[n] = ioff[ni];
		} else {
			if (T.dup) memcpy(T.dup, idup, n);
			if (T.rec_off) memcpy(T.rec_off, ioff, ((size_t) n + 1) * 8);
		}
	}
	if (n_recs) *n_recs = T.n_recs;
	T.open = false;
	h->tk_open = h->tk[0].open || h->tk[1].open;
	h->tk_info = par;      // fqsk_sorted_prefix / fqsk_pair_info now describe this segment
	return FQSK_OK;
}

// The worker loop of one reads_block (application.cpp:617-662) over the asynchronous pair: fqsk_block_start, then segment k + 1 is
// submitted before segment k is collected -- the point where the host-side coder would consume the records of k.  Same calls a host makes
// one by one (host/fqsk_live.h does), in one C call per block.
int fqsk_block_host(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads, const uint32_t *seg_end, uint32_t n_segs,
                    fqsk_base_rec *recs, uint64_t rec_cap, uint8_t *dup, uint64_t *seg_rec_off, uint64_t *seg_n_recs) {
	if (!h || !seg_end || !n_segs || !seg_rec_off || !seg_n_recs || (n_reads && (!slab || !reads || !recs))) return FQSK_E_INVAL;
	if (seg_end[n_segs - 1] != n_reads) return fail(h, FQSK_E_INVAL, "fqsk_block_host: the last segment must end at the last read");
	uint64_t at = 0;
	for (uint32_t k = 0, a = 0; k < n_segs; a = seg_end[k], ++k) {
		if (seg_end[k] < a) return fail(h, FQSK_E_INVAL, "fqsk_block_host: segment ends must not decrease");
		seg_rec_off[k] = at;
		for (uint32_t r = a; r < seg_end[k]; ++r) at += reads[r].dna_len;      // upper bound of the coded positions
	}
	if (at > rec_cap) return fail(h, FQSK_E_CAPACITY, "record buffer holds %llu, the block can produce %llu", (unsigned long long) rec_cap, (unsigned long long) at);
	CKR(fqsk_block_start(h));
	uint64_t ticket[2] = {0, 0};
	auto first_of = [&](uint32_t k) { return k ? seg_end[k - 1] : 0u; };
	auto submit = [&](uint32_t k) {
		const uint32_t a = first_of(k), n = seg_end[k] - a;
		const uint64_t cap = (k + 1 < n_segs ? seg_rec_off[k + 1] : at) - seg_rec_off[k];
		return fqsk_submit(h, slab, slab_size, reads + a, n, recs + seg_rec_off[k], cap, dup ? dup + a : nullptr, nullptr, &ticket[k & 1]);
	};
	CKR(submit(0));
	for (uint32_t k = 0; k < n_segs; ++k) {
		if (k + 1 < n_segs) CKR(submit(k + 1));      // the engine runs ahead of the consumer
		CKR(fqsk_collect(h, ticket[k & 1], &seg_n_recs[k]));
	}
	return FQSK_OK;
}

// fqsk_block_host without the drain at the block end: the last segment of the block stays in flight and is collected by the NEXT call (or
// by fqsk_collect), so that its records travel to the host while the first segments of the next reads_block are evaluated -- the worker
// loop of application.cpp:617-662 running over consecutive blocks, the engine one segment ahead of the consumer throughout.
int fqsk_block_stream(fqsk_handle *h, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads, const uint32_t *seg_end, uint32_t n_segs,
                      fqsk_base_rec *recs, fqsk_ctx_rec *ctx, uint64_t rec_cap, uint8_t *dup, uint64_t *seg_rec_off, uint64_t *seg_n_recs,
                      uint64_t *carry_ticket, uint64_t *carry_n_recs) {
	if (!h || !seg_end || !n_segs || !seg_rec_off || !seg_n_recs || !carry_ticket || (n_reads && (!slab || !reads || (!recs == !ctx)))) return FQSK_E_INVAL;
	if (seg_end[n_segs - 1] != n_reads) return fail(h, FQSK_E_INVAL, "fqsk_block_stream: the last segment must end at the last read");
	uint64_t at = 0;
	for (uint32_t k = 0, a = 0; k < n_segs; a = seg_end[k], ++k) {
		if (seg_end[k] < a) return fail(h, FQSK_E_INVAL, "fqsk_block_stream: segment ends must not decrease");
		seg_rec_off[k] = at;
		for (uint32_t r = a; r < seg_end[k]; ++r) at += reads[r].dna_len;      // upper bound of the coded positions
	}
	if (at > rec_cap) return fail(h, FQSK_E_CAPACITY, "record buffer holds %llu, the block can produce %llu", (unsigned long long) rec_cap, (unsigned long long) at);
	CKR(fqsk_block_start(h));
	uint64_t pend = *carry_ticket, pend_k = ~0ull;      // pend_k: segment of THIS block the open ticket belongs to (~0: the carried one)
	for (uint32_t k = 0, a = 0; k < n_segs; a = seg_end[k], ++k) {
		const uint32_t n = seg_end[k] - a;
		const uint64_t cap = (k + 1 < n_segs ? seg_rec_off[k + 1] : at) - seg_rec_off[k];
		uint64_t t = 0;
		if (ctx) CKR(fqsk_submit_ctx(h, slab, slab_size, reads + a, n, ctx + seg_rec_off[k], cap, dup ? dup + a : nullptr, nullptr, &t));
		else CKR(fqsk_submit(h, slab, slab_size, reads + a, n, recs + seg_rec_off[k], cap, dup ? dup + a : nullptr, nullptr, &t));
		if (pend) {
			uint64_t nr = 0;
			CKR(fqsk_collect(h, pend, &nr));
			if (pend_k == ~0ull) { if (carry_n_recs) *carry_n_recs = nr; } else seg_n_recs[pend_k] = nr;
		}
		pend = t; pend_k = k;
	}
	*carry_ticket = pend;
	return FQSK_OK;
}

// ---- sorted-mode front end (SURVEY.md section 8 row f3) ------------------------------------------------------------------------
// rank[i] of read i: an integer order-isomorphic to the comparator of CSortedFASTQFile::sort_reads (io.h:499-528); see fqsk_front.cuh.
// Needs no engine: its own stream and scratch on `device`, released before it returns (one call per bin file of a sorted-order job).
int fqsk_sort_ranks(int device, const uint8_t *slab, uint64_t slab_size, const fqsk_read_desc *reads, uint32_t n_reads, uint32_t *rank) {
	if ((!slab || !reads || !rank) && n_reads) return FQSK_E_INVAL;
	if (!n_reads) return FQSK_OK;
	for (uint32_t i = 0; i < n_reads; ++i) if (reads[i].dna_off > slab_size || reads[i].dna_len > slab_size - reads[i].dna_off) return FQSK_E_INVAL;
	int n_dev = 0;
	if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) { cudaGetLastError(); g_create_error = "fqsk_sort_ranks: no CUDA device"; return FQSK_E_NO_DEVICE; }
	if (device < 0 || device >= n_dev) return FQSK_E_INVAL;
	struct Scratch {
		std::vector<void *> ptrs; cudaStream_t st = nullptr;
		~Scratch() { for (void *p : ptrs) cudaFree(p); if (st) cudaStreamDestroy(st); }
		int get(void **p, size_t bytes) { void *q = nullptr; if (cudaMalloc(&q, std::max<size_t>(bytes, 16)) != cudaSuccess) { cudaGetLastError(); return FQSK_E_NOMEM; } ptrs.push_back(q); *p = q; return FQSK_OK; }
	} X;
#define FCK(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { g_create_error = std::string("fqsk_sort_ranks: ") + cudaGetErrorString(e_); cudaGetLastError(); return FQSK_E_CUDA; } } while (0)
	FCK(cudaSetDevice(device));
	FCK(cudaStreamCreateWithFlags(&X.st, cudaStreamNonBlocking));
	const uint32_t n = n_reads, tiles = nblk(n, RDX_TILE);
	uint8_t *d_slab = nullptr; fqsk_read_desc *d_reads = nullptr;
	unsigned long long *k0 = nullptr, *k1 = nullptr; uint32_t *v0 = nullptr, *v1 = nullptr, *gs = nullptr, *ge = nullptr, *d_rank = nullptr, *hist = nullptr, *d_max = nullptr;
	CKR(X.get((void **) &d_slab, slab_size)); CKR(X.get((void **) &d_reads, (size_t) n * sizeof(fqsk_read_desc)));
	CKR(X.get((void **) &k0, (size_t) n * 8)); CKR(X.get((void **) &k1, (size_t) n * 8)); CKR(X.get((void **) &v0, (size_t) n * 4)); CKR(X.get((void **) &v1, (size_t) n * 4));
	CKR(X.get((void **) &gs, (size_t) n * 4)); CKR(X.get((void **) &ge, (size_t) n * 4)); CKR(X.get((void **) &d_rank, (size_t) n * 4));
	CKR(X.get((void **) &hist, (((size_t) tiles + 1) << 8) * 4)); CKR(X.get((void **) &d_max, 4));
	FCK(cudaMemcpyAsync(d_slab, slab, slab_size, cudaMemcpyHostToDevice, X.st));
	FCK(cudaMemcpyAsync(d_reads, reads, (size_t) n * sizeof(fqsk_read_desc), cudaMemcpyHostToDevice, X.st));
	FCK(cudaMemsetAsync(d_max, 0, 4, X.st));
	FCK(pdl(k_front_key, nblk(n, 256), 256, X.st, (const uint8_t *) d_slab, (const fqsk_read_desc *) d_reads, n, k0));
	// stable LSD radix sort of (key, read) by all 64 bits, 8 bits a pass (the engine's own partition kernels, fqsk_sort.cuh)
	const unsigned long long *ks = k0; const uint32_t *vs = nullptr;
	for (int p = 0; p < 8; ++p) {
		unsigned long long *kd = (p & 1) ? k0 : k1; uint32_t *vd = (p & 1) ? v0 : v1;
		uint32_t *totals = hist + ((size_t) tiles << 8);
		const BitsOp op{(uint32_t) (8 * p), 0xFFu};
		FCK(pdl(k_rdx_hist<8, BitsOp>, tiles, RDX_THREADS, X.st, ks, n, tiles, hist, op));
		FCK(pdl(k_rdx_rowscan, 256u, 256, X.st, hist, tiles, totals));
		FCK(pdl(k_rdx_scatter<8, BitsOp>, tiles, RDX_THREADS, X.st, ks, vs, kd, vd, n, tiles, (const uint32_t *) hist, (const uint32_t *) totals, op));
		ks = kd; vs = vd;
	}
	// 8 passes: the result is in (k0, v0)
	FCK(pdl(k_front_group, nblk(n, 256), 256, X.st, (const unsigned long long *) k0, n, gs, ge, d_max));
	uint32_t max_run = 0;
	FCK(cudaMemcpyAsync(&max_run, d_max, 4, cudaMemcpyDeviceToHost, X.st));
	FCK(cudaStreamSynchronize(X.st));
	if (max_run > (1u << 16)) {      // the members of a run are ranked by comparing each with all others: bounded, never approximated
		g_create_error = "fqsk_sort_ranks: more than 65536 reads share their first 32 symbols; not supported";
		return FQSK_E_UNSUPPORTED;
	}
	FCK(pdl(k_front_rank, nblk(n, 128), 128, X.st, (const uint8_t *) d_slab, (const fqsk_read_desc *) d_reads, (const uint32_t *) v0, (const uint32_t *) gs, (const uint32_t *) ge, n, d_rank));
	FCK(cudaMemcpyAsync(rank, d_rank, (size_t) n * 4, cudaMemcpyDeviceToHost, X.st));
	FCK(cudaStreamSynchronize(X.st));
#undef FCK
	return FQSK_OK;
}

// ---- sharded operation --------------------------------------------------------------------------------------------
int fqsk_shard_export(fqsk_handle *h, fqsk_shard_desc *out) {
	if (!h || !out) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->world <= 1) return fail(h, FQSK_E_INVAL, "not a sharded engine");
	if (h->grow_pending) {      // after FQSK_RESHARD and the caller's barrier: every peer has closed its mappings of the tables that double now
		if (h->pending || h->tk_open) return fail(h, FQSK_E_INVAL, "fqsk_shard_export after FQSK_RESHARD: before the next segment");
		if (h->grow_all & 1u) CKR(table_double(h, h->ts));
		if (h->grow_all & 2u) CKR(table_double(h, h->tb));
		if (h->grow_all & 4u) CKR(pair_resize(h, (h->pair.mask + 1) * 2));
		h->grow_pending = false; h->grow_all = 0; h->grow_local = 0;
	}
	memset(out, 0, sizeof *out);
	out->rank = h->rank; out->world_size = h->world;
	out->geometry[0] = h->tb.d.B; out->geometry[1] = h->tb.d.stash_log2; out->geometry[2] = h->ts.d.B; out->geometry[3] = h->ts.d.stash_log2;
	out->geometry[4] = h->siv.key_bits;
	uint32_t pl2 = 0;
	if (h->pair.keys) while ((1ull << pl2) < h->pair.mask + 1) ++pl2;
	out->geometry[5] = pl2;
	out->inbox_cap = h->inbox_cap;
	void *ptrs[8] = {h->tb.d.main, h->tb.d.stash, h->ts.d.main, h->ts.d.stash, h->siv.w, h->inbox, h->pair.keys, h->pair.vcs};
	static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
	for (int q = 0; q < (h->pair.keys ? 8 : 6); ++q) CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t *) out->ipc[q], ptrs[q]));
	CK(cudaStreamSynchronize(h->st));      // the shards are zero-filled before anybody maps them
	return FQSK_OK;
}

int fqsk_shard_attach(fqsk_handle *h, const fqsk_shard_desc *peer) {
	if (!h || !peer) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->world <= 1 || peer->world_size != h->world || peer->rank >= h->world) return fail(h, FQSK_E_INVAL, "descriptor of rank %u / %u does not belong to this group", peer->rank, peer->world_size);
	if (peer->rank == h->rank) return FQSK_OK;
	if (peer->geometry[0] != h->tb.d.B || peer->geometry[1] != h->tb.d.stash_log2 || peer->geometry[2] != h->ts.d.B || peer->geometry[3] != h->ts.d.stash_log2 ||
	    peer->geometry[4] != h->siv.key_bits || peer->inbox_cap != h->inbox_cap || (h->pair.keys && (1ull << peer->geometry[5]) != h->pair.mask + 1))
		return fail(h, FQSK_E_INVAL, "rank %u was created with a different table geometry", peer->rank);
	const uint32_t r = peer->rank;
	for (int q = 0; q < (h->pair.keys ? 8 : 6); ++q) {
		if (h->peer_ptrs[r][q]) continue;
		cudaIpcMemHandle_t hd; memcpy(&hd, peer->ipc[q], 64);
		CK(cudaIpcOpenMemHandle(&h->peer_ptrs[r][q], hd, cudaIpcMemLazyEnablePeerAccess));
	}
	h->tb.d.peer_main[r] = (const uint32_t *) h->peer_ptrs[r][0]; h->tb.d.peer_stash[r] = (const unsigned long long *) h->peer_ptrs[r][1];
	h->ts.d.peer_main[r] = (const uint32_t *) h->peer_ptrs[r][2]; h->ts.d.peer_stash[r] = (const unsigned long long *) h->peer_ptrs[r][3];
	h->siv.peer_w[r] = (const uint32_t *) h->peer_ptrs[r][4];
	h->peer_inbox[r] = (unsigned long long *) h->peer_ptrs[r][5];
	if (h->pair.keys) { h->pair.peer_keys[r] = (const unsigned long long *) h->peer_ptrs[r][6]; h->pair.peer_vcs[r] = (const unsigned long long *) h->peer_ptrs[r][7]; }
	h->attached |= 1u << r;
	return FQSK_OK;
}

// fqsk_shard_attach for two handles of ONE process (a host with one worker thread per GPU -- host/fqsk_live.h at -t N): CUDA IPC handles
// cannot be opened by the process that exported them, and need not be -- with peer access enabled the peer's allocations are directly
// addressable (unified virtual addressing).  Same effect and same preconditions as fqsk_shard_attach; after FQSK_RESHARD it is called
// again once BOTH handles have passed their fqsk_shard_export.
int fqsk_shard_attach_local(fqsk_handle *h, fqsk_handle *peer) {
	if (!h || !peer) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->world <= 1 || peer->world != h->world || peer->rank >= h->world) return fail(h, FQSK_E_INVAL, "fqsk_shard_attach_local: the two handles do not belong to one group");
	if (peer == h || peer->rank == h->rank) return peer == h ? FQSK_OK : fail(h, FQSK_E_INVAL, "fqsk_shard_attach_local: two handles with rank %u", h->rank);
	if (peer->grow_pending || h->grow_pending) return fail(h, FQSK_E_INVAL, "fqsk_shard_attach_local: fqsk_shard_export (the doubling) comes first on both handles");
	if (peer->tb.d.B != h->tb.d.B || peer->tb.d.stash_log2 != h->tb.d.stash_log2 || peer->ts.d.B != h->ts.d.B || peer->ts.d.stash_log2 != h->ts.d.stash_log2 ||
	    peer->siv.key_bits != h->siv.key_bits || peer->inbox_cap != h->inbox_cap || !peer->pair.keys != !h->pair.keys || (h->pair.keys && peer->pair.mask != h->pair.mask))
		return fail(h, FQSK_E_INVAL, "rank %u was created with a different table geometry", peer->rank);
	if (peer->P.device != h->P.device) {
		int can = 0;
		CK(cudaDeviceCanAccessPeer(&can, h->P.device, peer->P.device));
		if (!can) return fail(h, FQSK_E_UNSUPPORTED, "device %d cannot access device %d (no NVLink / PCIe peer path)", h->P.device, peer->P.device);
		cudaError_t e = cudaDeviceEnablePeerAccess(peer->P.device, 0);
		if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError(); else CK(e);
	}
	const uint32_t r = peer->rank;
	h->tb.d.peer_main[r] = peer->tb.d.main; h->tb.d.peer_stash[r] = peer->tb.d.stash;
	h->ts.d.peer_main[r] = peer->ts.d.main; h->ts.d.peer_stash[r] = peer->ts.d.stash;
	h->siv.peer_w[r] = peer->siv.w;
	h->peer_inbox[r] = peer->inbox;
	if (h->pair.keys) { h->pair.peer_keys[r] = peer->pair.keys; h->pair.peer_vcs[r] = peer->pair.vcs; }
	h->attached |= 1u << r;
	return FQSK_OK;
}

int fqsk_sync_route(fqsk_handle *h) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->world <= 1) return fail(h, FQSK_E_INVAL, "not a sharded engine");
	CKR(seg_settle(h));
	++h->S.n_syncs;
	InboxDev I{};
	for (uint32_t i = 0; i < h->world; ++i) I.base[i] = h->peer_inbox[i];
	I.cap = h->inbox_cap; I.world = h->world; I.rank = h->rank;
	const bool have = h->pending && h->seg_reads;
	const unsigned long long *rows[3] = {h->row_p.as<unsigned long long>(), h->row_s[0].as<unsigned long long>(), h->row_b[0].as<unsigned long long>()};
	const uint32_t ns[3] = {have ? h->pend_p : 0, have ? h->pend_s : 0, have ? h->pend_b : 0};
	CK(h->route_hist.ensure(4 * 8 * 4));
	CK(cudaMemsetAsync(h->route_hist.p, 0, 4 * 8 * 4, h->st));
	CK(cudaMemsetAsync(h->status->flags, 0, 8 * sizeof(int), h->st));
	{   // p / s / b rows: owner histogram per chunk, then every k-mer straight to its place in its owner's inbox (fqsk_kernels.cuh)
		RouteRows R{};
		uint32_t n_max = 0;
		for (int t = 0; t < 3; ++t) { R.row[t] = rows[t]; R.n[t] = ns[t]; n_max = std::max(n_max, ns[t]); }
		R.pshift = 2 * h->P.pmer_len - 12;
		const uint32_t chunks = std::max<uint32_t>(nblk(n_max, ROUTE_CHUNK), 1);
		const uint32_t chunks_max = std::max<uint32_t>(chunks, nblk((uint32_t) row_reserve(h, n_max), ROUTE_CHUNK));
		CK(h->route_chunks.ensure((size_t) 3 * chunks_max * 8 * 4));
		if (n_max) { CK(pdl(k_route_count, dim3(chunks, 3), 256, h->st, R, h->world, chunks_max, h->route_chunks.as<uint32_t>())); LAUNCHED(h); }
		CK(pdl(k_route_move, dim3(chunks, 3), 256, h->st, R, chunks_max, (const uint32_t *) h->route_chunks.as<uint32_t>(), I, h->status->flags)); LAUNCHED(h);
	}
	if (h->pair.keys) {
		// paired end: the distinct (key, value) pairs of the segment with summed weights, routed by (fmix64(key) >> 48) % world as three
		// planes (key / value / weight = inbox tables 3 / 4 / 5) sorted with the same owner keys (stable: the planes stay aligned)
		uint32_t nu = 0;
		uint32_t *hist = h->route_hist.as<uint32_t>() + 8 * 3;
		const uint32_t nt = have ? h->pe_nt : 0;
		if (nt) {
			CK(h->pe_uk.ensure((size_t) nt * 8)); CK(h->pe_uv.ensure((size_t) nt * 8)); CK(h->pe_uc.ensure((size_t) nt * 8));
			uint32_t *d_nu = &h->status->pe_pool.used;
			CK(cudaMemsetAsync(d_nu, 0, 4, h->st));
			CK(pdl(k_pair_heads, nblk(nt, 256), 256, h->st, pe_seg(h), h->pair.vm, h->pe_uk.as<unsigned long long>(), h->pe_uv.as<unsigned long long>(), h->pe_uc.as<unsigned long long>(), d_nu)); LAUNCHED(h);
			CK(cudaMemcpyAsync(&h->look->st.pe_pool.used, d_nu, 4, cudaMemcpyDeviceToHost, h->st));
			CK(cudaStreamSynchronize(h->st));
			nu = h->look->st.pe_pool.used;
		}
		if (nu) {
			CK(h->route_keys.ensure(nu)); CK(h->route_keys2.ensure(nu)); CK(h->route_sorted.ensure((size_t) nu * 8));
			CK(pdl(k_pair_owner_keys, nblk(nu, 256), 256, h->st, (const unsigned long long *) h->pe_uk.as<unsigned long long>(), nu, h->world, h->route_keys.as<uint8_t>(), hist)); LAUNCHED(h);
		}
		const unsigned long long *planes[3] = {h->pe_uk.as<unsigned long long>(), h->pe_uv.as<unsigned long long>(), h->pe_uc.as<unsigned long long>()};
		if (nu) {      // the permutation that groups the key plane by owner (stable), then every plane is gathered through it
			CKR(rdx_scratch(h, nu, true));
			CK(h->route_perm.ensure((size_t) nu * 4));
			CKR((rdx_pass<3, OwnerOp>(h, h->st, planes[0], nullptr, h->rdx_k.as<unsigned long long>(), h->route_perm.as<uint32_t>(), nu, OwnerOp{2u, 0u, h->world})));
		}
		for (int q = 0; q < 3; ++q) {
			if (nu) { CK(pdl(k_pe_gather, nblk(nu, 256), 256, h->st, planes[q], (const uint32_t *) h->route_perm.as<uint32_t>(), h->route_sorted.as<unsigned long long>(), nu)); LAUNCHED(h); }
			CK(pdl(k_route_scatter, nblk(std::max<uint32_t>(nu, 8), 256), 256, h->st, (const unsigned long long *) h->route_sorted.as<unsigned long long>(), nu, (const uint32_t *) hist, I, (uint32_t) (3 + q), h->status->flags)); LAUNCHED(h);
		}
		h->pe_nt = 0;
	}
	// rows [rank][*] are on their way: post this sync's number at every owner (no host look: a row too long for its slot -- flags[4] -- is
	// reported by the first look of fqsk_sync_apply, and the owner sees the oversized length itself)
	CK(pdl(k_post_seq, 1, 32, h->st, I, ++h->sync_seq)); LAUNCHED(h);
	h->routed = true;
	return FQSK_OK;
}

int fqsk_sync_apply(fqsk_handle *h, uint64_t *fresh, uint64_t *updates) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->world <= 1 || !h->routed) return fail(h, FQSK_E_INVAL, "fqsk_sync_apply needs fqsk_sync_route on a sharded engine first");
	// The thread-local PRNG streams of THIS worker advance with its own pushes above thr, whoever owns them (ht_kmer.h:433-436 via
	// dna.cpp:826, 837, 862, 872): the ranks of the segment's pushes are counted now (no host look), the event counts come back with
	// the look below, and only a segment that has such pushes (low-complexity reads) pays for the ordered evaluation.
	const bool account = h->pending && h->seg_reads && !h->hot;
	if (account) { CK(cudaMemsetAsync(&h->status->hot, 0, sizeof h->status->hot, h->st)); CKR(hot_rank(h, 1)); CKR(hot_rank(h, 0)); }
	// every source has posted this sync's number once its rows were in our inbox (k_post_seq): wait for them on the device, then read
	// the posted slot lengths, the route's flags and the event counts with ONE look
	int *d_err = &h->status->wait_err;      // cleared at create; set means the group is lost anyway
	CK(pdl(k_wait_seq, 1, 32, h->st, (const unsigned long long *) h->inbox, h->world, h->sync_seq, d_err)); LAUNCHED(h);
	unsigned long long cnt[48];
	EngineStatus &seen = h->look->st;
	CK(cudaMemcpyAsync(cnt, h->inbox, sizeof cnt, cudaMemcpyDeviceToHost, h->st));
	CK(cudaMemcpyAsync(&seen, h->status, sizeof seen, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	if (seen.wait_err) return fail(h, FQSK_E_CUDA, "sharded sync: a peer did not post its rows within the time limit");
	if (seen.flags[4]) return fail(h, FQSK_E_CAPACITY, "an exchange row is longer than the inbox slot (%llu k-mers): create the engines with a larger reserve_bytes", (unsigned long long) h->inbox_cap);
	const uint32_t hot_en[2] = {seen.hot.ev[0], seen.hot.ev[1]};      // [0] b-stream events, [1] s-stream events
	uint64_t tot[3] = {0, 0, 0};
	for (int t = 0; t < 6; ++t) for (uint32_t i = 0; i < h->world; ++i)
		if (cnt[t * 8 + i] > h->inbox_cap) return fail(h, FQSK_E_CAPACITY, "rank %u posted an exchange row longer than the inbox slot: create the engines with a larger reserve_bytes", i);
	for (int t = 0; t < 3; ++t) for (uint32_t i = 0; i < h->world; ++i) tot[t] += cnt[t * 8 + i];
	for (int t = 0; t < 3; ++t) if (tot[t] >= 0x80000000ull) return fail(h, FQSK_E_INVAL, "more than 2^31 k-mers in one sync row");
	// rows [*][rank] in source order: one contiguous row per table
	CK(h->row_p.ensure((tot[0] + 1) * 8)); CK(h->row_s[0].ensure((tot[1] + 1) * 8)); CK(h->row_b[0].ensure((tot[2] + 1) * 8));
	unsigned long long *dst[3] = {h->row_p.as<unsigned long long>(), h->row_s[0].as<unsigned long long>(), h->row_b[0].as<unsigned long long>()};
	// (the segment's own rows lived in these buffers; fqsk_sync_route has copied them out)
	for (int t = 0; t < 3; ++t) {
		uint64_t at = 0;
		for (uint32_t i = 0; i < h->world; ++i) {
			const uint64_t c = cnt[t * 8 + i];
			if (c) CK(cudaMemcpyAsync(dst[t] + at, inbox_slot(h->inbox, h->inbox_cap, h->world, (uint32_t) t, i), c * 8, cudaMemcpyDeviceToDevice, h->st));
			at += c;
		}
	}
	if (account) { if (hot_en[1]) CKR(hot_account(h, 1)); if (hot_en[0]) CKR(hot_account(h, 0)); }      // rare: redoes the ranks, then evaluates in order
	h->hot_seen[0] = h->hot_seen[1] = false;
	CK(cudaMemsetAsync(&h->status->siv_fresh, 0, 8, h->st));
	if (tot[0]) {
		Phase ph(h, FQSK_PH_SYNC_SIV);
		CK(pdl(k_siv_increment, nblk(tot[0], 256), 256, h->st, h->siv, dst[0], tot[0], &h->status->siv_fresh, (const SyncIn *) nullptr)); LAUNCHED(h);
	}
	if (tot[1]) { bool fast = true; CKR(apply_inserts(h, h->ts, h->rng[ST_S], dst[1], (uint32_t) tot[1], &fast)); }
	if (tot[2]) CKR(apply_row(h, h->tb, h->rng[ST_B], dst[2], (uint32_t) tot[2]));
	if (h->pair.keys) {   // pair rows [*][rank], one source after the other (each holds distinct pairs; the insertion is commutative)
		uint64_t incoming = 0;
		for (uint32_t i = 0; i < h->world; ++i) incoming += cnt[3 * 8 + i];
		CKR(pair_reserve(h, incoming));
		unsigned long long *d_items = &h->status->pair_items;
		for (uint32_t i = 0; i < h->world; ++i) {
			const uint32_t c = (uint32_t) cnt[3 * 8 + i];
			if (!c) continue;
			CK(pdl(k_pair_insert_list, nblk(c, 256), 256, h->st, h->pair, (const unsigned long long *) inbox_slot(h->inbox, h->inbox_cap, h->world, 3, i),
			       (const unsigned long long *) inbox_slot(h->inbox, h->inbox_cap, h->world, 4, i), (const unsigned long long *) inbox_slot(h->inbox, h->inbox_cap, h->world, 5, i), c, d_items)); LAUNCHED(h);
		}
		CK(cudaMemcpyAsync(&h->look->st.pair_items, d_items, 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		h->pair_items = h->look->st.pair_items;
	}
	unsigned long long acc[2] = {0, 0}, grow_word = 0;
	h->sync_updates = tot[0] + h->hidden_p;
	if (h->dev_finish) {
		// this rank's inserts are enqueued: add its statistics to everybody's accumulators and post the sync's number (k_post_applied), then
		// wait -- on the device -- until every rank has done the same: no lookup of the next segment can see a half-applied sync
		InboxDev I{};
		for (uint32_t i = 0; i < h->world; ++i) I.base[i] = h->peer_inbox[i];
		I.cap = h->inbox_cap; I.world = h->world; I.rank = h->rank;
		GrowLim lim;
		for (int k = 0; k < 2; ++k) {      // [0, 1] b-mer table, [2, 3] s-mer table: the thresholds of table_crowded
			const Table &t = k ? h->ts : h->tb;
			lim.v[2 * k] = table_can_double(t) ? crowd_main(h, t) : ~0ull; lim.v[2 * k + 1] = table_can_double(t) ? crowd_stash(t) : ~0ull;
		}
		lim.v[4] = h->pair.keys ? (h->pair.mask + 1) / 2 : ~0ull;
		CK(pdl(k_post_applied, 1, 32, h->st, I, h->sync_seq, (const unsigned long long *) &h->status->siv_fresh, (unsigned long long) h->sync_updates,
		       (const unsigned long long *) h->status->items, (const unsigned long long *) (h->pair.keys ? &h->status->pair_items : nullptr), lim)); LAUNCHED(h);
		CK(pdl(k_wait_applied, 1, 32, h->st, (const unsigned long long *) h->inbox, h->world, h->sync_seq, d_err)); LAUNCHED(h);
		CK(cudaMemcpyAsync(acc, h->inbox + INBOX_ACC + 2 * (h->sync_seq & 1), 16, cudaMemcpyDeviceToHost, h->st));
		CK(cudaMemcpyAsync(&grow_word, h->inbox + INBOX_GROW + (h->sync_seq & 1), 8, cudaMemcpyDeviceToHost, h->st));
	}
	CK(cudaMemcpyAsync(&seen, h->status, sizeof seen, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	resolve_phases(h);
	if (h->dev_finish && seen.wait_err) return fail(h, FQSK_E_CUDA, "sharded sync: a peer did not finish its inserts within the time limit");
	// shards double together: what this rank's shards ask for (three-step form: fqsk_shard_grow_request), resp. what all ranks asked for
	// through the accumulators (device form)
	h->grow_local = 0;
	if (table_crowded(h, h->ts, seen.items[2], seen.items[3]) && table_can_double(h->ts)) h->grow_local |= 1u;
	if (table_crowded(h, h->tb, seen.items[0], seen.items[1]) && table_can_double(h->tb)) h->grow_local |= 2u;
	if (h->pair.keys && h->pair_items > (h->pair.mask + 1) / 2) h->grow_local |= 4u;
	h->grow_all = 0;
	if (h->dev_finish) h->grow_all = ((grow_word & 0xFFFFull) ? 1u : 0u) | (((grow_word >> 16) & 0xFFFFull) ? 2u : 0u) | (((grow_word >> 32) & 0xFFFFull) ? 4u : 0u);
	h->sync_fresh = seen.siv_fresh;
	h->siv_local_filled += seen.siv_fresh;
	h->hidden_p = 0;
	if (fresh) *fresh = h->dev_finish ? acc[0] : h->sync_fresh;
	if (updates) *updates = h->dev_finish ? acc[1] : h->sync_updates;
	h->applied = true;
	return FQSK_OK;
}

// The whole sharded sync in one call and without a collective library: fqsk_sync_route, fqsk_sync_apply with the device-side second
// barrier (k_post_applied / k_wait_applied: the global p-mer statistics travel as NVLink atomics), fqsk_sync_finish.
int fqsk_sync_device(fqsk_handle *h) {
	if (!h) return FQSK_E_INVAL;
	CKR(fqsk_sync_route(h));
	h->dev_finish = true;
	uint64_t fresh_all = 0, updates_all = 0;
	const int rc = fqsk_sync_apply(h, &fresh_all, &updates_all);
	h->dev_finish = false;
	if (rc != FQSK_OK) return rc;
	return fqsk_sync_finish(h, fresh_all, updates_all);
}

int fqsk_sync_finish(fqsk_handle *h, uint64_t fresh_all, uint64_t updates_all) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->world <= 1 || !h->applied) return fail(h, FQSK_E_INVAL, "fqsk_sync_finish needs fqsk_sync_apply on a sharded engine first");
	h->S.siv_no_filled += fresh_all;       // bit_vec.h:212-220: global atomics in the reference, read by every worker (dna.cpp:376)
	h->S.siv_no_updates += updates_all;
	for (int i = 0; i < 4; ++i) h->S.draws[i] = h->rng[i].consumed;
	CKR(stream_keep_ahead(h, h->rng[ST_B], 12u << 20)); CKR(stream_prefetch(h, h->rng[ST_S], 1u << 18));
	h->pending = false; h->pend_b = h->pend_s = h->pend_p = 0; h->seg_reads = 0;
	h->routed = h->applied = false;
	resolve_phases(h);
	if (h->grow_all) {
		// Some rank's shard is past half full: every shard of that table doubles (one geometry per table).  The sync is complete and this
		// rank's streams are idle (the apply step ended with a look), so the mappings of the peers' old tables can be closed here; the
		// doubling itself waits for the caller's barrier -- a table must not be freed while a peer still maps it -- and happens in the
		// fqsk_shard_export that follows.
		// (all three tables are remapped, doubled or not: one rule, and the p-mer shards and inboxes -- never reallocated -- stay mapped)
		for (uint32_t r = 0; r < h->world; ++r) {
			if (r == h->rank) continue;
			for (int q : {0, 1, 2, 3, 6, 7}) {      // ipc slots of the b-mer, s-mer and pair tables (fqsk_shard_desc)
				void *&pp = h->peer_ptrs[r][q];
				if (pp) { CK(cudaIpcCloseMemHandle(pp)); pp = nullptr; }
			}
			h->tb.d.peer_main[r] = nullptr; h->tb.d.peer_stash[r] = nullptr; h->ts.d.peer_main[r] = nullptr; h->ts.d.peer_stash[r] = nullptr;
			if (h->pair.keys) { h->pair.peer_keys[r] = nullptr; h->pair.peer_vcs[r] = nullptr; }
		}
		h->attached = 1u << h->rank;
		h->grow_pending = true;
		return FQSK_RESHARD;
	}
	return FQSK_OK;
}

int fqsk_shard_grow_request(fqsk_handle *h, uint32_t *request) {
	if (!h || !request) return FQSK_E_INVAL;
	if (h->world <= 1 || !h->applied) return fail(h, FQSK_E_INVAL, "fqsk_shard_grow_request: between fqsk_sync_apply and fqsk_sync_finish of a sharded engine");
	*request = h->grow_local;
	return FQSK_OK;
}
int fqsk_shard_grow(fqsk_handle *h, uint32_t request_all_ranks) {
	if (!h || request_all_ranks > 7u) return FQSK_E_INVAL;
	if (h->world <= 1 || !h->applied) return fail(h, FQSK_E_INVAL, "fqsk_shard_grow: between fqsk_sync_apply and fqsk_sync_finish of a sharded engine");
	if ((request_all_ranks & 4u) && !h->pair.keys) return fail(h, FQSK_E_INVAL, "fqsk_shard_grow: no pair table");
	h->grow_all = request_all_ranks;
	return FQSK_OK;
}

static int dump_sorted(fqsk_handle *h, uint64_t n, uint64_t *keys, uint64_t *vals) {
	std::vector<unsigned long long> k(n), v(n);
	if (n) {
		CK(cudaMemcpyAsync(k.data(), h->dump_k.p, n * 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaMemcpyAsync(v.data(), h->dump_v.p, n * 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
	}
	std::vector<uint64_t> order(n);
	for (uint64_t i = 0; i < n; ++i) order[i] = i;
	std::sort(order.begin(), order.end(), [&](uint64_t a, uint64_t b) { return k[a] < k[b]; });
	for (uint64_t i = 0; i < n; ++i) { keys[i] = k[order[i]]; vals[i] = v[order[i]]; }
	return FQSK_OK;
}

static int dump_pairs(fqsk_handle *h, uint64_t *keys, uint64_t *vals, uint64_t cap, uint64_t *n) {
	if (!h->pair.keys) return fail(h, FQSK_E_INVAL, "not a paired-end engine");
	const uint64_t slots = h->pair.mask + 1;
	std::vector<unsigned long long> k(slots), v(slots);
	CK(cudaMemcpyAsync(k.data(), h->pair.keys, slots * 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaMemcpyAsync(v.data(), h->pair.vcs, slots * 8, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	std::vector<std::pair<unsigned long long, unsigned long long>> items;
	for (uint64_t i = 0; i < slots; ++i) if (k[i] != PAIR_EMPTY) items.emplace_back(k[i], v[i]);
	*n = items.size();
	if (!keys) return FQSK_OK;
	if (items.size() > cap) return fail(h, FQSK_E_CAPACITY, "dump buffer holds %llu, table has %llu", (unsigned long long) cap, (unsigned long long) items.size());
	std::sort(items.begin(), items.end());
	for (size_t i = 0; i < items.size(); ++i) { keys[i] = items[i].first; vals[i] = items[i].second; }
	return FQSK_OK;
}

int fqsk_dump(fqsk_handle *h, int table, uint64_t *keys, uint64_t *vals, uint64_t cap, uint64_t *n) {
	if (!h || !n) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (h->pending && h->spec_prefix) return fail(h, FQSK_E_INVAL, "fqsk_dump between a segment and its sync: call fqsk_sync first");
	CKR(seg_settle(h));
	if (table == FQSK_TABLE_SMER || table == FQSK_TABLE_BMER) {
		Table &t = table == FQSK_TABLE_SMER ? h->ts : h->tb;
		uint64_t cnt = 0;
		CKR(table_dump_device(h, t, &cnt));
		*n = cnt;
		if (!keys) return FQSK_OK;
		if (cnt > cap) return fail(h, FQSK_E_CAPACITY, "dump needs %llu entries", (unsigned long long) cnt);
		return dump_sorted(h, cnt, keys, vals);
	}
	if (table == FQSK_TABLE_SIV) {
		uint64_t cnt = h->world > 1 ? h->siv_local_filled : h->S.siv_no_filled;
		*n = cnt;
		if (!keys) return FQSK_OK;
		if (cnt > cap) return fail(h, FQSK_E_CAPACITY, "dump needs %llu entries", (unsigned long long) cnt);
		CK(h->dump_k.ensure((cnt + 1) * 8)); CK(h->dump_v.ensure((cnt + 1) * 8));
		CK(cudaMemsetAsync(&h->status->dump_n, 0, 8, h->st));
		uint64_t nw = h->world > 1 ? ((((uint64_t) 4096 + h->world - 1) / h->world) << h->siv.top_shift) >> 4 : (1ull << h->siv.key_bits) >> 4;
		CK(pdl(k_dump_siv, nblk(nw, 256), 256, h->st, h->siv, h->dump_k.as<unsigned long long>(), h->dump_v.as<unsigned long long>(), cnt, &h->status->dump_n));
		LAUNCHED(h);
		unsigned long long got = 0;
		CK(cudaMemcpyAsync(&got, &h->status->dump_n, 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		if (got != cnt) return fail(h, FQSK_E_CUDA, "p-mer dump found %llu fields, no_filled says %llu", got, (unsigned long long) cnt);
		return dump_sorted(h, cnt, keys, vals);
	}
	if (table == FQSK_TABLE_PAIR) return dump_pairs(h, keys, vals, cap, n);
	return fail(h, FQSK_E_UNSUPPORTED, "table %d cannot be dumped", table);
}

int fqsk_stats_get(fqsk_handle *h, fqsk_stats *out) {
	if (!h || !out) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	CKR(seg_settle(h));
	unsigned long long c[4];
	CK(cudaMemcpyAsync(c, h->status->items, sizeof c, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	h->S.n_bmers = c[0] + c[1]; h->S.bmer_stash_used = c[1];
	h->S.n_smers = c[2] + c[3]; h->S.smer_stash_used = c[3];
	h->S.bmer_buckets = 1ull << h->tb.d.B; h->S.smer_buckets = 1ull << h->ts.d.B;
	for (int i = 0; i < 4; ++i) h->S.draws[i] = h->rng[i].consumed;
	*out = h->S;
	return FQSK_OK;
}

int fqsk_timer_begin(fqsk_handle *h) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	if (!h->t0) { CK(cudaEventCreate(&h->t0)); CK(cudaEventCreate(&h->t1)); }
	CK(cudaStreamSynchronize(h->st));
	CK(cudaEventRecord(h->t0, h->st));
	return FQSK_OK;
}
int fqsk_timer_end(fqsk_handle *h, double *ms) {
	if (!h || !ms || !h->t0) return FQSK_E_INVAL;
	CK(cudaEventRecord(h->t1, h->st));
	CK(cudaEventSynchronize(h->t1));
	float f = 0;
	CK(cudaEventElapsedTime(&f, h->t0, h->t1));
	*ms = f;
	return FQSK_OK;
}

// on != 0: start collecting; on == 0: synchronise the device and print one line per launch since the start (kernel, stream, begin and
// end in microseconds after the first launch) to stderr
int fqsk_timeline(fqsk_handle *h, int on) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	static std::vector<TimelineEntry> store;
	if (on) { CK(cudaDeviceSynchronize()); store.clear(); g_timeline = &store; return FQSK_OK; }
	g_timeline = nullptr;
	CK(cudaDeviceSynchronize());
	std::vector<cudaStream_t> streams;
	for (auto &e : store) {
		float a = 0, b = 0;
		cudaError_t ra = cudaEventElapsedTime(&a, store[0].a, e.a), rb = cudaEventElapsedTime(&b, store[0].a, e.b);
		if (ra != cudaSuccess || rb != cudaSuccess) { fprintf(stderr, "[fqsk timeline] cudaEventElapsedTime: %s / %s\n", cudaGetErrorString(ra), cudaGetErrorString(rb)); cudaGetLastError(); }
		size_t si = 0;
		while (si < streams.size() && streams[si] != e.st) ++si;
		if (si == streams.size()) streams.push_back(e.st);
		const char *name = "?";
		cudaFuncGetName(&name, e.fn);
		char shortname[48]; size_t q = 0;
		const char *k = strstr(name, "k_");      // mangled: ...<length>k_name<E or I>...
		size_t len = 40;
		if (k && k > name && isdigit((unsigned char) k[-1])) { const char *d = k; while (d > name && isdigit((unsigned char) d[-1])) --d; len = (size_t) atoi(d); }
		for (const char *c = k ? k : name; *c && q < len && q + 1 < sizeof shortname; ++c) shortname[q++] = *c;
		shortname[q] = 0;
		fprintf(stderr, "[fqsk timeline] %-22s stream %zu  %9.1f %9.1f  (%.1f us)\n", shortname, si, 1e3 * a, 1e3 * b, 1e3 * (b - a));
	}
	for (auto &e : store) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
	store.clear();
	return FQSK_OK;
}

int fqsk_profile(fqsk_handle *h, double *ms, uint32_t n) {
	if (!h || !ms) return FQSK_E_INVAL;
	for (uint32_t i = 0; i < n && i < FQSK_PH_COUNT; ++i) ms[i] = h->ph_ms[i];
	return FQSK_OK;
}

// ---- table-level batch mirrors ----------------------------------------------------------------------------------
static Table *pick(fqsk_handle *h, int table) { return table == FQSK_TABLE_SMER ? &h->ts : table == FQSK_TABLE_BMER ? &h->tb : nullptr; }

// the table-level calls work on the tables between segments: not while a segment's rows are pending or a ticket is open
static int unit_call_ok(fqsk_handle *h, const void *a, const void *b, uint64_t n) {
	if (h->pending || h->tk_open) return fail(h, FQSK_E_INVAL, "table-level call between a segment and its sync (or with a ticket open)");
	if (n && (!a || !b)) return fail(h, FQSK_E_INVAL, "null array");
	if (n > 0xFFFFFFFFull) return fail(h, FQSK_E_INVAL, "more than 2^32 - 1 elements in one call");
	return FQSK_OK;
}

int fqsk_ht_insert(fqsk_handle *h, int table, const uint64_t *kmers, uint64_t n) {
	if (!h) return FQSK_E_INVAL;
	Table *t = pick(h, table);
	if (!t) return fail(h, FQSK_E_INVAL, "bad table");
	CK(cudaSetDevice(h->P.device));
	CKR(unit_call_ok(h, kmers, kmers, n));
	if (!n) return FQSK_OK;
	CK(h->q3.ensure(n * 8));
	CK(cudaMemcpyAsync(h->q3.p, kmers, n * 8, cudaMemcpyHostToDevice, h->st));
	if (table == FQSK_TABLE_SMER) {   // same route as fqsk_sync: atomic fast path that checks itself, ordered path as the fallback
		bool fast = true;
		CKR(apply_inserts(h, *t, h->rng[ST_S], h->q3.as<unsigned long long>(), (uint32_t) n, &fast));
	} else CKR(apply_row(h, *t, h->rng[ST_B], h->q3.as<unsigned long long>(), (uint32_t) n));
	CKR(table_grow_if_needed(h, *t));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}

int fqsk_ht_find(fqsk_handle *h, int table, const uint64_t *kmer_dir, const uint64_t *kmer_rc, const uint32_t *cur_size, uint64_t n, uint32_t *counts) {
	if (!h) return FQSK_E_INVAL;
	Table *t = pick(h, table);
	if (!t) return fail(h, FQSK_E_INVAL, "bad table");
	CK(cudaSetDevice(h->P.device));
	CKR(unit_call_ok(h, kmer_dir, kmer_rc, n)); CKR(unit_call_ok(h, cur_size, counts, n));
	if (!n) return FQSK_OK;
	Stream &rng = h->rng[table == FQSK_TABLE_SMER ? ST_S : ST_B];
	if (n > (uint64_t) SCAN_CHAIN_MAX * SCAN_U32_CHUNK) return fail(h, FQSK_E_INVAL, "more than %u queries in one fqsk_ht_find call", SCAN_CHAIN_MAX * SCAN_U32_CHUNK);
	CK(h->q0.ensure((n + 1) * 8)); CK(h->q1.ensure((n + 1) * 8)); CK(h->q2.ensure((n + 1) * 16)); CK(h->q3.ensure((n + 1) * 16)); CK(h->q4.ensure((n + 1) * 8));
	unsigned long long *d_dir = h->q0.as<unsigned long long>(), *d_rc = h->q1.as<unsigned long long>(), *d_guess = h->q2.as<unsigned long long>(), *d_scan2 = h->q2.as<unsigned long long>() + (n + 1);
	uint32_t *d_counts = h->q3.as<uint32_t>();
	uint32_t *d_cur = h->q4.as<uint32_t>(), *d_used = h->q4.as<uint32_t>() + (n + 1);
	CK(cudaMemcpyAsync(d_dir, kmer_dir, n * 8, cudaMemcpyHostToDevice, h->st));
	CK(cudaMemcpyAsync(d_rc, kmer_rc, n * 8, cudaMemcpyHostToDevice, h->st));
	CK(cudaMemcpyAsync(d_cur, cur_size, n * 4, cudaMemcpyHostToDevice, h->st));
	CK(cudaMemsetAsync(d_guess, 0, (n + 1) * 8, h->st));
	CKR(stream_ensure(h, rng, 1u << 16));
	std::vector<unsigned long long> prev(n + 1, 0), now(n + 1, 0);
	for (int it = 0;; ++it) {
		if (it > 32) return fail(h, FQSK_E_NO_CONVERGE, "find: draw offsets did not settle");
		CK(cudaMemsetAsync(h->status->flags, 0, 4 * sizeof(int), h->st));
		CK(cudaMemsetAsync(d_used + n, 0, 4, h->st));
		CK(pdl(k_find, nblk(n, 128), 128, h->st, t->d, t->ci, d_dir, d_rc, d_cur, (uint32_t) n, d_counts, rng.buf, rng.cap - 1, rng.consumed, stream_avail(rng), d_guess, d_used, h->status->flags));
		LAUNCHED(h);
		int fl[4];
		CKR(read_flags(h, fl, 4));
		if (fl[0]) { CKR(stream_ensure(h, rng, 2 * stream_avail(rng) + (1u << 16))); --it; continue; }
		{   // per-query draw counts -> exclusive offsets (d_guess[n] = total)
			ScanChain sc; CKR(scan_chain(h, sc));
			CK(pdl(k_scan_draws, std::max<uint32_t>(nblk((uint32_t) n, SCAN_U32_CHUNK), 1), 1024, h->st, (uint32_t) n, (const uint32_t *) d_used, d_guess, (const uint32_t *) d_used, d_scan2,
			       h->status->scratch, (int *) nullptr, sc)); LAUNCHED(h);
		}
		CK(cudaMemcpyAsync(now.data(), d_guess, (n + 1) * 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
		if (now == prev) break;
		prev = now;
	}
	rng.consumed += now[n];
	CK(cudaMemcpyAsync(counts, d_counts, n * 16, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}

int fqsk_ht_count(fqsk_handle *h, int table, const uint64_t *kmers, uint64_t n, uint32_t *out) {
	if (!h) return FQSK_E_INVAL;
	Table *t = pick(h, table);
	if (!t) return fail(h, FQSK_E_INVAL, "bad table");
	CK(cudaSetDevice(h->P.device));
	CKR(unit_call_ok(h, kmers, out, n));
	if (!n) return FQSK_OK;
	CK(h->q0.ensure(n * 8)); CK(h->q1.ensure(n * 4));
	CK(cudaMemcpyAsync(h->q0.p, kmers, n * 8, cudaMemcpyHostToDevice, h->st));
	CK(pdl(k_count, nblk(n, 256), 256, h->st, t->d, h->q0.as<unsigned long long>(), (uint32_t) n, h->q1.as<uint32_t>()));
	LAUNCHED(h);
	CK(cudaMemcpyAsync(out, h->q1.p, n * 4, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}

int fqsk_siv_increment(fqsk_handle *h, const uint64_t *idx, uint64_t n, uint64_t *n_new) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	CKR(unit_call_ok(h, idx, idx, n));
	for (uint64_t i = 0; i < n; ++i) {      // a p-mer index outside 4^p, or one another rank owns, would be written outside this rank's array
		if (idx[i] >> h->siv.key_bits) return fail(h, FQSK_E_INVAL, "p-mer index %llu does not fit %u bits", (unsigned long long) idx[i], h->siv.key_bits);
		if (h->world > 1 && (idx[i] >> h->siv.top_shift) % h->world != h->rank) return fail(h, FQSK_E_INVAL, "p-mer index %llu belongs to another rank's shard", (unsigned long long) idx[i]);
	}
	unsigned long long fresh = 0;
	if (n) {
		CK(h->q0.ensure(n * 8));
		CK(cudaMemcpyAsync(h->q0.p, idx, n * 8, cudaMemcpyHostToDevice, h->st));
		CK(cudaMemsetAsync(&h->status->siv_fresh, 0, 8, h->st));
		CK(pdl(k_siv_increment, nblk(n, 256), 256, h->st, h->siv, h->q0.as<unsigned long long>(), n, &h->status->siv_fresh, (const SyncIn *) nullptr));
		LAUNCHED(h);
		CK(cudaMemcpyAsync(&fresh, &h->status->siv_fresh, 8, cudaMemcpyDeviceToHost, h->st));
		CK(cudaStreamSynchronize(h->st));
	}
	h->S.siv_no_filled += fresh; h->S.siv_no_updates += n;
	if (n_new) *n_new = fresh;
	return FQSK_OK;
}

static int siv_query(fqsk_handle *h, int what, const uint64_t *idx, const uint32_t *bits, uint64_t n, void *out) {
	CK(cudaSetDevice(h->P.device));
	CKR(unit_call_ok(h, idx, out, n));
	if (what == 2 && n && !bits) return fail(h, FQSK_E_INVAL, "null array");
	for (uint64_t i = 0; i < n; ++i) {
		const uint32_t kb = what == 2 ? bits[i] : h->siv.key_bits;
		if (kb > h->siv.key_bits || (kb < 64 && (idx[i] >> kb)) || (what == 2 && h->world > 1 && kb < 12)) return fail(h, FQSK_E_INVAL, "p-mer index / prefix %llu out of range", (unsigned long long) idx[i]);
	}
	if (!n) return FQSK_OK;
	CK(h->q0.ensure(n * 8)); CK(h->q1.ensure(n * 16)); CK(h->q2.ensure(n * 4));
	CK(cudaMemcpyAsync(h->q0.p, idx, n * 8, cudaMemcpyHostToDevice, h->st));
	if (bits) CK(cudaMemcpyAsync(h->q2.p, bits, n * 4, cudaMemcpyHostToDevice, h->st));
	size_t ob;
	if (what == 0) { CK(pdl(k_siv_test, nblk(n, 256), 256, h->st, h->siv, h->q0.as<unsigned long long>(), (uint32_t) n, h->q1.as<uint32_t>())); ob = n * 4; }
	else if (what == 1) { CK(pdl(k_siv_counts, nblk(n, 256), 256, h->st, h->siv, h->q0.as<unsigned long long>(), (uint32_t) n, h->q1.as<uint32_t>())); ob = n * 16; }
	else { CK(pdl(k_siv_prefix, nblk(n, 256), 256, h->st, h->siv, h->q0.as<unsigned long long>(), h->q2.as<uint32_t>(), (uint32_t) n, h->q1.as<unsigned long long>())); ob = n * 8; }
	LAUNCHED(h);
	CK(cudaMemcpyAsync(out, h->q1.p, ob, cudaMemcpyDeviceToHost, h->st));
	CK(cudaStreamSynchronize(h->st));
	return FQSK_OK;
}
int fqsk_siv_test(fqsk_handle *h, const uint64_t *idx, uint64_t n, uint32_t *out) { return h ? siv_query(h, 0, idx, nullptr, n, out) : FQSK_E_INVAL; }
int fqsk_siv_counts(fqsk_handle *h, const uint64_t *idx, uint64_t n, uint32_t *out4) { return h ? siv_query(h, 1, idx, nullptr, n, out4) : FQSK_E_INVAL; }
int fqsk_siv_test_shorter(fqsk_handle *h, const uint64_t *idx, const uint32_t *size_bits, uint64_t n, uint64_t *out) { return h ? siv_query(h, 2, idx, size_bits, n, out) : FQSK_E_INVAL; }

int fqsk_host_alloc(uint64_t bytes, void **out) {
	if (!out) return FQSK_E_INVAL;
	*out = nullptr;
	cudaError_t e = cudaMallocHost(out, bytes ? bytes : 1);
	if (e != cudaSuccess) { g_create_error = std::string("cudaMallocHost: ") + cudaGetErrorString(e); return e == cudaErrorMemoryAllocation ? FQSK_E_NOMEM : FQSK_E_CUDA; }
	return FQSK_OK;
}
void fqsk_host_free(void *p) { if (p) cudaFreeHost(p); }

int fqsk_mt_stream(fqsk_handle *h, uint64_t n, uint32_t *out) {
	if (!h) return FQSK_E_INVAL;
	CK(cudaSetDevice(h->P.device));
	// a scratch stream: same seed, generated from scratch so the engine's own streams are untouched
	Stream s;
	uint64_t cap = 1u << 16;
	while (cap < n + 1248) cap <<= 1;
	CKR(stream_init(h, s, cap));
	int rc = stream_ensure(h, s, n);
	if (rc == FQSK_OK && n) {
		cudaError_t e = cudaMemcpyAsync(out, s.buf, n * 4, cudaMemcpyDeviceToHost, h->st);
		if (e == cudaSuccess) e = cudaStreamSynchronize(h->st);
		if (e != cudaSuccess) rc = fail(h, FQSK_E_CUDA, "mt_stream copy: %s", cudaGetErrorString(e));
	}
	cudaStreamSynchronize(h->st_mt);
	if (s.buf) cudaFree(s.buf);
	if (s.state) cudaFree(s.state);
	if (s.jstates) cudaFree(s.jstates);
	if (s.ev) cudaEventDestroy(s.ev);
	return rc;
}

}  // extern "C"
