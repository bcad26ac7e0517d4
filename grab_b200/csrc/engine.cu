// engine.cu -- host side of libgscan.so: contexts, batch planning, staging, kernel orchestration and
// the extern "C" surface declared in include/gscan.h.
//
// Mirrors the reference's ownership model: a gscan_ctx is what a FileGrep object is in
// /root/reference/src/grab.cc (one per host thread, main.cc:195-199) -- it owns its stream, its
// device buffers and its last error string (FileGrep::why, grab.h:61-64).  Errors never throw
// across the ABI and never abort: int 0 / -1 + message.
#include <cuda_runtime.h>
#include <unistd.h>

#include <cerrno>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "../../include/gscan.h"
#include "device_types.h"
#include "kernels.h"
#include "pattern.h"

using namespace gscan;

// ------------------------------------------------------------------------------------------
// objects behind the opaque handles
// ------------------------------------------------------------------------------------------
struct gscan_pattern {
	Program prog;
	// host images of the device tables (FIXED engine)
	std::vector<uint16_t> seq_len;
	std::vector<uint32_t> seq_off, seq_pos, cls_bm;
	FixedParams fixed; // device pointers filled per context
	HashParams hash;
	RunParams run;
};

template <class T>
struct DevBuf {
	T *p = nullptr;
	size_t cap = 0; // elements
	cudaError_t ensure(size_t n)
	{
		if (n <= cap) return cudaSuccess;
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
		size_t want = std::max<size_t>(n, 1024);
		cudaError_t e = cudaMalloc(&p, want * sizeof(T));
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinnedBuf {
	void *p = nullptr;
	size_t cap = 0;
	cudaError_t ensure(size_t bytes)
	{
		if (bytes <= cap) return cudaSuccess;
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
		size_t want = std::max<size_t>(bytes, 1 << 16);
		cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct gscan_batch {
	uint32_t n_units = 0;        // units with len > 0, in caller order
	TileDesc *d_tiles = nullptr;
	DevUnit *d_units = nullptr;
	uint8_t *d_arena = nullptr;  // staged copies of host units (owned)
	uint32_t n_tiles = 0;
	uint32_t tile_shift = kMaxTileShift; // tiles of this batch are 2^tile_shift bytes (device_types.h)
	uint64_t bytes = 0;
	float h2d_ms = 0;
	bool pooled = false;         // device buffers belong to the context (gscan_scan_batch's transient batches)
};

struct gscan_ctx {
	int device = 0;
	int num_sms = 0;
	cudaStream_t stream = nullptr;
	cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
	std::string err;
	gscan_stats stats;

	DevBuf<SegEntry> segs;
	uint32_t seg_tag = 0;      // generation of the last scan that wrote segs (0: table freshly zeroed)
	DevBuf<Cand> cand;
	DevBuf<Cand> scratch;
	DevBuf<OutRec> ord;
	DevBuf<FinalRec> out;
	// pinned result buffers handed to the caller (gscan_match arrays), recycled by gscan_free_matches
	struct ResultBuf { void *p; size_t cap; bool lent; };
	std::vector<ResultBuf> results;
	DevBuf<uint32_t> unit_start, unit_out, blk, chain, vm_flag, vm_unit_start;
	DevBuf<OutRec> vm_ord;
	DevBuf<unsigned long long> vm_budget;
	DevBuf<unsigned long long> cursor; // [0] cursor, then 2 x u32 totals behind it
	DevBuf<uint8_t> pat_tables, hash_tables, vm_tables;
	const uint32_t *vm_code = nullptr, *vm_sets = nullptr;
	uint64_t pat_id = 0;
	FixedParams pat_fixed; // with this context's device pointers
	HashParams pat_hash;
	PinnedBuf readback;
	DevBuf<unsigned long long> probe_sum;
	DevBuf<uint8_t> needle;
	// staging of pageable host memory (the reference's mmap windows): helper threads, each with its own stream,
	// two pinned bounce buffers and two events
	struct StageLane { cudaStream_t stream = nullptr; void *buf[2] = {nullptr, nullptr}; cudaEvent_t ev[2] = {nullptr, nullptr}; };
	std::vector<StageLane> lanes;
	std::vector<void *> stage_slabs; // the lanes' bounce buffers are carved out of few big pinned allocations (one cudaHostAlloc per growth, not two per lane)
	// pools behind the transient batches of gscan_scan_batch (grow-only: no cudaMalloc/cudaFree per call)
	DevBuf<uint8_t> pool_arena;
	DevBuf<TileDesc> pool_tiles;
	DevBuf<DevUnit> pool_units;
	// the job of gscan_scan_batch_async (one in flight)
	std::thread job;
	bool job_active = false;
	int job_rc = 0;
	gscan_match *job_out = nullptr;
	size_t job_n = 0;
};

static thread_local std::string g_last_error;

static int fail(gscan_ctx *ctx, const std::string &msg)
{
	if (ctx) ctx->err = msg;
	g_last_error = msg;
	return -1;
}

#define CK(ctx, call)                                                                                  \
	do {                                                                                               \
		cudaError_t e__ = (call);                                                                      \
		if (e__ != cudaSuccess)                                                                        \
			return fail(ctx, std::string("gscan: ") + #call + ": " + cudaGetErrorString(e__));        \
	} while (0)

static inline uint32_t rep4(uint8_t b) { return (uint32_t)b * 0x01010101u; }
static inline uint32_t round16(uint32_t x) { return (x + 15u) & ~15u; }

// ------------------------------------------------------------------------------------------
// pattern
// ------------------------------------------------------------------------------------------
extern "C" int gscan_compile(const char *pattern, size_t len, uint32_t flags, gscan_pattern **out)
{
	if (!pattern || !out) { g_last_error = "gscan_compile: null argument"; return -1; }
	*out = nullptr;
	gscan_pattern *p = new (std::nothrow) gscan_pattern;
	if (!p) { g_last_error = "gscan_compile: out of memory"; return -1; }
	std::string err;
	if (!compile_pattern(pattern, len, flags, p->prog, err)) {
		g_last_error = "gscan_compile: " + err;
		delete p;
		return -1;
	}
	const Program &pr = p->prog;
	memset(&p->fixed, 0, sizeof(p->fixed));
	memset(&p->run, 0, sizeof(p->run));
	memset(&p->hash, 0, sizeof(p->hash));
	if (pr.kind == ENGINE_FIXED && !pr.vm_dense) {
		FixedParams &F = p->fixed;
		F.one = 1;
		F.ntests = (uint32_t)pr.tests.size();
		F.exact = 1;
		for (auto &t : pr.tests) if (t.m0 != 0xff || (pr.delta && t.m1 != 0xff)) F.exact = 0;
		if (!pr.delta) F.exact = 0; // single-byte filter: the second term must vanish through its zero mask
		F.n2 = (uint32_t)pr.triples.size();
		F.d2 = (uint32_t)pr.delta2;
		F.stage1_triples = pr.stage1_triples ? 1u : 0u;
		F.sh1 = 8u * (uint32_t)pr.delta;
		F.sh2 = 8u * (uint32_t)pr.delta2;
		F.exact3 = 1;
		for (int k = 0; k < 16; k++) { F.t2_m0[k] = 0; F.t2_v0[k] = 0xffffffffu; F.t2_m1[k] = 0; F.t2_v1[k] = 0; F.t2_m2[k] = 0; F.t2_v2[k] = 0; }
		for (auto &t : pr.triples) if (t.m0 != 0xff || t.m1 != 0xff || t.m2 != 0xff) F.exact3 = 0;
		for (size_t k = 0; k < pr.triples.size(); k++) {
			F.t2_m0[k] = rep4(pr.triples[k].m0); F.t2_v0[k] = rep4(pr.triples[k].v0);
			F.t2_m1[k] = rep4(pr.triples[k].m1); F.t2_v1[k] = rep4(pr.triples[k].v1);
			F.t2_m2[k] = rep4(pr.triples[k].m2); F.t2_v2[k] = rep4(pr.triples[k].v2);
		}
		for (int k = 0; k < 8; k++) { // unused slots: a test no byte can pass
			F.m0[k] = 0; F.v0[k] = 0xffffffffu; F.m1[k] = 0; F.v1[k] = 0;
		}
		for (size_t k = 0; k < pr.tests.size(); k++) {
			F.m0[k] = rep4(pr.tests[k].m0); F.v0[k] = rep4(pr.tests[k].v0);
			F.m1[k] = rep4(pr.tests[k].m1); F.v1[k] = rep4(pr.tests[k].v1);
		}
		{ // balanced pair filter (FixedBEngine): exact byte pairs, 2..8 tests; stage 2 needs one third-byte test per pair test
			F.b_engine = 0; F.b_aligned = 0; F.b_sh2 = 8u * (uint32_t)pr.delta2;
			for (int k = 0; k < 8; k++) { F.b_c0[k] = 0; F.b_c1[k] = 0; F.b_x0[k] = 0; F.b_x1[k] = 0; F.b_m2[k] = 0; F.b_v2[k] = 0xffffffffu; }
			const size_t nt = pr.tests.size();
			bool aligned = !pr.triples.empty() && pr.triples.size() == nt;
			for (size_t k = 0; k < nt && k < 8; k++) {
				const FilterTest &t = pr.tests[k];
				F.b_c0[k] = 0u - rep4(t.v0 & 0x7f); F.b_c1[k] = 0u - rep4(t.v1 & 0x7f);
				F.b_x0[k] = rep4(t.v0 | 0x80); F.b_x1[k] = rep4(t.v1 | 0x80);
				int hit = -1, hits = 0;
				for (size_t j = 0; j < pr.triples.size(); j++) {
					const Program::Triple &q = pr.triples[j];
					if (q.m0 == t.m0 && q.v0 == t.v0 && q.m1 == t.m1 && q.v1 == t.v1) { hit = (int)j; hits++; }
				}
				if (hits != 1) aligned = false;
				else { F.b_m2[k] = rep4(pr.triples[(size_t)hit].m2); F.b_v2[k] = rep4(pr.triples[(size_t)hit].v2); }
			}
			F.b_aligned = aligned ? 1u : 0u;
			const char *off = getenv("GSCAN_NO_FIXEDB"); // A/B switch for measurements
			if (F.exact && nt >= 2 && nt <= 8 && pr.delta >= 1 && pr.delta <= 4 && !pr.use_hash && !(off && *off == '1') &&
			    (aligned || pr.pair_flag_prior * 512.0 <= 0.01))
				F.b_engine = 1;
		}
		F.anchor = (uint32_t)pr.anchor;
		F.nseq = (uint32_t)pr.seqs.size();
		// the longest candidate sequence: what a verification may read behind a candidate decides between the slice in shared
		// memory and global memory.  NOT pr.maxlen: for general patterns (the sequences are only the leading bytes) that is -1,
		// which made every verification read shared memory -- past the resident slice for a candidate on a slice's last bytes,
		// i.e. whatever an earlier slice had left there: a candidate lost or invented per few thousand, depending on history
		// (found by tools/tile_edge_diag.py in round 2; FIXED patterns proper were never affected)
		size_t longest = 0;
		for (auto &s : pr.seqs) longest = std::max(longest, s.size());
		F.maxlen = (uint32_t)longest;
		bool uniform = true;
		for (auto &s : pr.seqs) uniform = uniform && s.size() == pr.seqs[0].size();
		F.uniform_len = uniform ? (uint32_t)pr.seqs[0].size() : 0u;
		std::vector<ByteSet> classes;
		for (auto &s : pr.seqs) {
			p->seq_len.push_back((uint16_t)s.size());
			p->seq_off.push_back((uint32_t)p->seq_pos.size());
			for (auto &cls : s) {
				MaskedEq e = masked_superset(cls);
				if (e.exact) {
					p->seq_pos.push_back((uint32_t)e.mask | ((uint32_t)e.val << 8) | (0xffffu << 16));
				} else {
					size_t id = 0;
					for (; id < classes.size(); id++) if (classes[id] == cls) break;
					if (id == classes.size()) classes.push_back(cls);
					p->seq_pos.push_back((uint32_t)id << 16);
				}
			}
		}
		for (auto &c : classes) for (int i = 0; i < 8; i++) p->cls_bm.push_back(c.w[i]);
		if (pr.use_hash) {
			HashParams &H = p->hash;
			H.mulsh = pr.hash_mul << (8 * (4 - pr.hash_len));
			H.nslots = pr.hash_slots;
			H.stride = hash_table_copies(pr.hash_slots) * 4u;
			H.neg1 = 0xffffffffu;
			H.pow2_shift = H.pow2_mask = 0;
			if (H.stride == 128u && (H.nslots & (H.nslots - 1u)) == 0u && H.nslots >= 2u) {
				uint32_t lg = 0;
				while ((1u << lg) < H.nslots) lg++;
				H.pow2_shift = 32u - lg - 7u;          // slot = h >> (32 - lg); row offset = slot * 128
				H.pow2_mask = (H.nslots - 1u) << 7;
			}
			H.uniform_len = F.uniform_len;
			H.maxlen = F.maxlen;
			// class prefilter of the sparse path: one byte range that holds every key byte
			H.one = 1;
			H.hash_len = (uint32_t)pr.hash_len;
			uint32_t lo = 255, hi = 0;
			for (uint32_t k : pr.hash_table) {
				if (k == 0xffffffffu) continue;
				for (int i = 0; i < pr.hash_len; i++) {
					const uint32_t b = (k >> (8 * i)) & 0xffu;
					lo = std::min(lo, b);
					hi = std::max(hi, b);
				}
			}
			const char *pre_off = getenv("GSCAN_HASH_PRE");
			H.pre_enable = lo >= 1 && hi <= 0x7d && hi - lo < 48 && !(pre_off && *pre_off == '0');
			H.pre_ge = (0x80u - lo) * 0x01010101u;
			H.pre_gt = (0x7eu - hi) * 0x01010101u;
			for (int k = 0; k < 7; k++) H.pre_mul[k] = 1u << (25 + k);
			H.tail = nullptr;
		}
	} else if (pr.kind == ENGINE_RUN) {
		RunParams &R = p->run;
		R.one = 1;
		// two low ranges [a,b] and [a+0x20,b+0x20] inside one 64-byte block with bit 5 clear / set throughout
		// ([A-Z] and [a-z]) collapse into one test of x | 0x20 against the upper range: exact, one range cheaper
		std::vector<ByteRange> low = pr.ranges_low;
		R.nfold = 0;
		for (size_t i = 0; i < low.size() && !R.nfold; i++)
			for (size_t j = 0; j < low.size() && !R.nfold; j++) {
				const ByteRange a = low[i], b = low[j];
				if (i != j && b.lo == a.lo + 0x20 && b.hi == a.hi + 0x20 && !(a.lo & 0x20) && !(a.hi & 0x20) && (a.lo >> 6) == (a.hi >> 6)) {
					R.nfold = 1;
					R.add_ge_fold = rep4((uint8_t)(0x80 - b.lo));
					R.add_gt_fold = rep4((uint8_t)(0x7f - b.hi));
					low.erase(low.begin() + (long)std::max(i, j));
					low.erase(low.begin() + (long)std::min(i, j));
				}
			}
		R.nlo = (uint32_t)low.size();
		R.nhi = (uint32_t)pr.ranges_high.size();
		for (size_t i = 0; i < low.size(); i++) {
			R.add_ge_lo[i] = rep4((uint8_t)(0x80 - low[i].lo));
			R.add_gt_lo[i] = rep4((uint8_t)(0x7f - low[i].hi));
		}
		for (size_t i = 0; i < pr.ranges_high.size(); i++) {
			R.add_ge_hi[i] = rep4((uint8_t)(0x80 - (pr.ranges_high[i].lo - 0x80)));
			R.add_gt_hi[i] = rep4((uint8_t)(0x7f - (pr.ranges_high[i].hi - 0x80)));
		}
		R.run_min = (uint32_t)pr.run_min;
		{ // AND-with-shift schedule for "at least nf consecutive ones": doubling while 2*len <= nf, then the remainder
			const uint32_t nf = std::min<uint32_t>((uint32_t)pr.run_min, 17u);
			uint32_t len = 1;
			int k = 0;
			for (int i = 0; i < 5; i++) R.sh[i] = 0;
			while (len * 2 <= nf) { R.sh[k++] = len; len *= 2; }
			if (len < nf) R.sh[k++] = nf - len;
		}
		for (int i = 0; i < 8; i++) R.bitmap[i] = pr.run_class.w[i];
	}
	*out = p;
	return 0;
}

extern "C" void gscan_free_pattern(gscan_pattern *p) { delete p; }
extern "C" int gscan_minlen(const gscan_pattern *p) { return p ? p->prog.minlen : -1; }
extern "C" const char *gscan_last_error(void) { return g_last_error.c_str(); }
extern "C" int gscan_abi_version(void) { return GSCAN_ABI_VERSION; }

extern "C" int gscan_pattern_get_info(const gscan_pattern *p, gscan_pattern_info *o)
{
	if (!p || !o) return -1;
	o->minlen = p->prog.minlen;
	o->maxlen = p->prog.maxlen;
	o->captures = p->prog.captures;
	o->engine = p->prog.use_vm ? GSCAN_ENGINE_VM : (int32_t)p->prog.kind;
	o->n_sequences = (int32_t)p->prog.seqs.size();
	o->n_filter_tests = p->prog.use_hash ? -(int32_t)p->prog.hash_slots : (int32_t)p->prog.tests.size();
	o->filter_anchor = p->prog.anchor;
	o->filter_delta = p->prog.delta;
	o->scan_variant = 0;
	if (p->prog.kind == ENGINE_NONE || (p->prog.use_vm && p->prog.vm_dense)) o->scan_kernel = GSCAN_KERNEL_NONE;
	else if (p->prog.kind == ENGINE_RUN) o->scan_kernel = GSCAN_KERNEL_RUN;
	else if (p->prog.use_hash) o->scan_kernel = GSCAN_KERNEL_HASH;
	else if (p->fixed.b_engine) o->scan_kernel = GSCAN_KERNEL_BALANCED;
	else o->scan_kernel = p->fixed.stage1_triples ? GSCAN_KERNEL_TRIPLE : GSCAN_KERNEL_PAIR;
	// what launch_scan_fixed / launch_scan_hash / launch_scan_run dispatch on (layout: include/gscan.h)
	if (o->scan_kernel == GSCAN_KERNEL_RUN) {
		const RunParams &R = p->run;
		o->scan_variant = (int32_t)(R.nlo | R.nhi << 4 | R.nfold << 6 | (R.run_min > 17u ? GSCAN_SV_RUN_LONG : 0u));
	} else if (o->scan_kernel == GSCAN_KERNEL_HASH) {
		const HashParams &H = p->hash;
		o->scan_variant = (int32_t)(H.hash_len | (H.pre_enable ? GSCAN_SV_HASH_SPARSE : 0u) | (H.stride / 4u) << 3);
	} else if (o->scan_kernel != GSCAN_KERNEL_NONE) {
		const FixedParams &F = p->fixed;
		o->scan_variant = (int32_t)(F.ntests | (uint32_t)p->prog.delta << 4 | (F.exact ? GSCAN_SV_EXACT : 0u) |
		                            (F.b_engine ? GSCAN_SV_BALANCED : 0u) | (F.b_aligned ? GSCAN_SV_ALIGNED : 0u) |
		                            (F.stage1_triples ? GSCAN_SV_STAGE1_TRIPLES : 0u) | F.n2 << 11 | (F.exact3 ? GSCAN_SV_EXACT3 : 0u));
	}
	return 0;
}

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
extern "C" gscan_ctx *gscan_open(int device)
{
	// GSCAN_TRACE_OPEN=1: where the start-up time goes (driver initialisation / primary context / the rest), on stderr
	const bool trace = getenv("GSCAN_TRACE_OPEN") != nullptr;
	auto t0 = std::chrono::steady_clock::now();
	auto lap = [&](const char *what) {
		if (!trace) return;
		const auto t1 = std::chrono::steady_clock::now();
		fprintf(stderr, "[gscan_open] %-44s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
		t0 = t1;
	};
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	lap("cudaGetDeviceCount (driver initialisation)");
	if (e != cudaSuccess || n == 0) {
		g_last_error = std::string("gscan_open: no CUDA device (") + cudaGetErrorString(e) +
		               "): the scan has no CPU fallback";
		return nullptr;
	}
	if (device < 0 || device >= n) { g_last_error = "gscan_open: bad device index"; return nullptr; }
	gscan_ctx *c = new (std::nothrow) gscan_ctx;
	if (!c) { g_last_error = "gscan_open: out of memory"; return nullptr; }
	c->device = device;
	memset(&c->stats, 0, sizeof(c->stats));
	int major = 0, minor = 0, sms = 0;
	if ((e = cudaSetDevice(device)) == cudaSuccess) e = cudaFree(nullptr); // creates the primary context
	lap("cudaSetDevice + cudaFree(0) (primary context)");
	// three attributes, not cudaGetDeviceProperties (which queries every property of the device)
	if (e == cudaSuccess) e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
	if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device);
	if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
	if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
	if (e != cudaSuccess) {
		g_last_error = std::string("gscan_open: ") + cudaGetErrorString(e);
		delete c;
		return nullptr;
	}
	if (major != 10) {
		g_last_error = "gscan_open: this library is built for sm_100a (B200) only; device is sm_" +
		               std::to_string(major) + std::to_string(minor);
		cudaStreamDestroy(c->stream);
		delete c;
		return nullptr;
	}
	c->num_sms = sms;
	for (auto &ev : c->ev) cudaEventCreate(&ev);
	lap("attributes, stream, events");
	return c;
}

extern "C" void gscan_close(gscan_ctx *c)
{
	if (!c) return;
	if (c->job_active) { c->job.join(); c->job_active = false; }
	cudaSetDevice(c->device);
	cudaStreamSynchronize(c->stream);
	c->segs.release(); c->cand.release(); c->scratch.release(); c->ord.release(); c->out.release();
	c->unit_start.release(); c->unit_out.release(); c->blk.release(); c->chain.release(); c->vm_flag.release(); c->vm_unit_start.release(); c->vm_ord.release(); c->vm_budget.release(); c->cursor.release(); c->pat_tables.release(); c->hash_tables.release(); c->vm_tables.release();
	c->probe_sum.release(); c->needle.release();
	c->pool_arena.release(); c->pool_tiles.release(); c->pool_units.release();
	c->readback.release();
	for (auto &rb : c->results) if (rb.p) cudaFreeHost(rb.p);
	for (auto &l : c->lanes) {
		for (int i = 0; i < 2; i++) if (l.ev[i]) cudaEventDestroy(l.ev[i]);
		if (l.stream) cudaStreamDestroy(l.stream);
	}
	for (void *slab : c->stage_slabs) cudaFreeHost(slab);
	for (auto &ev : c->ev) if (ev) cudaEventDestroy(ev);
	cudaStreamDestroy(c->stream);
	delete c;
}

extern "C" const char *gscan_why(const gscan_ctx *c) { return c ? c->err.c_str() : g_last_error.c_str(); }

extern "C" int gscan_last_stats(const gscan_ctx *c, gscan_stats *o)
{
	if (!c || !o) return -1;
	*o = c->stats;
	return 0;
}

// ------------------------------------------------------------------------------------------
// batches
// ------------------------------------------------------------------------------------------
extern "C" void gscan_batch_free(gscan_ctx *ctx, gscan_batch *b)
{
	if (!b) return;
	if (ctx) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
	if (!b->pooled) {
		if (b->d_tiles) cudaFree(b->d_tiles);
		if (b->d_units) cudaFree(b->d_units);
		if (b->d_arena) cudaFree(b->d_arena);
	}
	delete b;
}

static int batch_create(gscan_ctx *ctx, const gscan_unit *units, size_t n_units, bool pooled, gscan_batch **out);

// ---- feed path for pageable host memory (SURVEY.md 8(f) f1) ----
// A single memcpy into a pinned bounce buffer runs at ~8 GB/s, PCIe Gen5 takes ~55 GB/s: several helper threads
// copy disjoint 4 MiB chunks into their own pinned buffers and queue the H2D copies on their own streams.
// fd >= 0: the bytes are the `len` bytes at offset `foff` of that descriptor (GSCAN_UNIT_FD), read with pread() straight
// into the bounce buffer: no mapping, no page faults in the helper threads, no munmap under mmap_lock afterwards
struct StagePiece { const uint8_t *src; uint8_t *dst; size_t len; int fd; uint64_t foff; };
// one bounce-buffer load: pieces [first, first + count) whose arena range [dst, dst + span) is at most kStageChunk --
// many small units (1 MiB files) travel as ONE 4 MiB copy instead of four
struct StageJob { size_t first, count; uint8_t *dst; size_t span; };
constexpr size_t kStageChunk = 4u << 20;

static int stage_pageable(gscan_ctx *ctx, const std::vector<StagePiece> &pieces)
{
	// group consecutive pieces (ascending arena addresses) into bounce-buffer loads
	std::vector<StageJob> jobs;
	size_t total = 0;
	for (size_t i = 0; i < pieces.size(); i++) {
		total += pieces[i].len;
		if (!jobs.empty()) {
			StageJob &j = jobs.back();
			const uint8_t *end = pieces[i].dst + pieces[i].len;
			if (pieces[i].dst >= j.dst + j.span && (size_t)(end - j.dst) <= kStageChunk) { j.count++; j.span = (size_t)(end - j.dst); continue; }
		}
		jobs.push_back(StageJob{i, 1, pieces[i].dst, pieces[i].len});
	}
	int want = 12; // measured on the B200 box (tools/stage_sweep.py): 4 -> 33, 8 -> 35/49, 12 -> 38/50, 16 -> 38/49, 24 -> 32/39 GB/s (1 MiB / 64 MiB units)
	if (const char *e = getenv("GSCAN_STAGE_THREADS")) want = atoi(e);
	const int hw = (int)std::thread::hardware_concurrency();
	if (hw > 0 && want > hw) want = hw;
	if (want < 1 || total < (16u << 20)) want = 1;
	if ((size_t)want > jobs.size()) want = (int)jobs.size();
	if ((int)ctx->lanes.size() < want) {
		// all missing lanes' buffers in ONE pinned allocation instead of two per lane (the first batch of a process spends
		// 40-80 ms staging against 8 ms for the following ones: allocations, not copies)
		const size_t missing = (size_t)want - ctx->lanes.size();
		void *slab = nullptr;
		CK(ctx, cudaHostAlloc(&slab, missing * 2 * kStageChunk, cudaHostAllocDefault));
		ctx->stage_slabs.push_back(slab);
		for (size_t m = 0; m < missing; m++) {
			gscan_ctx::StageLane l;
			CK(ctx, cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
			for (int i = 0; i < 2; i++) {
				l.buf[i] = static_cast<uint8_t *>(slab) + (2 * m + (size_t)i) * kStageChunk;
				CK(ctx, cudaEventCreateWithFlags(&l.ev[i], cudaEventDisableTiming));
			}
			ctx->lanes.push_back(l);
		}
	}
	std::atomic<int> err{(int)cudaSuccess};
	std::atomic<int> io_errno{0}; // first pread failure (GSCAN_UNIT_FD units); -1: the file ended early
	auto work = [&](int t) {
		cudaSetDevice(ctx->device);
		gscan_ctx::StageLane &l = ctx->lanes[t];
		bool used[2] = {false, false};
		int k = 0;
		for (size_t j = (size_t)t; j < jobs.size() && err.load() == (int)cudaSuccess && !io_errno.load(); j += (size_t)want, k ^= 1) {
			cudaError_t e = cudaSuccess;
			if (used[k]) e = cudaEventSynchronize(l.ev[k]);
			if (e == cudaSuccess) {
				const StageJob &job = jobs[j];
				for (size_t q = job.first; q < job.first + job.count; q++) { // the gaps between units (256-byte alignment) travel as they are
					uint8_t *to = static_cast<uint8_t *>(l.buf[k]) + (pieces[q].dst - job.dst);
					if (pieces[q].fd < 0) { memcpy(to, pieces[q].src, pieces[q].len); continue; }
					for (size_t done = 0; done < pieces[q].len;) {
						const ssize_t r = pread(pieces[q].fd, to + done, pieces[q].len - done, (off_t)(pieces[q].foff + done));
						if (r < 0 && errno == EINTR) continue;
						if (r <= 0) {
							int want_no = 0;
							io_errno.compare_exchange_strong(want_no, r < 0 ? errno : -1);
							break;
						}
						done += (size_t)r;
					}
				}
				if (io_errno.load()) break;
				e = cudaMemcpyAsync(job.dst, l.buf[k], job.span, cudaMemcpyHostToDevice, l.stream);
			}
			if (e == cudaSuccess) e = cudaEventRecord(l.ev[k], l.stream);
			used[k] = true;
			if (e != cudaSuccess) err.store((int)e);
		}
		const cudaError_t e = cudaStreamSynchronize(l.stream);
		if (e != cudaSuccess) err.store((int)e);
	};
	std::vector<std::thread> th;
	for (int t = 1; t < want; t++) th.emplace_back(work, t);
	work(0);
	for (auto &x : th) x.join();
	if (err.load() != (int)cudaSuccess)
		return fail(ctx, std::string("gscan: staging host memory: ") + cudaGetErrorString((cudaError_t)err.load()));
	if (io_errno.load())
		return fail(ctx, std::string("gscan: reading a descriptor unit: ") + (io_errno.load() < 0 ? "file shorter than the unit" : strerror(io_errno.load())));
	return 0;
}

extern "C" int gscan_batch_create(gscan_ctx *ctx, const gscan_unit *units, size_t n_units, gscan_batch **out)
{
	return batch_create(ctx, units, n_units, false, out);
}

static int batch_create(gscan_ctx *ctx, const gscan_unit *units, size_t n_units, bool pooled, gscan_batch **out)
{
	if (!ctx || !out || (n_units && !units)) return fail(ctx, "gscan_batch_create: null argument");
	*out = nullptr;
	CK(ctx, cudaSetDevice(ctx->device));
	gscan_batch *b = new (std::nothrow) gscan_batch;
	if (!b) return fail(ctx, "gscan_batch_create: out of memory");
	b->pooled = pooled;
	struct Guard { gscan_ctx *c; gscan_batch *b; ~Guard() { if (b) gscan_batch_free(c, b); } } guard{ctx, b};

	// pass 1: validate, size the staging arena
	uint64_t arena_bytes = 0, n_tiles64 = 0;
	std::vector<uint64_t> arena_off(n_units, 0);
	{ // tile size: the power of two next to the average unit length, 4 KiB .. 64 KiB (many small files: no empty slices)
		uint64_t total = 0, live = 0;
		for (size_t i = 0; i < n_units; i++) if (units[i].len) { total += units[i].len; live++; }
		const uint64_t avg = live ? (total + live - 1) / live : 0;
		uint32_t sh = kMinTileShift;
		while (sh < (uint32_t)kMaxTileShift && (1ull << sh) < avg) sh++;
		if (const char *e = getenv("GSCAN_TILE_SHIFT")) { // tests: every tile size against the oracle
			const int v = atoi(e);
			if (v >= kMinTileShift && v <= kMaxTileShift) sh = (uint32_t)v;
		}
		b->tile_shift = sh;
	}
	const uint64_t tile_bytes = 1ull << b->tile_shift;
	for (size_t i = 0; i < n_units; i++) {
		const gscan_unit &u = units[i];
		if (u.len == 0) continue;
		if (u.len > (1ull << 31)) return fail(ctx, "gscan_batch_create: unit longer than 2 GiB (the reference's chunks are <= 1 GiB, grab.h:48)");
		if (!u.ptr && !(u.flags & GSCAN_UNIT_FD)) return fail(ctx, "gscan_batch_create: unit with null pointer");
		if ((u.flags & GSCAN_UNIT_FD) && ((u.flags & GSCAN_UNIT_DEVICE) || (intptr_t)u.ptr < 0 || (intptr_t)u.ptr > 0x7fffffff))
			return fail(ctx, "gscan_batch_create: descriptor unit with a bad descriptor");
		if (u.flags & GSCAN_UNIT_DEVICE) {
			if ((uintptr_t)u.ptr & 15u) return fail(ctx, "gscan_batch_create: device unit pointer must be 16-byte aligned");
		} else {
			arena_off[i] = arena_bytes;
			arena_bytes += (u.len + 255u) & ~255ull;
		}
		n_tiles64 += (u.len + tile_bytes - 1) >> b->tile_shift;
	}
	if ((n_tiles64 << (b->tile_shift - 9)) >= (1ull << 32)) return fail(ctx, "gscan_batch_create: batch too large (2 TiB of tiles or more)");
	if (arena_bytes) {
		if (pooled) { CK(ctx, ctx->pool_arena.ensure(arena_bytes + 256)); b->d_arena = ctx->pool_arena.p; }
		else CK(ctx, cudaMalloc(&b->d_arena, arena_bytes + 256));
	}

	// pass 2: stage host units, build tile and unit tables
	std::vector<TileDesc> tiles;
	std::vector<DevUnit> dunits;
	tiles.reserve((size_t)n_tiles64);
	auto t0 = std::chrono::steady_clock::now();
	std::vector<StagePiece> jobs;
	const uint8_t *run_src = nullptr;
	uint8_t *run_dst = nullptr;
	size_t run_len = 0;
	const uint8_t *prev_pinned_end = nullptr;
	for (size_t i = 0; i < n_units; i++) {
		const gscan_unit &u = units[i];
		if (u.len == 0) continue;
		const uint8_t *dptr;
		if (u.flags & GSCAN_UNIT_DEVICE) {
			dptr = u.ptr;
		} else {
			uint8_t *dst = b->d_arena + arena_off[i];
			dptr = dst;
			// pinned (page-locked) host memory can be copied from directly.  A unit that starts where the previous
			// pinned unit ended is taken to be pinned too (one driver query per contiguous run, not per unit; a
			// wrong guess only costs speed: cudaMemcpyAsync stages pageable memory itself)
			bool pinned;
			if (u.flags & GSCAN_UNIT_FD) {
				pinned = false;
			} else if (prev_pinned_end && u.ptr == prev_pinned_end) {
				pinned = true;
			} else {
				cudaPointerAttributes attr;
				pinned = cudaPointerGetAttributes(&attr, u.ptr) == cudaSuccess && attr.type == cudaMemoryTypeHost;
				cudaGetLastError();
			}
			prev_pinned_end = pinned ? u.ptr + u.len : nullptr;
			if (pinned) {
				// host units that are contiguous in memory (and 256-byte multiples, so contiguous in the arena too) go as one copy
				if (run_len && run_src + run_len == u.ptr && run_dst + run_len == dst && run_len < ((size_t)1 << 30)) {
					run_len += u.len;
				} else {
					if (run_len) CK(ctx, cudaMemcpyAsync(run_dst, run_src, run_len, cudaMemcpyHostToDevice, ctx->stream));
					run_src = u.ptr; run_dst = dst; run_len = u.len;
				}
			} else {
				// pageable memory (the reference's mmap windows): staged after this loop by the helper lanes
				const bool is_fd = (u.flags & GSCAN_UNIT_FD) != 0;
				for (uint64_t o = 0; o < u.len; o += kStageChunk)
					jobs.push_back(StagePiece{is_fd ? nullptr : u.ptr + o, dst + o, (size_t)std::min<uint64_t>(kStageChunk, u.len - o),
					                          is_fd ? (int)(intptr_t)u.ptr : -1, u.base_off + o});
			}
		}
		DevUnit du;
		du.ptr = (uint64_t)(uintptr_t)dptr;
		du.base_off = u.base_off;
		du.len = (uint32_t)u.len;
		du.first_tile = (uint32_t)tiles.size();
		du.file_id = u.file_id;
		du.pad = 0;
		const uint32_t unit_index = (uint32_t)dunits.size();
		dunits.push_back(du);
		for (uint64_t off = 0; off < u.len; off += tile_bytes) {
			TileDesc t;
			t.src = du.ptr + off;
			t.unit = unit_index;
			t.off = (uint32_t)off;
			t.len = (uint32_t)std::min<uint64_t>(tile_bytes, u.len - off);
			t.ulen = (uint32_t)u.len;
			t.pad[0] = t.pad[1] = 0;
			tiles.push_back(t);
		}
		b->bytes += u.len;
	}
	if (run_len) CK(ctx, cudaMemcpyAsync(run_dst, run_src, run_len, cudaMemcpyHostToDevice, ctx->stream));
	if (!jobs.empty() && stage_pageable(ctx, jobs) < 0) return -1;
	b->n_tiles = (uint32_t)tiles.size();
	b->n_units = (uint32_t)dunits.size();
	if (!tiles.empty()) {
		if (pooled) {
			CK(ctx, ctx->pool_tiles.ensure(tiles.size()));
			CK(ctx, ctx->pool_units.ensure(dunits.size()));
			b->d_tiles = ctx->pool_tiles.p;
			b->d_units = ctx->pool_units.p;
		} else {
			CK(ctx, cudaMalloc(&b->d_tiles, tiles.size() * sizeof(TileDesc)));
			CK(ctx, cudaMalloc(&b->d_units, dunits.size() * sizeof(DevUnit)));
		}
		CK(ctx, cudaMemcpyAsync(b->d_tiles, tiles.data(), tiles.size() * sizeof(TileDesc), cudaMemcpyHostToDevice, ctx->stream));
		CK(ctx, cudaMemcpyAsync(b->d_units, dunits.data(), dunits.size() * sizeof(DevUnit), cudaMemcpyHostToDevice, ctx->stream));
	}
	CK(ctx, cudaStreamSynchronize(ctx->stream)); // host buffers are consumed when this returns (grab.cc:215)
	b->h2d_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
	guard.b = nullptr;
	*out = b;
	return 0;
}

// the segment table is never cleared between scans: entries carry a 16-bit generation tag.  It is zeroed (with
// plain stores) when it is (re)allocated and when the tag wraps.
static int ensure_segs(gscan_ctx *ctx, uint32_t n_segs)
{
	const size_t before = ctx->segs.cap;
	CK(ctx, ctx->segs.ensure(n_segs));
	if (ctx->segs.cap != before || ctx->seg_tag >= 0xfffeu) {
		CK(ctx, launch_fill_u32(reinterpret_cast<uint32_t *>(ctx->segs.p), ctx->segs.cap * 2, 0u, ctx->stream));
		ctx->seg_tag = 0;
	}
	ctx->seg_tag++;
	return 0;
}

static int ensure_pattern(gscan_ctx *ctx, const gscan_pattern *pat)
{
	if (ctx->pat_id == pat->prog.id) return 0;
	if (pat->prog.kind == ENGINE_FIXED && !pat->prog.vm_dense) {
		const size_t b_len = (pat->seq_len.size() * 2 + 15) & ~(size_t)15;
		const size_t b_off = pat->seq_off.size() * 4, b_pos = pat->seq_pos.size() * 4, b_bm = pat->cls_bm.size() * 4;
		const size_t total = b_len + b_off + b_pos + b_bm + 64;
		CK(ctx, ctx->pat_tables.ensure(total));
		uint8_t *d = ctx->pat_tables.p;
		CK(ctx, cudaMemcpyAsync(d, pat->seq_len.data(), pat->seq_len.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
		CK(ctx, cudaMemcpyAsync(d + b_len, pat->seq_off.data(), b_off, cudaMemcpyHostToDevice, ctx->stream));
		CK(ctx, cudaMemcpyAsync(d + b_len + b_off, pat->seq_pos.data(), b_pos, cudaMemcpyHostToDevice, ctx->stream));
		if (b_bm) CK(ctx, cudaMemcpyAsync(d + b_len + b_off + b_pos, pat->cls_bm.data(), b_bm, cudaMemcpyHostToDevice, ctx->stream));
		CK(ctx, cudaStreamSynchronize(ctx->stream)); // the host vectors may die with the pattern
		ctx->pat_fixed = pat->fixed;
		ctx->pat_fixed.seq_len = reinterpret_cast<const uint16_t *>(d);
		ctx->pat_fixed.seq_off = reinterpret_cast<const uint32_t *>(d + b_len);
		ctx->pat_fixed.seq_pos = reinterpret_cast<const uint32_t *>(d + b_len + b_off);
		ctx->pat_fixed.cls_bm = reinterpret_cast<const uint32_t *>(d + b_len + b_off + b_pos);
		if (pat->prog.use_hash) {
			const Program &pr = pat->prog;
			const size_t nt = pr.hash_table.size() * 4, ns = pr.slot_seqs.size() * 4;
			const size_t ns16 = (ns + 15) & ~(size_t)15; // the tail table behind it is read as uint4
			CK(ctx, ctx->hash_tables.ensure(3 * nt + ns16 + 4 * nt + 64));
			uint8_t *h = ctx->hash_tables.p;
			std::vector<uint32_t> hashed(pr.hash_table.size()); // the device table holds the hash of the slot's key
			for (size_t i = 0; i < hashed.size(); i++)
				hashed[i] = pr.hash_table[i] == 0xffffffffu ? 0xffffffffu : pr.hash_table[i] * pat->hash.mulsh;
			CK(ctx, cudaMemcpyAsync(h, hashed.data(), nt, cudaMemcpyHostToDevice, ctx->stream));
			CK(ctx, cudaMemcpyAsync(h + nt, pr.slot_first.data(), nt, cudaMemcpyHostToDevice, ctx->stream));
			CK(ctx, cudaMemcpyAsync(h + 2 * nt, pr.slot_count.data(), nt, cudaMemcpyHostToDevice, ctx->stream));
			if (ns) CK(ctx, cudaMemcpyAsync(h + 3 * nt, pr.slot_seqs.data(), ns, cudaMemcpyHostToDevice, ctx->stream));
			// tail table: what the 7 bytes at a key position must look like for ANY alternative of the key to match -- byte i is
			// pinned when every alternative of the slot has an exact byte there and they agree (i below their shortest length)
			std::vector<uint32_t> tail(pr.hash_table.size() * 4, 0u);
			for (size_t sl = 0; sl < pr.hash_table.size(); sl++) {
				if (pr.hash_table[sl] == 0xffffffffu || pr.slot_count[sl] == 0) continue;
				uint64_t mask = 0, val = 0;
				for (int i = 0; i < 7; i++) { // byte 7 is never pinned: its val byte carries the length flag below
					int byte = -1;
					bool pinned = true;
					for (uint32_t k = 0; k < pr.slot_count[sl] && pinned; k++) {
						const Sequence &sq = pr.seqs[pr.slot_seqs[pr.slot_first[sl] + k]];
						if ((size_t)i >= sq.size() || sq[i].count() != 1) { pinned = false; break; }
						int b = 0;
						while (!sq[i].has((unsigned)b)) b++;
						if (byte >= 0 && byte != b) pinned = false;
						byte = b;
					}
					if (pinned && byte >= 0) { mask |= 0xffull << (8 * i); val |= (uint64_t)byte << (8 * i); }
				}
				// the slot's only alternative, all literal, at most 7 bytes: the entry is the whole verification; byte 7 of val
				// (never compared: its mask byte is 0) then carries the length
				if (pr.slot_count[sl] == 1) {
					const Sequence &sq = pr.seqs[pr.slot_seqs[pr.slot_first[sl]]];
					bool lit = sq.size() <= 7;
					for (size_t i = 0; lit && i < sq.size(); i++) lit = sq[i].count() == 1;
					if (lit) val |= (uint64_t)sq.size() << 56;
				}
				tail[4 * sl + 0] = (uint32_t)mask; tail[4 * sl + 1] = (uint32_t)val;
				tail[4 * sl + 2] = (uint32_t)(mask >> 32); tail[4 * sl + 3] = (uint32_t)(val >> 32);
			}
			CK(ctx, cudaMemcpyAsync(h + 3 * nt + ns16, tail.data(), 4 * nt, cudaMemcpyHostToDevice, ctx->stream));
			CK(ctx, cudaStreamSynchronize(ctx->stream));
			ctx->pat_hash = pat->hash;
			ctx->pat_hash.tail = reinterpret_cast<const uint4 *>(h + 3 * nt + ns16);
			ctx->pat_hash.table = reinterpret_cast<const uint32_t *>(h);
			ctx->pat_hash.slot_first = reinterpret_cast<const uint32_t *>(h + nt);
			ctx->pat_hash.slot_count = reinterpret_cast<const uint32_t *>(h + 2 * nt);
			ctx->pat_hash.slot_seqs = reinterpret_cast<const uint32_t *>(h + 3 * nt);
			ctx->pat_hash.seq_len = ctx->pat_fixed.seq_len;
			ctx->pat_hash.seq_off = ctx->pat_fixed.seq_off;
			ctx->pat_hash.seq_pos = ctx->pat_fixed.seq_pos;
			ctx->pat_hash.cls_bm = ctx->pat_fixed.cls_bm;
		}
	}
	if (pat->prog.use_vm) { // general patterns (either scan engine): VM program and byte classes
		const size_t nc = pat->prog.vm_code.size() * 4, nsb = pat->prog.vm_sets.size() * 4;
		CK(ctx, ctx->vm_tables.ensure(nc + nsb + 64));
		CK(ctx, cudaMemcpyAsync(ctx->vm_tables.p, pat->prog.vm_code.data(), nc, cudaMemcpyHostToDevice, ctx->stream));
		CK(ctx, cudaMemcpyAsync(ctx->vm_tables.p + nc, pat->prog.vm_sets.data(), nsb, cudaMemcpyHostToDevice, ctx->stream));
		CK(ctx, cudaStreamSynchronize(ctx->stream));
		ctx->vm_code = reinterpret_cast<const uint32_t *>(ctx->vm_tables.p);
		ctx->vm_sets = reinterpret_cast<const uint32_t *>(ctx->vm_tables.p + nc);
	}
	ctx->pat_id = pat->prog.id;
	return 0;
}

extern "C" int gscan_batch_scan(gscan_ctx *ctx, const gscan_pattern *pat, gscan_batch *b, uint32_t mode,
                                gscan_match **out, size_t *n_out)
{
	if (!ctx || !pat || !b || !out || !n_out) return fail(ctx, "gscan_batch_scan: null argument");
	if (mode > GSCAN_MODE_LINE) return fail(ctx, "gscan_batch_scan: bad mode");
	*out = nullptr;
	*n_out = 0;
	auto t0 = std::chrono::steady_clock::now();
	CK(ctx, cudaSetDevice(ctx->device));
	gscan_stats &S = ctx->stats;
	memset(&S, 0, sizeof(S));
	S.bytes_scanned = b->bytes;
	S.n_units = b->n_units;
	S.n_tiles = b->n_tiles;
	S.h2d_ms = b->h2d_ms;
	if (pat->prog.kind == ENGINE_NONE || b->n_tiles == 0) {
		S.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
		return 0;
	}
	if (ensure_pattern(ctx, pat) < 0) return -1;

	const bool hashed = pat->prog.kind == ENGINE_FIXED && pat->prog.use_hash;
	const uint32_t table_bytes = hashed ? pat->prog.hash_slots * 4u * hash_table_copies(pat->prog.hash_slots) : 0u;
	const bool fixedb = pat->prog.kind == ENGINE_FIXED && !hashed && pat->fixed.b_engine;
	const ScanGeom geom = scan_geom(hashed ? 4 : (fixedb ? 5 : (int)pat->prog.kind), pat->prog.kind == ENGINE_FIXED ? (uint32_t)pat->prog.tests.size() : 99u);
	uint32_t spt_shift = b->tile_shift;
	for (int sl = geom.slice; sl > 1; sl >>= 1) spt_shift--; // log2(tile bytes / slice bytes)
	const uint32_t n_segs = b->n_tiles << spt_shift;
	const int grid = (int)std::min<uint32_t>((uint32_t)ctx->num_sms, b->n_tiles);
	if (ensure_segs(ctx, n_segs) < 0) return -1;
	CK(ctx, ctx->scratch.ensure((size_t)ctx->num_sms * geom.warps * geom.slice));
	CK(ctx, ctx->cursor.ensure(2));
	CK(ctx, ctx->readback.ensure(64));
	{ // candidate buffer: sized to the batch (1 per 2 KiB, 1 Mi .. 64 Mi entries); grown on demand by the retry loop below
		const size_t want = std::min<size_t>(std::max<size_t>(b->bytes / 2048, 1u << 20), 64u << 20);
		if (ctx->cand.cap < want) CK(ctx, ctx->cand.ensure(want));
	}

	ScanArgs A;
	A.tiles = b->d_tiles;
	A.n_tiles = b->n_tiles;
	A.cursor = ctx->cursor.p;
	A.segs = ctx->segs.p;
	A.scratch = ctx->scratch.p;
	A.extra_smem = table_bytes;
	A.spt_shift = spt_shift;
	A.tag = ctx->seg_tag;

	unsigned long long *h_cursor = reinterpret_cast<unsigned long long *>(ctx->readback.p);
	unsigned long long total_cand = 0;
	// general patterns without a candidate filter: no scan kernel -- the VM walk tries the positions itself
	const bool dense = pat->prog.use_vm && pat->prog.vm_dense;
	if (dense) {
		CK(ctx, launch_fill_u32(reinterpret_cast<uint32_t *>(ctx->cursor.p), 8, 0u, ctx->stream));
		CK(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
		S.total_launches += 1;
	}
	for (int attempt = 0; !dense; attempt++) {
		A.cand = ctx->cand.p;
		A.cand_cap = (uint32_t)std::min<size_t>(ctx->cand.cap, 0xffffffffu);
		// a warp reserves candidate slots a chunk at a time; all warps' unused tails together stay below an eighth of the buffer
		A.chunk = (uint32_t)std::min<size_t>(std::max<size_t>(A.cand_cap / ((size_t)8 * (size_t)grid * (size_t)geom.warps), 32), 1024);
		CK(ctx, launch_fill_u32(reinterpret_cast<uint32_t *>(ctx->cursor.p), 8, 0u, ctx->stream));
		CK(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
		if (hashed) CK(ctx, launch_scan_hash(A, ctx->pat_hash, grid, ctx->stream));
		else if (pat->prog.kind == ENGINE_FIXED) CK(ctx, launch_scan_fixed(A, ctx->pat_fixed, pat->prog.delta, geom, grid, ctx->stream));
		else CK(ctx, launch_scan_run(A, pat->run, geom, grid, ctx->stream));
		CK(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
		CK(ctx, cudaMemcpyAsync(h_cursor, ctx->cursor.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
		CK(ctx, cudaStreamSynchronize(ctx->stream));
		float ms = 0;
		cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
		S.scan_kernel_ms += ms;
		S.scan_launches++;
		S.total_launches += 2; // cursor fill + scan kernel
		total_cand = *h_cursor;
		if (total_cand <= A.cand_cap) break;
		// candidate buffer too small: never truncate -- grow to what the kernel asked for and re-scan
		if (attempt >= 2 || total_cand >= 0xffffffffull)
			return fail(ctx, "gscan_batch_scan: candidate buffer overflow (pattern matches almost everywhere); split the batch");
		CK(ctx, ctx->cand.ensure((size_t)(total_cand + total_cand / 8 + 1024)));
	}
	S.n_candidates = total_cand; // slots reserved; replaced by the exact count once the segments are summed

	size_t n = 0;
	gscan_match *m = nullptr;
	static_assert(sizeof(FinalRec) == sizeof(gscan_match), "device records are gscan_match");
	if (total_cand || dense) {
		const uint32_t nb_seg = (n_segs + 2047) / 2048, nb_u = (uint32_t)((b->n_units + 2047) / 2048);
		CK(ctx, ctx->ord.ensure((size_t)total_cand));
		CK(ctx, ctx->unit_start.ensure((size_t)b->n_units + 1));
		CK(ctx, ctx->unit_out.ensure((size_t)b->n_units + 1));
		CK(ctx, ctx->blk.ensure((size_t)nb_seg + nb_u + (size_t)(total_cand / 2048 + 2) + 8));
		ResolveArgs R;
		R.tiles = b->d_tiles;
		R.segs = ctx->segs.p;
		R.n_segs = n_segs;
		R.spt_shift = spt_shift;
		R.tag = ctx->seg_tag;
		R.cand = ctx->cand.p;
		R.units = b->d_units;
		R.n_units = b->n_units;
		R.ord = ctx->ord.p;
		R.out = nullptr;
		R.unit_start = ctx->unit_start.p;
		R.unit_out = ctx->unit_out.p;
		R.blk = ctx->blk.p;
		R.totals = reinterpret_cast<uint32_t *>(ctx->cursor.p + 1);
		R.mode = mode;
		R.minlen = (uint32_t)pat->prog.minlen;
		R.engine = pat->prog.use_vm ? (uint32_t)GSCAN_ENGINE_VM : (uint32_t)pat->prog.kind;
		R.vm_code = ctx->vm_code;
		R.vm_sets = ctx->vm_sets;
		R.vm_runstart = pat->prog.vm_runstart ? 1u : 0u;
		R.flat = (mode == GSCAN_MODE_ALL && !pat->prog.use_vm && (pat->prog.kind == ENGINE_RUN || pat->prog.disjoint)) ? 1u : 0u;
		// chain path: FIXED patterns whose replay is sequential (overlapping matches, or LINE mode) with many candidates per
		// unit -- one thread per unit would walk them alone (a 1 GiB window of a log file with a million hits: seconds)
		R.chain = 0; R.chain_levels = 0; R.chain_cap = 0; R.chain_buf = nullptr;
		R.vm_par = 0; R.vm_ord = nullptr; R.vm_unit_start = nullptr; R.vm_flag = nullptr; R.vm_budget = nullptr;
		{
			// general patterns take the same path when their attempts do not depend on the search start (vm_start_free) and
			// the candidates come from a leading-sequence filter: one VM attempt per candidate, all at once, then the chain
			// over the candidates that matched (any mode) -- instead of one thread replaying a huge unit's attempts alone
			// RUN in LINE mode too: the search resumes behind a line remainder, possibly inside a run (chain_entry)
			const bool fixed_ok = !pat->prog.use_vm && ((pat->prog.kind == ENGINE_FIXED && (mode == GSCAN_MODE_ALL || mode == GSCAN_MODE_LINE)) ||
			                                            (pat->prog.kind == ENGINE_RUN && mode == GSCAN_MODE_LINE));
			const bool vm_ok = pat->prog.use_vm && !pat->prog.vm_runstart && pat->prog.vm_start_free;
			const bool eligible = !R.flat && !dense && (fixed_ok || vm_ok) && total_cand > 0;
			bool want = eligible && total_cand >= 65536 && total_cand / std::max<uint64_t>(b->n_units, 1) >= 1024;
			if (const char *e = getenv("GSCAN_CHAIN")) // tests: force the path on small inputs / switch it off
				want = eligible && *e == '1';
			uint32_t levels = 2; // at least two tables: the second one doubles as the RUN entry positions
			while ((1ull << levels) < total_cand) levels++;
			if (want && (uint64_t)(levels + 2) * total_cand * 4 <= (4ull << 30)) {
				CK(ctx, ctx->chain.ensure((size_t)(levels + 2) * (size_t)total_cand));
				R.chain = 1; R.chain_levels = levels; R.chain_cap = (uint32_t)total_cand; R.chain_buf = ctx->chain.p;
				if (vm_ok) {
					CK(ctx, ctx->vm_ord.ensure((size_t)total_cand));
					CK(ctx, ctx->vm_flag.ensure((size_t)total_cand));
					CK(ctx, ctx->vm_unit_start.ensure((size_t)b->n_units + 1));
					CK(ctx, ctx->vm_budget.ensure((size_t)b->n_units));
					R.vm_budget = ctx->vm_budget.p;
					R.vm_par = 1; R.vm_ord = ctx->vm_ord.p; R.vm_flag = ctx->vm_flag.p; R.vm_unit_start = ctx->vm_unit_start.p;
				}
			}
		}
		R.run_min = (uint32_t)pat->prog.run_min;
		for (int i = 0; i < 8; i++) R.bitmap[i] = dense ? pat->prog.first_set.w[i] : pat->prog.run_class.w[i];
		R.vm_dense = dense ? 1u : 0u;
		R.total_cand = (uint32_t)total_cand;
		R.vm_ready = 0; R.dense_blocks = 0; R.dense_tile_shift = b->tile_shift;
		uint32_t nl = 0;
		uint32_t *h_tot = reinterpret_cast<uint32_t *>((uint8_t *)ctx->readback.p + 16);
		bool resolved_empty = false;
		if (dense && pat->prog.vm_start_free) {
			// dense general pattern, big units: the attempts of all positions in parallel (k_vm_dense, twice: count / write), then
			// the chain over the matching positions -- one thread per unit would walk a 1 GiB window for minutes
			const uint64_t blocks = (uint64_t)b->n_tiles << (b->tile_shift - 6);
			bool want = b->bytes / std::max<uint64_t>(b->n_units, 1) >= (1u << 20);
			if (const char *e = getenv("GSCAN_CHAIN")) want = *e == '1'; // tests: force the path on small inputs / switch it off
			if (want && b->bytes <= (4ull << 30) && blocks < (1ull << 31)) {
				const uint32_t nb_u = (uint32_t)((b->n_units + 2047) / 2048);
				CK(ctx, ctx->vm_flag.ensure((size_t)blocks + 1));
				CK(ctx, ctx->vm_budget.ensure((size_t)b->n_units));
				CK(ctx, ctx->vm_unit_start.ensure((size_t)b->n_units + 1));
				CK(ctx, ctx->blk.ensure((size_t)(blocks / 2048 + 2) + nb_u + 16));
				R.blk = ctx->blk.p;
				R.dense_blocks = (uint32_t)blocks;
				R.vm_flag = ctx->vm_flag.p; R.vm_budget = ctx->vm_budget.p; R.vm_unit_start = ctx->vm_unit_start.p;
				CK(ctx, launch_vm_dense_count(R, ctx->stream, &nl));
				S.total_launches += nl;
				uint32_t *h8 = reinterpret_cast<uint32_t *>((uint8_t *)ctx->readback.p + 32);
				CK(ctx, cudaMemcpyAsync(h8, R.totals, 32, cudaMemcpyDeviceToHost, ctx->stream));
				CK(ctx, cudaStreamSynchronize(ctx->stream));
				const uint64_t hits = h8[4];
				uint32_t levels = 2;
				while ((1ull << levels) < hits) levels++;
				if (hits == 0) {
					h_tot[0] = 0; h_tot[1] = 0; h_tot[2] = h8[2];
					resolved_empty = true;
				} else if ((uint64_t)(levels + 2) * hits * 4 <= (4ull << 30)) {
					CK(ctx, ctx->vm_ord.ensure((size_t)hits));
					CK(ctx, ctx->chain.ensure((size_t)(levels + 2) * (size_t)hits));
					CK(ctx, ctx->blk.ensure((size_t)(blocks / 2048 + 2) + nb_u + (size_t)(hits / 2048 + 2) + 16));
					R.blk = ctx->blk.p;
					R.vm_ord = ctx->vm_ord.p;
					CK(ctx, launch_vm_dense_write(R, ctx->stream, &nl));
					S.total_launches += nl;
					R.vm_par = 1; R.vm_ready = 1; R.vm_dense = 0;
					R.chain = 1; R.chain_levels = levels; R.chain_cap = (uint32_t)hits; R.chain_buf = ctx->chain.p;
					R.total_cand = (uint32_t)hits;
					S.n_candidates = hits; // positions where an attempt matched
				} // else: more matching positions than the chain tables may hold -- the per-unit walk below serves the batch
			}
		}
		if (!resolved_empty) {
			CK(ctx, launch_resolve_count(R, ctx->stream, &nl));
			S.total_launches += nl;
			CK(ctx, cudaMemcpyAsync(h_tot, R.totals, 12, cudaMemcpyDeviceToHost, ctx->stream));
			CK(ctx, cudaStreamSynchronize(ctx->stream));
		}
		// a unit on which the backtracking VM ran out of stack or steps stops there, like the reference's loop when
		// pcre_exec reports a match-limit error (rc < 0 => break, grab.cc:179, quirk Q5); the other units are unaffected
		S.vm_limit_hit = h_tot[2] ? 1u : 0u;
		if (!dense && h_tot[0] > (uint32_t)total_cand) return fail(ctx, "gscan_batch_scan: internal: more candidates in the segments than slots reserved");
		if (!dense) { S.n_candidates = h_tot[0]; R.total_cand = h_tot[0]; }
		n = h_tot[1];
		if (n) {
			// the records are written on the device in their final form and land in a pinned buffer that is lent
			// to the caller until gscan_free_matches()
			gscan_ctx::ResultBuf *rb = nullptr;
			for (auto &x : ctx->results) if (!x.lent && (!rb || x.cap > rb->cap)) rb = &x;
			if (!rb) { ctx->results.push_back(gscan_ctx::ResultBuf{nullptr, 0, false}); rb = &ctx->results.back(); }
			if (rb->cap < n * sizeof(gscan_match)) {
				if (rb->p) cudaFreeHost(rb->p);
				rb->p = nullptr;
				rb->cap = 0;
				const size_t want = std::max<size_t>(n * sizeof(gscan_match) * 5 / 4, (size_t)1 << 16);
				CK(ctx, cudaHostAlloc(&rb->p, want, cudaHostAllocDefault));
				rb->cap = want;
			}
			CK(ctx, ctx->out.ensure(n));
			R.out = ctx->out.p;
			CK(ctx, launch_resolve_write(R, ctx->stream, &nl));
			S.total_launches += nl;
			CK(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
			CK(ctx, cudaMemcpyAsync(rb->p, ctx->out.p, n * sizeof(FinalRec), cudaMemcpyDeviceToHost, ctx->stream));
			rb->lent = true;
			m = static_cast<gscan_match *>(rb->p);
		} else {
			CK(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
		}
		CK(ctx, cudaStreamSynchronize(ctx->stream));
		float ms = 0;
		cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]);
		S.resolve_ms = ms;
	}
	*out = m;
	*n_out = n;
	S.n_matches = n;
	S.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
	return 0;
}

extern "C" int gscan_scan_batch(gscan_ctx *ctx, const gscan_pattern *pat, const gscan_unit *units, size_t n_units,
                                uint32_t mode, gscan_match **out, size_t *n_out)
{
	if (!ctx || !pat || !out || !n_out) return fail(ctx, "gscan_scan_batch: null argument");
	auto t0 = std::chrono::steady_clock::now();
	gscan_batch *b = nullptr;
	if (batch_create(ctx, units, n_units, true, &b) < 0) return -1;
	int rc = gscan_batch_scan(ctx, pat, b, mode, out, n_out);
	gscan_batch_free(ctx, b);
	ctx->stats.total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
	return rc;
}

extern "C" int gscan_last_device_matches(gscan_ctx *ctx, const gscan_match **dptr, size_t *n)
{
	if (!ctx || !dptr || !n) return fail(ctx, "gscan_last_device_matches: null argument");
	*n = (size_t)ctx->stats.n_matches;
	*dptr = *n ? reinterpret_cast<const gscan_match *>(ctx->out.p) : nullptr;
	return 0;
}

extern "C" int gscan_scan_batch_async(gscan_ctx *ctx, const gscan_pattern *pat, const gscan_unit *units, size_t n_units, uint32_t mode)
{
	if (!ctx || !pat) return fail(ctx, "gscan_scan_batch_async: null argument");
	if (ctx->job_active) return fail(ctx, "gscan_scan_batch_async: a job is already in flight on this context (call gscan_scan_wait)");
	ctx->job_rc = 0;
	ctx->job_out = nullptr;
	ctx->job_n = 0;
	try {
		ctx->job = std::thread([ctx, pat, units, n_units, mode] {
			ctx->job_rc = gscan_scan_batch(ctx, pat, units, n_units, mode, &ctx->job_out, &ctx->job_n);
		});
	} catch (const std::exception &e) {
		return fail(ctx, std::string("gscan_scan_batch_async: cannot start the worker: ") + e.what());
	}
	ctx->job_active = true;
	return 0;
}

extern "C" int gscan_scan_wait(gscan_ctx *ctx, gscan_match **out, size_t *n_out)
{
	if (!ctx || !out || !n_out) return fail(ctx, "gscan_scan_wait: null argument");
	if (!ctx->job_active) return fail(ctx, "gscan_scan_wait: no job in flight");
	ctx->job.join(); // the worker's writes (results, error text, statistics) happen-before this returns
	ctx->job_active = false;
	*out = ctx->job_out;
	*n_out = ctx->job_n;
	return ctx->job_rc;
}

extern "C" void gscan_free_matches(gscan_ctx *ctx, gscan_match *m)
{
	if (!ctx || !m) return;
	for (auto &rb : ctx->results) if (rb.p == m) rb.lent = false;
}

// ------------------------------------------------------------------------------------------
// utilities
// ------------------------------------------------------------------------------------------
extern "C" void *gscan_host_alloc(size_t bytes)
{
	void *p = nullptr;
	if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
	return p;
}
extern "C" void gscan_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" void *gscan_device_alloc(gscan_ctx *ctx, size_t bytes)
{
	if (!ctx) return nullptr;
	void *p = nullptr;
	if (cudaSetDevice(ctx->device) != cudaSuccess || cudaMalloc(&p, bytes) != cudaSuccess) {
		fail(ctx, std::string("gscan_device_alloc: ") + cudaGetErrorString(cudaGetLastError()));
		return nullptr;
	}
	return p;
}
extern "C" void gscan_device_free(gscan_ctx *ctx, void *d)
{
	if (ctx) cudaSetDevice(ctx->device);
	if (d) cudaFree(d);
}
extern "C" int gscan_memcpy_d2h(gscan_ctx *ctx, void *dst, const void *dsrc, size_t bytes)
{
	if (!ctx) return -1;
	CK(ctx, cudaSetDevice(ctx->device));
	CK(ctx, cudaMemcpyAsync(dst, dsrc, bytes, cudaMemcpyDeviceToHost, ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}
extern "C" int gscan_memcpy_h2d(gscan_ctx *ctx, void *ddst, const void *src, size_t bytes)
{
	if (!ctx) return -1;
	CK(ctx, cudaSetDevice(ctx->device));
	CK(ctx, cudaMemcpyAsync(ddst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

extern "C" int gscan_synth_corpus(gscan_ctx *ctx, void *dptr, uint64_t seed, uint64_t first_file_id, uint64_t n_files,
                                  uint64_t file_len, uint64_t stride, const uint8_t *needle, uint32_t needle_len,
                                  uint32_t needle_every)
{
	if (!ctx || !dptr) return fail(ctx, "gscan_synth_corpus: null argument");
	if ((file_len & 15u) || (stride & 15u) || ((uintptr_t)dptr & 15u)) return fail(ctx, "gscan_synth_corpus: lengths and pointer must be multiples of 16");
	CK(ctx, cudaSetDevice(ctx->device));
	const uint8_t *dn = nullptr;
	if (needle && needle_len && needle_every) {
		CK(ctx, ctx->needle.ensure(needle_len));
		CK(ctx, cudaMemcpyAsync(ctx->needle.p, needle, needle_len, cudaMemcpyHostToDevice, ctx->stream));
		dn = ctx->needle.p;
	}
	CK(ctx, launch_synth_corpus((uint8_t *)dptr, seed, first_file_id, n_files, file_len, stride, dn, needle_len, needle_every, ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	return 0;
}

extern "C" int gscan_tma_probe(gscan_ctx *ctx, gscan_batch *b, int geom, float *ms)
{
	if (!ctx || !b || !b->n_tiles) return fail(ctx, "gscan_tma_probe: null argument");
	CK(ctx, cudaSetDevice(ctx->device));
	const ScanGeom g = geom == 0 ? ScanGeom{GeomStream::kWarps, GeomStream::kRing, GeomStream::kSlice}
	                             : ScanGeom{GeomBalanced::kWarps, GeomBalanced::kRing, GeomBalanced::kSlice};
	uint32_t spt_shift = b->tile_shift;
	for (int sl = g.slice; sl > 1; sl >>= 1) spt_shift--;
	const uint32_t n_segs = b->n_tiles << spt_shift;
	if (ensure_segs(ctx, n_segs) < 0) return -1;
	CK(ctx, ctx->scratch.ensure((size_t)ctx->num_sms * g.warps * g.slice));
	CK(ctx, ctx->cursor.ensure(2));
	if (ctx->cand.cap == 0) CK(ctx, ctx->cand.ensure(1u << 20));
	ScanArgs A;
	A.tiles = b->d_tiles; A.n_tiles = b->n_tiles; A.cand = ctx->cand.p; A.cand_cap = (uint32_t)ctx->cand.cap;
	A.cursor = ctx->cursor.p; A.segs = ctx->segs.p; A.scratch = ctx->scratch.p; A.extra_smem = 0; A.tag = ctx->seg_tag; A.spt_shift = spt_shift; A.chunk = 64;
	CK(ctx, launch_fill_u32(reinterpret_cast<uint32_t *>(ctx->cursor.p), 8, 0u, ctx->stream));
	CK(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
	CK(ctx, launch_scan_null(A, geom, (int)std::min<uint32_t>((uint32_t)ctx->num_sms, b->n_tiles), ctx->stream));
	CK(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	float t = 0;
	cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[1]);
	if (ms) *ms = t;
	return 0;
}

extern "C" int gscan_read_probe(gscan_ctx *ctx, const void *dptr, uint64_t bytes, float *ms, uint64_t *checksum)
{
	if (!ctx || !dptr) return fail(ctx, "gscan_read_probe: null argument");
	CK(ctx, cudaSetDevice(ctx->device));
	CK(ctx, ctx->probe_sum.ensure(1));
	CK(ctx, cudaMemsetAsync(ctx->probe_sum.p, 0, 8, ctx->stream));
	CK(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
	CK(ctx, launch_read_probe(dptr, bytes, ctx->probe_sum.p, ctx->num_sms * 4, ctx->stream));
	CK(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
	unsigned long long h = 0;
	CK(ctx, cudaMemcpyAsync(&h, ctx->probe_sum.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	float t = 0;
	cudaEventElapsedTime(&t, ctx->ev[0], ctx->ev[1]);
	if (ms) *ms = t;
	if (checksum) *checksum = h;
	return 0;
}
