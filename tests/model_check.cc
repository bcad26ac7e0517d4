// model_check.cc -- CPU check of what the pattern compiler (grab_b200/csrc/pattern.cc) hands to the device, against
// the oracle: the compiled Program is interpreted on the host exactly as the resolve kernels interpret it -- FIXED:
// first sequence in preference order at the leftmost position; RUN: greedy class run of at least run_min; general
// patterns: the device VM, whose source is extracted verbatim from resolve_kernels.cu by tests/test_model.py
// (vm_snippet.inc) and compiled here for the host -- inside the reference's loop (moving search start, strict '<'
// guard, grab.cc:175-213).  Then the same with the device's own per-unit walk kernels (k_walk / k_walk_vm, same
// extraction) fed with the candidates the scan kernels deliver by contract, in all three modes (ALL / FIRST / LINE).  Also checks that the candidate filter of general patterns (leading-byte sequences / run
// starts) never rejects a position where the VM matches.
// Usage: model_check PATTERN_FILE   (one pattern per line)
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>

#include "../include/gscan.h"
#include "../grab_b200/csrc/pattern.h"
#include "../grab_b200/csrc/kernels.h" // ResolveArgs, DevUnit, FinalRec, OutRec (host-includable: PODs + launcher prototypes)
extern "C" {
#include "../oracle/grab_oracle.h"
}

// the extracted device source (VM + the per-unit walk kernels of resolve_kernels.cu) compiled for the host: CUDA's
// qualifiers vanish, the thread index is a global we set to the unit under test, atomicOr is a plain OR
#undef __device__
#undef __global__
#undef __forceinline__
#undef __launch_bounds__
#define __device__
#define __global__
#define __forceinline__ inline
#define __launch_bounds__(...)
namespace gscan {
struct ModelIdx { uint32_t x; };
static ModelIdx model_blockIdx{0}, model_blockDim{1}, model_threadIdx{0};
#define blockIdx model_blockIdx
#define blockDim model_blockDim
#define threadIdx model_threadIdx
static inline uint32_t atomicOr(uint32_t *p, uint32_t v) { const uint32_t o = *p; *p |= v; return o; }
static inline unsigned long long atomicAdd(unsigned long long *p, unsigned long long v) { const unsigned long long o = *p; *p += v; return o; }
#include "vm_snippet.inc"
#undef blockIdx
#undef blockDim
#undef threadIdx
} // namespace gscan

using namespace gscan;

static uint64_t rng_state = 0x1234567ull;
static uint32_t rnd() { rng_state ^= rng_state << 13; rng_state ^= rng_state >> 7; rng_state ^= rng_state << 17; return (uint32_t)(rng_state >> 9); }

struct M { uint64_t pos; uint32_t len; };

static bool seq_at(const Sequence &q, const uint8_t *s, size_t len, size_t pos)
{
	if (pos + q.size() > len) return false;
	for (size_t i = 0; i < q.size(); i++) if (!q[i].has(s[pos + i])) return false;
	return true;
}

// 0 ok, -1 VM limit, -2 filter soundness violated
static int emulate(const Program &p, const uint8_t *s, size_t len, std::vector<M> &out, std::string &why)
{
	ResolveArgs R;
	memset(&R, 0, sizeof R);
	R.vm_code = p.vm_code.data();
	R.vm_sets = p.vm_sets.data();
	size_t start = 0;
	while (start + (size_t)p.minlen < len) { // grab.cc:175
		bool found = false;
		size_t pos = start, mend = 0;
		VmBudget budget(len);
		for (; pos < len; pos++) {
			if (p.use_vm) {
				uint32_t e = 0;
				const int rc = vm_exec(R, s + start, (uint32_t)(len - start), (uint32_t)(pos - start), &e, budget);
				if (rc < 0) return -1;
				if (rc == 1) { found = true; mend = start + e; }
			} else if (p.kind == ENGINE_RUN) {
				size_t k = 0;
				while (pos + k < len && p.run_class.has(s[pos + k])) k++;
				if (k >= (size_t)p.run_min) { found = true; mend = pos + k; }
			} else {
				for (auto &q : p.seqs)
					if (seq_at(q, s, len, pos)) { found = true; mend = pos + q.size(); break; }
			}
			if (found) break;
		}
		if (!found) break;
		if (p.use_vm) { // the scan kernel (dense: the first-byte test of the walk) must have offered this position to the VM walk
			bool offered = false;
			if (p.vm_dense) offered = p.first_set.has(s[pos]);
			else if (p.vm_runstart) offered = p.run_class.has(s[pos]) && (pos == start || !p.run_class.has(s[pos - 1]));
			else for (auto &q : p.seqs) offered = offered || seq_at(q, s, len, pos);
			if (!offered) { why = "candidate filter rejects a matching position"; return -2; }
		}
		if (mend <= pos) { why = "empty match"; return -2; }
		out.push_back(M{pos, (uint32_t)(mend - pos)});
		start = mend;
	}
	return 0;
}

// What the scan kernels deliver for one unit, by contract (scan_kernels.cu): FIXED -- every position where an
// alternative (for general patterns: a leading-byte prefix) lies entirely inside the unit, with the length of the first
// one in preference order; RUN (and general patterns that begin with a class repeat) -- the first byte of every maximal
// class run of at least run_min bytes.  Position order.
static void candidates(const Program &p, const uint8_t *s, size_t len, std::vector<OutRec> &ord)
{
	const bool runs = p.kind == ENGINE_RUN || (p.use_vm && p.vm_runstart);
	for (size_t pos = 0; pos < len; pos++) {
		if (runs) {
			if (!p.run_class.has(s[pos]) || (pos > 0 && p.run_class.has(s[pos - 1]))) continue;
			size_t k = 0;
			while (pos + k < len && p.run_class.has(s[pos + k])) k++;
			if (k >= (size_t)p.run_min) ord.push_back(OutRec{0, (uint32_t)pos, 0, 0});
		} else {
			for (auto &q : p.seqs)
				if (seq_at(q, s, len, pos)) { ord.push_back(OutRec{0, (uint32_t)pos, (uint32_t)q.size(), 0}); break; }
		}
	}
}

static int g_flat_checks = 0, g_chain_checks = 0, g_vmpar_checks = 0, g_densepar_checks = 0;
// count pass, slot scan (one unit: slot 0), write pass -- the device code of resolve_kernels.cu, on the host.
// 0 ok, -1 VM limit
static int walk(const Program &p, const uint8_t *s, size_t len, uint32_t mode, std::vector<M> &out)
{
	std::vector<OutRec> ord;
	if (!(p.use_vm && p.vm_dense)) candidates(p, s, len, ord);
	DevUnit du;
	memset(&du, 0, sizeof du);
	du.ptr = (uint64_t)(uintptr_t)s;
	du.len = (uint32_t)len;
	uint32_t unit_start[2] = {0, (uint32_t)ord.size()}, unit_out[1] = {0}, totals[4] = {0, 0, 0, 0};
	ResolveArgs R;
	memset(&R, 0, sizeof R);
	R.units = &du;
	R.n_units = 1;
	R.ord = ord.empty() ? nullptr : ord.data();
	R.unit_start = unit_start;
	R.unit_out = unit_out;
	R.totals = totals;
	R.mode = mode;
	R.minlen = (uint32_t)p.minlen;
	R.engine = p.use_vm ? (uint32_t)GSCAN_ENGINE_VM : (uint32_t)p.kind;
	R.run_min = (uint32_t)p.run_min;
	for (int i = 0; i < 8; i++) R.bitmap[i] = (p.use_vm && p.vm_dense) ? p.first_set.w[i] : p.run_class.w[i];
	R.vm_code = p.vm_code.data();
	R.vm_sets = p.vm_sets.data();
	R.vm_runstart = p.vm_runstart ? 1u : 0u;
	R.vm_dense = (p.use_vm && p.vm_dense) ? 1u : 0u;
	model_threadIdx.x = 0;
	if (p.use_vm) k_walk_vm<false>(R); else k_walk<false>(R);
	if (totals[2]) return -1;
	std::vector<FinalRec> fin(unit_out[0] + 1);
	const uint32_t n = unit_out[0];
	unit_out[0] = 0;
	R.out = fin.data();
	if (p.use_vm) k_walk_vm<true>(R); else k_walk<true>(R);
	if (totals[2]) return -1;
	for (uint32_t i = 0; i < n; i++) out.push_back(M{fin[i].start, fin[i].len});
	// the flat write pass (one thread per candidate) wherever the engine would choose it: same records
	if (mode == GSCAN_MODE_ALL && !p.use_vm && (p.kind == ENGINE_RUN || p.disjoint)) {
		R.flat = 1;
		R.total_cand = (uint32_t)ord.size();
		R.out = nullptr;
		unit_out[0] = 0;
		model_threadIdx.x = 0;
		k_walk<false>(R);
		const uint32_t nf = unit_out[0];
		std::vector<FinalRec> ff(nf + 1);
		unit_out[0] = 0;
		R.out = ff.data();
		for (uint32_t i = 0; i < ord.size(); i++) { model_threadIdx.x = i; k_write_flat(R); }
		model_threadIdx.x = 0;
		bool same = nf == n;
		for (uint32_t i = 0; same && i < n; i++) same = ff[i].start == fin[i].start && ff[i].len == fin[i].len;
		if (!same) return -3;
		g_flat_checks++;
	}
	// the chain path (pointer doubling over the candidates) wherever it applies: same records as the serial replay
	if (!p.use_vm && ((p.kind == ENGINE_FIXED && (mode == GSCAN_MODE_ALL || mode == GSCAN_MODE_LINE)) || (p.kind == ENGINE_RUN && mode == GSCAN_MODE_LINE)) && !ord.empty()) {
		const uint32_t cap = (uint32_t)ord.size();
		uint32_t levels = 2;
		while ((1u << levels) < cap) levels++;
		std::vector<uint32_t> buf((size_t)(levels + 2) * cap, 0u);
		R.flat = 0;
		R.chain = 1; R.chain_levels = levels; R.chain_cap = cap; R.chain_buf = buf.data();
		totals[0] = cap;
		R.out = nullptr;
		auto each = [&](auto fn) { for (uint32_t i = 0; i < cap; i++) { model_threadIdx.x = i; fn(); } model_threadIdx.x = 0; };
		each([&] { k_chain_next(R); });
		for (uint32_t k = 1; k < levels; k++) each([&] { k_chain_double(R, k); });
		model_threadIdx.x = 0;
		k_chain_heads(R);
		for (uint32_t k = levels; k-- > 0;) each([&] { k_chain_spread(R, k); });
		if (p.kind == ENGINE_RUN) { each([&] { k_chain_entry_init(R); }); each([&] { k_chain_entry(R); }); }
		uint32_t *mark = buf.data() + (size_t)levels * cap, *rank = mark + cap;
		uint32_t acc = 0;
		for (uint32_t i = 0; i < cap; i++) { rank[i] = acc; acc += mark[i]; } // the device uses its block-scan kernels here
		k_chain_count(R);
		const uint32_t nc = unit_out[0];
		unit_out[0] = 0;
		std::vector<FinalRec> fc(nc + 1);
		R.out = fc.data();
		R.total_cand = cap;
		each([&] { k_chain_write(R); });
		bool same = nc == n;
		for (uint32_t i = 0; same && i < n; i++) same = fc[i].start == fin[i].start && fc[i].len == fin[i].len;
		if (!same) return -4;
		g_chain_checks++;
	}
	// general patterns on the chain path (vm_par): one attempt per candidate, compaction of the candidates that matched,
	// chain over those -- wherever the engine may choose it (start-free program, candidates from the leading-sequence
	// filter), in every mode: same records as the serial replay
	if (p.use_vm && !p.vm_dense && !p.vm_runstart && p.vm_start_free && !ord.empty()) {
		std::vector<OutRec> cand;
		candidates(p, s, len, cand); // fresh: the serial count pass above recorded its outcomes in ord
		const uint32_t cap = (uint32_t)cand.size();
		uint32_t levels = 2;
		while ((1u << levels) < cap) levels++;
		std::vector<uint32_t> buf((size_t)(levels + 2) * cap, 0u), flag(cap, 0u);
		std::vector<OutRec> vord(cap);
		uint32_t vus[2] = {0, 0}, us2[2] = {0, cap}, tot[8] = {cap, 0, 0, 0, 0, 0, 0, 0}, uo[1] = {0};
		ResolveArgs V = R;
		V.flat = 0;
		V.ord = cand.data(); V.unit_start = us2; V.unit_out = uo; V.totals = tot; V.out = nullptr; V.total_cand = cap;
		V.chain = 1; V.chain_levels = levels; V.chain_cap = cap; V.chain_buf = buf.data();
		unsigned long long vbud[1] = {0};
		V.vm_par = 1; V.vm_ord = vord.data(); V.vm_flag = flag.data(); V.vm_unit_start = vus; V.vm_budget = vbud;
		model_threadIdx.x = 0;
		k_vm_budget_init(V);
		const unsigned long long bud0 = vbud[0];
		auto each = [&](auto fn) { for (uint32_t i = 0; i < cap; i++) { model_threadIdx.x = i; fn(); } model_threadIdx.x = 0; };
		each([&] { k_vm_attempts(V); });
		if (tot[2]) return -1;
		if (vbud[0] > bud0 || vbud[0] == 0) return -5; // every attempt hands back what it did not use: never more than there was
		uint32_t acc = 0;
		for (uint32_t i = 0; i < cap; i++) { const uint32_t f = flag[i]; flag[i] = acc; acc += f; } // device: block-scan kernels
		tot[4] = acc;
		each([&] { k_vm_compact(V); });
		for (uint32_t u = 0; u <= 1; u++) { model_threadIdx.x = u; k_vm_unit_starts(V); }
		model_threadIdx.x = 0;
		ResolveArgs C = V;
		C.ord = V.vm_ord; C.unit_start = V.vm_unit_start; C.totals = V.totals + 4; // chain_view() of resolve_kernels.cu
		const bool follow = mode != GSCAN_MODE_FIRST;
		if (follow) {
			each([&] { k_chain_next(C); });
			for (uint32_t k = 1; k < levels; k++) each([&] { k_chain_double(C, k); });
		}
		model_threadIdx.x = 0;
		k_chain_heads(C);
		if (follow) for (uint32_t k = levels; k-- > 0;) each([&] { k_chain_spread(C, k); });
		each([&] { k_chain_unmark(C); });
		uint32_t *mark = buf.data() + (size_t)levels * cap, *rank = mark + cap;
		acc = 0;
		for (uint32_t i = 0; i < cap; i++) { rank[i] = acc; acc += mark[i]; }
		k_chain_count(C);
		const uint32_t nc = uo[0];
		uo[0] = 0;
		std::vector<FinalRec> fc(nc + 1);
		C.out = fc.data();
		each([&] { k_chain_write(C); });
		bool same = nc == n;
		for (uint32_t i = 0; same && i < n; i++) same = fc[i].start == fin[i].start && fc[i].len == fin[i].len;
		if (!same) return -5;
		g_vmpar_checks++;
	}
	// dense general patterns on the chain path (vm_ready): the attempts of all positions in blocks of 64 (count pass, prefix
	// sum, write pass), then the chain over the matching positions -- wherever the engine may choose it (start-free program
	// without a candidate filter), in every mode: same records as the serial walk
	if (p.use_vm && p.vm_dense && p.vm_start_free) {
		// tiles of 256 bytes (the device's are 4 .. 64 KiB; the block -> tile -> unit arithmetic is the same): the longer
		// subjects span several tiles, the last one partly filled
		const uint32_t tshift = 8;
		std::vector<TileDesc> tds;
		for (size_t off = 0; off < len || tds.empty(); off += (size_t)1 << tshift) {
			TileDesc t;
			memset(&t, 0, sizeof t);
			t.src = du.ptr + off; t.unit = 0; t.off = (uint32_t)off;
			t.len = (uint32_t)std::min<size_t>((size_t)1 << tshift, len - off); t.ulen = (uint32_t)len;
			tds.push_back(t);
		}
		const uint32_t blocks = (uint32_t)tds.size() << (tshift - 6);
		std::vector<uint32_t> flag(blocks + 1, 0u);
		uint32_t vus[2] = {0, 0}, tot[8] = {0, 0, 0, 0, 0, 0, 0, 0}, uo[1] = {0};
		unsigned long long vbud[1] = {0};
		ResolveArgs V = R;
		V.flat = 0; V.vm_dense = 0; V.tiles = tds.data(); V.dense_tile_shift = tshift; V.dense_blocks = blocks;
		V.unit_out = uo; V.totals = tot; V.out = nullptr;
		V.vm_flag = flag.data(); V.vm_unit_start = vus; V.vm_budget = vbud;
		auto blocks_each = [&](auto fn) { for (uint32_t b = 0; b < blocks; b++) { model_threadIdx.x = b; fn(); } model_threadIdx.x = 0; };
		model_threadIdx.x = 0;
		k_vm_budget_init(V);
		blocks_each([&] { k_vm_dense<false>(V); });
		if (tot[2]) return -1;
		uint32_t acc = 0;
		for (uint32_t b = 0; b < blocks; b++) { const uint32_t f = flag[b]; flag[b] = acc; acc += f; }
		tot[4] = acc;
		const uint32_t cap = acc;
		std::vector<FinalRec> fc(1);
		uint32_t nc = 0;
		if (cap) {
			std::vector<OutRec> vord(cap);
			uint32_t levels = 2;
			while ((1u << levels) < cap) levels++;
			std::vector<uint32_t> buf((size_t)(levels + 2) * cap, 0u);
			V.vm_ord = vord.data();
			{ // the write pass with LESS budget than the count pass had (the attempts of a unit share it: on the device the two
			  // passes can run out at different places): never more records than counted, what is missing padded with
			  // chain-ending entries, nothing written past the list, the limit reported
				std::vector<OutRec> guarded(cap + 4);
				for (auto &g : guarded) g = OutRec{0xdeadbeefu, 0xdeadbeefu, 0xdeadbeefu, 0xdeadbeefu};
				ResolveArgs W = V;
				uint32_t wtot[8];
				memcpy(wtot, tot, sizeof wtot);
				wtot[2] = 0;
				W.totals = wtot;
				W.vm_ord = guarded.data();
				vbud[0] = 40; // steps for the whole unit
				blocks_each([&] { k_vm_dense<true>(W); });
				bool ok = true; // (40 steps can be enough for a tiny subject: then nothing is flagged and the list is complete)
				for (uint32_t i = 0; ok && i < cap; i++) ok = guarded[i].unit == 0 && guarded[i].pos < len && guarded[i].pad >= 1 && guarded[i].pad <= 3;
				for (uint32_t i = cap; ok && i < cap + 4; i++) ok = guarded[i].unit == 0xdeadbeefu;
				if (!ok) return -6;
			}
			k_vm_budget_init(V);
			blocks_each([&] { k_vm_dense<true>(V); });
			for (uint32_t u = 0; u <= 1; u++) { model_threadIdx.x = u; k_vm_dense_unit_starts(V); }
			model_threadIdx.x = 0;
			V.vm_par = 1; V.vm_ready = 1;
			V.chain = 1; V.chain_levels = levels; V.chain_cap = cap; V.chain_buf = buf.data(); V.total_cand = cap;
			ResolveArgs C = V;
			C.ord = V.vm_ord; C.unit_start = V.vm_unit_start; C.totals = V.totals + 4;
			auto each = [&](auto fn) { for (uint32_t i = 0; i < cap; i++) { model_threadIdx.x = i; fn(); } model_threadIdx.x = 0; };
			const bool follow = mode != GSCAN_MODE_FIRST;
			if (follow) {
				each([&] { k_chain_next(C); });
				for (uint32_t k = 1; k < levels; k++) each([&] { k_chain_double(C, k); });
			}
			model_threadIdx.x = 0;
			k_chain_heads(C);
			if (follow) for (uint32_t k = levels; k-- > 0;) each([&] { k_chain_spread(C, k); });
			each([&] { k_chain_unmark(C); });
			uint32_t *mark = buf.data() + (size_t)levels * cap, *rank = mark + cap;
			acc = 0;
			for (uint32_t i = 0; i < cap; i++) { rank[i] = acc; acc += mark[i]; }
			k_chain_count(C);
			nc = uo[0];
			uo[0] = 0;
			fc.resize(nc + 1);
			C.out = fc.data();
			each([&] { k_chain_write(C); });
		}
		bool same = nc == n;
		for (uint32_t i = 0; same && i < n; i++) same = fc[i].start == fin[i].start && fc[i].len == fin[i].len;
		if (!same) return -6;
		g_densepar_checks++;
	}
	return 0;
}

// Two units in one batch on the chain paths (candidate chain, class runs in LINE mode, parallel VM attempts): the unit borders
// in the binary search, the heads, the ranks and the output slots.  Expected: the per-unit serial walks (checked against
// the oracle by the caller).  0 ok / not applicable, -1 VM limit, -7 mismatch
static int g_two_unit_checks = 0;
static int walk2(const Program &p, const std::vector<uint8_t> &a, const std::vector<uint8_t> &b, uint32_t mode)
{
	const bool fixed_chain = !p.use_vm && ((p.kind == ENGINE_FIXED && (mode == GSCAN_MODE_ALL || mode == GSCAN_MODE_LINE)) || (p.kind == ENGINE_RUN && mode == GSCAN_MODE_LINE));
	const bool vm_chain = p.use_vm && !p.vm_dense && !p.vm_runstart && p.vm_start_free;
	if (!fixed_chain && !vm_chain) return 0;
	std::vector<M> want[2];
	if (walk(p, a.data(), a.size(), mode, want[0]) != 0 || walk(p, b.data(), b.size(), mode, want[1]) != 0) return -1;
	const std::vector<uint8_t> *subj[2] = {&a, &b};
	DevUnit du[2];
	std::vector<OutRec> ord;
	uint32_t unit_start[3] = {0, 0, 0};
	for (uint32_t u = 0; u < 2; u++) {
		memset(&du[u], 0, sizeof du[u]);
		du[u].ptr = (uint64_t)(uintptr_t)subj[u]->data();
		du[u].len = (uint32_t)subj[u]->size();
		du[u].base_off = 1000u * u; // absolute offsets differ per unit
		du[u].file_id = 7 + u;
		std::vector<OutRec> c;
		candidates(p, subj[u]->data(), subj[u]->size(), c);
		for (auto &o : c) { o.unit = u; ord.push_back(o); }
		unit_start[u + 1] = (uint32_t)ord.size();
	}
	if (ord.empty()) return 0;
	const uint32_t cap = (uint32_t)ord.size();
	uint32_t levels = 2;
	while ((1u << levels) < cap) levels++;
	std::vector<uint32_t> buf((size_t)(levels + 2) * cap, 0u), flag(cap, 0u);
	std::vector<OutRec> vord(cap);
	uint32_t vus[3] = {0, 0, 0}, tot[8] = {cap, 0, 0, 0, 0, 0, 0, 0}, uo[2] = {0, 0};
	unsigned long long vbud[2] = {0, 0};
	ResolveArgs R;
	memset(&R, 0, sizeof R);
	R.units = du; R.n_units = 2; R.ord = ord.data(); R.unit_start = unit_start; R.unit_out = uo; R.totals = tot;
	R.mode = mode; R.minlen = (uint32_t)p.minlen; R.engine = p.use_vm ? (uint32_t)GSCAN_ENGINE_VM : (uint32_t)p.kind; R.run_min = (uint32_t)p.run_min;
	for (int i = 0; i < 8; i++) R.bitmap[i] = p.run_class.w[i];
	R.vm_code = p.vm_code.data(); R.vm_sets = p.vm_sets.data();
	R.chain = 1; R.chain_levels = levels; R.chain_cap = cap; R.chain_buf = buf.data(); R.total_cand = cap;
	auto each = [&](auto fn) { for (uint32_t i = 0; i < cap; i++) { model_threadIdx.x = i; fn(); } model_threadIdx.x = 0; };
	auto units_each = [&](uint32_t n, auto fn) { for (uint32_t u = 0; u < n; u++) { model_threadIdx.x = u; fn(); } model_threadIdx.x = 0; };
	ResolveArgs C = R;
	if (vm_chain) {
		R.vm_par = 1; R.vm_ord = vord.data(); R.vm_flag = flag.data(); R.vm_unit_start = vus; R.vm_budget = vbud;
		units_each(2, [&] { k_vm_budget_init(R); });
		each([&] { k_vm_attempts(R); });
		if (tot[2]) return -1;
		uint32_t acc = 0;
		for (uint32_t i = 0; i < cap; i++) { const uint32_t f = flag[i]; flag[i] = acc; acc += f; }
		tot[4] = acc;
		each([&] { k_vm_compact(R); });
		units_each(3, [&] { k_vm_unit_starts(R); });
		C = R;
		C.ord = R.vm_ord; C.unit_start = R.vm_unit_start; C.totals = R.totals + 4;
	}
	const bool follow = mode != GSCAN_MODE_FIRST;
	if (follow) {
		each([&] { k_chain_next(C); });
		for (uint32_t k = 1; k < levels; k++) each([&] { k_chain_double(C, k); });
	}
	units_each(2, [&] { k_chain_heads(C); });
	if (follow) for (uint32_t k = levels; k-- > 0;) each([&] { k_chain_spread(C, k); });
	if (vm_chain) each([&] { k_chain_unmark(C); });
	if (!vm_chain && p.kind == ENGINE_RUN) { each([&] { k_chain_entry_init(C); }); each([&] { k_chain_entry(C); }); }
	uint32_t *mark = buf.data() + (size_t)levels * cap, *rank = mark + cap;
	uint32_t acc = 0;
	for (uint32_t i = 0; i < cap; i++) { rank[i] = acc; acc += mark[i]; }
	units_each(2, [&] { k_chain_count(C); });
	const uint32_t n0 = uo[0], n1 = uo[1];
	uo[0] = 0; uo[1] = n0; // the device: exclusive scan of the per-unit counts
	std::vector<FinalRec> out(n0 + n1 + 1);
	C.out = out.data();
	each([&] { k_chain_write(C); });
	bool same = n0 == want[0].size() && n1 == want[1].size();
	for (uint32_t u = 0; same && u < 2; u++)
		for (size_t i = 0; same && i < want[u].size(); i++) {
			const FinalRec &r = out[(u ? n0 : 0) + i];
			same = r.start == du[u].base_off + want[u][i].pos && r.len == want[u][i].len && r.file_id == du[u].file_id;
		}
	if (!same) return -7;
	g_two_unit_checks++;
	return 0;
}

int main(int argc, char **argv)
{
	if (argc < 2) return 2;
	std::ifstream f(argv[1]);
	std::string pat;
	std::vector<std::vector<uint8_t>> subjects;
	const char *alphas[] = {"abc", "abcx \n", "ab", "abc abc\n\n", "aabbcc_x1 \t\n", "ab\n"};
	const int lens[] = {1, 2, 3, 4, 5, 7, 9, 16, 17, 33, 64, 130, 257};
	for (int k = 0; k < 78; k++) {
		const char *al = alphas[k % 6];
		const size_t na = strlen(al), ln = (size_t)lens[k % 13];
		std::vector<uint8_t> b(ln);
		for (auto &c : b) c = (uint8_t)al[rnd() % na];
		subjects.push_back(b);
	}
	// lines longer than the 511 bytes the reference prints behind a match (grab.cc:194-196): in LINE mode the search resumes
	// in the middle of the line, for class runs possibly in the middle of a run
	for (int k = 0; k < 6; k++) {
		const char *al = k % 3 == 0 ? "ab" : (k % 3 == 1 ? "abc " : "aab_1 ");
		const size_t na = strlen(al), ln = k < 3 ? 700 : 1500;
		std::vector<uint8_t> b(ln);
		for (auto &c : b) c = (uint8_t)al[rnd() % na];
		if (k >= 3) b[ln / 2] = '\n';
		subjects.push_back(b);
	}
	// binary subjects: uniform bytes, the ASCII alphabets with bit 7 or bit 5 flipped (what SWAR filters that ignore a bit
	// let through), and text with NUL bytes and a run of NULs
	for (int k = 0; k < 40; k++) {
		const char *al = alphas[k % 6];
		const size_t na = strlen(al), ln = (size_t)lens[(k * 7) % 13] + (k & 1) * 200;
		std::vector<uint8_t> b(ln);
		for (auto &c : b) {
			const uint8_t a = (uint8_t)al[rnd() % na];
			switch (k / 10) {
			case 0: c = (uint8_t)rnd(); break;
			case 1: c = rnd() % 3 ? a : (uint8_t)(a ^ 0x80); break;
			case 2: c = rnd() % 3 ? a : (uint8_t)(a ^ 0x20); break;
			default: c = rnd() % 4 ? a : 0; break;
			}
		}
		if (k / 10 == 3) for (size_t i = ln / 3; i < ln / 3 + ln / 4; i++) b[i] = 0;
		subjects.push_back(b);
	}
	int n_dense = 0, n_pat = 0, n_served = 0, n_vm = 0, n_cmp = 0, n_walk = 0, n_limit = 0, bad = 0, n_strict = 0;
	while (std::getline(f, pat)) {
		if (pat.empty()) continue;
		n_pat++;
		Program p;
		std::string err;
		if (!compile_pattern(pat.data(), pat.size(), 0, p, err)) continue; // rejected loudly: nothing to check
		char oerr[200];
		go_regex *re = go_compile(pat.data(), pat.size(), 0, oerr, sizeof oerr);
		if (!re) continue;
		if (go_nullable(re)) { printf("MISMATCH %s: compiled but the oracle says it can match the empty string\n", pat.c_str()); bad++; go_free(re); continue; }
		if (go_minlen(re) != p.minlen) { printf("MISMATCH %s: minlen %d, oracle %d\n", pat.c_str(), p.minlen, go_minlen(re)); bad++; }
		n_served++;
		n_vm += p.use_vm;
		n_dense += p.use_vm && p.vm_dense;
		for (auto &sb : subjects) {
			go_matches want = {0, 0, 0};
			if (go_scan_window(re, sb.data(), sb.size(), 0, 0, GO_MODE_ALL, 0, &want) != 0) { go_matches_free(&want); n_limit++; continue; }
			std::vector<M> got;
			std::string why;
			const int rc = emulate(p, sb.data(), sb.size(), got, why);
			if (rc == -1) { n_limit++; go_matches_free(&want); continue; }
			bool same = rc == 0 && got.size() == want.n;
			for (size_t i = 0; same && i < got.size(); i++) same = got[i].pos == want.v[i].start && got[i].len == want.v[i].len;
			n_cmp++;
			if (!same) {
				bad++;
				printf("MISMATCH %s (engine %d vm %d runstart %d) on \"", pat.c_str(), (int)p.kind, (int)p.use_vm, (int)p.vm_runstart);
				for (uint8_t c : sb) printf(c == '\n' ? "\\n" : c == '\t' ? "\\t" : "%c", c);
				printf("\": %s got %zu want %zu\n", why.c_str(), got.size(), want.n);
				if (bad > 20) { go_matches_free(&want); go_free(re); return 1; }
			}
			go_matches_free(&want);
			// the device's own walk code in all three modes
			const int modes[3] = {GO_MODE_ALL, GO_MODE_FIRST, GO_MODE_LINE};
			const uint32_t dmodes[3] = {GSCAN_MODE_ALL, GSCAN_MODE_FIRST, GSCAN_MODE_LINE};
			for (int m = 0; m < 3; m++) {
				go_matches w2 = {0, 0, 0};
				if (go_scan_window(re, sb.data(), sb.size(), 0, 0, modes[m], 0, &w2) != 0) { go_matches_free(&w2); continue; }
				std::vector<M> g2;
				const int wrc = walk(p, sb.data(), sb.size(), dmodes[m], g2);
				if (wrc == -3) { printf("FLAT WALK MISMATCH %s\n", pat.c_str()); bad++; go_matches_free(&w2); continue; }
				if (wrc == -4) { printf("CHAIN WALK MISMATCH %s mode %d\n", pat.c_str(), m); bad++; go_matches_free(&w2); continue; }
				if (wrc == -6) {
					printf("DENSE VM CHAIN MISMATCH %s mode %d on \"", pat.c_str(), m);
					for (uint8_t c : sb) printf(c == '\n' ? "\\n" : c == '\t' ? "\\t" : "%c", c);
					printf("\"\n");
					bad++; go_matches_free(&w2); continue;
				}
				if (wrc == -5) {
					printf("VM CHAIN MISMATCH %s mode %d on \"", pat.c_str(), m);
					for (uint8_t c : sb) printf(c == '\n' ? "\\n" : c == '\t' ? "\\t" : "%c", c);
					printf("\"\n");
					bad++; go_matches_free(&w2); continue;
				}
				if (wrc != 0) { go_matches_free(&w2); n_limit++; continue; }
				bool ok = g2.size() == w2.n;
				for (size_t i = 0; ok && i < g2.size(); i++) ok = g2[i].pos == w2.v[i].start && g2[i].len == w2.v[i].len;
				n_walk++;
				if (!ok) {
					bad++;
					printf("WALK MISMATCH %s mode %d (engine %d vm %d runstart %d) on \"", pat.c_str(), m, (int)p.kind, (int)p.use_vm, (int)p.vm_runstart);
					for (uint8_t c : sb) printf(c == '\n' ? "\\n" : c == '\t' ? "\\t" : "%c", c);
					printf("\": got %zu want %zu\n", g2.size(), w2.n);
					if (bad > 20) { go_matches_free(&w2); go_free(re); return 1; }
				}
				go_matches_free(&w2);
			}
		}
		// two units in one batch on the chain paths: consecutive subjects pairwise, all modes
		for (size_t k = 0; k + 1 < subjects.size(); k += 5) {
			const uint32_t dmodes[3] = {GSCAN_MODE_ALL, GSCAN_MODE_FIRST, GSCAN_MODE_LINE};
			for (int m = 0; m < 3; m++) {
				const int rc2 = walk2(p, subjects[k], subjects[k + 1], dmodes[m]);
				if (rc2 == -7) { printf("TWO-UNIT CHAIN MISMATCH %s mode %d subjects %zu,%zu\n", pat.c_str(), m, k, k + 1); bad++; }
			}
		}
		// Q2 in full (STRICT_REF): patterns with capturing groups -- the first match in which a group took part ends the
		// window; the device walk kernels against the oracle with strict_q2 on
		if (p.captures > 0) {
			Program ps;
			std::string e2;
			if (compile_pattern(pat.data(), pat.size(), GSCAN_STRICT_REF, ps, e2)) {
				n_strict++;
				for (auto &sb : subjects) {
					const int modes[3] = {GO_MODE_ALL, GO_MODE_FIRST, GO_MODE_LINE};
					const uint32_t dmodes[3] = {GSCAN_MODE_ALL, GSCAN_MODE_FIRST, GSCAN_MODE_LINE};
					for (int m = 0; m < 3; m++) {
						go_matches w2 = {0, 0, 0};
						if (go_scan_window(re, sb.data(), sb.size(), 0, 0, modes[m], 1, &w2) != 0) { go_matches_free(&w2); continue; }
						std::vector<M> g2;
						const int src = ps.kind != ENGINE_NONE ? walk(ps, sb.data(), sb.size(), dmodes[m], g2) : 0;
						if (src == -6) { printf("STRICT DENSE VM CHAIN MISMATCH %s mode %d\n", pat.c_str(), m); bad++; go_matches_free(&w2); continue; }
						if (src == -5) { printf("STRICT VM CHAIN MISMATCH %s mode %d\n", pat.c_str(), m); bad++; go_matches_free(&w2); continue; }
						if (src != 0) { go_matches_free(&w2); n_limit++; continue; }
						bool ok = g2.size() == w2.n;
						for (size_t i = 0; ok && i < g2.size(); i++) ok = g2[i].pos == w2.v[i].start && g2[i].len == w2.v[i].len;
						n_walk++;
						if (!ok) {
							bad++;
							printf("STRICT WALK MISMATCH %s mode %d (engine %d vm %d) on \"", pat.c_str(), m, (int)ps.kind, (int)ps.use_vm);
							for (uint8_t c : sb) printf(c == '\n' ? "\\n" : c == '\t' ? "\\t" : "%c", c);
							printf("\": got %zu want %zu\n", g2.size(), w2.n);
							if (bad > 20) { go_matches_free(&w2); go_free(re); return 1; }
						}
						go_matches_free(&w2);
					}
				}
			}
		}
		go_free(re);
	}
	printf("two-unit chain checks %d; dense vm chain checks %d; vm chain checks %d; chain checks %d; dense VM patterns %d; ", g_two_unit_checks, g_densepar_checks, g_vmpar_checks, g_chain_checks, n_dense);
	printf("flat write checks %d; strict (Q2) patterns %d; ", g_flat_checks, n_strict);
	printf("patterns %d, served %d (%d through the VM), comparisons %d + %d through the walk kernels, limit skips %d, mismatches %d\n", n_pat, n_served, n_vm, n_cmp, n_walk, n_limit, bad);
	if (bad == 0) printf("model ok\n");
	return bad ? 1 : 0;
}
