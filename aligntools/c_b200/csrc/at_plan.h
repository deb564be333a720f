// at_plan.h -- the BATCH PLAN of a shard: which kernel runs each pair, which pairs share a warp, how the pairs are cut
// into chunks whose traceback pointers fit the arena, the order of K2's task queue, and where each pair's pointer block,
// boundary slabs and traceback scratch lie.  Every kernel trusts these numbers: overlapping pointer blocks, a wrong
// layout-class byte or a task queued behind the stripe it waits for would corrupt results or deadlock.
//
// Host code (the uniform closed form is host + device), no CUDA includes, no environment: the runtime (setup_shard,
// at_runtime.cu) reads its knobs and passes them in.  tests/test_plan_cpu.py compiles this header with g++ and checks
// the plans against a port of the planning loop and against the invariants above, without a GPU.
#pragma once
#include <stdint.h>
#include <algorithm>
#include <vector>
#include "../../../include/aligntools_b200.h"      // AT_GLOBAL .. AT_EDIT, at_params
#include "at_ptr_layout.h"
#include "at_band.h"

namespace atb2 {

constexpr int MAXR = 8;      // rows per lane of K1 (32 * MAXR = 256 rows: longer reads run on K2)

struct FillJob { uint32_t a, b; };     // K1: pair indices; b == a for int32 lanes or a packed job without partner

// One unit of K2 work: stripe `stripe` of pair `pair`.  `prev` is the queue index of the same pair's stripe above it (its
// own index for stripe 0): the affine kernel waits on that task's progress word.
struct alignas(16) WaveTask { uint32_t pair, stripe, prev, reserved; };
static_assert(sizeof(WaveTask) == 16, "K2 loads a task as one 16-byte vector");

struct PairBand { int32_t lo, hi; };      // a pair's band clipped by band_clip (at_band.h); the device reads it as int2
static_assert(sizeof(PairBand) == 8, "uploaded as int2");

inline uint32_t rclass_of(uint32_t l1) { uint32_t r = (l1 + 31) / 32; return r < 1 ? 1 : (r > (uint32_t)MAXR ? MAXR : r); }

// Packed s16x2 lanes (two pairs per warp): local mode, scores x8 must fit int16, 8|m-u| < 256 (symbols are << 8).  Global /
// fit (without jump state) also carry -inf inside the 16 bits (AT_NEG16 = -30000, at_cell.cuh): finite values must stay
// above -24000 and a -inf value may drift by a few steps' worth of the largest parameter.
struct P16Rule {
	bool on = false, local = false;
	int64_t maxabs = 1;
	bool ok(uint32_t l1, uint32_t l2) const      // + 40: K1 also computes up to 34 columns past l2
	{
		return on && l1 <= 32u * MAXR && l2 <= 60000u && 8 * (int64_t)(l1 + l2 + 42) * maxabs < (local ? 32000 : 24000);
	}
};
inline P16Rule p16_rule(int mode, const at_params &p, bool jump, bool no_p16)
{
	auto iabs = [](int64_t x) { return x < 0 ? -x : x; };
	P16Rule r;
	r.local = mode == AT_LOCAL;
	r.maxabs = std::max<int64_t>({iabs(p.m), iabs(p.u), iabs(p.o), iabs(p.e), 1});
	r.on = (r.local || mode == AT_GLOBAL || (mode == AT_FIT && !jump)) && iabs((int64_t)p.m - p.u) <= 31 && (r.local || r.maxabs <= 31) && !no_p16;
	return r;
}
// Substitution-matrix scoring (at_batch_*_scored): `mat_maxabs` = max |s(a, b)| stands for m and u.  Packed lanes then run only
// the profile variant, whose words hold the matrix values themselves, so the symbol-shift limit on |m - u| does not apply.
inline P16Rule p16_rule(int mode, const at_params &p, bool jump, bool no_p16, int64_t mat_maxabs)
{
	auto iabs = [](int64_t x) { return x < 0 ? -x : x; };
	P16Rule r;
	r.local = mode == AT_LOCAL;
	r.maxabs = std::max<int64_t>({mat_maxabs, iabs(p.o), iabs(p.e), 1});
	r.on = (r.local || mode == AT_GLOBAL || (mode == AT_FIT && !jump)) && (r.local || r.maxabs <= 31) && !no_p16;
	return r;
}

// Bit-parallel edit distance: r = 32-row blocks per lane, 1024 r rows per stripe.  One column step of a lane is a serial
// chain through its r blocks, so few long pairs want r = 1 (more stripes in flight); 4 blocks per lane amortise the
// per-step overhead once there are tasks for every resident warp (warp_slots = SMs x 8 x AT_WAVE_WARPS).  Decided for the
// whole shard before the arena is sized: an edit path's pointer layout depends on it.
inline uint32_t choose_bits_r(const uint32_t *l1, uint32_t n, uint64_t warp_slots)
{
	for (uint32_t r : {4u, 2u}) {
		uint64_t tasks = 0;
		for (uint32_t k = 0; k < n; ++k) tasks += (l1[k] + edit_bits_rows(r) - 1) / edit_bits_rows(r);
		if (tasks >= 2 * warp_slots) return r;
	}
	return 1;
}

// A banded pair's stripe is queued when it has a window; the last stripe always is (it writes the end cell; banded
// global: the end diagonal is in band, so the last stripe has a window).
inline bool band_stripe_queued(uint32_t l1, uint32_t l2, PairBand b, uint32_t rows, uint32_t s)
{
	BandWin w;
	return s + 1 >= (l1 + rows - 1) / rows || band_stripe(l1, l2, b.lo, b.hi, rows, s, w);
}

// Contiguous slices of [lo, hi) with (nearly) equal numbers of cells, from running cell counts prefix[k] = sum of l1*l2
// over pairs < k; cut receives parts + 1 entries.  Slice d ends after the first pair at which the running count reaches
// d / parts of the range's total.  `prefix` is not read when parts <= 1.
inline void cut_by_prefix(const std::vector<uint64_t> &prefix, uint64_t lo, uint64_t hi, size_t parts, std::vector<uint64_t> &cut)
{
	cut.assign(parts + 1, lo);
	cut[parts] = hi;
	if (parts <= 1) return;
	const uint64_t base = prefix[lo], total = prefix[hi] - base;
	for (size_t d = 1; d < parts; ++d) {
		// smallest k in [lo, hi) with (prefix[k+1] - base) * parts >= total * d; the slice ends after it
		uint64_t a = lo, b = hi;
		while (a < b) {
			const uint64_t mid = a + (b - a) / 2;
			if ((unsigned __int128)(prefix[mid + 1] - base) * parts >= (unsigned __int128)total * d) b = mid; else a = mid + 1;
		}
		cut[d] = a < hi ? a + 1 : hi;
	}
	for (size_t d = 1; d <= parts; ++d) cut[d] = std::max(cut[d], cut[d - 1]);
}

// Queue order of the K2 tasks of one launch.  The persistent warps claim tasks in queue order, and a stripe can only run
// as far as the stripe above it has got.  Pair after pair (round 1) puts a pair's stripes next to each other in the
// queue: they are claimed within microseconds of each other and run as ONE tightly coupled chain, each stripe 64 columns
// behind the one above -- the chain advances at the pace of its momentarily slowest warp and the others poll (ncu on
// C3, 2 048 pairs: 21 % of all warp samples in the progress poll and its warp-sync).  Stripe after stripe ACROSS the
// launch's pairs -- all stripes 0, then all stripes 1, ... -- puts as many other tasks between a stripe and its
// predecessor as the launch has pairs: with more pairs than resident warps the predecessor has finished (or is far
// ahead) when the stripe is claimed and nothing ever polls; with fewer pairs the chains are as long as they have to be
// to fill the GPU and no longer.  A task's predecessor still precedes it in the queue, so a claimed task only ever
// waits for a running one (deadlock freedom as before).  In: tasks collected pair by pair, stripes ascending.
// `pair_major` keeps the old order (AT_WAVE_ORDER=pair, A/B runs).
inline void order_wave_tasks(std::vector<WaveTask> &t, bool pair_major)
{
	const size_t n = t.size();
	if (pair_major || n == 0) {
		for (size_t x = 0; x < n; ++x) t[x].prev = (uint32_t)(t[x].stripe ? x - 1 : x);
		return;
	}
	struct Run { uint32_t pair, n, last; size_t x0; };      // x0: the pair's first task in `t` (its stripes need not start at 0: banded pairs)
	std::vector<Run> active;
	for (size_t x = 0; x < n;) { size_t y = x; while (y < n && t[y].pair == t[x].pair) ++y; active.push_back(Run{t[x].pair, (uint32_t)(y - x), 0, x}); x = y; }
	std::vector<WaveTask> out;
	out.reserve(n);
	for (uint32_t s = 0; !active.empty(); ++s) {
		size_t keep = 0;
		for (Run &r : active) {
			const uint32_t idx = (uint32_t)out.size();
			out.push_back(WaveTask{r.pair, t[r.x0 + s].stripe, s ? r.last : idx, 0});
			r.last = idx;
			if (s + 1 < r.n) active[keep++] = r;
		}
		active.resize(keep);
	}
	t.swap(out);
}

// What the plan is made from: the shard's pairs and the run's settings.
struct PlanIn {
	uint32_t n = 0;
	const uint32_t *l1 = nullptr, *l2 = nullptr;      // read and target lengths of the shard's pairs
	int mode = AT_GLOBAL;
	bool traceback = false, jump = false;
	const PairBand *band = nullptr;                    // clipped bands, nullptr: unbanded
	bool bits = false;                                 // bit-parallel edit distance (at_wave_edit_bits) ...
	uint32_t bits_r = 1;                               // ... with its 32-row blocks per lane (choose_bits_r)
	P16Rule p16;                                       // which pairs may share a warp on packed lanes
	bool allow_uniform = true;                         // AT_NO_UNIFORM_PLAN clears it
	bool pair_major = false;                           // order_wave_tasks
	uint64_t budget_words = UINT64_MAX;                // pointer words a chunk may take (the arena)

	// banded global pairs all run on K2's affine kernel, short ones included: R = 8 rows per lane, 8-step pointer groups
	bool band_affine() const { return band && mode == AT_GLOBAL; }
	bool bits_path() const { return bits && traceback; }      // edit paths on at_wave_edit_bits: K3 reads R from the pair's class
	uint32_t rclass(uint32_t k) const { return band_affine() ? (uint32_t)MAXR : bits_path() ? bits_r : rclass_of(l1[k]); }
	// DP cells of pair k as K1 / K2 sweep them (banded: in-band cells)
	uint64_t cells(uint32_t k) const { return band ? band_cells(l1[k], l2[k], band[k].lo, band[k].hi) : (uint64_t)l1[k] * l2[k]; }
	// words of pair k's pointer block (not packed); overlap and edit on the cell-by-cell kernel store 2-bit codes, the
	// affine modes nibbles
	uint64_t ptr_words(uint32_t k) const
	{
		if (bits_path()) return edit_bits_pair_words(l1[k], l2[k], bits_r);
		const uint32_t code_sh = mode >= AT_OVERLAP ? PTR_SH_2BIT : PTR_SH_NIB;
		return band ? band_pair_words(l1[k], l2[k], band[k].lo, band[k].hi, 32u * rclass(k), code_sh) : ptr_pair_words(l1[k], l2[k], rclass(k), code_sh, jump);
	}
	// what pair k asks of the arena: its block + the rounding slack of the packed layout
	uint64_t arena_words(uint32_t k) const { return traceback ? ptr_words(k) + 64ull * rclass(k) : 0; }
	// every pair of the same shape and on K1: the plan is closed form (uniform_pair)
	bool uniform() const
	{
		if (!allow_uniform || mode > AT_FIT || l1[0] > 32u * MAXR || band_affine()) return false;
		for (uint32_t k = 1; k < n; ++k) if (l1[k] != l1[0] || l2[k] != l2[0]) return false;
		return true;
	}
};

// The pointer words the whole shard asks of the arena (the runtime sizes the budget by it)
inline uint64_t need_words(const PlanIn &in)
{
	if (in.uniform()) return (uint64_t)in.n * in.arena_words(0);
	uint64_t w = 0;
	for (uint32_t k = 0; k < in.n; ++k) w += in.arena_words(k);
	return w;
}

// One kernel launch of a chunk: the jobs of one (kernel kind, rows-per-lane) class.
enum { LK_INT32 = 0, LK_PACKED = 1, LK_WAVE = 2, LK_BITS = 3 };   // LK_BITS: bit-parallel edit distance (K2 task geometry, 1024*r rows per stripe)
struct PlanLaunch {
	int kind = LK_INT32, r = 1;
	uint64_t cells = 0;
	uint32_t n = 0;                     // jobs (K1) or tasks (K2) of the launch
	std::vector<FillJob> jobs;          // LK_INT32: one pair per warp (a == b); LK_PACKED: two pairs per warp (empty: uniform_pair)
	std::vector<WaveTask> tasks;        // LK_WAVE / LK_BITS: (pair, stripe) in queue order (order_wave_tasks)
	uint64_t prog_base = 0;             // first progress word of this launch in the shard's progress words
};

struct PlanChunk {
	uint32_t k0 = 0, k1 = 0;            // shard-local pair range
	std::vector<PlanLaunch> launches;
	// chunk-local, one entry per pair (empty for a uniform shard: uniform_pair): the pair's pointer block (words), the
	// element offset of its two boundary slabs (K2), its traceback scratch slot (words; with traceback only)
	std::vector<uint64_t> ptr_off, bnd_off, scratch_off;
	uint64_t ptr_words = 0, bnd_elems = 0, prog_words = 0, scratch_words = 0;
};

// A uniform shard's plan in closed form: one chunk, one K1 launch.  packed: jobs are pairs (2k, 2k + 1), a last odd pair
// runs alone.
struct UniformPlan { bool packed = false; uint32_t R = 1; uint64_t words_per_job = 0, scratch_per_pair = 0; };
struct UniformPair { uint64_t ptr_off, scratch_off; uint8_t rclass; bool writes_job; uint32_t job; FillJob fj; };
AT_HD UniformPair uniform_pair(const UniformPlan &u, uint32_t n, uint32_t k)
{
	UniformPair p;
	p.job = u.packed ? k >> 1 : k;
	p.ptr_off = (uint64_t)p.job * u.words_per_job;
	p.scratch_off = (uint64_t)k * u.scratch_per_pair;
	p.rclass = ptr_class(u.R, u.packed ? ((k & 1u) ? 2u : 1u) : 0u);
	p.writes_job = !u.packed || !(k & 1u);
	p.fj = FillJob{k, u.packed && (k | 1u) < n ? k + 1u : k};
	return p;
}

struct Plan {
	std::vector<PlanChunk> chunks;
	bool uniform = false;
	UniformPlan u;                      // uniform: the device writes jobs, offsets and class bytes (at_plan_uniform)
	std::vector<uint8_t> rclass;        // not uniform: the layout-class byte of every pair (at_ptr_layout.h)
	uint64_t cells = 0;
	// what the shard-level buffers are sized by: the largest chunk's pointer words, scratch words, boundary elements,
	// progress words and pairs
	uint64_t max_chunk_words = 0, max_scratch_words = 0, max_bnd_elems = 0, max_prog_words = 0;
	uint32_t max_pairs = 0;
	// a pair that needs more than the budget on its own (the plan is then incomplete)
	uint32_t fail_pair = UINT32_MAX;
	uint64_t fail_words = 0;
};

inline Plan make_plan(const PlanIn &in)
{
	Plan p;
	const uint32_t n = in.n;
	// ---- uniform shard: every pair has the same shape and runs on K1 in one chunk ----
	if (in.uniform() && (uint64_t)n * in.arena_words(0) <= in.budget_words) {      // else several chunks: the general plan
		const uint32_t l1 = in.l1[0], l2 = in.l2[0];
		p.uniform = true;
		p.u.packed = in.p16.ok(l1, l2) && n >= 2;
		p.u.R = rclass_of(l1);
		p.u.words_per_job = !in.traceback ? 0 : p.u.packed ? ptr_packed_job_words(l2, p.u.R) : in.ptr_words(0);
		p.u.scratch_per_pair = in.traceback ? (uint64_t)l1 + l2 : 0;
		p.cells = (uint64_t)n * l1 * l2;
		PlanLaunch l;
		l.kind = p.u.packed ? LK_PACKED : LK_INT32; l.r = (int)p.u.R; l.cells = p.cells; l.n = p.u.packed ? (n + 1) / 2 : n;
		PlanChunk c;
		c.k0 = 0; c.k1 = n;
		c.ptr_words = p.u.words_per_job * l.n;
		c.scratch_words = p.u.scratch_per_pair * n;
		c.launches.push_back(std::move(l));
		p.max_chunk_words = c.ptr_words; p.max_scratch_words = c.scratch_words; p.max_pairs = n;
		p.chunks.push_back(std::move(c));
		return p;
	}
	p.rclass.resize(n);
	for (uint32_t k = 0; k < n; ++k) { p.rclass[k] = ptr_class(in.rclass(k), 0); p.cells += in.cells(k); }
	// ---- chunks by pointer-arena budget ----
	{
		PlanChunk cur;
		uint64_t words = 0;
		for (uint32_t k = 0; k < n; ++k) {
			const uint64_t w = in.arena_words(k);
			if (w > in.budget_words) { p.fail_pair = k; p.fail_words = w; return p; }
			if (words + w > in.budget_words && k > cur.k0) {
				cur.k1 = k; p.chunks.push_back(std::move(cur));
				cur = PlanChunk(); cur.k0 = k; words = 0;
			}
			words += w;
		}
		cur.k1 = n; p.chunks.push_back(std::move(cur));
	}
	const bool linear = in.mode >= AT_OVERLAP;          // single-plane modes run on K2 at every length
	auto cells_of = [&](uint32_t k) { return (uint64_t)in.l1[k] * in.l2[k]; };
	auto by_cells = [&](std::vector<uint32_t> &v) {   // largest pairs first (dynamic queue => good tail balance)
		bool ragged = false;
		for (size_t x = 1; x < v.size() && !ragged; ++x) ragged = cells_of(v[x]) != cells_of(v[0]);
		if (ragged) std::stable_sort(v.begin(), v.end(), [&](uint32_t x, uint32_t y) { return cells_of(x) > cells_of(y); });
	};
	for (PlanChunk &c : p.chunks) {
		const uint32_t nc = c.k1 - c.k0;
		PlanLaunch l32[MAXR + 1], l16[MAXR + 1], lwv[MAXR + 1], lbit[MAXR + 1];
		std::vector<uint32_t> scalar_pairs, wave_pairs, cand;
		for (uint32_t k = c.k0; k < c.k1; ++k) {
			if (linear || in.band_affine() || in.l1[k] > 32u * MAXR) wave_pairs.push_back(k);
			else if (in.p16.ok(in.l1[k], in.l2[k])) cand.push_back(k);
			else scalar_pairs.push_back(k);
		}
		// ---- packed jobs (K1, s16x2): partners must share the rows-per-lane class and l2 ----
		{
			// local: the partners share the rows-per-lane class and l2; global / fit: l1 as well (one lane holds the last row of both)
			auto key = [&](uint32_t k) { return ((uint64_t)(in.p16.local ? p.rclass[k] : in.l1[k]) << 32) | in.l2[k]; };
			bool sorted = true;
			for (size_t x = 1; x < cand.size() && sorted; ++x) sorted = key(cand[x - 1]) >= key(cand[x]);
			if (!sorted) std::stable_sort(cand.begin(), cand.end(), [&](uint32_t x, uint32_t y) { return key(x) > key(y); });
			for (size_t x = 0; x < cand.size();) {
				if (x + 1 < cand.size() && key(cand[x]) == key(cand[x + 1])) {
					const int r = ptr_class_r(p.rclass[cand[x]]);
					l16[r].jobs.push_back(FillJob{cand[x], cand[x + 1]});
					l16[r].cells += cells_of(cand[x]) + cells_of(cand[x + 1]);
					x += 2;
				} else { scalar_pairs.push_back(cand[x]); x += 1; }
			}
		}
		// ---- int32 jobs (K1) per R class ----
		by_cells(scalar_pairs);
		for (uint32_t k : scalar_pairs) { const int r = ptr_class_r(p.rclass[k]); l32[r].jobs.push_back(FillJob{k, k}); l32[r].cells += cells_of(k); }
		// ---- wavefront tasks (K2): (pair, stripe), collected pair by pair, then put in queue order (order_wave_tasks) ----
		by_cells(wave_pairs);
		c.bnd_off.assign(nc, 0);
		for (uint32_t k : wave_pairs) {
			const uint32_t l1 = in.l1[k], l2 = in.l2[k];
			const int r = in.bits ? (int)in.bits_r : ptr_class_r(p.rclass[k]);
			const uint32_t rows = in.bits ? edit_bits_rows(r) : 32u * r;
			PlanLaunch &lw = in.bits ? lbit[r] : lwv[r];
			const uint32_t n_stripes = (l1 + rows - 1) / rows;
			uint32_t queued = 0;
			for (uint32_t s = 0; s < n_stripes; ++s) {
				if (in.band && !band_stripe_queued(l1, l2, in.band[k], rows, s)) continue;
				lw.tasks.push_back(WaveTask{k, s, 0, 0});
				++queued;
			}
			lw.cells += in.band ? in.cells(k) : cells_of(k);
			if (queued > 1) { c.bnd_off[k - c.k0] = c.bnd_elems; c.bnd_elems += 2ull * ((l2 + 4u) & ~3u); }
		}
		for (int r = 1; r <= MAXR; ++r) {
			if (!l32[r].jobs.empty()) { l32[r].kind = LK_INT32; l32[r].r = r; l32[r].n = (uint32_t)l32[r].jobs.size(); c.launches.push_back(std::move(l32[r])); }
			if (!l16[r].jobs.empty()) { l16[r].kind = LK_PACKED; l16[r].r = r; l16[r].n = (uint32_t)l16[r].jobs.size(); c.launches.push_back(std::move(l16[r])); }
			for (PlanLaunch *lw : {&lwv[r], &lbit[r]}) {
				order_wave_tasks(lw->tasks, in.pair_major);
				if (lw->tasks.empty()) continue;
				lw->kind = lw == &lwv[r] ? LK_WAVE : LK_BITS; lw->r = r; lw->n = (uint32_t)lw->tasks.size();
				lw->prog_base = c.prog_words; c.prog_words += lw->n;
				c.launches.push_back(std::move(*lw));
			}
		}
		// ---- pointer blocks: one per int32 / wavefront pair, one per packed job (shared by its two pairs) ----
		c.ptr_off.assign(nc, 0);
		if (in.traceback) {
			for (const PlanLaunch &l : c.launches) {
				if (l.kind == LK_PACKED) {
					for (const FillJob &jb : l.jobs) {
						c.ptr_off[jb.a - c.k0] = c.ptr_words; c.ptr_off[jb.b - c.k0] = c.ptr_words;
						p.rclass[jb.a] = ptr_class(l.r, 1); p.rclass[jb.b] = ptr_class(l.r, 2);
						c.ptr_words += ptr_packed_job_words(in.l2[jb.a], l.r);
					}
				} else if (l.kind == LK_INT32) {
					for (const FillJob &jb : l.jobs) { c.ptr_off[jb.a - c.k0] = c.ptr_words; c.ptr_words += in.ptr_words(jb.a); }
				} else {
					// a pair's block goes where its first task is queued (stripe 0 unless the band leaves stripe 0 out)
					std::vector<uint8_t> placed(nc, 0);
					for (const WaveTask &tk : l.tasks) {
						if (placed[tk.pair - c.k0]) continue;
						placed[tk.pair - c.k0] = 1;
						c.ptr_off[tk.pair - c.k0] = c.ptr_words; c.ptr_words += in.ptr_words(tk.pair);
					}
				}
			}
			// traceback scratch: a slot of l1+l2 run-length ops per pair (an alignment has at most l1+l2 columns)
			c.scratch_off.resize(nc);
			for (uint32_t k = 0; k < nc; ++k) { c.scratch_off[k] = c.scratch_words; c.scratch_words += (uint64_t)in.l1[c.k0 + k] + in.l2[c.k0 + k]; }
		}
		p.max_chunk_words = std::max(p.max_chunk_words, c.ptr_words);
		p.max_scratch_words = std::max(p.max_scratch_words, c.scratch_words);
		p.max_bnd_elems = std::max(p.max_bnd_elems, c.bnd_elems);
		p.max_prog_words = std::max(p.max_prog_words, c.prog_words);
		p.max_pairs = std::max(p.max_pairs, nc);
	}
	return p;
}

}  // namespace atb2
