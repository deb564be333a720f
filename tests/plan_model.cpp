// Host build of aligntools/c_b200/csrc/at_plan.h (the batch plan of a shard) for tests/test_plan_cpu.py: plain C entry
// points over the header's functions.  A plan is returned as one flat list of integers (plan_model_plan).
#include "../aligntools/c_b200/csrc/at_plan.h"

using namespace atb2;

static PlanIn plan_in(uint32_t n, const uint32_t *l1, const uint32_t *l2, int mode, int traceback, int jump, const int32_t *lo,
                      const int32_t *hi, int bits, uint32_t bits_r, const int32_t *prm, int no_p16, int allow_uniform, int pair_major,
                      uint64_t budget, std::vector<PairBand> &bands)
{
	PlanIn in;
	in.n = n; in.l1 = l1; in.l2 = l2; in.mode = mode; in.traceback = traceback != 0; in.jump = jump != 0;
	if (lo) {
		bands.resize(n);
		for (uint32_t k = 0; k < n; ++k) band_clip(l1[k], l2[k], lo[k], hi[k], bands[k].lo, bands[k].hi);
		in.band = bands.data();
	}
	in.bits = bits != 0; in.bits_r = bits_r;
	at_params p{prm[0], prm[1], prm[2], prm[3], 0, jump};
	in.p16 = p16_rule(mode, p, in.jump, no_p16 != 0);
	in.allow_uniform = allow_uniform != 0; in.pair_major = pair_major != 0;
	in.budget_words = budget;
	return in;
}

extern "C" {
// lo / hi: the caller's bands (NULL: unbanded), clipped here as the runtime does; prm: m, u, o, e.  Writes need_words and
// the plan, serialised as below, into out[0 .. cap) and returns the number of words it takes.
uint64_t plan_model_plan(uint32_t n, const uint32_t *l1, const uint32_t *l2, int mode, int traceback, int jump, const int32_t *lo,
                         const int32_t *hi, int bits, uint32_t bits_r, const int32_t *prm, int no_p16, int allow_uniform, int pair_major,
                         uint64_t budget, uint64_t *out, uint64_t cap)
{
	std::vector<PairBand> bands;
	const PlanIn in = plan_in(n, l1, l2, mode, traceback, jump, lo, hi, bits, bits_r, prm, no_p16, allow_uniform, pair_major, budget, bands);
	const Plan p = make_plan(in);
	std::vector<uint64_t> v;
	auto vec = [&](const std::vector<uint64_t> &x) { v.push_back(x.size()); v.insert(v.end(), x.begin(), x.end()); };
	v.push_back(need_words(in));
	v.insert(v.end(), {(uint64_t)p.uniform, (uint64_t)p.u.packed, p.u.R, p.u.words_per_job, p.u.scratch_per_pair, p.cells, p.max_chunk_words,
	                   p.max_scratch_words, p.max_bnd_elems, p.max_prog_words, p.max_pairs, p.fail_pair, p.fail_words});
	v.push_back(p.rclass.size());
	v.insert(v.end(), p.rclass.begin(), p.rclass.end());
	v.push_back(p.chunks.size());
	for (const PlanChunk &c : p.chunks) {
		v.insert(v.end(), {c.k0, c.k1, c.ptr_words, c.bnd_elems, c.prog_words, c.scratch_words, c.launches.size()});
		for (const PlanLaunch &l : c.launches) {
			v.insert(v.end(), {(uint64_t)l.kind, (uint64_t)l.r, l.cells, l.n, l.prog_base, l.jobs.size()});
			for (const FillJob &j : l.jobs) v.insert(v.end(), {j.a, j.b});
			v.push_back(l.tasks.size());
			for (const WaveTask &t : l.tasks) v.insert(v.end(), {t.pair, t.stripe, t.prev, t.reserved});
		}
		vec(c.ptr_off); vec(c.bnd_off); vec(c.scratch_off);
	}
	for (uint64_t k = 0; k < v.size() && k < cap; ++k) out[k] = v[k];
	return v.size();
}

// The uniform closed form of pair k: ptr_off, scratch_off, class byte, whether it writes a job, the job and its pair indices
void plan_model_uniform_pair(int packed, uint32_t R, uint64_t words_per_job, uint64_t scratch_per_pair, uint32_t n, uint32_t k, uint64_t *out)
{
	UniformPlan u;
	u.packed = packed != 0; u.R = R; u.words_per_job = words_per_job; u.scratch_per_pair = scratch_per_pair;
	const UniformPair p = uniform_pair(u, n, k);
	const uint64_t r[] = {p.ptr_off, p.scratch_off, p.rclass, p.writes_job, p.job, p.fj.a, p.fj.b};
	for (int x = 0; x < 7; ++x) out[x] = r[x];
}

void plan_model_cut(const uint64_t *prefix, uint64_t n, uint64_t lo, uint64_t hi, uint64_t parts, uint64_t *cut)
{
	std::vector<uint64_t> pre(prefix, prefix + n + 1), c;
	cut_by_prefix(pre, lo, hi, parts, c);
	for (uint64_t d = 0; d <= parts; ++d) cut[d] = c[d];
}

uint32_t plan_model_bits_r(const uint32_t *l1, uint32_t n, uint64_t warp_slots) { return choose_bits_r(l1, n, warp_slots); }
}
