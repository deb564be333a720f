// Host build of aligntools/c_b200/csrc/at_band.h (the banded overlap geometry shared by the runtime, K2 and K3) for
// tests/test_banded_oracle.py: plain C entry points over the header's functions.
#include "../aligntools/c_b200/csrc/at_band.h"

using namespace atb2;

extern "C" {
void band_model_clip(uint32_t l1, uint32_t l2, int64_t lo, int64_t hi, int32_t *out) { band_clip(l1, l2, lo, hi, out[0], out[1]); }
// out: c0, c1, t0, groups, t_last; returns 1 when the stripe has a window
int band_model_stripe(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, uint32_t *out)
{
	BandWin w;
	if (!band_stripe(l1, l2, elo, ehi, RPP, s, w)) return 0;
	out[0] = w.c0; out[1] = w.c1; out[2] = w.t0; out[3] = w.groups; out[4] = band_t_last(w);
	return 1;
}
uint64_t band_model_words(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s) { return band_stripe_words(l1, l2, elo, ehi, RPP, s); }
uint64_t band_model_off(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s) { return band_stripe_off(l1, l2, elo, ehi, RPP, s); }
uint64_t band_model_pair_words(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP) { return band_pair_words(l1, l2, elo, ehi, RPP); }
uint64_t band_model_cells(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi) { return band_cells(l1, l2, elo, ehi); }
uint32_t band_model_first_wait(uint32_t c0, uint32_t c1, uint32_t t0, uint32_t lag)
{
	BandWin p = {c0, c1, 0, 0};
	return band_first_wait(p, t0, lag);
}
}
