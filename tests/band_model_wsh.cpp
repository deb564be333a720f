// Host build of aligntools/c_b200/csrc/at_band.h with an explicit pointer-word shift (wsh = 4: overlap's 16 steps per
// word; wsh = 3: the affine kernel's 8 steps per word, banded global) for tests/test_banded_global_oracle.py.
#include "../aligntools/c_b200/csrc/at_band.h"

using namespace atb2;

extern "C" {
// out: c0, c1, t0, groups, t_last; returns 1 when the stripe has a window
int band_wsh_stripe(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, uint32_t wsh, uint32_t *out)
{
	BandWin w;
	if (!band_stripe(l1, l2, elo, ehi, RPP, s, w, wsh)) return 0;
	out[0] = w.c0; out[1] = w.c1; out[2] = w.t0; out[3] = w.groups; out[4] = band_t_last(w);
	return 1;
}
uint64_t band_wsh_words(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, uint32_t wsh) { return band_stripe_words(l1, l2, elo, ehi, RPP, s, wsh); }
uint64_t band_wsh_off(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, uint32_t wsh) { return band_stripe_off(l1, l2, elo, ehi, RPP, s, wsh); }
uint64_t band_wsh_pair_words(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t wsh) { return band_pair_words(l1, l2, elo, ehi, RPP, wsh); }
}
