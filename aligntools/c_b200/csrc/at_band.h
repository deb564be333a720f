// at_band.h -- geometry of a BANDED pair (overlap or global): the caller's static band lo <= j - i <= hi on the diagonals
// of the DP matrix, and what it means for K2's stripes and K3's pointer blocks.  Host + device: the runtime sizes pointer
// blocks and counts cells, K2 fills and hands off, K3 walks with these functions and nothing else
// (tests/test_banded_oracle.py compiles this header with g++ and checks the properties below without a GPU).
//
// A stripe (RPP rows) sweeps only its column WINDOW [c0, c1]: the columns of its in-band cells.  The window of rows
// ia..ib is [max(1, ia + lo), min(l2, ib + hi)]; stripes without in-band cells form a run at the top and one at the
// bottom of the pair (the in-band rows are one interval).  The stripe's steps start at t0 = (c0 - 1) rounded down to a
// 32-column hand-off block (lane 0 primes its diagonal input at column c0 - 1, as at column 0 unbanded) and end at
// (c1 + 31) | 31.  Pointer words are stored relative to t0: `groups` blocks of 2^wsh steps, 32 * R words each, stripes
// packed one after the other (wsh = 4: overlap's 2-bit pointers, 16 steps per word; wsh = 3: the affine kernel's nibbles,
// 8 steps per word).  A stripe publishes the last row of its window; every other column of that row is out of
// band (-inf), so the stripe below waits only for columns in [c0, c1] of the stripe above.
#pragma once
#include <stdint.h>
#include "at_cell.cuh"      // AT_HD

namespace atb2 {

struct BandWin {
	uint32_t c0, c1;        // column window, 1 <= c0 <= c1 <= l2
	uint32_t t0;            // first step: a multiple of 32, <= c0 - 1
	uint32_t groups;        // pointer groups (2^wsh steps) of the stripe
};

// The band clipped to the matrix's diagonals [1 - l1, l2 - 1], in 64 bits (int32 extremes do not overflow); an empty
// band comes back as (1, 0).  The clipped values fit int32 (l1, l2 < 2^27).
AT_HD void band_clip(uint32_t l1, uint32_t l2, int64_t lo, int64_t hi, int32_t &elo, int32_t &ehi)
{
	const int64_t a = lo > 1 - (int64_t)l1 ? lo : 1 - (int64_t)l1;
	const int64_t b = hi < (int64_t)l2 - 1 ? hi : (int64_t)l2 - 1;
	if (a > b) { elo = 1; ehi = 0; return; }
	elo = (int32_t)a; ehi = (int32_t)b;
}

// Window of stripe s (rows s*RPP+1 .. min((s+1)*RPP, l1)) of a clipped band; false when the stripe has no in-band cell.
AT_HD bool band_stripe(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, BandWin &w, uint32_t wsh = 4)
{
	if (elo > ehi) return false;
	const int64_t ia = (int64_t)s * RPP + 1, ibx = ((int64_t)s + 1) * RPP, ib = ibx < (int64_t)l1 ? ibx : (int64_t)l1;
	if (ia > ib) return false;
	const int64_t a = ia + elo > 1 ? ia + elo : 1, b = ib + ehi < (int64_t)l2 ? ib + ehi : (int64_t)l2;
	if (a > b) return false;
	w.c0 = (uint32_t)a; w.c1 = (uint32_t)b;
	w.t0 = (w.c0 - 1u) & ~31u;
	w.groups = ((w.c1 + 31u - w.t0) >> wsh) + 1u;
	return true;
}

AT_HD uint32_t band_t_last(const BandWin &w) { return (w.c1 + 31u) | 31u; }

// pointer words of stripe s (0 when it is empty)
AT_HD uint64_t band_stripe_words(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, uint32_t wsh = 4)
{
	BandWin w;
	return band_stripe(l1, l2, elo, ehi, RPP, s, w, wsh) ? (uint64_t)w.groups * RPP : 0;
}

// word offset of stripe s in the pair's pointer block (the words of the stripes above it)
AT_HD uint64_t band_stripe_off(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t s, uint32_t wsh = 4)
{
	uint64_t off = 0;
	for (uint32_t x = 0; x < s; ++x) off += band_stripe_words(l1, l2, elo, ehi, RPP, x, wsh);
	return off;
}

AT_HD uint64_t band_pair_words(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi, uint32_t RPP, uint32_t wsh = 4)
{
	return band_stripe_off(l1, l2, elo, ehi, RPP, (l1 + RPP - 1) / RPP, wsh);
}

// The column the first stripe below a producer waits for before it starts (three hand-off blocks past its own first
// step, or `lag` columns if that is more), kept inside the producer's window: the producer publishes exactly [c0, c1].
AT_HD uint32_t band_first_wait(const BandWin &prod, uint32_t t0, uint32_t lag)
{
	const uint32_t c = t0 + (lag > 96u ? lag : 96u);
	return c < prod.c0 ? prod.c0 : (c > prod.c1 ? prod.c1 : c);
}

// cells (i, j), 1 <= i <= l1, 1 <= j <= l2, with j - i <= D
AT_HD uint64_t band_cells_below(int64_t l1, int64_t l2, int64_t D)
{
	uint64_t n = 0;
	const int64_t a = 1 - D > 1 ? 1 - D : 1, b = l2 - D < l1 ? l2 - D : l1;      // rows with 1 <= i + D <= l2
	if (a <= b) n += (uint64_t)((b - a + 1) * (a + b + 2 * D) / 2);
	const int64_t f = l2 - D + 1 > 1 ? l2 - D + 1 : 1;                                // rows with i + D > l2: whole rows
	if (f <= l1) n += (uint64_t)(l1 - f + 1) * (uint64_t)l2;
	return n;
}

// in-band cells of a pair (clipped band)
AT_HD uint64_t band_cells(uint32_t l1, uint32_t l2, int32_t elo, int32_t ehi)
{
	if (elo > ehi) return 0;
	return band_cells_below(l1, l2, ehi) - band_cells_below(l1, l2, (int64_t)elo - 1);
}

}  // namespace atb2
