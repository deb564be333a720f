// Host build of aligntools/c_b200/csrc/at_ptr_layout.h (the unbanded pointer-block layouts shared by the runtime, K1, K2
// and K3) for tests/test_ptr_layout_cpu.py: plain C entry points over the header's functions.
#include "../aligntools/c_b200/csrc/at_ptr_layout.h"

using namespace atb2;

extern "C" {
uint32_t ptr_model_last_step(uint32_t l2, uint32_t sh, int jump) { return ptr_last_step(l2, sh, jump != 0); }
uint32_t ptr_model_groups(uint32_t last, uint32_t sh) { return ptr_groups(last, sh); }
uint64_t ptr_model_plane_words(uint32_t stripes, uint32_t G, uint32_t R) { return ptr_plane_words(stripes, G, R); }
uint64_t ptr_model_pair_words(uint32_t l1, uint32_t l2, uint32_t R, uint32_t sh, int jump) { return ptr_pair_words(l1, l2, R, sh, jump != 0); }
uint64_t ptr_model_packed_job_words(uint32_t l2, uint32_t R) { return ptr_packed_job_words(l2, R); }
uint32_t ptr_model_edit_bits_groups(uint32_t l2) { return edit_bits_groups(l2); }
uint32_t ptr_model_edit_bits_last_step(uint32_t l2) { return edit_bits_last_step(l2); }
uint64_t ptr_model_edit_bits_words(uint32_t l1, uint32_t l2, uint32_t R) { return edit_bits_pair_words(l1, l2, R); }
uint32_t ptr_model_class(uint32_t R, uint32_t half) { return ptr_class(R, half); }
uint32_t ptr_model_class_r(uint32_t c) { return ptr_class_r((uint8_t)c); }
uint32_t ptr_model_class_half(uint32_t c) { return ptr_class_half((uint8_t)c); }

// Every cell (i, j) of an l1 x l2 pair, row-major, in a plane of 2^sh-step words of `bits`-bit codes with G groups per
// stripe: word[] relative to the plane and shift[] as K3 reads them (ptr_row, PtrRow::base, ptr_shift).  Returns the
// number of cells whose word differs from the one the fill stores (ptr_index).
uint64_t ptr_model_cells(uint32_t l1, uint32_t l2, uint32_t R, uint32_t G, uint32_t sh, uint32_t bits, uint64_t *word, uint32_t *shift)
{
	uint64_t bad = 0, k = 0;
	for (uint32_t i = 1; i <= l1; ++i) {
		const PtrRow w = ptr_row(i, R);
		for (uint32_t j = 1; j <= l2; ++j, ++k) {
			const uint32_t t = j + w.lane;
			word[k] = w.base(G, R) + (uint64_t)(t >> sh) * (32u * R);
			shift[k] = ptr_shift(t, sh, bits);
			bad += word[k] != ptr_index(w.stripe, G, t >> sh, (int)w.lane, (int)R, (int)w.r);
		}
	}
	return bad;
}

// The same for a bit-parallel edit block: uint2 index and bit of every cell (edit_bits_index)
void ptr_model_edit_bits_cells(uint32_t l1, uint32_t l2, uint32_t R, uint32_t G, uint64_t *slot, uint32_t *bit)
{
	uint64_t k = 0;
	for (uint32_t i = 1; i <= l1; ++i)
		for (uint32_t j = 1; j <= l2; ++j, ++k) slot[k] = edit_bits_index(i, j, R, G, bit[k]);
}
}
