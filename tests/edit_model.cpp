// edit_model.cpp -- TEST INFRASTRUCTURE: host-side model of the edit-path pointer derivations.
//
// Compiles aligntools/c_b200/csrc/at_cell.cuh with g++ and runs its two edit-path helpers over whole matrices:
//   edit_bits_model  the bit-parallel column update of at_wave_edit_bits (32-row blocks, the horizontal difference carried
//                    from block to block as in the kernel) with edit_bits_ptr deriving the pointer planes;
//   edit_cell_model  the cell-by-cell min3 of at_wave_linear<MODE_EDIT, .., PTR> with edit_min3_tagged.
// Both return the 2-bit code (LEFT 0, DIAG 1, UP 2) of every cell; tests/test_edit_model.py compares them with a scalar
// min3 on random cases.  Not part of the product.
//   g++ -O2 -shared -fPIC -o tests/_build/libedit_model.so tests/edit_model.cpp
#include "../aligntools/c_b200/csrc/at_cell.cuh"

#include <vector>

using namespace atb2;

// s1: rows (l1), s2: columns (l2).  top[j-1] in {-1, 0, +1}: M(0, j) - M(0, j-1), the horizontal difference entering the
// first block (the row above a stripe); M(i, 0) = i.  code[(i-1) * l2 + (j-1)]; last[j] = M(l1, j), j = 0..l2.
extern "C" int edit_bits_model(const uint8_t *s1, int l1, const uint8_t *s2, int l2, const int8_t *top, uint8_t *code, int32_t *last)
{
	const int nb = (l1 + 31) / 32;
	std::vector<uint32_t> Pv(nb, 0xffffffffu), Mv(nb, 0u);
	last[0] = l1;
	for (int j = 1; j <= l2; ++j) {
		uint32_t hp = top[j - 1] > 0, hn = top[j - 1] < 0;
		for (int r = 0; r < nb; ++r) {
			uint32_t eq = 0;
			for (int b = 0; b < 32; ++b)
				if (32 * r + b < l1 && s1[32 * r + b] == s2[j - 1]) eq |= 1u << b;
			// the kernel's column update (at_wavefront.cuh, at_wave_edit_bits: `column`)
			uint32_t Eq = eq;
			const uint32_t Xv = Eq | Mv[r];
			Eq |= hn;
			const uint32_t Xh = (((Eq & Pv[r]) + Pv[r]) ^ Pv[r]) | Eq;
			uint32_t Ph = Mv[r] | ~(Xh | Pv[r]);
			uint32_t Mh = Pv[r] & Xh;
			uint32_t left, diag;
			edit_bits_ptr(eq, Pv[r], Ph, Mh, left, diag);
			for (int b = 0; b < 32 && 32 * r + b < l1; ++b) {
				const int i = 32 * r + b + 1;
				code[(size_t)(i - 1) * l2 + (j - 1)] = (uint8_t)(((left >> b) & 1u) ? 0 : ((diag >> b) & 1u) ? 1 : 2);
				if (i == l1) last[j] = last[j - 1] + (int)((Ph >> b) & 1u) - (int)((Mh >> b) & 1u);
			}
			const uint32_t op = Ph >> 31, on = Mh >> 31;
			Ph = (Ph << 1) | hp;
			Mh = (Mh << 1) | hn;
			Pv[r] = Mh | ~(Xv | Ph);
			Mv[r] = Ph & Xv;
			hp = op; hn = on;
		}
	}
	return 0;
}

// min3 with substitution cost u on a mismatch (0 on a match), unit gaps, M(i, 0) = i, M(0, j) = j.  Returns M(l1, l2).
extern "C" int edit_cell_model(const uint8_t *s1, int l1, const uint8_t *s2, int l2, int u, uint8_t *code)
{
	std::vector<int> prev(l2 + 1), cur(l2 + 1);
	for (int j = 0; j <= l2; ++j) prev[j] = j;
	for (int i = 1; i <= l1; ++i) {
		cur[0] = i;
		for (int j = 1; j <= l2; ++j) {
			const int s = s1[i - 1] == s2[j - 1] ? 0 : u;
			const int vt = edit_min3_tagged(cur[j - 1], prev[j - 1] + s, prev[j]);
			cur[j] = vt >> 2;
			code[(size_t)(i - 1) * l2 + (j - 1)] = (uint8_t)(vt & 3);
		}
		prev.swap(cur);
	}
	return prev[l2];
}
