// at_ptr_layout.h -- layout of an UNBANDED pair's traceback pointer block: how many words the runtime reserves for it,
// where the fill kernels (K1, K2) store a cell's code and where the walker (K3) reads it back.  Host + device, no CUDA
// includes (tests/test_ptr_layout_cpu.py compiles this header with g++ and checks the properties below without a GPU).
// Banded blocks (at_band.h) count their groups from a stripe's first step, with the word shifts named here.
//
// Steps.  A warp sweeps a STRIPE of RPP = 32 R rows over all columns; lane k owns rows k R .. k R + R - 1 of the stripe
// and at step t works on column j = t - k, so codes are stored in SKEWED coordinates (step = column + lane).  Lane 31
// reaches column l2 at step l2 + 31; a stripe's block runs to that step rounded up to a whole word.
//
// Words.  The codes of 2^sh consecutive steps of one row are packed into a 32-bit word, the earliest step in the top
// bits, and a stripe's words form `groups` blocks of 2^sh steps, stored as
//   word[((stripe * G + group) * 32 + lane) * R + r]
// with the R words of a lane's block contiguous: a warp flush writes one dense 128 R-byte run, and a diagonal traceback
// move (row - 1, column - 1) stays inside the same 32-byte sector most of the time.  The layouts:
//   * int32 nibbles (K1 int32 lanes, K2 affine): one nibble per cell, bits 0-1 = pointerM (0 LOW, 1 MID, 2 UPP,
//     3 HOME|JUMP), bit 2 = pointerL is MID (gap opened), bit 3 = pointerU is UPP (gap extended); reference planes:
//     src/alignment.h:44-47, values :27-34.  8 steps per word.
//   * the jump plane (fit+jump): one bit per cell (pointerJ is JUMP), 32 steps per word, the same addressing with its own
//     groups, placed after the nibble plane's stripes * G * RPP words.  Both planes end on the same step, (l2 + 31) | 31.
//   * packed s16x2 (K1 packed lanes): the nibbles of 4 steps of pair A in bits 0-15 and of pair B in bits 16-31 of one
//     word; one stripe, one block for the job's two pairs.
//   * 2-bit codes (overlap, edit paths of the cell-by-cell kernel): 16 steps per word.
//   * bit-parallel edit paths (at_wave_edit_bits<R, true>): every block column yields min3's argmin for its 32 cells as
//     two bit planes (edit_bits_ptr, at_cell.cuh: LEFT = Ph, DIAG = ~Ph & (Eq | (Pv & ~Mh)), UP = neither), stored as one
//     uint2 (LEFT, DIAG) per (32-row block, step) in skewed coordinates -- step t = j + 2 lane + 1, as the lanes run:
//       uint2 index = (((stripe * G + t / 16) * R + r) * 16 + t % 16) * 32 + lane,
//     so one store per block column writes 256 contiguous bytes across the warp (full sectors, no staging).  A stripe is
//     1024 R rows (32 lanes x R blocks of 32 rows) and runs to step (l2 + 63) | 15, so a pair's block is 2 bits per cell
//     of its stripes (rows rounded up to 1024 R).
//
// Layout class: one byte per pair from the runtime to K3, R in bits 0-3; bits 4-5: 0 = int32 / 2-bit / bit-parallel
// layout, 1 / 2 = packed s16x2 layout, the pair in the low / high half.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include "at_cell.cuh"      // AT_HD

namespace atb2 {

// log2 of the steps per pointer word; banded blocks (at_band.h) take wsh = PTR_SH_2BIT (overlap) or PTR_SH_NIB (global)
constexpr uint32_t PTR_SH_PACKED = 2u;     // packed s16x2 nibbles
constexpr uint32_t PTR_SH_NIB = 3u;        // int32 nibbles
constexpr uint32_t PTR_SH_2BIT = 4u;       // 2-bit codes
constexpr uint32_t PTR_SH_JUMP = 5u;       // jump plane

// last step of a stripe's block of 2^sh-step words; with the jump plane rounded up to a whole jump word.  K1 runs its
// steps to this one.
AT_HD uint32_t ptr_last_step(uint32_t l2, uint32_t sh, bool jump = false)
{
	const uint32_t mask = jump ? 31u : (1u << sh) - 1u;
	return (l2 + 31u) | mask;
}
// groups of a stripe (words per row) for steps 0 .. last in words of 2^sh steps
AT_HD uint32_t ptr_groups(uint32_t last, uint32_t sh) { return (last >> sh) + 1u; }
AT_HD uint32_t ptr_stripes(uint32_t l1, uint32_t R) { return (l1 + 32u * R - 1u) / (32u * R); }
// words of `stripes` stripes of G groups: one plane of a pair's block, and the offset of the plane after it
AT_HD uint64_t ptr_plane_words(uint32_t stripes, uint32_t G, uint32_t R) { return (uint64_t)stripes * G * (32u * R); }

// words of a pair's int32-nibble (sh = PTR_SH_NIB, + the jump plane with `jump`) or 2-bit (PTR_SH_2BIT) block
AT_HD uint64_t ptr_pair_words(uint32_t l1, uint32_t l2, uint32_t R, uint32_t sh, bool jump)
{
	const uint32_t stripes = ptr_stripes(l1, R), last = ptr_last_step(l2, sh, jump);
	return ptr_plane_words(stripes, ptr_groups(last, sh), R) + (jump ? ptr_plane_words(stripes, ptr_groups(last, PTR_SH_JUMP), R) : 0u);
}
// words of a packed job's block (one stripe, shared by the job's two pairs)
AT_HD uint64_t ptr_packed_job_words(uint32_t l2, uint32_t R) { return ptr_plane_words(1u, ptr_groups(ptr_last_step(l2, PTR_SH_PACKED), PTR_SH_PACKED), R); }

// word index of row r of `lane`'s block of `group` in `stripe`
AT_HD size_t ptr_index(uint32_t stripe, uint32_t G, uint32_t group, int lane, int R, int r = 0)
{
	return ((size_t)(stripe * G + group) * 32 + lane) * R + r;
}
// the fills' stores: the lane's R words of `group`, and the start of the plane after `stripes` stripes (the jump plane)
template <typename T> AT_HD T *ptr_at(T *p, uint32_t stripe, uint32_t G, uint32_t group, int lane, int R) { return p + ptr_index(stripe, G, group, lane, R); }
template <typename T> AT_HD T *ptr_plane(T *p, uint32_t stripes, uint32_t G, uint32_t R) { return p + ptr_plane_words(stripes, G, R); }

// Cell (i, j), i >= 1: row i - 1 is row r of `lane` in `stripe` (ptr_row).  Its code is in word base(G, R) + (t >> sh) * RPP
// of the plane, t = j + lane, at bit ptr_shift(t, sh, bits) (packed: + 16 for pair B) -- the word ptr_index(stripe, G,
// t >> sh, lane, R, r) the fill stored.
struct PtrRow {
	uint32_t stripe, lane, r;
	AT_HD size_t base(uint32_t G, uint32_t R) const { return (size_t)stripe * G * (32u * R) + (size_t)lane * R + r; }
};
AT_HD PtrRow ptr_row(uint32_t i, uint32_t R)
{
	const uint32_t ri = i - 1, stripe = ri / (32u * R), rem = ri - stripe * (32u * R), lane = rem / R;
	return PtrRow{stripe, lane, rem - lane * R};
}
// bit of step t's code (`bits` wide) in its word of 2^sh steps: the earliest step in the top bits
AT_HD uint32_t ptr_shift(uint32_t t, uint32_t sh, uint32_t bits) { return bits * ((1u << sh) - 1u - (t & ((1u << sh) - 1u))); }

// layout class byte: R and the packed half (0: not packed, 1 / 2: pair A / B)
AT_HD uint8_t ptr_class(uint32_t R, uint32_t half) { return (uint8_t)(R | (half << 4)); }
AT_HD uint32_t ptr_class_r(uint8_t c) { return c & 15u; }
AT_HD uint32_t ptr_class_half(uint8_t c) { return (c >> 4) & 3u; }

// bit-parallel edit paths (stripes of G = edit_bits_groups(l2) groups of 16 steps)
AT_HD constexpr uint32_t edit_bits_rows(uint32_t R) { return 1024u * R; }           // rows per stripe
AT_HD uint32_t edit_bits_last_step(uint32_t l2) { return (l2 + 63u) | 15u; }     // lane 31 reaches column l2 at step l2 + 63
AT_HD uint32_t edit_bits_groups(uint32_t l2) { return (edit_bits_last_step(l2) >> 4) + 1u; }
AT_HD uint64_t edit_bits_pair_words(uint32_t l1, uint32_t l2, uint32_t R)
{
	const uint64_t stripes = (l1 + edit_bits_rows(R) - 1u) / edit_bits_rows(R);
	return stripes * edit_bits_groups(l2) * edit_bits_rows(R);
}
// uint2 index of block r of `lane` at step t of `stripe`
AT_HD size_t edit_bits_slot(uint32_t stripe, uint32_t G, uint32_t t, uint32_t R, uint32_t r, uint32_t lane)
{
	return ((((size_t)stripe * G + (t >> 4)) * R + r) * 16 + (t & 15u)) * 32 + lane;
}
// uint2 index of cell (i, j), i, j >= 1; `bit` receives the cell's bit
AT_HD size_t edit_bits_index(uint32_t i, uint32_t j, uint32_t R, uint32_t G, uint32_t &bit)
{
	const uint32_t ri = i - 1, RPP = edit_bits_rows(R), s = ri / RPP, rem = ri - s * RPP;
	const uint32_t lane = rem / (32u * R), r = (rem >> 5) - lane * R, t = j + 2u * lane + 1u;
	bit = rem & 31u;
	return edit_bits_slot(s, G, t, R, r, lane);
}

}  // namespace atb2
