// at_kernels.cuh -- sm_100a device code of the alignTools DP core.
//
// K1  at_fill_affine<MODE,R,JUMP,PACKED,PROF> : Gotoh M/L/U(/J) fill of short pairs (l1 <= 256), one pair
//                                    (or two, packed s16x2) per warp; PROF = query profile in shared
//                                    memory for targets of <= 4 distinct bytes   (at_fill_affine.cuh)
// K2  at_wave_affine<MODE,JUMP,PROF> : the same recurrences for long pairs: stripes of 256 rows
//     at_wave_linear<MODE,R,PROF>    pipelined over warps / CTAs, TMA-staged target tiles; the
//                                    single-plane kernel (overlap max-plus / edit min-plus) serves
//                                    every length;
//     at_wave_edit_bits<R>         : bit-parallel (Myers) unit-cost edit distance in the same stripe
//                                    pipeline                                   (at_wavefront.cuh)
//     SCORED (last template flag of K1 / K2's affine and linear kernels): substitution-matrix scoring -- the profile
//                                    from the matrix (PROF), or a compact byte table in shared memory (SubstArgs)
// K3  at_traceback_walk            : device traceback, one thread per pair chases the pointers
//                                    once and leaves the reversed run-length ops in scratch;
//     at_traceback_emit            : one warp per pair writes the dense CIGAR and replays it over
//                                    the sequences into the gapped strings r1 / r2.
// helpers: at_scan_offsets (offsets of the dense outputs), at_symbol_set (which bytes occur: picks the
//     PROF / bit-parallel variants), at_build_jmask (jump blacklist), at_unpack_2bit (at_runtime.cu).
//
// Geometry (SURVEY.md Appendix D).  Rows i <-> read s1, columns j <-> target s2.  A warp
// sweeps a STRIPE of 32*R rows over all columns as a systolic array: lane k owns rows
// row0+k*R .. +R-1 and at step t works on column j = t - k, so the 32 lanes sit on one
// anti-diagonal of R-row blocks.  The last row of each lane (M+o, L, H=max(L,M,U[,J]) and
// the 2-bit argmax code of H) moves to lane k+1 with __shfl_up_sync once per step; lane 31
// parks it in a boundary row that lane 0 reads back on the next stripe (reads longer than
// 32*R rows).  Per-row state (M+o, U, H, code, J of column j-1) stays in registers.
//
// Traceback pointers: at_ptr_layout.h defines every pointer-block layout the fills store and K3 reads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "at_cell.cuh"      // Lanes<>, cell_update(), AT_NEG: the cell arithmetic shared by K1 and K2
#include "at_ptr_layout.h"  // pointer-block layouts shared by the runtime, K1, K2 and K3
#include "at_band.h"        // banded overlap / global: stripe windows and pointer layout shared by the runtime, K2 and K3

// traceback walker's look-ahead: how far ahead (steps) and how often (every PERIOD-th step, a power of two) it prefetches
#ifndef AT_TB_PF_AHEAD
#define AT_TB_PF_AHEAD 24
#endif
#ifndef AT_TB_PF_PERIOD
#define AT_TB_PF_PERIOD 8
#endif

namespace atb2 {

enum { MODE_GLOBAL = 0, MODE_LOCAL = 1, MODE_FIT = 2, MODE_OVERLAP = 3, MODE_EDIT = 4 };
enum { ST_LOW = 0, ST_MID = 1, ST_UPP = 2, ST_JUMP = 3 };   // also the 2-bit pointerM codes
enum { CIG_M = 0, CIG_I = 1, CIG_D = 2, CIG_N = 3 };

// Substitution-matrix scoring (at_batch_*_scored), read by the SCORED instantiations of K1 and K2 only.  Profile variants
// read `matrix` when they build their profile; the table variants copy `table` into shared memory and index it with
// qrow[read byte] + tcol[target byte] (byte offsets: the shard's alphabets compacted to codes, rows of int16 values).
struct SubstArgs {
	const int8_t   *matrix;       // the caller's 256 x 256 table, s(a, b) = matrix[a * 256 + b]
	const int16_t  *table;        // [read code][target code]: 8 s (affine kernels) or 4 s (overlap)
	const uint32_t *qrow;         // read byte -> byte offset of its row in `table`
	const uint16_t *tcol;         // target byte -> byte offset of its column within a row (2 x code)
	uint32_t        table_bytes;  // size of `table`, a multiple of 16
};

}  // namespace atb2
#include "at_fill_affine.cuh"
#include "at_wavefront.cuh"
namespace atb2 {

// ------------------------------------------------------------------------------------
// K3 traceback (reference: trace_back_gla :372-412, trace_back_fit_affine_jump :558-592,
// trace_back_local_affine :766-800, trace_back_overlap :896-922).  The pointer is read at
// the cell BEFORE the move; local emits the HOME cell's column; global flushes the
// remaining target then read symbols after the loop.
// ------------------------------------------------------------------------------------
struct TraceArgs {
	const uint8_t  *q;  const uint64_t *q_off;  const uint32_t *q_len;
	const uint8_t  *t;  const uint64_t *t_off;  const uint32_t *t_len;
	const uint32_t *ptr; const uint64_t *ptr_off;
	const uint8_t  *rclass;    // [pair] layout class (at_ptr_layout.h: ptr_class): the fill's R and packed half
	uint32_t        pair_base, n_pairs;   // chunk
	const uint32_t *end_i, *end_j; const uint8_t *end_state;
	uint32_t       *beg_i, *beg_j;
	uint32_t       *n_ops, *n_cols;       // [pair]
	uint32_t       *scratch;              // reversed run-length ops, slot of l1+l2 ops per pair
	const uint64_t *scratch_off;          // [n_chunk] chunk-local slot offsets
	const uint64_t *ops_off, *cols_off;   // [n_chunk+1] exclusive scans (chunk-local index)
	uint32_t       *cigar;                // dense ops of the chunk
	uint8_t        *aln1, *aln2;          // dense columns of the chunk
	int             mode, jump;
	int             lookahead;             // few, long walks (latency-bound): prefetch the pointer sectors ahead of the walker
	int             twobit;                // q / t hold 2-bit codes (four symbols per byte, A C G T = 0..3; byte-aligned records)
	const int2     *band;                  // banded walker: [pair] clipped band (lo, hi) on j - i (at_band.h)
};

// Cursor over a pair's pointer block (layout: at_ptr_layout.h).  The word of cell (i, j) is
//   ptr[rowA(i) + ((j + lane(i)) >> SH) * RPP],   rowA(i) = PtrRow::base,
// with stripe / lane / r the position of row i-1 in the fill's geometry.  A traceback only ever moves
// to row i-1, so rowA is kept incrementally (it just decrements, except across a stripe) instead of
// being re-derived with two integer divisions per visited cell.
struct PtrView {
	const uint32_t *ptr, *ptrJ;
	uint32_t R, RPP, G, GJ, half;
	uint32_t r, lane;            // position of row i-1: row within the lane, lane within the stripe
	size_t rowA, rowJ;           // word offsets of row i-1 in the nibble / 2-bit block and in the jump-bit plane
	__device__ __forceinline__ void seek(uint32_t i) {            // i >= 1
		const PtrRow w = ptr_row(i, R);
		lane = w.lane; r = w.r;
		rowA = w.base(G, R);
		rowJ = w.base(GJ, R);
	}
	__device__ __forceinline__ void up() {                        // row i-1 -> row i-2 (no-op bookkeeping when leaving row 0)
		if (r) { --r; --rowA; --rowJ; return; }
		r = R - 1;
		if (lane) { --lane; --rowA; --rowJ; return; }
		lane = 31;                                                // previous stripe: its last lane, last row
		rowA = rowA - (size_t)G * RPP + (RPP - 1);
		rowJ = rowJ - (size_t)GJ * RPP + (RPP - 1);
	}
	// Pull the sectors the walk will most likely need AHEAD steps from now into L2/L1: the path mostly runs
	// along the diagonal (rows and columns both move back) or along a row (gap / jump runs).  A thread-serial
	// pointer chase otherwise pays a full HBM round trip per new sector.
	__device__ __forceinline__ void prefetch(uint32_t i, uint32_t j, int sh) const {
		constexpr uint32_t AHEAD = AT_TB_PF_AHEAD;
		if (i <= AHEAD + 1 || j <= AHEAD + 1 || rowA < AHEAD) return;
		const uint32_t lane_then = lane - min(lane, (AHEAD + R - 1 - r) / R);               // rows per lane: R (approximate across a stripe edge)
		const uint32_t *diag = ptr + (rowA - AHEAD) + (size_t)((j - AHEAD + lane_then) >> sh) * RPP;
		const uint32_t *row = ptr + rowA + (size_t)((j - AHEAD + lane) >> sh) * RPP;
		asm volatile("prefetch.global.L2 [%0];" :: "l"(diag));
		asm volatile("prefetch.global.L2 [%0];" :: "l"(row));
	}
	__device__ __forceinline__ uint32_t nib(uint32_t j) const {
		const uint32_t t = j + lane;
		if (half) {   // packed s16x2: 4 steps x 2 pairs per word, single stripe
			const uint32_t w = __ldg(ptr + rowA + (size_t)(t >> PTR_SH_PACKED) * RPP);
			return (w >> (16 * (half - 1) + ptr_shift(t, PTR_SH_PACKED, 4))) & 15u;
		}
		const uint32_t w = __ldg(ptr + rowA + (size_t)(t >> PTR_SH_NIB) * RPP);
		return (w >> ptr_shift(t, PTR_SH_NIB, 4)) & 15u;
	}
	__device__ __forceinline__ uint32_t jbit(uint32_t j) const {
		const uint32_t t = j + lane;
		const uint32_t w = __ldg(ptrJ + rowJ + (size_t)(t >> PTR_SH_JUMP) * RPP);
		return (w >> ptr_shift(t, PTR_SH_JUMP, 1)) & 1u;
	}
	// Banded pairs (at_band.h): stripe s's words start at off(s) and count groups of 2^wsh steps (overlap 16, global 8) from
	// the stripe's first step t0, so rowA folds in - (t0 >> wsh) * RPP and two() / nib() stay as they are.  Crossing to the
	// stripe above moves `off` back by that stripe's words.
	uint32_t l1, l2, stripe, t0, wsh;
	int32_t elo, ehi;
	uint64_t off;
	__device__ __forceinline__ void band_base() {                 // rowA of row 0 of lane 0 of `stripe` (row -1 of a stripe without a window: never read)
		BandWin w;
		const uint32_t t = band_stripe(l1, l2, elo, ehi, RPP, stripe, w, wsh) ? w.t0 : 0u;
		t0 = t;
		rowA = (size_t)off - (size_t)(t >> wsh) * RPP;
	}
	__device__ __forceinline__ void seek_band(uint32_t i) {       // i >= 1
		const uint32_t ri = i - 1, rem = ri % RPP;
		stripe = ri / RPP; lane = rem / R; r = rem - lane * R;
		off = band_stripe_off(l1, l2, elo, ehi, RPP, stripe, wsh);
		band_base();
		rowA += (size_t)lane * R + r;
	}
	__device__ __forceinline__ void up_band() {
		if (r) { --r; --rowA; return; }
		r = R - 1;
		if (lane) { --lane; --rowA; return; }
		lane = 31;
		if (stripe == 0) return;                                  // leaving row 1: the walk stops at row 0
		--stripe;
		off -= band_stripe_words(l1, l2, elo, ehi, RPP, stripe, wsh);
		band_base();
		rowA += RPP - 1;
	}
	__device__ __forceinline__ uint32_t two(uint32_t j) const {   // overlap: 2 bits, 16 steps per word
		const uint32_t t = j + lane;
		const uint32_t w = __ldg(ptr + rowA + (size_t)(t >> PTR_SH_2BIT) * RPP);
		return (w >> ptr_shift(t, PTR_SH_2BIT, 2)) & 3u;
	}
};

// run-length encoder writing ops in walk (= reverse) order
struct RunWriter {
	uint32_t *dst; uint32_t n_ops, n_cols, run, op;
	__device__ __forceinline__ void flush() { if (run) dst[n_ops++] = (run << 4) | op; run = 0; }
	__device__ __forceinline__ void col(uint32_t o) { if (run && o != op) flush(); op = o; ++run; ++n_cols; }
};

// One thread per pair: chase the pointers once, leave the reversed CIGAR in the pair's scratch slot.
// BESIDE_FILL only makes two distinct functions: the <true> instances are given the fill kernels'
// shared-memory carve-out (they run beside another stream's persistent fill grid in the pipelined
// path), the <false> instances keep the default carve-out -- the walk lives on L1 hits.
// BANDED (overlap or global with a per-pair band): the pointer block has the banded layout (PtrView::seek_band / up_band)
// and a walk that reaches a cell outside the band stops, as at row 0 -- cells on a finite path are in band.  Global's
// flush after the walk is the unbanded one.
// EDIT (AT_OUT_EDIT_PATH; a.mode is ignored): the edit walk over the layout of the kernel that filled the shard --
// EDIT_WALK_LIN: at_wave_linear<MODE_EDIT, .., PTR>, overlap's 2-bit codes (LEFT 0, DIAG 1, UP 2);
// EDIT_WALK_BITS: at_wave_edit_bits<R, PTR>, a uint2 (LEFT, DIAG) of bit planes per block column (at_ptr_layout.h).
// From (l1, l2) while i > 0 && j > 0: LEFT -> D, DIAG -> M, UP -> I; then global's flush.
enum { EDIT_WALK_NONE = 0, EDIT_WALK_LIN = 1, EDIT_WALK_BITS = 2 };

template <bool BESIDE_FILL, bool BANDED = false, int EDIT = EDIT_WALK_NONE>
__global__ void __launch_bounds__(128) at_traceback_walk(const TraceArgs a)
{
	// Few long walks: ONE walker per warp (lane 0), so that a walk is not held back at every step by the
	// slowest of 31 unrelated walks sharing its warp (divergent states, the odd cache miss).  Many short
	// walks: one per thread.
	const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x;
	if (a.lookahead && (threadIdx.x & 31u)) return;
	const uint32_t k = a.lookahead ? gtid >> 5 : gtid;
	if (k >= a.n_pairs) return;
	const uint32_t p = a.pair_base + k;
	const uint32_t l1 = a.q_len[p], l2 = a.t_len[p];
	PtrView pv;
	pv.R = ptr_class_r(a.rclass[p]); pv.RPP = 32 * pv.R; pv.half = ptr_class_half(a.rclass[p]);
	const uint32_t n_stripes = ptr_stripes(l1, pv.R);
	const bool jump = a.jump != 0;
	if (a.mode == MODE_OVERLAP) { pv.G = ptr_groups(ptr_last_step(l2, PTR_SH_2BIT), PTR_SH_2BIT); pv.GJ = 0; }
	else if (pv.half) { pv.G = ptr_groups(ptr_last_step(l2, PTR_SH_PACKED), PTR_SH_PACKED); pv.GJ = 0; }
	else { const uint32_t tl = ptr_last_step(l2, PTR_SH_NIB, jump); pv.G = ptr_groups(tl, PTR_SH_NIB); pv.GJ = ptr_groups(tl, PTR_SH_JUMP); }
	pv.ptr = a.ptr + a.ptr_off[k];
	pv.ptrJ = ptr_plane(pv.ptr, n_stripes, pv.G, pv.R);
	RunWriter w;
	w.dst = a.scratch + a.scratch_off[k]; w.n_ops = w.n_cols = w.run = 0; w.op = 0;
	uint32_t i = a.end_i[p], j = a.end_j[p], state = a.end_state[p], tick = 3;
	if constexpr (EDIT == EDIT_WALK_BITS) {
		const uint32_t R = pv.R, G = edit_bits_groups(l2);
		const uint2 *base = (const uint2 *)(a.ptr + a.ptr_off[k]);
		while (i > 0 && j > 0) {
			// the path mostly runs along the diagonal: pull the word AT_TB_PF_AHEAD cells up-left into L2
			if (a.lookahead && !(++tick & (AT_TB_PF_PERIOD - 1u)) && i > AT_TB_PF_AHEAD && j > AT_TB_PF_AHEAD) {
				uint32_t b2;
				asm volatile("prefetch.global.L2 [%0];" :: "l"(base + edit_bits_index(i - AT_TB_PF_AHEAD, j - AT_TB_PF_AHEAD, R, G, b2)));
			}
			uint32_t b;
			const uint2 pl = __ldg(base + edit_bits_index(i, j, R, G, b));
			if ((pl.x >> b) & 1u)      { --j; w.col(CIG_D); }                 // LEFT
			else if ((pl.y >> b) & 1u) { --i; --j; w.col(CIG_M); }            // DIAG
			else                       { --i; w.col(CIG_I); }                 // UP
		}
	} else if constexpr (EDIT == EDIT_WALK_LIN) {
		pv.G = ptr_groups(ptr_last_step(l2, PTR_SH_2BIT), PTR_SH_2BIT); pv.GJ = 0;
		if (i) pv.seek(i);
		while (i > 0 && j > 0) {
			if (a.lookahead && !(++tick & (AT_TB_PF_PERIOD - 1u))) pv.prefetch(i, j, PTR_SH_2BIT);
			const uint32_t c = pv.two(j);                                      // bit 1: UP, bit 0: DIAG, 0: LEFT
			if (c & 2u)      { --i; pv.up(); w.col(CIG_I); }
			else if (c & 1u) { --i; pv.up(); --j; w.col(CIG_M); }
			else             { --j; w.col(CIG_D); }
		}
	} else if constexpr (BANDED) {
		const bool ov = a.mode == MODE_OVERLAP;
		pv.l1 = l1; pv.l2 = l2; pv.elo = a.band[p].x; pv.ehi = a.band[p].y; pv.wsh = ov ? PTR_SH_2BIT : PTR_SH_NIB;
		if (i && j) pv.seek_band(i);
		while (j > 0) {
			if (i == 0) break;
			if ((int)j - (int)i < pv.elo || (int)j - (int)i > pv.ehi) break;      // out of band: not on a finite path
			if (a.lookahead && !(++tick & (AT_TB_PF_PERIOD - 1u)) && pv.lane * pv.R + pv.r >= AT_TB_PF_AHEAD && j > pv.t0 + AT_TB_PF_AHEAD + 1)
				pv.prefetch(i, j, (int)pv.wsh);                                    // rows and columns of the look-ahead stay in the stripe's block
			if (ov) {
				const uint32_t c = pv.two(j);
				if (c & 2u)      { --i; pv.up_band(); w.col(CIG_I); }
				else if (c & 1u) { --i; pv.up_band(); --j; w.col(CIG_M); }
				else             { --j; w.col(CIG_D); }
			} else {                                                               // global (:377-397)
				const uint32_t nb = pv.nib(j);
				if (state == ST_LOW)      { state = (nb & 4u) ? ST_MID : ST_LOW; --i; pv.up_band(); w.col(CIG_I); }
				else if (state == ST_MID) { state = nb & 3u; --i; pv.up_band(); --j; w.col(CIG_M); }
				else if (state == ST_UPP) { state = (nb & 8u) ? ST_UPP : ST_MID; --j; w.col(CIG_D); }
				else break;                                                        // no JUMP / HOME state in global: corrupt pointers
			}
		}
	} else {
	if (i) pv.seek(i);

	if (a.mode == MODE_OVERLAP) {
		while (j > 0) {                                   // :899
			if (i == 0) break;                            // row 0 is -inf (:937): unreachable on a finite path
			if (a.lookahead && !(++tick & (AT_TB_PF_PERIOD - 1u))) pv.prefetch(i, j, PTR_SH_2BIT);      // every AT_TB_PF_PERIOD-th step: a sector holds eight rows of a lane block
			const uint32_t c = pv.two(j);                 // bit 1: RIGHT beat both; bit 0: DIAGONAL beat LEFT
			if (c & 2u)      { --i; pv.up(); w.col(CIG_I); }                  // RIGHT
			else if (c & 1u) { --i; pv.up(); --j; w.col(CIG_M); }             // DIAGONAL
			else             { --j; w.col(CIG_D); }                           // LEFT
		}
	} else {
		bool home = false;
		for (;;) {
			const bool go = a.mode == MODE_FIT ? (i > 0) : (i > 0 && j > 0);   // :562 | :377, :771
			if (!go || home) break;
			if (j == 0 && state != ST_LOW) break;         // only reachable with corrupt pointers: never index s2[-1]
			if (state == ST_JUMP && jump) {               // a jump run reads only the 1-bit plane (32 columns per word)
				if (a.lookahead && j > 160u) asm volatile("prefetch.global.L2 [%0];" :: "l"(pv.ptrJ + pv.rowJ + (size_t)((j - 128u + pv.lane) >> PTR_SH_JUMP) * pv.RPP));
				state = pv.jbit(j) ? ST_JUMP : ST_MID; --j; w.col(CIG_N);
				continue;
			}
			if (a.lookahead && !(++tick & (AT_TB_PF_PERIOD - 1u))) pv.prefetch(i, j, pv.half ? PTR_SH_PACKED : PTR_SH_NIB);
			const uint32_t nb = pv.nib(j);
			if (state == ST_LOW)      { state = (nb & 4u) ? ST_MID : ST_LOW; --i; pv.up(); w.col(CIG_I); }
			else if (state == ST_MID) {
				const uint32_t pm = nb & 3u;
				--i; pv.up(); --j; w.col(CIG_M);
				if (pm == 3 && a.mode == MODE_LOCAL) home = true;              // HOME: column emitted, then stop (:788-791)
				else state = pm;
			}
			else if (state == ST_UPP) { state = (nb & 8u) ? ST_UPP : ST_MID; --j; w.col(CIG_D); }
			else                      { state = pv.jbit(j) ? ST_JUMP : ST_MID; --j; w.col(CIG_N); }
		}
	}
	}
	a.beg_i[p] = i; a.beg_j[p] = j;
	if (EDIT || a.mode == MODE_GLOBAL) {                  // flush (:398-407): rest of the target, then rest of the read
		while (j > 0) { --j; w.col(CIG_D); }
		while (i > 0) { --i; w.col(CIG_I); }
	}
	w.flush();
	a.n_ops[p] = w.n_ops; a.n_cols[p] = w.n_cols;
}

// One warp per pair: reverse the scratch ops into the dense CIGAR and, on request, replay them
// forward over the two sequences to write the gapped strings r1 / r2 (coalesced).
// Edit paths are launched with a.mode = MODE_GLOBAL: like global's, they start at (0, 0) after the flush.
template <bool BESIDE_FILL>
__global__ void __launch_bounds__(128) at_traceback_emit(const TraceArgs a)
{
	const uint32_t k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const int lane = threadIdx.x & 31;
	if (k >= a.n_pairs) return;
	const uint32_t p = a.pair_base + k;
	const uint32_t n = a.n_ops[p];
	const uint32_t *src = a.scratch + a.scratch_off[k];
	if (a.cigar) {
		uint32_t *dst = a.cigar + a.ops_off[k];
		for (uint32_t x = lane; x < n; x += 32) dst[x] = src[n - 1 - x];
	}
	if (a.aln1) {
		const uint8_t *q = a.q + a.q_off[p], *tg = a.t + a.t_off[p];
		uint8_t *a1 = a.aln1 + a.cols_off[k], *a2 = a.aln2 + a.cols_off[k];
		uint32_t i = a.mode == MODE_GLOBAL ? 0 : a.beg_i[p], j = a.mode == MODE_GLOBAL ? 0 : a.beg_j[p], col = 0;
		for (uint32_t x = 0; x < n; ++x) {
			const uint32_t op = src[n - 1 - x], len = op >> 4, code = op & 15u;
			const bool gap1 = code == CIG_D || code == CIG_N, gap2 = code == CIG_I;
			for (uint32_t c = lane; c < len; c += 32) {
				uint8_t x = (uint8_t)'-', y = (uint8_t)'-';
				if (!gap1) { const uint32_t k = i + c; x = a.twobit ? (uint8_t)"ACGT"[(q[k >> 2] >> (2 * (k & 3))) & 3] : q[k]; }
				if (!gap2) { const uint32_t k = j + c; y = a.twobit ? (uint8_t)"ACGT"[(tg[k >> 2] >> (2 * (k & 3))) & 3] : tg[k]; }
				a1[col + c] = x; a2[col + c] = y;
			}
			col += len; if (!gap1) i += len; if (!gap2) j += len;
		}
	}
}

// Exclusive offsets of two per-pair count arrays (CIGAR ops, alignment columns) of a chunk:
// off[0] = 0, off[k+1] = off[k] + cnt[k].  Block 0 scans the ops, block 1 the columns; one block of
// 256 threads walks its array 2048 counts at a time.  Used for chunks of up to a few 100 k pairs
// (larger ones go through CUB): unlike a library kernel it can be given the fill kernels'
// shared-memory carve-out, so it runs beside a persistent fill grid of another stream.
__global__ void __launch_bounds__(256) at_scan_offsets(const uint32_t *cnt_ops, const uint32_t *cnt_cols, uint32_t n,
                                                       uint64_t *off_ops, uint64_t *off_cols)
{
	// 256 threads x 8 counts per pass: small enough in threads and registers to sit beside a fill grid
	constexpr uint32_t IPT = 8, TILE = 256 * IPT;
	const uint32_t *cnt = blockIdx.x ? cnt_cols : cnt_ops;
	uint64_t *off = blockIdx.x ? off_cols : off_ops;
	__shared__ uint64_t warp_sum[8];
	__shared__ uint64_t carry_sh;
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	if (threadIdx.x == 0) { carry_sh = 0; off[0] = 0; }
	__syncthreads();
	for (uint32_t base = 0; base < n; base += TILE) {
		const uint32_t k0 = base + threadIdx.x * IPT;
		uint64_t v[IPT];
		uint64_t run = 0;
#pragma unroll
		for (uint32_t x = 0; x < IPT; ++x) { run += (k0 + x < n) ? cnt[k0 + x] : 0u; v[x] = run; }
		uint64_t incl = run;                                  // inclusive scan of the thread totals over the warp
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) { const uint64_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
		if (lane == 31) warp_sum[wid] = incl;
		__syncthreads();
		uint64_t before_warps = 0;
#pragma unroll
		for (int w = 0; w < 8; ++w) if (w < wid) before_warps += warp_sum[w];
		const uint64_t before = carry_sh + before_warps + (incl - run);
#pragma unroll
		for (uint32_t x = 0; x < IPT; ++x) if (k0 + x < n) off[k0 + x + 1] = before + v[x];
		__syncthreads();
		if (threadIdx.x == 255) carry_sh = before + run;
		__syncthreads();
	}
}

// Which byte values occur in a buffer (256-bit set).  The fill kernels switch to their query-profile
// variant when the shard's targets use at most four distinct symbols.
__global__ void __launch_bounds__(256) at_symbol_set(const uint8_t *bytes, uint64_t n, uint32_t *set8)
{
	__shared__ uint32_t sh[8];
	if (threadIdx.x < 8) sh[threadIdx.x] = 0;
	__syncthreads();
	uint32_t loc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
	const uint64_t n16 = n / 16;
	const uint4 *v = (const uint4 *)bytes;                  // device buffers are 256-byte aligned
	for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n16; k += (uint64_t)gridDim.x * blockDim.x) {
		const uint4 x = __ldg(v + k);
		const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
		for (int q = 0; q < 4; ++q)
#pragma unroll
			for (int b = 0; b < 4; ++b) { const uint32_t c = (w[q] >> (8 * b)) & 255u; loc[c >> 5] |= 1u << (c & 31u); }
	}
	if (blockIdx.x == 0)
		for (uint64_t k = n16 * 16 + threadIdx.x; k < n; k += blockDim.x) { const uint32_t c = bytes[k]; loc[c >> 5] |= 1u << (c & 31u); }
#pragma unroll
	for (int q = 0; q < 8; ++q) if (loc[q]) atomicOr(&sh[q], loc[q]);
	__syncthreads();
	if (threadIdx.x < 8 && sh[threadIdx.x]) atomicOr(&set8[threadIdx.x], sh[threadIdx.x]);
}

// Plan arrays of a UNIFORM shard (every pair has the same l1 and the same l2, all on K1): what the host otherwise
// builds pair by pair and uploads -- the job list, the pointer-block / scratch offsets, the layout class -- is
// closed form (uniform_pair, at_plan.h), so the device writes it itself (no host loops, no pageable uploads on the
// set-up path).
__global__ void at_plan_uniform(uint32_t n, const UniformPlan u, FillJob *jobs, uint64_t *ptr_off, uint64_t *bnd_off, uint64_t *scratch_off, uint8_t *rclass)
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= n) return;
	const UniformPair p = uniform_pair(u, n, k);
	ptr_off[k] = p.ptr_off;
	bnd_off[k] = 0;
	if (scratch_off) scratch_off[k] = p.scratch_off;
	rclass[k] = p.rclass;
	if (p.writes_job) jobs[p.job] = p.fj;
}

// fit+jump: expand the per-pair blacklists into a byte mask aligned with the target bytes.
// `mark`: 1 = the listed indices are barred (the reference's behaviour), 0 = they are the only ones allowed (whitelist:
// the mask was preset to ones).
__global__ void at_build_jmask(const int32_t *sites, const uint64_t *site_off, const uint64_t *t_off,
                               const uint32_t *t_len, uint32_t n_pairs, uint8_t *jmask, uint8_t mark)
{
	const uint32_t p = blockIdx.x;
	if (p >= n_pairs) return;
	const uint64_t lo = site_off[p], hi = site_off[p + 1];
	for (uint64_t k = lo + threadIdx.x; k < hi; k += blockDim.x) {
		const int32_t s = sites[k];
		if (s >= 0 && (uint32_t)s < t_len[p]) jmask[t_off[p] + s] = mark;
	}
}

}  // namespace atb2
