// at_fill_affine.cuh -- K1: Gotoh M/L/U(/J) fill for global / local / fit (+jump), sm_100a.
// (included by at_kernels.cuh after the constants)
//
// Inter-pair kernel for SHORT reads (l1 <= 256 rows = 32 lanes x R <= 8 rows); longer reads go
// to the stripe-pipelined K2 (at_wavefront.cuh).  One kernel template, two kinds of score lanes:
//   Lanes<false>  int32   : one pair per warp, every mode.
//   Lanes<true>   s16x2   : TWO pairs per warp, pair A in bits 0-15 and pair B in bits 16-31 of
//                           every register (VIADDMNMX.U16x2 / VIMNMX3.U16x2 DPX instructions);
//                           every mode but fit + jump.  Both pairs share l2 (global / fit: l1 as well, so that
//                           one lane holds the last row of both); -inf is AT_NEG16 inside the 16 bits.
//
// Geometry: lane k owns R consecutive rows; at step t it works on column j = t - k (anti-diagonal
// of R-row blocks).  Per step each lane hands the last row of its strip -- M+o, L and H = max(L, M, U[, J]),
// whose low bits carry its argmax -- to lane k+1 with three __shfl_up_sync.  Target symbols are staged
// through a per-warp shared-memory ring (one entry per column).
//
// The cell itself -- tagged values, one VIADDMNMX per max, pointer nibbles assembled on the FMA pipe -- is
// cell_update() of at_cell.cuh; what this file adds around it:
//   * PROF variant (target alphabet of the shard has at most 4 distinct bytes -- DNA): a per-warp QUERY
//     PROFILE in shared memory, rebuilt per job: word[comb][lane][r] = 8*s(read row, target symbol) for
//     pair A (+ the same for pair B in the high half, comb = codeA*4 + codeB), so the substitution score is one
//     LDS; the target ring holds the byte offset of the column's `comb`.  The ring's first entries are
//     mirrored behind its end, so the steps of one pointer word read it at constant offsets from one base;
//   * fallback variant (any byte alphabet): symbols are pre-shifted (<<8 / <<16), so
//     min(a ^ b, 8|m-u|)  is 0 on a match and the whole substitution penalty otherwise;
//   * lane 0 takes matrix row 0 instead of a neighbour's row through a multiply-add with a 0/1 lane mask
//     (FMA pipe), not a select;
//   * local mode keeps the lane's running maximum of  8*M + (7 - row_in_lane)  with one
//     VIADDMNMX per cell: larger score first, then the smaller row -- together with "first step
//     at which the key reached its final value" this is the reference's first maximum in
//     row-major order (src/alignment.h:830-833).
//
// Reference recurrences: src/alignment.h:451-462 (global), :635-667 (fit), :825-841 (local);
// tie rules SURVEY.md A.0:  M: first strictly greater in order L,M,U,(J|HOME);  L: extend wins
// ties;  U: open wins ties;  J: enter wins ties, entering forbidden on listed target indices.
#pragma once
#include "at_plan.h"      // FillJob

namespace atb2 {

#define AT_RING 512        // target ring entries per warp (two 256-column blocks)
#define AT_RING_MIRROR 8   // its first entries again behind the end: a pointer word's steps never wrap
#define AT_FILL_WARPS 4

// query-profile geometry: words per lane (>= R, even, half of it odd: conflict-free 64-bit loads)
__host__ __device__ constexpr int prof_lane_stride(int R) { return R <= 2 ? 2 : (R <= 6 ? 6 : 10); }
// K1 only: an odd R keeps its rows unpadded and reads them with 32-bit loads (an odd lane stride is
// conflict-free too); the smaller table lets a fifth CTA fit an SM for R = 5
__host__ __device__ constexpr int k1_lane_stride(int R) { return (R & 1) ? R : prof_lane_stride(R); }
__host__ __device__ constexpr int prof_combs(bool packed) { return packed ? 16 : 4; }
// dynamic shared memory of one CTA of at_fill_affine<.., R, .., PACKED, PROF>
__host__ __device__ constexpr size_t fill_smem_bytes(int R, bool packed, bool prof)
{
	return (size_t)AT_FILL_WARPS * (prof ? (size_t)(AT_RING + AT_RING_MIRROR) * 2 + (size_t)prof_combs(packed) * 32 * k1_lane_stride(R) * 4
	                                     : (size_t)(AT_RING + AT_RING_MIRROR) * 4);
}
// ... and of at_fill_affine<.., R, false, false, false, true> (table variant): the same, then the shard's compact table
__host__ __device__ constexpr size_t fill_smem_bytes_table(int R, uint32_t table_bytes) { return fill_smem_bytes(R, false, false) + table_bytes; }

struct FillArgs2 {
	const uint8_t  *q;       const uint64_t *q_off;  const uint32_t *q_len;
	const uint8_t  *t;       const uint64_t *t_off;  const uint32_t *t_len;
	const uint8_t  *jmask;   // fit+jump: 1 where entering J is forbidden, one byte per target symbol
	const uint64_t *j_off;   // [pair] offset of the pair's mask (byte-encoded targets: the same array as t_off)
	const uint8_t  *symmap;  // PROF: byte -> code 0..3 of the shard's target alphabet (256 entries)
	uint32_t        syms;    // PROF: the byte of code c in bits 8c..8c+7
	const FillJob  *jobs;
	uint32_t        n_jobs;
	uint32_t       *counter;
	uint32_t       *ptr;     const uint64_t *ptr_off;   uint32_t pair_base;
	int32_t        *score;   uint32_t *end_i;  uint32_t *end_j;  uint8_t *end_state;
	int             m, u, o, e, jp;
	int             want_ptr;
	uint32_t        k_and, k_or;   // cell_k_and / cell_k_or of the lane type (at_cell.cuh: constants that must stay in registers)
	int             twobit;  // PROF: q / t hold 2-bit codes (AT_SEQ_2BIT, four symbols per byte, byte-aligned records; *_off are byte offsets)
	SubstArgs       sub;     // SCORED: the substitution matrix (at_kernels.cuh)
};

// packed lanes with up to five rows per lane (the 150-row reads of BASELINE config 2 are R = 5): hold ptxas to the 96 registers
// that let five CTAs share an SM -- the shared-memory profile allows exactly five; the other variants to 128 / 168 / 255
// SCORED (substitution matrix, at_batch_*_scored): with PROF the profile words come from the matrix row of the read symbol
// (the cell is unchanged); without PROF (int32 lanes only) the TABLE variant: ac[r] holds the byte offset of the row's read
// code in the shard's compact table (shared memory, after the warps' rings), the ring holds 2 x the column's target code
// (| blacklist bit), and 8 s(i, j) is one LDS.S16 from their sum.
template <int MODE, int R, bool JUMP, bool PACKED, bool PROF, bool SCORED = false>
__global__ void __launch_bounds__(32 * AT_FILL_WARPS, (PACKED && R <= 5) ? 5 : (JUMP && R > 5) ? 2 : (JUMP || R > 6) ? 3 : 4) at_fill_affine(const FillArgs2 a)
{
	static_assert(!SCORED || PROF || !PACKED, "the table variant runs on int32 lanes");
	constexpr bool TABLE = SCORED && !PROF;
	typedef Lanes<PACKED> V;
	typedef typename V::T T;
	static_assert(!PACKED || !JUMP, "packed lanes: no jump state");
	constexpr bool LOCAL = MODE == MODE_LOCAL;
	constexpr uint32_t SPW = V::STEPS_PER_WORD;
	constexpr uint32_t SH = PACKED ? PTR_SH_PACKED : PTR_SH_NIB;           // pointer layout (at_ptr_layout.h)
	static_assert(SPW == 1u << SH, "a lane assembles one pointer word per SPW steps");
	constexpr int LS = k1_lane_stride(R), NC = prof_combs(PACKED);
	constexpr uint32_t COMB_BYTES = 32u * LS * 4u;             // one comb's slice of the profile
	constexpr size_t WARP_BYTES = fill_smem_bytes(R, PACKED, PROF) / AT_FILL_WARPS;
	constexpr int SHIFT = PACKED ? 8 : 16;                     // fallback variant: where a symbol sits in its lane half

	extern __shared__ __align__(16) unsigned char fill_smem[];
	const int lane = threadIdx.x & 31;
	unsigned char *warp_smem = fill_smem + (threadIdx.x >> 5) * WARP_BYTES;
	uint32_t *ring = (uint32_t *)warp_smem;                                   // !PROF: one u32 per column
	uint16_t *ring16 = (uint16_t *)warp_smem;                                 // PROF: byte offset of the column's comb (| blacklist bit)
	uint32_t *prof = (uint32_t *)(warp_smem + (AT_RING + AT_RING_MIRROR) * 2);   // PROF: [NC][32][LS]
	const unsigned char *prof_lane = (const unsigned char *)(prof + lane * LS);
	const unsigned char *tab = fill_smem + (TABLE ? fill_smem_bytes(R, false, false) : 0);      // TABLE: [read code][target code] of 8 s
	if constexpr (TABLE) {
		for (uint32_t x = threadIdx.x; x < a.sub.table_bytes / 16u; x += blockDim.x)
			((uint4 *)tab)[x] = __ldg((const uint4 *)a.sub.table + x);
		__syncthreads();
	}

	const int m = a.m, u = a.u, o = a.o, e = a.e;
	CellConst<PACKED> cc;
	cc.set(o, e, a.jp, a.k_and, a.k_or);
	const T o8 = V::delta(o), e8 = V::delta(e), m8 = V::delta(m);
	T nz = lane ? 1 : 0;                                                      // lane 0 takes matrix row 0 instead of a neighbour
	asm volatile("" : "+r"(nz));                                              // opaque: keep x * nz + b0 a multiply-add (FMA pipe), not a SEL
	const uint32_t mu8 = (uint32_t)(8 * (m >= u ? m - u : u - m)) * (PACKED ? 0x10001u : 1u);     // per half; < 1 << SHIFT (host-checked)
	const int nsg = m >= u ? -1 : 1;                                    // s = m - penalty  (or + when u > m)
	const T ZERO = V::value(0);
	const T NEGV = PACKED ? (T)((uint32_t)(AT_NEG16 * 0x10001) + 0x80008000u) : (T)AT_NEG;      // -inf stand-in (at_cell.cuh)
	const bool want_ptr = a.want_ptr != 0;
	const bool twobit = PROF && a.twobit != 0;

	for (;;) {
		uint32_t job = 0;
		if (lane == 0) job = atomicAdd(a.counter, 1u);
		job = __shfl_sync(0xffffffffu, job, 0);
		if (job >= a.n_jobs) break;
		const FillJob jb = a.jobs[job];
		const uint32_t pA = jb.a, pB = PACKED ? jb.b : jb.a;
		const uint32_t l1A = a.q_len[pA], l1B = a.q_len[pB], l2 = a.t_len[pA];
		const uint8_t *__restrict__ qA = a.q + a.q_off[pA], *__restrict__ qB = a.q + a.q_off[pB];
		const uint8_t *__restrict__ tA = a.t + a.t_off[pA], *__restrict__ tB = a.t + a.t_off[pB];
		const uint8_t *__restrict__ jm = JUMP ? a.jmask + a.j_off[pA] : nullptr;
		uint32_t *__restrict__ ptr = a.ptr + a.ptr_off[pA - a.pair_base];
		const uint32_t t_last = ptr_last_step(l2, SH, JUMP);                  // also the last step the warp runs
		const uint32_t G = ptr_groups(t_last, SH);
		uint32_t *__restrict__ ptrJ = ptr_plane(ptr, 1u, G, R);

		// ring[(j-1) & 511]: packed (tA << 8) | (tB << 24); int32 (tA << 16) | blacklist bit;
		// PROF: byte offset of the column's comb in the profile | blacklist bit
		auto load_block = [&](uint32_t blk) {
			const uint32_t base = blk * 256u;
			if (PROF && twobit) {
				// 2-bit targets resident in HBM: 256 columns = 64 bytes per pair.  Records that start on a 16-byte boundary are
				// read with one 128-bit load per 64 columns (lanes 0-3: pair A, lanes 4-7: pair B) and handed round by shuffle;
				// others with two byte loads per lane.  Lane k turns columns base + 8k .. + 7 into ring entries.
				const uint8_t *pa = tA + (base >> 2), *pb = tB + (base >> 2);
				uint32_t wa = 0, wb = 0;
				if (base < l2) {
					if ((((uintptr_t)tA | (uintptr_t)tB) & 15u) == 0) {
						uint4 v = make_uint4(0, 0, 0, 0);
						const uint32_t need = (min(l2 - base, 256u) + 63u) >> 6;             // 16-byte groups that hold columns of this block
						if (lane < 8 && (uint32_t)(lane & 3) < need) v = __ldg((const uint4 *)((lane < 4 ? pa : pb) + 16 * (lane & 3)));
						const int src = lane >> 3, comp = (lane >> 1) & 3, hi = (lane & 1) * 16;
						const uint32_t xa0 = __shfl_sync(0xffffffffu, v.x, src), xa1 = __shfl_sync(0xffffffffu, v.y, src),
						               xa2 = __shfl_sync(0xffffffffu, v.z, src), xa3 = __shfl_sync(0xffffffffu, v.w, src);
						wa = ((comp == 0 ? xa0 : comp == 1 ? xa1 : comp == 2 ? xa2 : xa3) >> hi) & 0xffffu;
						if (PACKED) {
							const uint32_t xb0 = __shfl_sync(0xffffffffu, v.x, src + 4), xb1 = __shfl_sync(0xffffffffu, v.y, src + 4),
							               xb2 = __shfl_sync(0xffffffffu, v.z, src + 4), xb3 = __shfl_sync(0xffffffffu, v.w, src + 4);
							wb = ((comp == 0 ? xb0 : comp == 1 ? xb1 : comp == 2 ? xb2 : xb3) >> hi) & 0xffffu;
						}
					} else if (base + 8u * lane < l2) {
						wa = (uint32_t)__ldg(pa + 2 * lane) | ((uint32_t)__ldg(pa + 2 * lane + 1) << 8);     // (one byte of slack behind the last record)
						if (PACKED) wb = (uint32_t)__ldg(pb + 2 * lane) | ((uint32_t)__ldg(pb + 2 * lane + 1) << 8);
					}
				}
#pragma unroll
				for (int k = 0; k < 8; ++k) {
					const uint32_t idx = base + 8u * lane + k, slot = idx & (AT_RING - 1);
					uint32_t v = (wa >> (2 * k)) & 3u;
					if (PACKED) v = v * 4u + ((wb >> (2 * k)) & 3u);
					v = idx < l2 ? v * COMB_BYTES : 0u;
					if (JUMP && idx < l2) v |= __ldg(jm + idx) ? 1u : 0u;
					ring16[slot] = (uint16_t)v;
					if (slot < AT_RING_MIRROR) ring16[AT_RING + slot] = (uint16_t)v;
				}
				return;
			}
#pragma unroll
			for (int k = 0; k < 8; ++k) {
				const uint32_t idx = base + k * 32u + lane, slot = idx & (AT_RING - 1);
				if (PROF) {
					uint32_t v = 0;                            // past the end: any comb (those cells are never read back)
					if (idx < l2) {
						v = __ldg(a.symmap + __ldg(tA + idx));
						if (PACKED) v = v * 4u + __ldg(a.symmap + __ldg(tB + idx));
						v *= COMB_BYTES;
						if (JUMP) v |= __ldg(jm + idx) ? 1u : 0u;
					}
					ring16[slot] = (uint16_t)v;
					if (slot < AT_RING_MIRROR) ring16[AT_RING + slot] = (uint16_t)v;
				} else {
					uint32_t v = PACKED ? 0x00010001u : TABLE ? 0u : 0x2u;      // past the end: never equals a symbol (TABLE: target code 0)
					if (idx < l2) {
						if (PACKED) v = ((uint32_t)__ldg(tA + idx) << 8) | ((uint32_t)__ldg(tB + idx) << 24);
						else {
							v = TABLE ? (uint32_t)__ldg(a.sub.tcol + __ldg(tA + idx)) : (uint32_t)__ldg(tA + idx) << 16;
							if (JUMP) v |= __ldg(jm + idx) ? 1u : 0u;
						}
					}
					ring[slot] = v;
					if (slot < AT_RING_MIRROR) ring[AT_RING + slot] = v;
				}
			}
		};

		const uint32_t row0 = lane * R;
		__syncwarp();
		load_block(0);
		load_block(1);

		RowState<PACKED, JUMP> st[R];
		T crow[R];
		uint32_t ac[R];
#pragma unroll
		for (int r = 0; r < R; ++r) {
			const uint32_t ri = row0 + r;
			const int i = (int)ri + 1;
			ac[r] = 0;
			if (PACKED) {
				if (!PROF) {      // fallback variant: the read symbols, pre-shifted (the PROF variant reads them into its profile below)
					const uint32_t ca = ri < l1A ? ((uint32_t)qA[ri] << SHIFT) : 0x0002u;
					const uint32_t cb = ri < l1B ? ((uint32_t)qB[ri] << SHIFT) : 0x0002u;
					ac[r] = ca | (cb << 16);
				}
				// running-max key offset on top of Mk = 8 M + 2: 5 - r for real rows (key = 8 M + 7 - r); -0x8000 sinks
				// padded rows below every real key (per half, two's complement)
				const uint32_t ka = ri < l1A ? (uint32_t)(5 - r) : 0x8000u, kb = ri < l1B ? (uint32_t)(5 - r) : 0x8000u;
				crow[r] = (T)((ka & 0xffffu) | ((kb & 0xffffu) << 16));
			} else {
				if (TABLE) ac[r] = ri < l1A ? __ldg(a.sub.qrow + qA[ri]) : 0u;      // padded rows: any row of the table
				else if (!PROF) ac[r] = ri < l1A ? ((uint32_t)qA[ri] << SHIFT) : 0x4u;
				crow[r] = (T)(ri < l1A ? 5 - r : -(1 << 28));
			}
			// column 0 (left border), tags as cell_update leaves them: mo 3, u 1, h = the winner's
			if (MODE == MODE_GLOBAL)     { st[r].mo = NEGV | V::rep(3); st[r].u = NEGV | V::rep(1); st[r].h = V::value(o + e * i) | V::rep(TAG_L); }   // :432-436
			else if (MODE == MODE_LOCAL) { st[r].mo = ZERO + o8 + V::rep(3); st[r].u = ZERO | V::rep(1); st[r].h = ZERO | V::rep(TAG_L); }             // calloc zeros
			else                         { st[r].mo = NEGV | V::rep(3); st[r].u = NEGV | V::rep(1); st[r].h = NEGV | V::rep(TAG_M); }                  // :612-617
			st[r].j = NEGV; st[r].x = 0; st[r].xj = 0;
			if (PROF) {     // this lane's rows of the query profile: 8*s(read symbol, target symbol of code c)
				uint32_t qa = 0x100u, qb = 0x100u;          // byte of the read symbol (2-bit reads: its code), 0x100 = no such row
				if (ri < l1A) qa = twobit ? ((uint32_t)qA[ri >> 2] >> (2 * (ri & 3))) & 3u : (uint32_t)qA[ri];
				if (PACKED && ri < l1B) qb = twobit ? ((uint32_t)qB[ri >> 2] >> (2 * (ri & 3))) & 3u : (uint32_t)qB[ri];
				int sa[4], sb[4];
#pragma unroll
				for (int c = 0; c < 4; ++c) {
					const uint32_t sy = twobit ? (uint32_t)c : (a.syms >> (8 * c)) & 255u;
					if constexpr (SCORED) {      // the matrix entries of the read and target BYTES (2-bit codes stand for A C G T)
						const uint32_t ty = twobit ? (0x54474341u >> (8 * c)) & 255u : sy;
						const uint32_t ya = twobit ? (0x54474341u >> (8 * (qa & 3u))) & 255u : qa & 255u, yb = twobit ? (0x54474341u >> (8 * (qb & 3u))) & 255u : qb & 255u;
						sa[c] = qa < 0x100u ? 8 * (int)__ldg(a.sub.matrix + ya * 256u + ty) : 0;
						sb[c] = qb < 0x100u ? 8 * (int)__ldg(a.sub.matrix + yb * 256u + ty) : 0;
					} else { sa[c] = 8 * (qa == sy ? m : u); sb[c] = 8 * (qb == sy ? m : u); }
				}
#pragma unroll
				for (int c = 0; c < NC; ++c)
					prof[(c * 32 + lane) * LS + r] = !PACKED ? (uint32_t)sa[c]
					                                 : LOCAL ? (((uint32_t)sa[c >> 2] & 0xffffu) | ((uint32_t)sb[c & 3] << 16))      // fused add: per half
					                                         : (uint32_t)(sa[c >> 2] + sb[c & 3] * 65536);                         // plain add: exact sum
			}
		}
		__syncwarp();
		// what this lane hands down before its first column: its last row at column 0
		T sM = st[R - 1].mo, sH = st[R - 1].h;
		T sL = MODE == MODE_GLOBAL ? (V::value(o + e * (int)(row0 + R)) | V::rep(3)) : (MODE == MODE_LOCAL ? (ZERO | V::rep(3)) : (NEGV | V::rep(3)));
		T pH;      // H(row0, 0): the row above this lane's strip at column 0
		if (row0 == 0) {
			if (MODE == MODE_GLOBAL)     pH = V::value(o < 0 ? 0 : o) | V::rep(o < 0 ? TAG_M : TAG_L);      // max5(L = o, M = 0, U = o)
			else if (MODE == MODE_LOCAL) pH = ZERO | V::rep(TAG_L);
			else                         pH = ZERO | V::rep(TAG_M);                                        // M[0][0] = U[0][0] = 0
		} else {
			if (MODE == MODE_GLOBAL)     pH = V::value(o + e * (int)row0) | V::rep(TAG_L);
			else if (MODE == MODE_LOCAL) pH = ZERO | V::rep(TAG_L);
			else                         pH = NEGV | V::rep(TAG_M);
		}
		// matrix row 0 as lane 0 sees it (zero in every other lane: x = neighbour * nz + b0)
		T b0M, b0L, b0H, b0E = 0;
		if (MODE == MODE_GLOBAL)     { b0M = NEGV | V::rep(3); b0L = NEGV | V::rep(3); b0H = V::value(o) | V::rep(TAG_U); b0E = e8; }      // :437-441, U[0][j] = o + e j
		else if (MODE == MODE_LOCAL) { b0M = ZERO + o8 + V::rep(3); b0L = ZERO | V::rep(3); b0H = ZERO | V::rep(TAG_L); }
		else                         { b0M = ZERO + o8 + V::rep(3); b0L = NEGV | V::rep(3); b0H = ZERO | V::rep(TAG_M); }                  // :619-624
		if (lane) { b0M = 0; b0L = 0; b0H = 0; b0E = 0; }
		const int cap_r = (!LOCAL && lane == (int)((l1A - 1) / R)) ? (int)((l1A - 1) % R) : -1;      // packed global / fit jobs: l1A == l1B
		int hot[R];
#pragma unroll
		for (int r = 0; r < R; ++r) hot[r] = r == cap_r ? 1 : 0;
		T kbest = PACKED ? (T)0 : (T)AT_NEG_INIT;     // below every real key
		T tbest = 0;
		int capM = AT_NEG_INIT, capMj = 0, capL = AT_NEG_INIT, capLj = 0;      // fit, int32 lanes
		T capM2 = 0, capL2 = 0, capMj2 = 0, capLj2 = 0;                        // fit, packed lanes (biased: 0 is below every value)
		T gH = 0;                                                              // global

		// first step at which the running key took its (so far) final value -> column of the running maximum
		auto note_best = [&](const T before, const T after, const uint32_t t) {
			if (PACKED) { const T chg = (T)__vminu2((uint32_t)(after ^ before), 0x10001u) * 0xffffu; tbest = (tbest & ~chg) | ((T)(t * 0x10001u) & chg); }
			else if (after != before) tbest = (T)t;
		};
		// one step of the systolic array.  ring_k: PROF, unchecked: address of the column's ring entry (a constant offset
		// from the word's base); mul / mulj: see cell_update
		// tail: unchecked steps past the last column.  Cells of columns > l2 are computed like any other (on whatever the
		// ring holds there): no cell of the matrix depends on them, their pointers are never read and the end-cell
		// searches test the column -- only local mode's running maximum must not see them.
		auto step = [&](const uint32_t t, const bool checked, const uint16_t *ring_k, const uint32_t mul, const uint32_t mulj, const bool tail) {
			const int j = (int)t - lane;
			// neighbour's last row, or matrix row 0 at column j = t in lane 0 (multiply-add: keeps the ALU pipe free)
			const T rM = __shfl_up_sync(0xffffffffu, sM, 1) * nz + b0M;
			const T rL = __shfl_up_sync(0xffffffffu, sL, 1) * nz + b0L;
			T rH = __shfl_up_sync(0xffffffffu, sH, 1) * nz + b0H;
			if (MODE == MODE_GLOBAL) rH += b0E * (T)t;
			if (checked && t == 0) rH = pH;                // step 0 only primes the pipeline: keep H(row0, 0)
			T D = pH;
			pH = rH;
			if (!checked || (j >= 1 && j <= (int)l2)) {
				uint32_t c;
				if (PROF) c = checked ? (uint32_t)ring16[(uint32_t)(j - 1) & (AT_RING - 1)] : (uint32_t)*ring_k;
				else c = ring[(uint32_t)(j - 1) & (AT_RING - 1)];
				T jadd = 0;
				if (JUMP) { jadd = (c & 1u) ? cc.j_barred : cc.j_enter; c &= ~1u; }      // M[i][j-1] + jump, or barred (:659-665)
				uint32_t pw[LS + 1];                            // PROF: the profile words of this lane's rows for the column's comb
				if (PROF) {
					if (LS & 1) {
						const uint32_t *pp = (const uint32_t *)(prof_lane + c);
#pragma unroll
						for (int r2 = 0; r2 < R; ++r2) pw[r2] = pp[r2];
					} else {
						const uint2 *pp = (const uint2 *)(prof_lane + c);
#pragma unroll
						for (int r2 = 0; r2 < (R + 1) / 2; ++r2) { const uint2 v2 = pp[r2]; pw[2 * r2] = v2.x; pw[2 * r2 + 1] = v2.y; }
					}
				}
				T lup = rL, mo_up = rM;
				T rowM = 0, rowL = 0;                          // fit: M, L of the pair's last row
				const T kold = kbest;
				CellOut<PACKED> out;
#pragma unroll
				for (int r = 0; r < R; ++r) {
					T s8;                                      // 8 s(i, j)
					if (PROF) s8 = (T)pw[r];
					else if (TABLE) s8 = (T)*(const int16_t *)(tab + ac[r] + c);
					else {                                     // tt: 0 on a match, 8|m-u| otherwise (per half); plain-add form
						const T tt = PACKED ? (T)__vminu2(ac[r] ^ c, mu8) : (T)min(ac[r] ^ c, mu8);
						s8 = tt * (T)nsg + m8;
					}
					D = cell_update<LOCAL, JUMP, PACKED, PROF>(cc, st[r], D, s8, lup, mo_up, jadd, mul, mulj, out);
					lup = out.lk; mo_up = out.mo;
					if (LOCAL) kbest = V::addmax(out.mk, crow[r], kbest);
					// fit: the pair's last row is row cap_r of ONE lane: pick its values with a one-hot multiply-add per
					// row (FMA pipe) instead of compares and selects in every row; the search itself runs once per step
					if (MODE == MODE_FIT) { rowM += out.mk * (T)hot[r]; rowL += out.lk * (T)hot[r]; }
					if (MODE == MODE_GLOBAL) { if (r == cap_r && j == (int)l2) gH = out.h; }   // (cheaper than the one-hot form here)
				}
				sM = out.mo; sL = out.lk; sH = out.h;
				if (MODE == MODE_FIT && !PACKED && cap_r >= 0 && j < (int)l2) {       // column l2 excluded (:677, :684)
					const int rm = (int)rowM & ~7, rl = (int)rowL & ~7;               // drop the tags: M and L are compared with each other at the end
					if (rm > capM) { capM = rm; capMj = j; }
					if (rl > capL) { capL = rl; capLj = j; }
				}
				if (MODE == MODE_FIT && PACKED) {      // both pairs at once; lanes without the last row carry 0, which never wins
					const bool in = j >= 1 && j < (int)l2;
					const T rm = in ? (rowM & ~V::rep(7)) : (T)0, rl = in ? (rowL & ~V::rep(7)) : (T)0;
					const T j2 = (T)((uint32_t)j * 0x10001u);
					const T nm = V::vmax(capM2, rm), nl = V::vmax(capL2, rl);         // strictly greater only: the smallest column among maxima
					const T cm = (T)__vminu2((uint32_t)(nm ^ capM2), 0x10001u) * 0xffffu, cl = (T)__vminu2((uint32_t)(nl ^ capL2), 0x10001u) * 0xffffu;
					capMj2 = (capMj2 & ~cm) | (j2 & cm); capLj2 = (capLj2 & ~cl) | (j2 & cl);
					capM2 = nm; capL2 = nl;
				}
				if (LOCAL && tail) kbest = j > (int)l2 ? kold : kbest;
				if (LOCAL) note_best(kold, kbest, t);
			} else {
#pragma unroll
				for (int r = 0; r < R; ++r) { st[r].x *= mul; if (JUMP) st[r].xj *= mulj; }
			}
		};

		for (uint32_t tb = 0; tb <= t_last; tb += SPW) {
			if ((tb & 255u) == 32u && tb > 32u) {     // block tb/256 - 1 is dead: refill its slots two blocks ahead
				__syncwarp();
				load_block(tb / 256u + 1u);
				__syncwarp();
			}
			if (tb >= 32u) {      // every lane is inside the matrix or past its last column: no range checks
				const uint16_t *rb = ring16 + ((tb - (uint32_t)lane - 1u) & (AT_RING - 1));      // column j - 1 of step tb; + k for step tb + k (mirrored tail)
				if (tb + SPW - 1u <= l2) {
					if (PACKED) {
#pragma unroll
						for (uint32_t k = 0; k < SPW; ++k) step(tb + k, false, rb + k, k == 0 ? 0u : 16u, 2u, false);
					} else {      // int32 lanes: 8 steps per word; unroll by 4 only (instruction-cache footprint)
#pragma unroll 4
						for (uint32_t k = 0; k < SPW; ++k) step(tb + k, false, rb + k, 16u, 2u, false);
					}
				} else if (PACKED) {      // the last ~32 steps: some lanes are past column l2
#pragma unroll
					for (uint32_t k = 0; k < SPW; ++k) step(tb + k, false, rb + k, k == 0 ? 0u : 16u, 2u, true);
				} else {
#pragma unroll 2
					for (uint32_t k = 0; k < SPW; ++k) step(tb + k, false, rb + k, 16u, 2u, true);
				}
			} else {
#pragma unroll 1
				for (uint32_t k = 0; k < SPW; ++k) step(tb + k, true, nullptr, (PACKED && k == 0) ? 0u : 16u, 2u, false);
			}
			if (want_ptr) {
				uint32_t *w = ptr_at(ptr, 0u, 0u, tb >> SH, lane, R);          // one stripe
#pragma unroll
				for (int r = 0; r < R; ++r) w[r] = ptr_word(st[r].x);
			}
			if (JUMP && want_ptr && ((tb + SPW - 1u) & 31u) == 31u) {
				uint32_t *w = ptr_at(ptrJ, 0u, 0u, tb >> PTR_SH_JUMP, lane, R);
#pragma unroll
				for (int r = 0; r < R; ++r) w[r] = jump_word(st[r].xj);
			}
		}

		// ---- end cell (reference: :466-469 global, :673-690 fit, running max :830-833 local) ----
		if (LOCAL) {
#pragma unroll
			for (int h = 0; h < (PACKED ? 2 : 1); ++h) {
				int key, tcol;
				if (PACKED) { key = (int)((kbest >> (16 * h)) & 0xffffu) - 0x8000; tcol = (int)((tbest >> (16 * h)) & 0xffffu) - lane; }
				else { key = (int)kbest; tcol = (int)tbest - lane; }
				int sc = -1, row = 0x7fffffff, col = 0;
				if (key >= 0) { sc = key >> 3; row = (int)row0 + (7 - (key & 7)) + 1; col = tcol; }
#pragma unroll
				for (int d = 16; d >= 1; d >>= 1) {
					const int osc = __shfl_xor_sync(0xffffffffu, sc, d);
					const int orow = __shfl_xor_sync(0xffffffffu, row, d);
					const int ocol = __shfl_xor_sync(0xffffffffu, col, d);
					if (osc > sc || (osc == sc && orow < row)) { sc = osc; row = orow; col = ocol; }
				}
				const uint32_t p = h ? pB : pA;
				if (lane == 0 && (h == 0 || pB != pA)) { a.score[p] = sc; a.end_i[p] = row; a.end_j[p] = col; a.end_state[p] = ST_MID; }
			}
		} else {
			const int owner = (int)((l1A - 1) / R);
			if (lane == owner) {
#pragma unroll
				for (int h = 0; h < (PACKED ? 2 : 1); ++h) {
					const uint32_t p = h ? pB : pA;
					if (h && pB == pA) break;
					auto half = [&](T v) -> int { return PACKED ? (int)(((uint32_t)v >> (16 * h)) & 0xffffu) - 0x8000 : (int)v; };
					if (MODE == MODE_GLOBAL) { const int g = half(gH); a.score[p] = g >> 3; a.end_i[p] = l1A; a.end_j[p] = l2; a.end_state[p] = (uint8_t)(3 - (g & 3)); }
					else {
						const int cM = PACKED ? half(capM2) : capM, cL = PACKED ? half(capL2) : capL;
						const int jM = PACKED ? (int)(((uint32_t)capMj2 >> (16 * h)) & 0xffffu) : capMj, jL = PACKED ? (int)(((uint32_t)capLj2 >> (16 * h)) & 0xffffu) : capLj;
						const bool useL = cL > cM;            // L replaces M only when strictly greater (:685)
						a.score[p] = (useL ? cL : cM) >> 3; a.end_i[p] = l1A; a.end_j[p] = useL ? jL : jM;
						a.end_state[p] = useL ? ST_LOW : ST_MID;
					}
				}
			}
		}
		__syncwarp();
	}
}

}  // namespace atb2
