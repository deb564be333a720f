// at_wavefront.cuh -- K2: intra-pair anti-diagonal wavefront fill for long sequences, sm_100a.
// (included by at_kernels.cuh after the constants)
//
// A pair is cut into STRIPES of 32*R rows.  Every (pair, stripe) is a task; the persistent grid
// claims tasks IN ORDER from an atomic queue, one warp per task.  The queue lists stripe after stripe
// across the launch's pairs (order_wave_tasks, at_plan.h): stripes of one pair that happen to be
// resident together run concurrently on different warps / CTAs / SMs, each at least two 32-column blocks
// behind the one above; stripes claimed later find their predecessor finished.  Inside a
// stripe the warp is the same systolic array as K1 (lane k owns R rows, column j = t - k).
//
//   * target tiles (and the jump blacklist) are staged by TMA: one elected lane issues
//     cp.async.bulk global -> shared for the next 256-column tile into a two-slot ring and the
//     warp waits on the slot's mbarrier just before the first lane enters the tile; 2-bit resident
//     targets arrive as 64 packed bytes per tile and are expanded into the same byte ring;
//   * the last row of a stripe (lane 31) is parked in a shared-memory stage, flushed 32 columns
//     at a time with one coalesced store to the pair's boundary slab (L2 resident, two slabs
//     alternating by stripe parity) and published with a release of the task's progress word;
//   * the next stripe polls that word, pulls the 32-column block with one coalesced
//     ld.global.cg a block ahead of its use and feeds lane 0 from a shared-memory ring;
//   * traceback pointers go to HBM exactly as in K1 (nibbles / 2-bit codes in skewed coordinates,
//     one dense 128*R-byte run per warp flush), so K3 walks both kernels' output.
//
// Deadlock freedom: tasks are claimed in queue order by warps that are all resident (grid =
// occupancy x SMs), a warp only ever waits for a task that precedes its own in the queue (WaveTask::prev),
// and stripe 0 of a pair waits for nothing.
//
// Reference recurrences: src/alignment.h:451-462 (global), :635-667 (fit), :825-841 (local),
// :940-949 (overlap), :303-311 (edit); tie rules SURVEY.md A.0.
#pragma once
#include <type_traits>
#include "at_plan.h"      // WaveTask

namespace atb2 {

#define AT_WAVE_WARPS 4
#ifndef AT_WAVE_AFFINE_MINB
#define AT_WAVE_AFFINE_MINB 4      // resident CTAs per SM the affine kernel is compiled for (128 registers)
#endif
#ifndef AT_WAVE_AFFINE_BANDED_MINB
#define AT_WAVE_AFFINE_BANDED_MINB 3      // the banded instantiation: its band masks spill at 128 registers
#endif
#ifndef AT_WAVE_UNROLL_AFFINE_N
#define AT_WAVE_UNROLL_AFFINE_N 2
#endif
constexpr int AT_WAVE_UNROLL_AFFINE = AT_WAVE_UNROLL_AFFINE_N;     // steps per loop body (instruction-cache footprint, see the loops)
constexpr int AT_WAVE_UNROLL_OVERLAP = 4, AT_WAVE_UNROLL_EDIT = 8;
#define AT_PROG_DONE 0xffffffffu

struct WaveArgs {
	const uint8_t  *q;       const uint64_t *q_off;  const uint32_t *q_len;
	const uint8_t  *t;       const uint64_t *t_off;  const uint32_t *t_len;
	const uint8_t  *jmask;   // fit+jump: 1 where entering J is forbidden, one byte per target symbol
	const uint64_t *j_off;   // [pair] offset of the pair's mask (byte-encoded targets: the same array as t_off)
	const WaveTask *tasks;   // the queue: a pair's stripes in ascending order (the host interleaves the pairs, at_plan.h)
	uint32_t        n_tasks;
	uint32_t       *counter; // task queue head
	uint32_t       *prog;    // [n_tasks] columns of the task's last row that are visible in its slab
	uint32_t       *ptr;     const uint64_t *ptr_off;   uint32_t pair_base;
	void           *bnd;     // boundary slabs: int4 (affine) or int32 (single plane) per column
	const uint64_t *bnd_off; // [pair - pair_base] element offset of the pair's two slabs
	int32_t        *chain;   // [pair - pair_base][4] local mode: best (score, row, column) of the stripes so far
	int32_t        *score;   uint32_t *end_i;  uint32_t *end_j;  uint8_t *end_state;
	int             m, u, o, e, jp;
	int             want_ptr;
	const uint8_t  *symmap;  // at_wave_edit_bits: byte -> code 0..7 of the shard's READ alphabet, 8 = not in it;
	                         // at_wave_linear<.., PROF>: byte -> code 0..3 of the shard's TARGET alphabet
	uint32_t        syms;    // PROF: the byte of code c in bits 8c..8c+7
	uint32_t        k_and, k_or;   // affine kernel: cell_k_and / cell_k_or (at_cell.cuh: constants that must stay in registers)
	int             twobit;  // q / t hold 2-bit codes (AT_SEQ_2BIT resident: four symbols per byte, A C G T = 0..3, byte-aligned records)
	uint32_t        start_lag;   // a stripe starts once the stripe above it has published this many columns (0: as soon as it can)
	const int2     *band;        // at_wave_linear<.., BANDED>: [pair] clipped band (lo, hi) on j - i (at_band.h)
	SubstArgs       sub;         // SCORED: the substitution matrix (at_kernels.cuh)
};

// SCORED && !PROF (table variant): dynamic shared memory of a CTA -- the target byte -> column offset map, then the table
__host__ __device__ constexpr size_t wave_smem_bytes_table(uint32_t table_bytes) { return 512u + table_bytes; }
// copy the map and the table (every thread of the CTA; the caller synchronises)
__device__ __forceinline__ void wave_table_load(const SubstArgs &s, unsigned char *dyn)
{
	for (uint32_t x = threadIdx.x; x < 256u; x += blockDim.x) ((uint16_t *)dyn)[x] = __ldg(s.tcol + x);
	for (uint32_t x = threadIdx.x; x < s.table_bytes / 16u; x += blockDim.x) ((uint4 *)(dyn + 512))[x] = __ldg((const uint4 *)s.table + x);
}

// ---- TMA (bulk async copy) + mbarrier + release/acquire helpers ----
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             :: "r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
	uint32_t ok;
	do {
		asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
		             : "=r"(ok) : "r"(smem_addr(bar)), "r"(parity) : "memory");
	} while (!ok);
}
// Progress word of the predecessor stripe (affine kernel): polled with relaxed loads, then ONE ld.acquire once
// the awaited column is there -- the acquire pairs with the producer's st.release.gpu and orders the boundary
// loads behind it; polling with ld.acquire itself would invalidate L1 (CCTL.IVALL) on every iteration.
__device__ __forceinline__ uint32_t ld_progress(const uint32_t *p)
{
	uint32_t v;
	asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ uint32_t ld_acquire(const uint32_t *p)
{
	uint32_t v;
	asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
	return v;
}
// tagged hand-off words of the single-plane kernels: 64-bit accesses are single-copy atomic, so a word that
// carries its own tag needs neither a fence on the producer's side nor a flag on the consumer's
__device__ __forceinline__ void st_relaxed_u64(uint64_t *p, uint64_t v)
{
	asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t *p)
{
	uint64_t v;
	asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ void st_release(uint32_t *p, uint32_t v)
{
	asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// Per-warp target ring: two 256-byte slots per plane, slot c & 1 holds tile c of the target
// (bytes base + 256*c .. +255 where base is the pair's target address rounded DOWN to 16 bytes,
// as cp.async.bulk wants; `sh` = the rounding, so target index x lives at ring[(x + sh) & 511]).
// 2-bit resident targets: a tile is 64 packed bytes; TMA stages them in pk[] and the warp expands them into the
// byte ring once per 256 columns (ring_expand), so the column loops read the same bytes either way.  `sh` is then
// four times the rounding of the packed address.
template <bool JUMP> struct __align__(16) WaveRing {
	uint8_t  tring[512];
	uint8_t  jring[JUMP ? 512 : 16];
	uint8_t  pk[2][64];
	uint64_t bar[2];
};

template <bool JUMP>
__device__ __forceinline__ void ring_issue(WaveRing<JUMP> &rg, const uint8_t *tbase16, const uint8_t *jbase16, uint32_t c, int lane, bool twobit)
{
	if (lane == 0) {
		fence_proxy_async_smem();      // the slot's previous contents were read through the generic proxy
		uint64_t *bar = &rg.bar[c & 1];
		mbar_expect_tx(bar, (twobit ? 64u : 256u) + (JUMP ? 256u : 0u));
		if (twobit) tma_load_1d(rg.pk[c & 1], tbase16 + 64ull * c, 64u, bar);
		else tma_load_1d(rg.tring + 256u * (c & 1), tbase16 + 256ull * c, 256u, bar);
		if (JUMP) tma_load_1d(rg.jring + 256u * (c & 1), jbase16 + 256ull * c, 256u, bar);
	}
}

__device__ __forceinline__ uint32_t sym_of_code(uint32_t code) { return (0x54474341u >> (8u * code)) & 255u; }      // "ACGT"[code]

// tile c has landed in pk[c & 1]: 64 packed bytes -> 256 symbols of the byte ring (two packed bytes per lane)
template <bool JUMP>
__device__ __forceinline__ void ring_expand(WaveRing<JUMP> &rg, uint32_t c, int lane)
{
	const uint32_t two = ((const uint16_t *)rg.pk[c & 1])[lane];
	uint32_t lo = 0, hi = 0;
#pragma unroll
	for (int k = 0; k < 4; ++k) {
		lo |= sym_of_code((two >> (2 * k)) & 3u) << (8 * k);
		hi |= sym_of_code((two >> (8 + 2 * k)) & 3u) << (8 * k);
	}
	((uint2 *)(rg.tring + 256u * (c & 1)))[lane] = make_uint2(lo, hi);
	__syncwarp();
}

// symbol ri of a read: a byte, or "ACGT"[its 2-bit code]
__device__ __forceinline__ uint32_t read_sym(const uint8_t *__restrict__ q, uint32_t ri, bool twobit)
{
	return twobit ? sym_of_code(((uint32_t)q[ri >> 2] >> (2u * (ri & 3u))) & 3u) : (uint32_t)q[ri];
}

// Wait until the predecessor task has published column `need` (warp-uniform; `seen` caches the last value read).
__device__ __forceinline__ void wait_columns(const uint32_t *prog, uint32_t need, uint32_t &seen, int lane)
{
	if (seen >= need) return;
	uint32_t v = 0;
	if (lane == 0) {
		v = ld_progress(prog);
		while (v < need) { __nanosleep(100); v = ld_progress(prog); }
		v = ld_acquire(prog);                  // progress only grows: still >= need
	}
	seen = __shfl_sync(0xffffffffu, v, 0);
	__syncwarp();                              // orders the other lanes' loads after lane 0's acquire
}

// =====================================================================================
// Affine kernel: global / local / fit (+jump), int32 lanes, R = 8 rows per lane.
// =====================================================================================
// The cell is cell_update() of at_cell.cuh (tagged values, pointer nibbles assembled on the FMA pipe), as in K1.
// PROF (targets of the shard use at most four distinct bytes): query profile in shared memory as in K1,
// prof[code][lane][r] = 8 * s(read row, target symbol); otherwise the xor / min form.
// Lane 0's upper neighbour is matrix row 0 (first stripe) or the boundary row of the stripe above (a predicated
// LDS from the boundary ring); it enters through a multiply-add with a 0/1 lane mask, not a branch.
// Boundary element (int4 per column): x = M + o (tag 3), y = L (tag 3), z = H (tagged), w unused.
//
// BANDED (global only): the pair's band (at_band.h, 8-step pointer groups: wsh = PTR_SH_NIB) limits every stripe to its column
// window.  The band holds the end diagonal l2 - l1 (the host checks it), so the stripes without a window are a run at the
// top of the pair and the host queues none of them.  The steps run from the window's t0 to (c1 + 31) | 31; 8-step blocks
// whose cells may leave the band force M, L and U of those cells to -inf, blocks wholly inside the band run the plain body.
// With t0 > 0 every cell left of the window is out of band: the lanes' left state and lane 0's diagonal start at -inf.
// The first stripe with a window below empty ones has no predecessor: its row above is -inf at every column j >= 1 and
// keeps the column-0 border H(row0, 0).  A stripe publishes the window columns of its last row; the stripe below waits
// only for columns inside the producer's window and takes -inf for the others (the slab entries outside the window hold
// values of the stripe two above).  Target tiles keep their absolute numbering, only those the window reads are staged.
// Pointer words are stored relative to t0 at the stripe's offset in the pair's block (band_stripe_off).
//
// SCORED (substitution matrix, unbanded): PROF builds the profile from the matrix row of the read symbol; otherwise the
// TABLE variant: ac[r] = byte offset of the row's read code in the compact table (dynamic shared memory), the column's
// target code comes from the shared map of its ring byte, and 8 s(i, j) is one LDS.S16 per cell.
template <int MODE, bool JUMP, bool PROF, bool BANDED = false, bool SCORED = false>
__global__ void __launch_bounds__(32 * AT_WAVE_WARPS, BANDED ? AT_WAVE_AFFINE_BANDED_MINB : AT_WAVE_AFFINE_MINB) at_wave_affine(const WaveArgs a)
{
	static_assert(!BANDED || (MODE == MODE_GLOBAL && !JUMP), "banded affine kernel: global alignment only");
	static_assert(!BANDED || !SCORED, "no band with a substitution matrix");
	constexpr bool TABLE = SCORED && !PROF;
	extern __shared__ __align__(16) unsigned char wave_dyn[];          // TABLE: wave_smem_bytes_table
	const uint16_t *tmap_s = (const uint16_t *)wave_dyn;
	const unsigned char *tab = wave_dyn + 512;
	typedef Lanes<false> V;
	constexpr int R = 8, RPP = 32 * R;
	constexpr bool LOCAL = MODE == MODE_LOCAL;
	constexpr int LS = prof_lane_stride(R);
	struct __align__(16) Smem { int prof[PROF ? 4 : 1][PROF ? 32 : 1][PROF ? LS : 2]; WaveRing<JUMP> rg; int4 cring[64]; int4 stage[64]; };
	__shared__ Smem sm_all[AT_WAVE_WARPS];
	__shared__ uint8_t symmap_s[PROF ? 256 : 16];
	Smem &sm = sm_all[threadIdx.x >> 5];
	const int lane = threadIdx.x & 31;
	if (PROF) { for (int x = threadIdx.x; x < 256; x += blockDim.x) symmap_s[x] = a.symmap[x]; }
	if (TABLE) wave_table_load(a.sub, wave_dyn);
	if (lane == 0) { mbar_init(&sm.rg.bar[0], 1); mbar_init(&sm.rg.bar[1], 1); fence_proxy_async_smem(); }
	__syncthreads();
	uint32_t ring_par = 0;      // bit s: parity of the next completion of slot s's mbarrier

	const int m = a.m, u = a.u, o = a.o, e = a.e;
	CellConst<false> cc;
	cc.set(o, e, a.jp, a.k_and, a.k_or);
	const int m8 = 8 * m, o8 = 8 * o, e8 = 8 * e;
	const uint32_t mu8 = (uint32_t)(8 * (m >= u ? m - u : u - m));
	const int nsg = m >= u ? -1 : 1;
	const int ZERO = 0, NEGV = AT_NEG;
	const bool want_ptr = a.want_ptr != 0;
	int nz = lane ? 1 : 0;                                                     // lane 0 takes the row above the stripe instead of a neighbour
	asm volatile("" : "+r"(nz));                                               // opaque: keep x * nz + b a multiply-add (FMA pipe), not a SEL

	for (;;) {
		uint32_t job = 0;
		if (lane == 0) job = atomicAdd(a.counter, 1u);
		job = __shfl_sync(0xffffffffu, job, 0);
		if (job >= a.n_tasks) break;
		const WaveTask tk = a.tasks[job];
		const uint32_t p = tk.pair, stripe = tk.stripe;
		const uint32_t l1 = a.q_len[p], l2 = a.t_len[p];
		const uint8_t *__restrict__ q = a.q + a.q_off[p];
		const bool twobit = a.twobit != 0;
		const uint8_t *tbase = a.t + a.t_off[p];
		const uint32_t sh16 = (uint32_t)((uintptr_t)tbase & 15u);
		const uint8_t *tbase16 = tbase - sh16;
		const uint32_t sh = twobit ? 4u * sh16 : sh16;                        // ring position of target index 0
		const uint32_t tile_wait = twobit ? 192u : 224u;                      // step (mod 256) at which the next tile must have landed: lane 0 is up to sh + 1 columns ahead of the step counter
		const uint8_t *jbase16 = JUMP ? a.jmask + a.j_off[p] - sh : nullptr;     // the host lays the masks out with the targets' ring alignment
		uint32_t n_tiles = (l2 + sh + 255u) >> 8;
		uint32_t *__restrict__ ptr = a.ptr + a.ptr_off[p - a.pair_base];
		const uint32_t t_ptr_last = ptr_last_step(l2, PTR_SH_NIB, JUMP);
		const uint32_t G = ptr_groups(t_ptr_last, PTR_SH_NIB), GJ = ptr_groups(t_ptr_last, PTR_SH_JUMP);
		uint32_t t_last = (l2 + 31u) | 31u;
		const uint32_t n_stripes = (l1 + RPP - 1) / RPP;
		uint32_t *__restrict__ ptrJ = ptr_plane(ptr, n_stripes, G, R);
		const bool last_stripe = stripe + 1 == n_stripes;
		// banded: this stripe's window (bw), the one above (bwp), whether the stripe above takes part
		BandWin bw = {1u, l2, 0u, G}, bwp = bw;
		int32_t elo = 0, ehi = 0;
		bool has_prev = stripe > 0;
		if constexpr (BANDED) {
			const int2 bd = a.band[p];
			elo = bd.x; ehi = bd.y;
			band_stripe(l1, l2, elo, ehi, RPP, stripe, bw, PTR_SH_NIB);     // queued stripes have a window
			has_prev = stripe > 0 && band_stripe(l1, l2, elo, ehi, RPP, stripe - 1u, bwp, PTR_SH_NIB);
			t_last = band_t_last(bw);
			n_tiles = min(n_tiles, ((bw.c1 - 1u + sh) >> 8) + 1u);         // tiles the window reads
			if (want_ptr) ptr += band_stripe_off(l1, l2, elo, ehi, RPP, stripe, PTR_SH_NIB);
		}
		const uint32_t tile0 = bw.t0 >> 8;                                 // first tile the stripe reads (0 unbanded)
		const uint32_t slab = (l2 + 4u) & ~3u;
		int4 *bnd_pair = (int4 *)a.bnd + a.bnd_off[p - a.pair_base];
		int4 *bnd_out = bnd_pair + (size_t)(stripe & 1u) * slab;
		const int4 *bnd_in = bnd_pair + (size_t)((stripe & 1u) ^ 1u) * slab;
		const uint32_t *prog_in = a.prog + tk.prev;
		uint32_t seen = 0;
		const uint32_t row0 = stripe * RPP + lane * R;
		const bool feed = lane == 0 && has_prev;                           // this lane reads the boundary ring
		const bool park = lane == 31 && !last_stripe;                      // this lane parks its last row for the next stripe
		const bool left_neg = BANDED && bw.t0 > 0;                         // banded: the cells left of the window are -inf

		__syncwarp();
		if (n_tiles > tile0) ring_issue<JUMP>(sm.rg, tbase16, jbase16, tile0, lane, twobit);
		if (n_tiles > tile0 + 1u) ring_issue<JUMP>(sm.rg, tbase16, jbase16, tile0 + 1u, lane, twobit);

		RowState<false, JUMP> st[R];
		int crow[R];
		uint32_t ac[R];
#pragma unroll
		for (int r = 0; r < R; ++r) {
			const uint32_t ri = row0 + r;
			const int i = (int)ri + 1;
			if (TABLE) ac[r] = ri < l1 ? __ldg(a.sub.qrow + read_sym(q, ri, twobit)) : 0u;      // padded rows: any row of the table
			else ac[r] = ri < l1 ? (read_sym(q, ri, twobit) << 16) : 0x4u;
			if (PROF) {
				const uint32_t qa = ri < l1 ? read_sym(q, ri, twobit) : 0x100u;
#pragma unroll
				for (int c = 0; c < 4; ++c) {
					const uint32_t sy = (a.syms >> (8 * c)) & 255u;
					if (SCORED) sm.prof[c][lane][r] = qa < 0x100u ? 8 * (int)__ldg(a.sub.matrix + qa * 256u + sy) : 0;
					else sm.prof[c][lane][r] = 8 * (qa == sy ? m : u);
				}
			}
			crow[r] = ri < l1 ? 5 - r : -(1 << 28);                       // on top of Mk = 8 M + 2: key = 8 M + 7 - r
			// column 0 (left border), tags as cell_update leaves them
			if (left_neg)                { st[r].mo = NEGV | 3; st[r].u = NEGV | 1; st[r].h = NEGV | TAG_M; }
			else if (MODE == MODE_GLOBAL) { st[r].mo = NEGV | 3; st[r].u = NEGV | 1; st[r].h = 8 * (o + e * i) | TAG_L; }     // :432-436
			else if (MODE == MODE_LOCAL) { st[r].mo = ZERO + o8 + 3; st[r].u = ZERO | 1; st[r].h = ZERO | TAG_L; }            // calloc zeros
			else                         { st[r].mo = NEGV | 3; st[r].u = NEGV | 1; st[r].h = NEGV | TAG_M; }                 // :612-617
			st[r].j = NEGV; st[r].x = 0; st[r].xj = 0;
		}
		if (PROF) __syncwarp();
		int sM = st[R - 1].mo, sH = st[R - 1].h;
		int sL = MODE == MODE_GLOBAL ? (8 * (o + e * (int)(row0 + R)) | 3) : (MODE == MODE_LOCAL ? (ZERO | 3) : (NEGV | 3));
		if (left_neg) sL = NEGV | 3;
		int pH;      // H(row0, 0): the row above this lane's strip, column 0 (banded, t0 > 0: H(row0, t0 - 1) = -inf)
		if (left_neg) pH = NEGV | TAG_M;
		else if (row0 == 0) {
			if (MODE == MODE_GLOBAL)     pH = 8 * (o < 0 ? 0 : o) | (o < 0 ? TAG_M : TAG_L);                                 // max5(L=o, M=0, U=o)
			else if (MODE == MODE_LOCAL) pH = ZERO | TAG_L;
			else                         pH = ZERO | TAG_M;                                                                  // M[0][0]=U[0][0]=0
		} else {
			if (MODE == MODE_GLOBAL)     pH = 8 * (o + e * (int)row0) | TAG_L;
			else if (MODE == MODE_LOCAL) pH = ZERO | TAG_L;
			else                         pH = NEGV | TAG_M;
		}
		// what lane 0 adds instead of a neighbour's row (zero in every other lane): matrix row 0 in the first stripe,
		// the boundary ring's element of the column otherwise (loaded per step by lane 0 alone)
		// (banded, first stripe with a window below empty ones: the row above is out of band, -inf)
		int4 bq = make_int4(0, 0, 0, 0);
		int b0E = 0;
		const int4 neg4 = make_int4(NEGV | 3, NEGV | 3, NEGV | TAG_M, 0);      // banded: a boundary column outside the producer's window
		if (lane == 0 && stripe == 0) {
			if (MODE == MODE_GLOBAL)     { bq.x = NEGV | 3; bq.y = NEGV | 3; bq.z = 8 * o | TAG_U; b0E = e8; }                // :437-441, U[0][j] = o + e j
			else if (MODE == MODE_LOCAL) { bq.x = ZERO + o8 + 3; bq.y = ZERO | 3; bq.z = ZERO | TAG_L; }
			else                         { bq.x = ZERO + o8 + 3; bq.y = NEGV | 3; bq.z = ZERO | TAG_M; }                      // :619-624
		} else if (BANDED && lane == 0 && !has_prev) bq = neg4;
		const int cap_r = (last_stripe && lane == (int)(((l1 - 1) % RPP) / R)) ? (int)((l1 - 1) % R) : -1;
		int hot[R];
#pragma unroll
		for (int r = 0; r < R; ++r) hot[r] = r == cap_r ? 1 : 0;
		int kbest = AT_NEG_INIT, tbest = 0;                                         // local
		int capM = AT_NEG_INIT, capMj = 0, capL = AT_NEG_INIT, capLj = 0;           // fit
		int gH = 0;                                                                 // global

		// first boundary block of the stripe above
		// (banded: the columns [in0, in1] the stripe above publishes -- its window; only those are awaited and read)
		const uint32_t in0 = BANDED ? bwp.c0 : 1u, in1 = BANDED ? bwp.c1 : l2;
		int4 pre = make_int4(0, 0, 0, 0);
		if (has_prev) {
			if constexpr (BANDED) {
				wait_columns(prog_in, min(max(bw.t0 + max(31u, a.start_lag), in0), in1), seen, lane);
				const uint32_t col = bw.t0 + lane;
				pre = col >= in0 && col <= in1 ? __ldcg(bnd_in + col) : neg4;
			} else {
				wait_columns(prog_in, min(l2, max(31u, a.start_lag)), seen, lane);
				if ((uint32_t)lane <= l2) pre = __ldcg(bnd_in + lane);
			}
		}
		mbar_wait(&sm.rg.bar[tile0 & 1u], (ring_par >> (tile0 & 1u)) & 1u); ring_par ^= 1u << (tile0 & 1u);
		if (twobit) ring_expand(sm.rg, tile0, lane);
		if (BANDED && (bw.t0 & 255u) > tile_wait && tile0 + 1u < n_tiles) {      // the window starts past the point where the next tile is awaited
			const uint32_t c = tile0 + 1u;
			mbar_wait(&sm.rg.bar[c & 1u], (ring_par >> (c & 1u)) & 1u); ring_par ^= 1u << (c & 1u); if (twobit) ring_expand(sm.rg, c, lane);
		}

		// `cap`: std::true_type in the pair's last stripe -- only there can a lane hold the row whose cells the
		// end-cell search looks at; the other stripes run a body without it
		// `msk`: std::true_type where cells of the step may lie outside the pair's band (BANDED only): they become -inf
		auto step = [&](const uint32_t t, const bool checked, auto cap, auto msk) {
			constexpr bool CAP = decltype(cap)::value;
			constexpr bool MSK = decltype(msk)::value;
			const int j = (int)t - lane;
			if (feed) bq = sm.cring[t & 63u];
			const int rM = __shfl_up_sync(0xffffffffu, sM, 1) * nz + bq.x;
			const int rL = __shfl_up_sync(0xffffffffu, sL, 1) * nz + bq.y;
			int rH = __shfl_up_sync(0xffffffffu, sH, 1) * nz + bq.z;
			if (MODE == MODE_GLOBAL) rH += b0E * (int)t;
			if (checked && t == 0) rH = pH;                   // step 0 only primes the pipeline: keep H(row0, 0)
			int D = pH;
			pH = rH;
			if (!checked || (j >= 1 && j <= (int)l2)) {
				const uint32_t y = (uint32_t)(j - 1) + sh;
				const uint32_t c = PROF ? (uint32_t)symmap_s[sm.rg.tring[y & 511u]] : TABLE ? (uint32_t)tmap_s[sm.rg.tring[y & 511u]] : (uint32_t)sm.rg.tring[y & 511u] << 16;
				int pw[LS];                                                       // PROF: 8 * s of this lane's rows against the column's symbol
				if (PROF) {
					const int2 *pp = (const int2 *)&sm.prof[c][lane][0];
#pragma unroll
					for (int r2 = 0; r2 < R / 2; ++r2) { const int2 v2 = pp[r2]; pw[2 * r2] = v2.x; pw[2 * r2 + 1] = v2.y; }
				}
				int jadd = 0;
				if (JUMP) jadd = sm.rg.jring[y & 511u] ? cc.j_barred : cc.j_enter;       // M[i][j-1] + jump, or barred (:659-665)
				int lup = rL, mo_up = rM;
				int rowM = 0, rowL = 0;
				const int kold = kbest;
				CellOut<false> out;
#pragma unroll
				for (int r = 0; r < R; ++r) {
					int s8;                                                       // 8 s(i, j)
					if (PROF) s8 = pw[r];
					else if (TABLE) s8 = *(const int16_t *)(tab + ac[r] + c);
					else { const int tt = (int)min(ac[r] ^ c, mu8); s8 = tt * nsg + m8; }   // tt: 0 on a match, 8|m-u| otherwise
					D = cell_update<LOCAL, JUMP, false, true>(cc, st[r], D, s8, lup, mo_up, jadd, 16u, 2u, out);
					if (MSK && (uint32_t)(j - (int)row0 - 1 - r - elo) > (uint32_t)(ehi - elo)) {     // d = j - i out of band
						out.mo = out.lk = NEGV | 3; out.h = NEGV | TAG_M;
						st[r].mo = out.mo; st[r].u = NEGV | 1; st[r].h = out.h;
					}
					lup = out.lk; mo_up = out.mo;
					if (LOCAL) kbest = __viaddmax_s32(out.mk, crow[r], kbest);
					if (MODE == MODE_FIT && CAP) { rowM += out.mk * hot[r]; rowL += out.lk * hot[r]; }      // one-hot pick of the pair's last row (FMA pipe)
					if (MODE == MODE_GLOBAL && CAP) { if (r == cap_r && j == (int)l2) gH = out.h; }
				}
				sM = out.mo; sL = out.lk; sH = out.h;
				if (MODE == MODE_FIT && CAP) {
					if (cap_r >= 0 && j < (int)l2) {                              // column l2 excluded (:677, :684)
						rowM &= ~7; rowL &= ~7;                                   // drop the tags: M and L are compared with each other at the end
						if (rowM > capM) { capM = rowM; capMj = j; }
						if (rowL > capL) { capL = rowL; capLj = j; }
					}
				}
				if (LOCAL) { if (kbest != kold) tbest = (int)t; }
				if (park) sm.stage[(uint32_t)j & 63u] = make_int4(sM, sL, sH, 0);
			} else {
#pragma unroll
				for (int r = 0; r < R; ++r) { st[r].x *= 16u; if (JUMP) st[r].xj *= 2u; }
			}
		};

		// columns this stripe publishes (banded: its window)
		const int pub0 = (int)bw.c0, pub1 = (int)bw.c1;
		for (uint32_t tb = bw.t0; tb <= t_last; tb += 8) {
			if ((tb & 31u) == 0) {
				__syncwarp();
				if (!last_stripe && tb >= 64u) {      // lane 31 has finished the columns up to tb-32: flush (tb-64, tb-32]
					const int cidx = (int)tb - 63 + lane;
					if (cidx >= pub0 && cidx <= pub1) __stcg(bnd_out + cidx, sm.stage[(uint32_t)cidx & 63u]);
					__syncwarp();
					if (lane == 0) st_release(a.prog + job, min(tb - 32u, l2));
				}
				if (has_prev) {                       // block tb of the stripe above -> ring; fetch block tb+32
					sm.cring[(tb + lane) & 63u] = pre;
					const uint32_t nxt = tb + 32u + lane;
					if constexpr (BANDED) {
						if (tb + 32u <= in1 && tb + 63u >= in0) wait_columns(prog_in, min(in1, tb + 63u), seen, lane);
						pre = nxt >= in0 && nxt <= in1 ? __ldcg(bnd_in + nxt) : neg4;
					} else if (tb + 32u <= l2) {
						wait_columns(prog_in, min(l2, tb + 63u), seen, lane);
						if (nxt <= l2) pre = __ldcg(bnd_in + nxt);
					}
					__syncwarp();
				}
			}
			if ((tb & 255u) == 32u && (BANDED ? (tb >> 8) > tile0 : tb > 32u)) {     // tile tb/256 - 1 is dead: refill its slot two tiles ahead
				const uint32_t c = (tb >> 8) + 1u;
				__syncwarp();
				if (c < n_tiles) ring_issue<JUMP>(sm.rg, tbase16, jbase16, c, lane, twobit);
			}
			if ((tb & 255u) == tile_wait) {           // the first lane enters tile tb/256 + 1 within the next 32 steps (2-bit: 64, sh <= 60)
				const uint32_t c = (tb >> 8) + 1u;
				if (c < n_tiles) { mbar_wait(&sm.rg.bar[c & 1u], (ring_par >> (c & 1u)) & 1u); ring_par ^= 1u << (c & 1u); if (twobit) ring_expand(sm.rg, c, lane); }
			}
			// two steps per loop body: 8 rows x 2 steps already is ~400 instructions; a fully unrolled pointer
			// word (8 steps) overflows the instruction cache (ncu: stall_no_instruction was the top stall)
			// banded: d = j - i of the block's cells spans [tb - row(stripe) - RPP - 31, tb + 6 - row(stripe)]
			const bool inner = !BANDED || ((int64_t)tb - (int64_t)stripe * RPP - RPP - 31 >= elo && (int64_t)tb + 6 - (int64_t)stripe * RPP <= ehi);
			if (tb >= 32u && tb + 7u <= l2 && inner) {
				if (last_stripe) {
#pragma unroll AT_WAVE_UNROLL_AFFINE
					for (uint32_t k = 0; k < 8; ++k) step(tb + k, false, std::true_type(), std::false_type());
				} else {
#pragma unroll AT_WAVE_UNROLL_AFFINE
					for (uint32_t k = 0; k < 8; ++k) step(tb + k, false, std::false_type(), std::false_type());
				}
			} else if (BANDED && tb >= 32u && tb + 7u <= l2) {
				if (last_stripe) {
#pragma unroll AT_WAVE_UNROLL_AFFINE
					for (uint32_t k = 0; k < 8; ++k) step(tb + k, false, std::true_type(), std::true_type());
				} else {
#pragma unroll AT_WAVE_UNROLL_AFFINE
					for (uint32_t k = 0; k < 8; ++k) step(tb + k, false, std::false_type(), std::true_type());
				}
			} else {
#pragma unroll 1
				for (uint32_t k = 0; k < 8; ++k) step(tb + k, true, std::true_type(), std::integral_constant<bool, BANDED>());
			}
			if constexpr (BANDED) {
				if (want_ptr && ((tb - bw.t0) >> PTR_SH_NIB) < bw.groups) {
					uint32_t *w = ptr_at(ptr, 0u, 0u, (tb - bw.t0) >> PTR_SH_NIB, lane, R);
#pragma unroll
					for (int r = 0; r < R; ++r) w[r] = ptr_word(st[r].x);
				}
			} else if (want_ptr && (tb >> PTR_SH_NIB) < G) {
				uint32_t *w = ptr_at(ptr, stripe, G, tb >> PTR_SH_NIB, lane, R);
#pragma unroll
				for (int r = 0; r < R; ++r) w[r] = ptr_word(st[r].x);
			}
			if (JUMP && want_ptr && (tb & 31u) == 24u && (tb >> PTR_SH_JUMP) < GJ) {
				uint32_t *w = ptr_at(ptrJ, stripe, GJ, tb >> PTR_SH_JUMP, lane, R);
#pragma unroll
				for (int r = 0; r < R; ++r) w[r] = jump_word(st[r].xj);
			}
		}
		__syncwarp();

		if (!last_stripe) {       // rest of the boundary row: columns (t_last-63, t_last-31], and t_last-31 >= l2 (banded: >= c1)
			const int cidx = (int)t_last - 62 + lane;
			if (cidx >= pub0 && cidx <= pub1) __stcg(bnd_out + cidx, sm.stage[(uint32_t)cidx & 63u]);
			__syncwarp();
			if (lane == 0) st_release(a.prog + job, l2);
		}

		// ---- end cell (reference: :466-469 global, :673-690 fit, running max :830-833 local) ----
		if (LOCAL) {
			int sc = -1, row = 0x7fffffff, col = 0;
			if (kbest >= 0) { sc = kbest >> 3; row = (int)row0 + (7 - (kbest & 7)) + 1; col = tbest - lane; }
#pragma unroll
			for (int d = 16; d >= 1; d >>= 1) {
				const int osc = __shfl_xor_sync(0xffffffffu, sc, d);
				const int orow = __shfl_xor_sync(0xffffffffu, row, d);
				const int ocol = __shfl_xor_sync(0xffffffffu, col, d);
				if (osc > sc || (osc == sc && orow < row)) { sc = osc; row = orow; col = ocol; }
			}
			if (n_stripes > 1) {      // fold into the pair's chain: earlier stripes hold smaller rows and win ties
				int32_t *ch = a.chain + 4 * (size_t)(p - a.pair_base);
				if (stripe) {
					wait_columns(prog_in, AT_PROG_DONE, seen, lane);
					const int psc = __ldcg(ch + 0), prow = __ldcg(ch + 1), pcol = __ldcg(ch + 2);
					if (psc >= sc) { sc = psc; row = prow; col = pcol; }
				}
				if (!last_stripe) {
					if (lane == 0) { __stcg(ch + 0, sc); __stcg(ch + 1, row); __stcg(ch + 2, col); }
					__syncwarp();
					if (lane == 0) st_release(a.prog + job, AT_PROG_DONE);
				}
			}
			if (last_stripe && lane == 0) { a.score[p] = sc; a.end_i[p] = row; a.end_j[p] = col; a.end_state[p] = ST_MID; }
		} else if (last_stripe) {
			const int owner = (int)(((l1 - 1) % RPP) / R);
			if (lane == owner) {
				if (MODE == MODE_GLOBAL) { a.score[p] = gH >> 3; a.end_i[p] = l1; a.end_j[p] = l2; a.end_state[p] = (uint8_t)(3 - (gH & 3)); }
				else {
					const bool useL = capL > capM;            // L replaces M only when strictly greater (:685)
					a.score[p] = (useL ? capL : capM) >> 3; a.end_i[p] = l1; a.end_j[p] = useL ? capLj : capMj;
					a.end_state[p] = useL ? ST_LOW : ST_MID;
				}
			}
		}
		__syncwarp();
	}
}

// =====================================================================================
// Single-plane kernel: overlap (max-plus, linear gap, 2-bit pointers) and edit distance
// (min-plus, unit gaps; score only unless PTR, below), int32 lanes, R = 1..8 rows per lane.
//
// Overlap runs lin_update() of at_cell.cuh: scores x4, every cell carries A = 4*M + 4*o, the argmax of the one
// VIMNMX3 rides in the two spare bits (LEFT 2, DIAGONAL 1, RIGHT 0: the reference's order with
// first-strictly-greater ties, :944-947) and the 2-bit pointers are accumulated on the FMA pipe.
// Edit distance is min3 (:280-286) with one VIADDMNMX and one VIMNMX per cell.
// =====================================================================================
// PROF (targets of the shard use at most four distinct bytes): the substitution term comes from a per-warp
// query profile in shared memory, prof[code][lane][r] (overlap: 4 (s - o) - 1, the diagonal's tag included; edit: 0 on a
// match, the mismatch cost otherwise), as in K1 -- one 64-bit LDS per two rows; a.symmap maps target bytes to codes.
// Lane 0's upper neighbour (matrix row 0, or the stripe above through the boundary ring) enters through a
// multiply-add with a 0/1 lane mask, not a branch.
// (no minimum-blocks hint: ptxas's own choice, 72-80 registers = 6 CTAs per SM, measured best on C4 -- 24.6 ms against
// 26.3 ms when held to 64 registers for 8 CTAs and 27.8 ms with a hint of 1; profiles/ab_wave_linear_occupancy_r02.txt)
//
// BANDED (overlap only): the pair's band (at_band.h) limits every stripe to its column window.  The steps run from the
// window's t0 to (c1 + 31) | 31; 16-step blocks whose cells may leave the band force those cells to -inf (the band
// test is one unsigned compare per cell), blocks wholly inside the band run the plain body.  Target tiles keep their
// absolute numbering (tile c = ring bytes 256 c ..), only those the window reads are staged.  The stripe above is the
// predecessor when it has a window; otherwise the row above is -inf, as row 0 is.  Pointer words are stored relative to
// t0 at the stripe's offset in the pair's block.  A queued stripe without a window is the pair's last one: it only
// writes the end cell M[l1][0] = 0.
//
// PTR (edit only, AT_OUT_EDIT_PATH): the cell is edit_min3_tagged() of at_cell.cuh -- the three candidates x4 with min3's
// argmin code in the low bits (LEFT 0, DIAGONAL 1, UP 2), one VIMNMX3 -- and the codes are stored in overlap's layout
// (2 bits, 16 steps per word, code = the tag itself), so K3 walks them with overlap's reader.
//
// SCORED (overlap with a substitution matrix, unbanded): PROF builds 4 (s - o) - 1 from the matrix; otherwise the TABLE
// variant as in at_wave_affine, whose table holds 4 s (one add of -4 o - 1 per cell).
template <int MODE, int R, bool PROF, bool BANDED = false, bool PTR = false, bool SCORED = false>
__global__ void __launch_bounds__(32 * AT_WAVE_WARPS) at_wave_linear(const WaveArgs a)
{
	static_assert(!PTR || (MODE == MODE_EDIT && !BANDED), "PTR: the edit kernel's pointers (overlap stores its own)");
	static_assert(!SCORED || (MODE == MODE_OVERLAP && !BANDED), "substitution matrix: unbanded overlap only");
	constexpr bool TABLE = SCORED && !PROF;
	extern __shared__ __align__(16) unsigned char wave_dyn[];          // TABLE: wave_smem_bytes_table
	const uint16_t *tmap_s = (const uint16_t *)wave_dyn;
	const unsigned char *tab = wave_dyn + 512;
	constexpr int RPP = 32 * R;
	constexpr bool OV = MODE == MODE_OVERLAP;
	constexpr bool STORE = OV || PTR;      // the kernel writes 2-bit pointer words
	constexpr int UNR = OV ? AT_WAVE_UNROLL_OVERLAP : AT_WAVE_UNROLL_EDIT;
	constexpr int LS = prof_lane_stride(R);
	struct __align__(16) Smem { int prof[PROF ? 4 : 1][PROF ? 32 : 1][PROF ? LS : 2]; WaveRing<false> rg; int cring[64]; int stage[64]; };
	__shared__ Smem sm_all[AT_WAVE_WARPS];
	__shared__ uint8_t symmap_s[PROF ? 256 : 16];
	Smem &sm = sm_all[threadIdx.x >> 5];
	const int lane = threadIdx.x & 31;
	if (PROF) { for (int x = threadIdx.x; x < 256; x += blockDim.x) symmap_s[x] = a.symmap[x]; }
	if (TABLE) wave_table_load(a.sub, wave_dyn);
	if (lane == 0) { mbar_init(&sm.rg.bar[0], 1); mbar_init(&sm.rg.bar[1], 1); fence_proxy_async_smem(); }
	__syncthreads();
	uint32_t ring_par = 0;

	// overlap: S = 4, step cost o, substitution m / u; edit: S = 1, step cost +1, substitution 0 / u
	const int S = OV ? 4 : 1;
	const int gap = OV ? S * a.o : 1;
	const int pw_match = OV ? S * (a.m - a.o) - 1 : 0;               // substitution term of a match (overlap: carried value -> tagged diagonal candidate)
	const uint32_t pen = OV ? (uint32_t)(S * (a.m >= a.u ? a.m - a.u : a.u - a.m)) : (uint32_t)(a.u >= 0 ? a.u : -a.u);
	const int nsg = OV ? (a.m >= a.u ? -1 : 1) : (a.u >= 0 ? 1 : -1);
	const int sub_add = -S * a.o - 1;                                  // TABLE: 4 s + sub_add = 4 (s - o) - 1
	const bool want_ptr = STORE && a.want_ptr != 0;
	int nz = lane ? 1 : 0;                                            // lane 0 takes the row above the stripe instead of a neighbour
	asm volatile("" : "+r"(nz));                                      // opaque: keep x * nz + b a multiply-add (FMA pipe), not a SEL

	for (;;) {
		uint32_t job = 0;
		if (lane == 0) job = atomicAdd(a.counter, 1u);
		job = __shfl_sync(0xffffffffu, job, 0);
		if (job >= a.n_tasks) break;
		const WaveTask tk = a.tasks[job];
		const uint32_t p = tk.pair, stripe = tk.stripe;
		const uint32_t l1 = a.q_len[p], l2 = a.t_len[p];
		const uint8_t *__restrict__ q = a.q + a.q_off[p];
		const bool twobit = a.twobit != 0;
		const uint8_t *tbase = a.t + a.t_off[p];
		const uint32_t sh16 = (uint32_t)((uintptr_t)tbase & 15u);
		const uint8_t *tbase16 = tbase - sh16;
		const uint32_t sh = twobit ? 4u * sh16 : sh16;                        // ring position of target index 0
		const uint32_t tile_wait = twobit ? 192u : 224u;                      // step (mod 256) at which the next tile must have landed: lane 0 is up to sh + 1 columns ahead of the step counter
		uint32_t n_tiles = (l2 + sh + 255u) >> 8;
		uint32_t *__restrict__ ptr = STORE ? a.ptr + a.ptr_off[p - a.pair_base] : nullptr;
		const uint32_t G = ptr_groups(ptr_last_step(l2, PTR_SH_2BIT), PTR_SH_2BIT);
		uint32_t t_last = (l2 + 31u) | 31u;
		const uint32_t n_stripes = (l1 + RPP - 1) / RPP;
		const bool last_stripe = stripe + 1 == n_stripes;
		// banded: this stripe's window (bw), the one above (pw), whether the stripes above / below take part
		BandWin bw = {1u, l2, 0u, G}, bwp = bw, bwn = bw;
		int32_t elo = 0, ehi = 0;
		bool has_prev = stripe > 0, has_next = !last_stripe;
		if constexpr (BANDED) {
			const int2 bd = a.band[p];
			elo = bd.x; ehi = bd.y;
			if (!band_stripe(l1, l2, elo, ehi, RPP, stripe, bw, PTR_SH_2BIT)) {
				if (lane == 0) { a.score[p] = 0; a.end_i[p] = l1; a.end_j[p] = 0; a.end_state[p] = ST_MID; }      // M[l1][0] (:938)
				__syncwarp();
				continue;
			}
			has_prev = stripe > 0 && band_stripe(l1, l2, elo, ehi, RPP, stripe - 1u, bwp, PTR_SH_2BIT);
			has_next = !last_stripe && band_stripe(l1, l2, elo, ehi, RPP, stripe + 1u, bwn, PTR_SH_2BIT);
			t_last = band_t_last(bw);
			n_tiles = min(n_tiles, ((bw.c1 - 1u + sh) >> 8) + 1u);         // tiles the window reads
			if (want_ptr) ptr += band_stripe_off(l1, l2, elo, ehi, RPP, stripe, PTR_SH_2BIT);
		}
		const uint32_t tile0 = bw.t0 >> 8;                                 // first tile the stripe reads (0 unbanded)
		const uint32_t slab = (l2 + 4u) & ~3u;
		// boundary hand-off without fences: one 64-bit word per column = (stripe + 1) << 32 | value; the consumer
		// validates the tag of every word it loads (the slabs are zeroed by the host before each run)
		uint64_t *bnd_pair = (uint64_t *)a.bnd + a.bnd_off[p - a.pair_base];
		uint64_t *bnd_out = bnd_pair + (size_t)(stripe & 1u) * slab;
		const uint64_t *bnd_in = bnd_pair + (size_t)((stripe & 1u) ^ 1u) * slab;
		const uint64_t tag_out = (uint64_t)(stripe + 1u) << 32;
		const uint32_t tag_in = stripe;                                   // the predecessor's (stripe - 1) + 1
		const uint32_t row0 = stripe * RPP + lane * R;
		const bool feed = lane == 0 && has_prev;                          // this lane reads the boundary ring
		const bool park = lane == 31 && has_next;                         // this lane parks its last row for the next stripe

		__syncwarp();
		if (n_tiles > tile0) ring_issue<false>(sm.rg, tbase16, nullptr, tile0, lane, twobit);
		if (n_tiles > tile0 + 1u) ring_issue<false>(sm.rg, tbase16, nullptr, tile0 + 1u, lane, twobit);

		// carried value: overlap a = 4*M + 4*o (LinRow keeps a + 2), edit M.  Column 0: M[i][0] = 0 (:938) | i (:301)
		uint32_t ac[R];
		LinRow stl[R];
		int Vl[R];
#pragma unroll
		for (int r = 0; r < R; ++r) {
			const uint32_t ri = row0 + r;
			if (TABLE) ac[r] = ri < l1 ? __ldg(a.sub.qrow + read_sym(q, ri, twobit)) : 0u;      // padded rows: any row of the table
			else ac[r] = ri < l1 ? (read_sym(q, ri, twobit) << 16) : 0x4u;
			Vl[r] = (int)ri + 1;
			stl[r].a2 = gap + 2; stl[r].x = 0;
			if (PROF) {
				const uint32_t qa = ri < l1 ? read_sym(q, ri, twobit) : 0x100u;
#pragma unroll
				for (int c = 0; c < 4; ++c) {
					const uint32_t sy = (a.syms >> (8 * c)) & 255u;
					if (SCORED) sm.prof[c][lane][r] = qa < 0x100u ? S * ((int)__ldg(a.sub.matrix + qa * 256u + sy) - a.o) - 1 : 0;
					else sm.prof[c][lane][r] = pw_match + (qa == sy ? 0 : (int)pen * nsg);
				}
			}
		}
		if (PROF) __syncwarp();
		int sV = OV ? gap : Vl[R - 1];
		int pD = 0;                                               // diagonal input of the lane's first row (set at the step with j = 0)
		const int col0 = OV ? gap : (int)row0;                    // value of the row above this lane's strip at column 0
		const int dadd = OV ? 2 : 0;                              // overlap: the diagonal input is a + 2
		const int cap_r = (last_stripe && lane == (int)(((l1 - 1) % RPP) / R)) ? (int)((l1 - 1) % R) : -1;
		int hot[R];
#pragma unroll
		for (int r = 0; r < R; ++r) hot[r] = r == cap_r ? 1 : 0;
		int capV = OV ? gap : 0, capJ = 0;                        // overlap: M[l1][0] = 0 seeds the search (:954-959)
		// what lane 0 adds instead of a neighbour's row (zero in every other lane): matrix row 0 in the first stripe
		// (overlap: -inf, :937; edit: j, :302), the boundary ring's element otherwise (loaded per step by lane 0 alone)
		int bq = 0, b0E = 0;
		if (lane == 0 && !has_prev) { if (OV) bq = AT_NEGL; else b0E = 1; }

		uint64_t pre = 0;
		if (has_prev) {
			// start lag: three hand-off blocks behind the predecessor, so that blocks requested one block ahead are valid on arrival
			if (lane == 0) {
				const uint32_t c = BANDED ? band_first_wait(bwp, bw.t0, a.start_lag) : min(l2, max(96u, a.start_lag));
				while ((uint32_t)(ld_relaxed_u64(bnd_in + c) >> 32) != tag_in) __nanosleep(200);
			}
			__syncwarp();
			if (bw.t0 + (uint32_t)lane <= l2) pre = ld_relaxed_u64(bnd_in + bw.t0 + lane);
		}
		mbar_wait(&sm.rg.bar[tile0 & 1u], (ring_par >> (tile0 & 1u)) & 1u); ring_par ^= 1u << (tile0 & 1u);
		if (twobit) ring_expand(sm.rg, tile0, lane);
		if (BANDED && (bw.t0 & 255u) > tile_wait && tile0 + 1u < n_tiles) {      // the window starts past the point where the next tile is awaited
			const uint32_t c = tile0 + 1u;
			mbar_wait(&sm.rg.bar[c & 1u], (ring_par >> (c & 1u)) & 1u); ring_par ^= 1u << (c & 1u); if (twobit) ring_expand(sm.rg, c, lane);
		}

		// `cap`: std::true_type in the pair's last stripe (only there can a lane hold the pair's last row)
		// `msk`: std::true_type where cells of the step may lie outside the pair's band (BANDED only): they become -inf
		auto step = [&](const uint32_t t, const bool checked, auto cap, auto msk) {
			constexpr bool CAP = decltype(cap)::value;
			constexpr bool MSK = decltype(msk)::value;
			const int j = (int)t - lane;
			if (feed) bq = sm.cring[t & 63u];
			int rV = __shfl_up_sync(0xffffffffu, sV, 1) * nz + bq;
			if (!OV) rV += b0E * (int)t;
			if (checked && t == 0) rV = col0;
			int D = pD;
			pD = rV + dadd;
			if (!checked || (j >= 1 && j <= (int)l2)) {
				const uint32_t y = (uint32_t)(j - 1) + sh;
				const uint32_t c = PROF ? (uint32_t)symmap_s[sm.rg.tring[y & 511u]] : TABLE ? (uint32_t)tmap_s[sm.rg.tring[y & 511u]] : (uint32_t)sm.rg.tring[y & 511u] << 16;
				int pw[LS];                                                       // PROF: substitution terms of this lane's rows
				if (PROF) {
					const int2 *pp = (const int2 *)&sm.prof[c][lane][0];
#pragma unroll
					for (int r2 = 0; r2 < (R + 1) / 2; ++r2) { const int2 v2 = pp[r2]; pw[2 * r2] = v2.x; pw[2 * r2 + 1] = v2.y; }
				}
				int Vup = rV, v = 0, rowV = 0;
#pragma unroll
				for (int r = 0; r < R; ++r) {
					int sub;                                                      // substitution term
					if (PROF) sub = pw[r];
					else if (TABLE) sub = (int)*(const int16_t *)(tab + ac[r] + c) + sub_add;
					else { const int tt = (int)min(ac[r] ^ c, pen); sub = tt * nsg + pw_match; }   // tt: 0 on a match
					if (OV) {
						int dn;
						v = lin_update(stl[r], D, sub, Vup, gap, dn);
						D = dn;
						if (MSK && (uint32_t)(j - (int)row0 - 1 - r - elo) > (uint32_t)(ehi - elo)) { v = AT_NEGL; stl[r].a2 = AT_NEGL + 2; }   // d = j - i out of band
					} else if (PTR) {
						const int vt = edit_min3_tagged(Vl[r], D + sub, Vup);     // min3 (:280-286) + its argmin code
						D = Vl[r];
						v = vt >> 2;
						stl[r].x = stl[r].x * 4u + (uint32_t)(vt & 3);
						Vl[r] = v;
					} else {
						const int diag = D + sub;
						D = Vl[r];
						v = __viaddmin_s32(min(Vl[r], Vup), 1, diag);             // min3 (:280-286)
						Vl[r] = v;
					}
					Vup = v;
					if (CAP) rowV += v * hot[r];                                  // one-hot pick of the pair's last row (FMA pipe)
				}
				sV = v;
				if (park) sm.stage[(uint32_t)j & 63u] = sV;
				if (CAP && cap_r >= 0) {                                          // the pair's last row lives in this lane
					if (OV) { if (j < (int)l2 && rowV > capV) { capV = rowV; capJ = j; } }   // column l2 excluded (:955)
					else if (j == (int)l2) capV = rowV;
				}
			} else if (STORE) {
#pragma unroll
				for (int r = 0; r < R; ++r) stl[r].x *= 4u;
			}
		};

		// columns this stripe publishes, and those it takes from the stripe above (banded: their windows; the rest is -inf)
		const int pub0 = BANDED ? (int)bw.c0 : 1, pub1 = BANDED ? (int)bw.c1 : (int)l2;
		const uint32_t in0 = BANDED ? bwp.c0 : 1u, in1 = BANDED ? bwp.c1 : l2;
		for (uint32_t tb = bw.t0; tb <= t_last; tb += 16) {
			if ((tb & 31u) == 0) {
				__syncwarp();
				if (has_next && tb >= 64u) {
					const int cidx = (int)tb - 63 + lane;
					if (cidx >= pub0 && cidx <= pub1) st_relaxed_u64(bnd_out + cidx, tag_out | (uint32_t)sm.stage[(uint32_t)cidx & 63u]);
				}
				if (has_prev) {
					const uint32_t col = tb + lane;                       // `pre` was requested a block ago: make sure it is the predecessor's
					if (col >= in0 && col <= in1)
						while ((uint32_t)(pre >> 32) != tag_in) { __nanosleep(40); pre = ld_relaxed_u64(bnd_in + col); }
					sm.cring[col & 63u] = BANDED && (col < in0 || col > in1) ? AT_NEGL : (int)(uint32_t)pre;
					const uint32_t nxt = col + 32u;
					if (nxt <= l2) pre = ld_relaxed_u64(bnd_in + nxt);
					__syncwarp();
				}
			}
			if ((tb & 255u) == 32u && (BANDED ? (tb >> 8) > tile0 : tb > 32u)) {
				const uint32_t c = (tb >> 8) + 1u;
				__syncwarp();
				if (c < n_tiles) ring_issue<false>(sm.rg, tbase16, nullptr, c, lane, twobit);
			}
			if ((tb & 255u) == tile_wait) {
				const uint32_t c = (tb >> 8) + 1u;
				if (c < n_tiles) { mbar_wait(&sm.rg.bar[c & 1u], (ring_par >> (c & 1u)) & 1u); ring_par ^= 1u << (c & 1u); if (twobit) ring_expand(sm.rg, c, lane); }
			}
			// banded: d = j - i of the block's cells spans [tb - row(stripe) - RPP - 31, tb + 14 - row(stripe)]
			const bool inner = !BANDED || ((int64_t)tb - (int64_t)stripe * RPP - RPP - 31 >= elo && (int64_t)tb + 14 - (int64_t)stripe * RPP <= ehi);
			if (tb >= 32u && tb + 15u <= l2 && inner) {
				if (last_stripe) {
#pragma unroll UNR
					for (uint32_t k = 0; k < 16; ++k) step(tb + k, false, std::true_type(), std::false_type());
				} else {
#pragma unroll UNR
					for (uint32_t k = 0; k < 16; ++k) step(tb + k, false, std::false_type(), std::false_type());
				}
			} else if (BANDED && tb >= 32u && tb + 15u <= l2) {
				if (last_stripe) {
#pragma unroll UNR
					for (uint32_t k = 0; k < 16; ++k) step(tb + k, false, std::true_type(), std::true_type());
				} else {
#pragma unroll UNR
					for (uint32_t k = 0; k < 16; ++k) step(tb + k, false, std::false_type(), std::true_type());
				}
			} else {
#pragma unroll 1
				for (uint32_t k = 0; k < 16; ++k) step(tb + k, true, std::true_type(), std::integral_constant<bool, BANDED>());
			}
			if constexpr (BANDED) {
				if (want_ptr && ((tb - bw.t0) >> PTR_SH_2BIT) < bw.groups) {
					uint32_t *w = ptr_at(ptr, 0u, 0u, (tb - bw.t0) >> PTR_SH_2BIT, lane, R);
#pragma unroll
					for (int r = 0; r < R; ++r) w[r] = lin_word(stl[r].x);
				}
			} else if (want_ptr && (tb >> PTR_SH_2BIT) < G) {
				uint32_t *w = ptr_at(ptr, stripe, G, tb >> PTR_SH_2BIT, lane, R);
#pragma unroll
				for (int r = 0; r < R; ++r) w[r] = PTR ? stl[r].x : lin_word(stl[r].x);      // edit: the code is the tag
			}
		}
		__syncwarp();

		if (has_next) {
			const int cidx = (int)t_last - 62 + lane;
			if (cidx >= pub0 && cidx <= pub1) st_relaxed_u64(bnd_out + cidx, tag_out | (uint32_t)sm.stage[(uint32_t)cidx & 63u]);
		} else if (cap_r >= 0) {
			if (OV) { a.score[p] = (capV - gap) / S; a.end_i[p] = l1; a.end_j[p] = capJ; a.end_state[p] = ST_MID; }
			else { a.score[p] = capV; a.end_i[p] = l1; a.end_j[p] = l2; a.end_state[p] = ST_MID; }
		}
		__syncwarp();
	}
}

// =====================================================================================
// Bit-parallel edit distance (Myers 1999 / Hyyro 2003 block formulation) for `edit -u 1`, the
// unit-cost case of src/alignment.h:291-315:  M[i][j] = min(M[i][j-1]+1, M[i-1][j-1]+(eq?0:1),
// M[i-1][j]+1),  M[i][0] = i,  M[0][j] = j.  Column j of a 32-row block is held as two bit vectors
// of vertical differences (Pv: +1, Mv: -1); one column step of a block is ~14 logic/add
// instructions for 32 cells and passes a horizontal difference in {-1,0,+1} to the block below.
// Same stripe pipeline as the other K2 kernels: lane k owns R consecutive blocks (32*R rows), a
// stripe is 1024*R rows, the last block's horizontal difference travels to lane k+1 by shuffle.
// The match vectors Eq[symbol] of a lane's blocks live in a per-warp shared-memory table, rebuilt
// per task; target tiles come in by TMA as in the other kernels.  Needs a read alphabet of at
// most 8 distinct bytes (DNA); anything else runs through at_wave_linear<MODE_EDIT>.
//
// Stripe hand-off WITHOUT fences: the boundary row is 2 bits per column, so 16 columns and a tag
// travel in ONE 64-bit word (single-copy atomic): word g of the slab = (stripe + 1) << 32 | the
// differences of columns 16g+1 .. 16g+16.  The producer's lane 31 stores it with one st.relaxed;
// the consumer's lane 0 polls the word itself until the tag is its predecessor's.  The slabs are
// zeroed by the host before every run.  (The release/acquire protocol of the other kernels cost a
// membar per 32 columns -- 22 % of this kernel's stall samples when it was first written that way.)
//   score = M[l1][l2] = l1 + sum over j of the horizontal difference at row l1.     SURVEY.md 8(f) #4.
//
// PTR (AT_OUT_EDIT_PATH): every block column also stores min3's argmin for its 32 cells in the bit-parallel edit layout of
// at_ptr_layout.h.  K3's bit-parallel walker reads it.
// =====================================================================================
template <int R, bool PTR = false>
__global__ void __launch_bounds__(32 * AT_WAVE_WARPS) at_wave_edit_bits(const WaveArgs a)
{
	constexpr int RPP = edit_bits_rows(R);        // rows per stripe
	constexpr int NSYM = 9;                       // 8 symbols + "matches nothing"
	struct __align__(16) Smem { uint32_t eq[NSYM][32][R]; WaveRing<false> rg; };
	__shared__ Smem sm_all[AT_WAVE_WARPS];
	__shared__ uint8_t symmap_s[256];
	Smem &sm = sm_all[threadIdx.x >> 5];
	const int lane = threadIdx.x & 31;
	for (int k = threadIdx.x; k < 256; k += blockDim.x) symmap_s[k] = a.symmap[k];
	if (lane == 0) { mbar_init(&sm.rg.bar[0], 1); mbar_init(&sm.rg.bar[1], 1); fence_proxy_async_smem(); }
	__syncthreads();
	uint32_t ring_par = 0;

	for (;;) {
		uint32_t job = 0;
		if (lane == 0) job = atomicAdd(a.counter, 1u);
		job = __shfl_sync(0xffffffffu, job, 0);
		if (job >= a.n_tasks) break;
		const WaveTask tk = a.tasks[job];
		const uint32_t p = tk.pair, stripe = tk.stripe;
		const uint32_t l1 = a.q_len[p], l2 = a.t_len[p];
		const uint8_t *__restrict__ q = a.q + a.q_off[p];
		const bool twobit = a.twobit != 0;
		const uint8_t *tbase = a.t + a.t_off[p];
		const uint32_t sh16 = (uint32_t)((uintptr_t)tbase & 15u);
		const uint8_t *tbase16 = tbase - sh16;
		const uint32_t sh = twobit ? 4u * sh16 : sh16;                        // ring position of target index 0
		const uint32_t tile_wait = twobit ? 192u : 224u;                      // step (mod 256) at which the next tile must have landed: lane 0 is up to sh + 1 columns ahead of the step counter
		const uint32_t n_tiles = (l2 + sh + 255u) >> 8;
		const uint32_t n_stripes = (l1 + RPP - 1) / RPP;
		const bool last_stripe = stripe + 1 == n_stripes;
		const uint32_t n_groups = (l2 + 15u) / 16u;                        // words per slab (the host reserves far more)
		uint64_t *bnd_pair = (uint64_t *)a.bnd + a.bnd_off[p - a.pair_base];
		uint64_t *bnd_out = bnd_pair + (size_t)(stripe & 1u) * n_groups;
		const uint64_t *bnd_in = bnd_pair + (size_t)((stripe & 1u) ^ 1u) * n_groups;
		const uint64_t tag_in = (uint64_t)stripe << 32;                    // the predecessor's tag: (stripe - 1) + 1
		const uint64_t tag_out = (uint64_t)(stripe + 1u) << 32;
		const uint32_t row0 = stripe * RPP + lane * 32u * R;
		// PTR: this lane's words of the stripe, edit_bits_slot(stripe, G, 0, R, 0, lane); store_ptr adds (t, r)'s offset.
		// Spelled out here: through the helper, nvcc orders this kernel's address arithmetic differently.
		uint2 *__restrict__ pp = nullptr;
		if constexpr (PTR) pp = (uint2 *)(a.ptr + a.ptr_off[p - a.pair_base]) + (size_t)stripe * edit_bits_groups(l2) * R * 512 + lane;

		__syncwarp();
		if (n_tiles > 0) ring_issue<false>(sm.rg, tbase16, nullptr, 0, lane, twobit);
		if (n_tiles > 1) ring_issue<false>(sm.rg, tbase16, nullptr, 1, lane, twobit);

		// match vectors of this lane's blocks: bit i of eq[c][lane][r] <=> read[row0 + 32 r + i] == symbol c
#pragma unroll
		for (int c = 0; c < NSYM; ++c)
#pragma unroll
			for (int r = 0; r < R; ++r) sm.eq[c][lane][r] = 0;
		for (int r = 0; r < R; ++r)
			for (uint32_t i = 0; i < 32u; ++i) {
				const uint32_t ri = row0 + 32u * r + i;
				if (ri < l1) sm.eq[symmap_s[read_sym(q, ri, twobit)]][lane][r] |= 1u << i;
			}
		__syncwarp();

		uint32_t Pv[R], Mv[R];
#pragma unroll
		for (int r = 0; r < R; ++r) { Pv[r] = 0xffffffffu; Mv[r] = 0; }      // M[i][0] = i (:301)
		// the pair's last row: which lane / block / bit holds it (last stripe only)
		const uint32_t lr = (l1 - 1) % RPP;
		const int own_r = (last_stripe && lane == (int)(lr / (32u * R))) ? (int)((lr % (32u * R)) / 32u) : -1;
		const uint32_t own_b = lr & 31u;
		int dist = (int)l1;                                                 // M[l1][0]

		// Horizontal differences travel as two bits: hp (+1) and hn (-1).  In a hand-off word column x of a
		// group has hp at bit 2x and hn at bit 2x+1.
		// lane 0: the predecessor's word holding the column in hand; lane 31: the word being assembled
		uint32_t in_bits = 0, in_group = 0xffffffffu, out_bits = 0, pf_group = 0xffffffffu;
		uint64_t pf_word = 0;                                              // lane 0: next group's word, requested a call ahead
		auto group_bits = [&](const uint32_t g) -> uint32_t {              // lane 0, stripe > 0: the predecessor's word of group g
			if (g != in_group) {
				uint64_t w = g == pf_group ? pf_word : ld_relaxed_u64(bnd_in + g);
				while ((w & 0xffffffff00000000ull) != tag_in) { __nanosleep(40); w = ld_relaxed_u64(bnd_in + g); }
				in_bits = (uint32_t)w; in_group = g;
			}
			return in_bits;
		};
		mbar_wait(&sm.rg.bar[0], ring_par & 1u); ring_par ^= 1u;
		if (twobit) ring_expand(sm.rg, 0, lane);
		// Start lag: follow the predecessor four groups behind, so that the words requested one call ahead
		// already carry its tag -- a follower on the predecessor's heels pays an L2 round trip per group.
		if (stripe && lane == 0) {
			const uint32_t g = min(3u, n_groups - 1u);
			while ((ld_relaxed_u64(bnd_in + g) & 0xffffffff00000000ull) != tag_in) __nanosleep(200);
		}
		__syncwarp();

		// Lane k works on column j = t - 2k - 1: a skew of TWO steps per lane.  What lane k-1 produces at step t
		// is needed by lane k only at step t+2, so the shuffle that carries it (about 28 cycles) is off the
		// critical path -- the chain per step is the column update alone.  inA / inB: the neighbour's outputs
		// received at the end of the previous two steps (inA is the one due now).
		uint32_t sP = 0, sN = 0, inA_p = 0, inA_n = 0, inB_p = 0, inB_n = 0;
		uint32_t lft[R], dg[R];                                            // PTR: pointer planes of the column just computed
		// one column of the lane's R blocks; eq[] = match vectors of the column's symbol, (hp, hn) = horizontal
		// difference entering the first block, replaced by the one leaving the last block
		auto column = [&](const uint32_t (&eq)[R], uint32_t &hp, uint32_t &hn) {
#pragma unroll
			for (int r = 0; r < R; ++r) {
				uint32_t Eq = eq[r];
				const uint32_t Xv = Eq | Mv[r];
				Eq |= hn;
				const uint32_t Xh = (((Eq & Pv[r]) + Pv[r]) ^ Pv[r]) | Eq;
				uint32_t Ph = Mv[r] | ~(Xh | Pv[r]);
				uint32_t Mh = Pv[r] & Xh;
				if constexpr (PTR) edit_bits_ptr(eq[r], Pv[r], Ph, Mh, lft[r], dg[r]);
				if (r == own_r) dist += (int)((Ph >> own_b) & 1u) - (int)((Mh >> own_b) & 1u);
				const uint32_t op = Ph >> 31, on = Mh >> 31;
				Ph = (Ph << 1) | hp;
				Mh = (Mh << 1) | hn;
				Pv[r] = Mh | ~(Xv | Ph);
				Mv[r] = Ph & Xv;
				hp = op; hn = on;
			}
		};
		auto pass_on = [&]() {                                             // end of a step: send this step's output down, age the queue
			inA_p = inB_p; inA_n = inB_n;
			inB_p = __shfl_up_sync(0xffffffffu, sP, 1); inB_n = __shfl_up_sync(0xffffffffu, sN, 1);
		};
		auto store_ptr = [&](const uint32_t t) {                          // PTR: the planes of step t's column
			uint2 *w = pp + ((size_t)(t >> 4) * R * 16 + (t & 15u)) * 32;
#pragma unroll
			for (int r = 0; r < R; ++r) w[r * 512] = make_uint2(lft[r], dg[r]);
		};
		auto step = [&](const uint32_t t) {                                // any step: range-checked
			const int j = (int)t - 2 * lane - 1;
			const bool on = j >= 1 && j <= (int)l2;
			uint32_t hp = inA_p, hn = inA_n;
			if (lane == 0 && on) {
				if (stripe == 0) { hp = 1; hn = 0; }                               // M[0][j] - M[0][j-1] = 1 (:302)
				else { const uint32_t w = group_bits(((uint32_t)j - 1u) >> 4) >> (2u * (((uint32_t)j - 1u) & 15u)); hp = w & 1u; hn = (w >> 1) & 1u; }
			}
			if (on) {
				const uint32_t y = (uint32_t)(j - 1) + sh;
				const uint32_t c = symmap_s[sm.rg.tring[y & 511u]];
				uint32_t eq[R];
#pragma unroll
				for (int r = 0; r < R; ++r) eq[r] = sm.eq[c][lane][r];
				column(eq, hp, hn);
				if constexpr (PTR) store_ptr(t);
				sP = hp; sN = hn;
				if (lane == 31 && !last_stripe) {
					out_bits |= (hp | (hn << 1)) << (2u * (((uint32_t)j - 1u) & 15u));
					if ((((uint32_t)j - 1u) & 15u) == 15u || j == (int)l2) { st_relaxed_u64(bnd_out + (((uint32_t)j - 1u) >> 4), tag_out | out_bits); out_bits = 0; }
				}
			}
			pass_on();
		};
		// 16 in-range steps (tb a multiple of 16, every lane inside the matrix: tb >= 64, tb + 14 <= l2).
		// Everything that is not on the serial chain is done up front: the shared-memory reads, and lane 0's
		// sixteen boundary inputs (columns tb-1, tb close the group in hand, tb+1 .. tb+14 open the next).
		// Lane 31's columns tb-63 .. tb-48 are exactly one group: one 64-bit store, no fence.
		auto steps16 = [&](const uint32_t tb) {
			uint64_t nw = 0;                                               // lane 0 requests the NEXT call's group now
			const uint32_t ng = (tb >> 4) + 1u;
			const bool pf = lane == 0 && stripe && ng < n_groups;
			if (pf) nw = ld_relaxed_u64(bnd_in + ng);
			uint32_t eq[16][R];
#pragma unroll
			for (int k = 0; k < 16; ++k) {
				const uint32_t y = (uint32_t)((int)(tb + k) - 2 * lane - 2) + sh;
				const uint32_t c = symmap_s[sm.rg.tring[y & 511u]];
#pragma unroll
				for (int r = 0; r < R; ++r) eq[k][r] = sm.eq[c][lane][r];
			}
			uint32_t tops = 0x55555555u;                                   // stripe 0: +1 in every column
			if (lane == 0 && stripe) {
				const uint32_t w0 = group_bits((tb - 2u) >> 4) >> 28;              // columns tb-1, tb: the last two of their group
				tops = w0 | (group_bits(tb >> 4) << 4);                            // columns tb+1 .. tb+14
			}
			const bool first = lane == 0;
			uint32_t packed = 0;
#pragma unroll
			for (int k = 0; k < 16; ++k) {
				uint32_t hp = inA_p, hn = inA_n;
				if (first) { hp = (tops >> (2 * k)) & 1u; hn = (tops >> (2 * k + 1)) & 1u; }
				column(eq[k], hp, hn);
				if constexpr (PTR) store_ptr(tb + k);
				sP = hp; sN = hn;
				packed |= (hp | (hn << 1)) << (2 * k);
				pass_on();
			}
			if (lane == 31 && !last_stripe) st_relaxed_u64(bnd_out + ((tb - 64u) >> 4), tag_out | packed);
			if (pf) { pf_word = nw; pf_group = ng; }
		};

		const uint32_t t_end = edit_bits_last_step(l2);
		for (uint32_t tb = 0; tb <= t_end; tb += 16) {
			if ((tb & 255u) == 96u && tb > 96u) {                          // lane 31 has left tile tb/256 - 1: refill its slot two tiles ahead
				const uint32_t c = (tb >> 8) + 1u;
				__syncwarp();
				if (c < n_tiles) ring_issue<false>(sm.rg, tbase16, nullptr, c, lane, twobit);
			}
			if ((tb & 255u) == tile_wait) {                                // lane 0 enters tile tb/256 + 1 within the next 32 steps (2-bit: 64)
				const uint32_t c = (tb >> 8) + 1u;
				if (c < n_tiles) { mbar_wait(&sm.rg.bar[c & 1u], (ring_par >> (c & 1u)) & 1u); ring_par ^= 1u << (c & 1u); if (twobit) ring_expand(sm.rg, c, lane); }
			}
			if (tb >= 64u && tb + 14u <= l2) {
				steps16(tb);
			} else {
#pragma unroll 1
				for (uint32_t k = 0; k < 16; ++k) step(tb + k);
			}
		}
		__syncwarp();

		if (own_r >= 0) { a.score[p] = dist; a.end_i[p] = l1; a.end_j[p] = l2; a.end_state[p] = ST_MID; }
		__syncwarp();
	}
}

}  // namespace atb2
