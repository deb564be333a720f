// at_cell.cuh -- the Gotoh cell update shared by K1 (at_fill_affine.cuh) and K2's affine kernel
// (at_wavefront.cuh): one cell of M / L / U (/ J) with the argmax of every max carried in the low bits of
// the values and the traceback pointers assembled on the FMA pipe.  Host + device: the same source is compiled
// by g++ into tests/cell_model (tests/test_cell_model.py checks it against the oracle without a GPU).
//
// Why it looks like this (ncu / SASS of round 1's kernels: the ALU pipe -- VIMNMX, VIADDMNMX, LOP3, IADD3 -- was
// 90 % busy while the FMA pipe -- IMAD -- idled; both issue one warp instruction per two cycles per SM
// sub-partition, so work moved from the ALU to the FMA pipe is free until the two are level):
//
//   * scores are kept x8: the three spare low bits of every value carry a TAG.  A candidate enters its max with
//     a tie-break tag, so ONE VIADDMNMX gives the value AND its argmax (first-strictly-greater rules of max5,
//     src/alignment.h:90-100, reproduced by the order of the tags):
//         H tags = 3 - pointer code:  L 3, M 2, U 1, JUMP / HOME 0   (L wins ties, then M, then U: SURVEY A.0)
//         Mo' = M + o carries tag 3;  L: extend (tag 3 + 4 = 7) beats open (3) on ties (:456);
//         U: open (3) beats extend (1) on ties (:460);  J: enter (3 - 2 = 1) beats stay (0) on ties (:660);
//         local M: the diagonal (tag >= 1) beats HOME = 0.0 (tag 0) on ties (:825).
//   * one LOP3 per propagated value drops the tag again (Lk = Lt & ~4, Uk = Ut & ~2, Mk = (Mt & ~3) | 2,
//     Jk = Jt & ~1); these CLEAN values are what the next cells consume;
//   * the pointer nibble of a cell is a LINEAR function of (tagged - clean):
//         nibble = 13 + (Mk + Lk + 4 Uk) - (Mt + Lt + 4 Ut)
//       = (3 - tag of M) + 4 [L opened] + 8 [U extended]      (K3's layout, at_ptr_layout.h)
//     so the kernels keep one accumulator per row, X = 16 X + (Mk + Lk + 4 Uk) - (Mt + Lt + 4 Ut) -- six
//     adds / multiply-adds on the FMA pipe, no shifts / masks / selects on the ALU pipe -- and store
//     X + 0xDDDDDDDD once per pointer word.  All of it is arithmetic mod 2^32, also for packed s16x2 lanes:
//     the per-half nibble sums never exceed 16 bits, so carries between the halves cancel in the sum.
//     The jump-bit plane works the same way: XJ = 2 XJ + (Jt - Jk), word = ~XJ.
//
// Reference recurrences: src/alignment.h:451-462 (global), :635-667 (fit + jump), :825-841 (local).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define AT_HD __host__ __device__ __forceinline__
#else
#define AT_HD inline
#endif

namespace atb2 {

enum { TAG_J = 0, TAG_U = 1, TAG_M = 2, TAG_L = 3 };      // tag of the winner of H = max(L, M, U[, J]); pointer code = 3 - tag
#define AT_PTR_BIAS 0xDDDDDDDDu                            // 13 per nibble (see above)

// -INFINITY stand-in (SURVEY.md A.7) in the x8-scaled score domain of the int32 lanes: a NEG-like value (AT_NEG
// plus up to B = 8 (l1+l2+2) max|param| of drift) never beats a finite one (>= -B) as long as 2 B < 2^29, i.e.
// (l1+l2+2)*max|param| < 2^25, which the host checks (validate_batch -> AT_E_RANGE).
#define AT_NEG (-(1 << 29))
#define AT_NEG_INIT (-(1 << 30) - (1 << 29))
// The same inside one half of the packed s16x2 lanes (x8 domain, before the 0x8000 bias): finite values stay above
// -24000 (host check), a -inf value lives for at most two steps next to a border before a finite candidate replaces
// it, so its drift stays far inside [-32768, -24000).
#define AT_NEG16 (-30000)

template <bool PACKED> struct Lanes;

// int32 lanes: one pair per warp
template <> struct Lanes<false> {
	typedef int32_t T;
	static constexpr uint32_t STEPS_PER_WORD = 8;
	static AT_HD T rep(int v) { return v; }                                  // small constant in every lane half
	static AT_HD T value(int v) { return 8 * v; }                            // a score
	static AT_HD T delta(int v) { return 8 * v; }                            // score difference, for plain adds
	static AT_HD T delta_h(int v) { return 8 * v; }                          // score difference, for the fused add of addmax
	static AT_HD T addmax(T a, T b, T c)
	{
#ifdef __CUDA_ARCH__
		return __viaddmax_s32(a, b, c);
#else
		const T s = (T)((uint32_t)a + (uint32_t)b); return s > c ? s : c;
#endif
	}
	static AT_HD T vmax(T a, T b) { return a > b ? a : b; }
	static AT_HD T vmax3(T a, T b, T c)
	{
#ifdef __CUDA_ARCH__
		return __vimax3_s32(a, b, c);
#else
		return vmax(vmax(a, b), c);
#endif
	}
};

// packed s16x2 lanes: TWO pairs per warp, pair A in bits 0-15 and pair B in bits 16-31 of every register.
// Values are BIASED by 0x8000 per half and compared unsigned (VIADDMNMX.U16x2 / VIMNMX3.U16x2), so every plain
// add / subtract is an ordinary 32-bit integer instruction: no carry crosses the halves while the values stay in
// range, which the host checks.
template <> struct Lanes<true> {
	typedef uint32_t T;
	static constexpr uint32_t STEPS_PER_WORD = 4;
	static AT_HD T rep(int v) { return (uint32_t)v * 0x10001u; }
	static AT_HD T value(int v) { return (uint32_t)(8 * v * 0x10001) + 0x80008000u; }
	static AT_HD T delta(int v) { return (uint32_t)(8 * v * 0x10001); }                     // exact 32-bit sum of both halves
	static AT_HD T delta_h(int v) { return ((uint32_t)(8 * v) & 0xffffu) * 0x10001u; }      // two's complement per half
	static AT_HD T addmax(T a, T b, T c)
	{
#ifdef __CUDA_ARCH__
		return __viaddmax_u16x2(a, b, c);
#else
		const uint32_t lo = (a + b) & 0xffffu, hi = ((a >> 16) + (b >> 16)) & 0xffffu;
		const uint32_t clo = c & 0xffffu, chi = c >> 16;
		return (lo > clo ? lo : clo) | ((hi > chi ? hi : chi) << 16);
#endif
	}
	static AT_HD T vmax(T a, T b)
	{
#ifdef __CUDA_ARCH__
		return __vmaxu2(a, b);
#else
		const uint32_t lo = (a & 0xffffu) > (b & 0xffffu) ? (a & 0xffffu) : (b & 0xffffu);
		const uint32_t hi = (a >> 16) > (b >> 16) ? (a >> 16) : (b >> 16);
		return lo | (hi << 16);
#endif
	}
	static AT_HD T vmax3(T a, T b, T c)
	{
#ifdef __CUDA_ARCH__
		return __vimax3_u16x2(a, b, c);
#else
		return vmax(vmax(a, b), c);
#endif
	}
};

// Hide a value's provenance from the compiler (no instruction is emitted).  Without it LLVM rewrites
// (ut & ~2) * 4 as (ut * 4) & ~8 to share the shift with ut * 4 -- one IMAD less, one LOP3 more, on the pipe that
// binds these kernels.
template <typename T> AT_HD T opaque(T v)
{
#ifdef __CUDA_ARCH__
	asm("" : "+r"(v));
#endif
	return v;
}

// Which kernels spell the pointer algebra's adds as explicit multiply-adds (FMA pipe) instead of leaving the choice of
// pipe to the compiler.  Measured (profiles/ab_fma_adds_r02.txt): the packed kernel is ALU-bound and gains 1.2 % (C2 fill
// 31.11 -> 30.75 ms); the int32 kernels already lean on the FMA pipe and LOSE (C3 46.0 -> 54.2 ms, global 150 x 150
// 1.35 -> 1.43 ms).  Hence: packed lanes only.
// The jump-plane accumulator of the int32 kernels on the FMA pipe alone (A/B knob, see DESIGN.md)
#ifndef AT_CELL_FMA_XJ
#define AT_CELL_FMA_XJ 0
#endif
#ifndef AT_CELL_FMA_ADDS
#define AT_CELL_FMA_ADDS(PACKED) (PACKED)
#endif

// a * b + c as ONE multiply-add on the FMA pipe.  Written in PTX so that neither LLVM nor ptxas re-associates it into
// IADD3 / LOP3 forms (ALU pipe); with b a register holding +-1 it is how these kernels add without touching the ALU pipe.
AT_HD uint32_t fma_mad(uint32_t a, uint32_t b, uint32_t c)
{
#ifdef __CUDA_ARCH__
	uint32_t d;
	asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
	return d;
#else
	return a * b + c;
#endif
}

// values of the k_and / k_or kernel arguments (see CellConst::set)
template <bool PACKED> AT_HD uint32_t cell_k_and() { return (uint32_t)~Lanes<PACKED>::rep(3); }
template <bool PACKED> AT_HD uint32_t cell_k_or() { return (uint32_t)Lanes<PACKED>::rep(TAG_M); }

// Constants of one kernel instance (they live in registers / uniform registers).
template <bool PACKED> struct CellConst {
	typedef typename Lanes<PACKED>::T T;
	T zero;        // local: the HOME candidate 0.0 (tag 0)
	T e_l;         // 8 e + 4, fused-add form: L extends with tag 3 + 4 = 7
	T e_u;         // 8 e, fused-add form: U extends with tag 1
	T o_m;         // 8 o + 1, plain-add form: Mo' = Mk + o_m carries tag 3
	T m_and, m_or; // Mk = (Mt & m_and) | m_or = clean | 2, as registers
	T j_enter;     // 8 (jump - o) - 2, fused-add form: entering J from Mo' carries tag 1
	T j_barred;    // the same on a black-listed target index: -inf
	uint32_t one, neg1;   // +1 / -1 the compiler cannot see through (derived from k_or): multipliers of fma_mad
	// k_and / k_or: ~3 and TAG_M in every lane half, handed in as KERNEL ARGUMENTS: constants the compiler can see
	// become immediates, and a LOP3 takes only one -- (x & c1) | c2 would be two instructions on the binding pipe;
	// with both in registers it is one
	AT_HD void set(int o, int e, int jp, uint32_t k_and, uint32_t k_or)
	{
		typedef Lanes<PACKED> V;
		zero = V::value(0);
		e_l = V::delta_h(e) + V::rep(4);
		e_u = V::delta_h(e);
		o_m = V::delta(o) + V::rep(1);
		m_and = (T)k_and;
		m_or = (T)k_or;
		one = (k_or >> 1) & 1u;      // TAG_M = 2 in the low half: always 1, but only at run time
		neg1 = 0u - one;
		j_enter = PACKED ? (T)0 : (T)(8 * (jp - o) - 2);
		j_barred = PACKED ? (T)0 : (T)AT_NEG;
	}
};

// State of one row between two columns (registers of the lane that owns the row).
template <bool PACKED, bool JUMP> struct RowState {
	typedef typename Lanes<PACKED>::T T;
	T mo;          // M(i, j-1) + o, tag 3
	T u;           // U(i, j-1), tag 1
	T h;           // H(i, j-1) = max(L, M, U[, J]), tag of the winner
	T j;           // J(i, j-1), tag 0 (JUMP only)
	uint32_t x;    // pointer-word accumulator: 16 x + (clean - tagged) per step
	uint32_t xj;   // jump-bit plane accumulator: 2 xj + (tagged - clean) per step (JUMP only)
};

// What a cell hands to the row below it (same column) and to the kernel's end-cell logic.
template <bool PACKED> struct CellOut {
	typedef typename Lanes<PACKED>::T T;
	T lk;          // L(i, j) clean, tag 3     -> Lup of row i+1
	T mo;          // M(i, j) + o, tag 3       -> MoUp of row i+1
	T mk;          // M(i, j) clean, tag 2     (local: running maximum; fit: last-row search)
	T h;           // H(i, j), tagged          (global: the corner)
};

// One cell.  d: H(i-1, j-1) tagged; pw: 8 s(i, j) (LOCAL && FUSED: fused-add form, else plain-add form);
// lup / mo_up: L(i-1, j) clean and M(i-1, j) + o; jadd: c.j_enter or c.j_barred for this column; mul: 16, or 0 on the
// first step of a pointer word (packed lanes restart their accumulators: the halves must not spill into each
// other); mulj: 2, or 0 on the first step of a jump-plane word.  Returns the new D for the row below: H(i, j-1).
template <int MODE_LOCAL_, bool JUMP, bool PACKED, bool FUSED>
AT_HD typename Lanes<PACKED>::T cell_update(const CellConst<PACKED> &c, RowState<PACKED, JUMP> &st, const typename Lanes<PACKED>::T d,
                                            const typename Lanes<PACKED>::T pw, const typename Lanes<PACKED>::T lup,
                                            const typename Lanes<PACKED>::T mo_up, const typename Lanes<PACKED>::T jadd,
                                            const uint32_t mul, const uint32_t mulj, CellOut<PACKED> &out)
{
	typedef Lanes<PACKED> V;
	typedef typename V::T T;
	T mt;
	if (MODE_LOCAL_) mt = FUSED ? V::addmax(d, pw, c.zero) : V::vmax((T)(d + pw), c.zero);      // HOME: 0.0 strictly greater (:825)
	else mt = d + pw;                                                                           // the diagonal's tag rides along
	const T lt = V::addmax(lup, c.e_l, mo_up);           // tag 7: extended (ties included, :456), 3: opened
	const T ut = V::addmax(st.u, c.e_u, st.mo);          // tag 1: extended, 3: opened (ties included, :460)
	const T mk = opaque<T>((mt & c.m_and) | c.m_or);
	const T lk = opaque<T>(lt & ~V::rep(4));
	const T uk = opaque<T>(ut & ~V::rep(2));
	const T mo = AT_CELL_FMA_ADDS(PACKED) ? (T)fma_mad((uint32_t)mk, c.one, (uint32_t)c.o_m) : (T)(mk + c.o_m);
	T h = V::vmax3(lk, mk, uk);
	T jk = 0, jt = 0;
	if (JUMP) {
		jt = V::addmax(st.mo, jadd, st.j);               // tag 1: entered from M(i, j-1) (ties included, :660), 0: stayed
		jk = opaque<T>(jt & ~V::rep(1));
		h = V::vmax(h, jk);                              // J is the last argument of max5: it wins only when strictly greater
	}
	// pointer accumulator (FMA pipe): clean minus tagged, earliest step in the top nibble
	if (AT_CELL_FMA_ADDS(PACKED)) {
		uint32_t dx = fma_mad((uint32_t)mk, c.one, (uint32_t)lk);
		dx = fma_mad((uint32_t)mt, c.neg1, dx);
		dx = fma_mad((uint32_t)lt, c.neg1, dx);
		dx = (uint32_t)uk * 4u + dx;
		dx = (uint32_t)ut * 0xfffffffcu + dx;
		st.x = st.x * mul + dx;
	} else {
		st.x = st.x * mul + (((uint32_t)(lk + mk) - (uint32_t)(lt + mt)) + (uint32_t)uk * 4u - (uint32_t)ut * 4u);
	}
	if (JUMP) {
		if (AT_CELL_FMA_XJ && !PACKED) {      // both terms as multiply-adds: the compiler's own choice is x + x on the FMA pipe and an IADD3 on the ALU pipe
			const uint32_t t2 = fma_mad(st.xj, mulj, (uint32_t)jt);
			st.xj = fma_mad((uint32_t)jk, c.neg1, t2);
		} else st.xj = st.xj * mulj + ((uint32_t)jt - (uint32_t)jk);
	}
	const T d_next = st.h;
	st.h = h; st.u = uk; st.mo = mo;
	if (JUMP) st.j = jk;
	out.lk = lk; out.mo = mo; out.mk = mk; out.h = h;
	return d_next;
}

// the word a row stores after STEPS_PER_WORD steps / after 32 steps of the jump plane
AT_HD uint32_t ptr_word(uint32_t x) { return x + AT_PTR_BIAS; }
AT_HD uint32_t jump_word(uint32_t xj) { return ~xj; }

// ------------------------------------------------------------------------------------------------
// Single-plane cell (overlap: max-plus with a linear gap, src/alignment.h:940-949), int32 lanes.
// Values are kept x4 and every cell carries A = 4 M + 4 o (what its right and lower neighbours add anyway).
// Tags in the two spare bits reproduce max5's order LEFT, DIAGONAL, RIGHT (:944-947, first strictly greater):
//     LEFT 2, DIAGONAL 1, RIGHT 0;   pointer code (K3: bit 1 RIGHT, bit 0 DIAGONAL) = 2 - tag.
// A cell hands on its value in two forms: `a` (tag 0: the RIGHT candidate of the row below) and `a2` = a + 2 (its own
// LEFT candidate one column later, and the diagonal input of the row below, whose profile word carries - 1).
//     vt = max3(a2(i, j-1), a2(i-1, j-1) + 4 (s - o) - 1, a(i-1, j))        one VIMNMX3: value + argmax
//     x  = 4 x + (vt - (vt & ~3))                                           the 2-bit pointers: word = 0xAAAAAAAA - x
// ------------------------------------------------------------------------------------------------
#define AT_NEGL (-(1 << 30))       // -inf stand-in of the single-plane kernel (scores x4 stay below 2^29)
#define AT_LIN_BIAS 0xAAAAAAAAu    // 2 per 2-bit field

struct LinRow { int a2; uint32_t x; };      // A(i, j-1) + 2 and the pointer accumulator of one row

// d2: a2(i-1, j-1); pw: 4 (s(i, j) - o) - 1; a_up: a(i-1, j); gap = 4 o.  Returns a(i, j); st.a2 is replaced by
// a2(i, j) and the OLD st.a2 -- the diagonal input of the row below -- comes back through d2_next.
AT_HD int lin_update(LinRow &st, const int d2, const int pw, const int a_up, const int gap, int &d2_next)
{
	const int diag = d2 + pw;
#ifdef __CUDA_ARCH__
	const int vt = __vimax3_s32(st.a2, diag, a_up);
#else
	int vt = st.a2 > diag ? st.a2 : diag; vt = vt > a_up ? vt : a_up;
#endif
	const int vk = opaque<int>(vt & ~3);
	st.x = st.x * 4u + ((uint32_t)vt - (uint32_t)vk);
	d2_next = st.a2;
	st.a2 = vk + (gap + 2);
	return vk + gap;
}
AT_HD uint32_t lin_word(uint32_t x) { return AT_LIN_BIAS - x; }

// ------------------------------------------------------------------------------------------------
// Edit distance paths (AT_OUT_EDIT_PATH).  The pointer of a cell is min3's argmin (src/alignment.h:280-286) with the
// first-strictly-smaller rule in argument order: LEFT 0, DIAGONAL 1, UP 2 -- the 2-bit code overlap's walker reads
// (bit 1 UP, bit 0 DIAGONAL), so the cell-by-cell kernel stores it in overlap's layout.
// Cell-by-cell: the candidates x4 with the code in the two low bits; one VIMNMX3 gives value (vt >> 2) and code (vt & 3).
// ------------------------------------------------------------------------------------------------
AT_HD int edit_min3_tagged(const int left, const int diag, const int up)      // M(i, j-1), M(i-1, j-1) + s, M(i-1, j)
{
	const int a = 4 * left + 4, b = 4 * diag + 1, c = 4 * up + 6;
#ifdef __CUDA_ARCH__
	return __vimin3_s32(a, b, c);
#else
	int v = a < b ? a : b; return v < c ? v : c;
#endif
}

// Bit-parallel kernel (`edit -u 1`): the two pointer planes of one 32-row block column, from the vectors the column update
// holds.  pv: vertical +1 deltas of column j-1 (before the update); ph / mh: horizontal +1 / -1 deltas of column j at the
// block's rows (before the shift); eq: the PURE match vector of column j's symbol (without the carried-in hn).
//   LEFT  iff M(i, j) = M(i, j-1) + 1, i.e. the horizontal delta is +1;
//   DIAG  iff not LEFT and M(i, j) - M(i-1, j-1) = s(i, j).  That difference, d = dh(i, j) + dv(i, j-1), is 0 or 1;
//         on a match s = 0 and d = 0 always, on a mismatch s = 1 and, with dh in {0, -1}, d = 1 iff dh = 0 and dv = +1.
//   UP    otherwise.
AT_HD void edit_bits_ptr(const uint32_t eq, const uint32_t pv, const uint32_t ph, const uint32_t mh, uint32_t &left, uint32_t &diag)
{
	left = ph;
	diag = ~ph & (eq | (pv & ~mh));
}

}  // namespace atb2
