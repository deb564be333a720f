/* aligntools_b200.h -- C-ABI of the B200-native alignTools DP core.
 *
 * Drop-in boundary for the hot path of r3fang/alignTools.C: the Gotoh M/L/U(/J) matrix
 * fill and traceback behind `global | local | fit [-s -j] | overlap | edit`.  The
 * reference has no FFI; its de-facto operator interface is the five static-inline
 * functions in src/alignment.h, called from the printf argument of each main_<mode>
 * (src/alignment.h:345, 509, 736, 885, 1000).  This header gives
 *
 *   (1) single-pair shims with the reference's own signatures (section B), so the five
 *       main_<mode> drivers can stay byte-for-byte and only the callee changes;
 *   (2) a batched entry (section C) that takes thousands..millions of read/target pairs,
 *       packs them into device buffers and runs fill + traceback on one or more B200s.
 *
 * Plain C types only.  There is NO CPU fallback: every entry fails with AT_E_CUDA when
 * no sm_100 device / driver is usable.
 *
 * Conventions (SURVEY.md Appendix A): s1 = first FASTA record = rows i = "read";
 * s2 = second record = columns j = "target".  Scoring is raw byte equality
 * (src/alignment.h:449, 632, 824, 943, 305); at_batch_*_scored (section C) takes a substitution
 * matrix instead.  All results are bit-exact with the reference, quirks included (A.6).
 */
#ifndef ALIGNTOOLS_B200_H
#define ALIGNTOOLS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ A. common ---- */

/* sub-commands of src/main.c:40-44 */
enum at_mode {
	AT_GLOBAL  = 0,   /* align_gla               src/alignment.h:417-473 */
	AT_LOCAL   = 1,   /* align_local_affine      src/alignment.h:805-847 */
	AT_FIT     = 2,   /* align_fit_affine_jump   src/alignment.h:596-694 (jump iff params.jump) */
	AT_OVERLAP = 3,   /* align_overlap           src/alignment.h:926-964 */
	AT_EDIT    = 4    /* edit_dist               src/alignment.h:291-315 */
};

/* return codes (0 ok, <0 error).  The CLI host maps them onto the reference's die()
 * messages / exit codes (src/alignment.h:69-79). */
enum at_rc {
	AT_OK        =  0,
	AT_E_ARG     = -1,  /* NULL / malformed argument ("parameter error", :419)             */
	AT_E_CUDA    = -2,  /* no usable sm_100 device, or a CUDA call failed (no CPU fallback) */
	AT_E_NOMEM   = -3,  /* host or device allocation failed ("mycalloc failure", :85)       */
	AT_E_FITLEN  = -4,  /* fit: l1 > l2 ("first sequence must be shorter...", :599)         */
	AT_E_NOSPACE = -5,  /* caller's output buffer too small                                 */
	AT_E_RANGE   = -6,  /* (l1+l2)*max|param| does not fit the int32 score lanes            */
	AT_E_UNDEF   = -7   /* input on which the reference itself is undefined (empty record,
	                       fit with l2 < 2: uninitialised j_max, SURVEY.md A.3)             */
};

/* opt_t without the host-only members (src/alignment.h:57-65); defaults = init_opt() :102-114 */
typedef struct at_params {
	int32_t m;      /* match score        [ 1]  */
	int32_t u;      /* mismatch           [-2]  */
	int32_t o;      /* gap open           [-5]  */
	int32_t e;      /* gap extension      [-1]  */
	int32_t j;      /* jump penalty       [-10] */
	int32_t jump;   /* 0 = no jump state; 1 = `-s` given (the reference stores this as opt->s == true == 0): the site
	                   list is a BLACKLIST, bit-exact with the reference (SURVEY.md A.3); 2 = jump state with the
	                   site list as a WHITELIST -- entering J only on the listed target indices, the semantics
	                   the reference's own comments describe (src/alignment.h:542-544) but do not implement */
} at_params;

void        at_default_params(at_params *p);
const char *at_strerror(int rc);
/* version string + compiled arch, e.g. "aligntools-b200 0.1 (sm_100a)" */
const char *at_version(void);

typedef struct at_handle at_handle;

/* devices == NULL or n_devices <= 0: use device 0 only.  One host thread + stream per
 * device; pairs are sharded as contiguous slices, no inter-GPU communication.
 * Threading: a handle serves one batch operation at a time (at_batch_align serialises its callers;
 * at_batch_create / run / fetch of DIFFERENT batches on one handle must not overlap in time).  Use one
 * handle per host thread for concurrent work; handles are independent. */
int         at_create(const int *devices, int n_devices, at_handle **out);
void        at_destroy(at_handle *h);
const char *at_last_error(const at_handle *h);
int         at_device_count(const at_handle *h);
/* number of kernels of THIS library launched through the handle so far */
uint64_t    at_launch_count(const at_handle *h);

/* ------------------------------------------- B. single-pair, reference signatures ---- */

/* layout-compatible with kstring_t (src/kstring.h:56-59) */
typedef struct at_kstring_t { size_t l, m; char *s; } at_kstring_t;
/* layout-compatible with junction_t / opt_t (src/alignment.h:51-65); `s` follows the
 * reference's enum: 0 means jump enabled ("true"), 1 means disabled ("false"). */
typedef struct at_junction_t { size_t size; int *pos; } at_junction_t;
typedef struct at_opt_t { int o, e, m, u, j; int s; at_junction_t sites; } at_opt_t;

/* Each replaces the reference function of the same suffix.  Ownership as in the
 * reference (SURVEY.md 8b): the caller allocates r1->s / r2->s with at least l1+l2
 * bytes; on return r->s has been REPLACED by a fresh malloc'ed NUL-terminated string
 * (the old block is freed, as strrev does at :176-183) and r->l is the alignment length.
 * Errors follow die(): "FATAL ERROR: ..." on stderr and exit(-1). */
double at_align_gla(at_kstring_t *s1, at_kstring_t *s2, at_kstring_t *r1, at_kstring_t *r2, at_opt_t *opt);             /* :417 */
double at_align_local_affine(at_kstring_t *s1, at_kstring_t *s2, at_kstring_t *r1, at_kstring_t *r2, at_opt_t *opt);    /* :805 */
double at_align_fit_affine_jump(at_kstring_t *s1, at_kstring_t *s2, at_kstring_t *r1, at_kstring_t *r2, at_opt_t *opt); /* :596 */
double at_align_overlap(at_kstring_t *s1, at_kstring_t *s2, at_kstring_t *r1, at_kstring_t *r2, at_opt_t *opt);         /* :926 */
int    at_edit_dist(at_kstring_t *s1, at_kstring_t *s2, at_opt_t *opt);                                                 /* :291 */

/* ------------------------------------------------------------- C. batched entry ---- */

enum at_seq_encoding {
	AT_SEQ_BYTES = 0,  /* one byte per symbol, any alphabet, compared verbatim            */
	AT_SEQ_2BIT  = 1   /* four symbols per byte (A,C,G,T -> 0..3, symbol k of a record in
	                      bits 2*(k&3) of byte k>>2); every record starts on a byte boundary
	                      and *_off are BYTE offsets.  See at_pack_2bit().  The records stay
	                      packed in device memory and every kernel reads the codes directly;
	                      records on 16-byte boundaries are read with 128-bit loads.       */
};

typedef struct at_batch_input {
	uint64_t        n_pairs;
	uint32_t        encoding;   /* enum at_seq_encoding */
	const uint8_t  *q;          /* reads   (s1), concatenated                              */
	const uint64_t *q_off;      /* [n_pairs]  offset of pair p's read in q                 */
	const uint32_t *q_len;      /* [n_pairs]  l1 in symbols                                */
	const uint8_t  *t;          /* targets (s2), concatenated                              */
	const uint64_t *t_off;      /* [n_pairs]                                               */
	const uint32_t *t_len;      /* [n_pairs]  l2 in symbols                                */
	const int32_t  *sites;      /* fit+jump: 0-based target indices where ENTERING the jump
	                               state is forbidden (blacklist, SURVEY.md A.3); may be NULL */
	const uint64_t *site_off;   /* [n_pairs+1] slice of `sites` per pair; NULL iff sites NULL */
} at_batch_input;

enum at_out_flags {
	AT_OUT_SCORE = 0,        /* score, end cell and end state are always produced           */
	AT_OUT_CIGAR = 1u << 0,  /* run traceback, emit run-length ops                          */
	AT_OUT_ALN   = 1u << 1,  /* run traceback, emit the two gapped strings (r1, r2)         */
	AT_OUT_EDIT_PATH = 1u << 2   /* AT_EDIT: honour AT_OUT_CIGAR / AT_OUT_ALN (below); other
	                                modes ignore it                                           */
};

/* Edit paths.  AT_EDIT runs its traceback only when AT_OUT_EDIT_PATH is set together with AT_OUT_CIGAR and/or AT_OUT_ALN,
 * which then select the outputs as for the other modes.  Without AT_OUT_EDIT_PATH an edit batch is score-only whatever the
 * other flags say: no pointers are stored (at_timing.ptr_bytes 0) and cigar_off / aln_off come back all zero -- so callers
 * that pass CIGAR | ALN for every mode do not start writing 2 bits per cell (2.5 GB for a 100 kbp x 100 kbp pair).
 * The path is the traceback edit_dist (src/alignment.h:291-315) would have, with the conventions of the other modes:
 *   - the recurrence and borders are unchanged: M[i][0] = i, M[0][j] = j,
 *     M[i][j] = min3(M[i][j-1] + 1, M[i-1][j-1] + (s1[i-1] == s2[j-1] ? 0 : u), M[i-1][j] + 1);
 *   - a cell's pointer is min3's argmin, first strictly smaller in argument order: LEFT wins ties, then DIAG, then UP;
 *   - the walk starts at (l1, l2) and, reading the pointer of the cell before each move, runs while i > 0 && j > 0:
 *     LEFT emits (-, s2[--j]) as AT_CIG_D, DIAG (s1[--i], s2[--j]) as AT_CIG_M, UP (s1[--i], -) as AT_CIG_I;
 *   - then the rest of the target (AT_CIG_D) and the rest of the read (AT_CIG_I) are flushed, as global's traceback does.
 * end = (l1, l2), end state MID; beg_i / beg_j = the cell where the walk stopped, before the flush; the score is unchanged.
 * The path's cost -- 0 per equal M column, u per unequal one, 1 per I or D column -- equals the score for every u.
 * The bit-parallel kernel (u = 1, reads of <= 8 distinct bytes) and the cell-by-cell one give identical results.
 * at_timing.ptr_bytes reports the pointers (about l1 * l2 / 4 bytes per pair); they are chunked by the pointer arena as
 * for the other modes. */

/* CIGAR op = (run_length << 4) | code; columns left to right (SURVEY.md A.8) */
enum at_cigar_op { AT_CIG_M = 0 /* (x,y) */, AT_CIG_I = 1 /* (x,-) LOW */,
                   AT_CIG_D = 2 /* (-,y) UPP/LEFT */, AT_CIG_N = 3 /* (-,y) JUMP */ };

typedef struct at_batch_output {
	int32_t  *score;      /* [n]   DP score / edit distance                               */
	uint32_t *end_i;      /* [n]   matrix cell the traceback starts from; may be NULL     */
	uint32_t *end_j;
	uint32_t *beg_i;      /* [n]   matrix cell where the traceback stopped; may be NULL   */
	uint32_t *beg_j;
	uint32_t *cigar;      /* dense ops of all pairs; NULL to skip                         */
	uint64_t  cigar_cap;  /* capacity of `cigar` in ops                                   */
	uint64_t *cigar_off;  /* [n+1] pair p owns cigar[cigar_off[p] .. cigar_off[p+1])      */
	char     *aln1;       /* dense gapped strings r1 / r2 (no terminators); NULL to skip  */
	char     *aln2;
	uint64_t  aln_cap;    /* capacity of aln1 and of aln2 in bytes                        */
	uint64_t *aln_off;    /* [n+1] pair p owns aln?[aln_off[p] .. aln_off[p+1])           */
} at_batch_output;

typedef struct at_timing {
	double   fill_ms;        /* device time in the fill kernels (CUDA events), max over devices      */
	double   traceback_ms;   /* device time in the traceback kernels, max over devices               */
	double   device_ms;      /* first kernel start -> last kernel end, max over devices              */
	uint64_t cells;          /* sum of l1*l2 over all pairs; banded batches: the in-band cells exactly */
	uint64_t launches;       /* kernels launched by this run                                         */
	uint64_t ptr_bytes;      /* traceback-pointer bytes written to HBM                               */
	double   fill_kernel_ms; /* average duration of ONE launch of the dominant fill kernel           */
	uint64_t fill_kernel_cells; /* cells one such launch processes                                   */
	uint32_t fill_kernel_kind;  /* which kernel that was: enum at_kernel_kind                            */
	uint32_t fill_kernel_rows;  /* its rows per lane (AT_K_EDIT_BITS: 32-row blocks per lane)            */
	uint32_t fill_kernel_flags; /* bit 0: query-profile variant, bit 1: jump state, bit 2: sequences 2-bit packed in HBM, bit 3: substitution matrix */
	uint32_t reserved_;
} at_timing;

/* kernels a fill launch can be (at_timing.fill_kernel_kind) */
enum at_kernel_kind {
	AT_K_FILL_INT32  = 0,  /* at_fill_affine, int32 lanes, one pair per warp            */
	AT_K_FILL_S16X2  = 1,  /* at_fill_affine, packed s16x2 lanes, two pairs per warp    */
	AT_K_WAVE        = 2,  /* at_wave_affine / at_wave_linear, stripes of one pair      */
	AT_K_EDIT_BITS   = 3   /* at_wave_edit_bits, bit-parallel unit-cost edit distance   */
};

typedef struct at_batch at_batch;

/* Validate, pack and upload (H2D) a batch.  out_flags: OR of at_out_flags. */
int  at_batch_create(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                     uint32_t out_flags, at_batch **out);
/* Fill + traceback on the device(s); inputs are already resident.  May be called
 * repeatedly (benchmark steps); results of the last run are kept for at_batch_fetch. */
int  at_batch_run(at_batch *b, at_timing *timing /* may be NULL */);
/* Totals of the last run, to size the dense output buffers. */
int  at_batch_sizes(const at_batch *b, uint64_t *cigar_ops, uint64_t *aln_bytes);
/* D2H of the last run's results into caller memory. */
int  at_batch_fetch(at_batch *b, at_batch_output *out);
void at_batch_free(at_batch *b);

/* One-shot: create + run + fetch + free (host buffers in, host buffers out). */
int  at_batch_align(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                    uint32_t out_flags, at_batch_output *out, at_timing *timing);

/* Banded overlap alignment: pair p only fills the cells (i, j) of its band lo[p] <= j - i <= hi[p] (diagonals of the DP
 * matrix, 1 <= i <= l1, 1 <= j <= l2; the band is clipped to [1 - l1, l2 - 1] in 64 bits, and may be empty).  Cells
 * outside it are -inf; row 0 stays -inf and M[i][0] = 0, ties, the end search (last row, columns 0 .. l2-1) and the
 * traceback are the reference's.  An empty band gives score 0, end cell (l1, 0) and an empty alignment.
 * Identity: when every cell of the unbanded traceback path (its end cell included, its column-0 start excluded) lies
 * in the band, the banded result equals the unbanded one in every field -- a full band gives exactly at_batch_align's.
 * Only K2's stripe windows are filled and only their pointers are stored, so a caller that knows where the overlap lies
 * (seed or minimizer chains) pays for the band, not for l1 x l2.  at_timing.cells counts the in-band cells; ptr_bytes is
 * what the banded pointer blocks took.  band == NULL is the unbanded path.  AT_E_ARG (at_last_error names the reason
 * and the pair): a band with a mode other than AT_OVERLAP or AT_GLOBAL, a NULL lo or hi, lo[p] > hi[p], a global pair
 * whose band misses its end diagonal (below).  Results are sized and fetched with at_batch_run / at_batch_sizes /
 * at_batch_fetch as for any batch.
 *
 * Banded global alignment (mode AT_GLOBAL, affine gaps): a cell (i, j), 1 <= i <= l1, 1 <= j <= l2, whose diagonal
 * j - i lies outside the band (clipped as above) is -inf in M, L and U and its pointer is never read.  Everything else
 * is the reference's: row 0 and column 0 keep their border values, the end cell is (l1, l2) with max5's end state, and
 * the traceback, then the flush of the rest of the target and of the read, follow trace_back_gla.  The band must hold
 * the end diagonal, lo[p] <= l2 - l1 <= hi[p] (else AT_E_ARG; checked per pair after lo > hi): then every in-band cell
 * is finite and a banded global result always exists.  Identity: when every cell (i >= 1, j >= 1) of the unbanded
 * traceback path, end cell included, lies in the band, the banded result equals the unbanded one in every field.
 * Banded global pairs all run on the wavefront kernel (K2), short ones included; at_timing.cells and ptr_bytes are as
 * for overlap.  Local, fit and edit take no band. */
typedef struct at_band {
	const int32_t *lo;     /* [n_pairs] lowest diagonal d = j - i of the band  */
	const int32_t *hi;     /* [n_pairs] highest diagonal                        */
} at_band;
int  at_batch_create_banded(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                            const at_band *band, uint32_t out_flags, at_batch **out);
int  at_batch_align_banded(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                           const at_band *band, uint32_t out_flags, at_batch_output *out, at_timing *timing);

/* Substitution scores: s(a, b) = matrix[a * 256 + b] for read byte a (s1, rows) and target byte b (s2, columns).
 * Any byte may occur, the table need not be symmetric, and p->m / p->u are ignored; o, e, j and jump keep their meaning.
 * AT_SEQ_2BIT input: codes 0..3 stand for the bytes 'A', 'C', 'G', 'T'.
 * sc == NULL behaves exactly like at_batch_create / at_batch_align.  Modes AT_GLOBAL, AT_LOCAL, AT_FIT (jump 0, 1 or 2) and
 * AT_OVERLAP keep the reference's recurrence, borders, max5 first-strictly-greater ties, end-cell search (fit still excludes
 * column l2), traceback and flush; only s(i, j) = s(s1[i-1], s2[j-1]) comes from the table instead of m / u.  Identity: with
 * matrix[a * 256 + b] = (a == b ? m : u) the results equal at_batch_align's in every field.
 * AT_E_ARG (at_last_error names the reason): AT_EDIT with a matrix, a NULL matrix.  AT_E_RANGE: the score-range bound of
 * at_batch_create with max(|o|, |e|, |j|, max |matrix entry|) in place of max(|m|, |u|, ...).
 * Kernels: when a shard's targets use at most 4 distinct bytes (DNA, every 2-bit batch) the query-profile variants run with
 * profiles built from the matrix (no extra work per cell); otherwise the table variants look s up per cell in a compact
 * [read symbol][target symbol] table in shared memory (at_timing.fill_kernel_flags bit 3 marks a scored run, bit 0 the
 * profile variant).  Results are sized and fetched with at_batch_run / at_batch_sizes / at_batch_fetch as for any batch. */
typedef struct at_scoring {
	const int8_t *matrix;  /* [256 * 256] */
} at_scoring;
int  at_batch_create_scored(at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                            const at_scoring *sc, uint32_t out_flags, at_batch **out);
int  at_batch_align_scored (at_handle *h, int mode, const at_params *p, const at_batch_input *in,
                            const at_scoring *sc, uint32_t out_flags, at_batch_output *out, at_timing *timing);

/* Sharding plan (SURVEY.md 8e): cut pairs [0, n) into `parts` CONTIGUOUS slices holding nearly equal
 * numbers of DP cells (sum of l1*l2).  cut[] receives parts+1 ascending indices, cut[0] = 0 and
 * cut[parts] = n; slice r is [cut[r], cut[r+1]).  at_batch_create shards a batch over the handle's
 * devices with exactly this plan; a multi-process host (one rank per GPU) calls it to find each
 * rank's slice.  Pure host code. */
int  at_plan_slices(const uint32_t *q_len, const uint32_t *t_len, uint64_t n_pairs, uint32_t parts, uint64_t *cut);

/* Page-locked host memory for the caller's batch buffers: with pinned inputs and outputs the copies of at_batch_align
 * overlap its kernels (pageable memory works too, through the driver's staging buffers).  NULL when the allocation
 * fails.  Pure convenience over cudaHostAlloc / cudaFreeHost, so that a C host needs no CUDA headers. */
void *at_host_alloc(size_t bytes);
void  at_host_free(void *p);
/* Page-lock memory the caller already owns (e.g. a shared-memory segment several ranks write their slices into);
 * 0 on success.  Undo with at_host_unregister before the memory is released. */
int   at_host_register(void *p, size_t bytes);
int   at_host_unregister(void *p);

/* Helpers: 2-bit packing (returns number of bytes written = (n+3)/4, or <0 when a symbol
 * is not one of ACGT/acgt... only upper-case ACGT are accepted: the reference compares
 * bytes verbatim, so folding case would change results) and CIGAR rendering. */
int64_t at_pack_2bit(const char *seq, uint64_t n, uint8_t *dst);
int64_t at_cigar_to_string(const uint32_t *ops, uint64_t n_ops, char *dst, uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* ALIGNTOOLS_B200_H */
