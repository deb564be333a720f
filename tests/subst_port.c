/* Substitution-matrix scoring, CPU restatement for the tests (tests/subst_port.py): affine_align and overlap_align of
 * oracle/at_oracle.c (global / local / fit [+jump] and overlap, with their borders, max5 ties, end searches, tracebacks
 * and flushes), copied as they are except for one line each: the substitution score of cell (i, j) is
 * mat[s1[i-1] * 256 + s2[j-1]] (include/aligntools_b200.h, at_scoring) instead of m / u. */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { AT_GLOBAL = 0, AT_LOCAL = 1, AT_FIT = 2, AT_OVERLAP = 3 };
enum { P_NONE = 0, P_LOW = 1, P_MID = 2, P_UPP = 3, P_JUMP = 4, P_HOME = 5,
       P_LEFT = 1, P_DIAG = 2, P_RIGHT = 3 };

#define NEG (INT64_MIN / 4)
static inline int64_t norm(int64_t v) { return v < NEG / 2 ? NEG : v; }
static inline int64_t addn(int64_t v, int64_t d) { return v == NEG ? NEG : v + d; }

/* max5 (:90-100): scan in order, replace only when strictly greater, start at -inf.
 * Returns the winning index or -1 when every argument is -inf (the reference leaves
 * `state` uninitialised there; such cells are never visited by a traceback). */
static inline int max5i(int64_t *res, int64_t a1, int64_t a2, int64_t a3, int64_t a4, int64_t a5)
{
	int st = -1; *res = NEG;
	if (a1 > *res) { *res = a1; st = 0; }
	if (a2 > *res) { *res = a2; st = 1; }
	if (a3 > *res) { *res = a3; st = 2; }
	if (a4 > *res) { *res = a4; st = 3; }
	if (a5 > *res) { *res = a5; st = 4; }
	return st;
}

typedef struct {
	int64_t score;
	int32_t end_i, end_j;   /* cell the traceback starts from (1-based matrix indices) */
	int32_t beg_i, beg_j;   /* matrix indices after the last emitted column            */
	size_t aln_len;
} at_oracle_result;

/* pointer byte layout: bits0-2 pM, bit3-4 pL (0 none,1 LOW,2 MID), bit5-6 pU (0,1 MID,2 UPP)
 * and a second plane byte for pJ (0 none,1 MID,2 JUMP) when jump is enabled. */
#define PM(b) ((b) & 7)
#define PL(b) (((b) >> 3) & 3)
#define PU(b) (((b) >> 5) & 3)

static void reverse_bytes(char *s, size_t n)
{
	size_t i;
	for (i = 0; i < n / 2; i++) { char c = s[i]; s[i] = s[n - 1 - i]; s[n - 1 - i] = c; }
}

/* blacklist test of :659 -- isvalueinarray() returns the enum `true` (== 0) when the
 * value IS found, so `if (isvalueinarray(...))` takes the "may enter J" branch exactly
 * when j-1 is NOT listed (SURVEY.md A.3 / A.6 item 1). */
static uint8_t *build_site_mask(const int *sites, size_t n_sites, size_t l2, int whitelist)
{
	uint8_t *mask = (uint8_t *)calloc(l2 + 1, 1);
	size_t k;
	/* jump == 2: the semantics the reference's comments describe (:542-544, "we allow pointer move from M to J only
	 * at given positions on s2") but its inverted `bool` does not implement: entering J is barred everywhere
	 * EXCEPT on the listed target indices.  Equivalent to the blacklist mode run on the complement of the list. */
	if (whitelist) memset(mask, 1, l2 + 1);
	for (k = 0; k < n_sites; k++)
		if (sites[k] >= 0 && (size_t)sites[k] < l2) mask[sites[k]] = whitelist ? 0 : 1;
	return mask;
}

/* Affine three/four-state fill shared by global / local / fit (the recurrences at
 * :451-462, :635-667, :825-841 are textually the same apart from the 4th max5 argument
 * of M and the border initialisation). */
static int affine_align(int mode, const uint8_t *s1, size_t l1, const uint8_t *s2, size_t l2,
                        const int8_t *mat, int64_t o, int64_t e, int64_t jp, int jump,
                        const int *sites, size_t n_sites,
                        at_oracle_result *res, char *r1, char *r2, char *ops)
{
	size_t W = l2 + 1, i, j;
	uint8_t *P = (uint8_t *)calloc((l1 + 1) * W, 1);
	uint8_t *PJ = (mode == AT_FIT && jump) ? (uint8_t *)calloc((l1 + 1) * W, 1) : NULL;
	uint8_t *smask = (mode == AT_FIT && jump) ? build_site_mask(sites, n_sites, l2, jump == 2) : NULL;
	int64_t *buf = (int64_t *)malloc(sizeof(int64_t) * 8 * W);
	int64_t *Mp = buf, *Lp = buf + W, *Up = buf + 2 * W, *Jp = buf + 3 * W;
	int64_t *Mc = buf + 4 * W, *Lc = buf + 5 * W, *Uc = buf + 6 * W, *Jc = buf + 7 * W;
	int64_t best = NEG; int32_t bi = 0, bj = 0; int bstate = P_NONE;
	int64_t fitM_best = NEG, fitL_best = NEG;
	if (!P || !buf) { free(P); free(PJ); free(smask); free(buf); return -2; }

	/* row 0 */
	for (j = 0; j <= l2; j++) {
		switch (mode) {
		case AT_GLOBAL:   /* :428-441 */
			Mp[j] = j == 0 ? 0 : NEG; Lp[j] = j == 0 ? o : NEG; Up[j] = o + e * (int64_t)j; if (j == 0) Up[j] = o;
			Jp[j] = NEG; break;
		case AT_LOCAL:    /* no initialisation: calloc zeros (A.2) */
			Mp[j] = Lp[j] = Up[j] = 0; Jp[j] = NEG; break;
		default:          /* fit :612-624, row-0 loop runs after the column-0 loop */
			Mp[j] = 0; Up[j] = 0; Lp[j] = NEG; Jp[j] = NEG; break;
		}
	}
	for (i = 1; i <= l1; i++) {
		/* column 0 of row i */
		switch (mode) {
		case AT_GLOBAL: Lc[0] = o + e * (int64_t)i; Mc[0] = NEG; Uc[0] = NEG; Jc[0] = NEG; break;
		case AT_LOCAL:  Lc[0] = Mc[0] = Uc[0] = 0; Jc[0] = NEG; break;
		default:        Lc[0] = Mc[0] = Uc[0] = Jc[0] = NEG; break;
		}
		for (j = 1; j <= l2; j++) {
			int64_t s = mat[s1[i - 1] * 256 + s2[j - 1]], v;      /* the only change: s from the table */
			int idx; uint8_t b = 0;
			int64_t x4 = NEG;
			if (mode == AT_LOCAL) x4 = 0;
			else if (mode == AT_FIT && jump) x4 = addn(Jp[j - 1], s);
			idx = max5i(&v, addn(Lp[j - 1], s), addn(Mp[j - 1], s), addn(Up[j - 1], s), x4, NEG);
			Mc[j] = norm(v);
			if (idx == 0) b |= P_LOW; else if (idx == 1) b |= P_MID; else if (idx == 2) b |= P_UPP;
			else if (idx == 3) b |= (mode == AT_LOCAL) ? P_HOME : P_JUMP;
			if (mode == AT_LOCAL && Mc[j] > best) { best = Mc[j]; bi = (int32_t)i; bj = (int32_t)j; } /* :830-833 */
			idx = max5i(&v, addn(Lp[j], e), addn(Mp[j], o), NEG, NEG, NEG);
			Lc[j] = norm(v);
			if (idx == 0) b |= 1 << 3; else if (idx == 1) b |= 2 << 3;
			idx = max5i(&v, NEG, addn(Mc[j - 1], o), addn(Uc[j - 1], e), NEG, NEG);
			Uc[j] = norm(v);
			if (idx == 1) b |= 1 << 5; else if (idx == 2) b |= 2 << 5;
			P[i * W + j] = b;
			if (PJ) {
				if (!smask[j - 1]) {   /* j-1 not listed -> may enter J (:659-662) */
					idx = max5i(&v, NEG, addn(Mc[j - 1], jp), NEG, Jc[j - 1], NEG);
					Jc[j] = norm(v);
					PJ[i * W + j] = idx == 1 ? 1 : (idx == 3 ? 2 : 0);
				} else {               /* :664-665 */
					idx = max5i(&v, NEG, NEG, NEG, Jc[j - 1], NEG);
					Jc[j] = norm(v);
					PJ[i * W + j] = idx == 3 ? 2 : 0;
				}
			} else Jc[j] = NEG;
		}
		if (i == l1 && mode == AT_FIT) {   /* end search over the last row, column l2 excluded (:676-690) */
			for (j = 0; j < l2; j++) if (fitM_best < Mc[j]) { fitM_best = Mc[j]; best = Mc[j]; bj = (int32_t)j; bstate = P_MID; }
			fitL_best = best;
			for (j = 0; j < l2; j++) if (fitL_best < Lc[j]) { fitL_best = Lc[j]; best = Lc[j]; bj = (int32_t)j; bstate = P_LOW; }
			bi = (int32_t)l1;
		}
		if (i == l1 && mode == AT_GLOBAL) { /* :466-469 */
			int64_t v; int idx = max5i(&v, Lc[l2], Mc[l2], Uc[l2], NEG, NEG);
			best = v; bstate = idx == 0 ? P_LOW : idx == 1 ? P_MID : P_UPP; bi = (int32_t)l1; bj = (int32_t)l2;
		}
		{ int64_t *t; t = Mp; Mp = Mc; Mc = t; t = Lp; Lp = Lc; Lc = t; t = Up; Up = Uc; Uc = t; t = Jp; Jp = Jc; Jc = t; }
	}
	if (l1 == 0 && mode == AT_GLOBAL) {
		int64_t v; int idx = max5i(&v, Lp[l2], Mp[l2], Up[l2], NEG, NEG);
		best = v; bstate = idx == 0 ? P_LOW : idx == 1 ? P_MID : P_UPP; bi = 0; bj = (int32_t)l2;
	}
	if (mode == AT_LOCAL) bstate = P_MID;
	if (mode == AT_FIT && bstate == P_NONE) { free(P); free(PJ); free(smask); free(buf); return -3; } /* no finite end cell (A.3) */

	/* traceback: pointer is read at the cell BEFORE the move (:377-397, :562-587, :771-795) */
	{
		size_t cur = 0; int state = bstate; int32_t ti = bi, tj = bj;
		res->score = best; res->end_i = bi; res->end_j = bj;
		for (;;) {
			int go = (mode == AT_FIT) ? (ti > 0) : (ti > 0 && tj > 0);
			uint8_t b;
			if (!go) break;
			b = P[(size_t)ti * W + tj];
			if (state == P_LOW) {
				int p = PL(b); state = p == 1 ? P_LOW : p == 2 ? P_MID : P_NONE;
				r1[cur] = (char)s1[--ti]; r2[cur] = '-'; if (ops) ops[cur] = 'I'; cur++;
			} else if (state == P_MID) {
				state = PM(b);
				r1[cur] = (char)s1[--ti]; r2[cur] = (char)s2[--tj]; if (ops) ops[cur] = 'M'; cur++;
			} else if (state == P_UPP) {
				int p = PU(b); state = p == 1 ? P_MID : p == 2 ? P_UPP : P_NONE;
				r1[cur] = '-'; r2[cur] = (char)s2[--tj]; if (ops) ops[cur] = 'D'; cur++;
			} else if (state == P_JUMP && PJ) {
				int p = PJ[(size_t)ti * W + tj]; state = p == 1 ? P_MID : p == 2 ? P_JUMP : P_NONE;
				r1[cur] = '-'; r2[cur] = (char)s2[--tj]; if (ops) ops[cur] = 'N'; cur++;
			} else if (state == P_HOME && mode == AT_LOCAL) {
				break;   /* the reference sets i = j = 0 (:788-791); beg_i/beg_j report where the walk stopped */
			} else { /* unset pointer: the reference would spin forever; cannot happen on a finite path */
				free(P); free(PJ); free(smask); free(buf); return -4;
			}
		}
		res->beg_i = ti; res->beg_j = tj;
		if (mode == AT_GLOBAL) {   /* flush (:398-407) */
			while (tj > 0) { r1[cur] = '-'; r2[cur] = (char)s2[--tj]; if (ops) ops[cur] = 'D'; cur++; }
			while (ti > 0) { r2[cur] = '-'; r1[cur] = (char)s1[--ti]; if (ops) ops[cur] = 'I'; cur++; }
		}
		reverse_bytes(r1, cur); reverse_bytes(r2, cur); if (ops) { reverse_bytes(ops, cur); ops[cur] = 0; }
		r1[cur] = 0; r2[cur] = 0; res->aln_len = cur;
	}
	free(P); free(PJ); free(smask); free(buf);
	return 0;
}

/* align_overlap (:926-964) + trace_back_overlap (:896-922): one plane, linear gap `o`. */
static int overlap_align(const uint8_t *s1, size_t l1, const uint8_t *s2, size_t l2,
                         const int8_t *mat, int64_t o,
                         at_oracle_result *res, char *r1, char *r2, char *ops)
{
	size_t W = l2 + 1, i, j, cur = 0;
	uint8_t *P = (uint8_t *)calloc((l1 + 1) * W, 1);
	int64_t *prev = (int64_t *)malloc(sizeof(int64_t) * 2 * W), *cur_row = prev + W;
	int64_t best = NEG; int32_t bj = 0, ti, tj;
	if (!P || !prev) { free(P); free(prev); return -2; }
	for (j = 0; j <= l2; j++) prev[j] = NEG;     /* :937 */
	prev[0] = 0;                                 /* :938 */
	for (i = 1; i <= l1; i++) {
		cur_row[0] = 0;
		for (j = 1; j <= l2; j++) {
			int64_t s = mat[s1[i - 1] * 256 + s2[j - 1]], v;      /* the only change: s from the table */
			int idx = max5i(&v, addn(cur_row[j - 1], o), addn(prev[j - 1], s), addn(prev[j], o), NEG, NEG);
			cur_row[j] = norm(v);
			P[i * W + j] = idx == 0 ? P_LEFT : idx == 1 ? P_DIAG : idx == 2 ? P_RIGHT : 0;
		}
		{ int64_t *t = prev; prev = cur_row; cur_row = t; }
	}
	for (j = 0; j < l2; j++) if (best < prev[j]) { best = prev[j]; bj = (int32_t)j; }  /* :954-959 */
	if (l2 == 0) { free(P); free(prev < cur_row ? prev : cur_row); return -3; }
	res->score = best; res->end_i = (int32_t)l1; res->end_j = bj;
	ti = (int32_t)l1; tj = bj;
	while (tj > 0) {
		uint8_t p = P[(size_t)ti * W + tj];
		if (p == P_LEFT) { r2[cur] = (char)s2[--tj]; r1[cur] = '-'; if (ops) ops[cur] = 'D'; cur++; }
		else if (p == P_DIAG) { r1[cur] = (char)s1[--ti]; r2[cur] = (char)s2[--tj]; if (ops) ops[cur] = 'M'; cur++; }
		else if (p == P_RIGHT) { r1[cur] = (char)s1[--ti]; r2[cur] = '-'; if (ops) ops[cur] = 'I'; cur++; }
		else { free(P); free(prev < cur_row ? prev : cur_row); return -4; }
	}
	res->beg_i = ti; res->beg_j = tj;
	reverse_bytes(r1, cur); reverse_bytes(r2, cur); if (ops) { reverse_bytes(ops, cur); ops[cur] = 0; }
	r1[cur] = 0; r2[cur] = 0; res->aln_len = cur;
	free(P); free(prev < cur_row ? prev : cur_row);
	return 0;
}

/* One pair.  r1 / r2 / ops hold l1 + l2 + 1 bytes; coords: end_i, end_j, beg_i, beg_j.  0 or < 0 as at_oracle_align. */
int subst_port_align(int mode, const uint8_t *s1, size_t l1, const uint8_t *s2, size_t l2, const int8_t *mat,
                     int o, int e, int j, int jump, const int *sites, size_t n_sites,
                     int64_t *score, int32_t *coords, char *r1, char *r2, char *ops, size_t *aln_len)
{
	at_oracle_result res; int rc;
	memset(&res, 0, sizeof(res));
	if (mode == AT_FIT && l1 > l2) return -3;
	if (mode == AT_OVERLAP) rc = overlap_align(s1, l1, s2, l2, mat, o, &res, r1, r2, ops);
	else if (mode >= AT_GLOBAL && mode <= AT_FIT) rc = affine_align(mode, s1, l1, s2, l2, mat, o, e, j, jump, sites, n_sites, &res, r1, r2, ops);
	else return -1;
	if (rc) return rc;
	*score = res.score;
	coords[0] = res.end_i; coords[1] = res.end_j; coords[2] = res.beg_i; coords[3] = res.beg_j;
	*aln_len = res.aln_len;
	return 0;
}

/* ---- many pairs over threads; slot p of r1 / r2 / ops starts at aln_off[p] (>= q_len + t_len + 1 bytes) ---- */
typedef struct {
	int mode, o, e, j, jump; size_t lo_p, hi_p; const int8_t *mat;
	const uint8_t *q; const uint64_t *q_off; const uint32_t *q_len;
	const uint8_t *t; const uint64_t *t_off; const uint32_t *t_len;
	const int *sites; const uint64_t *site_off;
	int64_t *score; int32_t *coords; char *r1, *r2, *ops; const uint64_t *aln_off; uint32_t *aln_len;
	int rc;
} job_t;

static void *worker(void *arg)
{
	job_t *b = (job_t *)arg; size_t p;
	for (p = b->lo_p; p < b->hi_p; p++) {
		size_t al = 0;
		int rc = subst_port_align(b->mode, b->q + b->q_off[p], b->q_len[p], b->t + b->t_off[p], b->t_len[p], b->mat, b->o, b->e, b->j,
		                          b->jump, b->sites ? b->sites + b->site_off[p] : NULL, b->sites ? (size_t)(b->site_off[p + 1] - b->site_off[p]) : 0,
		                          &b->score[p], b->coords + 4 * p, b->r1 + b->aln_off[p], b->r2 + b->aln_off[p], b->ops + b->aln_off[p], &al);
		b->aln_len[p] = (uint32_t)al;
		if (rc) b->rc = rc;
	}
	return NULL;
}

int subst_port_batch(int mode, const int8_t *mat, int o, int e, int j, int jump, size_t n,
                     const uint8_t *q, const uint64_t *q_off, const uint32_t *q_len, const uint8_t *t, const uint64_t *t_off,
                     const uint32_t *t_len, const int *sites, const uint64_t *site_off, int64_t *score, int32_t *coords,
                     char *r1, char *r2, char *ops, const uint64_t *aln_off, uint32_t *aln_len, int n_threads)
{
	pthread_t th[64]; job_t jobs[64]; int k, rc = 0;
	if (n_threads < 1) n_threads = 1;
	if (n_threads > 64) n_threads = 64;
	for (k = 0; k < n_threads; k++) {
		job_t *b = &jobs[k];
		b->mode = mode; b->o = o; b->e = e; b->j = j; b->jump = jump; b->mat = mat;
		b->lo_p = n * (size_t)k / n_threads; b->hi_p = n * (size_t)(k + 1) / n_threads;
		b->q = q; b->q_off = q_off; b->q_len = q_len; b->t = t; b->t_off = t_off; b->t_len = t_len;
		b->sites = sites; b->site_off = site_off; b->score = score; b->coords = coords;
		b->r1 = r1; b->r2 = r2; b->ops = ops; b->aln_off = aln_off; b->aln_len = aln_len; b->rc = 0;
		if (n_threads == 1) worker(b); else pthread_create(&th[k], NULL, worker, b);
	}
	for (k = 0; k < n_threads; k++) { if (n_threads > 1) pthread_join(th[k], NULL); if (jobs[k].rc) rc = jobs[k].rc; }
	return rc;
}
