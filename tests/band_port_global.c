/* Banded global alignment, CPU restatement for the tests (tests/band_port_global.py): align_gla (src/alignment.h:428-469)
 * and trace_back_gla (:372-412) as oracle/at_oracle.c's affine_align runs them for AT_GLOBAL, plus the band of
 * include/aligntools_b200.h (at_band): a cell (i, j >= 1) whose diagonal j - i lies outside [lo, hi] is -inf in M, L and
 * U and its pointer is never set.  Nothing else changes: row 0 and column 0 keep their border values, max5's
 * first-strictly-greater ties, the end cell (l1, l2) with max5's end state, the traceback and the flush of the rest of
 * the target, then the rest of the read.  banded == 0 is the unbanded recurrence. */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NEG (INT64_MIN / 4)

static inline int64_t addn(int64_t v, int64_t d) { return v == NEG ? NEG : v + d; }

static void reverse_bytes(char *s, size_t n)
{
	size_t i;
	for (i = 0; i < n / 2; i++) { char c = s[i]; s[i] = s[n - 1 - i]; s[n - 1 - i] = c; }
}

enum { G_NONE = 0, G_LOW = 1, G_MID = 2, G_UPP = 3 };
#define PM(b) ((b) & 7)
#define PL(b) (((b) >> 3) & 3)
#define PU(b) (((b) >> 5) & 3)

static inline int64_t norm(int64_t v) { return v < NEG / 2 ? NEG : v; }

/* max5 (:90-100) over three arguments: first strictly greater, from -inf; -1 when all are -inf */
static inline int max3i(int64_t *res, int64_t a1, int64_t a2, int64_t a3)
{
	int st = -1; *res = NEG;
	if (a1 > *res) { *res = a1; st = 0; }
	if (a2 > *res) { *res = a2; st = 1; }
	if (a3 > *res) { *res = a3; st = 2; }
	return st;
}

/* coords: end_i, end_j, beg_i, beg_j.  r1 / r2 / ops hold l1 + l2 + 1 bytes.  0 or <0 (-2 memory, -4 unset pointer) */
int band_port_global(const uint8_t *s1, size_t l1, const uint8_t *s2, size_t l2, int m, int u, int o, int e,
                     int banded, int64_t lo, int64_t hi, int64_t *score, int32_t *coords, char *r1, char *r2, char *ops,
                     size_t *aln_len)
{
	size_t W = l2 + 1, i, j, cur = 0;
	uint8_t *P = (uint8_t *)calloc((l1 + 1) * W, 1);
	int64_t *buf = (int64_t *)malloc(sizeof(int64_t) * 6 * W);
	int64_t *Mp = buf, *Lp = buf + W, *Up = buf + 2 * W, *Mc = buf + 3 * W, *Lc = buf + 4 * W, *Uc = buf + 5 * W;
	int64_t best = NEG; int state = G_NONE; int32_t ti, tj;
	if (!P || !buf) { free(P); free(buf); return -2; }
	for (j = 0; j <= l2; j++) {                  /* row 0 (:428-441) */
		Mp[j] = j == 0 ? 0 : NEG; Lp[j] = j == 0 ? o : NEG; Up[j] = j == 0 ? o : o + e * (int64_t)j;
	}
	for (i = 1; i <= l1; i++) {
		Lc[0] = o + e * (int64_t)i; Mc[0] = NEG; Uc[0] = NEG;      /* column 0 */
		for (j = 1; j <= l2; j++) {
			const int64_t d = (int64_t)j - (int64_t)i;
			int64_t s, v;
			int idx; uint8_t b = 0;
			if (banded && (d < lo || d > hi)) { Mc[j] = Lc[j] = Uc[j] = NEG; continue; }
			s = (s1[i - 1] == s2[j - 1]) ? m : u;
			idx = max3i(&v, addn(Lp[j - 1], s), addn(Mp[j - 1], s), addn(Up[j - 1], s));      /* :451-462 */
			Mc[j] = norm(v);
			if (idx == 0) b |= G_LOW; else if (idx == 1) b |= G_MID; else if (idx == 2) b |= G_UPP;
			idx = max3i(&v, addn(Lp[j], e), addn(Mp[j], o), NEG);
			Lc[j] = norm(v);
			if (idx == 0) b |= 1 << 3; else if (idx == 1) b |= 2 << 3;
			idx = max3i(&v, NEG, addn(Mc[j - 1], o), addn(Uc[j - 1], e));
			Uc[j] = norm(v);
			if (idx == 1) b |= 1 << 5; else if (idx == 2) b |= 2 << 5;
			P[i * W + j] = b;
		}
		if (i == l1) {                           /* end cell (:466-469) */
			int idx = max3i(&best, Lc[l2], Mc[l2], Uc[l2]);
			state = idx == 0 ? G_LOW : idx == 1 ? G_MID : G_UPP;
		}
		{ int64_t *t; t = Mp; Mp = Mc; Mc = t; t = Lp; Lp = Lc; Lc = t; t = Up; Up = Uc; Uc = t; }
	}
	*score = best; coords[0] = (int32_t)l1; coords[1] = (int32_t)l2;
	ti = (int32_t)l1; tj = (int32_t)l2;
	while (ti > 0 && tj > 0) {                   /* :377-397: the pointer is read at the cell before the move */
		uint8_t b = P[(size_t)ti * W + tj];
		if (state == G_LOW) {
			int p = PL(b); state = p == 1 ? G_LOW : p == 2 ? G_MID : G_NONE;
			r1[cur] = (char)s1[--ti]; r2[cur] = '-'; ops[cur] = 'I'; cur++;
		} else if (state == G_MID) {
			state = PM(b);
			r1[cur] = (char)s1[--ti]; r2[cur] = (char)s2[--tj]; ops[cur] = 'M'; cur++;
		} else if (state == G_UPP) {
			int p = PU(b); state = p == 1 ? G_MID : p == 2 ? G_UPP : G_NONE;
			r1[cur] = '-'; r2[cur] = (char)s2[--tj]; ops[cur] = 'D'; cur++;
		} else { free(P); free(buf); return -4; }
	}
	coords[2] = ti; coords[3] = tj;
	while (tj > 0) { r1[cur] = '-'; r2[cur] = (char)s2[--tj]; ops[cur] = 'D'; cur++; }      /* flush (:398-407) */
	while (ti > 0) { r2[cur] = '-'; r1[cur] = (char)s1[--ti]; ops[cur] = 'I'; cur++; }
	reverse_bytes(r1, cur); reverse_bytes(r2, cur); reverse_bytes(ops, cur);
	*aln_len = cur;
	free(P); free(buf);
	return 0;
}

/* ---- many pairs over threads; slot p of r1 / r2 / ops starts at aln_off[p] (>= q_len + t_len + 1 bytes) ---- */
typedef struct {
	int m, u, o, e, banded; size_t lo_p, hi_p;
	const uint8_t *q; const uint64_t *q_off; const uint32_t *q_len;
	const uint8_t *t; const uint64_t *t_off; const uint32_t *t_len;
	const int32_t *band_lo, *band_hi;
	int64_t *score; int32_t *coords; char *r1, *r2, *ops; const uint64_t *aln_off; uint32_t *aln_len;
	int rc;
} job_t;

static void *worker(void *arg)
{
	job_t *b = (job_t *)arg; size_t p;
	for (p = b->lo_p; p < b->hi_p; p++) {
		size_t al = 0;
		int rc = band_port_global(b->q + b->q_off[p], b->q_len[p], b->t + b->t_off[p], b->t_len[p], b->m, b->u, b->o, b->e, b->banded,
		                          b->banded ? b->band_lo[p] : 0, b->banded ? b->band_hi[p] : 0, &b->score[p], b->coords + 4 * p,
		                          b->r1 + b->aln_off[p], b->r2 + b->aln_off[p], b->ops + b->aln_off[p], &al);
		b->aln_len[p] = (uint32_t)al;
		if (rc) b->rc = rc;
	}
	return NULL;
}

int band_port_global_batch(int m, int u, int o, int e, size_t n, const uint8_t *q, const uint64_t *q_off, const uint32_t *q_len,
                           const uint8_t *t, const uint64_t *t_off, const uint32_t *t_len, const int32_t *band_lo, const int32_t *band_hi,
                           int64_t *score, int32_t *coords, char *r1, char *r2, char *ops, const uint64_t *aln_off, uint32_t *aln_len,
                           int n_threads)
{
	pthread_t th[64]; job_t jobs[64]; int k, rc = 0;
	if (n_threads < 1) n_threads = 1;
	if (n_threads > 64) n_threads = 64;
	for (k = 0; k < n_threads; k++) {
		job_t *b = &jobs[k];
		b->m = m; b->u = u; b->o = o; b->e = e; b->banded = band_lo != NULL;
		b->lo_p = n * (size_t)k / n_threads; b->hi_p = n * (size_t)(k + 1) / n_threads;
		b->q = q; b->q_off = q_off; b->q_len = q_len; b->t = t; b->t_off = t_off; b->t_len = t_len;
		b->band_lo = band_lo; b->band_hi = band_hi; b->score = score; b->coords = coords;
		b->r1 = r1; b->r2 = r2; b->ops = ops; b->aln_off = aln_off; b->aln_len = aln_len; b->rc = 0;
		if (n_threads == 1) worker(b); else pthread_create(&th[k], NULL, worker, b);
	}
	for (k = 0; k < n_threads; k++) { if (n_threads > 1) pthread_join(th[k], NULL); if (jobs[k].rc) rc = jobs[k].rc; }
	return rc;
}
