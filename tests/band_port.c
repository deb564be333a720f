/* Banded overlap alignment, CPU restatement for the tests (tests/band_port.py): align_overlap (src/alignment.h:926-964)
 * and trace_back_overlap (:896-922) written as oracle/at_oracle.c writes them, plus the band of
 * include/aligntools_b200.h (at_band): a cell (i, j >= 1) whose diagonal j - i lies outside [lo, hi] is -inf and its
 * pointer is never set.  Nothing else changes: row 0 is -inf, M[i][0] = 0, first-strictly-greater ties in the order
 * LEFT, DIAGONAL, RIGHT, the end search over the last row's columns 0 .. l2-1, the traceback.
 * banded == 0 is the unbanded recurrence. */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NEG (INT64_MIN / 4)
enum { P_LEFT = 1, P_DIAG = 2, P_RIGHT = 3 };

static inline int64_t addn(int64_t v, int64_t d) { return v == NEG ? NEG : v + d; }

static void reverse_bytes(char *s, size_t n)
{
	size_t i;
	for (i = 0; i < n / 2; i++) { char c = s[i]; s[i] = s[n - 1 - i]; s[n - 1 - i] = c; }
}

/* coords: end_i, end_j, beg_i, beg_j.  r1 / r2 / ops hold l1 + l2 + 1 bytes.  0 or <0 (-2 memory, -4 unset pointer) */
int band_port_align(const uint8_t *s1, size_t l1, const uint8_t *s2, size_t l2, int m, int u, int o,
                    int banded, int64_t lo, int64_t hi, int64_t *score, int32_t *coords, char *r1, char *r2, char *ops,
                    size_t *aln_len)
{
	size_t W = l2 + 1, i, j, cur = 0;
	uint8_t *P = (uint8_t *)calloc((l1 + 1) * W, 1);
	int64_t *buf = (int64_t *)malloc(sizeof(int64_t) * 2 * W), *prev = buf, *row = buf + W;
	int64_t best = NEG; int32_t bj = 0, ti, tj;
	if (!P || !buf) { free(P); free(buf); return -2; }
	for (j = 0; j <= l2; j++) prev[j] = NEG;     /* :937 */
	prev[0] = 0;                                 /* :938 */
	for (i = 1; i <= l1; i++) {
		row[0] = 0;
		for (j = 1; j <= l2; j++) {
			const int64_t d = (int64_t)j - (int64_t)i;
			int64_t v, s, c[3];
			int k, idx = -1;
			if (banded && (d < lo || d > hi)) { row[j] = NEG; continue; }
			s = (s1[i - 1] == s2[j - 1]) ? m : u;
			c[0] = addn(row[j - 1], o); c[1] = addn(prev[j - 1], s); c[2] = addn(prev[j], o);
			v = NEG;
			for (k = 0; k < 3; k++) if (c[k] > v) { v = c[k]; idx = k; }      /* max5: first strictly greater */
			row[j] = v < NEG / 2 ? NEG : v;
			P[i * W + j] = idx == 0 ? P_LEFT : idx == 1 ? P_DIAG : idx == 2 ? P_RIGHT : 0;
		}
		{ int64_t *t = prev; prev = row; row = t; }
	}
	for (j = 0; j < l2; j++) if (best < prev[j]) { best = prev[j]; bj = (int32_t)j; }   /* :954-959 */
	*score = best; coords[0] = (int32_t)l1; coords[1] = bj;
	ti = (int32_t)l1; tj = bj;
	while (tj > 0) {
		uint8_t p = P[(size_t)ti * W + tj];
		if (p == P_LEFT) { r2[cur] = (char)s2[--tj]; r1[cur] = '-'; ops[cur] = 'D'; cur++; }
		else if (p == P_DIAG) { r1[cur] = (char)s1[--ti]; r2[cur] = (char)s2[--tj]; ops[cur] = 'M'; cur++; }
		else if (p == P_RIGHT) { r1[cur] = (char)s1[--ti]; r2[cur] = '-'; ops[cur] = 'I'; cur++; }
		else { free(P); free(buf); return -4; }
	}
	coords[2] = ti; coords[3] = tj;
	reverse_bytes(r1, cur); reverse_bytes(r2, cur); reverse_bytes(ops, cur);
	*aln_len = cur;
	free(P); free(buf);
	return 0;
}

/* ---- many pairs over threads; slot p of r1 / r2 / ops starts at aln_off[p] (>= q_len + t_len + 1 bytes) ---- */
typedef struct {
	int m, u, o, banded; size_t lo_p, hi_p;
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
		int rc = band_port_align(b->q + b->q_off[p], b->q_len[p], b->t + b->t_off[p], b->t_len[p], b->m, b->u, b->o, b->banded,
		                         b->banded ? b->band_lo[p] : 0, b->banded ? b->band_hi[p] : 0, &b->score[p], b->coords + 4 * p,
		                         b->r1 + b->aln_off[p], b->r2 + b->aln_off[p], b->ops + b->aln_off[p], &al);
		b->aln_len[p] = (uint32_t)al;
		if (rc) b->rc = rc;
	}
	return NULL;
}

int band_port_batch(int m, int u, int o, size_t n, const uint8_t *q, const uint64_t *q_off, const uint32_t *q_len,
                    const uint8_t *t, const uint64_t *t_off, const uint32_t *t_len, const int32_t *band_lo, const int32_t *band_hi,
                    int64_t *score, int32_t *coords, char *r1, char *r2, char *ops, const uint64_t *aln_off, uint32_t *aln_len,
                    int n_threads)
{
	pthread_t th[64]; job_t jobs[64]; int k, rc = 0;
	if (n_threads < 1) n_threads = 1;
	if (n_threads > 64) n_threads = 64;
	for (k = 0; k < n_threads; k++) {
		job_t *b = &jobs[k];
		b->m = m; b->u = u; b->o = o; b->banded = band_lo != NULL;
		b->lo_p = n * (size_t)k / n_threads; b->hi_p = n * (size_t)(k + 1) / n_threads;
		b->q = q; b->q_off = q_off; b->q_len = q_len; b->t = t; b->t_off = t_off; b->t_len = t_len;
		b->band_lo = band_lo; b->band_hi = band_hi; b->score = score; b->coords = coords;
		b->r1 = r1; b->r2 = r2; b->ops = ops; b->aln_off = aln_off; b->aln_len = aln_len; b->rc = 0;
		if (n_threads == 1) worker(b); else pthread_create(&th[k], NULL, worker, b);
	}
	for (k = 0; k < n_threads; k++) { if (n_threads > 1) pthread_join(th[k], NULL); if (jobs[k].rc) rc = jobs[k].rc; }
	return rc;
}
