/* Edit distance with a path, CPU restatement for the tests (tests/edit_port.py): edit_dist (src/alignment.h:291-315)
 * as oracle/at_oracle.c writes it, plus the traceback include/aligntools_b200.h defines for AT_OUT_EDIT_PATH:
 *   - M[i][0] = i, M[0][j] = j, M[i][j] = min3(M[i][j-1] + 1, M[i-1][j-1] + (eq ? 0 : u), M[i-1][j] + 1);
 *   - the pointer of a cell is min3's first strictly smaller argument: LEFT, then DIAG, then UP on ties;
 *   - the walk starts at (l1, l2) and runs while i > 0 && j > 0 (LEFT: D, DIAG: M, UP: I), then flushes the rest of the
 *     target (D) and the rest of the read (I), as trace_back_gla does.
 * coords: end_i, end_j, beg_i, beg_j (beg = where the walk stopped, before the flush).  Pointers: 2 bits per cell. */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { P_LEFT = 0, P_DIAG = 1, P_UP = 2 };

static void reverse_bytes(char *s, size_t n)
{
	size_t i;
	for (i = 0; i < n / 2; i++) { char c = s[i]; s[i] = s[n - 1 - i]; s[n - 1 - i] = c; }
}

/* r1 / r2 / ops hold l1 + l2 + 1 bytes (NULL: score only).  0, or -2 when out of memory */
int edit_port_align(const uint8_t *s1, size_t l1, const uint8_t *s2, size_t l2, int u, int64_t *score, int32_t *coords,
                    char *r1, char *r2, char *ops, size_t *aln_len)
{
	const int path = ops != NULL;
	const size_t W = l2 + 1;
	uint8_t *P = path ? (uint8_t *)calloc(((l1 + 1) * W + 3) / 4, 1) : NULL;
	int64_t *buf = (int64_t *)malloc(sizeof(int64_t) * 2 * W), *prev = buf, *row = buf + W;
	size_t i, j, cur = 0, ti, tj;
	if (!buf || (path && !P)) { free(P); free(buf); return -2; }
	for (j = 0; j <= l2; j++) prev[j] = (int64_t)j;            /* :302 */
	for (i = 1; i <= l1; i++) {
		row[0] = (int64_t)i;                                   /* :301 */
		for (j = 1; j <= l2; j++) {
			const int64_t c0 = row[j - 1] + 1, c1 = prev[j - 1] + (s1[i - 1] == s2[j - 1] ? 0 : u), c2 = prev[j] + 1;
			int64_t v = c0; int k = P_LEFT;
			if (c1 < v) { v = c1; k = P_DIAG; }
			if (c2 < v) { v = c2; k = P_UP; }
			row[j] = v;
			if (path) { const size_t x = i * W + j; P[x >> 2] |= (uint8_t)(k << (2 * (x & 3))); }
		}
		{ int64_t *t = prev; prev = row; row = t; }
	}
	*score = prev[l2];
	coords[0] = (int32_t)l1; coords[1] = (int32_t)l2; coords[2] = (int32_t)l1; coords[3] = (int32_t)l2;
	if (!path) { free(buf); return 0; }
	ti = l1; tj = l2;
	while (ti > 0 && tj > 0) {
		const size_t x = ti * W + tj;
		const int k = (P[x >> 2] >> (2 * (x & 3))) & 3;
		if (k == P_LEFT) { r1[cur] = '-'; r2[cur] = (char)s2[--tj]; ops[cur] = 'D'; }
		else if (k == P_DIAG) { r1[cur] = (char)s1[--ti]; r2[cur] = (char)s2[--tj]; ops[cur] = 'M'; }
		else { r1[cur] = (char)s1[--ti]; r2[cur] = '-'; ops[cur] = 'I'; }
		cur++;
	}
	coords[2] = (int32_t)ti; coords[3] = (int32_t)tj;
	while (tj > 0) { r1[cur] = '-'; r2[cur] = (char)s2[--tj]; ops[cur] = 'D'; cur++; }
	while (ti > 0) { r1[cur] = (char)s1[--ti]; r2[cur] = '-'; ops[cur] = 'I'; cur++; }
	reverse_bytes(r1, cur); reverse_bytes(r2, cur); reverse_bytes(ops, cur);
	*aln_len = cur;
	free(P); free(buf);
	return 0;
}

/* ---- many pairs over threads; slot p of r1 / r2 / ops starts at aln_off[p] (>= q_len + t_len + 1 bytes) ---- */
typedef struct {
	int u; size_t lo_p, hi_p;
	const uint8_t *q; const uint64_t *q_off; const uint32_t *q_len;
	const uint8_t *t; const uint64_t *t_off; const uint32_t *t_len;
	int64_t *score; int32_t *coords; char *r1, *r2, *ops; const uint64_t *aln_off; uint32_t *aln_len;
	int rc;
} job_t;

static void *worker(void *arg)
{
	job_t *b = (job_t *)arg; size_t p;
	for (p = b->lo_p; p < b->hi_p; p++) {
		size_t al = 0;
		int rc = edit_port_align(b->q + b->q_off[p], b->q_len[p], b->t + b->t_off[p], b->t_len[p], b->u, &b->score[p], b->coords + 4 * p,
		                         b->r1 + b->aln_off[p], b->r2 + b->aln_off[p], b->ops + b->aln_off[p], &al);
		b->aln_len[p] = (uint32_t)al;
		if (rc) b->rc = rc;
	}
	return NULL;
}

int edit_port_batch(int u, size_t n, const uint8_t *q, const uint64_t *q_off, const uint32_t *q_len,
                    const uint8_t *t, const uint64_t *t_off, const uint32_t *t_len,
                    int64_t *score, int32_t *coords, char *r1, char *r2, char *ops, const uint64_t *aln_off, uint32_t *aln_len,
                    int n_threads)
{
	pthread_t th[64]; job_t jobs[64]; int k, rc = 0;
	if (n_threads < 1) n_threads = 1;
	if (n_threads > 64) n_threads = 64;
	for (k = 0; k < n_threads; k++) {
		job_t *b = &jobs[k];
		b->u = u;
		b->lo_p = n * (size_t)k / n_threads; b->hi_p = n * (size_t)(k + 1) / n_threads;
		b->q = q; b->q_off = q_off; b->q_len = q_len; b->t = t; b->t_off = t_off; b->t_len = t_len;
		b->score = score; b->coords = coords;
		b->r1 = r1; b->r2 = r2; b->ops = ops; b->aln_off = aln_off; b->aln_len = aln_len; b->rc = 0;
		if (n_threads == 1) worker(b); else pthread_create(&th[k], NULL, worker, b);
	}
	for (k = 0; k < n_threads; k++) { if (n_threads > 1) pthread_join(th[k], NULL); if (jobs[k].rc) rc = jobs[k].rc; }
	return rc;
}
