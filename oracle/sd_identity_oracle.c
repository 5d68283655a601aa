/* sd_identity_oracle.c -- CPU oracle for the identity rescoring row (SURVEY §8 f1).
 *
 * TEST INFRASTRUCTURE ONLY: used by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg as the
 * checker.  The product (stringdecomposer_b200) never links, imports or executes this file.
 *
 * What it restates: main.py:29-60 (`edist` / `aai`): edlib.align(interval, monomer, mode="NW", task="path"),
 * identity = (sum of '=' run lengths) / (sum of all CIGAR run lengths) * 100.  edlib is third-party code the
 * reference vendors as src/edlib.cpp (the Python wheel `edlib` wraps the same library); its NW path is
 *   - the unit-cost global edit-distance matrix D over (query rows, target columns) with D[-1][j] = j+1,
 *     D[i][-1] = i+1 (edlib.cpp:994-998 boundary scores),
 *   - walked back from the bottom-right cell, testing at every cell, in this order (edlib.cpp:1036-1133):
 *       up    (query char alone,  EDLIB_EDOP_INSERT)  if D[i-1][j] + 1 == D[i][j]
 *       left  (target char alone, EDLIB_EDOP_DELETE)  if D[i][j-1] + 1 == D[i][j]
 *       diagonal, a match ('=') if D[i-1][j-1] == D[i][j], else a mismatch ('X').
 *     The band edlib computes (k = the optimal distance) contains every cell of every optimal path with its
 *     exact value, and a neighbour outside it can never satisfy the equalities, so the walk is a function of
 *     the full matrix.  Above 1 MiB of traceback state edlib switches to Hirschberg splitting
 *     (edlib.cpp:1189-1191), which may choose another optimal path: sdo_nw_uses_traceback() says which side
 *     a pair is on; the pinning below only covers the traceback side.
 * sdo_nw_prefix_counts gives the triple of every prefix pair from one matrix (for the cell-by-cell tests of the
 * kernel, tests/test_identity_tables.py) and sdo_nw_path_counts_batch runs the walk over a pair list in parallel.
 * Parity: PINNED -- against the reference's own edlib.cpp compiled into oracle/_ref/libedlib_ref.so
 * (tests/test_identity_oracle.py, random and adversarial pairs) and, through oracle/sd_convert_oracle.py,
 * against all 12 columns of the reference's golden file test_data/final_decomposition_fc89af8.tsv. */
#include <stdlib.h>
#include <string.h>
#include "sd_oracle.h"

int sdo_nw_uses_traceback(int qlen, int tlen)
{
    long long blocks = (qlen + 63) / 64;                                            /* edlib.cpp:1176 */
    long long bytes = (2ll * 8 + 4) * blocks * tlen + 2ll * 4 * tlen;               /* edlib.cpp:1187-1188 */
    return bytes < 1024 * 1024;
}

/* The unit-cost NW matrix with its boundary: a (qlen+1) x (tlen+1) table, D[i][j] at [(i+1)*(tlen+1) + j+1]. */
static int *nw_matrix(const char *q, int qlen, const char *t, int tlen)
{
    size_t W = (size_t)tlen + 1;
    int *D = (int *)malloc(sizeof(int) * (size_t)(qlen + 1) * W);
    if (!D) return NULL;
#define AT(i, j) D[(size_t)((i) + 1) * W + (size_t)((j) + 1)]
    for (int j = -1; j < tlen; ++j) AT(-1, j) = j + 1;
    for (int i = 0; i < qlen; ++i) {
        AT(i, -1) = i + 1;
        for (int j = 0; j < tlen; ++j) {
            int d = AT(i - 1, j - 1) + (q[i] != t[j]);
            int u = AT(i - 1, j) + 1, l = AT(i, j - 1) + 1;
            if (u < d) d = u;
            if (l < d) d = l;
            AT(i, j) = d;
        }
    }
    return D;
}

/* Returns the edit distance; *matches = number of '=' columns, *columns = alignment length.
 * Either sequence empty: main.py:30-33 returns (-1, "") -> identity 0; reported here as -1. */
int sdo_nw_path_counts(const char *q, int qlen, const char *t, int tlen, int *matches, int *columns)
{
    *matches = 0; *columns = 0;
    if (qlen <= 0 || tlen <= 0) return -1;
    size_t W = (size_t)tlen + 1;
    int *D = nw_matrix(q, qlen, t, tlen);
    if (!D) return -2;
    int i = qlen - 1, j = tlen - 1, m = 0, c = 0;
    while (i >= 0 || j >= 0) {
        int cur = AT(i, j);
        if (i >= 0 && AT(i - 1, j) + 1 == cur) --i;                 /* up first    (edlib.cpp:1038) */
        else if (j >= 0 && AT(i, j - 1) + 1 == cur) --j;            /* then left   (edlib.cpp:1068) */
        else { if (AT(i - 1, j - 1) == cur) ++m; --i; --j; }        /* else diagonal (edlib.cpp:1098-1099) */
        ++c;
    }
    int dist = AT(qlen - 1, tlen - 1);
    free(D);
    *matches = m; *columns = c;
    return dist;
}

/* The triple of every prefix pair (q[:i+1], t[:j+1]) at once, into qlen x tlen row-major arrays.  With edlib's
 * boundary the matrix of a prefix pair is the top-left block of the full one, and the walk above is memoryless, so
 * the triple of (i, j) is that of the walk started at (i, j): one step of the walk (the same tests in the same order)
 * from the already-known triple of the cell it moves to.  A boundary cell (i, -1) or (-1, j) walks straight to the
 * corner: no '=' column, i + 1 or j + 1 columns.  Returns 0, -1 when either sequence is empty, -2 without memory. */
int sdo_nw_prefix_counts(const char *q, int qlen, const char *t, int tlen, int32_t *dist, int32_t *matches, int32_t *columns)
{
    if (qlen <= 0 || tlen <= 0) return -1;
    size_t W = (size_t)tlen + 1, T = (size_t)tlen;
    int *D = nw_matrix(q, qlen, t, tlen);
    if (!D) return -2;
#define CELL(i, j) ((size_t)(i) * T + (size_t)(j))
    for (int i = 0; i < qlen; ++i)
        for (int j = 0; j < tlen; ++j) {
            int cur = AT(i, j), pi, pj, eq = 0;
            if (AT(i - 1, j) + 1 == cur) { pi = i - 1; pj = j; }
            else if (AT(i, j - 1) + 1 == cur) { pi = i; pj = j - 1; }
            else { eq = AT(i - 1, j - 1) == cur; pi = i - 1; pj = j - 1; }
            int pm = 0, pc = pi + pj + 2;                               /* boundary: i + 1 or j + 1 columns */
            if (pi >= 0 && pj >= 0) { pm = matches[CELL(pi, pj)]; pc = columns[CELL(pi, pj)]; }
            dist[CELL(i, j)] = cur; matches[CELL(i, j)] = pm + eq; columns[CELL(i, j)] = pc + 1;
        }
#undef CELL
#undef AT
    free(D);
    return 0;
}

/* sdo_nw_path_counts over a pair list of packed sequences (offsets as sd_identity takes them), in parallel.
 * Returns 0, or -2 when a pair's matrix could not be allocated. */
int sdo_nw_path_counts_batch(const char *qtext, const int64_t *qoff, const char *ttext, const int64_t *toff,
                             const int32_t *pair_q, const int32_t *pair_t, int64_t npairs,
                             int32_t *dist, int32_t *matches, int32_t *columns)
{
    int status = 0;
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t p = 0; p < npairs; ++p) {
        const int64_t qi = pair_q[p], ti = pair_t[p];
        int m, c;
        int d = sdo_nw_path_counts(qtext + qoff[qi], (int)(qoff[qi + 1] - qoff[qi]), ttext + toff[ti],
                                   (int)(toff[ti + 1] - toff[ti]), &m, &c);
        if (d == -2) {
#pragma omp atomic write
            status = -2;
        }
        dist[p] = d; matches[p] = m; columns[p] = c;
    }
    return status;
}
