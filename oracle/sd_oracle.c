/*
 * sd_oracle.c -- CPU restatement of the StringDecomposer string-decomposition DP.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is on the product path: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may build,
 * load or run it, and there only as the checker / the timed CPU arm.  The product
 * (stringdecomposer_b200/csrc) never links or calls this file.
 *
 * Parity status: PINNED.  tests/test_oracle.py checks this restatement against
 *   (1) the reference's only golden vector, test_data/final_decomposition_fc89af8.tsv cols 1-4
 *       (committed as tests/golden/config1_cols1-4.tsv), and
 *   (2) the unmodified reference binary compiled from /root/reference by oracle/Makefile
 *       into oracle/_ref/dp (full raw TSV incl. score/gap/length columns, many edge cases;
 *       outputs committed as fixtures under tests/golden/ by tests/golden/make_golden.py).
 *
 * The --ed_thr pre-filter (main.cpp:128-149) is restated too; its edit distance comes from edlib (vendored by the
 * reference as src/edlib.cpp) and is restated from edlib's published definition of the HW mode as the textbook
 * infix DP; it is pinned by the reference runs with argc == 11 in tests/golden/edge_cases.json.
 *
 * Every function cites the reference lines it restates (paths relative to
 * /root/reference/stringdecomposer/src/main.cpp).  This is a restatement in plain C with flat
 * arrays, not a copy: the reference is C++ with nested std::vector and std::string.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "sd_oracle.h"

#define SDO_NEG_INF (-1000000) /* main.cpp:156 "INF" */

#define CELL(i, r, k) tab[(int64_t)(i) * width + row_off[r] + (k)]
#define ROWLEN(r) (row_off[(r) + 1] - row_off[r])

/* ---------------------------------------------------------------------------------------
 * The forward DP of one segment against all DP rows: allocation main.cpp:158-169, row 0 :171-182, sweep :183-208.
 * rows: concatenated row strings (forward monomers then reverse complements), row r occupies
 * rows[row_off[r] .. row_off[r+1]).  Returns the flat table (cell (i, r, k) at i*row_off[R] + row_off[r] + k) and
 * sets *jump_out to jump[i] = dp[i][monomers_num][0]; both malloc'd.  NULL if an allocation failed.
 * ------------------------------------------------------------------------------------- */
static int64_t *fill_table(const char *seg, int n, const char *rows, const int *row_off, int R,
                           int ins, int del, int mismatch, int match, int64_t **jump_out)
{
    const int64_t width = row_off[R];           /* total cells of one column */
    int64_t *tab = (int64_t *)malloc(sizeof(int64_t) * (size_t)n * (size_t)width);
    int64_t *jump = (int64_t *)malloc(sizeof(int64_t) * (size_t)n);
    if (!tab || !jump) { free(tab); free(jump); return NULL; }
    for (int64_t x = 0; x < (int64_t)n * width; ++x) tab[x] = SDO_NEG_INF;       /* :160-166 */
    for (int i = 0; i < n; ++i) jump[i] = SDO_NEG_INF;                            /* :167-168 */

    /* row 0, main.cpp:171-182 (note del*(k-1), not del*k) */
    for (int r = 0; r < R; ++r) {
        const char *m = rows + row_off[r];
        const int L = ROWLEN(r);
        CELL(0, r, 0) = (m[0] == seg[0]) ? match : mismatch;
        for (int k = 1; k < L; ++k) {
            int64_t sub = (m[k] == seg[0]) ? match : mismatch;
            int64_t a = CELL(0, r, k - 1) + del;
            int64_t b = (int64_t)(del * (k - 1) + sub);
            CELL(0, r, k) = a > b ? a : b;
        }
    }
    /* columns 1..n-1, main.cpp:183-208 */
    for (int i = 1; i < n; ++i) {
        for (int r = 0; r < R; ++r) {                                             /* :184-186 */
            int64_t e = CELL(i - 1, r, ROWLEN(r) - 1);
            if (e > jump[i]) jump[i] = e;
        }
        for (int r = 0; r < R; ++r) {
            const char *m = rows + row_off[r];
            const int L = ROWLEN(r);
            for (int k = 0; k < L; ++k) {
                int64_t best = SDO_NEG_INF;
                int sub = (m[k] == seg[i]) ? match : mismatch;                    /* :190 */
                if (jump[i] > SDO_NEG_INF) {                                      /* :191-193 */
                    int64_t c = jump[i] + sub + (int64_t)k * del;
                    if (c > best) best = c;
                }
                if (k > 0) {                                                      /* :194-204 */
                    if (CELL(i - 1, r, k - 1) > SDO_NEG_INF) {
                        int64_t c = CELL(i - 1, r, k - 1) + sub;
                        if (c > best) best = c;
                    }
                    if (CELL(i - 1, r, k) > SDO_NEG_INF) {
                        int64_t c = CELL(i - 1, r, k) + ins;
                        if (c > best) best = c;
                    }
                    if (CELL(i, r, k - 1) > SDO_NEG_INF) {
                        int64_t c = CELL(i, r, k - 1) + del;
                        if (c > best) best = c;
                    }
                }
                CELL(i, r, k) = best;
            }
        }
    }
    *jump_out = jump;
    return tab;
}

/* ---------------------------------------------------------------------------------------
 * One segment against all DP rows.  Restates MonomersAligner::AlignPartClassicDP,
 * main.cpp:151-270: forward DP (fill_table) :156-208, final argmax :209-216, equality-test traceback :217-267,
 * reversal :268.  Output records are in read order, positions relative to the segment.  Returns the record count,
 * or -1 if out is too small / allocation failed.
 * ------------------------------------------------------------------------------------- */
int sdo_align_segment(const char *seg, int n, const char *rows, const int *row_off, int R,
                      int ins, int del, int mismatch, int match, sdo_rec *out, int cap)
{
    if (n <= 0 || R <= 0) return 0;
    const int64_t width = row_off[R];
    int64_t *jump = NULL;
    int64_t *tab = fill_table(seg, n, rows, row_off, R, ins, del, mismatch, match, &jump);
    if (!tab) return -1;

    /* final argmax, main.cpp:209-216: int max_score, strict '<', lowest row wins */
    int top = SDO_NEG_INF, top_row = R;
    for (int r = 0; r < R; ++r) {
        int64_t e = CELL(n - 1, r, ROWLEN(r) - 1);
        if ((int64_t)top < e) { top = (int)e; top_row = r; }
    }
    if (top_row == R) { free(tab); free(jump); return -2; } /* reference would index out of range */

    /* traceback, main.cpp:217-267.  State (i, r, k); r == R is the jump state. */
    int cnt = 0, fail = 0;
    int64_t i = n - 1, r = top_row, k = ROWLEN(top_row) - 1;
    int fresh = 1;                       /* "monomer_changed" */
    sdo_rec cur; memset(&cur, 0, sizeof cur);
    while (i >= 0) {
        if (r != R && k == ROWLEN(r) - 1 && fresh) {                              /* :224-227 */
            cur.row = (int)r; cur.start = (int)i; cur.end = (int)i;
            cur.score = (float)CELL(i, r, k);
            fresh = 0;
        }
        if (r == R) {                                                             /* :228-240 */
            if (i != 0) {
                int found = 0;
                for (int p = 0; p < R; ++p) {
                    if (CELL(i - 1, p, ROWLEN(p) - 1) == jump[i]) {
                        --i; r = p; k = ROWLEN(p) - 1; found = 1;
                        break;
                    }
                }
                if (!found) { fail = 1; break; } /* reference would spin forever */
            } else {
                --i;
            }
            continue;
        }
        if (k != 0 && CELL(i, r, k) == CELL(i, r, k - 1) + del) {                 /* :242 */
            --k;
        } else if (i != 0 && CELL(i, r, k) == CELL(i - 1, r, k) + ins) {          /* :245 (no k guard) */
            --i;
        } else {
            int sub = (rows[row_off[r] + k] == seg[i]) ? match : mismatch;        /* :248 */
            if (i != 0 && k != 0 && CELL(i, r, k) == CELL(i - 1, r, k - 1) + sub) { /* :249 */
                --i; --k;
            } else {
                fresh = 1;                                                        /* :252 */
                if (cnt >= cap) { fail = 1; break; }
                if (i != 0 && jump[i] + (int64_t)k * del + sub == CELL(i, r, k)) { /* :253-257 */
                    cur.start = (int)i;
                    cur.score = cur.score - (float)jump[i];
                    out[cnt++] = cur;
                    r = R; k = 0;
                } else {                                                          /* :258-262 */
                    cur.start = (int)i;
                    out[cnt++] = cur;
                    --i;
                }
            }
        }
    }
    free(tab); free(jump);
    if (fail) return -1;
    for (int a = 0, b = cnt - 1; a < b; ++a, --b) { sdo_rec t = out[a]; out[a] = out[b]; out[b] = t; } /* :268 */
    return cnt;
}

/* ---------------------------------------------------------------------------------------
 * The DP table of one segment as the reference's traceback reads it (main.cpp:217-267), cell by cell:
 *   code[i * row_off[R] + row_off[r] + k]: the move the traceback takes at (i, r, k), in the order of :242-253:
 *     0 the deletion equality holds (k != 0), else 1 the insertion equality (i != 0; no k guard, :245), else 2 the
 *     diagonal equality (i != 0, k != 0), else 3 (close the alignment)
 *   J[i], i = 1..n-1: jump[i] = max_r dp[i-1][r][last];  J[n]: the final maximum (:209-216)
 *   argJ[i]: the lowest row attaining J[i] -- the row the jump state picks (:230-236); argJ[n] = top row (:212)
 * J[0] and argJ[0] are set to 0.  Returns 0, or -1 if an allocation failed.
 * ------------------------------------------------------------------------------------- */
int sdo_dp_tables(const char *seg, int n, const char *rows, const int *row_off, int R,
                  int ins, int del, int mismatch, int match, int8_t *code, int64_t *J, int *argJ)
{
    if (n <= 0 || R <= 0) return 0;
    const int64_t width = row_off[R];
    int64_t *jump = NULL;
    int64_t *tab = fill_table(seg, n, rows, row_off, R, ins, del, mismatch, match, &jump);
    if (!tab) return -1;
    for (int i = 0; i < n; ++i)
        for (int r = 0; r < R; ++r) {
            const char *m = rows + row_off[r];
            for (int k = 0; k < ROWLEN(r); ++k) {
                const int64_t h = CELL(i, r, k);
                const int sub = (m[k] == seg[i]) ? match : mismatch;
                int c = 3;
                if (k != 0 && h == CELL(i, r, k - 1) + del) c = 0;                                /* :242 */
                else if (i != 0 && h == CELL(i - 1, r, k) + ins) c = 1;                           /* :245 */
                else if (i != 0 && k != 0 && h == CELL(i - 1, r, k - 1) + sub) c = 2;             /* :249 */
                code[(int64_t)i * width + row_off[r] + k] = (int8_t)c;
            }
        }
    J[0] = 0; argJ[0] = 0;
    for (int i = 1; i <= n; ++i) {
        J[i] = SDO_NEG_INF; argJ[i] = R;
        for (int r = 0; r < R; ++r) {
            const int64_t e = CELL(i - 1, r, ROWLEN(r) - 1);
            if (e > J[i]) { J[i] = e; argJ[i] = r; }                                     /* strict: lowest row */
        }
    }
    free(tab); free(jump);
    return 0;
}
#undef CELL
#undef ROWLEN

/* ---------------------------------------------------------------------------------------
 * MonomerEditDistance, main.cpp:128-133: edlibAlign(monomer, segment, k = -1, EDLIB_MODE_HW,
 * EDLIB_TASK_DISTANCE).  edlib (vendored by the reference as src/edlib.cpp, Myers bit-vector) returns the
 * unit-cost edit distance between the query and the best-matching substring of the target ("infix" / HW
 * mode: gaps before and after the query's image in the target are free).  Restated here from that published
 * definition as the textbook O(n*m) dynamic program: D[0][j] = 0, D[i][0] = i, answer = min_j D[m][j].
 * ------------------------------------------------------------------------------------- */
int sdo_hw_distance(const char *query, int m, const char *target, int n)
{
    int *prev = (int *)malloc(sizeof(int) * (size_t)(n + 1)), *cur = (int *)malloc(sizeof(int) * (size_t)(n + 1));
    for (int j = 0; j <= n; ++j) prev[j] = 0;
    for (int i = 1; i <= m; ++i) {
        cur[0] = i;
        for (int j = 1; j <= n; ++j) {
            int a = prev[j - 1] + (query[i - 1] != target[j - 1]);
            int b = prev[j] + 1, c = cur[j - 1] + 1;
            cur[j] = a < b ? (a < c ? a : c) : (b < c ? b : c);
        }
        int *t = prev; prev = cur; cur = t;
    }
    int best = prev[0];
    for (int j = 1; j <= n; ++j) if (prev[j] < best) best = prev[j];
    free(prev); free(cur);
    return best;
}

/* FilterMonomersForRead, main.cpp:135-149: rows sorted by (distance, index); element 0 is always kept (:142), the
 * others when distance <= ed_thr (:143-147).  keep[] receives the kept row indices in their new order. */
typedef struct { int dist, idx; } sdo_di;
static int cmp_di(const void *a, const void *b)
{
    const sdo_di *x = (const sdo_di *)a, *y = (const sdo_di *)b;
    if (x->dist != y->dist) return x->dist < y->dist ? -1 : 1;
    return x->idx < y->idx ? -1 : (x->idx > y->idx);
}
int sdo_filter_rows(const char *seg, int n, const char *rows, const int *row_off, int R, int ed_thr, int *keep)
{
    sdo_di *v = (sdo_di *)malloc(sizeof(sdo_di) * (size_t)R);
    for (int r = 0; r < R; ++r) { v[r].dist = sdo_hw_distance(rows + row_off[r], row_off[r + 1] - row_off[r], seg, n); v[r].idx = r; }
    qsort(v, (size_t)R, sizeof(sdo_di), cmp_di);
    int nk = 0;
    keep[nk++] = v[0].idx;
    for (int x = 1; x < R; ++x) if (v[x].dist <= ed_thr) keep[nk++] = v[x].idx;
    free(v);
    return nk;
}

/* ---------------------------------------------------------------------------------------
 * Segmentation of one read, main.cpp:73-79.  The condition at :74 mixes int and size_t; it is
 * evaluated here with the same conversions (size_t arithmetic, int operands converted).
 * Returns the number of segments; offs/lens may be NULL to count only.
 * ------------------------------------------------------------------------------------- */
int sdo_segment_read(long read_len, int part_size, int overlap, int *offs, int *lens, int cap)
{
    int cnt = 0;
    if (part_size <= 0) return -1;   /* the reference loops forever */
    size_t len = (size_t)read_len;
    for (size_t i = 0; i < len; i += (size_t)part_size) {
        int keep = ((size_t)(int)len - i >= (size_t)overlap) || (len < (size_t)overlap);
        if (keep) {
            int rest = (int)(len - i);
            int want = part_size + overlap;
            int take = want < rest ? want : rest;
            if (take < 0) take = rest; /* substr(i, npos) */
            if (offs && cnt < cap) { offs[cnt] = (int)i; lens[cnt] = take; }
            ++cnt;
        }
    }
    return cnt;
}

/* Overlap resolution, main.cpp:287-302 (PostProcessing).  in/out may not alias. */
int sdo_postprocess(const sdo_rec *in, int n, sdo_rec *out)
{
    int m = 0;
    size_t i = 0, N = (size_t)n;
    while (i < N) {
        size_t hi = i + 7 < N ? i + 7 : N;
        for (size_t j = i + 1; j < hi; ++j) {
            if ((in[i].end - in[j].start) * 2 > (in[j].end - in[j].start)) {
                out[m++] = in[i];
                i = j + 1;
                break;
            }
        }
        if (i < N) out[m++] = in[i];
        ++i;
    }
    return m;
}

/* ----------------------------------------------------------------------------------------
 * FASTA loading, main.cpp:314-346.  Name = first whitespace token of the header (:321-325),
 * sequence lines appended raw (:327), alphabet {A,C,G,T,N} validated afterwards (:330-341).
 * -------------------------------------------------------------------------------------- */
typedef struct { char *name; char *seq; size_t len, cap; } sdo_seq;
typedef struct { sdo_seq *v; int n, cap; } sdo_seqs;

static void seqs_free(sdo_seqs *s)
{
    for (int i = 0; i < s->n; ++i) { free(s->v[i].name); free(s->v[i].seq); }
    free(s->v); s->v = NULL; s->n = s->cap = 0;
}

static sdo_seq *seqs_push(sdo_seqs *s, const char *name, size_t name_len)
{
    if (s->n == s->cap) { s->cap = s->cap ? s->cap * 2 : 16; s->v = (sdo_seq *)realloc(s->v, sizeof(sdo_seq) * (size_t)s->cap); }
    sdo_seq *q = &s->v[s->n++];
    q->name = (char *)malloc(name_len + 1); memcpy(q->name, name, name_len); q->name[name_len] = 0;
    q->cap = 256; q->len = 0; q->seq = (char *)malloc(q->cap); q->seq[0] = 0;
    return q;
}

/* returns 0 ok, 255 on illegal symbol (message on err).  A missing file yields zero sequences
 * (main.cpp:315-319: the ifstream simply never delivers a line). */
static int load_fasta_file(const char *path, sdo_seqs *out, FILE *err)
{
    memset(out, 0, sizeof *out);
    FILE *f = fopen(path, "rb");
    if (f) {
        char *line = NULL; size_t lcap = 0; ssize_t got;
        while ((got = getline(&line, &lcap, f)) >= 0) {
            size_t L = (size_t)got;
            if (L && line[L - 1] == '\n') --L;      /* std::getline drops '\n' only; '\r' stays */
            if (L > 0 && line[0] == '>') {
                size_t a = 1;
                while (a < L && (line[a] == ' ' || line[a] == '\t' || line[a] == '\r' || line[a] == '\v' || line[a] == '\f')) ++a;
                size_t b = a;
                while (b < L && !(line[b] == ' ' || line[b] == '\t' || line[b] == '\r' || line[b] == '\v' || line[b] == '\f')) ++b;
                seqs_push(out, line + a, b - a);    /* empty header would be UB upstream */
            } else if (out->n > 0) {
                sdo_seq *q = &out->v[out->n - 1];
                if (q->len + L + 1 > q->cap) { while (q->len + L + 1 > q->cap) q->cap *= 2; q->seq = (char *)realloc(q->seq, q->cap); }
                memcpy(q->seq + q->len, line, L); q->len += L; q->seq[q->len] = 0;
            } /* a sequence line before any header is UB upstream (seqs[-1]); ignored here */
        }
        free(line); fclose(f);
    }
    int has_n = 0;
    for (int i = 0; i < out->n; ++i) {
        const sdo_seq *q = &out->v[i];
        for (size_t x = 0; x < q->len; ++x) {
            char c = q->seq[x];
            if (!(c == 'A' || c == 'C' || c == 'G' || c == 'T' || c == 'N')) {   /* :333-336 */
                fprintf(err, "ERROR: Sequence %s contains undefined symbol (not ACGT): %c\n", q->name, c);
                return 255;
            }
            if (c == 'N') has_n = 1;
        }
    }
    if (has_n)                                                                     /* :342-344 */
        fprintf(err, "WARNING: sequences in %s contain N symbol. It will be counted as a separate symbol in scoring!\n", path);
    return 0;
}

static char comp_base(char c) /* main.cpp:350 */
{
    switch (c) { case 'A': return 'T'; case 'T': return 'A'; case 'G': return 'C'; case 'C': return 'G'; default: return 'N'; }
}

/* growable text buffer */
typedef struct { char *p; size_t n, cap; } sdo_buf;
static void buf_add(sdo_buf *b, const char *s, size_t n)
{
    if (b->n + n + 1 > b->cap) { size_t c = b->cap ? b->cap : 4096; while (b->n + n + 1 > c) c *= 2; b->p = (char *)realloc(b->p, c); b->cap = c; }
    memcpy(b->p + b->n, s, n); b->n += n; b->p[b->n] = 0;
}

/* ----------------------------------------------------------------------------------------
 * Whole `dp` run.  Restates main(), main.cpp:374-402 (argument handling is done by the caller,
 * see sdo_cli_main), add_reverse_complement :364-371, AlignReadsSet :67-122 (segments in read
 * order; per read: offsets added :110, PostProcessing :116, SaveBatch :117 / :272-285).
 * The OpenMP chunking of :85-103 does not influence the output and is replaced by a plain
 * parallel loop over all segments.  raw TSV goes to *tsv (malloc'd, caller frees).
 * -------------------------------------------------------------------------------------- */
int sdo_run_files(const char *reads_path, const char *monomers_path, int threads, int part_size, int overlap,
                  int ins, int del, int mismatch, int match, int ed_thr, char **tsv, size_t *tsv_len, FILE *err)
{
    sdo_seqs reads, mons;
    *tsv = NULL; *tsv_len = 0;
    int st = load_fasta_file(reads_path, &reads, err);
    if (st) { seqs_free(&reads); return st; }
    st = load_fasta_file(monomers_path, &mons, err);
    if (st) { seqs_free(&reads); seqs_free(&mons); return st; }

    /* rows = forward monomers in file order, then all reverse complements (name + "'") */
    const int M = mons.n, R = 2 * M;
    int *row_off = (int *)malloc(sizeof(int) * (size_t)(R + 1));
    size_t tot = 0;
    for (int j = 0; j < M; ++j) tot += mons.v[j].len;
    char *rows = (char *)malloc(2 * tot + 1);
    row_off[0] = 0;
    for (int j = 0; j < M; ++j) { memcpy(rows + row_off[j], mons.v[j].seq, mons.v[j].len); row_off[j + 1] = row_off[j] + (int)mons.v[j].len; }
    for (int j = 0; j < M; ++j) {
        int L = (int)mons.v[j].len;
        for (int x = 0; x < L; ++x) rows[row_off[M + j] + x] = comp_base(mons.v[j].seq[L - 1 - x]);
        row_off[M + j + 1] = row_off[M + j] + L;
    }

    /* segmentation of all reads, :70-81 */
    int nseg = 0, *first = (int *)malloc(sizeof(int) * (size_t)(reads.n + 1));
    for (int p = 0; p < reads.n; ++p) {
        first[p] = nseg;
        int c = sdo_segment_read((long)reads.v[p].len, part_size, overlap, NULL, NULL, 0);
        if (c < 0) { fprintf(err, "oracle: part_size must be positive\n"); st = 2; goto done0; }
        nseg += c;
    }
    first[reads.n] = nseg;
    {
        int *soff = (int *)malloc(sizeof(int) * (size_t)(nseg + 1)), *slen = (int *)malloc(sizeof(int) * (size_t)(nseg + 1));
        int *sread = (int *)malloc(sizeof(int) * (size_t)(nseg + 1)), *scnt = (int *)calloc((size_t)nseg + 1, sizeof(int));
        sdo_rec **srec = (sdo_rec **)calloc((size_t)nseg + 1, sizeof(sdo_rec *));
        for (int p = 0; p < reads.n; ++p) {
            sdo_segment_read((long)reads.v[p].len, part_size, overlap, soff + first[p], slen + first[p], nseg - first[p]);
            for (int s = first[p]; s < first[p + 1]; ++s) sread[s] = p;
        }
        fprintf(err, "Prepared reads\n");                                           /* :82 */
        int bad = 0;
        if (threads < 1) threads = 1;
#ifdef _OPENMP
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
#endif
        for (int s = 0; s < nseg; ++s) {
            sdo_rec *buf = (sdo_rec *)malloc(sizeof(sdo_rec) * (size_t)(slen[s] + 1));
            const char *segp = reads.v[sread[s]].seq + soff[s];
            int c = 0;
            if (R > 0 && ed_thr > -1) {                                              /* main.cpp:91-93 */
                int *keep = (int *)malloc(sizeof(int) * (size_t)R), *foff = (int *)malloc(sizeof(int) * (size_t)(R + 1));
                int nk = sdo_filter_rows(segp, slen[s], rows, row_off, R, ed_thr, keep);
                char *frows = (char *)malloc((size_t)row_off[R] + 1);
                foff[0] = 0;
                for (int x = 0; x < nk; ++x) {
                    int L = row_off[keep[x] + 1] - row_off[keep[x]];
                    memcpy(frows + foff[x], rows + row_off[keep[x]], (size_t)L);
                    foff[x + 1] = foff[x] + L;
                }
                c = sdo_align_segment(segp, slen[s], frows, foff, nk, ins, del, mismatch, match, buf, slen[s] + 1);
                for (int x = 0; x < c; ++x) buf[x].row = keep[buf[x].row];            /* back to rows of the full set */
                free(keep); free(foff); free(frows);
            } else if (R > 0) {
                c = sdo_align_segment(segp, slen[s], rows, row_off, R, ins, del, mismatch, match, buf, slen[s] + 1);
            }
            if (c < 0) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
                bad = 1;
                c = 0;
            }
            srec[s] = buf; scnt[s] = c;
        }
        if (bad) { fprintf(err, "oracle: segment alignment failed (out of the reference's domain)\n"); st = 3; }
        sdo_buf outb; memset(&outb, 0, sizeof outb);
        for (int p = 0; p < reads.n && !st; ++p) {
            int total = 0;
            for (int s = first[p]; s < first[p + 1]; ++s) total += scnt[s];
            if (first[p + 1] == first[p] || total == 0) continue; /* reference: UB (batch[0] of empty vector), App. B */
            sdo_rec *all = (sdo_rec *)malloc(sizeof(sdo_rec) * (size_t)total), *kept = (sdo_rec *)malloc(sizeof(sdo_rec) * (size_t)total);
            int a = 0;
            for (int s = first[p]; s < first[p + 1]; ++s)
                for (int x = 0; x < scnt[s]; ++x) { all[a] = srec[s][x]; all[a].start += soff[s]; all[a].end += soff[s]; ++a; }  /* :110 */
            fprintf(err, "%zu%%: Aligned %s\n", (size_t)(p + 1) * 100 / (size_t)reads.n, reads.v[p].name);      /* :115 */
            int m = sdo_postprocess(all, total, kept);
            int prev_end = 0;                                                       /* :273 */
            for (int x = 0; x < m; ++x) {
                const sdo_rec *q = &kept[x];
                const sdo_seq *mono = &mons.v[q->row < M ? q->row : q->row - M];
                char line[256];
                buf_add(&outb, reads.v[p].name, strlen(reads.v[p].name)); buf_add(&outb, "\t", 1);
                buf_add(&outb, mono->name, strlen(mono->name));
                if (q->row >= M) buf_add(&outb, "'", 1);
                int w = snprintf(line, sizeof line, "\t%d\t%d\t%f\t%d\t%d\n", q->start, q->end, (double)q->score, q->start - prev_end, q->end - q->start);
                buf_add(&outb, line, (size_t)w);
                prev_end = q->end;
            }
            free(all); free(kept);
        }
        if (!outb.p) buf_add(&outb, "", 0);
        *tsv = outb.p; *tsv_len = outb.n;
        for (int s = 0; s < nseg; ++s) free(srec[s]);
        free(srec); free(scnt); free(sread); free(soff); free(slen);
    }
done0:
    free(first); free(rows); free(row_off);
    seqs_free(&reads); seqs_free(&mons);
    return st;
}

/* The `dp` command line, main.cpp:374-402, including the argc==10 / argc==11 quirk (:381-391). */
int sdo_cli_main(int argc, char **argv)
{
    if (argc < 5) {
        fputs("Failed to process. Number of arguments < 5\n", stdout);
        fputs("./decompose <reads> <monomers> <threads> <part-size> <overlap> [<ins-score> <del-score> <mismatch-score> <match-score>]\n", stdout);
        return 255;
    }
    if (argc == 5) { fprintf(stderr, "oracle: missing <overlap> (the reference aborts on a NULL argv)\n"); return 134; }
    int ins = -1, del = -1, mismatch = -1, match = 1;
    if (argc == 10) { ins = atoi(argv[6]); del = atoi(argv[7]); mismatch = atoi(argv[8]); match = atoi(argv[9]); }
    int ed_thr = -1;
    if (argc == 11) ed_thr = atoi(argv[10]);
    fprintf(stderr, "Scores: insertion=%d deletion=%d mismatch=%d match=%d\n", ins, del, mismatch, match);
    char *tsv; size_t n;
    int st = sdo_run_files(argv[1], argv[2], atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), ins, del, mismatch, match, ed_thr, &tsv, &n, stderr);
    if (tsv) { fwrite(tsv, 1, n, stdout); free(tsv); }
    return st;
}

#ifdef SDO_MAIN
int main(int argc, char **argv) { return sdo_cli_main(argc, argv); }
#endif
