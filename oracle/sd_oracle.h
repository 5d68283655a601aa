/* sd_oracle.h -- CPU oracle for the string-decomposition DP.  TEST INFRASTRUCTURE ONLY
 * (see the header of sd_oracle.c).  Restates /root/reference/stringdecomposer/src/main.cpp. */
#ifndef SD_ORACLE_H
#define SD_ORACLE_H
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#ifdef __cplusplus
extern "C" {
#endif

/* One monomer alignment of a segment: MonomerAlignment of main.cpp:37-49 with the monomer kept
 * as a DP-row index (rows 0..M-1 forward in FASTA order, M..2M-1 reverse complements). */
typedef struct { int row; int start; int end; float score; } sdo_rec;

int sdo_align_segment(const char *seg, int n, const char *rows, const int *row_off, int R,
                      int ins, int del, int mismatch, int match, sdo_rec *out, int cap);
int sdo_dp_tables(const char *seg, int n, const char *rows, const int *row_off, int R,
                  int ins, int del, int mismatch, int match, int8_t *code, int64_t *J, int *argJ);
int sdo_segment_read(long read_len, int part_size, int overlap, int *offs, int *lens, int cap);
int sdo_postprocess(const sdo_rec *in, int n, sdo_rec *out);
int sdo_hw_distance(const char *query, int m, const char *target, int n);
int sdo_filter_rows(const char *seg, int n, const char *rows, const int *row_off, int R, int ed_thr, int *keep);
int sdo_run_files(const char *reads_path, const char *monomers_path, int threads, int part_size, int overlap,
                  int ins, int del, int mismatch, int match, int ed_thr, char **tsv, size_t *tsv_len, FILE *err);
int sdo_cli_main(int argc, char **argv);
/* identity rescoring (sd_identity_oracle.c; main.py:29-60) */
int sdo_nw_path_counts(const char *q, int qlen, const char *t, int tlen, int *matches, int *columns);
int sdo_nw_uses_traceback(int qlen, int tlen);
int sdo_nw_prefix_counts(const char *q, int qlen, const char *t, int tlen, int32_t *dist, int32_t *matches, int32_t *columns);
int sdo_nw_path_counts_batch(const char *qtext, const int64_t *qoff, const char *ttext, const int64_t *toff,
                             const int32_t *pair_q, const int32_t *pair_t, int64_t npairs,
                             int32_t *dist, int32_t *matches, int32_t *columns);

#ifdef __cplusplus
}
#endif
#endif
