/*
 * sd_b200.h -- C ABI of the B200-native string-decomposition DP (libsd_b200.so).
 *
 * The reference (ablab/stringdecomposer v1.1.2) has no FFI: its boundary is the process CLI of the `dp`
 * binary that stringdecomposer/main.py:194 spawns.  The entry points below are what a binding for that
 * path would need; each cites the reference code it replaces (main.cpp = stringdecomposer/src/main.cpp,
 * main.py = stringdecomposer/main.py, edlib.cpp = stringdecomposer/src/edlib.cpp).  Plain C types only, caller-owned inputs, library-owned outputs that
 * are released with sd_free(), integer status codes (0 = ok), no exceptions cross the boundary.
 * A handle may be used from one host thread at a time.  There is no CPU fallback: sd_create() fails
 * with SD_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef SD_B200_H
#define SD_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct sd_handle sd_handle;

enum {
    SD_OK = 0,
    SD_ERR_ARG = 1,          /* bad argument (NULL, negative size, symbol outside ACGTN, ...) */
    SD_ERR_NO_DEVICE = 2,    /* no usable CUDA device / CUDA runtime error at start-up */
    SD_ERR_UNSUPPORTED = 3,  /* outside the supported domain (monomer set too large for this build, scores reaching
                                the reference's INF sentinel, a segment whose DP needs more device memory than the
                                device has, a sequence too long for sd_identity) */
    SD_ERR_CUDA = 4,         /* CUDA failure while running */
    SD_ERR_INTERNAL = 5,
    SD_ERR_INPUT = 255       /* illegal FASTA symbol: the reference exits with status 255 (main.cpp:333-336) */
};

/* One monomer alignment of a segment -- MonomerAlignment (main.cpp:37-49) with the monomer kept as a DP-row
 * index: rows 0..M-1 are the forward monomers in input order, rows M..2M-1 their reverse complements in the
 * same order (add_reverse_complement, main.cpp:364-371).  start/end are segment-relative read positions
 * (main.cpp:225,254,259), score is the `identity` field the raw TSV prints (main.cpp:225,255,279). */
typedef struct { int32_t row, start, end, score; } sd_record;

typedef struct {
    double sweep_ms, traceback_ms;      /* CUDA-event time of the kernels, max over devices, accumulated */
    double h2d_ms, d2h_ms;
    int64_t h2d_bytes, d2h_bytes;
    int64_t cells;                      /* cell updates computed: sum over segments n_seg * sum of row lengths */
    int64_t segments, columns;
    int64_t launches;                   /* kernels launched */
    int32_t n_devices;
    int32_t packed;                     /* 1: s16x2 sweep, 0: s32 sweep (last call) */
    int32_t C, T, NS, NT;               /* launch geometry of the last call */
    int32_t NG, lat, scanw;             /* CTAs per segment; 1 = deferred-jump sweep; carry window of the scan */
    int32_t stream;                     /* 1: the sweep read the segment symbols from global memory as it went (segments
                                           too long for shared memory); 0: they were staged in shared memory */
    int64_t sweep_store_bytes;          /* bytes the sweep writes per pass over the last batch: 2-bit codes (incl. slot
                                           padding) + 8 B per column, summed over devices -- computed from the layout */
    int32_t dev_segments[8];            /* segments each device got in the last batch (AlignReadsSet's gather,
                                           main.cpp:84-121, is the concatenation in device order) */
} sd_stats;

/* Replaces the MonomersAligner constructor (main.cpp:59-65) + add_reverse_complement (main.cpp:364-371).
 * monomers: the forward monomers as upper-case ACGTN text, concatenated; monomer j is
 * monomers[offsets[j] .. offsets[j+1]).  device_ids may be NULL (n_devices = 0 -> device 0; n_devices = -1 ->
 * all visible devices). */
int sd_create(const char *monomers, const int64_t *offsets, int32_t n_monomers,
              int32_t ins, int32_t del, int32_t mismatch, int32_t match,
              const int32_t *device_ids, int32_t n_devices, sd_handle **out);

/* Replaces the per-segment calls of AlignPartClassicDP (main.cpp:151-270) that AlignReadsSet issues under OpenMP
 * (main.cpp:87-102).  segments: ACGTN text of all segments back to back, segment s = [offsets[s], offsets[s+1]).
 * On success *records holds the alignments of all segments in segment order, each segment's in read order,
 * and (*rec_offsets)[s .. s+1] delimits segment s (n_segments+1 entries).  Release both with sd_free().
 * Segment length is limited only by the score domain and by device memory, not by shared memory: segments too long to
 * be staged in shared memory are swept with their symbols read from device memory (sd_stats.stream).  A segment whose
 * scores can reach the reference's INF sentinel -- length * max(|ins|, |mismatch|) + 2 * longest monomer * |del| +
 * 2 * |mismatch| + |match| must stay below 999,000, about 998 kb with the default scores -- returns
 * SD_ERR_UNSUPPORTED, and so does a segment whose backpointers (0.25 B per cell of every monomer row, with slot
 * padding) exceed the memory that was free on its device when the handle was created; sd_last_error() then gives the
 * segment length and the bytes needed and available. */
int sd_decompose(sd_handle *h, const char *segments, const int64_t *offsets, int64_t n_segments,
                 sd_record **records, int64_t **rec_offsets);

/* The same call split in three so that the kernels can be timed with inputs resident in HBM:
 * sd_stage copies the segments to the device(s), sd_run_staged runs sweep + traceback (may be repeated),
 * sd_fetch_staged returns the records.  Only valid when the batch fits one wave per device. */
int sd_stage(sd_handle *h, const char *segments, const int64_t *offsets, int64_t n_segments);
int sd_run_staged(sd_handle *h, double *kernel_ms);
int sd_fetch_staged(sd_handle *h, sd_record **records, int64_t **rec_offsets);

/* Replaces AlignReadsSet's segmentation (main.cpp:70-81).  Returns the number of segments of a read of
 * read_len symbols; fills offs/lens (capacity cap) when they are not NULL.  Negative on bad arguments. */
int64_t sd_segment_read(int64_t read_len, int32_t part_size, int32_t overlap, int64_t *offs, int32_t *lens, int64_t cap);

/* Replaces PostProcessing (main.cpp:287-302) on read-relative records.  Returns the number kept (<= n). */
int64_t sd_postprocess(const sd_record *in, int64_t n, sd_record *out);

/* Replaces main() of the `dp` binary (main.cpp:374-402) after argument parsing: load_fasta of both files
 * (main.cpp:314-346), reverse complements, segmentation, DP, overlap resolution, SaveBatch (main.cpp:272-285).
 * The raw TSV goes to out_fd, the reference's diagnostics to err_fd.  Returns the process exit status the
 * reference would produce (0, or 255 for an illegal symbol) or an SD_ERR_* code.  part_size may be as large as the
 * longest read (one segment per read); the segment-length limits of sd_decompose apply, and both return
 * SD_ERR_UNSUPPORTED (3) with an "ERROR: ..." line on err_fd and no output. */
int sd_run_files(const char *reads_path, const char *monomers_path, int32_t threads, int32_t part_size,
                 int32_t overlap, int32_t ins, int32_t del, int32_t mismatch, int32_t match, int32_t ed_thr,
                 int out_fd, int err_fd);

/* Replaces FilterMonomersForRead (main.cpp:135-149), the optional --ed_thr pre-filter: for every segment the DP rows
 * are sorted by (infix edit distance to the segment, row), the closest row and every row with distance <= ed_thr are
 * kept, and the DP runs on that re-ordered subset (so arg-max ties follow the new order).  ed_thr < 0 switches it
 * off (default).  Records keep reporting rows of the full set. */
int sd_set_ed_thr(sd_handle *h, int32_t ed_thr);

/* Replaces MonomerEditDistance (main.cpp:128-133): infix (edlib "HW") unit-cost edit distance of `query` against the
 * best substring of `target`; host-side helper (the pre-filter itself runs on the device).  -1 on bad arguments. */
int32_t sd_hw_distance(const char *query, int32_t query_len, const char *target, int32_t target_len);

/* Replaces edist / aai (stringdecomposer/main.py:29-60), the per-alignment `edlib.align(interval, monomer, mode="NW",
 * task="path")` of the final-TSV stage (convert_read, main.py:107-147): for every (query, target) pair the unit-cost
 * global alignment edlib would report -- its edit distance, the number of '=' columns and the alignment length, so
 * that identity = 100 * matches / columns -- computed on `device` for the whole batch at once.
 *   queries / targets   concatenated bytes (compared verbatim, like edlib's default equality) + n+1 offsets
 *   pair_query/_target  n_pairs index pairs; both NULL: every query against every target, query-major
 *                       (n_pairs must then be n_queries * n_targets)
 *   matches, columns    caller-allocated [n_pairs]; distance may be NULL.  A pair with an empty side gets
 *                       matches = columns = 0, distance = -1 (main.py:30-33 -> identity 0)
 *   hirschberg_pairs    optional: number of pairs so large that edlib would leave its traceback for Hirschberg
 *                       splitting (edlib.cpp:1187-1191) and might report another optimal path; they are still
 *                       computed with the traceback rule.  Lengths above 16382 are refused (SD_ERR_UNSUPPORTED).
 *   kernel_ms           optional: device time of the kernel */
int sd_identity(const char *queries, const int64_t *query_offsets, int64_t n_queries,
                const char *targets, const int64_t *target_offsets, int64_t n_targets,
                const int32_t *pair_query, const int32_t *pair_target, int64_t n_pairs,
                int32_t *matches, int32_t *columns, int32_t *distance,
                int32_t device, int64_t *hirschberg_pairs, double *kernel_ms);

/* Replaces convert_tsv / print_read / convert_read / classify (stringdecomposer/main.py:96-184): turns the raw `dp`
 * text into the final TSV (12 columns, main.py:158-162) on out_fd and, with light == 0 (--second-best), the per-monomer
 * `_alt` lines (main.py:163-166) on alt_fd.  All alignments of a chunk of lines go through sd_identity on `device`.
 *   raw, raw_len          the text `dp` wrote; as in the reference only its first four columns are read, names are cut
 *                         at the first blank and only newline-terminated lines count (main.py:173-176)
 *   read_names/reads      ids and (upper-case) sequences of the reads, concatenated + n_reads+1 offsets each
 *   mono_names/monos      the monomers in add_rc_monomers() order (main.py:80-85: each followed by its reverse
 *                         complement, named with a trailing quote), concatenated + n_monomers+1 offsets each
 *   min_identity          lines with identity below it are dropped (main.py:157)
 * Returns SD_OK or an SD_ERR_* code (sd_convert_error() has the text; a read or monomer of the raw text that is not in
 * the inputs -- a KeyError in the reference -- is SD_ERR_ARG).  Byte-identical to the Python mirror convert.convert_tsv. */
typedef struct sd_convert_stats {
    int64_t lines_in, lines_out, pairs, hirschberg_pairs;
    double kernel_ms;
} sd_convert_stats;
int sd_convert(const char *raw, int64_t raw_len,
               const char *read_names, const int64_t *read_name_off, const char *reads, const int64_t *read_off, int64_t n_reads,
               const char *mono_names, const int64_t *mono_name_off, const char *monos, const int64_t *mono_off, int32_t n_monomers,
               int32_t min_identity, int32_t light, int32_t device, int out_fd, int alt_fd, sd_convert_stats *stats);
const char *sd_convert_error(void);

int sd_get_stats(sd_handle *h, sd_stats *out);
void sd_reset_stats(sd_handle *h);
const char *sd_last_error(sd_handle *h);       /* h may be NULL: error of the last failed sd_create/sd_run_files */
void sd_free(void *p);
/* Optional page-locked host buffers for the caller's inputs (segment text of sd_decompose / sd_stage): copies from them
 * are plain DMA, without the driver's staging pass that pageable memory needs (the reference has no counterpart: its
 * reads live in std::string, main.cpp:283-330).  Any host pointer is accepted by every entry point; these only make
 * the copy-in cheaper.  NULL when the allocation fails. */
void *sd_host_alloc(int64_t bytes);
void sd_host_free(void *p);
void sd_destroy(sd_handle *h);
int sd_device_count(void);
const char *sd_version(void);

/* Measures the integer-pipe issue rate (lane-ops per second) the roofline is quoted against: streams of
 * independent VIADDMNMX.S16x2 (ALU pipe) and IMAD (FMA pipe) instructions on every SM of `device`. */
int sd_int_peak(int32_t device, double *alu_lane_ops_per_s, double *alu_fma_lane_ops_per_s, double *sm_clock_mhz);

#ifdef __cplusplus
}
#endif
#endif
