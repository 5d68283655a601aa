// common.h -- host-side types shared by the planner, the pipeline, the CUDA backend and the test emulator.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "sweep_core.cuh"

namespace sdb {

struct Scoring { int ins = -1, del = -1, mismatch = -1, match = 1; };   // main.cpp:380 defaults

// Symbol codes: A C G T N -> 0..4 (N is a fifth symbol that matches itself, main.cpp:190,330).
inline int base_code(char c)
{
    switch (c) { case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': return 3; case 'N': return 4; default: return -1; }
}

// DP rows: forward monomers in input order, then the reverse complement of each (main.cpp:364-371).
struct MonomerSet {
    int M = 0;                       // forward monomers; rows = 2M
    std::vector<uint8_t> rows;       // symbol codes of all 2M rows, concatenated
    std::vector<int> row_off;        // 2M+1 offsets into rows
    int Lmax = 0, Lmin = 0;
    int nrows() const { return 2 * M; }
    int rowlen(int r) const { return row_off[r + 1] - row_off[r]; }
};

// Everything a backend needs that depends only on (monomers, scoring, launch geometry).
struct Plan {
    Geometry g{};
    Scoring sc;
    int deadz = 0;                       // "minus infinity" in tag-3 form
    int nsl = 0;                         // slot lanes per segment = nslots*T
    int qp = 0;                          // uint4 per lane row of the profile: C/4 padded to an odd count (bank-conflict-free LDS.128)
    std::vector<uint32_t> prof;          // [5 symbols][nsl][qp][4] profile words 4*s''-1 (pad cells: very negative)
    std::vector<int> slot_len;           // row length of each slot
    std::vector<int> slot_endadd;        // (L-1)*del of each slot
    // deferred-jump sweep (Geometry::lat): profile rows carry p and, right behind it, the tagged prefix maximum PT of
    // the jump candidates: [5 symbols][nsl][qp2][4] with words [0,C) = p, [C,2C) = PT
    std::vector<uint32_t> prof2;
    int qp2 = 0;                         // uint4 per lane row of prof2: ceil(2C/4) padded to an odd count
    int kj[5] = {0, 0, 0, 0, 0};         // per symbol: best key of a jump-derived row end, relative to the jump base
    int lat_th = 0;                      // rebase threshold of the deferred form (SD_REBASE_TH minus one column step)
    size_t smem_bytes(int seg_stride) const;
};

// A batch of segments to decompose: upper-case ACGTN text of all segments back to back.  `text` may point into
// caller-owned memory (sd_decompose hands the caller's buffer straight to the H2D copy; the symbols are encoded
// and validated on the device) or into `own`.
struct Batch {
    const uint8_t *text = nullptr;
    std::vector<uint8_t> own;
    std::vector<int64_t> off;            // nseg+1, relative to text
    int nseg() const { return (int)off.size() - 1; }
    int len(int s) const { return (int)(off[s + 1] - off[s]); }
};

// A C G T N -> 0..4, anything else -> 255; shared by the device staging code and the emulator
SD_HD int ascii_code(unsigned c)
{
    return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : c == 'N' ? 4 : 255;
}
// Symbol code of a segment byte for the sweeps: a byte outside ACGTN sets *bad (the host then refuses the wave) and
// reads as 0, so the sweep stays in range until then
SD_HD int symbol_code(unsigned c, int *bad)
{
    int code = ascii_code(c);
    if (code > 4) { *bad = 1; code = 0; }
    return code;
}

struct BatchResult {
    std::vector<Record> recs;            // per segment in read order (already reversed), positions segment-relative
    std::vector<int64_t> rec_off;        // nseg+1
};

struct PlanError { std::string msg; };
// A traceback met a jump row outside the DP rows (a wrong column key).  The C ABI reports messages that start with
// "internal error:" as SD_ERR_INTERNAL.
constexpr const char *SD_MSG_TB_BAD_ROW = "internal error: the traceback met a jump to a row outside the monomer set";

// plan.cpp
void build_monomer_set(const std::vector<std::string> &forward, MonomerSet &ms);     // throws PlanError
// nseg_hint/n_hint steer the geometry heuristic (few long segments -> more lanes per slot).
Plan make_plan(const MonomerSet &ms, const Scoring &sc, int max_seg_len, int64_t nseg_hint);  // throws PlanError
bool packed_range_ok(const MonomerSet &ms, const Scoring &sc, int *deadz, int *pad_s);
bool geometry_compiled(int packed, int C, int T);
bool lat_geometry_compiled(int C, int T);
// per symbol: max over the DP rows of ((best s'' of the row for that symbol) + (L-1)*del) * 4096 + 4095 - tie-break index;
// rank_of_row: the --ed_thr ranks of one segment ([row] -> position in the filtered list, -1 = filtered out) or null
void lat_jump_keys(const MonomerSet &ms, const Scoring &sc, const int *rank_of_row, int out[5]);
// lanes a lane of a slot must look back so that the windowed deletion carry equals the full prefix maximum
int scan_window(const MonomerSet &ms, const Scoring &sc, int packed, int C, int T);
// CTA bookkeeping shared by backend and emulator
struct CtaLayout {
    std::vector<int> cta_nmax;           // longest segment of each CTA
    std::vector<int64_t> cta_code_off;   // word offset of each CTA's backpointer block (+1 sentinel)
    std::vector<int64_t> seg_j_off;      // offset of each segment's J/argJ arrays (n+1 entries each) (+1 sentinel)
    std::vector<int64_t> seg_rec_off;    // scratch record offset of each segment (cap = n) (+1 sentinel)
};
CtaLayout make_cta_layout(const Plan &p, const Batch &b, int seg_begin, int seg_end);
// SD_DUMP_TABLES=<directory> (tests): the directory into which every wave's sweep output is written, or null.
// dump_wave_tables writes one wave as <directory>/wave_<first segment, 8 digits>.bin (little-endian):
//   int32 packed, C, T, nslots, M, NS, NT, CW, NG, SG, lat, scanw, stream (Geometry), first segment, nseg, nctas;
//   int64 cta_code_off[nctas + 1], seg_j_off[nseg + 1]; uint32 codes[cta_code_off[nctas]]; int32 {j, row}[seg_j_off[nseg]]
const char *dump_tables_dir();
void dump_wave_tables(const char *dir, const Geometry &g, int first, const CtaLayout &l, const uint32_t *codes, const JR *jr);

// Backend interface.  configure() binds a plan; stage() copies a range of segments to the device;
// execute() runs sweep + traceback with inputs and outputs resident; fetch() brings the records back.
class Backend {
public:
    virtual ~Backend() {}
    virtual const char *name() const = 0;
    virtual void configure(const Plan &p, const MonomerSet &ms) = 0;
    virtual int64_t wave_bytes(const Batch &b, int seg_begin, int seg_end) const = 0;   // device bytes stage() would need
    virtual int64_t wave_budget() const = 0;                                            // bytes one wave may use
    // device memory a wave can never exceed: the CUDA backend reports what was free when it was created (never the
    // SD_WAVE_BYTES override); the host emulator keeps the fixed 1 GiB its wave budget was written for
    virtual int64_t device_bytes() const { return (int64_t)1 << 30; }
    // --ed_thr pre-filter (FilterMonomersForRead, main.cpp:135-149): -1 = off.  Applied by stage() to every segment.
    virtual void set_filter(int ed_thr) { ed_thr_ = ed_thr; }
    virtual void stage(const Batch &b, int seg_begin, int seg_end) = 0;
    virtual void execute() = 0;
    virtual void fetch(BatchResult &out) = 0;       // appends to out.recs / out.rec_off (out.rec_off starts as {0})
    // Pipelined form: submit() enqueues copy-in, kernels and copy-out of one wave on wave slot `slot` and returns at
    // once; collect() waits for that wave and appends its records.  A backend with wave_slots() == 2 overlaps the
    // copies of one wave with the kernels of the other.  Default: the synchronous three-step path.
    virtual int wave_slots() const { return 1; }
    virtual void reserve(int slot, const Batch &b, int seg_begin, int seg_end) { (void)slot; (void)b; (void)seg_begin; (void)seg_end; }   // size a slot's buffers for its largest wave up front
    virtual void submit(int slot, const Batch &b, int seg_begin, int seg_end) { (void)slot; stage(b, seg_begin, seg_end); execute(); }
    virtual void collect(int slot, BatchResult &out) { (void)slot; fetch(out); }
    double sweep_ms = 0, traceback_ms = 0, h2d_ms = 0, d2h_ms = 0;     // accumulated since reset_stats()
    int64_t h2d_bytes = 0, d2h_bytes = 0, launches = 0;
    int group_slots = 0;            // group sweep: most slot groups (CTA groups that loop over segment blocks) of a launch
    int ed_thr_ = -1;
    void reset_stats() { sweep_ms = traceback_ms = h2d_ms = d2h_ms = 0; h2d_bytes = d2h_bytes = launches = 0; group_slots = 0; }
};

// rank tables of the pre-filter for one segment: rows sorted by (distance, row); the first one and every row with
// distance <= ed_thr are kept (main.cpp:141-147).  rank_of_row[r] = position in the kept list or -1.
void build_filter_tables(const int *dist, int R, int ed_thr, int *rank_of_row, int *row_of_rank);

Backend *make_cuda_backend(int device_id, std::string &err);    // sweep_kernels.cu (product)
Backend *make_emu_backend();                                    // emu.cpp (CPU test-suite only; absent from libsd_b200.so)

} // namespace sdb
