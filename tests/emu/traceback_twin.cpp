// traceback_twin.cpp -- the host twin of tests/cuda/traceback_probe.cu: the same file (tests/cuda/tb_file.h) walked by
// sweep_core.cuh: traceback_segment + fetch_code, the walk the emulator runs.  CPU TEST-SUITE ONLY (built by
// tests/test_traceback.py), so that the tables the tests construct, the file format and the emulator's walker can be
// checked without a GPU.
//
//   traceback_twin IN...      (writes IN.out for every IN)
#include <cstdio>
#include <string>
#include <vector>

#include "../cuda/tb_file.h"

static int run_one(const char *in, const char *out_path)
{
    using namespace sdb;
    TbFile f;
    if (!read_tb_file(in, f)) { fprintf(stderr, "%s: short or missing input\n", in); return 1; }
    const Geometry &g = f.g;
    const std::vector<int64_t> rec_off = f.seg_rec_off();
    std::vector<Record> scratch((size_t)rec_off[f.nseg]), dense;
    std::vector<int> counts((size_t)f.nseg, 0);
    int error = 0, total = 0;
    for (int s = 0; s < f.nseg; ++s) {
        const int n = (int)(f.seg_off[s + 1] - f.seg_off[s]);
        auto code_at = [&](int i, int row, int rowlen, int k) {
            const RowPlace pl = place_row(g, g.NG > 1 ? 0 : s % g.NS, row);
            const int cta = g.NG > 1 ? s * g.NG + pl.grp : s / g.NS;
            return fetch_code(f.codes.data() + f.cta_code_off[cta] + (size_t)i * g.NT * g.CW, g, pl, rowlen, k);
        };
        Record *out = scratch.data() + rec_off[s];
        const int c = traceback_segment(n, f.jr.data() + f.seg_j_off[s], f.bases.data() + f.seg_off[s], f.rows.data(), f.row_off.data(),
                                        f.ins, f.del, f.mismatch, f.match, code_at, out, n, true,
                                        f.with_r2r ? f.r2r.data() + (size_t)s * 2 * g.M : nullptr, 2 * g.M);
        if (c == SD_TB_BAD_ROW) { error = 1; continue; }
        if (c < 0) { counts[(size_t)s] = -1; total = -1; continue; }
        counts[(size_t)s] = c;
        if (total >= 0) total += c;
        for (int x = c - 1; x >= 0; --x) dense.push_back(out[x]);
    }
    if (total < 0) dense.clear();
    if (!write_tb_result(out_path, error, total, counts.data(), f.nseg, dense.data())) { perror(out_path); return 1; }
    return 0;
}

int main(int argc, char **argv)
{
    if (argc < 2) { fprintf(stderr, "usage: traceback_twin IN...\n"); return 1; }
    for (int a = 1; a < argc; ++a)
        if (const int st = run_one(argv[a], (std::string(argv[a]) + ".out").c_str())) return st;
    return 0;
}
