// tb_file.h -- the file format of traceback_probe.cu (the traceback and gather kernels on the GPU) and of its host twin
// tests/emu/traceback_twin.cpp (sweep_core.cuh: traceback_segment + fetch_code), so that tests/test_traceback.py can
// hand both the same tables.
//
// IN (little-endian): int32 packed, C, T, nslots, M, NS, NT, CW, NG, SG, lat, scanw, stream (Geometry), ins, del,
//                     mismatch, match, nseg, nctas, with_r2r; int64 seg_off[nseg+1]; int32 row_off[2M+1]; the segments'
//                     bytes; the rows' bytes (ASCII); int64 cta_code_off[nctas+1]; uint32 codes[cta_code_off[nctas]];
//                     int64 seg_j_off[nseg+1]; int32 {j, row}[seg_j_off[nseg]]; int32 rank2row[nseg][2M] if with_r2r
// OUT:                int32 error (a jump to a row outside the monomer set), total (-1: a record buffer overflowed),
//                     counts[nseg]; int32 {row, start, end, score}[total], each segment's records in read order
#pragma once
#include <cstdio>
#include <vector>

#include "common.h"

struct TbFile {
    sdb::Geometry g{};
    int ins = 0, del = 0, mismatch = 0, match = 0, nseg = 0, nctas = 0, with_r2r = 0;
    std::vector<int64_t> seg_off, cta_code_off, seg_j_off;
    std::vector<int> row_off, r2r;
    std::vector<uint8_t> bases, rows;
    std::vector<uint32_t> codes;
    std::vector<sdb::JR> jr;
    std::vector<int64_t> seg_rec_off() const       // scratch records of a segment: at most one per column
    {
        std::vector<int64_t> o(seg_off.size(), 0);
        for (int s = 0; s < nseg; ++s) o[s + 1] = o[s] + (seg_off[s + 1] - seg_off[s]);
        return o;
    }
};

template <class T> static bool tb_get(FILE *f, std::vector<T> &v, size_t n) { v.resize(n); return fread(v.data(), sizeof(T), n, f) == n; }

static bool read_tb_file(const char *path, TbFile &t)
{
    FILE *f = fopen(path, "rb");
    if (!f) return false;
    std::vector<int> h;
    bool ok = tb_get(f, h, 20);
    if (ok) {
        sdb::Geometry &g = t.g;
        int *gf[13] = {&g.packed, &g.C, &g.T, &g.nslots, &g.M, &g.NS, &g.NT, &g.CW, &g.NG, &g.SG, &g.lat, &g.scanw, &g.stream};
        for (int x = 0; x < 13; ++x) *gf[x] = h[x];
        t.ins = h[13]; t.del = h[14]; t.mismatch = h[15]; t.match = h[16]; t.nseg = h[17]; t.nctas = h[18]; t.with_r2r = h[19];
        const size_t R = 2 * (size_t)g.M;
        ok = tb_get(f, t.seg_off, t.nseg + 1) && tb_get(f, t.row_off, R + 1) && tb_get(f, t.bases, t.seg_off[t.nseg]) &&
             tb_get(f, t.rows, t.row_off[R]) && tb_get(f, t.cta_code_off, t.nctas + 1) && tb_get(f, t.codes, t.cta_code_off[t.nctas]) &&
             tb_get(f, t.seg_j_off, t.nseg + 1) && tb_get(f, t.jr, t.seg_j_off[t.nseg]) && tb_get(f, t.r2r, t.with_r2r ? t.nseg * R : 0);
    }
    fclose(f);
    return ok;
}

static bool write_tb_result(const char *path, int error, int total, const int *counts, int nseg, const sdb::Record *recs)
{
    FILE *f = fopen(path, "wb");
    if (!f) return false;
    const int hdr[2] = {error, total};
    bool ok = fwrite(hdr, 4, 2, f) == 2 && fwrite(counts, 4, nseg, f) == (size_t)nseg &&
              (total <= 0 || fwrite(recs, sizeof(sdb::Record), total, f) == (size_t)total);
    return fclose(f) == 0 && ok;
}
