// traceback_probe.cu -- runs the traceback and gather kernels (traceback_kernels.cuh) on the tables of one file and writes
// what the host gets back from a wave: the error word, the total, the counts and the dense records (tb_file.h), so that
// tests/test_traceback.py can compare the walk with a walker written from the reference on constructed tables.
//
//   traceback_probe IN...      (writes IN.out for every IN: one process, one CUDA context, many files)
#include <cstdio>
#include <string>
#include <vector>

#include "traceback_kernels.cuh"
#include "tb_file.h"

#define CK(x)                                                                                        \
    do {                                                                                             \
        cudaError_t e_ = (x);                                                                        \
        if (e_ != cudaSuccess) { fprintf(stderr, "%s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 3; } \
    } while (0)

template <class T> static cudaError_t to_device(const std::vector<T> &h, T **d)
{
    cudaError_t e = cudaMalloc(d, h.size() * sizeof(T) + 16);
    if (e == cudaSuccess && !h.empty()) e = cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
}

static int run_one(const char *in, const char *out_path)
{
    using namespace sdb;
    TbFile f;
    if (!read_tb_file(in, f)) { fprintf(stderr, "%s: short or missing input\n", in); return 1; }
    const std::vector<int64_t> rec_off = f.seg_rec_off();
    const int nseg = f.nseg;
    TbArgs t{};
    t.g = f.g; t.nseg = nseg;
    uint32_t *codes; int64_t *cta_code_off, *seg_j_off, *seg_off, *seg_rec_off; JR *jr; uint8_t *bases, *rows; int *row_off, *r2r = nullptr;
    CK(to_device(f.codes, &codes)); CK(to_device(f.cta_code_off, &cta_code_off)); CK(to_device(f.jr, &jr));
    CK(to_device(f.seg_j_off, &seg_j_off)); CK(to_device(f.bases, &bases)); CK(to_device(f.seg_off, &seg_off));
    CK(to_device(f.rows, &rows)); CK(to_device(f.row_off, &row_off)); CK(to_device(rec_off, &seg_rec_off));
    if (f.with_r2r) CK(to_device(f.r2r, &r2r));
    t.codes = codes; t.cta_code_off = cta_code_off; t.jr = jr; t.seg_j_off = seg_j_off; t.bases = bases; t.seg_off = seg_off;
    t.rows = rows; t.row_off = row_off; t.ins = f.ins; t.del = f.del; t.mismatch = f.mismatch; t.match = f.match;
    t.seg_rec_off = seg_rec_off; t.rank2row = r2r;
    // the result block of a wave: int32 header {0, 0, total, error}, counts[nseg], the dense records
    const size_t nrec = (size_t)rec_off[nseg], out_bytes = 16 + (size_t)nseg * 4 + nrec * sizeof(Record);
    Record *scratch; char *out;
    CK(cudaMalloc(&scratch, nrec * sizeof(Record) + 16));
    CK(cudaMalloc(&out, out_bytes + 16));
    CK(cudaMemset(out, 0, 16));
    int *hdr = reinterpret_cast<int *>(out), *counts = hdr + 4;
    Record *dense = reinterpret_cast<Record *>(counts + nseg);
    t.scratch = scratch; t.counts = counts; t.error = hdr + 3;
    cudaStream_t st;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    try { CK(launch_traceback(t, st)); } catch (PlanError &e) { fprintf(stderr, "%s\n", e.msg.c_str()); return 2; }
    gather_kernel<<<1, 1024, 0, st>>>(scratch, seg_rec_off, counts, dense, nseg, hdr + 2);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    std::vector<char> h(out_bytes);
    CK(cudaMemcpy(h.data(), out, out_bytes, cudaMemcpyDeviceToHost));
    cudaStreamDestroy(st);
    for (void *p : {(void *)codes, (void *)cta_code_off, (void *)jr, (void *)seg_j_off, (void *)bases, (void *)seg_off, (void *)rows,
                    (void *)row_off, (void *)seg_rec_off, (void *)r2r, (void *)scratch, (void *)out})
        cudaFree(p);
    const int *hh = reinterpret_cast<const int *>(h.data());
    if (!write_tb_result(out_path, hh[3], hh[2], hh + 4, nseg, reinterpret_cast<const Record *>(hh + 4 + nseg))) { perror(out_path); return 1; }
    return 0;
}

int main(int argc, char **argv)
{
    if (argc < 2) { fprintf(stderr, "usage: traceback_probe IN...\n"); return 1; }
    for (int a = 1; a < argc; ++a)
        if (const int st = run_one(argv[a], (std::string(argv[a]) + ".out").c_str())) return st;
    return 0;
}
