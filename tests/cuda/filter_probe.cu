// filter_probe.cu -- runs the --ed_thr pre-filter kernels (filter_kernels.cuh: launch_filter) on inputs from a file and
// writes their tables, so that tests/test_batch_scale.py can compare them with the oracle entry by entry.
//
//   filter_probe IN OUT
// IN (little-endian): int32 nseg, R, ed_thr, with_kj; int64 seg_off[nseg+1]; int32 row_off[R+1]; the segments' bytes;
//                     the rows' bytes (ASCII); int32 kjbase[R][5] if with_kj
// OUT:                int32 dist[nseg][R], rank_of_row[nseg][R], row_of_rank[nseg][R], seg_kj[nseg][5]
// Every output word starts as 0x7f7f7f7f, so an entry the kernels never write is visible.
#include <cstdio>
#include <cstring>
#include <vector>

#include "filter_kernels.cuh"

#define CK(x)                                                                                        \
    do {                                                                                             \
        cudaError_t e_ = (x);                                                                        \
        if (e_ != cudaSuccess) { fprintf(stderr, "%s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); return 3; } \
    } while (0)

template <class T> static bool get(FILE *f, T *p, size_t n) { return fread(p, sizeof(T), n, f) == n; }

template <class T> static cudaError_t to_device(const std::vector<T> &h, T **d)
{
    cudaError_t e = cudaMalloc(d, h.size() * sizeof(T) + 16);
    if (e == cudaSuccess && !h.empty()) e = cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
    return e;
}

int main(int argc, char **argv)
{
    if (argc != 3) { fprintf(stderr, "usage: filter_probe IN OUT\n"); return 1; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 1; }
    int hdr[4];
    if (!get(f, hdr, 4)) { fprintf(stderr, "short header\n"); return 1; }
    const int nseg = hdr[0], R = hdr[1], ed_thr = hdr[2], with_kj = hdr[3];
    std::vector<int64_t> seg_off((size_t)nseg + 1);
    std::vector<int> row_off((size_t)R + 1);
    bool ok = get(f, seg_off.data(), seg_off.size()) && get(f, row_off.data(), row_off.size());
    std::vector<uint8_t> bases(ok ? (size_t)seg_off[nseg] : 0), rows(ok ? (size_t)row_off[R] : 0);
    std::vector<int> kjbase(with_kj ? (size_t)R * 5 : 0);
    ok = ok && get(f, bases.data(), bases.size()) && get(f, rows.data(), rows.size()) && get(f, kjbase.data(), kjbase.size());
    fclose(f);
    if (!ok) { fprintf(stderr, "short input\n"); return 1; }
    int Lmax = 0, nmax = 0;
    for (int r = 0; r < R; ++r) Lmax = std::max(Lmax, row_off[r + 1] - row_off[r]);
    for (int s = 0; s < nseg; ++s) nmax = std::max(nmax, (int)(seg_off[s + 1] - seg_off[s]));

    uint8_t *d_bases, *d_rows; int64_t *d_segoff; int *d_rowoff, *d_kj = nullptr;
    CK(to_device(bases, &d_bases)); CK(to_device(rows, &d_rows)); CK(to_device(seg_off, &d_segoff)); CK(to_device(row_off, &d_rowoff));
    if (with_kj) CK(to_device(kjbase, &d_kj));
    const size_t np = (size_t)nseg * R, nout = 3 * np + (size_t)nseg * 5;
    int *d_out;
    CK(cudaMalloc(&d_out, nout * 4));
    CK(cudaMemset(d_out, 0x7f, nout * 4));
    cudaStream_t st;
    CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CK(sdb::launch_filter(d_bases, d_segoff, nseg, nmax, d_rows, d_rowoff, R, Lmax, ed_thr, d_kj, d_out, d_out + np, d_out + 2 * np,
                          d_out + 3 * np, st));
    CK(cudaStreamSynchronize(st));
    std::vector<int> out(nout);
    CK(cudaMemcpy(out.data(), d_out, nout * 4, cudaMemcpyDeviceToHost));
    cudaStreamDestroy(st);
    cudaFree(d_out); cudaFree(d_bases); cudaFree(d_rows); cudaFree(d_segoff); cudaFree(d_rowoff); cudaFree(d_kj);
    FILE *g = fopen(argv[2], "wb");
    if (!g || fwrite(out.data(), 4, nout, g) != nout) { perror(argv[2]); return 1; }
    fclose(g);
    return 0;
}
