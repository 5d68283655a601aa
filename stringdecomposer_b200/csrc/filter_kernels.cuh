// filter_kernels.cuh -- the --ed_thr pre-filter on the device (FilterMonomersForRead, main.cpp:135-149): the infix edit
// distance of every DP row against every segment of a wave, then per segment the ranks of the rows and the kept list.
// sweep_kernels.cu runs it for every wave; tests/cuda/filter_probe.cu runs it on its own so that the tests can compare
// its tables with the oracle directly.  The kernels below are ordinary (non-inline) __global__ definitions: within
// libsd_b200.so only sweep_kernels.cu may include this header, or the link fails on duplicate symbols.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cstdint>

#include "common.h"

namespace sdb {

// Step 1: infix edit distance of every DP row against every staged segment.  Generic form: one thread per pair, state
// in local memory (rows of up to 1536 symbols).
__global__ void hw_distance_kernel(const uint8_t *bases, const int64_t *seg_off, int nseg, const uint8_t *rows, const int *row_off,
                                   int R, int *dist)
{
    const int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= (int64_t)nseg * R) return;
    const int s = (int)(x / R), r = (int)(x - (int64_t)s * R);
    dist[x] = hw_distance(rows + row_off[r], row_off[r + 1] - row_off[r], bases + seg_off[s], (int)(seg_off[s + 1] - seg_off[s]));
}

// The same for rows of at most 64*NB symbols (NB <= 4: alpha-satellite monomers need 3): a CTA takes one segment and 128
// rows, one row per thread.  The segment's symbols pass through shared memory in tiles of HWF_TILE (one barrier per tile,
// so a segment of any length fits) and are broadcast; the match masks of the CTA's rows live in shared memory as
// [symbol][word][thread] (conflict-free 8-byte loads); the Myers/Hyyro column state stays in registers.  Same recurrence
// as sweep_core.cuh: hw_distance (edlib's HW mode, distance only).
constexpr int HWF_ROWS = 128;
constexpr int HWF_TILE = 4096;
template <int NB>
__global__ void __launch_bounds__(HWF_ROWS) hw_distance_rows_kernel(const uint8_t *bases, const int64_t *seg_off, const uint8_t *rows,
                                                                    const int *row_off, int R, int *dist)
{
    extern __shared__ unsigned long long hwf_smem[];
    unsigned long long *peq = hwf_smem;                                  // [5][NB][HWF_ROWS]
    uint8_t *stext = reinterpret_cast<uint8_t *>(peq + 5 * NB * HWF_ROWS);     // [HWF_TILE]
    const int s = blockIdx.x, tid = threadIdx.x;
    const int r = blockIdx.y * HWF_ROWS + tid;
    const int64_t o = seg_off[s];
    const int n = (int)(seg_off[s + 1] - o);
#pragma unroll
    for (int q = 0; q < 5 * NB; ++q) peq[q * HWF_ROWS + tid] = 0ull;
    int m = 0;
    if (r < R) {
        const uint8_t *pat = rows + row_off[r];
        m = row_off[r + 1] - row_off[r];
        for (int i = 0; i < m; ++i) {
            const unsigned ch = pat[i];
            const int c = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : 4;
            peq[(c * NB + (i >> 6)) * HWF_ROWS + tid] |= 1ull << (i & 63);
        }
    }
    const int B = (m + 63) >> 6;
    unsigned long long pv[NB], mv[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) { pv[b] = ~0ull; mv[b] = 0ull; }
    const unsigned long long last_bit = 1ull << ((m - 1) & 63);
    int score = m, best = m;
    for (int j0 = 0; j0 < n; j0 += HWF_TILE) {
        const int len = min(HWF_TILE, n - j0);
        __syncthreads();                                                  // the previous tile is consumed (first: peq is built)
        for (int x = tid; x < len; x += HWF_ROWS) { const int c = ascii_code(bases[o + j0 + x]); stext[x] = (uint8_t)(c > 4 ? 4 : c); }
        __syncthreads();
        if (r >= R) continue;
        for (int j = 0; j < len; ++j) {
            const int c = stext[j];
            int hin = 0;
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                if (b < B) {
                    unsigned long long eq = peq[(c * NB + b) * HWF_ROWS + tid];
                    const unsigned long long p = pv[b], mm = mv[b];
                    const unsigned long long xv = eq | mm;
                    if (hin < 0) eq |= 1ull;
                    const unsigned long long xh = (((eq & p) + p) ^ p) | eq;
                    unsigned long long ph = mm | ~(xh | p);
                    unsigned long long mh = p & xh;
                    const unsigned long long top = (b == B - 1) ? last_bit : (1ull << 63);
                    const int hout = (ph & top) ? 1 : ((mh & top) ? -1 : 0);
                    ph <<= 1; mh <<= 1;
                    if (hin < 0) mh |= 1ull; else if (hin > 0) ph |= 1ull;
                    pv[b] = mh | ~(xv | ph);
                    mv[b] = ph & xv;
                    hin = hout;
                }
            }
            score += hin;
            best = min(best, score);
        }
    }
    if (r < R) dist[(size_t)s * R + r] = best;
}

// Step 2: per segment, the rows sorted by (distance, row); the closest row and every row within ed_thr are kept
// (main.cpp:141-147).  rank_of_row[r] = position in the kept list or -1; row_of_rank[pos] = r or -1.  The position is
// found by counting (R is at most 4096), so no sort and no trip to the host.  For the deferred-jump sweep the best
// jump-derived row-end key per symbol of the kept rows is formed on the way (plan.cpp: lat_jump_keys):
// kjbase[r][sym] = key of row r with tie-break index 0, the rank is subtracted here.
__global__ void __launch_bounds__(256) filter_rank_kernel(const int *dist, int R, int ed_thr, int *rank_of_row, int *row_of_rank,
                                                          const int *kjbase, int *seg_kj)
{
    extern __shared__ int frk_d[];
    __shared__ int s_kj[5];
    const int s = blockIdx.x, tid = threadIdx.x;
    const int *d = dist + (size_t)s * R;
    for (int r = tid; r < R; r += 256) frk_d[r] = d[r];
    if (tid < 5) s_kj[tid] = INT_MIN;
    __syncthreads();
    for (int r = tid; r < R; r += 256) {
        const int dr = frk_d[r];
        int pos = 0;
        for (int q = 0; q < R; ++q) { const int dq = frk_d[q]; pos += (dq < dr) || (dq == dr && q < r); }
        const bool keep = pos == 0 || dr <= ed_thr;
        rank_of_row[(size_t)s * R + r] = keep ? pos : -1;
        row_of_rank[(size_t)s * R + pos] = keep ? r : -1;
        if (keep && kjbase)
            for (int sym = 0; sym < 5; ++sym) atomicMax(&s_kj[sym], kjbase[r * 5 + sym] - pos);
    }
    __syncthreads();
    if (seg_kj && tid < 5) seg_kj[(size_t)s * 5 + tid] = s_kj[tid];
}

// Both steps for the nseg segments of a wave, asynchronous on `stream`.  Device pointers: bases/seg_off the segments
// (ASCII, offsets into bases), rows/row_off the R DP rows (ASCII), Lmax the longest row, nmax the longest segment.
// Outputs [nseg][R] dist, rank_of_row and row_of_rank; kjbase [R][5] and seg_kj [nseg][5] may be null (the deferred-jump
// sweep's keys).  Returns the first launch error.
inline cudaError_t launch_filter(const uint8_t *bases, const int64_t *seg_off, int nseg, int nmax, const uint8_t *rows, const int *row_off,
                                 int R, int Lmax, int ed_thr, const int *kjbase, int *dist, int *rank_of_row, int *row_of_rank,
                                 int *seg_kj, cudaStream_t stream)
{
    const size_t np = (size_t)nseg * R;
    const int NB = (Lmax + 63) / 64;
    if (NB <= 4) {
        const size_t smem = (size_t)5 * NB * HWF_ROWS * 8 + (size_t)std::min(HWF_TILE, (nmax + 16) / 16 * 16);
        const void *k = NB == 1 ? (const void *)hw_distance_rows_kernel<1> : NB == 2 ? (const void *)hw_distance_rows_kernel<2>
                      : NB == 3 ? (const void *)hw_distance_rows_kernel<3> : (const void *)hw_distance_rows_kernel<4>;
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        int Rv = R;
        void *args[] = {(void *)&bases, (void *)&seg_off, (void *)&rows, (void *)&row_off, (void *)&Rv, (void *)&dist};
        e = cudaLaunchKernel(k, dim3((unsigned)nseg, (unsigned)((R + HWF_ROWS - 1) / HWF_ROWS)), dim3(HWF_ROWS), args, smem, stream);
        if (e != cudaSuccess) return e;
    } else {
        hw_distance_kernel<<<(unsigned)((np + 63) / 64), 64, 0, stream>>>(bases, seg_off, nseg, rows, row_off, R, dist);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    filter_rank_kernel<<<(unsigned)nseg, 256, (size_t)R * 4, stream>>>(dist, R, ed_thr, rank_of_row, row_of_rank, kjbase, seg_kj);
    return cudaGetLastError();
}

} // namespace sdb
