// traceback_kernels.cuh -- the traceback of a wave (main.cpp:217-267 through the sweep's 2-bit backpointers) and the
// compaction of its records.  sweep_kernels.cu runs them for every wave; tests/cuda/traceback_probe.cu runs them on
// their own, on tables the tests construct, so that the walk can be compared with a walker written from the reference.
// The kernels below are ordinary (non-inline) __global__ definitions: within libsd_b200.so only sweep_kernels.cu may
// include this header, or the link fails on duplicate symbols.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "common.h"

namespace sdb {

struct TbArgs {
    Geometry g;
    const uint32_t *codes; const int64_t *cta_code_off;
    const JR *jr; const int64_t *seg_j_off;
    const uint8_t *bases; const int64_t *seg_off; int nseg;
    const uint8_t *rows; const int *row_off;
    int ins, del, mismatch, match;
    Record *scratch; const int64_t *seg_rec_off; int *counts;
    const int *rank2row;    // --ed_thr pre-filter: [segment][rank] -> row of the full set, or null
    int *error;             // set to 1 when a jump names a row outside the monomer set (SD_MSG_TB_BAD_ROW)
    int invC;               // ceil(65536 / C): pos / C == (pos * invC) >> 16 for every pos < C*T (checked on the host)
};

// Warp-cooperative traceback (reference main.cpp:217-267 through the 2-bit backpointers; same state machine as
// sweep_core.cuh: traceback_segment, which the host emulator runs).
// One warp per segment.  Lane d of the warp owns column i0-d of a 32-column window and keeps, in registers, the
// three consecutive backpointer words around the cell the diagonal through the current position predicts.  Every
// round all lanes decode "their" cell on that diagonal at once; a ballot finds the first column whose move is not
// diagonal, the walk jumps over the whole diagonal run, and only the odd move (deletion, insertion, close, k==0)
// is handled serially.  Windows further down the diagonal are fetched ahead with cp.async (see TB_RING).
constexpr int TB_WARPS = 4;
__global__ void __launch_bounds__(TB_WARPS * 32) traceback_kernel(const TbArgs a)
{
    const int s = blockIdx.x * TB_WARPS + (threadIdx.x >> 5);
    if (s >= a.nseg) return;
    const int lane = threadIdx.x & 31;
    const Geometry g = a.g;
    const int cta0 = g.NG > 1 ? s * g.NG : s / g.NS, seg_local = g.NG > 1 ? 0 : s % g.NS;
    const int64_t o = a.seg_off[s];
    const int n = (int)(a.seg_off[s + 1] - o);
    const uint8_t *seg = a.bases + o;
    const JR *jr = a.jr + a.seg_j_off[s];
    const size_t cstride = (size_t)g.NT * g.CW;
    const int C = g.C, CW = g.CW, cshift = g.packed ? 3 : 4, cpw = 1 << cshift, invC = a.invC;
    const int maxwl = g.T * CW - 1;
    Record *out = a.scratch + a.seg_rec_off[s];

    // walk state (warp-uniform)
    const int *r2r = a.rank2row ? a.rank2row + (size_t)s * (2 * g.M) : nullptr;
    // the row of a jump comes from the sweep's column key: one outside the DP rows is reported, not used as an index
    auto row_of = [&](int kr) { return (unsigned)kr >= (unsigned)(2 * g.M) ? -1 : r2r ? r2r[kr] : kr; };
    int i = n - 1;
    int r = row_of(jr[n].row);
    if (r < 0) {
        if (lane == 0) { *a.error = 1; a.counts[s] = 0; }
        return;
    }
    int last = a.row_off[r + 1] - a.row_off[r] - 1;
    int k = last, end = i, end_score = jr[n].j, cnt = 0;
    // Window (per lane): the three words around this lane's cell, and a ring of look-ahead windows further down the
    // same diagonal (columns i0-32j-lane).  A clean 32-column window is consumed in ~150 cycles, a tenth of an HBM
    // round trip, and the backpointers left L2 long ago, so the walk is bound by how many windows one round trip
    // brings in.  A refill therefore fetches TB_RING windows at once -- for a 171-bp monomer the whole row -- with
    // cp.async into shared memory: unlike a register ring, nothing touches the data (and stalls on it) before the
    // window is adopted.  Every lane reads back only what it copied itself, so no barrier is involved.
    constexpr int TB_RING = 8;
    __shared__ uint32_t s_ring[TB_WARPS][TB_RING][4][32];          // [.][.][0..2] words, [3] = word base | valid << 31
    uint32_t (*ring)[4][32] = s_ring[threadIdx.x >> 5];
    int i0 = -1000, row0 = -1, half = 0, ni0 = -2000, cur = 0;
    uint32_t w0 = 0, w1 = 0, w2 = 0; int wb = 0; bool colok = false;
    const uint32_t *rowbase = nullptr;                  // first word of the current row's slot in column 0
    auto issue_window = [&](int slot, int iw, int kw) {
        const int c = iw - lane;
        const bool xok = c >= 0 && kw >= 1;             // kw < 1: the window lies before the start of the row
        int xb = 0;
        if (xok) {
            const int kp = max(kw - lane, 0);
            const int t = (kp * invC) >> 16;
            const int wl = t * CW + ((kp - t * C) >> cshift);
            xb = min(max(wl - 1, 0), max(maxwl - 2, 0));
            const uint32_t *col = rowbase + (size_t)c * cstride;
            const uint32_t d0 = (uint32_t)__cvta_generic_to_shared(&ring[slot][0][lane]);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0), "l"(col + xb) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0 + 128u), "l"(col + min(xb + 1, maxwl)) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d0 + 256u), "l"(col + min(xb + 2, maxwl)) : "memory");
        }
        ring[slot][3][lane] = (uint32_t)xb | (xok ? 0x80000000u : 0u);
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    for (;;) {
        if (k == 0) {
            // k == 0: the insertion equality is tested although the forward pass never takes that move (main.cpp:245
            // vs :194); decide it from J and the symbols involved, else close the alignment (main.cpp:252-262)
            bool ins_move = false;
            if (i != 0) {
                const uint8_t m0 = a.rows[a.row_off[r]];
                const int s_here = m0 == seg[i] ? a.match : a.mismatch;
                const int s_prev = m0 == seg[i - 1] ? a.match : a.mismatch;
                const int h_here = jr[i].j + s_here;
                const int h_prev = (i == 1) ? s_prev : jr[i - 1].j + s_prev;
                ins_move = (h_here == h_prev + a.ins);
            }
            if (ins_move) { --i; continue; }
        } else {
            if (r != row0 || i > i0 || i <= i0 - 32) {
                if (r == row0 && i == ni0) {
                    // the walk ran straight into the next window of the ring: adopt it (if the path drifted out of its
                    // three words the decode below notices and forces a refill) and reuse the freed slot for the
                    // window TB_RING-1 further down
                    i0 = ni0;
                    const int freed = cur;
                    cur = cur + 1 == TB_RING ? 0 : cur + 1;
                    issue_window(freed, i0 - 32 * (TB_RING - 1), k - 32 * (TB_RING - 1));
                } else {
                    // refill: lane d fetches the words around cell k-d of column i-d, and of the windows behind it
                    i0 = i; row0 = r;
                    const RowPlace pl = place_row(g, seg_local, r);
                    half = pl.half;
                    rowbase = a.codes + a.cta_code_off[cta0 + (g.NG > 1 ? pl.grp : 0)] + (size_t)lane_tid(g.T, pl.ginst, 0) * CW;
                    asm volatile("cp.async.wait_all;" ::: "memory");     // nothing of an abandoned ring may land later
                    cur = 0;
#pragma unroll
                    for (int j = 0; j < TB_RING; ++j) issue_window(j, i - 32 * j, k - 32 * j);
                }
                ni0 = i0 - 32;
                asm volatile("cp.async.wait_group %0;" ::"n"(TB_RING - 1) : "memory");
                w0 = ring[cur][0][lane]; w1 = ring[cur][1][lane]; w2 = ring[cur][2][lane];
                const uint32_t meta = ring[cur][3][lane];
                wb = (int)(meta & 0x7fffffffu); colok = (meta >> 31) != 0;
            }
            const int dcur = i0 - i;
            const int kd = k - (lane - dcur);
            bool ok = colok && lane >= dcur && kd >= 1;
            int code = 2;
            {
                const int kq = max(kd, 0);
                const int t = (kq * invC) >> 16;
                const int kk = kq - t * C;
                const int wi = kk >> cshift;
                const int rel = t * CW + wi - wb;
                ok = ok && (unsigned)rel < 3u;
                const uint32_t w = rel == 0 ? w0 : rel == 1 ? w1 : w2;
                const int cc = kk & (cpw - 1);
                const int ncell = min(cpw, C - (wi << cshift));
                code = decode_code(w, g.packed, ncell, cc, half);
            }
            const bool stop = lane >= dcur && (!ok || code != 2);
            const unsigned ball = __ballot_sync(0xffffffffu, stop);
            const int f = ball ? __ffs(ball) - 1 : 32;
            const int steps = f - dcur;                       // diagonal moves (main.cpp:249-250)
            i -= steps; k -= steps;
            if (f == 32) continue;                            // ran off the window: refill at the top
            const int okf = __shfl_sync(0xffffffffu, (int)ok, f);
            const int codef = __shfl_sync(0xffffffffu, code, f);
            if (!okf) {
                if (k >= 1) row0 = -1;                        // cell outside the cached words: force a refill
                continue;                                     // (k == 0 is handled at the top)
            }
            if (codef == 0) { --k; continue; }                // deletion (main.cpp:242-243)
            if (codef == 1) { --i; continue; }                // insertion (main.cpp:245-246)
        }
        // close the alignment (main.cpp:252-262)
        if (cnt >= n) { cnt = -1; break; }
        Record rec;
        rec.row = r; rec.start = i; rec.end = end;
        if (i == 0) { rec.score = end_score; if (lane == 0) out[cnt] = rec; ++cnt; break; }
        const JR ji = jr[i];
        rec.score = end_score - ji.j;
        if (lane == 0) out[cnt] = rec;
        ++cnt;
        end_score = ji.j;
        r = row_of(ji.row);
        if (r < 0) {
            if (lane == 0) *a.error = 1;
            cnt = 0;
            break;
        }
        --i;
        last = a.row_off[r + 1] - a.row_off[r] - 1;
        k = last; end = i;
    }
    if (lane == 0) a.counts[s] = cnt;
}

// Compaction of the per-segment records into one dense array (in segment order, each segment reversed: main.cpp:268)
// plus the total, so that one device->host copy brings a whole wave back.  One CTA: the exclusive prefix of the counts
// is formed chunk by chunk with a block scan, then every warp copies segments.
//   dense[prefix[s] + x] = scratch[seg_rec_off[s] + cnt[s]-1-x];   *total = sum of counts, or -1 if a traceback overflowed
__global__ void __launch_bounds__(1024) gather_kernel(const Record *scratch, const int64_t *seg_rec_off, const int *counts, Record *dense,
                                                      int nseg, int *total)
{
    __shared__ int s_warp[32];
    __shared__ int s_base, s_bad;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_base = 0; s_bad = 0; }
    __syncthreads();
    for (int c0 = 0; c0 < nseg; c0 += 1024) {
        const int s = c0 + tid;
        const int c = s < nseg ? counts[s] : 0;
        if (c < 0) s_bad = 1;
        int v = c < 0 ? 0 : c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) v += o; }
        if (lane == 31) s_warp[warp] = v;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += o; }
            s_warp[lane] = w;
        }
        __syncthreads();
        const int start = s_base + (warp ? s_warp[warp - 1] : 0) + v - (c < 0 ? 0 : c);     // exclusive prefix of segment s
        // every thread copies its own segment (a few dozen 16-byte records)
        if (s < nseg && c > 0) {
            const Record *src = scratch + seg_rec_off[s];
            Record *dst = dense + start;
            for (int x = 0; x < c; ++x) dst[x] = src[c - 1 - x];
        }
        __syncthreads();
        if (tid == 0) s_base += s_warp[31];
        __syncthreads();
    }
    if (tid == 0) *total = s_bad ? -1 : s_base;
}

// The traceback of the t.nseg segments of a wave, asynchronous on `stream`; t.invC is set here.  Throws PlanError when the
// reciprocal division of the geometry is not exact; returns the launch error.
inline cudaError_t launch_traceback(TbArgs t, cudaStream_t stream)
{
    const Geometry &g = t.g;
    t.invC = (65536 + g.C - 1) / g.C;
    for (int pos = 0; pos < g.C * g.T; ++pos)
        if (((pos * t.invC) >> 16) != pos / g.C) throw PlanError{"internal: reciprocal division inexact"};
    traceback_kernel<<<(t.nseg + TB_WARPS - 1) / TB_WARPS, TB_WARPS * 32, 0, stream>>>(t);
    return cudaGetLastError();
}

} // namespace sdb
