// sweep_kernels.cu -- sm_100a kernels of the string-decomposition DP and the CUDA backend that drives them.
//
//   sweep_kernel<P,C,T>       (sweep_kernel.cuh) column-synchronous forward sweep, one CTA per NS segments.  Every DP row
//                             pair (Packed16: forward monomer + reverse complement in the two s16 halves of a register) or
//                             row (Scalar32) is a slot of T lanes x C cells held in registers.  Per column: chain-free
//                             candidates (DPX VIADDMNMX), windowed carry of the deletion chain across the lanes (warp
//                             shuffles), chain + 2-bit backpointers, per-segment max/argmax of the row ends on a
//                             (score,row) key (CREDUX + one shared-memory word per warp), one barrier.
//   sweep_group_kernel        the same for monomer sets that need several CTAs per segment (keys meet in global memory).
//   sweep_lat_kernel<P,C,T,W> (sweep_lat_kernel.cuh) deferred-jump form, one segment per thread-block cluster, keys
//                             exchanged through distributed shared memory one column ahead of their use.
//   traceback_kernel          walks the 2-bit backpointers (sweep_core.cuh: traceback_segment).
//   hw_distance_rows_kernel, filter_rank_kernel    (filter_kernels.cuh) the --ed_thr pre-filter (distances, ranks) on the device.
//   gather_kernel             compacts + reverses the per-segment records into the result block of a wave.
//   int_peak_kernel           integer-pipe issue-rate probe the roofline is quoted against.
// and the CUDA backend: two wave slots per device, streams for copy-in / sweep / traceback / copy-out.
//
// Reference semantics: stringdecomposer/src/main.cpp:151-270 (AlignPartClassicDP); see sweep_core.cuh.
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>      // header-only; ranges cost nothing unless a profiler is attached

#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "sweep_kernel.cuh"
#include "sweep_lat_kernel.cuh"
#include "filter_kernels.cuh"
#include "cuda_scope.h"
#include "block_cache.h"

namespace sdb {

#define SD_CUDA(x)                                                                                              \
    do {                                                                                                        \
        cudaError_t e_ = (x);                                                                                   \
        if (e_ != cudaSuccess) throw PlanError{std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " +  \
                                               __FILE__ + ":" + std::to_string(__LINE__)};                      \
    } while (0)

// ---------------------------------------------------------------------------------------------
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

// ---------------------------------------------------------------------------------------------
template <int MODE> __global__ void int_peak_kernel(unsigned *out, unsigned seed)
{
    unsigned r[8];
    const unsigned b = seed * 3u + threadIdx.x;
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = threadIdx.x * 17u + j * 1315423911u + seed;
    for (int it = 0; it < 2048; ++it) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const unsigned nb = r[(j + 1) & 7];
            if (MODE == 0) r[j] = __viaddmax_s16x2(r[j], b, nb);                       // ALU pipe only
            else { r[j] = __viaddmax_s16x2(r[j], b, nb); r[j] = r[j] * b + nb; }       // ALU + FMA(IMAD) pipes
        }
    }
    unsigned acc = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc ^= r[j];
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

// ---------------------------------------------------------------------------------------------
// The sweep kernel compiled for a geometry, or null.  fast, multi: the classic sweep's FAST and MULTI variants
// (sweep_kernel.cuh); timing: the instrumented twin of the deferred-jump sweep (SD_LAT_TIMING; packed, staged only).
static const void *sweep_kernel_for(const Geometry &g, bool fast, bool multi, bool timing)
{
    // [policy: s32, p16][variant: !FAST, FAST, FAST + MULTI][symbols: staged, streamed]
    static const SweepLookup classic[2][3][2] = {
        {{sweep_lookup_s32_f0_m0, sweep_lookup_s32_f0_m0_st}, {sweep_lookup_s32_f1_m0, sweep_lookup_s32_f1_m0_st},
         {sweep_lookup_s32_f1_m1, sweep_lookup_s32_f1_m1_st}},
        {{sweep_lookup_p16_f0_m0, sweep_lookup_p16_f0_m0_st}, {sweep_lookup_p16_f1_m0, sweep_lookup_p16_f1_m0_st},
         {sweep_lookup_p16_f1_m1, sweep_lookup_p16_f1_m1_st}}};
    // [policy]
    static const SweepLookup group[2] = {sweep_group_lookup_s32, sweep_group_lookup_p16};
    // [policy][symbols]
    static const SweepLookup lat[2][2] = {{sweep_lat_lookup_s32, sweep_lat_lookup_s32_st}, {sweep_lat_lookup_p16, sweep_lat_lookup_p16_st}};
    const int pol = g.packed ? 1 : 0, st = g.stream ? 1 : 0;
    if (g.lat && timing) return pol && !st ? sweep_lat_timing_lookup_p16(g) : nullptr;
    if (g.lat) return lat[pol][st](g);
    if (g.NG > 1) return group[pol](g);
    return classic[pol][fast ? (multi ? 2 : 1) : 0][st](g);
}

namespace {

struct DevBuf {
    void *p = nullptr; size_t cap = 0; int dev = -1;
    void release()
    {
        if (!p) return;
        if (!BlockCache::get().give(BlockCache::Device, dev, p, cap)) cudaFree(p);
        p = nullptr; cap = 0;
    }
    void need(size_t bytes)
    {
        if (bytes <= cap) return;
        if (p) { cudaDeviceSynchronize(); release(); }       // nothing in flight may still use the old block (cudaFree used to imply this)
        const size_t want = bytes + bytes / 8 + 256;
        int d = 0;
        SD_CUDA(cudaGetDevice(&d));
        size_t got = 0;
        void *q = BlockCache::get().take(BlockCache::Device, d, want, &got);
        if (!q) {
            if (cudaMalloc(&q, want) != cudaSuccess) {
                cudaGetLastError();
                for (void *old : BlockCache::get().flush(BlockCache::Device, d)) cudaFree(old);
                SD_CUDA(cudaMalloc(&q, want));
            }
            got = want;
        }
        p = q; cap = got; dev = d;
    }
    template <class U> U *as() { return reinterpret_cast<U *>(p); }
    ~DevBuf() { release(); }
};
struct PinnedBuf {          // page-locked host memory: the result block of a wave lands here with one asynchronous copy
    void *p = nullptr; size_t cap = 0; int dev = -1;
    void release()
    {
        if (!p) return;
        if (!BlockCache::get().give(BlockCache::Pinned, dev, p, cap)) cudaFreeHost(p);
        p = nullptr; cap = 0;
    }
    void need(size_t bytes)
    {
        if (bytes <= cap) return;
        if (p) { cudaDeviceSynchronize(); release(); }
        const size_t want = bytes + bytes / 4 + 4096;
        int d = 0;
        SD_CUDA(cudaGetDevice(&d));
        size_t got = 0;
        void *q = BlockCache::get().take(BlockCache::Pinned, d, want, &got);
        if (!q) {
            if (cudaHostAlloc(&q, want, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                for (void *old : BlockCache::get().flush(BlockCache::Pinned, d)) cudaFreeHost(old);
                SD_CUDA(cudaHostAlloc(&q, want, cudaHostAllocDefault));
            }
            got = want;
        }
        p = q; cap = got; dev = d;
    }
    template <class U> U *as() { return reinterpret_cast<U *>(p); }
    ~PinnedBuf() { release(); }
};
struct MetaView { void *p = nullptr; template <class U> U *as() { return reinterpret_cast<U *>(p); } };

// Result block of a wave in device memory: header, per-segment counts, then the dense records.
//   int32 flag[2] (bad symbol, exchange time-out), int32 total, int32 traceback row error, int32 counts[nseg] (padded to
//   16 B), Record dense[]
constexpr size_t OUT_HDR = 16;
inline size_t out_counts_bytes(int nseg) { return ((size_t)nseg * 4 + 15) & ~size_t(15); }
// Checks the header's flags (the first error in this order is reported) and returns the record total
inline int64_t wave_total(const int *hdr)
{
    if (hdr[1]) throw PlanError{"CUDA: sweep timed out waiting for a partner CTA (internal error)"};
    if (hdr[3]) throw PlanError{SD_MSG_TB_BAD_ROW};
    if (hdr[0]) throw PlanError{"segment contains a symbol outside ACGTN"};
    if (hdr[2] < 0) throw PlanError{"traceback overflowed its record buffer (internal error)"};
    return hdr[2];
}

// One wave in flight: its device buffers, its layout and its events.  Two slots per device let the host->device copy of
// wave w+1 and the device->host copy of wave w-1 run while wave w computes (three streams: in, compute, out).
struct WaveSlot {
    DevBuf d_bases, d_meta, d_codes, d_jr, d_scratch, d_out, d_dist, d_rank, d_r2r, d_segkj, d_xchg, d_dbg;
    MetaView d_segoff, d_ctanmax, d_ctacode, d_segj, d_segrec;     // slices of d_meta
    PinnedBuf h_out;
    std::vector<char> hmeta;
    std::vector<int64_t> hoff;
    CtaLayout lay;
    int s0 = 0, s1 = 0, nseg = 0, nmax = 0;
    bool filter_on = false, staged = false;
    size_t nb = 0, rec_guess = 0;
    int end_idx = -1, prev_end = -1;      // this wave's and its predecessor's entry in the backend's ring of sweep-end events
    cudaEvent_t ev[7]{};            // 0 h2d begin, 1 h2d end, 2 sweep begin, 3 sweep end, 4 traceback end, 5 d2h end, 6 traceback begin
};

class CudaBackend : public Backend {
public:
    explicit CudaBackend(int dev) : dev_(dev)
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        SD_CUDA(cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking));
        SD_CUDA(cudaStreamCreateWithFlags(&st_in_, cudaStreamNonBlocking));
        SD_CUDA(cudaStreamCreateWithFlags(&st_out_, cudaStreamNonBlocking));
        SD_CUDA(cudaStreamCreateWithFlags(&st_tb_, cudaStreamNonBlocking));
        SD_CUDA(cudaStreamCreateWithFlags(&st2_, cudaStreamNonBlocking));
        for (auto &w : slot_) for (auto &e : w.ev) SD_CUDA(cudaEventCreate(&e));
        for (auto &e : endev_) SD_CUDA(cudaEventCreate(&e));
        SD_CUDA(cudaGetDeviceProperties(&prop_, dev_));
        if (prop_.major != 10) throw PlanError{"CUDA device is not sm_100 class: this library carries sm_100a code only (no PTX for other architectures)"};
        size_t fr = 0, tot = 0;
        SD_CUDA(cudaMemGetInfo(&fr, &tot));
        free_at_start_ = (int64_t)fr;
        budget_ = std::min<int64_t>((int64_t)(fr * 0.85), (int64_t)96 << 30);
    }
    ~CudaBackend() override
    {
        DeviceScope scope_(dev_);
        cudaDeviceSynchronize();          // the blocks of this backend go back to the process-wide cache: nothing may still use them
        for (auto &w : slot_) for (auto &e : w.ev) cudaEventDestroy(e);
        for (auto &e : endev_) cudaEventDestroy(e);
        cudaStreamDestroy(st2_);
        cudaStreamDestroy(st_); cudaStreamDestroy(st_in_); cudaStreamDestroy(st_out_); cudaStreamDestroy(st_tb_);
    }
    const char *name() const override { return "cuda"; }

    void configure(const Plan &p, const MonomerSet &ms) override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        plan_ = p; ms_ = ms;
        const Geometry &g = p.g;
        const int spw = 32 / g.T;
        fast_ = (g.nslots % spw == 0) && (g.nslots / spw <= 4) && g.NS <= 15;     // 15 named barriers besides barrier 0
        if (getenv("SD_NOFAST")) fast_ = false;
        lat_timing_ = g.lat && getenv("SD_LAT_TIMING") && sweep_kernel_for(g, fast_, false, true);
        kernel_ = sweep_kernel_for(g, fast_, fast_ && g.NS > 1, lat_timing_);
        if (g.lat && (g.NT / 32) * g.NG > 32) throw PlanError{"internal: a deferred-jump cluster holds at most 32 warps"};
        if (!kernel_) throw PlanError{"no sweep kernel compiled for this geometry"};
        cudaFuncAttributes fa;
        SD_CUDA(cudaFuncGetAttributes(&fa, kernel_));
        // registers are handed out per warp in units of 8 per thread
        const int nthreads = g.NT * (g.NG > 1 && !g.lat ? g.NS : 1);
        if ((int64_t)((fa.numRegs + 7) / 8 * 8) * nthreads > 65536 || fa.maxThreadsPerBlock < nthreads)
            throw PlanError{"sweep geometry exceeds the register file (regs*threads > 64K)"};
        const std::vector<uint32_t> &table = g.lat ? p.prof2 : p.prof;
        d_prof_.need(table.size() * 4);
        SD_CUDA(cudaMemcpyAsync(d_prof_.p, table.data(), table.size() * 4, cudaMemcpyHostToDevice, st_));
        d_slotlen_.need(p.slot_len.size() * 4); d_slotend_.need(p.slot_endadd.size() * 4);
        SD_CUDA(cudaMemcpyAsync(d_slotlen_.p, p.slot_len.data(), p.slot_len.size() * 4, cudaMemcpyHostToDevice, st_));
        SD_CUDA(cudaMemcpyAsync(d_slotend_.p, p.slot_endadd.data(), p.slot_endadd.size() * 4, cudaMemcpyHostToDevice, st_));
        d_rows_.need(ms.rows.size()); d_rowoff_.need(ms.row_off.size() * 4);
        rows_ascii_.resize(ms.rows.size());           // the traceback compares row and segment symbols as text
        for (size_t x = 0; x < ms.rows.size(); ++x) rows_ascii_[x] = (uint8_t)"ACGTN"[ms.rows[x]];
        SD_CUDA(cudaMemcpyAsync(d_rows_.p, rows_ascii_.data(), rows_ascii_.size(), cudaMemcpyHostToDevice, st_));
        SD_CUDA(cudaMemcpyAsync(d_rowoff_.p, ms.row_off.data(), ms.row_off.size() * 4, cudaMemcpyHostToDevice, st_));
        if (g.lat) {
            // per row and symbol: the key of its best jump-derived row end with tie-break index 0 (plan.cpp: lat_jump_keys);
            // the --ed_thr pre-filter subtracts the row's rank on the device
            const int R = ms.nrows();
            kjbase_.assign((size_t)R * 5, 0);
            std::vector<int> one((size_t)R, -1);
            for (int r = 0; r < R; ++r) {
                one[(size_t)r] = 0;
                lat_jump_keys(ms, p.sc, one.data(), kjbase_.data() + (size_t)r * 5);
                one[(size_t)r] = -1;
            }
            d_kjbase_.need(kjbase_.size() * 4);
            SD_CUDA(cudaMemcpyAsync(d_kjbase_.p, kjbase_.data(), kjbase_.size() * 4, cudaMemcpyHostToDevice, st_));
        }
        SD_CUDA(cudaStreamSynchronize(st_));
    }

    int64_t wave_bytes(const Batch &b, int s0, int s1) const override
    {
        CtaLayout l = make_cta_layout(plan_, b, s0, s1);
        int64_t bytes = l.cta_code_off.back() * 4 + l.seg_j_off.back() * 8 + l.seg_rec_off.back() * 32 + (b.off[s1] - b.off[s0]);
        if (ed_thr_ >= 0) bytes += (int64_t)(s1 - s0) * ms_.nrows() * 12;      // pre-filter tables: distance, rank, rank -> row
        return bytes;
    }
    int64_t wave_budget() const override
    {
        if (const char *e = getenv("SD_WAVE_BYTES")) if (atoll(e) > 0) return atoll(e);
        return budget_;        // 85 % of the memory that was free when the backend was created (cudaMemGetInfo costs ms)
    }
    int64_t device_bytes() const override { return free_at_start_; }
    int wave_slots() const override { return 2; }

    // Buffers of a slot sized for the largest wave it will see: growing them later would mean cudaFree (a device-wide
    // synchronisation) in the middle of the pipeline.
    void reserve(int slot, const Batch &b, int s0, int s1) override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        WaveSlot &w = slot_[slot & 1];
        const CtaLayout lay = make_cta_layout(plan_, b, s0, s1);
        const int nseg = s1 - s0;
        w.d_bases.need((size_t)(b.off[s1] - b.off[s0]) + 16);
        w.d_codes.need((size_t)lay.cta_code_off.back() * 4 + 16);
        w.d_jr.need((size_t)lay.seg_j_off.back() * sizeof(JR) + 16);
        w.d_scratch.need((size_t)lay.seg_rec_off.back() * sizeof(Record) + 16);
        w.d_out.need(OUT_HDR + out_counts_bytes(nseg) + (size_t)lay.seg_rec_off.back() * sizeof(Record) + 64);
        w.h_out.need(OUT_HDR + out_counts_bytes(nseg) + ((size_t)(b.off[s1] - b.off[s0]) / 48 + (size_t)nseg * 4 + 64) * sizeof(Record));
    }

    // ---- the three stages of a wave, each asynchronous on its own stream ----------------------------------------
    void enqueue_h2d(WaveSlot &w, const Batch &b, int s0, int s1)
    {
        w.s0 = s0; w.s1 = s1; w.nseg = s1 - s0;
        w.lay = make_cta_layout(plan_, b, s0, s1);
        w.nmax = 0;
        for (int v : w.lay.cta_nmax) w.nmax = std::max(w.nmax, v);
        // inputs: bases of [s0,s1) and their offsets rebased to the staged buffer
        const int64_t base = b.off[s0];
        w.nb = (size_t)(b.off[s1] - base);
        w.hoff.resize((size_t)w.nseg + 1);
        for (int s = 0; s <= w.nseg; ++s) w.hoff[s] = b.off[s0 + s] - base;
        w.d_bases.need(w.nb + 16);
        // the five small per-wave tables travel as one block
        const size_t msz[5] = {w.hoff.size() * 8, w.lay.cta_nmax.size() * 4, w.lay.cta_code_off.size() * 8, w.lay.seg_j_off.size() * 8,
                               w.lay.seg_rec_off.size() * 8};
        const void *msrc[5] = {w.hoff.data(), w.lay.cta_nmax.data(), w.lay.cta_code_off.data(), w.lay.seg_j_off.data(), w.lay.seg_rec_off.data()};
        MetaView *mdst[5] = {&w.d_segoff, &w.d_ctanmax, &w.d_ctacode, &w.d_segj, &w.d_segrec};
        size_t mtotal = 0, moff[5];
        for (int x = 0; x < 5; ++x) { moff[x] = mtotal; mtotal += (msz[x] + 255) & ~size_t(255); }
        w.d_meta.need(mtotal + 16);
        w.hmeta.resize(mtotal);
        for (int x = 0; x < 5; ++x) { memcpy(w.hmeta.data() + moff[x], msrc[x], msz[x]); mdst[x]->p = w.d_meta.as<char>() + moff[x]; }
        w.d_codes.need((size_t)w.lay.cta_code_off.back() * 4 + 16);
        w.d_jr.need((size_t)w.lay.seg_j_off.back() * sizeof(JR) + 16);
        w.d_scratch.need((size_t)w.lay.seg_rec_off.back() * sizeof(Record) + 16);
        // result block: counts + a guess of the dense records (an alignment per ~64 columns plus slack); fetch copies the
        // rest in a second step in the rare case the guess was too small
        w.rec_guess = (size_t)(w.nb / 48) + (size_t)w.nseg * 4 + 64;
        w.d_out.need(OUT_HDR + out_counts_bytes(w.nseg) + (size_t)w.lay.seg_rec_off.back() * sizeof(Record) + 64);
        SD_CUDA(cudaEventRecord(w.ev[0], st_in_));
        SD_CUDA(cudaMemcpyAsync(w.d_bases.p, b.text + base, w.nb, cudaMemcpyHostToDevice, st_in_));
        SD_CUDA(cudaMemcpyAsync(w.d_meta.p, w.hmeta.data(), mtotal, cudaMemcpyHostToDevice, st_in_));
        SD_CUDA(cudaMemsetAsync(w.d_out.p, 0, OUT_HDR, st_in_));
        SD_CUDA(cudaEventRecord(w.ev[1], st_in_));
        h2d_bytes += (int64_t)(w.nb + mtotal);
        w.filter_on = ed_thr_ >= 0;
        if (w.filter_on) build_filter(w);
        w.staged = true;
    }

    // FilterMonomersForRead (main.cpp:135-149): distances, ranks and (deferred-jump sweep) the per-segment jump keys, all
    // on the device and all asynchronous on the copy-in stream
    void build_filter(WaveSlot &w)
    {
        const int R = ms_.nrows();
        const size_t np = (size_t)w.nseg * R;
        w.d_dist.need(np * 4); w.d_rank.need(np * 4); w.d_r2r.need(np * 4);
        int *segkj = nullptr;
        if (plan_.g.lat) { w.d_segkj.need((size_t)w.nseg * 5 * 4); segkj = w.d_segkj.as<int>(); }
        SD_CUDA(launch_filter(w.d_bases.as<uint8_t>(), w.d_segoff.as<int64_t>(), w.nseg, w.nmax, d_rows_.as<uint8_t>(), d_rowoff_.as<int>(),
                              R, ms_.Lmax, ed_thr_, plan_.g.lat ? d_kjbase_.as<int>() : nullptr, w.d_dist.as<int>(), w.d_rank.as<int>(),
                              w.d_r2r.as<int>(), segkj, st_in_));
        SD_CUDA(cudaEventRecord(w.ev[1], st_in_));
        launches += 2;
    }

    // the argument fields that SweepArgs, GroupArgs and LatArgs share
    template <class A> void fill_common_args(A &a, WaveSlot &w)
    {
        const Geometry &g = plan_.g;
        a.bases = w.d_bases.as<uint8_t>(); a.seg_off = w.d_segoff.as<int64_t>(); a.nseg = w.nseg;
        a.cta_code_off = w.d_ctacode.as<int64_t>(); a.seg_j_off = w.d_segj.as<int64_t>();
        a.codes = w.d_codes.as<uint32_t>(); a.jr = w.d_jr.as<JR>();
        a.slot_len = d_slotlen_.as<int>(); a.slot_endadd = d_slotend_.as<int>();
        a.nslots = g.nslots; a.M = g.M; a.NT = g.NT; a.CW = g.CW;
        a.ins = plan_.sc.ins; a.del = plan_.sc.del; a.deadz = plan_.deadz;
        a.tr = g.packed ? tag_regs<Packed16>() : tag_regs<Scalar32>();
        a.bad_symbol = w.d_out.as<int>();
        a.rank = w.filter_on ? w.d_rank.as<int>() : nullptr;
    }

    void launch_single(WaveSlot &w, int seg_stride, cudaStream_t stream)
    {
        const Geometry &g = plan_.g;
        SweepArgs a;
        fill_common_args(a, w);
        a.prof = d_prof_.as<uint4>(); a.prof_u4 = (int)(plan_.prof.size() / 4);
        a.cta_nmax = w.d_ctanmax.as<int>();
        a.NS = g.NS; a.nsl = plan_.nsl; a.qp = plan_.qp;
        a.seg_stride = seg_stride;
        const int spw = 32 / g.T;
        a.wps = fast_ ? g.nslots / spw : 1;
        a.kstride = fast_ ? g.NS * 4 : (g.NS + 3) / 4 * 4;
        a.scanw = getenv("SD_FULL_SCAN") ? 64 : g.scanw;
        const size_t smem = plan_.prof.size() * 4 + (size_t)3 * a.kstride * 4 + (g.stream ? 0 : (size_t)g.NS * a.seg_stride);
        if (smem > (size_t)prop_.sharedMemPerBlockOptin) throw PlanError{"sweep geometry needs more shared memory than the SM has"};
        SD_CUDA(cudaFuncSetAttribute(kernel_, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int nctas = (int)w.lay.cta_nmax.size();
        void *args[] = {(void *)&a};
        SD_CUDA(cudaLaunchKernel(kernel_, dim3(nctas), dim3(g.NT), args, smem, stream));
    }

    void launch_group(WaveSlot &w)
    {
        const Geometry &g = plan_.g;
        GroupArgs a;
        fill_common_args(a, w);
        a.prof = d_prof_.as<uint4>(); a.nsl_total = plan_.nsl; a.qp = plan_.qp;
        a.NG = g.NG; a.SG = g.SG; a.NS = g.NS;
        a.scanw = getenv("SD_FULL_SCAN") ? 64 : g.scanw;
        a.error = w.d_out.as<int>() + 1;
        const int spw = 32 / g.T, wps = g.NT / 32;
        const size_t sgt = (size_t)wps * spw * g.T;
        const size_t smem = (size_t)5 * sgt * plan_.qp * 16 + ((size_t)g.NS * wps + g.NS + 8) * 4;
        if (smem > (size_t)prop_.sharedMemPerBlockOptin) throw PlanError{"group sweep needs more shared memory than the SM has"};
        SD_CUDA(cudaFuncSetAttribute(kernel_, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        SD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel_, g.NS * g.NT, smem));
        const int capacity = per_sm * prop_.multiProcessorCount;
        if (capacity < g.NG) throw PlanError{"monomer set too large: the CTAs of one segment cannot be co-resident on this GPU"};
        const int nblocks = (w.nseg + g.NS - 1) / g.NS;
        a.ngslots = std::min(nblocks, capacity / g.NG);
        // SD_GROUP_GSLOTS=n (tests): at most n slot groups, so that each sweeps several segment blocks
        if (const char *e = getenv("SD_GROUP_GSLOTS")) if (atoi(e) > 0) a.ngslots = std::min(a.ngslots, atoi(e));
        group_slots = std::max(group_slots, a.ngslots);
        const size_t xwords = (size_t)a.ngslots * 2 * g.NG * g.NS;
        w.d_xchg.need(xwords * 8);
        a.xbuf = w.d_xchg.as<unsigned long long>();
        SD_CUDA(cudaMemsetAsync(a.xbuf, 0, xwords * 8, st_));    // epoch 0 = nothing published
        void *args[] = {(void *)&a};
        SD_CUDA(cudaLaunchCooperativeKernel(kernel_, dim3(a.ngslots * g.NG), dim3(g.NS * g.NT), args, smem, st_));
    }

    void launch_lat(WaveSlot &w, int seg_stride)
    {
        const Geometry &g = plan_.g;
        LatArgs a;
        fill_common_args(a, w);
        a.prof2 = d_prof_.as<uint4>(); a.nsl_total = plan_.nsl; a.qp2 = plan_.qp2;
        a.NG = g.NG; a.SG = g.SG;
        a.lat_th = plan_.lat_th; a.scanw = g.scanw;
        for (int q = 0; q < 5; ++q) a.kj[q] = plan_.kj[q];
        a.seg_kj = w.filter_on ? w.d_segkj.as<int>() : nullptr;
        a.seg_stride = seg_stride;
        a.error = w.d_out.as<int>() + 1;
        const int spw = 32 / g.T, wpc = g.NT / 32;
        a.dbg = nullptr;
        if (lat_timing_) { w.d_dbg.need((size_t)w.nseg * g.NG * wpc * 64); a.dbg = w.d_dbg.as<long long>(); SD_CUDA(cudaMemsetAsync(a.dbg, 0, (size_t)w.nseg * g.NG * wpc * 64, st_)); }
        const size_t sgt = (size_t)wpc * spw * g.T;
        const size_t smem = (size_t)5 * sgt * plan_.qp2 * 16 + (size_t)LAT_NBUF * 32 * 8 + 32 + (g.stream ? 0 : (size_t)seg_stride);
        if (smem > (size_t)prop_.sharedMemPerBlockOptin) throw PlanError{"deferred-jump sweep needs more shared memory than the SM has"};
        SD_CUDA(cudaFuncSetAttribute(kernel_, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(w.nseg * g.NG)); cfg.blockDim = dim3((unsigned)g.NT);
        cfg.dynamicSmemBytes = smem; cfg.stream = st_;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)g.NG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        void *args[] = {(void *)&a};
        SD_CUDA(cudaLaunchKernelExC(&cfg, kernel_, args));
        if (lat_timing_) {
            const size_t nw = (size_t)w.nseg * g.NG * wpc;
            std::vector<long long> h(nw * 8);
            SD_CUDA(cudaMemcpyAsync(h.data(), a.dbg, nw * 64, cudaMemcpyDeviceToHost, st_));
            SD_CUDA(cudaStreamSynchronize(st_));
            double acc[6] = {0, 0, 0, 0, 0, 0}, cols = 0;
            for (size_t x = 0; x < nw; ++x) { for (int q = 0; q < 6; ++q) acc[q] += (double)h[x * 8 + q]; cols += (double)h[x * 8 + 6]; }
            fprintf(stderr, "[sd_b200 lat timing] cycles per column and warp: scan %.1f chain %.1f key+publish %.1f receive %.1f J+merge+store %.1f pre %.1f  (total %.1f)\n",
                    acc[0] / cols, acc[1] / cols, acc[2] / cols, acc[3] / cols, acc[4] / cols, acc[5] / cols,
                    (acc[0] + acc[1] + acc[2] + acc[3] + acc[4] + acc[5]) / cols);
        }
    }

    // sweep + traceback + compaction of the records into the result block; waits (on the device) for the wave's inputs
    void enqueue_kernels(WaveSlot &w)
    {
        const Geometry &g = plan_.g;
        const int seg_stride = (w.nmax + 16) / 16 * 16;
        // The classic sweeps of the two wave slots go to two streams: the CTAs of the next wave fill the SMs that the
        // last CTAs of this wave leave idle (a CTA runs for milliseconds, so the tail of a wave is a sizeable part of a
        // small wave).  The cluster and group kernels need the whole device to themselves and stay on one stream.
        const bool own_stream = !g.lat && g.NG == 1 && &w == &slot_[1];
        cudaStream_t ss = own_stream ? st2_ : st_;
        SD_CUDA(cudaStreamWaitEvent(ss, w.ev[1], 0));
        SD_CUDA(cudaEventRecord(w.ev[2], ss));
        if (g.lat) launch_lat(w, seg_stride); else if (g.NG > 1) launch_group(w); else launch_single(w, seg_stride, ss);
        SD_CUDA(cudaEventRecord(w.ev[3], ss));
        w.prev_end = last_end_;
        w.end_idx = (int)(wave_seq_++ & 3);
        SD_CUDA(cudaEventRecord(endev_[w.end_idx], ss));
        last_end_ = w.end_idx;
        // the traceback (a latency-bound walk, one warp per segment) and the compaction run on their own stream: the
        // sweep of the next wave starts as soon as this one's sweep is done and the two overlap
        SD_CUDA(cudaStreamWaitEvent(st_tb_, w.ev[3], 0));
        SD_CUDA(cudaEventRecord(w.ev[6], st_tb_));
        TbArgs t;
        t.g = g; t.codes = w.d_codes.as<uint32_t>(); t.cta_code_off = w.d_ctacode.as<int64_t>(); t.jr = w.d_jr.as<JR>();
        t.seg_j_off = w.d_segj.as<int64_t>();
        t.bases = w.d_bases.as<uint8_t>(); t.seg_off = w.d_segoff.as<int64_t>(); t.nseg = w.nseg;
        t.rows = d_rows_.as<uint8_t>(); t.row_off = d_rowoff_.as<int>();
        t.ins = plan_.sc.ins; t.del = plan_.sc.del; t.mismatch = plan_.sc.mismatch; t.match = plan_.sc.match;
        t.scratch = w.d_scratch.as<Record>(); t.seg_rec_off = w.d_segrec.as<int64_t>();
        t.counts = reinterpret_cast<int *>(w.d_out.as<char>() + OUT_HDR);
        t.rank2row = w.filter_on ? w.d_r2r.as<int>() : nullptr;
        t.error = w.d_out.as<int>() + 3;
        t.invC = (65536 + g.C - 1) / g.C;
        for (int pos = 0; pos < g.C * g.T; ++pos)
            if (((pos * t.invC) >> 16) != pos / g.C) throw PlanError{"internal: reciprocal division inexact"};
        traceback_kernel<<<(w.nseg + TB_WARPS - 1) / TB_WARPS, TB_WARPS * 32, 0, st_tb_>>>(t);
        SD_CUDA(cudaGetLastError());
        SD_CUDA(cudaEventRecord(w.ev[4], st_tb_));
        launches += 2;
    }

    void enqueue_gather(WaveSlot &w)
    {
        char *ob = w.d_out.as<char>();
        Record *dense = reinterpret_cast<Record *>(ob + OUT_HDR + out_counts_bytes(w.nseg));
        gather_kernel<<<1, 1024, 0, st_tb_>>>(w.d_scratch.as<Record>(), w.d_segrec.as<int64_t>(), reinterpret_cast<int *>(ob + OUT_HDR),
                                          dense, w.nseg, reinterpret_cast<int *>(ob) + 2);
        SD_CUDA(cudaGetLastError());
        launches += 1;
    }

    // device -> host: header + counts + the guessed share of the records in one copy into page-locked memory
    void enqueue_d2h(WaveSlot &w)
    {
        const size_t first = OUT_HDR + out_counts_bytes(w.nseg) + w.rec_guess * sizeof(Record);
        const size_t cap = OUT_HDR + out_counts_bytes(w.nseg) + (size_t)w.lay.seg_rec_off.back() * sizeof(Record);
        w.h_out.need(std::min(first, cap));
        SD_CUDA(cudaEventRecord(w.ev[5], st_tb_));                                 // compute done ...
        SD_CUDA(cudaStreamWaitEvent(st_out_, w.ev[5], 0));                        // ... before the copy starts
        SD_CUDA(cudaMemcpyAsync(w.h_out.p, w.d_out.p, std::min(first, cap), cudaMemcpyDeviceToHost, st_out_));
        SD_CUDA(cudaEventRecord(w.ev[5], st_out_));
    }

    // wait for the wave, check its flags, append its records
    void finish(WaveSlot &w, BatchResult &out)
    {
        SD_CUDA(cudaEventSynchronize(w.ev[5]));
        const int64_t total = wave_total(w.h_out.as<int>());
        const size_t rec_off = OUT_HDR + out_counts_bytes(w.nseg);
        const size_t base = out.recs.size();
        out.recs.resize(base + (size_t)total);
        const size_t have = std::min<size_t>((size_t)total, w.rec_guess);
        if (have) memcpy(out.recs.data() + base, w.h_out.as<char>() + rec_off, have * sizeof(Record));
        if ((size_t)total > have) {              // the guess was too small (very short monomers): fetch the rest
            SD_CUDA(cudaMemcpyAsync(out.recs.data() + base + have, w.d_out.as<char>() + rec_off + have * sizeof(Record),
                                    ((size_t)total - have) * sizeof(Record), cudaMemcpyDeviceToHost, st_out_));
            SD_CUDA(cudaStreamSynchronize(st_out_));
        }
        const int *cnt = reinterpret_cast<const int *>(w.h_out.as<char>() + OUT_HDR);
        int64_t run = (int64_t)base;
        for (int s = 0; s < w.nseg; ++s) { run += cnt[s]; out.rec_off.push_back(run); }
        float ms = 0;
        SD_CUDA(cudaEventElapsedTime(&ms, w.ev[0], w.ev[1])); h2d_ms += ms;
        SD_CUDA(cudaEventElapsedTime(&ms, w.ev[2], w.ev[3]));
        if (w.prev_end >= 0) {                  // sweeps of consecutive waves overlap: count the overlap once
            float since_prev = 0;
            SD_CUDA(cudaEventElapsedTime(&since_prev, endev_[w.prev_end], w.ev[3]));
            ms = std::min(ms, std::max(since_prev, 0.0f));
        }
        sweep_ms += ms;
        SD_CUDA(cudaEventElapsedTime(&ms, w.ev[6], w.ev[4])); traceback_ms += ms;
        d2h_bytes += (int64_t)(rec_off + (size_t)total * sizeof(Record));
        w.staged = false;
    }

    // ---- Backend interface --------------------------------------------------------------------------------------
    void submit(int slot, const Batch &b, int s0, int s1) override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        WaveSlot &w = slot_[slot & 1];
        nvtxRangePushA("sd_b200: wave copy-in");
        enqueue_h2d(w, b, s0, s1);
        nvtxRangePop();
        nvtxRangePushA("sd_b200: wave sweep + traceback");
        enqueue_kernels(w);
        enqueue_gather(w);
        nvtxRangePop();
        nvtxRangePushA("sd_b200: wave copy-out");
        enqueue_d2h(w);
        nvtxRangePop();
    }
    void collect(int slot, BatchResult &out) override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        nvtxRangePushA("sd_b200: wave collect");
        try { finish(slot_[slot & 1], out); } catch (...) { nvtxRangePop(); throw; }
        nvtxRangePop();
    }
    // the resident path (sd_stage / sd_run_staged / sd_fetch_staged): one wave on slot 0, each step synchronous
    void stage(const Batch &b, int s0, int s1) override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        enqueue_h2d(slot_[0], b, s0, s1);
        SD_CUDA(cudaStreamSynchronize(st_in_));
        float ms = 0; SD_CUDA(cudaEventElapsedTime(&ms, slot_[0].ev[0], slot_[0].ev[1])); h2d_ms += ms;
    }
    void execute() override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        WaveSlot &w = slot_[0];
        SD_CUDA(cudaMemsetAsync(w.d_out.p, 0, OUT_HDR, st_));
        enqueue_kernels(w);
        int hdr[4] = {0, 0, 0, 0};
        SD_CUDA(cudaMemcpyAsync(hdr, w.d_out.p, OUT_HDR, cudaMemcpyDeviceToHost, st_tb_));
        SD_CUDA(cudaStreamSynchronize(st_tb_));
        wave_total(hdr);                  // the records are compacted by fetch(): the total is still 0 here
        float ms = 0;
        SD_CUDA(cudaEventElapsedTime(&ms, w.ev[2], w.ev[3])); sweep_ms += ms;
        SD_CUDA(cudaEventElapsedTime(&ms, w.ev[6], w.ev[4])); traceback_ms += ms;
    }
    void fetch(BatchResult &out) override
    {
        DeviceScope scope_(dev_); SD_CUDA(scope_.status);
        WaveSlot &w = slot_[0];
        const double sw = sweep_ms, tb = traceback_ms, h2 = h2d_ms;
        enqueue_gather(w);
        enqueue_d2h(w);
        finish(w, out);
        sweep_ms = sw; traceback_ms = tb; h2d_ms = h2;          // already accounted for by stage() / execute()
    }

private:
    int dev_;
    cudaStream_t st_{}, st_in_{}, st_out_{}, st_tb_{};      // sweep, copy-in, copy-out, traceback + compaction
    cudaStream_t st2_{};                                     // classic sweeps of wave slot 1
    cudaEvent_t endev_[4]{};                                 // sweep-end events of the last four waves (ring)
    uint64_t wave_seq_ = 0; int last_end_ = -1;
    cudaDeviceProp prop_{};
    Plan plan_; MonomerSet ms_;
    const void *kernel_ = nullptr;
    bool fast_ = false, lat_timing_ = false;
    std::vector<uint8_t> rows_ascii_;
    int64_t budget_ = 0;
    int64_t free_at_start_ = 0;        // device memory that was free when the backend was created
    DevBuf d_prof_, d_slotlen_, d_slotend_, d_rows_, d_rowoff_, d_kjbase_;
    std::vector<int> kjbase_;
    WaveSlot slot_[2];
};

} // namespace

Backend *make_cuda_backend(int device_id, std::string &err)
{
    try { return new CudaBackend(device_id); }
    catch (PlanError &e) { err = e.msg; return nullptr; }
}

} // namespace sdb

int cuda_device_count()
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

// page-locked host memory for callers that want their inputs to travel by DMA without the driver's staging copy
void *cuda_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void cuda_host_free(void *p) { cudaFreeHost(p); }

int cuda_int_peak(int device, double *alu, double *both, double *mhz, std::string &err)
{
    using namespace sdb;
    try {
        DeviceScope scope_(device); SD_CUDA(scope_.status);
        cudaDeviceProp p; SD_CUDA(cudaGetDeviceProperties(&p, device));
        const int nblk = p.multiProcessorCount * 2, nthr = 512;
        unsigned *d; SD_CUDA(cudaMalloc(&d, (size_t)nblk * nthr * 4));
        cudaEvent_t e0, e1; SD_CUDA(cudaEventCreate(&e0)); SD_CUDA(cudaEventCreate(&e1));
        double res[2] = {0, 0};
        for (int mode = 0; mode < 2; ++mode) {
            float best = 1e30f;
            for (int rep = 0; rep < 5; ++rep) {
                SD_CUDA(cudaEventRecord(e0));
                if (mode == 0) int_peak_kernel<0><<<nblk, nthr>>>(d, 1234u); else int_peak_kernel<1><<<nblk, nthr>>>(d, 1234u);
                SD_CUDA(cudaEventRecord(e1));
                SD_CUDA(cudaEventSynchronize(e1));
                float ms; SD_CUDA(cudaEventElapsedTime(&ms, e0, e1));
                if (rep > 0) best = std::min(best, ms);
            }
            const double ops = (double)nblk * nthr * 2048.0 * 8.0 * (mode == 0 ? 1.0 : 2.0);
            res[mode] = ops / (best * 1e-3);
        }
        if (alu) *alu = res[0];
        if (both) *both = res[1];
        if (mhz) *mhz = res[0] / ((double)p.multiProcessorCount * 64.0) / 1e6;     // ALU pipe: 64 lanes/clk/SM (measured)
        cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    } catch (PlanError &e) { err = e.msg; return 4; }
    return 0;
}
