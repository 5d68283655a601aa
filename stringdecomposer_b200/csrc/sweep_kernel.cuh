// sweep_kernel.cuh -- the sm_100a column-sweep kernel template (instantiated in sweep_inst_*.cu).
#pragma once
#include <cuda_runtime.h>
#include <climits>

#include "common.h"

namespace sdb {

struct SweepArgs {
    const uint4 *prof; int prof_u4;                    // [5][nsl][qp] uint4
    const uint8_t *bases; const int64_t *seg_off;      // seg_off indexed by segment id within the staged wave
    int nseg;
    const int *cta_nmax; const int64_t *cta_code_off; const int64_t *seg_j_off;
    uint32_t *codes; JR *jr;
    const int *slot_len; const int *slot_endadd;
    int nslots, M, NS, NT, CW, nsl, qp;
    int ins, del, deadz;
    int seg_stride;
    int wps;                // warps per segment (FAST only, <= 4)
    int kstride;            // ints per key buffer
    const int *rank;        // --ed_thr pre-filter: [segment][row] position in the filtered list, -1 = filtered out; or null
    int *bad_symbol;        // set to 1 when a segment holds a symbol outside ACGTN
    TagRegs tr;             // TAGMASK / ONE of the policy, passed as run-time values (sweep_core.cuh: TagRegs)
    int scanw;              // carry window of the deletion scan (plan.cpp: scan_window)
};

// Carry of the deletion chain into a lane: exclusive prefix maximum of the lane maxima over the lanes of its slot.
// Only the W nearest lanes on the left can matter (W = plan.cpp: scan_window, a property of the monomer set, so the
// branches below are uniform over the whole launch): W independent shuffles and a small max tree -- one shuffle
// latency -- instead of a scan over all T lanes.  Windows wider than 8 fall back to a log-depth scan.
template <class P, int T, int N>
__device__ __forceinline__ uint32_t flat_window(uint32_t E, int t, uint32_t dead)
{
    uint32_t r[N];
#pragma unroll
    for (int d = 1; d <= N; ++d) { r[d - 1] = __shfl_up_sync(0xffffffffu, E, d); if (t < d) r[d - 1] = dead; }
    return tree_max<P, N>(r);
}
template <class P, int T>
__device__ __forceinline__ uint32_t slot_scan_window(uint32_t E, int t, uint32_t dead, int W)
{
    if (T == 1) return dead;
    if (T == 2) { const uint32_t pv = __shfl_up_sync(0xffffffffu, E, 1); return t == 0 ? dead : pv; }
    if (T >= 3 && W <= 2) return flat_window<P, T, 2>(E, t, dead);
    if (T >= 5 && W <= 4) return flat_window<P, T, (T >= 5 ? 4 : 1)>(E, t, dead);
    if (T >= 9 && W <= 8) return flat_window<P, T, (T >= 9 ? 8 : 1)>(E, t, dead);
    uint32_t pv = __shfl_up_sync(0xffffffffu, E, 1);
    if (t == 0) pv = dead;
#pragma unroll
    for (int d = 1; d < T; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, pv, d);
        if (t >= d) pv = P::max2(pv, o);
    }
    return pv;
}

// Profile words of one lane for one column: (C+3)/4 uint4 loads from the lane's row of the symbol (the words past C are
// padding).
template <int C>
__device__ __forceinline__ void load_profile_row(uint32_t (&pw)[(C + 3) / 4 * 4], const uint4 *row)
{
#pragma unroll
    for (int q = 0; q < (C + 3) / 4; ++q) {
        const uint4 v = row[q];
        pw[4 * q] = v.x; pw[4 * q + 1] = v.y; pw[4 * q + 2] = v.z; pw[4 * q + 3] = v.w;
    }
}

// One lane's backpointer words of one column: a single vector store where the word count allows it.
template <int NW>
__device__ __forceinline__ void store_code_words(uint32_t *cptr, const uint32_t (&cw)[NW])
{
    if (NW == 2) *reinterpret_cast<uint2 *>(cptr) = make_uint2(cw[0], cw[1]);
    else if (NW == 4) *reinterpret_cast<uint4 *>(cptr) = make_uint4(cw[0], cw[1], cw[2], cw[3]);
    else {
#pragma unroll
        for (int w = 0; w < NW; ++w) cptr[w] = cw[w];
    }
}

// First cell of the lane for the next column (lane_pre_first): it needs the left lane's row-end value.
template <class P, int C, int T>
__device__ __forceinline__ uint32_t next_first_cell(uint32_t uend, uint32_t pn0, uint32_t ufirst, uint32_t deadu, int t,
                                                    bool kill_first, bool kill_last)
{
    uint32_t prevU = deadu;
    if (T > 1) { prevU = __shfl_up_sync(0xffffffffu, uend, 1); if (t == 0) prevU = deadu; }
    return lane_pre_first<P>(prevU, pn0, ufirst, deadu, kill_first, C == 1 && kill_last);
}

// FAST: every warp serves exactly one segment and a segment has <= 4 warps: the per-column (score,row) key is
// reduced with CREDUX inside the warp and exchanged through one aligned int4 row of shared memory.
// MULTI (with FAST): several segments share the CTA and its profile table but synchronise separately (named barriers).
// !FAST: arbitrary lane->segment mapping; keys meet in shared-memory atomicMax (three rotating buffers).
// STREAM: the segment symbols are not staged in shared memory (whose size then does not depend on the segment length):
// every thread loads the symbol of column i+2 from global memory while it sweeps column i, the same symbol for all
// lanes of a segment (one L1 broadcast), and validates and encodes it as the staging loop does.
template <class P, int C, int T, bool FAST, bool MULTI, bool STREAM = false>
__device__ __forceinline__ void sweep_body(const SweepArgs &a)
{
    extern __shared__ uint4 smem_u4[];
    uint4 *sprof = smem_u4;
    int *skey = reinterpret_cast<int *>(sprof + a.prof_u4);             // key buffers, 16-byte aligned rows
    const int NS = a.NS, NT = a.NT;
    const int kstride = a.kstride;
    uint8_t *schar = reinterpret_cast<uint8_t *>(skey + 3 * kstride);

    const int tid = threadIdx.x, cta = blockIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    constexpr int SPW = 32 / T;
    const int siw = lane / T, t = lane - siw * T;
    const bool lane_ok = siw < SPW;
    const int ginst = warp * SPW + (lane_ok ? siw : 0);
    int seg_local = ginst / a.nslots;
    const int slot = ginst - seg_local * a.nslots;
    const int first = cta * NS;                                         // first segment of the CTA (within the launch)
    const bool active = lane_ok && seg_local < NS && first + seg_local < a.nseg;
    if (seg_local >= NS) seg_local = 0;
    const int nmax = a.cta_nmax[cta];
    int n_seg = 0;
    if (active) n_seg = (int)(a.seg_off[first + seg_local + 1] - a.seg_off[first + seg_local]);

    // stage profile, segment symbols and keys
    for (int x = tid; x < a.prof_u4; x += NT) sprof[x] = a.prof[x];
    for (int s = 0; s < (STREAM ? 0 : NS); ++s) {
        int n = 0; const uint8_t *src = nullptr;
        if (first + s < a.nseg) {
            const int64_t o = a.seg_off[first + s];
            n = (int)(a.seg_off[first + s + 1] - o);
            src = a.bases + o;
        }
        for (int x = tid; x < a.seg_stride; x += NT) schar[s * a.seg_stride + x] = (uint8_t)((x < n) ? symbol_code(src[x], a.bad_symbol) : 0);
    }
    for (int x = tid; x < 3 * kstride; x += NT) skey[x] = INT_MIN;
    __syncthreads();

    const int L = a.slot_len[slot];
    const int endadd = a.slot_endadd[slot];
    const uint32_t deadu = P::splat(a.deadz - 1);
    const TagRegs tr = a.tr;
    const bool kill_first = (t == 0), kill_last = (t == T - 1 && L == 1);
    const bool j_writer = active && slot == 0 && t == 0;
    const bool is_end = active && t == T - 1;
    const SlotKey sk = slot_key<P>(active, is_end, endadd, slot, a.M, a.rank, first, seg_local, -0x800);
    JR *jptr = a.jr + (active ? a.seg_j_off[first + seg_local] : 0);
    uint32_t *cptr = a.codes + a.cta_code_off[cta] + (size_t)tid * a.CW;
    const size_t cstride = (size_t)NT * a.CW;
    const uint8_t *cp = schar + seg_local * a.seg_stride;               // symbol of the column being prepared
    // STREAM: the segment's text in global memory; columns past its end read as symbol 0, like the 0-padded buffer
    const uint8_t *src = a.bases + (active ? a.seg_off[first + seg_local] : 0);
    auto symbol = [&](int i) { return (i < n_seg) ? symbol_code(__ldg(src + i), a.bad_symbol) : 0; };
    const uint4 *myprof = sprof + (size_t)(slot * T + t) * a.qp;
    const int sym_stride = a.nsl * a.qp;
    // FAST: segment s of the CTA owns int4 row s of each key buffer, its warps write one int each.  Raw shared-space
    // addresses keep the exchange to one STS / one LDS.128 (no generic-address arithmetic in the loop).
    const int wseg = FAST ? warp / a.wps : 0;
    const uint32_t skey_s = (uint32_t)__cvta_generic_to_shared(skey);
    const uint32_t key_wr_s = skey_s + 4u * (uint32_t)(FAST ? wseg * 4 + (warp - wseg * a.wps) : seg_local);
    const uint32_t key_rd_s = skey_s + 4u * (uint32_t)(FAST ? wseg * 4 : seg_local);
    const uint32_t kbytes = 4u * (uint32_t)kstride;
    const int bar_id = 1 + wseg, bar_threads = a.wps * 32;

    uint32_t X[C], pw[(C + 3) / 4 * 4];
#pragma unroll
    for (int kk = 0; kk < C; ++kk) X[kk] = deadu;
    auto load_profile = [&](int sym) { load_profile_row<C>(pw, myprof + sym * sym_stride); };

    int sym_next = 0;
    if (STREAM) { load_profile(symbol(0)); sym_next = symbol(1); }
    else load_profile(*cp++);
    lane_pre_col0<P, C>(X, pw, a.del, L, deadu, kill_first, kill_last);
    int jbase = a.ins;            // Bref + i*ins: J[i+1] = vmax + jbase
    int jump0 = 0;                // 4*(B[i] - Bref)
    uint32_t kboff = 0;           // byte offset of the key buffer in use (FAST: 2 buffers alternate; else 3 rotate)
#pragma unroll 1
    for (int i = 0; i < nmax; ++i) {
        const uint32_t E = lane_post<P, C>(X, pw, P::splat(jump0 + 1), deadu, tr);
        // profile of the next column (the symbol buffer is 0-padded, so the round after the last column is harmless);
        // issued here so that the loads fly during the scan
        if (STREAM) { load_profile(sym_next); sym_next = symbol(i + 2); }
        else load_profile(*cp++);
        const uint32_t carry = slot_scan_window<P, T>(E, t, deadu, a.scanw);
        constexpr int NW = (C + P::CELLS_PER_WORD - 1) / P::CELLS_PER_WORD;
        uint32_t cw[NW];
        uint32_t ufirst;
        const uint32_t uend = lane_pass2_pre<P, C>(X, carry, cw, tr, pw, deadu, kill_last, &ufirst);

        // one segment per CTA (FAST without MULTI): every column is live; else a shorter segment idles past its end
        const bool live = active && ((FAST && !MULTI) || i < n_seg);
        if (live) store_code_words(cptr, cw);
        cptr += cstride;

        // row ends -> (score,row) key of the segment: key = (u >> 2) * 4096 + (endadd * 4096 + 4095 - row)
        const int key = lane_key<P>(uend, sk.kc_lo, sk.kc_hi, sk.counted);
        if (FAST) {
            const int wk = __reduce_max_sync(0xffffffffu, key);
            if (lane == 0) asm volatile("st.shared.b32 [%0], %1;" ::"r"(key_wr_s + kboff), "r"(wk) : "memory");
        } else {
            // reset the buffer of the NEXT column: it was last read two columns ago, and every thread has passed a
            // barrier since (the buffer of the previous column may still be being read by a slower warp)
            const uint32_t kclr = (kboff == 2 * kbytes) ? 0 : kboff + kbytes;
            if (tid < NS) asm volatile("st.shared.b32 [%0], %1;" ::"r"(skey_s + kclr + 4u * tid), "r"(INT_MIN) : "memory");
            if (is_end) atomicMax(reinterpret_cast<int *>(reinterpret_cast<char *>(skey) + kboff) + seg_local, key);
        }
        X[0] = next_first_cell<P, C, T>(uend, pw[0], ufirst, deadu, t, kill_first, kill_last);
        // (ptxas schedules these J-independent max-plus ops behind the barrier, where they cover the latency of the
        // key load that follows it)

        // FAST: only the warps of this segment meet (named barrier 1 + segment), so the segments that share a CTA
        // (and its profile table) run decoupled; otherwise the whole CTA synchronises
        if (FAST && MULTI) asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(bar_threads) : "memory");
        else __syncthreads();
        int k2;
        if (FAST) {
            int4 v;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(key_rd_s + kboff) : "memory");
            k2 = max(max(v.x, v.y), max(v.z, v.w));
            kboff ^= kbytes;
        } else {
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(k2) : "r"(key_rd_s + kboff) : "memory");
            kboff = (kboff == 2 * kbytes) ? 0 : kboff + kbytes;
        }
        const int vmax = k2 >> 12;
        ++jptr;
        if (live && j_writer) *jptr = JR{vmax + jbase, SD_KEY_ROWS - 1 - (k2 & (SD_KEY_ROWS - 1))};
        jbase += a.ins;
        jump0 = 4 * (vmax + a.del);
        if (jump0 > SD_REBASE_TH || jump0 < -SD_REBASE_TH) {
            lane_rebase<P, C>(X, jump0);
            jbase += jump0 >> 2;
            jump0 = 0;
        }
    }
}


template <class P, int C, int T, bool FAST, bool MULTI, bool STREAM>
__global__ void sweep_kernel(const SweepArgs a) { sweep_body<P, C, T, FAST, MULTI, STREAM>(a); }

// The same kernel with its register budget pinned at 80: saturated launches (several segments per CTA, C <= 24) then fit
// two 384-thread CTAs per SM; left alone ptxas settles on 96 registers and halves the occupancy (measured: 3.95 -> 4.11
// TCUPS on 4,000 segments).  Only used for CTAs of at most 768 threads.
template <class P, int C, int T, bool FAST, bool MULTI, bool STREAM>
__global__ void __maxnreg__(80) sweep_kernel_r80(const SweepArgs a) { sweep_body<P, C, T, FAST, MULTI, STREAM>(a); }

// ---------------------------------------------------------------------------------------------------------------
// Group sweep: monomer sets that do not fit one CTA (threads, registers, or the shared-memory profile table).
// The slots are split into NG groups.  CTA (gslot, grp) holds the profile slice of group `grp` and sweeps that group
// for NS segments at a time (segment blocks gslot, gslot+ngslots, ...; the NS segments share the profile slice and the
// column exchange, which amortises its latency).  The NG CTAs of a block meet once per column in global memory:
// every CTA publishes (epoch, key) per segment in its own slots with relaxed 64-bit stores and warp 0 polls the
// NG*NS slots of the current buffer (no atomics, two buffers, bounded spin).  All CTAs are co-resident (cooperative
// launch), so the spin cannot deadlock; a time-out raises *error instead of hanging.
struct GroupArgs {
    const uint4 *prof; int nsl_total, qp;              // [5][nsl_total][qp] uint4
    const uint8_t *bases; const int64_t *seg_off; int nseg;
    const int64_t *cta_code_off; const int64_t *seg_j_off;
    uint32_t *codes; JR *jr;
    const int *slot_len; const int *slot_endadd;
    int nslots, M, NT, CW, NG, SG, NS;                 // NT: threads per (segment, group) = layout stride; block = NS*NT
    int ins, del, deadz;
    TagRegs tr;
    int *bad_symbol;
    int scanw;                                          // carry window of the deletion scan (plan.cpp: scan_window)
    unsigned long long *xbuf;                           // [ngslots][2][NG][NS] exchange slots, zeroed before the launch
    const int *rank;                                    // --ed_thr pre-filter ranks [segment][row] or null
    int ngslots;
    int *error;
};

template <class P, int C, int T>
__global__ void sweep_group_kernel(const GroupArgs a)
{
    extern __shared__ uint4 smem_u4[];
    constexpr int SPW = 32 / T;
    const int NT = a.NT, NG = a.NG, NS = a.NS;
    const int wps = NT >> 5;                             // warps per segment in this CTA
    const int sgt = wps * SPW * T;                       // profile rows kept per CTA (slot lanes)
    uint4 *sprof = smem_u4;                              // [5][sgt][qp]
    int *swk = reinterpret_cast<int *>(sprof + (size_t)5 * sgt * a.qp);     // [NS][wps] warp keys
    int *sres = swk + NS * wps;                          // [NS] block-wide keys of the column

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gslot = blockIdx.x / NG, grp = blockIdx.x - gslot * NG;
    const int seg_local = warp / wps, wseg = warp - seg_local * wps;
    const int siw = lane / T, t = lane - siw * T;
    const bool lane_ok = siw < SPW;
    const int ginst = wseg * SPW + (lane_ok ? siw : 0);
    int slot = grp * a.SG + ginst;
    const bool slot_ok = lane_ok && ginst < a.SG && slot < a.nslots;
    if (slot >= a.nslots) slot = a.nslots - 1;

    // profile slice of this group: rows [grp*SG*T, grp*SG*T + sgt) of every symbol (clamped at the table end)
    for (int x = tid; x < 5 * sgt * a.qp; x += NS * NT) {
        const int sym = x / (sgt * a.qp), r = x - sym * (sgt * a.qp);
        const int row = min(grp * a.SG * T + r / a.qp, a.nsl_total - 1);
        sprof[x] = a.prof[((size_t)sym * a.nsl_total + row) * a.qp + (r % a.qp)];
    }
    const int L = a.slot_len[slot];
    const int endadd = a.slot_endadd[slot];
    const uint32_t deadu = P::splat(a.deadz - 1);
    const TagRegs tr = a.tr;
    const bool kill_first = (t == 0), kill_last = (t == T - 1 && L == 1);
    const uint4 *myprof = sprof + (size_t)(ginst * T + t) * a.qp;
    const int sym_stride = sgt * a.qp;
    unsigned long long *xbuf = a.xbuf + (size_t)gslot * 2 * NG * NS;
    unsigned gcol = 0;                                   // columns this CTA group has exchanged so far
    __syncthreads();

    uint32_t X[C], pw[(C + 3) / 4 * 4];
    auto load_profile = [&](int sym) { load_profile_row<C>(pw, myprof + sym * sym_stride); };
    const int nblocks = (a.nseg + NS - 1) / NS;
    for (int blk = gslot; blk < nblocks; blk += a.ngslots) {
        // the NS segments of the block advance in lockstep; a shorter (or missing) one idles past its end
        const int seg = blk * NS + seg_local;
        const bool seg_ok = seg < a.nseg;
        const int64_t o = seg_ok ? a.seg_off[seg] : 0;
        const int n = seg_ok ? (int)(a.seg_off[seg + 1] - o) : 0;
        int nmax = 0;
        for (int q = 0; q < NS; ++q) {
            const int sq = blk * NS + q;
            if (sq < a.nseg) nmax = max(nmax, (int)(a.seg_off[sq + 1] - a.seg_off[sq]));
        }
        const bool active = slot_ok && seg_ok;
        const bool is_end = active && t == T - 1;
        const bool j_writer = seg_ok && grp == 0 && wseg == 0 && lane == 0;
        const SlotKey sk = slot_key<P>(active, is_end, endadd, slot, a.M, a.rank, seg, 0, -0x800);
        JR *jptr = a.jr + (seg_ok ? a.seg_j_off[seg] : 0);
        uint32_t *cptr = a.codes + (seg_ok ? a.cta_code_off[(size_t)seg * NG + grp] : 0) + (size_t)(wseg * 32 + lane) * a.CW;
        const size_t cstride = (size_t)NT * a.CW;
        // symbols are streamed from global memory (one byte per column, the same for all lanes of the segment)
        const uint8_t *src = a.bases + o;
        auto symbol = [&](int i) { return (i < n) ? symbol_code(__ldg(src + i), a.bad_symbol) : 0; };
#pragma unroll
        for (int kk = 0; kk < C; ++kk) X[kk] = deadu;
        load_profile(symbol(0));
        lane_pre_col0<P, C>(X, pw, a.del, L, deadu, kill_first, kill_last);
        int jbase = a.ins, jump0 = 0;
        int sym_next = symbol(1);
#pragma unroll 1
        for (int i = 0; i < nmax; ++i) {
            const uint32_t E = lane_post<P, C>(X, pw, P::splat(jump0 + 1), deadu, tr);
            load_profile(sym_next);
            sym_next = symbol(i + 2);
            const uint32_t carry = slot_scan_window<P, T>(E, t, deadu, a.scanw);
            constexpr int NW = (C + P::CELLS_PER_WORD - 1) / P::CELLS_PER_WORD;
            uint32_t cw[NW];
            uint32_t ufirst;
            const uint32_t uend = lane_pass2_pre<P, C>(X, carry, cw, tr, pw, deadu, kill_last, &ufirst);
            const bool live = active && i < n;
            if (live) {
#pragma unroll
                for (int w = 0; w < NW; ++w) cptr[w] = cw[w];
            }
            cptr += cstride;
            const int key = lane_key<P>(uend, sk.kc_lo, sk.kc_hi, sk.counted);
            const int wk = __reduce_max_sync(0xffffffffu, key);
            if (lane == 0) swk[seg_local * wps + wseg] = wk;
            X[0] = next_first_cell<P, C, T>(uend, pw[0], ufirst, deadu, t, kill_first, kill_last);
            __syncthreads();
            // Column exchange between the NG CTAs of the block (see the comment above the kernel).  Two buffers
            // suffice: a CTA can only be one column ahead of the slowest reader, because it needs everybody's key of
            // column c to leave column c.
            if (warp == 0) {
                const unsigned epoch = gcol + 1u;
                unsigned long long *buf = xbuf + (size_t)(gcol & 1u) * NG * NS;
                if (lane < NS) {
                    int k = swk[lane * wps];
                    for (int w = 1; w < wps; ++w) k = max(k, swk[lane * wps + w]);
                    const unsigned long long v = ((unsigned long long)epoch << 32) | (unsigned)k;
                    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(buf + grp * NS + lane), "l"(v) : "memory");
                    sres[lane] = INT_MIN;
                }
                __syncwarp();
                // every lane owns the slots lane, lane+32, ...; the loads of one polling round are issued back to back
                // so that a round costs one L2 round trip however many slots a lane owns
                const int nx = NG * NS;
                unsigned pending = 0;                            // bit j: slot lane + 32*j not seen yet
                for (int j = 0; lane + 32 * j < nx; ++j) pending |= 1u << j;
                unsigned spins = 0;
                while (__any_sync(0xffffffffu, pending != 0)) {
                    unsigned long long v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (pending & (1u << j))
                            asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v[j]) : "l"(buf + lane + 32 * j) : "memory");
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if ((pending & (1u << j)) && (unsigned)(v[j] >> 32) == epoch) {
                            atomicMax(&sres[(lane + 32 * j) % NS], (int)(unsigned)v[j]);
                            pending &= ~(1u << j);
                        }
                    if (++spins > (1u << 21)) { *a.error = 1; break; }
                }
            }
            __syncthreads();
            const int k2 = sres[seg_local];
            ++gcol;
            const int vmax = k2 >> 12;
            ++jptr;
            if (j_writer && i < n) *jptr = JR{vmax + jbase, SD_KEY_ROWS - 1 - (k2 & (SD_KEY_ROWS - 1))};
            jbase += a.ins;
            jump0 = 4 * (vmax + a.del);
            if (i >= n) jump0 = 0;                       // an idle segment keeps its registers bounded
            if (jump0 > SD_REBASE_TH || jump0 < -SD_REBASE_TH) {
                lane_rebase<P, C>(X, jump0);
                jbase += jump0 >> 2;
                jump0 = 0;
            }
        }
    }
}

// Lookup tables of the instantiations, one translation unit per (policy, FAST, MULTI, STREAM) so that they build in
// parallel: the kernel compiled for the geometry, or null.  sweep_kernels.cu: sweep_kernel_for picks the table.
using SweepLookup = const void *(*)(const Geometry &g);
const void *sweep_lookup_p16_f1_m0(const Geometry &g);
const void *sweep_lookup_p16_f1_m1(const Geometry &g);
const void *sweep_lookup_p16_f0_m0(const Geometry &g);
const void *sweep_lookup_s32_f1_m0(const Geometry &g);
const void *sweep_lookup_s32_f1_m1(const Geometry &g);
const void *sweep_lookup_s32_f0_m0(const Geometry &g);
const void *sweep_lookup_p16_f1_m0_st(const Geometry &g);
const void *sweep_lookup_p16_f1_m1_st(const Geometry &g);
const void *sweep_lookup_p16_f0_m0_st(const Geometry &g);
const void *sweep_lookup_s32_f1_m0_st(const Geometry &g);
const void *sweep_lookup_s32_f1_m1_st(const Geometry &g);
const void *sweep_lookup_s32_f0_m0_st(const Geometry &g);
const void *sweep_group_lookup_p16(const Geometry &g);
const void *sweep_group_lookup_s32(const Geometry &g);

// the register-capped twin is instantiated only where it is used: several segments per CTA (LL) and C <= 24
template <class POLICY, int CC, int TT, bool FAST, bool LL, bool ST> static const void *sweep_pick(bool cap80)
{
    if constexpr (LL && CC <= 24) { if (cap80) return (const void *)sweep_kernel_r80<POLICY, CC, TT, FAST, LL, ST>; }
    (void)cap80;
    return (const void *)sweep_kernel<POLICY, CC, TT, FAST, LL, ST>;
}
#define SD_SWEEP_PICK(POLICY, CC, TT, FAST, LL, ST) sweep_pick<POLICY, CC, TT, FAST, LL, ST>(cap80)
#define SD_INSTANTIATE_SWEEP(NAME, POLICY, FAST, LL, ST)                                                             \
    template <int C> static const void *NAME##_t(int T, bool cap80)                                                  \
    {                                                                                                                 \
        switch (T) {                                                                                                  \
        case 1: return SD_SWEEP_PICK(POLICY, C, 1, FAST, LL, ST);                                                     \
        case 2: return SD_SWEEP_PICK(POLICY, C, 2, FAST, LL, ST);                                                     \
        case 4: return SD_SWEEP_PICK(POLICY, C, 4, FAST, LL, ST);                                                     \
        case 8: return SD_SWEEP_PICK(POLICY, C, 8, FAST, LL, ST);                                                     \
        case 10: return SD_SWEEP_PICK(POLICY, C, 10, FAST, LL, ST);                                                   \
        case 16: return SD_SWEEP_PICK(POLICY, C, 16, FAST, LL, ST);                                                   \
        case 32: return SD_SWEEP_PICK(POLICY, C, 32, FAST, LL, ST);                                                   \
        }                                                                                                             \
        return nullptr;                                                                                               \
    }                                                                                                                 \
    const void *NAME(const Geometry &g)                                                                               \
    {                                                                                                                 \
        const int T = g.T;                                                                                            \
        const bool cap80 = g.NT <= 768;                                                                               \
        switch (g.C) {                                                                                                \
        case 8: return NAME##_t<8>(T, cap80); case 12: return NAME##_t<12>(T, cap80); case 16: return NAME##_t<16>(T, cap80);   \
        case 19: return NAME##_t<19>(T, cap80); case 20: return NAME##_t<20>(T, cap80); case 24: return NAME##_t<24>(T, cap80); \
        case 32: return NAME##_t<32>(T, cap80);                                                                       \
        case 48: return NAME##_t<48>(T, cap80);                                                                       \
        }                                                                                                             \
        return nullptr;                                                                                               \
    }

#define SD_INSTANTIATE_GROUP(NAME, POLICY)                                                                           \
    template <int C> static const void *NAME##_t(int T)                                                              \
    {                                                                                                                 \
        switch (T) {                                                                                                  \
        case 1: return (const void *)sweep_group_kernel<POLICY, C, 1>;                                                \
        case 2: return (const void *)sweep_group_kernel<POLICY, C, 2>;                                                \
        case 4: return (const void *)sweep_group_kernel<POLICY, C, 4>;                                                \
        case 8: return (const void *)sweep_group_kernel<POLICY, C, 8>;                                                \
        case 10: return (const void *)sweep_group_kernel<POLICY, C, 10>;                                              \
        case 16: return (const void *)sweep_group_kernel<POLICY, C, 16>;                                              \
        case 32: return (const void *)sweep_group_kernel<POLICY, C, 32>;                                              \
        }                                                                                                             \
        return nullptr;                                                                                               \
    }                                                                                                                 \
    const void *NAME(const Geometry &g)                                                                               \
    {                                                                                                                 \
        const int T = g.T;                                                                                            \
        switch (g.C) {                                                                                                \
        case 8: return NAME##_t<8>(T); case 12: return NAME##_t<12>(T); case 16: return NAME##_t<16>(T);              \
        case 19: return NAME##_t<19>(T); case 20: return NAME##_t<20>(T); case 24: return NAME##_t<24>(T);              \
        case 32: return NAME##_t<32>(T);            \
        case 48: return NAME##_t<48>(T);                                                                              \
        }                                                                                                             \
        return nullptr;                                                                                               \
    }

} // namespace sdb
