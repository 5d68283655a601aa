// sweep_lat_kernel.cuh -- deferred-jump column sweep: one segment per thread-block cluster (sm_100a).
//
// The classic sweep (sweep_kernel.cuh) keeps a segment inside one CTA and pays, every column, the full round trip
// "row ends -> key -> barrier -> J[i] -> first dependent instruction".  That is fine when an SM hosts several segments,
// but with few segments (BASELINE config 1: 19; one 2 Mb array shared by 8 GPUs: 50 per GPU) most of the GPU idles and
// the run time is 5500 x (per-column latency).  Here a segment is spread over NG CTAs x NT/32 warps (a cluster; the
// CTAs land on different SMs) and uses the deferred form of the recurrence (sweep_core.cuh: lat_total / lat_chain /
// lat_merge): the vector work of column i does not need J[i] until its very last instruction per register, so the key of
// column i is published one whole column before it is consumed and the exchange -- distributed shared memory inside
// the cluster, one 8-byte (column, key) word per warp and destination CTA -- is off the critical path.
//
//   per column and warp:   lane totals -> windowed carry (plan.cpp: scan_window) -> chain -> key of the row ends ->
//                          CREDUX -> st.shared::cluster to every CTA of the cluster            (publish K0[i])
//                          poll own shared memory for K0[i-1] of all warps -> J[i], jump operand  (published long ago)
//                          merge + re-tag + 2-bit codes -> store; profile row i+1; candidates of column i+1
//
// No barrier of any kind inside the column loop: the (column, key) words carry their own epoch, four buffers rotate
// (a warp can run at most two columns ahead of the slowest one, see the comment at `publish`).
// Reference semantics: stringdecomposer/src/main.cpp:171-216 (forward sweep, per-column jump maximum, final argmax).
#pragma once
#include <cuda_runtime.h>
#include <climits>

#include "common.h"
#include "sweep_kernel.cuh"

namespace sdb {

struct LatArgs {
    const uint4 *prof2; int nsl_total, qp2;            // [5][nsl_total][qp2] uint4: words [0,C) = p, [C,2C) = PT
    const uint8_t *bases; const int64_t *seg_off; int nseg;
    const int64_t *cta_code_off; const int64_t *seg_j_off;
    uint32_t *codes; JR *jr;
    const int *slot_len; const int *slot_endadd;
    int nslots, M, NT, CW, NG, SG;
    int ins, del, deadz, lat_th, scanw;
    int kj[5];                                          // best jump-derived row-end key per symbol (plan.cpp: lat_jump_keys)
    const int *seg_kj;                                  // [segment][5]: the same per segment when --ed_thr re-ranks the rows, or null
    const int *rank;                                    // --ed_thr pre-filter ranks [segment][row] or null
    int seg_stride;                                     // bytes of the symbol buffer
    TagRegs tr;
    int *bad_symbol, *error;
    long long *dbg;                                     // SD_LAT_TIMING: [warp][8] cycles per phase, summed over the columns
};

constexpr int LAT_NBUF = 4;

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Carry of the deletion chain into a lane: maximum of the lane totals of the WN nearest lanes on its left inside the slot
// (exact when WN >= plan.cpp: scan_window; a larger window is always correct).  WN independent shuffles, each masked by
// the shuffle's own "source lane in range" flag, then a ternary max tree -- one shuffle latency, no compares.
// WN == 0: log-depth scan over the whole slot (any window).
template <class P, int T, int WN>
__device__ __forceinline__ uint32_t window_carry(uint32_t total, int t, uint32_t dead)
{
    if (T == 1) return dead;
    if (WN > 0) {
        constexpr int N = WN <= 0 ? 1 : (WN < T - 1 ? WN : T - 1);
        uint32_t r[N];
        if ((T & (T - 1)) == 0) {
            constexpr int cseg = (32 - T) << 8;         // shfl.up clamp: segments of T lanes
#pragma unroll
            for (int d = 1; d <= N; ++d)
                asm volatile("{ .reg .pred q; .reg .b32 v; shfl.sync.up.b32 v|q, %1, %2, %3, 0xffffffff; selp.b32 %0, v, %4, q; }"
                             : "=r"(r[d - 1]) : "r"(total), "r"(d), "r"(cseg), "r"(dead));
        } else {
#pragma unroll
            for (int d = 1; d <= N; ++d) { r[d - 1] = __shfl_up_sync(0xffffffffu, total, d); if (t < d) r[d - 1] = dead; }
        }
        return tree_max<P, N>(r);
    }
    uint32_t pv = __shfl_up_sync(0xffffffffu, total, 1);
    if (t == 0) pv = dead;
#pragma unroll
    for (int d = 1; d < T; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, pv, d);
        if (t >= d) pv = P::max2(pv, o);
    }
    return pv;
}

// ST: the segment symbols are not staged in shared memory (whose size then does not depend on the segment length):
// every thread loads the symbol of column i+2 from global memory while it sweeps column i (one L1 broadcast per warp);
// column i uses the symbol of column i+1 for its look-ahead profile load, so the load has a whole column to land.
template <class P, int C, int T, int WN, bool TM = false, bool ST = false>
__global__ void sweep_lat_kernel(const LatArgs a)
{
    extern __shared__ uint4 smem_u4[];
    constexpr int SPW = 32 / T;
    const int NT = a.NT, NG = a.NG;
    const int wpc = NT >> 5;                             // warps per CTA
    const int nwtot = wpc * NG;                          // warps of the segment (all CTAs of the cluster), <= 32
    const int sgt = wpc * SPW * T;                       // profile rows (slot lanes) kept by this CTA
    uint4 *sprof = smem_u4;                              // [5][sgt][qp2]
    unsigned long long *xkey = reinterpret_cast<unsigned long long *>(sprof + (size_t)5 * sgt * a.qp2);   // [LAT_NBUF][32]
    int *skj = reinterpret_cast<int *>(xkey + LAT_NBUF * 32);                                                // [8]
    uint8_t *schar = reinterpret_cast<uint8_t *>(skj + 8);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int seg = blockIdx.x / NG;
    const int grp = NG > 1 ? (int)cluster_ctarank() : 0;
    const int siw = lane / T, t = lane - siw * T;
    const bool lane_ok = siw < SPW;
    const int ginst = warp * SPW + (lane_ok ? siw : 0);
    int slot = (NG > 1 ? grp * a.SG : 0) + ginst;
    const bool active = lane_ok && ginst < a.SG && slot < a.nslots;
    if (slot >= a.nslots) slot = a.nslots - 1;

    const int64_t o = a.seg_off[seg];
    const int n = (int)(a.seg_off[seg + 1] - o);

    // stage: profile slice of this CTA's slots, the segment's symbols, the per-symbol jump keys, empty exchange words
    for (int x = tid; x < 5 * sgt * a.qp2; x += NT) {
        const int sym = x / (sgt * a.qp2), r = x - sym * (sgt * a.qp2);
        const int row = min((NG > 1 ? grp * a.SG * T : 0) + r / a.qp2, a.nsl_total - 1);
        sprof[x] = a.prof2[((size_t)sym * a.nsl_total + row) * a.qp2 + (r % a.qp2)];
    }
    for (int x = tid; x < (ST ? 0 : a.seg_stride); x += NT) schar[x] = (uint8_t)((x < n) ? symbol_code(a.bases[o + x], a.bad_symbol) : 0);
    if (tid < 5) skj[tid] = a.seg_kj ? a.seg_kj[(size_t)seg * 5 + tid] : a.kj[tid];
    for (int x = tid; x < LAT_NBUF * 32; x += NT) xkey[x] = 0ull;            // column tag 0 = nothing published
    __syncthreads();
    if (NG > 1) cluster_sync_all();                      // nobody may store into a CTA that has not cleared its words yet

    const int L = a.slot_len[slot];
    const int endadd = a.slot_endadd[slot];
    const uint32_t deadu = P::splat(a.deadz - 1);
    const TagRegs tr = a.tr;
    const bool kill_first = (t == 0), kill_last = (t == T - 1 && L == 1);
    const bool is_end = active && t == T - 1;
    const bool j_writer = grp == 0 && tid == 0;
    // key = (half << 10) + const: the row-end word is U (tag 2: 0x800 too much) in column 0, g (tag 3: 0xC00) afterwards
    const SlotKey sk = slot_key<P>(active, is_end, endadd, slot, a.M, a.rank, seg, 0, 0);
    const int kc3_lo = sk.kc_lo - 0xC00, kc3_hi = sk.kc_hi - 0xC00;
    JR *jptr = a.jr + a.seg_j_off[seg];
    uint32_t *cptr = a.codes + a.cta_code_off[(size_t)seg * NG + grp] + (size_t)tid * a.CW;
    const size_t cstride = (size_t)NT * a.CW;
    const uint32_t myprof = (uint32_t)__cvta_generic_to_shared(sprof + (size_t)(ginst * T + t) * a.qp2);
    const uint32_t sym_stride = 16u * (uint32_t)(sgt * a.qp2);         // bytes between the rows of two symbols

    // exchange: warp w of CTA c owns word [buf][c*wpc + w] in EVERY CTA of the cluster; lane c of a warp stores to CTA c.
    // Lanes >= nwtot read (again) the word of warp lane % nwtot, so that all lanes of a warp run the same poll.
    const uint32_t xkey_s = (uint32_t)__cvta_generic_to_shared(xkey);
    uint32_t xremote = xkey_s;
    if (NG > 1 && lane < NG) asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(xremote) : "r"(xkey_s), "r"(lane));
    // generic pointer of this lane's destination word in buffer 0: {shared::cluster offset, window high word}; the
    // buffers are 256 B apart and the window is aligned, so the per-column offset is added to the low word only
    uint32_t pub_lo, pub_hi;
    {
        unsigned long long gen;
        asm volatile("{ .reg .u64 a; cvt.u64.u32 a, %1; cvta.shared::cluster.u64 %0, a; }" : "=l"(gen) : "r"(xremote + 8u * (uint32_t)(grp * wpc + warp)));
        pub_lo = (uint32_t)gen; pub_hi = (uint32_t)(gen >> 32);
    }
    const uint32_t rcv_addr = xkey_s + 8u * (uint32_t)(lane % nwtot);
    const bool pub_lane = lane < NG;
    // A warp publishes K0[i] and only then waits for K0[i-1]; when it publishes K0[i+3] everybody has published
    // K0[i+1], hence consumed K0[i-1] -- the word it overwrites (buffer (i+3) & 3 == (i-1) & 3) is no longer needed.
    auto publish = [&](uint32_t boff, int tag, int key) {                          // boff = 256 * (column & 3)
        unsigned long long dst;
        asm("mov.b64 %0, {%1, %2};" : "=l"(dst) : "r"(pub_lo + boff), "r"(pub_hi));
        if (pub_lane) asm volatile("st.relaxed.cluster.v2.b32 [%0], {%1, %2};" ::"l"(dst), "r"(key), "r"(tag) : "memory");
    };
    // every lane polls one word; the warp leaves the loop together (a vote keeps the control flow convergent, so the
    // shuffles and reductions further down need no divergence checks)
    auto receive = [&](uint32_t boff, int tag) {
        const uint32_t src = rcv_addr + boff;
        int key, got;
        unsigned spins = 0;
        for (;;) {
            asm volatile("ld.volatile.shared.v2.b32 {%0, %1}, [%2];" : "=r"(key), "=r"(got) : "r"(src) : "memory");
            if (__all_sync(0xffffffffu, got == tag)) break;
            if (++spins > (1u << 22)) { *a.error = 1; break; }                  // a partner died: fail instead of hanging
        }
        return __reduce_max_sync(0xffffffffu, key);
    };

    constexpr int CQ2 = (2 * C + 3) / 4;                 // uint4 per profile row
    constexpr int QP_END = (C + 3) / 4;                  // uint4 [0, QP_END) hold p
    constexpr int QT_BEG = C / 4;                        // uint4 [QT_BEG, CQ2) hold PT
    uint32_t X[C], pw[C], pt[C];
    // profile rows are addressed in the shared window directly (a generic pointer would be re-converted every column)
    auto lds128 = [](uint32_t addr) {
        uint4 v;
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
        return v;
    };
    auto load_p = [&](uint32_t pp) {
#pragma unroll
        for (int q = 0; q < QP_END; ++q) {
            const uint4 v = lds128(pp + 16u * q);
            if (4 * q + 0 < C) pw[4 * q + 0] = v.x;
            if (4 * q + 1 < C) pw[4 * q + 1] = v.y;
            if (4 * q + 2 < C) pw[4 * q + 2] = v.z;
            if (4 * q + 3 < C) pw[4 * q + 3] = v.w;
        }
    };
    auto load_pt = [&](uint32_t pp) {
#pragma unroll
        for (int q = QT_BEG; q < CQ2; ++q) {
            const uint4 v = lds128(pp + 16u * q);
            if (4 * q + 0 >= C && 4 * q + 0 < 2 * C) pt[4 * q + 0 - C] = v.x;
            if (4 * q + 1 >= C && 4 * q + 1 < 2 * C) pt[4 * q + 1 - C] = v.y;
            if (4 * q + 2 >= C && 4 * q + 2 < 2 * C) pt[4 * q + 2 - C] = v.z;
            if (4 * q + 3 >= C && 4 * q + 3 < 2 * C) pt[4 * q + 3 - C] = v.w;
        }
    };
    constexpr int NW = (C + P::CELLS_PER_WORD - 1) / P::CELLS_PER_WORD;
    uint32_t cw[NW];
    auto store_codes = [&]() {
        if (active) store_code_words(cptr, cw);
        cptr += cstride;
    };

    // ST: symbols past the end of the segment read as 0, like the 0-padded buffer
    auto symbol = [&](int i) { return (i < n) ? symbol_code(__ldg(a.bases + o + i), a.bad_symbol) : 0; };

    // ---- column 0 in the classic form: its jump base (row-0 rule, main.cpp:171-182) needs no exchange -------------
#pragma unroll
    for (int kk = 0; kk < C; ++kk) X[kk] = deadu;
    load_p(myprof + (ST ? symbol(0) : schar[0]) * sym_stride);
    lane_pre_col0<P, C>(X, pw, a.del, L, deadu, kill_first, kill_last);
    {
        const uint32_t E = lane_post<P, C>(X, pw, P::splat(1), deadu, tr);
        const uint32_t carry = window_carry<P, T, 0>(E, t, deadu);
        const uint32_t pn = myprof + (ST ? symbol(1) : schar[1]) * sym_stride;
        load_p(pn);
        load_pt(pn);
        uint32_t ufirst;
        const uint32_t uend = lane_pass2_pre<P, C>(X, carry, cw, tr, pw, deadu, kill_last, &ufirst);
        store_codes();
        publish(0u, 1, __reduce_max_sync(0xffffffffu, lane_key<P>(uend, sk.kc_lo, sk.kc_hi, sk.counted, 0x800)));
        X[0] = next_first_cell<P, C, T>(uend, pw[0], ufirst, deadu, t, kill_first, kill_last);
    }

    int jbase = a.ins;            // Bref + (i-1)*ins when J[i] is formed
    int jump0 = 0;                // 4*(B[i] - Bref)
    int kjprev = INT_MIN;         // key of the best jump-derived row end of the previous column (none in column 0)
    int adjk = 0;                 // rebase after the key in flight was published: that key is still in the old frame
    // loop invariants pinned in registers (ptxas would otherwise re-read them from the constant bank every column)
    int th, th2, del4p1, ins;
    TagRegs trr;
    asm volatile("mov.b32 %0, %1;" : "=r"(th) : "r"(a.lat_th));
    asm volatile("mov.b32 %0, %1;" : "=r"(th2) : "r"(2 * a.lat_th));
    asm volatile("mov.b32 %0, %1;" : "=r"(del4p1) : "r"(4 * a.del + 1));
    asm volatile("mov.b32 %0, %1;" : "=r"(ins) : "r"(a.ins));
    asm volatile("mov.b32 %0, %1;" : "=r"(trr.mask3) : "r"(tr.mask3));
    asm volatile("mov.b32 %0, %1;" : "=r"(trr.one) : "r"(tr.one));
    long long tacc[7] = {0, 0, 0, 0, 0, 0, 0}, tprev = 0;
    auto tick = [&](int ph) { if (TM) { const long long c = clock64(); tacc[ph] += c - tprev; tprev = c; } };
    if (TM) tprev = clock64();
    const uint8_t *sp = schar + 2;
    int sym = ST ? symbol(1) : schar[1];
    int sym_ahead = ST ? symbol(2) : 0;       // ST: symbol of column i+1, loaded one column before it is needed
    uint32_t boff = 256u, boff_prev = 0u;                  // 256 * (i & 3), 256 * ((i-1) & 3)
#pragma unroll 1
    for (int i = 1; i < n; ++i, ++sp) {
        // J-independent part of column i (X holds max(diag, up))
        const uint32_t total = lat_total<P, C>(X, trr);
        const int symn = ST ? sym_ahead : sp[0];
        if (ST) sym_ahead = symbol(i + 2);
        const uint32_t pn = myprof + (uint32_t)symn * sym_stride;
        const uint32_t carry = window_carry<P, T, WN>(total, t, deadu);
        tick(0);
        load_p(pn);                                       // flies during the chain
        const uint32_t g = lat_chain<P, C>(X, carry, trr);
        tick(1);
        publish(boff, i + 1, __reduce_max_sync(0xffffffffu, lane_key<P, true>(g, kc3_lo, kc3_hi, sk.counted)));
        tick(2);

        // J[i] from the key of column i-1, published one column ago
        const int k2 = max(receive(boff_prev, i) - adjk, kjprev);
        tick(3);
        boff_prev = boff; boff = (boff + 256u) & 0x300u;
        adjk = 0;
        const int vmax = k2 >> 12;
        ++jptr;                                            // J[i], lowest row attaining it: one predicated 8-byte store
        asm volatile("{ .reg .pred q; setp.ne.b32 q, %0, 0; @q st.global.v2.b32 [%1], {%2, %3}; }"
                     ::"r"((int)j_writer), "l"(jptr), "r"(vmax + jbase), "r"(~k2 & (SD_KEY_ROWS - 1)) : "memory");
        jbase += ins;
        const int j1 = 4 * vmax + del4p1;                 // jump0 + 1
        jump0 = j1 - 1;
        kjprev = (jump0 >> 2) * SD_KEY_ROWS + skj[sym];

        lat_merge<P, C>(X, pt, P::splat(j1), cw, trr);
        store_codes();
        tick(4);
        load_pt(pn);
        if ((unsigned)(jump0 + th) > (unsigned)th2) {
            lane_rebase<P, C>(X, jump0);
            jbase += jump0 >> 2; adjk = (jump0 >> 2) * SD_KEY_ROWS; jump0 = 0;
            kjprev = skj[sym];
        }
        sym = symn;
        // candidates of column i+1
        uint32_t prevU = deadu;
        if (T > 1 && (T & (T - 1)) == 0) {
            constexpr int cseg = (32 - T) << 8;
            asm volatile("{ .reg .pred q; .reg .b32 v; shfl.sync.up.b32 v|q, %1, 1, %2, 0xffffffff; selp.b32 %0, v, %3, q; }"
                         : "=r"(prevU) : "r"(X[C - 1]), "r"(cseg), "r"(deadu));
        } else if (T > 1) {
            prevU = __shfl_up_sync(0xffffffffu, X[C - 1], 1);
            if (t == 0) prevU = deadu;
        }
        lane_pre<P, C>(X, prevU, pw, deadu, kill_first, kill_last);
        tick(5);
    }
    if (TM && a.dbg && lane == 0) {
#pragma unroll
        for (int q = 0; q < 6; ++q) a.dbg[((size_t)blockIdx.x * wpc + warp) * 8 + q] = tacc[q];
        a.dbg[((size_t)blockIdx.x * wpc + warp) * 8 + 6] = n - 1;
    }
    {
        const int k2 = max(receive(256u * (uint32_t)((n - 1) & (LAT_NBUF - 1)), n) - adjk, kjprev);
        if (j_writer) jptr[1] = JR{(k2 >> 12) + jbase, ~k2 & (SD_KEY_ROWS - 1)};          // jptr points at J[n-1]
    }
    if (NG > 1) cluster_sync_all();                      // no CTA may retire while partners still store into it
}

// WN: carry window the kernel is compiled for (0 = any, log-depth scan)
const void *sweep_lat_lookup_p16(const Geometry &g);
const void *sweep_lat_lookup_s32(const Geometry &g);
const void *sweep_lat_lookup_p16_st(const Geometry &g);                  // ST: symbols streamed from global memory
const void *sweep_lat_lookup_s32_st(const Geometry &g);
const void *sweep_lat_timing_lookup_p16(const Geometry &g);             // instrumented twins (SD_LAT_TIMING=1, exploration only)

// smallest compiled window >= W (= g.scanw)
#define SD_LAT_PICK(POLICY, CC, TT, TMF, STF)                                                                        \
    if (C == CC && T == TT) {                                                                                         \
        if (W <= 2) return (const void *)sweep_lat_kernel<POLICY, CC, TT, 2, TMF, STF>;                               \
        if (W <= 4) return (const void *)sweep_lat_kernel<POLICY, CC, TT, 4, TMF, STF>;                               \
        if (W <= 8) return (const void *)sweep_lat_kernel<POLICY, CC, TT, 8, TMF, STF>;                               \
        return (const void *)sweep_lat_kernel<POLICY, CC, TT, 0, TMF, STF>;                                           \
    }

#define SD_INSTANTIATE_LAT(NAME, POLICY, STF)                                                                        \
    const void *NAME(const Geometry &g)                                                                               \
    {                                                                                                                 \
        const int C = g.C, T = g.T, W = g.scanw;                                                                      \
        SD_LAT_PICK(POLICY, 6, 32, false, STF) SD_LAT_PICK(POLICY, 12, 16, false, STF)                                \
        SD_LAT_PICK(POLICY, 12, 32, false, STF) SD_LAT_PICK(POLICY, 24, 8, false, STF)                                \
        SD_LAT_PICK(POLICY, 24, 16, false, STF) SD_LAT_PICK(POLICY, 24, 32, false, STF)                               \
        SD_LAT_PICK(POLICY, 48, 32, false, STF)                                                                       \
        return nullptr;                                                                                               \
    }

} // namespace sdb
