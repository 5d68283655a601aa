// tests/emu/emu.cpp -- host emulation of the sweep and traceback kernels.  CPU TEST-SUITE ONLY (built by tests/emu/Makefile).
//
// Runs the very same per-lane functions as the sm_100a kernels (sweep_core.cuh) with the CTA-level
// choreography (shuffles, prefix-max scan across the lanes of a slot, key exchange, barrier) replaced by
// loops over an array of lane states.  It is linked into libsd_emu.so, which only tests/ load; the product
// library libsd_b200.so does not contain it and fails loudly without a CUDA device.
#include <algorithm>
#include <climits>
#include <cstring>
#include <type_traits>

#include "common.h"
#include "identity_core.cuh"

namespace sdb {

namespace {

int &bad_symbol() { static thread_local int f = 0; return f; }
bool &window_violation() { static thread_local bool f = false; return f; }
bool &key_violation() { static thread_local bool f = false; return f; }

template <class P, int C, int T>
void emu_cta(const Plan &p, const Batch &b, int seg_first, int nseg_cta, int nmax,
             uint32_t *const *codes, JR *const *jr, const int *rank)
{
    // rank: pre-filter ranks of the rows of the CTA's segments ([segment][row], -1 = filtered out) or nullptr
    // NG == 1: one CTA of NT threads, `codes[0]` its backpointer block.  NG > 1: the NG CTAs that share the segment are
    // emulated side by side (thread tid belongs to group tid / NT); the only coupling between them is the column key.
    const Geometry &g = p.g;
    const int NTC = g.NT, NS = g.NS, NG = g.NG;
    const int NT = NTC * NG;
    constexpr int SPW = 32 / T;
    const uint32_t deadu = P::splat(p.deadz - 1);
    std::vector<uint32_t> Xall((size_t)NT * C, deadu), PWall((size_t)NT * C, 0u);
    std::vector<uint32_t> E(NT), carry(NT);
    std::vector<int> bref(NS, p.sc.ins), jump0(NS, 0);
    // key: the column key formed with a select over the counted row ends; dkey: the same with the kernels' arithmetic
    std::vector<int> key(NS, INT_MIN), dkey(NS, INT_MIN);
    uint32_t (*X)[C] = reinterpret_cast<uint32_t (*)[C]>(Xall.data());
    uint32_t (*PW)[C] = reinterpret_cast<uint32_t (*)[C]>(PWall.data());
    uint32_t cw[8];
    struct LaneId { bool ok; int seg_local, slot, t, sl; bool active; int n; };
    auto lane_id = [&](int tid) {
        LaneId l;
        const int grp = tid / NTC, tin = tid % NTC;
        const int warp = tin / 32, lane = tin % 32, siw = lane / T;
        l.t = lane - siw * T;
        l.ok = siw < SPW;
        const int ginst = warp * SPW + (l.ok ? siw : 0);
        if (NG > 1) {
            l.seg_local = 0; l.slot = grp * g.SG + ginst;
            l.active = l.ok && ginst < g.SG && l.slot < g.nslots && nseg_cta > 0;
            if (l.slot >= g.nslots) l.slot = g.nslots - 1;
        } else {
            l.seg_local = ginst / g.nslots; l.slot = ginst % g.nslots;
            l.active = l.ok && l.seg_local < NS && l.seg_local < nseg_cta;
        }
        if (l.seg_local >= NS) l.seg_local = 0;
        l.sl = l.slot * T + l.t;
        l.n = (l.seg_local < nseg_cta) ? b.len(seg_first + l.seg_local) : 0;
        return l;
    };
    auto load_profile = [&](int tid, const LaneId &l, int i) {
        const int sym = (i < l.n) ? symbol_code(b.text[b.off[seg_first + l.seg_local] + i], &bad_symbol()) : 0;
        for (int kk = 0; kk < C; ++kk)
            PW[tid][kk] = p.prof[(((size_t)sym * p.nsl + l.sl) * p.qp + kk / 4) * 4 + (kk % 4)];
    };
    // prologue: column 0
    for (int tid = 0; tid < NT; ++tid) {
        const LaneId l = lane_id(tid);
        const int L = p.slot_len[l.slot];
        load_profile(tid, l, 0);
        lane_pre_col0<P, C>(X[tid], PW[tid], p.sc.del, L, deadu, l.t == 0, l.t == T - 1 && L == 1);
    }
    std::vector<uint32_t> ufirst(NT), uend(NT);
    for (int i = 0;; ++i) {
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            E[tid] = lane_post<P, C>(X[tid], PW[tid], P::splat(jump0[l.seg_local] + 1), deadu, tag_regs<P>());
        }
        // exclusive prefix max of E inside each slot, restricted to the carry window (slot_scan_window on the device);
        // the full prefix maximum is formed too and any difference on a live lane is reported
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            uint32_t full = deadu, win = deadu;
            for (int d = 1; d <= l.t; ++d) { full = P::max2(full, E[tid - d]); if (d <= std::max(g.scanw, 2)) win = P::max2(win, E[tid - d]); }
            if (full != win && l.active) window_violation() = true;
            carry[tid] = win;
        }
        std::fill(key.begin(), key.end(), INT_MIN);
        std::fill(dkey.begin(), dkey.end(), INT_MIN);
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            load_profile(tid, l, i + 1);                      // profile of the next column (0-padded past the end)
            uend[tid] = lane_pass2_pre<P, C>(X[tid], carry[tid], cw, tag_regs<P>(), PW[tid], deadu,
                                             l.t == T - 1 && p.slot_len[l.slot] == 1, &ufirst[tid]);
            if (l.active && i < l.n)
                for (int w = 0; w < g.CW; ++w) codes[tid / NTC][((size_t)i * NTC + tid % NTC) * g.CW + w] = cw[w];
            const bool is_end = l.active && l.t == T - 1;
            const uint32_t u = uend[tid];
            const int R = 2 * g.M;
            int row_lo = l.slot, row_hi = g.M + l.slot;                      // tie-break index of the two rows of the slot
            if (rank && l.active) { row_lo = rank[l.seg_local * R + row_lo]; row_hi = (P::ROWS == 2) ? rank[l.seg_local * R + row_hi] : -1; }
            if (is_end) {
                int k0 = INT_MIN;
                if (row_lo >= 0) k0 = make_key(P::lo(u), p.slot_endadd[l.slot], row_lo);
                if (P::ROWS == 2 && row_hi >= 0) k0 = std::max(k0, make_key(P::hi(u), p.slot_endadd[l.slot], row_hi));
                key[l.seg_local] = std::max(key[l.seg_local], k0);
            }
            // the kernels' key of every lane (an idle lane counts towards the segment of its warp, as in the warp reduction)
            if (l.seg_local < nseg_cta) {
                const SlotKey sk = slot_key<P>(l.active, is_end, p.slot_endadd[l.slot], l.slot, g.M, rank, 0, l.seg_local, -0x800);
                dkey[l.seg_local] = std::max(dkey[l.seg_local], lane_key<P>(u, sk.kc_lo, sk.kc_hi, sk.counted));
            }
        }
        for (int s = 0; s < nseg_cta; ++s)
            if (i < b.len(seg_first + s) && dkey[s] != key[s]) key_violation() = true;
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            const uint32_t prevU = (l.t == 0) ? deadu : uend[tid - 1];
            X[tid][0] = lane_pre_first<P>(prevU, PW[tid][0], ufirst[tid], deadu, l.t == 0,
                                          C == 1 && l.t == T - 1 && p.slot_len[l.slot] == 1);
        }
        // "barrier": keys visible
        std::vector<int> shift(NS, 0);
        for (int s = 0; s < nseg_cta; ++s) {
            const int vmax = key_value(key[s]);
            if (i + 1 <= b.len(seg_first + s)) {
                jr[s][i + 1].j = vmax + bref[s] + i * p.sc.ins;
                jr[s][i + 1].row = key_row(key[s]);
            }
            jump0[s] = 4 * (vmax + p.sc.del);
            if (jump0[s] > SD_REBASE_TH || jump0[s] < -SD_REBASE_TH) { shift[s] = jump0[s]; bref[s] += jump0[s] >> 2; jump0[s] = 0; }
        }
        if (i + 1 == nmax) break;
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            if (l.seg_local < nseg_cta && shift[l.seg_local]) lane_rebase<P, C>(X[tid], shift[l.seg_local]);
        }
    }
}

// Deferred-jump sweep (sweep_lat_kernel): the CTAs of the segment's cluster side by side; the only coupling between
// the warps is the column key, published at column i and consumed at column i+1 (sweep_core.cuh: lat_*).
const int *&emu_kj() { static thread_local const int *p = nullptr; return p; }

template <class P, int C, int T>
void emu_cta_lat(const Plan &p, const Batch &b, int seg_first, int nseg_cta, int nmax,
                 uint32_t *const *codes, JR *const *jr, const int *rank)
{
    (void)nseg_cta;
    const Geometry &g = p.g;
    const int NTC = g.NT, NG = g.NG, NT = NTC * NG;
    constexpr int SPW = 32 / T;
    const TagRegs tr = tag_regs<P>();
    const uint32_t deadu = P::splat(p.deadz - 1);
    const int n = b.len(seg_first);
    std::vector<uint32_t> Xall((size_t)NT * C, deadu), PWall((size_t)NT * C, 0u), PTall((size_t)NT * C, 0u);
    uint32_t (*X)[C] = reinterpret_cast<uint32_t (*)[C]>(Xall.data());
    uint32_t (*PW)[C] = reinterpret_cast<uint32_t (*)[C]>(PWall.data());
    uint32_t (*PT)[C] = reinterpret_cast<uint32_t (*)[C]>(PTall.data());
    struct LaneId { bool ok; int slot, t, sl; bool active; };
    auto lane_id = [&](int tid) {
        LaneId l;
        const int grp = tid / NTC, tin = tid % NTC;
        const int warp = tin / 32, lane = tin % 32, siw = lane / T;
        l.t = lane - siw * T;
        l.ok = siw < SPW;
        const int ginst = warp * SPW + (l.ok ? siw : 0);
        l.slot = (NG > 1 ? grp * g.SG : 0) + ginst;
        l.active = l.ok && ginst < g.SG && l.slot < g.nslots;
        if (l.slot >= g.nslots) l.slot = g.nslots - 1;
        l.sl = l.slot * T + l.t;
        return l;
    };
    auto symbol = [&](int i) { return (i < n) ? symbol_code(b.text[b.off[seg_first] + i], &bad_symbol()) : 0; };
    auto load_profile = [&](int tid, const LaneId &l, int i) {
        const uint32_t *row = p.prof2.data() + (((size_t)symbol(i) * p.nsl + l.sl) * p.qp2) * 4;
        for (int kk = 0; kk < C; ++kk) { PW[tid][kk] = row[kk]; PT[tid][kk] = row[C + kk]; }
    };
    const int *kj = emu_kj() ? emu_kj() : p.kj;          // per-segment keys when the --ed_thr filter re-ranks the rows
    const int R = 2 * g.M;
    auto tie_lo = [&](const LaneId &l) { return rank ? rank[l.slot] : l.slot; };
    auto tie_hi = [&](const LaneId &l) { return P::ROWS == 2 ? (rank ? rank[g.M + l.slot] : g.M + l.slot) : -1; };
    (void)R;
    std::vector<uint32_t> E(NT), carry(NT), uend(NT), ufirst(NT), gout(NT);
    uint32_t cw[8];
    // column 0 in the classic form (row-0 rule, main.cpp:171-182): its jump base does not depend on any exchange
    for (int tid = 0; tid < NT; ++tid) {
        const LaneId l = lane_id(tid);
        const int L = p.slot_len[l.slot];
        load_profile(tid, l, 0);
        lane_pre_col0<P, C>(X[tid], PW[tid], p.sc.del, L, deadu, l.t == 0, l.t == T - 1 && L == 1);
        E[tid] = lane_post<P, C>(X[tid], PW[tid], P::splat(0 + 1), deadu, tr);
    }
    for (int tid = 0; tid < NT; ++tid) carry[tid] = (lane_id(tid).t == 0) ? deadu : P::max2(carry[tid - 1], E[tid - 1]);
    // the kernel's key of a lane (sweep_lat_kernel: kc_lo / kc3_lo); tag_off 0x800 in column 0, 0xC00 afterwards
    auto device_key = [&](const LaneId &l, uint32_t u, int tag_off, auto floor) {
        const SlotKey sk = slot_key<P>(l.active, l.active && l.t == T - 1, p.slot_endadd[l.slot], l.slot, g.M, rank, 0, 0, 0);
        return lane_key<P, decltype(floor)::value>(u, sk.kc_lo, sk.kc_hi, sk.counted, tag_off);
    };
    int kpub = INT_MIN;                                  // key published for the column just swept
    int dkey = INT_MIN;
    for (int tid = 0; tid < NT; ++tid) {
        const LaneId l = lane_id(tid);
        load_profile(tid, l, 1);
        uend[tid] = lane_pass2_pre<P, C>(X[tid], carry[tid], cw, tr, PW[tid], deadu, l.t == T - 1 && p.slot_len[l.slot] == 1, &ufirst[tid]);
        if (l.active)
            for (int w = 0; w < g.CW; ++w) codes[tid / NTC][((size_t)0 * NTC + tid % NTC) * g.CW + w] = cw[w];
        if (l.active && l.t == T - 1) {
            if (tie_lo(l) >= 0) kpub = std::max(kpub, make_key(P::lo(uend[tid]), p.slot_endadd[l.slot], tie_lo(l)));
            if (tie_hi(l) >= 0) kpub = std::max(kpub, make_key(P::hi(uend[tid]), p.slot_endadd[l.slot], tie_hi(l)));
        }
        dkey = std::max(dkey, device_key(l, uend[tid], 0x800, std::false_type()));
    }
    if (dkey != kpub) key_violation() = true;
    for (int tid = 0; tid < NT; ++tid) {
        const LaneId l = lane_id(tid);
        const uint32_t prevU = (l.t == 0) ? deadu : uend[tid - 1];
        X[tid][0] = lane_pre_first<P>(prevU, PW[tid][0], ufirst[tid], deadu, l.t == 0, C == 1 && l.t == T - 1 && p.slot_len[l.slot] == 1);
    }
    int jbase = p.sc.ins, jump0 = 0, kjprev = INT_MIN, adj = 0;
    auto consume = [&](int i) {                          // K[i-1] -> J[i], jump operand of column i
        const int k = std::max(kpub - adj * SD_KEY_ROWS, kjprev);
        adj = 0;
        const int vmax = key_value(k);
        jr[0][i].j = vmax + jbase; jr[0][i].row = key_row(k);
        jbase += p.sc.ins;
        jump0 = 4 * (vmax + p.sc.del);
    };
    for (int i = 1; i < nmax; ++i) {
        // a. J-independent part of column i: lane totals, windowed carry, chain
        for (int tid = 0; tid < NT; ++tid) E[tid] = lat_total<P, C>(X[tid], tr);
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            uint32_t full = deadu, win = deadu;
            for (int d = 1; d <= l.t; ++d) { full = P::max2(full, E[tid - d]); if (d <= g.scanw) win = P::max2(win, E[tid - d]); }
            if (full != win && l.active) window_violation() = true;
            carry[tid] = win;
        }
        int knew = INT_MIN;
        dkey = INT_MIN;
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            gout[tid] = lat_chain<P, C>(X[tid], carry[tid], tr);
            if (l.active && l.t == T - 1) {
                if (tie_lo(l) >= 0) knew = std::max(knew, make_key(P::ROWS == 2 ? P::lo(gout[tid]) : key_floor(P::lo(gout[tid])), p.slot_endadd[l.slot], tie_lo(l)));
                if (tie_hi(l) >= 0) knew = std::max(knew, make_key(P::hi(gout[tid]), p.slot_endadd[l.slot], tie_hi(l)));
            }
            dkey = std::max(dkey, device_key(l, gout[tid], 0xC00, std::true_type()));
        }
        if (dkey != knew) key_violation() = true;
        // c. the key of column i-1 arrives: J[i]
        consume(i);
        kpub = knew;
        kjprev = (jump0 >> 2) * SD_KEY_ROWS + kj[symbol(i)];
        // d. merge, codes
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            uend[tid] = lat_merge<P, C>(X[tid], PT[tid], P::splat(jump0 + 1), cw, tr);
            if (l.active)
                for (int w = 0; w < g.CW; ++w) codes[tid / NTC][((size_t)i * NTC + tid % NTC) * g.CW + w] = cw[w];
        }
        // e. rebase (the key published above is still in the old frame: adj)
        if (jump0 > p.lat_th || jump0 < -p.lat_th) {
            for (int tid = 0; tid < NT; ++tid) lane_rebase<P, C>(X[tid], jump0);
            jbase += jump0 >> 2; adj = jump0 >> 2; jump0 = 0;
            kjprev = kj[symbol(i)];
            for (int tid = 0; tid < NT; ++tid) uend[tid] = X[tid][C - 1];
        }
        // f. J-independent candidates of column i+1
        for (int tid = 0; tid < NT; ++tid) {
            const LaneId l = lane_id(tid);
            load_profile(tid, l, i + 1);
            const uint32_t prevU = (l.t == 0) ? deadu : uend[tid - 1];
            lane_pre<P, C>(X[tid], prevU, PW[tid], deadu, l.t == 0, l.t == T - 1 && p.slot_len[l.slot] == 1);
        }
    }
    consume(nmax);
}

template <class P> using CtaFn = void (*)(const Plan &, const Batch &, int, int, int, uint32_t *const *, JR *const *, const int *);

template <class P, int C> CtaFn<P> pick_t(int T)
{
    switch (T) {
    case 1: return emu_cta<P, C, 1>; case 2: return emu_cta<P, C, 2>; case 4: return emu_cta<P, C, 4>;
    case 8: return emu_cta<P, C, 8>; case 10: return emu_cta<P, C, 10>; case 16: return emu_cta<P, C, 16>;
    case 32: return emu_cta<P, C, 32>;
    }
    return nullptr;
}
template <class P> CtaFn<P> pick(int C, int T)
{
    switch (C) {
    case 8: return pick_t<P, 8>(T); case 12: return pick_t<P, 12>(T); case 16: return pick_t<P, 16>(T);
    case 19: return pick_t<P, 19>(T); case 20: return pick_t<P, 20>(T); case 24: return pick_t<P, 24>(T); case 32: return pick_t<P, 32>(T);
    case 48: return pick_t<P, 48>(T);
    }
    return nullptr;
}

template <class P> CtaFn<P> pick_lat(int C, int T)
{
    if (C == 6 && T == 32) return emu_cta_lat<P, 6, 32>;
    if (C == 12 && T == 16) return emu_cta_lat<P, 12, 16>;
    if (C == 12 && T == 32) return emu_cta_lat<P, 12, 32>;
    if (C == 24 && T == 8) return emu_cta_lat<P, 24, 8>;
    if (C == 24 && T == 16) return emu_cta_lat<P, 24, 16>;
    if (C == 24 && T == 32) return emu_cta_lat<P, 24, 32>;
    if (C == 48 && T == 32) return emu_cta_lat<P, 48, 32>;
    return nullptr;
}

class EmuBackend : public Backend {
public:
    const char *name() const override { return "emu"; }
    void configure(const Plan &p, const MonomerSet &ms) override { plan_ = p; ms_ = ms; }
    int64_t wave_bytes(const Batch &b, int s0, int s1) const override
    {
        CtaLayout l = make_cta_layout(plan_, b, s0, s1);
        return l.cta_code_off.back() * 4 + l.seg_j_off.back() * 8 + l.seg_rec_off.back() * 16;
    }
    int64_t wave_budget() const override
    {
        if (const char *e = getenv("SD_WAVE_BYTES")) if (atoll(e) > 0) return atoll(e);
        return (int64_t)1 << 30;
    }
    void stage(const Batch &b, int s0, int s1) override
    {
        batch_ = &b; s0_ = s0; s1_ = s1; lay_ = make_cta_layout(plan_, b, s0, s1);
        rank_.clear(); r2r_.clear();
        if (ed_thr_ < 0) return;
        // FilterMonomersForRead (main.cpp:135-149) on the host
        const int R = ms_.nrows(), nseg = s1 - s0;
        std::vector<uint8_t> rows((size_t)ms_.rows.size());
        for (size_t x = 0; x < rows.size(); ++x) rows[x] = (uint8_t)"ACGTN"[ms_.rows[x]];
        rank_.assign((size_t)nseg * R, -1); r2r_.assign((size_t)nseg * R, -1);
        std::vector<int> dist((size_t)R);
        for (int s = 0; s < nseg; ++s) {
            for (int r = 0; r < R; ++r)
                dist[(size_t)r] = hw_distance(rows.data() + ms_.row_off[r], ms_.rowlen(r), b.text + b.off[s0 + s], b.len(s0 + s));
            build_filter_tables(dist.data(), R, ed_thr_, rank_.data() + (size_t)s * R, r2r_.data() + (size_t)s * R);
        }
    }
    void execute() override
    {
        const Geometry &g = plan_.g;
        const Batch &b = *batch_;
        codes_.assign((size_t)lay_.cta_code_off.back(), 0u);
        jr_.assign((size_t)lay_.seg_j_off.back(), JR{0, 0});
        const int nseg = s1_ - s0_, nctas = (int)lay_.cta_nmax.size();
        EmuFlags::overflow() = false;
        bad_symbol() = 0;
        const int nunits = g.NG > 1 ? nseg : nctas;          // group mode: one emulated unit per segment (all its CTAs)
        for (int c = 0; c < nunits; ++c) {
            int first = g.NG > 1 ? c : c * g.NS, cnt = g.NG > 1 ? 1 : std::min(g.NS, nseg - first);
            std::vector<JR *> jp(g.NS, nullptr);
            for (int s = 0; s < cnt; ++s) jp[s] = jr_.data() + lay_.seg_j_off[first + s];
            std::vector<uint32_t *> cp(g.NG);
            for (int q = 0; q < g.NG; ++q) cp[q] = codes_.data() + lay_.cta_code_off[g.NG > 1 ? c * g.NG + q : c];
            const int nmax = lay_.cta_nmax[g.NG > 1 ? c * g.NG : c];
            const int *rk = rank_.empty() ? nullptr : rank_.data() + (size_t)first * ms_.nrows();
            if (g.lat) {
                int kj[5];
                if (rk) { lat_jump_keys(ms_, plan_.sc, rk, kj); emu_kj() = kj; } else emu_kj() = nullptr;
                if (g.packed) pick_lat<Packed16>(g.C, g.T)(plan_, b, s0_ + first, cnt, nmax, cp.data(), jp.data(), rk);
                else pick_lat<Scalar32>(g.C, g.T)(plan_, b, s0_ + first, cnt, nmax, cp.data(), jp.data(), rk);
                emu_kj() = nullptr;
                continue;
            }
            if (g.packed) pick<Packed16>(g.C, g.T)(plan_, b, s0_ + first, cnt, nmax, cp.data(), jp.data(), rk);
            else pick<Scalar32>(g.C, g.T)(plan_, b, s0_ + first, cnt, nmax, cp.data(), jp.data(), rk);
        }
        overflowed_ = g.packed && EmuFlags::overflow();
        if (window_violation()) { window_violation() = false; throw PlanError{"emulator: windowed deletion carry differs from the full prefix maximum (scan_window too small)"}; }
        if (key_violation()) { key_violation() = false; throw PlanError{"emulator: the kernels' column key differs from the select-based key (key_violation)"}; }
        if (bad_symbol()) throw PlanError{"segment contains a symbol outside ACGTN"};
        // the traceback compares segment and row symbols: bring the rows to the same (ASCII) alphabet
        rows_ascii_.resize(ms_.rows.size());
        for (size_t x = 0; x < ms_.rows.size(); ++x) rows_ascii_[x] = (uint8_t)"ACGTN"[ms_.rows[x]];
        launches += 2;
        // traceback
        recs_.assign((size_t)lay_.seg_rec_off.back(), Record{});
        cnt_.assign(nseg, 0);
        // SD_EMU_BAD_JUMP_ROW=1 (tests): the last jump of the first segment names row 4095, as a wrong column key would
        if (getenv("SD_EMU_BAD_JUMP_ROW") && atoi(getenv("SD_EMU_BAD_JUMP_ROW")) && nseg > 0)
            jr_[(size_t)lay_.seg_j_off[0] + b.len(s0_)].row = SD_KEY_ROWS - 1;
        for (int s = 0; s < nseg; ++s) {
            const int n = b.len(s0_ + s);
            if (n == 0) continue;
            auto code_at = [&](int i, int row, int rowlen, int k) {
                const RowPlace pl = place_row(g, g.NG > 1 ? 0 : s % g.NS, row);
                const int cta = g.NG > 1 ? s * g.NG + pl.grp : s / g.NS;
                const uint32_t *cbase = codes_.data() + lay_.cta_code_off[cta];
                return fetch_code(cbase + (size_t)i * g.NT * g.CW, g, pl, rowlen, k);
            };
            cnt_[s] = traceback_segment(n, jr_.data() + lay_.seg_j_off[s],
                                        b.text + b.off[s0_ + s], rows_ascii_.data(), ms_.row_off.data(),
                                        plan_.sc.ins, plan_.sc.del, plan_.sc.mismatch, plan_.sc.match, code_at,
                                        recs_.data() + lay_.seg_rec_off[s], n, true,
                                        r2r_.empty() ? nullptr : r2r_.data() + (size_t)s * ms_.nrows(), ms_.nrows());
        }
        if (const char *dir = dump_tables_dir()) dump_wave_tables(dir, g, s0_, lay_, codes_.data(), jr_.data());
    }
    void fetch(BatchResult &out) override
    {
        if (overflowed_) throw PlanError{"emulator: 16-bit overflow in the packed sweep (range proof violated)"};
        const int nseg = s1_ - s0_;
        for (int s = 0; s < nseg; ++s) {
            if (cnt_[s] == SD_TB_BAD_ROW) throw PlanError{SD_MSG_TB_BAD_ROW};
            if (cnt_[s] < 0) throw PlanError{"emulator: traceback record overflow"};
            const Record *r = recs_.data() + lay_.seg_rec_off[s];
            for (int x = cnt_[s] - 1; x >= 0; --x) out.recs.push_back(r[x]);
            out.rec_off.push_back((int64_t)out.recs.size());
        }
    }

private:
    Plan plan_; MonomerSet ms_;
    const Batch *batch_ = nullptr; int s0_ = 0, s1_ = 0;
    CtaLayout lay_;
    std::vector<uint32_t> codes_; std::vector<JR> jr_; std::vector<uint8_t> rows_ascii_; std::vector<int> rank_, r2r_; std::vector<Record> recs_; std::vector<int> cnt_;
    bool overflowed_ = false;
};

} // namespace

Backend *make_emu_backend() { return new EmuBackend(); }

// Host emulation of identity_kernel<R, L> (identity_kernels.cu): the same strips, tiles, wavefront steps and spill
// row, with the L lanes of a group walked in descending order so that lane l reads lane l-1's bottom cell of the
// previous step, exactly what the SHFL.UP delivers on the device.
template <int R, int L>
static void emu_identity_pair(const char *q, int qlen, const char *t, int tlen, std::vector<uint32_t> &scratch, int &m, int &d)
{
    const int ntiles = (qlen + L * R - 1) / (L * R);
    NwLane<R> st[L];
    uint32_t bottom[L];
    for (int tile = 0; tile < ntiles; ++tile) {
        const int base = tile * L * R;
        for (int l = 0; l < L; ++l) { nw_lane_init<R>(st[l], q, qlen, base + l * R); bottom[l] = 0; }
        const int nl = std::min(L, (qlen - base + R - 1) / R);
        const bool spill = tile + 1 < ntiles;
        for (int s = 0; s < tlen + nl - 1; ++s)
            for (int l = L - 1; l >= 0; --l) {
                uint32_t top = bottom[l ? l - 1 : 0];
                const int j = s - l;
                if (j < 0 || j >= tlen) continue;
                if (l == 0) top = tile == 0 ? (uint32_t)(j + 1) << NW_DSHIFT : scratch[j];
                bottom[l] = nw_lane_step<R>(st[l], top, (uint32_t)(uint8_t)t[j]);
                if (spill && l == L - 1) scratch[j] = bottom[l];
            }
    }
    const int fr = qlen - 1 - (ntiles - 1) * L * R;
    const uint32_t v = st[fr / R].left[fr % R];
    d = (int)(v >> NW_DSHIFT); m = (int)(v & 0xffffu);
}

int emu_identity(const IdentityArgs &a, int max_qlen, int max_tlen, double *kernel_ms, std::string &err)
{
    (void)max_qlen;
    int L = 0, R = 0;
    if (!nw_choose_geometry(a.qoff, a.nq, L, R)) { err = "unsupported SD_NW_GEOM"; return 4; }
    if (getenv("SD_PROFILE")) fprintf(stderr, "[sd_b200 profile] sd_identity (emulator): pairs %ld L %d R %d\n", (long)a.npairs, L, R);
    auto pair = emu_identity_pair<6, 32>;                   // one per NW_GEOMS entry
    if (L == 8 && R == 8) pair = emu_identity_pair<8, 8>;
    else if (L == 8 && R == 16) pair = emu_identity_pair<16, 8>;
    else if (L == 8 && R == 24) pair = emu_identity_pair<24, 8>;
    else if (L == 16 && R == 12) pair = emu_identity_pair<12, 16>;
    std::vector<uint32_t> scratch((size_t)max_tlen + 32);
    for (int64_t p = 0; p < a.npairs; ++p) {
        const int64_t qi = a.pair_q ? a.pair_q[p] : p / a.nt, ti = a.pair_q ? a.pair_t[p] : p % a.nt;
        const char *q = a.qtext + a.qoff[qi], *t = a.ttext + a.toff[ti];
        const int qlen = (int)(a.qoff[qi + 1] - a.qoff[qi]), tlen = (int)(a.toff[ti + 1] - a.toff[ti]);
        int m = 0, d = -1;
        if (qlen > 0 && tlen > 0) pair(q, qlen, t, tlen, scratch, m, d);
        a.matches[p] = m; a.columns[p] = d < 0 ? 0 : m + d;
        if (a.distance) a.distance[p] = d;
    }
    if (kernel_ms) *kernel_ms = 0;
    return 0;
}

} // namespace sdb
