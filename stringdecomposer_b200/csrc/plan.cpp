// plan.cpp -- DP-row construction, score-range analysis (s16x2 vs s32), launch geometry, profile table.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <climits>
#include <cstring>

#include "common.h"

namespace sdb {

// Rows = forward monomers in input order followed by the reverse complement of each, in the same order.
// Restates add_reverse_complement / reverse_complement (main.cpp:348-371): this order is the arg-max
// tie-break order of the whole DP (main.cpp:212, :230-236).
void build_monomer_set(const std::vector<std::string> &forward, MonomerSet &ms)
{
    ms.M = (int)forward.size();
    ms.rows.clear(); ms.row_off.assign(1, 0);
    ms.Lmax = 0; ms.Lmin = 1 << 30;
    for (int pass = 0; pass < 2; ++pass) {
        for (const std::string &m : forward) {
            int L = (int)m.size();
            if (L == 0) throw PlanError{"empty monomer sequence (the reference indexes seq[0] of it, main.cpp:173)"};
            for (int x = 0; x < L; ++x) {
                int c = base_code(pass == 0 ? m[x] : m[L - 1 - x]);
                if (c < 0) throw PlanError{"monomer contains a symbol outside ACGTN"};
                if (pass == 1 && c < 4) c = 3 - c;            // A<->T, C<->G, N stays N (main.cpp:350)
                ms.rows.push_back((uint8_t)c);
            }
            ms.row_off.push_back((int)ms.rows.size());
            ms.Lmax = std::max(ms.Lmax, L); ms.Lmin = std::min(ms.Lmin, L);
        }
    }
    if (ms.M == 0) { ms.Lmax = ms.Lmin = 0; }
}

// Range proof for the packed s16x2 representation (DESIGN.md "score range").  With D=-del>=0, I=-ins>=0:
//   live relative cells  rel in [min(s''min,0), D*(Lmax+1) + I + max(smax,0)]          (s'' = s + I + D)
//   column shift         |delta| <= D*(Lmax+1) + I + max(|smax|,|smin|) + 1
//   registers are relative to Bref with |4*(B[i]-Bref)| <= SD_REBASE_TH (rebase otherwise)
//   pad/dead level       s''pad = -(relmax + |s''min| + TH/4 + 2)
// Every intermediate of lane_pre/post/pass2/rebase is (value +- 4*delta +- TH +- small), so 16 bits suffice when
//   4*(|s''pad| + relmax + 2*dmax) + 2*TH + 64 <= 32767.
// The host emulator traps any 16-bit overflow, which is how the tests keep this proof honest.
bool packed_range_ok(const MonomerSet &ms, const Scoring &sc, int *deadz, int *pad_s)
{
    if (sc.ins > 0 || sc.del > 0) return false;
    const int64_t D = -(int64_t)sc.del, I = -(int64_t)sc.ins;
    const int64_t smax = std::max(sc.match, sc.mismatch), smin = std::min(sc.match, sc.mismatch);
    const int64_t s2max = smax + I + D, s2min = smin + I + D;
    const int64_t L = std::max(ms.Lmax, 2);
    const int64_t relmax = D * (L + 2) + I + std::max<int64_t>(smax, 0) + 2 * std::max(std::llabs(s2min), std::llabs(s2max)) + 4;
    const int64_t dmax = D * (L + 1) + I + std::max(std::llabs(smax), std::llabs(smin)) + 1;
    const int64_t pad = relmax + std::llabs(s2min) + SD_REBASE_TH / 4 + 2;
    if (4 * (pad + relmax + 2 * dmax) + 2 * SD_REBASE_TH + 64 > 32767) return false;
    if (deadz) *deadz = (int)(-4 * pad + 3);
    if (pad_s) *pad_s = (int)(-pad);
    return true;
}

// Kernel instantiations compiled into the library (sweep_kernels.cu instantiates exactly this table).
static const int kC[] = {8, 12, 16, 19, 20, 24, 32, 48};
static const int kT[] = {1, 2, 4, 8, 10, 16, 32};
bool geometry_compiled(int packed, int C, int T)
{
    (void)packed;
    bool c = false, t = false;
    for (int x : kC) c |= (x == C);
    for (int x : kT) t |= (x == T);
    return c && t;
}

// (C, T) pairs the deferred-jump kernel is compiled for (sweep_inst_lat_*.cu instantiates exactly this table)
static const int kLatGeom[][2] = {{6, 32}, {12, 16}, {12, 32}, {24, 8}, {24, 16}, {24, 32}, {48, 32}};
bool lat_geometry_compiled(int C, int T)
{
    for (auto &g : kLatGeom) if (g[0] == C && g[1] == T) return true;
    return false;
}

void lat_jump_keys(const MonomerSet &ms, const Scoring &sc, const int *rank_of_row, int out[5])
{
    const int shift = -sc.ins - sc.del;
    for (int sym = 0; sym < 5; ++sym) {
        int best = INT_MIN;
        for (int r = 0; r < ms.nrows(); ++r) {
            const int tb = rank_of_row ? rank_of_row[r] : r;
            if (tb < 0) continue;
            int s2 = INT_MIN;
            for (int k = ms.row_off[r]; k < ms.row_off[r + 1]; ++k) s2 = std::max(s2, (ms.rows[k] == sym ? sc.match : sc.mismatch) + shift);
            best = std::max(best, make_key(4 * s2, (ms.rowlen(r) - 1) * sc.del, tb));
        }
        out[sym] = best;
    }
}

// Windowed deletion carry.  The carry into lane t of a slot is the maximum of the lane totals of ALL lanes on its left.
// Scores along a row never decrease in the shifted domain (deletions are free), so a candidate of an earlier lane is
// dominated by any later candidate of the same or a better score class: "up" candidates by the nearest lane, diagonal
// and jump candidates of the better class (match, normally) by the nearest lane that holds a position of that class
// for the column's symbol, those of the worse class by either.  The window is the largest such distance over all
// symbols, slots, lanes and (packed) both rows of a slot; it is a property of the monomer set, not of the reads.
int scan_window(const MonomerSet &ms, const Scoring &sc, int packed, int C, int T)
{
    if (T <= 1) return 0;
    const int nslots = packed ? ms.M : 2 * ms.M;
    const int SL = C * T;
    int W = 1;
    for (int slot = 0; slot < nslots; ++slot) {
        const int L = ms.rowlen(slot), lead = (L == 1) ? SL - 1 : 0;
        for (int half = 0; half < (packed ? 2 : 1); ++half) {
            const uint8_t *row = ms.rows.data() + ms.row_off[half ? ms.M + slot : slot];
            for (int sym = 0; sym < 5; ++sym) {
                // nearest lane so far that holds a position of the better / the worse score class (pad cells: neither --
                // the lanes behind a short row must look all the way back to its last real cells)
                int last_hi = -1, last_lo = -1;
                for (int t = 0; t < T; ++t) {
                    if (t > 0) {
                        const int need = last_hi >= 0 ? last_hi : last_lo;
                        if (need >= 0) W = std::max(W, t - need);
                    }
                    for (int kk = 0; kk < C; ++kk) {
                        const int k = t * C + kk - lead;
                        if (k < 0 || k >= L) continue;
                        const int s = row[k] == sym ? sc.match : sc.mismatch;
                        if (s >= std::max(sc.match, sc.mismatch)) last_hi = t; else last_lo = t;
                    }
                }
            }
        }
    }
    return std::min(W, T - 1);
}

static const size_t kSmemLimit = 200 * 1024;

size_t Plan::smem_bytes(int seg_stride) const
{
    return prof.size() * 4 + (size_t)g.NS * (size_t)seg_stride + 3 * (size_t)g.NS * 4 + 64;
}

// Cost model used to pick (C, T, NS), calibrated on B200 runs (DESIGN.md section 6).  The sweep is bound by the
// ALU pipe (every DPX/VIMNMX/LOP3 instruction issues at 16 lanes/clk per SM sub-partition): a warp needs
//   alu = 2 * (4.5*C + 43 + 4*ceil(log2 T))   ALU-pipe cycles per column,
// a sub-partition hosting w warps advances them one column in max(w*alu/0.75, lat) cycles (0.75: the pipe
// utilisation reached with the CTA-wide column barrier), and an SM hosts k CTAs (k limited by shared memory --
// the profile table is per CTA -- and registers).  Small launches are quantised: the slowest SM sets the time.
static double geometry_cost(int C, int T, int NS, int NT, size_t smem_bytes, int64_t nseg, int nmax)
{
    const int lg = (T > 1) ? 32 - __builtin_clz((unsigned)(T - 1)) : 0;
    const int W = NT / 32;
    const double alu = 2.0 * (4.5 * C + 43.0 + 4.0 * lg);
    const double lat = 330.0 + 9.0 * C + (T <= 10 ? 30.0 : 75.0) * lg;     // measured: (19,10) 620, (24,8) 650, (12,16) 750 cycles
    int kmax = (int)std::min<size_t>((227u * 1024u) / std::max<size_t>(smem_bytes, 1), 32);
    kmax = std::min(kmax, 65536 / (NT * (2 * C + 40)));       // registers: X[C] + profile[C] + ~40
    kmax = std::min(kmax, 64 / W);
    if (kmax < 1) return 1e300;
    const int64_t ncta = (nseg + NS - 1) / NS;
    auto col_cost = [&](int k) { return std::max(std::ceil(k * W / 4.0) * alu / 0.75, lat); };
    if (ncta <= (int64_t)148 * kmax) return (double)nmax * col_cost((int)((ncta + 147) / 148));
    return (double)nmax * ((double)ncta / (148.0 * kmax)) * col_cost(kmax);
}

Plan make_plan(const MonomerSet &ms, const Scoring &sc, int max_seg_len, int64_t nseg_hint)
{
    Plan p;
    p.sc = sc;
    if (ms.M <= 0) throw PlanError{"no monomers"};
    if (ms.nrows() > SD_KEY_ROWS) throw PlanError{"more than 2048 monomers are not supported by this build"};
    // The reference guards every candidate with '> INF' (INF=-1000000, main.cpp:156,191-201); those guards are
    // no-ops only while every true score stays above INF.  Refuse instead of diverging silently.
    {
        int64_t a = std::max(std::abs(sc.ins), std::abs(sc.mismatch));
        int64_t lo = (int64_t)max_seg_len * a + 2ll * ms.Lmax * std::abs(sc.del) + 2ll * std::abs(sc.mismatch) + std::abs(sc.match);
        int64_t hi = ((int64_t)max_seg_len + ms.Lmax) * std::max({std::abs(sc.match), std::abs(sc.mismatch), std::abs(sc.ins), std::abs(sc.del)});
        if (lo >= 999000) throw PlanError{"scores can reach the reference's INF sentinel (-1000000): outside the supported domain"};
        if (hi >= (1 << 23)) throw PlanError{"scores exceed the exact float range of the reference's output"};
    }
    int pad_s = 0;
    int packed = packed_range_ok(ms, sc, &p.deadz, &pad_s) ? 1 : 0;
    if (const char *e = getenv("SD_FORCE_S32")) if (atoi(e)) packed = 0;
    if (!packed) { pad_s = -(1 << 26); p.deadz = 4 * pad_s + 3; }

    const int nslots = packed ? ms.M : 2 * ms.M;
    int bestC = 0, bestT = 0, bestNS = 0, bestNT = 0; double best = 1e300;
    int fC = 0, fT = 0, fNS = 0;
    if (const char *e = getenv("SD_GEOM")) sscanf(e, "%d,%d,%d", &fC, &fT, &fNS);
    // Symbols of the segments: staged in shared memory (NS * (max_seg_len + 64) bytes) wherever that fits, streamed from
    // global memory (no length term) where it does not.  SD_STREAM_SYMBOLS=1 (tests) streams on every shape.
    const bool force_stream = getenv("SD_STREAM_SYMBOLS") && atoi(getenv("SD_STREAM_SYMBOLS")) > 0;
    int stream = force_stream ? 1 : 0;
    // lanes with more than 24 cells run into register-limited occupancy and long dependent chains (measured);
    // they are only considered for rows that need them
    const bool need_big = ms.Lmax > 24 * 32;
    auto classic_search = [&](bool streamed) {
        for (int C : kC) for (int T : kT) {
            if (fC && (C != fC || T != fT)) continue;
            if (C * T < ms.Lmax) continue;
            if (!fC && C > 24 && !need_big) continue;
            int ls = nslots * T;                        // lanes per segment
            if (ls > 1024) continue;
            const int qpc = ((C + 3) / 4) | 1;
            size_t prof_bytes = (size_t)5 * qpc * ls * 16;
            for (int NS = 1; NS <= 16; ++NS) {
                if (fNS && NS != fNS) continue;
                const int spw = 32 / T;
                int NT = (NS * nslots + spw - 1) / spw * 32;
                if (NT > 1024) break;
                if ((int64_t)NT * (2 * C + 40) > 65536) continue;   // register file (verified against the real kernel at configure time)
                size_t smem = prof_bytes + (streamed ? 0 : (size_t)NS * ((size_t)max_seg_len + 64)) + 256;
                if (smem > kSmemLimit) continue;
                double cost = geometry_cost(C, T, NS, NT, smem, std::max<int64_t>(nseg_hint, 1), std::max(max_seg_len, 1));
                cost *= 1.0 + 0.002 * (NS - 1);           // ties: prefer fewer segments per CTA
                if (cost < best) { best = cost; bestC = C; bestT = T; bestNS = NS; bestNT = NT; }
            }
        }
    };
    classic_search(stream);
    Geometry &g = p.g;
    g.NG = 1;
    int force_sg = 0;
    if (const char *e = getenv("SD_GROUP_SLOTS")) force_sg = atoi(e);
    const bool lat_forced = getenv("SD_LAT") && atoi(getenv("SD_LAT")) > 0;
    if (lat_forced && !bestC) { bestC = 6; bestT = 32; bestNS = 1; bestNT = 32; }      // placeholder, replaced below
    else if (!bestC || force_sg > 0) {
        // The monomer set does not fit one CTA (threads, registers or the shared-memory profile table): split the slots
        // into NG groups, one CTA each; the per-column key then meets in global memory (sweep_group_kernel).
        // fewest partner CTAs per segment first (the exchange latency grows with them), then least padding
        int gC = 0, gT = 0, gNG = 1 << 30;
        for (int C : kC) for (int T : kT) {
            if (fC && (C != fC || T != fT)) continue;
            if (C * T < ms.Lmax || (C > 24 && !need_big && !fC)) continue;
            const int spw_c = 32 / T, qp_c = ((C + 3) / 4) | 1;
            int sg_c = (int)std::min<size_t>((size_t)(140 * 1024) / ((size_t)5 * qp_c * T * 16), (size_t)8 * spw_c);
            sg_c = std::max(sg_c / spw_c * spw_c, spw_c);
            const int ng_c = (nslots + sg_c - 1) / sg_c;
            if (ng_c < gNG || (ng_c == gNG && C * T < gC * gT)) { gC = C; gT = T; gNG = ng_c; }
        }
        if (!gC) throw PlanError{"monomers longer than 1536 bp are not supported by this build"};
        const int spw = 32 / gT, qpc = ((gC + 3) / 4) | 1;
        const size_t per_slot = (size_t)5 * qpc * gT * 16;
        // The per-column exchange costs ~1-2 us whatever the CTA computes and grows with the number of partner CTAs, so
        // groups are large (8 warps per segment) and a CTA sweeps its group for two segments at once (they share the
        // profile slice).  Measured on 1000 monomers: 8 warps x 2 segments 1.11 TCUPS, 12 x 1 1.07, 5 x 3 0.70.
        int sg = (int)std::min<size_t>((size_t)(140 * 1024) / per_slot, (size_t)8 * spw);
        sg = std::max(sg / spw * spw, spw);
        if (force_sg > 0) sg = std::max(force_sg / spw * spw, spw);
        sg = std::min(sg, (nslots + spw - 1) / spw * spw);
        const int ng = (nslots + sg - 1) / sg;
        if (ng > 1) {
            bestC = gC; bestT = gT; bestNT = (sg + spw - 1) / spw * 32;
            bestNS = std::max(1, std::min({2, 65536 / (bestNT * 112), 256 / ng}));   // registers; <= 256 exchange slots
            if (fNS) bestNS = std::min(fNS, 1024 / bestNT);
            bestNS = (int)std::max<int64_t>(1, std::min<int64_t>(bestNS, nseg_hint));
            g.NG = ng;
            g.SG = sg;
        } else if (!bestC) {
            // one group covers the set: only the segment length kept the symbols out of shared memory
            classic_search(true);
            if (!bestC) throw PlanError{"internal: no launch geometry for this monomer set"};
            stream = 1;
        }                                    // a forced group size that covers every slot is the ordinary single-CTA sweep
    }
    g.packed = packed; g.C = bestC; g.T = bestT; g.nslots = nslots; g.M = ms.M; g.NS = bestNS; g.NT = bestNT;
    if (g.NG == 1) g.SG = nslots;
    g.lat = 0;
    g.stream = g.NG > 1 ? 0 : stream;         // the group sweep always reads its symbols from global memory
    // Deferred-jump sweep (sweep_core.cuh: lat_*): a segment is spread over many warps -- a cluster of CTAs that exchange
    // the column key through distributed shared memory -- and runs at the latency of one column instead of at the
    // throughput of a loaded SM.  It pays when there are too few segments to fill the GPU with classic CTAs (config 1,
    // or one array shared by several GPUs); it costs 5.5 instead of 4.5 ALU instructions per register.
    {
        int lat_mode = -1, lat_warps = 0;
        if (const char *e = getenv("SD_LAT")) lat_mode = atoi(e);
        if (const char *e = getenv("SD_LAT_WARPS")) lat_warps = atoi(e);
        const int64_t nseg = std::max<int64_t>(nseg_hint, 1);
        double lbest = 1e300; int lC = 0, lT = 0, lNT = 0, lNG = 0, lSG = 0, lW = 0;
        auto lat_search = [&](bool streamed) {
            if (lat_mode == 0 || force_sg > 0) return;
            for (auto &cand : kLatGeom) {
                const int C = cand[0], T = cand[1];
                if (fC && (C != fC || T != fT)) continue;
                if (C * T < ms.Lmax) continue;
                if (!fC && C * T >= 2 * std::max(ms.Lmax, 96) && C * T > 192) continue;       // far too much padding
                const int spw = 32 / T, ws = (nslots + spw - 1) / spw;                        // warps per segment
                if (ws > 32) continue;                                                          // one exchange word per warp, polled by one lane each
                const int W = scan_window(ms, sc, packed, C, T);
                // warps per CTA: one per scheduler unless that needs more than 8 CTAs per cluster
                int wc = lat_warps > 0 ? lat_warps : std::min(ws, 4);
                while ((ws + wc - 1) / wc > 8 && wc < 32) ++wc;
                if (wc > 32 || (ws + wc - 1) / wc > 8) continue;
                wc = (ws + (ws + wc - 1) / wc - 1) / ((ws + wc - 1) / wc);                    // even out the CTAs of a cluster
                const int ng = (ws + wc - 1) / wc, sg = wc * spw;
                const int qp2c = ((2 * C + 3) / 4) | 1;
                const size_t smem = (size_t)5 * sg * T * qp2c * 16 + (streamed ? 0 : (size_t)max_seg_len) + 4096;
                if (smem > kSmemLimit) continue;
                // Measured on the B200 (tools/lat_probe.py, profiles/r02_lat_timing.txt, 12 DXZ1 monomers).  With one CTA
                // per SM a column takes 415 cycles at (6,32), 510 at (12,16), 605 at (24,8); every further CTA that has
                // to share the SM stretches it by 0.3 (C/6)^0.6 -- 520 / 690 / 855 cycles for 2 / 3 / 4 CTAs at (6,32),
                // 705 for 2 at (12,16), 1080 for 2 at (24,8): the warps then compete for issue slots.
                static const double kBaseC[] = {6, 12, 24, 48}, kBaseCycles[] = {415, 510, 605, 900};
                double base = kBaseCycles[3];
                for (int q = 0; q < 3; ++q)
                    if (C <= kBaseC[q + 1]) { base = kBaseCycles[q] + (kBaseCycles[q + 1] - kBaseCycles[q]) * std::max(0.0, C - kBaseC[q]) / (kBaseC[q + 1] - kBaseC[q]); break; }
                const int ctas_sm = (int)((nseg * ng + 147) / 148);
                const double cost = (double)std::max(max_seg_len, 1) * base * (1.0 + 0.3 * std::pow(C / 6.0, 0.6) * (ctas_sm - 1));
                if (cost < lbest) { lbest = cost; lC = C; lT = T; lNT = wc * 32; lNG = ng; lSG = sg; lW = W; }
            }
        };
        // streamed candidates only where the classic sweep streams too, or where SD_LAT=1 finds no staged one
        lat_search(stream);
        int lstream = stream;
        if (!lC && !stream && lat_mode > 0) { lat_search(true); lstream = 1; }
        const bool want = lat_mode > 0 || (lat_mode < 0 && lC && g.NG == 1 && nseg <= 2 * 148 && lbest < 0.97 * best);
        if (want && lC) {
            g.lat = 1; g.C = lC; g.T = lT; g.NS = 1; g.NT = lNT; g.NG = lNG; g.SG = lNG > 1 ? lSG : nslots; g.scanw = lW;
            g.stream = lstream;
        } else if (lat_mode > 0) {
            throw PlanError{"SD_LAT=1: no deferred-jump geometry fits this monomer set"};
        }
    }
    {
        // the lanes of a CTA must cover its slots: NS*nslots slot instances (single CTA) or SG (group sweep)
        const int spw = 32 / g.T;
        const int need = g.NG > 1 ? (g.SG + spw - 1) / spw * 32 : (g.NS * nslots + spw - 1) / spw * 32;
        if (g.NT < need || g.NT * (g.NG > 1 ? g.NS : 1) > 1024 || g.C * g.T < ms.Lmax)
            throw PlanError{"internal: inconsistent launch geometry"};
    }
    const int cpw = packed ? 8 : 16;
    g.CW = (g.C + cpw - 1) / cpw;
    p.nsl = nslots * g.T;
    if (!g.lat) g.scanw = scan_window(ms, sc, packed, g.C, g.T);
    {
        const int64_t D = -(int64_t)sc.del, I = -(int64_t)sc.ins;
        const int64_t dmax = std::llabs(D) * (std::max(ms.Lmax, 2) + 1) + std::llabs(I) + std::max(std::abs(sc.match), std::abs(sc.mismatch)) + 1;
        p.lat_th = (int)std::max<int64_t>(0, SD_REBASE_TH - 4 * dmax);
    }
    lat_jump_keys(ms, sc, nullptr, p.kj);

    // profile words: prof[sym][sl][q][e] = 4*s''(sym, row cell k) - 1 with k = t*C + 4q + e; pad cells get 4*pad_s - 1.
    const int C = g.C, T = g.T, SL = C * T;
    p.qp = ((C + 3) / 4) | 1;
    p.prof.assign((size_t)5 * p.nsl * p.qp * 4, 0u);
    p.slot_len.resize(nslots); p.slot_endadd.resize(nslots);
    const int shift = -sc.ins - sc.del;
    for (int slot = 0; slot < nslots; ++slot) {
        const int L = ms.rowlen(slot);              // packed: forward row `slot`, its RC row M+slot has the same length
        p.slot_len[slot] = L;
        p.slot_endadd[slot] = (L - 1) * sc.del;
        const int lead = (L == 1) ? SL - 1 : 0;     // length-1 rows sit in the last cell of their slot
        for (int sym = 0; sym < 5; ++sym)
            for (int pos = 0; pos < SL; ++pos) {
                int k = pos - lead;
                int lo = pad_s, hi = pad_s;
                if (k >= 0 && k < L) {
                    lo = (ms.rows[ms.row_off[slot] + k] == sym ? sc.match : sc.mismatch) + shift;
                    if (packed) hi = (ms.rows[ms.row_off[ms.M + slot] + k] == sym ? sc.match : sc.mismatch) + shift;
                }
                uint32_t w = packed ? (((uint32_t)(4 * lo - 1) & 0xffffu) | ((uint32_t)(4 * hi - 1) << 16)) : (uint32_t)(4 * lo - 1);
                int t = pos / C, kk = pos % C, q = kk / 4, e = kk % 4;
                int sl = slot * T + t;
                p.prof[(((size_t)sym * p.nsl + sl) * p.qp + q) * 4 + e] = w;
            }
    }
    if (g.lat) {
        // rows of the deferred form: [p | PT], PT[pos] = max(p[pos], max_{pos' < pos} p[pos'] + 3) per half (sweep_core.cuh)
        p.qp2 = ((2 * C + 3) / 4) | 1;
        p.prof2.assign((size_t)5 * p.nsl * p.qp2 * 4, 0u);
        auto word = [&](int sym, int slot, int pos) { return p.prof[(((size_t)sym * p.nsl + slot * T + pos / C) * p.qp + (pos % C) / 4) * 4 + (pos % C) % 4]; };
        for (int sym = 0; sym < 5; ++sym)
            for (int slot = 0; slot < nslots; ++slot) {
                int run_lo = INT_MIN, run_hi = INT_MIN;         // max over earlier positions of p + 3
                for (int pos = 0; pos < SL; ++pos) {
                    const uint32_t w = word(sym, slot, pos);
                    const int lo = packed ? (int)(int16_t)(w & 0xffffu) : (int)w, hi = packed ? (int)(int16_t)(w >> 16) : 0;
                    const int plo = std::max(lo, run_lo), phi = std::max(hi, run_hi);
                    run_lo = std::max(run_lo, lo + 3); run_hi = std::max(run_hi, hi + 3);
                    const uint32_t pt = packed ? (((uint32_t)plo & 0xffffu) | ((uint32_t)phi << 16)) : (uint32_t)plo;
                    uint32_t *row = p.prof2.data() + (((size_t)sym * p.nsl + slot * T + pos / C) * p.qp2) * 4;
                    row[pos % C] = w;
                    row[C + pos % C] = pt;
                }
            }
    }
    return p;
}

void build_filter_tables(const int *dist, int R, int ed_thr, int *rank_of_row, int *row_of_rank)
{
    std::vector<std::pair<int, int>> v((size_t)R);
    for (int r = 0; r < R; ++r) v[(size_t)r] = {dist[r], r};
    std::sort(v.begin(), v.end());
    int nf = 0;
    for (int r = 0; r < R; ++r) { rank_of_row[r] = -1; row_of_rank[r] = -1; }
    for (int x = 0; x < R; ++x)
        if (x == 0 || v[(size_t)x].first <= ed_thr) { rank_of_row[v[(size_t)x].second] = nf; row_of_rank[nf] = v[(size_t)x].second; ++nf; }
}

CtaLayout make_cta_layout(const Plan &p, const Batch &b, int seg_begin, int seg_end)
{
    CtaLayout l;
    const Geometry &g = p.g;
    const int nseg = seg_end - seg_begin;
    // logical CTAs: NG == 1: one per NS segments; NG > 1: CTA seg*NG + grp sweeps slot group grp of segment seg
    const int nctas = g.NG > 1 ? nseg * g.NG : (nseg + g.NS - 1) / g.NS;
    l.cta_nmax.assign(nctas, 0);
    l.cta_code_off.assign(nctas + 1, 0);
    l.seg_j_off.assign(nseg + 1, 0);
    l.seg_rec_off.assign(nseg + 1, 0);
    for (int s = 0; s < nseg; ++s) {
        int n = b.len(seg_begin + s);
        if (g.NG > 1) for (int q = 0; q < g.NG; ++q) l.cta_nmax[s * g.NG + q] = n;
        else l.cta_nmax[s / g.NS] = std::max(l.cta_nmax[s / g.NS], n);
        l.seg_j_off[s + 1] = l.seg_j_off[s] + n + 1;
        l.seg_rec_off[s + 1] = l.seg_rec_off[s] + n;
    }
    for (int c = 0; c < nctas; ++c)
        l.cta_code_off[c + 1] = l.cta_code_off[c] + (int64_t)l.cta_nmax[c] * g.NT * g.CW;
    return l;
}

} // namespace sdb
