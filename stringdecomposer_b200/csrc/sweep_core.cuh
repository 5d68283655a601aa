// sweep_core.cuh -- per-lane arithmetic of the column sweep and the traceback walk.
//
// Shared verbatim by the sm_100a kernels (sweep_kernels.cu) and by the host emulator used in the
// CPU test-suite (emu.cpp, tests only), so the algebra can be checked without a GPU.
//
// The recurrence restated (reference: stringdecomposer/src/main.cpp:171-208, SURVEY App. A):
//   H[i][k] = max( H[i][k-1]+del, H[i-1][k]+ins, H[i-1][k-1]+s, J[i]+k*del+s )      k>=1, i>=1
// Shift every cell by its position, Hh[i][k] = H[i][k] - i*ins - k*del, and the moves become
//   left: Hh[i][k-1]          up: Hh[i-1][k]          diag: Hh[i-1][k-1] + s''
//   jump: B[i] + s''          with s'' = s - ins - del and B[i] = J[i] - (i-1)*ins + del,
// i.e. the deletion chain is a pure prefix-max and the insertion move is free.  Values are multiplied by 4 and
// carry a 2-bit priority tag in the low bits (left/del=3 > up/ins=2 > diag=1 > jump=0), so that a plain
// integer max reproduces the reference's traceback priority del > ins > diag > jump
// (main.cpp:242-253) and the backpointer is (3 - tag) = reference code {0:del,1:ins,2:diag,3:jump}.
// State registers hold U = 4*rel + 2 ("tag-2 form": already the insertion candidate of the next column);
// rel is relative to a per-segment reference base Bref that is moved ("rebase") only when the jump operand
// 4*(B[i]-Bref) leaves +-SD_REBASE_TH, so no per-column renormalisation work is needed.
// Per register (two DP cells when packed) and column the sweep issues, on the integer ALU pipe:
//   VIADDMNMX  m = max(U[k-1] + p[k], U[k])      diag vs up; independent of J[i]  (lane_pre / lane_pass2_pre)
//   VIADDMNMX  m = max(p[k] + j, m)              jump candidate                    (lane_post)
//   1/2 VIMNMX3                                  lane maximum for the cross-lane scan
//   VIADDMNMX  h = max(Uleft + 1, m)             deletion chain, left wins ties    (lane_pass2_pre)
//   LOP3       U = (h | 3) ^ 1                   re-tag
// and on the FMA pipe IMAD + IMAD.IADD for the backpointer digits w = w*4 + U - h.
#pragma once
#include <climits>
#include <stdint.h>

#if defined(__CUDACC__)
#define SD_HD __host__ __device__ __forceinline__
#else
#define SD_HD inline
#endif

namespace sdb {

// --------------------------------------------------------------------------------------------
// Host-side emulation of the DPX instructions, with an optional overflow trap for the tests.
// --------------------------------------------------------------------------------------------
#ifndef __CUDA_ARCH__
struct EmuFlags { static inline bool &overflow() { static thread_local bool f = false; return f; } };
static inline int16_t emu_s16(int v) { if (v < -32768 || v > 32767) EmuFlags::overflow() = true; return (int16_t)v; }
static inline uint32_t emu_pack(int lo, int hi) { return (uint32_t)(uint16_t)emu_s16(lo) | ((uint32_t)(uint16_t)emu_s16(hi) << 16); }
static inline int emu_lo(uint32_t a) { return (int16_t)(a & 0xffffu); }
static inline int emu_hi(uint32_t a) { return (int16_t)(a >> 16); }
static inline int emu_max(int a, int b) { return a > b ? a : b; }
#endif

// Two DP rows per 32-bit register (lo half = forward monomer, hi half = its reverse complement).
struct Packed16 {
    static constexpr int ROWS = 2;             // DP rows per slot
    static constexpr int CELLS_PER_WORD = 8;   // backpointer cells per 32-bit word (per half: 8 x 2 bit)
    static constexpr uint32_t TAGMASK = 0x00030003u;
    static constexpr uint32_t ONE = 0x00010001u;
    static SD_HD uint32_t splat(int v)
    {
#ifdef __CUDA_ARCH__
        return __byte_perm((uint32_t)v, 0u, 0x1010);   // one PRMT
#else
        return ((uint32_t)v & 0xffffu) | ((uint32_t)v << 16);
#endif
    }
    static SD_HD int lo(uint32_t a) { return (int)(int16_t)(a & 0xffffu); }
    static SD_HD int hi(uint32_t a) { return (int)(int16_t)(a >> 16); }
    static SD_HD uint32_t addmax(uint32_t a, uint32_t b, uint32_t c) {   // per half: max(a+b, c)   VIADDMNMX.S16x2
#ifdef __CUDA_ARCH__
        return __viaddmax_s16x2(a, b, c);
#else
        return emu_pack(emu_max(emu_lo(a) + emu_lo(b), emu_lo(c)), emu_max(emu_hi(a) + emu_hi(b), emu_hi(c)));
#endif
    }
    static SD_HD uint32_t max2(uint32_t a, uint32_t b) {                 // VIMNMX.S16x2
#ifdef __CUDA_ARCH__
        return __vmaxs2(a, b);
#else
        return emu_pack(emu_max(emu_lo(a), emu_lo(b)), emu_max(emu_hi(a), emu_hi(b)));
#endif
    }
    static SD_HD uint32_t max3(uint32_t a, uint32_t b, uint32_t c) {     // VIMNMX3.S16x2
#ifdef __CUDA_ARCH__
        return __vimax3_s16x2(a, b, c);
#else
        return max2(max2(a, b), c);
#endif
    }
    static SD_HD uint32_t add(uint32_t a, uint32_t b) {                  // per half add
#ifdef __CUDA_ARCH__
        return __vadd2(a, b);
#else
        return emu_pack(emu_lo(a) + emu_lo(b), emu_hi(a) + emu_hi(b));
#endif
    }
};

// One DP row per 32-bit register; used when the score range does not provably fit 14+2 bits.
struct Scalar32 {
    static constexpr int ROWS = 1;
    static constexpr int CELLS_PER_WORD = 16;
    static constexpr uint32_t TAGMASK = 3u;
    static constexpr uint32_t ONE = 1u;
    static SD_HD uint32_t splat(int v) { return (uint32_t)v; }
    static SD_HD int lo(uint32_t a) { return (int)a; }
    static SD_HD int hi(uint32_t a) { return (int)a; }
    static SD_HD uint32_t addmax(uint32_t a, uint32_t b, uint32_t c) {   // VIADDMNMX
#ifdef __CUDA_ARCH__
        return (uint32_t)__viaddmax_s32((int)a, (int)b, (int)c);
#else
        int s = (int)a + (int)b; return (uint32_t)(s > (int)c ? s : (int)c);
#endif
    }
    static SD_HD uint32_t max2(uint32_t a, uint32_t b) { return (uint32_t)((int)a > (int)b ? (int)a : (int)b); }
    static SD_HD uint32_t max3(uint32_t a, uint32_t b, uint32_t c) {
#ifdef __CUDA_ARCH__
        return (uint32_t)__vimax3_s32((int)a, (int)b, (int)c);
#else
        return max2(max2(a, b), c);
#endif
    }
    static SD_HD uint32_t add(uint32_t a, uint32_t b) { return a + b; }
};

// TAGMASK and ONE as run-time register values: ptxas then folds (h | TAGMASK) ^ ONE into one three-register LOP3
// instead of two LOP3 with an immediate each.
struct TagRegs { uint32_t mask3, one; };
template <class P> SD_HD TagRegs tag_regs() { TagRegs r; r.mask3 = P::TAGMASK; r.one = P::ONE; return r; }

constexpr int SD_REBASE_TH = 4096;      // |4*(B[i]-Bref)| above this triggers a rebase of the lane registers

// Pass 1a ("pre", independent of J[i]): X[kk] <- max(diag, up) for the lane's C cells.
//   X[kk] in : U (tag-2 form) of the previous column        X[kk] out: max(U[k-1] + p[k], U[k])   (tags 1 / 2)
//   prevU    : previous-column U of the cell left of X[0] (the left lane's X[C-1]; dead for lane 0 of a slot)
//   pw       : profile words p = 4*s'' - 1 (packed per half) for this column's read symbol; pad cells very negative
//   kill_first / kill_last: the cell is a k==0 cell -- no insertion candidate (main.cpp:194)
template <class P, int C>
SD_HD void lane_pre(uint32_t (&X)[C], uint32_t prevU, const uint32_t *pw, uint32_t deadu, bool kill_first, bool kill_last)
{
    uint32_t prev = prevU;
#pragma unroll
    for (int kk = 0; kk < C; ++kk) {
        uint32_t up = X[kk];
        const uint32_t keep = up;
        if (kk == 0 && kill_first) up = deadu;
        if (kk == C - 1 && kill_last) up = deadu;
        X[kk] = P::addmax(prev, pw[kk], up);
        prev = keep;
    }
}

// Pass 1a of column 0, where every cell of the previous column is dead and the base is B[0] = ins (row-0 rule,
// main.cpp:180).  A row's k==0 cell is s(0,0) itself (main.cpp:173-177), one `del` more than the generic jump
// candidate, so the profile word of the slot's first cell (the last cell of a length-1 row) gets 4*del added first.
// del is taken by reference so that a kernel reads its parameter where it uses it: passed by value, the load moves
// ahead of the two branches and the kernels' machine code changes.
template <class P, int C>
SD_HD void lane_pre_col0(uint32_t (&X)[C], uint32_t *pw, const int &del, int L, uint32_t deadu, bool kill_first, bool kill_last)
{
    if (kill_first && L > 1) pw[0] = P::add(pw[0], P::splat(4 * del));
    if (kill_last) pw[C - 1] = P::add(pw[C - 1], P::splat(4 * del));
    lane_pre<P, C>(X, deadu, pw, deadu, kill_first, kill_last);
}

// Pass 1b ("post"): add the jump candidate 4*(B[i]-Bref) + 4*s'' (tag 0) once J[i] is known.
// jump0p1 = splat(4*(B[i]-Bref) + 1) (the +1 undoes the -1 folded into the profile words).
// Returns the lane maximum in tag-2 form: what the lane hands to the lanes on its right (deletion chain).
// Maximum of n registers as a ternary tree (depth ~log3 n instead of a serial chain of VIMNMX3).
template <class P, int N> SD_HD uint32_t tree_max(const uint32_t (&v)[N])
{
    uint32_t a[N];
#pragma unroll
    for (int j = 0; j < N; ++j) a[j] = v[j];
    int n = N;
#pragma unroll
    for (int level = 0; level < 6; ++level) {
        if (n <= 1) break;
        const int m = (n + 2) / 3;
#pragma unroll
        for (int j = 0; j < (N + 2) / 3; ++j) {
            if (j < m) {
                const int b = 3 * j;
                uint32_t r = a[b];
                if (b + 2 < n) r = P::max3(a[b], a[b + 1], a[b + 2]);
                else if (b + 1 < n) r = P::max2(a[b], a[b + 1]);
                a[j] = r;
            }
        }
        n = m;
    }
    return a[0];
}

template <class P, int C>
SD_HD uint32_t lane_post(uint32_t (&X)[C], const uint32_t *pw, uint32_t jump0p1, uint32_t deadu, TagRegs tr)
{
    (void)deadu;
#pragma unroll
    for (int kk = 0; kk < C; ++kk) X[kk] = P::addmax(pw[kk], jump0p1, X[kk]);
    const uint32_t E = tree_max<P, C>(X);
    return (E | tr.mask3) ^ tr.one;
}

// Backpointer words hold the digits (U - h) in {-1..2} accumulated as w = w*4 + digit (mod 2^32); adding this
// constant turns an n-cell word into the 2-bit codes (U + 1 - h).  The sweep stores the raw word; the decoder adds
// the bias (one add per decoded cell in the traceback instead of one per word in the sweep).
SD_HD uint32_t code_bias(int packed, int ncell)
{
    const uint32_t v = 0x55555555u >> (32 - 2 * ncell);       // (4^ncell - 1) / 3, ncell in 1..16
    return v * (packed ? 0x00010001u : 1u);
}
// code of cell c (0-based) of an ncell-cell word; half = 16 for the reverse-complement row of a packed word
SD_HD int decode_code(uint32_t w, int packed, int ncell, int c, int half)
{
    return (int)(((w + code_bias(packed, ncell)) >> (2 * (ncell - 1 - c) + half)) & 3u);
}

// Pass 2 fused with pass 1a of the NEXT column.  The deletion chain (prefix max) runs through the lane with the carry
// from the lanes on its left:
//   h = max(Uleft + 1, m2)      tagged winner (left has tag 3 and wins ties: main.cpp:242 comes first)
//   U = (h | 3) ^ 1             new state, tag-2 form                 code = U + 1 - h  in {0,1,2,3}
// Backpointer word layout: word wi holds cells [wi*CPW, wi*CPW + ncell); cell c of the word sits at bits 2*(ncell-1-c)
// (Packed16: forward row in bits 0..15, reverse-complement row in bits 16..31); see decode_code().
// While the chain runs (two dependent ALU ops per cell), the J-independent candidates of column i+1 are formed from
// the fresh U values:
//   X[kk] <- max(U[kk-1] + pn[kk], U[kk])      kk >= 1        (pn: profile words of column i+1)
// Cell 0 needs the left lane's last U (a shuffle), so the caller finishes it with lane_pre_first().
// Returns U[C-1] (row-end value for the jump key and the right neighbour's diagonal); *u_first gets U[0].
template <class P, int C>
SD_HD uint32_t lane_pass2_pre(uint32_t (&X)[C], uint32_t carryU, uint32_t *codes, TagRegs tr, const uint32_t *pn,
                              uint32_t deadu, bool kill_last, uint32_t *u_first)
{
    constexpr int CPW = P::CELLS_PER_WORD;
    uint32_t ul = carryU, uprev = 0;
    uint32_t w = 0;
#pragma unroll
    for (int kk = 0; kk < C; ++kk) {
        const uint32_t h = P::addmax(ul, tr.one, X[kk]);
        ul = (h | tr.mask3) ^ tr.one;
        w = w * 4u + ul - h;
        if ((kk + 1) % CPW == 0 || kk == C - 1) { codes[kk / CPW] = w; w = 0; }     // unbiased digits; see decode_code()
        if (kk == 0) *u_first = ul;
        else X[kk] = P::addmax(uprev, pn[kk], (kk == C - 1 && kill_last) ? deadu : ul);
        uprev = ul;
    }
    return ul;
}

template <class P>
SD_HD uint32_t lane_pre_first(uint32_t prevU, uint32_t pn0, uint32_t u_first, uint32_t deadu, bool kill_first, bool kill_only)
{
    // kill_only: C == 1 and the single cell is also the slot's last cell of a length-1 row
    return P::addmax(prevU, pn0, (kill_first || kill_only) ? deadu : u_first);
}

// --------------------------------------------------------------------------------------------
// Deferred-jump ("latency") form of the same column, used when a segment is spread over many warps / CTAs and the
// per-column exchange of the jump value J[i] would otherwise sit on the critical path.
//
// In the shifted domain a jump can only win at a row's first cell and where the profile rises (everywhere else the
// left neighbour holds at least the same jump-derived value and wins the tie), so column i factors into
//   h[k] = max( h0[k] , JT[k] )     h0[k] = max( g[k], m[k] ),  g[k] = max_{k'<k} (m[k'] | 3)    -- independent of J[i]
//                                   JT[k] = PT[k] + 4*(B[i]-Bref) + 1,  PT[k] = max( p[k], max_{k'<k} p[k'] + 3 )
// with m[k] = max(U[k-1] + p[k], U[k]) as before and PT a second, static profile (the tagged prefix maximum of the
// jump candidates of the slot).  This is the same tagged maximum the classic form computes -- (x | 3) distributes over
// max -- so values, tie-breaks and backpointer codes are identical.  What changes is the dependency: the vector work
// of column i needs B[i-1] only through U[i-1]; B[i] enters in one VIADDMNMX per register at the very end.  The key of
// the J-independent row ends (K0[i]) is therefore published one whole column before anybody needs it:
//   B[i+1] <- max( K0[i] , B[i] + KJ[sym_i] )      KJ: static per symbol (best jump-derived row end)
// Per register: VIADDMNMX (m), LOP3 + VIMNMX/VIMNMX3 + VIMNMX (chain), VIADDMNMX (merge), LOP3 (re-tag) + 1/2 VIMNMX3
// (lane total) = 6.5 ALU-pipe instructions (classic: 4.5) -- the price of taking the exchange latency off the
// critical path; it pays only where the sweep is bound by latency, not by the ALU pipe.
//
// lat_total: the lane's contribution to the left candidates of the lanes on its right, tag 3.
template <class P, int C> SD_HD uint32_t lat_total(const uint32_t (&M)[C], TagRegs tr) { return tree_max<P, C>(M) | tr.mask3; }

// Deletion chain of the J-independent part, in place: X[kk] = m[kk] -> h0[kk] = max(g[kk], m[kk]) with
// g[kk] = max(carry, m[0..kk) | 3).  carry: maximum of lat_total over the lanes on the left (tag 3; dead for the first
// lane of a slot).  The sweep runs at the latency of a lone warp, so the chain is kept shallow: the left candidates
// m3 = m | 3 are formed up front (independent), the running maximum advances two cells per VIMNMX3, and h0 is taken off
// the chain -- 3 instructions per register at a third of the depth of the obvious two-instruction recurrence.
// Returns g after the last cell = (h0 of the lane's last cell) | 3.
template <class P, int C>
SD_HD uint32_t lat_chain(uint32_t (&X)[C], uint32_t carry, TagRegs tr)
{
    uint32_t m3[C], g[C + 1];
#pragma unroll
    for (int kk = 0; kk < C; ++kk) m3[kk] = X[kk] | tr.mask3;
    g[0] = carry;
#pragma unroll
    for (int kk = 0; kk < C; kk += 2) {
        g[kk + 1] = P::max2(g[kk], m3[kk]);
        if (kk + 1 < C) g[kk + 2] = P::max3(g[kk], m3[kk], m3[kk + 1]);
    }
#pragma unroll
    for (int kk = 0; kk < C; ++kk) X[kk] = P::max2(g[kk], X[kk]);
    return g[C];
}

// Merge with the jump-derived candidates and re-tag, in place: X[kk] = h0 -> U (tag-2 form); backpointer digits as in
// lane_pass2_pre.  pt: the PT words of the column, jump0p1 = splat(4*(B[i]-Bref) + 1).  Returns U[C-1].
template <class P, int C>
SD_HD uint32_t lat_merge(uint32_t (&X)[C], const uint32_t *pt, uint32_t jump0p1, uint32_t *codes, TagRegs tr)
{
    constexpr int CPW = P::CELLS_PER_WORD;
    uint32_t w = 0;
#pragma unroll
    for (int kk = 0; kk < C; ++kk) {
        const uint32_t h = P::addmax(pt[kk], jump0p1, X[kk]);
        X[kk] = (h | tr.mask3) ^ tr.one;
        w = w * 4u + X[kk] - h;
        if ((kk + 1) % CPW == 0 || kk == C - 1) { codes[kk / CPW] = w; w = 0; }
    }
    return X[C - 1];
}

// Rebase: shift every register of the lane by -shift4 (packed per half).
template <class P, int C>
SD_HD void lane_rebase(uint32_t (&X)[C], int shift4)
{
    const uint32_t d = P::splat(-shift4);
#pragma unroll
    for (int kk = 0; kk < C; ++kk) X[kk] = P::add(X[kk], d);
}

// Jump key of an end cell: (relative end score + (L-1)*del) * 4096 + (4095 - row): a plain integer max
// over the keys yields max score and, on ties, the lowest row (main.cpp:212 strict '<', :230-236 first match).
constexpr int SD_KEY_ROWS = 4096;
SD_HD int make_key(int z_end, int endadd, int row) { return ((z_end >> 2) + endadd) * SD_KEY_ROWS + (SD_KEY_ROWS - 1 - row); }
SD_HD int key_const(int endadd, int row) { return endadd * SD_KEY_ROWS + (SD_KEY_ROWS - 1 - row); }      // key = (u>>2)*4096 + const
SD_HD int key_value(int key) { return key >> 12; }
// In the deferred form the J-independent part of a row end can be "minus infinity" (a length-1 row has nothing but its
// jump candidate); with 32-bit lanes that value times 4096 would wrap, so it is clamped before the key is formed.
// Real row ends stay far above: a row end scores at least J[i] + (L-1)*del + min(mismatch, 0) and Bref follows J
// within SD_REBASE_TH/4, so rel = (row end - Bref) - (L-1)*del stays above about -2^10 + min(mismatch, 0), far from
// the floor's -2^18.  Only length-1 rows, whose endadd is 0, reach it.  The floor is a tag-3 word like the g it
// replaces, so that its key decodes to the lane's own row.
constexpr int SD_KEY_FLOOR = -(1 << 20) + 3;
SD_HD int key_floor(int z) { return z > SD_KEY_FLOOR ? z : SD_KEY_FLOOR; }
SD_HD int key_row(int key) { return SD_KEY_ROWS - 1 - (key & (SD_KEY_ROWS - 1)); }

// Column key of one lane, the operand of the sweep's per-column maximum (CREDUX / atomicMax).
//   u       the lane's last word: U (tag 2) in the classic sweeps and in column 0 of the deferred sweep, g (tag 3)
//           afterwards.  (u << 10) is rel*4096 + (tag << 10).
//   kc      key_const(endadd, tie-break row) - (tag << 10) of a lane that holds a counted row end; SD_KEY_NONE for any
//           other lane (not the last lane of its slot, or a row the --ed_thr filter dropped).  tag_off: a part of
//           (tag << 10) that kc does not include yet
//   counted whether the lane holds a counted row end (the forward row of the slot for Scalar32)
//   FLOOR   deferred sweep after column 0: clamp the J-independent value first (key_floor; Scalar32 only)
// Packed16: |rel| < 2^13 by the range proof (packed_range_ok), so a lane with kc = SD_KEY_NONE stays below every real
// key without a select.  Scalar32 has no such bound: in the shifted domain a row never decreases, so an interior cell
// carries about the row end's rel = (row end - Bref) - (L-1)*del, and (L-1)*|del| reaches 499,500 within the planner's
// INF check; such a lane gets INT_MIN through a select.  A counted row end's key is its true score relative to Bref
// (|.| < 2^19 for the same reason) times 4096 and fits 32 bits, while rel*4096 alone may not: the shift and the add
// are done modulo 2^32.
constexpr int SD_KEY_NONE = -(1 << 30);
template <class P, bool FLOOR = false>
SD_HD int lane_key(uint32_t u, int kc_lo, int kc_hi, bool counted, int tag_off = 0)
{
    if (P::ROWS == 2) {
        const int klo = ((int)(u << 16) >> 6) + kc_lo - tag_off;
        const int khi = ((int)(u & 0xffff0000u) >> 6) + kc_hi - tag_off;
        return klo > khi ? klo : khi;
    }
    (void)kc_hi;
    if (FLOOR) u = (uint32_t)key_floor((int)u);
    return counted ? (int)((u << 10) + (uint32_t)kc_lo - (uint32_t)tag_off) : INT_MIN;
}

// lane_key's constants for one lane of a slot.  is_end: the lane is the active last lane of its slot.  Ties between
// rows break on the row itself, or with the --ed_thr pre-filter on its position in the segment's filtered list
// (main.cpp:141-147): rank is the [segment][row] -> position table (-1 = filtered out) or null, read only for an active
// lane, at segment first + seg (a classic sweep CTA holds segments first, first+1, ...).  kc_off is added to the
// constant of every counted row (the part of -(tag << 10) the caller folds in).  The segment comes in two parts and M
// by reference for the reason given at lane_pre_col0: the kernels then form the rank address and read M inside the
// branches that use them.
struct SlotKey { int kc_lo, kc_hi; bool counted; };
template <class P>
SD_HD SlotKey slot_key(bool active, bool is_end, int endadd, int slot, const int &M, const int *rank, int first, int seg, int kc_off)
{
    int tb_lo = slot, tb_hi = M + slot;
    if (rank && active) {
        const int *rk = rank + (size_t)(first + seg) * (2 * M);
        tb_lo = rk[slot]; tb_hi = (P::ROWS == 2) ? rk[M + slot] : -1;
    }
    SlotKey k;
    k.counted = is_end && tb_lo >= 0;
    k.kc_lo = k.counted ? key_const(endadd, tb_lo) + kc_off : SD_KEY_NONE;
    k.kc_hi = (is_end && tb_hi >= 0) ? key_const(endadd, tb_hi) + kc_off : SD_KEY_NONE;
    return k;
}

// --------------------------------------------------------------------------------------------
// Geometry of one launch: how DP rows map onto lanes and where backpointers live.
// --------------------------------------------------------------------------------------------
struct Geometry {
    int packed;      // 1: Packed16 (slot = forward row + its reverse complement), 0: Scalar32 (slot = one row)
    int C, T;        // cells per lane, lanes per slot; slot length SL = C*T >= longest row
    int nslots;      // slots per segment
    int M;           // forward monomers (rows = 2M)
    int NS;          // segments per CTA
    int NT;          // threads per CTA
    int CW;          // backpointer words per lane per column
    int NG;          // CTAs (slot groups) that share one segment; 1 = the whole monomer set fits one CTA
    int SG;          // slots per group (== nslots when NG == 1)
    int lat;         // 1: deferred-jump sweep (sweep_lat_kernel; a segment = a cluster of NG CTAs, NS == 1), 0: classic
    int scanw;       // lanes a lane must look back for the deletion carry (windowed scan; see plan.cpp: scan_window)
    int stream;      // 1: the classic / deferred-jump sweep reads the segment symbols from global memory as it goes
                     // (shared memory independent of the segment length); 0: they are staged in shared memory first
};

struct Record { int32_t row, start, end, score; };
struct JR { int32_t j, row; };      // per column i: J[i] = max_r H[i-1][r][last] and the lowest row attaining it

// Lanes of a slot never straddle a warp: a warp holds 32/T whole slots (the remaining lanes idle when T does not
// divide 32), slot instance g of the CTA lives in warp g / spw at lane (g % spw)*T + t.
SD_HD int slots_per_warp(int T) { return 32 / T; }
SD_HD int lane_tid(int T, int ginst, int t) { const int spw = 32 / T; return (ginst / spw) * 32 + (ginst % spw) * T + t; }

// Where the backpointers of DP row `row` live: the slot, the group (CTA) that owns it when the monomer set is split
// over several CTAs, the slot instance inside that CTA, and the half of the packed word.
struct RowPlace { int grp, ginst, half; };
SD_HD RowPlace place_row(const Geometry &g, int seg_local, int row)
{
    RowPlace r;
    const int slot = g.packed ? (row < g.M ? row : row - g.M) : row;
    r.half = (g.packed && row >= g.M) ? 16 : 0;
    r.grp = slot / g.SG;
    r.ginst = (g.NG > 1) ? slot - r.grp * g.SG : seg_local * g.nslots + slot;
    return r;
}

// Decode the backpointer of cell k of a row placed at `pl`; codes_col points at the first word of column i of the
// CTA that owns the row.
SD_HD int fetch_code(const uint32_t *codes_col, const Geometry &g, RowPlace pl, int rowlen, int k)
{
    int pos = (rowlen == 1) ? (g.C * g.T - 1) : k;     // length-1 rows are right-aligned in their slot
    int t = pos / g.C, kk = pos - t * g.C;
    int cpw = g.packed ? 8 : 16;
    int wi = kk / cpw, c = kk - wi * cpw;
    int ncell = g.C - wi * cpw; if (ncell > cpw) ncell = cpw;
    int tid = lane_tid(g.T, pl.ginst, t);
    uint32_t w = codes_col[(size_t)tid * g.CW + wi];
    return decode_code(w, g.packed, ncell, c, pl.half);
}

// Infix ("HW") edit distance of a DP row against a segment: unit-cost edit distance between the row and the best
// substring of the segment.  This is what the reference's --ed_thr pre-filter asks edlib for
// (MonomerEditDistance, main.cpp:128-133: edlibAlign(monomer, segment, k=-1, EDLIB_MODE_HW, EDLIB_TASK_DISTANCE)); the
// distance is unique, so any exact algorithm agrees with edlib.  Myers/Hyyro bit-vector algorithm, 64 rows per word,
// rows of up to 64*SD_HW_BLOCKS symbols.
constexpr int SD_HW_BLOCKS = 24;
SD_HD int hw_distance(const uint8_t *pat, int m, const uint8_t *text, int n, int (*code_of)(unsigned) = nullptr)
{
    (void)code_of;
    const int B = (m + 63) / 64;
    unsigned long long peq[5][SD_HW_BLOCKS], pv[SD_HW_BLOCKS], mv[SD_HW_BLOCKS];
    for (int b = 0; b < B; ++b) { pv[b] = ~0ull; mv[b] = 0ull; for (int c = 0; c < 5; ++c) peq[c][b] = 0ull; }
    for (int i = 0; i < m; ++i) {
        const unsigned ch = pat[i];
        const int c = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : 4;
        peq[c][i >> 6] |= 1ull << (i & 63);
    }
    const unsigned long long last_bit = 1ull << ((m - 1) & 63);
    int score = m, best = m;
    for (int j = 0; j < n; ++j) {
        const unsigned ch = text[j];
        const int c = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : 4;
        int hin = 0;                                     // row 0 of the HW table is all zeros: no horizontal delta
        for (int b = 0; b < B; ++b) {
            unsigned long long eq = peq[c][b];
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
        score += hin;
        if (score < best) best = score;
    }
    return best;
}

// Traceback of one segment from the 2-bit backpointers (SURVEY App. A.3; reference main.cpp:217-267).
//   jr[i], i=1..n : J[i] = max_r H[i-1][r][last] (jr[n].j is the final score) and its lowest row.
//   k == 0 cells are decided here from J and the two symbols involved (main.cpp:245 tests the insertion
//   equality at k==0 although the forward pass never takes that move, main.cpp:194).
// Records come out last-to-first (the caller reverses, main.cpp:268).  Returns the count, -1 on overflow, or
// SD_TB_BAD_ROW when a jump names a row outside the nrows DP rows, or a filtered-out rank (a wrong column key;
// row_off is not read then).
constexpr int SD_TB_BAD_ROW = -2;
template <class CodeAt>
SD_HD int traceback_segment(int n, const JR *jr, const uint8_t *seg, const uint8_t *rows,
                            const int *row_off, int ins, int del, int mismatch, int match,
                            CodeAt code_at, Record *out, int cap, bool writer = true, const int *rank2row = nullptr,
                            int nrows = SD_KEY_ROWS)
{
    // rank2row: with the --ed_thr pre-filter the DP rows of a segment are a re-ordered subset (main.cpp:135-149) and
    // jr[].row holds the position in that list; rank2row maps it back to the row of the full set (-1 past its end)
    (void)del;
    auto row_of = [&](int kr) { return (unsigned)kr >= (unsigned)nrows ? -1 : rank2row ? rank2row[kr] : kr; };
    int cnt = 0;
    int i = n - 1;
    int r = row_of(jr[n].row);
    if (r < 0) return SD_TB_BAD_ROW;
    int last = row_off[r + 1] - row_off[r] - 1;
    int k = last;
    int end = i;
    int end_score = jr[n].j;
    for (;;) {
        int code;
        if (k == 0) {
            code = 3;
            if (i != 0) {
                int s_here = rows[row_off[r]] == seg[i] ? match : mismatch;
                int s_prev = rows[row_off[r]] == seg[i - 1] ? match : mismatch;
                int h_here = jr[i].j + s_here;                               // H[i][r][0], main.cpp:191-193
                int h_prev = (i == 1) ? s_prev : jr[i - 1].j + s_prev;       // H[i-1][r][0] (row 0: main.cpp:173-177)
                if (h_here == h_prev + ins) code = 1;
            }
        } else {
            code = code_at(i, r, last + 1, k);
        }
        if (code == 0) { --k; continue; }
        if (code == 1) { --i; continue; }
        if (code == 2) { --i; --k; continue; }
        if (cnt >= cap) return -1;
        Record rec;
        rec.row = r; rec.start = i; rec.end = end;
        if (i == 0) { rec.score = end_score; if (writer) out[cnt] = rec; ++cnt; break; }      // main.cpp:258-262
        rec.score = end_score - jr[i].j;                                      // main.cpp:253-257
        if (writer) out[cnt] = rec;
        ++cnt;
        end_score = jr[i].j;
        r = row_of(jr[i].row);
        if (r < 0) return SD_TB_BAD_ROW;
        --i;
        last = row_off[r + 1] - row_off[r] - 1;
        k = last; end = i;
    }
    return cnt;
}

} // namespace sdb
