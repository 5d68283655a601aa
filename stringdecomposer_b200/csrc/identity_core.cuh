// identity_core.cuh -- per-lane algebra of the identity rescoring kernel (SURVEY §8 f1), shared by the CUDA kernel
// (identity_kernels.cu) and the host emulator of the CPU test-suite (tests/emu/emu.cpp).
//
// Replaces edist/aai of the reference (stringdecomposer/main.py:29-60): edlib.align(interval, monomer, mode="NW",
// task="path"), identity = '=' columns / alignment columns.  edlib walks its unit-cost matrix back from the
// bottom-right cell taking, at every cell, the first move that explains the value: up (query character alone),
// then left (target character alone), then the diagonal (vendored edlib.cpp:1036-1133).  The number of '='
// columns on that walk obeys a forward recurrence over the same matrix,
//     pred(i,j) = up if D[i-1][j]+1 == D[i][j], else left if D[i][j-1]+1 == D[i][j], else diagonal
//     M[i][j]   = M[pred(i,j)] + (diagonal taken and q[i] == t[j]),      columns = M + D at the last cell,
// so no traceback state is stored at all.  One 32-bit word per cell carries both: D in bits 18..31, M in bits
// 0..15; bits 16..17 hold the move priority inside the three candidates only, so ONE unsigned minimum picks the
// smallest distance and, among equal distances, edlib's preferred move, and drags that move's M along.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#if defined(__CUDACC__)
#define SDI_HD __host__ __device__ __forceinline__
#else
#define SDI_HD inline
#endif

namespace sdb {

constexpr int SD_NW_MAXLEN = 16382;                 // every candidate D + 1 <= max(len) + 1 must fit 14 bits; M < 2^16
constexpr uint32_t NW_DSHIFT = 18;
constexpr uint32_t NW_K_UP = 1u << 18;                              // +1, priority 0
constexpr uint32_t NW_K_LEFT = (1u << 18) | (1u << 16);             // +1, priority 1
constexpr uint32_t NW_K_DIAG_EQ = (2u << 16) + 1u;                  // +0, priority 2, one more '=' column
constexpr uint32_t NW_K_DIAG_NE = (1u << 18) | (2u << 16);          // +1, priority 2
constexpr uint32_t NW_CLEAR = ~(3u << 16);
constexpr uint32_t NW_NOCHAR = 0xffffu;                             // query padding: equals no target byte

SDI_HD uint32_t nw_addmin(uint32_t a, uint32_t b, uint32_t c)       // min(a + b, c)     VIADDMNMX.U32
{
#if defined(__CUDA_ARCH__)
    return __viaddmin_u32(a, b, c);
#else
    const uint32_t s = a + b;
    return s < c ? s : c;
#endif
}

// The R consecutive query rows one lane owns, at the column it finished last.
template <int R>
struct NwLane {
    uint32_t left[R];      // cells of the previous column
    uint32_t qc[R];        // query characters (NW_NOCHAR beyond the end)
    uint32_t up_prev;      // cell above the first row, previous column
};

template <int R>
SDI_HD void nw_lane_init(NwLane<R> &st, const char *q, int qlen, int row0)
{
#pragma unroll
    for (int r = 0; r < R; ++r) {
        st.qc[r] = row0 + r < qlen ? (uint32_t)(uint8_t)q[row0 + r] : NW_NOCHAR;
        st.left[r] = (uint32_t)(row0 + r + 1) << NW_DSHIFT;         // D[i][-1] = i + 1
    }
    st.up_prev = (uint32_t)row0 << NW_DSHIFT;                       // D[row0-1][-1] = row0
}

// One column for this lane: `top` is the cell above the first row in this column, tc the target character.
template <int R>
SDI_HD uint32_t nw_lane_step(NwLane<R> &st, uint32_t top, uint32_t tc)
{
    // diagonal candidates first: they only read the previous column, so they are independent of the chain below
    uint32_t cd[R];
#pragma unroll
    for (int r = 0; r < R; ++r)
        cd[r] = (r ? st.left[r - 1] : st.up_prev) + (st.qc[r] == tc ? NW_K_DIAG_EQ : NW_K_DIAG_NE);
    uint32_t up = top;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t v = nw_addmin(up, NW_K_UP, nw_addmin(st.left[r], NW_K_LEFT, cd[r])) & NW_CLEAR;
        st.left[r] = v;
        up = v;
    }
    st.up_prev = top;
    return up;              // bottom cell of the strip
}

// A pair is swept by a group of NW_LANES lanes (four pairs per warp), each lane owning R consecutive query rows:
// long strips amortise the per-step bookkeeping and the SHFL over many cells and keep the wavefront fill small
// (171 columns + 7 fill steps), while the 2-deep dependent chain per cell leaves enough independent work per warp.
constexpr int NW_LANES = 8;
// Rows per lane for a batch: the strip length (8, 16 or 24) that minimises tiles x instructions per step summed
// over the batch's queries (a query longer than NW_LANES * R rows is swept in several tiles).
inline int nw_choose_rows(const int64_t *qoff, int64_t nq)
{
    int best_r = 24;
    double best = 1e300;
    for (int cand : {8, 16, 24}) {
        double cost = 0;
        for (int64_t i = 0; i < nq; ++i) {
            const int64_t ql = qoff[i + 1] - qoff[i];
            cost += (double)((ql + NW_LANES * cand - 1) / (NW_LANES * cand)) * (7.0 * cand + 25.0);
        }
        if (cost < best) { best = cost; best_r = cand; }
    }
    return best_r;
}

// The geometries compiled into the library, as (lanes per pair L, rows per lane R).
constexpr int NW_GEOMS[5][2] = {{8, 8}, {8, 16}, {8, 24}, {16, 12}, {32, 6}};

// (L, R) of a batch, for the launcher and the emulator alike: NW_LANES lanes with the strip nw_choose_rows picks,
// unless SD_NW_GEOM=L,R asks for another geometry (tests and experiments).  Returns false, with L and R as asked,
// when that geometry is not compiled.
inline bool nw_choose_geometry(const int64_t *qoff, int64_t nq, int &L, int &R)
{
    L = NW_LANES; R = nw_choose_rows(qoff, nq);
    if (const char *e = getenv("SD_NW_GEOM")) { int l = 0, r = 0; if (sscanf(e, "%d,%d", &l, &r) == 2) { L = l; R = r; } }
    for (const auto &g : NW_GEOMS) if (g[0] == L && g[1] == R) return true;
    return false;
}

// Above 1 MiB of traceback state edlib switches to Hirschberg splitting (edlib.cpp:1187-1191), whose path may differ.
SDI_HD bool nw_edlib_traceback_domain(int qlen, int tlen)
{
    const long long blocks = (qlen + 63) / 64;
    return 20ll * blocks * tlen + 8ll * tlen < 1024ll * 1024ll;
}

struct IdentityArgs {
    const char *qtext; const int64_t *qoff; int64_t nq;
    const char *ttext; const int64_t *toff; int64_t nt;
    const int32_t *pair_q, *pair_t; int64_t npairs;        // pair_q == nullptr: all queries x all targets, query-major
    int32_t *matches, *columns, *distance;                 // distance may be nullptr
    uint32_t *scratch; int64_t scratch_stride;             // one row of max target length per lane group (tiled queries)
};

} // namespace sdb
