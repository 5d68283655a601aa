// tests/emu/plan_probe.cpp -- CPU TEST-SUITE ONLY.  Compiled together with a checkout's csrc/plan.cpp into a small
// shared library by tests/golden/make_golden_plans.py (for the planner table) and by tests/test_long_segments.py.
//
// The launch geometry make_plan picks for a monomer set, a longest segment and a segment count on one device -- the
// geometry fields sd_get_stats reports after a call of that shape -- without materialising the segments (40,000
// segments of 100 kb would not fit a test machine).  It builds against planners that predate Geometry::stream too
// (stream then reads 0), so that the table can be written from an older commit.
#include <cstring>
#include <string>
#include <vector>

#include "common.h"

namespace {
template <class G> auto stream_of(const G &g, int) -> decltype(g.stream) { return g.stream; }
template <class G> int stream_of(const G &, long) { return 0; }
}

// out[10]: packed C T NS NT NG lat scanw SG stream.  Returns 0, or 3 with the planner's message in msg (capacity msg_cap).
extern "C" int sd_plan_probe(const char *monomers, const int64_t *offsets, int32_t n_monomers, int32_t ins, int32_t del,
                             int32_t mismatch, int32_t match, int32_t max_seg_len, int64_t nseg, int32_t *out, char *msg,
                             int32_t msg_cap)
{
    using namespace sdb;
    try {
        std::vector<std::string> mons;
        for (int32_t j = 0; j < n_monomers; ++j) mons.emplace_back(monomers + offsets[j], monomers + offsets[j + 1]);
        MonomerSet ms;
        build_monomer_set(mons, ms);
        Scoring sc; sc.ins = ins; sc.del = del; sc.mismatch = mismatch; sc.match = match;
        const Plan p = make_plan(ms, sc, max_seg_len, nseg);
        const Geometry &g = p.g;
        const int32_t v[10] = {g.packed, g.C, g.T, g.NS, g.NT, g.NG, g.lat, g.scanw, g.SG, (int32_t)stream_of(g, 0)};
        for (int x = 0; x < 10; ++x) out[x] = v[x];
        return 0;
    } catch (PlanError &e) {
        if (msg && msg_cap > 0) { strncpy(msg, e.msg.c_str(), (size_t)msg_cap - 1); msg[msg_cap - 1] = 0; }
        return 3;
    }
}
