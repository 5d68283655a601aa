// pipeline.cpp -- host driver around the device sweep: FASTA ingest, segmentation, per-device scheduling,
// overlap resolution and the raw TSV writer.  Reference behaviour restated from stringdecomposer/src/main.cpp
// (line numbers cited per function); the data structures and control flow are this project's own.
#include <algorithm>
#include <cerrno>
#include <cstring>
#include <fstream>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <exception>
#include <future>
#include <mutex>
#include <stdexcept>
#include <thread>
#include <sys/stat.h>
#include <unistd.h>

#include "pipeline.h"

namespace sdb {

// ---------------------------------------------------------------------------------------------
// FASTA: name = first whitespace-delimited token of the header (main.cpp:321-325); sequence lines are
// appended verbatim (main.cpp:327) -- the toupper in Seq's constructor only ever sees "" (main.cpp:29,325),
// so lower case and '\r' are illegal symbols; alphabet check and messages main.cpp:330-344.
// ---------------------------------------------------------------------------------------------
// Chunked reader: the file is read in 4 MiB pieces and handed on line by line, so that neither pass over a reads file
// needs more memory than one chunk (plus, in the second pass, the read being assembled).
//   on_header(first, last)   a '>' line: [first,last) is the text after '>'
//   on_line(first, last)     any other line (the reference appends it to the current record verbatim, main.cpp:327)
template <class OnHeader, class OnLine>
static bool scan_fasta(const std::string &path, OnHeader on_header, OnLine on_line)
{
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) return false;                                   // the reference reads nothing from a missing file (main.cpp:315-319)
    std::vector<char> buf((size_t)4 << 20);
    std::string carry;                                      // unfinished last line of the previous chunk
    auto emit = [&](const char *p, const char *le) { if (le > p && *p == '>') on_header(p + 1, le); else on_line(p, le); };
    size_t got;
    while ((got = fread(buf.data(), 1, buf.size(), f)) > 0) {
        const char *p = buf.data(), *end = p + got;
        while (p < end) {
            const char *nl = static_cast<const char *>(memchr(p, '\n', (size_t)(end - p)));
            if (!nl) { carry.append(p, end); break; }
            if (!carry.empty()) { carry.append(p, nl); emit(carry.data(), carry.data() + carry.size()); carry.clear(); }
            else emit(p, nl);
            p = nl + 1;
        }
    }
    if (!carry.empty()) emit(carry.data(), carry.data() + carry.size());      // last line without a newline, like getline
    fclose(f);
    return true;
}

static inline bool is_space(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n' || c == '\v' || c == '\f'; }
static std::string header_name(const char *a, const char *le)      // name = first token (main.cpp:321-325)
{
    while (a < le && is_space(*a)) ++a;
    const char *b = a;
    while (b < le && !is_space(*b)) ++b;
    return std::string(a, b);
}

// Alphabet check of one line in a single branch-free pass (a table look-up OR-ed over the line): bit 0 = an N was
// seen, bit 1 = a symbol outside ACGTN.  Only a line with bit 1 set is looked at again, for the position of the symbol.
struct SymbolClass {
    uint8_t t[256];
    SymbolClass() { for (int c = 0; c < 256; ++c) t[c] = base_code((char)c) < 0 ? 2 : (c == 'N' ? 1 : 0); }
};
static inline unsigned classify_line(const char *p, const char *le)
{
    static const SymbolClass sc;
    const uint8_t *t = sc.t;
    const unsigned char *a = reinterpret_cast<const unsigned char *>(p), *e = reinterpret_cast<const unsigned char *>(le);
    unsigned f0 = 0, f1 = 0, f2 = 0, f3 = 0;
    for (; a + 8 <= e; a += 8) {
        f0 |= t[a[0]] | t[a[4]]; f1 |= t[a[1]] | t[a[5]]; f2 |= t[a[2]] | t[a[6]]; f3 |= t[a[3]] | t[a[7]];
    }
    for (; a < e; ++a) f0 |= t[*a];
    return f0 | f1 | f2 | f3;
}

// First pass over a FASTA file: names, lengths, the alphabet check and the N warning of load_fasta (main.cpp:330-344)
// without keeping any sequence.  Returns 0, or 255 after writing the reference's error line to diag.
struct FastaIndex { std::vector<std::string> names; std::vector<int64_t> lens; };
static int index_fasta(const std::string &path, FastaIndex &out, std::string &diag)
{
    out.names.clear(); out.lens.clear();
    bool has_n = false;
    int bad_seq = -1; char bad_char = 0;
    scan_fasta(path,
        [&](const char *a, const char *le) { out.names.push_back(header_name(a, le)); out.lens.push_back(0); },
        [&](const char *p, const char *le) {
            if (out.lens.empty()) return;                   // text before the first header belongs to no record
            if (bad_seq < 0) {
                const unsigned f = classify_line(p, le);
                has_n |= (f & 1) != 0;
                if (f & 2)
                    for (const char *c = p; c < le; ++c)
                        if (base_code(*c) < 0) { bad_seq = (int)out.lens.size() - 1; bad_char = *c; break; }
            }
            out.lens.back() += le - p;
        });
    if (bad_seq >= 0) {
        // the reference reports the first offending sequence in file order, and in it the first offending symbol
        diag += "ERROR: Sequence " + out.names[(size_t)bad_seq] + " contains undefined symbol (not ACGT): " + std::string(1, bad_char) + "\n";
        return 255;
    }
    if (has_n) diag += "WARNING: sequences in " + path + " contain N symbol. It will be counted as a separate symbol in scoring!\n";
    return 0;
}

int load_fasta(const std::string &path, FastaSet &out, std::string &diag)
{
    out.names.clear(); out.seqs.clear();
    bool has_n = false;
    int bad_seq = -1; char bad_char = 0;
    scan_fasta(path,
        [&](const char *a, const char *le) { out.names.push_back(header_name(a, le)); out.seqs.emplace_back(); },
        [&](const char *p, const char *le) {
            if (out.seqs.empty()) return;
            if (bad_seq < 0) {
                const unsigned f = classify_line(p, le);
                has_n |= (f & 1) != 0;
                if (f & 2)
                    for (const char *c = p; c < le; ++c)
                        if (base_code(*c) < 0) { bad_seq = (int)out.seqs.size() - 1; bad_char = *c; break; }
            }
            out.seqs.back().append(p, le);                  // lines appended raw (main.cpp:327), checked at :330-341
        });
    if (bad_seq >= 0) {
        diag += "ERROR: Sequence " + out.names[(size_t)bad_seq] + " contains undefined symbol (not ACGT): " + std::string(1, bad_char) + "\n";
        return 255;
    }
    if (has_n) diag += "WARNING: sequences in " + path + " contain N symbol. It will be counted as a separate symbol in scoring!\n";
    return 0;
}

// main.cpp:73-79.  The test at :74 is evaluated in size_t (int operands converted), as written there.
int64_t segment_read(int64_t read_len, int part_size, int overlap, std::vector<std::pair<int, int>> *out)
{
    if (part_size <= 0) return -1;
    int64_t cnt = 0;
    const size_t len = (size_t)read_len;
    for (size_t i = 0; i < len; i += (size_t)part_size) {
        bool keep = ((size_t)(int)len - i >= (size_t)overlap) || (len < (size_t)overlap);
        if (!keep) continue;
        int rest = (int)(len - i), want = part_size + overlap;
        int take = std::min(want, rest);
        if (take < 0) take = rest;
        if (out) out->emplace_back((int)i, take);
        ++cnt;
    }
    return cnt;
}

// main.cpp:287-302
void postprocess(const std::vector<Record> &in, std::vector<Record> &out)
{
    out.clear();
    size_t i = 0; const size_t n = in.size();
    while (i < n) {
        for (size_t j = i + 1; j < std::min(i + 7, n); ++j) {
            if ((in[i].end - in[j].start) * 2 > (in[j].end - in[j].start)) {
                out.push_back(in[i]);
                i = j + 1;
                break;
            }
        }
        if (i < n) out.push_back(in[i]);
        ++i;
    }
}

// ---------------------------------------------------------------------------------------------
// One host thread per device, kept for the life of the engine: with kernels in the millisecond range the cost of
// spawning and joining a thread per device and call (tens of microseconds each) would show in the multi-GPU numbers.
// So would a condition-variable wake-up per device and call (30-60 us on a sleeping thread): a thread that has just
// finished a job keeps polling for the next one for half a millisecond before it goes to sleep, the caller's own thread
// drives device 0, and the caller polls briefly for the others before it blocks.
class DevicePool {
public:
    explicit DevicePool(int n) : n_(n)
    {
        for (int d = 1; d < n; ++d) th_.emplace_back([this, d] { loop(d); });
    }
    ~DevicePool()
    {
        stop_.store(true);
        { std::lock_guard<std::mutex> l(mu_); }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    // runs fn(d) for every device d (device 0 on the calling thread, the others on their own) and waits for all of them
    void run(const std::function<void(int)> &fn)
    {
        fn_ = &fn;
        pending_.store(n_ - 1);
        epoch_.fetch_add(1);
        { std::lock_guard<std::mutex> l(mu_); }          // a thread between its check and its wait holds the mutex
        cv_.notify_all();
        std::exception_ptr thrown;                      // the workers hold references into the caller's frame: always wait for them
        try { fn(0); } catch (...) { thrown = std::current_exception(); }
        bool all_done = false;
        for (int spin = 0; spin < (1 << 14) && !all_done; ++spin) { all_done = pending_.load() == 0; if (!all_done) relax(); }
        if (!all_done) {
            std::unique_lock<std::mutex> l(mu_);
            done_.wait(l, [this] { return pending_.load() == 0; });
        }
        if (thrown) std::rethrow_exception(thrown);
    }

private:
    static void relax()
    {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#else
        std::this_thread::yield();
#endif
    }
    void loop(int d)
    {
        uint64_t seen = 0;
        for (;;) {
            const auto t0 = std::chrono::steady_clock::now();
            bool got = false;
            for (int spin = 0; !got; ++spin) {
                if (stop_.load()) return;
                if (epoch_.load() != seen) { got = true; break; }
                relax();
                if ((spin & 255) == 255 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(500)) break;
            }
            if (!got) {
                std::unique_lock<std::mutex> l(mu_);
                cv_.wait(l, [&] { return stop_.load() || epoch_.load() != seen; });
                if (stop_.load()) return;
            }
            seen = epoch_.load();
            (*fn_)(d);
            if (pending_.fetch_sub(1) == 1) {
                { std::lock_guard<std::mutex> l(mu_); }
                done_.notify_all();
            }
        }
    }
    int n_;
    std::vector<std::thread> th_;
    const std::function<void(int)> *fn_ = nullptr;
    std::atomic<uint64_t> epoch_{0};
    std::atomic<int> pending_{0};
    std::atomic<bool> stop_{false};
    std::mutex mu_;
    std::condition_variable cv_, done_;
};

Engine::Engine(const std::vector<std::string> &forward_monomers, const Scoring &sc, std::vector<std::unique_ptr<Backend>> devs)
    : sc_(sc), devs_(std::move(devs))
{
    build_monomer_set(forward_monomers, ms_);
    if (devs_.empty()) throw PlanError{"no device backend"};
    if (devs_.size() > 1) pool_.reset(new DevicePool((int)devs_.size()));
}

Engine::~Engine() {}

void Engine::on_devices(const std::function<void(int)> &fn)
{
    if (ndev() == 1) fn(0);
    else pool_->run(fn);
}

void Engine::set_ed_thr(int ed_thr)
{
    if (ed_thr > -1 && ms_.Lmax > 64 * SD_HW_BLOCKS) throw PlanError{"--ed_thr needs monomers of at most 1536 bp"};
    for (auto &d : devs_) d->set_filter(ed_thr < 0 ? -1 : ed_thr);
}

void Engine::set_plan_hint(int max_seg_len, int64_t nseg_total) { hint_maxlen_ = max_seg_len; hint_nseg_ = nseg_total; }

void Engine::plan_for(const Batch &b)
{
    int maxlen = 0;
    for (int s = 0; s < b.nseg(); ++s) maxlen = std::max(maxlen, b.len(s));
    int64_t per_dev = (b.nseg() + ndev() - 1) / ndev();
    // a streamed run (run_files) announces the shape of the whole job: one plan for all its chunks
    if (hint_nseg_ > 0 && maxlen <= hint_maxlen_) { maxlen = hint_maxlen_; per_dev = std::max<int64_t>(per_dev, std::min<int64_t>((hint_nseg_ + ndev() - 1) / ndev(), 1 << 20)); }
    // re-plan only when the shape changes enough to matter (geometry depends on segment count and length)
    if (have_plan_ && maxlen <= plan_maxlen_ && maxlen * 2 > plan_maxlen_ && per_dev == plan_nseg_) return;
    plan_ = make_plan(ms_, sc_, maxlen, per_dev);
    plan_maxlen_ = maxlen; plan_nseg_ = per_dev; have_plan_ = true;
    for (auto &d : devs_) d->configure(plan_, ms_);
    stats.g = plan_.g;
}

void Engine::note_split(const Batch &b, const std::vector<int> &bounds)
{
    stats.sweep_store_bytes = 0;
    for (int d = 0; d < 8; ++d) stats.dev_segments[d] = 0;
    for (int d = 0; d < ndev(); ++d) {
        if (d < 8) stats.dev_segments[d] = bounds[d + 1] - bounds[d];
        if (bounds[d] == bounds[d + 1]) continue;
        const CtaLayout l = make_cta_layout(plan_, b, bounds[d], bounds[d + 1]);
        stats.sweep_store_bytes += l.cta_code_off.back() * 4 + l.seg_j_off.back() * (int64_t)sizeof(JR);
    }
}

// contiguous, column-balanced ranges, one per device (SURVEY 8e: segments are independent, no collective)
void Engine::split(const Batch &b, std::vector<int> &bounds) const
{
    const int nd = ndev(), nseg = b.nseg();
    bounds.assign(nd + 1, nseg);
    bounds[0] = 0;
    const int64_t total = b.off[nseg] - b.off[0];
    int s = 0;
    for (int d = 1; d < nd; ++d) {
        const int64_t target = b.off[0] + total * d / nd;
        while (s < nseg && b.off[s] < target) ++s;
        int cut = s / plan_.g.NS * plan_.g.NS;           // keep CTAs whole
        bounds[d] = std::max(bounds[d - 1], std::min(cut, nseg));
    }
}

// The wave loop below forms a wave of at least NS segments (one CTA) even when that exceeds the soft wave budget.  Such a
// minimum wave that exceeds the memory the device had free is refused up front, before anything is allocated, instead
// of failing in the middle of a run.  Every minimum wave is one of the NS-aligned blocks of a device's range.
static void check_device_fit(const Backend &dev, const Batch &b, int s0, int s1, int NS)
{
    const int64_t cap = dev.device_bytes();
    for (int s = s0; s < s1; s += NS) {
        const int e = std::min(s1, s + NS);
        const int64_t need = dev.wave_bytes(b, s, e);
        if (need <= cap) continue;
        int longest = 0;
        for (int q = s; q < e; ++q) longest = std::max(longest, b.len(q));
        char msg[256];
        snprintf(msg, sizeof msg, "segment of %d bp needs %lld bytes of device memory for its sweep; %lld bytes are available "
                 "(segment the reads with a smaller -b)", longest, (long long)need, (long long)cap);
        throw PlanError{msg};
    }
}

void Engine::decompose(const Batch &b, BatchResult &out)
{
    out.recs.clear(); out.rec_off.assign(1, 0);
    if (b.nseg() == 0) return;
    for (int s = 0; s < b.nseg(); ++s) if (b.len(s) <= 0) throw PlanError{"empty segment"};
    plan_for(b);
    std::vector<int> bounds; split(b, bounds);
    note_split(b, bounds);
    const int nd = ndev();
    for (int d = 0; d < nd; ++d) check_device_fit(*devs_[d], b, bounds[d], bounds[d + 1], plan_.g.NS);
    std::vector<BatchResult> part(nd);
    std::vector<std::string> errs(nd);
    auto work = [&](int d) {
        try {
            Backend &dev = *devs_[d];
            dev.reset_stats();
            part[d].rec_off.assign(1, 0);
            const int s_end = bounds[d + 1];
            const int nsl = dev.wave_slots();
            // waves: as many segments as fit the budget of one wave slot (with two slots each gets half the memory, and
            // the copies of one wave overlap the kernels of the other)
            const int64_t budget = dev.wave_budget() / nsl;
            const bool prof = getenv("SD_PROFILE") != nullptr;
            std::vector<std::pair<int, int>> waves;
            // The copy-in of the first wave is the only one that cannot hide behind kernels (a segment takes ~10x longer to
            // sweep than to copy), so a large share starts with a small wave and doubles from there: 1/16, 1/8, 1/4, ...
            // of the share, each at most what the memory budget of a wave slot allows.
            const int share = s_end - bounds[d];
            int ramp = (nsl > 1 && share >= 4096) ? std::max(1024, share / 16) / plan_.g.NS * plan_.g.NS : share;
            for (int s0 = bounds[d]; s0 < s_end;) {
                int lo = std::min(s_end, s0 + plan_.g.NS), hi = std::min(s_end, s0 + std::max(ramp, plan_.g.NS));
                if (s_end - hi < ramp / 2) hi = s_end;                 // no tiny last wave
                if (dev.wave_bytes(b, s0, hi) > budget) {
                    while (hi - lo > plan_.g.NS) {
                        int mid = lo + (hi - lo) / 2 / plan_.g.NS * plan_.g.NS;
                        if (mid <= lo) break;
                        if (dev.wave_bytes(b, s0, mid) <= budget) lo = mid; else hi = mid;
                    }
                    hi = lo;
                }
                waves.emplace_back(s0, hi);
                s0 = hi;
                if (ramp < share) ramp *= 2;
            }
            if (waves.size() > 2)
                for (int sl = 0; sl < nsl; ++sl) {              // each slot's buffers sized once, for the largest wave it will hold
                    int best = -1; int64_t bytes = -1;
                    for (size_t w = (size_t)sl; w < waves.size(); w += (size_t)nsl) {
                        const int64_t wb = dev.wave_bytes(b, waves[w].first, waves[w].second);
                        if (wb > bytes) { bytes = wb; best = (int)w; }
                    }
                    if (best >= 0) dev.reserve(sl, b, waves[(size_t)best].first, waves[(size_t)best].second);
                }
            auto now = [] { return std::chrono::steady_clock::now(); };
            auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            const auto t0 = now();
            for (size_t w = 0; w < waves.size(); ++w) {
                dev.submit((int)(w % (size_t)nsl), b, waves[w].first, waves[w].second);
                if (nsl == 1) dev.collect(0, part[d]);
                else if (w >= 1) dev.collect((int)((w - 1) % (size_t)nsl), part[d]);
            }
            if (nsl > 1 && !waves.empty()) dev.collect((int)((waves.size() - 1) % (size_t)nsl), part[d]);
            if (prof) fprintf(stderr, "[sd_b200 profile] dev %d: %zu wave(s), segments [%d,%d): %.3f ms host wall (sweep %.3f traceback %.3f h2d %.3f ms on the device), %d group slot(s)\n",
                              d, waves.size(), bounds[d], s_end, ms(t0, now()), dev.sweep_ms, dev.traceback_ms, dev.h2d_ms, dev.group_slots);
        } catch (PlanError &e) { errs[d] = e.msg.empty() ? "error" : e.msg; }
        catch (std::exception &e) { errs[d] = e.what(); }
    };
    on_devices(work);
    for (int d = 0; d < nd; ++d) if (!errs[d].empty()) throw PlanError{errs[d]};
    double sw = 0, tb = 0, h2d = 0, d2h = 0;
    for (int d = 0; d < nd; ++d) {
        if (nd == 1) { out.recs.swap(part[0].recs); out.rec_off.swap(part[0].rec_off); }    // one device: no merge copy
        else {
            const int64_t base = (int64_t)out.recs.size();
            out.recs.insert(out.recs.end(), part[d].recs.begin(), part[d].recs.end());
            for (size_t x = 1; x < part[d].rec_off.size(); ++x) out.rec_off.push_back(base + part[d].rec_off[x]);
        }
        sw = std::max(sw, devs_[d]->sweep_ms); tb = std::max(tb, devs_[d]->traceback_ms);
        h2d = std::max(h2d, devs_[d]->h2d_ms); d2h = std::max(d2h, devs_[d]->d2h_ms);
        stats.h2d_bytes += devs_[d]->h2d_bytes; stats.d2h_bytes += devs_[d]->d2h_bytes; stats.launches += devs_[d]->launches;
    }
    stats.sweep_ms += sw; stats.traceback_ms += tb; stats.h2d_ms += h2d; stats.d2h_ms += d2h;
    const int64_t cols = b.off[b.nseg()] - b.off[0];
    stats.columns += cols; stats.segments += b.nseg(); stats.cells += cols * (int64_t)ms_.rows.size();
}

void Engine::stage(const Batch &b)
{
    if (b.nseg() == 0) throw PlanError{"nothing to stage"};
    staged_ = b;
    if (staged_.own.empty() && b.nseg()) staged_.own.assign(b.text, b.text + b.off[b.nseg()]);   // outlive the caller's buffer
    staged_.text = staged_.own.data();
    plan_for(staged_);
    split(staged_, staged_bounds_);
    note_split(staged_, staged_bounds_);
    for (int d = 0; d < ndev(); ++d) {
        if (staged_bounds_[d] == staged_bounds_[d + 1]) continue;
        if (devs_[d]->wave_bytes(staged_, staged_bounds_[d], staged_bounds_[d + 1]) > devs_[d]->wave_budget())
            throw PlanError{"staged batch does not fit one wave on the device"};
    }
    std::vector<std::string> errs(ndev());
    auto work = [&](int d) {
        try { if (staged_bounds_[d] < staged_bounds_[d + 1]) devs_[d]->stage(staged_, staged_bounds_[d], staged_bounds_[d + 1]); }
        catch (PlanError &e) { errs[d] = e.msg.empty() ? "error" : e.msg; }
        catch (std::exception &e) { errs[d] = e.what(); }
    };
    on_devices(work);
    for (auto &e : errs) if (!e.empty()) throw PlanError{e};
}

double Engine::run_staged()
{
    if (staged_.nseg() == 0) throw PlanError{"nothing staged"};
    std::vector<std::string> errs(ndev());
    auto work = [&](int d) {
        try {
            devs_[d]->reset_stats();
            if (staged_bounds_[d] < staged_bounds_[d + 1]) devs_[d]->execute();
        } catch (PlanError &e) { errs[d] = e.msg.empty() ? "error" : e.msg; }
        catch (std::exception &e) { errs[d] = e.what(); }
    };
    on_devices(work);
    for (auto &e : errs) if (!e.empty()) throw PlanError{e};
    double ms = 0, sw = 0, tb = 0;
    for (auto &d : devs_) { ms = std::max(ms, d->sweep_ms + d->traceback_ms); sw = std::max(sw, d->sweep_ms); tb = std::max(tb, d->traceback_ms); stats.launches += d->launches; }
    stats.sweep_ms += sw; stats.traceback_ms += tb;
    const int64_t cols = staged_.off[staged_.nseg()] - staged_.off[0];
    stats.columns += cols; stats.segments += staged_.nseg(); stats.cells += cols * (int64_t)ms_.rows.size();
    return ms;
}

void Engine::fetch_staged(BatchResult &out)
{
    out.recs.clear(); out.rec_off.assign(1, 0);
    for (int d = 0; d < ndev(); ++d) {
        if (staged_bounds_[d] == staged_bounds_[d + 1]) continue;
        devs_[d]->fetch(out);
    }
}

// ---------------------------------------------------------------------------------------------
namespace {

struct FdWriter {
    int fd; std::string buf;
    explicit FdWriter(int f) : fd(f) { buf.reserve(1 << 20); }
    bool failed = false;             // a write() error other than EINTR: the output is incomplete (ENOSPC, EPIPE, ...)
    bool flush()
    {
        if (fd < 0) return true;
        size_t o = 0;
        while (o < buf.size()) {
            ssize_t w = ::write(fd, buf.data() + o, buf.size() - o);
            if (w < 0 && errno == EINTR) continue;
            if (w <= 0) { failed = true; break; }
            o += (size_t)w;
        }
        buf.clear();
        return !failed;
    }
    void add(const std::string &s) { buf += s; if (buf.size() > (1 << 20)) flush(); }
    void add_int(long v) { char t[24]; int n = 0; bool neg = v < 0; unsigned long u = neg ? 0ul - (unsigned long)v : (unsigned long)v;
        do { t[n++] = (char)('0' + u % 10); u /= 10; } while (u); if (neg) t[n++] = '-'; while (n) buf.push_back(t[--n]); }
    ~FdWriter() { flush(); }
};

} // namespace

// A bounded hand-over between two stages of the host pipeline (reader -> device -> writer).
template <class T> class Handoff {
public:
    explicit Handoff(size_t cap) : cap_(cap) {}
    void push(T v)
    {
        std::unique_lock<std::mutex> l(mu_);
        room_.wait(l, [&] { return q_.size() < cap_ || closed_; });
        if (closed_) return;
        q_.push_back(std::move(v));
        item_.notify_one();
    }
    bool pop(T &out)                                        // false once the producer has finished and the queue is empty
    {
        std::unique_lock<std::mutex> l(mu_);
        item_.wait(l, [&] { return !q_.empty() || done_ || closed_; });
        if (q_.empty()) return false;
        out = std::move(q_.front()); q_.erase(q_.begin());
        room_.notify_one();
        return true;
    }
    void finish() { std::lock_guard<std::mutex> l(mu_); done_ = true; item_.notify_all(); }
    void close() { std::lock_guard<std::mutex> l(mu_); closed_ = true; q_.clear(); item_.notify_all(); room_.notify_all(); }   // a stage failed

private:
    size_t cap_;
    std::vector<T> q_;
    std::mutex mu_;
    std::condition_variable item_, room_;
    bool done_ = false, closed_ = false;
};

// A chunk of work: whole segments of consecutive reads (a long read may straddle chunks), packed for the device.
struct Chunk {
    Batch b;
    std::vector<int> seg_read;              // read index of each segment
    std::vector<int> seg_off;               // offset of each segment in its read
    BatchResult res;
};

int run_files(const std::string &reads_path, const std::string &monomers_path, int threads, int part_size, int overlap,
              const Scoring &sc, int ed_thr, DeviceOpener open_devices, int out_fd, int err_fd, std::string &error)
{
    (void)threads;     // OpenMP width in the reference (main.cpp:85,88); the output does not depend on it
    FdWriter err(err_fd);
    std::vector<std::unique_ptr<Backend>> devs;
    std::string dev_error;
    std::future<int> dev_ready = std::async(std::launch::async, [&] { return open_devices(devs, dev_error); });
    err.add("Scores: insertion=" + std::to_string(sc.ins) + " deletion=" + std::to_string(sc.del) + " mismatch=" +
            std::to_string(sc.mismatch) + " match=" + std::to_string(sc.match) + "\n");                  // main.cpp:393
    err.flush();
    const bool prof = getenv("SD_PROFILE") != nullptr;
    auto tnow = [] { return std::chrono::steady_clock::now(); };
    auto tms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    const auto t_begin = tnow();

    // Pass 1 over the reads (while the devices are being opened): names, lengths, alphabet check.  The reference loads and
    // checks both files completely before it aligns anything (main.cpp:394-395), so an illegal symbol anywhere means no
    // output at all; the sequences themselves are only read in pass 2, chunk by chunk.
    FastaIndex ridx;
    FastaSet mons;
    std::string diag;
    int st = index_fasta(reads_path, ridx, diag);
    err.add(diag); err.flush(); diag.clear();
    if (st) return st;
    st = load_fasta(monomers_path, mons, diag);
    err.add(diag); err.flush();
    if (st) return st;
    if (part_size <= 0) { error = "part-size must be positive"; err.add("ERROR: " + error + "\n"); return 1; }

    // segmentation of all reads, in read order (main.cpp:70-81): counts only
    const size_t nreads = ridx.lens.size();
    std::vector<int64_t> read_nseg(nreads, 0);
    int64_t nseg_total = 0;
    int max_seg_len = 0;
    for (size_t p = 0; p < nreads; ++p) {
        read_nseg[p] = segment_read(ridx.lens[p], part_size, overlap, nullptr);
        nseg_total += read_nseg[p];
        if (read_nseg[p]) max_seg_len = (int)std::max<int64_t>(max_seg_len, std::min<int64_t>(ridx.lens[p], (int64_t)part_size + overlap));
    }
    err.add("Prepared reads\n"); err.flush();                                                                    // main.cpp:82
    if (nseg_total == 0) return 0;
    if (mons.seqs.empty()) { error = "no monomers"; err.add("ERROR: " + error + "\n"); return 1; }
    const auto t_indexed = tnow();

    // Pass 2: reader thread -> device (this thread) -> writer thread.  A chunk holds up to chunk_cols read symbols, so
    // that the three stages overlap on anything larger than a few tens of megabases; host memory is bounded by the
    // chunks in flight (two per hand-over) plus the read being assembled, whatever the size of the file.  The reader
    // starts now, while the devices are still being opened: the first chunks are waiting when the context is up.
    int64_t chunk_cols = (int64_t)32 << 20;
    if (const char *e = getenv("SD_CHUNK_BASES")) if (atoll(e) > 0) chunk_cols = atoll(e);
    Handoff<std::unique_ptr<Chunk>> to_device(2), to_writer(2);
    std::string reader_error, writer_error;

    std::thread reader([&] {
        try {
            std::unique_ptr<Chunk> cur(new Chunk);
            cur->b.off.push_back(0);
            int ridx_now = -1;
            std::string seq;
            std::vector<std::pair<int, int>> cuts;
            auto flush_read = [&] {                                   // cut the finished read into segments (main.cpp:73-79)
                if (ridx_now < 0) return;
                cuts.clear();
                segment_read((int64_t)seq.size(), part_size, overlap, &cuts);
                for (auto &c : cuts) {
                    if ((int64_t)cur->b.own.size() + c.second > chunk_cols && !cur->seg_read.empty()) {
                        cur->b.text = cur->b.own.data();
                        to_device.push(std::move(cur));
                        cur.reset(new Chunk); cur->b.off.push_back(0);
                    }
                    cur->b.own.insert(cur->b.own.end(), seq.begin() + c.first, seq.begin() + c.first + c.second);
                    cur->b.off.push_back((int64_t)cur->b.own.size());
                    cur->seg_read.push_back(ridx_now); cur->seg_off.push_back(c.first);
                }
            };
            scan_fasta(reads_path,
                [&](const char *, const char *) { flush_read(); ++ridx_now; seq.clear(); if (ridx_now < (int)nreads) seq.reserve((size_t)ridx.lens[(size_t)ridx_now]); },
                [&](const char *p, const char *le) { if (ridx_now >= 0) seq.append(p, le); });
            flush_read();
            if (!cur->seg_read.empty()) { cur->b.text = cur->b.own.data(); to_device.push(std::move(cur)); }
        } catch (std::exception &e) { reader_error = e.what(); }
        to_device.finish();
    });
    struct JoinOnExit {                              // early returns below: stop the reader before its captures go away
        Handoff<std::unique_ptr<Chunk>> &q; std::thread &t;
        ~JoinOnExit() { if (t.joinable()) { q.close(); t.join(); } }
    } reader_guard{to_device, reader};

    if (int dst = dev_ready.get()) {                 // no usable device: fail loudly, there is no CPU path
        error = dev_error;
        err.add("ERROR: " + error + "\n");
        return dst;
    }
    const auto t_device = tnow();
    std::unique_ptr<Engine> eng;
    try {
        eng.reset(new Engine(mons.seqs, sc, std::move(devs)));
        eng->set_ed_thr(ed_thr);          // FilterMonomersForRead (main.cpp:91-93,135-149) when ed_thr > -1
        eng->set_plan_hint(max_seg_len, nseg_total);
    } catch (PlanError &e) {
        error = e.msg;
        err.add("ERROR: " + error + "\n");
        return 3;
    }

    const int M = (int)mons.seqs.size();
    FdWriter outw(out_fd);
    std::thread writer([&] {
        // per read: add segment offsets (main.cpp:110), PostProcessing (:116), SaveBatch (:117, :272-285), in read order
        try {
            std::unique_ptr<Chunk> c;
            std::vector<Record> all, kept;
            int cur_read = -1; int64_t seen = 0;
            auto finish_read = [&] {
                if (cur_read < 0 || all.empty()) { all.clear(); return; }     // a read without alignments: the reference has UB here (SURVEY App. B)
                err.add(std::to_string(((size_t)cur_read + 1) * 100 / nreads) + "%: Aligned " + ridx.names[(size_t)cur_read] + "\n");   // main.cpp:115
                err.flush();
                postprocess(all, kept);
                int prev_end = 0;
                const std::string &rname = ridx.names[(size_t)cur_read];
                for (const Record &r : kept) {
                    outw.buf += rname; outw.buf.push_back('\t');
                    outw.buf += mons.names[(size_t)(r.row < M ? r.row : r.row - M)];
                    if (r.row >= M) outw.buf.push_back('\'');
                    outw.buf.push_back('\t'); outw.add_int(r.start);
                    outw.buf.push_back('\t'); outw.add_int(r.end);
                    outw.buf.push_back('\t'); outw.add_int(r.score); outw.buf += ".000000";      // to_string(float), main.cpp:279
                    outw.buf.push_back('\t'); outw.add_int(r.start - prev_end);
                    outw.buf.push_back('\t'); outw.add_int(r.end - r.start);
                    outw.buf.push_back('\n');
                    prev_end = r.end;
                }
                if (outw.buf.size() > (1 << 20) && !outw.flush()) throw std::runtime_error(std::string("writing the raw decomposition failed: ") + strerror(errno));
                all.clear();
            };
            while (to_writer.pop(c)) {
                for (size_t sgi = 0; sgi < c->seg_read.size(); ++sgi) {
                    if (c->seg_read[sgi] != cur_read) { finish_read(); cur_read = c->seg_read[sgi]; seen = 0; }
                    for (int64_t x = c->res.rec_off[sgi]; x < c->res.rec_off[sgi + 1]; ++x) {
                        Record r = c->res.recs[(size_t)x];
                        r.start += c->seg_off[sgi]; r.end += c->seg_off[sgi];
                        all.push_back(r);
                    }
                    if (++seen == read_nseg[(size_t)cur_read]) { finish_read(); cur_read = -1; }
                }
            }
            finish_read();
            if (!outw.flush()) throw std::runtime_error(std::string("writing the raw decomposition failed: ") + strerror(errno));
        } catch (std::exception &e) { writer_error = e.what(); to_writer.close(); }
    });

    std::string engine_error;
    double dev_ms = 0;
    {
        std::unique_ptr<Chunk> c;
        while (to_device.pop(c)) {
            if (!engine_error.empty() || !writer_error.empty()) continue;          // drain
            try {
                const auto t0 = tnow();
                eng->decompose(c->b, c->res);
                dev_ms += tms(t0, tnow());
                c->b.own.clear(); c->b.own.shrink_to_fit();
                to_writer.push(std::move(c));
            } catch (PlanError &e) { engine_error = e.msg.empty() ? "error" : e.msg; to_device.close(); }
            catch (std::exception &e) { engine_error = e.what(); to_device.close(); }
        }
    }
    to_writer.finish();
    reader.join();
    writer.join();
    const auto t_done = tnow();
    if (!engine_error.empty() || !reader_error.empty()) {
        error = !engine_error.empty() ? engine_error : reader_error;
        err.add("ERROR: " + error + "\n");
        return 3;
    }
    if (!writer_error.empty()) {                    // ENOSPC / EPIPE ...: a truncated raw TSV must not look like success
        error = writer_error;
        err.add("ERROR: " + error + "\n");
        return 5;
    }
    if (getenv("SD_VERBOSE")) {
        const EngineStats &es = eng->stats;
        char line[512];
        // with several waves the traceback of one wave shares the device with the sweep of the next: its time is then
        // mostly waiting for free SMs and lies inside the sweep time, so the rates are quoted on the sweep and on the calls
        snprintf(line, sizeof line, "[sd_b200] devices=%d geometry packed=%d lat=%d C=%d T=%d NS=%d NT=%d NG=%d segments=%ld cells=%ld sweep=%.3f ms traceback=%.3f ms -> %.1f GCUPS (sweep), %.1f GCUPS (device calls with copies, %.1f ms)\n",
                 eng->ndev(), es.g.packed, es.g.lat, es.g.C, es.g.T, es.g.NS, es.g.NT, es.g.NG, (long)es.segments, (long)es.cells, es.sweep_ms, es.traceback_ms,
                 es.cells / (es.sweep_ms * 1e6 + 1e-9), es.cells / (dev_ms * 1e6 + 1e-9), dev_ms);
        err.add(line);
    }
    if (const char *pj = getenv("SD_PERF_JSON")) {
        // machine-readable summary of the run, appended to a side file (stdout is the data channel, SURVEY section 5)
        if (FILE *f = fopen(pj, "a")) {
            const EngineStats &es = eng->stats;
            int64_t read_bp = 0;
            for (int64_t l : ridx.lens) read_bp += l;
            const double wall = tms(t_begin, t_done);
            fprintf(f, "{\"reads\": %zu, \"read_bp\": %ld, \"segments\": %ld, \"columns\": %ld, \"cells\": %ld, \"devices\": %d, "
                       "\"sweep_ms\": %.3f, \"traceback_ms\": %.3f, \"h2d_ms\": %.3f, \"device_calls_ms\": %.3f, \"wall_ms\": %.3f, "
                       "\"wait_for_device_ms\": %.3f, \"sweep_gcups\": %.2f, \"wall_mbp_per_s\": %.3f, "
                       "\"geometry\": {\"packed\": %d, \"lat\": %d, \"C\": %d, \"T\": %d, \"NS\": %d, \"NT\": %d, \"NG\": %d, \"scanw\": %d}}\n",
                    nreads, (long)read_bp, (long)es.segments, (long)es.columns, (long)es.cells, eng->ndev(), es.sweep_ms, es.traceback_ms, es.h2d_ms,
                    dev_ms, wall, tms(t_indexed, t_device), es.cells / (es.sweep_ms * 1e6 + 1e-9), read_bp / (wall * 1e3 + 1e-9),
                    es.g.packed, es.g.lat, es.g.C, es.g.T, es.g.NS, es.g.NT, es.g.NG, es.g.scanw);
            fclose(f);
        }
    }
    if (prof) {
        char line[320];
        snprintf(line, sizeof line, "[sd_b200 profile] run_files: index %.1f wait-for-device %.1f stream+decompose+write %.1f ms (device calls %.1f ms; %ld segments)\n",
                 tms(t_begin, t_indexed), tms(t_indexed, t_device), tms(t_device, t_done), dev_ms, (long)nseg_total);
        err.add(line);
    }
    // The `dp` process exits right after this call: its device buffers need no orderly release (dp_main.cpp).
    if (getenv("SD_FAST_EXIT")) (void)eng.release();
    return 0;
}

} // namespace sdb
