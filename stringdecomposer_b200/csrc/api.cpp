// api.cpp -- the C ABI declared in include/sd_b200.h.
#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <cstdio>
#include <mutex>
#include <unistd.h>

#include "../../include/sd_b200.h"
#include "pipeline.h"
#include "identity_core.cuh"

using namespace sdb;

#ifdef SD_EMULATOR_BUILD
static const bool kEmu = true;      // libsd_emu.so: CPU test-suite only
#else
static const bool kEmu = false;     // libsd_b200.so: CUDA only, no fallback
#endif

struct sd_handle {
    std::unique_ptr<Engine> eng;
    std::string err;
    int n_devices = 0;
};

static std::string g_err;
static std::mutex g_mu;
static void set_global_error(const std::string &e) { std::lock_guard<std::mutex> l(g_mu); g_err = e; }

#ifndef SD_EMULATOR_BUILD
namespace sdb { Backend *make_emu_backend() { return nullptr; } }
int cuda_device_count();
void *cuda_host_alloc(size_t bytes);
void cuda_host_free(void *p);
int cuda_int_peak(int device, double *alu, double *both, double *mhz, std::string &err);
namespace sdb { int cuda_identity(const IdentityArgs &h, int max_qlen, int max_tlen, int device, double *kernel_ms, std::string &err); }
static int run_identity(const IdentityArgs &h, int mq, int mt, int device, double *ms, std::string &err) { return cuda_identity(h, mq, mt, device, ms, err); }
#else
namespace sdb { int emu_identity(const IdentityArgs &h, int max_qlen, int max_tlen, double *kernel_ms, std::string &err); }
static int run_identity(const IdentityArgs &h, int mq, int mt, int, double *ms, std::string &err) { return emu_identity(h, mq, mt, ms, err); }
namespace sdb { Backend *make_cuda_backend(int, std::string &err) { err = "emulator build"; return nullptr; } }
static int cuda_device_count() { return 1; }
static void *cuda_host_alloc(size_t bytes) { return malloc(bytes ? bytes : 1); }
static void cuda_host_free(void *p) { free(p); }
static int cuda_int_peak(int, double *, double *, double *, std::string &err) { err = "emulator build has no device"; return SD_ERR_NO_DEVICE; }
#endif

static int make_backends(const int32_t *ids, int32_t n, std::vector<std::unique_ptr<Backend>> &out, std::string &err)
{
    if (kEmu) { out.emplace_back(make_emu_backend()); return SD_OK; }
    std::vector<int> dev;
    const int avail = cuda_device_count();
    if (avail <= 0) { err = "no CUDA device is visible: libsd_b200 has no CPU path"; return SD_ERR_NO_DEVICE; }
    if (n == 0) dev.push_back(0);
    else if (n < 0) for (int d = 0; d < avail; ++d) dev.push_back(d);
    else for (int i = 0; i < n; ++i) dev.push_back(ids ? ids[i] : i);
    for (int d : dev) {
        if (d < 0 || d >= avail) { err = "device id out of range"; return SD_ERR_ARG; }
        Backend *b = make_cuda_backend(d, err);
        if (!b) return SD_ERR_NO_DEVICE;
        out.emplace_back(b);
    }
    return SD_OK;
}

static int to_batch(const char *segments, const int64_t *offsets, int64_t n, Batch &b, std::string &err)
{
    if (n < 0 || (n > 0 && (!segments || !offsets))) { err = "bad segment arguments"; return SD_ERR_ARG; }
    b.off.assign((size_t)n + 1, 0);
    const int64_t base = n ? offsets[0] : 0;
    for (int64_t s = 0; s <= n && n; ++s) {
        b.off[(size_t)s] = offsets[s] - base;
        if (s && offsets[s] <= offsets[s - 1]) { err = "segments must be non-empty and offsets increasing"; return SD_ERR_ARG; }
    }
    b.text = reinterpret_cast<const uint8_t *>(segments) + base;     // encoded and validated on the device
    return SD_OK;
}

static int status_of(const std::string &msg)
{
    if (msg.find("symbol outside") != std::string::npos) return SD_ERR_INPUT;
    if (msg.rfind("internal error:", 0) == 0) return SD_ERR_INTERNAL;
    if (msg.find("CUDA") != std::string::npos) return SD_ERR_CUDA;
    return SD_ERR_UNSUPPORTED;
}

static int export_result(const BatchResult &res, sd_record **records, int64_t **rec_offsets)
{
    static_assert(sizeof(sd_record) == sizeof(Record), "record layout");
    sd_record *r = (sd_record *)malloc(sizeof(sd_record) * std::max<size_t>(res.recs.size(), 1));
    int64_t *o = (int64_t *)malloc(sizeof(int64_t) * res.rec_off.size());
    if (!r || !o) { free(r); free(o); return SD_ERR_INTERNAL; }
    if (!res.recs.empty()) memcpy(r, res.recs.data(), sizeof(sd_record) * res.recs.size());
    memcpy(o, res.rec_off.data(), sizeof(int64_t) * res.rec_off.size());
    *records = r; *rec_offsets = o;
    return SD_OK;
}

extern "C" {

int sd_create(const char *monomers, const int64_t *offsets, int32_t n_monomers, int32_t ins, int32_t del,
              int32_t mismatch, int32_t match, const int32_t *device_ids, int32_t n_devices, sd_handle **out)
{
    if (!out) return SD_ERR_ARG;
    *out = nullptr;
    if (!monomers || !offsets || n_monomers <= 0) { set_global_error("bad monomer arguments"); return SD_ERR_ARG; }
    std::vector<std::string> fwd;
    for (int j = 0; j < n_monomers; ++j) {
        if (offsets[j + 1] <= offsets[j]) { set_global_error("monomers must be non-empty"); return SD_ERR_ARG; }
        fwd.emplace_back(monomers + offsets[j], (size_t)(offsets[j + 1] - offsets[j]));
    }
    std::string err;
    std::vector<std::unique_ptr<Backend>> devs;
    int st = make_backends(device_ids, n_devices, devs, err);
    if (st) { set_global_error(err); return st; }
    try {
        std::unique_ptr<sd_handle> h(new sd_handle);
        h->n_devices = (int)devs.size();
        Scoring sc; sc.ins = ins; sc.del = del; sc.mismatch = mismatch; sc.match = match;
        h->eng.reset(new Engine(fwd, sc, std::move(devs)));
        *out = h.release();
    } catch (PlanError &e) { set_global_error(e.msg); return SD_ERR_ARG; }
    return SD_OK;
}

int sd_decompose(sd_handle *h, const char *segments, const int64_t *offsets, int64_t n_segments,
                 sd_record **records, int64_t **rec_offsets)
{
    if (!h || !records || !rec_offsets) return SD_ERR_ARG;
    Batch b;
    const auto t0 = std::chrono::steady_clock::now();
    int st = to_batch(segments, offsets, n_segments, b, h->err);
    if (st) return st;
    const auto t1 = std::chrono::steady_clock::now();
    BatchResult res;
    try { h->eng->decompose(b, res); }
    catch (PlanError &e) { h->err = e.msg; return status_of(e.msg); }
    catch (std::exception &e) { h->err = e.what(); return SD_ERR_INTERNAL; }
    const auto t2 = std::chrono::steady_clock::now();
    st = export_result(res, records, rec_offsets);
    if (getenv("SD_PROFILE")) {
        const auto t3 = std::chrono::steady_clock::now();
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        fprintf(stderr, "[sd_b200 profile] sd_decompose: encode %.3f decompose %.3f export %.3f ms\n", ms(t0, t1), ms(t1, t2), ms(t2, t3));
    }
    return st;
}

int sd_stage(sd_handle *h, const char *segments, const int64_t *offsets, int64_t n_segments)
{
    if (!h) return SD_ERR_ARG;
    Batch b;
    int st = to_batch(segments, offsets, n_segments, b, h->err);
    if (st) return st;
    try { h->eng->stage(b); }
    catch (PlanError &e) { h->err = e.msg; return status_of(e.msg); }
    catch (std::exception &e) { h->err = e.what(); return SD_ERR_INTERNAL; }
    return SD_OK;
}

int sd_run_staged(sd_handle *h, double *kernel_ms)
{
    if (!h) return SD_ERR_ARG;
    try { double ms = h->eng->run_staged(); if (kernel_ms) *kernel_ms = ms; }
    catch (PlanError &e) { h->err = e.msg; return status_of(e.msg); }
    catch (std::exception &e) { h->err = e.what(); return SD_ERR_INTERNAL; }
    return SD_OK;
}

int sd_fetch_staged(sd_handle *h, sd_record **records, int64_t **rec_offsets)
{
    if (!h || !records || !rec_offsets) return SD_ERR_ARG;
    BatchResult res;
    try { h->eng->fetch_staged(res); }
    catch (PlanError &e) { h->err = e.msg; return SD_ERR_CUDA; }
    catch (std::exception &e) { h->err = e.what(); return SD_ERR_INTERNAL; }
    return export_result(res, records, rec_offsets);
}

int64_t sd_segment_read(int64_t read_len, int32_t part_size, int32_t overlap, int64_t *offs, int32_t *lens, int64_t cap)
{
    if (read_len < 0) return -1;
    std::vector<std::pair<int, int>> v;
    int64_t n = segment_read(read_len, part_size, overlap, &v);
    if (n < 0) return n;
    if (offs && lens) for (int64_t i = 0; i < n && i < cap; ++i) { offs[i] = v[(size_t)i].first; lens[i] = v[(size_t)i].second; }
    return n;
}

int64_t sd_postprocess(const sd_record *in, int64_t n, sd_record *out)
{
    if (n < 0 || (n && (!in || !out))) return -1;
    std::vector<Record> a((size_t)n), b;
    if (n) memcpy(a.data(), in, sizeof(Record) * (size_t)n);
    postprocess(a, b);
    if (!b.empty()) memcpy(out, b.data(), sizeof(Record) * b.size());
    return (int64_t)b.size();
}

int sd_run_files(const char *reads_path, const char *monomers_path, int32_t threads, int32_t part_size, int32_t overlap,
                 int32_t ins, int32_t del, int32_t mismatch, int32_t match, int32_t ed_thr, int out_fd, int err_fd)
{
    if (!reads_path || !monomers_path) return SD_ERR_ARG;
    std::string err;
    int32_t ndev = 0;
    if (const char *e = getenv("SD_DEVICES")) ndev = (strcmp(e, "all") == 0) ? -1 : atoi(e);
    auto open_devices = [ndev](std::vector<std::unique_ptr<Backend>> &devs, std::string &e) { return make_backends(nullptr, ndev, devs, e); };
    Scoring sc; sc.ins = ins; sc.del = del; sc.mismatch = mismatch; sc.match = match;
    int st = run_files(reads_path, monomers_path, threads, part_size, overlap, sc, ed_thr, open_devices, out_fd, err_fd, err);
    if (!err.empty()) set_global_error(err);
    return st;
}

int sd_set_ed_thr(sd_handle *h, int32_t ed_thr)
{
    if (!h) return SD_ERR_ARG;
    try { h->eng->set_ed_thr(ed_thr); }
    catch (PlanError &e) { h->err = e.msg; return SD_ERR_UNSUPPORTED; }
    return SD_OK;
}

int32_t sd_hw_distance(const char *query, int32_t query_len, const char *target, int32_t target_len)
{
    if (!query || !target || query_len <= 0 || target_len < 0 || query_len > 64 * SD_HW_BLOCKS) return -1;
    return hw_distance(reinterpret_cast<const uint8_t *>(query), query_len, reinterpret_cast<const uint8_t *>(target), target_len);
}

int sd_identity(const char *queries, const int64_t *qoff, int64_t nq, const char *targets, const int64_t *toff, int64_t nt,
                const int32_t *pair_q, const int32_t *pair_t, int64_t npairs, int32_t *matches, int32_t *columns,
                int32_t *distance, int32_t device, int64_t *hirschberg_pairs, double *kernel_ms)
{
    std::string err;
    auto fail = [&](int st, const char *msg) { set_global_error(msg); return st; };
    if (nq < 0 || nt < 0 || npairs < 0 || !qoff || !toff || (npairs > 0 && (!matches || !columns))) return fail(SD_ERR_ARG, "sd_identity: bad arguments");
    if ((pair_q == nullptr) != (pair_t == nullptr)) return fail(SD_ERR_ARG, "sd_identity: pair_query and pair_target go together");
    if (!pair_q && npairs != nq * nt) return fail(SD_ERR_ARG, "sd_identity: n_pairs must be n_queries * n_targets without a pair list");
    if (nq > INT32_MAX || nt > INT32_MAX) return fail(SD_ERR_ARG, "sd_identity: too many sequences");
    int max_q = 0, max_t = 0;
    for (int64_t i = 0; i < nq; ++i) {
        const int64_t l = qoff[i + 1] - qoff[i];
        if (l < 0) return fail(SD_ERR_ARG, "sd_identity: query offsets must not decrease");
        if (l > SD_NW_MAXLEN) return fail(SD_ERR_UNSUPPORTED, "sd_identity: sequence longer than 16382");
        max_q = std::max<int>(max_q, (int)l);
    }
    for (int64_t i = 0; i < nt; ++i) {
        const int64_t l = toff[i + 1] - toff[i];
        if (l < 0) return fail(SD_ERR_ARG, "sd_identity: target offsets must not decrease");
        if (l > SD_NW_MAXLEN) return fail(SD_ERR_UNSUPPORTED, "sd_identity: sequence longer than 16382");
        max_t = std::max<int>(max_t, (int)l);
    }
    if ((qoff[nq] > qoff[0] && !queries) || (toff[nt] > toff[0] && !targets) || qoff[0] != 0 || toff[0] != 0) return fail(SD_ERR_ARG, "sd_identity: bad text buffers");
    int64_t hb = 0;
    for (int64_t p = 0; p < npairs; ++p) {
        const int64_t qi = pair_q ? pair_q[p] : p / nt, ti = pair_q ? pair_t[p] : p % nt;
        if (qi < 0 || qi >= nq || ti < 0 || ti >= nt) return fail(SD_ERR_ARG, "sd_identity: pair index out of range");
        if (!nw_edlib_traceback_domain((int)(qoff[qi + 1] - qoff[qi]), (int)(toff[ti + 1] - toff[ti]))) ++hb;
    }
    if (hirschberg_pairs) *hirschberg_pairs = hb;
    if (kernel_ms) *kernel_ms = 0;
    if (npairs == 0) return SD_OK;
    if (!kEmu && (device < 0 || device >= cuda_device_count())) return fail(SD_ERR_NO_DEVICE, "sd_identity: no such CUDA device (libsd_b200 has no CPU path)");
    IdentityArgs a{};
    a.qtext = queries; a.qoff = qoff; a.nq = nq; a.ttext = targets; a.toff = toff; a.nt = nt;
    a.pair_q = pair_q; a.pair_t = pair_t; a.npairs = npairs; a.matches = matches; a.columns = columns; a.distance = distance;
    const int st = run_identity(a, max_q, max_t, device, kernel_ms, err);
    if (st) { set_global_error(err); return st == 2 ? SD_ERR_NO_DEVICE : SD_ERR_CUDA; }
    return SD_OK;
}

int sd_get_stats(sd_handle *h, sd_stats *o)
{
    if (!h || !o) return SD_ERR_ARG;
    const EngineStats &s = h->eng->stats;
    memset(o, 0, sizeof *o);
    o->sweep_ms = s.sweep_ms; o->traceback_ms = s.traceback_ms; o->h2d_ms = s.h2d_ms; o->d2h_ms = s.d2h_ms;
    o->h2d_bytes = s.h2d_bytes; o->d2h_bytes = s.d2h_bytes; o->cells = s.cells; o->segments = s.segments;
    o->columns = s.columns; o->launches = s.launches; o->n_devices = h->n_devices;
    o->packed = s.g.packed; o->C = s.g.C; o->T = s.g.T; o->NS = s.g.NS; o->NT = s.g.NT;
    o->NG = s.g.NG; o->lat = s.g.lat; o->scanw = s.g.scanw; o->stream = s.g.stream;
    o->sweep_store_bytes = s.sweep_store_bytes;
    for (int d = 0; d < 8; ++d) o->dev_segments[d] = s.dev_segments[d];
    return SD_OK;
}

void sd_reset_stats(sd_handle *h)
{
    if (!h) return;
    const EngineStats old = h->eng->stats;
    h->eng->stats = EngineStats();
    h->eng->stats.g = old.g; h->eng->stats.sweep_store_bytes = old.sweep_store_bytes;
    for (int d = 0; d < 8; ++d) h->eng->stats.dev_segments[d] = old.dev_segments[d];
}

const char *sd_last_error(sd_handle *h)
{
    if (h) return h->err.c_str();
    std::lock_guard<std::mutex> l(g_mu);
    static thread_local std::string copy;
    copy = g_err;
    return copy.c_str();
}

void sd_free(void *p) { free(p); }
void *sd_host_alloc(int64_t bytes) { return bytes < 0 ? nullptr : cuda_host_alloc((size_t)bytes); }
void sd_host_free(void *p) { if (p) cuda_host_free(p); }
void sd_destroy(sd_handle *h) { delete h; }
int sd_device_count(void) { return kEmu ? 0 : cuda_device_count(); }
const char *sd_version(void) { return kEmu ? "stringdecomposer_b200 0.1 (host emulator, tests only)" : "stringdecomposer_b200 0.1 (sm_100a)"; }

int sd_int_peak(int32_t device, double *alu, double *both, double *mhz)
{
    std::string err;
    int st = cuda_int_peak(device, alu, both, mhz, err);
    if (st) set_global_error(err);
    return st;
}

} // extern "C"
