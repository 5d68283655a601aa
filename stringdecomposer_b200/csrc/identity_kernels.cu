// identity_kernels.cu -- batched global-alignment identity on the device (SURVEY §8 f1; replaces the per-alignment
// edlib.align calls of stringdecomposer/main.py:29-60,96-150).  Eight lanes per (interval, monomer) pair, four pairs
// per warp: a lane owns a strip of R query rows and the group sweeps the target columns as a skewed wavefront; the
// only cross-lane traffic is one SHFL.UP per step.  No matrix and no traceback state ever leave the registers (identity_core.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <string>
#include <vector>

#include "common.h"
#include "cuda_scope.h"
#include "identity_core.cuh"

namespace sdb {

#define SDI_CUDA(x)                                                                                             \
    do {                                                                                                        \
        cudaError_t e_ = (x);                                                                                   \
        if (e_ != cudaSuccess) throw PlanError{std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " +  \
                                               __FILE__ + ":" + std::to_string(__LINE__)};                      \
    } while (0)

template <int R, int L>
__global__ void __launch_bounds__(256) identity_kernel(IdentityArgs a)
{
    constexpr int G = 32 / L;
    const int lane = threadIdx.x & 31, gl = lane % L, sub = lane / L;
    const unsigned mask = (0xffffffffu >> (32 - L)) << (sub * L);     // this group's lanes; no shift by 32 when L = 32
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t group = warp * G + sub, ngroups = (((int64_t)gridDim.x * blockDim.x) >> 5) * G;
    uint32_t *scratch = a.scratch ? a.scratch + group * a.scratch_stride : nullptr;
    for (int64_t p = group; p < a.npairs; p += ngroups) {
        const int64_t qi = a.pair_q ? a.pair_q[p] : p / a.nt, ti = a.pair_q ? a.pair_t[p] : p % a.nt;
        const char *q = a.qtext + a.qoff[qi], *t = a.ttext + a.toff[ti];
        const int qlen = (int)(a.qoff[qi + 1] - a.qoff[qi]), tlen = (int)(a.toff[ti + 1] - a.toff[ti]);
        if (qlen == 0 || tlen == 0) {                       // main.py:30-33: no alignment, identity 0
            if (gl == 0) { a.matches[p] = 0; a.columns[p] = 0; a.distance[p] = -1; }
            continue;
        }
        const int ntiles = (qlen + L * R - 1) / (L * R);
        NwLane<R> st;
        for (int tile = 0; tile < ntiles; ++tile) {
            const int base = tile * L * R;
            nw_lane_init<R>(st, q, qlen, base + gl * R);
            const int nl = min(L, (qlen - base + R - 1) / R);           // lanes that own at least one row
            const bool spill = tile + 1 < ntiles;                       // the last lane's bottom row feeds the next tile
            uint32_t bottom = 0;
            const int nsteps = tlen + nl - 1;
            for (int s = 0; s < nsteps; ++s) {
                uint32_t top = __shfl_up_sync(mask, bottom, 1, L);
                const int j = s - gl;
                if (j >= 0 && j < tlen) {
                    if (gl == 0) top = tile == 0 ? (uint32_t)(j + 1) << NW_DSHIFT : scratch[j];
                    bottom = nw_lane_step<R>(st, top, (uint32_t)(uint8_t)__ldg(t + j));
                    if (spill && gl == L - 1) scratch[j] = bottom;
                }
            }
            __syncwarp(mask);
        }
        const int fr = qlen - 1 - (ntiles - 1) * L * R;
        uint32_t v = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) if (r == fr % R) v = st.left[r];
        v = __shfl_sync(mask, v, fr / R, L);
        if (gl == 0) {
            const int d = (int)(v >> NW_DSHIFT), m = (int)(v & 0xffffu);
            a.matches[p] = m; a.columns[p] = m + d; a.distance[p] = d;
        }
    }
}

namespace {
// One grow-only device arena per GPU, kept between calls: convert_tsv issues many calls of similar size and
// cudaMalloc / cudaFree would otherwise cost more than the kernel.
struct Arena {
    char *base = nullptr; size_t cap = 0, used = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    void reserve(size_t n) {
        used = 0;
        if (n <= cap) return;
        if (base) { cudaFree(base); base = nullptr; cap = 0; }
        n += n / 4;
        SDI_CUDA(cudaMalloc(&base, n));
        cap = n;
    }
    template <class T> T *take(size_t count) {
        T *p = reinterpret_cast<T *>(base + used);
        used += (count * sizeof(T) + 255) & ~size_t(255);
        return p;
    }
};
std::mutex g_arena_mu;
Arena g_arena[64];
size_t pad(size_t n) { return (n + 255) & ~size_t(255); }
} // namespace

// Host launcher behind sd_identity.  Buffers are validated by the caller (api.cpp).
int cuda_identity(const IdentityArgs &h, int max_qlen, int max_tlen, int device, double *kernel_ms, std::string &err)
{
    std::lock_guard<std::mutex> lock(g_arena_mu);
    try {
        if (device < 0 || device >= 64) { err = "device id out of range"; return 2; }
        DeviceScope scope(device);                       // the caller's current device is restored on return
        SDI_CUDA(scope.status);
        int major = 0, sms = 0;
        SDI_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
        SDI_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        if (major != 10) { err = "libsd_b200 carries sm_100a code only"; return 2; }
        const bool prof = getenv("SD_PROFILE") != nullptr;
        const auto t_begin = std::chrono::steady_clock::now();
        auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
        const size_t qbytes = (size_t)h.qoff[h.nq], tbytes = (size_t)h.toff[h.nt];
        int L = 0, R = 0;
        if (!nw_choose_geometry(h.qoff, h.nq, L, R)) { err = "unsupported SD_NW_GEOM"; return 4; }
        void (*kernel)(IdentityArgs) = identity_kernel<6, 32>;      // one per NW_GEOMS entry
        if (L == 8 && R == 8) kernel = identity_kernel<8, 8>;
        else if (L == 8 && R == 16) kernel = identity_kernel<16, 8>;
        else if (L == 8 && R == 24) kernel = identity_kernel<24, 8>;
        else if (L == 16 && R == 12) kernel = identity_kernel<12, 16>;
        const int threads = 256, wpb = threads / 32 * (32 / L);                                    // pairs in flight per block
        int resident = 1;                                           // grid-stride kernel: exactly one resident wave of blocks
        SDI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kernel, threads, 0));
        int64_t blocks = std::min<int64_t>((h.npairs + wpb - 1) / wpb, (int64_t)sms * std::max(1, resident));
        if (blocks < 1) blocks = 1;
        const size_t stride = max_qlen > L * R ? (size_t)((max_tlen + 31) & ~31) : 0;
        const size_t np = (size_t)h.npairs;
        Arena &ar = g_arena[device];
        ar.reserve(pad(qbytes) + pad(tbytes) + pad(8 * (h.nq + 1)) + pad(8 * (h.nt + 1)) + 5 * pad(4 * np) +
                   pad(4 * stride * (size_t)(blocks * wpb)) + 4096);
        if (!ar.e0) { SDI_CUDA(cudaEventCreate(&ar.e0)); SDI_CUDA(cudaEventCreate(&ar.e1)); }
        IdentityArgs a = h;
        char *dq = ar.take<char>(qbytes), *dt = ar.take<char>(tbytes);
        int64_t *dqo = ar.take<int64_t>(h.nq + 1), *dto = ar.take<int64_t>(h.nt + 1);
        int32_t *dout = ar.take<int32_t>(3 * np);                      // matches | columns | distance, one copy back
        SDI_CUDA(cudaMemcpyAsync(dq, h.qtext, qbytes, cudaMemcpyHostToDevice));
        SDI_CUDA(cudaMemcpyAsync(dqo, h.qoff, sizeof(int64_t) * (h.nq + 1), cudaMemcpyHostToDevice));
        SDI_CUDA(cudaMemcpyAsync(dt, h.ttext, tbytes, cudaMemcpyHostToDevice));
        SDI_CUDA(cudaMemcpyAsync(dto, h.toff, sizeof(int64_t) * (h.nt + 1), cudaMemcpyHostToDevice));
        a.qtext = dq; a.qoff = dqo; a.ttext = dt; a.toff = dto;
        a.matches = dout; a.columns = dout + np; a.distance = dout + 2 * np;
        if (h.pair_q) {
            int32_t *dpq = ar.take<int32_t>(np), *dpt = ar.take<int32_t>(np);
            SDI_CUDA(cudaMemcpyAsync(dpq, h.pair_q, 4 * np, cudaMemcpyHostToDevice));
            SDI_CUDA(cudaMemcpyAsync(dpt, h.pair_t, 4 * np, cudaMemcpyHostToDevice));
            a.pair_q = dpq; a.pair_t = dpt;
        }
        a.scratch = stride ? ar.take<uint32_t>(stride * (size_t)(blocks * wpb)) : nullptr;
        a.scratch_stride = (int64_t)stride;
        const double t_h2d = since();
        SDI_CUDA(cudaEventRecord(ar.e0));
        kernel<<<(unsigned)blocks, threads>>>(a);
        SDI_CUDA(cudaGetLastError());
        SDI_CUDA(cudaEventRecord(ar.e1));
        SDI_CUDA(cudaMemcpyAsync(h.matches, a.matches, 4 * np, cudaMemcpyDeviceToHost));
        SDI_CUDA(cudaMemcpyAsync(h.columns, a.columns, 4 * np, cudaMemcpyDeviceToHost));
        if (h.distance) SDI_CUDA(cudaMemcpyAsync(h.distance, a.distance, 4 * np, cudaMemcpyDeviceToHost));
        SDI_CUDA(cudaStreamSynchronize(nullptr));
        float ms = 0; SDI_CUDA(cudaEventElapsedTime(&ms, ar.e0, ar.e1));
        if (kernel_ms) *kernel_ms = ms;
        if (prof) fprintf(stderr, "[sd_b200 profile] sd_identity: pairs %ld L %d R %d blocks %ld x %d pairs  h2d issue %.2f ms, kernel %.3f ms, total %.2f ms\n",
                          (long)h.npairs, L, R, (long)blocks, wpb, t_h2d, ms, since());
    } catch (PlanError &e) { err = e.msg; return 4; }
    return 0;
}

} // namespace sdb
