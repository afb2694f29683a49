// runtime.hpp -- host helpers shared by the phi engine (engine.cu) and gen.gc/occ/rec (gc_engine.cu): error
// reporting, the device arena cache, the staged device-to-host copy and the per-device fan-out.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdint>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/genlib_cuda.h"

#pragma GCC visibility push(hidden)          // internal to the library: nothing here is exported
namespace genlib {

extern thread_local std::string g_err;       // genlib_last_error

inline int fail(int code, const std::string &msg) { g_err = msg; return code; }

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(e_ == cudaErrorMemoryAllocation ? GENLIB_ENOMEM : GENLIB_ECUDA,       \
                        std::string(#call) + ": " + cudaGetErrorString(e_));                  \
    } while (0)

inline double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

struct DeviceGuard {
    int prev = -1;
    bool active = false;
    int enter(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) return fail(GENLIB_ECUDA, "no usable CUDA device (cudaGetDevice failed)");
        if (dev >= 0 && dev != prev) {
            if (cudaSetDevice(dev) != cudaSuccess) return fail(GENLIB_ECUDA, "cudaSetDevice failed");
            active = true;
        }
        return GENLIB_OK;
    }
    ~DeviceGuard() { if (active) cudaSetDevice(prev); }
};

inline size_t pad256(size_t b) { return (std::max<size_t>(b, 1) + 255) / 256 * 256; }

// ---- device arena: ONE allocation per engine, cached across calls -------------------------
// cudaMalloc / cudaFree of tens of GB cost hundreds of milliseconds; a repeated gen.phi call
// (and the one-shot genlib_phi) reuses the previous arena when it is large enough.
struct Arena {
    void *base = nullptr;
    size_t size = 0;
    int device = -1;
    bool exported = false;      // a CUDA-IPC handle of it was handed out: peer processes may keep it mapped
};

class ArenaCache {
    std::mutex mu_;
    std::vector<Arena> free_;
public:
    cudaError_t acquire(int device, size_t bytes, Arena &out) {
        {
            std::lock_guard<std::mutex> g(mu_);
            int best = -1;
            for (int i = 0; i < (int)free_.size(); i++)
                if (free_[i].device == device && free_[i].size >= bytes && (best < 0 || free_[i].size < free_[best].size)) best = i;
            if (best >= 0) { out = free_[best]; free_.erase(free_.begin() + best); return cudaSuccess; }
        }
        // Nothing cached fits.  The smaller cached arenas of this device are given back first (a long-lived
        // process would otherwise pin one arena per size it ever needed) -- except those a peer process may
        // still have mapped (CUDA IPC: freeing exported memory under an open mapping is undefined); these go
        // only when the device is out of memory.
        release_device(device, /*also_exported=*/false);
        out = Arena{nullptr, bytes, device, false};
        cudaError_t ce = cudaMalloc(&out.base, bytes);
        if (ce == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            release_device(device, true);
            ce = cudaMalloc(&out.base, bytes);
        }
        return ce;
    }
    void release(Arena a) {
        if (!a.base) return;
        std::lock_guard<std::mutex> g(mu_);
        free_.push_back(a);
    }
    void release_device(int device, bool also_exported = true) {
        std::lock_guard<std::mutex> g(mu_);
        for (size_t i = 0; i < free_.size();) {
            if ((device < 0 || free_[i].device == device) && (also_exported || !free_[i].exported)) {
                int prev = -1; cudaGetDevice(&prev);
                cudaSetDevice(free_[i].device); cudaFree(free_[i].base);
                if (prev >= 0) cudaSetDevice(prev);
                free_.erase(free_.begin() + (long)i);
            } else i++;
        }
    }
};
extern ArenaCache g_arenas;

// An arena of `bytes` on `device` from the cache.  Out of device memory fails with GENLIB_ENOMEM and the message
// describe(free bytes on the device).
template <class Describe>
int acquire_arena(int device, size_t bytes, Arena &out, Describe &&describe) {
    if (g_arenas.acquire(device, bytes, out) == cudaSuccess) return GENLIB_OK;
    out = Arena();
    cudaGetLastError();
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    return fail(GENLIB_ENOMEM, describe(free_b));
}

// non-owning typed view into the arena
template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    static size_t padded(size_t count) { return (std::max<size_t>(count, 1) * sizeof(T) + 255) / 256 * 256; }
    void place(unsigned char *&cursor, size_t count) { p = reinterpret_cast<T *>(cursor); n = count; cursor += padded(count); }
    cudaError_t upload(const std::vector<T> &h, cudaStream_t s) {
        if (h.empty()) return cudaSuccess;
        return cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s);
    }
};

constexpr size_t kFetchStageBytes = (size_t)64 << 20;

// `items` items to host memory in blocks of `per`, through two device staging buffers: gather(stage, i0, n) enqueues
// the gather of items [i0, i0 + n) into `stage` on stream `st`, copy(stage, i0, n) enqueues their copy to the host on
// `cst` and returns its status.  The gather of block b+1 overlaps the copy of block b; block b+2 waits for it.
// A failure is GENLIB_ECUDA "<what> failed: <CUDA error>".
template <typename O, class Gather, class Copy>
int staged_d2h(cudaStream_t st, cudaStream_t cst, O *stage0, O *stage1, int64_t items, int64_t per, const char *what,
               Gather &&gather, Copy &&copy) {
    O *stage[2] = {stage0, stage1};
    cudaEvent_t done[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    cudaError_t ce = cudaSuccess;
    for (int b = 0; b < 2 && ce == cudaSuccess; b++) {
        ce = cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming);
    }
    int blk = 0;
    for (int64_t i0 = 0; i0 < items && ce == cudaSuccess; i0 += per, blk++) {
        const int b = blk & 1;
        const int64_t nb = std::min(per, items - i0);
        if (blk >= 2 && (ce = cudaStreamWaitEvent(st, copied[b], 0)) != cudaSuccess) break;
        gather(stage[b], i0, nb);
        if ((ce = cudaGetLastError()) != cudaSuccess) break;
        cudaEventRecord(done[b], st);
        cudaStreamWaitEvent(cst, done[b], 0);
        ce = copy(stage[b], i0, nb);
        cudaEventRecord(copied[b], cst);
    }
    const cudaError_t e1 = cudaStreamSynchronize(st), e2 = cudaStreamSynchronize(cst);
    for (int b = 0; b < 2; b++) { if (done[b]) cudaEventDestroy(done[b]); if (copied[b]) cudaEventDestroy(copied[b]); }
    if (ce != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess)
        return fail(GENLIB_ECUDA, std::string(what) + " failed: " + cudaGetErrorString(ce != cudaSuccess ? ce : e1 != cudaSuccess ? e1 : e2));
    return GENLIB_OK;
}

// Checks a device list given by the caller: every entry a device of this host, none listed twice.  With
// `negative_is_current` a negative entry names the current device and is replaced by its number.
inline int resolve_devices(const std::string &who, int32_t n_dev, const int32_t *devices, bool negative_is_current,
                           std::vector<int> &out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(GENLIB_ECUDA, "no CUDA device: libgenlib_cuda has no CPU fallback");
    out.assign(devices, devices + n_dev);
    for (int g = 0; g < n_dev; g++) {
        int &d = out[(size_t)g];
        if (d < 0 && negative_is_current && cudaGetDevice(&d) != cudaSuccess) return fail(GENLIB_ECUDA, "no usable CUDA device (cudaGetDevice failed)");
        if (d < 0 || d >= ndev) return fail(GENLIB_EINVAL, who + ": no such device");
        for (int h = 0; h < g; h++) if (out[(size_t)h] == d) return fail(GENLIB_EINVAL, who + ": a device is listed twice");
    }
    return GENLIB_OK;
}

// What fn(g) returned for device g of a fan-out, and the message of a failure.
struct DeviceStatus {
    int status = GENLIB_OK;
    std::string message;
};

// fn(g) for g in [0, n): on the calling thread for one device, otherwise on one host thread per device.
template <class Fn>
std::vector<DeviceStatus> on_devices(int n, Fn &&fn) {
    std::vector<DeviceStatus> r((size_t)n);
    auto one = [&](int g) {
        DeviceStatus &s = r[(size_t)g];
        s.status = fn(g);
        if (s.status != GENLIB_OK) s.message = g_err;
    };
    if (n == 1) one(0);
    else {
        std::vector<std::thread> th;
        for (int g = 0; g < n; g++) th.emplace_back(one, g);
        for (auto &t : th) t.join();
    }
    return r;
}

}  // namespace genlib
#pragma GCC visibility pop
