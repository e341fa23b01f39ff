// common.cuh -- handle, stream-ordered temporaries, host/device pointer staging.
#pragma once
#include <cuda_runtime.h>

#include <chrono>
#include <climits>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/mfgp.h"

#define MFGP_ERR_ARG (-1)
#define MFGP_ERR_CUDA (-2)
#define MFGP_ERR_UNSUPPORTED (-3)

// Where a call's temporaries come from (mfgp_workspace in include/mfgp.h).  POOL: stream-ordered allocations from the device's
// default memory pool.  MEASURE: the same, and the bytes of every call are summed (need = the largest call).  FIXED: bump
// allocation from ONE arena that was allocated outside any stream capture; every call that opens at the depth where the
// mode was entered starts again at offset 0 (its predecessor's temporaries are dead in stream order).  Captured into a
// CUDA graph, a FIXED call contains no allocation nodes: the graph owns no memory that would outlive it.
struct mfgp_ws_state {
    int mode = MFGP_WS_POOL;
    int depth = 0;       // live Scopes on this handle
    int base_depth = 0;  // depth at which the mode was entered
    size_t cur = 0, need = 0;
    char* arena = nullptr;
    size_t cap = 0, off = 0;
    size_t spilled = 0;  // FIXED: bytes that did not fit and were served by the pool
};
inline thread_local mfgp_ws_state* mfgp_tl_ws = nullptr;  // workspace of the innermost live Scope of this thread

// MFGP_WS_DEBUG=1: every outermost call reports its wall time, the time spent inside the allocator and allocations slower
// than 0.5 ms on stderr (how the pool-growth and host-noise outliers in the wall-clock bench legs were told apart).
inline bool mfgp_ws_debug() { static const bool on = getenv("MFGP_WS_DEBUG") != nullptr; return on; }
inline double& mfgp_dbg_malloc_ms() { static thread_local double ms = 0; return ms; }
inline cudaError_t mfgp_ws_malloc_impl(void** p, size_t bytes, cudaStream_t s);
inline cudaError_t mfgp_ws_malloc(void** p, size_t bytes, cudaStream_t s) {
    if (!mfgp_ws_debug()) return mfgp_ws_malloc_impl(p, bytes, s);
    const auto t0 = std::chrono::steady_clock::now();
    const cudaError_t e = mfgp_ws_malloc_impl(p, bytes, s);
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    mfgp_dbg_malloc_ms() += ms;
    if (ms > 0.5) fprintf(stderr, "[mfgp ws] malloc %zu bytes took %.2f ms\n", bytes, ms);
    return e;
}
inline cudaError_t mfgp_ws_malloc_impl(void** p, size_t bytes, cudaStream_t s) {
    mfgp_ws_state* w = mfgp_tl_ws;
    const size_t a = (bytes + 255) & ~(size_t)255;
    if (w && w->mode == MFGP_WS_FIXED) {
        if (w->off + a <= w->cap) {
            *p = w->arena + w->off;
            w->off += a;
            return cudaSuccess;
        }
        w->spilled += a;
    } else if (w && w->mode == MFGP_WS_MEASURE) {
        w->cur += a;
        if (w->cur > w->need) w->need = w->cur;
    }
    return cudaMallocAsync(p, bytes, s);
}
inline cudaError_t mfgp_ws_free(void* p, cudaStream_t s) {
    const mfgp_ws_state* w = mfgp_tl_ws;
    if (w && w->arena && static_cast<char*>(p) >= w->arena && static_cast<char*>(p) < w->arena + w->cap) return cudaSuccess;
    return cudaFreeAsync(p, s);
}

struct mfgp_handle {
    mfgp_ws_state ws;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaStream_t aux_stream = nullptr;  // look-ahead stream for the panel chain; H2D stream of the pipelined batched call
    cudaStream_t copy_stream = nullptr; // D2H stream of the pipelined batched call
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int async = 0;
    int sm_count = 148;
    int* d_info = nullptr;   // device: first failing pivot (1-based), 0 = ok
    int* h_info = nullptr;   // pinned mirror
    char err[512] = {0};
};

inline int mfgp_fail(mfgp_handle* h, int code, const char* fmt, ...) {
    if (h) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(h->err, sizeof(h->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

#define CUDA_TRY(h, expr)                                                                        \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return mfgp_fail((h), MFGP_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,    \
                             cudaGetErrorString(_e));                                            \
    } while (0)

#define MFGP_TRY(expr)            \
    do {                          \
        int _rc = (expr);         \
        if (_rc != 0) return _rc; \
    } while (0)

// ---- per-device launch state -------------------------------------------------------------------
// Function attributes and device properties belong to a DEVICE, and one process may hold one handle per GPU
// (include/mfgp.h threading contract): every cache below is a per-device table behind a mutex.
constexpr int MFGP_MAX_DEVICES = 64;

struct mfgp_dev_info {
    int sms = 0;         // multiprocessors
    int smem_optin = 0;  // cudaDevAttrMaxSharedMemoryPerBlockOptin
};
inline mfgp_dev_info mfgp_current_dev_info() {
    static std::mutex mu;
    static mfgp_dev_info tab[MFGP_MAX_DEVICES];
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    mfgp_dev_info local;
    mfgp_dev_info& e = (dev >= 0 && dev < MFGP_MAX_DEVICES) ? tab[dev] : local;
    if (!e.sms) {
        cudaDeviceGetAttribute(&e.sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&e.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    return e;
}
// Raises cudaFuncAttributeMaxDynamicSharedMemorySize of one kernel to >= bytes on the CURRENT device, once per device.
struct SmemOptIn {
    std::mutex mu;
    int have[MFGP_MAX_DEVICES] = {};
    template <typename Kernel>
    bool ensure(Kernel func, size_t bytes) {
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lock(mu);
        const bool cached = dev >= 0 && dev < MFGP_MAX_DEVICES;
        if (cached && (int)bytes <= have[dev]) return true;
        if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return false;
        if (cached) have[dev] = (int)bytes;
        return true;
    }
};

inline bool mfgp_is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// Per-call scope: stream-ordered temporaries (cudaMallocAsync pool) + staged host I/O.
struct Scope {
    mfgp_handle* h;
    std::vector<void*> temps;
    struct Pending {
        void* host;
        const void* dev;
        size_t bytes;
    };
    std::vector<Pending> outs;
    bool ok = true;
    bool host_out = false;
    mfgp_ws_state* prev_ws;
    std::chrono::steady_clock::time_point t_open = std::chrono::steady_clock::now();
    explicit Scope(mfgp_handle* hh) : h(hh), prev_ws(mfgp_tl_ws) {
        mfgp_ws_state& w = h->ws;
        if (w.depth == w.base_depth) w.off = w.cur = 0;  // a new call at the level the workspace mode was entered
        ++w.depth;
        mfgp_tl_ws = &w;
    }
    ~Scope() {
        if (mfgp_ws_debug() && h->ws.depth == 1) {
            const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_open).count();
            fprintf(stderr, "[mfgp ws] call: %.2f ms wall, %.2f ms in malloc, %zu temporaries\n", ms, mfgp_dbg_malloc_ms(), temps.size());
            mfgp_dbg_malloc_ms() = 0;
        }
        for (void* p : temps) mfgp_ws_free(p, h->stream);
        --h->ws.depth;
        mfgp_tl_ws = prev_ws;
    }
    Scope(const Scope&) = delete;
    Scope& operator=(const Scope&) = delete;
    template <typename T>
    T* alloc(size_t count, bool zero = false) {
        void* p = nullptr;
        size_t bytes = (count ? count : 1) * sizeof(T);
        if (mfgp_ws_malloc(&p, bytes, h->stream) != cudaSuccess) {
            snprintf(h->err, sizeof(h->err), "cudaMallocAsync(%zu bytes) failed: %s", bytes,
                     cudaGetErrorString(cudaGetLastError()));
            ok = false;
            return nullptr;
        }
        temps.push_back(p);
        if (zero) cudaMemsetAsync(p, 0, bytes, h->stream);
        return static_cast<T*>(p);
    }
    // input: returns a device pointer holding `count` elements of `p` (copy if p is host)
    template <typename T>
    const T* in(const T* p, size_t count) {
        if (!p) return nullptr;
        if (mfgp_is_device_ptr(p)) return p;
        T* d = alloc<T>(count);
        if (!d) return nullptr;
        if (cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) ok = false;
        return d;
    }
    // output: returns a device pointer; if p is host the copy-back is queued for finish()
    template <typename T>
    T* out(T* p, size_t count, bool zero = false) {
        if (!p) return nullptr;
        if (mfgp_is_device_ptr(p)) {
            if (zero) cudaMemsetAsync(p, 0, count * sizeof(T), h->stream);
            return p;
        }
        T* d = alloc<T>(count, zero);
        if (!d) return nullptr;
        outs.push_back({p, d, count * sizeof(T)});
        host_out = true;
        return d;
    }
    // in/out buffer: staged to the device now and copied back by finish() when p is host memory
    template <typename T>
    T* inout(T* p, size_t count) {
        if (!p) return nullptr;
        if (mfgp_is_device_ptr(p)) return p;
        T* d = alloc<T>(count);
        if (!d) return nullptr;
        if (cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) ok = false;
        outs.push_back({p, d, count * sizeof(T)});
        host_out = true;
        return d;
    }
    // copy results back, synchronise unless (async && no host outputs), collect info
    int finish() {
        if (!ok) {
            if (!h->err[0]) snprintf(h->err, sizeof(h->err), "allocation / staging failed");
            return MFGP_ERR_CUDA;  // h->err already holds the message of the failing allocation / copy
        }
        for (auto& o : outs) CUDA_TRY(h, cudaMemcpyAsync(o.host, o.dev, o.bytes, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaGetLastError());
        if (h->async && !host_out) return 0;
        CUDA_TRY(h, cudaMemcpyAsync(h->h_info, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        int info = *h->h_info;
        if (info != 0) {
            CUDA_TRY(h, cudaMemsetAsync(h->d_info, 0, sizeof(int), h->stream));
            snprintf(h->err, sizeof(h->err), "Cholesky decomposition was not successful (pivot %d not positive)", info);
        }
        return info;
    }
};

__host__ __device__ inline long round_up(long x, long m) { return (x + m - 1) / m * m; }

// Items per chunk of a chunked call: as many as take at most half of the free device memory at per_item bytes each,
// clamped to [lo, hi].
inline long chunk_by_free_memory(size_t per_item, long lo, long hi) {
    size_t freeb = 0, totb = 0;
    cudaMemGetInfo(&freeb, &totb);
    long chunk = (long)((freeb / 2) / per_item);
    if (chunk < lo) chunk = lo;
    if (chunk > hi) chunk = hi;
    return chunk;
}
