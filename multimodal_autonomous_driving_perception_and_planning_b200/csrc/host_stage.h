// The host/device boundary of the context-free entry points: error reporting, device selection, and host memory in and
// out (staging of ordinary pageable memory for H2D and D2H copies, per-device scratch).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "cuda_owned.h"
#include "lane_common.cuh"

// Host frames in ordinary (pageable) memory: cudaMemcpy from such memory runs at ~11 GB/s on this platform (the
// driver stages it single-threaded).  The library stages them itself instead: a few worker threads copy 32 MB
// pieces into a small ring of pinned buffers while the previous piece is on its way over PCIe.
struct CopyPool {
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv_work, cv_done;
    uint8_t *dst = nullptr;
    const uint8_t *src = nullptr;
    size_t bytes = 0;
    unsigned long generation = 0;
    int pending = 0;
    bool stop = false;

    explicit CopyPool(int n)
    {
        for (int t = 0; t < n; t++)
            th.emplace_back([this, t, n] {
                unsigned long seen = 0;
                for (;;) {
                    std::unique_lock<std::mutex> lk(m);
                    cv_work.wait(lk, [&] { return stop || generation != seen; });
                    if (stop) return;
                    seen = generation;
                    uint8_t *d = dst;
                    const uint8_t *s0 = src;
                    const size_t nb = bytes;
                    lk.unlock();
                    const size_t per = ((nb + n - 1) / n + 4095) & ~(size_t)4095, a = std::min(nb, per * t), b = std::min(nb, a + per);
                    if (b > a) memcpy(d + a, s0 + a, b - a);
                    lk.lock();
                    if (--pending == 0) cv_done.notify_one();
                }
            });
    }
    void run(uint8_t *d, const uint8_t *s0, size_t nb)
    {
        std::unique_lock<std::mutex> lk(m);
        dst = d; src = s0; bytes = nb;
        pending = (int)th.size();
        generation++;
        cv_work.notify_all();
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    ~CopyPool()
    {
        {
            std::lock_guard<std::mutex> lk(m);
            stop = true;
        }
        cv_work.notify_all();
        for (auto &t : th) t.join();
    }
};

// What the driver knows of host address `p`: cudaMemoryTypeHost for page-locked or registered memory,
// cudaMemoryTypeUnregistered for ordinary memory (or an address it cannot query).
inline cudaMemoryType host_memory_type(const void *p)
{
    cudaPointerAttributes pa{};
    const cudaMemoryType t = cudaPointerGetAttributes(&pa, p) == cudaSuccess ? pa.type : cudaMemoryTypeUnregistered;
    cudaGetLastError();
    return t;
}

// One staging ring per device, shared by the contexts and the context-free entry points on it; the worker threads and
// pinned buffers are created by the first staged copy.  h2d() is blocking on the host side only as far as the memcpy
// into pinned memory goes; the DMA itself is asynchronous on `st`.
struct HostStager {
    static constexpr int SLOTS = 3;
    static constexpr size_t PIECE = (size_t)32 << 20;
    CopyPool *pool = nullptr;
    uint8_t *stage[SLOTS] = {};
    cudaEvent_t ev[SLOTS] = {};
    bool used[SLOTS] = {};
    int next = 0;                     // slot of the next h2d() piece: consecutive calls go round the ring
    std::mutex mu;
    bool ok = true;

    bool ready()                      // under mu; false: the ring could not be allocated, copies take the DMA directly
    {
        if (pool) return ok;
        const unsigned hc = std::thread::hardware_concurrency();
        pool = new CopyPool((int)std::max(1u, std::min(8u, hc ? hc / 2 : 4u)));
        for (int i = 0; i < SLOTS; i++)
            ok = ok && cudaHostAlloc((void **)&stage[i], PIECE, cudaHostAllocDefault) == cudaSuccess &&
                 cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) == cudaSuccess;
        cudaGetLastError();
        return ok;
    }
    // Whether a transfer of `bytes` to or from host `p` should go through the ring: ordinary memory, 24 MB or more.
    // Pinned or registered memory goes straight to the copy engine, and small transfers (a single frame) are quicker
    // through the driver's own path than through worker wake-ups.
    static bool pageable(const void *p, size_t bytes)
    {
        return host_memory_type(p) == cudaMemoryTypeUnregistered && bytes >= ((size_t)24 << 20);
    }
    // Through the ring, whatever the size (the caller has decided with pageable()).
    cudaError_t h2d(uint8_t *dst, const uint8_t *src, size_t bytes, cudaStream_t st)
    {
        std::lock_guard<std::mutex> lk(mu);
        if (!ready()) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
        for (size_t done = 0; done < bytes; done += PIECE) {
            const int slot = next;
            next = (next + 1) % SLOTS;
            const size_t nb = std::min(PIECE, bytes - done);
            cudaError_t e;
            if (used[slot] && (e = cudaEventSynchronize(ev[slot]))) return e;    // its last DMA has left
            pool->run(stage[slot], src + done, nb);
            if ((e = cudaMemcpyAsync(dst + done, stage[slot], nb, cudaMemcpyHostToDevice, st))) return e;
            if ((e = cudaEventRecord(ev[slot], st))) return e;
            used[slot] = true;
        }
        return cudaSuccess;
    }
    // The reverse direction, for a pageable destination (the caller has checked pageable()): the DMA on `st` fills a
    // slot, and the pool copies the slot into `dst` once the slot's event has fired, while the DMA of the next pieces
    // is under way.  Pieces are a quarter slot so that even one 32 MB chunk overlaps the two copies.  Blocking: returns
    // when all `bytes` are in `dst`.
    cudaError_t d2h(uint8_t *dst, const uint8_t *src, size_t bytes, cudaStream_t st)
    {
        cudaError_t e;
        std::lock_guard<std::mutex> lk(mu);
        if (!ready()) return (e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st)) ? e : cudaStreamSynchronize(st);
        constexpr size_t D2H_PIECE = PIECE / 4;
        const size_t pieces = (bytes + D2H_PIECE - 1) / D2H_PIECE;
        auto issue = [&](size_t p) {
            const int slot = (int)(p % SLOTS);
            cudaError_t r;
            if (used[slot] && (r = cudaEventSynchronize(ev[slot]))) return r;      // an h2d() may still read it
            const size_t off = p * D2H_PIECE;
            if ((r = cudaMemcpyAsync(stage[slot], src + off, std::min(D2H_PIECE, bytes - off), cudaMemcpyDeviceToHost, st)))
                return r;
            used[slot] = true;
            return cudaEventRecord(ev[slot], st);
        };
        for (size_t p = 0; p < std::min(pieces, (size_t)SLOTS); p++)
            if ((e = issue(p))) return e;
        for (size_t p = 0; p < pieces; p++) {
            const int slot = (int)(p % SLOTS);
            if ((e = cudaEventSynchronize(ev[slot]))) return e;
            const size_t off = p * D2H_PIECE;
            pool->run(dst + off, stage[slot], std::min(D2H_PIECE, bytes - off));
            if (p + SLOTS < pieces && (e = issue(p + SLOTS))) return e;
        }
        return cudaSuccess;
    }
};

// Everything the context-free entry points keep per device, until exit.  `mu` serialises the blocking calls that use
// the scratch buffer or the copy stream; each returns with both idle.
struct LaneDeviceHost {
    std::mutex mu;
    HostStager stager;
    DeviceArray<uint8_t> scratch;     // grow-only: host round trips, frame statistics' sums, egress's conversion slots
    CudaStream copy_st;               // egress to host memory: copies out beside the conversions on the caller's stream
    CudaEvent converted[2], copied[2];
    // Drawing's upload block (primitive lists or lane points), written by the host into write-combined pinned memory and
    // copied to the device in one piece; grow-only.  Its own lock: a draw call holds it across lane_host_round_trip,
    // which takes `mu`.
    std::mutex draw_mu;
    DeviceArray<uint8_t> draw_d;
    PinnedArray<uint8_t> draw_h;

    cudaError_t init_copy_stream()
    {
        if (copy_st) return cudaSuccess;
        cudaError_t e;
        for (int i = 0; i < 2; i++)
            if ((e = converted[i].create(cudaEventDisableTiming)) || (e = copied[i].create(cudaEventDisableTiming))) return e;
        return copy_st.create(cudaStreamNonBlocking);
    }
    // Under draw_mu: `cap` bytes on both sides unless `need` are already there.
    cudaError_t reserve_draw(size_t need, size_t cap)
    {
        if (draw_d.size() >= need) return cudaSuccess;
        draw_h.reset();
        cudaError_t e = draw_d.alloc(cap);
        if (!e) e = draw_h.alloc(cap, cudaHostAllocWriteCombined);
        if (e) {
            draw_d.reset();
            cudaGetLastError();
        }
        return e;
    }
};

// One record per device, created on first use and never destroyed: no CUDA call may run from a static destructor at
// process exit.
inline LaneDeviceHost &lane_device_host(int device)      // device: checked by lane_api_device
{
    static std::mutex mu;
    static LaneDeviceHost *all[LANE_MAX_DEVICES] = {};
    std::lock_guard<std::mutex> lk(mu);
    if (!all[device]) all[device] = new LaneDeviceHost();
    return *all[device];
}

// Reports a context-free call's failure: lane_last_error(NULL) reads "<who>: <what>[: <CUDA error>]".
inline int lane_api_fail(int code, const char *who, const char *what, cudaError_t e = cudaSuccess)
{
    char buf[256];
    snprintf(buf, sizeof buf, "%s: %s%s%s", who, what, e ? ": " : "", e ? cudaGetErrorString(e) : "");
    lane_set_global_error(buf);
    return code;
}

// Selects `device` for a context-free call, after its argument checks.
inline int lane_api_device(const char *who, int device)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return lane_api_fail(LANE_ERR_NO_DEVICE, who, "no CUDA device visible: this library has no CPU fallback");
    if (device < 0 || device >= std::min(ndev, LANE_MAX_DEVICES)) return lane_api_fail(LANE_ERR_INVALID, who, "device out of range");
    const cudaError_t e = cudaSetDevice(device);
    return e ? lane_api_fail(LANE_ERR_CUDA, who, "cudaSetDevice", e) : LANE_OK;
}

// The blocking host round trip of a context-free call, through the device's scratch buffer: `in_bytes` from host `in`
// to d_in, launch(d_in, d_out) on `st`, `out_bytes` from d_out back to host `out`, synchronise.  No upload when `in` is
// null (the generator clears its frames on the device), no download when `out` is null (frame statistics copy their
// few sums themselves), and d_out == d_in when in == out (drawing on host frames).  Pageable buffers of 24 MB or more
// go through the staging ring, all others straight to the DMA.  launch returns LANE_OK or a code it has reported.
template <class Launch>
int lane_host_round_trip(const char *who, int device, cudaStream_t st, const void *in, size_t in_bytes, void *out,
                         size_t out_bytes, Launch &&launch)
{
    LaneDeviceHost &h = lane_device_host(device);
    std::lock_guard<std::mutex> lk(h.mu);
    const size_t in_span = in && in != out ? (in_bytes + 255) & ~(size_t)255 : 0;
    cudaError_t e;
    if ((e = h.scratch.grow(std::max<size_t>(in_span + out_bytes, 1)))) return lane_api_fail(LANE_ERR_CUDA, who, "scratch allocation", e);
    uint8_t *d_in = h.scratch, *d_out = h.scratch + in_span;
    int rc = LANE_OK;
    if (in) {
        e = HostStager::pageable(in, in_bytes) ? h.stager.h2d(d_in, (const uint8_t *)in, in_bytes, st)
                                               : cudaMemcpyAsync(d_in, in, in_bytes, cudaMemcpyHostToDevice, st);
        if (e) rc = lane_api_fail(LANE_ERR_CUDA, who, "H2D", e);
    }
    if (!rc) rc = launch(d_in, d_out);
    if (!rc && out) {
        e = HostStager::pageable(out, out_bytes) ? h.stager.d2h((uint8_t *)out, d_out, out_bytes, st)
                                                 : cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, st);
        if (e) rc = lane_api_fail(LANE_ERR_CUDA, who, "D2H", e);
    }
    if ((e = cudaStreamSynchronize(st)) && !rc) rc = lane_api_fail(LANE_ERR_CUDA, who, "host round trip", e);
    return rc;
}
