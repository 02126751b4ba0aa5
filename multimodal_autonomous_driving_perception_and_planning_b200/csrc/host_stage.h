// Host-side staging of ordinary (pageable) memory for H2D and D2H copies.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

// Host frames in ordinary (pageable) memory: cudaMemcpy from such memory runs at ~11 GB/s on this platform (the
// driver stages it single-threaded).  The context stages them itself instead: a few worker threads copy 32 MB
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


// Context-free entry points (resize, frame statistics, egress) share one staging ring per device.  h2d() is blocking on the
// host side only as far as the memcpy into pinned memory goes; the DMA itself is asynchronous on `st`.
struct HostStager {
    static constexpr int SLOTS = 3;
    static constexpr size_t PIECE = (size_t)32 << 20;
    CopyPool pool;
    uint8_t *stage[SLOTS] = {};
    cudaEvent_t ev[SLOTS] = {};
    bool used[SLOTS] = {};
    std::mutex mu;
    bool ok = true;

    HostStager() : pool((int)std::max(1u, std::min(8u, std::thread::hardware_concurrency() ? std::thread::hardware_concurrency() / 2 : 4u)))
    {
        for (int i = 0; i < SLOTS; i++)
            ok = ok && cudaHostAlloc((void **)&stage[i], PIECE, cudaHostAllocDefault) == cudaSuccess &&
                 cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) == cudaSuccess;
    }
    static bool pageable(const void *p, size_t bytes)
    {
        cudaPointerAttributes pa{};
        const bool un = cudaPointerGetAttributes(&pa, p) != cudaSuccess || pa.type == cudaMemoryTypeUnregistered;
        cudaGetLastError();
        return un && bytes >= ((size_t)24 << 20);
    }
    cudaError_t h2d(uint8_t *dst, const uint8_t *src, size_t bytes, cudaStream_t st)
    {
        if (!ok || !pageable(src, bytes)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
        std::lock_guard<std::mutex> lk(mu);
        int piece = 0;
        for (size_t done = 0; done < bytes; done += PIECE, piece++) {
            const int slot = piece % SLOTS;
            const size_t nb = std::min(PIECE, bytes - done);
            cudaError_t e;
            if (used[slot] && (e = cudaEventSynchronize(ev[slot]))) return e;
            pool.run(stage[slot], src + done, nb);
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
        if (!ok) return (e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st)) ? e : cudaStreamSynchronize(st);
        constexpr size_t D2H_PIECE = PIECE / 4;
        std::lock_guard<std::mutex> lk(mu);
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
            pool.run(dst + off, stage[slot], std::min(D2H_PIECE, bytes - off));
            if (p + SLOTS < pieces && (e = issue(p + SLOTS))) return e;
        }
        return cudaSuccess;
    }
};

inline HostStager *lane_host_stager(int device)      // one per device, created on first use, lives until exit
{
    static std::mutex mu;
    static HostStager *all[64] = {};
    if (device < 0 || device >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    if (!all[device]) all[device] = new HostStager();
    return all[device];
}
