// Host <-> device staging for the host-buffer entry points (lb_import_batch, lb_doc_json).
//
// The caller's blobs are ~100k separate pageable allocations; the JSON result is one large pageable buffer.
// Each direction goes through a small process-wide ring of pinned slots: worker threads gather/scatter one slot
// while the copy engine moves the other, so the PCIe transfer overlaps the host memcpy and no batch-sized pinned
// allocation (seconds for several GB) is ever made.
#pragma once
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <functional>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

namespace lbstage {
// Internal linkage: the statics of inline functions below (rings, caches, worker pool) would otherwise be GNU-unique
// symbols, which the dynamic loader shares between every library of the process that defines them -- a second build
// of the engine loaded next to this one (the emulated test build, a tuning variant) would hand this one its pinned
// slots and CUDA events.
namespace {

constexpr size_t SLOT_BYTES = 32u << 20;
constexpr int N_SLOTS = 4;

struct Ring {
    uint8_t* slot[N_SLOTS] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev[N_SLOTS];
    bool ready = false;
    std::mutex mu;
    bool init() {
        if (ready) return true;
        for (int i = 0; i < N_SLOTS; i++) {
            if (cudaMallocHost((void**)&slot[i], SLOT_BYTES) != cudaSuccess) return false;
            if (cudaEventCreate(&ev[i]) != cudaSuccess) return false;
        }
        ready = true;
        return true;
    }
};

// One ring per direction: PCIe is full duplex, and with two imports in flight (api.MultiBatch, or any host that calls
// the C ABI from two threads) the upload of one batch runs while the other's JSON / exported blobs come home.  A
// download of JSON (second stream, its own thread) and one of exported blobs still take turns on the download ring.
inline Ring& ring(int dir) {
    static Ring r[2];
    return r[dir & 1];
}

// LB_STAGE_SLOT (bytes, testing hook) shrinks the slot so that small inputs exercise the multi-slot, multi-thread paths.
inline size_t slot_bytes() {
    static size_t v = [] {
        const char* e = getenv("LB_STAGE_SLOT");
        size_t x = e ? (size_t)strtoull(e, nullptr, 10) : 0;
        return (x >= 64 && x <= SLOT_BYTES) ? x : SLOT_BYTES;
    }();
    return v;
}

inline unsigned n_workers() {
    unsigned hc = std::thread::hardware_concurrency();
    return std::max(1u, std::min(16u, hc ? hc : 1u));
}

// Result buffers (JSON, exported blobs) are GBs of pageable memory: a fresh malloc of that size is page-faulted
// in on first touch every time.  Freed result buffers are kept (a few, size-matched) for the next batch.
struct HostCache {
    struct Hdr { size_t cap; size_t pad; };
    std::mutex mu;
    std::vector<void*> free_;
    void* take(size_t n) {
        {
            std::lock_guard<std::mutex> g(mu);
            int best = -1;
            for (size_t i = 0; i < free_.size(); i++) {
                size_t cap = ((Hdr*)free_[i])->cap;
                if (cap >= n && cap <= 2 * n + (1u << 20) && (best < 0 || cap < ((Hdr*)free_[best])->cap)) best = (int)i;
            }
            if (best >= 0) {
                void* h = free_[best];
                free_[best] = free_.back();
                free_.pop_back();
                return (char*)h + sizeof(Hdr);
            }
        }
        Hdr* h = (Hdr*)malloc(n + sizeof(Hdr));
        if (!h) return nullptr;
        h->cap = n;
        return (char*)h + sizeof(Hdr);
    }
    void give(void* p) {
        if (!p) return;
        Hdr* h = (Hdr*)((char*)p - sizeof(Hdr));
        std::lock_guard<std::mutex> g(mu);
        free_.push_back(h);
        while (free_.size() > 4) {   // drop the smallest
            size_t k = 0;
            for (size_t i = 1; i < free_.size(); i++)
                if (((Hdr*)free_[i])->cap < ((Hdr*)free_[k])->cap) k = i;
            free(free_[k]);
            free_[k] = free_.back();
            free_.pop_back();
        }
    }
};
inline HostCache& host_cache() {
    static HostCache c;
    return c;
}

// The gather / scatter workers are persistent: a 32 MB slot is handed to them every few milliseconds (540 slots per step of
// config C3), and starting 16 threads per slot put ~0.4 ms of thread creation on the critical path of every slot.
// The pool is process-wide and lives as long as the process (detached workers; callers from several threads -- one ring
// per direction, two imports in flight -- share it through one queue).  Workers are created by the first caller, after
// lb_numa_bind if the host called it, so they inherit its CPU affinity.
struct WorkerPool {
    std::mutex mu;
    std::condition_variable cv;
    std::deque<std::function<void()>> q;
    unsigned n = 0;
    void ensure(unsigned want) {
        std::lock_guard<std::mutex> g(mu);
        for (; n < want; n++)
            std::thread([this] {
                for (;;) {
                    std::function<void()> job;
                    {
                        std::unique_lock<std::mutex> lk(mu);
                        cv.wait(lk, [this] { return !q.empty(); });
                        job = std::move(q.front());
                        q.pop_front();
                    }
                    job();
                }
            }).detach();
    }
    void submit(std::function<void()> job) {
        {
            std::lock_guard<std::mutex> g(mu);
            q.push_back(std::move(job));
        }
        cv.notify_one();
    }
};
inline WorkerPool& pool() {
    static WorkerPool* p = new WorkerPool();   // never destroyed: its detached workers may outlive static destructors
    return *p;
}

template <class F>
inline void parallel_ranges(size_t lo, size_t hi, F&& f) {
    unsigned T = n_workers();
    size_t n = hi - lo;
    if (n < std::min<size_t>(1u << 20, slot_bytes() / 2) || T == 1) { f(lo, hi); return; }
    WorkerPool& wp = pool();
    wp.ensure(T);
    size_t per = (n + T - 1) / T;
    struct Done { std::mutex mu; std::condition_variable cv; unsigned left; } done;
    unsigned parts = 0;
    for (unsigned t = 0; t < T; t++)
        if (lo + t * per < hi) parts++;
    done.left = parts;
    for (unsigned t = 1; t < parts; t++) {
        size_t a = lo + t * per, b = std::min(hi, a + per);
        wp.submit([&f, &done, a, b] {
            f(a, b);
            std::lock_guard<std::mutex> g(done.mu);
            if (--done.left == 0) done.cv.notify_one();
        });
    }
    f(lo, std::min(hi, lo + per));            // the caller takes the first part itself
    std::unique_lock<std::mutex> lk(done.mu);
    if (--done.left != 0) done.cv.wait(lk, [&done] { return done.left == 0; });
}

// Copy bytes [lo,hi) of the virtual stream "blob i at offs[i], zero padded up to offs[i+1]" into dst (dst[0] = lo).
struct BlobView { const uint8_t* ptr; size_t len; };
inline void gather(const BlobView* blobs, const uint64_t* offs, size_t n_blobs, size_t lo, size_t hi, uint8_t* dst) {
    size_t i = std::upper_bound(offs, offs + n_blobs + 1, (uint64_t)lo) - offs;
    i = i ? i - 1 : 0;
    size_t pos = lo;
    while (pos < hi && i < n_blobs) {
        size_t b0 = offs[i], bdata = b0 + blobs[i].len, b1 = offs[i + 1];
        if (pos < bdata) {
            size_t e = std::min(hi, bdata);
            std::memcpy(dst + (pos - lo), blobs[i].ptr + (pos - b0), e - pos);
            pos = e;
        }
        if (pos < hi && pos < b1) {
            size_t e = std::min(hi, b1);
            std::memset(dst + (pos - lo), 0, e - pos);
            pos = e;
        }
        i++;
    }
    if (pos < hi) std::memset(dst + (pos - lo), 0, hi - pos);
}

// Host blobs -> one contiguous device buffer.  Returns false on a CUDA error.
inline bool upload_blobs(const BlobView* blobs, const uint64_t* offs, size_t n_blobs, uint8_t* d_dst, cudaStream_t st) {
    Ring& r = ring(0);
    std::lock_guard<std::mutex> g(r.mu);
    if (!r.init()) return false;
    size_t total = offs[n_blobs];
    const size_t SB = slot_bytes();
    int k = 0;
    for (size_t lo = 0; lo < total; lo += SB, k++) {
        size_t hi = std::min(total, lo + SB);
        int s = k % N_SLOTS;
        if (k >= N_SLOTS && cudaEventSynchronize(r.ev[s]) != cudaSuccess) return false;
        uint8_t* buf = r.slot[s];
        parallel_ranges(lo, hi, [&](size_t a, size_t b) { gather(blobs, offs, n_blobs, a, b, buf + (a - lo)); });
        if (cudaMemcpyAsync(d_dst + lo, buf, hi - lo, cudaMemcpyHostToDevice, st) != cudaSuccess) return false;
        if (cudaEventRecord(r.ev[s], st) != cudaSuccess) return false;
    }
    // the slots are reused by the next caller: drain before releasing the ring
    return cudaStreamSynchronize(st) == cudaSuccess;
}

// Device buffer -> pageable host buffer.
inline bool download(const uint8_t* d_src, uint8_t* dst, size_t total, cudaStream_t st) {
    Ring& r = ring(1);
    std::lock_guard<std::mutex> g(r.mu);
    if (!r.init()) return false;
    const size_t SB = slot_bytes();
    size_t n_chunks = (total + SB - 1) / SB;
    auto drain = [&](size_t c) -> bool {
        int s = (int)(c % N_SLOTS);
        if (cudaEventSynchronize(r.ev[s]) != cudaSuccess) return false;
        size_t lo = c * SB, hi = std::min(total, lo + SB);
        const uint8_t* buf = r.slot[s];
        parallel_ranges(lo, hi, [&](size_t a, size_t b) { std::memcpy(dst + a, buf + (a - lo), b - a); });
        return true;
    };
    for (size_t c = 0; c < n_chunks; c++) {
        if (c >= (size_t)N_SLOTS && !drain(c - N_SLOTS)) return false;
        int s = (int)(c % N_SLOTS);
        size_t lo = c * SB, hi = std::min(total, lo + SB);
        if (cudaMemcpyAsync(r.slot[s], d_src + lo, hi - lo, cudaMemcpyDeviceToHost, st) != cudaSuccess) return false;
        if (cudaEventRecord(r.ev[s], st) != cudaSuccess) return false;
    }
    for (size_t c = n_chunks > (size_t)N_SLOTS ? n_chunks - N_SLOTS : 0; c < n_chunks; c++)
        if (!drain(c)) return false;
    return true;
}

}  // namespace
}  // namespace lbstage
