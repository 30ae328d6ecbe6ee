// C ABI (include/snarkvm_b200.h): the three drop-in symbols of the reference FFI
// (/root/reference/algorithms/cuda/src/lib.rs:42-69) plus the device-resident extended API.
// Error contract (SURVEY §5, §8b): never throw or abort across the boundary; return a
// cudaError_t code; leave outputs untouched on failure so the Rust caller can fall back.
#include "../../include/snarkvm_b200.h"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include <cuda_runtime.h>
#include <pthread.h>
#include <sched.h>
#include <cstdio>

#include "host_ec.hpp"
#include "msm.cuh"
#include "ntt.cuh"
#include "poly.cuh"

namespace b200 { void host_stream_copy(void* dst, const void* src, size_t n); }      // hostcopy.cpp: memcpy with non-temporal stores
using namespace b200;

namespace {

snarkvm_error_t make_error(int code) {
    snarkvm_error_t e;
    e.code = code;
    e.message = nullptr;
    if (code != 0) {
        const char* s = cudaGetErrorString((cudaError_t)code);
        if (s) { size_t n = strlen(s) + 1; e.message = (char*)malloc(n); if (e.message) memcpy(e.message, s, n); }
    }
    return e;
}

// One non-blocking stream per (host thread, device): the FFI is entered concurrently from many
// rayon workers (sonic_pc/mod.rs:186-245), so calls must not serialise on the default stream.
struct ThreadCtx {
    cudaStream_t stream[64] = {};
    bool have[64] = {};
    cudaStream_t copy_stream[64] = {};
    bool have_copy[64] = {};
    ~ThreadCtx() {}
};
thread_local ThreadCtx t_ctx;

int thread_stream(cudaStream_t* out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    dev &= 63;
    if (!t_ctx.have[dev]) {
        e = cudaStreamCreateWithFlags(&t_ctx.stream[dev], cudaStreamNonBlocking);
        if (e != cudaSuccess) return (int)e;
        t_ctx.have[dev] = true;
    }
    *out = t_ctx.stream[dev];
    return 0;
}

// second stream of the calling thread: uploads that overlap the kernels of the first
int thread_copy_stream(cudaStream_t* out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    dev &= 63;
    if (!t_ctx.have_copy[dev]) {
        e = cudaStreamCreateWithFlags(&t_ctx.copy_stream[dev], cudaStreamNonBlocking);
        if (e != cudaSuccess) return (int)e;
        t_ctx.have_copy[dev] = true;
    }
    *out = t_ctx.copy_stream[dev];
    return 0;
}

// Registered (resident) bases: the SRS powers of a proving key are constant, and the reference re-passes the same
// host slice on every commitment (kzg10/mod.rs:119,149).  A caller may register that slice once; snarkvm_msm then
// recognises the pointer and skips the 104 B/point upload.  Opt-in: the caller promises not to mutate the slice.
// Entries are shared_ptr-owned: a call that found an entry keeps it (device copy, tables) alive until it returns, so a
// concurrent unregister / re-register only drops the map's reference and the memory goes when the last call ends.
struct PrecomputedBases { uint32_t* table; size_t n; MsmPlan plan; int device; };
struct ResidentBases {
    void* d_ptr = nullptr;
    size_t npoints = 0, stride = 0;
    int device = 0;
    std::atomic<PrecomputedBases*> tables{nullptr};
    uint8_t head[104] = {}, tail[104] = {};       // first and last point of the host slice at registration (stale-address check)
    ~ResidentBases() {
        int cur = 0;
        cudaGetDevice(&cur);
        if (cur != device) cudaSetDevice(device);
        if (d_ptr) cudaFree(d_ptr);
        if (PrecomputedBases* t = tables.load()) { cudaFree(t->table); delete t; }
        if (cur != device) cudaSetDevice(cur);
    }
};
std::mutex g_bases_mu;
std::map<const void*, std::shared_ptr<ResidentBases>> g_bases;

std::shared_ptr<ResidentBases> find_resident(const void* host, size_t npoints, size_t stride) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    std::shared_ptr<ResidentBases> r;
    {
        std::lock_guard<std::mutex> lock(g_bases_mu);
        auto it = g_bases.find(host);
        if (it == g_bases.end()) return nullptr;
        r = it->second;
    }
    if (r->device != dev || r->stride != stride || r->npoints < npoints) return nullptr;
    // a freed and re-used host buffer at the same address would silently compute with stale bases: compare the end points
    if (memcmp(r->head, host, 104) != 0) return nullptr;
    if (memcmp(r->tail, (const uint8_t*)host + (r->npoints - 1) * stride, 104) != 0) return nullptr;
    return r;
}

void write_infinity(void* out144) {
    host::Xyzz inf = host::xyzz_inf();
    host::xyzz_to_normalised_projective(inf, (uint64_t*)out144);
}

// Runs `njobs` sums through ONE msm_core pass and finishes them on the host: one D2H of njobs·sets XYZZ points plus the
// overflow flag, ONE stream synchronisation, then the Horner fold per job (253 doublings on 64-bit host limbs ≈ 0.1 ms,
// exactly where the reference's own plugin finishes, snarkvm.cu:290-295).  out144s: njobs × 144 B of HOST memory.
int msm_jobs_impl(void* out144s, const MsmPlan& plan, const MsmBases* bases, int nbases, const uint32_t* table, size_t table_n,
                  const MsmSegment* segs, int nsegs, int njobs, cudaStream_t stream) {
    const size_t sets = table ? 1 : (size_t)plan.nwin;
    const size_t npts = (size_t)njobs * sets;
    uint32_t* d_buf = nullptr;
    cudaError_t e = pool_alloc(&d_buf, npts * 192 + 256, stream);
    if (e != cudaSuccess) return (int)e;
    uint32_t* d_flags = d_buf + npts * 48;
    int rc = (int)cudaMemsetAsync(d_flags, 0, 256, stream);
    if (rc == 0) rc = msm_core(d_buf, d_flags, plan, bases, nbases, table, table_n, segs, nsegs, njobs, stream);
    // the window sums come back through a small pinned buffer of the calling thread when they fit (a pageable destination makes
    // the driver stage the copy: ≈ 15 µs of a 0.5 ms small MSM)
    static thread_local void* t_result_pinned = nullptr;
    constexpr size_t RESULT_PINNED_BYTES = (size_t)64 << 10;
    const size_t result_bytes = npts * 192 + 256;
    if (!t_result_pinned && result_bytes <= RESULT_PINNED_BYTES && cudaHostAlloc(&t_result_pinned, RESULT_PINNED_BYTES, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError(); t_result_pinned = nullptr;
    }
    std::vector<host::Xyzz> sums(npts + 2);
    void* land = (t_result_pinned && result_bytes <= RESULT_PINNED_BYTES) ? t_result_pinned : (void*)sums.data();
    if (rc == 0) rc = (int)cudaMemcpyAsync(land, d_buf, result_bytes, cudaMemcpyDeviceToHost, stream);
    cudaFreeAsync(d_buf, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc != 0) return rc;
    if (land != (void*)sums.data()) memcpy(sums.data(), land, result_bytes);
    uint32_t flags = 0;
    memcpy(&flags, sums.data() + npts, 4);
    if (flags & 1u) return (int)cudaErrorInvalidValue;           // a scalar ≥ 2^253: not a canonical Fr, let the caller fall back
    auto finish = [&](int j) {
        host::Xyzz total = table ? sums[(size_t)j] : host::horner_windows(sums.data() + (size_t)j * sets, plan.nwin, plan.c);
        host::xyzz_to_normalised_projective(total, (uint64_t*)((uint8_t*)out144s + (size_t)j * 144));
    };
    if (njobs <= 2) { for (int j = 0; j < njobs; j++) finish(j); }
    else {
        const int nt = njobs < 8 ? njobs : 8;
        std::vector<std::thread> th;
        std::atomic<int> next{0};
        for (int t = 0; t < nt; t++) th.emplace_back([&] { for (int j; (j = next.fetch_add(1)) < njobs;) finish(j); });
        for (auto& t : th) t.join();
    }
    return 0;
}

int msm_device_impl(void* out144, const void* d_points, size_t npoints, const void* d_scalars, size_t stride, int mont,
                    cudaStream_t stream) {
    if (npoints == 0) { write_infinity(out144); return 0; }
    if (stride < 104 || (stride & 7)) return (int)cudaErrorInvalidValue;
    MsmPlan plan = msm_make_plan(npoints);
    MsmBases b{d_points, stride, npoints};
    MsmSegment sg{d_scalars, npoints, 0u, 0u, mont};
    return msm_jobs_impl(out144, plan, &b, 1, nullptr, 0, &sg, 1, 1, stream);
}

// ----------------------------------------------------------------------------------------
// Host → device uploads.  A Rust Vec is PAGEABLE memory: cudaMemcpyAsync from it goes through the driver's own
// staging at a fraction of the link rate and blocks the calling thread.  Pageable sources therefore go through a ring
// of pinned buffers owned by the calling thread, filled by a small pool of copy threads (several cores are needed to
// feed PCIe Gen5) and drained by async DMA on the thread's copy stream; pinned sources (cudaHostAlloc / registered)
// are copied directly.
// ----------------------------------------------------------------------------------------
// CPUs on the NUMA node of the current device (sysfs `local_cpulist` of its PCI function) ∩ the CPUs this process may use.
// With one process per GPU on a two-socket host, copy threads that wander between the sockets push every staged byte over the
// inter-socket links twice: 4 ranks staged 51 GB/s in total (177 ms per 2^24-point step against 113 ms alone, r2ad_bench_n4).
// The pool's threads and the pinned staging ring are therefore kept on the device's node (SNARKVM_B200_COPY_NUMA=0 disables).
static bool device_local_cpus(cpu_set_t* out) {
    // default: only under a one-process-per-GPU launch (torchrun exports LOCAL_WORLD_SIZE) — a single process that drives several
    // GPUs shares one pool, and tying it to the first device's node would hurt the others; SNARKVM_B200_COPY_NUMA=1 / 0 forces it
    if (const char* e = getenv("SNARKVM_B200_COPY_NUMA")) { if (atoi(e) == 0) return false; }
    else { const char* lws = getenv("LOCAL_WORLD_SIZE"); if (!lws || atoi(lws) <= 1) return false; }
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return false; }
    char bus[64] = {};
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus - 1, dev) != cudaSuccess) { cudaGetLastError(); return false; }
    for (char* c = bus; *c; c++) if (*c >= 'A' && *c <= 'Z') *c = (char)(*c - 'A' + 'a');
    char path[160];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/local_cpulist", bus);
    FILE* f = fopen(path, "r");
    if (!f) return false;
    char line[4096] = {};
    const bool got = fgets(line, sizeof line, f) != nullptr;
    fclose(f);
    if (!got) return false;
    cpu_set_t allowed, local;
    CPU_ZERO(&local);
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return false;
    for (const char* p = line; *p;) {                              // "0-31,64-95"
        while (*p == ',' || *p == ' ') p++;
        if (*p < '0' || *p > '9') break;
        char* end = nullptr;
        long a = strtol(p, &end, 10), b = a;
        if (*end == '-') b = strtol(end + 1, &end, 10);
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) if (CPU_ISSET((int)c, &allowed)) CPU_SET((int)c, &local);
        p = end;
    }
    if (CPU_COUNT(&local) < 2 || CPU_COUNT(&local) == CPU_COUNT(&allowed)) return false;     // nothing to gain (single node / cpuset)
    *out = local;
    return true;
}

class CopyPool {
public:
    // the device-local CPU set the pool was bound to, if any
    bool numa_cpus(cpu_set_t* out) const { if (have_numa_) *out = numa_; return have_numa_; }
    static CopyPool& get() { static CopyPool* p = new CopyPool(); return *p; }      // leaked on purpose: threads outlive static destructors
    // memcpy(dst, src, bytes) split over the pool and the caller; returns when all of it is done
    void parallel_memcpy(void* dst, const void* src, size_t bytes) {
        const size_t piece = (size_t)2 << 20;
        if (bytes <= piece || nthreads_ == 0) { host_stream_copy(dst, src, bytes); return; }
        Batch batch;
        batch.dst = (uint8_t*)dst; batch.src = (const uint8_t*)src; batch.bytes = bytes; batch.piece = piece;
        batch.npieces = (bytes + piece - 1) / piece;
        run(batch);
    }
    // `rows` rows of `width` bytes, row r at dst + r·dpitch ← src + r·spitch (a column range of a row-major matrix)
    void parallel_rows(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows) {
        if (rows == 0 || width == 0) return;
        Batch batch;
        batch.dst = (uint8_t*)dst; batch.src = (const uint8_t*)src; batch.bytes = rows * width; batch.piece = width;
        batch.npieces = rows; batch.dpitch = dpitch; batch.spitch = spitch; batch.rows = true;
        if (nthreads_ == 0) { work(batch); return; }
        run(batch);
    }
private:
    struct Batch;
    void run(Batch& batch) {
        {
            std::lock_guard<std::mutex> lock(mu_);
            queue_.push_back(&batch);
        }
        cv_.notify_all();
        work(batch);                                              // the caller copies too
        std::unique_lock<std::mutex> lock(mu_);
        for (auto it = queue_.begin(); it != queue_.end(); ++it) if (*it == &batch) { queue_.erase(it); break; }
        // no worker can pick the batch up any more; wait for the ones inside it
        done_cv_.wait(lock, [&] { return batch.active == 0; });
    }
    struct Batch {
        uint8_t* dst; const uint8_t* src; size_t bytes, piece, npieces;
        size_t dpitch = 0, spitch = 0;
        bool rows = false;
        std::atomic<size_t> next{0};
        int active = 0;                                           // workers inside work(); guarded by mu_
    };
    CopyPool() {
        int n = 12;                                              // 2^24-point pageable snarkvm_msm: 6 → 128 ms, 12 → 114–120 ms, 24/48 no better (profiles/r2i_e2e_pageable.log)
        // one process per GPU on a shared host (torchrun exports LOCAL_WORLD_SIZE): do not oversubscribe the cores with copy threads
        if (const char* lws = getenv("LOCAL_WORLD_SIZE")) {
            const int procs = atoi(lws), cores = (int)std::thread::hardware_concurrency();
            if (procs > 1 && cores > 0) { int per = cores / procs - 1; if (per < 2) per = 2; if (per < n) n = per; }
        }
        if (const char* e = getenv("SNARKVM_B200_COPY_THREADS")) { int v = atoi(e); if (v >= 0 && v <= 64) n = v; }
        nthreads_ = n;
        have_numa_ = device_local_cpus(&numa_);
        for (int i = 0; i < n; i++) std::thread([this] { loop(); }).detach();
    }
    static void work(Batch& b) {
        for (;;) {
            size_t k = b.next.fetch_add(1);
            if (k >= b.npieces) return;
            if (b.rows) { host_stream_copy(b.dst + k * b.dpitch, b.src + k * b.spitch, b.piece); continue; }
            size_t off = k * b.piece, len = b.bytes - off < b.piece ? b.bytes - off : b.piece;
            host_stream_copy(b.dst + off, b.src + off, len);
        }
    }
    void loop() {
        if (have_numa_) pthread_setaffinity_np(pthread_self(), sizeof numa_, &numa_);       // best effort
        std::unique_lock<std::mutex> lock(mu_);
        for (;;) {
            cv_.wait(lock, [&] { return !queue_.empty(); });
            Batch* b = queue_.front();
            if (b->next.load() >= b->npieces) { queue_.pop_front(); continue; }      // nothing left to claim in it
            b->active++;
            lock.unlock();
            work(*b);
            lock.lock();
            if (--b->active == 0) done_cv_.notify_all();
        }
    }
    std::mutex mu_;
    std::condition_variable cv_, done_cv_;
    std::deque<Batch*> queue_;
    int nthreads_ = 0;
    cpu_set_t numa_;
    bool have_numa_ = false;
};

static bool host_is_pinned(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
}

// per-thread ring of pinned staging buffers
struct StageRing {
    static constexpr int SLOTS = 4;
    static constexpr size_t SLOT_BYTES = (size_t)32 << 20;
    void* buf[SLOTS] = {};
    cudaEvent_t ev[SLOTS] = {};
    bool used[SLOTS] = {};
    int next = 0;
    int init() {
        if (buf[0]) return 0;
        // the slots are allocated (= pinned, first-touched) while the calling thread sits on the device's NUMA node
        cpu_set_t local, old;
        const bool moved = CopyPool::get().numa_cpus(&local) && sched_getaffinity(0, sizeof old, &old) == 0 &&
                           sched_setaffinity(0, sizeof local, &local) == 0;
        int rc = 0;
        for (int i = 0; i < SLOTS && rc == 0; i++) {
            cudaError_t e = cudaHostAlloc(&buf[i], SLOT_BYTES, cudaHostAllocDefault);
            if (e == cudaSuccess) { memset(buf[i], 0, SLOT_BYTES); e = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming); }
            if (e != cudaSuccess) rc = (int)e;
        }
        if (moved) sched_setaffinity(0, sizeof old, &old);
        return rc;
    }
};
thread_local StageRing t_ring;

// dst (device) ← src (host), enqueued on `copy`: direct DMA for pinned sources, staged for pageable ones
int upload(void* d_dst, const void* h_src, size_t bytes, cudaStream_t copy, bool pinned) {
    if (bytes == 0) return 0;
    static const bool no_stage = getenv("SNARKVM_B200_NO_STAGING") != nullptr;
    if (pinned || no_stage || bytes < ((size_t)1 << 20)) return (int)cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, copy);
    int rc = t_ring.init();
    if (rc) return rc;
    for (size_t off = 0; off < bytes; off += StageRing::SLOT_BYTES) {
        const size_t len = bytes - off < StageRing::SLOT_BYTES ? bytes - off : StageRing::SLOT_BYTES;
        const int sl = t_ring.next;
        t_ring.next = (sl + 1) % StageRing::SLOTS;
        if (t_ring.used[sl] && (rc = (int)cudaEventSynchronize(t_ring.ev[sl])) != 0) return rc;     // its previous DMA has drained
        CopyPool::get().parallel_memcpy(t_ring.buf[sl], (const uint8_t*)h_src + off, len);
        if ((rc = (int)cudaMemcpyAsync((uint8_t*)d_dst + off, t_ring.buf[sl], len, cudaMemcpyHostToDevice, copy)) != 0) return rc;
        if ((rc = (int)cudaEventRecord(t_ring.ev[sl], copy)) != 0) return rc;
        t_ring.used[sl] = true;
    }
    return 0;
}
// src (device) → dst (host) after everything already enqueued on `stream`; returns when dst is complete
int download(void* h_dst, const void* d_src, size_t bytes, cudaStream_t stream, bool pinned) {
    if (bytes == 0) return (int)cudaStreamSynchronize(stream);
    static const bool no_stage = getenv("SNARKVM_B200_NO_STAGING") != nullptr;
    if (pinned || no_stage || bytes < ((size_t)1 << 20)) {
        int rc = (int)cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, stream);
        return rc ? rc : (int)cudaStreamSynchronize(stream);
    }
    int rc = t_ring.init();
    if (rc) return rc;
    for (int i = 0; i < StageRing::SLOTS; i++)                                // uploads of this thread that may still be reading a slot
        if (t_ring.used[i] && (rc = (int)cudaEventSynchronize(t_ring.ev[i])) != 0) return rc;
    // DMA slot k+1 while the copy threads unload slot k
    const size_t nslices = (bytes + StageRing::SLOT_BYTES - 1) / StageRing::SLOT_BYTES;
    auto slice_len = [&](size_t k) { size_t off = k * StageRing::SLOT_BYTES; return bytes - off < StageRing::SLOT_BYTES ? bytes - off : StageRing::SLOT_BYTES; };
    for (size_t k = 0; k < nslices && k < 2; k++) {
        if ((rc = (int)cudaMemcpyAsync(t_ring.buf[k & 1], (const uint8_t*)d_src + k * StageRing::SLOT_BYTES, slice_len(k), cudaMemcpyDeviceToHost, stream)) != 0) return rc;
        if ((rc = (int)cudaEventRecord(t_ring.ev[k & 1], stream)) != 0) return rc;
    }
    for (size_t k = 0; k < nslices; k++) {
        if ((rc = (int)cudaEventSynchronize(t_ring.ev[k & 1])) != 0) return rc;
        CopyPool::get().parallel_memcpy((uint8_t*)h_dst + k * StageRing::SLOT_BYTES, t_ring.buf[k & 1], slice_len(k));
        if (k + 2 < nslices) {
            if ((rc = (int)cudaMemcpyAsync(t_ring.buf[k & 1], (const uint8_t*)d_src + (k + 2) * StageRing::SLOT_BYTES, slice_len(k + 2), cudaMemcpyDeviceToHost, stream)) != 0) return rc;
            if ((rc = (int)cudaEventRecord(t_ring.ev[k & 1], stream)) != 0) return rc;
        }
    }
    for (int i = 0; i < StageRing::SLOTS; i++) t_ring.used[i] = false;      // every slot is idle again
    return (int)cudaStreamSynchronize(stream);
}

// NN is native (bit reversal fused into the last pass); the other orders add explicit derange passes:
// R-input ⇒ permute before, R-output ⇒ permute after.
int ntt_ordered(void* d, uint32_t lg, int order, int dir, int type, void* scratch, cudaStream_t stream) {
    if (order < 0 || order > 3) return (int)cudaErrorInvalidValue;
    int rc = 0;
    if (order == SNARKVM_NTT_RN || order == SNARKVM_NTT_RR) rc = fr_bitrev_device(d, lg, stream);
    if (rc == 0) rc = ntt_device(d, lg, dir, type, scratch, stream);
    if (rc == 0 && (order == SNARKVM_NTT_NR || order == SNARKVM_NTT_RR)) rc = fr_bitrev_device(d, lg, stream);
    return rc;
}

// snarkvm_ntt for large NN transforms: the host buffer crosses PCIe by COLUMN RANGES underneath the first and the last pass.
// Pass 0 works on tiles that are column ranges of the 2^S0 × 2^(lg−S0) row-major view of the input, the last pass produces
// column ranges of the 2^SL × 2^t0 view of the output (ntt.cu): range k + 1 is uploaded while pass 0 runs on range k, and range
// k is downloaded while the last pass runs on range k + 1.  A 2^24 transform is 2 × 9.6 ms of PCIe around 4.1 ms of kernels; this
// hides the 2.7 ms of the two outer passes.  Pageable buffers go through the thread's pinned ring, row by row.
// The passes before the last are checked for errors BEFORE the first byte is written back (the Rust caller falls back to its CPU
// path on an error code and needs its input intact).
int ntt_host_pipelined(void* inout, uint32_t lg, int dir, int type, cudaStream_t stream, bool pinned) {
    NttPass passes[8];
    int P = 0, rc = ntt_make_passes(lg, passes, &P);
    if (rc) return rc;
    const size_t n = (size_t)1 << lg, bytes = n * 32;
    const NttPass &p0 = passes[0], &pl = passes[P - 1];
    const size_t rows0 = (size_t)1 << p0.S, cols0 = n >> p0.S, rowsL = (size_t)1 << pl.S, colsL = n >> pl.S;
    // chunks: whole tiles, ≤ one staging slot per chunk for pageable buffers
    size_t K = 8;
    while ((bytes / K) > StageRing::SLOT_BYTES && !pinned) K <<= 1;
    while (K > 1 && ((p0.tiles % K) || (pl.tiles % K))) K >>= 1;
    if (P < 2 || K < 2 || (!pinned && bytes / K > StageRing::SLOT_BYTES)) return -1;       // not applicable: the caller takes the plain path
    cudaStream_t copy = nullptr;
    void *d = nullptr, *scratch = nullptr;
    std::vector<cudaEvent_t> ev(2 * K + 1, nullptr);
    rc = thread_copy_stream(&copy);
    if (rc == 0) rc = (int)pool_alloc(&d, bytes, stream);
    if (rc == 0) rc = (int)pool_alloc(&scratch, bytes, stream);
    for (auto& e : ev) if (rc == 0) rc = (int)cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (rc == 0 && !pinned) rc = t_ring.init();
    if (rc == 0) rc = (int)cudaEventRecord(ev[2 * K], stream);                       // the allocations are ordered on `stream`
    if (rc == 0) rc = (int)cudaStreamWaitEvent(copy, ev[2 * K], 0);
    uint8_t* h = (uint8_t*)inout;
    // ---- upload by column ranges, pass 0 right behind each ----
    for (size_t k = 0; k < K && rc == 0; k++) {
        const size_t c0 = cols0 / K * k, nc = cols0 / K, width = nc * 32, pitch = cols0 * 32;
        if (pinned) {
            rc = (int)cudaMemcpy2DAsync((uint8_t*)d + c0 * 32, pitch, h + c0 * 32, pitch, width, rows0, cudaMemcpyHostToDevice, copy);
        } else {
            const int sl = t_ring.next;
            t_ring.next = (sl + 1) % StageRing::SLOTS;
            if (t_ring.used[sl]) rc = (int)cudaEventSynchronize(t_ring.ev[sl]);
            if (rc == 0) {
                CopyPool::get().parallel_rows(t_ring.buf[sl], width, h + c0 * 32, pitch, width, rows0);
                rc = (int)cudaMemcpy2DAsync((uint8_t*)d + c0 * 32, pitch, t_ring.buf[sl], width, width, rows0, cudaMemcpyHostToDevice, copy);
            }
            if (rc == 0) rc = (int)cudaEventRecord(t_ring.ev[sl], copy);
            t_ring.used[sl] = true;
        }
        if (rc == 0) rc = (int)cudaEventRecord(ev[k], copy);
        if (rc == 0) rc = (int)cudaStreamWaitEvent(stream, ev[k], 0);
        if (rc == 0) rc = ntt_launch_pass(d, scratch, lg, dir, type, 0, p0.tiles / K * k, p0.tiles / K, stream);
    }
    for (int p = 1; p + 1 < P && rc == 0; p++) rc = ntt_launch_pass(d, scratch, lg, dir, type, p, 0, passes[p].tiles, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);                            // everything so far succeeded: the output may start to land
    // ---- last pass by column ranges, download right behind each ----
    struct Pending { int slot; size_t c0; };
    std::deque<Pending> pending;                                                      // pageable: slots whose DMA is in flight, oldest first
    const size_t ncL = colsL / K, widthL = ncL * 32, pitchL = colsL * 32;
    auto unstage = [&](const Pending& pd) -> int {
        int r = (int)cudaEventSynchronize(t_ring.ev[pd.slot]);
        if (r == 0) CopyPool::get().parallel_rows(h + pd.c0 * 32, pitchL, t_ring.buf[pd.slot], widthL, widthL, rowsL);
        t_ring.used[pd.slot] = false;
        return r;
    };
    if (rc == 0 && !pinned)
        for (int i = 0; i < StageRing::SLOTS && rc == 0; i++) { if (t_ring.used[i]) rc = (int)cudaEventSynchronize(t_ring.ev[i]); t_ring.used[i] = false; }
    for (size_t k = 0; k < K && rc == 0; k++) {
        const size_t c0 = ncL * k;
        rc = ntt_launch_pass(d, scratch, lg, dir, type, P - 1, pl.tiles / K * k, pl.tiles / K, stream);
        if (rc == 0) rc = (int)cudaEventRecord(ev[K + k], stream);
        if (rc == 0) rc = (int)cudaStreamWaitEvent(copy, ev[K + k], 0);
        if (rc != 0) break;
        if (pinned) {
            rc = (int)cudaMemcpy2DAsync(h + c0 * 32, pitchL, (uint8_t*)d + c0 * 32, pitchL, widthL, rowsL, cudaMemcpyDeviceToHost, copy);
        } else {
            if ((int)pending.size() == StageRing::SLOTS) { rc = unstage(pending.front()); pending.pop_front(); if (rc) break; }
            int sl = -1;
            for (int i = 0; i < StageRing::SLOTS; i++) if (!t_ring.used[i]) { sl = i; break; }
            rc = (int)cudaMemcpy2DAsync(t_ring.buf[sl], widthL, (uint8_t*)d + c0 * 32, pitchL, widthL, rowsL, cudaMemcpyDeviceToHost, copy);
            if (rc == 0) rc = (int)cudaEventRecord(t_ring.ev[sl], copy);
            t_ring.used[sl] = true;
            pending.push_back(Pending{sl, c0});
        }
    }
    while (rc == 0 && !pending.empty()) { rc = unstage(pending.front()); pending.pop_front(); }
    if (copy) { int rs = (int)cudaStreamSynchronize(copy); if (rc == 0) rc = rs; }
    { int rs = (int)cudaStreamSynchronize(stream); if (rc == 0) rc = rs; }
    if (!pinned) for (int i = 0; i < StageRing::SLOTS; i++) t_ring.used[i] = false;
    for (auto& e : ev) if (e) cudaEventDestroy(e);
    if (d) cudaFreeAsync(d, stream);
    if (scratch) cudaFreeAsync(scratch, stream);
    return rc;
}

int polymul_device_impl(void* d_out, size_t pcount, const void* const* d_polys, const size_t* plens, size_t ecount,
                        const void* const* d_evals, const size_t* elens, uint32_t lg, cudaStream_t stream) {
    const size_t n = (size_t)1 << lg, bytes = n * 32;
    if (pcount + ecount == 0) return 0;
    for (size_t i = 0; i < pcount; i++) if (plens[i] > n) return (int)cudaErrorInvalidValue;
    for (size_t i = 0; i < ecount; i++) if (elens[i] != n) return (int)cudaErrorInvalidValue;   // polynomial.cuh:95
    void *tmp = nullptr, *scratch = nullptr;
    cudaError_t e;
    if ((e = pool_alloc(&tmp, bytes, stream)) != cudaSuccess) return (int)e;
    if ((e = pool_alloc(&scratch, bytes, stream)) != cudaSuccess) { cudaFreeAsync(tmp, stream); return (int)e; }
    int rc = 0;
    bool have = false;
    for (size_t i = 0; i < pcount && rc == 0; i++) {
        void* dst = have ? tmp : d_out;
        rc = (int)cudaMemsetAsync(dst, 0, bytes, stream);
        if (rc == 0 && plens[i]) rc = (int)cudaMemcpyAsync(dst, d_polys[i], plens[i] * 32, cudaMemcpyDeviceToDevice, stream);
        if (rc == 0) rc = ntt_device(dst, lg, NTT_FORWARD, NTT_STANDARD, scratch, stream);
        if (rc == 0 && have) rc = fr_pointwise_mul_device(d_out, tmp, n, stream);
        have = true;
    }
    for (size_t i = 0; i < ecount && rc == 0; i++) {
        if (have) rc = fr_pointwise_mul_device(d_out, d_evals[i], n, stream);
        else rc = (int)cudaMemcpyAsync(d_out, d_evals[i], bytes, cudaMemcpyDeviceToDevice, stream);
        have = true;
    }
    if (rc == 0) rc = ntt_device(d_out, lg, NTT_INVERSE, NTT_STANDARD, scratch, stream);
    cudaFreeAsync(tmp, stream);
    cudaFreeAsync(scratch, stream);
    return rc;
}

}  // namespace

extern "C" {

const char* snarkvm_b200_version(void) { return "snarkvm_b200 0.1 (sm_100a)"; }
uint64_t snarkvm_b200_launch_count(void) { return launch_count(); }

// ----------------------------------------------------------------------------------------
// PART 1 — drop-in symbols
// ----------------------------------------------------------------------------------------
snarkvm_error_t snarkvm_ntt(void* inout, uint32_t lg, snarkvm_ntt_order_t order, snarkvm_ntt_direction_t dir,
                            snarkvm_ntt_type_t type) {
    if (lg > NTT_MAX_LG || !inout || (int)order < 0 || (int)order > 3) return make_error((int)cudaErrorInvalidValue);
    cudaStream_t stream;
    int rc = thread_stream(&stream);
    if (rc) return make_error(rc);
    const size_t bytes = ((size_t)1 << lg) * 32;
    const bool pinned = host_is_pinned(inout);
    static const bool no_pipe = getenv("SNARKVM_B200_NTT_NO_PIPELINE") != nullptr;
    if (lg >= 20 && order == SNARKVM_NTT_NN && !no_pipe) {
        rc = ntt_host_pipelined(inout, lg, (int)dir, (int)type, stream, pinned);
        if (rc != -1) {
            int rs = (int)cudaStreamSynchronize(stream);
            return make_error(rc ? rc : rs);
        }
        rc = 0;
    }
    void *d = nullptr, *scratch = nullptr;
    rc = (int)pool_alloc(&d, bytes, stream);
    if (rc == 0) rc = (int)pool_alloc(&scratch, bytes, stream);
    if (rc == 0) rc = upload(d, inout, bytes, stream, pinned);
    if (rc == 0) rc = ntt_ordered(d, lg, (int)order, (int)dir, (int)type, scratch, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);          // only copy back on success (snarkvm.cu:178-183)
    if (rc == 0) rc = download(inout, d, bytes, stream, pinned);
    if (d) cudaFreeAsync(d, stream);
    if (scratch) cudaFreeAsync(scratch, stream);
    int rs = (int)cudaStreamSynchronize(stream);
    return make_error(rc ? rc : rs);
}

snarkvm_error_t snarkvm_polymul(void* out, size_t pcount, const void* polynomials, const void* plens_v, size_t ecount,
                                const void* evaluations, const void* elens_v, uint32_t lg) {
    if (pcount + ecount == 0) return make_error(0);                 // snarkvm.cu:195-197
    if (lg > NTT_MAX_LG || !out) return make_error((int)cudaErrorInvalidValue);
    const void* const* polys = (const void* const*)polynomials;
    const void* const* evals = (const void* const*)evaluations;
    const size_t* plens = (const size_t*)plens_v;
    const size_t* elens = (const size_t*)elens_v;
    const size_t n = (size_t)1 << lg, bytes = n * 32;
    for (size_t i = 0; i < pcount; i++) if (plens[i] > n) return make_error((int)cudaErrorInvalidValue);
    for (size_t i = 0; i < ecount; i++) if (elens[i] != n) return make_error((int)cudaErrorInvalidValue);
    cudaStream_t stream;
    int rc = thread_stream(&stream);
    if (rc) return make_error(rc);
    std::vector<void*> dbuf(pcount + ecount, nullptr);
    std::vector<const void*> dp(pcount), de(ecount);
    void* d_out = nullptr;
    rc = (int)pool_alloc(&d_out, bytes, stream);
    for (size_t i = 0; i < pcount && rc == 0; i++) {
        size_t b = plens[i] ? plens[i] * 32 : 32;
        rc = (int)pool_alloc(&dbuf[i], b, stream);
        if (rc == 0 && plens[i]) rc = upload(dbuf[i], polys[i], plens[i] * 32, stream, host_is_pinned(polys[i]));
        dp[i] = dbuf[i];
    }
    for (size_t i = 0; i < ecount && rc == 0; i++) {
        rc = (int)pool_alloc(&dbuf[pcount + i], bytes, stream);
        if (rc == 0) rc = upload(dbuf[pcount + i], evals[i], bytes, stream, host_is_pinned(evals[i]));
        de[i] = dbuf[pcount + i];
    }
    if (rc == 0) rc = polymul_device_impl(d_out, pcount, dp.data(), plens, ecount, de.data(), elens, lg, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc == 0) rc = download(out, d_out, bytes, stream, host_is_pinned(out));
    for (void* p : dbuf) if (p) cudaFreeAsync(p, stream);
    if (d_out) cudaFreeAsync(d_out, stream);
    int rs = (int)cudaStreamSynchronize(stream);
    return make_error(rc ? rc : rs);
}

// Large host-buffer MSMs are cut into point ranges: range k+1 crosses PCIe on the thread's copy stream while range k is in
// the Pippenger kernels (an MSM is a sum over points: every range is a complete MSM with its own plan and the results add).
// 2^24 points: 2.28 GB of upload, ≈ 40 ms, of which only the first range's share stays exposed — so the first range is small
// (1/16 of the points), then 1/8, 1/4 and the rest (swept in profiles/r2i_e2e_pageable.log).  SNARKVM_B200_MSM_CHUNKS = "1", "2" (equal parts) or weights like "1:3:4".
static std::vector<size_t> msm_ranges(size_t npoints) {
    std::vector<size_t> w;
    if (npoints >= ((size_t)1 << 23)) w = {1, 2, 4, 9};
    if (const char* e = getenv("SNARKVM_B200_MSM_CHUNKS")) {
        std::vector<size_t> v;
        for (const char* p = e; *p;) {
            char* end = nullptr;
            long x = strtol(p, &end, 10);
            if (end == p || x < 1 || x > 1024) { v.clear(); break; }
            v.push_back((size_t)x);
            p = *end == ':' ? end + 1 : end;
            if (*end && *end != ':') { v.clear(); break; }
        }
        if (v.size() == 1) v.assign(v[0] <= 64 ? v[0] : 64, 1);            // "k" = k equal parts
        if (!v.empty()) w = v;
    }
    size_t total = 0;
    for (size_t x : w) total += x;
    std::vector<size_t> bounds{0};                                        // range k = [bounds[k], bounds[k+1])
    size_t acc = 0;
    for (size_t x : w) {
        acc += x;
        size_t b = (size_t)((unsigned __int128)npoints * acc / total);
        if (b > bounds.back()) bounds.push_back(b);                       // empty ranges are dropped
    }
    if (bounds.back() != npoints) bounds.push_back(npoints);
    return bounds;
}

snarkvm_error_t snarkvm_msm(void* out, const void* points, size_t npoints, const void* scalars, size_t ffi_affine_sz) {
    if (!out) return make_error((int)cudaErrorInvalidValue);
    if (npoints == 0) { write_infinity(out); return make_error(0); }
    if (!points || !scalars || ffi_affine_sz < 104 || (ffi_affine_sz & 7)) return make_error((int)cudaErrorInvalidValue);
    cudaStream_t stream;
    int rc = thread_stream(&stream);
    if (rc) return make_error(rc);
    void *d_points = nullptr, *d_scalars = nullptr;
    std::shared_ptr<ResidentBases> rb = find_resident(points, npoints, ffi_affine_sz);     // kept alive until this call returns
    const bool resident = rb != nullptr;
    std::vector<size_t> bounds{0, npoints};
    if (!resident) bounds = msm_ranges(npoints);
    const int chunks = (int)bounds.size() - 1;
    const bool pin_s = host_is_pinned(scalars), pin_p = resident || host_is_pinned(points);
    if (!resident) rc = (int)pool_alloc(&d_points, npoints * ffi_affine_sz, stream);
    if (rc == 0) rc = (int)pool_alloc(&d_scalars, npoints * 32, stream);
    uint64_t result[18];
    if (chunks == 1) {
        if (rc == 0) rc = upload(d_scalars, scalars, npoints * 32, stream, pin_s);
        if (rc == 0 && !resident) rc = upload(d_points, points, npoints * ffi_affine_sz, stream, pin_p);
        if (rc == 0 && resident && rb->tables.load()) rc = snarkvm_b200_msm_precomputed_device(result, rb->tables.load(), d_scalars, npoints, stream);
        else if (rc == 0) rc = msm_device_impl(result, resident ? rb->d_ptr : d_points, npoints, d_scalars, ffi_affine_sz, 0, stream);
    } else {
        cudaStream_t copy = nullptr;
        if (rc == 0) rc = thread_copy_stream(&copy);
        std::vector<MsmPlan> plans;
        std::vector<size_t> sum_off{0};                                   // in XYZZ points
        for (int k = 0; k < chunks; k++) {
            plans.push_back(msm_make_plan(bounds[k + 1] - bounds[k]));
            sum_off.push_back(sum_off.back() + (size_t)plans.back().nwin);
        }
        std::vector<cudaEvent_t> ev((size_t)chunks + 1, nullptr);
        for (auto& e : ev) if (rc == 0) rc = (int)cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        uint32_t* d_sums = nullptr;
        const size_t nsums = sum_off.back();
        if (rc == 0) rc = (int)pool_alloc(&d_sums, nsums * 192 + 256, stream);
        uint32_t* d_flags = d_sums ? d_sums + nsums * 48 : nullptr;
        if (rc == 0) rc = (int)cudaMemsetAsync(d_flags, 0, 256, stream);
        // the pool allocations above are ordered on `stream`; the copy stream may touch them only after this point
        if (rc == 0) rc = (int)cudaEventRecord(ev[chunks], stream);
        if (rc == 0) rc = (int)cudaStreamWaitEvent(copy, ev[chunks], 0);
        // Issue order: upload of range k, then the kernels of range k.  A pageable upload keeps this thread busy (staging)
        // until its last slice is on its way, so the kernels of range k−1 — already enqueued — run underneath it.
        for (int k = 0; k < chunks && rc == 0; k++) {
            const size_t i0 = bounds[k], cn = bounds[k + 1] - i0;
            rc = upload((uint8_t*)d_scalars + i0 * 32, (const uint8_t*)scalars + i0 * 32, cn * 32, copy, pin_s);
            if (rc == 0) rc = upload((uint8_t*)d_points + i0 * ffi_affine_sz, (const uint8_t*)points + i0 * ffi_affine_sz, cn * ffi_affine_sz, copy, pin_p);
            if (rc == 0) rc = (int)cudaEventRecord(ev[k], copy);
            if (rc == 0) rc = (int)cudaStreamWaitEvent(stream, ev[k], 0);
            if (rc == 0) rc = msm_window_sums_device(d_sums + sum_off[k] * 48, d_flags, plans[k], (const uint8_t*)d_points + i0 * ffi_affine_sz,
                                                     ffi_affine_sz, (const uint8_t*)d_scalars + i0 * 32, cn, stream);
        }
        std::vector<host::Xyzz> sums(nsums + 2);
        if (rc == 0) rc = (int)cudaMemcpyAsync(sums.data(), d_sums, nsums * 192 + 256, cudaMemcpyDeviceToHost, stream);
        if (d_sums) cudaFreeAsync(d_sums, stream);
        // on any failure the copy stream may still be writing: drain it before the buffers go back to the pool
        if (copy) { int rs = (int)cudaStreamSynchronize(copy); if (rc == 0) rc = rs; }
        if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        if (rc == 0) {
            uint32_t flags = 0;
            memcpy(&flags, sums.data() + nsums, 4);
            if (flags & 1u) rc = (int)cudaErrorInvalidValue;
        }
        if (rc == 0) {
            host::Xyzz total = host::xyzz_inf();
            for (int k = 0; k < chunks; k++) host::xyzz_add(total, host::horner_windows(sums.data() + sum_off[k], plans[k].nwin, plans[k].c));
            host::xyzz_to_normalised_projective(total, result);
        }
    }
    if (d_points) cudaFreeAsync(d_points, stream);
    if (d_scalars) cudaFreeAsync(d_scalars, stream);
    int rs = (int)cudaStreamSynchronize(stream);
    if (rc == 0 && rs == 0) memcpy(out, result, 144);
    return make_error(rc ? rc : rs);
}

// ----------------------------------------------------------------------------------------
// PART 2 — extended device-resident API
// ----------------------------------------------------------------------------------------
int snarkvm_b200_ntt_device(void* d_inout, uint32_t lg, int order, int dir, int type, void* d_scratch, void* stream) {
    if (lg > NTT_MAX_LG) return (int)cudaErrorInvalidValue;
    return ntt_ordered(d_inout, lg, order, dir, type, d_scratch, (cudaStream_t)stream);
}

int snarkvm_b200_polymul_device(void* d_out, size_t pcount, const void* const* d_polys, const size_t* plens, size_t ecount,
                                const void* const* d_evals, const size_t* elens, uint32_t lg, void* stream) {
    if (lg > NTT_MAX_LG) return (int)cudaErrorInvalidValue;
    return polymul_device_impl(d_out, pcount, d_polys, plens, ecount, d_evals, elens, lg, (cudaStream_t)stream);
}

int snarkvm_b200_msm_plan(size_t npoints, int* c, int* nwin, uint32_t* cap) {
    MsmPlan p = msm_make_plan(npoints);
    if (c) *c = p.c;
    if (nwin) *nwin = p.nwin;
    if (cap) *cap = p.cap;
    return 0;
}

int snarkvm_b200_msm_plan_levels(size_t npoints) { return msm_make_plan(npoints).levels; }

int snarkvm_b200_msm_device(void* out144, const void* d_points, size_t npoints, const void* d_scalars, size_t stride,
                            void* stream) {
    if (!out144) return (int)cudaErrorInvalidValue;
    return msm_device_impl(out144, d_points, npoints, d_scalars, stride, 0, (cudaStream_t)stream);
}

// `count` MSMs over the SAME resident bases in one pass: one digit/sort keyed by (vector, window, bucket), one set of pair
// levels, count × nwin window sums, one D2H + one synchronisation, Horner per vector on the host.
static int msm_batch_impl(void* out144s, const void* d_points, size_t stride, const void* const* d_scalars, const size_t* nscalars,
                          size_t count, int mont, const void* d_points2, const void* const* d_scalars2, const size_t* nscalars2,
                          cudaStream_t stream) {
    if (count == 0) return 0;
    if (!out144s || !d_scalars || !nscalars || stride < 104 || (stride & 7)) return (int)cudaErrorInvalidValue;
    // empty vectors commit to the identity; the rest become jobs
    std::vector<MsmSegment> segs;
    std::vector<size_t> job_of(count, (size_t)-1);
    size_t max_n = 0, total_n = 0, max_n2 = 0;
    uint32_t njobs = 0;
    for (size_t i = 0; i < count; i++) {
        const size_t n2 = (d_scalars2 && nscalars2) ? nscalars2[i] : 0;
        if (nscalars[i] == 0 && n2 == 0) { write_infinity((uint8_t*)out144s + i * 144); continue; }
        job_of[i] = njobs;
        if (nscalars[i]) segs.push_back(MsmSegment{d_scalars[i], nscalars[i], 0u, njobs, mont});
        if (nscalars[i] > max_n) max_n = nscalars[i];
        if (n2 > max_n2) max_n2 = n2;
        total_n += nscalars[i] + n2;
        njobs++;
    }
    if (njobs == 0) return 0;
    if (max_n >= (1ull << 31)) return (int)cudaErrorInvalidValue;
    // second segments (the blinding polynomials against powers_of_beta_times_gamma_g) index the bases after the first array
    for (size_t i = 0; i < count; i++) {
        const size_t n2 = (d_scalars2 && nscalars2) ? nscalars2[i] : 0;
        if (n2) segs.push_back(MsmSegment{d_scalars2[i], n2, (uint32_t)max_n, (uint32_t)job_of[i], mont});
    }
    MsmBases bases[2] = {{d_points, stride, max_n}, {d_points2, stride, max_n2}};
    const int nbases = max_n2 ? 2 : 1;
    if (max_n2 && !d_points2) return (int)cudaErrorInvalidValue;
    size_t job_max = max_n + max_n2;
    MsmPlan plan = msm_make_plan_batch(job_max ? job_max : 1, total_n);
    std::vector<uint8_t> outs((size_t)njobs * 144);
    int rc = msm_jobs_impl(outs.data(), plan, bases, nbases, nullptr, 0, segs.data(), (int)segs.size(), (int)njobs, stream);
    if (rc != 0) return rc;
    for (size_t i = 0; i < count; i++) if (job_of[i] != (size_t)-1) memcpy((uint8_t*)out144s + i * 144, outs.data() + job_of[i] * 144, 144);
    return 0;
}

int snarkvm_b200_msm_batch_device(void* out144s, const void* d_points, size_t stride, const void* const* d_scalars, const size_t* nscalars,
                                  size_t count, void* stream) {
    return msm_batch_impl(out144s, d_points, stride, d_scalars, nscalars, count, 0, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int snarkvm_b200_msm_window_sums_device(void* d_window_sums, const void* d_points, size_t npoints, const void* d_scalars,
                                        size_t stride, void* stream) {
    return snarkvm_b200_msm_window_sums_plan_device(d_window_sums, nullptr, npoints, d_points, npoints, d_scalars, stride, stream);
}

// Window sums under the plan of `plan_npoints` (every rank of a sharded MSM passes the SAME plan_npoints — the largest shard —
// so all ranks use one window size whatever their own shard length; an empty shard contributes infinity sums).
// d_flags: device u32 (zeroed here) that gets bit 0 set if a scalar has bits 253..255 set, or NULL.
int snarkvm_b200_msm_window_sums_plan_device(void* d_window_sums, uint32_t* d_flags, size_t plan_npoints, const void* d_points,
                                             size_t npoints, const void* d_scalars, size_t stride, void* stream_v) {
    if (!d_window_sums || stride < 104 || (stride & 7) || plan_npoints == 0 || npoints > plan_npoints) return (int)cudaErrorInvalidValue;
    cudaStream_t stream = (cudaStream_t)stream_v;
    MsmPlan plan = msm_make_plan(plan_npoints);
    uint32_t* own_flags = nullptr;
    int rc = 0;
    if (!d_flags) { rc = (int)pool_alloc(&own_flags, 256, stream); if (rc) return rc; d_flags = own_flags; }
    rc = (int)cudaMemsetAsync(d_flags, 0, 4, stream);
    if (rc == 0 && npoints == 0) rc = (int)cudaMemsetAsync(d_window_sums, 0, (size_t)plan.nwin * 192, stream);     // XYZZ infinity = zeros
    else if (rc == 0) rc = msm_window_sums_device((uint32_t*)d_window_sums, d_flags, plan, d_points, stride, d_scalars, npoints, stream);
    if (own_flags) cudaFreeAsync(own_flags, stream);
    return rc;
}

// Host-buffer form of the sharded building block: uploads this rank's shard (point ranges overlapped with the kernels of the
// previous range, pageable sources staged through pinned buffers) and leaves its window sums under the plan of `plan_npoints`
// in HBM — nothing is synchronised, so the caller can enqueue its collective right behind it.
int snarkvm_b200_msm_window_sums_host(void* d_window_sums, uint32_t* d_flags, size_t plan_npoints, const void* h_points, size_t npoints,
                                      const void* h_scalars, size_t stride, void* stream_v) {
    if (!d_window_sums || stride < 104 || (stride & 7) || plan_npoints == 0 || npoints > plan_npoints) return (int)cudaErrorInvalidValue;
    cudaStream_t stream = (cudaStream_t)stream_v;
    MsmPlan plan = msm_make_plan(plan_npoints);
    uint32_t* own_flags = nullptr;
    int rc = 0;
    if (!d_flags) { rc = (int)pool_alloc(&own_flags, 256, stream); if (rc) return rc; d_flags = own_flags; }
    rc = (int)cudaMemsetAsync(d_flags, 0, 4, stream);
    if (npoints == 0) {
        if (rc == 0) rc = (int)cudaMemsetAsync(d_window_sums, 0, (size_t)plan.nwin * 192, stream);
        if (own_flags) cudaFreeAsync(own_flags, stream);
        return rc;
    }
    if (!h_points || !h_scalars) { if (own_flags) cudaFreeAsync(own_flags, stream); return (int)cudaErrorInvalidValue; }
    std::vector<size_t> bounds = msm_ranges(npoints);
    const int chunks = (int)bounds.size() - 1;
    const bool pin_s = host_is_pinned(h_scalars), pin_p = host_is_pinned(h_points);
    cudaStream_t copy = nullptr;
    void *d_points = nullptr, *d_scalars = nullptr;
    uint32_t* d_parts = nullptr;
    std::vector<cudaEvent_t> ev((size_t)chunks + 1, nullptr);
    if (rc == 0) rc = thread_copy_stream(&copy);
    if (rc == 0) rc = (int)pool_alloc(&d_points, npoints * stride, stream);
    if (rc == 0) rc = (int)pool_alloc(&d_scalars, npoints * 32, stream);
    if (rc == 0 && chunks > 1) rc = (int)pool_alloc(&d_parts, (size_t)chunks * plan.nwin * 192, stream);
    for (auto& e : ev) if (rc == 0) rc = (int)cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (rc == 0) rc = (int)cudaEventRecord(ev[chunks], stream);
    if (rc == 0) rc = (int)cudaStreamWaitEvent(copy, ev[chunks], 0);
    for (int k = 0; k < chunks && rc == 0; k++) {
        const size_t i0 = bounds[k], cn = bounds[k + 1] - i0;
        rc = upload((uint8_t*)d_scalars + i0 * 32, (const uint8_t*)h_scalars + i0 * 32, cn * 32, copy, pin_s);
        if (rc == 0) rc = upload((uint8_t*)d_points + i0 * stride, (const uint8_t*)h_points + i0 * stride, cn * stride, copy, pin_p);
        if (rc == 0) rc = (int)cudaEventRecord(ev[k], copy);
        if (rc == 0) rc = (int)cudaStreamWaitEvent(stream, ev[k], 0);
        uint32_t* dst = chunks > 1 ? d_parts + (size_t)k * plan.nwin * 48 : (uint32_t*)d_window_sums;
        if (rc == 0) rc = msm_window_sums_device(dst, d_flags, plan, (const uint8_t*)d_points + i0 * stride, stride,
                                                 (const uint8_t*)d_scalars + i0 * 32, cn, stream);
    }
    if (rc == 0 && chunks > 1) rc = xyzz_sum_ranks_device((uint32_t*)d_window_sums, d_parts, chunks, plan.nwin, stream);
    if (rc != 0 && copy) cudaStreamSynchronize(copy);              // a failed call must not leave copies writing into freed buffers
    if (d_parts) cudaFreeAsync(d_parts, stream);
    if (d_points) cudaFreeAsync(d_points, stream);
    if (d_scalars) cudaFreeAsync(d_scalars, stream);
    if (own_flags) cudaFreeAsync(own_flags, stream);
    for (auto& e : ev) if (e) cudaEventDestroy(e);
    return rc;
}

int snarkvm_b200_xyzz_sum_ranks_device(void* d_out, const void* d_in, int nranks, int count, void* stream) {
    if (nranks < 1 || count < 1) return (int)cudaErrorInvalidValue;
    return xyzz_sum_ranks_device((uint32_t*)d_out, (const uint32_t*)d_in, nranks, count, (cudaStream_t)stream);
}

int snarkvm_b200_msm_finish(void* out144, const void* h_window_sums, int nwin, int c) {
    if (!out144 || !h_window_sums || nwin < 1 || c < 0) return (int)cudaErrorInvalidValue;
    std::vector<host::Xyzz> sums((size_t)nwin);
    memcpy(sums.data(), h_window_sums, (size_t)nwin * 192);
    host::Xyzz total = host::horner_windows(sums.data(), nwin, c);
    host::xyzz_to_normalised_projective(total, (uint64_t*)out144);
    return 0;
}

int snarkvm_b200_msm_scratch_stats(size_t* limit_bytes, size_t* in_use_bytes, size_t* peak_bytes) {
    return msm_scratch_stats(limit_bytes, in_use_bytes, peak_bytes);
}
int snarkvm_b200_msm_set_scratch_limit(size_t limit_bytes) { return msm_set_scratch_limit(limit_bytes); }

// KZG10::commit core: the Montgomery → canonical conversion (to_bigint, kzg10/mod.rs:469-474) happens inside the digit kernel
int snarkvm_b200_kzg_commit_device(void* out144, const void* d_powers, size_t stride, const void* d_coeffs_mont,
                                   size_t ncoeffs, void* stream_v) {
    if (!out144) return (int)cudaErrorInvalidValue;
    return msm_device_impl(out144, d_powers, ncoeffs, d_coeffs_mont, stride, 1, (cudaStream_t)stream_v);
}

// Precomputed tables for a fixed base set (an SRS): handle = {table, n, plan}.  One-time cost: (nwin−1)·c doublings and
// nwin−1 inversions per point; memory npoints·nwin·128 B.
int snarkvm_b200_msm_precompute_device(void** handle_out, const void* d_points, size_t npoints, size_t stride, void* stream_v) {
    if (!handle_out || !d_points || npoints == 0 || stride < 104 || (stride & 7)) return (int)cudaErrorInvalidValue;
    cudaStream_t stream = (cudaStream_t)stream_v;
    MsmPlan plan = msm_make_plan_precomputed(npoints);
    if (npoints * (size_t)plan.nwin >= (1ull << 31)) return (int)cudaErrorInvalidValue;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    uint32_t* table = nullptr;
    if ((e = cudaMalloc(&table, npoints * (size_t)plan.nwin * 128)) != cudaSuccess) return (int)e;
    int rc = msm_precompute_tables_device(table, plan, d_points, stride, npoints, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc != 0) { cudaFree(table); return rc; }
    *handle_out = new PrecomputedBases{table, npoints, plan, dev};
    return 0;
}

int snarkvm_b200_msm_precomputed_free(void* handle) {
    if (!handle) return (int)cudaErrorInvalidValue;
    PrecomputedBases* h = (PrecomputedBases*)handle;
    cudaError_t e = cudaFree(h->table);
    delete h;
    return (int)e;
}

int snarkvm_b200_msm_precomputed_info(const void* handle, size_t* npoints, int* c, int* nwin, size_t* table_bytes) {
    if (!handle) return (int)cudaErrorInvalidValue;
    const PrecomputedBases* h = (const PrecomputedBases*)handle;
    if (npoints) *npoints = h->n;
    if (c) *c = h->plan.c;
    if (nwin) *nwin = h->plan.nwin;
    if (table_bytes) *table_bytes = h->n * (size_t)h->plan.nwin * 128;
    return 0;
}

static int msm_precomputed_impl(void* out144, const void* handle, const void* d_scalars, size_t nscalars, int mont, cudaStream_t stream) {
    if (!out144 || !handle) return (int)cudaErrorInvalidValue;
    const PrecomputedBases* h = (const PrecomputedBases*)handle;
    if (nscalars > h->n) return (int)cudaErrorInvalidValue;
    if (nscalars == 0) { write_infinity(out144); return 0; }
    if (!d_scalars) return (int)cudaErrorInvalidValue;
    MsmSegment sg{d_scalars, nscalars, 0u, 0u, mont};
    return msm_jobs_impl(out144, h->plan, nullptr, 0, h->table, h->n, &sg, 1, 1, stream);
}
int snarkvm_b200_msm_precomputed_device(void* out144, const void* handle, const void* d_scalars, size_t nscalars, void* stream_v) {
    return msm_precomputed_impl(out144, handle, d_scalars, nscalars, 0, (cudaStream_t)stream_v);
}
int snarkvm_b200_kzg_commit_precomputed_device(void* out144, const void* handle, const void* d_coeffs_mont, size_t ncoeffs, void* stream_v) {
    return msm_precomputed_impl(out144, handle, d_coeffs_mont, ncoeffs, 1, (cudaStream_t)stream_v);
}
// all commitments of a round over the tables of the resident powers: one pass, one bucket set per polynomial
int snarkvm_b200_kzg_commit_batch_precomputed_device(void* out144s, const void* handle, const void* const* d_coeffs_mont, const size_t* ncoeffs,
                                                     size_t count, void* stream_v) {
    if (count == 0) return 0;
    if (!out144s || !handle || !d_coeffs_mont || !ncoeffs) return (int)cudaErrorInvalidValue;
    const PrecomputedBases* h = (const PrecomputedBases*)handle;
    std::vector<MsmSegment> segs;
    std::vector<size_t> job_of(count, (size_t)-1);
    uint32_t njobs = 0;
    for (size_t i = 0; i < count; i++) {
        if (ncoeffs[i] > h->n) return (int)cudaErrorInvalidValue;
        if (ncoeffs[i] == 0) { write_infinity((uint8_t*)out144s + i * 144); continue; }
        job_of[i] = njobs;
        segs.push_back(MsmSegment{d_coeffs_mont[i], ncoeffs[i], 0u, njobs++, 1});
    }
    if (njobs == 0) return 0;
    std::vector<uint8_t> outs((size_t)njobs * 144);
    int rc = msm_jobs_impl(outs.data(), h->plan, nullptr, 0, h->table, h->n, segs.data(), (int)segs.size(), (int)njobs, (cudaStream_t)stream_v);
    if (rc != 0) return rc;
    for (size_t i = 0; i < count; i++) if (job_of[i] != (size_t)-1) memcpy((uint8_t*)out144s + i * 144, outs.data() + job_of[i] * 144, 144);
    return 0;
}

// KZG10::commit with a hiding bound (polycommit/kzg10/mod.rs:98-156): commitment to the plaintext polynomial against
// powers_of_beta_g plus the commitment to the blinding polynomial against powers_of_beta_times_gamma_g.  The caller samples the
// blinding polynomial (KZGRandomness::rand, :129-140) and passes its Montgomery coefficients; nblinding = 0 is the non-hiding
// commit.  Zero coefficients contribute nothing, so skip_leading_zeros_and_convert_to_bigints (:455-467) needs no special path.
// Both MSMs run as ONE pass: the blinding terms are a second scalar segment of the same job whose digits point at the gamma
// powers appended to the dense base array, so they land in the same buckets and the sum comes out of one Horner fold.
int snarkvm_b200_kzg_commit_hiding_device(void* out144, const void* d_powers, size_t stride, const void* d_coeffs_mont, size_t ncoeffs,
                                          const void* d_gamma_powers, const void* d_blinding_mont, size_t nblinding, void* stream) {
    if (!out144) return (int)cudaErrorInvalidValue;
    const void* c1[1] = {d_coeffs_mont};
    const void* c2[1] = {d_blinding_mont};
    return msm_batch_impl(out144, d_powers, stride, c1, &ncoeffs, 1, 1, d_gamma_powers, c2, &nblinding, (cudaStream_t)stream);
}

// All commitments of one prover round share powers_of_beta_g (sonic_pc/mod.rs:177-257): count polynomials, ONE pass over the
// resident bases.  out144s: count × 144 B of HOST memory.
int snarkvm_b200_kzg_commit_batch_device(void* out144s, const void* d_powers, size_t stride, const void* const* d_coeffs_mont,
                                         const size_t* ncoeffs, size_t count, void* stream) {
    return msm_batch_impl(out144s, d_powers, stride, d_coeffs_mont, ncoeffs, count, 1, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}
// ... with hiding: polynomial i also gets Σ blinding_i[j]·gamma_powers[j] (nblinding[i] may be 0)
int snarkvm_b200_kzg_commit_batch_hiding_device(void* out144s, const void* d_powers, size_t stride, const void* const* d_coeffs_mont,
                                                const size_t* ncoeffs, const void* d_gamma_powers, const void* const* d_blinding_mont,
                                                const size_t* nblinding, size_t count, void* stream) {
    return msm_batch_impl(out144s, d_powers, stride, d_coeffs_mont, ncoeffs, count, 1, d_gamma_powers, d_blinding_mont, nblinding, (cudaStream_t)stream);
}

// SonicKZG10::commit for all polynomials of a round (sonic_pc/mod.rs:177-257) in ONE msm_core pass.  Polynomial i is committed
// against the base array the reference would pick for it — ck.powers() (d_bases[i] = the powers), ck.shifted_powers_of_beta_g(bound)
// (the powers advanced by max_degree − bound points, mod.rs:229-233, data_structures.rs:310-331) or a Lagrange basis
// (mod.rs:215-227) — plus, when hiding, Σ_j blinding_i[j]·gamma_i[j] (kzg10/mod.rs:129-150).  The slices may overlap (shifted powers
// are suffixes of one SRS): they are merged into disjoint arrays and every scalar vector becomes a segment with its offset.
int snarkvm_b200_sonic_commit_batch_device(void* out144s, size_t stride, const void* const* d_bases, const void* const* d_coeffs_mont,
                                           const size_t* ncoeffs, const void* const* d_gamma_bases, const void* const* d_blinding_mont,
                                           const size_t* nblinding, size_t count, void* stream_v) {
    cudaStream_t stream = (cudaStream_t)stream_v;
    if (count == 0) return 0;
    if (!out144s || !d_bases || !d_coeffs_mont || !ncoeffs || stride < 104 || (stride & 7)) return (int)cudaErrorInvalidValue;
    struct Use { const uint8_t* p; size_t n; const void* scal; uint32_t job; };
    std::vector<Use> uses;
    std::vector<size_t> job_of(count, (size_t)-1), job_n;
    uint32_t njobs = 0;
    size_t total_n = 0;
    for (size_t i = 0; i < count; i++) {
        const size_t n1 = ncoeffs[i], n2 = (d_blinding_mont && nblinding) ? nblinding[i] : 0;
        if (n1 == 0 && n2 == 0) { write_infinity((uint8_t*)out144s + i * 144); continue; }
        if ((n1 && (!d_bases[i] || !d_coeffs_mont[i])) || (n2 && (!d_gamma_bases || !d_gamma_bases[i] || !d_blinding_mont[i]))) return (int)cudaErrorInvalidValue;
        job_of[i] = njobs;
        if (n1) uses.push_back(Use{(const uint8_t*)d_bases[i], n1, d_coeffs_mont[i], njobs});
        if (n2) uses.push_back(Use{(const uint8_t*)d_gamma_bases[i], n2, d_blinding_mont[i], njobs});
        job_n.push_back(n1 + n2);
        total_n += n1 + n2;
        njobs++;
    }
    if (njobs == 0) return 0;
    // merge the base slices into disjoint arrays: sort by address, join a slice that starts inside (or right at the end of) the
    // running array on the same stride grid
    std::vector<size_t> order(uses.size());
    for (size_t k = 0; k < order.size(); k++) order[k] = k;
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return uses[a].p < uses[b].p; });
    std::vector<MsmBases> arrays;
    std::vector<size_t> array_first;                       // index of the array's first point in the concatenation
    std::vector<uint32_t> base0(uses.size(), 0);
    size_t concat = 0;
    for (size_t k : order) {
        const Use& u = uses[k];
        bool joined = false;
        if (!arrays.empty()) {
            MsmBases& a = arrays.back();
            const uint8_t* a0 = (const uint8_t*)a.d_points;
            const size_t off = (size_t)(u.p - a0);
            if (off <= a.n * stride && off % stride == 0) {
                const size_t first = off / stride;
                if (first + u.n > a.n) { concat += first + u.n - a.n; a.n = first + u.n; }
                base0[k] = (uint32_t)(array_first.back() + first);
                joined = true;
            } else if (off < a.n * stride) return (int)cudaErrorInvalidValue;      // overlapping arrays on different grids
        }
        if (!joined) {
            array_first.push_back(concat);
            arrays.push_back(MsmBases{u.p, stride, u.n});
            base0[k] = (uint32_t)concat;
            concat += u.n;
        }
        if (concat >= (1ull << 31)) return (int)cudaErrorInvalidValue;
    }
    std::vector<MsmSegment> segs;
    for (size_t k = 0; k < uses.size(); k++) segs.push_back(MsmSegment{uses[k].scal, uses[k].n, base0[k], uses[k].job, 1});
    size_t job_max = 1;
    for (size_t v : job_n) if (v > job_max) job_max = v;
    MsmPlan plan = msm_make_plan_batch(job_max, total_n);
    std::vector<uint8_t> outs((size_t)njobs * 144);
    int rc = msm_jobs_impl(outs.data(), plan, arrays.data(), (int)arrays.size(), nullptr, 0, segs.data(), (int)segs.size(), (int)njobs, stream);
    if (rc != 0) return rc;
    for (size_t i = 0; i < count; i++) if (job_of[i] != (size_t)-1) memcpy((uint8_t*)out144s + i * 144, outs.data() + job_of[i] * 144, 144);
    return 0;
}

// VariableBase::msm for G2 (Affine<G2> images: x.c0 x.c1 y.c0 y.c1 infinity, stride ≥ 200; canonical scalars) — the curves the
// reference routes to standard::msm (msm/variable_base/mod.rs:44-47).  out288: HOST memory, the normalised projective image
// (x, y, 1) or (0, 1, 0) over Fq2.
static int msm_g2_impl(void* out288, const void* d_points, size_t npoints, const void* d_scalars, size_t stride, cudaStream_t stream) {
    if (!out288) return (int)cudaErrorInvalidValue;
    if (npoints == 0) { host::Xyzz2 inf = host::xyzz_inf_t<host::Fq2>(); host::xyzz_to_normalised_projective(inf, (uint64_t*)out288); return 0; }
    if (!d_points || !d_scalars || stride < 200 || (stride & 7)) return (int)cudaErrorInvalidValue;
    MsmPlan plan = msm_make_plan(npoints);
    const size_t nw = (size_t)plan.nwin;
    uint32_t* d_buf = nullptr;
    cudaError_t e = pool_alloc(&d_buf, nw * 384 + 256, stream);
    if (e != cudaSuccess) return (int)e;
    uint32_t* d_flags = d_buf + nw * 96;
    int rc = (int)cudaMemsetAsync(d_flags, 0, 256, stream);
    if (rc == 0) rc = msm_g2_window_sums_device(d_buf, d_flags, plan, d_points, stride, d_scalars, npoints, 0, stream);
    std::vector<host::Xyzz2> sums(nw + 1);
    if (rc == 0) rc = (int)cudaMemcpyAsync(sums.data(), d_buf, nw * 384 + 256, cudaMemcpyDeviceToHost, stream);
    cudaFreeAsync(d_buf, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc != 0) return rc;
    uint32_t flags = 0;
    memcpy(&flags, sums.data() + nw, 4);
    if (flags & 1u) return (int)cudaErrorInvalidValue;
    host::Xyzz2 total = host::horner_windows(sums.data(), plan.nwin, plan.c);
    host::xyzz_to_normalised_projective(total, (uint64_t*)out288);
    return 0;
}
int snarkvm_b200_msm_g2_device(void* out288, const void* d_points, size_t npoints, const void* d_scalars, size_t stride, void* stream) {
    return msm_g2_impl(out288, d_points, npoints, d_scalars, stride, (cudaStream_t)stream);
}
// host-buffer form with the drop-in symbol's contract (outputs untouched on failure, error struct by value)
snarkvm_error_t snarkvm_b200_msm_g2(void* out, const void* points, size_t npoints, const void* scalars, size_t ffi_affine_sz) {
    if (!out) return make_error((int)cudaErrorInvalidValue);
    uint64_t result[36];
    if (npoints == 0) { int rc0 = msm_g2_impl(result, nullptr, 0, nullptr, 200, nullptr); if (rc0 == 0) memcpy(out, result, 288); return make_error(rc0); }
    if (!points || !scalars || ffi_affine_sz < 200 || (ffi_affine_sz & 7)) return make_error((int)cudaErrorInvalidValue);
    cudaStream_t stream;
    int rc = thread_stream(&stream);
    if (rc) return make_error(rc);
    void *d_points = nullptr, *d_scalars = nullptr;
    rc = (int)pool_alloc(&d_points, npoints * ffi_affine_sz, stream);
    if (rc == 0) rc = (int)pool_alloc(&d_scalars, npoints * 32, stream);
    if (rc == 0) rc = upload(d_scalars, scalars, npoints * 32, stream, host_is_pinned(scalars));
    if (rc == 0) rc = upload(d_points, points, npoints * ffi_affine_sz, stream, host_is_pinned(points));
    if (rc == 0) rc = msm_g2_impl(result, d_points, npoints, d_scalars, ffi_affine_sz, stream);
    if (d_points) cudaFreeAsync(d_points, stream);
    if (d_scalars) cudaFreeAsync(d_scalars, stream);
    int rs = (int)cudaStreamSynchronize(stream);
    if (rc == 0 && rs == 0) memcpy(out, result, 288);
    return make_error(rc ? rc : rs);
}
int snarkvm_b200_generate_bases_g2_device(void* d_points, size_t npoints, size_t stride, uint64_t seed, void* stream) {
    return msm_generate_bases_g2_device(d_points, npoints, stride, seed, (cudaStream_t)stream);
}

int snarkvm_b200_g1_ntt_device(void* d_out, size_t out_stride, const void* d_in, size_t in_stride, uint32_t lg, int direction, void* stream) {
    return g1_ntt_device(d_out, out_stride, d_in, in_stride, lg, direction, (cudaStream_t)stream);
}
int snarkvm_b200_fr_batch_inversion_and_mul_device(void* d_v, size_t n, const void* coeff_mont_host, void* stream) {
    return fr_batch_inversion_and_mul_device(d_v, n, coeff_mont_host, (cudaStream_t)stream);
}
int snarkvm_b200_poly_divide_by_vanishing_device(void* d_q, void* d_r, const void* d_p, size_t m, size_t n, void* stream) {
    return poly_divide_by_vanishing_device(d_q, d_r, d_p, m, n, (cudaStream_t)stream);
}
int snarkvm_b200_poly_divide_by_linear_device(void* d_q, const void* d_p, size_t m, const void* point_mont_host, void* stream) {
    return poly_divide_by_linear_device(d_q, d_p, m, point_mont_host, (cudaStream_t)stream);
}
int snarkvm_b200_sparse_matvec_device(void* d_out, const void* d_row_ptr, const void* d_cols, const void* d_vals, size_t nrows, const void* d_x,
                                      size_t nvars, void* stream) {
    return sparse_matvec_device(d_out, d_row_ptr, d_cols, d_vals, nrows, d_x, nvars, (cudaStream_t)stream);
}
int snarkvm_b200_fr_vec_op_device(void* d_out, const void* d_a, const void* d_b, size_t n, int op, void* stream) {
    return fr_vec_op_device(d_out, d_a, d_b, n, op, (cudaStream_t)stream);
}
int snarkvm_b200_fr_vec_scalar_op_device(void* d_out, const void* d_a, const void* scalar_mont_host, size_t n, int op, void* stream) {
    return fr_vec_scalar_op_device(d_out, d_a, scalar_mont_host, n, op, (cudaStream_t)stream);
}
int snarkvm_b200_domain_elements_device(void* d_out, uint32_t lg, void* stream) {
    return domain_elements_device(d_out, lg, (cudaStream_t)stream);
}
int snarkvm_b200_index_arithmetize_device(int mode, const void* const* d_row_ptr, const void* const* d_cols, const void* const* d_vals,
                                          const size_t* nnz, const uint32_t* lg_k, size_t num_constraints, size_t num_variables,
                                          size_t num_public, void* const* d_io, void* sums_mont_host, void* stream) {
    return index_arithmetize_device(mode, d_row_ptr, d_cols, d_vals, nnz, lg_k, num_constraints, num_variables, num_public, d_io,
                                    sums_mont_host, (cudaStream_t)stream);
}
int snarkvm_b200_poly_evaluate_device(void* out_mont_host, const void* d_coeffs, size_t m, const void* point_mont_host, void* stream) {
    return poly_evaluate_device(out_mont_host, d_coeffs, m, point_mont_host, (cudaStream_t)stream);
}

int snarkvm_b200_fr_from_mont_device(void* d_out, const void* d_in, size_t n, void* stream) {
    return fr_from_mont_device(d_out, d_in, n, (cudaStream_t)stream);
}
int snarkvm_b200_fr_to_mont_device(void* d_out, const void* d_in, size_t n, void* stream) {
    return fr_to_mont_device(d_out, d_in, n, (cudaStream_t)stream);
}

int snarkvm_b200_srs_decode_device(void* d_out, size_t stride, const void* d_in96, size_t npoints, uint32_t* d_invalid, void* stream) {
    if (!d_out || !d_in96 || !d_invalid) return (int)cudaErrorInvalidValue;
    return srs_decode_device(d_out, stride, d_in96, npoints, d_invalid, (cudaStream_t)stream);
}

int snarkvm_b200_register_bases(const void* host_points, size_t npoints, size_t stride) {
    if (!host_points || npoints == 0 || stride < 104 || (stride & 7)) return (int)cudaErrorInvalidValue;
    auto rb = std::make_shared<ResidentBases>();
    cudaError_t e = cudaGetDevice(&rb->device);
    if (e != cudaSuccess) return (int)e;
    if ((e = cudaMalloc(&rb->d_ptr, npoints * stride)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(rb->d_ptr, host_points, npoints * stride, cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    rb->npoints = npoints; rb->stride = stride;
    memcpy(rb->head, host_points, 104);
    memcpy(rb->tail, (const uint8_t*)host_points + (npoints - 1) * stride, 104);
    std::lock_guard<std::mutex> lock(g_bases_mu);
    g_bases[host_points] = rb;                                  // a previous registration of this address is released by its last user
    return 0;
}
int snarkvm_b200_unregister_bases(const void* host_points) {
    std::shared_ptr<ResidentBases> old;
    {
        std::lock_guard<std::mutex> lock(g_bases_mu);
        auto it = g_bases.find(host_points);
        if (it == g_bases.end()) return (int)cudaErrorInvalidValue;
        old = it->second;
        g_bases.erase(it);
    }
    return 0;                                                    // `old` frees the device memory here unless a call still holds it
}
// register + build the fixed-base tables (snarkvm_b200_msm_precompute_device) from the uploaded copy: later snarkvm_msm calls
// on this slice run over the tables (one bucket set, wider windows).  Costs npoints·nwin·128 B of HBM and seconds of set-up.
int snarkvm_b200_register_bases_precomputed(const void* host_points, size_t npoints, size_t stride) {
    int rc = snarkvm_b200_register_bases(host_points, npoints, stride);
    if (rc != 0) return rc;
    std::shared_ptr<ResidentBases> rb;
    {
        std::lock_guard<std::mutex> lock(g_bases_mu);
        auto it = g_bases.find(host_points);
        if (it == g_bases.end()) return (int)cudaErrorInvalidValue;
        rb = it->second;
    }
    cudaStream_t stream;
    if ((rc = thread_stream(&stream)) != 0) return rc;
    void* tables = nullptr;
    rc = snarkvm_b200_msm_precompute_device(&tables, rb->d_ptr, npoints, stride, stream);
    if (rc != 0) { snarkvm_b200_unregister_bases(host_points); return rc; }
    // the entry a concurrent call may already hold just gains its tables (atomic pointer); both forms stay valid until the
    // last holder lets go
    PrecomputedBases* expected = nullptr;
    if (!rb->tables.compare_exchange_strong(expected, (PrecomputedBases*)tables)) { snarkvm_b200_msm_precomputed_free(tables); }
    return 0;
}

// device self-test of the warp-cooperative field arithmetic: returns 0 and *mismatches = number of failing warps
// Host-only self-test of the staging copies (copy pool + non-temporal stores, hostcopy.cpp): contiguous copies and column-range
// copies of random sizes and alignments against memcpy.  Needs no GPU; *mismatches receives the number of differing cases.
int snarkvm_b200_selftest_host_copy(size_t max_bytes, uint64_t seed, uint32_t* mismatches) {
    if (!mismatches || max_bytes < 4096) return (int)cudaErrorInvalidValue;
    std::vector<uint8_t> src(max_bytes + 256), dst(max_bytes + 256), ref(max_bytes + 256);
    uint64_t x = seed | 1;
    auto rnd = [&x]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
    for (size_t i = 0; i < src.size(); i++) src[i] = (uint8_t)rnd();
    uint32_t bad = 0;
    const size_t sizes[] = {0, 1, 31, 32, 33, 4095, 4096, 4097, 65537, ((size_t)2 << 20) - 1, ((size_t)2 << 20) + 5, max_bytes};
    for (size_t n : sizes) {
        if (n > max_bytes) continue;
        for (int rep = 0; rep < 3; rep++) {
            const size_t so = rnd() % 64, doff = rnd() % 64;
            memset(dst.data(), 0xA5, dst.size()); memset(ref.data(), 0xA5, ref.size());
            memcpy(ref.data() + doff, src.data() + so, n);
            CopyPool::get().parallel_memcpy(dst.data() + doff, src.data() + so, n);
            if (memcmp(dst.data(), ref.data(), dst.size()) != 0) bad++;
        }
    }
    for (int rep = 0; rep < 6; rep++) {                             // rows: a column range of a row-major matrix
        const size_t width = 32 * (1 + rnd() % 700) + (rep & 1 ? 8 : 0), rows = 1 + rnd() % 97;
        const size_t spitch = width + 32 * (rnd() % 9), dpitch = width + 8 * (rnd() % 5);
        if (rows * spitch > max_bytes || rows * dpitch > max_bytes) continue;
        memset(dst.data(), 0x5A, dst.size()); memset(ref.data(), 0x5A, ref.size());
        for (size_t r = 0; r < rows; r++) memcpy(ref.data() + r * dpitch, src.data() + r * spitch, width);
        CopyPool::get().parallel_rows(dst.data(), dpitch, src.data(), spitch, width, rows);
        if (memcmp(dst.data(), ref.data(), dst.size()) != 0) bad++;
    }
    *mismatches = bad;
    return 0;
}

int snarkvm_b200_selftest_coop(uint32_t nwarps, uint64_t seed, uint32_t* mismatches, void* stream_v) {
    if (!mismatches || nwarps == 0) return (int)cudaErrorInvalidValue;
    cudaStream_t stream = (cudaStream_t)stream_v;
    uint32_t* d = nullptr;
    int rc = (int)pool_alloc(&d, 256, stream);
    if (rc == 0) rc = selftest_coop_device(nwarps, seed, d, stream);
    if (rc == 0) rc = (int)cudaMemcpyAsync(mismatches, d, 4, cudaMemcpyDeviceToHost, stream);
    if (d) cudaFreeAsync(d, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    return rc;
}

int snarkvm_b200_profile_enable(int on) { prof_enable(on != 0); return 0; }
int snarkvm_b200_profile_collect(int kind, double* total_ms, uint64_t* count) { return prof_collect(kind, total_ms, count); }

int snarkvm_b200_generate_bases_device(void* d_points, size_t npoints, size_t stride, uint64_t seed, void* stream) {
    return msm_generate_bases_device(d_points, npoints, stride, seed, (cudaStream_t)stream);
}

// P_i = s_i·G for n canonical scalars (32 B each) in HBM → the reference Affine layout; test/bench set-up of an SRS with a known trapdoor
int snarkvm_b200_generator_mul_device(void* d_points, size_t stride, const void* d_scalars, size_t npoints, void* stream) {
    if (npoints && (!d_points || !d_scalars)) return (int)cudaErrorInvalidValue;
    return msm_generator_mul_device(d_points, npoints, stride, d_scalars, (cudaStream_t)stream);
}

}  // extern "C"
