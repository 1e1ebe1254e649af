// runtime.cu -- host runtime and C ABI of libb200df.so (see include/b200df.h for the contract).
//
// One bdf_ctx per GPU (one process per GPU).  Three non-blocking streams: h2d (uploads), compute (all
// kernels, all stream-ordered allocations), d2h (downloads).  Columns are device-resident lists of Arrow
// chunks carved out of two arenas (values, validity).  Chunks become ready in *groups*; every group has
// an event, so the kernels of group g run while group g+1 is still crossing PCIe and group g-1 is
// already on its way back.  When all inputs are already resident an operator is ONE batched launch over
// every chunk of the column.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <new>
#include <deque>
#include <limits>
#include <sys/mman.h>
#include <thread>

#include "runtime.cuh"

// ---------------------------------------------------------------------------------------------------
// errors

thread_local std::string g_err;

int fail(int status, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return status;
}

namespace bdf {
int set_error(int status, const char* msg) {   // for the host-only translation units of the library (ipc.cu)
    g_err = msg;
    return status;
}
}  // namespace bdf

// Set by the communicator layer (comm.cu reports NCCL failures as text + cudaErrorUnknown): turns the next
// fail_cuda into BDF_NCCL.
static thread_local std::string g_nccl_err;
static int fail_cuda(cudaError_t e, const char* what) {
    if (!g_nccl_err.empty()) {
        const std::string m = g_nccl_err;
        g_nccl_err.clear();
        return fail(BDF_NCCL, "%s: %s", what, m.c_str());
    }
    return fail(cuda_status(e), "%s failed: %s", what, cudaGetErrorString(e));
}

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------------
// objects

// Persistent host threads for the staged copies of PAGEABLE buffers (Arrow MutableBuffers, a mapped IPC file): a copy
// is cut into 512 KiB jobs that the workers and the calling thread pull until it is done.  (Spawning threads per 8 MiB
// slot, the first version, stopped scaling at 4 threads because the spawn/join cost was comparable to the copy.)
class CopyPool {
  public:
    explicit CopyPool(int workers) {
        for (int i = 0; i < workers; i++) th_.emplace_back([this] { work(); });
    }
    ~CopyPool() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; }
        cv_work_.notify_all();
        for (auto& t : th_) t.join();
    }
    int workers() const { return (int)th_.size(); }
    // populate: the destination may be memory nobody has touched yet (a fresh Arrow MutableBuffer): every job first asks
    // the kernel for its pages in ONE call (MADV_POPULATE_WRITE) instead of taking a fault per 4 KiB page inside the
    // copy -- 18 -> 31 GB/s into fresh memory with 8 threads (benchmarks/staging_probe2.cu); a no-op for resident pages.
    static void job_copy(char* dst, const char* src, size_t n, bool populate) {
        if (populate) {
            const uintptr_t a = ((uintptr_t)dst + 4095) & ~(uintptr_t)4095, b = ((uintptr_t)dst + n) & ~(uintptr_t)4095;
            if (b > a) madvise((void*)a, b - a, 23 /* MADV_POPULATE_WRITE (Linux 5.14+); an error only means: fault as usual */);
        }
        memcpy(dst, src, n);
    }
    void copy(char* dst, const char* src, size_t n, bool populate = false) {
        constexpr size_t kJob = (size_t)512 << 10;
        if (th_.empty() || n < 2 * kJob) { job_copy(dst, src, n, populate); return; }
        std::unique_lock<std::mutex> lk(m_);
        populate_ = populate;
        dst_ = dst; src_ = src; n_ = n; next_ = 0; jobs_ = (n + kJob - 1) / kJob; done_ = 0;
        lk.unlock();
        cv_work_.notify_all();
        lk.lock();
        while (next_ < jobs_) {   // the caller works too
            const size_t j = next_++;
            lk.unlock();
            job_copy(dst + j * kJob, src + j * kJob, std::min(kJob, n - j * kJob), populate);
            lk.lock();
            done_++;
        }
        cv_done_.wait(lk, [this] { return done_ == jobs_; });
        jobs_ = 0; next_ = 0; done_ = 0;
    }

  private:
    void work() {
        constexpr size_t kJob = (size_t)512 << 10;
        std::unique_lock<std::mutex> lk(m_);
        for (;;) {
            cv_work_.wait(lk, [this] { return stop_ || next_ < jobs_; });
            if (stop_) return;
            const size_t j = next_++;
            char* d = dst_; const char* s = src_; const size_t n = n_;
            const bool pop = populate_;
            lk.unlock();
            job_copy(d + j * kJob, s + j * kJob, std::min(kJob, n - j * kJob), pop);
            lk.lock();
            if (++done_ == jobs_) cv_done_.notify_all();
        }
    }
    std::mutex m_;
    std::condition_variable cv_work_, cv_done_;
    std::vector<std::thread> th_;
    char* dst_ = nullptr; const char* src_ = nullptr;
    size_t n_ = 0, next_ = 0, jobs_ = 0, done_ = 0;
    bool stop_ = false, populate_ = false;
};

bdf_ctx::bdf_ctx() = default;
bdf_ctx::~bdf_ctx() = default;

static constexpr int kAggSlots = 4096;

// ---------------------------------------------------------------------------------------------------
// small helpers

static inline size_t value_bytes(int dtype, int64_t len, int bit_off) {
    return dtype == kBool ? (size_t)((len + bit_off + 7) / 8) : (size_t)len * dtype_width(dtype);
}

// The first check of every entry that takes columns: a context, and columns that context made.  Reads only what is fixed
// when a column is made, so it runs before the context's lock is taken.
static int check_cols(const bdf_ctx* c, int64_t n, const bdf_col* const* cols) {
    if (!c) return fail(BDF_INVALID, "null context");
    for (int64_t i = 0; i < n; i++) {
        if (!cols[i]) return fail(BDF_INVALID, "null argument");
        if (cols[i]->owner != c) return fail(BDF_INVALID, "a column may only be passed to the context that made it");
    }
    return BDF_OK;
}
static int check_cols(const bdf_ctx* c, std::initializer_list<const bdf_col*> cols) { return check_cols(c, (int64_t)cols.size(), cols.begin()); }

// Host chunks: a count, and views with sane lengths and offsets.
static int check_views(int64_t n, const bdf_view* v) {
    if (n < 0 || (n && !v)) return fail(BDF_INVALID, "bad arguments");
    for (int64_t i = 0; i < n; i++)
        if (v[i].len < 0 || v[i].offset < 0 || (v[i].len > 0 && !v[i].values)) return fail(BDF_INVALID, "bad view %lld", (long long)i);
    return BDF_OK;
}

// Descriptor ring: host writes descriptors into pinned memory, one async copy moves them to the same offset
// of the device ring, kernels read them there.  No per-call allocation.
static int ring_alloc(bdf_ctx* c, size_t bytes, void** host, void** dev) {
    bytes = align_up(std::max<size_t>(bytes, 1), 256);
    if (bytes > c->ring_cap) return fail(BDF_OOM, "descriptor ring too small for %zu bytes", bytes);
    if (c->ring_head + bytes > c->ring_cap) {
        CK(cudaStreamSynchronize(c->s_desc));
        CK(cudaStreamSynchronize(c->s_compute));  // everything that read the ring has finished
        c->ring_head = 0;
    }
    *host = c->ring + c->ring_head;
    *dev = c->dring + c->ring_head;
    c->ring_head += bytes;
    return BDF_OK;
}

static cudaError_t ev_get(bdf_ctx* c, cudaEvent_t* ev) {
    if (!c->ev_pool.empty()) { *ev = c->ev_pool.back(); c->ev_pool.pop_back(); return cudaSuccess; }
    return cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
}
static void ev_put(bdf_ctx* c, cudaEvent_t ev) { if (ev) c->ev_pool.push_back(ev); }

// Copy descriptors host ring -> device ring on the descriptor stream and make the compute stream wait for
// them: the copy itself runs while the previous kernel is still busy.
static cudaError_t desc_upload(bdf_ctx* c, void* dev, const void* host, size_t bytes) {
    if (!bytes) return cudaSuccess;
    cudaError_t e = cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, c->s_desc);
    cudaEvent_t ev = nullptr;
    if (e == cudaSuccess) e = ev_get(c, &ev);
    if (e == cudaSuccess) e = cudaEventRecord(ev, c->s_desc);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c->s_compute, ev, 0);
    ev_put(c, ev);  // the wait has captured this record; re-recording later does not affect it
    return e;
}

struct LaunchTimer {  // brackets one launch with events when profiling is on
    bdf_ctx* c;
    ProfEntry e{};
    bool on;
    LaunchTimer(bdf_ctx* ctx, int kernel, int dtype, int64_t rows, int64_t bytes) : c(ctx), on(ctx->profiling) {
        c->launches++;
        if (!on) return;
        e.rec.kernel = kernel; e.rec.dtype = dtype; e.rec.rows = rows; e.rec.bytes = bytes; e.rec.ms = 0.f;
        // timing events come from a pool (bdf_profile_read returns them): creating two events per launch cost more host time
        // than the launch itself and showed up as a few percent of the headline step at 8 GPUs
        auto take = [&](cudaEvent_t* ev) {
            if (!c->prof_pool.empty()) { *ev = c->prof_pool.back(); c->prof_pool.pop_back(); } else cudaEventCreate(ev);
        };
        take(&e.e0); take(&e.e1);
        cudaEventRecord(e.e0, c->s_compute);
    }
    ~LaunchTimer() {
        if (!on) return;
        cudaEventRecord(e.e1, c->s_compute);
        c->prof.push_back(e);
    }
};

static void col_destroy_host(bdf_ctx* c, bdf_col* col) {
    for (auto& g : col->groups) ev_put(c, g.ev);
    delete col;
}

// Free device memory of a column in stream order on the compute stream.
static void col_release(bdf_ctx* c, bdf_col* col) {
    if (!col) return;
    if (col->dl_tmp) { cudaStreamSynchronize(c->s_d2h); col_release(c, col->dl_tmp); col->dl_tmp = nullptr; }
    if (!col->dl_counts.empty()) cudaStreamSynchronize(c->s_d2h);  // a split download is still writing into it
    for (auto& g : col->groups) if (g.ev) cudaStreamWaitEvent(c->s_compute, g.ev, 0);
    if (col->arena_values) cudaFreeAsync(col->arena_values, c->s_compute);
    if (col->arena_validity) cudaFreeAsync(col->arena_validity, c->s_compute);
    if (col->d_warp_counts) cudaFreeAsync(col->d_warp_counts, c->s_compute);
    col_destroy_host(c, col);
}

struct ChunkPlan {
    int64_t len;
    bool has_validity;
};

// Allocate arenas for a column with the given chunk plan (validity at bit offset `bit_off[i]`).
// tile_elems > 0: the column will be produced by a kernel with that tile size (per-warp valid counts are kept).
static int col_alloc(bdf_ctx* c, int dtype, const std::vector<ChunkPlan>& plan, const std::vector<int32_t>* bit_offs,
                     int64_t tile_elems, bdf_col** out) {
    bdf_col* col = new (std::nothrow) bdf_col();
    if (!col) return fail(BDF_OOM, "host allocation failed");
    col->owner = c;
    col->dtype = dtype;
    const int w = dtype_width(dtype);
    const size_t n = plan.size();
    std::vector<size_t> voff(n), boff(n);
    size_t vbytes = 0, bbytes = 0;
    for (size_t i = 0; i < n; i++) {
        voff[i] = vbytes;
        vbytes += align_up(value_bytes(dtype, plan[i].len, bit_offs ? (*bit_offs)[i] : 0) + (dtype == kBool ? 8 : 0), 256);
        boff[i] = bbytes;
        if (plan[i].has_validity) {
            const int bo = bit_offs ? (*bit_offs)[i] : 0;
            bbytes += align_up(((size_t)plan[i].len + bo + 7) / 8 + 8, 256);
        }
        col->total_len += plan[i].len;
    }
    cudaError_t e = cudaSuccess;
    if (vbytes) e = cudaMallocAsync((void**)&col->arena_values, vbytes, c->s_compute);
    if (e == cudaSuccess && bbytes) e = cudaMallocAsync((void**)&col->arena_validity, bbytes, c->s_compute);
    col->tile_elems = tile_elems;
    col->tile0.assign(n + 1, 0);
    if (tile_elems > 0)
        for (size_t i = 0; i < n; i++) col->tile0[i + 1] = col->tile0[i] + (plan[i].len + tile_elems - 1) / tile_elems;
    const size_t n_tiles = (size_t)col->tile0[n];
    if (e == cudaSuccess && bbytes && n_tiles)
        e = cudaMallocAsync((void**)&col->d_warp_counts, n_tiles * kWarpsPerCta * sizeof(uint32_t), c->s_compute);
    if (e == cudaSuccess && bbytes) e = cudaMemsetAsync(col->arena_validity, 0, bbytes, c->s_compute);
    if (e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, col);
        return fail(cuda_status(e), "device allocation of %zu bytes failed: %s", vbytes + bbytes, cudaGetErrorString(e));
    }
    col->chunks.resize(n);
    col->null_counts.assign(n, 0);
    for (size_t i = 0; i < n; i++) {
        DevChunk& ch = col->chunks[i];
        ch.values = col->arena_values ? col->arena_values + voff[i] : nullptr;
        ch.validity = plan[i].has_validity ? (uint32_t*)(col->arena_validity + boff[i]) : nullptr;
        ch.len = plan[i].len;
        ch.bit_off = bit_offs ? (*bit_offs)[i] : 0;
        ch.val_bit_off = (dtype == kBool && bit_offs) ? (*bit_offs)[i] : 0;
    }
    *out = col;
    return BDF_OK;
}

// True when every group event of the column has already fired.
static bool col_complete(const bdf_col* col) {
    for (auto& g : col->groups)
        if (cudaEventQuery(g.ev) != cudaSuccess) { cudaGetLastError(); return false; }
    return true;
}

static void wait_groups(cudaStream_t s, const bdf_col* col, int64_t begin, int64_t end) {
    for (auto& g : col->groups)
        if (g.begin < end && g.end > begin) cudaStreamWaitEvent(s, g.ev, 0);
}

// Group boundaries for an operator over `n` chunks: a single group when the inputs are resident, else
// the union of the inputs' group ends (so work starts as soon as its own inputs have landed).
static std::vector<int64_t> plan_groups(int64_t n, std::initializer_list<const bdf_col*> inputs) {
    bool all_done = true;
    for (auto* col : inputs) all_done = all_done && col_complete(col);
    std::vector<int64_t> ends;
    if (!all_done)
        for (auto* col : inputs)
            for (auto& g : col->groups)
                if (g.end < n) ends.push_back(g.end);
    ends.push_back(n);
    std::sort(ends.begin(), ends.end());
    ends.erase(std::unique(ends.begin(), ends.end()), ends.end());
    return ends;
}

static int64_t bitmap_bytes(int64_t len) { return (len + 7) / 8; }

// Fold the per-warp valid counts of every chunk into null_counts (host side; chunk i owns tiles [tile0[i], tile0[i+1])).
static void fold_counts(bdf_col* col, const uint32_t* counts) {
    const size_t n = col->chunks.size();
    for (size_t i = 0; i < n; i++) {
        if (!col->chunks[i].validity) { col->null_counts[i] = 0; continue; }
        int64_t valid = 0;
        for (int64_t k = col->tile0[i] * kWarpsPerCta; k < col->tile0[i + 1] * kWarpsPerCta; k++) valid += counts[k];
        col->null_counts[i] = col->chunks[i].len - valid;
    }
    col->counts_on_device = false;
}

// Mirror kernel-written valid counts into host null_counts (one small D2H + sync on the compute stream).
static int fetch_counts(bdf_ctx* c, bdf_col* col) {
    if (!col->counts_on_device) return BDF_OK;
    const size_t n = col->chunks.size();
    const size_t total = (size_t)col->tile0[n] * kWarpsPerCta;
    std::vector<uint32_t> tmp(std::max<size_t>(total, 1));
    if (total) {
        wait_groups(c->s_compute, col, 0, (int64_t)n);
        CK(cudaMemcpyAsync(tmp.data(), col->d_warp_counts, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
    }
    fold_counts(col, tmp.data());
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// reduce plumbing

static int64_t reduce_bytes(const bdf_col* col, int64_t begin, int64_t end) {
    int64_t b = 0;
    const int w = dtype_width(col->dtype);
    for (int64_t i = begin; i < end; i++)
        b += col->chunks[i].len * w + (col->chunks[i].validity ? bitmap_bytes(col->chunks[i].len) : 0);
    return b;
}

// Launch one reduce over chunks [begin,end) of col into *result (device-mapped host memory: c->h_agg_dev + slot, or a
// device record that a collective will read).  Caller has made the stream wait.
static int reduce_range(bdf_ctx* c, const bdf_col* col, int64_t begin, int64_t end, AggDev* result) {
    const int64_t n = end - begin;
    const int tile = elems_per_tile(col->dtype);
    void *hp = nullptr, *dp = nullptr;
    TRY(ring_alloc(c, (size_t)n * sizeof(RedDesc), &hp, &dp));
    RedDesc* hd = (RedDesc*)hp;
    int64_t tiles = 0, rows = 0;
    for (int64_t i = 0; i < n; i++) {
        const DevChunk& ch = col->chunks[begin + i];
        hd[i].in = ch.values; hd[i].vin = ch.validity; hd[i].len = ch.len; hd[i].tile0 = tiles; hd[i].off = ch.bit_off; hd[i].pad = 0;
        tiles += (ch.len + tile - 1) / tile;
        rows += ch.len;
    }
    RedDesc* dd = (RedDesc*)dp;
    CK(desc_upload(c, dd, hd, (size_t)n * sizeof(RedDesc)));
    if ((size_t)tiles > c->red_part_cap) {  // grow the per-CTA partials buffer (rare): drain its users first
        CK(cudaStreamSynchronize(c->s_compute));
        if (c->d_partials) CK(cudaFree(c->d_partials));
        c->d_partials = nullptr; c->red_part_cap = 0;
        const size_t cap = std::max<size_t>((size_t)tiles * 2, 65536);
        CK(cudaMalloc((void**)&c->d_partials, cap * sizeof(AggDev)));
        c->red_part_cap = cap;
    }
    {
        LaunchTimer t(c, BDF_K_REDUCE, col->dtype, rows, reduce_bytes(col, begin, end));  // k_reduce + k_finish
        CK(launch_reduce(col->dtype, dd, (int)n, tiles, c->d_partials, c->s_compute));
        c->launches++;
        CK(launch_finish(dtype_is_float(col->dtype), c->d_partials, reduce_partials(col->dtype, tiles), c->sm_count, c->d_stage2, c->d_ticket, result, c->s_compute));
    }
    return BDF_OK;
}

// Make sure every chunk's null count is known on the host (metadata for count / would_panic).
static int ensure_null_counts(bdf_ctx* c, bdf_col* col) {
    TRY(fetch_counts(c, col));
    std::vector<int64_t> unknown;
    for (size_t i = 0; i < col->chunks.size(); i++)
        if (col->null_counts[i] < 0) unknown.push_back((int64_t)i);
    if (unknown.empty()) return BDF_OK;
    if (col->dtype == kBool) return fail(BDF_UNSUPPORTED, "null count of an uploaded boolean column is unknown: pass null_count in the view");
    wait_groups(c->s_compute, col, 0, (int64_t)col->chunks.size());
    for (size_t k = 0; k < unknown.size(); k += kAggSlots) {
        const size_t m = std::min<size_t>(kAggSlots, unknown.size() - k);
        for (size_t j = 0; j < m; j++) TRY(reduce_range(c, col, unknown[k + j], unknown[k + j] + 1, c->h_agg_dev + j));
        CK(cudaStreamSynchronize(c->s_compute));
        for (size_t j = 0; j < m; j++) {
            const int64_t i = unknown[k + j];
            col->null_counts[i] = col->chunks[i].len - (int64_t)c->h_agg[j].count;
        }
    }
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// pageable host memory: staged copies

static constexpr size_t kStageBytes = (size_t)8 << 20;
static constexpr int kStageSlots = 6;
static constexpr size_t kStageMin = (size_t)1 << 20;  // smaller copies go straight through the driver

static bool is_pageable(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return attr.type == cudaMemoryTypeUnregistered;
}

static int ensure_stage(bdf_ctx* c) {
    if (!c->stage.empty()) return BDF_OK;
    // built in locals and committed to the context only when complete: a failure part-way leaves the context unstaged
    std::vector<bdf_ctx::StageSlot> slots(kStageSlots);
    cudaError_t e = cudaSuccess;
    for (auto& sl : slots) {
        if (e == cudaSuccess) e = cudaHostAlloc((void**)&sl.p, kStageBytes, cudaHostAllocDefault);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl.ev, cudaEventDisableTiming);
    }
    const char* t = getenv("BDF_COPY_THREADS");
    const int hw = (int)std::thread::hardware_concurrency();
    const int threads = t && atoi(t) > 0 ? atoi(t) : std::max(1, std::min(8, hw > 0 ? hw : 8));
    std::unique_ptr<CopyPool> pool;
    if (e == cudaSuccess) pool.reset(new (std::nothrow) CopyPool(threads - 1));   // the calling thread is the last worker
    if (e != cudaSuccess || !pool) {
        cudaGetLastError();
        for (auto& sl : slots) { if (sl.p) cudaFreeHost(sl.p); if (sl.ev) cudaEventDestroy(sl.ev); }
        return e != cudaSuccess ? fail(cuda_status(e), "pinned staging allocation failed: %s", cudaGetErrorString(e)) : fail(BDF_OOM, "host allocation failed");
    }
    c->copy_threads = threads;
    c->pool = std::move(pool);
    c->stage = std::move(slots);
    return BDF_OK;
}

// host -> device on the h2d stream; pageable sources are staged through pinned slots (the source has been read
// completely when this returns).
static cudaError_t h2d_copy(bdf_ctx* c, void* dst, const void* src, size_t bytes) {
    if (bytes < kStageMin || !is_pageable(src)) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->s_h2d);
    if (ensure_stage(c) != BDF_OK) return cudaErrorMemoryAllocation;
    for (size_t off = 0; off < bytes; off += kStageBytes) {
        const size_t n = std::min(kStageBytes, bytes - off);
        bdf_ctx::StageSlot& sl = c->stage[c->stage_next++ % kStageSlots];
        if (sl.busy) { cudaError_t e = cudaEventSynchronize(sl.ev); if (e != cudaSuccess) return e; }
        c->pool->copy(sl.p, (const char*)src + off, n);
        cudaError_t e = cudaMemcpyAsync((char*)dst + off, sl.p, n, cudaMemcpyHostToDevice, c->s_h2d);
        if (e == cudaSuccess) e = cudaEventRecord(sl.ev, c->s_h2d);
        if (e != cudaSuccess) return e;
        sl.busy = true;
    }
    return cudaSuccess;
}

// device -> pageable host, pipelined: DMA into slot k+1.. while host threads drain slot k into the user's buffer.
static cudaError_t d2h_staged(bdf_ctx* c, const std::vector<bdf_col::StagedCopy>& copies) {
    if (copies.empty()) return cudaSuccess;
    if (ensure_stage(c) != BDF_OK) return cudaErrorMemoryAllocation;
    struct Pending { bdf_ctx::StageSlot* sl; char* dst; size_t n; };
    std::deque<Pending> pending;
    auto retire = [&]() -> cudaError_t {
        Pending p = pending.front();
        pending.pop_front();
        cudaError_t e = cudaEventSynchronize(p.sl->ev);
        if (e == cudaSuccess) c->pool->copy(p.dst, p.sl->p, p.n, true);
        p.sl->busy = false;
        return e;
    };
    for (auto& cp : copies)
        for (size_t off = 0; off < cp.bytes; off += kStageBytes) {
            const size_t n = std::min(kStageBytes, cp.bytes - off);
            if ((int)pending.size() >= kStageSlots - 1) { cudaError_t e = retire(); if (e != cudaSuccess) return e; }
            bdf_ctx::StageSlot& sl = c->stage[c->stage_next++ % kStageSlots];
            if (sl.busy) { cudaError_t e = cudaEventSynchronize(sl.ev); if (e != cudaSuccess) return e; }  // an earlier upload's slot
            cudaError_t e = cudaMemcpyAsync(sl.p, (const char*)cp.src + off, n, cudaMemcpyDeviceToHost, c->s_d2h);
            if (e == cudaSuccess) e = cudaEventRecord(sl.ev, c->s_d2h);
            if (e != cudaSuccess) return e;
            sl.busy = true;
            pending.push_back(Pending{&sl, (char*)cp.dst + off, n});
        }
    while (!pending.empty()) { cudaError_t e = retire(); if (e != cudaSuccess) return e; }
    return cudaSuccess;
}

// ---------------------------------------------------------------------------------------------------
// upload / download

struct UploadSpec {
    int dtype;
    int64_t n;
    const bdf_view* views;
};

// Upload K columns with their chunks interleaved (a0,b0,a1,b1,...) so that a binary operator can start on
// chunk i as soon as BOTH of its inputs have landed.
static int upload_many(bdf_ctx* c, const std::vector<UploadSpec>& specs, bool async, std::vector<bdf_col*>& cols) {
    cols.assign(specs.size(), nullptr);
    int64_t max_n = 0;
    auto cleanup = [&]() { for (auto*& col : cols) { col_release(c, col); col = nullptr; } };
    for (size_t k = 0; k < specs.size(); k++) {
        const UploadSpec& s = specs[k];
        std::vector<ChunkPlan> plan((size_t)s.n);
        std::vector<int32_t> offs((size_t)s.n);
        for (int64_t i = 0; i < s.n; i++) {
            const bdf_view& v = s.views[i];
            plan[i] = {v.len, v.validity != nullptr};
            offs[i] = (int32_t)(v.offset & 7);
        }
        int st = col_alloc(c, s.dtype, plan, &offs, 0, &cols[k]);
        if (st != BDF_OK) { cleanup(); return st; }
        for (int64_t i = 0; i < s.n; i++)
            cols[k]->null_counts[i] = s.views[i].validity ? (s.views[i].null_count >= 0 ? s.views[i].null_count : -1) : 0;
        max_n = std::max(max_n, s.n);
    }
    // allocations are stream-ordered on the compute stream: let the copy stream see them
    cudaError_t e = cudaEventRecord(c->ev_tmp, c->s_compute);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c->s_h2d, c->ev_tmp, 0);
    size_t pending = 0;
    int64_t group_begin = 0;
    for (int64_t i = 0; i < max_n && e == cudaSuccess; i++) {
        for (size_t k = 0; k < specs.size() && e == cudaSuccess; k++) {
            if (i >= specs[k].n) continue;
            const bdf_view& v = specs[k].views[i];
            const DevChunk& ch = cols[k]->chunks[i];
            const int w = dtype_width(specs[k].dtype);
            if (v.len) {
                const bool is_bool = specs[k].dtype == kBool;
                const size_t vb = value_bytes(specs[k].dtype, v.len, (int)(v.offset & 7));
                e = h2d_copy(c, ch.values, (const char*)v.values + (is_bool ? (v.offset >> 3) : v.offset * w), vb);
                pending += vb;
                if (e == cudaSuccess && v.validity)
                    e = cudaMemcpyAsync(ch.validity, v.validity + (v.offset >> 3), (size_t)((v.len + (v.offset & 7) + 7) / 8),
                                        cudaMemcpyHostToDevice, c->s_h2d);
            }
        }
        if (e == cudaSuccess && (pending >= c->pipeline_bytes || i == max_n - 1)) {
            for (size_t k = 0; k < specs.size() && e == cudaSuccess; k++) {
                const int64_t b = std::min(group_begin, specs[k].n), en = std::min(i + 1, specs[k].n);
                if (en <= b) continue;
                Group g{b, en, nullptr};
                e = ev_get(c, &g.ev);
                if (e == cudaSuccess) e = cudaEventRecord(g.ev, c->s_h2d);
                cols[k]->groups.push_back(g);
            }
            pending = 0;
            group_begin = i + 1;
        }
    }
    if (e == cudaSuccess && !async) e = cudaStreamSynchronize(c->s_h2d);
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaStreamSynchronize(c->s_h2d);
        cleanup();
        return fail(cuda_status(e), "upload failed: %s", cudaGetErrorString(e));
    }
    return BDF_OK;
}

static int realign(bdf_ctx* c, const bdf_col* in, bdf_col** out);  // identity cast: bit offset -> 0

// Downloads are split in two so that callers can overlap them with later work: enqueue puts the D2H copies
// on the d2h stream behind the group events; finish waits for them and fills in the metadata.
static int download_enqueue(bdf_ctx* c, bdf_col* col, bdf_out* out) {
    bool misaligned = false;
    for (auto& ch : col->chunks) misaligned = misaligned || (ch.validity && ch.bit_off != 0) || ch.val_bit_off != 0;
    if (misaligned) {  // an uploaded slice downloaded as-is: shift its bitmap to offset 0 first
        bdf_col* tmp = nullptr;
        TRY(realign(c, col, &tmp));
        int st = download_enqueue(c, tmp, out);
        if (st != BDF_OK) { col_release(c, tmp); return st; }
        col->dl_tmp = tmp;
        return BDF_OK;
    }
    const int w = dtype_width(col->dtype);
    const int64_t n = (int64_t)col->chunks.size();
    for (int64_t i = 0; i < n; i++) {
        const DevChunk& ch = col->chunks[i];
        if (out[i].len != ch.len) return fail(BDF_INVALID, "output chunk %lld has capacity %lld, result has %lld rows", (long long)i, (long long)out[i].len, (long long)ch.len);
        if (ch.len && !out[i].values) return fail(BDF_INVALID, "output chunk %lld has no values buffer", (long long)i);
        if (ch.validity && ch.len && !out[i].validity) return fail(BDF_INVALID, "output chunk %lld needs a validity buffer", (long long)i);
    }
    for (auto& g : col->groups) {
        CK(cudaStreamWaitEvent(c->s_d2h, g.ev, 0));
        for (int64_t i = g.begin; i < g.end; i++) {
            const DevChunk& ch = col->chunks[i];
            if (!ch.len) continue;
            const size_t vbytes = value_bytes(col->dtype, ch.len, 0);
            if (vbytes >= kStageMin && is_pageable(out[i].values)) col->dl_staged.push_back({out[i].values, ch.values, vbytes});
            else CK(cudaMemcpyAsync(out[i].values, ch.values, vbytes, cudaMemcpyDeviceToHost, c->s_d2h));
            if (ch.validity) CK(cudaMemcpyAsync(out[i].validity, ch.validity, (size_t)bitmap_bytes(ch.len), cudaMemcpyDeviceToHost, c->s_d2h));
        }
    }
    if (col->counts_on_device && col->tile0[n] > 0) {
        col->dl_counts.resize((size_t)col->tile0[n] * kWarpsPerCta);
        CK(cudaMemcpyAsync(col->dl_counts.data(), col->d_warp_counts, col->dl_counts.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->s_d2h));
    }
    return BDF_OK;
}

static int download_finish(bdf_ctx* c, bdf_col* col, bdf_out* out) {
    if (col->dl_tmp) {
        bdf_col* tmp = col->dl_tmp;
        col->dl_tmp = nullptr;
        int st = download_finish(c, tmp, out);
        col_release(c, tmp);
        return st;
    }
    const int64_t n = (int64_t)col->chunks.size();
    if (!col->dl_staged.empty()) {  // the d2h stream already waits for the group events of this column
        cudaError_t e = d2h_staged(c, col->dl_staged);
        col->dl_staged.clear();
        if (e != cudaSuccess) { cudaGetLastError(); return fail(cuda_status(e), "staged download failed: %s", cudaGetErrorString(e)); }
    }
    CK(cudaStreamSynchronize(c->s_d2h));
    if (col->counts_on_device && (int64_t)col->dl_counts.size() == col->tile0[n] * kWarpsPerCta) {
        fold_counts(col, col->dl_counts.data());
        col->dl_counts.clear();
    }
    TRY(ensure_null_counts(c, col));
    for (int64_t i = 0; i < n; i++) {
        out[i].len = col->chunks[i].len;
        out[i].has_validity = col->chunks[i].validity != nullptr;
        out[i].null_count = col->null_counts[i];
    }
    return BDF_OK;
}

static int download(bdf_ctx* c, bdf_col* col, bdf_out* out) {
    TRY(download_enqueue(c, col, out));
    return download_finish(c, col, out);
}

// ---------------------------------------------------------------------------------------------------
// operators on device columns

static bool cast_is_fallible(int from, int to) {
    if (from == to || dtype_is_float(to)) return false;
    if (dtype_is_float(from)) return true;
    const bool fs = dtype_is_signed_int(from), ts = dtype_is_signed_int(to);
    const int fw = dtype_width(from), tw = dtype_width(to);
    if (fs == ts) return tw < fw;
    if (fs) return true;        // signed -> unsigned: negatives fail
    return tw <= fw;            // unsigned -> signed: needs a strictly wider target
}

static int future_new(bdf_ctx* c, int dtype, int fused, int64_t rows, bdf_future** out, int n = 1);
static bool is_global(const bdf_ctx* c) { return c->comm != nullptr && c->collective; }
static AggDev* future_target(bdf_ctx* c, const bdf_future* f, int i);
static cudaError_t future_combine(bdf_ctx* c, bdf_future* f, cudaStream_t s);
// The DivideByZero flag of a sharded divide: max over the ranks, so that every rank returns the same status.
static cudaError_t flag_allreduce(bdf_ctx* c) {
    std::string err;
    c->collectives++;
    cudaError_t e = comm_allreduce_max_i32(c->comm, c->d_flag, 1, c->s_compute, &err);
    if (e != cudaSuccess && !err.empty()) g_nccl_err = err;
    return e;
}

// One of three rotating per-tile partial buffers (K5 and fused expressions): grown on demand, reused once the
// k_finish that last read it has run.
static cudaError_t part_acquire(bdf_ctx* c, int64_t total_tiles, bdf_ctx::PartBuf** out) {
    bdf_ctx::PartBuf* pb = &c->part[c->part_next++ % 3];
    cudaError_t e = cudaSuccess;
    const size_t need = std::max<size_t>(1, (size_t)total_tiles);
    if (pb->cap < need) {  // grow (rare): nothing may still be using the old buffer
        cudaStreamSynchronize(c->s_fin); cudaStreamSynchronize(c->s_compute);
        if (pb->p) cudaFree(pb->p);
        pb->p = nullptr; pb->cap = 0;
        e = cudaMalloc((void**)&pb->p, need * sizeof(AggDev));
        if (e == cudaSuccess) pb->cap = need;
    }
    if (e == cudaSuccess && !pb->done) e = cudaEventCreateWithFlags(&pb->done, cudaEventDisableTiming);
    if (e == cudaSuccess && pb->used) e = cudaStreamWaitEvent(c->s_compute, pb->done, 0);  // its previous k_finish has read it
    *out = pb;
    return e;
}

static int binary_dev(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, bdf_col** out, bdf_future** fut = nullptr) {
    if (op < 0 || op >= BDF_NBINARY) return fail(BDF_INVALID, "invalid binary op %d", op);
    if (l->dtype != r->dtype) return fail(BDF_INVALID, "binary op on columns of different types (%d, %d)", l->dtype, r->dtype);
    if (l->dtype == kBool) return fail(BDF_UNSUPPORTED, "arithmetic on a boolean column");
    const int dtype = l->dtype;
    if (op > BDF_DIV && !dtype_is_float(dtype)) return fail(BDF_UNSUPPORTED, "atan2/hypot/log need a float column (T::Native: Float)");
    const int64_t n = std::min<int64_t>((int64_t)l->chunks.size(), (int64_t)r->chunks.size());  // zip()
    for (int64_t i = 0; i < n; i++)
        if (l->chunks[i].len != r->chunks[i].len)
            return fail(BDF_LENGTH_MISMATCH, "Cannot perform math operation on arrays of different length");
    std::vector<ChunkPlan> plan((size_t)n);
    for (int64_t i = 0; i < n; i++)
        plan[i] = {l->chunks[i].len, op > BDF_DIV || l->chunks[i].validity || r->chunks[i].validity};
    bdf_col* o = nullptr;
    const int tile = elems_per_tile_binary(op, dtype);
    TRY(col_alloc(c, dtype, plan, nullptr, tile, &o));
    o->counts_on_device = o->d_warp_counts != nullptr;

    const int w = dtype_width(dtype);
    void *hp = nullptr, *dp = nullptr;
    int st = ring_alloc(c, (size_t)n * sizeof(BinDesc), &hp, &dp);
    BinDesc* dd = (BinDesc*)dp;
    cudaError_t e = cudaSuccess;
    // K5: aggregate of the output fused into the same pass -> one partial per tile, folded by k_finish
    AggDev* partials = nullptr;
    bdf_ctx::PartBuf* pb = nullptr;
    int64_t total_tiles = 0, tile_base = 0;
    bdf_future* f = nullptr;
    if (fut && st == BDF_OK) {
        if (op > BDF_DIV) { col_release(c, o); return fail(BDF_UNSUPPORTED, "fused aggregate is available for add/subtract/multiply/divide"); }
        for (int64_t i = 0; i < n; i++) total_tiles += (l->chunks[i].len + tile - 1) / tile;
        st = future_new(c, dtype, 1, o->total_len, &f);
        if (st == BDF_OK) {
            e = part_acquire(c, total_tiles, &pb);
            partials = pb->p;
        }
    }
    if (st == BDF_OK && e == cudaSuccess) {
        BinDesc* hd = (BinDesc*)hp;
        const std::vector<int64_t> ends = plan_groups(n, {l, r});
        if (op == BDF_DIV) e = cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->s_compute);
        int64_t begin = 0;
        for (size_t gi = 0; gi < ends.size() && e == cudaSuccess; gi++) {
            const int64_t end = ends[gi];
            int64_t tiles = 0, rows = 0, bytes = 0;
            for (int64_t i = begin; i < end; i++) {
                const DevChunk &a = l->chunks[i], &b = r->chunks[i], &oc = o->chunks[i];
                hd[i] = BinDesc{a.values, b.values, oc.values, a.validity, b.validity, oc.validity, a.len, tiles, a.bit_off, b.bit_off};
                tiles += (a.len + tile - 1) / tile;
                rows += a.len;
                bytes += 3 * a.len * w + ((a.validity ? 1 : 0) + (b.validity ? 1 : 0) + (oc.validity ? 1 : 0)) * bitmap_bytes(a.len);
            }
            wait_groups(c->s_compute, l, begin, end);
            wait_groups(c->s_compute, r, begin, end);
            if (end > begin) {
                e = desc_upload(c, dd + begin, hd + begin, (size_t)(end - begin) * sizeof(BinDesc));
                if (e == cudaSuccess) {
                    LaunchTimer t(c, BDF_K_BINARY, dtype, rows, bytes);
                    e = launch_binary(op, dtype, dd + begin, (int)(end - begin), tiles, o->d_warp_counts ? o->d_warp_counts + o->tile0[begin] * kWarpsPerCta : nullptr, c->d_flag, c->s_compute, partials ? partials + tile_base : nullptr);
                }
            }
            if (e == cudaSuccess) {
                Group g{begin, end, nullptr};
                e = ev_get(c, &g.ev);
                if (e == cudaSuccess) e = cudaEventRecord(g.ev, c->s_compute);
                o->groups.push_back(g);
            }
            begin = end;
            tile_base += tiles;
        }
        if (e == cudaSuccess && f) {
            // fold the per-tile partials on the finish stream: the next operator on the compute stream does not wait
            c->launches++;
            for (auto& g : o->groups) cudaStreamWaitEvent(c->s_fin, g.ev, 0);
            e = launch_finish(dtype_is_float(dtype), partials, total_tiles, c->sm_count, c->d_stage, c->d_ticket + 1, future_target(c, f, 0), c->s_fin);
            if (e == cudaSuccess) e = cudaEventRecord(pb->done, c->s_fin);
            pb->used = true;
            f->chunks[0] = (uint32_t)n;
            if (e == cudaSuccess) e = future_combine(c, f, c->s_fin);   // ranks of a communicator: one grouped NCCL reduction
            if (e == cudaSuccess) e = cudaEventRecord(f->ev, c->s_fin);
        }
        if (e == cudaSuccess && op == BDF_DIV) {
            // DivideByZero must be returned INSTEAD of data: wait for the flag (every rank of a communicator takes the same exit).
            if (is_global(c)) e = flag_allreduce(c);
            if (e == cudaSuccess) e = cudaMemcpyAsync(c->h_flag, c->d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->s_compute);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->s_compute);
            if (e == cudaSuccess && *c->h_flag) {
                col_release(c, o);
                if (f) { ev_put(c, f->ev); delete f; }
                return fail(BDF_DIVIDE_BY_ZERO, "Divide by zero error");
            }
        }
    }
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        if (f) { ev_put(c, f->ev); delete f; }
        return st != BDF_OK ? st : fail_cuda(e, "binary op");
    }
    *out = o;
    if (fut) *fut = f;
    return BDF_OK;
}

// Shared body of unary ops and casts (one input column, one output column).
static int map_dev(bdf_ctx* c, bool is_cast, int op_or_to, const bdf_col* in, bdf_col** out) {
    const int from = in->dtype;
    int to = from;
    if (from == kBool) return fail(BDF_UNSUPPORTED, "numeric function on a boolean column");
    if (is_cast) {
        to = op_or_to;
    } else {
        const int op = op_or_to;
        if (op < 0 || op >= BDF_NUNARY) return fail(BDF_INVALID, "invalid unary op %d", op);
        if (op == BDF_ABS) {
            if (!dtype_is_float(from) && !dtype_is_signed_int(from)) return fail(BDF_UNSUPPORTED, "abs needs a signed type (T::Native: Signed)");
        } else if (!dtype_is_float(from)) {
            return fail(BDF_UNSUPPORTED, "float function on a non-float column (T::Native: Float)");
        }
    }
    const int64_t n = (int64_t)in->chunks.size();
    const bool fallible = is_cast && cast_is_fallible(from, to);
    std::vector<ChunkPlan> plan((size_t)n);
    for (int64_t i = 0; i < n; i++) plan[i] = {in->chunks[i].len, in->chunks[i].validity != nullptr || fallible};
    bdf_col* o = nullptr;
    const int tile = is_cast ? elems_per_tile_cast(from, to) : elems_per_tile_unary(op_or_to, from);
    TRY(col_alloc(c, to, plan, nullptr, tile, &o));
    o->counts_on_device = o->d_warp_counts != nullptr;

    const int wf = dtype_width(from), wt = dtype_width(to);
    void *hp = nullptr, *dp = nullptr;
    int st = ring_alloc(c, (size_t)n * sizeof(UnDesc), &hp, &dp);
    UnDesc* dd = (UnDesc*)dp;
    cudaError_t e = cudaSuccess;
    if (st == BDF_OK) {
        UnDesc* hd = (UnDesc*)hp;
        const std::vector<int64_t> ends = plan_groups(n, {in});
        int64_t begin = 0;
        for (size_t gi = 0; gi < ends.size() && e == cudaSuccess; gi++) {
            const int64_t end = ends[gi];
            int64_t tiles = 0, rows = 0, bytes = 0;
            for (int64_t i = begin; i < end; i++) {
                const DevChunk &a = in->chunks[i], &oc = o->chunks[i];
                hd[i] = UnDesc{a.values, oc.values, a.validity, oc.validity, a.len, tiles, a.bit_off, 0};
                tiles += (a.len + tile - 1) / tile;
                rows += a.len;
                bytes += a.len * (wf + wt) + ((a.validity ? 1 : 0) + (oc.validity ? 1 : 0)) * bitmap_bytes(a.len);
            }
            wait_groups(c->s_compute, in, begin, end);
            if (end > begin) {
                e = desc_upload(c, dd + begin, hd + begin, (size_t)(end - begin) * sizeof(UnDesc));
                if (e == cudaSuccess) {
                    LaunchTimer t(c, is_cast ? BDF_K_CAST : BDF_K_UNARY, to, rows, bytes);
                    e = is_cast ? launch_cast(from, to, dd + begin, (int)(end - begin), tiles, o->d_warp_counts ? o->d_warp_counts + o->tile0[begin] * kWarpsPerCta : nullptr, c->s_compute)
                                : launch_unary(op_or_to, from, dd + begin, (int)(end - begin), tiles, o->d_warp_counts ? o->d_warp_counts + o->tile0[begin] * kWarpsPerCta : nullptr, c->s_compute);
                }
            }
            if (e == cudaSuccess) {
                Group g{begin, end, nullptr};
                e = ev_get(c, &g.ev);
                if (e == cudaSuccess) e = cudaEventRecord(g.ev, c->s_compute);
                o->groups.push_back(g);
            }
            begin = end;
        }
    }
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return st != BDF_OK ? st : fail(cuda_status(e), "%s failed: %s", is_cast ? "cast" : "unary op", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

static int boolean_dev(bdf_ctx* c, int op, const bdf_col* a, const bdf_col* b, bdf_col** out);
static int realign(bdf_ctx* c, const bdf_col* in, bdf_col** out) {
    if (in->dtype == kBool) return boolean_dev(c, 1 /* OR: x | x = x, validity AND itself */, in, in, out);
    return map_dev(c, true, in->dtype, in, out);
}

// A future over n aggregates.  On a context that is a rank of a communicator (collective mode) the kernels write their
// per-rank records to device memory (d_local) and future_combine enqueues the grouped NCCL reduction that delivers the
// GLOBAL records to the pinned slots; otherwise the kernels write the pinned slots themselves.
static int future_new(bdf_ctx* c, int dtype, int fused, int64_t rows, bdf_future** out, int n) {
    if (n < 1 || n > kCommMaxCols) return fail(BDF_INVALID, "an aggregate call takes 1..%d columns", kCommMaxCols);
    bdf_future* f = new (std::nothrow) bdf_future();
    if (!f) return fail(BDF_OOM, "host allocation failed");
    f->n = n; f->fused = fused; f->global = is_global(c);
    f->dtypes.assign((size_t)n, dtype); f->rows.assign((size_t)n, rows); f->panics.assign((size_t)n, 0u); f->chunks.assign((size_t)n, 1u);
    const int words = f->global ? 2 * n : n;
    if (c->fut_next % kAggSlots + words > kAggSlots) c->fut_next += kAggSlots - c->fut_next % kAggSlots;  // keep the block contiguous
    f->slot = kAggSlots + c->fut_next % kAggSlots;  // upper half of h_agg is the future ring
    c->fut_next += words;
    if (f->global) {
        if (c->local_next % kAggSlots + n > kAggSlots) c->local_next += kAggSlots - c->local_next % kAggSlots;
        f->lslot = c->local_next % kAggSlots;
        c->local_next += n;
    }
    cudaError_t e = ev_get(c, &f->ev);
    if (e != cudaSuccess) { delete f; return fail(cuda_status(e), "event creation failed: %s", cudaGetErrorString(e)); }
    *out = f;
    return BDF_OK;
}

// Where the kernels of aggregate i of the future deliver their folded record.
static AggDev* future_target(bdf_ctx* c, const bdf_future* f, int i) {
    return f->global ? c->d_local + f->lslot + i : c->h_agg_dev + f->slot + i;
}

// Global futures: enqueue the ONE grouped collective on the stream that produced the records (no host round trip).
static cudaError_t future_combine(bdf_ctx* c, bdf_future* f, cudaStream_t s) {
    if (!f->global) return cudaSuccess;
    unsigned long long fmask = 0, rows[kCommMaxCols];
    for (int i = 0; i < f->n; i++) {
        if (dtype_is_float(f->dtypes[i])) fmask |= 1ull << i;
        rows[i] = (unsigned long long)f->rows[i];
    }
    std::string err;
    c->collectives++;
    c->launches += 2;  // pack + unpack (the NCCL kernel itself is not ours)
    cudaError_t e = comm_combine(c->comm, fmask, f->n, c->d_local + f->lslot, rows, f->panics.data(), f->chunks.data(), c->h_agg_dev + f->slot, s, &err);
    if (e != cudaSuccess && !err.empty()) g_nccl_err = err;
    return e;
}

// AggDev (device format) -> bdf_agg4 (ABI format: T::Native bit patterns)
static void convert_agg(int dtype, int fused, const AggDev& a, int64_t rows, bdf_agg4* out) {
    memset(out, 0, sizeof *out);
    const int w = dtype_width(dtype);
    const uint64_t mask = w == 8 ? ~0ull : ((1ull << (8 * w)) - 1ull);
    if (dtype == BDF_F64) {
        out->sum = a.sum_bits;
    } else if (dtype == BDF_F32) {
        double d; memcpy(&d, &a.sum_bits, 8);
        const float f = (float)d;
        uint32_t fb; memcpy(&fb, &f, 4);
        out->sum = fb;
    } else {
        // k_binary AGG (fused == 1) keys flip the sign bit of T; k_reduce (fused == 2) keys flip bit 63 of the extended value
        const uint64_t flip = !dtype_is_signed_int(dtype) ? 0ull : (fused == 1 ? (1ull << (8 * w - 1)) : (1ull << 63));
        out->sum = a.sum_bits & mask;
        out->min = (a.min_bits ^ flip) & mask;
        out->max = (a.max_bits ^ flip) & mask;
    }
    out->count = (int64_t)a.count;
    out->rows = rows;
    out->any_valid = a.count > 0;
}

// sum/min/max/count of several columns with as few launches as possible: the columns of one dtype share ONE k_reduce launch
// (their chunk descriptors are concatenated, every column starting on a CTA boundary), and ONE k_finish_many folds every
// column's partials.  BASELINE config 3 (8 x Int64) is 2 launches instead of 16 -- what matters once the rows are split
// over 8 GPUs and a column's reduction takes 17 us.
static int reduce_columns(bdf_ctx* c, int n_cols, bdf_col* const* cols, bdf_future* f) {
    struct Range { int64_t cta0, ctas; };
    std::vector<Range> range((size_t)n_cols);
    int64_t total_ctas = 0, total_chunks = 0;
    for (int k = 0; k < n_cols; k++) total_chunks += (int64_t)cols[k]->chunks.size();
    void *hp = nullptr, *dp = nullptr;
    TRY(ring_alloc(c, (size_t)total_chunks * sizeof(RedDesc), &hp, &dp));
    RedDesc* hd = (RedDesc*)hp;
    RedDesc* dd = (RedDesc*)dp;
    struct Launch { int dtype; int64_t desc0, n_desc, tiles, cta0; int64_t rows, bytes; };
    std::vector<Launch> launches;
    std::vector<char> done((size_t)n_cols, 0);
    int64_t di = 0;
    for (int k0 = 0; k0 < n_cols; k0++) {
        if (done[k0]) continue;
        const int dtype = cols[k0]->dtype;
        const int K = reduce_tiles_per_cta(dtype), tile = elems_per_tile(dtype);
        Launch L{dtype, di, 0, 0, total_ctas, 0, 0};
        int64_t tiles = 0;
        for (int k = k0; k < n_cols; k++) {
            if (done[k] || cols[k]->dtype != dtype) continue;
            done[k] = 1;
            tiles = (tiles + K - 1) / K * K;   // the column starts on a CTA boundary
            const int64_t col_tile0 = tiles;
            for (const DevChunk& ch : cols[k]->chunks) {
                hd[di] = RedDesc{ch.values, ch.validity, ch.len, tiles, ch.bit_off, 0};
                di++;
                tiles += (ch.len + tile - 1) / tile;
                L.rows += ch.len;
            }
            L.bytes += reduce_bytes(cols[k], 0, (int64_t)cols[k]->chunks.size());
            range[k] = Range{L.cta0 + col_tile0 / K, (tiles - col_tile0 + K - 1) / K};
        }
        L.n_desc = di - L.desc0;
        L.tiles = tiles;
        total_ctas += (tiles + K - 1) / K;
        launches.push_back(L);
    }
    CK(desc_upload(c, dd, hd, (size_t)total_chunks * sizeof(RedDesc)));
    if ((size_t)total_ctas > c->red_part_cap) {
        CK(cudaStreamSynchronize(c->s_compute));
        if (c->d_partials) CK(cudaFree(c->d_partials));
        c->d_partials = nullptr; c->red_part_cap = 0;
        const size_t cap = std::max<size_t>((size_t)total_ctas * 2, 65536);
        CK(cudaMalloc((void**)&c->d_partials, cap * sizeof(AggDev)));
        c->red_part_cap = cap;
    }
    if (!c->d_stage_many) {
        CK(cudaMalloc((void**)&c->d_stage_many, (size_t)kFinishMany * c->sm_count * sizeof(AggDev)));
        CK(cudaMalloc((void**)&c->d_tickets_many, kFinishMany * sizeof(unsigned int)));
        CK(cudaMemset(c->d_tickets_many, 0, kFinishMany * sizeof(unsigned int)));
    }
    for (const Launch& L : launches) {
        LaunchTimer t(c, BDF_K_REDUCE, L.dtype, L.rows, L.bytes);
        CK(launch_reduce(L.dtype, dd + L.desc0, (int)L.n_desc, L.tiles, c->d_partials + L.cta0, c->s_compute));
    }
    FinishJob jobs[kFinishMany];
    for (int k = 0; k < n_cols; k++)
        jobs[k] = FinishJob{c->d_partials + range[k].cta0, (long long)range[k].ctas, future_target(c, f, k), dtype_is_float(cols[k]->dtype) ? 1 : 0, 0};
    c->launches++;
    CK(launch_finish_many(n_cols, jobs, c->sm_count, c->d_stage_many, c->d_tickets_many, c->s_compute));
    return BDF_OK;
}

// Chunks of the column that are empty or all-null: the reference's max/min .unwrap() a None there (aggregate.rs:19,29).
static int count_panic_chunks(bdf_ctx* c, bdf_col* col, uint32_t* out) {
    TRY(ensure_null_counts(c, col));
    uint32_t k = 0;
    for (size_t i = 0; i < col->chunks.size(); i++)
        if (col->chunks[i].len - col->null_counts[i] == 0) k++;
    *out = k;
    return BDF_OK;
}

// sum/min/max/count of n columns: one k_reduce + k_finish per column on the compute stream and -- on a rank of a
// communicator -- ONE grouped collective for all of them.  need_counts: also evaluate the would-panic rule (may
// synchronise to learn null counts of uploaded columns).
static int aggregate_many_dev_async(bdf_ctx* c, int n_cols, bdf_col* const* cols, bool need_counts, bdf_future** fut) {
    for (int k = 0; k < n_cols; k++)
        if (cols[k]->dtype == kBool) return fail(BDF_UNSUPPORTED, "aggregate of a boolean column");
    std::vector<uint32_t> panics((size_t)n_cols, 0u);
    if (need_counts)
        for (int k = 0; k < n_cols; k++) TRY(count_panic_chunks(c, cols[k], &panics[k]));
    bdf_future* f = nullptr;
    TRY(future_new(c, cols[0]->dtype, 2, 0, &f, n_cols));
    int st = BDF_OK;
    for (int k = 0; k < n_cols; k++) {
        bdf_col* col = cols[k];
        const int64_t n = (int64_t)col->chunks.size();
        f->dtypes[k] = col->dtype; f->rows[k] = col->total_len; f->panics[k] = panics[k]; f->chunks[k] = (uint32_t)n;
        wait_groups(c->s_compute, col, 0, n);
    }
    if (n_cols == 1) st = reduce_range(c, cols[0], 0, (int64_t)cols[0]->chunks.size(), future_target(c, f, 0));
    else st = reduce_columns(c, n_cols, cols, f);
    cudaError_t e = cudaSuccess;
    if (st == BDF_OK) e = future_combine(c, f, c->s_compute);
    if (st == BDF_OK && e == cudaSuccess) e = cudaEventRecord(f->ev, c->s_compute);
    if (st != BDF_OK || e != cudaSuccess) {
        ev_put(c, f->ev); delete f;
        return st != BDF_OK ? st : fail_cuda(e, "aggregate");
    }
    *fut = f;
    return BDF_OK;
}

// Waits for the future, converts its n records into out[0..n) and consumes it.
static int future_wait(bdf_ctx* c, bdf_future* f, bdf_agg4* out) {
    cudaError_t e = cudaEventSynchronize(f->ev);
    if (e == cudaSuccess && out)
        for (int i = 0; i < f->n; i++) {
            if (f->global) {
                const AggDev& x = c->h_agg[f->slot + 2 * i + 1];   // {rows, panics, chunks} summed over the ranks
                convert_agg(f->dtypes[i], f->fused, c->h_agg[f->slot + 2 * i], (int64_t)x.sum_bits, &out[i]);
                out[i].would_panic = x.min_bits != 0;
                out[i].n_chunks = (int64_t)x.max_bits;
            } else {
                convert_agg(f->dtypes[i], f->fused, c->h_agg[f->slot + i], f->rows[i], &out[i]);
                out[i].would_panic = f->panics[i] != 0;
                out[i].n_chunks = (int64_t)f->chunks[i];
            }
        }
    ev_put(c, f->ev);
    delete f;
    if (e != cudaSuccess) return fail(cuda_status(e), "waiting for an aggregate failed: %s", cudaGetErrorString(e));
    return BDF_OK;
}

static int aggregate_all_dev(bdf_ctx* c, bdf_col* col, bool need_counts, bdf_agg4* out) {
    bdf_future* f = nullptr;
    TRY(aggregate_many_dev_async(c, 1, &col, need_counts, &f));
    return future_wait(c, f, out);
}

// count is metadata (aggregate.rs:70-80); on a rank of a communicator the other ranks' chunks count too.
static int count_global(bdf_ctx* c, int64_t* total) {
    if (!is_global(c)) return BDF_OK;
    std::vector<int64_t> all((size_t)comm_world(c->comm));
    std::string err;
    c->collectives++;
    cudaError_t e = comm_host_allgather(c->comm, total, all.data(), sizeof(int64_t), c->s_compute, &err);
    if (e != cudaSuccess) { g_nccl_err = err; return fail_cuda(e, "count"); }
    *total = 0;
    for (int64_t v : all) *total += v;
    return BDF_OK;
}

static int aggregate_dev(bdf_ctx* c, int op, bdf_col* col, void* out_scalar, int32_t* is_some) {
    const int dtype = col->dtype;
    const int w = dtype_width(dtype);
    if (op == BDF_COUNT) {  // metadata only, as in the reference (aggregate.rs:70-80)
        TRY(ensure_null_counts(c, col));
        int64_t total = 0;
        for (size_t i = 0; i < col->chunks.size(); i++) total += col->chunks[i].len - col->null_counts[i];
        TRY(count_global(c, &total));
        *(int64_t*)out_scalar = total;
        *is_some = 1;
        return BDF_OK;
    }
    bdf_agg4 a;
    TRY(aggregate_all_dev(c, col, op != BDF_SUM, &a));
    if (op == BDF_SUM) {
        memcpy(out_scalar, &a.sum, (size_t)w);
        *is_some = 1;
        return BDF_OK;
    }
    if (a.would_panic) return fail(BDF_WOULD_PANIC, "max/min on an empty or all-null chunk: the reference unwraps None");
    *is_some = a.n_chunks == 0 ? 0 : 1;   // Iterator::max of an empty Vec is None
    if (*is_some) memcpy(out_scalar, op == BDF_MIN ? &a.min : &a.max, (size_t)w);
    return BDF_OK;
}

// avg (aggregate.rs:32-65): per-chunk mean from an exact/double sum and the valid count, then the
// reference's weighted merge in chunk order.
static int avg_dev(bdf_ctx* c, bdf_col* col, double* out, int32_t* is_some) {
    const int dtype = col->dtype;
    if (dtype == BDF_I64 || dtype == BDF_U64) return fail(BDF_UNSUPPORTED, "avg needs f64: From<T::Native>");
    const int64_t n = (int64_t)col->chunks.size();
    wait_groups(c->s_compute, col, 0, n);
    double mean = 0.0;
    int64_t count = 0;
    for (int64_t k = 0; k < n; k += kAggSlots) {
        const int64_t m = std::min<int64_t>(kAggSlots, n - k);
        for (int64_t j = 0; j < m; j++) TRY(reduce_range(c, col, k + j, k + j + 1, c->h_agg_dev + j));
        CK(cudaStreamSynchronize(c->s_compute));
        for (int64_t j = 0; j < m; j++) {
            const AggDev& a = c->h_agg[j];
            const int64_t len = (int64_t)a.count;
            double s;
            if (dtype_is_float(dtype)) memcpy(&s, &a.sum_bits, 8);
            else if (dtype_is_signed_int(dtype)) s = (double)(int64_t)a.sum_bits;
            else s = (double)a.sum_bits;
            const double mch = len ? s / (double)len : 0.0;
            // A rank of a communicator sees only SOME chunks of the column: an empty local chunk contributes nothing there
            // (the reference's 0/0 = NaN when the column's FIRST chunk has no valid slot is a statement about the whole
            // column's chunk order; the one-GPU context and the multi-GPU context reproduce it, see fleet_avg_dev).
            if (len == 0 && is_global(c)) continue;
            count += len;
            mean = mean + ((mch - mean) * (double)len) / (double)count;
        }
    }
    if (is_global(c)) {
        // The reference merges per-chunk means in chunk order (aggregate.rs:44-63); the chunks of the other ranks are
        // merged as one (mean, count) pair per rank, in rank order, with the same formula.
        struct Pair { double mean; int64_t count; } mine{mean, count};
        std::vector<Pair> all((size_t)comm_world(c->comm));
        std::string err;
        c->collectives++;
        cudaError_t e = comm_host_allgather(c->comm, &mine, all.data(), sizeof(Pair), c->s_compute, &err);
        if (e != cudaSuccess) { g_nccl_err = err; return fail_cuda(e, "avg"); }
        mean = 0.0; count = 0;
        for (const Pair& p : all) {
            if (!p.count) continue;
            count += p.count;
            mean = mean + ((p.mean - mean) * (double)p.count) / (double)count;
        }
    }
    *is_some = count != 0;
    *out = mean;
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// N2: BooleanFilter comparisons, boolean kernels, filter (k_filter.cu)

namespace bdf {
cudaError_t launch_compare(int op, const BinDesc* d, int n, int64_t tiles, int ta, int tb, bool scalar_rhs, double scalar, uint32_t* wc,
                           cudaStream_t s);
int compare_tile_elems();
int bool_tile_elems();
cudaError_t launch_boolean(int op, const void* d, int n, int64_t tiles, uint32_t* wc, cudaStream_t s);
cudaError_t launch_filter_count(const void* d, int n, int64_t tiles, int tile_elems, unsigned int* tile_counts, long long* tile_offsets,
                                long long* chunk_totals, cudaStream_t s);
cudaError_t launch_filter_scatter(int dtype, const void* d, int n, int64_t tiles, const long long* tile_offsets, cudaStream_t s);
size_t filter_desc_size();
size_t bool_desc_size();
void fill_filter_desc(void* base, int64_t i, const void* in, void* out, const uint32_t* vin, uint32_t* vout, const uint32_t* mval,
                      const uint32_t* mvalid, int64_t len, int64_t tile0, int off, int moff, int mvoff);
void fill_bool_desc(void* base, int64_t i, const uint32_t* a, const uint32_t* b, uint32_t* out, const uint32_t* va, const uint32_t* vb,
                    uint32_t* vout, int64_t len, int64_t tile0, int offa, int offb, int voffa, int voffb);
}  // namespace bdf

static cudaError_t finish_single_group(bdf_ctx* c, bdf_col* o) {
    Group g{0, (int64_t)o->chunks.size(), nullptr};
    cudaError_t e = ev_get(c, &g.ev);
    if (e == cudaSuccess) e = cudaEventRecord(g.ev, c->s_compute);
    o->groups.push_back(g);
    return e;
}

// BooleanFilter::{Gt,..,Le}: cast both sides to Float64 (as the reference does, expression.rs:820-845), compare.
static int compare_dev(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, double scalar, bdf_col** out) {
    if (op < 0 || op > 5) return fail(BDF_INVALID, "invalid comparison op %d", op);
    if (l->dtype == kBool || (r && r->dtype == kBool)) return fail(BDF_UNSUPPORTED, "comparison of boolean columns is not part of this path");
    auto cleanup = [] {};  // (the Float64 casts of the reference are fused into the kernel's loads)
    const int64_t n = r ? std::min<int64_t>((int64_t)l->chunks.size(), (int64_t)r->chunks.size()) : (int64_t)l->chunks.size();
    for (int64_t i = 0; r && i < n; i++)
        if (l->chunks[i].len != r->chunks[i].len) { cleanup(); return fail(BDF_LENGTH_MISMATCH, "Cannot perform math operation on arrays of different length"); }
    std::vector<ChunkPlan> plan((size_t)n);
    for (int64_t i = 0; i < n; i++) plan[i] = {l->chunks[i].len, l->chunks[i].validity != nullptr || (r && r->chunks[i].validity != nullptr)};
    const int tile = compare_tile_elems();
    bdf_col* o = nullptr;
    int st = col_alloc(c, kBool, plan, nullptr, tile, &o);
    if (st != BDF_OK) { cleanup(); return st; }
    o->counts_on_device = o->d_warp_counts != nullptr;
    void *hp = nullptr, *dp = nullptr;
    st = ring_alloc(c, (size_t)n * sizeof(BinDesc), &hp, &dp);
    cudaError_t e = cudaSuccess;
    if (st == BDF_OK) {
        BinDesc* hd = (BinDesc*)hp;
        int64_t tiles = 0, rows = 0, bytes = 0;
        for (int64_t i = 0; i < n; i++) {
            const DevChunk& a = l->chunks[i];
            const DevChunk* b = r ? &r->chunks[i] : nullptr;
            const DevChunk& oc = o->chunks[i];
            hd[i] = BinDesc{a.values, b ? b->values : nullptr, oc.values, a.validity, b ? b->validity : nullptr, oc.validity, a.len, tiles,
                            a.bit_off, b ? b->bit_off : 0};
            tiles += (a.len + tile - 1) / tile;
            rows += a.len;
            bytes += (dtype_width(l->dtype) + (b ? dtype_width(r->dtype) : 0)) * a.len +
                     bitmap_bytes(a.len) * (1 + (a.validity ? 1 : 0) + (b && b->validity ? 1 : 0) + (oc.validity ? 1 : 0));
        }
        wait_groups(c->s_compute, l, 0, n);
        if (r) wait_groups(c->s_compute, r, 0, n);
        e = desc_upload(c, dp, hd, (size_t)n * sizeof(BinDesc));
        if (e == cudaSuccess) {
            LaunchTimer t(c, BDF_K_COMPARE, kBool, rows, bytes);
            e = launch_compare(op, (const BinDesc*)dp, (int)n, tiles, l->dtype, r ? r->dtype : BDF_F64, r == nullptr, scalar, o->d_warp_counts, c->s_compute);
        }
        if (e == cudaSuccess) e = finish_single_group(c, o);
    }
    cleanup();
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return st != BDF_OK ? st : fail(cuda_status(e), "compare failed: %s", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

static int boolean_dev(bdf_ctx* c, int op, const bdf_col* a, const bdf_col* b, bdf_col** out) {
    if (op < 0 || op > 2) return fail(BDF_INVALID, "invalid boolean op %d", op);
    if (a->dtype != kBool || (op != 2 && (!b || b->dtype != kBool))) return fail(BDF_UNSUPPORTED, "and/or/not need boolean columns");
    if (op == 2) b = nullptr;
    const int64_t n = b ? std::min<int64_t>((int64_t)a->chunks.size(), (int64_t)b->chunks.size()) : (int64_t)a->chunks.size();
    for (int64_t i = 0; b && i < n; i++)
        if (a->chunks[i].len != b->chunks[i].len) return fail(BDF_LENGTH_MISMATCH, "Cannot perform math operation on arrays of different length");
    std::vector<ChunkPlan> plan((size_t)n);
    for (int64_t i = 0; i < n; i++) plan[i] = {a->chunks[i].len, a->chunks[i].validity != nullptr || (b && b->chunks[i].validity != nullptr)};
    const int tile = bool_tile_elems();
    bdf_col* o = nullptr;
    TRY(col_alloc(c, kBool, plan, nullptr, tile, &o));
    o->counts_on_device = o->d_warp_counts != nullptr;
    void *hp = nullptr, *dp = nullptr;
    int st = ring_alloc(c, (size_t)n * bool_desc_size(), &hp, &dp);
    cudaError_t e = cudaSuccess;
    if (st == BDF_OK) {
        int64_t tiles = 0, rows = 0;
        for (int64_t i = 0; i < n; i++) {
            const DevChunk& x = a->chunks[i];
            const DevChunk* y = b ? &b->chunks[i] : nullptr;
            const DevChunk& oc = o->chunks[i];
            fill_bool_desc(hp, i, (const uint32_t*)x.values, y ? (const uint32_t*)y->values : nullptr, (uint32_t*)oc.values, x.validity,
                           y ? y->validity : nullptr, oc.validity, x.len, tiles, x.val_bit_off, y ? y->val_bit_off : 0, x.bit_off, y ? y->bit_off : 0);
            tiles += (x.len + tile - 1) / tile;
            rows += x.len;
        }
        wait_groups(c->s_compute, a, 0, n);
        if (b) wait_groups(c->s_compute, b, 0, n);
        e = desc_upload(c, dp, hp, (size_t)n * bool_desc_size());
        if (e == cudaSuccess) {
            LaunchTimer t(c, BDF_K_COMPARE, kBool, rows, rows / 8 * (b ? 3 : 2));
            e = launch_boolean(op, dp, (int)n, tiles, o->d_warp_counts, c->s_compute);
        }
        if (e == cudaSuccess) e = finish_single_group(c, o);
    }
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return st != BDF_OK ? st : fail(cuda_status(e), "boolean op failed: %s", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

// ChunkedArray::filter: arrow compute::filter(chunk, mask chunk) for every chunk pair (src/table.rs:97-107).
static int filter_dev(bdf_ctx* c, const bdf_col* values, const bdf_col* mask, bdf_col** out) {
    if (mask->dtype != kBool) return fail(BDF_INVALID, "the filter mask must be a boolean column");
    if (values->dtype == kBool) return fail(BDF_UNSUPPORTED, "filtering a boolean column is not part of this path");
    const int64_t n = std::min<int64_t>((int64_t)values->chunks.size(), (int64_t)mask->chunks.size());  // zip()
    for (int64_t i = 0; i < n; i++)
        if (values->chunks[i].len != mask->chunks[i].len)
            return fail(BDF_LENGTH_MISMATCH, "Filter array must have the same length as the data");
    const int dtype = values->dtype;
    const int tile = elems_per_tile(dtype);
    int64_t tiles = 0, rows = 0;
    std::vector<int64_t> tile0((size_t)n + 1, 0);
    for (int64_t i = 0; i < n; i++) { tile0[i] = tiles; tiles += (values->chunks[i].len + tile - 1) / tile; rows += values->chunks[i].len; }
    void *hp = nullptr, *dp = nullptr;
    TRY(ring_alloc(c, (size_t)n * filter_desc_size(), &hp, &dp));
    unsigned int* d_counts = nullptr; long long *d_offsets = nullptr, *d_totals = nullptr;
    auto free_scratch = [&]() {
        if (d_counts) cudaFreeAsync(d_counts, c->s_compute);
        if (d_offsets) cudaFreeAsync(d_offsets, c->s_compute);
        if (d_totals) cudaFreeAsync(d_totals, c->s_compute);
    };
    {   // three scratch arrays; a failure part-way frees what was already obtained
        cudaError_t ea = cudaMallocAsync((void**)&d_counts, std::max<size_t>(1, (size_t)tiles) * sizeof(unsigned int), c->s_compute);
        if (ea == cudaSuccess) ea = cudaMallocAsync((void**)&d_offsets, std::max<size_t>(1, (size_t)tiles) * sizeof(long long), c->s_compute);
        if (ea == cudaSuccess) ea = cudaMallocAsync((void**)&d_totals, std::max<size_t>(1, (size_t)n) * sizeof(long long), c->s_compute);
        if (ea != cudaSuccess) {
            cudaGetLastError();
            free_scratch();
            return fail(cuda_status(ea), "filter scratch allocation failed: %s", cudaGetErrorString(ea));
        }
    }
    // pass 1: counts + scan (output pointers are not needed yet)
    for (int64_t i = 0; i < n; i++) {
        const DevChunk &v = values->chunks[i], &m = mask->chunks[i];
        fill_filter_desc(hp, i, v.values, nullptr, v.validity, nullptr, (const uint32_t*)m.values, m.validity, v.len, tile0[i], v.bit_off, m.val_bit_off, m.bit_off);
    }
    wait_groups(c->s_compute, values, 0, n);
    wait_groups(c->s_compute, mask, 0, n);
    cudaError_t e = desc_upload(c, dp, hp, (size_t)n * filter_desc_size());
    std::vector<long long> totals((size_t)std::max<int64_t>(n, 1), 0);
    if (e == cudaSuccess) {
        LaunchTimer t(c, BDF_K_FILTER, dtype, rows, rows / 4);
        c->launches++;  // count + scan
        e = launch_filter_count(dp, (int)n, tiles, tile, d_counts, d_offsets, d_totals, c->s_compute);
    }
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(totals.data(), d_totals, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost, c->s_compute);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->s_compute);  // output lengths are needed to size the result
    if (e != cudaSuccess) { cudaGetLastError(); free_scratch(); return fail(cuda_status(e), "filter (count) failed: %s", cudaGetErrorString(e)); }
    std::vector<ChunkPlan> plan((size_t)n);
    int64_t kept = 0;
    for (int64_t i = 0; i < n; i++) { plan[i] = {(int64_t)totals[i], values->chunks[i].validity != nullptr}; kept += totals[i]; }
    bdf_col* o = nullptr;
    int st = col_alloc(c, dtype, plan, nullptr, 0, &o);
    if (st != BDF_OK) { free_scratch(); return st; }
    for (int64_t i = 0; i < n; i++) o->null_counts[i] = o->chunks[i].validity ? -1 : 0;  // counted on demand
    // pass 2: scatter
    void *hp2 = nullptr, *dp2 = nullptr;
    st = ring_alloc(c, (size_t)n * filter_desc_size(), &hp2, &dp2);
    if (st == BDF_OK) {
        for (int64_t i = 0; i < n; i++) {
            const DevChunk &v = values->chunks[i], &m = mask->chunks[i], &oc = o->chunks[i];
            fill_filter_desc(hp2, i, v.values, oc.values, v.validity, oc.validity, (const uint32_t*)m.values, m.validity, v.len, tile0[i], v.bit_off, m.val_bit_off, m.bit_off);
        }
        e = desc_upload(c, dp2, hp2, (size_t)n * filter_desc_size());
        if (e == cudaSuccess) {
            const int w = dtype_width(dtype);
            LaunchTimer t(c, BDF_K_FILTER, dtype, rows, rows * w + kept * w + rows / 4);
            e = launch_filter_scatter(dtype, dp2, (int)n, tiles, d_offsets, c->s_compute);
        }
        if (e == cudaSuccess) e = finish_single_group(c, o);
    }
    free_scratch();
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return st != BDF_OK ? st : fail(cuda_status(e), "filter (scatter) failed: %s", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// N3: a chain of Calculations fused into one pass (k_expr.cu)

namespace bdf {
int expr_tile_elems();
int expr_max_inputs();
int expr_max_nodes();
size_t expr_desc_size();
void fill_expr_desc(void* base, int64_t i, int n_inputs, const void* const* in, const uint32_t* const* vin, const int32_t* off, double* out,
                    uint32_t* vout, int64_t len, int64_t tile0);
size_t expr_prog_size();
void expr_prog_stats(const void* prog, int* n_instructions, int* n_temporaries);
int expr_compile(int n_inputs, const int* in_dtypes, int n_nodes, const int* op, const int* a, const int* b, void* prog);
cudaError_t launch_expr(const void* descs, int n_chunks, int64_t tiles, const void* prog, uint32_t* warp_counts, int* flags, AggDev* tile_partials,
                        cudaStream_t s);
}  // namespace bdf

// Validation + host compilation of a fused program (shared by the evaluation entry and bdf_expr_check; needs no device).
static int expr_prepare(int n_inputs, const int* in_dtypes, int n_nodes, const bdf_expr_node* nodes, unsigned char (&prog)[256], bool* has_div) {
    if (n_inputs < 1 || n_inputs > expr_max_inputs()) return fail(BDF_INVALID, "an expression takes 1..%d input columns", expr_max_inputs());
    if (n_nodes < 1 || n_nodes > expr_max_nodes()) return fail(BDF_INVALID, "an expression has 1..%d nodes", expr_max_nodes());
    std::vector<int> op(n_nodes), a(n_nodes), b(n_nodes);
    *has_div = false;
    for (int k = 0; k < n_nodes; k++) {
        op[k] = nodes[k].op; a[k] = nodes[k].a; b[k] = nodes[k].b;
        const bool unary = op[k] >= BDF_EXPR_UNARY;
        if (unary ? (op[k] - BDF_EXPR_UNARY >= BDF_NUNARY) : (op[k] < 0 || op[k] >= BDF_NBINARY)) return fail(BDF_INVALID, "node %d: invalid op %d", k, op[k]);
        if (a[k] < 0 || a[k] >= n_inputs + k || (!unary && (b[k] < 0 || b[k] >= n_inputs + k)))
            return fail(BDF_INVALID, "node %d refers to a slot that is not computed yet", k);
        if (unary) b[k] = a[k];
        *has_div = *has_div || op[k] == BDF_DIV;
    }
    static_assert(sizeof(prog) >= 8 + 2 * 40, "ExprProg must fit");
    if (expr_prog_size() > sizeof(prog)) return fail(BDF_INVALID, "internal: expression program too large");
    for (int i = 0; i < n_inputs; i++)
        if (in_dtypes[i] < 0 || in_dtypes[i] >= BDF_NTYPES) return fail(BDF_UNSUPPORTED, "fused expressions take numeric columns");
    switch (expr_compile(n_inputs, in_dtypes, n_nodes, op.data(), a.data(), b.data(), prog)) {
        case 0: return BDF_OK;
        case 1: return fail(BDF_INVALID, "a node's result is never used: the materialised chain would still evaluate it, split the expression");
        case 2: return fail(BDF_UNSUPPORTED, "the expression keeps more than two intermediates alive at once: split it");
        default: return fail(BDF_UNSUPPORTED, "the expression is too long to fuse: split it");
    }
}

// prog: the program expr_prepare compiled.  out == nullptr (only with fut): aggregate only, the result column is never written.
static int expr_dev(bdf_ctx* c, int n_inputs, const bdf_col* const* inputs, const unsigned char* prog, bool has_div, bdf_col** out,
                    bdf_future** fut) {
    int64_t n = (int64_t)inputs[0]->chunks.size();
    for (int i = 0; i < n_inputs; i++) {
        n = std::min<int64_t>(n, (int64_t)inputs[i]->chunks.size());
    }
    for (int64_t ch = 0; ch < n; ch++)
        for (int i = 1; i < n_inputs; i++)
            if (inputs[i]->chunks[ch].len != inputs[0]->chunks[ch].len)
                return fail(BDF_LENGTH_MISMATCH, "Cannot perform math operation on arrays of different length");
    std::vector<ChunkPlan> plan((size_t)n);
    for (int64_t ch = 0; ch < n; ch++) {
        bool hv = false;
        for (int i = 0; i < n_inputs; i++) hv = hv || inputs[i]->chunks[ch].validity != nullptr;
        plan[ch] = {inputs[0]->chunks[ch].len, hv};
    }
    const int tile = expr_tile_elems();
    bdf_col* o = nullptr;
    if (out) {
        TRY(col_alloc(c, BDF_F64, plan, nullptr, tile, &o));
        o->counts_on_device = o->d_warp_counts != nullptr;
    }
    int64_t total_tiles = 0, total_rows = 0;
    for (int64_t ch = 0; ch < n; ch++) { total_tiles += (plan[ch].len + tile - 1) / tile; total_rows += plan[ch].len; }
    void *hp = nullptr, *dp = nullptr;
    int st = ring_alloc(c, (size_t)n * expr_desc_size(), &hp, &dp);
    cudaError_t e = cudaSuccess;
    bdf_future* f = nullptr;
    bdf_ctx::PartBuf* pb = nullptr;
    if (fut && st == BDF_OK) {
        st = future_new(c, BDF_F64, 1, total_rows, &f);
        if (st == BDF_OK) e = part_acquire(c, total_tiles, &pb);
    }
    cudaEvent_t ev_done = nullptr;   // the launch's completion on the compute stream, for the finish stream
    if (st == BDF_OK && e == cudaSuccess) {
        int64_t tiles = 0, bytes = 0;
        for (int64_t ch = 0; ch < n; ch++) {
            const void* in[8]; const uint32_t* vin[8]; int32_t off[8];
            const int64_t len = plan[ch].len;
            for (int i = 0; i < n_inputs; i++) {
                const DevChunk& x = inputs[i]->chunks[ch];
                in[i] = x.values; vin[i] = x.validity; off[i] = x.bit_off;
                if ((uintptr_t)x.values & 15) e = cudaErrorMisalignedAddress;
                bytes += (int64_t)dtype_width(inputs[i]->dtype) * x.len + (x.validity ? bitmap_bytes(x.len) : 0);
            }
            double* po = o ? (double*)o->chunks[ch].values : nullptr;
            uint32_t* vo = o ? o->chunks[ch].validity : nullptr;
            fill_expr_desc(hp, ch, n_inputs, in, vin, off, po, vo, len, tiles);
            tiles += (len + tile - 1) / tile;
            if (o) bytes += 8 * len + (vo ? bitmap_bytes(len) : 0);
        }
        for (int i = 0; i < n_inputs; i++) wait_groups(c->s_compute, inputs[i], 0, n);
        if (e == cudaSuccess) e = desc_upload(c, dp, hp, (size_t)n * expr_desc_size());
        if (e == cudaSuccess && has_div) e = cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->s_compute);
        if (e == cudaSuccess) {
            LaunchTimer t(c, BDF_K_EXPR, BDF_F64, total_rows, bytes);
            e = launch_expr(dp, (int)n, total_tiles, prog, o ? o->d_warp_counts : nullptr, c->d_flag, pb ? pb->p : nullptr, c->s_compute);
        }
        if (e == cudaSuccess && o) e = finish_single_group(c, o);
        if (e == cudaSuccess && f) {
            // fold the per-tile partials on the finish stream, like K5
            c->launches++;
            e = ev_get(c, &ev_done);
            if (e == cudaSuccess) e = cudaEventRecord(ev_done, c->s_compute);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(c->s_fin, ev_done, 0);
            if (e == cudaSuccess) e = launch_finish(true, pb->p, total_tiles, c->sm_count, c->d_stage, c->d_ticket + 1, future_target(c, f, 0), c->s_fin);
            if (e == cudaSuccess) e = cudaEventRecord(pb->done, c->s_fin);
            pb->used = true;
            f->chunks[0] = (uint32_t)n;
            if (e == cudaSuccess) e = future_combine(c, f, c->s_fin);
            if (e == cudaSuccess) e = cudaEventRecord(f->ev, c->s_fin);
            if (ev_done) ev_put(c, ev_done);
        }
        if (e == cudaSuccess && has_div) {
            if (is_global(c)) e = flag_allreduce(c);
            if (e == cudaSuccess) e = cudaMemcpyAsync(c->h_flag, c->d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->s_compute);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->s_compute);
            if (e == cudaSuccess && *c->h_flag) {
                if (o) col_release(c, o);
                if (f) { ev_put(c, f->ev); delete f; }
                return fail(BDF_DIVIDE_BY_ZERO, "Divide by zero error");
            }
        }
    }
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        if (o) col_release(c, o);
        if (f) { ev_put(c, f->ev); delete f; }
        return st != BDF_OK ? st : fail_cuda(e, "fused expression");
    }
    if (out) *out = o;
    if (fut) *fut = f;
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// DataFrame::sort = lexsort_to_indices + take (k_sort.cu)

namespace bdf {
size_t sort_chunk_size();
void fill_sort_chunk(void* base, int64_t i, const void* values, const uint32_t* validity, int64_t start, int32_t bit_off, int32_t val_bit_off);
int sort_tile_elems();
int take_tile_elems();
int sort_pass_ctas(int64_t n, int sm_count);
cudaError_t launch_iota(uint32_t* out, int64_t n, int sm_count, cudaStream_t s);
int sort_key_bytes(int dtype);
cudaError_t launch_sort_keys(int dtype, const void* chunks, int n_chunks, const uint32_t* idx, int64_t n, int mode, int descending,
                             void* keys, unsigned long long* agree, int sm_count, cudaStream_t s);
cudaError_t launch_radix_pass(int key_bytes, const void* keys_in, const uint32_t* idx_in, int64_t n, int shift, unsigned int* block_hist,
                              void* keys_out, uint32_t* idx_out, int sm_count, cudaStream_t s);
cudaError_t launch_take(int dtype, const void* vals, int n_vals, const void* idxs, int n_idxs, int64_t n, int64_t n_rows_values, void* out,
                        uint32_t* vout, uint32_t* warp_counts, int* flags, cudaStream_t s);
}  // namespace bdf

// The chunk table of a column in the concatenated row space (descriptor ring, uploaded on the descriptor stream).
static int sort_table(bdf_ctx* c, const bdf_col* col, void** dev, int* n_chunks, bool* nullable) {
    const int64_t n = (int64_t)col->chunks.size();
    void* hp = nullptr;
    TRY(ring_alloc(c, (size_t)std::max<int64_t>(n, 1) * sort_chunk_size(), &hp, dev));
    int64_t start = 0;
    bool any = false;
    for (int64_t i = 0; i < n; i++) {
        const DevChunk& ch = col->chunks[i];
        fill_sort_chunk(hp, i, ch.values, ch.validity, start, ch.bit_off, ch.val_bit_off);
        start += ch.len;
        any = any || ch.validity != nullptr;
    }
    if (n == 0) fill_sort_chunk(hp, 0, nullptr, nullptr, 0, 0, 0);
    wait_groups(c->s_compute, col, 0, n);
    cudaError_t e = desc_upload(c, *dev, hp, (size_t)std::max<int64_t>(n, 1) * sort_chunk_size());
    if (e != cudaSuccess) return fail(cuda_status(e), "descriptor upload failed: %s", cudaGetErrorString(e));
    *n_chunks = (int)std::max<int64_t>(n, 1);
    if (nullable) *nullable = any;
    return BDF_OK;
}

static int sort_indices_dev(bdf_ctx* c, int n_keys, const bdf_sort_key* keys, bdf_col** out) {
    if (n_keys < 1) return fail(BDF_INVALID, "Sort criteria cannot be empty");
    for (int k = 0; k < n_keys; k++) {
        const int dt = keys[k].column->dtype;
        if (dt < 0 || dt >= BDF_NTYPES) return fail(BDF_UNSUPPORTED, "sort criteria must be numeric columns");
        if (keys[k].column->total_len != keys[0].column->total_len) return fail(BDF_LENGTH_MISMATCH, "sort columns have different lengths");
    }
    const int64_t n = keys[0].column->total_len;
    if (n > 0xffffffffLL) return fail(BDF_UNSUPPORTED, "sort indices are UInt32: at most 2^32-1 rows");
    bdf_col* o = nullptr;
    TRY(col_alloc(c, BDF_U32, {ChunkPlan{n, false}}, nullptr, sort_tile_elems(), &o));
    cudaError_t e = cudaSuccess;
    int st = BDF_OK;
    unsigned long long* kbuf[2] = {nullptr, nullptr};
    uint32_t* ibuf[2] = {nullptr, nullptr};
    unsigned int* block_hist = nullptr;
    unsigned long long* agree = nullptr;   // [0] OR, [1] AND of the keys of the current criterion
    if (n > 0) {
        if (!c->h_sort_agree) e = cudaHostAlloc((void**)&c->h_sort_agree, 2 * sizeof(unsigned long long), cudaHostAllocDefault);
        for (int b = 0; b < 2 && e == cudaSuccess; b++) {
            e = cudaMallocAsync((void**)&kbuf[b], (size_t)n * 8, c->s_compute);
            if (e == cudaSuccess) e = cudaMallocAsync((void**)&ibuf[b], (size_t)n * 4, c->s_compute);
        }
        if (e == cudaSuccess) e = cudaMallocAsync((void**)&block_hist, (size_t)256 * sort_pass_ctas(n, c->sm_count) * sizeof(unsigned int), c->s_compute);
        if (e == cudaSuccess) e = cudaMallocAsync((void**)&agree, 2 * sizeof(unsigned long long), c->s_compute);
        int cur = 0;
        int64_t passes = 0, pass_bytes = 0;
        if (e == cudaSuccess) {
            LaunchTimer t(c, BDF_K_SORT, keys[0].column->dtype, n, 0);
            e = launch_iota(ibuf[0], n, c->sm_count, c->s_compute);
            for (int k = n_keys - 1; k >= 0 && e == cudaSuccess && st == BDF_OK; k--) {
                const bdf_col* col = keys[k].column;
                void* table = nullptr; int nch = 0; bool nullable = false;
                st = sort_table(c, col, &table, &nch, &nullable);
                for (int mode = 0; mode < (nullable ? 2 : 1) && e == cudaSuccess && st == BDF_OK; mode++) {
                    e = cudaMemsetAsync(agree, 0, sizeof(unsigned long long), c->s_compute);
                    if (e == cudaSuccess) e = cudaMemsetAsync(agree + 1, 0xff, sizeof(unsigned long long), c->s_compute);
                    if (e == cudaSuccess) e = launch_sort_keys(col->dtype, table, nch, ibuf[cur], n, mode, keys[k].descending != 0, kbuf[cur], agree, c->sm_count, c->s_compute);
                    if (e == cudaSuccess) e = cudaMemcpyAsync(c->h_sort_agree, agree, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->s_compute);
                    if (e == cudaSuccess) e = cudaStreamSynchronize(c->s_compute);
                    const int digits = mode ? 1 : dtype_width(col->dtype);
                    const unsigned long long differ = e == cudaSuccess ? (c->h_sort_agree[0] ^ c->h_sort_agree[1]) : 0ull;   // bits that are not the same in all keys
                    for (int d = 0; d < digits && e == cudaSuccess; d++) {
                        if (((differ >> (8 * d)) & 0xff) == 0) continue;   // every key has the same digit: the pass would be the identity
                        const int kb = sort_key_bytes(col->dtype);
                        e = launch_radix_pass(kb, kbuf[cur], ibuf[cur], n, 8 * d, block_hist, kbuf[cur ^ 1], ibuf[cur ^ 1], c->sm_count, c->s_compute);
                        cur ^= 1;
                        passes++;
                        pass_bytes += (int64_t)(3 * kb + 8) * n;   // histogram read + keys and indices read and written
                    }
                }
            }
            if (e == cudaSuccess && st == BDF_OK)
                e = cudaMemcpyAsync(o->chunks[0].values, ibuf[cur], (size_t)n * 4, cudaMemcpyDeviceToDevice, c->s_compute);
            c->last_sort_passes = passes;
        }
        if (c->profiling && !c->prof.empty() && c->prof.back().rec.kernel == BDF_K_SORT) c->prof.back().rec.bytes = 8 * n + pass_bytes + 4 * n;
        for (int b = 0; b < 2; b++) { if (kbuf[b]) cudaFreeAsync(kbuf[b], c->s_compute); if (ibuf[b]) cudaFreeAsync(ibuf[b], c->s_compute); }
        if (block_hist) cudaFreeAsync(block_hist, c->s_compute);
        if (agree) cudaFreeAsync(agree, c->s_compute);
    }
    if (e == cudaSuccess && st == BDF_OK) e = finish_single_group(c, o);
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return st != BDF_OK ? st : fail(cuda_status(e), "sort failed: %s", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

static int take_dev(bdf_ctx* c, const bdf_col* values, const bdf_col* indices, bdf_col** out) {
    if (indices->dtype != BDF_U32) return fail(BDF_UNSUPPORTED, "take indices must be a UInt32 column");
    const int64_t n = indices->total_len;
    void *vt = nullptr, *it = nullptr;
    int nv = 0, ni = 0;
    bool vnull = false, inull = false;
    TRY(sort_table(c, values, &vt, &nv, &vnull));
    TRY(sort_table(c, indices, &it, &ni, &inull));
    bdf_col* o = nullptr;
    TRY(col_alloc(c, values->dtype, {ChunkPlan{n, vnull || inull}}, nullptr, take_tile_elems(), &o));
    o->counts_on_device = o->d_warp_counts != nullptr;
    cudaError_t e = cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->s_compute);
    if (e == cudaSuccess) {
        const int w = values->dtype == kBool ? 1 : dtype_width(values->dtype);
        LaunchTimer t(c, BDF_K_TAKE, values->dtype, n, n * (4 + 2 * (int64_t)w));
        e = launch_take(values->dtype, vt, nv, it, ni, n, values->total_len, o->chunks[0].values, o->chunks[0].validity, o->d_warp_counts, c->d_flag, c->s_compute);
    }
    if (e == cudaSuccess) e = finish_single_group(c, o);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c->h_flag, c->d_flag, sizeof(int), cudaMemcpyDeviceToHost, c->s_compute);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->s_compute);
    if (e == cudaSuccess && *c->h_flag) { col_release(c, o); return fail(BDF_INVALID, "take: index out of bounds"); }
    if (e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return fail(cuda_status(e), "take failed: %s", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// group-by aggregate (k_group.cu): sort the key, gather, mark group heads, compact keys and group starts, one warp per group

namespace bdf {
cudaError_t launch_group_heads(int dtype, const void* key, const uint32_t* kvalid, long long n, uint32_t* words, cudaStream_t s);
cudaError_t launch_group_reduce(int dtype, const void* val, const uint32_t* vvalid, const uint32_t* starts, long long n_groups, long long n_rows,
                                void* sum, long long* count, void* mn, void* mx, uint32_t* mm_valid, void* scratch, int sm_count, cudaStream_t s);
size_t group_big_scratch_bytes(long long n_rows);
}  // namespace bdf

static int group_aggregate_dev(bdf_ctx* c, const bdf_col* key, int n_values, const bdf_col* const* values, bdf_col** out_keys,
                               bdf_group_out* outs, int64_t* n_groups_out) {
    if (key->dtype < 0 || key->dtype >= BDF_NTYPES) return fail(BDF_UNSUPPORTED, "the group key must be a numeric column");
    for (int j = 0; j < n_values; j++) {
        if (values[j]->dtype < 0 || values[j]->dtype >= BDF_NTYPES) return fail(BDF_UNSUPPORTED, "aggregated columns must be numeric");
        if (values[j]->total_len != key->total_len) return fail(BDF_LENGTH_MISMATCH, "key and value columns have different lengths");
    }
    const int64_t n = key->total_len;
    std::vector<bdf_col*> tmp;   // everything made on the way; released at the end whatever happens
    std::vector<bdf_col*> made;  // the results (released only on failure)
    auto cleanup = [&](bool fail_too) {
        for (bdf_col* t : tmp) col_release(c, t);
        if (fail_too) for (bdf_col* t : made) col_release(c, t);
    };
    int st = BDF_OK;
    cudaError_t e = cudaSuccess;
    bdf_col *idx = nullptr, *skey = nullptr, *head = nullptr, *iota = nullptr, *starts = nullptr, *ukeys = nullptr;
    const bdf_sort_key sk{key, 0};
    st = sort_indices_dev(c, 1, &sk, &idx);
    if (st == BDF_OK) { tmp.push_back(idx); st = take_dev(c, key, idx, &skey); }
    if (st == BDF_OK) { tmp.push_back(skey); st = col_alloc(c, kBool, {ChunkPlan{n, false}}, nullptr, 0, &head); }
    if (st == BDF_OK) {
        tmp.push_back(head);
        wait_groups(c->s_compute, skey, 0, 1);
        c->launches++;
        e = launch_group_heads(skey->dtype, skey->chunks[0].values, skey->chunks[0].validity, n, (uint32_t*)head->chunks[0].values, c->s_compute);
        if (e == cudaSuccess) e = finish_single_group(c, head);
        if (e != cudaSuccess) st = fail_cuda(e, "group heads");
    }
    if (st == BDF_OK) st = filter_dev(c, skey, head, &ukeys);                       // the distinct keys, ascending, null key last
    if (st == BDF_OK) { made.push_back(ukeys); st = col_alloc(c, BDF_U32, {ChunkPlan{n, false}}, nullptr, 0, &iota); }
    if (st == BDF_OK) {
        tmp.push_back(iota);
        c->launches++;
        e = n > 0 ? launch_iota((uint32_t*)iota->chunks[0].values, n, c->sm_count, c->s_compute) : cudaSuccess;
        if (e == cudaSuccess) e = finish_single_group(c, iota);
        if (e != cudaSuccess) st = fail_cuda(e, "group iota");
    }
    if (st == BDF_OK) st = filter_dev(c, iota, head, &starts);                     // first sorted row of every group
    int64_t n_groups = 0;
    if (st == BDF_OK) { tmp.push_back(starts); n_groups = starts->chunks.empty() ? 0 : starts->chunks[0].len; }
    for (int j = 0; j < n_values && st == BDF_OK; j++) {
        const int dt = values[j]->dtype;
        const bool is_float = dtype_is_float(dt);
        bdf_col* sval = nullptr;
        st = take_dev(c, values[j], idx, &sval);
        if (st != BDF_OK) break;
        tmp.push_back(sval);
        bdf_col *csum = nullptr, *ccnt = nullptr, *cmin = nullptr, *cmax = nullptr;
        st = col_alloc(c, dt, {ChunkPlan{n_groups, false}}, nullptr, 0, &csum);
        if (st == BDF_OK) { made.push_back(csum); st = col_alloc(c, BDF_I64, {ChunkPlan{n_groups, false}}, nullptr, 0, &ccnt); }
        if (st == BDF_OK) made.push_back(ccnt);
        if (st == BDF_OK && !is_float) {
            st = col_alloc(c, dt, {ChunkPlan{n_groups, true}}, nullptr, 0, &cmin);
            if (st == BDF_OK) { made.push_back(cmin); st = col_alloc(c, dt, {ChunkPlan{n_groups, true}}, nullptr, 0, &cmax); }
            if (st == BDF_OK) made.push_back(cmax);
        }
        if (st != BDF_OK) break;
        wait_groups(c->s_compute, sval, 0, 1);
        wait_groups(c->s_compute, starts, 0, 1);
        {
            const int w = dtype_width(dt);
            LaunchTimer t(c, BDF_K_GROUP, dt, n, n * w + (sval->chunks[0].validity ? bitmap_bytes(n) : 0) + n_groups * (4 + (is_float ? 1 : 3) * w + 8));
            void* scratch = nullptr;
            e = cudaMallocAsync(&scratch, group_big_scratch_bytes(n), c->s_compute);
            c->launches += 2;   // hot keys: k_group_big + k_group_big_finish
            if (e == cudaSuccess)
                e = launch_group_reduce(dt, sval->chunks[0].values, sval->chunks[0].validity, (const uint32_t*)starts->chunks[0].values, n_groups, n,
                                        csum->chunks[0].values, (long long*)ccnt->chunks[0].values, cmin ? cmin->chunks[0].values : nullptr,
                                        cmax ? cmax->chunks[0].values : nullptr, cmin ? cmin->chunks[0].validity : nullptr, scratch, c->sm_count, c->s_compute);
            if (scratch) cudaFreeAsync(scratch, c->s_compute);
        }
        // max shares min's validity pattern: copy the bitmap rather than set it twice with atomics
        if (e == cudaSuccess && cmin && n_groups)
            e = cudaMemcpyAsync(cmax->chunks[0].validity, cmin->chunks[0].validity, (size_t)bitmap_bytes(n_groups), cudaMemcpyDeviceToDevice, c->s_compute);
        for (bdf_col* r : {csum, ccnt, cmin, cmax})
            if (r && e == cudaSuccess) {
                e = finish_single_group(c, r);
                if (r == cmin || r == cmax) r->null_counts[0] = -1;   // learnt on demand (ensure_null_counts)
            }
        if (e != cudaSuccess) { st = fail_cuda(e, "group aggregate"); break; }
        outs[j].sum = csum; outs[j].count = ccnt; outs[j].min = cmin; outs[j].max = cmax;
    }
    if (st != BDF_OK) {
        const std::string keep = g_err;
        cudaGetLastError();
        cleanup(true);
        for (int j = 0; j < n_values; j++) outs[j] = bdf_group_out{nullptr, nullptr, nullptr, nullptr};
        g_err = keep;
        return st;
    }
    cleanup(false);
    *out_keys = ukeys;
    if (n_groups_out) *n_groups_out = n_groups;
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// C ABI
//
// Every entry has one shape: the checks that need no device (context, pointers, counts, dtype codes, host views, the owner of
// every column), then the dispatch of a multi-GPU context to fleet.cu, then ENTER and the one-GPU implementation.

// sum/min/max/count: a known op, and min/max only where T::Native: Ord.
static int check_agg_op(int op, int dtype) {
    if (op < 0 || op >= BDF_NAGG) return fail(BDF_INVALID, "invalid aggregate op %d", op);
    if ((op == BDF_MIN || op == BDF_MAX) && dtype_is_float(dtype)) return fail(BDF_UNSUPPORTED, "min/max need T::Native: Ord (integers only)");
    return BDF_OK;
}

// Host in / host out on one GPU: upload the inputs, run fn on the device columns (a result column fn leaves in *o is downloaded
// into out), release everything.
static int host_call(bdf_ctx* c, const std::vector<UploadSpec>& specs, bdf_out* out, const std::function<int(bdf_col* const*, bdf_col**)>& fn) {
    std::vector<bdf_col*> cols;
    TRY(upload_many(c, specs, true, cols));
    bdf_col* o = nullptr;
    int st = fn(cols.data(), &o);
    if (st == BDF_OK && o) st = download(c, o, out);
    cudaStreamSynchronize(c->s_h2d);  // host inputs must not be touched after return
    col_release(c, o);
    for (bdf_col* col : cols) col_release(c, col);
    return st;
}

namespace bdf { int ctx_attach_comm(bdf_ctx* c, Comm* cm) { c->comm = cm; c->collective = true; c->collectives = 0; return BDF_OK; } }

#define ENTER(ctx)                                                   \
    if (!(ctx)) return fail(BDF_INVALID, "null context");           \
    std::lock_guard<std::mutex> _lock((ctx)->mu);                    \
    CK(cudaSetDevice((ctx)->device));

extern "C" {

int bdf_abi_version(void) { return BDF_ABI_VERSION; }

const char* bdf_last_error(void) { return g_err.c_str(); }

void bdf_destroy(bdf_ctx* c) {
    if (!c) return;
    if (c->fleet) { fleet_destroy(c); return; }
    cudaSetDevice(c->device);
    if (c->s_compute) cudaStreamSynchronize(c->s_compute);
    if (c->s_h2d) cudaStreamSynchronize(c->s_h2d);
    if (c->s_d2h) cudaStreamSynchronize(c->s_d2h);
    if (c->s_desc) cudaStreamSynchronize(c->s_desc);
    if (c->s_fin) cudaStreamSynchronize(c->s_fin);
    for (auto& p : c->prof) { cudaEventDestroy(p.e0); cudaEventDestroy(p.e1); }
    for (auto ev : c->prof_pool) cudaEventDestroy(ev);
    for (auto ev : c->ev_pool) cudaEventDestroy(ev);
    c->pool.reset();
    for (auto& sl : c->stage) { if (sl.p) cudaFreeHost(sl.p); if (sl.ev) cudaEventDestroy(sl.ev); }
    for (auto& b : c->part) { if (b.p) cudaFree(b.p); if (b.done) cudaEventDestroy(b.done); }
    if (c->ring) cudaFreeHost(c->ring);
    if (c->dring) cudaFree(c->dring);
    if (c->d_stage) cudaFree(c->d_stage);
    if (c->h_agg) cudaFreeHost(c->h_agg);
    if (c->h_flag) cudaFreeHost(c->h_flag);
    if (c->h_sort_agree) cudaFreeHost(c->h_sort_agree);
    if (c->d_partials) cudaFree(c->d_partials);
    if (c->d_stage2) cudaFree(c->d_stage2);
    if (c->d_stage_many) cudaFree(c->d_stage_many);
    if (c->d_tickets_many) cudaFree(c->d_tickets_many);
    if (c->d_ticket) cudaFree(c->d_ticket);
    if (c->d_flag) cudaFree(c->d_flag);
    if (c->flush_buf) cudaFree(c->flush_buf);
    if (c->comm) { comm_destroy(c->comm); c->comm = nullptr; }
    if (c->d_local) cudaFree(c->d_local);
    if (c->ev_tmp) cudaEventDestroy(c->ev_tmp);
    if (c->ev_t0) cudaEventDestroy(c->ev_t0);
    if (c->ev_t1) cudaEventDestroy(c->ev_t1);
    if (c->s_compute) cudaStreamDestroy(c->s_compute);
    if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
    if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
    if (c->s_desc) cudaStreamDestroy(c->s_desc);
    if (c->s_fin) cudaStreamDestroy(c->s_fin);
    delete c;
}

static int init_impl(bdf_ctx* c, int device) {
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(BDF_CUDA, "no usable CUDA device (%s); this library has no CPU fallback", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n_dev) return fail(BDF_INVALID, "device %d out of range (0..%d)", device, n_dev - 1);
    c->device = device;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount; c->cc_major = prop.major; c->cc_minor = prop.minor; c->hbm_bytes = prop.totalGlobalMem;
    if (prop.major != 10) return fail(BDF_CUDA, "device %d is sm_%d%d; libb200df is built for sm_100a only", device, prop.major, prop.minor);
    CK(cudaStreamCreateWithFlags(&c->s_compute, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->s_desc, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->s_fin, cudaStreamNonBlocking));
    cudaMemPool_t pool;
    CK(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = ~0ull;  // keep freed arenas cached: operators allocate their outputs per call
    CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    c->ring_cap = (size_t)32 << 20;  // ~400k chunk descriptors per operator call
    CK(cudaHostAlloc((void**)&c->ring, c->ring_cap, cudaHostAllocDefault));
    CK(cudaMalloc((void**)&c->dring, c->ring_cap));
    CK(cudaHostAlloc((void**)&c->h_agg, 2 * kAggSlots * sizeof(AggDev), cudaHostAllocMapped));
    CK(cudaHostGetDevicePointer((void**)&c->h_agg_dev, c->h_agg, 0));
    CK(cudaHostAlloc((void**)&c->h_flag, sizeof(int), cudaHostAllocDefault));
    CK(cudaMalloc((void**)&c->d_stage2, (size_t)c->sm_count * sizeof(AggDev)));
    CK(cudaMalloc((void**)&c->d_stage, (size_t)c->sm_count * sizeof(AggDev)));
    CK(cudaMalloc((void**)&c->d_ticket, 4 * sizeof(unsigned int)));
    CK(cudaMalloc((void**)&c->d_flag, sizeof(int)));
    CK(cudaMalloc((void**)&c->d_local, (size_t)kAggSlots * sizeof(AggDev)));
    CK(cudaMemset(c->d_ticket, 0, 4 * sizeof(unsigned int)));
    CK(cudaMemset(c->d_flag, 0, sizeof(int)));
    CK(cudaEventCreateWithFlags(&c->ev_tmp, cudaEventDisableTiming));
    CK(cudaEventCreate(&c->ev_t0));
    CK(cudaEventCreate(&c->ev_t1));
    // experiment knob: L2 fetch granularity hint (32 / 64 / 128 bytes) -- random gathers (take) fetch whole 128-byte lines by default
    if (const char* fg = getenv("BDF_L2_FETCH")) { if (atoi(fg) > 0) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(fg)); cudaGetLastError(); }
    const char* pb = getenv("BDF_PIPELINE_BYTES");
    if (pb && atoll(pb) > 0) c->pipeline_bytes = (size_t)atoll(pb);
    return BDF_OK;
}

int bdf_init(int device, bdf_ctx** out) {
    if (!out) return fail(BDF_INVALID, "null out pointer");
    *out = nullptr;
    bdf_ctx* c = new (std::nothrow) bdf_ctx();
    if (!c) return fail(BDF_OOM, "host allocation failed");
    int st = init_impl(c, device);
    if (st != BDF_OK) { std::string keep = g_err; bdf_destroy(c); g_err = keep; return st; }
    *out = c;
    return BDF_OK;
}

int bdf_synchronize(bdf_ctx* c) {
    if (c && c->fleet) return fleet_each_gpu(c, bdf_synchronize);
    ENTER(c);
    CK(cudaStreamSynchronize(c->s_h2d));
    CK(cudaStreamSynchronize(c->s_compute));
    CK(cudaStreamSynchronize(c->s_fin));
    CK(cudaStreamSynchronize(c->s_d2h));
    return BDF_OK;
}

int bdf_device_info(bdf_ctx* c, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* hbm_bytes) {
    if (c && c->fleet) return fleet_device_info(c, sm_count, cc_major, cc_minor, hbm_bytes);
    if (!c) return fail(BDF_INVALID, "null context");
    if (sm_count) *sm_count = c->sm_count;
    if (cc_major) *cc_major = c->cc_major;
    if (cc_minor) *cc_minor = c->cc_minor;
    if (hbm_bytes) *hbm_bytes = (int64_t)c->hbm_bytes;
    return BDF_OK;
}

int bdf_host_alloc(bdf_ctx* c, size_t bytes, void** out) {
    if (c && c->fleet) return bdf_host_alloc(fleet_first_gpu(c), bytes, out);   // pinned memory is usable from every GPU (unified addressing)
    ENTER(c);
    if (!out) return fail(BDF_INVALID, "null out pointer");
    CK(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return BDF_OK;
}
int bdf_host_free(bdf_ctx* c, void* p) {
    if (c && c->fleet) return bdf_host_free(fleet_first_gpu(c), p);
    ENTER(c);
    if (p) CK(cudaFreeHost(p));
    return BDF_OK;
}
int bdf_host_register(bdf_ctx* c, void* p, size_t bytes) {
    if (c && c->fleet) return bdf_host_register(fleet_first_gpu(c), p, bytes);
    ENTER(c);
    CK(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
    return BDF_OK;
}
int bdf_host_unregister(bdf_ctx* c, void* p) {
    if (c && c->fleet) return bdf_host_unregister(fleet_first_gpu(c), p);
    ENTER(c);
    CK(cudaHostUnregister(p));
    return BDF_OK;
}

// ---- multi-GPU: communicator -------------------------------------------------------------------------

int bdf_comm_unique_id(uint8_t* id) {
    if (!id) return fail(BDF_INVALID, "null id");
    std::string err;
    if (comm_unique_id(id, &err) != 0) return fail(BDF_NCCL, "%s", err.c_str());
    return BDF_OK;
}

int bdf_comm_attach(bdf_ctx* c, const uint8_t* id, int rank, int world) {
    if (c && c->fleet) return fail(BDF_INVALID, "a multi-GPU context already owns its communicator (ncclCommInitAll)");
    ENTER(c);
    if (!id || world < 1 || rank < 0 || rank >= world) return fail(BDF_INVALID, "bad communicator arguments (rank %d of %d)", rank, world);
    if (c->comm) return fail(BDF_INVALID, "the context already belongs to a communicator");
    CK(cudaStreamSynchronize(c->s_compute));
    std::string err;
    Comm* cm = comm_create(id, rank, world, &err);
    if (!cm) return fail(BDF_NCCL, "%s", err.c_str());
    c->comm = cm;
    c->collective = true;
    c->collectives = 0;
    // The combine itself can run over NVLink peer memory instead of NCCL (comm.cuh); every rank reads the same environment.
    const char* mode = getenv("BDF_COMBINE");
    if (world > 1 && !(mode && strcmp(mode, "nccl") == 0)) {
        std::string perr;
        // Default transport: the mailboxes up to 4 ranks, NCCL above unless asked for.  Measured on NVSwitch B200 boxes
        // (profiles/r2_*): a blocking combine costs 10 / 13 / 13 us over the mailboxes and 17 / 23 / 31 us over NCCL at
        // 2 / 4 / 8 GPUs and the strong series gains 10 % at 8, but the pipelined weak series at 8 GPUs ran 8 % slower with
        // the mailboxes in the one 8-GPU comparison this round could afford (0.400 vs 0.369-0.379 ms per step).
        if (comm_enable_p2p(cm, &perr) == 0) comm_set_p2p(cm, world <= 4 || (mode && strcmp(mode, "p2p") == 0));
        else if (mode && strcmp(mode, "p2p") == 0) { comm_destroy(cm); c->comm = nullptr; return fail(BDF_NCCL, "BDF_COMBINE=p2p: %s", perr.c_str()); }
    }
    return BDF_OK;
}

int bdf_comm_set_combine(bdf_ctx* c, int mode) {
    if (c && c->fleet) return fleet_each_gpu(c, [mode](bdf_ctx* k) { return bdf_comm_set_combine(k, mode); });
    ENTER(c);
    if (mode != 0 && mode != 1) return fail(BDF_INVALID, "combine mode is 0 (NCCL) or 1 (peer memory)");
    if (!c->comm) return mode == 0 ? BDF_OK : fail(BDF_UNSUPPORTED, "the context is not a rank of a communicator");
    CK(cudaStreamSynchronize(c->s_compute));
    CK(cudaStreamSynchronize(c->s_fin));
    if (comm_set_p2p(c->comm, mode == 1) != 0) return fail(BDF_UNSUPPORTED, "peer-memory mailboxes are not available on this communicator");
    return BDF_OK;
}

int bdf_comm_get_combine(bdf_ctx* c) {
    if (c && c->fleet) return bdf_comm_get_combine(fleet_first_gpu(c));
    return c && c->comm && comm_uses_p2p(c->comm) ? 1 : 0;
}

int bdf_comm_detach(bdf_ctx* c) {
    if (c && c->fleet) return fail(BDF_INVALID, "the communicator of a multi-GPU context lives as long as the context");
    ENTER(c);
    if (!c->comm) return BDF_OK;
    CK(cudaStreamSynchronize(c->s_compute));
    CK(cudaStreamSynchronize(c->s_fin));
    comm_destroy(c->comm);
    c->comm = nullptr;
    return BDF_OK;
}

int bdf_comm_info(bdf_ctx* c, int32_t* rank, int32_t* world, int32_t* nccl_version, int64_t* collectives) {
    if (c && c->fleet) return fleet_comm_info(c, rank, world, nccl_version, collectives);
    if (!c) return fail(BDF_INVALID, "null context");
    if (rank) *rank = c->comm ? comm_rank(c->comm) : 0;
    if (world) *world = c->comm ? comm_world(c->comm) : 1;
    if (nccl_version) *nccl_version = c->comm ? comm_version() : 0;
    if (collectives) *collectives = c->collectives;
    return BDF_OK;
}

int bdf_comm_collective(bdf_ctx* c, int on) {
    if (c && c->fleet) return on ? BDF_OK : fail(BDF_UNSUPPORTED, "a multi-GPU context always returns the aggregates of the whole column");
    ENTER(c);
    c->collective = on != 0;
    return BDF_OK;
}

int bdf_comm_all_reduce_f64(bdf_ctx* c, int op, int64_t n, double* inout) {
    if (c && c->fleet) return BDF_OK;   // one process: the caller's value is already the job's value
    ENTER(c);
    if (n < 0 || (n && !inout) || (op != BDF_SUM && op != BDF_MIN && op != BDF_MAX)) return fail(BDF_INVALID, "bad arguments");
    if (!c->comm || n == 0) return BDF_OK;   // a lone GPU: the value is already the result
    std::string err;
    c->collectives++;
    cudaError_t e = comm_host_allreduce_f64(c->comm, op == BDF_SUM ? 0 : op == BDF_MIN ? 1 : 2, inout, (int)n, c->s_compute, &err);
    if (e != cudaSuccess) { g_nccl_err = err; return fail_cuda(e, "all-reduce"); }
    return BDF_OK;
}

int bdf_comm_barrier(bdf_ctx* c) {
    if (c && c->fleet) return bdf_synchronize(c);
    {
        ENTER(c);
        CK(cudaStreamSynchronize(c->s_h2d));
        CK(cudaStreamSynchronize(c->s_compute));
        CK(cudaStreamSynchronize(c->s_fin));
        CK(cudaStreamSynchronize(c->s_d2h));
    }
    double one = 1.0;
    return bdf_comm_all_reduce_f64(c, BDF_SUM, 1, &one);   // returns once every rank has arrived
}

int bdf_aggregate_all_many_dev_async(bdf_ctx* c, int32_t n_cols, const bdf_col* const* cols, bdf_future** fut) {
    if (!cols || !fut) return fail(BDF_INVALID, "null argument");
    if (n_cols < 1 || n_cols > kCommMaxCols) return fail(BDF_INVALID, "an aggregate call takes 1..%d columns", kCommMaxCols);
    TRY(check_cols(c, n_cols, cols));
    if (c->fleet) return fleet_aggregate_many(c, n_cols, cols, fut);
    ENTER(c);
    return aggregate_many_dev_async(c, n_cols, const_cast<bdf_col* const*>(cols), false, fut);
}

int bdf_aggregate_all_many_dev(bdf_ctx* c, int32_t n_cols, const bdf_col* const* cols, bdf_agg4* out) {
    if (!cols || !out) return fail(BDF_INVALID, "null argument");
    if (n_cols < 1 || n_cols > kCommMaxCols) return fail(BDF_INVALID, "an aggregate call takes 1..%d columns", kCommMaxCols);
    TRY(check_cols(c, n_cols, cols));
    if (c->fleet) return fleet_aggregate_all_blocking(c, n_cols, cols, out);
    ENTER(c);
    bdf_future* f = nullptr;
    TRY(aggregate_many_dev_async(c, n_cols, const_cast<bdf_col* const*>(cols), true, &f));
    return future_wait(c, f, out);
}

int bdf_future_count(const bdf_future* fut) { return fut ? fut->n : 0; }

// ---- device-resident API -----------------------------------------------------------------------

int bdf_upload(bdf_ctx* c, int dtype, int64_t n_chunks, const bdf_view* in, int flags, bdf_col** out) {
    const int32_t dt = dtype;
    return bdf_upload_many(c, 1, &dt, &n_chunks, &in, flags, out);
}

int bdf_upload_many(bdf_ctx* c, int64_t n_cols, const int32_t* dtypes, const int64_t* n_chunks, const bdf_view* const* in,
                    int flags, bdf_col** out) {
    if (n_cols < 0 || (n_cols && (!dtypes || !n_chunks || !in || !out))) return fail(BDF_INVALID, "bad arguments");
    for (int64_t k = 0; k < n_cols; k++) {
        if (dtypes[k] != kBool) TRY(check_dtype(dtypes[k]));
        TRY(check_views(n_chunks[k], in[k]));
    }
    if (c && c->fleet) return fleet_upload_many(c, n_cols, dtypes, n_chunks, in, flags, out);
    ENTER(c);
    std::vector<UploadSpec> specs;
    for (int64_t k = 0; k < n_cols; k++) specs.push_back(UploadSpec{dtypes[k], n_chunks[k], in[k]});
    std::vector<bdf_col*> cols;
    TRY(upload_many(c, specs, (flags & BDF_ASYNC) != 0, cols));
    for (int64_t k = 0; k < n_cols; k++) out[k] = cols[k];
    return BDF_OK;
}

int bdf_col_wait(bdf_ctx* c, const bdf_col* col) {
    TRY(check_cols(c, {col}));
    if (c->fleet) return fleet_col_wait(c, col);
    ENTER(c);
    for (auto& g : col->groups) CK(cudaEventSynchronize(g.ev));
    return BDF_OK;
}

int bdf_col_describe(const bdf_col* col, int32_t* dtype, int64_t* n_chunks, int64_t* total_len) {
    if (!col) return fail(BDF_INVALID, "null column");
    if (dtype) *dtype = col->dtype;
    if (n_chunks) *n_chunks = col_chunk_count(col);
    if (total_len) *total_len = col->total_len;
    return BDF_OK;
}

int bdf_col_chunk_info(bdf_ctx* c, const bdf_col* col, int64_t chunk, int64_t* len, int64_t* null_count, int32_t* has_validity) {
    TRY(check_cols(c, {col}));
    if (chunk < 0 || chunk >= col_chunk_count(col)) return fail(BDF_INVALID, "bad chunk index");
    if (c->fleet) return fleet_chunk_info(c, col, chunk, len, null_count, has_validity);
    ENTER(c);
    if (len) *len = col->chunks[chunk].len;
    if (has_validity) *has_validity = col->chunks[chunk].validity != nullptr;
    if (null_count) {
        TRY(ensure_null_counts(c, const_cast<bdf_col*>(col)));
        *null_count = col->null_counts[chunk];
    }
    return BDF_OK;
}

int bdf_binary_dev(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {l, r}));
    if (c->fleet) return fleet_binary_dev(c, op, l, r, out, nullptr);
    ENTER(c);
    return binary_dev(c, op, l, r, out);
}

int bdf_unary_dev(bdf_ctx* c, int op, const bdf_col* in, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {in}));
    if (c->fleet) return fleet_map_dev(c, false, op, in, out);
    ENTER(c);
    return map_dev(c, false, op, in, out);
}

int bdf_cast_dev(bdf_ctx* c, int to, const bdf_col* in, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {in}));
    TRY(check_dtype(to));
    if (c->fleet) return fleet_map_dev(c, true, to, in, out);
    ENTER(c);
    return map_dev(c, true, to, in, out);
}

int bdf_aggregate_dev(bdf_ctx* c, int op, const bdf_col* in, void* out_scalar, int32_t* is_some) {
    if (!out_scalar || !is_some) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {in}));
    TRY(check_agg_op(op, in->dtype));
    if (c->fleet) return fleet_aggregate_dev(c, op, in, out_scalar, is_some);
    ENTER(c);
    return aggregate_dev(c, op, const_cast<bdf_col*>(in), out_scalar, is_some);
}

int bdf_aggregate_all_dev(bdf_ctx* c, const bdf_col* in, bdf_agg4* out) { return bdf_aggregate_all_many_dev(c, 1, &in, out); }

int bdf_avg_dev(bdf_ctx* c, const bdf_col* in, double* out, int32_t* is_some) {
    if (!out || !is_some) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {in}));
    if (c->fleet) return fleet_avg_dev(c, in, out, is_some);
    ENTER(c);
    return avg_dev(c, const_cast<bdf_col*>(in), out, is_some);
}

int bdf_binary_agg_dev_async(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, bdf_col** out, bdf_future** fut) {
    if (!out || !fut) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {l, r}));
    if (c->fleet) return fleet_binary_dev(c, op, l, r, out, fut);
    ENTER(c);
    return binary_dev(c, op, l, r, out, fut);
}

int bdf_binary_agg_dev(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, bdf_col** out, bdf_agg4* agg) {
    if (!agg) return fail(BDF_INVALID, "null argument");
    bdf_future* f = nullptr;
    TRY(bdf_binary_agg_dev_async(c, op, l, r, out, &f));
    return bdf_future_wait(c, f, agg);
}

// The two expression entries (fut == nullptr: bdf_eval_expr_dev).
static int expr_entry(bdf_ctx* c, int n_inputs, const bdf_col* const* inputs, int n_nodes, const bdf_expr_node* nodes, bdf_col** out,
                      bdf_future** fut) {
    if (!inputs || !nodes) return fail(BDF_INVALID, "null argument");
    int in_dtypes[8] = {0};
    const int n = std::max(0, std::min(n_inputs, 8));   // expr_prepare rejects any other count
    TRY(check_cols(c, n, inputs));
    for (int i = 0; i < n; i++) in_dtypes[i] = inputs[i]->dtype;
    alignas(8) unsigned char prog[256];
    bool has_div = false;
    TRY(expr_prepare(n_inputs, in_dtypes, n_nodes, nodes, prog, &has_div));
    if (c->fleet) return fleet_eval_expr(c, n_inputs, inputs, n_nodes, nodes, out, fut);
    ENTER(c);
    return expr_dev(c, n_inputs, inputs, prog, has_div, out, fut);
}

int bdf_eval_expr_agg_dev_async(bdf_ctx* c, int32_t n_inputs, const bdf_col* const* inputs, int32_t n_nodes, const bdf_expr_node* nodes,
                                bdf_col** out, bdf_future** fut) {
    if (!fut) return fail(BDF_INVALID, "null argument");
    return expr_entry(c, n_inputs, inputs, n_nodes, nodes, out, fut);
}

int bdf_eval_expr_agg_dev(bdf_ctx* c, int32_t n_inputs, const bdf_col* const* inputs, int32_t n_nodes, const bdf_expr_node* nodes, bdf_col** out,
                          bdf_agg4* agg) {
    if (!agg) return fail(BDF_INVALID, "null argument");
    bdf_future* f = nullptr;
    TRY(bdf_eval_expr_agg_dev_async(c, n_inputs, inputs, n_nodes, nodes, out, &f));
    return bdf_future_wait(c, f, agg);
}

int bdf_aggregate_all_dev_async(bdf_ctx* c, const bdf_col* in, bdf_future** fut) { return bdf_aggregate_all_many_dev_async(c, 1, &in, fut); }

int bdf_future_wait(bdf_ctx* c, bdf_future* fut, bdf_agg4* out) {
    if (!fut) return fail(BDF_INVALID, "null future");
    if (c && c->fleet) return fleet_future_wait(c, fut, out);
    ENTER(c);
    return future_wait(c, fut, out);
}

int bdf_expr_check(int32_t n_inputs, const int32_t* input_dtypes, int32_t n_nodes, const bdf_expr_node* nodes, int32_t* n_instructions,
                   int32_t* n_temporaries) {
    if (!nodes) return fail(BDF_INVALID, "null argument");
    int dt[8];
    for (int i = 0; i < 8; i++) dt[i] = (input_dtypes && i < n_inputs) ? input_dtypes[i] : BDF_F64;
    alignas(8) unsigned char prog[256];
    bool has_div = false;
    TRY(expr_prepare(n_inputs, dt, n_nodes, nodes, prog, &has_div));
    int ni = 0, nt = 0;
    expr_prog_stats(prog, &ni, &nt);
    if (n_instructions) *n_instructions = ni;
    if (n_temporaries) *n_temporaries = nt;
    return BDF_OK;
}

int bdf_eval_expr_dev(bdf_ctx* c, int32_t n_inputs, const bdf_col* const* inputs, int32_t n_nodes, const bdf_expr_node* nodes, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    return expr_entry(c, n_inputs, inputs, n_nodes, nodes, out, nullptr);
}

int bdf_sort_indices_dev(bdf_ctx* c, int32_t n_keys, const bdf_sort_key* keys, bdf_col** indices) {
    if (!keys || !indices) return fail(BDF_INVALID, "null argument");
    for (int32_t k = 0; k < n_keys; k++) TRY(check_cols(c, {keys[k].column}));
    if (c && c->fleet) return fail(BDF_UNSUPPORTED, "sort / take / filter move rows between chunks: use a one-GPU context (bdf_init) for them");
    ENTER(c);
    return sort_indices_dev(c, n_keys, keys, indices);
}

int bdf_group_aggregate_dev(bdf_ctx* c, const bdf_col* key, int32_t n_values, const bdf_col* const* values, bdf_col** out_keys, bdf_group_out* out,
                            int64_t* n_groups) {
    if (!out_keys || (n_values && (!values || !out))) return fail(BDF_INVALID, "null argument");
    if (n_values < 0 || n_values > 64) return fail(BDF_INVALID, "0..64 value columns");
    TRY(check_cols(c, {key}));
    TRY(check_cols(c, n_values, values));
    if (c->fleet) return fail(BDF_UNSUPPORTED, "group-by moves rows between chunks: use a one-GPU context (bdf_init) for it");
    ENTER(c);
    return group_aggregate_dev(c, key, n_values, values, out_keys, out, n_groups);
}

int bdf_take_dev(bdf_ctx* c, const bdf_col* values, const bdf_col* indices, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {values, indices}));
    if (c->fleet) return fail(BDF_UNSUPPORTED, "sort / take / filter move rows between chunks: use a one-GPU context (bdf_init) for them");
    ENTER(c);
    return take_dev(c, values, indices, out);
}

int bdf_compare_dev(bdf_ctx* c, int op, const bdf_col* left, const bdf_col* right, double scalar, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {left}));
    if (right) TRY(check_cols(c, {right}));
    if (c->fleet) return fleet_compare_dev(c, op, left, right, scalar, out);
    ENTER(c);
    return compare_dev(c, op, left, right, scalar, out);
}

int bdf_boolean_dev(bdf_ctx* c, int op, const bdf_col* a, const bdf_col* b, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {a}));
    if (b) TRY(check_cols(c, {b}));
    if (c->fleet) return fleet_boolean_dev(c, op, a, b, out);
    ENTER(c);
    return boolean_dev(c, op, a, b, out);
}

int bdf_filter_dev(bdf_ctx* c, const bdf_col* values, const bdf_col* mask, bdf_col** out) {
    if (!out) return fail(BDF_INVALID, "null argument");
    TRY(check_cols(c, {values, mask}));
    if (c->fleet) return fail(BDF_UNSUPPORTED, "sort / take / filter move rows between chunks: use a one-GPU context (bdf_init) for them");
    ENTER(c);
    return filter_dev(c, values, mask, out);
}

// The three download entries (phase 0 both halves, 1 begin, 2 end).
static int download_entry(bdf_ctx* c, const bdf_col* col, bdf_out* out, int phase) {
    TRY(check_cols(c, {col}));
    if (!out && col_chunk_count(col)) return fail(BDF_INVALID, "null argument");
    if (c->fleet) return fleet_download(c, col, out, phase);
    ENTER(c);
    bdf_col* m = const_cast<bdf_col*>(col);
    return phase == 1 ? download_enqueue(c, m, out) : phase == 2 ? download_finish(c, m, out) : download(c, m, out);
}

int bdf_download_begin(bdf_ctx* c, const bdf_col* col, bdf_out* out) { return download_entry(c, col, out, 1); }
int bdf_download_end(bdf_ctx* c, const bdf_col* col, bdf_out* out) { return download_entry(c, col, out, 2); }
int bdf_download(bdf_ctx* c, const bdf_col* col, bdf_out* out) { return download_entry(c, col, out, 0); }

void bdf_col_free(bdf_ctx* c, bdf_col* col) {
    if (!c || !col) return;
    if (c->fleet) { fleet_col_free(c, col); return; }
    std::lock_guard<std::mutex> lock(c->mu);
    cudaSetDevice(c->device);
    col_release(c, col);
}

// ---- host in / host out ------------------------------------------------------------------------

int bdf_binary(bdf_ctx* c, int op, int dtype, int64_t n_left, const bdf_view* left, int64_t n_right, const bdf_view* right, bdf_out* out) {
    TRY(check_dtype(dtype));
    if (n_left < 0 || n_right < 0 || (n_left && !left) || (n_right && !right)) return fail(BDF_INVALID, "bad arguments");
    const int64_t n = std::min(n_left, n_right);   // zip()
    if (n && !out) return fail(BDF_INVALID, "bad arguments");
    TRY(check_views(n, left));
    TRY(check_views(n, right));
    for (int64_t i = 0; i < n; i++)  // reject before moving a byte
        if (left[i].len != right[i].len) return fail(BDF_LENGTH_MISMATCH, "Cannot perform math operation on arrays of different length");
    if (c && c->fleet) return fleet_binary_host(c, op, dtype, n, left, right, out);
    ENTER(c);
    return host_call(c, {UploadSpec{dtype, n, left}, UploadSpec{dtype, n, right}}, out,
                     [&](bdf_col* const* in, bdf_col** o) { return binary_dev(c, op, in[0], in[1], o); });
}

int bdf_unary(bdf_ctx* c, int op, int dtype, int64_t n, const bdf_view* in, bdf_out* out) {
    TRY(check_dtype(dtype));
    TRY(check_views(n, in));
    if (c && c->fleet) return fleet_map_host(c, false, op, dtype, n, in, out);
    ENTER(c);
    return host_call(c, {UploadSpec{dtype, n, in}}, out, [&](bdf_col* const* cols, bdf_col** o) { return map_dev(c, false, op, cols[0], o); });
}

int bdf_cast(bdf_ctx* c, int from, int to, int64_t n, const bdf_view* in, bdf_out* out) {
    TRY(check_dtype(from));
    TRY(check_dtype(to));
    TRY(check_views(n, in));
    if (c && c->fleet) return fleet_map_host(c, true, to, from, n, in, out);
    ENTER(c);
    return host_call(c, {UploadSpec{from, n, in}}, out, [&](bdf_col* const* cols, bdf_col** o) { return map_dev(c, true, to, cols[0], o); });
}

int bdf_aggregate(bdf_ctx* c, int op, int dtype, int64_t n, const bdf_view* in, void* out_scalar, int32_t* is_some) {
    TRY(check_dtype(dtype));
    TRY(check_views(n, in));
    if (!out_scalar || !is_some) return fail(BDF_INVALID, "bad arguments");
    TRY(check_agg_op(op, dtype));
    if (c && c->fleet) return fleet_aggregate_host(c, dtype, n, in, [&](const bdf_col* col) { return bdf_aggregate_dev(c, op, col, out_scalar, is_some); });
    ENTER(c);
    if (op == BDF_COUNT) {  // metadata only when every null_count is known: no bytes move
        bool known = true;
        int64_t total = 0;
        for (int64_t i = 0; i < n; i++) {
            if (in[i].validity && in[i].null_count < 0) known = false;
            total += in[i].len - (in[i].validity ? in[i].null_count : 0);
        }
        if (known) { TRY(count_global(c, &total)); *(int64_t*)out_scalar = total; *is_some = 1; return BDF_OK; }
    }
    return host_call(c, {UploadSpec{dtype, n, in}}, nullptr,
                     [&](bdf_col* const* cols, bdf_col**) { return aggregate_dev(c, op, cols[0], out_scalar, is_some); });
}

int bdf_aggregate_all(bdf_ctx* c, int dtype, int64_t n, const bdf_view* in, bdf_agg4* out) {
    TRY(check_dtype(dtype));
    TRY(check_views(n, in));
    if (!out) return fail(BDF_INVALID, "bad arguments");
    if (c && c->fleet) return fleet_aggregate_host(c, dtype, n, in, [&](const bdf_col* col) { return bdf_aggregate_all_dev(c, col, out); });
    ENTER(c);
    return host_call(c, {UploadSpec{dtype, n, in}}, nullptr, [&](bdf_col* const* cols, bdf_col**) { return aggregate_all_dev(c, cols[0], true, out); });
}

int bdf_avg(bdf_ctx* c, int dtype, int64_t n, const bdf_view* in, double* out, int32_t* is_some) {
    TRY(check_dtype(dtype));
    TRY(check_views(n, in));
    if (!out || !is_some) return fail(BDF_INVALID, "bad arguments");
    if (c && c->fleet) return fleet_aggregate_host(c, dtype, n, in, [&](const bdf_col* col) { return bdf_avg_dev(c, col, out, is_some); });
    ENTER(c);
    return host_call(c, {UploadSpec{dtype, n, in}}, nullptr, [&](bdf_col* const* cols, bdf_col**) { return avg_dev(c, cols[0], out, is_some); });
}

// ---- measurement support -------------------------------------------------------------------------

int bdf_profile_enable(bdf_ctx* c, int on) {
    if (c && c->fleet) return fleet_each_gpu(c, [on](bdf_ctx* k) { return bdf_profile_enable(k, on); });
    ENTER(c);
    c->profiling = on != 0;
    return BDF_OK;
}

int bdf_profile_read(bdf_ctx* c, bdf_launch_record* buf, int64_t cap, int64_t* n) {
    if (c && c->fleet) return fleet_profile_read(c, buf, cap, n);
    ENTER(c);
    CK(cudaStreamSynchronize(c->s_compute));
    int64_t k = 0;
    for (auto& p : c->prof) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, p.e0, p.e1);
        p.rec.ms = ms;
        if (buf && k < cap) buf[k++] = p.rec;
        c->prof_pool.push_back(p.e0); c->prof_pool.push_back(p.e1);
    }
    c->prof.clear();
    if (n) *n = k;
    return BDF_OK;
}

int64_t bdf_launch_count(bdf_ctx* c) {
    if (c && c->fleet) return fleet_launch_count(c);
    return c ? c->launches : 0;
}

int bdf_timer_start(bdf_ctx* c) {
    if (c && c->fleet) return fleet_each_gpu(c, bdf_timer_start);
    ENTER(c);
    CK(cudaEventRecord(c->ev_t0, c->s_compute));
    return BDF_OK;
}

int bdf_timer_stop(bdf_ctx* c, float* ms) {
    if (c && c->fleet) return fleet_timer_stop(c, ms);
    ENTER(c);
    CK(cudaEventRecord(c->ev_t1, c->s_compute));
    CK(cudaEventSynchronize(c->ev_t1));
    if (ms) CK(cudaEventElapsedTime(ms, c->ev_t0, c->ev_t1));
    return BDF_OK;
}

int bdf_flush_l2(bdf_ctx* c, size_t bytes) {
    if (c && c->fleet) return fleet_each_gpu(c, [bytes](bdf_ctx* k) { return bdf_flush_l2(k, bytes); });
    ENTER(c);
    if (bytes > c->flush_bytes) {
        if (c->flush_buf) CK(cudaFree(c->flush_buf));
        c->flush_buf = nullptr; c->flush_bytes = 0;
        CK(cudaMalloc(&c->flush_buf, bytes));
        c->flush_bytes = bytes;
    }
    CK(launch_fill(c->flush_buf, bytes, c->s_compute));
    return BDF_OK;
}

int bdf_generate(bdf_ctx* c, int dtype, int kind, double lo, double hi, uint64_t seed, uint64_t col_id, int64_t n_chunks,
                 const int64_t* chunk_lens, int64_t row0, uint32_t null_mod, bdf_col** out) {
    TRY(check_dtype(dtype));
    if (!out || n_chunks < 0 || (n_chunks && !chunk_lens) || kind < 0 || kind > 3) return fail(BDF_INVALID, "bad arguments");
    for (int64_t i = 0; i < n_chunks; i++)
        if (chunk_lens[i] < 0) return fail(BDF_INVALID, "negative chunk length");
    if (c && c->fleet) return fleet_generate(c, dtype, kind, lo, hi, seed, col_id, n_chunks, chunk_lens, row0, null_mod, out);
    ENTER(c);
    std::vector<ChunkPlan> plan((size_t)n_chunks);
    for (int64_t i = 0; i < n_chunks; i++) plan[i] = {chunk_lens[i], null_mod != 0};
    bdf_col* o = nullptr;
    const int tile = elems_per_tile(dtype);
    TRY(col_alloc(c, dtype, plan, nullptr, tile, &o));
    o->counts_on_device = o->d_warp_counts != nullptr;
    void *hp = nullptr, *dp = nullptr;
    int st = ring_alloc(c, (size_t)n_chunks * sizeof(GenDesc), &hp, &dp);
    cudaError_t e = cudaSuccess;
    GenDesc* dd = (GenDesc*)dp;
    if (st == BDF_OK) {
        GenDesc* hd = (GenDesc*)hp;
        int64_t tiles = 0, rows = 0;
        for (int64_t i = 0; i < n_chunks; i++) {
            hd[i] = GenDesc{o->chunks[i].values, o->chunks[i].validity, chunk_lens[i], tiles, row0 + rows};
            tiles += (chunk_lens[i] + tile - 1) / tile;
            rows += chunk_lens[i];
        }
        e = desc_upload(c, dd, hd, (size_t)n_chunks * sizeof(GenDesc));
        if (e == cudaSuccess) {
            LaunchTimer t(c, BDF_K_GENERATE, dtype, rows, rows * dtype_width(dtype));
            e = launch_generate(dtype, kind, lo, hi, seed, col_id, null_mod, dd, (int)n_chunks, tiles, o->d_warp_counts, c->s_compute);
        }
        if (e == cudaSuccess) {
            Group g{0, n_chunks, nullptr};
            e = ev_get(c, &g.ev);
            if (e == cudaSuccess) e = cudaEventRecord(g.ev, c->s_compute);
            o->groups.push_back(g);
        }
    }
    if (st != BDF_OK || e != cudaSuccess) {
        cudaGetLastError();
        col_release(c, o);
        return st != BDF_OK ? st : fail(cuda_status(e), "generate failed: %s", cudaGetErrorString(e));
    }
    *out = o;
    return BDF_OK;
}

}  // extern "C"
