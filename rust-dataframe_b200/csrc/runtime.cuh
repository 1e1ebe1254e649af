// runtime.cuh -- the objects behind the C ABI's handles and the error plumbing, shared by runtime.cu (the one-GPU runtime and
// the C ABI) and fleet.cu (the multi-GPU context).  Private to the library: nothing here is exported.
#pragma once

#include <cstdint>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200df.h"
#include "common.cuh"
#include "comm.cuh"

using namespace bdf;

// ---------------------------------------------------------------------------------------------------
// errors

extern thread_local std::string g_err;   // the message bdf_last_error returns (defined in runtime.cu)

int fail(int status, const char* fmt, ...);

static inline int cuda_status(cudaError_t e) { return e == cudaErrorMemoryAllocation ? BDF_OOM : BDF_CUDA; }

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t _e = (call);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            return fail(cuda_status(_e), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

#define TRY(expr)                  \
    do {                           \
        int _st = (expr);          \
        if (_st != BDF_OK) return _st; \
    } while (0)

static constexpr int kBool = 10;  // BDF_BOOL: bit-packed boolean column (N2)

static inline int check_dtype(int t) {
    if (t < 0 || t >= BDF_NTYPES) return fail(BDF_INVALID, "invalid dtype %d", t);
    return BDF_OK;
}

// ---------------------------------------------------------------------------------------------------
// objects

struct Group {
    int64_t begin, end;  // chunks [begin, end)
    cudaEvent_t ev;      // chunks are complete in HBM once ev has fired
};

struct DevChunk {
    char* values;
    uint32_t* validity;  // nullptr = no bitmap
    int64_t len;
    int32_t bit_off;      // residual bit offset of the validity bitmap
    int32_t val_bit_off;  // boolean columns only: residual bit offset of the VALUES bitmap
};

struct bdf_col {
    const bdf_ctx* owner = nullptr;                // the context that made the column; no other context accepts it
    int dtype = 0;
    int64_t total_len = 0;
    std::vector<DevChunk> chunks;
    char* arena_values = nullptr;
    char* arena_validity = nullptr;
    uint32_t* d_warp_counts = nullptr;             // valid slots per warp per tile ([tile][8]), written by the producing kernel
    int64_t tile_elems = 0;                        // tile size (elements) the producing kernel used
    std::vector<int64_t> tile0;                    // column-global first tile of each chunk (n+1 entries)
    bool counts_on_device = false;                 // d_warp_counts not yet folded into null_counts
    std::vector<int64_t> null_counts;              // -1 = unknown
    std::vector<Group> groups;
    std::vector<uint32_t> dl_counts;               // staging of d_warp_counts during a split download
    bdf_col* dl_tmp = nullptr;                     // re-aligned copy used by a split download of a sliced column
    struct StagedCopy { void* dst; const void* src; size_t bytes; };
    std::vector<StagedCopy> dl_staged;             // device->pageable-host copies carried out in download_finish
    // A column of a multi-GPU context (bdf_init_multi): the logical chunks are cut into row ranges, each range lives as one
    // chunk of a per-GPU sub-column.  Empty for the columns of a one-GPU context.
    struct Piece { int kid; int64_t local; int64_t row0, rows; };   // rows [row0, row0 + rows) of a logical chunk = chunk `local` of fparts[kid]
    std::vector<bdf_col*> fparts;                  // one sub-column per GPU (possibly without chunks)
    std::vector<std::vector<Piece>> fmap;          // per logical chunk, in row order
    std::vector<int64_t> flens;                    // logical chunk lengths
};

// The number of chunks the caller sees (a column of a multi-GPU context keeps its logical chunks in flens).
static inline int64_t col_chunk_count(const bdf_col* col) {
    return col->fparts.empty() ? (int64_t)col->chunks.size() : (int64_t)col->flens.size();
}

// Result of an aggregate that is still in flight (or done): a pinned slot + the event that guards it.
struct bdf_future {
    int n = 1;                   // number of aggregates the future carries (one per column of a multi-column call)
    int fused = 1;               // which kernel produced the keys: 1 = k_binary AGG, 2 = k_reduce (see convert_agg)
    int slot = 0;                // first index into h_agg: n records, or 2n ({AggDev, {rows, panics, chunks}}) when global
    bool global = false;         // combined across the ranks of the communicator (comm.cuh)
    int lslot = 0;               // global only: first index into d_local (the per-rank records the collective reads)
    std::vector<int> dtypes;
    std::vector<int64_t> rows;   // local rows per aggregate
    std::vector<uint32_t> panics;  // local chunks that are empty or all-null (max/min .unwrap() would panic)
    std::vector<uint32_t> chunks;  // local chunk count
    cudaEvent_t ev = nullptr;
    std::vector<bdf_future*> fparts;   // multi-GPU context: the per-GPU futures (every one yields the same, global, records)
};

struct ProfEntry {
    bdf_launch_record rec;
    cudaEvent_t e0, e1;
};

class CopyPool;   // staging threads of a one-GPU context (runtime.cu)
struct Fleet;     // the GPUs of a multi-GPU context (fleet.cu)

struct bdf_ctx {
    // defined where CopyPool is complete (runtime.cu); hidden, as b200df.h declares the struct among the library's exports
    __attribute__((visibility("hidden"))) bdf_ctx();
    __attribute__((visibility("hidden"))) ~bdf_ctx();
    int device = 0;
    int sm_count = 0, cc_major = 0, cc_minor = 0;
    size_t hbm_bytes = 0;
    cudaStream_t s_compute = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaStream_t s_desc = nullptr;  // descriptor copies: run ahead of the compute stream, off its critical path
    cudaStream_t s_fin = nullptr;   // k_finish of fused aggregates: overlaps the next operator
    std::mutex mu;
    // pinned staging: descriptor ring + small result area
    char* ring = nullptr;           // pinned host side of the descriptor ring
    char* dring = nullptr;          // device side, same offsets
    size_t ring_cap = 0, ring_head = 0;
    std::vector<cudaEvent_t> ev_pool;  // recycled cudaEventDisableTiming events
    AggDev* h_agg = nullptr;        // pinned + device-mapped: kernels write results straight into it
    AggDev* h_agg_dev = nullptr;    // device-side address of h_agg
    int* h_flag = nullptr;          // pinned
    unsigned long long* h_sort_agree = nullptr;   // pinned: OR and AND of the sort keys of one criterion
    int64_t last_sort_passes = 0;
    // device scratch
    AggDev* d_partials = nullptr;       // per-CTA partials of k_reduce (compute stream only)
    size_t red_part_cap = 0;
    AggDev* d_stage2 = nullptr;         // k_finish staging for the k_reduce path
    AggDev* d_stage_many = nullptr;     // k_finish_many staging (kFinishMany x sm_count) and tickets, allocated on first use
    unsigned int* d_tickets_many = nullptr;
    unsigned int* d_ticket = nullptr;   // k_finish tickets: [0] reduce path (compute stream), [1] fused aggregates (finish stream)
    AggDev* d_stage = nullptr;          // k_finish per-CTA staging, sm_count entries
    int* d_flag = nullptr;
    int fut_next = 0;                   // ring cursor over the future half of h_agg
    struct PartBuf { AggDev* p = nullptr; size_t cap = 0; cudaEvent_t done = nullptr; bool used = false; } part[3];
    int part_next = 0;                  // per-tile partials of fused aggregates: 3 persistent buffers in rotation
    // staging for PAGEABLE host buffers: pinned slots filled/drained by a few host threads while the DMA of the
    // previous slot is in flight (cudaMemcpyAsync straight from pageable memory is a single-threaded driver copy)
    struct StageSlot { char* p = nullptr; cudaEvent_t ev = nullptr; bool busy = false; };
    std::vector<StageSlot> stage;
    int stage_next = 0;
    int copy_threads = 8;
    std::unique_ptr<CopyPool> pool;
    cudaEvent_t ev_tmp = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
    void* flush_buf = nullptr;
    size_t flush_bytes = 0;
    size_t pipeline_bytes = (size_t)32 << 20;
    bool profiling = false;
    std::vector<ProfEntry> prof;
    std::vector<cudaEvent_t> prof_pool;   // recycled timing events
    int64_t launches = 0;
    // multi-GPU: the communicator this context is a rank of (nullptr = a lone GPU) -- comm.cuh
    Comm* comm = nullptr;
    bool collective = true;             // aggregates are combined across the ranks (every rank makes the same calls)
    AggDev* d_local = nullptr;          // per-rank aggregate records awaiting their collective (ring of kAggSlots)
    int local_next = 0;
    int64_t collectives = 0;            // grouped NCCL calls enqueued since the communicator was attached
    Fleet* fleet = nullptr;             // non-null: this is a multi-GPU context (bdf_init_multi); it owns no device itself
};

namespace bdf { int ctx_attach_comm(bdf_ctx* c, Comm* cm); }

// ---------------------------------------------------------------------------------------------------
// The multi-GPU context (fleet.cu): what each C entry runs when c->fleet is set.  The entries have checked their arguments
// (columns included) before they dispatch here.

void fleet_destroy(bdf_ctx* c);
int fleet_device_info(bdf_ctx* c, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* hbm_bytes);
bdf_ctx* fleet_first_gpu(bdf_ctx* c);
int fleet_each_gpu(bdf_ctx* c, const std::function<int(bdf_ctx*)>& fn);   // the entry on one GPU after the other, up to the first failure
int fleet_comm_info(bdf_ctx* c, int32_t* rank, int32_t* world, int32_t* nccl_version, int64_t* collectives);
int fleet_upload_many(bdf_ctx* c, int64_t n_cols, const int32_t* dtypes, const int64_t* n_chunks, const bdf_view* const* in, int flags, bdf_col** out);
int fleet_col_wait(bdf_ctx* c, const bdf_col* col);
int fleet_chunk_info(bdf_ctx* c, const bdf_col* col, int64_t chunk, int64_t* len, int64_t* null_count, int32_t* has_validity);
void fleet_col_free(bdf_ctx* c, bdf_col* col);
int fleet_download(bdf_ctx* c, const bdf_col* col, bdf_out* out, int phase /* 0 both, 1 begin, 2 end */);
int fleet_binary_dev(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, bdf_col** out, bdf_future** fut);
int fleet_map_dev(bdf_ctx* c, bool is_cast, int op_or_to, const bdf_col* in, bdf_col** out);
int fleet_compare_dev(bdf_ctx* c, int op, const bdf_col* left, const bdf_col* right, double scalar, bdf_col** out);
int fleet_boolean_dev(bdf_ctx* c, int op, const bdf_col* a, const bdf_col* b, bdf_col** out);
int fleet_eval_expr(bdf_ctx* c, int n_inputs, const bdf_col* const* inputs, int n_nodes, const bdf_expr_node* nodes, bdf_col** out,
                    bdf_future** fut);
int fleet_aggregate_many(bdf_ctx* c, int32_t n_cols, const bdf_col* const* cols, bdf_future** fut);
int fleet_aggregate_all_blocking(bdf_ctx* c, int32_t n_cols, const bdf_col* const* cols, bdf_agg4* out);
int fleet_aggregate_dev(bdf_ctx* c, int op, const bdf_col* col, void* out_scalar, int32_t* is_some);
int fleet_avg_dev(bdf_ctx* c, const bdf_col* col, double* out, int32_t* is_some);
int fleet_future_wait(bdf_ctx* c, bdf_future* fu, bdf_agg4* out);
int fleet_binary_host(bdf_ctx* c, int op, int dtype, int64_t n, const bdf_view* left, const bdf_view* right, bdf_out* out);
int fleet_map_host(bdf_ctx* c, bool is_cast, int op_or_to, int dtype, int64_t n, const bdf_view* in, bdf_out* out);
int fleet_aggregate_host(bdf_ctx* c, int dtype, int64_t n, const bdf_view* in, const std::function<int(const bdf_col*)>& fn);
int fleet_generate(bdf_ctx* c, int dtype, int kind, double lo, double hi, uint64_t seed, uint64_t col_id, int64_t n_chunks,
                   const int64_t* chunk_lens, int64_t row0, uint32_t null_mod, bdf_col** out);
int fleet_profile_read(bdf_ctx* c, bdf_launch_record* buf, int64_t cap, int64_t* n);
int64_t fleet_launch_count(bdf_ctx* c);
int fleet_timer_stop(bdf_ctx* c, float* ms);
