// fleet.cu -- the multi-GPU context (bdf_init_multi): ONE process, every GPU of the box.  The library owns the sharding that the
// reference leaves to rayon (par_iter over chunks, src/functions/scalar.rs:28-31,99-102): the rows of a call are cut into
// one contiguous range per GPU (cuts on 64-row boundaries inside a chunk, so a piece is a zero-copy Arrow slice whose
// validity starts on a byte boundary), every GPU runs the ordinary one-GPU path on its pieces -- its own PCIe link, its
// own staging threads -- and aggregates are combined by the grouped ncclAllReduce of comm.cu (ncclCommInitAll).
// A fleet context owns no device; its "kids" are complete one-GPU contexts driven by one persistent host thread each
// (a blocking collective must be entered by all ranks at once, and uploads of different GPUs should overlap).  Like ipc.cu,
// this file reaches the kids only through the C ABI; the C entries of runtime.cu check their arguments and dispatch here.
#include <algorithm>
#include <cctype>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <sched.h>
#include <thread>

#include "runtime.cuh"

struct Fleet {
    std::vector<bdf_ctx*> kids;
    struct Worker {
        std::thread th;
        std::mutex m;
        std::condition_variable cv;
        std::function<int()> job;
        bool has_job = false, done = false, stop = false;
        int status = BDF_OK;
        std::string err;
    };
    std::vector<std::unique_ptr<Worker>> workers;
    std::mutex run_mu;   // one fan-out at a time: two caller threads must not interleave their jobs (or the order of the kids' collectives)
};

static void fleet_worker_main(Fleet::Worker* w, int device) {
    // run near the GPU: host<->device copies and the staging threads this thread creates stay on the GPU's NUMA node
    char bus[32];
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) == cudaSuccess) {
        for (char* p = bus; *p; p++) *p = (char)tolower(*p);
        const std::string base = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
        int node = -1;
        if (FILE* f = fopen(base.c_str(), "r")) { if (fscanf(f, "%d", &node) != 1) node = -1; fclose(f); }
        if (node >= 0) {
            const std::string cl = "/sys/devices/system/node/node" + std::to_string(node) + "/cpulist";
            if (FILE* f = fopen(cl.c_str(), "r")) {
                char buf[4096];
                if (fgets(buf, sizeof buf, f)) {
                    cpu_set_t set, cur; CPU_ZERO(&set);
                    int n = 0;
                    for (char* tok = strtok(buf, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
                        int lo, hi;
                        if (sscanf(tok, "%d-%d", &lo, &hi) == 2) { for (int cpu = lo; cpu <= hi && cpu < CPU_SETSIZE; cpu++) { CPU_SET(cpu, &set); n++; } }
                        else if (sscanf(tok, "%d", &lo) == 1 && lo < CPU_SETSIZE) { CPU_SET(lo, &set); n++; }
                    }
                    if (n && sched_getaffinity(0, sizeof cur, &cur) == 0) {
                        CPU_AND(&set, &set, &cur);
                        if (CPU_COUNT(&set) > 0) sched_setaffinity(0, sizeof set, &set);
                    }
                }
                fclose(f);
            }
        }
    }
    cudaGetLastError();
    std::unique_lock<std::mutex> lk(w->m);
    for (;;) {
        w->cv.wait(lk, [w] { return w->has_job || w->stop; });
        if (w->stop) return;
        std::function<int()> job = std::move(w->job);
        w->has_job = false;
        lk.unlock();
        g_err.clear();
        int st;
        try { st = job(); } catch (...) { st = fail(BDF_INVALID, "internal error in a fleet worker"); }
        lk.lock();
        w->status = st;
        w->err = g_err;
        w->done = true;
        w->cv.notify_all();
    }
}

// Run fn(k) for every kid, each on its own thread, and wait.  The first failing status (lowest kid) is returned with its message.
static int fleet_run(Fleet* f, const std::function<int(int)>& fn) {
    std::lock_guard<std::mutex> one_at_a_time(f->run_mu);   // the jobs run on the workers and never fan out themselves: no recursion
    const int n = (int)f->kids.size();
    for (int k = 0; k < n; k++) {
        Fleet::Worker* w = f->workers[k].get();
        std::lock_guard<std::mutex> g(w->m);
        w->job = [&fn, k] { return fn(k); };
        w->has_job = true; w->done = false;
        w->cv.notify_all();
    }
    int status = BDF_OK;
    std::string err;
    for (int k = 0; k < n; k++) {
        Fleet::Worker* w = f->workers[k].get();
        std::unique_lock<std::mutex> lk(w->m);
        w->cv.wait(lk, [w] { return w->done; });
        if (w->status != BDF_OK && status == BDF_OK) { status = w->status; err = w->err; }
    }
    if (status != BDF_OK) g_err = err;
    return status;
}

// Cut the rows of the logical chunks into one contiguous range per kid (balanced by rows; cuts inside a chunk are
// multiples of 64 rows).  Returns the pieces per logical chunk; `local` numbers a kid's pieces in order.
static std::vector<std::vector<bdf_col::Piece>> fleet_plan(const std::vector<int64_t>& lens, int n_kids) {
    const size_t n = lens.size();
    int64_t total = 0;
    std::vector<int64_t> start(n + 1, 0);
    for (size_t i = 0; i < n; i++) { start[i] = total; total += lens[i]; }
    start[n] = total;
    auto snap = [&](int64_t g) {   // a global cut -> an aligned row of the chunk it falls into
        if (g <= 0) return (int64_t)0;
        if (g >= total) return total;
        size_t i = (size_t)(std::upper_bound(start.begin(), start.begin() + (ptrdiff_t)n, g) - start.begin()) - 1;
        return start[i] + (g - start[i]) / 64 * 64;
    };
    std::vector<int64_t> cut((size_t)n_kids + 1);
    for (int k = 0; k <= n_kids; k++) cut[k] = snap((int64_t)((__int128)total * k / n_kids));
    cut[n_kids] = total;
    std::vector<std::vector<bdf_col::Piece>> map(n);
    std::vector<int64_t> next_local((size_t)n_kids, 0);
    for (size_t i = 0; i < n; i++)
        for (int k = 0; k < n_kids; k++) {
            const int64_t b = std::max(cut[k], start[i]), e = std::min(cut[k + 1], start[i] + lens[i]);
            if (e > b) map[i].push_back(bdf_col::Piece{k, next_local[k]++, b - start[i], e - b});
        }
    // an empty logical chunk still needs a home (it keeps the chunk structure and the reference's panic rule intact)
    for (size_t i = 0; i < n; i++)
        if (lens[i] == 0) map[i].push_back(bdf_col::Piece{(int)(i % (size_t)n_kids), next_local[i % (size_t)n_kids]++, 0, 0});
    return map;
}

// The host views of kid k under a plan (zero-copy slices of the caller's chunks), in the kid's local chunk order (a kid's
// pieces are numbered 0, 1, ... without gaps).
static std::vector<bdf_view> fleet_views(const std::vector<std::vector<bdf_col::Piece>>& map, int kid, const bdf_view* in) {
    std::vector<bdf_view> out;
    for (size_t i = 0; i < map.size(); i++)
        for (const auto& pc : map[i])
            if (pc.kid == kid) {
                bdf_view v = in[i];
                v.offset += pc.row0;
                v.len = pc.rows;
                if (!(pc.row0 == 0 && pc.rows == in[i].len)) v.null_count = v.validity ? -1 : 0;   // a proper slice: unknown
                if ((size_t)pc.local >= out.size()) out.resize((size_t)pc.local + 1);
                out[(size_t)pc.local] = v;
            }
    return out;
}

static std::vector<bdf_out> fleet_outs(const std::vector<std::vector<bdf_col::Piece>>& map, int kid, int out_dtype, const bdf_out* out) {
    std::vector<bdf_out> res;
    const int w = out_dtype == kBool ? 0 : dtype_width(out_dtype);
    for (size_t i = 0; i < map.size(); i++)
        for (const auto& pc : map[i])
            if (pc.kid == kid) {
                bdf_out o = out[i];
                if (o.values) o.values = (char*)o.values + (out_dtype == kBool ? pc.row0 / 8 : pc.row0 * w);
                if (o.validity) o.validity = o.validity + pc.row0 / 8;   // row0 is a multiple of 64
                o.len = pc.rows;
                if ((size_t)pc.local >= res.size()) res.resize((size_t)pc.local + 1);
                res[(size_t)pc.local] = o;
            }
    return res;
}

// Fold the kids' per-piece results back into the caller's per-chunk bdf_out entries.
static void fleet_merge_outs(const std::vector<std::vector<bdf_col::Piece>>& map, const std::vector<std::vector<bdf_out>>& kid_outs,
                             const std::vector<int64_t>& lens, bdf_out* out) {
    for (size_t i = 0; i < map.size(); i++) {
        int64_t nulls = 0;
        int32_t hv = 0;
        for (const auto& pc : map[i]) {
            const bdf_out& o = kid_outs[(size_t)pc.kid][(size_t)pc.local];
            nulls += o.null_count;
            hv |= o.has_validity;
        }
        out[i].len = lens[i];
        out[i].null_count = nulls;
        out[i].has_validity = hv;
    }
}

static bool fleet_same_map(const bdf_col* a, const bdf_col* b, int64_t n) {
    for (int64_t i = 0; i < n; i++) {
        if (a->fmap[i].size() != b->fmap[i].size()) return false;
        for (size_t j = 0; j < a->fmap[i].size(); j++) {
            const auto &x = a->fmap[i][j], &y = b->fmap[i][j];
            if (x.kid != y.kid || x.local != y.local || x.row0 != y.row0 || x.rows != y.rows) return false;
        }
    }
    return true;
}

// The inputs of one operator must line up piece by piece.  *n_chunks: the chunks the operator zips.
static int fleet_check_inputs(int n_in, const bdf_col* const* in, int64_t* n_chunks) {
    const bdf_col* first = in[0];
    int64_t n = (int64_t)first->fmap.size();
    for (int j = 1; j < n_in; j++) n = std::min<int64_t>(n, (int64_t)in[j]->fmap.size());   // zip()
    for (int j = 1; j < n_in; j++)
        for (int64_t i = 0; i < n; i++)
            if (in[j]->flens[i] != first->flens[i]) return fail(BDF_LENGTH_MISMATCH, "Cannot perform math operation on arrays of different length");
    for (int j = 1; j < n_in; j++)
        if (!fleet_same_map(first, in[j], n))
            return fail(BDF_INVALID, "the columns are sharded differently over the GPUs (upload them in one bdf_upload_many call)");
    for (int j = 1; j < n_in; j++)
        if (in[j]->fmap.size() != first->fmap.size()) return fail(BDF_UNSUPPORTED, "columns with different numbers of chunks on a multi-GPU context");
    *n_chunks = n;
    return BDF_OK;
}

static bdf_col* fleet_col_new(bdf_ctx* c, int dtype) {
    bdf_col* col = new (std::nothrow) bdf_col();
    if (!col) return nullptr;
    col->owner = c;
    col->dtype = dtype;
    col->fparts.assign(c->fleet->kids.size(), nullptr);
    return col;
}

void fleet_col_free(bdf_ctx* c, bdf_col* col) {
    if (!col) return;
    for (size_t k = 0; k < col->fparts.size(); k++)
        if (col->fparts[k]) bdf_col_free(c->fleet->kids[k], col->fparts[k]);
    delete col;
}

// A column whose logical chunks have the lengths `lens`, cut over the kids by fleet_plan; its parts are still to be made.
static bdf_col* fleet_col_planned(bdf_ctx* c, int dtype, const std::vector<int64_t>& lens) {
    bdf_col* col = fleet_col_new(c, dtype);
    if (!col) return nullptr;
    col->fmap = fleet_plan(lens, (int)c->fleet->kids.size());
    col->flens = lens;
    for (int64_t v : lens) col->total_len += v;
    return col;
}

// A result column with the logical structure of `like` (elementwise operators keep it), parts filled by the kids.
static bdf_col* fleet_col_like(bdf_ctx* c, const bdf_col* like, int dtype, int64_t n_chunks) {
    bdf_col* col = fleet_col_new(c, dtype);
    if (!col) return nullptr;
    col->fmap.assign(like->fmap.begin(), like->fmap.begin() + (ptrdiff_t)n_chunks);
    col->flens.assign(like->flens.begin(), like->flens.begin() + (ptrdiff_t)n_chunks);
    for (int64_t v : col->flens) col->total_len += v;
    return col;
}

int fleet_upload_many(bdf_ctx* c, int64_t n_cols, const int32_t* dtypes, const int64_t* n_chunks, const bdf_view* const* in, int flags, bdf_col** out) {
    Fleet* f = c->fleet;
    const int nk = (int)f->kids.size();
    // all columns of one call share ONE plan when their chunk lengths agree (a RecordBatch list), so that operators over them line up
    std::vector<bdf_col*> cols((size_t)n_cols, nullptr);
    std::vector<std::vector<std::vector<bdf_view>>> views((size_t)n_cols);
    for (int64_t j = 0; j < n_cols; j++) {
        std::vector<int64_t> lens((size_t)n_chunks[j]);
        for (int64_t i = 0; i < n_chunks[j]; i++) lens[i] = in[j][i].len;
        cols[j] = fleet_col_planned(c, dtypes[j], lens);
        if (!cols[j]) { for (auto* x : cols) fleet_col_free(c, x); return fail(BDF_OOM, "host allocation failed"); }
        views[j].resize((size_t)nk);
        for (int k = 0; k < nk; k++) views[j][k] = fleet_views(cols[j]->fmap, k, in[j]);
    }
    int st = fleet_run(f, [&](int k) {
        std::vector<int32_t> dt((size_t)n_cols);
        std::vector<int64_t> cnt((size_t)n_cols);
        std::vector<const bdf_view*> ptr((size_t)n_cols);
        std::vector<bdf_col*> res((size_t)n_cols, nullptr);
        for (int64_t j = 0; j < n_cols; j++) { dt[j] = dtypes[j]; cnt[j] = (int64_t)views[j][k].size(); ptr[j] = views[j][k].data(); }
        int s2 = bdf_upload_many(f->kids[k], n_cols, dt.data(), cnt.data(), ptr.data(), flags, res.data());
        for (int64_t j = 0; j < n_cols; j++) cols[j]->fparts[k] = res[j];
        return s2;
    });
    if (st != BDF_OK) { const std::string keep = g_err; for (auto* x : cols) fleet_col_free(c, x); g_err = keep; return st; }
    for (int64_t j = 0; j < n_cols; j++) out[j] = cols[j];
    return BDF_OK;
}

int fleet_download(bdf_ctx* c, const bdf_col* col, bdf_out* out, int phase) {
    Fleet* f = c->fleet;
    const int nk = (int)f->kids.size();
    const int64_t n = (int64_t)col->fmap.size();
    for (int64_t i = 0; i < n; i++)
        if (out[i].len != col->flens[i]) return fail(BDF_INVALID, "output chunk %lld has capacity %lld, result has %lld rows", (long long)i, (long long)out[i].len, (long long)col->flens[i]);
    std::vector<std::vector<bdf_out>> kouts((size_t)nk);
    for (int k = 0; k < nk; k++) kouts[k] = fleet_outs(col->fmap, k, col->dtype, out);
    int st = fleet_run(f, [&](int k) {
        bdf_out dummy{};
        bdf_out* o = kouts[k].empty() ? &dummy : kouts[k].data();
        if (phase == 1) return bdf_download_begin(f->kids[k], col->fparts[k], o);
        if (phase == 2) return bdf_download_end(f->kids[k], col->fparts[k], o);
        return bdf_download(f->kids[k], col->fparts[k], o);
    });
    if (st != BDF_OK) return st;
    if (phase != 1) fleet_merge_outs(col->fmap, kouts, col->flens, out);
    return BDF_OK;
}

int fleet_col_wait(bdf_ctx* c, const bdf_col* col) {
    Fleet* f = c->fleet;
    return fleet_run(f, [f, col](int k) { return bdf_col_wait(f->kids[k], col->fparts[k]); });
}

int fleet_chunk_info(bdf_ctx* c, const bdf_col* col, int64_t chunk, int64_t* len, int64_t* null_count, int32_t* has_validity) {
    if (len) *len = col->flens[chunk];
    if (!null_count && !has_validity) return BDF_OK;
    int64_t nulls = 0; int32_t hv = 0;
    for (const auto& pc : col->fmap[chunk]) {   // a handful of pieces: the calling thread asks the kids in turn
        int64_t l = 0, nc = 0; int32_t h = 0;
        TRY(bdf_col_chunk_info(c->fleet->kids[pc.kid], col->fparts[pc.kid], pc.local, &l, null_count ? &nc : nullptr, &h));
        nulls += nc; hv |= h;
    }
    if (null_count) *null_count = nulls;
    if (has_validity) *has_validity = hv;
    return BDF_OK;
}

static bdf_future* fleet_future_new(bdf_ctx* c) {
    bdf_future* fu = new (std::nothrow) bdf_future();
    if (fu) fu->fparts.assign(c->fleet->kids.size(), nullptr);
    return fu;
}

int fleet_future_wait(bdf_ctx* c, bdf_future* fu, bdf_agg4* out) {
    Fleet* f = c->fleet;
    const int n = fu->n;
    std::vector<std::vector<bdf_agg4>> res(f->kids.size(), std::vector<bdf_agg4>((size_t)std::max(n, 1)));
    int st = fleet_run(f, [&](int k) { return fu->fparts[k] ? bdf_future_wait(f->kids[k], fu->fparts[k], res[k].data()) : BDF_OK; });
    if (st == BDF_OK && out) for (int i = 0; i < n; i++) out[i] = res[0][i];   // every rank holds the same global records
    delete fu;
    return st;
}

// One elementwise operator over fleet columns: `call(kid, k, &result part, &future part)` runs the one-GPU entry on kid k's parts.
// out == nullptr: no result column (an aggregate-only expression); fut == nullptr: no fused aggregate (the kid gets nullptr).
static int fleet_op(bdf_ctx* c, int out_dtype, int n_in, const bdf_col* const* in, bdf_col** out, bdf_future** fut,
                    const std::function<int(bdf_ctx*, int, bdf_col**, bdf_future**)>& call) {
    int64_t n = 0;
    TRY(fleet_check_inputs(n_in, in, &n));
    bdf_col* o = out ? fleet_col_like(c, in[0], out_dtype, n) : nullptr;
    bdf_future* fu = fut ? fleet_future_new(c) : nullptr;
    if ((out && !o) || (fut && !fu)) { fleet_col_free(c, o); delete fu; return fail(BDF_OOM, "host allocation failed"); }
    Fleet* f = c->fleet;
    int st = fleet_run(f, [&](int k) { return call(f->kids[k], k, o ? &o->fparts[k] : nullptr, fu ? &fu->fparts[k] : nullptr); });
    if (st != BDF_OK) {
        const std::string keep = g_err;
        if (fu) fleet_future_wait(c, fu, nullptr);
        fleet_col_free(c, o);
        g_err = keep;
        return st;
    }
    if (out) *out = o;
    if (fut) *fut = fu;
    return BDF_OK;
}

int fleet_binary_dev(bdf_ctx* c, int op, const bdf_col* l, const bdf_col* r, bdf_col** out, bdf_future** fut) {
    const bdf_col* in[2] = {l, r};
    return fleet_op(c, l->dtype, 2, in, out, fut, [=](bdf_ctx* kid, int k, bdf_col** o, bdf_future** fu) {
        return fu ? bdf_binary_agg_dev_async(kid, op, l->fparts[k], r->fparts[k], o, fu) : bdf_binary_dev(kid, op, l->fparts[k], r->fparts[k], o);
    });
}

int fleet_map_dev(bdf_ctx* c, bool is_cast, int op_or_to, const bdf_col* in, bdf_col** out) {
    return fleet_op(c, is_cast ? op_or_to : in->dtype, 1, &in, out, nullptr, [=](bdf_ctx* kid, int k, bdf_col** o, bdf_future**) {
        return is_cast ? bdf_cast_dev(kid, op_or_to, in->fparts[k], o) : bdf_unary_dev(kid, op_or_to, in->fparts[k], o);
    });
}

int fleet_compare_dev(bdf_ctx* c, int op, const bdf_col* left, const bdf_col* right, double scalar, bdf_col** out) {
    const bdf_col* in[2] = {left, right};
    return fleet_op(c, kBool, right ? 2 : 1, in, out, nullptr, [=](bdf_ctx* kid, int k, bdf_col** o, bdf_future**) {
        return bdf_compare_dev(kid, op, left->fparts[k], right ? right->fparts[k] : nullptr, scalar, o);
    });
}

int fleet_boolean_dev(bdf_ctx* c, int op, const bdf_col* a, const bdf_col* b, bdf_col** out) {
    if (op == BDF_NOT) b = nullptr;
    const bdf_col* in[2] = {a, b};
    return fleet_op(c, kBool, b ? 2 : 1, in, out, nullptr, [=](bdf_ctx* kid, int k, bdf_col** o, bdf_future**) {
        return bdf_boolean_dev(kid, op, a->fparts[k], b ? b->fparts[k] : nullptr, o);
    });
}

int fleet_eval_expr(bdf_ctx* c, int n_inputs, const bdf_col* const* inputs, int n_nodes, const bdf_expr_node* nodes, bdf_col** out,
                    bdf_future** fut) {
    return fleet_op(c, BDF_F64, n_inputs, inputs, out, fut, [=](bdf_ctx* kid, int k, bdf_col** o, bdf_future** fu) {
        const bdf_col* parts[8];
        for (int i = 0; i < n_inputs; i++) parts[i] = inputs[i]->fparts[k];
        return fu ? bdf_eval_expr_agg_dev_async(kid, n_inputs, parts, n_nodes, nodes, o, fu) : bdf_eval_expr_dev(kid, n_inputs, parts, n_nodes, nodes, o);
    });
}

// Aggregates of n columns: every kid reduces its parts, the collective inside the kids' call makes the result global.
int fleet_aggregate_many(bdf_ctx* c, int32_t n_cols, const bdf_col* const* cols, bdf_future** fut) {
    Fleet* f = c->fleet;
    bdf_future* fu = fleet_future_new(c);
    if (!fu) return fail(BDF_OOM, "host allocation failed");
    fu->n = n_cols;
    int st = fleet_run(f, [&](int k) {
        std::vector<const bdf_col*> parts((size_t)n_cols);
        for (int32_t j = 0; j < n_cols; j++) parts[j] = cols[j]->fparts[k];
        return bdf_aggregate_all_many_dev_async(f->kids[k], n_cols, parts.data(), &fu->fparts[k]);
    });
    if (st != BDF_OK) { const std::string keep = g_err; fleet_future_wait(c, fu, nullptr); g_err = keep; return st; }
    *fut = fu;
    return BDF_OK;
}

// Logical chunks of a fleet column without a valid slot (empty or all-null): the reference's max/min unwrap() a None there.
// Evaluated over the caller's chunks -- a piece may be all-null while its chunk is not.
static int fleet_panic_chunks(bdf_ctx* c, const bdf_col* col, int* out) {
    Fleet* f = c->fleet;
    const size_t n = col->fmap.size();
    std::vector<int64_t> valid(n, 0);
    std::mutex m;
    int st = fleet_run(f, [&](int k) {
        for (size_t i = 0; i < n; i++)
            for (const auto& pc : col->fmap[i])
                if (pc.kid == k) {
                    int64_t len = 0, nulls = 0; int32_t hv = 0;
                    int s2 = bdf_col_chunk_info(f->kids[k], col->fparts[k], pc.local, &len, &nulls, &hv);
                    if (s2 != BDF_OK) return s2;
                    std::lock_guard<std::mutex> g(m);
                    valid[i] += len - (hv ? nulls : 0);
                }
        return (int)BDF_OK;
    });
    if (st != BDF_OK) return st;
    int k = 0;
    for (size_t i = 0; i < n; i++) if (valid[i] == 0) k++;
    *out = k;
    return BDF_OK;
}

int fleet_aggregate_dev(bdf_ctx* c, int op, const bdf_col* col, void* out_scalar, int32_t* is_some) {
    const int dtype = col->dtype;
    if (dtype == kBool) return fail(BDF_UNSUPPORTED, "aggregate of a boolean column");
    bdf_future* fu = nullptr;
    TRY(fleet_aggregate_many(c, 1, &col, &fu));
    bdf_agg4 a;
    TRY(fleet_future_wait(c, fu, &a));
    const int w = dtype_width(dtype);
    if (op == BDF_COUNT) { *(int64_t*)out_scalar = a.count; *is_some = 1; return BDF_OK; }
    if (op == BDF_SUM) { memcpy(out_scalar, &a.sum, (size_t)w); *is_some = 1; return BDF_OK; }
    int panics = 0;
    TRY(fleet_panic_chunks(c, col, &panics));
    if (panics) return fail(BDF_WOULD_PANIC, "max/min on an empty or all-null chunk: the reference unwraps None");
    *is_some = col->fmap.empty() ? 0 : 1;
    if (*is_some) memcpy(out_scalar, op == BDF_MIN ? &a.min : &a.max, (size_t)w);
    return BDF_OK;
}

int fleet_aggregate_all_blocking(bdf_ctx* c, int32_t n_cols, const bdf_col* const* cols, bdf_agg4* out) {
    bdf_future* fu = nullptr;
    TRY(fleet_aggregate_many(c, n_cols, cols, &fu));
    TRY(fleet_future_wait(c, fu, out));
    for (int32_t j = 0; j < n_cols; j++) {
        int panics = 0;
        TRY(fleet_panic_chunks(c, cols[j], &panics));
        out[j].would_panic = panics != 0;
        out[j].n_chunks = (int64_t)cols[j]->fmap.size();
    }
    return BDF_OK;
}

int fleet_avg_dev(bdf_ctx* c, const bdf_col* col, double* out, int32_t* is_some) {
    Fleet* f = c->fleet;
    std::vector<double> v(f->kids.size(), 0.0);
    std::vector<int32_t> some(f->kids.size(), 0);
    TRY(fleet_run(f, [&](int k) { return bdf_avg_dev(f->kids[k], col->fparts[k], &v[k], &some[k]); }));
    *out = v[0]; *is_some = some[0];
    // aggregate.rs:57-60: `mean + (m - mean) * len / count` is 0/0 when the first chunk has no valid slot, and NaN sticks
    if (!col->fmap.empty()) {
        int64_t len = 0, nulls = 0; int32_t hv = 0;
        TRY(fleet_chunk_info(c, col, 0, &len, &nulls, &hv));
        if (len - (hv ? nulls : 0) == 0) *out = std::numeric_limits<double>::quiet_NaN();
    }
    return BDF_OK;
}

// Host in / host out over every GPU: shard the views of the inputs (lists of n chunks with the same lengths), run the one-GPU
// drop-in entry per kid on its pieces (its own PCIe link), fold the metadata into the caller's chunks.
static int fleet_host(bdf_ctx* c, int out_dtype, int64_t n, std::initializer_list<const bdf_view*> ins, bdf_out* out,
                      const std::function<int(bdf_ctx*, int64_t, const bdf_view* const*, bdf_out*)>& call) {
    Fleet* f = c->fleet;
    const int nk = (int)f->kids.size();
    std::vector<int64_t> lens((size_t)n);
    for (int64_t i = 0; i < n; i++) lens[i] = (*ins.begin())[i].len;
    const auto map = fleet_plan(lens, nk);
    std::vector<std::vector<std::vector<bdf_view>>> views((size_t)nk);   // [kid][input]
    std::vector<std::vector<bdf_out>> outs((size_t)nk);
    for (int k = 0; k < nk; k++) {
        for (const bdf_view* in : ins) views[k].push_back(fleet_views(map, k, in));
        outs[k] = fleet_outs(map, k, out_dtype, out);
    }
    TRY(fleet_run(f, [&](int k) {
        bdf_view dv{}; bdf_out dummy{};
        std::vector<const bdf_view*> v;
        for (const auto& x : views[k]) v.push_back(x.empty() ? &dv : x.data());
        return call(f->kids[k], (int64_t)outs[k].size(), v.data(), outs[k].empty() ? &dummy : outs[k].data());
    }));
    fleet_merge_outs(map, outs, lens, out);
    return BDF_OK;
}

int fleet_binary_host(bdf_ctx* c, int op, int dtype, int64_t n, const bdf_view* left, const bdf_view* right, bdf_out* out) {
    return fleet_host(c, dtype, n, {left, right}, out, [&](bdf_ctx* kid, int64_t m, const bdf_view* const* v, bdf_out* o) {
        return bdf_binary(kid, op, dtype, m, v[0], m, v[1], o);
    });
}

int fleet_map_host(bdf_ctx* c, bool is_cast, int op_or_to, int dtype, int64_t n, const bdf_view* in, bdf_out* out) {
    return fleet_host(c, is_cast ? op_or_to : dtype, n, {in}, out, [&](bdf_ctx* kid, int64_t m, const bdf_view* const* v, bdf_out* o) {
        return is_cast ? bdf_cast(kid, dtype, op_or_to, m, v[0], o) : bdf_unary(kid, op_or_to, dtype, m, v[0], o);
    });
}

// Aggregates of a host column: upload the pieces (every GPU its own), run fn on the fleet column, release it.
int fleet_aggregate_host(bdf_ctx* c, int dtype, int64_t n, const bdf_view* in, const std::function<int(const bdf_col*)>& fn) {
    bdf_col* col = nullptr;
    const int32_t dt = dtype;
    TRY(fleet_upload_many(c, 1, &dt, &n, &in, BDF_ASYNC, &col));
    const int st = fn(col);
    const std::string keep = g_err;
    fleet_col_wait(c, col);   // host inputs must not be touched after return
    fleet_col_free(c, col);
    g_err = keep;
    return st;
}

int fleet_generate(bdf_ctx* c, int dtype, int kind, double lo, double hi, uint64_t seed, uint64_t col_id, int64_t n_chunks,
                   const int64_t* chunk_lens, int64_t row0, uint32_t null_mod, bdf_col** out) {
    Fleet* f = c->fleet;
    const int nk = (int)f->kids.size();
    bdf_col* col = fleet_col_planned(c, dtype, std::vector<int64_t>(chunk_lens, chunk_lens + n_chunks));
    if (!col) return fail(BDF_OOM, "host allocation failed");
    // a kid's pieces cover one contiguous range of global rows: generate them as one column starting at that row
    std::vector<std::vector<int64_t>> klens((size_t)nk);
    std::vector<int64_t> krow0((size_t)nk, -1);
    int64_t start = 0;
    for (int64_t i = 0; i < n_chunks; i++) {
        for (const auto& pc : col->fmap[i]) {
            if ((int64_t)klens[pc.kid].size() <= pc.local) klens[pc.kid].resize((size_t)pc.local + 1, 0);
            klens[pc.kid][pc.local] = pc.rows;
            if (krow0[pc.kid] < 0 && pc.rows > 0) krow0[pc.kid] = start + pc.row0;
        }
        start += chunk_lens[i];
    }
    int st = fleet_run(f, [&](int k) {
        const int64_t dummy = 0;
        return bdf_generate(f->kids[k], dtype, kind, lo, hi, seed, col_id, (int64_t)klens[k].size(), klens[k].empty() ? &dummy : klens[k].data(),
                            row0 + std::max<int64_t>(krow0[k], 0), null_mod, &col->fparts[k]);
    });
    if (st != BDF_OK) { const std::string keep = g_err; fleet_col_free(c, col); g_err = keep; return st; }
    *out = col;
    return BDF_OK;
}

// ---- context, device and measurement entries: every GPU in turn ----------------------------------------

void fleet_destroy(bdf_ctx* c) {
    Fleet* f = c->fleet;
    for (auto& w : f->workers) {
        { std::lock_guard<std::mutex> g(w->m); w->stop = true; }
        w->cv.notify_all();
        if (w->th.joinable()) w->th.join();
    }
    for (bdf_ctx* k : f->kids) bdf_destroy(k);
    delete f;
    delete c;
}

bdf_ctx* fleet_first_gpu(bdf_ctx* c) { return c->fleet->kids[0]; }

int fleet_each_gpu(bdf_ctx* c, const std::function<int(bdf_ctx*)>& fn) {
    for (bdf_ctx* k : c->fleet->kids) TRY(fn(k));
    return BDF_OK;
}

int fleet_device_info(bdf_ctx* c, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* hbm_bytes) {   // the first GPU's shape, the HBM of all of them
    int64_t total = 0, one = 0;
    for (bdf_ctx* k : c->fleet->kids) { TRY(bdf_device_info(k, sm_count, cc_major, cc_minor, &one)); total += one; }
    TRY(bdf_device_info(c->fleet->kids[0], sm_count, cc_major, cc_minor, &one));
    if (hbm_bytes) *hbm_bytes = total;
    return BDF_OK;
}

int fleet_comm_info(bdf_ctx* c, int32_t* rank, int32_t* world, int32_t* nccl_version, int64_t* collectives) {
    TRY(bdf_comm_info(c->fleet->kids[0], rank, world, nccl_version, collectives));
    if (rank) *rank = 0;
    return BDF_OK;
}

int fleet_profile_read(bdf_ctx* c, bdf_launch_record* buf, int64_t cap, int64_t* n) {
    int64_t total = 0;   // the records of all GPUs, GPU by GPU
    for (bdf_ctx* k : c->fleet->kids) {
        int64_t got = 0;
        TRY(bdf_profile_read(k, buf ? buf + total : nullptr, buf ? cap - total : 0, &got));
        total += got;
    }
    if (n) *n = total;
    return BDF_OK;
}

int64_t fleet_launch_count(bdf_ctx* c) {
    int64_t t = 0;
    for (bdf_ctx* k : c->fleet->kids) t += bdf_launch_count(k);
    return t;
}

int fleet_timer_stop(bdf_ctx* c, float* ms) {
    float worst = 0.f;   // the slowest GPU
    for (bdf_ctx* k : c->fleet->kids) { float one = 0.f; TRY(bdf_timer_stop(k, &one)); worst = std::max(worst, one); }
    if (ms) *ms = worst;
    return BDF_OK;
}

extern "C" {

int bdf_init_multi(int n_gpus, const int* devices, bdf_ctx** out) {
    if (!out) return fail(BDF_INVALID, "null out pointer");
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(BDF_CUDA, "no usable CUDA device (%s); this library has no CPU fallback", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (n_gpus == 0) n_gpus = n_dev;
    if (n_gpus < 1 || n_gpus > n_dev) return fail(BDF_INVALID, "%d GPUs requested, %d visible", n_gpus, n_dev);
    std::vector<int> devs((size_t)n_gpus);
    for (int i = 0; i < n_gpus; i++) {
        devs[i] = devices ? devices[i] : i;
        if (devs[i] < 0 || devs[i] >= n_dev) return fail(BDF_INVALID, "device %d out of range (0..%d)", devs[i], n_dev - 1);
        for (int j = 0; j < i; j++) if (devs[j] == devs[i]) return fail(BDF_INVALID, "device %d listed twice", devs[i]);
    }
    bdf_ctx* c = new (std::nothrow) bdf_ctx();
    Fleet* f = new (std::nothrow) Fleet();
    if (!c || !f) { delete c; delete f; return fail(BDF_OOM, "host allocation failed"); }
    c->fleet = f;
    c->device = devs[0];
    int st = BDF_OK;
    for (int i = 0; i < n_gpus && st == BDF_OK; i++) {
        bdf_ctx* kid = nullptr;
        st = bdf_init(devs[i], &kid);
        if (st == BDF_OK) f->kids.push_back(kid);
    }
    if (st == BDF_OK && n_gpus > 1) {   // ncclCommInitAll: one communicator, one rank per GPU, all in this process
        std::vector<Comm*> comms((size_t)n_gpus, nullptr);
        std::string err;
        if (comm_create_all(n_gpus, devs.data(), comms.data(), &err) != 0) st = fail(BDF_NCCL, "%s", err.c_str());
        else {
            for (int i = 0; i < n_gpus; i++) ctx_attach_comm(f->kids[i], comms[i]);
            const char* mode = getenv("BDF_COMBINE");
            if (!(mode && strcmp(mode, "nccl") == 0)) {
                std::string perr;
                if (comm_enable_p2p_all(n_gpus, comms.data(), &perr) == 0) for (Comm* cm : comms) comm_set_p2p(cm, true);
                else if (mode && strcmp(mode, "p2p") == 0) st = fail(BDF_NCCL, "BDF_COMBINE=p2p: %s", perr.c_str());
            }
        }
    }
    if (st == BDF_OK)
        for (int i = 0; i < n_gpus; i++) {
            f->workers.emplace_back(new Fleet::Worker());
            Fleet::Worker* w = f->workers.back().get();
            w->th = std::thread(fleet_worker_main, w, devs[i]);
        }
    if (st != BDF_OK) { const std::string keep = g_err; fleet_destroy(c); g_err = keep; return st; }
    *out = c;
    return BDF_OK;
}

int bdf_fleet_size(bdf_ctx* c) { return c ? (c->fleet ? (int)c->fleet->kids.size() : 1) : 0; }

}  // extern "C"
