// comm.cuh -- the one exchange step of the path (SURVEY.md 8(e)): the per-GPU partial aggregates are combined
// with NCCL over NVLink / NVSwitch, enqueued on the stream that produced them (no host round trip between
// the reducing kernel and the collective).  Implemented in comm.cu; used by runtime.cu and fleet.cu only.
//
// Reference seam: the cross-chunk fold of AggregateFunctions::{sum,min,max,count}
// (src/functions/aggregate.rs:12-31,70-93) -- chunks live on different GPUs here, so the fold over chunks
// becomes [fold over this GPU's chunks] -> [all-reduce over GPUs].
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "common.cuh"

namespace bdf {

struct Comm;  // one NCCL communicator + its device scratch, owned by a bdf_ctx

constexpr int kCommMaxCols = 64;      // aggregates combined by ONE grouped collective
constexpr int kCommIdBytes = 128;     // == NCCL_UNIQUE_ID_BYTES

// ncclGetUniqueId (rank 0 makes it, every rank passes the same bytes to comm_create).
int comm_unique_id(unsigned char* id, std::string* err);
// ncclCommInitRank on the current device.  Returns nullptr and fills err on failure.
Comm* comm_create(const unsigned char* id, int rank, int world, std::string* err);
// Single-process form: ncclCommInitAll over `devices` (the current device is restored).  out[n] receives the comms.
int comm_create_all(int n, const int* devices, Comm** out, std::string* err);
void comm_destroy(Comm* c);
int comm_rank(const Comm* c);
int comm_world(const Comm* c);
int comm_version();   // NCCL version code of the loaded library (0 when it is not loaded)

// Combine n local aggregates (AggDev records in device memory, as k_finish writes them) across the ranks, on `s`, as
// ONE group of collectives:
//   ncclAllReduce ncclSum over {sum bits, valid count, rows, panics, chunks} (u64, wrapping), ncclMin over the min keys,
//   ncclMax over the max keys -- order independent, so integer results are identical for every world size;
//   float columns (bit i of float_mask): the partial sums are also ncclAllGather-ed and folded in rank order
//   (deterministic for a given world size; covered by the float-sum tolerance).
// local_rows / local_panics / local_chunks ride along (rows of column i on this rank; chunks of it that are empty or
// all-null -- the reference's max/min unwrap() would panic; number of chunks of it on this rank).
// Results: result[2*i] = the combined AggDev, result[2*i+1] = {rows, panics, chunks, 0} -- `result` may be
// device-mapped host memory (it is written by a kernel, followed by a system-scope fence).
cudaError_t comm_combine(Comm* c, unsigned long long float_mask, int n, const AggDev* d_local, const unsigned long long* local_rows,
                         const unsigned int* local_panics, const unsigned int* local_chunks, AggDev* result, cudaStream_t s,
                         std::string* err);

// The same combine over NVLink peer memory instead of NCCL (k_p2p_combine in comm.cu): every rank stores its record into
// every peer's mailbox and folds what it received in rank order -- one small launch, no library call.  Needs peer access
// between all GPUs of the communicator (NVSwitch boxes have it).  comm_enable_p2p is collective (every rank calls it).
int comm_enable_p2p(Comm* c, std::string* err);               // process per GPU: CUDA IPC handles travel through the communicator
int comm_enable_p2p_all(int n, Comm** comms, std::string* err);   // one process: direct peer pointers
bool comm_has_p2p(const Comm* c);
bool comm_uses_p2p(const Comm* c);
int comm_set_p2p(Comm* c, bool on);   // non-zero if the mailboxes are not set up

// In-place all-reduce of device memory on `s` (the DivideByZero flag: every rank must take the same exit).
cudaError_t comm_allreduce_max_i32(Comm* c, int* d_inout, int n, cudaStream_t s, std::string* err);
// Blocking host-side helpers (bench timing, avg merge): stage through device scratch on `s`, synchronise.
cudaError_t comm_host_allreduce_f64(Comm* c, int op /*0 sum, 1 min, 2 max*/, double* inout, int n, cudaStream_t s, std::string* err);
cudaError_t comm_host_allgather(Comm* c, const void* in, void* out /* world * bytes */, size_t bytes, cudaStream_t s, std::string* err);

}  // namespace bdf
