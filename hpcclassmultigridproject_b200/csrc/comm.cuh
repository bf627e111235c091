// comm.cuh -- one-process-per-GPU communication for the row-slab sharded solver.
//  * a thin layer over NCCL (loaded at run time from the process: torch.distributed has already
//    mapped libnccl.so.2, a single-GPU user never needs it): bootstrap (all-gather of CUDA IPC
//    handles) and the fallback transport (send/receive groups, all-reduce);
//  * the production transport: kernels that store rows into the peers' memory over NVLink and
//    synchronise through device-side counters (further down).
#pragma once
#include "common.cuh"

namespace mgb200 {

struct Comm;

// rank 0 creates the 128-byte NCCL unique id; the host (bench.py / tests) broadcasts it
int comm_unique_id(unsigned char out[128]);
int comm_create(Comm** out, int rank, int nranks, const unsigned char id[128]);
void comm_destroy(Comm* c);
int comm_rank(const Comm* c);
int comm_size(const Comm* c);

// a batch of sends/receives issued as one NCCL group on `s`
struct P2P { int peer; double* buf; size_t count; bool send; };
int comm_p2p(Comm* c, const P2P* ops, int nops, cudaStream_t s);
// `count` doubles from rank `root` to every rank, in place (set-up traffic over NVLink)
int comm_broadcast(Comm* c, double* buf, size_t count, int root, cudaStream_t s);
// in-place sum of `count` doubles on every rank
int comm_allreduce_sum(Comm* c, double* buf, size_t count, cudaStream_t s);
// every rank contributes `bytes` bytes (device memory); recv holds nranks * bytes
int comm_allgather_bytes(Comm* c, const void* send, void* recv, size_t bytes, cudaStream_t s);


// ---- peer-memory transfers (NVLink stores + device-side counters, no NCCL on the path) ---------
// One launch copies up to eight row blocks into other ranks' memory (mapped with CUDA IPC); its
// last CTA then increments a counter on each destination rank and, if asked, waits until enough
// increments have arrived in this rank's own counters.  Counter block of a rank (ints):
//   [0..7]   arrivals, incremented by the peers       (slot 0: from rank-1, 1: from rank+1,
//                                                      2: gather contributions, 3: scatter from rank 0,
//                                                      4: norm contributions, 5: norm result from rank 0)
//   [8..15]  arrivals this rank has consumed so far
//   [16]     CTA arrival counter of the running launch
//   [19]     set when a wait gave up (a peer never arrived within ~2 s: it died or left the sequence); the host
//            checks it after synchronising and reports MGB200_ERR_STATE
// Graph-replayable: every counter lives in device memory, nothing changes in the kernel arguments
// between cycles.  Never run two ranks of one communicator on the same GPU (the waiter would spin
// against a kernel that cannot be scheduled).
constexpr int SYNC_FROM_UP = 0, SYNC_FROM_DOWN = 1, SYNC_GATHER = 2, SYNC_SCATTER = 3, SYNC_NORM_UP = 4, SYNC_NORM_DOWN = 5,
              SYNC_ABORT = 19, SYNC_INTS = 32;
// spin budget of a device-side wait for a peer, in clock64 ticks (~2 s)
constexpr long long SYNC_SPIN_BUDGET = 4000000000LL;
struct PeerSeg { const double* src; double* dst; long count; };      // count doubles, multiple of 2, 16-byte aligned
struct PeerPush {
    PeerSeg seg[8];
    int nseg;
    int* raise[8];            // remote arrival counters to increment once the stores are out
    int nraise;
    int* sync;                // this rank's counter block
    int wait_slot[2];         // own slots to wait on ...
    int wait_count[2];        // ... for this many new arrivals each
    int nwait;
};
int launch_peer_push(const PeerPush& a, cudaStream_t s);

// Sum of one double per rank through rank 0, in rank order (deterministic, identical on every
// rank): the others store their term into rank 0's `red[rank]`, rank 0 adds them up and stores
// the total into everybody's `red[0]`.  One single-thread launch per rank.
constexpr int RED_DOUBLES = 16;
struct NormReduce {
    double* value;            // in: this rank's term, out: the total
    double* red;              // this rank's landing block (RED_DOUBLES doubles, IPC-shared)
    double* peer_red[8];      // rank 0: red of rank r at [r]; other ranks: rank 0's red at [0]
    int* sync;                // this rank's counter block
    int* peer_sync[8];        // same indexing as peer_red
    int rank, nranks;
};
int launch_norm_allreduce(const NormReduce& a, cudaStream_t s);

}  // namespace mgb200
