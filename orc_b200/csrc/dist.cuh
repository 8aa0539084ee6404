// dist.cuh — multi-GPU plumbing of the SIMPLE loop (SURVEY.md §8e): one process per GPU, NCCL over NVLink/NVSwitch.
// C1 halo exchange of cell fields (ncclSend/ncclRecv, one group per exchange), C2 small allreduces for the BiCGSTAB
// scalars and the iteration scalars, C4 partition-lagged recurrences. AMG below the fine level is built per partition.
#pragma once
#include "linalg.cuh"
#include "mesh_host.hpp"

namespace orc {

// NCCL is resolved at run time (dlopen "libnccl.so.2"): a single-GPU process never loads it, and inside a torch process
// the already-loaded NCCL of torch is reused.
// Symmetric peer memory (CUDA IPC over NVLink / NVSwitch): every rank of the node maps a window of every other rank. The two
// latency-critical collectives of the distributed BiCGSTAB go through it instead of NCCL:
//  * one-shot allreduce of a few doubles: ONE kernel writes this rank's values + a sequence number into every peer's mailbox, waits
//    for the peers' entries and adds them up in rank order (deterministic, the same bits on every rank), then derives the BiCGSTAB
//    scalar that follows (alpha / omega / beta / rho) in the same launch — NCCL needs an allreduce and a scalar kernel;
//  * halo exchange: the pack kernel stores straight into the neighbour's staging slot and publishes a sequence number; the
//    receiver's unpack kernel waits for it and copies the slice into its halo cells. Two launches, no NCCL group.
// Staging and mailboxes are double buffered by sequence parity: a rank can be at most one collective ahead of a peer (it needs
// the peer's entry of collective k to finish k), so slot k % 2 is never overwritten before its reader is done.
struct Peer {
    static constexpr int kMaxRanks = 8;
    static constexpr size_t kMailDoubles = 8;                       // per (slot, sender): [sequence, 6 values, pad]
    static constexpr size_t kMailBytes = 2 * kMaxRanks * kMailDoubles * sizeof(double);
    static constexpr size_t kFlagBytes = 256;                        // halo sequence numbers, one per sender
    static constexpr size_t kStageSlot = (size_t)8 << 20;            // bytes per (sender, parity) staging slot
    bool on = false;
    int rank = 0, nranks = 1;
    char* local = nullptr;
    char* remote[kMaxRanks] = {};
    unsigned long long ar_seq = 0, halo_seq = 0;
    static size_t window_bytes() { return kMailBytes + kFlagBytes + 2 * (size_t)kMaxRanks * kStageSlot; }
    void alloc_window(Ctx& c, int rank_, int nranks_, char handle_out64[64]);
    void open(Ctx& c, const char* all_handles /* nranks x 64 bytes */);
    void destroy();
};

// what a kernel needs for the one-shot allreduce over the peer windows (passed by value)
struct PeerAr {
    int rank = 0, nranks = 1;
    unsigned long long seq = 0;
    char* win[Peer::kMaxRanks] = {};
};
struct Comm {
    int rank = 0, nranks = 1;
    void* comm = nullptr;  // ncclComm_t
    Peer peer;             // optional fast path (same node); NCCL is used whenever it is off
    bool active() const { return nranks > 1 && comm != nullptr; }
    static void unique_id(char out128[128]);
    void init(Ctx& c, int rank_, int nranks_, const char id128[128]);
    void destroy();
    // in-place allreduce of `count` (<= 6) doubles at `dev`; post_op >= 0 derives the BiCGSTAB scalars of K systems from the reduced
    // values in the same launch when the peer path is on (linalg.cu: DistOp), otherwise the caller launches k_dist_scalar itself
    void allreduce(Ctx& c, double* dev, int count, int op /* 0 sum, 2 max, 3 min */);
    PeerAr next_allreduce();   // the arguments of the next one-shot allreduce (advances the sequence number); peer path only
};

#ifdef __CUDACC__
// One-shot allreduce of `count` (<= 6) doubles, in place at `vals` (global memory), by ONE warp. Lane r writes this rank's values and
// then the sequence number into rank r's mailbox (system-scope fence in between), spins on the local mailbox entry of sender r,
// and the values are combined in rank order — the same order on every rank, so all ranks get the same bits. op: 0 sum, 2 max, 3 min.
__device__ __forceinline__ void peer_allreduce_warp(const PeerAr& pa, double* vals, int count, int op, int* flags) {
    const int lane = threadIdx.x & 31;
    const int parity = (int)(pa.seq & 1ull);
    double v[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) v[q] = (q < count) ? vals[q] : 0.;
    if (lane < pa.nranks) {
        double* e = reinterpret_cast<double*>(pa.win[lane]) + ((size_t)parity * Peer::kMaxRanks + pa.rank) * Peer::kMailDoubles;
#pragma unroll
        for (int q = 0; q < 6; ++q) if (q < count) ((volatile double*)e)[1 + q] = v[q];
        __threadfence_system();
        *reinterpret_cast<volatile unsigned long long*>(e) = pa.seq;
        const double* mine = reinterpret_cast<const double*>(pa.win[pa.rank]) + ((size_t)parity * Peer::kMaxRanks + lane) * Peer::kMailDoubles;
        long long spins = 0;
        while (*reinterpret_cast<const volatile unsigned long long*>(mine) != pa.seq) {
            if (++spins > (1ll << 24)) { atomicOr(flags, DF_SPIN); break; }
        }
        __threadfence_system();
#pragma unroll
        for (int q = 0; q < 6; ++q) if (q < count) v[q] = ((const volatile double*)mine)[1 + q];
    }
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        if (q >= count) continue;
        double acc = __shfl_sync(0xffffffffu, v[q], 0);
        for (int r = 1; r < pa.nranks; ++r) {
            const double o = __shfl_sync(0xffffffffu, v[q], r);
            acc = (op == 0) ? acc + o : (op == 2 ? fmax(acc, o) : fmin(acc, o));
        }
        if (lane == 0) vals[q] = acc;
    }
    __syncwarp();
}
#endif

// device-side exchange plan of one partition (from PartPlan)
struct Halo {
    int64_t n_loc = 0, own_lo = 0, own_hi = 0;
    std::vector<int> nbr, send_ptr, recv_begin, recv_count;
    DBuf<int> send_idx;       // local ids of owned cells to pack, all neighbours back to back
    DBuf<double> sendbuf;     // kMaxFields * total send count
    DBuf<unsigned int> push_counter;   // last-block-done counter of the peer push kernel (self-resetting)
    bool peer_ok = true;               // every link of EVERY rank fits a staging slot (agreed on by all ranks, agree_on_peer)
    void agree_on_peer(Ctx& c, Comm& comm);   // collective: call once per partition mesh after the communicator exists
    // peer path: ONE push kernel (pack + store into the neighbours' staging slots + publish the sequence number) and ONE unpack
    // kernel (wait for the neighbours' sequence numbers, copy the slices into the halo cells); false = message too large, use NCCL
    bool exchange_peer(Ctx& c, Comm& comm, double* const* fields, int nfields, int stride);
    static constexpr int kMaxFields = 4;
    void build(Ctx& c, const PartPlan& p);
    // exchanges vectors of n_loc cells of `stride` doubles (1 = plain vector, 4 = a batch of three systems, linalg.cu Cell<3>) in
    // one NCCL group: owned values -> the neighbours' halo slots. Up to kMaxFields doubles per cell over all fields.
    void exchange(Ctx& c, Comm& comm, double* const* fields, int nfields, int stride = 1);
    void exchange(Ctx& c, Comm& comm, double* x, int stride = 1) { exchange(c, comm, &x, 1, stride); }
};

struct DistEnv {  // what a distributed solve needs besides the matrices
    Comm* comm = nullptr;
    Halo* halo = nullptr;
    bool on() const { return comm && halo && comm->active(); }
};

}  // namespace orc
