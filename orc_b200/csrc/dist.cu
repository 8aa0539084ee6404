// dist.cu — NCCL communicator (resolved with dlopen) and the halo exchange of a row-partitioned mesh.
#include "dist.cuh"

#include <dlfcn.h>

#include <cstring>

namespace orc {

namespace {
struct ncclUniqueId_ { char internal[128]; };
typedef int (*fn_get_uid)(ncclUniqueId_*);
typedef int (*fn_init_rank)(void**, int, ncclUniqueId_, int);
typedef int (*fn_destroy)(void*);
typedef int (*fn_group)(void);
typedef int (*fn_sendrecv)(void*, size_t, int, int, void*, cudaStream_t);
typedef int (*fn_allreduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef const char* (*fn_errstr)(int);
struct Nccl {
    void* lib = nullptr;
    fn_get_uid get_uid = nullptr;
    fn_init_rank init_rank = nullptr;
    fn_destroy destroy = nullptr;
    fn_group group_start = nullptr, group_end = nullptr;
    fn_sendrecv send = nullptr, recv = nullptr;
    fn_allreduce allreduce = nullptr;
    fn_errstr errstr = nullptr;
};
Nccl& nccl() {
    static Nccl n;
    if (n.lib) return n;
    n.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!n.lib) n.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!n.lib) n.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!n.lib) throw Error(ORC_E_NCCL, std::string("cannot load libnccl.so.2: ") + dlerror());
    auto sym = [&](const char* name) {
        void* p = dlsym(n.lib, name);
        if (!p) throw Error(ORC_E_NCCL, std::string("libnccl lacks ") + name);
        return p;
    };
    n.get_uid = (fn_get_uid)sym("ncclGetUniqueId");
    n.init_rank = (fn_init_rank)sym("ncclCommInitRank");
    n.destroy = (fn_destroy)sym("ncclCommDestroy");
    n.group_start = (fn_group)sym("ncclGroupStart");
    n.group_end = (fn_group)sym("ncclGroupEnd");
    n.send = (fn_sendrecv)sym("ncclSend");
    n.recv = (fn_sendrecv)sym("ncclRecv");
    n.allreduce = (fn_allreduce)sym("ncclAllReduce");
    n.errstr = (fn_errstr)sym("ncclGetErrorString");
    return n;
}
void nccl_check(int rc, const char* what) {
    if (rc != 0) throw Error(ORC_E_NCCL, std::string(what) + ": " + nccl().errstr(rc));
}
constexpr int kNcclFloat64 = 8;  // ncclDataType_t::ncclFloat64
}  // namespace

void Comm::unique_id(char out128[128]) {
    ncclUniqueId_ id;
    nccl_check(nccl().get_uid(&id), "ncclGetUniqueId");
    memcpy(out128, id.internal, 128);
}
void Comm::init(Ctx& c, int rank_, int nranks_, const char id128[128]) {
    ORC_REQUIRE(nranks_ >= 1 && rank_ >= 0 && rank_ < nranks_, ORC_E_INVALID, "bad rank / nranks");
    rank = rank_; nranks = nranks_;
    if (nranks == 1) return;
    ncclUniqueId_ id;
    memcpy(id.internal, id128, 128);
    ORC_CUDA(cudaSetDevice(c.device));
    nccl_check(nccl().init_rank(&comm, nranks, id, rank), "ncclCommInitRank");
}
void Comm::destroy() {
    peer.destroy();
    if (comm) nccl().destroy(comm);
    comm = nullptr;
}
// ---- symmetric peer windows over CUDA IPC ------------------------------------------------------------------------------
void Peer::alloc_window(Ctx& c, int rank_, int nranks_, char handle_out64[64]) {
    ORC_REQUIRE(nranks_ <= kMaxRanks, ORC_E_UNSUPPORTED, "peer windows support up to 8 ranks per node");
    rank = rank_; nranks = nranks_;
    ORC_CUDA(cudaSetDevice(c.device));
    ORC_CUDA(cudaMalloc(&local, window_bytes()));
    ORC_CUDA(cudaMemset(local, 0, window_bytes()));
    cudaIpcMemHandle_t h;
    ORC_CUDA(cudaIpcGetMemHandle(&h, local));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle_out64, &h, 64);
}
void Peer::open(Ctx& c, const char* all_handles) {
    ORC_REQUIRE(local != nullptr, ORC_E_INVALID, "peer window not allocated");
    ORC_CUDA(cudaSetDevice(c.device));
    for (int r = 0; r < nranks; ++r) {
        if (r == rank) { remote[r] = local; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, all_handles + 64 * (size_t)r, 64);
        void* p = nullptr;
        ORC_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        remote[r] = static_cast<char*>(p);
    }
    on = true;
}
void Peer::destroy() {
    for (int r = 0; r < nranks; ++r)
        if (r != rank && remote[r]) cudaIpcCloseMemHandle(remote[r]);
    if (local) cudaFree(local);
    local = nullptr; on = false;
    for (auto& p : remote) p = nullptr;
}
PeerAr Comm::next_allreduce() {
    PeerAr pa;
    pa.rank = peer.rank; pa.nranks = peer.nranks; pa.seq = ++peer.ar_seq;
    for (int r = 0; r < peer.nranks; ++r) pa.win[r] = peer.remote[r];
    return pa;
}
__global__ void k_peer_allreduce(PeerAr pa, double* vals, int count, int op, int* flags) { peer_allreduce_warp(pa, vals, count, op, flags); }

void Comm::allreduce(Ctx& c, double* dev, int count, int op) {
    if (!active()) return;
    ProfScope ps(c, PC_OTHER, 0.);
    if (peer.on && count <= 6) {
        k_peer_allreduce<<<1, 32, 0, c.stream>>>(next_allreduce(), dev, count, op, c.d_flags);
        c.after_launch("k_peer_allreduce");
        return;
    }
    nccl_check(nccl().allreduce(dev, dev, (size_t)count, kNcclFloat64, op, comm, c.stream), "ncclAllReduce");
    ++c.launches;
}

// -------------------------------------------------------------------------------------------------
// cells of four doubles (three systems + padding): one 32-byte gather per packed cell
struct alignas(32) HaloCell { double a, b, c, d; };
__global__ void k_halo_pack(int count, const int* __restrict__ idx, const double* __restrict__ x, double* __restrict__ out) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x) out[k] = x[idx[k]];
}

__global__ void k_halo_pack4(int count, const int* __restrict__ idx, const double* __restrict__ x, double* __restrict__ out) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < count; k += gridDim.x * blockDim.x)
        reinterpret_cast<HaloCell*>(out)[k] = reinterpret_cast<const HaloCell*>(x)[idx[k]];
}

// ---- peer halo exchange -------------------------------------------------------------------------------------------------
struct PushArgs {
    int nnbr, ns, nfields, elem;           // elem: doubles per packed element (1, or 4 for the cells of three systems)
    int send_ptr[Peer::kMaxRanks + 1];
    char* stage[Peer::kMaxRanks];          // the neighbour's staging slot for (sender = this rank, parity of seq)
    unsigned long long* flag[Peer::kMaxRanks];   // the neighbour's sequence word for sender = this rank
    const double* fields[Halo::kMaxFields];
    unsigned long long seq;
};
__global__ void k_peer_push(PushArgs a, const int* __restrict__ idx, unsigned int* counter) {
    const long long total = (long long)a.nfields * a.ns;
    for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
        const int f = (int)(k / a.ns), j = (int)(k - (long long)f * a.ns);
        int q = 0;
        while (q + 1 < a.nnbr && j >= a.send_ptr[q + 1]) ++q;
        const int cnt = a.send_ptr[q + 1] - a.send_ptr[q];
        const size_t dst = ((size_t)f * cnt + (size_t)(j - a.send_ptr[q])) * a.elem;
        const size_t src = (size_t)idx[j] * a.elem;
        double* out = reinterpret_cast<double*>(a.stage[q]);
        if (a.elem == 4) reinterpret_cast<HaloCell*>(out)[dst / 4] = reinterpret_cast<const HaloCell*>(a.fields[f])[src / 4];
        else out[dst] = a.fields[f][src];
    }
    if (last_block_done(counter)) {   // every block has fenced its stores: publish the sequence number to the neighbours
        __threadfence_system();
        if (threadIdx.x < a.nnbr) *reinterpret_cast<volatile unsigned long long*>(a.flag[threadIdx.x]) = a.seq;
    }
}
struct UnpackArgs {
    int nnbr, nfields, elem;
    int recv_begin[Peer::kMaxRanks], recv_count[Peer::kMaxRanks];
    const char* stage[Peer::kMaxRanks];                  // local staging slot of (sender = neighbour, parity)
    const unsigned long long* flag[Peer::kMaxRanks];     // local sequence word of that sender
    double* fields[Halo::kMaxFields];
    unsigned long long seq;
};
__global__ void k_peer_unpack(UnpackArgs a, int* flags) {
    if (threadIdx.x < a.nnbr) {
        long long spins = 0;
        while (*reinterpret_cast<const volatile unsigned long long*>(a.flag[threadIdx.x]) < a.seq) {
            if (++spins > (1ll << 24)) { atomicOr(flags, DF_SPIN); break; }
        }
        __threadfence_system();
    }
    __syncthreads();
    for (int q = 0; q < a.nnbr; ++q) {
        const long long total = (long long)a.nfields * a.recv_count[q];
        const double* in = reinterpret_cast<const double*>(a.stage[q]);
        for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x) {
            const int f = (int)(k / a.recv_count[q]), j = (int)(k - (long long)f * a.recv_count[q]);
            if (a.elem == 4) {   // L2 loads (the peer's stores land in this GPU's L2; never through a stale L1 line)
                const double2 lo = __ldcg(reinterpret_cast<const double2*>(in) + 2 * k), hi = __ldcg(reinterpret_cast<const double2*>(in) + 2 * k + 1);
                HaloCell cell; cell.a = lo.x; cell.b = lo.y; cell.c = hi.x; cell.d = hi.y;
                reinterpret_cast<HaloCell*>(a.fields[f])[a.recv_begin[q] + j] = cell;
            } else {
                a.fields[f][a.recv_begin[q] + j] = __ldcg(in + k);
            }
        }
    }
}
bool Halo::exchange_peer(Ctx& c, Comm& comm, double* const* fields, int nfields, int stride) {
    Peer& P = comm.peer;
    if (!P.on || !peer_ok) return false;   // peer_ok: all ranks agreed that every link fits a staging slot (the widest message is 32 B per cell)
    const int ns = send_ptr.back();
    const unsigned long long seq = ++P.halo_seq;
    const size_t par = (size_t)(seq & 1ull);
    auto stage_of = [&](char* win, int sender) { return win + Peer::kMailBytes + Peer::kFlagBytes + ((size_t)sender * 2 + par) * Peer::kStageSlot; };
    auto flag_of = [&](char* win, int sender) { return reinterpret_cast<unsigned long long*>(win + Peer::kMailBytes) + sender; };
    PushArgs pa{};
    pa.nnbr = (int)nbr.size(); pa.ns = ns; pa.nfields = nfields; pa.elem = stride; pa.seq = seq;
    UnpackArgs ua{};
    ua.nnbr = (int)nbr.size(); ua.nfields = nfields; ua.elem = stride; ua.seq = seq;
    for (size_t q = 0; q <= nbr.size(); ++q) pa.send_ptr[q] = send_ptr[q];
    int max_recv = 1;
    for (size_t q = 0; q < nbr.size(); ++q) {
        pa.stage[q] = stage_of(P.remote[nbr[q]], P.rank);
        pa.flag[q] = flag_of(P.remote[nbr[q]], P.rank);
        ua.stage[q] = stage_of(P.local, nbr[q]);
        ua.flag[q] = flag_of(P.local, nbr[q]);
        ua.recv_begin[q] = recv_begin[q]; ua.recv_count[q] = recv_count[q];
        max_recv = std::max(max_recv, recv_count[q]);
    }
    for (int f = 0; f < nfields; ++f) { pa.fields[f] = fields[f]; ua.fields[f] = fields[f]; }
    k_peer_push<<<grid_for(std::max((long long)nfields * ns, 1ll), 256, c.sm_count * 2), 256, 0, c.stream>>>(pa, send_idx, push_counter);
    c.after_launch("k_peer_push");
    k_peer_unpack<<<grid_for(std::max((long long)nfields * max_recv, 1ll), 256, c.sm_count * 2), 256, 0, c.stream>>>(ua, c.d_flags);
    c.after_launch("k_peer_unpack");
    return true;
}

void Halo::agree_on_peer(Ctx& c, Comm& comm) {
    if (!comm.active() || !comm.peer.on) return;
    double widest = (int)nbr.size() > Peer::kMaxRanks ? 1e300 : 0.;
    for (size_t q = 0; q < nbr.size(); ++q) widest = std::max(widest, 32. * std::max(send_ptr[q + 1] - send_ptr[q], recv_count[q]));
    DBuf<double> d(&c, 1);
    ORC_CUDA(cudaMemcpyAsync(d.p, &widest, sizeof(double), cudaMemcpyHostToDevice, c.stream));
    comm.allreduce(c, d.p, 1, 2);   // max over the ranks
    ORC_CUDA(cudaMemcpyAsync(&widest, d.p, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    peer_ok = widest <= (double)Peer::kStageSlot;
}

void Halo::build(Ctx& c, const PartPlan& p) {
    n_loc = p.n_lo + p.n_own + p.n_hi;
    own_lo = p.n_lo; own_hi = p.n_lo + p.n_own;
    nbr.assign(p.nbr_rank.begin(), p.nbr_rank.end());
    send_ptr.assign(p.send_ptr.begin(), p.send_ptr.end());
    recv_begin.assign(p.recv_begin.begin(), p.recv_begin.end());
    recv_count.assign(p.recv_count.begin(), p.recv_count.end());
    const size_t ns = p.send_idx.size();
    send_idx.alloc(&c, std::max<size_t>(ns, 1));
    if (ns) ORC_CUDA(cudaMemcpyAsync(send_idx.p, p.send_idx.data(), ns * sizeof(int), cudaMemcpyHostToDevice, c.stream));
    sendbuf.alloc(&c, std::max<size_t>(ns * kMaxFields, 1));
    push_counter.alloc(&c, 1);
    push_counter.zero();
    c.sync();
}

void Halo::exchange(Ctx& c, Comm& comm, double* const* fields, int nfields, int stride) {
    ORC_REQUIRE(stride == 1 || stride == 4, ORC_E_INTERNAL, "halo exchange: cells hold 1 or 4 doubles");
    if (!comm.active() || nbr.empty()) return;
    ORC_REQUIRE(nfields >= 1 && nfields * stride <= kMaxFields, ORC_E_INVALID, "halo exchange: too many fields");
    ProfScope ps(c, PC_OTHER, 0.);
    if (exchange_peer(c, comm, fields, nfields, stride)) return;
    const int ns = send_ptr.back();
    for (int f = 0; f < nfields; ++f) {
        double* out = sendbuf.p + (size_t)f * ns * stride;
        if (stride == 1) {
            k_halo_pack<<<grid_for(std::max(ns, 1), 256, c.sm_count * 4), 256, 0, c.stream>>>(ns, send_idx, fields[f], out);
            c.after_launch("k_halo_pack");
        } else {
            k_halo_pack4<<<grid_for(std::max(ns, 1), 256, c.sm_count * 4), 256, 0, c.stream>>>(ns, send_idx, fields[f], out);
            c.after_launch("k_halo_pack4");
        }
    }
    Nccl& n = nccl();
    nccl_check(n.group_start(), "ncclGroupStart");
    for (int f = 0; f < nfields; ++f)
        for (size_t q = 0; q < nbr.size(); ++q) {
            const size_t cnt = (size_t)(send_ptr[q + 1] - send_ptr[q]) * stride, rcnt = (size_t)recv_count[q] * stride;
            double* out = sendbuf.p + ((size_t)f * ns + send_ptr[q]) * stride;
            if (cnt > 0) nccl_check(n.send(out, cnt, kNcclFloat64, nbr[q], comm.comm, c.stream), "ncclSend");
            if (rcnt > 0) nccl_check(n.recv(fields[f] + (size_t)recv_begin[q] * stride, rcnt, kNcclFloat64, nbr[q], comm.comm, c.stream), "ncclRecv");
        }
    nccl_check(n.group_end(), "ncclGroupEnd");
    ++c.launches;
}

}  // namespace orc
