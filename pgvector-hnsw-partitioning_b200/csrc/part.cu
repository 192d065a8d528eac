// part.cu -- the hash-partitioned index behind the C ABI (hb_part_*): what the fork adds to pgvector.
//
// The reference mount has no source (/root/reference/README.md:1), so the contract is the one
// BASELINE.json states: a row belongs to partition splitmix64(heap_tid) mod P, every partition is an
// ordinary HNSW index, a query is broadcast to all partitions and the per-partition top-k lists are
// merged.  One process per GPU: rank r owns the partitions {p : p mod world == r}.
//
// Data path of one search batch on a rank (nothing returns to the host in between):
//   queries (already on every rank, or ncclBroadcast from the root rank)
//     -> one scan per owned partition (hb_search_batch_dev + TID mapping), on the slot's sub-streams
//     -> part_merge_kernel over the owned partitions' lists -> packed block [tids nq x k | dist nq x k]
//     -> ONE ncclAllGather of that block (12 bytes per result)      -- the only exchange
//     -> part_merge_kernel over the world's blocks -> result, identical on every rank.
// All collectives of a handle are issued on ONE exchange stream, in call order, so every rank issues the
// same NCCL sequence as long as every rank makes the same hb_part_search_* calls (SPMD, like any NCCL
// program).  Up to HB_PART_SLOTS batches are in flight: batch i's exchange and merge run under batch
// i+1's scans.  NCCL is loaded with dlopen at the first hb_part call that needs it (world > 1), so the
// library itself has no link-time dependency on it.
#include "index.h"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace hb {

// ---- NCCL, resolved at run time -------------------------------------------------------------
struct NcclApi {
    void *lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    std::string why;
};

static NcclApi *nccl_api()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char *names[] = { getenv("HB_NCCL_LIB"), "libnccl.so.2", "libnccl.so" };
        for (const char *nm : names) {
            if (!nm || !*nm) continue;
            api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (api.lib) break;
            api.why = dlerror();
        }
        if (!api.lib) return;
#define HB_SYM(field, name)                                                       \
        api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.lib, name)); \
        if (!api.field) { api.why = std::string("missing symbol ") + name; api.lib = nullptr; return; }
        HB_SYM(GetUniqueId, "ncclGetUniqueId")
        HB_SYM(CommInitRank, "ncclCommInitRank")
        HB_SYM(CommDestroy, "ncclCommDestroy")
        HB_SYM(AllGather, "ncclAllGather")
        HB_SYM(Broadcast, "ncclBroadcast")
        HB_SYM(GetErrorString, "ncclGetErrorString")
        HB_SYM(GetVersion, "ncclGetVersion")
#undef HB_SYM
    });
    if (!api.lib) { set_error("NCCL is not available (dlopen libnccl.so.2: %s)", api.why.c_str()); return nullptr; }
    return &api;
}

#define HB_NCCL(call)                                                                                     \
    do {                                                                                                  \
        ncclResult_t r__ = (call);                                                                        \
        if (r__ != ncclSuccess) {                                                                         \
            hb::set_error("%s failed: %s (%s:%d)", #call, nccl_api()->GetErrorString(r__), __FILE__, __LINE__); \
            return HB_ECUDA;                                                                              \
        }                                                                                                 \
    } while (0)

// ---- merge ----------------------------------------------------------------------------------
// A "block" is one list set for nq queries: [tids nq x k int64 | dist nq x k fp32], nearest-first, padded with
// tid -1 / +inf.  Greedy head merge of n_lists blocks (block l at base + l * stride bytes) ordered by
// (distance, tid): since the key is a total order the result does not depend on how the lists are grouped
// (merging per rank and then across ranks equals one flat merge over all partitions).
__global__ void part_merge_kernel(const char *__restrict__ base, int n_lists, size_t stride, int64_t nq, int k,
                                  char *__restrict__ out)
{
    const int64_t qi = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    constexpr int MAXL = 64;
    uint8_t head[MAXL];
    for (int l = 0; l < n_lists; l++) head[l] = 0;
    const size_t dist_off = (size_t) nq * k * sizeof(int64_t);
    int64_t *out_t = reinterpret_cast<int64_t *>(out) + qi * k;
    float *out_d = reinterpret_cast<float *>(out + dist_off) + qi * k;
    for (int o = 0; o < k; o++) {
        int best = -1;
        float bd = 0.f;
        int64_t bt = 0;
        for (int l = 0; l < n_lists; l++) {
            if (head[l] >= k) continue;
            const char *b = base + (size_t) l * stride;
            const int64_t t = reinterpret_cast<const int64_t *>(b)[qi * k + head[l]];
            if (t < 0) { head[l] = (uint8_t) k; continue; }      // pads end a list
            const float d = reinterpret_cast<const float *>(b + dist_off)[qi * k + head[l]];
            if (best < 0 || d < bd || (d == bd && t < bt)) { best = l; bd = d; bt = t; }
        }
        if (best < 0) {
            out_t[o] = -1;
            out_d[o] = __int_as_float(0x7f800000);
        } else {
            out_t[o] = bt;
            out_d[o] = bd;
            head[best]++;
        }
    }
}

__global__ void part_pad_kernel(char *__restrict__ out, int64_t nq, int k)
{
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq * k) return;
    reinterpret_cast<int64_t *>(out)[i] = -1;
    reinterpret_cast<float *>(out + (size_t) nq * k * sizeof(int64_t))[i] = __int_as_float(0x7f800000);
}

// fold a scan's error word (tie tail beyond HB_TIE_LIMIT) into the slot's status word
__global__ void part_status_kernel(const int32_t *__restrict__ err, int32_t *__restrict__ status)
{
    if (*err) atomicOr(status, 1);
}


// ---- the exchange over peer memory ------------------------------------------------------------
// With peer access between the ranks' GPUs (NVLink / NVSwitch; buffers opened through CUDA IPC at first use) the
// all-gather needs no collective kernel: the merge of a rank's owned partitions writes its packed block STRAIGHT INTO
// every rank's receive buffer (remote stores over NVLink), the last CTA publishes a per-source epoch flag with a
// system-scope release, and each rank's final merge waits for the world's flags with acquire loads.  A second set of
// flags acknowledges consumption, so a slot's receive buffer is not overwritten before its owner merged it.  No SM is
// held by a spinning collective while the persistent scan kernels fill the machine; the NCCL path stays as fallback
// (option "exchange" = 0, or when peer access cannot be established).
constexpr int PART_MAX_WORLD = 64;
struct PeerView {
    char *base[PART_MAX_WORLD];      // rank r's exchange buffer as mapped in this process (own buffer for r == rank)
    size_t blk_cap;                  // bytes reserved per source block
    size_t flags_off;                // int32 ready[world] | int32 ack[world] behind the blocks
    int rank, world;
};
__device__ __forceinline__ int ld_acquire_sys(const int *p)
{
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(int *p, int v)
{
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// one warp waits until flags[0 .. world) have all reached `epoch` (a kernel of its own, so that the waiting holds one
// warp and not the CTAs of the merge that follows it in the stream)
// A rank that never arrives (it failed, or the ranks' call sequences diverged) must not hang the GPU: after ~20 s the
// wait gives up and flags the slot's status word (bit 1), which hb_part_search_wait reports.
__global__ void part_wait_kernel(const int *flags, int world, int epoch, int32_t *status)
{
    const long long t0 = clock64();
    for (int r = threadIdx.x; r < world; r += 32)
        while (ld_acquire_sys(flags + r) < epoch) {
            if (clock64() - t0 > 40000000000ll) { atomicOr(status, 2); return; }
        }
}

// merge the owned partitions' lists (n_lists blocks at `lists`, stride `stride`; n_lists == 0: nothing owned) and
// store the result into block `rank` of every rank's buffer; then publish ready[rank] = epoch everywhere
__global__ void part_push_kernel(const char *__restrict__ lists, int n_lists, size_t stride, int64_t nq, int k, PeerView pv,
                                 int epoch, unsigned int *done_counter)
{
    // (part_wait_kernel ran before: every rank has consumed this slot's previous batch)
    const int64_t qi = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (qi < nq) {
        uint8_t head[PART_MAX_WORLD];
        for (int l = 0; l < n_lists; l++) head[l] = 0;
        const size_t dist_off = (size_t) nq * k * sizeof(int64_t);
        for (int o = 0; o < k; o++) {
            int best = -1;
            float bd = __int_as_float(0x7f800000);
            int64_t bt = -1;
            for (int l = 0; l < n_lists; l++) {
                if (head[l] >= k) continue;
                const char *b = lists + (size_t) l * stride;
                const int64_t t = reinterpret_cast<const int64_t *>(b)[qi * k + head[l]];
                if (t < 0) { head[l] = (uint8_t) k; continue; }
                const float d = reinterpret_cast<const float *>(b + dist_off)[qi * k + head[l]];
                if (best < 0 || d < bd || (d == bd && t < bt)) { best = l; bd = d; bt = t; }
            }
            if (best >= 0) head[best]++;
            else { bt = -1; bd = __int_as_float(0x7f800000); }
            for (int r = 0; r < pv.world; r++) {
                char *dst = pv.base[r] + (size_t) pv.rank * pv.blk_cap;
                reinterpret_cast<int64_t *>(dst)[qi * k + o] = bt;
                reinterpret_cast<float *>(dst + dist_off)[qi * k + o] = bd;
            }
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned prev = atomicAdd(done_counter, 1u);
        if (prev == gridDim.x - 1) {
            *done_counter = 0;
            __threadfence_system();
            for (int r = 0; r < pv.world; r++) st_release_sys(reinterpret_cast<int *>(pv.base[r] + pv.flags_off) + pv.rank, epoch);
        }
    }
}

// wait for every rank's block of this epoch, merge them, acknowledge
__global__ void part_pull_merge_kernel(PeerView pv, int64_t nq, int k, int epoch, char *__restrict__ out, unsigned int *done_counter)
{
    // (part_wait_kernel ran before: every rank's block of this epoch has arrived)
    const int64_t qi = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (qi < nq) {
        const char *base = pv.base[pv.rank];
        uint8_t head[PART_MAX_WORLD];
        for (int l = 0; l < pv.world; l++) head[l] = 0;
        const size_t dist_off = (size_t) nq * k * sizeof(int64_t);
        int64_t *out_t = reinterpret_cast<int64_t *>(out) + qi * k;
        float *out_d = reinterpret_cast<float *>(out + dist_off) + qi * k;
        for (int o = 0; o < k; o++) {
            int best = -1;
            float bd = 0.f;
            int64_t bt = 0;
            for (int l = 0; l < pv.world; l++) {
                if (head[l] >= k) continue;
                const char *b = base + (size_t) l * pv.blk_cap;
                // written by a peer over NVLink: read through L2, never from a stale L1 line of an earlier batch
                const int64_t t = __ldcg(reinterpret_cast<const long long *>(b) + qi * k + head[l]);
                if (t < 0) { head[l] = (uint8_t) k; continue; }
                const float d = __ldcg(reinterpret_cast<const float *>(b + dist_off) + qi * k + head[l]);
                if (best < 0 || d < bd || (d == bd && t < bt)) { best = l; bd = d; bt = t; }
            }
            if (best < 0) { out_t[o] = -1; out_d[o] = __int_as_float(0x7f800000); }
            else { out_t[o] = bt; out_d[o] = bd; head[best]++; }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned prev = atomicAdd(done_counter, 1u);
        if (prev == gridDim.x - 1) {
            *done_counter = 0;
            __threadfence_system();
            for (int r = 0; r < pv.world; r++) st_release_sys(reinterpret_cast<int *>(pv.base[r] + pv.flags_off) + pv.world + pv.rank, epoch);
        }
    }
}

constexpr int PART_SLOTS = 4;
constexpr int PART_SUBSTREAMS = 4;

struct PartSlot {
    cudaStream_t s = nullptr;                    // H2D of the queries, D2H of the results
    cudaStream_t sub[PART_SUBSTREAMS] = { nullptr, nullptr, nullptr, nullptr };   // partition scans
    cudaEvent_t ev_q = nullptr, ev_done = nullptr, ev_sub[PART_SUBSTREAMS] = { nullptr, nullptr, nullptr, nullptr };
    DevBuf q, elem, edist, cnt, lists, send, recv, out, status;
    int32_t *h_status = nullptr;                 // pinned
    // peer-memory exchange: this rank's buffer [world blocks | ready flags | ack flags], the peers' mapped in
    char *xbuf = nullptr;
    char *peer[PART_MAX_WORLD] = { nullptr };
    size_t xblk_cap = 0, xflags_off = 0;
    int epoch = 0;
    bool pending = false, tail_queued = false;
    int64_t nq = 0;
    int k = 0, ef = 0, nsub = 0, out_dev = 0;
    int64_t *out_tids = nullptr;
    float *out_dist = nullptr;
};

}   // namespace hb

using namespace hb;

struct hb_part {
    int device = 0, dim = 0, m = 0, efc = 0, metric = 0, dtype = 0, esize = 4;
    int P = 1, rank = 0, world = 1;
    std::vector<int> owned;                      // partition numbers, ascending
    std::vector<hb_index *> parts;               // handles of the owned partitions, same order
    ncclComm_t comm = nullptr;
    cudaStream_t xs = nullptr;                   // the exchange stream: every collective, in call order
    int exchange = 1;                            // 1 = stores into peer memory + flags, 0 = ncclAllGather
    bool peer_failed = false;                    // peer access could not be set up: NCCL from then on
    DevBuf xmisc;                                // counters of the push / pull kernels, handle exchange scratch
    PartSlot slots[PART_SLOTS];
    uint64_t issued = 0;                         // batches issued so far (diagnostics)
};

static size_t block_bytes(int64_t nq, int k) { return (((size_t) nq * k * 12) + 15) & ~(size_t) 15; }

static int slot_init(hb_part *pt, PartSlot &S)
{
    if (S.s) return HB_OK;
    HB_CK(cudaStreamCreateWithFlags(&S.s, cudaStreamNonBlocking));
    for (int j = 0; j < PART_SUBSTREAMS; j++) {
        HB_CK(cudaStreamCreateWithFlags(&S.sub[j], cudaStreamNonBlocking));
        HB_CK(cudaEventCreateWithFlags(&S.ev_sub[j], cudaEventDisableTiming));
    }
    HB_CK(cudaEventCreateWithFlags(&S.ev_q, cudaEventDisableTiming));
    HB_CK(cudaEventCreateWithFlags(&S.ev_done, cudaEventDisableTiming));
    HB_CK(cudaMallocHost(&S.h_status, 64));
    HB_CK(S.status.ensure(64));
    (void) pt;
    return HB_OK;
}

static void slot_release(PartSlot &S)
{
    DevBuf *b[] = { &S.q, &S.elem, &S.edist, &S.cnt, &S.lists, &S.send, &S.recv, &S.out, &S.status };
    for (auto x : b) x->release();
    if (S.h_status) cudaFreeHost(S.h_status);
    if (S.ev_q) cudaEventDestroy(S.ev_q);
    if (S.ev_done) cudaEventDestroy(S.ev_done);
    for (int j = 0; j < PART_SUBSTREAMS; j++) {
        if (S.ev_sub[j]) cudaEventDestroy(S.ev_sub[j]);
        if (S.sub[j]) cudaStreamDestroy(S.sub[j]);
    }
    if (S.s) cudaStreamDestroy(S.s);
    S = PartSlot();
}


// (Re)allocate slot S's exchange buffer for blocks of `blk` bytes and map every peer's into this process.  Collective:
// every rank calls it at the same point (the first batch of a slot, or a larger nq / k), because the IPC handles are
// exchanged with one ncclAllGather.  Returns HB_OK and sets pt->peer_failed when peer access is not available.
static void peer_close(hb_part *pt, PartSlot &S)
{
    for (int r = 0; r < pt->world; r++) {
        if (S.peer[r] && r != pt->rank) cudaIpcCloseMemHandle(S.peer[r]);
        S.peer[r] = nullptr;
    }
}
static void peer_unmap(hb_part *pt, PartSlot &S)
{
    peer_close(pt, S);
    if (S.xbuf) cudaFree(S.xbuf);
    S.xbuf = nullptr; S.xblk_cap = 0;
}
// every rank has closed its mappings of the others' buffers before anybody frees one
static void peer_barrier(hb_part *pt)
{
    NcclApi *nc = nccl_api();
    if (!nc || !pt->comm || !pt->xmisc.p) return;
    char *scratch = pt->xmisc.as<char>() + 256;
    if (nc->AllGather(scratch, scratch + 64, 4, ncclChar, pt->comm, pt->xs) == ncclSuccess) cudaStreamSynchronize(pt->xs);
}

static int peer_ensure(hb_part *pt, PartSlot &S, size_t blk)
{
    if (pt->peer_failed || blk <= S.xblk_cap) return HB_OK;
    NcclApi *nc = nccl_api();
    if (!nc) return HB_ECUDA;
    HB_CK(cudaDeviceSynchronize());                        // nothing of this handle is in flight on a buffer about to go
    if (S.xbuf) { peer_close(pt, S); peer_barrier(pt); }
    peer_unmap(pt, S);
    const int W = pt->world;
    const size_t cap = (blk + blk / 4 + 255) & ~(size_t) 255;
    const size_t flags_off = cap * W;
    const size_t total = flags_off + sizeof(int) * 2 * W + 64;
    HB_CK(cudaMalloc(&S.xbuf, total));
    HB_CK(cudaMemset(S.xbuf, 0, total));
    HB_CK(cudaDeviceSynchronize());                        // flags are zero before any peer can learn the address
    S.epoch = 0;
    cudaIpcMemHandle_t mine;
    bool ok = cudaIpcGetMemHandle(&mine, S.xbuf) == cudaSuccess;
    if (!ok) { cudaGetLastError(); memset(&mine, 0, sizeof mine); }
    // all-gather {ok, handle}
    struct Rec { int ok; int pad; cudaIpcMemHandle_t h; };
    HB_CK(pt->xmisc.ensure(256 + sizeof(Rec) * (size_t) (W + 1)));
    Rec *d_send = reinterpret_cast<Rec *>(pt->xmisc.as<char>() + 256), *d_recv = d_send + 1;
    Rec rec;
    rec.ok = ok ? 1 : 0; rec.pad = 0; rec.h = mine;
    std::vector<Rec> all(W);
    HB_CK(cudaMemcpyAsync(d_send, &rec, sizeof rec, cudaMemcpyHostToDevice, pt->xs));
    HB_NCCL(nc->AllGather(d_send, d_recv, sizeof(Rec), ncclChar, pt->comm, pt->xs));
    HB_CK(cudaMemcpyAsync(all.data(), d_recv, sizeof(Rec) * W, cudaMemcpyDeviceToHost, pt->xs));
    HB_CK(cudaStreamSynchronize(pt->xs));
    for (int r = 0; r < W; r++) ok = ok && all[r].ok;
    if (ok) {
        for (int r = 0; r < W && ok; r++) {
            if (r == pt->rank) { S.peer[r] = S.xbuf; continue; }
            void *ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, all[r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = false; }
            S.peer[r] = (char *) ptr;
        }
    }
    // agree on the outcome: one rank that cannot map a peer sends everybody to the NCCL path
    rec.ok = ok ? 1 : 0;
    HB_CK(cudaMemcpyAsync(d_send, &rec, sizeof rec, cudaMemcpyHostToDevice, pt->xs));
    HB_NCCL(nc->AllGather(d_send, d_recv, sizeof(Rec), ncclChar, pt->comm, pt->xs));
    HB_CK(cudaMemcpyAsync(all.data(), d_recv, sizeof(Rec) * W, cudaMemcpyDeviceToHost, pt->xs));
    HB_CK(cudaStreamSynchronize(pt->xs));
    for (int r = 0; r < W; r++) ok = ok && all[r].ok;
    if (!ok) {
        peer_unmap(pt, S);
        pt->peer_failed = true;
        return HB_OK;
    }
    S.xblk_cap = cap;
    S.xflags_off = flags_off;
    return HB_OK;
}

// the exchange + final merge of one batch, queued on the exchange stream
static int queue_tail(hb_part *pt, PartSlot &S)
{
    if (S.tail_queued) return HB_OK;
    const int64_t nq = S.nq;
    const int k = S.k;
    const size_t blk = block_bytes(nq, k);
    const int tgrid = (int) ((nq + 127) / 128);
    cudaStream_t xs = pt->xs;
    for (int j = 0; j < S.nsub; j++) HB_CK(cudaStreamWaitEvent(xs, S.ev_sub[j], 0));
    const int no = (int) pt->owned.size();
    char *result = nullptr;
    if (pt->world > 1 && pt->exchange == 1 && !pt->peer_failed && S.xbuf && blk <= S.xblk_cap) {
        // merge of the owned partitions pushed straight into every rank's receive block; flags instead of a collective
        PeerView pv;
        memset(&pv, 0, sizeof pv);
        for (int r = 0; r < pt->world; r++) pv.base[r] = S.peer[r];
        pv.blk_cap = S.xblk_cap; pv.flags_off = S.xflags_off; pv.rank = pt->rank; pv.world = pt->world;
        S.epoch++;
        unsigned int *counters = pt->xmisc.as<unsigned int>();
        const int *my_flags = reinterpret_cast<const int *>(S.xbuf + S.xflags_off);
        part_wait_kernel<<<1, 32, 0, xs>>>(my_flags + pt->world, pt->world, S.epoch - 1, S.status.as<int32_t>());          // acknowledgements of the slot's previous batch
        part_push_kernel<<<tgrid, 128, 0, xs>>>(S.lists.as<char>(), no, blk, nq, k, pv, S.epoch, counters + 2 * (int) (&S - pt->slots));
        HB_CK(cudaGetLastError());
        part_wait_kernel<<<1, 32, 0, xs>>>(my_flags, pt->world, S.epoch, S.status.as<int32_t>());                           // every rank's block of this batch
        part_pull_merge_kernel<<<tgrid, 128, 0, xs>>>(pv, nq, k, S.epoch, S.out.as<char>(), counters + 2 * (int) (&S - pt->slots) + 1);
        HB_CK(cudaGetLastError());
        result = S.out.as<char>();
    } else {
        char *local = nullptr;
        if (no == 0) {
            part_pad_kernel<<<(int) ((nq * k + 255) / 256), 256, 0, xs>>>(S.send.as<char>(), nq, k);
            local = S.send.as<char>();
        } else if (no == 1) {
            local = S.lists.as<char>();                      // one partition: its list is the rank's list
        } else {
            part_merge_kernel<<<tgrid, 128, 0, xs>>>(S.lists.as<char>(), no, blk, nq, k, S.send.as<char>());
            local = S.send.as<char>();
        }
        HB_CK(cudaGetLastError());
        result = local;
        if (pt->world > 1) {
            NcclApi *nc = nccl_api();
            if (!nc) return HB_ECUDA;
            HB_NCCL(nc->AllGather(local, S.recv.p, blk, ncclChar, pt->comm, xs));
            part_merge_kernel<<<tgrid, 128, 0, xs>>>(S.recv.as<char>(), pt->world, blk, nq, k, S.out.as<char>());
            HB_CK(cudaGetLastError());
            result = S.out.as<char>();
        }
    }
    HB_CK(cudaEventRecord(S.ev_done, xs));
    HB_CK(cudaStreamWaitEvent(S.s, S.ev_done, 0));
    const size_t tb = (size_t) nq * k * sizeof(int64_t), db = (size_t) nq * k * sizeof(float);
    const cudaMemcpyKind kind = S.out_dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    HB_CK(cudaMemcpyAsync(S.out_tids, result, tb, kind, S.s));
    HB_CK(cudaMemcpyAsync(S.out_dist, result + tb, db, kind, S.s));
    HB_CK(cudaMemcpyAsync(S.h_status, S.status.p, sizeof(int32_t), cudaMemcpyDeviceToHost, S.s));
    S.tail_queued = true;
    return HB_OK;
}

extern "C" {

int hb_part_unique_id(void *id_out)
{
    if (!id_out) { set_error("hb_part_unique_id: NULL argument"); return HB_EINVAL; }
    NcclApi *nc = nccl_api();
    if (!nc) return HB_ECUDA;
    static_assert(sizeof(ncclUniqueId) == HB_PART_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    HB_NCCL(nc->GetUniqueId(&id));
    memcpy(id_out, &id, sizeof id);
    return HB_OK;
}

void hb_part_free(hb_part *pt)
{
    if (!pt) return;
    cudaSetDevice(pt->device);
    cudaDeviceSynchronize();
    bool any_peer = false;
    for (auto &S : pt->slots) { if (S.xbuf) any_peer = true; peer_close(pt, S); }
    if (any_peer) peer_barrier(pt);
    for (auto &S : pt->slots) { peer_unmap(pt, S); slot_release(S); }
    pt->xmisc.release();
    if (pt->comm) { NcclApi *nc = nccl_api(); if (nc) nc->CommDestroy(pt->comm); }
    if (pt->xs) cudaStreamDestroy(pt->xs);
    for (hb_index *ix : pt->parts) hb_index_free(ix);
    delete pt;
}

hb_part *hb_part_create(int device, int dim, int m, int ef_construction, int metric, int dtype, int n_partitions,
                        int64_t capacity_per_partition, uint64_t seed, int rank, int world, const void *unique_id)
{
    if (n_partitions < 1 || n_partitions > 64 || world < 1 || rank < 0 || rank >= world || (world > 1 && !unique_id)) {
        set_error("hb_part_create: bad argument (1 <= partitions <= 64, 0 <= rank < world, unique_id needed when world > 1)");
        return nullptr;
    }
    hb_part *pt = new hb_part();
    pt->device = device; pt->dim = dim; pt->m = m; pt->efc = ef_construction; pt->metric = metric; pt->dtype = dtype;
    pt->esize = dtype == HB_F32 ? 4 : 2;
    pt->P = n_partitions; pt->rank = rank; pt->world = world;
    for (int p = rank; p < n_partitions; p += world) {
        // partition p draws its levels from its own seed, whatever rank builds it
        hb_index *ix = hb_index_create(device, dim, m, ef_construction, metric, dtype, capacity_per_partition, seed + (uint64_t) p);
        if (!ix) { hb_part_free(pt); return nullptr; }
        pt->owned.push_back(p);
        pt->parts.push_back(ix);
    }
    // the exchange stream gets the highest priority: the scans are persistent kernels that keep every SM full, and the
    // all-gather's and the merges' CTAs must not queue behind a whole batch of them
    int prio_lo = 0, prio_hi = 0;
    if (cudaSetDevice(device) == cudaSuccess) cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithPriority(&pt->xs, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
        set_error("hb_part_create: no CUDA device %d; there is no CPU fallback", device);
        hb_part_free(pt);
        return nullptr;
    }
    if (pt->xmisc.ensure(8192) != cudaSuccess || cudaMemset(pt->xmisc.p, 0, 8192) != cudaSuccess) {
        set_error("hb_part_create: out of device memory");
        hb_part_free(pt);
        return nullptr;
    }
    if (world > PART_MAX_WORLD) pt->exchange = 0;
    if (world > 1) {
        NcclApi *nc = nccl_api();
        if (!nc) { hb_part_free(pt); return nullptr; }
        ncclUniqueId id;
        memcpy(&id, unique_id, sizeof id);
        const ncclResult_t r = nc->CommInitRank(&pt->comm, world, id, rank);
        if (r != ncclSuccess) {
            set_error("ncclCommInitRank(rank %d of %d) failed: %s", rank, world, nc->GetErrorString(r));
            pt->comm = nullptr;
            hb_part_free(pt);
            return nullptr;
        }
    }
    return pt;
}

int hb_part_owned(const hb_part *pt, int32_t *partitions)
{
    if (!pt) return HB_EINVAL;
    if (partitions) for (size_t i = 0; i < pt->owned.size(); i++) partitions[i] = pt->owned[i];
    return (int) pt->owned.size();
}

hb_index *hb_part_index(hb_part *pt, int partition)
{
    if (!pt) return nullptr;
    for (size_t i = 0; i < pt->owned.size(); i++) if (pt->owned[i] == partition) return pt->parts[i];
    return nullptr;
}

int64_t hb_part_size(const hb_part *pt)
{
    if (!pt) return HB_EINVAL;
    int64_t n = 0;
    for (hb_index *ix : pt->parts) n += ix->n;
    return n;
}

int hb_part_set_option(hb_part *pt, const char *name, int value)
{
    if (!pt) return HB_EINVAL;
    if (name && !strcmp(name, "exchange")) { pt->exchange = value; return HB_OK; }      // 1 = peer-memory stores + flags, 0 = ncclAllGather
    for (hb_index *ix : pt->parts) { const int rc = hb_set_option(ix, name, value); if (rc) return rc; }
    return HB_OK;
}

int hb_part_get_counters(hb_part *pt, hb_counters *out, int reset)
{
    if (!pt || !out) return HB_EINVAL;
    memset(out, 0, sizeof *out);
    for (hb_index *ix : pt->parts) {
        hb_counters c;
        const int rc = hb_get_counters(ix, &c, reset);
        if (rc) return rc;
        out->n_dist += c.n_dist; out->n_hop0 += c.n_hop0; out->n_hopu += c.n_hopu; out->n_pair += c.n_pair; out->n_slow += c.n_slow;
    }
    return HB_OK;
}

// hnswbuild / hnswinsert of the partitioned index: every rank is handed the same tuples (or any superset
// of the ones it owns); a tuple is indexed by the rank that owns partition splitmix64(tid) mod P.  The
// partitions a rank owns are built concurrently, one host thread each (the handles share nothing), so
// that the latency-bound small batches at the start of every build overlap on the GPU.  No collective.
int64_t hb_part_build(hb_part *pt, const void *host_vecs, int64_t n, const int64_t *heap_tids)
{
    if (!pt || (!host_vecs && n > 0) || n < 0) { set_error("hb_part_build: bad argument"); return HB_EINVAL; }
    const int no = (int) pt->owned.size();
    if (no == 0 || n == 0) return 0;
    std::vector<int> slot_of(pt->P, -1);
    for (int i = 0; i < no; i++) slot_of[pt->owned[i]] = i;
    std::vector<std::vector<int64_t>> rows(no);
    for (auto &r : rows) r.reserve((size_t) (n / pt->P + n / (8 * pt->P) + 16));
    for (int64_t i = 0; i < n; i++) {
        const int64_t tid = heap_tids ? heap_tids[i] : i;
        const int s = slot_of[(int) (splitmix64((uint64_t) tid) % (uint64_t) pt->P)];
        if (s >= 0) rows[s].push_back(i);
    }
    const size_t row = (size_t) pt->dim * pt->esize;
    std::vector<int64_t> done(no, 0);
    std::vector<std::string> msg(no);
    auto work = [&](int s) {
        const std::vector<int64_t> &r = rows[s];
        if (r.empty()) return;
        if ((int64_t) r.size() == n) {
            // every tuple handed in belongs to this partition (a caller that routed already): index it in place
            done[s] = hb_insert(pt->parts[s], host_vecs, n, heap_tids);
        } else {
            std::unique_ptr<char[]> buf(new char[r.size() * row]);       // not value-initialised: written once below
            std::vector<int64_t> tids(r.size());
            for (size_t j = 0; j < r.size(); j++) {
                memcpy(buf.get() + j * row, (const char *) host_vecs + (size_t) r[j] * row, row);
                tids[j] = heap_tids ? heap_tids[r[j]] : r[j];
            }
            done[s] = hb_insert(pt->parts[s], buf.get(), (int64_t) r.size(), tids.data());
        }
        if (done[s] < 0) msg[s] = hb_last_error();       // the message lives in this thread: hand it over
    };
    if (no == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int s = 0; s < no; s++) th.emplace_back(work, s);
        for (auto &t : th) t.join();
    }
    int64_t total = 0;
    for (int s = 0; s < no; s++) {
        if (done[s] < 0) { set_error("hb_part_build: partition %d: %s", pt->owned[s], msg[s].c_str()); return done[s]; }
        total += done[s];
    }
    return total;
}

int hb_part_search_async(hb_part *pt, int slot, const void *queries, int queries_on_device, int root, int64_t nq,
                         int ef_search, int k, int64_t *out_tids, float *out_dist, int out_on_device)
{
    if (!pt || slot < 0 || slot >= PART_SLOTS || !out_tids || !out_dist || k < 1 || k > 255 || nq < 0 || root >= pt->world) {
        set_error("hb_part_search: bad argument (slot 0..%d, 1 <= k <= 255, root < world)", PART_SLOTS - 1);
        return HB_EINVAL;
    }
    if (ef_search < 1 || ef_search > 1000) { set_error("hnsw.ef_search must be in [1,1000] (got %d)", ef_search); return HB_EINVAL; }
    if (pt->world == 1) root = -1;
    const bool have_q = root < 0 || root == pt->rank;
    if (have_q && !queries && nq > 0) { set_error("hb_part_search: NULL queries"); return HB_EINVAL; }
    HB_CK(cudaSetDevice(pt->device));
    PartSlot &S = pt->slots[slot];
    int rc = slot_init(pt, S);
    if (rc) return rc;
    if (S.pending) { set_error("hb_part_search_async: slot %d still has a batch in flight", slot); return HB_ESTATE; }
    if (nq == 0) return HB_OK;
    const int no = (int) pt->owned.size();
    const size_t qbytes = (size_t) nq * pt->dim * pt->esize;
    const size_t blk = block_bytes(nq, k);
    HB_CK(S.q.ensure(qbytes));
    HB_CK(S.elem.ensure(sizeof(int32_t) * (size_t) std::max(no, 1) * nq * ef_search));
    HB_CK(S.edist.ensure(sizeof(float) * (size_t) std::max(no, 1) * nq * ef_search));
    HB_CK(S.cnt.ensure(sizeof(int32_t) * (size_t) std::max(no, 1) * nq));
    HB_CK(S.lists.ensure(blk * std::max(no, 1)));
    HB_CK(S.send.ensure(blk));
    if (pt->world > 1) {
        HB_CK(S.recv.ensure(blk * pt->world));
        HB_CK(S.out.ensure(blk));
        if (pt->exchange == 1) { rc = peer_ensure(pt, S, blk); if (rc) return rc; }
    }
    S.nq = nq; S.k = k; S.ef = ef_search; S.out_tids = out_tids; S.out_dist = out_dist; S.out_dev = out_on_device;
    S.nsub = std::min(std::max(no, 1), PART_SUBSTREAMS);
    S.tail_queued = false;
    HB_CK(cudaMemsetAsync(S.status.p, 0, sizeof(int32_t), S.s));

    // ---- the queries, on this rank's GPU
    const void *dq = nullptr;
    if (root < 0) {
        if (queries_on_device) dq = queries;
        else {
            HB_CK(cudaMemcpyAsync(S.q.p, queries, qbytes, cudaMemcpyHostToDevice, S.s));
            dq = S.q.p;
        }
        HB_CK(cudaEventRecord(S.ev_q, S.s));
    } else {
        NcclApi *nc = nccl_api();
        if (!nc) return HB_ECUDA;
        const void *src = S.q.p;
        if (root == pt->rank) {
            if (queries_on_device) src = queries;
            else HB_CK(cudaMemcpyAsync(S.q.p, queries, qbytes, cudaMemcpyHostToDevice, S.s));
        }
        HB_CK(cudaEventRecord(S.ev_q, S.s));
        HB_CK(cudaStreamWaitEvent(pt->xs, S.ev_q, 0));
        HB_NCCL(nc->Broadcast(src, S.q.p, qbytes, ncclChar, root, pt->comm, pt->xs));
        HB_CK(cudaEventRecord(S.ev_q, pt->xs));
        dq = S.q.p;
    }

    // ---- one scan per owned partition, spread over the slot's sub-streams
    for (int j = 0; j < S.nsub; j++) HB_CK(cudaStreamWaitEvent(S.sub[j], S.ev_q, 0));
    for (int i = 0; i < no; i++) {
        hb_index *ix = pt->parts[i];
        cudaStream_t t = S.sub[i % S.nsub];
        char *lst = S.lists.as<char>() + blk * i;
        int64_t *l_tids = reinterpret_cast<int64_t *>(lst);
        float *l_dist = reinterpret_cast<float *>(lst + (size_t) nq * k * sizeof(int64_t));
        if (ix->n == 0) {
            part_pad_kernel<<<(int) ((nq * k + 255) / 256), 256, 0, t>>>(lst, nq, k);
            HB_CK(cudaGetLastError());
            continue;
        }
        int32_t *elem = S.elem.as<int32_t>() + (size_t) i * nq * ef_search;
        float *edist = S.edist.as<float>() + (size_t) i * nq * ef_search;
        int32_t *cnt = S.cnt.as<int32_t>() + (size_t) i * nq;
        rc = hb_search_batch_dev(ix, dq, nq, ef_search, elem, edist, cnt, (void *) t);
        if (rc) return rc;
        rc = hb_elements_to_tids_dev(ix, elem, edist, nq, ef_search, k, l_tids, l_dist, (void *) t);
        if (rc) return rc;
        auto it = ix->stream_ws.find((void *) t);
        if (it != ix->stream_ws.end()) {
            part_status_kernel<<<1, 1, 0, t>>>(it->second->misc.as<int32_t>() + 3, S.status.as<int32_t>());
            HB_CK(cudaGetLastError());
        }
    }
    for (int j = 0; j < S.nsub; j++) HB_CK(cudaEventRecord(S.ev_sub[j], S.sub[j]));
    // the status word is cleared on S.s: scans must not fold into it before that
    S.pending = true;
    pt->issued++;

    if (root < 0) return queue_tail(pt, S);
    // Broadcast path: this batch's exchange is queued when the NEXT batch has been issued (or at its wait),
    // so that the next broadcast does not sit behind an all-gather that waits for this batch's scans.
    for (int o = 0; o < PART_SLOTS; o++) {
        PartSlot &O = pt->slots[o];
        if (o != slot && O.pending && !O.tail_queued) { rc = queue_tail(pt, O); if (rc) return rc; }
    }
    return HB_OK;
}

int hb_part_search_wait(hb_part *pt, int slot)
{
    if (!pt || slot < 0 || slot >= PART_SLOTS) { set_error("hb_part_search_wait: bad argument"); return HB_EINVAL; }
    PartSlot &S = pt->slots[slot];
    if (!S.pending) return HB_OK;
    HB_CK(cudaSetDevice(pt->device));
    if (!S.tail_queued) {
        // deferred exchanges are queued oldest first so that every rank issues the same NCCL sequence
        for (int o = 0; o < PART_SLOTS; o++) {
            PartSlot &O = pt->slots[o];
            if (o != slot && O.pending && !O.tail_queued) { const int rc = queue_tail(pt, O); if (rc) return rc; }
        }
        const int rc = queue_tail(pt, S);
        if (rc) return rc;
    }
    HB_CK(cudaStreamSynchronize(S.s));
    S.pending = false;
    if (*S.h_status & 2) {
        set_error("hb_part_search: a rank did not deliver its results within 20 s (failed rank, or the ranks' call sequences differ)");
        return HB_ECUDA;
    }
    if (*S.h_status) {
        set_error("a query has more than %d candidates tying exactly at the ef boundary", HB_TIE_LIMIT);
        return HB_ELIMIT;
    }
    return HB_OK;
}

int hb_part_search(hb_part *pt, const void *host_queries, int root, int64_t nq, int ef_search, int k, int64_t *out_tids,
                   float *out_dist)
{
    const int rc = hb_part_search_async(pt, 0, host_queries, 0, root, nq, ef_search, k, out_tids, out_dist, 0);
    if (rc) return rc;
    return hb_part_search_wait(pt, 0);
}

}   // extern "C"
