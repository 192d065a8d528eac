// index.h -- internal definition of the hb_index / hb_scan handles (host side).
#pragma once
#include "../../include/hnsw_b200.h"
#include "search_core.cuh"
#include <cuda_runtime.h>
#include <map>
#include <string>
#include <vector>

namespace hb {

void set_error(const char *fmt, ...);

#define HB_CK(call)                                                                              \
    do {                                                                                         \
        cudaError_t e__ = (call);                                                                \
        if (e__ != cudaSuccess) {                                                                \
            hb::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return HB_ECUDA;                                                                     \
        }                                                                                        \
    } while (0)

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

// everything one in-flight scan batch needs; one per user stream (device API) or per async slot
struct ScanWs {
    cudaStream_t own_stream = nullptr;      // slots of the host API own a stream
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    DevBuf q, qn, elem, dist, cnt, status, slow, misc, pq, tids, tdist, gbits, gwd, gwi, ep, ovf;
    bool timing_valid = false;
    // pending asynchronous host-API call
    int64_t pending_nq = 0;
    bool pending = false;
    int32_t *h_err = nullptr;               // pinned: error flag of the last batch
    char *h_pin = nullptr;                  // pinned staging of small host-API calls (query in, results out)
    size_t h_pin_cap = 0;
    DevBuf pack;                            // small calls: elem | dist | cnt contiguous, one D2H
    void release()
    {
        if (h_err) cudaFreeHost(h_err);
        if (h_pin) cudaFreeHost(h_pin);
        pack.release();
        DevBuf *b[] = { &q, &qn, &elem, &dist, &cnt, &status, &slow, &misc, &pq, &tids, &tdist, &gbits, &gwd, &gwi, &ep, &ovf };
        for (auto x : b) x->release();
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (own_stream) cudaStreamDestroy(own_stream);
    }
};
constexpr int ASYNC_SLOTS = 4;

}   // namespace hb

struct hb_index {
    int device = 0, dim = 0, m = 0, efc = 0, metric = 0, dtype = 0;
    int esize = 4, nvec = 0, num_sms = 148;
    size_t row_bytes = 0;
    int64_t cap = 0, n = 0, seq = 0;
    uint64_t seed = 0;
    int64_t upper_rows = 0, upper_cap = 0;
    int32_t entry = -1;
    int entry_level = -1;
    bool has_dups = false;
    uint64_t generation = 1;       // bumped by every mutation of the graph image (load, insert, delete, repair)
    void *bf = nullptr;            // exact-scan state (bruteforce.cu BfState), owned by the handle

    // graph image in HBM
    char *d_vecs = nullptr;
    int32_t *d_nbr0 = nullptr;
    float *d_nbr0d = nullptr;      // cached owner->neighbour distances (build only)
    int32_t *d_uoff = nullptr;
    int32_t *d_nbru = nullptr;
    float *d_nbrud = nullptr;
    // pair cache of the link phase (build only): distances among each list's members, strict lower
    // triangle by slot, + filled flag; absent when it would not fit (opt_pair_cache 0 disables)
    float *d_pc0 = nullptr, *d_pcu = nullptr;
    uint8_t *d_pv0 = nullptr, *d_pvu = nullptr;
    bool pair_cache_tried = false;
    int64_t *d_tid0 = nullptr;     // first heap TID of each element
    uint8_t *d_ntids = nullptr;
    int64_t *d_tidx = nullptr;     // remaining HB_HEAPTIDS-1 TIDs, allocated when duplicates exist

    // host mirrors of the small per-element state
    std::vector<uint8_t> h_level, h_ntids;
    std::vector<int64_t> h_tids;   // n x HB_HEAPTIDS
    std::vector<uint8_t> h_deleted;   // HnswElementTupleData.deleted: set by hb_vacuum_repair's MarkDeleted (may be shorter than n)

    // tuning knobs (0 = automatic)
    int opt_slots = 0, opt_grid = 0, opt_build_batch = 0, opt_per_query = 0;
    int opt_variant = 0;           // the scan path forced for tests (ScanVariant, scan_kernel.cuh)
    int opt_pair_cache = 1, opt_pair_fill = 1, opt_eval_table = 1;
    int opt_auto_grow = 1;         // inserts beyond the capacity grow the index (hb_index_reserve) instead of failing
    int opt_build_fraction = 16;   // a batch is at most 1/opt_build_fraction of the graph
    int opt_build_fraction_small = 0;    // the same while the graph holds fewer than 65536 elements (the latency-bound start-up); 0 = automatic
    int opt_vacuum_batch = 0;      // elements repaired concurrently by hb_vacuum_repair (0 = 2048, 1 = one after the other)
    int opt_link_kernel = 0;       // 0 automatic, 1 warp-per-segment, 2 CTA-per-segment (link_kernel.cuh)

    // workspaces
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    hb::DevBuf ws_q, ws_qn, ws_elem, ws_dist, ws_status, ws_misc;   // opclass support functions, build
    hb::DevBuf ws_gbits, ws_gwd, ws_gwi, ws_ovf;                    // build-search scratch
    hb::ScanWs *slot_ws[hb::ASYNC_SLOTS] = { nullptr, nullptr, nullptr, nullptr };
    std::map<void *, hb::ScanWs *> stream_ws;                       // device API: one workspace per user stream
    hb::ScanWs *last_ws = nullptr;
    hb::DevBuf ws_build[12];
    int32_t *h_flag = nullptr;                // pinned: per-batch flag word of the build pipeline
    cudaStream_t up_stream = nullptr;         // build: rows are uploaded ahead of the batch that indexes them
    cudaEvent_t up_event = nullptr;
    unsigned long long *d_totals = nullptr;   // n_dist, n_hop0, n_hopu, n_slow, n_pair, ...
    hb_counters host_totals = {0, 0, 0, 0, 0};
    bool timing_valid = false;

    hb::GraphView view() const
    {
        hb::GraphView g;
        g.vecs = d_vecs; g.row_bytes = row_bytes; g.dim = dim; g.nvec = nvec;
        g.nbr0 = d_nbr0; g.uoff = d_uoff; g.nbru = d_nbru; g.m = m;
        g.entry = entry; g.entry_level = entry_level; g.n = n;
        return g;
    }
};

struct hb_iter;
struct hb_scan {
    hb_index *ix = nullptr;
    int iter_mode = 0;              // hnsw.iterative_scan: HB_ITER_*
    int64_t max_scan_tuples = 20000;
    hb_iter *iter = nullptr;
    float prev_dist = 0.f;
    bool have_prev = false;
    std::vector<char> query;
    int ef = 0;
    bool bound = false, fetched = false;
    std::vector<int32_t> elem;
    std::vector<float> dist;
    int cnt = 0, pos = 0, tid_pos = -1;
};

namespace hb {
// implemented per (dtype, metric) translation unit
struct ScanParams;
struct ScanLaunchInfo;
typedef cudaError_t (*scan_launch_fn)(const ScanParams &, int num_sms, int max_grid, cudaStream_t, ScanLaunchInfo *);
// kind: 0 = squared L2, 1 = negative inner product (and cosine), 2 = L1 (metric_kind())
scan_launch_fn get_scan_launcher(int dtype, int kind, bool slow);
// register-list scan (scan_reg.cuh): R = registers per lane and field holding the W list
typedef cudaError_t (*scan_reg_launch_fn)(const ScanParams &, int R, int num_sms, int max_grid, cudaStream_t, ScanLaunchInfo *);
scan_reg_launch_fn get_scan_reg_launcher(int dtype, int kind);
// CTA-per-query scan for small batches (scan_cta.cuh)
typedef cudaError_t (*scan_cta_launch_fn)(const ScanParams &, int num_sms, cudaStream_t);
scan_cta_launch_fn get_scan_cta_launcher(int dtype, int kind);

struct DistBatchParams;
typedef cudaError_t (*dist_launch_fn)(const DistBatchParams &, cudaStream_t);
dist_launch_fn get_dist_launcher(int dtype, int kind);
inline int metric_kind(int metric) { return metric == HB_L2 ? 0 : (metric == HB_L1 ? 2 : 1); }

// api.cu: canonical l2_normalize of n rows resident in HBM
int normalize_dev(hb_index *ix, const void *dev_in, int64_t n, void *dev_out, cudaStream_t s);
// bruteforce.cu
void bruteforce_release(hb_index *ix);
// build.cu
int64_t build_insert(hb_index *ix, const void *host_vecs, int64_t n, const int64_t *heap_tids);
void release_pair_cache(hb_index *ix);
int level_for(uint64_t seed, int64_t seq, int m);
uint64_t splitmix64(uint64_t x);
}   // namespace hb
