// scan_kernel.cuh -- batched hnswgettuple: many queries' GetScanItems run concurrently, one
// warp per query, persistent CTAs pulling queries from a device work counter.
//
// Takes the role of hnswscan.c GetScanItems (entry point -> greedy descent with ef = 1 on layers
// entry_level..1 -> HnswSearchLayer with ef = hnsw.ef_search on layer 0) [RECALL; reference
// mount empty, /root/reference/README.md:1].
#pragma once
#include "search_core.cuh"
#include <cuda_runtime.h>
#include <type_traits>

namespace hb {

constexpr int SCAN_WARPS = 4;   // warps (= concurrent queries) per CTA
constexpr int MAX_CTAS_PER_SM = 12;   // cap on resident CTAs per SM (sizes the per-warp overflow tables)

// hb_set_option("variant"): the scan path forced for tests, so that every production kernel can be checked against
// the others on any shape.  All of them give identical results.
enum ScanVariant {
    SCAN_AUTO = 0,
    SCAN_NO_CTA = 6,            // never the CTA-per-query kernels of small batches (scan_cta.cuh)
    SCAN_CTA = 7,               // the CTA-per-query kernels for every row length, in the form the shape selects
    SCAN_SMEM_LIST = 9,         // the shared-memory-list warp kernel instead of the register-list one, no CTA kernels
    SCAN_CTA_SMEM_LIST = 17,    // as SCAN_CTA, with the list in shared memory
    SCAN_CTA_NO_STAGE = 27,     // as SCAN_CTA, the register list without row staging
};
inline bool is_scan_variant(int v)
{
    return v == SCAN_AUTO || v == SCAN_NO_CTA || v == SCAN_CTA || v == SCAN_SMEM_LIST || v == SCAN_CTA_SMEM_LIST ||
           v == SCAN_CTA_NO_STAGE;
}

struct ScanParams {
    GraphView g;
    const void *queries;       // nq x dim, index dtype, already normalised when cosine
    int64_t nq;
    const int32_t *qlist;      // slow path: work item -> query index
    const int32_t *qcount;     // slow path: number of work items (device)
    int ef, slots, upper_slots, capW;
    int32_t *out_elem;         // nq x out_stride
    float *out_dist;
    int32_t *out_cnt;
    int out_stride;
    int32_t *status;           // nq
    int32_t *slow_list;        // fast path appends queries whose visited table / tie tail overflowed
    int32_t *slow_count;
    int32_t *err;              // set to 1 when a query could not be completed (tie tail beyond HB_TIE_LIMIT)
    int32_t *per_query;        // optional nq x 4: n_dist, n_hop0, n_hopu, path
    unsigned long long *totals;   // n_dist, n_hop0, n_hopu, n_slow
    unsigned int *work;
    // slow-path scratch in HBM, one slice per resident warp
    uint32_t *ovf; int oslots;    // fast path: per-warp visited overflow table in HBM
    uint32_t *gbits; int gwords;
    float *gwd; uint32_t *gwi; int gcap;
    // single-layer mode (unit tests): explicit entry points
    const int32_t *ep; int nep; int layer;
    int variant;               // host only: the forced scan path (ScanVariant)
};

template <typename T> __host__ __device__ inline size_t scan_warp_smem(int nvec, int capW, int slots, bool slow)
{
    size_t b = (size_t) nvec * Vec<T>::VEC * 4;
    if (!slow) b += (size_t) capW * 8 + (size_t) slots * 4;
    return (b + 15) & ~(size_t) 15;
}

// SCAN_WARPS warps (= concurrent queries) per CTA: with rows of several kB one-warp CTAs measured 12 % slower
// (3.56 vs 4.05 M queries/s at 1M x 768 in the same run), while the register-list kernel for short rows gains 5-9 % from
// them (profiles/r2_experiments.md).
template <typename T, int IP, int NV, int G, bool SLOW, int MINB>
__global__ void __launch_bounds__(SCAN_WARPS * 32, MINB) scan_kernel(const ScanParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    const size_t wbytes = scan_warp_smem<T>(g.nvec, p.capW, p.slots, SLOW);
    unsigned char *base = smem + wbytes * warp;
    float *q = reinterpret_cast<float *>(base);

    using VS = typename std::conditional<SLOW, VisitedBitmap, VisitedHash>::type;
    WList w;
    VS vs;
    if constexpr (SLOW) {
        const size_t gw = (size_t) blockIdx.x * SCAN_WARPS + warp;
        vs.bits = p.gbits + gw * p.gwords;
        vs.words = p.gwords;
        w.d = p.gwd + gw * p.gcap;
        w.id = p.gwi + gw * p.gcap;
        w.cap = p.gcap;
    } else {
        unsigned char *s = base + (size_t) g.nvec * Vec<T>::VEC * 4;
        vs.tab = reinterpret_cast<uint32_t *>(s);
        vs.set_overflow(p.ovf + ((size_t) blockIdx.x * SCAN_WARPS + warp) * p.oslots, p.oslots);
        w.d = reinterpret_cast<float *>(s + (size_t) p.slots * 4);
        w.id = reinterpret_cast<uint32_t *>(s + (size_t) p.slots * 4 + (size_t) p.capW * 4);
        w.cap = p.capW;
    }

    const unsigned total = p.qlist ? (unsigned) *p.qcount : (unsigned) p.nq;
    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(p.work, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= total) break;
        const int64_t qi = p.qlist ? p.qlist[item] : (int64_t) item;

        __syncwarp();
        stage_query<T>(reinterpret_cast<const T *>(p.queries) + qi * g.dim, g.dim, g.nvec, q, lane);
        __syncwarp();

        QueryCounters ctr = { 0, 0, 0 };
        int st = ST_OK;
        int ef = p.ef;
        w.L = 0;
        if (p.ep == nullptr) {
            if (g.entry >= 0) {
                const float d0 = one_distance<T, IP, NV>(g, q, g.entry, lane);
                ctr.n_dist = 1;
                if (lane == 0) { w.d[0] = d0; w.id[0] = (uint32_t) g.entry; }
                w.L = 1;
                __syncwarp();
                vs.configure(p.upper_slots);
                for (int lc = g.entry_level; lc >= 1 && st == ST_OK; lc--) {
                    st = wlist_as_entries(w, vs, 1, lane);
                    if (st == ST_OK) st = search_layer<T, IP, NV, G>(g, w, vs, q, 1, lc, lane, ctr);
                }
                if (st == ST_OK) {
                    vs.configure(p.slots);
                    st = wlist_as_entries(w, vs, 1, lane);
                    if (st == ST_OK) st = search_layer<T, IP, NV, G>(g, w, vs, q, ef, 0, lane, ctr);
                }
            }
        } else {
            // one HnswSearchLayer call from explicit entry points (nep <= ef)
            int low = 0;
            for (int i = 0; i < p.nep && st == ST_OK; i++) {
                const int32_t e = p.ep[qi * p.nep + i];
                const float d = one_distance<T, IP, NV>(g, q, e, lane);
                ctr.n_dist++;
                st = wlist_insert(w, d, (uint32_t) e, p.nep > ef ? p.nep : ef, lane, low);
            }
            if (st == ST_OK) {
                vs.configure(p.layer == 0 ? p.slots : p.upper_slots);
                st = wlist_as_entries(w, vs, w.L, lane);
                if (st == ST_OK) st = search_layer<T, IP, NV, G>(g, w, vs, q, ef, p.layer, lane, ctr);
            }
        }

        if (st != ST_OK && !SLOW) {
            // hand the query to the large-visited-set path; nothing is written for it here
            if (lane == 0) {
                const int slot = atomicAdd(p.slow_count, 1);
                p.slow_list[slot] = (int32_t) qi;
                p.status[qi] = st;
            }
            continue;
        }
        const int cnt = st == ST_OK ? min(w.L, ef) : 0;
        for (int j = lane; j < p.out_stride; j += 32) {
            p.out_elem[qi * p.out_stride + j] = j < cnt ? (int32_t) (w.id[j] & ID_MASK) : -1;
            p.out_dist[qi * p.out_stride + j] = j < cnt ? w.d[j] : __int_as_float(0x7f800000);
        }
        if (lane == 0) {
            p.out_cnt[qi] = cnt;
            p.status[qi] = st == ST_OK ? 0 : -st;
            if (st != ST_OK) atomicExch(p.err, 1);
            atomicAdd(p.totals + 0, (unsigned long long) ctr.n_dist);
            atomicAdd(p.totals + 1, (unsigned long long) ctr.n_hop0);
            atomicAdd(p.totals + 2, (unsigned long long) ctr.n_hopu);
            if (SLOW) atomicAdd(p.totals + 3, 1ull);
            if (p.per_query) {
                p.per_query[qi * 4 + 0] = ctr.n_dist;
                p.per_query[qi * 4 + 1] = ctr.n_hop0;
                p.per_query[qi * 4 + 2] = ctr.n_hopu;
                p.per_query[qi * 4 + 3] = SLOW ? 1 : 0;
            }
        }
    }
}

// host-side launch helper -------------------------------------------------------------------
struct ScanLaunchInfo { int grid; size_t smem; int blocks_per_sm; };

// Persistent CTAs of WARPS warps that pull queries from p.work: as many CTAs as are resident, no more than `want` and,
// when max_grid > 0, no more than max_grid.  The kernel is a template argument so that each kernel caches its own
// occupancy.
template <void (*KERN)(ScanParams), int WARPS>
cudaError_t launch_persistent(const ScanParams &p, size_t smem, int64_t want, int num_sms, int max_grid, cudaStream_t stream,
                              ScanLaunchInfo *info)
{
    // the function attribute and the occupancy query cost several microseconds each: remember them per
    // device for the shared-memory size last used (a single scan is only ~350 us long); per host thread,
    // so that handles driven from different threads never share mutable state
    static thread_local size_t seen_smem[16];
    static thread_local int seen_bps[16];
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 15;
    int bps = 0;
    if (seen_bps[dev] > 0 && seen_smem[dev] == smem) bps = seen_bps[dev];
    else {
        cudaError_t e = cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, KERN, WARPS * 32, smem);
        if (e != cudaSuccess) return e;
        if (bps < 1) return cudaErrorInvalidConfiguration;
        seen_smem[dev] = smem; seen_bps[dev] = bps;
    }
    if (bps * WARPS > MAX_CTAS_PER_SM * SCAN_WARPS) bps = MAX_CTAS_PER_SM * SCAN_WARPS / WARPS;     // the overflow tables are sized for this many warps
    int grid = (int) (want < (int64_t) bps * num_sms ? want : (int64_t) bps * num_sms);
    if (max_grid > 0 && grid > max_grid) grid = max_grid;
    if (grid < 1) grid = 1;
    if (info) { info->grid = grid; info->smem = smem; info->blocks_per_sm = bps; }
    KERN<<<grid, WARPS * 32, smem, stream>>>(p);
    return cudaGetLastError();
}

// pick the chunks-per-lane specialisation: rows of exactly 32*NV 16-byte chunks get the unrolled
// kernels (NV, rows in flight G, min CTAs per SM); any other row length runs the generic loop.
#define HB_NV_TABLE(X) X(1, 8, 6) X(2, 8, 4) X(3, 4, 4) X(4, 4, 4) X(6, 4, 4) X(8, 2, 4)
inline int nv_of(int nvec)
{
    if (nvec % 32) return 0;
    const int nv = nvec / 32;
    return (nv == 1 || nv == 2 || nv == 3 || nv == 4 || nv == 6 || nv == 8) ? nv : 0;
}

template <typename T, int IP, bool SLOW>
cudaError_t launch_scan_t(const ScanParams &p, int num_sms, int max_grid, cudaStream_t stream,
                          ScanLaunchInfo *info)
{
    const size_t smem = scan_warp_smem<T>(p.g.nvec, p.capW, p.slots, SLOW) * SCAN_WARPS;
    const int64_t want = SLOW ? max_grid : (p.nq + SCAN_WARPS - 1) / SCAN_WARPS;
#define HB_LAUNCH(NVV, GG, MB) launch_persistent<scan_kernel<T, IP, NVV, GG, SLOW, MB>, SCAN_WARPS>(p, smem, want, num_sms, max_grid, stream, info)
    if constexpr (SLOW) return HB_LAUNCH(0, 2, 1);
    else {
        switch (nv_of(p.g.nvec)) {
#define HB_CASE(NVV, GG, MB) case NVV: return HB_LAUNCH(NVV, GG, MB);
            HB_NV_TABLE(HB_CASE)
#undef HB_CASE
        default: return HB_LAUNCH(0, 2, 4);
        }
    }
#undef HB_LAUNCH
}

// ---- the query-vs-neighbour-list distance kernel on its own (opclass FUNCTION 1, batched) ----
struct DistBatchParams {
    GraphView g;
    const void *queries;   // nq x dim, index dtype (normalised when cosine)
    int64_t nq;
    const int32_t *cand;   // nq x nc element ids (< 0 or >= n: +inf)
    int nc;
    float *out;            // nq x nc
};

template <typename T, int IP, int NV, int G>
__global__ void __launch_bounds__(SCAN_WARPS * 32) dist_batch_kernel(const DistBatchParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    float *q = reinterpret_cast<float *>(smem + scan_warp_smem<T>(g.nvec, 0, 0, true) * warp);
    const int chunks = (p.nc + 31) / 32;
    const int64_t items = p.nq * chunks;
    for (int64_t item = (int64_t) blockIdx.x * SCAN_WARPS + warp; item < items; item += (int64_t) gridDim.x * SCAN_WARPS) {
        const int64_t qi = item / chunks;
        const int c = (int) (item % chunks) * 32 + lane;
        __syncwarp();
        stage_query<T>(reinterpret_cast<const T *>(p.queries) + qi * g.dim, g.dim, g.nvec, q, lane);
        __syncwarp();
        const int32_t nb = c < p.nc ? p.cand[qi * p.nc + c] : -1;
        const unsigned mask = __ballot_sync(FULL, nb >= 0 && nb < g.n);
        const float d = eval_candidates<T, IP, NV, G>(g, q, nb, mask, lane);
        if (c < p.nc) p.out[qi * p.nc + c] = d;
    }
}

template <typename T, int IP>
cudaError_t launch_dist_t(const DistBatchParams &p, cudaStream_t stream)
{
    const size_t smem = scan_warp_smem<T>(p.g.nvec, 0, 0, true) * SCAN_WARPS;
    const int64_t items = p.nq * ((p.nc + 31) / 32);
    int64_t grid = (items + SCAN_WARPS - 1) / SCAN_WARPS;
    if (grid > 148 * 16) grid = 148 * 16;
    if (grid < 1) grid = 1;
    cudaError_t e = cudaSuccess;
#define HB_DCASE(NVV, GG)                                                                          \
    {                                                                                              \
        auto kern = dist_batch_kernel<T, IP, NVV, GG>;                                             \
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);   \
        if (e == cudaSuccess) {                                                                    \
            kern<<<(int) grid, SCAN_WARPS * 32, smem, stream>>>(p);                                \
            e = cudaGetLastError();                                                                \
        }                                                                                          \
    }
    switch (nv_of(p.g.nvec)) {
    case 1: HB_DCASE(1, 8) break;
    case 2: HB_DCASE(2, 8) break;
    case 3: HB_DCASE(3, 4) break;
    case 4: HB_DCASE(4, 4) break;
    case 6: HB_DCASE(6, 4) break;
    case 8: HB_DCASE(8, 2) break;
    default: HB_DCASE(0, 2) break;
    }
#undef HB_DCASE
    return e;
}

}   // namespace hb
