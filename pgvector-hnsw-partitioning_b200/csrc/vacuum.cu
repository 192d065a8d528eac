// vacuum.cu -- ambulkdelete's graph passes on the GPU: RepairGraph and MarkDeleted (hb_vacuum_repair).
//
// Takes the role of upstream pgvector's hnswvacuum.c RepairGraphEntryPoint / RepairGraph / RepairGraphElement /
// NeedsUpdated / MarkDeleted, of HnswFindElementNeighbors(existing = true) with its CountElement / RemoveElements
// rules, and of HnswUpdateNeighborsOnDisk(checkExisting = true) [RECALL; the reference mount has no source,
// /root/reference/README.md:1].  The first pass (RemoveHeapTids) is hb_bulk_delete (api.cu).
//
// Rules restated (oracle/hnsw_oracle.c orc_vacuum_repair is the CPU statement of the same thing):
//   * an element left without heap TIDs is "being deleted": searches still walk through it and keep it in W,
//     but it does not count towards ef, and it is removed from the result before neighbours are selected;
//   * an element needs repair when one of its neighbours is being deleted or its layer-0 list is not full;
//     its neighbours are recomputed from scratch by a search with ef_construction + 1 (it will find itself),
//     its lists are overwritten, and it is offered to each new neighbour: skipped when already listed, appended
//     when there is room, put in place of the first neighbour that is being deleted, else by the selection
//     heuristic over list + element;
//   * the entry point is repaired first (through the highest other live element) or replaced by that element
//     when it is being deleted; finally the emptied elements lose their lists and their vector.
// Elements are repaired in batches (option "vacuum_batch", default 2048; 1 = strictly one after the other, the
// graph is then identical to the sequential algorithm's): phase 1 searches and selects for the whole batch on
// the graph as it stands, phase 2 writes the new lists and the reverse links under per-target locks -- the
// relation concurrent backends have to one another.  Not on the throughput path: generic row loop, visited
// bitmaps and lists in HBM.
#include "index.h"
#include "build_kernel.cuh"

#include <algorithm>
#include <cstring>

namespace hb {

constexpr int VAC_WARPS = 4;
constexpr int VAC_GRID = 64;

struct RepairParams {
    GraphView g;                 // g.entry / g.entry_level: where the searches start (-1: no entry point)
    const int32_t *elems;        // B element ids
    const uint8_t *lev;          // B levels
    int B;
    const uint8_t *ntids;        // per element: 0 = being deleted
    int efc1;                    // ef_construction + 1
    int LS;                      // layer stride of the staging arrays (max level in the batch + 1)
    int32_t *need;               // B: 1 = new lists staged, 0 = left alone, -1 = W outgrew gcap (searched again with a larger one)
    int32_t *sel_id; float *sel_d; int32_t *sel_cnt;   // B x LS x lm0, B x LS
    // per-warp scratch in HBM
    uint32_t *gbits; int gwords;
    float *gwd; uint32_t *gwi; int gcap;
    int32_t *c_id; float *c_d; int32_t *wd_id; float *wd_d;   // gcap each per warp
    unsigned int *work;
    unsigned long long *totals;
    int32_t *nbr0; int32_t *nbru;   // writable views (phase 2)
    int32_t *locks;                  // per element
};

// HnswSearchLayer as vacuum calls it.  Precondition: w holds Lw entry candidates (sorted, unexpanded), vs their ids.
// Postcondition: w[0 .. Lw) = W nearest first (elements being deleted included).
template <typename T, int IP, int NV, int G, typename VS>
__device__ __forceinline__ int search_layer_vacuum(const GraphView &g, WList &w, VS &vs, const float *q, int ef, int lc, int lane,
                                                   QueryCounters &ctr, const uint8_t *ntids, int &Lw)
{
    const int deg = lc == 0 ? 2 * g.m : g.m;
    int wlen = 0;
    for (int base = 0; base < Lw; base += 32) {
        const int i = base + lane;
        wlen += __popc(__ballot_sync(FULL, i < Lw && ntids[w.id[i] & ID_MASK] != 0));
    }
    int low = 0;
    NoDiscard nd;
    for (;;) {
        int idx = -1;
        for (int base = low; base < w.L; base += 32) {
            const int i = base + lane;
            const unsigned b = __ballot_sync(FULL, i < w.L && !(w.id[i] & EXP_BIT));
            if (b) { idx = base + __ffs(b) - 1; break; }
        }
        if (idx < 0) break;
        const uint32_t cid = w.id[idx];
        __syncwarp();
        if (lane == 0) w.id[idx] = cid | EXP_BIT;
        __syncwarp();
        low = idx + 1;
        if (lc == 0) ctr.n_hop0++; else ctr.n_hopu++;
        const int32_t *list = lc == 0 ? g.nbr0 + (size_t) cid * deg : g.nbru + ((size_t) g.uoff[cid] + (lc - 1)) * g.m;
        for (int cb = 0; cb < deg; cb += 32) {
            const int i = cb + lane;
            const int32_t nb = i < deg ? __ldcg(list + i) : -1;
            bool isnew = false;
            if (nb >= 0) isnew = vs.insert((uint32_t) nb, false);
            const unsigned nmask = __ballot_sync(FULL, isnew);
            if (nmask == 0) continue;
            ctr.n_dist += __popc(nmask);
            const float myd = eval_candidates<T, IP, NV, G>(g, q, nb, nmask, lane);
            unsigned rem = nmask;
            while (rem) {
                const int s = __ffs(rem) - 1;
                rem &= rem - 1;
                const float ed = __shfl_sync(FULL, myd, s);
                const uint32_t eid = (uint32_t) __shfl_sync(FULL, nb, s);
                const bool always = wlen < ef;
                if (!(always || ed < w.d[Lw - 1])) continue;
                int newLw = Lw + 1;
                if (ntids[eid] != 0) {           // CountElement; wlen is never decremented
                    wlen++;
                    if (wlen > ef) newLw = Lw;
                }
                const int st = wlist_insert(w, ed, eid, newLw, lane, low, nd);
                if (st) return st;
                Lw = newLw;
            }
        }
    }
    return ST_OK;
}

// NeedsUpdated: a neighbour is being deleted, or layer 0 is not full
__device__ __forceinline__ bool needs_updated_warp(const GraphView &g, const int32_t *nbr0, const int32_t *nbru, int32_t e, int level,
                                                   const uint8_t *ntids, int lane)
{
    const int lm0 = 2 * g.m;
    bool hit = false;
    for (int lc = level; lc >= 0; lc--) {
        const int lm = lc == 0 ? lm0 : g.m;
        const int32_t *list = lc == 0 ? nbr0 + (size_t) e * lm0 : nbru + ((size_t) g.uoff[e] + (lc - 1)) * g.m;
        for (int jb = 0; jb < lm; jb += 32) {
            const int j = jb + lane;
            const int32_t nb = j < lm ? __ldcg(list + j) : -1;
            if (nb >= 0 && ntids[nb] == 0) hit = true;
        }
    }
    if (__any_sync(FULL, hit)) return true;
    return __ldcg(nbr0 + (size_t) e * lm0 + (lm0 - 1)) < 0;
}

// phase 1: NeedsUpdated, HnswFindElementNeighbors(existing = true) and SelectNeighbors per element; read-only
template <typename T, int IP>
__global__ void __launch_bounds__(VAC_WARPS * 32) repair_search_kernel(const RepairParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    const int lm0 = 2 * g.m;
    const size_t qbytes = (size_t) g.nvec * Vec<T>::VEC * 4;
    unsigned char *base = smem + ((qbytes + (size_t) lm0 * 8 + 15) & ~(size_t) 15) * warp;
    float *q = reinterpret_cast<float *>(base);
    int32_t *r_id = reinterpret_cast<int32_t *>(base + qbytes);
    float *r_d = reinterpret_cast<float *>(r_id + lm0);
    const size_t gw = (size_t) blockIdx.x * VAC_WARPS + warp;
    VisitedBitmap vs;
    vs.bits = p.gbits + gw * p.gwords;
    vs.words = p.gwords;
    WList w;
    w.d = p.gwd + gw * p.gcap;
    w.id = p.gwi + gw * p.gcap;
    w.cap = p.gcap;
    int32_t *c_id = p.c_id + gw * p.gcap;
    float *c_d = p.c_d + gw * p.gcap;
    int32_t *wd_id = p.wd_id + gw * p.gcap;
    float *wd_d = p.wd_d + gw * p.gcap;
    unsigned long long npair = 0;

    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(p.work, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= (unsigned) p.B) break;
        const int i = (int) item;
        const int32_t e = p.elems[i];
        int level = p.lev[i];
        if (lane == 0) p.need[i] = 0;
        if (e == g.entry) continue;                                             // "Skip if element is entry point"
        if (!needs_updated_warp(g, g.nbr0, g.nbru, e, level, p.ntids, lane)) continue;
        int32_t *s_cnt = p.sel_cnt + (size_t) i * p.LS;
        for (int lc = lane; lc <= level; lc += 32) s_cnt[lc] = 0;               // HnswInitNeighbors: every layer empty
        QueryCounters ctr = { 0, 0, 0 };
        int st = ST_OK;
        if (g.entry >= 0) {
            __syncwarp();
            stage_row<T>(g.vecs + (size_t) e * g.row_bytes, g.nvec, q, lane);
            __syncwarp();
            const float d0 = one_distance<T, IP, 0>(g, q, g.entry, lane);
            ctr.n_dist = 1;
            w.L = 1;
            if (lane == 0) { w.d[0] = d0; w.id[0] = (uint32_t) g.entry; }
            __syncwarp();
            int Lw = 1;
            for (int lc = g.entry_level; lc >= level + 1 && st == ST_OK; lc--) {
                st = wlist_as_entries(w, vs, Lw, lane);
                if (st == ST_OK) st = search_layer_vacuum<T, IP, 0, 2>(g, w, vs, q, 1, lc, lane, ctr, p.ntids, Lw);
            }
            if (level > g.entry_level) level = g.entry_level;
            for (int lc = level; lc >= 0 && st == ST_OK; lc--) {
                st = wlist_as_entries(w, vs, Lw, lane);
                if (st == ST_OK) st = search_layer_vacuum<T, IP, 0, 2>(g, w, vs, q, p.efc1, lc, lane, ctr, p.ntids, Lw);
                if (st != ST_OK) break;
                // RemoveElements: the element itself and elements being deleted are not candidates
                int nc = 0;
                for (int jb = 0; jb < Lw; jb += 32) {
                    const int j = jb + lane;
                    const int32_t id = j < Lw ? (int32_t) (w.id[j] & ID_MASK) : -1;
                    const bool keep = id >= 0 && id != e && p.ntids[id] != 0;
                    const unsigned km = __ballot_sync(FULL, keep);
                    if (keep) {
                        const int o = nc + __popc(km & ((1u << lane) - 1u));
                        c_id[o] = id; c_d[o] = w.d[j];
                    }
                    nc += __popc(km);
                }
                __syncwarp();
                const int lm = lc == 0 ? lm0 : g.m;
                int32_t pruned;
                const int nr = select_neighbors_warp<T, IP, 0, 2>(g, q, c_id, c_d, nc, lm, r_id, r_d, wd_id, wd_d, pruned, lane, npair);
                int32_t *oid = p.sel_id + ((size_t) i * p.LS + lc) * lm0;
                float *od = p.sel_d + ((size_t) i * p.LS + lc) * lm0;
                for (int j = lane; j < lm; j += 32) { oid[j] = j < nr ? r_id[j] : -1; od[j] = j < nr ? r_d[j] : 0.f; }
                if (lane == 0) s_cnt[lc] = nr;
                // the selection staged candidate rows over the query: put it back
                __syncwarp();
                stage_row<T>(g.vecs + (size_t) e * g.row_bytes, g.nvec, q, lane);
                __syncwarp();
            }
        }
        if (lane == 0) {
            p.need[i] = st == ST_OK ? 1 : -1;
            atomicAdd(p.totals + 0, (unsigned long long) ctr.n_dist);
            atomicAdd(p.totals + 1, (unsigned long long) ctr.n_hop0);
            atomicAdd(p.totals + 2, (unsigned long long) ctr.n_hopu);
        }
    }
    if (lane == 0 && npair) atomicAdd(p.totals + 4, npair);
}

// phase 2: overwrite the repaired elements' lists, then HnswUpdateNeighborsOnDisk(checkExisting = true)
template <typename T, int IP>
__global__ void __launch_bounds__(VAC_WARPS * 32) repair_apply_kernel(const RepairParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    const int lm0 = 2 * g.m, cap = lm0 + 1;
    const size_t qbytes = (size_t) g.nvec * Vec<T>::VEC * 4;
    unsigned char *base = smem + ((qbytes + (size_t) cap * 24 + (size_t) lm0 * 8 + 15) & ~(size_t) 15) * warp;
    float *q = reinterpret_cast<float *>(base);
    int32_t *l_id = reinterpret_cast<int32_t *>(base + qbytes);
    float *l_d = reinterpret_cast<float *>(l_id + cap);
    int32_t *s_id = reinterpret_cast<int32_t *>(l_d + cap);
    float *s_d = reinterpret_cast<float *>(s_id + cap);
    int32_t *wd_id = reinterpret_cast<int32_t *>(s_d + cap);
    float *wd_d = reinterpret_cast<float *>(wd_id + cap);
    int32_t *r_id = reinterpret_cast<int32_t *>(wd_d + cap);
    float *r_d = reinterpret_cast<float *>(r_id + lm0);
    unsigned long long npair = 0;

    for (int i = blockIdx.x * VAC_WARPS + warp; i < p.B; i += gridDim.x * VAC_WARPS) {
        if (p.need[i] != 1) continue;
        const int32_t e = p.elems[i];
        const int level = p.lev[i];
        // the element's own neighbour tuple
        for (int lc = 0; lc <= level; lc++) {
            const int lm = lc == 0 ? lm0 : g.m;
            int32_t *list = lc == 0 ? p.nbr0 + (size_t) e * lm0 : p.nbru + ((size_t) g.uoff[e] + (lc - 1)) * g.m;
            const int32_t *sid = p.sel_id + ((size_t) i * p.LS + lc) * lm0;
            const int nr = p.sel_cnt[(size_t) i * p.LS + lc];
            if (lane == 0) { while (atomicCAS(p.locks + e, 0, 1) != 0) { } __threadfence(); }
            __syncwarp();
            for (int j = lane; j < lm; j += 32) __stcg(list + j, j < nr ? sid[j] : -1);
            __syncwarp();
            if (lane == 0) { __threadfence(); atomicExch(p.locks + e, 0); }
        }
        // offer the element to each of its new neighbours, upper layers first, list order
        for (int lc = level; lc >= 0; lc--) {
            const int lm = lc == 0 ? lm0 : g.m;
            const int32_t *sid = p.sel_id + ((size_t) i * p.LS + lc) * lm0;
            const float *sd = p.sel_d + ((size_t) i * p.LS + lc) * lm0;
            const int nr = p.sel_cnt[(size_t) i * p.LS + lc];
            for (int k = 0; k < nr; k++) {
                const int32_t n = sid[k];
                const float d = sd[k];
                int32_t *gl = lc == 0 ? p.nbr0 + (size_t) n * lm0 : p.nbru + ((size_t) g.uoff[n] + (lc - 1)) * g.m;
                if (lane == 0) { while (atomicCAS(p.locks + n, 0, 1) != 0) { } __threadfence(); }
                __syncwarp();
                int cnt = 0;
                bool listed = false;
                for (int jb = 0; jb < lm; jb += 32) {
                    const int j = jb + lane;
                    int32_t v = -1;
                    if (j < lm) { v = __ldcg(gl + j); l_id[j] = v; }
                    cnt += __popc(__ballot_sync(FULL, v >= 0));
                    listed = listed || __any_sync(FULL, v == e);
                }
                __syncwarp();
                if (!listed) {
                    if (cnt < lm) {
                        if (lane == 0) __stcg(gl + cnt, e);
                    } else {
                        // distances owner -> members (recomputed, as the on-disk path does); first member being deleted goes
                        stage_row<T>(g.vecs + (size_t) n * g.row_bytes, g.nvec, q, lane);
                        __syncwarp();
                        int32_t pruned = -1;
                        for (int jb = 0; jb < lm; jb += 32) {
                            const int j = jb + lane;
                            const int32_t nb = j < lm ? l_id[j] : -1;
                            const unsigned mask = __ballot_sync(FULL, nb >= 0);
                            const float v = eval_candidates<T, IP, 0, 2>(g, q, nb, mask, lane);
                            if (j < lm) l_d[j] = v;
                            const unsigned dead = __ballot_sync(FULL, nb >= 0 && p.ntids[nb] == 0);
                            if (dead && pruned < 0) pruned = l_id[jb + __ffs(dead) - 1];
                        }
                        __syncwarp();
                        if (pruned < 0) {
                            if (lane == 0) { l_id[lm] = e; l_d[lm] = d; }
                            __syncwarp();
                            const int nc = lm + 1;
                            for (int ib = 0; ib < nc; ib += 32) {          // sortCandidates: (distance, id)
                                const int a = ib + lane;
                                if (a < nc) {
                                    const float da = l_d[a];
                                    const int32_t ia = l_id[a];
                                    int rank = 0;
                                    for (int j = 0; j < nc; j++) rank += (l_d[j] < da || (l_d[j] == da && l_id[j] < ia)) ? 1 : 0;
                                    s_id[rank] = ia; s_d[rank] = da;
                                }
                            }
                            __syncwarp();
                            select_neighbors_warp<T, IP, 0, 2>(g, q, s_id, s_d, nc, lm, r_id, r_d, wd_id, wd_d, pruned, lane, npair);
                        }
                        for (int jb = 0; jb < lm; jb += 32) {
                            const int j = jb + lane;
                            if (j < lm && l_id[j] == pruned) __stcg(gl + j, e);     // nothing happens when the element itself was pruned
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) { __threadfence(); atomicExch(p.locks + n, 0); }
                __syncwarp();
            }
        }
    }
    if (lane == 0 && npair) atomicAdd(p.totals + 4, npair);
}

// MarkDeleted: emptied elements lose their lists and their vector
__global__ void mark_deleted_kernel(const int32_t *__restrict__ elems, const uint8_t *__restrict__ lev, int B, GraphView g,
                                    int32_t *nbr0, int32_t *nbru, char *vecs)
{
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= B) return;
    const int32_t e = elems[i];
    const int lm0 = 2 * g.m;
    for (int j = lane; j < lm0; j += 32) nbr0[(size_t) e * lm0 + j] = -1;
    for (int lc = 1; lc <= lev[i]; lc++)
        for (int j = lane; j < g.m; j += 32) nbru[((size_t) g.uoff[e] + (lc - 1)) * g.m + j] = -1;
    uint4 *row = reinterpret_cast<uint4 *>(vecs + (size_t) e * g.row_bytes);
    for (int ch = lane; ch < g.nvec; ch += 32) row[ch] = make_uint4(0u, 0u, 0u, 0u);
}

template <typename T, int IP>
static int run_repair_t(hb_index *ix, RepairParams &p, cudaStream_t s)
{
    const int lm0 = 2 * ix->m, cap = lm0 + 1;
    const size_t qbytes = (size_t) ix->nvec * Vec<T>::VEC * 4;
    const size_t smem1 = ((qbytes + (size_t) lm0 * 8 + 15) & ~(size_t) 15) * VAC_WARPS;
    const size_t smem2 = ((qbytes + (size_t) cap * 24 + (size_t) lm0 * 8 + 15) & ~(size_t) 15) * VAC_WARPS;
    auto k1 = repair_search_kernel<T, IP>;
    auto k2 = repair_apply_kernel<T, IP>;
    HB_CK(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem1));
    HB_CK(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem2));
    const int grid = std::min(VAC_GRID, (p.B + VAC_WARPS - 1) / VAC_WARPS);
    k1<<<grid, VAC_WARPS * 32, smem1, s>>>(p);
    HB_CK(cudaGetLastError());
    k2<<<grid, VAC_WARPS * 32, smem2, s>>>(p);
    HB_CK(cudaGetLastError());
    return HB_OK;
}

static int run_repair(hb_index *ix, RepairParams &p, cudaStream_t s)
{
    const int kind = metric_kind(ix->metric);
    if (ix->dtype == HB_F32) return kind == 0 ? run_repair_t<float, 0>(ix, p, s) : kind == 1 ? run_repair_t<float, 1>(ix, p, s) : run_repair_t<float, 2>(ix, p, s);
    return kind == 0 ? run_repair_t<__half, 0>(ix, p, s) : kind == 1 ? run_repair_t<__half, 1>(ix, p, s) : run_repair_t<__half, 2>(ix, p, s);
}

}   // namespace hb

using namespace hb;

extern "C" int64_t hb_vacuum_repair(hb_index *ix, int64_t *repaired)
{
    if (!ix) { set_error("hb_vacuum_repair: NULL index"); return HB_EINVAL; }
    if (repaired) *repaired = 0;
    const int64_t n = ix->n;
    if (n == 0) return 0;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaDeviceSynchronize());
    cudaStream_t s = ix->stream;
    const int m = ix->m, lm0 = 2 * m;
    // what only inserts use is stale once lists change under it: cached distances, pair cache (as after hb_index_load)
    if (ix->d_nbr0d) { cudaFree(ix->d_nbr0d); ix->d_nbr0d = nullptr; }
    if (ix->d_nbrud) { cudaFree(ix->d_nbrud); ix->d_nbrud = nullptr; }
    release_pair_cache(ix);
    ix->h_deleted.resize((size_t) n, 0);

    const int bmax = ix->opt_vacuum_batch > 0 ? ix->opt_vacuum_batch : 2048;
    int max_level = 0;
    for (int64_t e = 0; e < n; e++) max_level = std::max<int>(max_level, ix->h_level[e]);
    const int LS = max_level + 1;
    const int64_t warps = (int64_t) VAC_GRID * VAC_WARPS;
    // per-warp W list: ef_construction + 1 + the tie allowance.  Emptied elements stay in W without counting towards
    // ef, so after heavy deletes a search can outgrow it; such an element is searched again alone with a larger list
    const int gcap = ix->efc + 1 + HB_TIE_LIMIT;
    const int gwords = (int) ((n + 31) / 32 + 1);
    DevBuf b_elems, b_lev, b_need, b_sel, b_scr, b_misc, b_locks, b_big;
    struct Release { DevBuf *b[8]; ~Release() { for (auto x : b) x->release(); } } rel{ { &b_elems, &b_lev, &b_need, &b_sel, &b_scr, &b_misc, &b_locks, &b_big } };
    HB_CK(b_elems.ensure(sizeof(int32_t) * (size_t) std::max<int64_t>(bmax, 1)));
    HB_CK(b_lev.ensure((size_t) bmax));
    HB_CK(b_need.ensure(sizeof(int32_t) * (size_t) bmax));
    HB_CK(b_sel.ensure((size_t) bmax * LS * lm0 * 8 + (size_t) bmax * LS * 4));
    HB_CK(b_scr.ensure((size_t) warps * ((size_t) gwords * 4 + (size_t) gcap * 24)));
    HB_CK(b_misc.ensure(64));
    HB_CK(b_locks.ensure(sizeof(int32_t) * (size_t) n));
    HB_CK(cudaMemsetAsync(b_locks.p, 0, sizeof(int32_t) * (size_t) n, s));
    HB_CK(cudaMemsetAsync(b_misc.p, 0, 64, s));

    RepairParams p;
    memset(&p, 0, sizeof p);
    p.ntids = ix->d_ntids;
    p.efc1 = ix->efc + 1;
    p.LS = LS;
    p.elems = b_elems.as<int32_t>();
    p.lev = b_lev.as<uint8_t>();
    p.need = b_need.as<int32_t>();
    p.sel_id = b_sel.as<int32_t>();
    p.sel_d = reinterpret_cast<float *>(p.sel_id + (size_t) bmax * LS * lm0);
    p.sel_cnt = reinterpret_cast<int32_t *>(p.sel_d + (size_t) bmax * LS * lm0);
    // per-warp scratch of `nw` warps with W lists of `cap` entries
    auto carve_scratch = [&](RepairParams &q, char *c, int64_t nw, int cap) {
        q.gbits = reinterpret_cast<uint32_t *>(c); c += (size_t) nw * gwords * 4;
        q.gwd = reinterpret_cast<float *>(c); c += (size_t) nw * cap * 4;
        q.gwi = reinterpret_cast<uint32_t *>(c); c += (size_t) nw * cap * 4;
        q.c_id = reinterpret_cast<int32_t *>(c); c += (size_t) nw * cap * 4;
        q.c_d = reinterpret_cast<float *>(c); c += (size_t) nw * cap * 4;
        q.wd_id = reinterpret_cast<int32_t *>(c); c += (size_t) nw * cap * 4;
        q.wd_d = reinterpret_cast<float *>(c);
        q.gwords = gwords; q.gcap = cap;
    };
    carve_scratch(p, b_scr.as<char>(), warps, gcap);
    unsigned int *misc = b_misc.as<unsigned int>();
    p.work = misc;
    p.totals = ix->d_totals;
    p.nbr0 = ix->d_nbr0; p.nbru = ix->d_nbru;
    p.locks = b_locks.as<int32_t>();

    std::vector<int32_t> h_need;
    int64_t n_repaired = 0;
    // both phases for elems[0 .. B) with the given entry point and scratch; h_need receives the phase-1 outcome
    auto launch = [&](RepairParams &q, const int32_t *elems, int B, int32_t entry, int entry_level) -> int {
        if (entry < -1 || entry >= n) { set_error("hb_vacuum_repair: entry point %d is not an element (n = %lld)", entry, (long long) n); return HB_EINVAL; }
        std::vector<uint8_t> lev(B);
        for (int i = 0; i < B; i++) lev[i] = ix->h_level[elems[i]];
        q.g = ix->view();
        q.g.entry = entry;
        q.g.entry_level = entry_level;
        q.B = B;
        HB_CK(cudaMemcpyAsync(b_elems.p, elems, sizeof(int32_t) * B, cudaMemcpyHostToDevice, s));
        HB_CK(cudaMemcpyAsync(b_lev.p, lev.data(), B, cudaMemcpyHostToDevice, s));
        HB_CK(cudaMemsetAsync(misc, 0, 4, s));
        const int rc = run_repair(ix, q, s);
        if (rc) return rc;
        h_need.resize(B);
        HB_CK(cudaMemcpyAsync(h_need.data(), b_need.p, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, s));
        HB_CK(cudaStreamSynchronize(s));
        return HB_OK;
    };
    // one batch through both phases; elements whose W outgrew gcap were left alone by phase 2 and are searched again,
    // one at a time in element order, on one CTA with W doubled until it fits (W holds distinct elements: n + 1 always does)
    auto run_batch = [&](const std::vector<int32_t> &elems, int32_t entry, int entry_level) -> int {
        const int B = (int) elems.size();
        if (B == 0) return HB_OK;
        int rc = launch(p, elems.data(), B, entry, entry_level);
        if (rc) return rc;
        std::vector<int32_t> again;
        for (int i = 0; i < B; i++) {
            if (h_need[i] > 0) n_repaired++;
            else if (h_need[i] < 0) again.push_back(elems[i]);
        }
        for (const int32_t e : again) {
            int cap = gcap;
            for (;;) {
                if (cap >= n + 1) {
                    set_error("hb_vacuum_repair: the repair search of element %d holds more than %d candidates", e, cap);
                    return HB_ELIMIT;
                }
                cap = (int) std::min<int64_t>(2 * (int64_t) cap, n + 1);
                HB_CK(b_big.ensure((size_t) VAC_WARPS * ((size_t) gwords * 4 + (size_t) cap * 24)));
                RepairParams q = p;
                carve_scratch(q, b_big.as<char>(), VAC_WARPS, cap);
                if ((rc = launch(q, &e, 1, entry, entry_level)) != 0) return rc;
                if (h_need[0] >= 0) { n_repaired += h_need[0]; break; }
            }
        }
        return HB_OK;
    };

    // RemoveHeapTids remembered the highest live element that is not the entry point (first one in page order)
    int32_t highest = -1;
    int hl = -1;
    for (int64_t e = 0; e < n; e++)
        if (ix->h_ntids[e] != 0 && e != ix->entry && ix->h_level[e] > hl) { highest = (int32_t) e; hl = ix->h_level[e]; }
    // RepairGraphEntryPoint
    int rc;
    if (highest >= 0 && (rc = run_batch({ highest }, ix->entry, ix->entry_level)) != 0) return rc;
    if (ix->entry >= 0) {
        if (ix->h_ntids[ix->entry] == 0) {
            ix->entry = highest;
            ix->entry_level = highest >= 0 ? ix->h_level[highest] : -1;
        } else if ((rc = run_batch({ ix->entry }, highest, highest >= 0 ? ix->h_level[highest] : -1)) != 0) return rc;
    }
    // RepairGraph: every live element in page order
    std::vector<int32_t> batch;
    batch.reserve(bmax);
    for (int64_t e = 0; e <= n; e++) {
        if (e < n && ix->h_ntids[e] != 0 && e != ix->entry) batch.push_back((int32_t) e);
        if ((int) batch.size() == bmax || (e == n && !batch.empty())) {
            if ((rc = run_batch(batch, ix->entry, ix->entry_level)) != 0) return rc;
            batch.clear();
        }
    }
    // MarkDeleted
    std::vector<int32_t> dead;
    for (int64_t e = 0; e < n; e++)
        if (ix->h_ntids[e] == 0 && !ix->h_deleted[e]) dead.push_back((int32_t) e);
    for (size_t lo = 0; lo < dead.size(); lo += (size_t) bmax) {
        const int B = (int) std::min<size_t>((size_t) bmax, dead.size() - lo);
        std::vector<uint8_t> lev(B);
        for (int i = 0; i < B; i++) lev[i] = ix->h_level[dead[lo + i]];
        HB_CK(cudaMemcpyAsync(b_elems.p, dead.data() + lo, sizeof(int32_t) * B, cudaMemcpyHostToDevice, s));
        HB_CK(cudaMemcpyAsync(b_lev.p, lev.data(), B, cudaMemcpyHostToDevice, s));
        mark_deleted_kernel<<<(B + 3) / 4, 128, 0, s>>>(b_elems.as<int32_t>(), b_lev.as<uint8_t>(), B, ix->view(), ix->d_nbr0, ix->d_nbru, ix->d_vecs);
        HB_CK(cudaGetLastError());
        HB_CK(cudaStreamSynchronize(s));
    }
    for (int32_t e : dead) ix->h_deleted[e] = 1;
    ix->generation++;
    if (repaired) *repaired = n_repaired;
    return (int64_t) dead.size();
}
