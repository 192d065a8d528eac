// build_kernel.cuh -- the index-build hot path, batched.
//
// Roles [RECALL; the reference mount has no source, /root/reference/README.md:1]:
//   build_search_kernel   <- hnswutils.c HnswFindElementNeighbors: greedy descent, then per layer
//                            HnswSearchLayer(ef_construction) and -- fused, on the W just produced --
//                            SelectNeighbors + CheckElementCloser (heuristic with pruned back-fill) and
//                            hnswbuild.c FindDuplicateInMemory, for a whole batch of new elements against
//                            the graph as it stood before the batch
//   build_commit_kernel   <- hnswutils.c AddConnections (build.cu)
//   link_memo_kernel /    <- hnswutils.c HnswUpdateConnection (reverse links; re-selection when the
//   link_pipe_kernel /       neighbour's list is full), one warp or CTA per (target, layer), edges
//   link_warp_kernel         applied in source-id order (link_kernel.cuh describes the three)
// A batch is what pgvector's parallel build workers are to each other: elements inserted
// concurrently do not see one another.
#pragma once
#include "scan_kernel.cuh"
#include "link_kernel.cuh"
#include <cuda_runtime.h>

namespace hb {

constexpr int BUILD_WARPS = 4;
#ifndef HB_MEMO_COLD_GENERIC
#define HB_MEMO_COLD_GENERIC 0     // link_memo_kernel: rarely taken distance evaluations use the run-time chunk loop (code size)
#endif
constexpr int DUP_SLOTS = 8;

struct BuildSearchParams {
    GraphView g;                 // the graph before the batch
    int64_t first;               // new element i lives in row first + i
    int B;
    const uint8_t *level;        // B
    const int32_t *ucand_row;    // B: first upper candidate row of element i (layers 1..), or -1
    int efc, slots, upper_slots, capW;
    int32_t *status, *slow_list, *slow_count;
    const int32_t *qlist, *qcount;
    unsigned long long *totals;
    unsigned int *work;
    uint32_t *ovf; int oslots;    // fast path: per-warp visited overflow table in HBM
    uint32_t *gbits; int gwords;
    float *gwd; uint32_t *gwi; int gcap;
    // SelectNeighbors runs on each layer's W as soon as that layer's search is done -- the selection
    // work of finished elements fills the tail of the batch's search -- so the candidate lists are
    // never written out
    int32_t *sel0_id; float *sel0_d; int32_t *sel0_cnt;     // B x 2m
    int32_t *selu_id; float *selu_d; int32_t *selu_cnt;     // UR x m
    int32_t *dup;                                           // B x DUP_SLOTS: leading byte-identical neighbours
    // evaluated-distance logs (search_core.cuh EvalLog), B x el_cap entries each + B counts; NULL = not kept
    uint32_t *el_id; float *el_d; int32_t *el_n; int el_cap;
};

template <typename T> __host__ __device__ inline size_t build_warp_smem(int nvec, int capW, int slots, bool slow)
{
    size_t b = (size_t) nvec * Vec<T>::VEC * 4;
    if (!slow) b += (size_t) capW * 8 + (size_t) slots * 4;
    return (b + 15) & ~(size_t) 15;
}

// per warp: build_warp_smem + the selection's scratch (candidate ids, pruned list, selected list)
template <typename T> __host__ __device__ inline size_t bsearch_warp_smem(int nvec, int capW, int slots, bool slow, int efc, int lm0)
{
    return build_warp_smem<T>(nvec, capW, slots, slow) + (((size_t) efc * 12 + (size_t) lm0 * 8 + 15) & ~(size_t) 15);
}

template <typename T, int IP, int NV, int G>
__device__ __forceinline__ int select_neighbors_warp(const GraphView &g, float *q, const int32_t *cand_id,
                                                     const float *cand_d, int nc, int lm, int32_t *r_id, float *r_d,
                                                     int32_t *wd_id, float *wd_d, int32_t &pruned, int lane,
                                                     unsigned long long &npair);

template <typename T, int IP, int NV, int G, bool SLOW>
__global__ void __launch_bounds__(BUILD_WARPS * 32, (NV == 1 ? 6 : 4)) build_search_kernel(const BuildSearchParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    const int lm0 = 2 * g.m;
    const size_t wbytes = bsearch_warp_smem<T>(g.nvec, p.capW, p.slots, SLOW, p.efc, lm0);
    unsigned char *base = smem + wbytes * warp;
    float *q = reinterpret_cast<float *>(base);
    int32_t *c_id = reinterpret_cast<int32_t *>(base + build_warp_smem<T>(g.nvec, p.capW, p.slots, SLOW));
    int32_t *wd_id = c_id + p.efc;
    float *wd_d = reinterpret_cast<float *>(wd_id + p.efc);
    int32_t *r_id = reinterpret_cast<int32_t *>(wd_d + p.efc);
    float *r_d = reinterpret_cast<float *>(r_id + lm0);
    unsigned long long npair = 0;
    using VS = typename std::conditional<SLOW, VisitedBitmap, VisitedHash>::type;
    WList w;
    VS vs;
    if constexpr (SLOW) {
        const size_t gw = (size_t) blockIdx.x * BUILD_WARPS + warp;
        vs.bits = p.gbits + gw * p.gwords;
        vs.words = p.gwords;
        w.d = p.gwd + gw * p.gcap;
        w.id = p.gwi + gw * p.gcap;
        w.cap = p.gcap;
    } else {
        unsigned char *s = base + (size_t) g.nvec * Vec<T>::VEC * 4;
        vs.tab = reinterpret_cast<uint32_t *>(s);
        vs.set_overflow(p.ovf + ((size_t) blockIdx.x * BUILD_WARPS + warp) * p.oslots, p.oslots);
        w.d = reinterpret_cast<float *>(s + (size_t) p.slots * 4);
        w.id = reinterpret_cast<uint32_t *>(s + (size_t) p.slots * 4 + (size_t) p.capW * 4);
        w.cap = p.capW;
    }
    const unsigned total = p.qlist ? (unsigned) *p.qcount : (unsigned) p.B;
    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(p.work, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= total) break;
        const int i = p.qlist ? p.qlist[item] : (int) item;
        __syncwarp();
        stage_row<T>(g.vecs + (size_t) (p.first + i) * g.row_bytes, g.nvec, q, lane);
        __syncwarp();

        QueryCounters ctr = { 0, 0, 0 };
        unsigned long long np_e = 0;      // pairs of this element's selections; counted once it completes
        int st = ST_OK;
        int level = p.level[i];
        const float d0 = one_distance<T, IP, NV>(g, q, g.entry, lane);
        ctr.n_dist = 1;
        w.L = 1;
        if (lane == 0) { w.d[0] = d0; w.id[0] = (uint32_t) g.entry; }
        __syncwarp();
        // 1st phase: greedy search to the insert level
        vs.configure(p.upper_slots);
        for (int lc = g.entry_level; lc >= level + 1 && st == ST_OK; lc--) {
            st = wlist_as_entries(w, vs, 1, lane);
            if (st == ST_OK) st = search_layer<T, IP, NV, G>(g, w, vs, q, 1, lc, lane, ctr);
        }
        if (level > g.entry_level) level = g.entry_level;
        // 2nd phase: ef_construction candidates per layer; the whole result is the next entry list
        vs.configure(p.slots);
        int keep = 1;
        EvalLog el;
        el.id = p.el_id ? p.el_id + (size_t) i * p.el_cap : nullptr;
        el.d = p.el_d ? p.el_d + (size_t) i * p.el_cap : nullptr;
        el.n = 0; el.cap = p.el_cap;
        for (int lc = level; lc >= 0 && st == ST_OK; lc--) {
            st = wlist_as_entries(w, vs, keep, lane);
            if (st != ST_OK) break;
            if (el.id) {
                NoDiscard nd;
                st = search_layer<T, IP, NV, G, VS, NoDiscard, EvalLog>(g, w, vs, q, p.efc, lc, lane, ctr, nd, el);
            } else st = search_layer<T, IP, NV, G>(g, w, vs, q, p.efc, lc, lane, ctr);
            if (st != ST_OK) break;
            keep = p.efc;
            const int cnt = min(w.L, p.efc);
            // SelectNeighbors on this layer's candidates (W is only read: it is the next layer's entry list)
            const int lm = lc == 0 ? lm0 : g.m;
            const size_t row = lc == 0 ? (size_t) i : (size_t) p.ucand_row[i] + (lc - 1);
            __syncwarp();
            for (int j = lane; j < cnt; j += 32) c_id[j] = (int32_t) (w.id[j] & ID_MASK);
            __syncwarp();
            int32_t pruned;
            const int nr = select_neighbors_warp<T, IP, NV, (G > 4 ? 4 : G)>(g, q, c_id, w.d, cnt, lm, r_id, r_d, wd_id, wd_d, pruned,
                                                                            lane, np_e);
            int32_t *oid = (lc == 0 ? p.sel0_id : p.selu_id) + row * lm;
            float *od = (lc == 0 ? p.sel0_d : p.selu_d) + row * lm;
            for (int j = lane; j < lm; j += 32) { oid[j] = j < nr ? r_id[j] : -1; od[j] = j < nr ? r_d[j] : 0.f; }
            if (lane == 0) (lc == 0 ? p.sel0_cnt : p.selu_cnt)[row] = nr;
            if (lc == 0) {
                // FindDuplicateInMemory: neighbours in stored order while byte-identical to the new row
                const uint4 *mine = reinterpret_cast<const uint4 *>(g.vecs + (size_t) (p.first + i) * g.row_bytes);
                int nd = 0;
                for (int j = 0; j < nr && nd < DUP_SLOTS; j++) {
                    const uint4 *other = reinterpret_cast<const uint4 *>(g.vecs + (size_t) r_id[j] * g.row_bytes);
                    bool same = true;
                    for (int ch = lane; ch < g.nvec; ch += 32) {
                        const uint4 a = mine[ch], b = other[ch];
                        same = same && a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w;
                    }
                    if (!__all_sync(FULL, same)) break;
                    if (lane == 0) p.dup[(size_t) i * DUP_SLOTS + nd] = r_id[j];
                    nd++;
                }
                if (lane == 0 && nd < DUP_SLOTS) p.dup[(size_t) i * DUP_SLOTS + nd] = -1;
            } else {
                // the selection staged candidate rows over the query: put the query back for the next layer
                __syncwarp();
                stage_row<T>(g.vecs + (size_t) (p.first + i) * g.row_bytes, g.nvec, q, lane);
                __syncwarp();
            }
        }
        if (st != ST_OK && !SLOW) {
            if (lane == 0) {
                const int slot = atomicAdd(p.slow_count, 1);
                p.slow_list[slot] = i;
                p.status[i] = st;
            }
            continue;
        }
        npair += np_e;
        if (lane == 0) {
            if (p.el_n) p.el_n[i] = st == ST_OK ? min(el.n, el.cap) : 0;
            p.status[i] = st == ST_OK ? 0 : -st;
            atomicAdd(p.totals + 0, (unsigned long long) ctr.n_dist);
            atomicAdd(p.totals + 1, (unsigned long long) ctr.n_hop0);
            atomicAdd(p.totals + 2, (unsigned long long) ctr.n_hopu);
            if (SLOW) atomicAdd(p.totals + 3, 1ull);
        }
    }
    if (lane == 0 && npair) atomicAdd(p.totals + 4, npair);
}

// ---- SelectNeighbors ------------------------------------------------------------------------
// cand_*: candidates nearest first (key order) in shared memory.  r_*: the selected list in
// upstream's list order (furthest-first when nc <= lm, else selection order then back-fill).
// `pruned` = the candidate upstream reports as pruned (-1 when nothing was dropped).
template <typename T, int IP, int NV, int G>
__device__ __forceinline__ int select_neighbors_warp(const GraphView &g, float *q, const int32_t *cand_id,
                                                     const float *cand_d, int nc, int lm, int32_t *r_id, float *r_d,
                                                     int32_t *wd_id, float *wd_d, int32_t &pruned, int lane,
                                                     unsigned long long &npair)
{
    pruned = -1;
    if (nc <= lm) {
        for (int j = lane; j < nc; j += 32) { r_id[j] = cand_id[nc - 1 - j]; r_d[j] = cand_d[nc - 1 - j]; }
        __syncwarp();
        return nc;
    }
    int nr = 0, nwd = 0, i = 0;
    while (i < nc && nr < lm) {
        const int32_t e = cand_id[i];
        const float ed = cand_d[i];
        i++;
        bool closer = true;
        if (nr > 0) {
            __syncwarp();
            stage_row<T>(g.vecs + (size_t) e * g.row_bytes, g.nvec, q, lane);
            __syncwarp();
            // CheckElementCloser: rejected as soon as one selected neighbour is at least as close
            // to e as the owner is; evaluated eight selected neighbours at a time
            for (int jb = 0; jb < nr && closer; jb += 8) {
                const int j = jb + lane;
                const int32_t nb = (lane < 8 && j < nr) ? r_id[j] : -1;
                const unsigned mask = __ballot_sync(FULL, nb >= 0);
                const float d = eval_candidates<T, IP, NV, G>(g, q, nb, mask, lane);
                // n_pair counts what the sequential loop evaluates: up to the first failure
                const unsigned fail = __ballot_sync(FULL, nb >= 0 && d <= ed);
                if (fail) { npair += __ffs(fail); closer = false; }
                else npair += __popc(mask);
            }
        }
        if (lane == 0) {
            if (closer) { r_id[nr] = e; r_d[nr] = ed; }
            else { wd_id[nwd] = e; wd_d[nwd] = ed; }
        }
        if (closer) nr++; else nwd++;
        __syncwarp();
    }
    int wdoff = 0;
    while (wdoff < nwd && nr < lm) {
        if (lane == 0) { r_id[nr] = wd_id[wdoff]; r_d[nr] = wd_d[wdoff]; }
        nr++; wdoff++;
    }
    __syncwarp();
    pruned = wdoff < nwd ? wd_id[wdoff] : cand_id[nc - 1];
    return nr;
}

template <typename T> __host__ __device__ inline size_t select_warp_smem(int nvec, int nc_max, int lm_max)
{
    size_t b = (size_t) nvec * Vec<T>::VEC * 4 + (size_t) nc_max * 16 + (size_t) lm_max * 8;
    return (b + 15) & ~(size_t) 15;
}

// ---- HnswUpdateConnection, one warp per segment (see link_kernel.cuh) --------------------------
template <typename T, int IP, int NV, int G>
__global__ void __launch_bounds__(BUILD_WARPS * 32) link_warp_kernel(const LinkParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    if (*p.flag) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    const int lm0 = 2 * g.m, cap = lm0 + 1;
    // per warp: query, list (id,d) x cap, sorted (id,d) x cap, wd (id,d) x cap, r (id,d) x lm0
    unsigned char *base = smem + select_warp_smem<T>(g.nvec, 3 * cap / 2 + 2, lm0) * warp;
    float *q = reinterpret_cast<float *>(base);
    int32_t *l_id = reinterpret_cast<int32_t *>(base + (size_t) g.nvec * Vec<T>::VEC * 4);
    float *l_d = reinterpret_cast<float *>(l_id + cap);
    int32_t *s_id = reinterpret_cast<int32_t *>(l_d + cap);
    float *s_d = reinterpret_cast<float *>(s_id + cap);
    int32_t *wd_id = reinterpret_cast<int32_t *>(s_d + cap);
    float *wd_d = reinterpret_cast<float *>(wd_id + cap);
    int32_t *r_id = reinterpret_cast<int32_t *>(wd_d + cap);
    float *r_d = reinterpret_cast<float *>(r_id + lm0);

    unsigned long long npair = 0;
    const int S = *p.nseg;
    for (int seg = blockIdx.x * BUILD_WARPS + warp; seg < S; seg += gridDim.x * BUILD_WARPS) {
        const int e0 = p.seg_start[seg];
        const unsigned long long key0 = p.edge_key[e0] >> LINK_KEY_SRC_BITS;
        const int lc = (int) (key0 >> 32);
        const int32_t target = (int32_t) (key0 & 0xffffffffu);
        const int lm = lc == 0 ? lm0 : g.m;
        int32_t *gl;
        float *gld;
        if (lc == 0) { gl = p.nbr0 + (size_t) target * lm0; gld = p.nbr0d + (size_t) target * lm0; }
        else {
            const size_t row = (size_t) g.uoff[target] + (lc - 1);
            gl = p.nbru + row * g.m; gld = p.nbrud + row * g.m;
        }
        __syncwarp();
        int cnt = 0;
        for (int jb = 0; jb < lm; jb += 32) {
            const int j = jb + lane;
            int32_t v = -1;
            if (j < lm) { v = gl[j]; l_id[j] = v; l_d[j] = gld[j]; }
            cnt += __popc(__ballot_sync(FULL, v >= 0));
        }
        __syncwarp();
        for (int e = e0; e < p.E; e++) {
            const unsigned long long key = p.edge_key[e];
            if ((key >> LINK_KEY_SRC_BITS) != key0) break;
            const int32_t src = (int32_t) (p.first + (int64_t) (key & ((1u << LINK_KEY_SRC_BITS) - 1)));
            const float d = p.edge_d[e];
            if (cnt < lm) {
                if (lane == 0) { l_id[cnt] = src; l_d[cnt] = d; }
                cnt++;
                __syncwarp();
                continue;
            }
            // shrink: candidates = list + new, sorted by (distance, id) [sortCandidates = true]
            if (lane == 0) { l_id[lm] = src; l_d[lm] = d; }
            __syncwarp();
            const int nc = lm + 1;
            for (int ib = 0; ib < nc; ib += 32) {
                const int i = ib + lane;
                if (i < nc) {
                    const float di = l_d[i];
                    const int32_t ii = l_id[i];
                    int rank = 0;
                    for (int j = 0; j < nc; j++) {
                        const float dj = l_d[j];
                        rank += (dj < di || (dj == di && l_id[j] < ii)) ? 1 : 0;
                    }
                    s_id[rank] = ii; s_d[rank] = di;
                }
            }
            __syncwarp();
            int32_t pruned;
            select_neighbors_warp<T, IP, NV, G>(g, q, s_id, s_d, nc, lm, r_id, r_d, wd_id, wd_d, pruned, lane, npair);
            // find and replace the pruned element (nothing happens when the new one is pruned)
            for (int jb = 0; jb < lm; jb += 32) {
                const int j = jb + lane;
                if (j < lm && l_id[j] == pruned) { l_id[j] = src; l_d[j] = d; }
            }
            __syncwarp();
        }
        for (int j = lane; j < lm; j += 32) {
            if (j < cnt) { gl[j] = l_id[j]; gld[j] = l_d[j]; }
        }
    }
    if (lane == 0 && npair) atomicAdd(p.totals + 4, npair);
}

// ---- HnswUpdateConnection with memoised pair distances ------------------------------------------
// A shrink replaces at most one member of the list, so the distances AMONG the members survive it:
// each list keeps the strict lower triangle of its members' distance matrix (by slot) in HBM.  A
// shrink then costs lm new pairs (new element <-> members: one staged row, one gather of lm rows)
// plus the selection replayed on the matrix, instead of the ~125 pairs CheckElementCloser asks for.
// The first shrink of a list fills its matrix (lm(lm-1)/2 pairs).  Results and n_pair are those of
// the sequential algorithm (the distances are the same numbers, computed once).  One warp per
// segment; per warp in shared memory: staged row, matrix, list, sort scratch.
template <typename T> __host__ __device__ inline size_t memo_warp_smem(int nvec, int lm0)
{
    const int cap = lm0 + 1;
    // two staged rows | matrix | second new element's row of the matrix | list | sort scratch
    size_t b = (size_t) 2 * nvec * Vec<T>::VEC * 4 + (size_t) cap * cap * 4 + (size_t) cap * 4 + (size_t) cap * 8 + ((cap + 7) & ~7);
    return (b + 15) & ~(size_t) 15;
}
// per CTA: triangle index -> (a << 8 | b), so that a list's triangle moves with flat coalesced accesses
__host__ __device__ inline size_t memo_lut_bytes(int lm0) { return ((size_t) lm0 * (lm0 - 1) / 2 * 2 + 15) & ~(size_t) 15; }

// the less travelled paths of link_memo_kernel (out of line they cost more in spills than they save in instruction cache: measured)
// first shrink of a list whose triangle the pre-pass did not fill: distances among its members
template <typename T, int IP, int NV, int G>
__device__ __forceinline__ void memo_fill_matrix(const GraphView &g, float *q0, float *D, int ld, const int32_t *l_id, int lm, int lane)
{
    for (int a = 1; a < lm; a++) {
        __syncwarp();
        stage_row_nv<T, NV>(g.vecs + (size_t) l_id[a] * g.row_bytes, g.nvec, q0, lane);
        __syncwarp();
        for (int jb = 0; jb < a; jb += 32) {
            const int j = jb + lane;
            const int32_t nb = j < a ? l_id[j] : -1;
            const float v = eval_candidates<T, IP, NV, G>(g, q0, nb, __ballot_sync(FULL, nb >= 0), lane);
            if (j < a) { D[a * ld + j] = v; D[j * ld + a] = v; }
        }
    }
}
// distances the tables did not hold: new element A (and B) against the members flagged in missA / missB
template <typename T, int IP, int NV, int G>
__device__ __forceinline__ void memo_eval_missing(const GraphView &g, const float *q0, const float *q1, int two, int32_t nb,
                                               unsigned missA, unsigned missB, int lane, float &vA, float &vB)
{
    if (two && (missA & missB)) {
        float cA, cB;
        eval_candidates2<T, IP, NV, (G > 2 ? 2 : G)>(g, q0, q1, nb, missA & missB, lane, cA, cB);
        if ((missA & missB) >> lane & 1u) { vA = cA; vB = cB; }
    }
    const unsigned onlyA = two ? (missA & ~missB) : missA, onlyB = two ? (missB & ~missA) : 0u;
    if (onlyA) {
        const float c = eval_candidates<T, IP, NV, G>(g, q0, nb, onlyA, lane);
        if (onlyA >> lane & 1u) vA = c;
    }
    if (onlyB) {
        const float c = eval_candidates<T, IP, NV, G>(g, q1, nb, onlyB, lane);
        if (onlyB >> lane & 1u) vB = c;
    }
}

template <typename T, int IP, int NV, int G>
__global__ void __launch_bounds__(BUILD_WARPS * 32, 5) link_memo_kernel(const LinkParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    if (*p.flag) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    const int lm0 = 2 * g.m, cap = lm0 + 1, ld = cap;
    const int qfloats = g.nvec * Vec<T>::VEC;
    uint16_t *lut = reinterpret_cast<uint16_t *>(smem);
    unsigned char *base = smem + memo_lut_bytes(lm0) + memo_warp_smem<T>(g.nvec, lm0) * warp;
    float *q0 = reinterpret_cast<float *>(base);
    float *q1 = q0 + qfloats;
    float *D = q1 + qfloats;
    float *D2 = D + cap * cap;                       // second new element <-> members
    int32_t *l_id = reinterpret_cast<int32_t *>(D2 + cap);
    float *l_d = reinterpret_cast<float *>(l_id + cap);
    uint8_t *ord = reinterpret_cast<uint8_t *>(l_d + cap);
    for (int a = 1 + (int) threadIdx.x; a < lm0; a += BUILD_WARPS * 32)
        for (int b = 0; b < a; b++) lut[a * (a - 1) / 2 + b] = (uint16_t) (a << 8 | b);
    __syncthreads();

    unsigned long long npair = 0;
    const int S = *p.nseg;
    const unsigned src_mask = (1u << LINK_KEY_SRC_BITS) - 1;
    for (int seg = blockIdx.x * BUILD_WARPS + warp; seg < S; seg += gridDim.x * BUILD_WARPS) {
        const int e0 = p.seg_start[seg];
        const unsigned long long key0 = p.edge_key[e0] >> LINK_KEY_SRC_BITS;
        const int lc = (int) (key0 >> 32);
        const int32_t target = (int32_t) (key0 & 0xffffffffu);
        const int lm = lc == 0 ? lm0 : g.m;
        const int tri = lm * (lm - 1) / 2;
        int32_t *gl;
        float *gld, *pc;
        uint8_t *pv;
        if (lc == 0) {
            gl = p.nbr0 + (size_t) target * lm0; gld = p.nbr0d + (size_t) target * lm0;
            pc = p.pc0 + (size_t) target * tri; pv = p.pv0 + target;
        } else {
            const size_t row = (size_t) g.uoff[target] + (lc - 1);
            gl = p.nbru + row * g.m; gld = p.nbrud + row * g.m;
            pc = p.pcu + row * tri; pv = p.pvu + row;
        }
        __syncwarp();
        const bool filled = *pv != 0;
        int cnt = 0;
        for (int jb = 0; jb < lm; jb += 32) {
            const int j = jb + lane;
            int32_t v = -1;
            if (j < lm) { v = gl[j]; l_id[j] = v; l_d[j] = gld[j]; }
            cnt += __popc(__ballot_sync(FULL, v >= 0));
        }
        __syncwarp();
        // the segment's edges: lanes read up to 32 of them at once (a longer segment reads again)
        int e = e0;
        bool have_matrix = false, more = true;
        while (more) {
            const int ee = e + lane;
            unsigned long long key = LINK_KEY_INVALID;
            float dk = 0.f;
            if (ee < p.E) { key = p.edge_key[ee]; dk = p.edge_d[ee]; }
            const unsigned in_seg = __ballot_sync(FULL, (key >> LINK_KEY_SRC_BITS) == key0);
            const int navail = in_seg == FULL ? 32 : __ffs(~in_seg) - 1;     // leading run
            more = navail == 32;
            int k = 0;
            // appends while the list has room
            while (k < navail && cnt < lm) {
                const int32_t src = (int32_t) (p.first + (int64_t) ((unsigned) __shfl_sync(FULL, key, k) & src_mask));
                const float d = __shfl_sync(FULL, dk, k);
                if (lane == 0) { l_id[cnt] = src; l_d[cnt] = d; }
                cnt++; k++;
            }
            __syncwarp();
            // shrinks, two new elements per pass over the members' rows
            while (k < navail) {
                const int two = k + 1 < navail ? 1 : 0;
                const int32_t srcA = (int32_t) (p.first + (int64_t) ((unsigned) __shfl_sync(FULL, key, k) & src_mask));
                const int32_t srcB = (int32_t) (p.first + (int64_t) ((unsigned) __shfl_sync(FULL, key, k + two) & src_mask));
                const float dA = __shfl_sync(FULL, dk, k), dB = __shfl_sync(FULL, dk, k + two);
                if (!have_matrix) {
                    if (filled) {
#pragma unroll 16
                        for (int idx = lane; idx < tri; idx += 32) {
                            const float v = __ldcs(pc + idx);
                            const int ab = lut[idx], a = ab >> 8, b = ab & 0xff;
                            D[a * ld + b] = v; D[b * ld + a] = v;
                        }
                    } else {
                        // cold (the fill pre-pass filled almost every triangle): the generic row loop keeps the kernel small
                        memo_fill_matrix<T, IP, (HB_MEMO_COLD_GENERIC ? 0 : NV), (HB_MEMO_COLD_GENERIC ? 2 : G)>(g, q0, D, ld, l_id, lm, lane);
                    }
                    have_matrix = true;
                }
                // the new elements against the members.  Their candidate searches expanded every neighbour
                // they selected, so these distances were evaluated already and sit in the searches' tables
                // (EvalTable); only what is missing there -- members that joined in this very batch, a
                // crowded table -- is computed, each member row fetched once for both new elements.
                EvalTable etA, etB;
                const bool have_et = p.et_key != nullptr;
                etA.key = etB.key = nullptr;
                if (have_et) {
                    etA.key = const_cast<uint32_t *>(p.et_key) + (size_t) (srcA - p.first) * p.et_slots;
                    etA.val = const_cast<float *>(p.et_val) + (size_t) (srcA - p.first) * p.et_slots;
                    etB.key = const_cast<uint32_t *>(p.et_key) + (size_t) (srcB - p.first) * p.et_slots;
                    etB.val = const_cast<float *>(p.et_val) + (size_t) (srcB - p.first) * p.et_slots;
                    etA.mask = etB.mask = (uint32_t) p.et_slots - 1u;
                }
                bool staged = false;
                for (int jb = 0; jb < lm; jb += 32) {
                    const int j = jb + lane;
                    const int32_t nb = j < lm ? l_id[j] : -1;
                    float vA = 0.f, vB = 0.f;
                    bool okA = false, okB = !two;
                    if (have_et && nb >= 0) {
                        okA = etA.get((uint32_t) nb, vA);
                        if (two) okB = etB.get((uint32_t) nb, vB);
                    }
                    const unsigned missA = __ballot_sync(FULL, nb >= 0 && !okA);
                    const unsigned missB = __ballot_sync(FULL, nb >= 0 && !okB);
#ifdef HB_LINK_PROFILE
                    {
                        const unsigned valid = __ballot_sync(FULL, nb >= 0);
                        if (lane == 0) {
                            atomicAdd(p.totals + 14, (unsigned long long) (__popc(valid) * (1 + two)));
                            atomicAdd(p.totals + 15, (unsigned long long) (__popc(missA) + (two ? __popc(missB) : 0)));
                        }
                    }
#endif
                    if ((missA | missB) && !staged) {
                        __syncwarp();
                        stage_row_nv<T, NV>(g.vecs + (size_t) srcA * g.row_bytes, g.nvec, q0, lane);
                        if (two) stage_row_nv<T, NV>(g.vecs + (size_t) srcB * g.row_bytes, g.nvec, q1, lane);
                        __syncwarp();
                        staged = true;
                    }
                    if (missA | missB) memo_eval_missing<T, IP, (HB_MEMO_COLD_GENERIC ? 0 : NV), (HB_MEMO_COLD_GENERIC ? 2 : G)>(g, q0, q1, two, nb, missA, missB, lane, vA, vB);
                    if (j < lm) { D[lm * ld + j] = vA; D[j * ld + lm] = vA; if (two) D2[j] = vB; }
                }
                float dAB = 0.f;
                if (two) {
                    if (!staged) {
                        __syncwarp();
                        stage_row_nv<T, NV>(g.vecs + (size_t) srcA * g.row_bytes, g.nvec, q0, lane);
                        stage_row_nv<T, NV>(g.vecs + (size_t) srcB * g.row_bytes, g.nvec, q1, lane);
                        __syncwarp();
                    }
                    dAB = staged_pair_distance<T, IP>(q0, q1, g.nvec, lane);
                }
                if (lane == 0) { l_id[lm] = srcA; l_d[lm] = dA; }
                __syncwarp();
                const int psA = link_select_slot(D, ld, l_id, l_d, ord, lm, lane, npair);
                if (psA != lm) {
                    // the new element takes the pruned member's slot: list entry, matrix row and column
                    for (int b = lane; b < lm; b += 32)
                        if (b != psA) { const float v = D[lm * ld + b]; D[psA * ld + b] = v; D[b * ld + psA] = v; }
                    if (lane == 0) { l_id[psA] = srcA; l_d[psA] = dA; }
                }
                __syncwarp();
                if (two) {
                    for (int b = lane; b < lm; b += 32) {
                        const float v = (b == psA) ? dAB : D2[b];
                        D[lm * ld + b] = v; D[b * ld + lm] = v;
                    }
                    if (lane == 0) { l_id[lm] = srcB; l_d[lm] = dB; }
                    __syncwarp();
                    const int psB = link_select_slot(D, ld, l_id, l_d, ord, lm, lane, npair);
                    if (psB != lm) {
                        for (int b = lane; b < lm; b += 32)
                            if (b != psB) { const float v = D[lm * ld + b]; D[psB * ld + b] = v; D[b * ld + psB] = v; }
                        if (lane == 0) { l_id[psB] = srcB; l_d[psB] = dB; }
                    }
                    __syncwarp();
                }
                k += 1 + two;
            }
            e += navail;
        }
        for (int j = lane; j < lm; j += 32)
            if (j < cnt) { gl[j] = l_id[j]; gld[j] = l_d[j]; }
        if (have_matrix) {
            for (int idx = lane; idx < tri; idx += 32) {
                const int ab = lut[idx];
                __stcs(pc + idx, D[(ab >> 8) * ld + (ab & 0xff)]);
            }
            if (lane == 0 && !filled) *pv = 1;
        }
    }
    if (lane == 0 && npair) atomicAdd(p.totals + 4, npair);
}

// cached owner->neighbour distances for a graph that was loaded rather than built here
struct NbrDistParams {
    GraphView g;
    int64_t rows;                 // n (layer 0) or upper rows
    int deg;
    const int32_t *owner_of_row;  // upper table: owning element of each row; NULL = row index
    const int32_t *nbr; float *nbrd;
};

template <typename T, int IP>
__global__ void __launch_bounds__(BUILD_WARPS * 32) nbr_dist_kernel(const NbrDistParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    float *q = reinterpret_cast<float *>(smem + build_warp_smem<T>(g.nvec, 0, 0, true) * warp);
    for (int64_t row = (int64_t) blockIdx.x * BUILD_WARPS + warp; row < p.rows; row += (int64_t) gridDim.x * BUILD_WARPS) {
        const int64_t owner = p.owner_of_row ? p.owner_of_row[row] : row;
        __syncwarp();
        stage_row<T>(g.vecs + (size_t) owner * g.row_bytes, g.nvec, q, lane);
        __syncwarp();
        for (int jb = 0; jb < p.deg; jb += 32) {
            const int j = jb + lane;
            const int32_t nb = j < p.deg ? p.nbr[row * p.deg + j] : -1;
            const unsigned mask = __ballot_sync(FULL, nb >= 0);
            const float d = eval_candidates<T, IP, 0, 2>(g, q, nb, mask, lane);
            if (j < p.deg) p.nbrd[row * p.deg + j] = nb >= 0 ? d : 0.f;
        }
    }
}

// ---- launch helpers ---------------------------------------------------------------------------
#define HB_NV_DISPATCH(nvec, CALL)                                                                 \
    switch (nv_of(nvec)) {                                                                         \
    case 1: CALL(1, 8); break;                                                                     \
    case 2: CALL(2, 8); break;                                                                     \
    case 3: CALL(3, 4); break;                                                                     \
    case 4: CALL(4, 4); break;                                                                     \
    case 6: CALL(6, 4); break;                                                                     \
    case 8: CALL(8, 2); break;                                                                     \
    default: CALL(0, 2); break;                                                                    \
    }

template <typename T, int IP, bool SLOW>
cudaError_t launch_build_search_t(const BuildSearchParams &p, int num_sms, int slow_grid, cudaStream_t stream)
{
    cudaError_t err = cudaSuccess;
#define HB_CALL(NVV, GG)                                                                           \
    {                                                                                              \
        auto kern = build_search_kernel<T, IP, SLOW ? 0 : NVV, SLOW ? 2 : GG, SLOW>;               \
        const size_t smem = bsearch_warp_smem<T>(p.g.nvec, p.capW, p.slots, SLOW, p.efc, 2 * p.g.m) * BUILD_WARPS; \
        err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem); \
        if (err == cudaSuccess) {                                                                  \
            int bps = 0;                                                                           \
            err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, BUILD_WARPS * 32, smem); \
            if (err == cudaSuccess) {                                                              \
                if (bps > MAX_CTAS_PER_SM) bps = MAX_CTAS_PER_SM;                                  \
                if (bps < 1) err = cudaErrorInvalidConfiguration;                                  \
                else {                                                                             \
                    int64_t want = SLOW ? slow_grid : (p.B + BUILD_WARPS - 1) / BUILD_WARPS;       \
                    int grid = (int) (want < (int64_t) bps * num_sms ? want : (int64_t) bps * num_sms); \
                    if (grid < 1) grid = 1;                                                        \
                    kern<<<grid, BUILD_WARPS * 32, smem, stream>>>(p);                             \
                    err = cudaGetLastError();                                                      \
                }                                                                                  \
            }                                                                                      \
        }                                                                                          \
    }
    HB_NV_DISPATCH(p.g.nvec, HB_CALL)
#undef HB_CALL
    return err;
}

// which: 0 = automatic: the memoising kernel when the pair cache is allocated and m <= 31, else the
// pipelined kernel when two stages of lm+1 rows fit shared memory, else the warp kernel;
// 1 = warp kernel, 2 = pipelined kernel, 3 = memoising kernel (error when the choice cannot run)
template <typename T, int IP>
cudaError_t launch_build_link_t(const LinkParams &p, int num_sms, int which, cudaStream_t stream)
{
    cudaError_t err = cudaSuccess;
    if (p.E <= 0) return err;
    const int lm0 = 2 * p.g.m;
    const size_t stage = link_stage_bytes(p.g.row_bytes, lm0), shared = link_shared_bytes(lm0);
    const size_t limit = 227 * 1024;
    int nstages = shared < limit ? (int) ((limit - shared) / stage) : 0;
    if (nstages > LINK_MAX_STAGES) nstages = LINK_MAX_STAGES;
    const bool can = lm0 <= LINK_MAX_LM && nstages >= 1 && link_num_tiles(LinkTile<T>::TA, lm0) <= LINK_MAX_TILES;
    if (which == 2 && !can) return cudaErrorInvalidConfiguration;
    const bool can_memo = p.pc0 != nullptr && lm0 <= LINK_MAX_LM;
    if (which == 3 && !can_memo) return cudaErrorInvalidConfiguration;
    if (which == 3 || (which == 0 && can_memo)) {
#define HB_CALL(NVV, GG)                                                                           \
    {                                                                                              \
        auto kern = link_memo_kernel<T, IP, NVV, (GG > 4 ? 4 : GG)>;                               \
        const size_t smem = memo_lut_bytes(lm0) + memo_warp_smem<T>(p.g.nvec, lm0) * BUILD_WARPS;  \
        err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem); \
        if (err == cudaSuccess) {                                                                  \
            int grid = (p.E + BUILD_WARPS - 1) / BUILD_WARPS;                                      \
            if (grid > num_sms * 8) grid = num_sms * 8;                                            \
            kern<<<grid, BUILD_WARPS * 32, smem, stream>>>(p);                                     \
            err = cudaGetLastError();                                                              \
        }                                                                                          \
    }
        HB_NV_DISPATCH(p.g.nvec, HB_CALL)
#undef HB_CALL
        return err;
    }
    if (which == 2 || (which == 0 && can && nstages >= 2)) {
        auto kern = link_pipe_kernel<T, IP>;
        const size_t smem = stage * nstages + shared;
        err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (err != cudaSuccess) return err;
        int64_t grid = num_sms;
        if (grid > (p.E + LINK_PREFETCH - 1) / LINK_PREFETCH) grid = (p.E + LINK_PREFETCH - 1) / LINK_PREFETCH;
        kern<<<(int) grid, LINK_THREADS, smem, stream>>>(p, nstages);
        return cudaGetLastError();
    }
#define HB_CALL(NVV, GG)                                                                           \
    {                                                                                              \
        auto kern = link_warp_kernel<T, IP, NVV, (GG > 4 ? 4 : GG)>;                               \
        const int cap = 2 * p.g.m + 1;                                                             \
        const size_t smem = select_warp_smem<T>(p.g.nvec, 3 * cap / 2 + 2, 2 * p.g.m) * BUILD_WARPS; \
        err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem); \
        if (err == cudaSuccess) {                                                                  \
            int grid = (p.E + BUILD_WARPS - 1) / BUILD_WARPS;                                      \
            if (grid > num_sms * 8) grid = num_sms * 8;                                            \
            kern<<<grid, BUILD_WARPS * 32, smem, stream>>>(p);                                     \
            err = cudaGetLastError();                                                              \
        }                                                                                          \
    }
    HB_NV_DISPATCH(p.g.nvec, HB_CALL)
#undef HB_CALL
    return err;
}

// pair-cache fill pre-pass: link_pipe_kernel in fill mode over p.fill_list.  Returns
// cudaErrorInvalidConfiguration when the pipelined kernel cannot run for this shape (the memoising
// kernel then fills in place).
template <typename T, int IP>
cudaError_t launch_pair_fill_t(const LinkParams &p, int num_sms, int max_items, cudaStream_t stream)
{
    const int lm0 = 2 * p.g.m;
    const size_t stage = link_stage_bytes(p.g.row_bytes, lm0), shared = link_shared_bytes(lm0);
    const size_t limit = 227 * 1024;
    int nstages = shared < limit ? (int) ((limit - shared) / stage) : 0;
    if (nstages > LINK_MAX_STAGES) nstages = LINK_MAX_STAGES;
    if (!(lm0 <= LINK_MAX_LM && nstages >= 1 && link_num_tiles(LinkTile<T>::TA, lm0) <= LINK_MAX_TILES) || !p.fill_list)
        return cudaErrorInvalidConfiguration;
    auto kern = link_pipe_kernel<T, IP>;
    const size_t smem = stage * nstages + shared;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (err != cudaSuccess) return err;
    int64_t grid = num_sms;
    if (grid > (max_items + LINK_PREFETCH - 1) / LINK_PREFETCH) grid = (max_items + LINK_PREFETCH - 1) / LINK_PREFETCH;
    if (grid < 1) grid = 1;
    kern<<<(int) grid, LINK_THREADS, smem, stream>>>(p, nstages);
    return cudaGetLastError();
}

template <typename T, int IP>
cudaError_t launch_nbr_dist_t(const NbrDistParams &p, int num_sms, cudaStream_t stream)
{
    if (p.rows <= 0) return cudaSuccess;
    auto kern = nbr_dist_kernel<T, IP>;
    const size_t smem = build_warp_smem<T>(p.g.nvec, 0, 0, true) * BUILD_WARPS;
    cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (err != cudaSuccess) return err;
    int64_t grid = (p.rows + BUILD_WARPS - 1) / BUILD_WARPS;
    if (grid > num_sms * 8) grid = num_sms * 8;
    kern<<<(int) grid, BUILD_WARPS * 32, smem, stream>>>(p);
    return cudaGetLastError();
}

}   // namespace hb
