// scan_reg.cuh -- the batched scan for short rows: HnswSearchLayer with the W/C list held in REGISTERS.
//
// Same algorithm, same expansion order and therefore the same ids, distances and counters as scan_kernel.cuh
// (role: hnswscan.c GetScanItems + hnswutils.c HnswSearchLayer [RECALL; reference mount empty,
// /root/reference/README.md:1]).  What differs is where the bookkeeping lives.  For 128..256-dimensional rows a
// distance evaluation is one or two 128-bit loads per lane, and ncu shows the shared-memory version of the
// search is bound by instruction issue, not by bytes (profiles/r2_scan128_before_ncu_summary.txt: 44 k warp
// instructions per query, 32 % of them in the sorted-list insertion, issue slots 48 % busy on one stream).  Here:
//   * W and C are one sorted list of up to 32*R (distance, id) entries spread over the warp's registers, slot
//     s = lane*R + r.  Finding the insert position is R ballots, the shift is ONE shuffle per field (each lane
//     passes its last entry up), trimming to ef + boundary ties is R ballots -- no shared-memory round trips.
//   * the candidates that passed the visited filter are compacted through 128 bytes of shared memory, so a
//     group of G rows gets its ids with one or two vector loads instead of G shuffles, and a group's G results
//     come back with one shuffle.
// Queries whose list outgrows the registers (tie tail) or whose visited set outgrows the tables are handed to
// the large-visited-set path exactly like scan_kernel does.
#pragma once
#include "scan_kernel.cuh"

namespace hb {

__device__ __forceinline__ unsigned lanemask_lt()
{
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

template <int R> struct RegW {
    static constexpr int CAP = 32 * R;
    static constexpr int SH = R == 1 ? 0 : (R == 2 ? 1 : (R == 4 ? 2 : 3));
    float d[R];
    uint32_t id[R];
    int L;          // warp-uniform
    float f;        // distance of entry ef-1 while L >= ef (warp-uniform)
    // Invariant: slots >= L hold (+inf, 0xffffffff) -- "further than anything, already expanded" -- so that neither the
    // position count, nor the search for the next unexpanded entry, nor the tie-run count needs an s < L test.
    __device__ __forceinline__ void reset()
    {
        L = 0;
        f = 0.f;
#pragma unroll
        for (int r = 0; r < R; r++) { d[r] = __int_as_float(0x7f800000); id[r] = 0xffffffffu; }
    }

    // this lane's entry r = j mod R, as a tree of two-way selects (a chain of compares is turned into an indexed
    // load by the compiler, which sends the whole list to local memory)
    template <typename V> __device__ __forceinline__ static V pick(const V (&a)[R], int j)
    {
        if constexpr (R == 1) return a[0];
        else if constexpr (R == 2) return (j & 1) ? a[1] : a[0];
        else if constexpr (R == 4) {
            const V lo = (j & 1) ? a[1] : a[0], hi = (j & 1) ? a[3] : a[2];
            return (j & 2) ? hi : lo;
        } else {
            const V v0 = (j & 1) ? a[1] : a[0], v1 = (j & 1) ? a[3] : a[2], v2 = (j & 1) ? a[5] : a[4], v3 = (j & 1) ? a[7] : a[6];
            const V lo = (j & 2) ? v1 : v0, hi = (j & 2) ? v3 : v2;
            return (j & 4) ? hi : lo;
        }
    }
    __device__ __forceinline__ float get_d(int j) const { return __shfl_sync(FULL, pick(d, j), j >> SH); }
    __device__ __forceinline__ uint32_t get_id(int j) const { return __shfl_sync(FULL, pick(id, j), j >> SH); }
    __device__ __forceinline__ void refresh_f(int ef) { if (L >= ef) f = get_d(ef - 1); }

    // insert (ed, eid) keeping (distance, id) order, then trim to ef + the run of entries tying with entry ef-1
    __device__ __forceinline__ int insert(float ed, uint32_t eid, int ef, int lane)
    {
        if (L + 1 > CAP) return ST_TAIL;
        int pos = 0;
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int s = lane * R + r;
            const bool lt = d[r] < ed || (d[r] == ed && (id[r] & ID_MASK) < eid);
            pos += __popc(__ballot_sync(FULL, lt));
            (void) s;
        }
        const float pd = __shfl_up_sync(FULL, d[R - 1], 1);
        const uint32_t pi = __shfl_up_sync(FULL, id[R - 1], 1);
#pragma unroll
        for (int r = R - 1; r >= 0; r--) {
            const int s = lane * R + r;
            const float nd = r ? d[r > 0 ? r - 1 : 0] : pd;
            const uint32_t ni = r ? id[r > 0 ? r - 1 : 0] : pi;
            if (s > pos) { d[r] = nd; id[r] = ni; }
            else if (s == pos) { d[r] = ed; id[r] = eid; }
        }
        L++;
        if (L >= ef) {
            f = get_d(ef - 1);
            if (L > ef) {
                int keep = 0;
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int s = lane * R + r;
                    keep += __popc(__ballot_sync(FULL, s >= ef && d[r] == f));
                }
                if (ef + keep < L) {             // something fell off the end: restore the invariant
#pragma unroll
                    for (int r = 0; r < R; r++)
                        if (lane * R + r >= ef + keep) { d[r] = __int_as_float(0x7f800000); id[r] = 0xffffffffu; }
                }
                L = ef + keep;
            }
        }
        return ST_OK;
    }

    // The candidates flagged in amask (lane j holds candidate j: myd, cj) inserted in ONE step: ranks by ballots, then a
    // scatter through shared memory (td, ti: CAP entries).  Inserting them one after the other in lane order gives the
    // same list PROVIDED no candidate's distance equals another key's: then the admission test `ed < f` never meets
    // equality, whatever was trimmed or skipped on the way lies beyond the final entry ef-1 as well, and the result is
    // the merge trimmed to ef + ties.  Returns -1 WITHOUT touching the list when that cannot be guaranteed (equal
    // distances, or the untrimmed merge would not fit): the caller then inserts one at a time.
    __device__ __forceinline__ int insert_many(float myd, uint32_t cj, unsigned amask, int ef, int lane, float *td, uint32_t *ti)
    {
        const int k = __popc(amask);
        if (L + k > CAP) return -1;
        int shift[R];
#pragma unroll
        for (int r = 0; r < R; r++) shift[r] = 0;
        const bool mine = (amask >> lane) & 1u;
        int mypos = 0;
        bool eq = false;
        for (unsigned rem = amask; rem; rem &= rem - 1) {
            const int s = __ffs(rem) - 1;
            const float ed = __shfl_sync(FULL, myd, s);
            const uint32_t eid = __shfl_sync(FULL, cj, s);
            int below = 0;
#pragma unroll
            for (int r = 0; r < R; r++) {
                const bool wlt = d[r] < ed || (d[r] == ed && (id[r] & ID_MASK) < eid);     // this entry stays before the candidate
                below += __popc(__ballot_sync(FULL, wlt));
                shift[r] += wlt ? 0 : 1;
                eq |= d[r] == ed;
            }
            if (s == lane) mypos += below;
            else if (mine) {
                mypos += (ed < myd || (ed == myd && eid < cj)) ? 1 : 0;
                eq |= ed == myd;
            }
        }
        if (__any_sync(FULL, eq)) return -1;
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int s = lane * R + r;
            if (s < L) { td[s + shift[r]] = d[r]; ti[s + shift[r]] = id[r]; }
        }
        if (mine) { td[mypos] = myd; ti[mypos] = cj; }
        __syncwarp();
        L += k;
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int s = lane * R + r;
            const bool in = s < L;
            d[r] = in ? td[in ? s : 0] : __int_as_float(0x7f800000);
            id[r] = in ? ti[in ? s : 0] : 0xffffffffu;
        }
        __syncwarp();
        if (L >= ef) {
            f = get_d(ef - 1);
            if (L > ef) {
                int keep = 0;
#pragma unroll
                for (int r = 0; r < R; r++) {
                    const int s = lane * R + r;
                    keep += __popc(__ballot_sync(FULL, s >= ef && d[r] == f));
                }
                if (ef + keep < L) {
#pragma unroll
                    for (int r = 0; r < R; r++)
                        if (lane * R + r >= ef + keep) { d[r] = __int_as_float(0x7f800000); id[r] = 0xffffffffu; }
                }
                L = ef + keep;
            }
        }
        return ST_OK;
    }
};

// entry list of the next HnswSearchLayer call = the list's first entry (keep = 1: the scan path)
template <int R, typename VS>
__device__ __forceinline__ int regw_as_entry(RegW<R> &w, VS &vs, int ef, int lane)
{
    if (w.L > 1) {
        w.L = 1;
#pragma unroll
        for (int r = 0; r < R; r++)
            if (lane * R + r >= 1) { w.d[r] = __int_as_float(0x7f800000); w.id[r] = 0xffffffffu; }
    }
    vs.clear(lane);
    if (!vs.room(w.L)) return ST_TABLE;
    const bool sp = vs.spill(w.L);
    if (lane == 0 && w.L > 0) {
        w.id[0] &= ID_MASK;
        vs.insert(w.id[0], sp);
    }
    vs.added(w.L, sp);
    __syncwarp();
    w.refresh_f(ef);
    return ST_OK;
}

// distances of the nnew candidates whose ids sit in cbuf[0 .. nnew) (shared memory, 16-byte aligned); lane j
// (j < nnew) receives candidate j's distance, other lanes +inf
template <typename T, int IP, int NV, int G>
__device__ __forceinline__ float eval_compact(const GraphView &g, const float *q, const int32_t *cbuf, int nnew, int lane)
{
    float myd = __int_as_float(0x7f800000);
    int g0 = 0;
#define HB_CGROUP(GG)                                                                              \
    {                                                                                              \
        int32_t ids[GG];                                                                           \
        if constexpr (GG >= 4) {                                                                   \
            _Pragma("unroll") for (int c = 0; c < GG; c += 4)                                      \
            {                                                                                      \
                const int4 v = *reinterpret_cast<const int4 *>(cbuf + g0 + c);                     \
                ids[c] = v.x; ids[c + 1] = v.y; ids[c + 2] = v.z; ids[c + 3] = v.w;                \
            }                                                                                      \
        } else if constexpr (GG == 2) {                                                            \
            const int2 v = *reinterpret_cast<const int2 *>(cbuf + g0);                             \
            ids[0] = v.x; ids[1] = v.y;                                                            \
        } else ids[0] = cbuf[g0];                                                                  \
        const float s = group_distance<T, IP, NV, GG>(g.vecs, (uint32_t) g.row_bytes, g.nvec, q, ids, lane); \
        const float v = __shfl_sync(FULL, s, ((lane - g0) * (32 / GG)) & 31);                      \
        if (lane >= g0 && lane < g0 + GG) myd = v;                                                 \
        g0 += GG;                                                                                  \
    }
    if constexpr (G >= 8) while (nnew - g0 >= 8) HB_CGROUP(8)
    if constexpr (G >= 4) while (nnew - g0 >= 4) HB_CGROUP(4)
    if constexpr (G >= 2) while (nnew - g0 >= 2) HB_CGROUP(2)
    while (nnew - g0 >= 1) HB_CGROUP(1)
#undef HB_CGROUP
    return myd;
}

template <typename T, int IP, int NV, int G, int R, typename VS>
__device__ __forceinline__ int search_layer_reg(const GraphView &g, RegW<R> &w, VS &vs, const float *q, int32_t *cbuf, int ef,
                                                int lc, int lane, QueryCounters &ctr)
{
    const int deg = lc == 0 ? 2 * g.m : g.m;
    const unsigned lt_mask = lanemask_lt();
    for (;;) {
        // nearest unexpanded entry: slots are lane-major, so the lowest lane that has one has the lowest slot
        int mys = 0x7fffffff;
#pragma unroll
        for (int r = R - 1; r >= 0; r--) {
            if (!(w.id[r] & EXP_BIT)) mys = lane * R + r;       // expanded entries and free slots carry the bit
        }
        const unsigned b = __ballot_sync(FULL, mys != 0x7fffffff);
        if (!b) break;
        const int src = __ffs(b) - 1;
        const int idx = __shfl_sync(FULL, mys, src);
        const uint32_t cid = __shfl_sync(FULL, RegW<R>::pick(w.id, mys), src);
#pragma unroll
        for (int r = 0; r < R; r++) if (lane * R + r == idx) w.id[r] |= EXP_BIT;
        if (lc == 0) ctr.n_hop0++; else ctr.n_hopu++;
        if (!vs.room(deg)) return ST_TABLE;
        const int32_t *list = lc == 0 ? g.nbr0 + (size_t) cid * deg : g.nbru + ((size_t) g.uoff[cid] + (lc - 1)) * g.m;
        for (int cb = 0; cb < deg; cb += 32) {
            const int i = cb + lane;
            const int32_t nb = i < deg ? list[i] : -1;
            const bool sp = vs.spill(min(32, deg - cb));
            bool isnew = false;
            if (nb >= 0) isnew = vs.insert((uint32_t) nb, sp);
            const unsigned nmask = __ballot_sync(FULL, isnew);
            if (nmask == 0) continue;
            const int nnew = __popc(nmask);
            vs.added(nnew, sp);
            ctr.n_dist += nnew;
            // compact the new candidates, neighbour order kept: candidate j sits in cbuf[j] and is lane j's
            if (isnew) cbuf[__popc(nmask & lt_mask)] = nb;
            __syncwarp();
            const uint32_t cj = lane < nnew ? (uint32_t) cbuf[lane] : 0u;
            const float myd = eval_compact<T, IP, NV, G>(g, q, cbuf, nnew, lane);
            __syncwarp();
            unsigned amask = __ballot_sync(FULL, lane < nnew && (w.L < ef || myd < w.f));
            while (amask) {
                const int s = __ffs(amask) - 1;
                amask &= amask - 1;
                const float ed = __shfl_sync(FULL, myd, s);
                const uint32_t eid = __shfl_sync(FULL, cj, s);
                if (w.L >= ef && !(ed < w.f)) continue;
                const int st = w.insert(ed, eid, ef, lane);
                if (st) return st;
            }
        }
    }
    return ST_OK;
}

template <typename T> __host__ __device__ inline size_t scan_reg_warp_smem(int nvec, int slots)
{
    return (((size_t) nvec * Vec<T>::VEC * 4 + (size_t) slots * 4 + 128) + 15) & ~(size_t) 15;
}

// One warp (= one concurrent query) per CTA: a CTA's resources come back the moment its last query is done, so the tail
// of one batch overlaps the start of the next at warp granularity (with four warps per CTA three idle warps wait for the
// straggler; measured in profiles/r2_experiments.md).
constexpr int SCAN_REG_WARPS = 1;

template <typename T, int IP, int NV, int G, int R, int MINB>
__global__ void __launch_bounds__(SCAN_REG_WARPS * 32, MINB) scan_reg_kernel(const ScanParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    unsigned char *base = smem + scan_reg_warp_smem<T>(g.nvec, p.slots) * warp;
    float *q = reinterpret_cast<float *>(base);
    int32_t *cbuf = reinterpret_cast<int32_t *>(base + (size_t) g.nvec * Vec<T>::VEC * 4);
    VisitedHash vs;
    vs.tab = reinterpret_cast<uint32_t *>(cbuf + 32);
    vs.set_overflow(p.ovf + ((size_t) blockIdx.x * SCAN_REG_WARPS + warp) * p.oslots, p.oslots);
    RegW<R> w;
    const int ef = p.ef;

    for (;;) {
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(p.work, 1u);
        item = __shfl_sync(FULL, item, 0);
        if (item >= (unsigned) p.nq) break;
        const int64_t qi = item;
        __syncwarp();
        stage_query<T>(reinterpret_cast<const T *>(p.queries) + qi * g.dim, g.dim, g.nvec, q, lane);
        __syncwarp();

        QueryCounters ctr = { 0, 0, 0 };
        int st = ST_OK;
        w.reset();
        if (g.entry >= 0) {
            const float d0 = one_distance<T, IP, NV>(g, q, g.entry, lane);
            ctr.n_dist = 1;
            if (lane == 0) { w.d[0] = d0; w.id[0] = (uint32_t) g.entry; }
            w.L = 1;
            vs.configure(p.upper_slots);
            for (int lc = g.entry_level; lc >= 1 && st == ST_OK; lc--) {
                st = regw_as_entry(w, vs, 1, lane);
                if (st == ST_OK) st = search_layer_reg<T, IP, NV, G, R>(g, w, vs, q, cbuf, 1, lc, lane, ctr);
            }
            if (st == ST_OK) {
                vs.configure(p.slots);
                st = regw_as_entry(w, vs, ef, lane);
                if (st == ST_OK) st = search_layer_reg<T, IP, NV, G, R>(g, w, vs, q, cbuf, ef, 0, lane, ctr);
            }
        }
        if (st != ST_OK) {
            // hand the query to the large-visited-set path; nothing is written for it here
            if (lane == 0) {
                const int slot = atomicAdd(p.slow_count, 1);
                p.slow_list[slot] = (int32_t) qi;
                p.status[qi] = st;
            }
            continue;
        }
        const int cnt = min(w.L, ef);
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int s = lane * R + r;
            if (s < p.out_stride) {
                p.out_elem[qi * p.out_stride + s] = s < cnt ? (int32_t) (w.id[r] & ID_MASK) : -1;
                p.out_dist[qi * p.out_stride + s] = s < cnt ? w.d[r] : __int_as_float(0x7f800000);
            }
        }
        if (lane == 0) {
            p.out_cnt[qi] = cnt;
            p.status[qi] = 0;
            atomicAdd(p.totals + 0, (unsigned long long) ctr.n_dist);
            atomicAdd(p.totals + 1, (unsigned long long) ctr.n_hop0);
            atomicAdd(p.totals + 2, (unsigned long long) ctr.n_hopu);
            if (p.per_query) {
                p.per_query[qi * 4 + 0] = ctr.n_dist;
                p.per_query[qi * 4 + 1] = ctr.n_hop0;
                p.per_query[qi * 4 + 2] = ctr.n_hopu;
                p.per_query[qi * 4 + 3] = 0;
            }
        }
    }
}

// rows short enough that bookkeeping, not bytes, bounds the scan (one or two 128-bit loads per lane): the
// register-list kernel when the list fits (ef + room for the tie tail <= 32 R)
inline int reg_list_R(int nvec, int ef, const void *ep, int variant)
{
    if (ep != nullptr || variant == SCAN_SMEM_LIST) return 0;      // single-layer test surface / forced shared-memory list
    const int nv = nv_of(nvec);
    if (nv != 1 && nv != 2) return 0;
    if (ef + 16 <= 64) return 2;
    if (ef + 24 <= 128) return 4;
    return 0;
}

template <typename T, int IP>
cudaError_t launch_scan_reg_t(const ScanParams &p, int R, int num_sms, int max_grid, cudaStream_t stream, ScanLaunchInfo *info)
{
    const size_t smem = scan_reg_warp_smem<T>(p.g.nvec, p.slots) * SCAN_REG_WARPS;
    const int64_t want = (p.nq + SCAN_REG_WARPS - 1) / SCAN_REG_WARPS;
    const int nv = nv_of(p.g.nvec);
#define HB_LAUNCH(NVV, RR, MB) launch_persistent<scan_reg_kernel<T, IP, NVV, 8, RR, MB>, SCAN_REG_WARPS>(p, smem, want, num_sms, max_grid, stream, info)
    if (nv == 1 && R == 2) return HB_LAUNCH(1, 2, 24);
    if (nv == 1 && R == 4) return HB_LAUNCH(1, 4, 24);
    if (nv == 2 && R == 2) return HB_LAUNCH(2, 2, 16);
    if (nv == 2 && R == 4) return HB_LAUNCH(2, 4, 16);
#undef HB_LAUNCH
    return cudaErrorInvalidConfiguration;
}

}   // namespace hb
