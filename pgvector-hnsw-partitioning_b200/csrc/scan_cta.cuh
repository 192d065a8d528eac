// scan_cta.cuh -- the scan for a HANDFUL of queries (one backend's amrescan + amgettuple, small batches): one CTA of
// four warps per query instead of one warp.
//
// Same algorithm and expansion order as scan_kernel.cuh (role: hnswscan.c GetScanItems + hnswutils.c HnswSearchLayer
// [RECALL; reference mount empty, /root/reference/README.md:1]), so ids, distances and counters are identical.  A single
// scan is a chain of dependent expansions; with few queries the GPU is idle and what matters is the length of one link
// of that chain, not throughput.  Per expansion:
//   warp 0   picks the nearest unexpanded entry, reads its neighbour list, filters it through the visited table and
//            compacts the new candidates into shared memory;
//   warp 1   meanwhile looks one expansion ahead: it reads the neighbour list of the NEXT nearest unexpanded entry and
//            asks the rows of its not-yet-visited neighbours into L2 (prefetch only: nothing observable changes), so
//            that when that entry is expanded next -- the usual case -- its list and rows come from L2, not HBM;
//   warps 0-3 evaluate the new candidates' distances, a quarter each (canonical order, so the same bits);
//   warp 0   admits and inserts in neighbour order, as the sequential loop does.
// Queries whose tie tail or visited set outgrow shared memory go to the large-visited-set path like everywhere else.
#pragma once
#include "scan_kernel.cuh"
#include "scan_reg.cuh"

namespace hb {

// -DHB_CTA_PROFILE: cycles of warp 0 per phase of an expansion, printed per layer-0 search (experiments only)
#ifdef HB_CTA_PROFILE
#define HB_CTA_PROF_DECL long long pt_[5] = { 0, 0, 0, 0, 0 }, pl_ = clock64(); int phit_ = 0, pn_ = 0, pprev_ = -2;
#define HB_CTA_PROF_MARK(k) { const long long t_ = clock64(); pt_[k] += t_ - pl_; pl_ = t_; }
#define HB_CTA_PROF_PRED(cid, nxt) { if (cid >= 0) { pn_++; phit_ += (cid == pprev_); } pprev_ = nxt; }
#define HB_CTA_PROF_DUMP if (threadIdx.x == 0 && lc == 0 && blockIdx.x == 0) printf("cta prof: hops %d predicted %d; cycles pick %lld list+filter %lld distances %lld insert %lld loop %lld\n", pn_, phit_, pt_[0], pt_[1], pt_[2], pt_[3], pt_[4]);
#else
#define HB_CTA_PROF_DECL
#define HB_CTA_PROF_MARK(k)
#define HB_CTA_PROF_PRED(cid, nxt)
#define HB_CTA_PROF_DUMP
#endif

constexpr int CTA_WARPS = 4;
constexpr int CTA_SLOTS = 8192;          // visited table of the layer-0 search (32 kB: one CTA per SM is plenty)

template <typename T> __host__ __device__ inline size_t scan_cta_smem(int nvec, int capW)
{
    // query | W (d, id) | visited table | cbuf ids | dbuf distances | control words
    return (((size_t) nvec * Vec<T>::VEC * 4 + (size_t) capW * 8 + (size_t) CTA_SLOTS * 4 + 64 * 8 + 64) + 15) & ~(size_t) 15;
}

template <typename T, int IP, int NV>
__device__ __forceinline__ int search_layer_cta(const GraphView &g, WList &w, VisitedHash &vs, const float *q, int32_t *cbuf,
                                                float *dbuf, volatile int *ctl, int ef, int lc, int lane, int warp,
                                                QueryCounters &ctr)
{
    // ctl[0] = candidate to expand (-1: layer done), ctl[1] = number of new candidates, ctl[2] = status,
    // ctl[3] = next nearest unexpanded candidate (-1: none)
    const int deg = lc == 0 ? 2 * g.m : g.m;
    int low = 0;                       // warp 0 only
    NoDiscard nd;
    HB_CTA_PROF_DECL
    for (;;) {
        HB_CTA_PROF_MARK(4)
        if (warp == 0) {
            int idx = -1, nxt = -1;
            for (int base = low; base < w.L && idx < 0; base += 32) {
                const int i = base + lane;
                const unsigned b = __ballot_sync(FULL, i < w.L && !(w.id[i] & EXP_BIT));
                if (b) {
                    idx = base + __ffs(b) - 1;
                    const unsigned b2 = b & (b - 1);
                    if (b2) nxt = (int) (w.id[base + __ffs(b2) - 1] & ID_MASK);
                }
            }
            int cid = -1;
            if (idx >= 0) {
                cid = (int) (w.id[idx] & ID_MASK);
                __syncwarp();
                if (lane == 0) w.id[idx] |= EXP_BIT;
                low = idx + 1;
                if (lc == 0) ctr.n_hop0++; else ctr.n_hopu++;
            }
            HB_CTA_PROF_PRED(cid, nxt)
            if (lane == 0) { ctl[0] = cid; ctl[3] = nxt; ctl[1] = 0; }
        }
        __syncthreads();
        HB_CTA_PROF_MARK(0)
        const int cid = ctl[0];
        if (cid < 0) break;
        const int32_t *list = lc == 0 ? g.nbr0 + (size_t) cid * deg : g.nbru + ((size_t) g.uoff[cid] + (lc - 1)) * g.m;
        // the neighbour list goes through in chunks of 32, each filtered, evaluated and inserted before the next one --
        // the order in which the sequential loop meets the neighbours
        for (int cb = 0; cb < deg; cb += 32) {
            if (warp == 0) {
                int st = ST_OK, nnew = 0;
                if (cb == 0 && !vs.room(deg)) st = ST_TABLE;
                if (st == ST_OK) {
                    const int i = cb + lane;
                    const int32_t nb = i < deg ? list[i] : -1;
                    bool isnew = false;
                    if (nb >= 0) isnew = vs.insert((uint32_t) nb, false);
                    const unsigned nmask = __ballot_sync(FULL, isnew);
                    if (isnew) cbuf[__popc(nmask & ((1u << lane) - 1u))] = nb;
                    nnew = __popc(nmask);
                    vs.added(nnew, false);
                    ctr.n_dist += nnew;
                }
                if (lane == 0) { ctl[1] = nnew; ctl[2] = st; }
            } else if (warp == 1 && cb == 0 && lc == 0 && deg <= 32) {
                // look ahead: rows the next expansion will most likely want, into L2 (reads of the visited table race
                // with warp 0's inserts: a stale answer only costs a useless prefetch)
                const int nxt = ctl[3];
                if (nxt >= 0) {
                    const int32_t nb = lane < deg ? __ldg(g.nbr0 + (size_t) nxt * deg + lane) : -1;
                    if (nb >= 0 && !vs.contains((uint32_t) nb)) prefetch_l2_bulk(g.vecs + (size_t) nb * g.row_bytes, (uint32_t) g.row_bytes);
                }
            }
            __syncthreads();
            HB_CTA_PROF_MARK(1)
            if (ctl[2] != ST_OK) return ctl[2];
            const int nnew = ctl[1];
            // distances: two candidates per warp and pass
            for (int j0 = warp * 2; j0 < nnew; j0 += CTA_WARPS * 2) {
                if (j0 + 1 < nnew) {
                    const int32_t ids[2] = { cbuf[j0], cbuf[j0 + 1] };
                    const float sd = group_distance<T, IP, NV, 2>(g.vecs, (uint32_t) g.row_bytes, g.nvec, q, ids, lane);
                    const float v1 = __shfl_sync(FULL, sd, 16);
                    if (lane == 0) { dbuf[j0] = sd; dbuf[j0 + 1] = v1; }
                } else {
                    const int32_t ids[1] = { cbuf[j0] };
                    const float sd = group_distance<T, IP, NV, 1>(g.vecs, (uint32_t) g.row_bytes, g.nvec, q, ids, lane);
                    if (lane == 0) dbuf[j0] = sd;
                }
            }
            __syncthreads();
            HB_CTA_PROF_MARK(2)
            if (warp == 0) {
                int st = ST_OK;
                for (int j = 0; j < nnew && st == ST_OK; j++) {
                    const float ed = dbuf[j];
                    const uint32_t eid = (uint32_t) cbuf[j];
                    if (w.L >= ef && !(ed < w.d[ef - 1])) continue;
                    st = wlist_insert(w, ed, eid, ef, lane, low, nd);
                }
                if (lane == 0) ctl[2] = st;
            }
            __syncthreads();
            HB_CTA_PROF_MARK(3)
            if (ctl[2] != ST_OK) return ctl[2];
        }
    }
    HB_CTA_PROF_DUMP
    return ST_OK;
}

template <typename T, int IP, int NV>
__global__ void __launch_bounds__(CTA_WARPS * 32, 1) scan_cta_kernel(const ScanParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    float *q = reinterpret_cast<float *>(smem);
    unsigned char *s = smem + (size_t) g.nvec * Vec<T>::VEC * 4;
    WList w;
    w.d = reinterpret_cast<float *>(s);
    w.id = reinterpret_cast<uint32_t *>(s + (size_t) p.capW * 4);
    w.cap = p.capW;
    VisitedHash vs;
    vs.tab = reinterpret_cast<uint32_t *>(s + (size_t) p.capW * 8);
    vs.set_overflow(nullptr, 0);
    int32_t *cbuf = reinterpret_cast<int32_t *>(vs.tab + CTA_SLOTS);
    float *dbuf = reinterpret_cast<float *>(cbuf + 64);
    volatile int *ctl = reinterpret_cast<volatile int *>(dbuf + 64);

    for (int64_t qi = blockIdx.x; qi < p.nq; qi += gridDim.x) {
        __syncthreads();
        // every warp stages the query (same values): no barrier needed before each warp's own reads... but the other
        // warps read it too, so stage once and synchronise
        if (warp == 0) stage_query<T>(reinterpret_cast<const T *>(p.queries) + qi * g.dim, g.dim, g.nvec, q, lane);
        __syncthreads();
        QueryCounters ctr = { 0, 0, 0 };
        int st = ST_OK;
        w.L = 0;
        if (g.entry >= 0) {
            if (warp == 0) {
                const float d0 = one_distance<T, IP, NV>(g, q, g.entry, lane);
                ctr.n_dist = 1;
                if (lane == 0) { w.d[0] = d0; w.id[0] = (uint32_t) g.entry; }
            }
            w.L = 1;
            for (int lc = g.entry_level; lc >= 0 && st == ST_OK; lc--) {
                const int ef = lc == 0 ? p.ef : 1;
                vs.configure(lc == 0 ? CTA_SLOTS : 1024);
                __syncthreads();
                if (warp == 0) {
                    st = wlist_as_entries(w, vs, 1, lane);
                    if (lane == 0) { ctl[2] = st; ctl[4] = w.L; }
                }
                __syncthreads();
                st = ctl[2];
                w.L = ctl[4];
                if (st == ST_OK) st = search_layer_cta<T, IP, NV>(g, w, vs, q, cbuf, dbuf, ctl, ef, lc, lane, warp, ctr);
                // warp 0 owns the list: its length and the table's fill are what the other warps must agree on next round
                __syncthreads();
                if (warp == 0 && lane == 0) { ctl[4] = w.L; ctl[5] = vs.count; }
                __syncthreads();
                w.L = ctl[4];
                vs.count = ctl[5];
            }
        }
        if (st != ST_OK) {
            if (threadIdx.x == 0) {
                const int slot = atomicAdd(p.slow_count, 1);
                p.slow_list[slot] = (int32_t) qi;
                p.status[qi] = st;
            }
            continue;
        }
        const int cnt = min(w.L, p.ef);
        for (int j = threadIdx.x; j < p.out_stride; j += CTA_WARPS * 32) {
            p.out_elem[qi * p.out_stride + j] = j < cnt ? (int32_t) (w.id[j] & ID_MASK) : -1;
            p.out_dist[qi * p.out_stride + j] = j < cnt ? w.d[j] : __int_as_float(0x7f800000);
        }
        if (threadIdx.x == 0) {
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

// ---- the same, with the list in warp 0's registers and one expansion of look-ahead staged in shared memory ----------
// (ef + room for the tie tail <= 128 entries: scan_reg.cuh's RegW<4>.)  What a single scan waits for is, per expansion,
// a neighbour-list read, a row gather and the insertions.  Here warp 1 reads the list of the entry that will be expanded
// NEXT while the current rows are evaluated, and -- once the current distances are known and none of them overtakes that
// entry -- copies the rows of its not-yet-visited neighbours into shared memory (cp.async.bulk, one mbarrier phase per
// expansion), so that the next expansion finds its list and its rows on chip.  Only the source of the bytes changes: the
// expansion order, the per-row summation order and therefore ids, distances and counters are those of every other kernel.
struct CtaSmem {
    int32_t *cbuf, *cslot, *nlist;      // new candidates (ids | positions in the list), two buffers each | the next expansion's list
    float *dbuf, *td;                   // distances of the new candidates | RegW::insert_many scratch
    uint32_t *ti;
    volatile int *ctl;                  // 0 cid | 1 nnew | 2 status | 3 next | 4 list already filtered | 5 rows staged | 6 list tag | 8 row tag |
                                        // 9 parity | 11 next's distance | 12 filtered-ahead tag | 13 its nnew | 14 visited count
    uint64_t *mbar;
    char *rows;                         // 32 x row_bytes (row staging enabled) or nullptr
};

struct CtaLook { uint32_t issued; bool pending; };       // warp 1: row batches issued, last one not yet seen complete

__device__ __forceinline__ uint32_t cta_smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void cta_mbar_wait(uint64_t *bar, uint32_t parity)
{
    // bounded: a protocol error must end the kernel with an error, not hang the device
    for (int spin = 0; spin < (1 << 22); spin++) {
        uint32_t done;
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(cta_smem_u32(bar)), "r"(parity) : "memory");
        if (done) return;
    }
    __trap();
}

template <typename T> __host__ __device__ inline size_t scan_cta_reg_smem(int nvec, size_t row_bytes, bool stage_rows)
{
    // query | visited table | cbuf x2, cslot x2, nlist, dbuf (32 words each) | merge scratch (128 d | 128 id) | control words |
    // mbarrier | staged rows
    return (((size_t) nvec * Vec<T>::VEC * 4 + (size_t) CTA_SLOTS * 4 + 6 * 128 + 1024 + 64 + 16 + (stage_rows ? 32 * row_bytes : 0)) + 15) & ~(size_t) 15;
}

template <typename T, int IP, int NV, int R>
__device__ __forceinline__ int search_layer_cta_reg(const GraphView &g, RegW<R> &w, VisitedHash &vs, const float *q,
                                                    const CtaSmem &S, int ef, int lc, int lane, int warp,
                                                    QueryCounters &ctr, CtaLook &lk)
{
    const int deg = lc == 0 ? 2 * g.m : g.m;
    const bool look = lc == 0 && deg <= 32;         // look-ahead: layer 0, lists of one chunk
    const uint32_t row_bytes = (uint32_t) g.row_bytes;
    const unsigned lt_mask = (1u << lane) - 1u;
    volatile int *ctl = S.ctl;
    if (threadIdx.x == 0) { ctl[6] = -1; ctl[8] = -1; ctl[12] = -1; }      // nothing read ahead yet
    __syncthreads();
    HB_CTA_PROF_DECL
    for (int hop = 0;; hop++) {
        HB_CTA_PROF_MARK(4)
        const int pb = hop & 1;
        int32_t *cbuf = S.cbuf + 32 * pb, *cslot = S.cslot + 32 * pb;
        if (warp == 0) {
            // nearest unexpanded entry, and the one after it
            int mys = 0x7fffffff, mys2 = 0x7fffffff;
#pragma unroll
            for (int r = R - 1; r >= 0; r--)
                if (!(w.id[r] & EXP_BIT)) { mys2 = mys; mys = lane * R + r; }
            const unsigned b = __ballot_sync(FULL, mys != 0x7fffffff);
            int cid = -1, nxt = -1, pre = 0, nnew = 0, staged = 0;
            float nxd = 0.f;
            if (b) {
                const int src = __ffs(b) - 1;
                const int idx = __shfl_sync(FULL, mys, src);
                cid = (int) __shfl_sync(FULL, RegW<R>::pick(w.id, mys), src);
                int idx2 = __shfl_sync(FULL, mys2, src);
                const unsigned b2 = b & (b - 1);
                if (b2) idx2 = min(idx2, __shfl_sync(FULL, mys, __ffs(b2) - 1));
                if (look && idx2 != 0x7fffffff) { nxt = (int) w.get_id(idx2); nxd = w.get_d(idx2); }
#pragma unroll
                for (int r = 0; r < R; r++) if (lane * R + r == idx) w.id[r] |= EXP_BIT;
                if (lc == 0) ctr.n_hop0++; else ctr.n_hopu++;
                if (look && ctl[12] == cid) {
                    // the look-ahead warp already filtered this entry's list through the visited table (it was certain
                    // to be expanded next): its new candidates wait in this expansion's buffers
                    pre = 1;
                    nnew = ctl[13];
                    vs.added(nnew, false);
                    ctr.n_dist += nnew;
                    staged = ctl[8] == cid;
                }
            }
            HB_CTA_PROF_PRED(cid, nxt)
            if (lane == 0) {
                ctl[0] = cid; ctl[3] = nxt; ctl[11] = __float_as_int(nxd); ctl[4] = pre;
                ctl[1] = nnew; ctl[2] = ST_OK; ctl[5] = staged;
                if (pre) ctl[14] = vs.count;
            }
        }
        __syncthreads();
        HB_CTA_PROF_MARK(0)
        const int cid = ctl[0];
        if (cid < 0) break;
        const int nxt = ctl[3];
        const bool pre = ctl[4] != 0;
        const int32_t *list = lc == 0 ? g.nbr0 + (size_t) cid * deg : g.nbru + ((size_t) g.uoff[cid] + (lc - 1)) * g.m;
        int32_t look_nb = -1;              // warp 1: the next expansion's list, in flight until the distances are done
        for (int cb = 0; cb < deg; cb += 32) {
            if (warp == 1 && look && nxt >= 0 && cb == 0)
                look_nb = lane < deg ? __ldg(g.nbr0 + (size_t) nxt * deg + lane) : -1;
            if (!pre) {
                if (warp == 0) {
                    int st = ST_OK, nnew = 0, staged = 0;
                    if (cb == 0 && !vs.room(deg)) st = ST_TABLE;
                    if (st == ST_OK) {
                        const int i = cb + lane;
                        int32_t nb;
                        if (look && ctl[6] == cid) nb = S.nlist[lane];           // read ahead by the previous expansion
                        else nb = i < deg ? list[i] : -1;
                        bool isnew = false;
                        if (nb >= 0) isnew = vs.insert((uint32_t) nb, false);
                        const unsigned nmask = __ballot_sync(FULL, isnew);
                        if (isnew) {
                            const int j = __popc(nmask & lt_mask);
                            cbuf[j] = nb;
                            cslot[j] = lane;
                        }
                        nnew = __popc(nmask);
                        vs.added(nnew, false);
                        ctr.n_dist += nnew;
                        staged = look && ctl[8] == cid;
                    }
                    if (lane == 0) { ctl[1] = nnew; ctl[2] = st; ctl[5] = staged; ctl[14] = vs.count; }
                }
                __syncthreads();
            }
            HB_CTA_PROF_MARK(1)
            if (ctl[2] != ST_OK) return ctl[2];
            const int nnew = ctl[1];
            const bool staged = ctl[5] != 0;
            // distances: two candidates per warp and pass; the rows come from shared memory when they were staged
            if (staged && warp * 2 < nnew) cta_mbar_wait(S.mbar, (uint32_t) ctl[9]);
            for (int j0 = warp * 2; j0 < nnew; j0 += CTA_WARPS * 2) {
                if (j0 + 1 < nnew) {
                    float sd;
                    if (staged) {
                        const int32_t ids[2] = { cslot[j0], cslot[j0 + 1] };
                        sd = group_distance<T, IP, NV, 2, true>(S.rows, row_bytes, g.nvec, q, ids, lane);
                    } else {
                        const int32_t ids[2] = { cbuf[j0], cbuf[j0 + 1] };
                        sd = group_distance<T, IP, NV, 2>(g.vecs, row_bytes, g.nvec, q, ids, lane);
                    }
                    const float v1 = __shfl_sync(FULL, sd, 16);
                    if (lane == 0) { S.dbuf[j0] = sd; S.dbuf[j0 + 1] = v1; }
                } else {
                    float sd;
                    if (staged) {
                        const int32_t ids[1] = { cslot[j0] };
                        sd = group_distance<T, IP, NV, 1, true>(S.rows, row_bytes, g.nvec, q, ids, lane);
                    } else {
                        const int32_t ids[1] = { cbuf[j0] };
                        sd = group_distance<T, IP, NV, 1>(g.vecs, row_bytes, g.nvec, q, ids, lane);
                    }
                    if (lane == 0) S.dbuf[j0] = sd;
                }
            }
            __syncthreads();
            HB_CTA_PROF_MARK(2)
            if (warp == 0) {
                // admit and insert in neighbour order, as the sequential loop does (several at once when that is the same)
                const float myd = lane < nnew ? S.dbuf[lane] : __int_as_float(0x7f800000);
                const uint32_t cj = lane < nnew ? (uint32_t) cbuf[lane] : 0u;
                unsigned amask = __ballot_sync(FULL, lane < nnew && (w.L < ef || myd < w.f));
                int st = ST_OK;
                if (amask & (amask - 1)) {
                    if (w.insert_many(myd, cj, amask, ef, lane, S.td, S.ti) == ST_OK) amask = 0;
                }
                while (amask && st == ST_OK) {
                    const int sl = __ffs(amask) - 1;
                    amask &= amask - 1;
                    const float ed = __shfl_sync(FULL, myd, sl);
                    const uint32_t eid = __shfl_sync(FULL, cj, sl);
                    if (w.L >= ef && !(ed < w.f)) continue;
                    st = w.insert(ed, eid, ef, lane);
                }
                if (lane == 0) ctl[2] = st;
            } else if (warp == 1 && look && cb == 0) {
                // Will the entry read ahead really be expanded next?  Yes unless a candidate just evaluated sorts before it
                // (W is ordered by (distance, id); entries inserted behind it cannot evict it).  Then its expansion is
                // certain, and its list can be filtered through the visited table now -- warp 0 only touches registers
                // in this phase -- and the rows of its new candidates copied into shared memory.
                // (the list read ahead is first needed here: waiting for it next to warp 0's insertions costs nothing, at the end
                // of the distance phase it held up all four warps -- profiles/r2_cta_reg_ncu_summary.txt)
                S.nlist[lane] = look_nb;
                if (lane == 0) ctl[6] = nxt;
                bool go = nxt >= 0;
                if (go) {
                    const float nxd = __int_as_float(ctl[11]);
                    const float myd = lane < nnew ? S.dbuf[lane] : __int_as_float(0x7f800000);
                    const bool first = lane < nnew && (myd < nxd || (myd == nxd && (uint32_t) cbuf[lane] < (uint32_t) nxt));
                    go = !__any_sync(FULL, first);
                }
                if (go && ctl[14] + deg <= vs.limit) {
                    const bool need = look_nb >= 0 && vs.insert((uint32_t) look_nb, false);
                    const unsigned nm = __ballot_sync(FULL, need);
                    const int cnt = __popc(nm);
                    if (need) {
                        const int j = __popc(nm & lt_mask);
                        S.cbuf[32 * (pb ^ 1) + j] = look_nb;
                        S.cslot[32 * (pb ^ 1) + j] = lane;
                    }
                    bool staged_next = false;
                    if (S.rows != nullptr && cnt) {
                        if (lk.pending) { cta_mbar_wait(S.mbar, (lk.issued - 1u) & 1u); lk.pending = false; }
                        if (lane == 0) {
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                                         ::"r"(cta_smem_u32(S.mbar)), "r"((uint32_t) cnt * row_bytes) : "memory");
                        }
                        __syncwarp();
                        if (need)
                            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                         ::"r"(cta_smem_u32(S.rows + (size_t) lane * row_bytes)),
                                           "l"(g.vecs + (size_t) (uint32_t) look_nb * row_bytes), "r"(row_bytes),
                                           "r"(cta_smem_u32(S.mbar)) : "memory");
                        if (lane == 0) ctl[9] = (int) (lk.issued & 1u);
                        lk.issued++;
                        lk.pending = true;
                        staged_next = true;
                    }
                    if (lane == 0) { ctl[12] = nxt; ctl[13] = cnt; ctl[8] = staged_next ? nxt : -1; }
                } else if (lane == 0) { ctl[12] = -1; ctl[8] = -1; }
            }
            __syncthreads();
            HB_CTA_PROF_MARK(3)
            if (ctl[2] != ST_OK) return ctl[2];
        }
    }
    HB_CTA_PROF_DUMP
    return ST_OK;
}

template <typename T, int IP, int NV, int R>
__global__ void __launch_bounds__(CTA_WARPS * 32, 1) scan_cta_reg_kernel(const ScanParams p, int stage_rows)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const GraphView &g = p.g;
    float *q = reinterpret_cast<float *>(smem);
    VisitedHash vs;
    vs.tab = reinterpret_cast<uint32_t *>(smem + (size_t) g.nvec * Vec<T>::VEC * 4);
    vs.set_overflow(nullptr, 0);
    CtaSmem S;
    S.cbuf = reinterpret_cast<int32_t *>(vs.tab + CTA_SLOTS);
    S.cslot = S.cbuf + 64;
    S.nlist = S.cslot + 64;
    S.dbuf = reinterpret_cast<float *>(S.nlist + 32);
    S.td = S.dbuf + 32;
    S.ti = reinterpret_cast<uint32_t *>(S.td + 128);
    S.ctl = reinterpret_cast<volatile int *>(S.ti + 128);
    S.mbar = reinterpret_cast<uint64_t *>(const_cast<int *>(S.ctl) + 16);
    S.rows = stage_rows ? reinterpret_cast<char *>(S.mbar + 2) : nullptr;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(cta_smem_u32(S.mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    RegW<R> w;                          // warp 0's; the other warps never read theirs
    CtaLook lk = { 0u, false };
    const int ef = p.ef;

    for (int64_t qi = blockIdx.x; qi < p.nq; qi += gridDim.x) {
        __syncthreads();
        if (warp == 0) stage_query<T>(reinterpret_cast<const T *>(p.queries) + qi * g.dim, g.dim, g.nvec, q, lane);
        __syncthreads();
        QueryCounters ctr = { 0, 0, 0 };
        int st = ST_OK;
        w.reset();
        if (g.entry >= 0) {
            if (warp == 0) {
                const float d0 = one_distance<T, IP, NV>(g, q, g.entry, lane);
                ctr.n_dist = 1;
                if (lane == 0) { w.d[0] = d0; w.id[0] = (uint32_t) g.entry; }
                w.L = 1;
            }
            for (int lc = g.entry_level; lc >= 0 && st == ST_OK; lc--) {
                const int efl = lc == 0 ? ef : 1;
                vs.configure(lc == 0 ? CTA_SLOTS : 1024);
                __syncthreads();                       // nobody still reads the previous layer's table
                if (warp == 0) {
                    st = regw_as_entry(w, vs, efl, lane);
                    if (lane == 0) S.ctl[2] = st;
                }
                __syncthreads();
                st = S.ctl[2];
                if (st == ST_OK) st = search_layer_cta_reg<T, IP, NV, R>(g, w, vs, q, S, efl, lc, lane, warp, ctr, lk);
            }
        }
        if (st != ST_OK) {
            if (threadIdx.x == 0) {
                const int slot = atomicAdd(p.slow_count, 1);
                p.slow_list[slot] = (int32_t) qi;
                p.status[qi] = st;
            }
            continue;
        }
        if (warp == 0) {
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
    // no copy may still be in flight towards this CTA's shared memory when it exits
    if (warp == 1 && lk.pending) cta_mbar_wait(S.mbar, (lk.issued - 1u) & 1u);
}

template <typename T, int IP, int NV>
cudaError_t launch_scan_cta_variant(const ScanParams &p, int num_sms, cudaStream_t stream)
{
    int grid = (int) (p.nq < (int64_t) num_sms * 2 ? p.nq : (int64_t) num_sms * 2);
    if (grid < 1) grid = 1;
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 15;
    if (p.variant != SCAN_CTA_SMEM_LIST && p.ef + 24 <= 128 && p.out_stride <= 128) {
        auto kern = scan_cta_reg_kernel<T, IP, NV, 4>;
        const bool stage = p.variant != SCAN_CTA_NO_STAGE && 2 * p.g.m <= 32 && scan_cta_reg_smem<T>(p.g.nvec, p.g.row_bytes, true) <= 200 * 1024;
        const size_t smem = scan_cta_reg_smem<T>(p.g.nvec, p.g.row_bytes, stage);
        static thread_local size_t seen_reg[16];
        if (seen_reg[dev] < smem) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
            if (e != cudaSuccess) return e;
            seen_reg[dev] = smem;
        }
        kern<<<grid, CTA_WARPS * 32, smem, stream>>>(p, stage ? 1 : 0);
        return cudaGetLastError();
    }
    auto kern = scan_cta_kernel<T, IP, NV>;
    const size_t smem = scan_cta_smem<T>(p.g.nvec, p.capW);
    static thread_local size_t seen[16];
    if (seen[dev] < smem) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (e != cudaSuccess) return e;
        seen[dev] = smem;
    }
    kern<<<grid, CTA_WARPS * 32, smem, stream>>>(p);
    return cudaGetLastError();
}

// batches small enough that the GPU is mostly idle: one CTA per query (shared memory must hold the list and the table)
inline bool use_cta_scan(const ScanParams &p, int num_sms, size_t row_smem_bytes, const void *ep, int variant)
{
    if (ep != nullptr || variant == SCAN_SMEM_LIST || variant == SCAN_NO_CTA) return false;
    if (p.nq > num_sms) return false;
    const bool forced = variant == SCAN_CTA || variant == SCAN_CTA_SMEM_LIST || variant == SCAN_CTA_NO_STAGE;
    // measured (profiles/r2_experiments.md): rows of 3 KB gain 15-20 % at 32..148 queries; rows of 512 B lose 15-25 %
    // to the register-list kernel, whose hop is shorter than this kernel's three block barriers.  SCAN_CTA forces it.
    if (p.g.nvec < 96 && !forced) return false;
    return row_smem_bytes + (size_t) p.capW * 8 + (size_t) CTA_SLOTS * 4 + 1024 <= 200 * 1024;
}

template <typename T, int IP>
cudaError_t launch_scan_cta_t(const ScanParams &p, int num_sms, cudaStream_t stream)
{
    switch (nv_of(p.g.nvec)) {
#define HB_CCASE(NVV, GG, MB) case NVV: return launch_scan_cta_variant<T, IP, NVV>(p, num_sms, stream);
        HB_NV_TABLE(HB_CCASE)
#undef HB_CCASE
    default: return launch_scan_cta_variant<T, IP, 0>(p, num_sms, stream);
    }
}

}   // namespace hb
