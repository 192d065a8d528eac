// build.cu -- host orchestration of the batched insert pipeline (hnswbuild.c InsertTupleInMemory /
// UpdateGraphInMemory / UpdateNeighborsInMemory, hnswutils.c HnswFindElementNeighbors
// [RECALL; reference mount empty, /root/reference/README.md:1]).
//
// Per batch, all on one stream with no host round trip in between (the rows of the NEXT batch are
// uploaded meanwhile on a second stream):
//   build_search_kernel (candidates per layer, SelectNeighbors fused in, duplicate detection; every
//   distance it evaluates is logged) -> eval_table_build_kernel (logs -> per-element hash tables)
//   -> build_check_kernel -> build_commit_kernel (AddConnections) -> edge_gen_kernel (reverse links as
//   sortable keys) -> radix sort by (layer, target, source) -> seg_heads_kernel -> fill_list_kernel +
//   link_pipe_kernel in fill mode (pair caches of lists shrunk for the first time) -> link_memo_kernel
//   (HnswUpdateConnection; link_kernel.cuh, build_kernel.cuh).
// The host assumes the batch holds no duplicate of an indexed vector (ids = arrival order) and
// reads one flag word back per batch; when the check kernel found a duplicate the kernels after it
// did nothing, the host folds the duplicates (FindDuplicateInMemory, <= 10 heap TIDs per element),
// renumbers and re-runs the tail.  The host only moves bookkeeping integers; every distance is
// evaluated on the GPU.  A batch is at most 1/16 of the current graph (8192, 16384 from 512k
// elements), and an element that would raise the entry level is inserted alone.
#include "index.h"
#include "build_kernel.cuh"
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <tuple>

namespace hb {

#define HB_DECLB(name)                                                                                   \
    cudaError_t build_search_##name(const BuildSearchParams &, int, int, cudaStream_t, bool slow);       \
    cudaError_t build_select_##name(const BuildSelectParams &, int, cudaStream_t);                       \
    cudaError_t build_link_##name(const LinkParams &, int, int, cudaStream_t);                            \
    cudaError_t pair_fill_##name(const LinkParams &, int, int, cudaStream_t);                           \
    cudaError_t nbr_dist_##name(const NbrDistParams &, int, cudaStream_t);
HB_DECLB(f32_l2) HB_DECLB(f32_ip) HB_DECLB(f16_l2) HB_DECLB(f16_ip) HB_DECLB(f32_l1) HB_DECLB(f16_l1)
#undef HB_DECLB

#define HB_PICK(fn, ix)                                                                                   \
    ((ix)->dtype == HB_F32 ? (metric_kind((ix)->metric) == 2 ? fn##_f32_l1 : metric_kind((ix)->metric) == 1 ? fn##_f32_ip : fn##_f32_l2) \
                           : (metric_kind((ix)->metric) == 2 ? fn##_f16_l1 : metric_kind((ix)->metric) == 1 ? fn##_f16_ip : fn##_f16_l2))

template <typename T>
__global__ void normalize_rows_kernel(const T *__restrict__ in, char *__restrict__ out_rows, size_t row_bytes,
                                      int64_t n, int dim);

// l2_normalize (canonical order, see api.cu normalize_kernel) writing into padded rows
template <typename T>
__global__ void normalize_rows_kernel(const T *__restrict__ in, char *__restrict__ out_rows, size_t row_bytes,
                                      int64_t n, int dim)
{
    constexpr int VEC = Vec<T>::VEC;
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t) blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= n) return;
    const T *src = in + row * dim;
    double acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; k++) acc[k] = 0.0;
    const int nch = (dim + VEC - 1) / VEC;
    for (int ch = lane; ch < nch; ch += 32) {
#pragma unroll
        for (int k = 0; k < VEC; k++) {
            const int e = ch * VEC + k;
            if (e < dim) {
                const double x = (double) (float) src[e];
                acc[k] = acc[k] + x * x;
            }
        }
    }
    double s;
    if constexpr (VEC == 4) s = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    else s = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
    for (int b = 16; b >= 1; b >>= 1) s = s + __shfl_xor_sync(FULL, s, b);
    const double norm = sqrt(s);
    T *dst = reinterpret_cast<T *>(out_rows + row * row_bytes);
    const int padded = (int) (row_bytes / sizeof(T));
    for (int e = lane; e < padded; e += 32) {
        float y = 0.f;
        if (e < dim) {
            const float x = (float) src[e];
            y = norm > 0.0 ? (float) ((double) x / norm) : x;
        }
        dst[e] = (T) y;
    }
}

void release_pair_cache(hb_index *ix)
{
    cudaFree(ix->d_pc0); cudaFree(ix->d_pcu); cudaFree(ix->d_pv0); cudaFree(ix->d_pvu);
    ix->d_pc0 = ix->d_pcu = nullptr; ix->d_pv0 = ix->d_pvu = nullptr;
    ix->pair_cache_tried = false;
}

// the pair cache costs lm0(lm0-1)/2 floats per element (2 kB at m = 16): taken only when it fits in a
// third of the free memory
static int ensure_pair_cache(hb_index *ix)
{
    if (ix->pair_cache_tried) return HB_OK;
    ix->pair_cache_tried = true;
    const int lm0 = 2 * ix->m;
    if (!ix->opt_pair_cache || lm0 > LINK_MAX_LM) return HB_OK;
    const size_t b0 = sizeof(float) * (size_t) ix->cap * (lm0 * (lm0 - 1) / 2);
    const size_t bu = sizeof(float) * (size_t) ix->upper_cap * (ix->m * (ix->m - 1) / 2);
    size_t free_b = 0, total_b = 0;
    HB_CK(cudaMemGetInfo(&free_b, &total_b));
    if (b0 + bu > free_b / 3) return HB_OK;
    HB_CK(cudaMalloc(&ix->d_pc0, b0));
    HB_CK(cudaMalloc(&ix->d_pcu, bu));
    HB_CK(cudaMalloc(&ix->d_pv0, ix->cap));
    HB_CK(cudaMalloc(&ix->d_pvu, ix->upper_cap));
    HB_CK(cudaMemset(ix->d_pv0, 0, ix->cap));
    HB_CK(cudaMemset(ix->d_pvu, 0, ix->upper_cap));
    return HB_OK;
}

static int ensure_build_arrays(hb_index *ix, cudaStream_t s)
{
    {
        const int rc = ensure_pair_cache(ix);
        if (rc) return rc;
    }
    if (ix->d_nbr0d) return HB_OK;
    const int m2 = 2 * ix->m;
    HB_CK(cudaMalloc(&ix->d_nbr0d, sizeof(float) * ix->cap * m2));
    HB_CK(cudaMalloc(&ix->d_nbrud, sizeof(float) * ix->upper_cap * ix->m));
    if (ix->n == 0) return HB_OK;
    // the graph was loaded: recompute the cached owner->neighbour distances
    NbrDistParams p;
    p.g = ix->view(); p.rows = ix->n; p.deg = m2; p.owner_of_row = nullptr; p.nbr = ix->d_nbr0; p.nbrd = ix->d_nbr0d;
    HB_CK(HB_PICK(nbr_dist, ix)(p, ix->num_sms, s));
    if (ix->upper_rows > 0) {
        std::vector<int32_t> uoff(ix->n), owner(ix->upper_rows, 0);
        HB_CK(cudaMemcpy(uoff.data(), ix->d_uoff, sizeof(int32_t) * ix->n, cudaMemcpyDeviceToHost));
        for (int64_t e = 0; e < ix->n; e++)
            for (int l = 0; l < ix->h_level[e]; l++) owner[uoff[e] + l] = (int32_t) e;
        HB_CK(ix->ws_build[11].ensure(sizeof(int32_t) * ix->upper_rows));
        HB_CK(cudaMemcpyAsync(ix->ws_build[11].p, owner.data(), sizeof(int32_t) * ix->upper_rows, cudaMemcpyHostToDevice, s));
        p.rows = ix->upper_rows; p.deg = ix->m; p.owner_of_row = ix->ws_build[11].as<int32_t>();
        p.nbr = ix->d_nbru; p.nbrd = ix->d_nbrud;
        HB_CK(HB_PICK(nbr_dist, ix)(p, ix->num_sms, s));
        HB_CK(cudaStreamSynchronize(s));
    }
    return HB_OK;
}

static bool all_zero(const char *row, size_t bytes, int esize)
{
    // a vector has zero norm iff every component is +-0 (squares of fp32/fp16 values do not
    // underflow in double)
    if (esize == 4) {
        const uint32_t *w = reinterpret_cast<const uint32_t *>(row);
        for (size_t i = 0; i < bytes / 4; i++) if (w[i] & 0x7fffffffu) return false;
    } else {
        const uint16_t *w = reinterpret_cast<const uint16_t *>(row);
        for (size_t i = 0; i < bytes / 2; i++) if (w[i] & 0x7fffu) return false;
    }
    return true;
}

// ---- small kernels of the batch tail (no distances here) ---------------------------------------
// flag bit 0: an insert hit the tie limit (error); bit 1: a new row is byte-identical to a neighbour
static __global__ void build_check_kernel(const int32_t *__restrict__ status, const int32_t *__restrict__ dup, int B,
                                          int32_t *flag)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    int f = 0;
    if (status[i] < 0) f |= 1;
    if (dup[(size_t) i * DUP_SLOTS] >= 0) f |= 2;
    if (f) atomicOr(flag, f);
}

constexpr int BUILD_SLOW_GRID = 16;

struct EdgeGenParams {
    int B, UR, m;
    int64_t first;
    const int32_t *final_id;        // B
    const int32_t *urow_owner;      // UR: batch index of the element owning upper candidate row r
    const int32_t *urow_layer;      // UR
    const int32_t *sel0_id; const float *sel0_d; const int32_t *sel0_cnt;
    const int32_t *selu_id; const float *selu_d; const int32_t *selu_cnt;
    unsigned long long *key; float *val;
    const int32_t *flag;
};

// one thread per selected-neighbour slot: the reverse link (layer, target = neighbour, source = new element)
static __global__ void edge_gen_kernel(const EdgeGenParams p)
{
    if (*p.flag) return;
    const int lm0 = 2 * p.m;
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n0 = (int64_t) p.B * lm0, total = n0 + (int64_t) p.UR * p.m;
    if (t >= total) return;
    unsigned long long key = LINK_KEY_INVALID;
    float d = 0.f;
    if (t < n0) {
        const int i = (int) (t / lm0), j = (int) (t % lm0);
        const int32_t f = p.final_id[i];
        if (f >= 0 && j < p.sel0_cnt[i]) {
            key = ((unsigned long long) (uint32_t) p.sel0_id[t] << LINK_KEY_SRC_BITS) | (unsigned long long) (f - p.first);
            d = p.sel0_d[t];
        }
    } else {
        const int64_t u = t - n0;
        const int r = (int) (u / p.m), j = (int) (u % p.m);
        const int32_t f = p.final_id[p.urow_owner[r]];
        if (f >= 0 && j < p.selu_cnt[r]) {
            key = ((unsigned long long) p.urow_layer[r] << (32 + LINK_KEY_SRC_BITS)) |
                  ((unsigned long long) (uint32_t) p.selu_id[u] << LINK_KEY_SRC_BITS) | (unsigned long long) (f - p.first);
            d = p.selu_d[u];
        }
    }
    p.key[t] = key;
    p.val[t] = d;
}

// segment = run of sorted edges with the same (layer, target); order of the segment list is free
static __global__ void seg_heads_kernel(const unsigned long long *__restrict__ key, int E, int32_t *seg_start,
                                        int32_t *nseg, const int32_t *flag)
{
    if (*flag) return;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const unsigned long long k = key[e];
    if (k == LINK_KEY_INVALID) return;
    if (e + 1 == E || key[e + 1] == LINK_KEY_INVALID) nseg[1] = e + 1;      // number of valid edges
    if (e == 0 || (key[e - 1] >> LINK_KEY_SRC_BITS) != (k >> LINK_KEY_SRC_BITS)) seg_start[atomicAdd(nseg, 1)] = e;
}

// evaluated-distance logs -> hash tables (search_core.cuh EvalTable), one warp per new element
static __global__ void eval_table_build_kernel(const uint32_t *__restrict__ el_id, const float *__restrict__ el_d,
                                               const int32_t *__restrict__ el_n, int el_cap, int B, uint32_t *et_key,
                                               float *et_val, int et_slots)
{
    const int lane = threadIdx.x & 31;
    const int i = (int) (((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (i >= B) return;
    EvalTable et;
    et.key = et_key + (size_t) i * et_slots; et.val = et_val + (size_t) i * et_slots; et.mask = (uint32_t) et_slots - 1u;
    const int n = el_n[i];
    for (int e = lane; e < n; e += 32) et.put(el_id[(size_t) i * el_cap + e], el_d[(size_t) i * el_cap + e], true);
}

// lists that this batch will shrink and whose pair cache is still unfilled: (layer << 32 | target)
static __global__ void fill_list_kernel(const unsigned long long *__restrict__ key, const int32_t *__restrict__ seg_start,
                                        const int32_t *__restrict__ nseg, int m, const int32_t *__restrict__ nbr0,
                                        const int32_t *__restrict__ uoff, const int32_t *__restrict__ nbru,
                                        const uint8_t *__restrict__ pv0, const uint8_t *__restrict__ pvu,
                                        unsigned long long *fill_list, int32_t *nfill, const int32_t *flag)
{
    if (*flag) return;
    const int sgm = blockIdx.x * blockDim.x + threadIdx.x;
    if (sgm >= *nseg) return;
    const unsigned long long key0 = key[seg_start[sgm]] >> LINK_KEY_SRC_BITS;
    const int lc = (int) (key0 >> 32);
    const int32_t target = (int32_t) (key0 & 0xffffffffu);
    bool want;
    if (lc == 0) want = pv0[target] == 0 && nbr0[(size_t) target * 2 * m + 2 * m - 1] >= 0;
    else {
        const size_t row = (size_t) uoff[target] + (lc - 1);
        want = pvu[row] == 0 && nbru[row * m + m - 1] >= 0;
    }
    if (want) fill_list[atomicAdd(nfill, 1)] = key0;
}

// AddConnections plus the per-element words of the new elements (uoff, first heap TID)
struct CommitParams {
    int B, UR, m;
    const int32_t *final_id;      // B: element id, or -1 for a tuple folded into a duplicate
    const int32_t *new_uoff;      // B
    const int64_t *tid;           // B
    const int32_t *dest_urow;     // UR: row in nbru, or -1
    const int32_t *sel0_id; const float *sel0_d;
    const int32_t *selu_id; const float *selu_d;
    int32_t *nbr0; float *nbr0d; int32_t *nbru; float *nbrud;
    int32_t *uoff; int64_t *tid0; uint8_t *ntids;
    uint8_t *pv0, *pvu;           // pair-cache filled flags (NULL without the cache): new lists start unfilled
    const int32_t *flag;
};

static __global__ void build_commit_kernel(const CommitParams p)
{
    if (*p.flag) return;
    const int lm0 = 2 * p.m;
    const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n0 = (int64_t) p.B * lm0;
    if (t < n0) {
        const int i = (int) (t / lm0), j = (int) (t % lm0);
        const int32_t f = p.final_id[i];
        if (f >= 0) {
            p.nbr0[(size_t) f * lm0 + j] = p.sel0_id[t]; p.nbr0d[(size_t) f * lm0 + j] = p.sel0_d[t];
            if (j == 0) { p.uoff[f] = p.new_uoff[i]; p.tid0[f] = p.tid[i]; p.ntids[f] = 1; if (p.pv0) p.pv0[f] = 0; }
        }
    } else if (t < n0 + (int64_t) p.UR * p.m) {
        const int64_t u = t - n0;
        const int r = (int) (u / p.m), j = (int) (u % p.m);
        const int32_t dr = p.dest_urow[r];
        if (dr >= 0) {
            p.nbru[(size_t) dr * p.m + j] = p.selu_id[u]; p.nbrud[(size_t) dr * p.m + j] = p.selu_d[u];
            if (j == 0 && p.pvu) p.pvu[dr] = 0;
        }
    }
}

template <typename V> static inline V *carve(char *&p, size_t count)
{
    V *r = reinterpret_cast<V *>(p);
    p += (count * sizeof(V) + 15) & ~(size_t) 15;
    return r;
}

int64_t build_insert(hb_index *ix, const void *host_vecs, int64_t n_in, const int64_t *heap_tids)
{
    if (n_in == 0) return 0;
    const double t_enter = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    HB_CK(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const size_t src_row = (size_t) ix->dim * ix->esize;
    const int m = ix->m, m2 = 2 * m, efc = ix->efc;

    // tuples to index, in order (HnswCheckNorm drops zero-norm vectors under the cosine opclass)
    std::vector<int64_t> todo;
    todo.reserve(n_in);
    for (int64_t i = 0; i < n_in; i++) {
        if (ix->metric == HB_COSINE && all_zero((const char *) host_vecs + i * src_row, src_row, ix->esize)) continue;
        todo.push_back(i);
    }
    if (ix->n + (int64_t) todo.size() > ix->cap) {
        if (!ix->opt_auto_grow) {
            set_error("index capacity %lld exceeded (%lld + %lld)", (long long) ix->cap, (long long) ix->n, (long long) todo.size());
            return HB_ENOMEM;
        }
        // a pgvector index has no capacity: grow (at least by half, so that single-row inserts do not regrow every time)
        const int64_t want = std::max<int64_t>(ix->n + (int64_t) todo.size(), ix->cap + ix->cap / 2 + 1024);
        const int grc = hb_index_reserve(ix, want);
        if (grc) return grc;
    }
    const double t_todo = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    int rc = ensure_build_arrays(ix, s);
    if (rc) return rc;
    const double t_arrays = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    ix->h_level.reserve(ix->n + todo.size());
    ix->h_ntids.reserve(ix->n + todo.size());
    ix->h_tids.reserve((ix->n + todo.size()) * HB_HEAPTIDS);
    if (!ix->h_flag) HB_CK(cudaMallocHost(&ix->h_flag, 16));

    // HB_BUILD_TRACE=1: where the host's wall time goes (enqueue vs waiting for the device)
    const bool trace = getenv("HB_BUILD_TRACE") != nullptr;
    double t_prep = 0, t_wait = 0, t_post = 0;
    int64_t n_batches = 0, n_segs = 0, n_edges = 0;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_begin = now();
    cudaEvent_t tev[5] = { nullptr, nullptr, nullptr, nullptr, nullptr };
    double t_dev[4] = { 0, 0, 0, 0 };   // upload+search | select | commit+edges+sort | link
    if (trace) for (auto &e : tev) HB_CK(cudaEventCreate(&e));

    // automatic batch cap: 8192 rows.  16384 once the graph holds 512k elements built 1M x 768 4 % faster but cost recall
    // against the sequentially built graph (10 000 queries, paired: -0.56 / -0.69 pt at ef_search 40 / 90 with 16384,
    // -0.30 / -0.39 pt with 8192; smaller caps bring nothing more: profiles/r2_build_recall_1m.txt)
    const int max_batch = std::min(ix->opt_build_batch > 0 ? ix->opt_build_batch : 8192, 1 << LINK_KEY_SRC_BITS);
    int64_t indexed = 0;
    size_t pos = 0;
    std::vector<char> stage, pack;
    std::vector<uint8_t> levels;
    std::vector<int32_t> ucand_row, dup;

    // workspaces are sized once for the largest batch this call can form (cudaFree inside the
    // loop would stall the pipeline); a batch with unusually many upper-layer rows regrows them
    // evaluated-distance table per new element: 32 x ef_construction slots (2048 at 64), 8 bytes each
    int et_slots = 1;
    while (et_slots < 32 * efc) et_slots <<= 1;
    auto size_workspaces = [&](int64_t b, int64_t UR1) -> int {
        hb::DevBuf *W = ix->ws_build;
        const int64_t E = b * m2 + UR1 * m;
        HB_CK(W[1].ensure(((size_t) 3 * b + 3 * UR1) * 4 + (size_t) b * 9 + 256));   // packed bookkeeping words
        HB_CK(W[3].ensure((size_t) b * efc * 8 + sizeof(int32_t) * b));       // cand0 id | d | cnt
        HB_CK(W[4].ensure((size_t) UR1 * efc * 8 + sizeof(int32_t) * UR1));
        HB_CK(W[5].ensure((size_t) b * m2 * 8 + sizeof(int32_t) * b));        // sel0 id | d | cnt
        HB_CK(W[6].ensure((size_t) UR1 * m * 8 + sizeof(int32_t) * UR1));     // selu id | d | cnt
        HB_CK(W[7].ensure(sizeof(int32_t) * b * DUP_SLOTS));
        HB_CK(W[8].ensure(sizeof(int32_t) * b * 2 + 64));                     // status | slow list
        HB_CK(W[9].ensure((size_t) E * (8 + 8 + 4 + 4 + 4 + 8) + 256));       // keys in/out | vals in/out | seg_start | fill list
        if (ix->opt_eval_table) HB_CK(W[2].ensure((size_t) b * et_slots * 16 + (size_t) b * 4));   // evaluated-distance tables (keys | values) | logs (ids | distances) | counts
        HB_CK(ix->ws_misc.ensure(256));
        return HB_OK;
    };
    {
        const int64_t bmax = std::min<int64_t>(max_batch, std::max<int64_t>(1, std::min<int64_t>((int64_t) todo.size(), (ix->n + (int64_t) todo.size()) / std::max(2, ix->opt_build_fraction))));
        rc = size_workspaces(bmax, std::max<int64_t>(bmax / 4, 64));
        if (rc) return rc;
        size_t sort_bytes = 0;
        HB_CK(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (unsigned long long *) nullptr, (unsigned long long *) nullptr,
                                              (float *) nullptr, (float *) nullptr, (int) (bmax * m2 + std::max<int64_t>(bmax / 4, 64) * m), 0, 64, s));
        HB_CK(ix->ws_build[10].ensure(sort_bytes + 16));
        // large-visited-set path of the candidate search: bitmaps sized for the final graph
        const int64_t slow_warps = (int64_t) BUILD_SLOW_GRID * BUILD_WARPS;
        HB_CK(ix->ws_gbits.ensure(sizeof(uint32_t) * slow_warps * ((ix->n + (int64_t) todo.size() + 31) / 32 + 2)));
    }

    // Rows are uploaded (and normalised under the cosine opclass) AHEAD of the batch that indexes
    // them, on a second stream, while the previous batch's kernels run: todo row t goes to slot
    // slot_base + t, which holds as long as no tuple folds into a duplicate (the duplicate path
    // re-bases and re-uploads).  The host blocks in the pageable-memory copy, the device does not.
    if (!ix->up_stream) HB_CK(cudaStreamCreateWithFlags(&ix->up_stream, cudaStreamNonBlocking));
    if (!ix->up_event) HB_CK(cudaEventCreateWithFlags(&ix->up_event, cudaEventDisableTiming));
    cudaStream_t up = ix->up_stream;
    cudaEvent_t up_ev = ix->up_event;
    int64_t uploaded = 0;                    // todo rows [0, uploaded) are in HBM or on their way
    int64_t slot_base = ix->n;
    const int64_t up_chunk = 16384;
    // the upload stream must not run ahead of whatever used these slots before this call
    HB_CK(cudaEventRecord(up_ev, s));
    HB_CK(cudaStreamWaitEvent(up, up_ev, 0));
    auto upload_upto = [&](int64_t want) -> int {
        want = std::min<int64_t>(want, (int64_t) todo.size());
        while (uploaded < want) {
            const int64_t c = std::min<int64_t>(std::min<int64_t>(up_chunk, max_batch), (int64_t) todo.size() - uploaded);
            const char *src = (const char *) host_vecs + todo[uploaded] * src_row;
            if (todo[uploaded + c - 1] - todo[uploaded] != c - 1) {       // a zero vector was skipped inside the chunk
                stage.resize((size_t) c * src_row);
                for (int64_t i = 0; i < c; i++) memcpy(&stage[i * src_row], (const char *) host_vecs + todo[uploaded + i] * src_row, src_row);
                src = stage.data();
            }
            char *rows = ix->d_vecs + (size_t) (slot_base + uploaded) * ix->row_bytes;
            if (ix->metric == HB_COSINE) {
                HB_CK(ix->ws_build[0].ensure((size_t) c * src_row));
                HB_CK(cudaMemcpyAsync(ix->ws_build[0].p, src, (size_t) c * src_row, cudaMemcpyHostToDevice, up));
                const int wpb = 8, grid = (int) ((c + wpb - 1) / wpb);
                if (ix->dtype == HB_F32)
                    normalize_rows_kernel<float><<<grid, wpb * 32, 0, up>>>(ix->ws_build[0].as<float>(), rows, ix->row_bytes, c, ix->dim);
                else
                    normalize_rows_kernel<__half><<<grid, wpb * 32, 0, up>>>(ix->ws_build[0].as<__half>(), rows, ix->row_bytes, c, ix->dim);
                HB_CK(cudaGetLastError());
            } else if (src_row == ix->row_bytes) {
                HB_CK(cudaMemcpyAsync(rows, src, src_row * c, cudaMemcpyHostToDevice, up));
            } else {
                HB_CK(cudaMemsetAsync(rows, 0, ix->row_bytes * c, up));
                HB_CK(cudaMemcpy2DAsync(rows, ix->row_bytes, src, src_row, src_row, c, cudaMemcpyHostToDevice, up));
            }
            uploaded += c;
        }
        HB_CK(cudaEventRecord(up_ev, up));
        return HB_OK;
    };

    const int64_t final_size = ix->n + (int64_t) todo.size();
    while (pos < todo.size()) {
        const double t0 = now();
        n_batches++;
        const int64_t cur = ix->n;
        // the latency-bound start-up: while the graph is small a batch may be 1/8 of it when the whole build stays small (recall of
        // such graphs is insensitive to it: profiles/r2_experiments.md), 1/16 otherwise
        const int frac_small = ix->opt_build_fraction_small > 0 ? ix->opt_build_fraction_small : (final_size < 262144 ? 8 : ix->opt_build_fraction);
        const int frac = cur < 65536 ? std::max(2, frac_small) : std::max(2, ix->opt_build_fraction);
        int64_t b = std::max<int64_t>(1, std::min<int64_t>(max_batch, cur / frac));
        b = std::min<int64_t>(b, (int64_t) todo.size() - pos);
        levels.resize(b);
        for (int64_t i = 0; i < b; i++) levels[i] = (uint8_t) level_for(ix->seed, ix->seq + i, m);
        // an element above the current entry level becomes the entry point: insert it alone; so does the first element
        // of a graph without an entry point (empty, or every element vacuumed away)
        if (ix->entry >= 0) {
            if (levels[0] > ix->entry_level) b = 1;
            else for (int64_t i = 1; i < b; i++) if (levels[i] > ix->entry_level) { b = i; break; }
        } else b = 1;
        levels.resize(b);

        // ---- rows into HBM at [cur, cur + b): normally already there (uploaded ahead, see below)
        rc = upload_upto((int64_t) pos + b);
        if (rc) return rc;
        HB_CK(cudaStreamWaitEvent(s, up_ev, 0));
        char *rows = ix->d_vecs + (size_t) cur * ix->row_bytes;

        auto tid_of = [&](int64_t i) { return heap_tids ? heap_tids[todo[pos + i]] : todo[pos + i]; };

        if (ix->entry < 0) {
            // first element of a graph without an entry point: slot cur (elements vacuumed away keep theirs), no
            // neighbours; it becomes the entry point
            const int lv = levels[0];
            const int64_t ur = ix->upper_rows;
            if (ur + lv > ix->upper_cap) {
                if (!ix->opt_auto_grow) { set_error("upper layer table full (%lld rows)", (long long) (ur + lv)); return HB_ENOMEM; }
                HB_CK(cudaStreamSynchronize(s));
                HB_CK(cudaStreamSynchronize(up));
                const int grc = hb_index_reserve(ix, ix->cap + ix->cap / 2 + 1024);
                if (grc) return grc;
                uploaded = (int64_t) pos;      // rows uploaded ahead lived in the old array: upload them again
                slot_base = ix->n - uploaded;
                continue;
            }
            const int64_t t0 = tid_of(0);
            const int32_t uo = lv > 0 ? (int32_t) ur : -1;
            const uint8_t one = 1;
            HB_CK(cudaMemcpyAsync(ix->d_uoff + cur, &uo, sizeof uo, cudaMemcpyHostToDevice, s));
            HB_CK(cudaMemcpyAsync(ix->d_tid0 + cur, &t0, sizeof t0, cudaMemcpyHostToDevice, s));
            HB_CK(cudaMemcpyAsync(ix->d_ntids + cur, &one, 1, cudaMemcpyHostToDevice, s));
            // stale lists and cached distances from a previous life of these rows
            HB_CK(cudaMemsetAsync(ix->d_nbr0 + (size_t) cur * m2, 0xff, sizeof(int32_t) * m2, s));
            HB_CK(cudaMemsetAsync(ix->d_nbr0d + (size_t) cur * m2, 0, sizeof(float) * m2, s));
            if (lv > 0) {
                HB_CK(cudaMemsetAsync(ix->d_nbru + (size_t) ur * m, 0xff, sizeof(int32_t) * (size_t) lv * m, s));
                HB_CK(cudaMemsetAsync(ix->d_nbrud + (size_t) ur * m, 0, sizeof(float) * (size_t) lv * m, s));
            }
            if (ix->d_pv0) HB_CK(cudaMemsetAsync(ix->d_pv0 + cur, 0, 1, s));
            if (ix->d_pvu && lv > 0) HB_CK(cudaMemsetAsync(ix->d_pvu + ur, 0, lv, s));
            HB_CK(cudaStreamSynchronize(s));
            ix->h_level.push_back((uint8_t) lv);
            ix->h_ntids.push_back(1);
            ix->h_tids.resize((size_t) (cur + 1) * HB_HEAPTIDS, 0);
            ix->h_tids[(size_t) cur * HB_HEAPTIDS] = t0;
            ix->n = cur + 1; ix->upper_rows = ur + lv;
            ix->entry = (int32_t) cur; ix->entry_level = lv; ix->seq += 1;
            ix->generation++;
            pos += 1; indexed += 1;
            continue;
        }
        // the candidate search starts at the entry point: it must be an element (a bad one would be read out of bounds)
        if (ix->entry >= cur || ix->entry_level < 0) {
            set_error("insert: entry point %d (level %d) is not an element of the %lld in the graph", ix->entry, ix->entry_level,
                      (long long) cur);
            return HB_EINVAL;
        }

        // ---- the batch's bookkeeping integers, assuming no tuple folds into a duplicate
        const int EL = ix->entry_level;
        ucand_row.assign(b, -1);
        int UR = 0;
        for (int64_t i = 0; i < b; i++) {
            const int l = std::min<int>(levels[i], EL);
            if (l > 0) { ucand_row[i] = UR; UR += l; }
        }
        const int UR1 = std::max(UR, 1);
        // host image of the packed words: ucand_row | final_id | new_uoff | dest_urow | urow_owner | urow_layer | tid | level
        const size_t pack_bytes = ((size_t) 3 * b + 3 * UR1) * 4 + 64 + (size_t) b * 8 + b + 16 * 8;
        pack.assign(pack_bytes, 0);
        char *hp = pack.data();
        int32_t *h_ucand = carve<int32_t>(hp, b);
        int32_t *h_final = carve<int32_t>(hp, b);
        int32_t *h_nuoff = carve<int32_t>(hp, b);
        int32_t *h_durow = carve<int32_t>(hp, UR1);
        int32_t *h_uown = carve<int32_t>(hp, UR1);
        int32_t *h_ulay = carve<int32_t>(hp, UR1);
        int64_t *h_tid = carve<int64_t>(hp, b);
        uint8_t *h_lev = carve<uint8_t>(hp, b);
        const size_t pack_used = (size_t) (hp - pack.data());
        int64_t urows = ix->upper_rows;
        for (int64_t i = 0; i < b; i++) {
            h_ucand[i] = ucand_row[i];
            h_final[i] = (int32_t) (cur + i);
            h_nuoff[i] = -1;
            h_tid[i] = tid_of(i);
            h_lev[i] = levels[i];
            if (levels[i] > 0) {
                h_nuoff[i] = (int32_t) urows;
                const int l = std::min<int>(levels[i], EL);
                for (int r = 0; r < l; r++) { h_durow[ucand_row[i] + r] = (int32_t) (urows + r); h_uown[ucand_row[i] + r] = (int32_t) i; h_ulay[ucand_row[i] + r] = r + 1; }
                urows += levels[i];
            }
        }
        if (UR == 0) h_durow[0] = -1;
        if (urows > ix->upper_cap) {
            // an unlucky run of level draws: more upper-layer rows than the n / (m - 1) expected ones
            if (!ix->opt_auto_grow) { set_error("upper layer table full (%lld rows)", (long long) urows); return HB_ENOMEM; }
            HB_CK(cudaStreamSynchronize(s));
            HB_CK(cudaStreamSynchronize(up));
            const int grc = hb_index_reserve(ix, ix->cap + ix->cap / 2 + 1024);
            if (grc) return grc;
            uploaded = (int64_t) pos;      // rows uploaded ahead lived in the old array: upload them again
            slot_base = ix->n - uploaded;
            continue;                      // form the batch again against the grown arrays
        }

        hb::DevBuf *W = ix->ws_build;
        const int64_t E = (int64_t) b * m2 + (int64_t) UR * m;
        rc = size_workspaces(b, UR1);
        if (rc) return rc;
        HB_CK(cudaMemcpyAsync(W[1].p, pack.data(), pack_used, cudaMemcpyHostToDevice, s));
        char *dp = W[1].as<char>();
        const int32_t *d_ucand = carve<int32_t>(dp, b);
        const int32_t *d_final = carve<int32_t>(dp, b);
        const int32_t *d_nuoff = carve<int32_t>(dp, b);
        const int32_t *d_durow = carve<int32_t>(dp, UR1);
        const int32_t *d_uown = carve<int32_t>(dp, UR1);
        const int32_t *d_ulay = carve<int32_t>(dp, UR1);
        const int64_t *d_tid = carve<int64_t>(dp, b);
        const uint8_t *d_lev = carve<uint8_t>(dp, b);
        // misc words: 0 work counter (fast) | 1 work counter (slow) | 2 slow count | 4 flag | 5 nseg | 6 valid edges | 7 lists to fill
        unsigned int *misc = ix->ws_misc.as<unsigned int>();
        HB_CK(cudaMemsetAsync(misc, 0, 32, s));
        int32_t *d_flag = reinterpret_cast<int32_t *>(misc + 4);
        int32_t *d_nseg = reinterpret_cast<int32_t *>(misc + 5);

        if (trace) cudaEventRecord(tev[0], s);
        // ---- candidate search
        BuildSearchParams sp;
        memset(&sp, 0, sizeof sp);
        sp.g = ix->view();
        sp.first = cur; sp.B = (int) b;
        sp.level = d_lev;
        sp.ucand_row = d_ucand;
        sp.efc = efc;
        sp.capW = ((efc + 16 + 3) / 4) * 4;
        {
            int slots = 1; while (slots < efc * 16) slots <<= 1;
            if (slots < 1024) slots = 1024;
            const size_t fixed = (size_t) ix->nvec * (ix->dtype == HB_F32 ? 4 : 8) * 4 + (size_t) sp.capW * 8 + 16 +
                                 (size_t) efc * 12 + (size_t) m2 * 8;
            // twice the table while the CTAs the register budget allows (launch bounds of build_search_kernel)
            // still fit shared memory: fewer searches spill into the overflow table in HBM
            const int ctas = ix->nvec == 32 ? 6 : 4;
            if (ix->opt_slots <= 0 && (fixed + (size_t) slots * 2 * 4) * BUILD_WARPS * ctas <= 216 * 1024) slots <<= 1;
            if (ix->opt_slots > 0) { slots = 1; while (slots < ix->opt_slots) slots <<= 1; }
            while (slots > 256 && (fixed + (size_t) slots * 4) * BUILD_WARPS > 200 * 1024) slots >>= 1;
            sp.slots = slots;
            sp.upper_slots = std::min(slots, 1024);
        }
        sp.cand0_id = W[3].as<int32_t>();
        sp.cand0_d = reinterpret_cast<float *>(sp.cand0_id + (size_t) b * efc);
        sp.cand0_cnt = reinterpret_cast<int32_t *>(sp.cand0_d + (size_t) b * efc);
        sp.candu_id = W[4].as<int32_t>();
        sp.candu_d = reinterpret_cast<float *>(sp.candu_id + (size_t) UR1 * efc);
        sp.candu_cnt = reinterpret_cast<int32_t *>(sp.candu_d + (size_t) UR1 * efc);
        sp.status = W[8].as<int32_t>();
        sp.slow_list = sp.status + b;
        sp.slow_count = reinterpret_cast<int32_t *>(misc + 2);
        sp.totals = ix->d_totals;
        sp.work = misc + 0;
        const int slow_grid = BUILD_SLOW_GRID;
        const int64_t slow_warps = (int64_t) slow_grid * BUILD_WARPS;
        sp.gwords = (int) ((cur + b + 31) / 32 + 1);
        sp.gcap = efc + HB_TIE_LIMIT;
        HB_CK(ix->ws_gbits.ensure(sizeof(uint32_t) * slow_warps * sp.gwords));
        HB_CK(ix->ws_gwd.ensure(sizeof(float) * slow_warps * sp.gcap));
        HB_CK(ix->ws_gwi.ensure(sizeof(uint32_t) * slow_warps * sp.gcap));
        sp.gbits = ix->ws_gbits.as<uint32_t>(); sp.gwd = ix->ws_gwd.as<float>(); sp.gwi = ix->ws_gwi.as<uint32_t>();
        sp.oslots = 4096;
        HB_CK(ix->ws_ovf.ensure(sizeof(uint32_t) * (size_t) ix->num_sms * MAX_CTAS_PER_SM * BUILD_WARPS * sp.oslots));
        sp.ovf = ix->ws_ovf.as<uint32_t>();
        // ---- neighbour selection: fused into the candidate search unless fused_select = 0
        BuildSelectParams lp;
        memset(&lp, 0, sizeof lp);
        lp.g = sp.g; lp.first = cur; lp.B = (int) b; lp.UR = UR; lp.efc = efc;
        lp.cand0_id = sp.cand0_id; lp.cand0_d = sp.cand0_d; lp.cand0_cnt = sp.cand0_cnt;
        lp.candu_id = sp.candu_id; lp.candu_d = sp.candu_d; lp.candu_cnt = sp.candu_cnt;
        lp.sel0_id = W[5].as<int32_t>();
        lp.sel0_d = reinterpret_cast<float *>(lp.sel0_id + (size_t) b * m2);
        lp.sel0_cnt = reinterpret_cast<int32_t *>(lp.sel0_d + (size_t) b * m2);
        lp.selu_id = W[6].as<int32_t>();
        lp.selu_d = reinterpret_cast<float *>(lp.selu_id + (size_t) UR1 * m);
        lp.selu_cnt = reinterpret_cast<int32_t *>(lp.selu_d + (size_t) UR1 * m);
        lp.dup = W[7].as<int32_t>();
        lp.totals = ix->d_totals;
        sp.fuse = ix->opt_fused_select;
        uint32_t *et_key = nullptr;
        float *et_val = nullptr;
        if (ix->opt_eval_table) {
            et_key = W[2].as<uint32_t>();
            et_val = reinterpret_cast<float *>(et_key + (size_t) b * et_slots);
            sp.el_id = reinterpret_cast<uint32_t *>(et_val + (size_t) b * et_slots);
            sp.el_d = reinterpret_cast<float *>(sp.el_id + (size_t) b * et_slots);
            sp.el_n = reinterpret_cast<int32_t *>(sp.el_d + (size_t) b * et_slots);
            sp.el_cap = et_slots / 2;            // a table is at most half full
            HB_CK(cudaMemsetAsync(et_key, 0xff, (size_t) b * et_slots * 4, s));
        }
        sp.sel0_id = lp.sel0_id; sp.sel0_d = lp.sel0_d; sp.sel0_cnt = lp.sel0_cnt;
        sp.selu_id = lp.selu_id; sp.selu_d = lp.selu_d; sp.selu_cnt = lp.selu_cnt; sp.dup = lp.dup;
        HB_CK(HB_PICK(build_search, ix)(sp, ix->num_sms, slow_grid, s, false));
        BuildSearchParams sps = sp;
        sps.work = misc + 1; sps.qlist = sp.slow_list; sps.qcount = sp.slow_count;
        HB_CK(HB_PICK(build_search, ix)(sps, ix->num_sms, slow_grid, s, true));

        if (et_key) {
            eval_table_build_kernel<<<(int) ((b * 32 + 255) / 256), 256, 0, s>>>(sp.el_id, sp.el_d, sp.el_n, sp.el_cap, (int) b, et_key,
                                                                                 et_val, et_slots);
            HB_CK(cudaGetLastError());
        }
        if (trace) cudaEventRecord(tev[1], s);
        if (!sp.fuse) HB_CK(HB_PICK(build_select, ix)(lp, ix->num_sms, s));
        build_check_kernel<<<(int) ((b + 255) / 256), 256, 0, s>>>(sp.status, lp.dup, (int) b, d_flag);
        HB_CK(cudaGetLastError());
        if (trace) cudaEventRecord(tev[2], s);

        // ---- the tail: AddConnections, reverse links.  Runs once when the no-duplicate assumption
        // held, a second time with the folded numbering otherwise.
        char *ep = W[9].as<char>();
        unsigned long long *key_in = carve<unsigned long long>(ep, E);
        unsigned long long *key_out = carve<unsigned long long>(ep, E);
        float *val_in = carve<float>(ep, E);
        float *val_out = carve<float>(ep, E);
        int32_t *seg_start = carve<int32_t>(ep, E);
        unsigned long long *fill_list = carve<unsigned long long>(ep, E);
        int32_t *d_nfill = reinterpret_cast<int32_t *>(misc + 7);
        int top_bit = 32 + LINK_KEY_SRC_BITS;
        for (int v = EL; v > 0; v >>= 1) top_bit++;
        size_t sort_bytes = 0;
        HB_CK(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, key_in, key_out, val_in, val_out, (int) E, 0, top_bit, s));
        HB_CK(W[10].ensure(sort_bytes + 16));

        auto run_tail = [&](int64_t next, int64_t urows_after) -> int {
            const int64_t nb_new = next - cur;
            if (nb_new <= 0) return HB_OK;
            // clean list rows for the new elements (an element above the old entry level has rows no search filled)
            HB_CK(cudaMemsetAsync(ix->d_nbr0 + (size_t) cur * m2, 0xff, sizeof(int32_t) * nb_new * m2, s));
            if (urows_after > ix->upper_rows)
                HB_CK(cudaMemsetAsync(ix->d_nbru + (size_t) ix->upper_rows * m, 0xff, sizeof(int32_t) * (urows_after - ix->upper_rows) * m, s));
            CommitParams cp;
            cp.B = (int) b; cp.UR = UR; cp.m = m;
            cp.final_id = d_final; cp.new_uoff = d_nuoff; cp.tid = d_tid; cp.dest_urow = d_durow;
            cp.sel0_id = lp.sel0_id; cp.sel0_d = lp.sel0_d; cp.selu_id = lp.selu_id; cp.selu_d = lp.selu_d;
            cp.nbr0 = ix->d_nbr0; cp.nbr0d = ix->d_nbr0d; cp.nbru = ix->d_nbru; cp.nbrud = ix->d_nbrud;
            cp.uoff = ix->d_uoff; cp.tid0 = ix->d_tid0; cp.ntids = ix->d_ntids;
            cp.pv0 = ix->d_pv0; cp.pvu = ix->d_pvu;
            cp.flag = d_flag;
            const int tgrid = (int) ((E + 255) / 256);
            build_commit_kernel<<<tgrid, 256, 0, s>>>(cp);
            HB_CK(cudaGetLastError());
            EdgeGenParams gp;
            gp.B = (int) b; gp.UR = UR; gp.m = m; gp.first = cur;
            gp.final_id = d_final; gp.urow_owner = d_uown; gp.urow_layer = d_ulay;
            gp.sel0_id = lp.sel0_id; gp.sel0_d = lp.sel0_d; gp.sel0_cnt = lp.sel0_cnt;
            gp.selu_id = lp.selu_id; gp.selu_d = lp.selu_d; gp.selu_cnt = lp.selu_cnt;
            gp.key = key_in; gp.val = val_in; gp.flag = d_flag;
            edge_gen_kernel<<<tgrid, 256, 0, s>>>(gp);
            HB_CK(cudaGetLastError());
            size_t sb = sort_bytes;
            HB_CK(cub::DeviceRadixSort::SortPairs(W[10].p, sb, key_in, key_out, val_in, val_out, (int) E, 0, top_bit, s));
            seg_heads_kernel<<<tgrid, 256, 0, s>>>(key_out, (int) E, seg_start, d_nseg, d_flag);
            HB_CK(cudaGetLastError());
            if (trace) cudaEventRecord(tev[3], s);
            LinkParams kp;
            memset(&kp, 0, sizeof kp);
            kp.g = ix->view();
            kp.g.n = next;
            kp.first = cur; kp.E = (int) E; kp.nseg = d_nseg; kp.seg_start = seg_start;
            kp.edge_key = key_out; kp.edge_d = val_out;
            kp.nbr0 = ix->d_nbr0; kp.nbr0d = ix->d_nbr0d; kp.nbru = ix->d_nbru; kp.nbrud = ix->d_nbrud;
            kp.totals = ix->d_totals; kp.flag = d_flag;
            kp.pc0 = ix->d_pc0; kp.pv0 = ix->d_pv0; kp.pcu = ix->d_pcu; kp.pvu = ix->d_pvu;
            // the tables are indexed by arrival order: usable only while ids = arrival order (no folded duplicates)
            if (et_key && next == cur + b) { kp.et_key = et_key; kp.et_val = et_val; kp.et_slots = et_slots; }
            if (ix->d_pc0 && (ix->opt_link_kernel == 0 || ix->opt_link_kernel == 3) && ix->opt_pair_fill) {
                // pair-cache fill pre-pass: triangles of the full, still unfilled lists this batch shrinks
                fill_list_kernel<<<tgrid, 256, 0, s>>>(key_out, seg_start, d_nseg, m, ix->d_nbr0, ix->d_uoff, ix->d_nbru,
                                                        ix->d_pv0, ix->d_pvu, fill_list, d_nfill, d_flag);
                HB_CK(cudaGetLastError());
                LinkParams fp = kp;
                fp.fill_list = fill_list; fp.nfill = d_nfill;
                const cudaError_t fe = HB_PICK(pair_fill, ix)(fp, ix->num_sms, (int) std::min<int64_t>(E, 2 * b + UR), s);
                if (fe != cudaSuccess && fe != cudaErrorInvalidConfiguration) HB_CK(fe);
            }
            HB_CK(HB_PICK(build_link, ix)(kp, ix->num_sms, ix->opt_link_kernel, s));
            return HB_OK;
        };

        rc = run_tail(cur + b, urows);
        if (rc) return rc;
        if (trace) cudaEventRecord(tev[4], s);
        HB_CK(cudaMemcpyAsync(ix->h_flag, d_flag, 12, cudaMemcpyDeviceToHost, s));
        // while the device works on this batch: the rows of the next one (at most ~cur/16 + a chunk ahead)
        rc = upload_upto((int64_t) pos + b + std::min<int64_t>(max_batch, (cur + b) / 8 + 1));
        if (rc) return rc;
        const double t1 = now();
        HB_CK(cudaStreamSynchronize(s));
        const double t2 = now();
        t_prep += t1 - t0; t_wait += t2 - t1;
        if (trace)
            for (int k = 0; k < 4; k++) {
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, tev[k], tev[k + 1]) == cudaSuccess) t_dev[k] += ms * 1e-3;
            }
        const int flag = ix->h_flag[0];
        n_segs += ix->h_flag[1]; n_edges += ix->h_flag[2];
        if (flag & 1) {
            set_error("insert: more than %d candidates tie exactly at the ef_construction boundary", HB_TIE_LIMIT);
            return HB_ELIMIT;
        }

        int64_t next = cur + b;
        std::vector<int32_t> dirty;
        if (flag & 2) {
            // FindDuplicateInMemory: fold a tuple into the first byte-identical neighbour with room
            dup.resize((size_t) b * DUP_SLOTS);
            HB_CK(cudaMemcpyAsync(dup.data(), lp.dup, sizeof(int32_t) * b * DUP_SLOTS, cudaMemcpyDeviceToHost, s));
            HB_CK(cudaStreamSynchronize(s));
            next = cur;
            urows = ix->upper_rows;
            for (int r = 0; r < UR1; r++) h_durow[r] = -1;
            bool any_fold = false;
            for (int64_t i = 0; i < b; i++) {
                int32_t into = -1;
                for (int k = 0; k < DUP_SLOTS; k++) {
                    const int32_t c = dup[i * DUP_SLOTS + k];
                    if (c < 0) break;
                    if (ix->h_ntids[c] < HB_HEAPTIDS) { into = c; break; }
                }
                h_nuoff[i] = -1;
                if (into >= 0) {
                    ix->h_tids[(size_t) into * HB_HEAPTIDS + ix->h_ntids[into]++] = tid_of(i);
                    dirty.push_back(into);
                    h_final[i] = -1;
                    any_fold = true;
                    continue;
                }
                h_final[i] = (int32_t) next++;
                if (levels[i] > 0) {
                    h_nuoff[i] = (int32_t) urows;
                    const int l = std::min<int>(levels[i], EL);
                    for (int r = 0; r < l; r++) h_durow[ucand_row[i] + r] = (int32_t) (urows + r);
                    urows += levels[i];
                }
            }
            if (any_fold && next > cur) {
                // close the gaps the folded tuples left in [cur, cur + b)
                HB_CK(ix->ws_build[11].ensure((size_t) b * ix->row_bytes));
                HB_CK(cudaMemcpyAsync(ix->ws_build[11].p, rows, (size_t) b * ix->row_bytes, cudaMemcpyDeviceToDevice, s));
                for (int64_t i = 0; i < b; i++)
                    if (h_final[i] >= 0 && h_final[i] != cur + i)
                        HB_CK(cudaMemcpyAsync(ix->d_vecs + (size_t) h_final[i] * ix->row_bytes,
                                              ix->ws_build[11].as<char>() + (size_t) i * ix->row_bytes, ix->row_bytes,
                                              cudaMemcpyDeviceToDevice, s));
            }
            HB_CK(cudaMemcpyAsync(W[1].p, pack.data(), pack_used, cudaMemcpyHostToDevice, s));
            HB_CK(cudaMemsetAsync(d_flag, 0, 16, s));     // flag, nseg, edge count, fill count
            rc = run_tail(next, urows);
            if (rc) return rc;
            HB_CK(cudaStreamSynchronize(s));
            if (next != cur + b) {
                // rows uploaded ahead sit at slots computed without the folds: re-base and upload again
                HB_CK(cudaStreamSynchronize(up));
                uploaded = (int64_t) pos + b;
                slot_base = next - uploaded;
            }
        }

        // ---- host mirrors
        for (int64_t i = 0; i < b; i++) {
            if (h_final[i] < 0) continue;
            ix->h_level.push_back(levels[i]);
            ix->h_ntids.push_back(1);
            ix->h_tids.resize(ix->h_tids.size() + HB_HEAPTIDS, 0);
            ix->h_tids[(size_t) h_final[i] * HB_HEAPTIDS] = tid_of(i);
            // entry point: the first element whose level exceeds the current entry level
            if (levels[i] > ix->entry_level) { ix->entry = h_final[i]; ix->entry_level = levels[i]; }
        }
        ix->n = next; ix->upper_rows = urows;
        ix->seq += b;
        ix->generation++;

        // heap TIDs of elements that absorbed a duplicate
        if (!dirty.empty()) {
            if (!ix->d_tidx) {
                HB_CK(cudaMalloc(&ix->d_tidx, sizeof(int64_t) * ix->cap * (HB_HEAPTIDS - 1)));
                HB_CK(cudaMemset(ix->d_tidx, 0, sizeof(int64_t) * ix->cap * (HB_HEAPTIDS - 1)));
                ix->has_dups = true;
            }
            for (int32_t c : dirty) {
                HB_CK(cudaMemcpy(ix->d_tidx + (size_t) c * (HB_HEAPTIDS - 1), &ix->h_tids[(size_t) c * HB_HEAPTIDS + 1],
                                 sizeof(int64_t) * (HB_HEAPTIDS - 1), cudaMemcpyHostToDevice));
                HB_CK(cudaMemcpy(ix->d_ntids + c, &ix->h_ntids[c], 1, cudaMemcpyHostToDevice));
                // slot 0 changes too when the element had been emptied by hb_bulk_delete
                HB_CK(cudaMemcpy(ix->d_tid0 + c, &ix->h_tids[(size_t) c * HB_HEAPTIDS], sizeof(int64_t), cudaMemcpyHostToDevice));
            }
        }
        pos += b;
        indexed += b;
        t_post += now() - t2;
    }
    if (trace) {
        fprintf(stderr, "[hb build] before the first batch: zero-vector scan %.3f s, build arrays %.3f s, workspaces %.3f s\n",
                t_todo - t_enter, t_arrays - t_todo, t_begin - t_arrays);
        fprintf(stderr, "[hb build] device time: search %.3f s, select %.3f s, commit+edges+sort %.3f s, link %.3f s\n",
                t_dev[0], t_dev[1], t_dev[2], t_dev[3]);
        for (auto &e : tev) cudaEventDestroy(e);
#ifdef HB_LINK_PROFILE
        unsigned long long t[16];
        cudaMemcpy(t, ix->d_totals, sizeof t, cudaMemcpyDeviceToHost);
        fprintf(stderr, "[hb build] evaluated-distance tables: %llu lookups, %llu misses\n", t[14], t[15]);
        fprintf(stderr, "[hb build] link pipeline, warp-cycles: consumers total %.3g = wait %.3g + tiles %.3g + finalize %.3g (of which extra edges %.3g; %llu finalizes); producer total %.3g, waiting for a free stage %.3g; finalize parts: sort %.3g masks %.3g select %.3g\n",
                (double) t[12], (double) t[6], (double) t[7], (double) t[8], (double) t[9], t[13], (double) t[11], (double) t[10],
                (double) t[14], (double) t[15], (double) t[5]);
#endif
    }
    if (trace)
        fprintf(stderr, "[hb build] %lld tuples in %lld batches: %.3f s total; host enqueue %.3f s, waiting for the device %.3f s, bookkeeping %.3f s; %lld reverse links in %lld (layer, target) segments\n",
                (long long) indexed, (long long) n_batches, now() - t_begin, t_prep, t_wait, t_post, (long long) n_edges, (long long) n_segs);
    return indexed;
}

}   // namespace hb
