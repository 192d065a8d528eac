// api.cu -- the C ABI (include/hnsw_b200.h): index handle, graph image in HBM, the scan path
// (ambeginscan / amrescan / amgettuple / amendscan and the batched extension), opclass support
// functions, partition routing and merge.  Host-side control only; all arithmetic on vectors
// happens in the kernels.  There is no CPU fallback: every entry point fails with HB_ECUDA when
// no device is present.
#include "index.h"
#include "scan_kernel.cuh"
#include "scan_reg.cuh"
#include "scan_cta.cuh"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>

namespace hb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

uint64_t splitmix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

// HnswGetMaxLevel / HnswInitElement [RECALL]: level = (int)(-log(U) * 1/ln(m)), capped by what a
// neighbour tuple can hold on an 8 kB page
static int max_level(int m)
{
    int v = (8192 - 24 - 8 - 8 - 4) / 6 / m - 2;
    return v > 255 ? 255 : (v < 0 ? 0 : v);
}

int level_for(uint64_t seed, int64_t seq, int m)
{
    const uint64_t r = splitmix64(seed ^ splitmix64((uint64_t) seq));
    const double u = ((double) (r >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    const double ml = 1.0 / log((double) m);
    const int level = (int) (-log(u) * ml);
    const int mx = max_level(m);
    return level > mx ? mx : level;
}

// ---- small kernels --------------------------------------------------------------------------

// l2_normalize in the canonical order: squared norm accumulated in double with the lane/slot
// pattern of distance.cuh, x / norm rounded to the storage type.  One warp per row.
template <typename T>
__global__ void normalize_kernel(const T *__restrict__ in, T *__restrict__ out, uint8_t *__restrict__ ok,
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
                acc[k] = acc[k] + x * x;   // the product is exact in double
            }
        }
    }
    double s;
    if constexpr (VEC == 4) s = (acc[0] + acc[1]) + (acc[2] + acc[3]);
    else s = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
    for (int b = 16; b >= 1; b >>= 1) s = s + __shfl_xor_sync(FULL, s, b);
    const double norm = sqrt(s);
    const bool good = norm > 0.0;
    T *dst = out + row * dim;
    for (int e = lane; e < dim; e += 32) {
        const float x = (float) src[e];
        const float y = good ? (float) ((double) x / norm) : x;
        dst[e] = (T) y;
    }
    if (ok && lane == 0) ok[row] = good ? 1 : 0;
}

// hnswgettuple's TID emission: elements nearest-first, each element's heap TIDs last-to-first
__global__ void elements_to_tids_kernel(const int32_t *__restrict__ elem, const float *__restrict__ dist,
                                        int64_t nq, int ef, int k, const int64_t *__restrict__ tid0,
                                        const uint8_t *__restrict__ ntids, const int64_t *__restrict__ tidx,
                                        int64_t *__restrict__ out_tids, float *__restrict__ out_dist,
                                        int32_t *__restrict__ out_cnt)
{
    const int64_t qi = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    int o = 0;
    for (int j = 0; j < ef && o < k; j++) {
        const int32_t e = elem[qi * ef + j];
        if (e < 0) break;
        const float d = dist[qi * ef + j];
        for (int t = (int) ntids[e] - 1; t >= 0 && o < k; t--) {
            out_tids[qi * k + o] = t == 0 ? tid0[e] : tidx[(int64_t) e * (HB_HEAPTIDS - 1) + (t - 1)];
            out_dist[qi * k + o] = d;
            o++;
        }
    }
    if (out_cnt) out_cnt[qi] = o;
    for (; o < k; o++) {
        out_tids[qi * k + o] = -1;
        out_dist[qi * k + o] = __int_as_float(0x7f800000);
    }
}

// merge P sorted lists of k into one of k; ties by (distance, partition)
__global__ void merge_topk_kernel(const int64_t *__restrict__ tids, const float *__restrict__ dist, int P,
                                  int64_t nq, int k, int64_t *__restrict__ out_tids, float *__restrict__ out_dist)
{
    const int64_t qi = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    constexpr int MAXP = 64;
    uint8_t head[MAXP];
    for (int p = 0; p < P; p++) head[p] = 0;
    for (int o = 0; o < k; o++) {
        int best = -1;
        float bd = __int_as_float(0x7f800000);
        for (int p = 0; p < P; p++) {
            if (head[p] >= k) continue;
            const int64_t off = ((int64_t) p * nq + qi) * k + head[p];
            if (tids[off] < 0) continue;
            const float d = dist[off];
            if (best < 0 || d < bd) { best = p; bd = d; }
        }
        if (best < 0) {
            out_tids[qi * k + o] = -1;
            out_dist[qi * k + o] = __int_as_float(0x7f800000);
        } else {
            const int64_t off = ((int64_t) best * nq + qi) * k + head[best];
            out_tids[qi * k + o] = tids[off];
            out_dist[qi * k + o] = bd;
            head[best]++;
        }
    }
}

// scan launchers (scan_<type>_<metric>.cu)
#define HB_DECL(name)                                                                                         \
    cudaError_t scan_fast_##name(const ScanParams &, int, int, cudaStream_t, ScanLaunchInfo *);               \
    cudaError_t scan_slow_##name(const ScanParams &, int, int, cudaStream_t, ScanLaunchInfo *);               \
    cudaError_t scan_reg_##name(const ScanParams &, int, int, int, cudaStream_t, ScanLaunchInfo *);           \
    cudaError_t scan_cta_##name(const ScanParams &, int, cudaStream_t);                                       \
    cudaError_t dist_##name(const DistBatchParams &, cudaStream_t);
HB_DECL(f32_l2) HB_DECL(f32_ip) HB_DECL(f16_l2) HB_DECL(f16_ip) HB_DECL(f32_l1) HB_DECL(f16_l1)
#undef HB_DECL

scan_launch_fn get_scan_launcher(int dtype, int kind, bool slow)
{
    static const scan_launch_fn tab[2][3][2] = {
        { { scan_fast_f32_l2, scan_slow_f32_l2 }, { scan_fast_f32_ip, scan_slow_f32_ip }, { scan_fast_f32_l1, scan_slow_f32_l1 } },
        { { scan_fast_f16_l2, scan_slow_f16_l2 }, { scan_fast_f16_ip, scan_slow_f16_ip }, { scan_fast_f16_l1, scan_slow_f16_l1 } } };
    return tab[dtype == HB_F32 ? 0 : 1][kind][slow ? 1 : 0];
}
scan_reg_launch_fn get_scan_reg_launcher(int dtype, int kind)
{
    static const scan_reg_launch_fn tab[2][3] = { { scan_reg_f32_l2, scan_reg_f32_ip, scan_reg_f32_l1 }, { scan_reg_f16_l2, scan_reg_f16_ip, scan_reg_f16_l1 } };
    return tab[dtype == HB_F32 ? 0 : 1][kind];
}
scan_cta_launch_fn get_scan_cta_launcher(int dtype, int kind)
{
    static const scan_cta_launch_fn tab[2][3] = { { scan_cta_f32_l2, scan_cta_f32_ip, scan_cta_f32_l1 }, { scan_cta_f16_l2, scan_cta_f16_ip, scan_cta_f16_l1 } };
    return tab[dtype == HB_F32 ? 0 : 1][kind];
}
dist_launch_fn get_dist_launcher(int dtype, int kind)
{
    static const dist_launch_fn tab[2][3] = { { dist_f32_l2, dist_f32_ip, dist_f32_l1 }, { dist_f16_l2, dist_f16_ip, dist_f16_l1 } };
    return tab[dtype == HB_F32 ? 0 : 1][kind];
}

constexpr int HB_OVERFLOW_SLOTS = 4096;
static size_t scan_warp_smem_bytes(const hb_index *ix, int capW, int slots)
{
    return ix->dtype == HB_F32 ? scan_warp_smem<float>(ix->nvec, capW, slots, false) : scan_warp_smem<__half>(ix->nvec, capW, slots, false);
}
int normalize_dev(hb_index *ix, const void *dev_in, int64_t n, void *dev_out, cudaStream_t s)
{
    const int wpb = 8;
    const int grid = (int) ((n + wpb - 1) / wpb);
    if (ix->dtype == HB_F32)
        normalize_kernel<float><<<grid, wpb * 32, 0, s>>>((const float *) dev_in, (float *) dev_out, nullptr, n, ix->dim);
    else
        normalize_kernel<__half><<<grid, wpb * 32, 0, s>>>((const __half *) dev_in, (__half *) dev_out, nullptr, n, ix->dim);
    HB_CK(cudaGetLastError());
    return HB_OK;
}

static int pow2ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }

// upload n rows of dim components into the padded row layout
static int upload_rows(hb_index *ix, int64_t first, const void *host, int64_t n, cudaStream_t s)
{
    const size_t src_row = (size_t) ix->dim * ix->esize;
    char *dst = ix->d_vecs + (size_t) first * ix->row_bytes;
    if (src_row == ix->row_bytes) {
        HB_CK(cudaMemcpyAsync(dst, host, src_row * n, cudaMemcpyHostToDevice, s));
    } else {
        HB_CK(cudaMemsetAsync(dst, 0, ix->row_bytes * n, s));
        HB_CK(cudaMemcpy2DAsync(dst, ix->row_bytes, host, src_row, src_row, n, cudaMemcpyHostToDevice, s));
    }
    return HB_OK;
}

}   // namespace hb

using namespace hb;

// =============================================================================================
extern "C" {

const char *hb_last_error(void) { return g_err; }
const char *hb_version(void) { return "hnsw_b200 0.1 (sm_100a)"; }

int hb_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        return HB_ECUDA;
    }
    return n;
}

static int index_alloc(hb_index *ix)
{
    const int64_t cap = ix->cap;
    const int m2 = 2 * ix->m;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaMalloc(&ix->d_vecs, (size_t) cap * ix->row_bytes));
    HB_CK(cudaMalloc(&ix->d_nbr0, sizeof(int32_t) * cap * m2));
    HB_CK(cudaMalloc(&ix->d_uoff, sizeof(int32_t) * cap));
    ix->upper_cap = cap / (ix->m > 2 ? ix->m - 1 : 1) + cap / 16 + 1024;   // E[rows] = cap / (m - 1)
    HB_CK(cudaMalloc(&ix->d_nbru, sizeof(int32_t) * ix->upper_cap * ix->m));
    HB_CK(cudaMalloc(&ix->d_tid0, sizeof(int64_t) * cap));
    HB_CK(cudaMalloc(&ix->d_ntids, cap));
    HB_CK(cudaMalloc(&ix->d_totals, sizeof(unsigned long long) * 16));
    HB_CK(cudaMemset(ix->d_totals, 0, sizeof(unsigned long long) * 16));
    HB_CK(cudaMemset(ix->d_nbr0, 0xff, sizeof(int32_t) * cap * m2));
    HB_CK(cudaMemset(ix->d_nbru, 0xff, sizeof(int32_t) * ix->upper_cap * ix->m));
    HB_CK(cudaMemset(ix->d_uoff, 0xff, sizeof(int32_t) * cap));
    HB_CK(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    HB_CK(cudaEventCreate(&ix->ev0));
    HB_CK(cudaEventCreate(&ix->ev1));
    cudaDeviceProp prop;
    HB_CK(cudaGetDeviceProperties(&prop, ix->device));
    ix->num_sms = prop.multiProcessorCount;
    return HB_OK;
}

hb_index *hb_index_create(int device, int dim, int m, int efc, int metric, int dtype, int64_t capacity,
                          uint64_t seed)
{
    if (dim < 1 || dim > (dtype == HB_F16 ? HB_MAX_DIM_HALF : HB_MAX_DIM) || m < 2 || m > 100 || efc < 4 || efc > 1000 || efc < 2 * m ||
        metric < HB_L2 || metric > HB_L1 || (dtype != HB_F32 && dtype != HB_F16) || capacity < 1 ||
        capacity > 0x7ffffff0LL) {
        set_error("hb_index_create: invalid parameters (dim=%d m=%d ef_construction=%d metric=%d dtype=%d capacity=%lld)",
                  dim, m, efc, metric, dtype, (long long) capacity);
        return nullptr;
    }
    int ndev = hb_device_count();
    if (ndev <= 0 || device < 0 || device >= ndev) {
        if (ndev >= 0) set_error("hb_index_create: no CUDA device %d (found %d); there is no CPU fallback", device, ndev);
        return nullptr;
    }
    hb_index *ix = new hb_index();
    ix->device = device; ix->dim = dim; ix->m = m; ix->efc = efc; ix->metric = metric; ix->dtype = dtype;
    ix->esize = dtype == HB_F32 ? 4 : 2;
    const int vec = dtype == HB_F32 ? 4 : 8;
    ix->nvec = (dim + vec - 1) / vec;
    ix->row_bytes = (size_t) ix->nvec * 16;
    ix->cap = capacity; ix->seed = seed;
    if (index_alloc(ix) != HB_OK) { hb_index_free(ix); return nullptr; }
    return ix;
}

void hb_index_free(hb_index *ix)
{
    if (!ix) return;
    cudaSetDevice(ix->device);
    bruteforce_release(ix);
    cudaFree(ix->d_vecs); cudaFree(ix->d_nbr0); cudaFree(ix->d_nbr0d); cudaFree(ix->d_uoff);
    cudaFree(ix->d_nbru); cudaFree(ix->d_nbrud); cudaFree(ix->d_tid0); cudaFree(ix->d_ntids);
    cudaFree(ix->d_tidx); cudaFree(ix->d_totals);
    hb::release_pair_cache(ix);
    hb::DevBuf *bufs[] = { &ix->ws_q, &ix->ws_qn, &ix->ws_elem, &ix->ws_dist, &ix->ws_status, &ix->ws_misc,
                           &ix->ws_gbits, &ix->ws_gwd, &ix->ws_gwi, &ix->ws_ovf };
    for (auto b : bufs) b->release();
    for (auto &w : ix->slot_ws) if (w) { w->release(); delete w; w = nullptr; }
    for (auto &kv : ix->stream_ws) { kv.second->release(); delete kv.second; }
    ix->stream_ws.clear();
    for (auto &b : ix->ws_build) b.release();
    if (ix->h_flag) cudaFreeHost(ix->h_flag);
    if (ix->up_event) cudaEventDestroy(ix->up_event);
    if (ix->up_stream) cudaStreamDestroy(ix->up_stream);
    if (ix->ev0) cudaEventDestroy(ix->ev0);
    if (ix->ev1) cudaEventDestroy(ix->ev1);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
}

int64_t hb_index_size(const hb_index *ix) { return ix ? ix->n : HB_EINVAL; }
int64_t hb_index_upper_rows(const hb_index *ix) { return ix ? ix->upper_rows : HB_EINVAL; }

int hb_index_entry(const hb_index *ix, int32_t *entry, int *entry_level)
{
    if (!ix) return HB_EINVAL;
    if (entry) *entry = ix->entry;
    if (entry_level) *entry_level = ix->entry_level;
    return HB_OK;
}

int hb_set_option(hb_index *ix, const char *name, int value)
{
    if (!ix || !name) return HB_EINVAL;
    if (!strcmp(name, "slots")) ix->opt_slots = value;
    else if (!strcmp(name, "grid")) ix->opt_grid = value;
    else if (!strcmp(name, "build_batch")) ix->opt_build_batch = value;
    else if (!strcmp(name, "per_query_counters")) ix->opt_per_query = value;
    else if (!strcmp(name, "variant")) {
        if (!is_scan_variant(value)) { set_error("hb_set_option: variant %d is not one of 0, 6, 7, 9, 17, 27", value); return HB_EINVAL; }
        ix->opt_variant = value;
    }
    else if (!strcmp(name, "link_kernel")) ix->opt_link_kernel = value;
    else if (!strcmp(name, "pair_cache")) ix->opt_pair_cache = value;
    else if (!strcmp(name, "pair_fill")) ix->opt_pair_fill = value;
    else if (!strcmp(name, "eval_table")) ix->opt_eval_table = value;
    else if (!strcmp(name, "build_fraction")) ix->opt_build_fraction = value > 0 ? value : 16;
    else if (!strcmp(name, "build_fraction_small")) ix->opt_build_fraction_small = value > 0 ? value : 0;
    else if (!strcmp(name, "auto_grow")) ix->opt_auto_grow = value;
    else if (!strcmp(name, "vacuum_batch")) ix->opt_vacuum_batch = value;
    else { set_error("hb_set_option: unknown option %s", name); return HB_EINVAL; }
    return HB_OK;
}

// grow one device array: new allocation, fill pattern, old contents copied, old array freed
extern "C++" {
template <typename V> int grow_array(V *&p, size_t old_used, size_t new_count, int fill)
{
    if (!p) return HB_OK;
    V *q = nullptr;
    HB_CK(cudaMalloc(&q, sizeof(V) * new_count));
    HB_CK(cudaMemset(q, fill, sizeof(V) * new_count));
    if (old_used) HB_CK(cudaMemcpy(q, p, sizeof(V) * old_used, cudaMemcpyDeviceToDevice));
    cudaFree(p);
    p = q;
    return HB_OK;
}
}   // extern "C++"

int hb_index_reserve(hb_index *ix, int64_t capacity)
{
    if (!ix || capacity < 1 || capacity > 0x7ffffff0LL) { set_error("hb_index_reserve: bad argument"); return HB_EINVAL; }
    if (capacity <= ix->cap) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaDeviceSynchronize());
    const int m = ix->m, m2 = 2 * m;
    const int64_t n = ix->n, ur = ix->upper_rows;
    const int64_t ucap = std::max<int64_t>(ix->upper_cap, capacity / (m > 2 ? m - 1 : 1) + capacity / 16 + 1024);
    const size_t tri0 = (size_t) m2 * (m2 - 1) / 2, triu = (size_t) m * (m - 1) / 2;
    int rc;
    {
        char *q = nullptr;
        HB_CK(cudaMalloc(&q, (size_t) capacity * ix->row_bytes));
        if (n) HB_CK(cudaMemcpy(q, ix->d_vecs, (size_t) n * ix->row_bytes, cudaMemcpyDeviceToDevice));
        cudaFree(ix->d_vecs);
        ix->d_vecs = q;
    }
    if ((rc = grow_array(ix->d_nbr0, (size_t) n * m2, (size_t) capacity * m2, 0xff))) return rc;
    if ((rc = grow_array(ix->d_uoff, (size_t) n, (size_t) capacity, 0xff))) return rc;
    if ((rc = grow_array(ix->d_nbru, (size_t) ur * m, (size_t) ucap * m, 0xff))) return rc;
    if ((rc = grow_array(ix->d_tid0, (size_t) n, (size_t) capacity, 0))) return rc;
    if ((rc = grow_array(ix->d_ntids, (size_t) n, (size_t) capacity, 0))) return rc;
    if ((rc = grow_array(ix->d_tidx, (size_t) n * (HB_HEAPTIDS - 1), (size_t) capacity * (HB_HEAPTIDS - 1), 0))) return rc;
    if ((rc = grow_array(ix->d_nbr0d, (size_t) n * m2, (size_t) capacity * m2, 0))) return rc;
    if ((rc = grow_array(ix->d_nbrud, (size_t) ur * m, (size_t) ucap * m, 0))) return rc;
    if ((rc = grow_array(ix->d_pc0, (size_t) n * tri0, (size_t) capacity * tri0, 0))) return rc;
    if ((rc = grow_array(ix->d_pcu, (size_t) ur * triu, (size_t) ucap * triu, 0))) return rc;
    if ((rc = grow_array(ix->d_pv0, (size_t) n, (size_t) capacity, 0))) return rc;
    if ((rc = grow_array(ix->d_pvu, (size_t) ur, (size_t) ucap, 0))) return rc;
    ix->cap = capacity;
    ix->upper_cap = ucap;
    return HB_OK;
}

int hb_index_trim(hb_index *ix)
{
    if (!ix) return HB_EINVAL;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaDeviceSynchronize());
    // everything only inserts use: cached neighbour distances, the pair cache, batch workspaces.  A later
    // hb_insert allocates them again (cached distances are recomputed, the pair cache refills lazily).
    if (ix->d_nbr0d) { cudaFree(ix->d_nbr0d); ix->d_nbr0d = nullptr; }
    if (ix->d_nbrud) { cudaFree(ix->d_nbrud); ix->d_nbrud = nullptr; }
    hb::release_pair_cache(ix);
    for (auto &b : ix->ws_build) b.release();
    ix->ws_gbits.release(); ix->ws_gwd.release(); ix->ws_gwi.release(); ix->ws_ovf.release();
    return HB_OK;
}

int hb_level_for(uint64_t seed, int64_t seq, int m) { return m >= 2 ? level_for(seed, seq, m) : HB_EINVAL; }

int hb_set_build_batch(hb_index *ix, int max_batch) { return hb_set_option(ix, "build_batch", max_batch); }

// ---- tids on the device --------------------------------------------------------------------
static int sync_tids_to_device(hb_index *ix, int64_t first, int64_t n)
{
    if (n <= 0) return HB_OK;
    std::vector<int64_t> t0(n);
    bool dups = ix->has_dups;
    for (int64_t i = 0; i < n; i++) {
        t0[i] = ix->h_tids[(first + i) * HB_HEAPTIDS];
        if (ix->h_ntids[first + i] > 1) dups = true;
    }
    HB_CK(cudaMemcpy(ix->d_tid0 + first, t0.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice));
    HB_CK(cudaMemcpy(ix->d_ntids + first, ix->h_ntids.data() + first, n, cudaMemcpyHostToDevice));
    if (dups) {
        if (!ix->d_tidx) {
            HB_CK(cudaMalloc(&ix->d_tidx, sizeof(int64_t) * ix->cap * (HB_HEAPTIDS - 1)));
            first = 0; n = ix->n;   // first time: upload everything
        }
        std::vector<int64_t> tx((size_t) n * (HB_HEAPTIDS - 1));
        for (int64_t i = 0; i < n; i++)
            memcpy(&tx[i * (HB_HEAPTIDS - 1)], &ix->h_tids[(first + i) * HB_HEAPTIDS + 1], sizeof(int64_t) * (HB_HEAPTIDS - 1));
        HB_CK(cudaMemcpy(ix->d_tidx + first * (HB_HEAPTIDS - 1), tx.data(), sizeof(int64_t) * tx.size(), cudaMemcpyHostToDevice));
        ix->has_dups = true;
    }
    return HB_OK;
}


// ---- ambulkdelete, first pass -----------------------------------------------------------------
// hnswvacuum.c RemoveHeapTids [RECALL]: dead heap TIDs leave their elements; an element left without TIDs
// stays in the graph as a routing node and returns nothing.  Graph repair (RepairGraph / MarkDeleted: new
// neighbours for elements that pointed at emptied ones, slot reuse) is not implemented.
int64_t hb_bulk_delete(hb_index *ix, const int64_t *dead_tids, int64_t n_dead)
{
    if (!ix || (!dead_tids && n_dead > 0) || n_dead < 0) { set_error("hb_bulk_delete: bad argument"); return HB_EINVAL; }
    if (n_dead == 0 || ix->n == 0) return 0;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaDeviceSynchronize());
    std::vector<int64_t> dead(dead_tids, dead_tids + n_dead);
    std::sort(dead.begin(), dead.end());
    int64_t removed = 0, lo = -1, hi = -1;
    for (int64_t e = 0; e < ix->n; e++) {
        int64_t *t = &ix->h_tids[(size_t) e * HB_HEAPTIDS];
        const int nt = ix->h_ntids[e];
        int w = 0;
        for (int k = 0; k < nt; k++)
            if (!std::binary_search(dead.begin(), dead.end(), t[k])) t[w++] = t[k];
        if (w != nt) {
            for (int k = w; k < HB_HEAPTIDS; k++) t[k] = 0;
            ix->h_ntids[e] = (uint8_t) w;
            removed += nt - w;
            if (lo < 0) lo = e;
            hi = e;
        }
    }
    if (removed > 0) {
        ix->generation++;
        const int rc = sync_tids_to_device(ix, lo, hi - lo + 1);
        if (rc) return rc;
    }
    return removed;
}

// ---- graph image ---------------------------------------------------------------------------
int hb_index_load(hb_index *ix, int64_t n, int64_t upper_rows, int32_t entry, const void *vecs,
                  const uint8_t *level, const int32_t *nbr0, const int32_t *uoff, const int32_t *nbru,
                  const uint8_t *ntids, const int64_t *tids)
{
    if (!ix || n < 0 || !vecs || !level || !nbr0 || !uoff || (upper_rows > 0 && !nbru)) {
        set_error("hb_index_load: NULL argument");
        return HB_EINVAL;
    }
    if ((n > ix->cap || upper_rows > ix->upper_cap) && ix->opt_auto_grow) {
        int64_t want = std::max<int64_t>(n, ix->cap);
        const int mm = ix->m > 2 ? ix->m - 1 : 1;
        while (want / mm + want / 16 + 1024 < upper_rows) want += want / 2 + 1024;     // upper_cap follows the capacity
        if (want == ix->cap) want = ix->cap + 1;
        const int grc = hb_index_reserve(ix, want);
        if (grc) return grc;
    }
    if (n > ix->cap || upper_rows > ix->upper_cap) {
        set_error("hb_index_load: graph (%lld elements, %lld upper rows) exceeds capacity", (long long) n, (long long) upper_rows);
        return HB_ENOMEM;
    }
    if (n > 0 && (entry < -1 || entry >= n)) { set_error("hb_index_load: entry point %d is not an element (n = %lld)", entry, (long long) n); return HB_EINVAL; }
    // no entry point with elements present: what vacuum leaves when it removed every element; only then
    if (n > 0 && entry < 0) {
        for (int64_t e = 0; e < n; e++)
            if (!ntids || ntids[e] > 0) {
                set_error("hb_index_load: no entry point, but element %lld holds heap TIDs", (long long) e);
                return HB_EINVAL;
            }
    }
    for (int64_t i = 0; i < n * 2 * ix->m; i++)
        if (nbr0[i] < -1 || nbr0[i] >= n) { set_error("hb_index_load: layer-0 neighbour id %d out of range", nbr0[i]); return HB_EINVAL; }
    for (int64_t i = 0; i < upper_rows * ix->m; i++)
        if (nbru[i] < -1 || nbru[i] >= n) { set_error("hb_index_load: upper-layer neighbour id %d out of range", nbru[i]); return HB_EINVAL; }
    for (int64_t e = 0; e < n; e++)
        if (uoff[e] < -1 || (level[e] > 0 && (uoff[e] < 0 || (int64_t) uoff[e] + level[e] > upper_rows))) {
            set_error("hb_index_load: element %lld: upper rows [%d, +%d) out of range", (long long) e, uoff[e], (int) level[e]);
            return HB_EINVAL;
        }
    HB_CK(cudaSetDevice(ix->device));
    int rc = upload_rows(ix, 0, vecs, n, 0);
    if (rc) return rc;
    HB_CK(cudaMemcpy(ix->d_nbr0, nbr0, sizeof(int32_t) * n * 2 * ix->m, cudaMemcpyHostToDevice));
    HB_CK(cudaMemcpy(ix->d_uoff, uoff, sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    if (upper_rows > 0)
        HB_CK(cudaMemcpy(ix->d_nbru, nbru, sizeof(int32_t) * upper_rows * ix->m, cudaMemcpyHostToDevice));
    ix->n = n; ix->seq = n; ix->upper_rows = upper_rows;
    ix->generation++;
    ix->entry = n > 0 ? entry : -1;
    ix->entry_level = ix->entry >= 0 ? level[ix->entry] : -1;
    ix->h_level.assign(level, level + n);
    ix->h_ntids.assign(n, 1);
    ix->h_deleted.clear();
    if (ntids) ix->h_ntids.assign(ntids, ntids + n);
    ix->h_tids.assign((size_t) n * HB_HEAPTIDS, 0);
    for (int64_t i = 0; i < n; i++) {
        if (tids) memcpy(&ix->h_tids[i * HB_HEAPTIDS], tids + i * HB_HEAPTIDS, sizeof(int64_t) * HB_HEAPTIDS);
        else ix->h_tids[i * HB_HEAPTIDS] = i;
    }
    // cached neighbour distances are unknown for a loaded graph; build.cu recomputes on demand
    if (ix->d_nbr0d) { cudaFree(ix->d_nbr0d); ix->d_nbr0d = nullptr; }
    if (ix->d_nbrud) { cudaFree(ix->d_nbrud); ix->d_nbrud = nullptr; }
    hb::release_pair_cache(ix);
    HB_CK(cudaDeviceSynchronize());
    return sync_tids_to_device(ix, 0, n);
}

int hb_index_export(const hb_index *ix, void *vecs, uint8_t *level, int32_t *nbr0, int32_t *uoff,
                    int32_t *nbru, uint8_t *ntids, int64_t *tids)
{
    if (!ix) return HB_EINVAL;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaDeviceSynchronize());
    const int64_t n = ix->n;
    if (vecs && n)
        HB_CK(cudaMemcpy2D(vecs, (size_t) ix->dim * ix->esize, ix->d_vecs, ix->row_bytes, (size_t) ix->dim * ix->esize, n,
                           cudaMemcpyDeviceToHost));
    if (level && n) memcpy(level, ix->h_level.data(), n);
    if (nbr0 && n) HB_CK(cudaMemcpy(nbr0, ix->d_nbr0, sizeof(int32_t) * n * 2 * ix->m, cudaMemcpyDeviceToHost));
    if (uoff && n) HB_CK(cudaMemcpy(uoff, ix->d_uoff, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    if (nbru && ix->upper_rows)
        HB_CK(cudaMemcpy(nbru, ix->d_nbru, sizeof(int32_t) * ix->upper_rows * ix->m, cudaMemcpyDeviceToHost));
    if (ntids && n) memcpy(ntids, ix->h_ntids.data(), n);
    if (tids && n) memcpy(tids, ix->h_tids.data(), sizeof(int64_t) * n * HB_HEAPTIDS);
    return HB_OK;
}

// ---- build / insert --------------------------------------------------------------------------
int64_t hb_build(hb_index *ix, const void *host_vecs, int64_t n, const int64_t *heap_tids)
{
    if (!ix || (!host_vecs && n > 0) || n < 0) { set_error("hb_build: bad argument"); return HB_EINVAL; }
    if (ix->n != 0) { set_error("hb_build: index is not empty (use hb_insert)"); return HB_ESTATE; }
    return build_insert(ix, host_vecs, n, heap_tids);
}

int64_t hb_insert(hb_index *ix, const void *host_vecs, int64_t n, const int64_t *heap_tids)
{
    if (!ix || (!host_vecs && n > 0) || n < 0) { set_error("hb_insert: bad argument"); return HB_EINVAL; }
    return build_insert(ix, host_vecs, n, heap_tids);
}

// ---- scan ------------------------------------------------------------------------------------
static int choose_slots(const hb_index *ix, int ef, int capW)
{
    // ~5-15 distance evaluations per unit of ef is typical.  At least 16*ef slots; more (up to 64*ef)
    // while a warp's shared memory stays within ~12 kB, so that 16 warps fit an SM; heavier queries
    // spill into the per-warp overflow table in HBM.
    const size_t fixed = (size_t) ix->nvec * (ix->dtype == HB_F32 ? 4 : 8) * 4 + (size_t) capW * 8 + 16;
    int slots;
    if (ix->opt_slots > 0) slots = (ix->opt_slots + 15) & ~15;          // any multiple of 16 (the home slot is a mulhi, not a mask)
    else {
        slots = std::max(1024, pow2ceil(ef * 16));
        const int cap = pow2ceil(ef * 64);
        while (slots < cap && fixed + (size_t) slots * 2 * 4 <= 12288) slots <<= 1;
    }
    if (slots < 64) slots = 64;
    // keep SCAN_WARPS warps within 200 kB of shared memory
    while (slots > 256 && (fixed + (size_t) slots * 4) * SCAN_WARPS > 200 * 1024) slots >>= 1;
    return slots;
}

static ScanWs *ws_for_stream(hb_index *ix, cudaStream_t s)
{
    auto it = ix->stream_ws.find((void *) s);
    if (it != ix->stream_ws.end()) return it->second;
    ScanWs *ws = new ScanWs();
    if (cudaEventCreate(&ws->ev0) != cudaSuccess || cudaEventCreate(&ws->ev1) != cudaSuccess ||
        cudaMallocHost(&ws->h_err, 64) != cudaSuccess) { delete ws; return nullptr; }
    ix->stream_ws[(void *) s] = ws;
    return ws;
}

static ScanWs *ws_for_slot(hb_index *ix, int slot)
{
    if (slot < 0 || slot >= ASYNC_SLOTS) return nullptr;
    if (ix->slot_ws[slot]) return ix->slot_ws[slot];
    ScanWs *ws = new ScanWs();
    if (cudaStreamCreateWithFlags(&ws->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ws->ev0) != cudaSuccess || cudaEventCreate(&ws->ev1) != cudaSuccess ||
        cudaMallocHost(&ws->h_err, 64) != cudaSuccess) { delete ws; return nullptr; }
    ix->slot_ws[slot] = ws;
    return ws;
}

// normalise queries on the device when the opclass is cosine; returns the pointer to scan with
static int prepare_queries(hb_index *ix, ScanWs &ws, const void *dev_q, int64_t nq, cudaStream_t s, const void **out)
{
    if (ix->metric != HB_COSINE) { *out = dev_q; return HB_OK; }
    HB_CK(ws.qn.ensure((size_t) nq * ix->dim * ix->esize));
    const int wpb = 8;
    const int grid = (int) ((nq + wpb - 1) / wpb);
    if (ix->dtype == HB_F32)
        normalize_kernel<float><<<grid, wpb * 32, 0, s>>>((const float *) dev_q, ws.qn.as<float>(), nullptr, nq, ix->dim);
    else
        normalize_kernel<__half><<<grid, wpb * 32, 0, s>>>((const __half *) dev_q, ws.qn.as<__half>(), nullptr, nq, ix->dim);
    HB_CK(cudaGetLastError());
    *out = ws.qn.p;
    return HB_OK;
}

static int scan_dev(hb_index *ix, ScanWs &ws, const void *dev_queries, int64_t nq, int ef, int32_t *out_elem, float *out_dist,
                    int32_t *out_cnt, cudaStream_t s, const int32_t *dev_ep, int nep, int layer)
{
    if (ef < 1 || ef > 1000) { set_error("hnsw.ef_search must be in [1,1000] (got %d)", ef); return HB_EINVAL; }
    if (nq <= 0) return HB_OK;
    if (nq > 0x7fffffff) { set_error("too many queries in one batch"); return HB_EINVAL; }
    HB_CK(cudaSetDevice(ix->device));
    const void *q = nullptr;
    int rc = prepare_queries(ix, ws, dev_queries, nq, s, &q);
    if (rc) return rc;

    ScanParams p;
    memset(&p, 0, sizeof p);
    p.g = ix->view();
    p.queries = q;
    p.nq = nq;
    p.ef = ef;
    p.capW = ((std::max(ef, nep) + 16 + 3) / 4) * 4;
    p.slots = choose_slots(ix, ef, p.capW);
    const int regR = reg_list_R(ix->nvec, ef, dev_ep, ix->opt_variant);
    if (regR && ix->opt_slots <= 0) {
        // register-list kernel, one warp per CTA: the visited table is what fills shared memory.  Size it so that 24
        // (128-d) / 16 (256-d) one-warp CTAs are resident per SM (each CTA also costs 1 kB of reserved shared memory)
        const int warps = ix->nvec <= 32 ? 24 : 16;
        const size_t per_cta = (size_t) 233472 / warps - 1024;
        const size_t fixed = (size_t) ix->nvec * (ix->dtype == HB_F32 ? 4 : 8) * 4 + 128 + 16;
        int sl = (int) ((per_cta - fixed) / 4) & ~15;
        sl = std::min(sl, pow2ceil(ef * 64));
        if (sl >= 256) p.slots = sl;
    }
    p.upper_slots = std::min(p.slots, 1024);
    p.out_elem = out_elem; p.out_dist = out_dist; p.out_cnt = out_cnt;
    p.out_stride = std::max(ef, nep);
    p.ep = dev_ep; p.nep = nep; p.layer = layer;
    p.variant = ix->opt_variant;

    HB_CK(ws.status.ensure(sizeof(int32_t) * nq));
    HB_CK(ws.slow.ensure(sizeof(int32_t) * nq));
    HB_CK(ws.misc.ensure(256));
    p.status = ws.status.as<int32_t>();
    p.slow_list = ws.slow.as<int32_t>();
    unsigned int *misc = ws.misc.as<unsigned int>();   // [0] work fast, [1] work slow, [2] slow_count
    p.slow_count = reinterpret_cast<int32_t *>(misc + 2);
    p.err = reinterpret_cast<int32_t *>(misc + 3);
    p.totals = ix->d_totals;
    if (ix->opt_per_query) {
        HB_CK(ws.pq.ensure(sizeof(int32_t) * 4 * nq));
        p.per_query = ws.pq.as<int32_t>();
    }
    HB_CK(cudaMemsetAsync(misc, 0, 16, s));

    // slow-path scratch: a bitmap of n bits and a long W list per resident warp
    const int slow_grid = 32;
    const int64_t slow_warps = (int64_t) slow_grid * SCAN_WARPS;
    p.gwords = (int) ((ix->n + 31) / 32 + 1);
    p.gcap = std::max(ef, nep) + HB_TIE_LIMIT;
    HB_CK(ws.gbits.ensure(sizeof(uint32_t) * slow_warps * p.gwords));
    HB_CK(ws.gwd.ensure(sizeof(float) * slow_warps * p.gcap));
    HB_CK(ws.gwi.ensure(sizeof(uint32_t) * slow_warps * p.gcap));
    p.gbits = ws.gbits.as<uint32_t>();
    p.gwd = ws.gwd.as<float>();
    p.gwi = ws.gwi.as<uint32_t>();

    // per-warp visited overflow tables for the fast path (one slice per resident warp; the launcher
    // keeps at most MAX_CTAS_PER_SM CTAs per SM resident)
    // Sized for the searches shared memory cannot hold: 64 slots per unit of ef_search (4096 .. 32768), so
    // that data on which a scan visits thousands of elements (iid high-dimensional rows: ~36 evaluations
    // per unit of ef) stays on the fast path instead of falling to the bitmap path.
    {
        int os = HB_OVERFLOW_SLOTS;
        while (os < ef * 64 && os < 32768) os <<= 1;
        p.oslots = os;
        // one slice per warp that can be resident: an upper bound from the smaller of the two kernels' per-warp
        // shared memory (the launchers clamp their grids to MAX_CTAS_PER_SM * SCAN_WARPS warps per SM)
        const size_t warp_smem = scan_warp_smem_bytes(ix, p.capW, p.slots) - (size_t) p.capW * 8;
        int warps = (int) std::min<size_t>((size_t) MAX_CTAS_PER_SM * SCAN_WARPS, (228 * 1024) / std::max<size_t>(warp_smem, 1));
        if (warps < SCAN_WARPS) warps = SCAN_WARPS;
        HB_CK(ws.ovf.ensure(sizeof(uint32_t) * (size_t) ix->num_sms * warps * p.oslots));
    }
    p.ovf = ws.ovf.as<uint32_t>();

    const int ip = metric_kind(ix->metric);
    HB_CK(cudaEventRecord(ws.ev0, s));
    p.work = misc + 0;
    ScanLaunchInfo info;
    const size_t qsmem = (size_t) ix->nvec * (ix->dtype == HB_F32 ? 4 : 8) * 4;
    if (use_cta_scan(p, ix->num_sms, qsmem, dev_ep, ix->opt_variant)) HB_CK(get_scan_cta_launcher(ix->dtype, ip)(p, ix->num_sms, s));
    else if (regR) HB_CK(get_scan_reg_launcher(ix->dtype, ip)(p, regR, ix->num_sms, ix->opt_grid, s, &info));
    else HB_CK(get_scan_launcher(ix->dtype, ip, false)(p, ix->num_sms, ix->opt_grid, s, &info));
    // queries whose tie tail (or overflow table) outgrew the fast path run again with a bitmap in HBM
    ScanParams ps = p;
    ps.work = misc + 1;
    ps.qlist = p.slow_list;
    ps.qcount = p.slow_count;
    HB_CK(get_scan_launcher(ix->dtype, ip, true)(ps, ix->num_sms, slow_grid, s, nullptr));
    HB_CK(cudaEventRecord(ws.ev1, s));
    ws.timing_valid = true;
    ix->last_ws = &ws;
    return HB_OK;
}

static int check_status(hb_index *ix, ScanWs &ws, int64_t nq, cudaStream_t s)
{
    (void) ix; (void) nq;
    HB_CK(cudaMemcpyAsync(ws.h_err, ws.misc.as<int32_t>() + 3, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    HB_CK(cudaStreamSynchronize(s));
    if (*ws.h_err) {
        set_error("a query has more than %d candidates tying exactly at the ef boundary", HB_TIE_LIMIT);
        return HB_ELIMIT;
    }
    return HB_OK;
}

int hb_search_batch_dev(hb_index *ix, const void *dev_queries, int64_t nq, int ef, int32_t *dev_out_elem,
                        float *dev_out_dist, int32_t *dev_out_cnt, void *stream)
{
    if (!ix || !dev_queries || !dev_out_elem || !dev_out_dist || !dev_out_cnt) { set_error("hb_search_batch_dev: NULL argument"); return HB_EINVAL; }
    ScanWs *ws = ws_for_stream(ix, (cudaStream_t) stream);
    if (!ws) { set_error("hb_search_batch_dev: cannot create the stream workspace"); return HB_ECUDA; }
    return scan_dev(ix, *ws, dev_queries, nq, ef, dev_out_elem, dev_out_dist, dev_out_cnt, (cudaStream_t) stream, nullptr, 0, 0);
}

// the error word of the last hb_search_batch_dev on `stream` (the device API cannot fail asynchronously otherwise):
// waits for the stream, HB_ELIMIT when a query of that batch exceeded HB_TIE_LIMIT boundary ties (its count is 0)
int hb_search_batch_status(hb_index *ix, void *stream)
{
    if (!ix) { set_error("hb_search_batch_status: NULL index"); return HB_EINVAL; }
    auto it = ix->stream_ws.find(stream);
    if (it == ix->stream_ws.end() || !it->second->misc.p) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    return check_status(ix, *it->second, 0, (cudaStream_t) stream);
}

int hb_search_batch_elements(hb_index *ix, const void *host_queries, int64_t nq, int ef, int32_t *out_elem,
                             float *out_dist, int32_t *out_cnt)
{
    if (!ix || !host_queries || !out_elem || !out_dist) { set_error("hb_search_batch_elements: NULL argument"); return HB_EINVAL; }
    if (ef < 1 || ef > 1000) { set_error("hnsw.ef_search must be in [1,1000] (got %d)", ef); return HB_EINVAL; }
    if (nq > 0x7fffffff) { set_error("too many queries in one batch"); return HB_EINVAL; }
    if (nq <= 0) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    ScanWs *wsp = ws_for_slot(ix, 0);
    if (!wsp) { set_error("cannot create the scan workspace"); return HB_ECUDA; }
    ScanWs &ws = *wsp;
    if (ws.pending) { set_error("hb_search_batch_elements: slot 0 still has a batch in flight"); return HB_ESTATE; }
    cudaStream_t s = ws.own_stream;
    const size_t qbytes = (size_t) nq * ix->dim * ix->esize;
    const size_t obytes = (size_t) nq * ef * 8 + (size_t) nq * 4;
    HB_CK(ws.q.ensure(qbytes));
    if (qbytes + obytes <= (256 << 10)) {
        // small call (one backend's amgettuple): the caller's pageable buffers would make every copy a
        // synchronous one; stage through pinned memory instead -- one H2D, one D2H, one synchronisation
        if (!ws.h_pin) { HB_CK(cudaMallocHost(&ws.h_pin, 512 << 10)); ws.h_pin_cap = 512 << 10; }
        HB_CK(ws.pack.ensure(obytes));
        memcpy(ws.h_pin, host_queries, qbytes);
        HB_CK(cudaMemcpyAsync(ws.q.p, ws.h_pin, qbytes, cudaMemcpyHostToDevice, s));
        int32_t *d_elem = ws.pack.as<int32_t>();
        float *d_dist = reinterpret_cast<float *>(d_elem + (size_t) nq * ef);
        int32_t *d_cnt = reinterpret_cast<int32_t *>(d_dist + (size_t) nq * ef);
        int rc = scan_dev(ix, ws, ws.q.p, nq, ef, d_elem, d_dist, d_cnt, s, nullptr, 0, 0);
        if (rc) return rc;
        char *h_out = ws.h_pin + qbytes;
        HB_CK(cudaMemcpyAsync(h_out, ws.pack.p, obytes, cudaMemcpyDeviceToHost, s));
        rc = check_status(ix, ws, nq, s);
        if (rc) return rc;
        memcpy(out_elem, h_out, (size_t) nq * ef * 4);
        memcpy(out_dist, h_out + (size_t) nq * ef * 4, (size_t) nq * ef * 4);
        if (out_cnt) memcpy(out_cnt, h_out + (size_t) nq * ef * 8, (size_t) nq * 4);
        return HB_OK;
    }
    HB_CK(ws.elem.ensure(sizeof(int32_t) * nq * ef));
    HB_CK(ws.dist.ensure(sizeof(float) * nq * ef));
    HB_CK(ws.cnt.ensure(sizeof(int32_t) * nq));
    HB_CK(cudaMemcpyAsync(ws.q.p, host_queries, qbytes, cudaMemcpyHostToDevice, s));
    int rc = scan_dev(ix, ws, ws.q.p, nq, ef, ws.elem.as<int32_t>(), ws.dist.as<float>(), ws.cnt.as<int32_t>(), s, nullptr, 0, 0);
    if (rc) return rc;
    HB_CK(cudaMemcpyAsync(out_elem, ws.elem.p, sizeof(int32_t) * nq * ef, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaMemcpyAsync(out_dist, ws.dist.p, sizeof(float) * nq * ef, cudaMemcpyDeviceToHost, s));
    if (out_cnt) HB_CK(cudaMemcpyAsync(out_cnt, ws.cnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, s));
    return check_status(ix, ws, nq, s);
}

int hb_elements_to_tids_dev(hb_index *ix, const int32_t *dev_elem, const float *dev_dist, int64_t nq, int ef, int k,
                            int64_t *dev_out_tids, float *dev_out_dist, void *stream)
{
    if (!ix || !dev_elem || !dev_dist || !dev_out_tids || !dev_out_dist || k < 1) { set_error("hb_elements_to_tids_dev: bad argument"); return HB_EINVAL; }
    if (nq <= 0) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    elements_to_tids_kernel<<<(int) ((nq + 127) / 128), 128, 0, (cudaStream_t) stream>>>(
        dev_elem, dev_dist, nq, ef, k, ix->d_tid0, ix->d_ntids, ix->d_tidx, dev_out_tids, dev_out_dist, nullptr);
    HB_CK(cudaGetLastError());
    return HB_OK;
}

// host buffers in / out, asynchronous: H2D, scan, TID mapping and D2H are queued on the slot's own
// stream; hb_search_batch_wait() completes the call.  Up to ASYNC_SLOTS batches can be in flight,
// so copies of one batch overlap the scan of another and one batch's tail overlaps the next one's
// ramp.  The host buffers must stay valid (and, to overlap, be pinned) until the wait.
int hb_search_batch_async(hb_index *ix, int slot, const void *host_queries, int64_t nq, int ef, int k, int64_t *out_tids,
                          float *out_dist, int32_t *out_cnt)
{
    if (!ix || !host_queries || !out_tids || !out_dist || k < 1) { set_error("hb_search_batch: bad argument"); return HB_EINVAL; }
    if (ef < 1 || ef > 1000) { set_error("hnsw.ef_search must be in [1,1000] (got %d)", ef); return HB_EINVAL; }
    if (nq > 0x7fffffff) { set_error("too many queries in one batch"); return HB_EINVAL; }
    HB_CK(cudaSetDevice(ix->device));
    ScanWs *wsp = ws_for_slot(ix, slot);
    if (!wsp) { set_error("hb_search_batch_async: bad slot %d (0..%d)", slot, ASYNC_SLOTS - 1); return HB_EINVAL; }
    ScanWs &ws = *wsp;
    if (ws.pending) { set_error("hb_search_batch_async: slot %d still has a batch in flight", slot); return HB_ESTATE; }
    if (nq <= 0) return HB_OK;
    cudaStream_t s = ws.own_stream;
    HB_CK(ws.q.ensure((size_t) nq * ix->dim * ix->esize));
    HB_CK(ws.elem.ensure(sizeof(int32_t) * nq * ef));
    HB_CK(ws.dist.ensure(sizeof(float) * nq * ef));
    HB_CK(ws.cnt.ensure(sizeof(int32_t) * nq));
    HB_CK(ws.tids.ensure(sizeof(int64_t) * nq * k));
    HB_CK(ws.tdist.ensure(sizeof(float) * nq * k));
    HB_CK(cudaMemcpyAsync(ws.q.p, host_queries, (size_t) nq * ix->dim * ix->esize, cudaMemcpyHostToDevice, s));
    int rc = scan_dev(ix, ws, ws.q.p, nq, ef, ws.elem.as<int32_t>(), ws.dist.as<float>(), ws.cnt.as<int32_t>(), s, nullptr, 0, 0);
    if (rc) return rc;
    elements_to_tids_kernel<<<(int) ((nq + 127) / 128), 128, 0, s>>>(ws.elem.as<int32_t>(), ws.dist.as<float>(), nq, ef, k,
                                                                      ix->d_tid0, ix->d_ntids, ix->d_tidx, ws.tids.as<int64_t>(),
                                                                      ws.tdist.as<float>(), ws.cnt.as<int32_t>());
    HB_CK(cudaGetLastError());
    HB_CK(cudaMemcpyAsync(out_tids, ws.tids.p, sizeof(int64_t) * nq * k, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaMemcpyAsync(out_dist, ws.tdist.p, sizeof(float) * nq * k, cudaMemcpyDeviceToHost, s));
    if (out_cnt) HB_CK(cudaMemcpyAsync(out_cnt, ws.cnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaMemcpyAsync(ws.h_err, ws.misc.as<int32_t>() + 3, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    ws.pending = true;
    ws.pending_nq = nq;
    return HB_OK;
}

int hb_search_batch_wait(hb_index *ix, int slot)
{
    if (!ix || slot < 0 || slot >= ASYNC_SLOTS) { set_error("hb_search_batch_wait: bad argument"); return HB_EINVAL; }
    ScanWs *wsp = ix->slot_ws[slot];
    if (!wsp || !wsp->pending) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaStreamSynchronize(wsp->own_stream));
    wsp->pending = false;
    if (*wsp->h_err) {
        set_error("a query has more than %d candidates tying exactly at the ef boundary", HB_TIE_LIMIT);
        return HB_ELIMIT;
    }
    return HB_OK;
}

int hb_search_batch(hb_index *ix, const void *host_queries, int64_t nq, int ef, int k, int64_t *out_tids,
                    float *out_dist, int32_t *out_cnt)
{
    if (!ix || !host_queries || !out_tids || !out_dist || k < 1) { set_error("hb_search_batch: bad argument"); return HB_EINVAL; }
    if (ef < 1 || ef > 1000) { set_error("hnsw.ef_search must be in [1,1000] (got %d)", ef); return HB_EINVAL; }
    const size_t qbytes = nq > 0 ? (size_t) nq * ix->dim * ix->esize : 0;
    const size_t obytes = nq > 0 ? (size_t) nq * k * 12 + (size_t) nq * 4 : 0;
    if (nq > 0 && qbytes + obytes <= (256 << 10)) {
        // small call: stage through pinned memory (see hb_search_batch_elements) -- one H2D, one D2H, one wait
        HB_CK(cudaSetDevice(ix->device));
        ScanWs *wsp = ws_for_slot(ix, 0);
        if (!wsp) { set_error("cannot create the scan workspace"); return HB_ECUDA; }
        ScanWs &ws = *wsp;
        if (ws.pending) { set_error("hb_search_batch: slot 0 still has a batch in flight"); return HB_ESTATE; }
        cudaStream_t s = ws.own_stream;
        if (!ws.h_pin) { HB_CK(cudaMallocHost(&ws.h_pin, 512 << 10)); ws.h_pin_cap = 512 << 10; }
        HB_CK(ws.q.ensure(qbytes));
        HB_CK(ws.elem.ensure(sizeof(int32_t) * nq * ef));
        HB_CK(ws.dist.ensure(sizeof(float) * nq * ef));
        HB_CK(ws.pack.ensure(obytes + 16));
        memcpy(ws.h_pin, host_queries, qbytes);
        HB_CK(cudaMemcpyAsync(ws.q.p, ws.h_pin, qbytes, cudaMemcpyHostToDevice, s));
        int64_t *d_tids = ws.pack.as<int64_t>();
        float *d_tdist = reinterpret_cast<float *>(d_tids + (size_t) nq * k);
        int32_t *d_cnt = reinterpret_cast<int32_t *>(d_tdist + (size_t) nq * k);
        int rc = scan_dev(ix, ws, ws.q.p, nq, ef, ws.elem.as<int32_t>(), ws.dist.as<float>(), d_cnt, s, nullptr, 0, 0);
        if (rc) return rc;
        elements_to_tids_kernel<<<(int) ((nq + 127) / 128), 128, 0, s>>>(ws.elem.as<int32_t>(), ws.dist.as<float>(), nq, ef, k,
                                                                          ix->d_tid0, ix->d_ntids, ix->d_tidx, d_tids, d_tdist, d_cnt);
        HB_CK(cudaGetLastError());
        char *h_out = ws.h_pin + qbytes;
        HB_CK(cudaMemcpyAsync(h_out, ws.pack.p, obytes, cudaMemcpyDeviceToHost, s));
        rc = check_status(ix, ws, nq, s);
        if (rc) return rc;
        memcpy(out_tids, h_out, (size_t) nq * k * 8);
        memcpy(out_dist, h_out + (size_t) nq * k * 8, (size_t) nq * k * 4);
        if (out_cnt) memcpy(out_cnt, h_out + (size_t) nq * k * 12, (size_t) nq * 4);
        return HB_OK;
    }
    int rc = hb_search_batch_async(ix, 0, host_queries, nq, ef, k, out_tids, out_dist, out_cnt);
    if (rc) return rc;
    return hb_search_batch_wait(ix, 0);
}

int hb_search_layer(hb_index *ix, const void *host_queries, int64_t nq, const int32_t *ep, int nep, int ef, int layer,
                    int32_t *out_elem, float *out_dist, int32_t *out_cnt)
{
    if (!ix || !host_queries || !ep || nep < 1 || nep > ef || !out_elem || !out_dist || layer < 0) {
        set_error("hb_search_layer: bad argument (need 1 <= nep <= ef)");
        return HB_EINVAL;
    }
    if (nq <= 0) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    ScanWs *wsp = ws_for_slot(ix, 0);
    if (!wsp) { set_error("cannot create the scan workspace"); return HB_ECUDA; }
    ScanWs &ws = *wsp;
    cudaStream_t s = ws.own_stream;
    const int stride = std::max(ef, nep);
    HB_CK(ws.q.ensure((size_t) nq * ix->dim * ix->esize));
    HB_CK(ws.ep.ensure(sizeof(int32_t) * nq * nep));
    HB_CK(ws.elem.ensure(sizeof(int32_t) * nq * stride));
    HB_CK(ws.dist.ensure(sizeof(float) * nq * stride));
    HB_CK(ws.cnt.ensure(sizeof(int32_t) * nq));
    HB_CK(cudaMemcpyAsync(ws.q.p, host_queries, (size_t) nq * ix->dim * ix->esize, cudaMemcpyHostToDevice, s));
    HB_CK(cudaMemcpyAsync(ws.ep.p, ep, sizeof(int32_t) * nq * nep, cudaMemcpyHostToDevice, s));
    int rc = scan_dev(ix, ws, ws.q.p, nq, ef, ws.elem.as<int32_t>(), ws.dist.as<float>(), ws.cnt.as<int32_t>(), s,
                      ws.ep.as<int32_t>(), nep, layer);
    if (rc) return rc;
    HB_CK(cudaMemcpyAsync(out_elem, ws.elem.p, sizeof(int32_t) * nq * stride, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaMemcpyAsync(out_dist, ws.dist.p, sizeof(float) * nq * stride, cudaMemcpyDeviceToHost, s));
    if (out_cnt) HB_CK(cudaMemcpyAsync(out_cnt, ws.cnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, s));
    return check_status(ix, ws, nq, s);
}

int hb_get_counters(hb_index *ix, hb_counters *out, int reset)
{
    if (!ix || !out) return HB_EINVAL;
    HB_CK(cudaSetDevice(ix->device));
    unsigned long long t[16];
    HB_CK(cudaDeviceSynchronize());
    HB_CK(cudaMemcpy(t, ix->d_totals, sizeof t, cudaMemcpyDeviceToHost));
    out->n_dist = (int64_t) t[0]; out->n_hop0 = (int64_t) t[1]; out->n_hopu = (int64_t) t[2];
    out->n_slow = (int64_t) t[3]; out->n_pair = (int64_t) t[4];
    if (reset) HB_CK(cudaMemset(ix->d_totals, 0, sizeof t));
    return HB_OK;
}

int hb_get_per_query_counters(hb_index *ix, int64_t nq, int32_t *out)
{
    if (!ix || !out || !ix->last_ws || !ix->last_ws->pq.p) { set_error("per-query counters are not enabled (hb_set_option per_query_counters 1)"); return HB_ESTATE; }
    HB_CK(cudaSetDevice(ix->device));
    HB_CK(cudaDeviceSynchronize());
    HB_CK(cudaMemcpy(out, ix->last_ws->pq.p, sizeof(int32_t) * 4 * nq, cudaMemcpyDeviceToHost));
    return HB_OK;
}

float hb_last_search_ms(const hb_index *ix)
{
    if (!ix || !ix->last_ws || !ix->last_ws->timing_valid) return -1.f;
    float ms = -1.f;
    cudaSetDevice(ix->device);
    if (cudaEventSynchronize(ix->last_ws->ev1) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, ix->last_ws->ev0, ix->last_ws->ev1) != cudaSuccess) return -1.f;
    return ms;
}

// ---- scan handle: ambeginscan / amrescan / amgettuple / amendscan ---------------------------
hb_scan *hb_beginscan(hb_index *ix)
{
    if (!ix) { set_error("hb_beginscan: NULL index"); return nullptr; }
    hb_scan *sc = new hb_scan();
    sc->ix = ix;
    return sc;
}

int hb_scan_set_iterative(hb_scan *sc, int mode, int64_t max_scan_tuples)
{
    if (!sc || mode < HB_ITER_OFF || mode > HB_ITER_STRICT || max_scan_tuples < 1) {
        set_error("hb_scan_set_iterative: bad argument");
        return HB_EINVAL;
    }
    sc->iter_mode = mode;
    sc->max_scan_tuples = max_scan_tuples;
    return HB_OK;
}

int hb_rescan(hb_scan *sc, const void *host_query, int ef)
{
    if (!sc || !host_query) { set_error("hb_rescan: NULL argument"); return HB_EINVAL; }
    if (ef < 1 || ef > 1000) { set_error("hnsw.ef_search must be in [1,1000] (got %d)", ef); return HB_EINVAL; }
    const size_t b = (size_t) sc->ix->dim * sc->ix->esize;
    sc->query.assign((const char *) host_query, (const char *) host_query + b);
    sc->ef = ef; sc->bound = true; sc->fetched = false; sc->cnt = 0; sc->pos = 0; sc->tid_pos = -1;
    if (sc->iter) { hb_iter_end(sc->iter); sc->iter = nullptr; }
    sc->have_prev = false;
    return HB_OK;
}

int hb_gettuple(hb_scan *sc, int64_t *heap_tid, float *distance)
{
    if (!sc || !heap_tid) { set_error("hb_gettuple: NULL argument"); return HB_EINVAL; }
    if (!sc->bound) { set_error("hb_gettuple: cannot scan hnsw index without order (no hb_rescan)"); return HB_ESTATE; }
    hb_index *ix = sc->ix;
    for (;;) {
        if (!sc->fetched || (sc->pos >= sc->cnt && sc->iter)) {
            // first call: GetScanItems; later, with hnsw.iterative_scan on: ResumeScanItems
            if (!sc->fetched && ix->n == 0) { sc->fetched = true; sc->cnt = 0; return 0; }
            sc->elem.resize(sc->ef); sc->dist.resize(sc->ef);
            int32_t cnt = 0;
            if (sc->iter_mode == HB_ITER_OFF) {
                int rc = hb_search_batch_elements(ix, sc->query.data(), 1, sc->ef, sc->elem.data(), sc->dist.data(), &cnt);
                if (rc) return rc;
            } else {
                if (!sc->iter) {
                    sc->iter = hb_iter_begin(ix, sc->query.data(), 1, sc->ef, sc->max_scan_tuples);
                    if (!sc->iter) return HB_ECUDA;
                }
                const int64_t got = hb_iter_next(sc->iter, sc->elem.data(), sc->dist.data(), &cnt);
                if (got < 0) return (int) got;
                if (got == 0) { hb_iter_end(sc->iter); sc->iter = nullptr; }
            }
            sc->cnt = cnt; sc->pos = 0; sc->tid_pos = -1; sc->fetched = true;
        }
        while (sc->pos < sc->cnt) {
            const int32_t e = sc->elem[sc->pos];
            if (sc->tid_pos < 0) sc->tid_pos = ix->h_ntids[e];
            if (sc->tid_pos > 0) {
                const float d = sc->dist[sc->pos];
                sc->tid_pos--;
                const int64_t tid = ix->h_tids[(int64_t) e * HB_HEAPTIDS + sc->tid_pos];
                if (sc->tid_pos == 0) { sc->pos++; sc->tid_pos = -1; }
                if (sc->iter_mode == HB_ITER_STRICT) {
                    if (sc->have_prev && d < sc->prev_dist) continue;       // out of order: dropped
                    sc->prev_dist = d; sc->have_prev = true;
                }
                *heap_tid = tid;
                if (distance) *distance = d;
                return 1;
            }
            sc->pos++; sc->tid_pos = -1;
        }
        if (!sc->iter) return 0;
    }
}

void hb_endscan(hb_scan *sc)
{
    if (!sc) return;
    if (sc->iter) hb_iter_end(sc->iter);
    delete sc;
}

// ---- opclass support functions ---------------------------------------------------------------
int hb_distance_batch(hb_index *ix, const void *host_queries, int64_t nq, const int32_t *cand, int nc, float *out)
{
    if (!ix || !host_queries || !cand || !out || nc < 1) { set_error("hb_distance_batch: bad argument"); return HB_EINVAL; }
    if (nq <= 0) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    HB_CK(ix->ws_q.ensure((size_t) nq * ix->dim * ix->esize));
    HB_CK(ix->ws_elem.ensure(sizeof(int32_t) * nq * nc));
    HB_CK(ix->ws_dist.ensure(sizeof(float) * nq * nc));
    HB_CK(cudaMemcpyAsync(ix->ws_q.p, host_queries, (size_t) nq * ix->dim * ix->esize, cudaMemcpyHostToDevice, s));
    HB_CK(cudaMemcpyAsync(ix->ws_elem.p, cand, sizeof(int32_t) * nq * nc, cudaMemcpyHostToDevice, s));
    const void *q = nullptr;
    ScanWs *wsp = ws_for_slot(ix, 0);
    if (!wsp) { set_error("cannot create the scan workspace"); return HB_ECUDA; }
    int rc = prepare_queries(ix, *wsp, ix->ws_q.p, nq, s, &q);
    if (rc) return rc;
    DistBatchParams p;
    p.g = ix->view(); p.queries = q; p.nq = nq; p.cand = ix->ws_elem.as<int32_t>(); p.nc = nc; p.out = ix->ws_dist.as<float>();
    HB_CK(get_dist_launcher(ix->dtype, metric_kind(ix->metric))(p, s));
    HB_CK(cudaMemcpyAsync(out, ix->ws_dist.p, sizeof(float) * nq * nc, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaStreamSynchronize(s));
    return HB_OK;
}

int hb_distance_batch_dev(hb_index *ix, const void *dev_queries, int64_t nq, const int32_t *dev_cand, int nc, float *dev_out,
                          void *stream)
{
    if (!ix || !dev_queries || !dev_cand || !dev_out || nc < 1) { set_error("hb_distance_batch_dev: bad argument"); return HB_EINVAL; }
    if (nq <= 0) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    DistBatchParams p;
    p.g = ix->view(); p.queries = dev_queries; p.nq = nq; p.cand = dev_cand; p.nc = nc; p.out = dev_out;
    HB_CK(get_dist_launcher(ix->dtype, metric_kind(ix->metric))(p, (cudaStream_t) stream));
    return HB_OK;
}

int hb_normalize(hb_index *ix, const void *host_in, int64_t n, void *host_out, uint8_t *ok)
{
    if (!ix || !host_in || !host_out) { set_error("hb_normalize: NULL argument"); return HB_EINVAL; }
    if (n <= 0) return HB_OK;
    HB_CK(cudaSetDevice(ix->device));
    cudaStream_t s = ix->stream;
    const size_t bytes = (size_t) n * ix->dim * ix->esize;
    HB_CK(ix->ws_q.ensure(bytes));
    HB_CK(ix->ws_qn.ensure(bytes));
    HB_CK(ix->ws_status.ensure(n));
    HB_CK(cudaMemcpyAsync(ix->ws_q.p, host_in, bytes, cudaMemcpyHostToDevice, s));
    const int wpb = 8, grid = (int) ((n + wpb - 1) / wpb);
    if (ix->dtype == HB_F32)
        normalize_kernel<float><<<grid, wpb * 32, 0, s>>>(ix->ws_q.as<float>(), ix->ws_qn.as<float>(), ix->ws_status.as<uint8_t>(), n, ix->dim);
    else
        normalize_kernel<__half><<<grid, wpb * 32, 0, s>>>(ix->ws_q.as<__half>(), ix->ws_qn.as<__half>(), ix->ws_status.as<uint8_t>(), n, ix->dim);
    HB_CK(cudaGetLastError());
    HB_CK(cudaMemcpyAsync(host_out, ix->ws_qn.p, bytes, cudaMemcpyDeviceToHost, s));
    if (ok) HB_CK(cudaMemcpyAsync(ok, ix->ws_status.p, n, cudaMemcpyDeviceToHost, s));
    HB_CK(cudaStreamSynchronize(s));
    return HB_OK;
}

// ---- partitions -------------------------------------------------------------------------------
int hb_partition_of(int64_t id, int n_partitions)
{
    if (n_partitions < 1) return HB_EINVAL;
    return (int) (splitmix64((uint64_t) id) % (uint64_t) n_partitions);
}

void hb_partition_route(const int64_t *ids, int64_t n, int n_partitions, int32_t *out_part)
{
    for (int64_t i = 0; i < n; i++) out_part[i] = hb_partition_of(ids[i], n_partitions);
}

int hb_merge_topk_dev(int device, const int64_t *dev_tids, const float *dev_dist, int n_parts, int64_t nq, int k,
                      int64_t *dev_out_tids, float *dev_out_dist, void *stream)
{
    if (!dev_tids || !dev_dist || !dev_out_tids || !dev_out_dist || n_parts < 1 || n_parts > 64 || k < 1 || k > 255) {
        set_error("hb_merge_topk_dev: bad argument (1 <= partitions <= 64, 1 <= k <= 255)");
        return HB_EINVAL;
    }
    if (nq <= 0) return HB_OK;
    HB_CK(cudaSetDevice(device));
    merge_topk_kernel<<<(int) ((nq + 127) / 128), 128, 0, (cudaStream_t) stream>>>(dev_tids, dev_dist, n_parts, nq, k, dev_out_tids,
                                                                                  dev_out_dist);
    HB_CK(cudaGetLastError());
    return HB_OK;
}

}   // extern "C"
